#!/usr/bin/env python
"""Triangular-multiplication measurement: B <- alpha op(A) B (Left) / alpha B op(A) (Right) through
dlaf_b200_triangular_multiplication_d with HOST buffers (the C entry's contract), the device time inside it, and cuBLAS
Dtrmm on device-resident data of the same shape (tools/cublas_trmm_ref). Flop model of the reference's miniapp
(miniapp_triangular_multiplication.cpp:141-144): m^2 n (Left) / m n^2 (Right) for real types. One JSON line, with the card
name and power limit read in the same run.
usage: python tools/bench_trmm.py [--n 16384] [--nrhs 16384] [--nb 512] [--side L --uplo L --op N]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=16384)
    ap.add_argument("--nrhs", type=int, default=16384)
    ap.add_argument("--nb", type=int, default=512)
    ap.add_argument("--side", default="L")
    ap.add_argument("--uplo", default="L")
    ap.add_argument("--op", default="N")
    ap.add_argument("--steps", type=int, default=3)
    a = ap.parse_args()
    import torch

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True).stdout.strip().splitlines()
    pkg = ge.load_package()
    pkg.initialize()
    ctx = pkg.create_grid(None, 1, 1, "C")
    n, nrhs, nb = a.n, a.nrhs, a.nb
    m, nn = (n, nrhs) if a.side == "L" else (nrhs, n)
    spd = np.zeros((n, n), order="F")
    pkg.set_random_hermitian_positive_definite(ctx, spd, n, nb)
    assert pkg.cholesky_factorization(ctx, a.uplo, spd, nb) == 0
    tri = np.tril if a.uplo == "L" else np.triu
    A = np.asfortranarray(tri(spd) / np.sqrt(n))  # O(1) entries
    del spd
    rng = np.random.default_rng(1)
    B = np.asfortranarray(rng.uniform(-1, 1, (m, nn)))
    times, dev_ms, launches, guard = [], [], 0, 0
    for i in range(1 + a.steps):
        X = B.copy(order="F")
        t0 = time.perf_counter()
        pkg.triangular_multiplication(ctx, a.side, a.uplo, a.op, "N", 1.0, A, X, nb, nb)
        dt = time.perf_counter() - t0
        if i:
            times.append(dt)
            dev_ms.append(pkg.last_solver_device_ms(ctx))
        launches, guard = pkg.last_solver_launch_count(ctx), pkg.last_inverse_guard_steps(ctx)
    flops = float(n) * n * nrhs
    # relative error against the dense fp64 product on the GPU
    opa = {"N": A, "T": A.T, "C": A.T}[a.op]
    dA, dB, dX = (torch.from_numpy(np.ascontiguousarray(v)).cuda() for v in (opa, B, X))
    ref = dA @ dB if a.side == "L" else dB @ dA
    rel = ((dX - ref).abs().max() / ref.abs().max()).item()
    del dA, dB, dX, ref
    torch.cuda.empty_cache()
    exe = os.path.join(ROOT, "tools", "cublas_trmm_ref")
    r = subprocess.run([exe, str(m), str(nn), a.side, a.uplo, a.op], capture_output=True, text=True)
    vendor = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else {"error": (r.stdout + r.stderr)[-500:]}
    e2e = min(times)
    line = {"metric": f"triangular multiplication TFLOP/s (fp64, {a.side}{a.uplo}{a.op}, n={n}, nrhs={nrhs}, nb={nb})",
            "value": flops / (min(dev_ms) * 1e-3) / 1e12, "ms_device": min(dev_ms), "unit": "TFLOP/s",
            "value_e2e_host_buffers": flops / e2e / 1e12, "ms_e2e": e2e * 1e3,
            "h2d_bytes": A.nbytes + B.nbytes, "d2h_bytes": B.nbytes, "launches": launches, "guard_steps": guard,
            "rel_err_vs_dense_fp64_product": rel, "eps": float(np.finfo(np.float64).eps),
            "gpu_library_reference": vendor, "card": card,
            "engine": os.environ.get("DLAF_B200_D_BULK", "ozaki")}
    print(json.dumps(line), flush=True)
    pkg.free_grid(ctx)


if __name__ == "__main__":
    main()
