"""Worker of the distributed triangular-multiplication tests (one process and GPU per rank, NCCL): every side / uplo / op /
diag combination and size of the reference's table with its distributed source rank (P-1, min(1, Q-1)),
test_multiplication_triangular.cpp:118, against the closed forms, plus one random case with config-sized tiles against
the oracle (tests/trmm_oracle.py). Prints "total failures N" on rank 0."""
import argparse
import itertools
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
import __graft_entry__ as ge  # noqa: E402
import trmm_oracle  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", default="2x1")
    ap.add_argument("--order", default="R")
    a = ap.parse_args()
    import torch
    import torch.distributed as dist

    P, Q = (int(x) for x in a.grid.split("x"))
    rank = int(os.environ["RANK"])
    pkg = ge.load_package()
    O = ge.load_oracle()
    lr = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(lr)
    dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
    pkg.initialize()
    comm = pkg.comm_create_from_torch()
    ctx = pkg.create_grid(comm, P, Q, a.order)
    _, _, myrow, mycol = pkg.grid_info(ctx)
    src = (P - 1, min(1, Q - 1))
    failures = []

    def run(side, uplo, op, diag, alpha, A, B, mb, nb):
        """this rank's part of the product (None outside the grid or for an empty local part)"""
        m, n = B.shape
        ba = mb if side == "L" else nb
        dt = B.dtype
        if rank < P * Q:
            la = np.asfortranarray(O.scatter_block_cyclic(A, ba, (P, Q), src)[(myrow, mycol)])
            lb = np.asfortranarray(O.scatter_block_cyclic_rect(B, mb, nb, (P, Q), src)[(myrow, mycol)])
        else:
            la = lb = np.zeros((1, 1), dtype=dt, order="F")
        if la.size == 0:
            la = np.zeros((max(1, la.shape[0]), max(1, la.shape[1])), dtype=dt, order="F")
        lbw = lb if lb.size else np.zeros((max(1, lb.shape[0]), max(1, lb.shape[1])), dtype=dt, order="F")
        pkg.triangular_multiplication(ctx, side, uplo, op, diag, alpha, la, lbw, mb, nb, m=m, n=n, isrc=src[0], jsrc=src[1])
        return lbw if (rank < P * Q and lb.size) else None

    for (m, n, mb, nb) in O.TRIANGULAR_TEST_SIZES:
        if m == 0 or n == 0:
            continue
        for t in "sdcz":
            dt = pkg.TYPES[t]
            alpha = O.TRIANGULAR_TEST_ALPHA if np.dtype(dt).kind == "c" else O.TRIANGULAR_TEST_ALPHA.real
            for side, uplo, op, diag in itertools.product("LR", "LU", "NTC", "NU"):
                A, B, expected = trmm_oracle.golden(O, side, uplo, op, diag, alpha, m, n, dt)
                out = run(side, uplo, op, diag, alpha, A, B, mb, nb)
                if out is not None:
                    tol = trmm_oracle.tolerance(m, dt)
                    ok, _, msg = O.check_near(O.scatter_block_cyclic_rect(expected, mb, nb, (P, Q), src)[(myrow, mycol)], out, tol, tol)
                    if not ok:
                        failures.append(("closed form", t, side, uplo, op, diag, m, n, mb, nb, msg))

    # one config-sized random case per element type family against the oracle
    rng = np.random.default_rng(23)
    for (m, n, mb, nb, t) in [(1100, 900, 256, 128, "d"), (520, 600, 64, 128, "z")]:
        dt = pkg.TYPES[t]
        for side, uplo, op in [("L", "L", "N"), ("L", "U", "C"), ("R", "L", "T"), ("R", "U", "N")]:
            na, ba = (m, mb) if side == "L" else (n, nb)
            A = rng.uniform(-1, 1, (na, na)) / np.sqrt(na)
            B = rng.uniform(-1, 1, (m, n))
            if np.dtype(dt).kind == "c":
                A = A + 1j * rng.uniform(-1, 1, (na, na)) / np.sqrt(na)
                B = B + 1j * rng.uniform(-1, 1, (m, n))
            A, B = np.asfortranarray(A.astype(dt)), np.asfortranarray(B.astype(dt))
            ref = B.copy(order="F")
            trmm_oracle.triangular_multiplication(side, uplo, op, "N", 1.0, A, ref, mb, nb)
            out = run(side, uplo, op, "N", 1.0, A, B, mb, nb)
            if out is not None:
                tol = trmm_oracle.tolerance(max(m, n), dt) * max(1.0, float(np.abs(ref).max()))
                ok, _, msg = O.check_near(O.scatter_block_cyclic_rect(ref, mb, nb, (P, Q), src)[(myrow, mycol)], out, tol, tol)
                if not ok:
                    failures.append(("random", t, side, uplo, op, m, n, mb, nb, msg))

    flag = torch.tensor([len(failures)], dtype=torch.int64, device="cuda")
    dist.all_reduce(flag)
    if failures:
        print(f"rank {rank} FAILURES: {failures[:5]}", flush=True)
    if rank == 0:
        print(f"trmm_dist_worker grid={P}x{Q} order={a.order} src={src}: total failures {int(flag.item())}", flush=True)
    pkg.free_grid(ctx)
    dist.destroy_process_group()
    sys.exit(1 if flag.item() else 0)


if __name__ == "__main__":
    main()
