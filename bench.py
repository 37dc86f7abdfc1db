#!/usr/bin/env python
"""bench.py — POTRF GFLOP/s (fp64, N=32768, nb=512) on 1/2/4/8 B200, the metric of BASELINE.json.

A "step" is one Cholesky factorization of the miniapp's random Hermitian positive definite matrix
(include/dlaf/util_matrix.h:410-453), timed like miniapp_cholesky.cpp:137-154 (input resident on the
device, factorization + all inter-GPU traffic + final drain), flop model N^3/3 (miniapp_cholesky.cpp:157-162).

  python bench.py --gpus 1 --steps K --warmup W            our arm (N>1: under torchrun, one rank per GPU)
  python bench.py --impl reference --steps K --warmup W    the reference algorithm on the host cores (oracle port)
  python bench.py ... --dump-outputs DIR                   also write a fixed sample of the last timed factor to DIR/*.npy

One JSON line on stdout (rank 0); everything else goes to stderr. Nothing is written into the source tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only; no __pycache__ in it from a benchmark run
import __graft_entry__ as ge  # noqa: E402

METRIC = "POTRF GFLOP/s (fp64, N=32768, nb=512)"
GRIDS = {1: (1, 1), 2: (2, 1), 4: (2, 2), 8: (2, 4)}
DUMP_SAMPLES = 1 << 21  # 16 MB of fp64 (32 MB complex128): the whole factor at N=32768 would be 8 GB
DUMP_SEED = 20240601


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference", "next-rows"],
                   help="ours / reference: the two arms of the contract; next-rows: child mode of the `next_rows` block")
    # (--matrix-size / --block-size are the miniapp's names; under torchrun use them: its own parser rejects "--n" as an
    # ambiguous abbreviation of --nnodes / --nproc-per-node even after the script name)
    p.add_argument("--n", "--matrix-size", dest="n", type=int, default=32768, help="matrix size (BASELINE metric: 32768)")
    p.add_argument("--nb", "--block-size", dest="nb", type=int, default=512, help="block size (BASELINE metric: 512)")
    p.add_argument("--grid-rows", type=int, default=0)
    p.add_argument("--grid-cols", type=int, default=0)
    p.add_argument("--type", default="d", choices=["s", "d", "c", "z"], help="element type (BASELINE metric: d)")
    p.add_argument("--e2e-steps", type=int, default=-1, help="end-to-end (host buffer) steps, default --steps")
    p.add_argument("--parity-n", type=int, default=8192, help="size of the element-wise oracle parity case run after the "
                   "timed region (non-zero source rank on grids; 0 = skip)")
    p.add_argument("--cpu-budget-s", type=float, default=240.0, help="time budget of the CPU arm (whole run)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-check", action="store_true")
    p.add_argument("--no-gpu-reference", action="store_true", help="skip the cuSOLVER Dpotrf timing (tools/cusolver_potrf_ref)")
    p.add_argument("--next-n", type=int, default=8192, help="size of the short measurements of the algorithms that consume the "
                   "factor (triangular solver, inverse, generalized -> standard; SURVEY 8f), 0 = skip; 1 GPU only")
    p.add_argument("--cpu-sample-n", type=int, default=0, help="force the CPU sample size")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the last one computed to DIR/<name>.npy: the factor's diagonal and "
                        f"{DUMP_SAMPLES} entries of its referenced triangle at positions drawn with a fixed seed (complex types as "
                        "(..., 2) real/imaginary pairs), so that two builds can be compared output for output")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    return a


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    f = [x.strip() for x in line.split(",")]
                    if len(f) >= 8:
                        self.rows.append(f)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[4 + i].lower().startswith("active") for r in self.rows)]
        pw = [float(r[3]) for r in self.rows if r[3].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "power_w_max": max(pw) if pw else None, "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------------
def cpu_reference_run(O, n: int, nb: int, threads: int, steps: int, warmup: int):
    """The reference algorithm (oracle port: same tile ops, same DAG/priorities, 1 BLAS thread per tile
    task, `threads` pool workers) on the host cores. Returns (GFLOP/s best-of-steps average, residual)."""
    a = O.set_random_hermitian_positive_definite(n, nb, np.float64)
    times = []
    res = None
    for i in range(warmup + steps):
        w = a.copy(order="F")
        t0 = time.perf_counter()
        info = O.cholesky_local("L", w, nb, threads)
        dt = time.perf_counter() - t0
        assert info == 0
        if i >= warmup:
            times.append(dt)
        if i == warmup + steps - 1:
            res = cpu_arm_residual(O, a, w, n)
    return n ** 3 / 3 / (sum(times) / len(times)) / 1e9, sum(times) / len(times), res


def cpu_arm_residual(O, a, w, n):
    """Residual of the CPU arm's own result (checker): oracle routine up to N=8192, above that the torch fp64 checker on
    the GPU when one is visible (not part of any timed region)."""
    if n <= 8192:
        return O.residual("L", a, w)
    try:
        import torch

        if not torch.cuda.is_available() or 2 * a.nbytes > 0.8 * torch.cuda.mem_get_info()[0]:
            return None
        da = torch.from_numpy(np.ascontiguousarray(a.T)).cuda()  # [col, row] views like run_ours
        dw = torch.from_numpy(np.ascontiguousarray(w.T)).cuda()
        return residual_check_torch(torch, da, dw, n)
    except Exception as e:  # pragma: no cover
        log(f"[cpu] residual check skipped: {e!r}")
        return None


def pick_cpu_sample(O, nb: int, threads: int, budget_s: float, n_max: int) -> int:
    """Largest N (multiple of nb, <= n_max) whose factorization is expected to stay within budget_s."""
    n0 = max(nb * 4, 2048)
    g, _, _ = cpu_reference_run(O, n0, nb, threads, 1, 1)
    n = int((budget_s * g * 1e9 * 3) ** (1 / 3))
    n = max(n0, min(n_max, n // nb * nb))
    log(f"[cpu] probe N={n0}: {g:.1f} GFLOP/s on {threads} threads -> sample N={n}")
    return n


def run_reference_arm(args):
    """The reference's CPU path (oracle port, see cpu_reference_run) on all usable host threads. Each step is a bounded
    sample of the workload: the largest N (multiple of nb, <= --n) whose warmup + steps fit the time budget; when the
    budget allows --n itself the arm runs the FULL configuration (same_config)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    O = ge.load_oracle()
    O.build()
    threads = O.max_pool_threads()
    per_step = max(2.0, args.cpu_budget_s / max(1, args.steps + args.warmup))
    n = args.cpu_sample_n or pick_cpu_sample(O, args.nb, threads, per_step, args.n)
    gf, sec, res = cpu_reference_run(O, n, args.nb, threads, args.steps, args.warmup)
    sample = (f"N={n} nb={args.nb} fp64, same generator, oracle port of impl.h:150-189 over OpenBLAS, {threads} pool threads x 1 "
              f"BLAS thread (OpenBLAS in the scipy wheel is built with MAX_THREADS=64, so at most 56 concurrent tile tasks)")
    line = {
        "impl": "reference", "metric": METRIC, "value": gf, "unit": "GFLOP/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"fp64 POTRF N={args.n} nb={args.nb} (CPU arm measured on N={n})",
                   "sample": sample, "same_config": n == args.n},
        "cpu_baseline": {"value": gf, "unit": "GFLOP/s", "cores": threads, "kind": "port", "sample": sample,
                         "blas": O.lib().oracle_blas_config().decode(), "residual": res,
                         "host_hw_threads": O.lib().oracle_hardware_threads()},
        "e2e": {"value": gf, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def residual_check_torch(torch, d_ref, d_fac, n: int, blk: int = 4096):
    """Checker (not product code): the miniapp's max|A - L L^T| / max|A| over the lower triangle
    (miniapp_cholesky.cpp:408-446), evaluated block column by block column with torch fp64 matmul.
    d_ref / d_fac are (n, n) torch views of column-major storage, i.e. indexed [col, row]."""
    max_a = 0.0
    max_d = 0.0
    # In the [col,row] view X[j, i] = A(i, j); the lower triangle of A is the upper triangle of X.
    Lt = torch.triu(d_fac)  # Lt[j, i] = L(i, j) for i >= j
    for j0 in range(0, n, blk):
        j1 = min(n, j0 + blk)
        # (L L^T)(i, j) for j in block, i >= j0:  sum_k L(i,k) L(j,k) -> Lt[:, i]^T Lt[:, j]
        prod = Lt[:j1, j0:j1].T @ Lt[:j1, j0:]  # [j, i], k < j1 suffices because L(j,k)=0 for k>j
        a_blk = d_ref[j0:j1, j0:]
        diff = torch.triu(a_blk - prod)  # keep i >= j (i index offset j0 on both axes)
        max_d = max(max_d, diff.abs().max().item())
        max_a = max(max_a, torch.triu(a_blk).abs().max().item())
        del prod, diff
    return max_d / max_a


def oracle_parity(pkg, ctx, torch, dist, rank, world, P, Q, myrow, mycol, n, nb, dtype):
    """Checker (never timed): the distributed factorization of the miniapp's matrix (size n) against the oracle's factor,
    element-wise on the referenced triangle, plus the untouched other triangle and the product's own grid residual."""
    O = ge.load_oracle()
    src = (max(0, P - 1), min(1, Q - 1)) if world > 1 else (0, 0)
    dt = np.dtype(dtype)
    tdt = {"f": {4: torch.float32, 8: torch.float64}, "c": {8: torch.complex64, 16: torch.complex128}}[dt.kind][dt.itemsize]
    t0 = time.perf_counter()
    if rank == 0:
        O.build()
        A = O.set_random_hermitian_positive_definite(n, nb, dt)
        expect = A.copy(order="F")
        assert O.cholesky_local("L", expect, nb, O.max_pool_threads()) == 0
        both = torch.from_numpy(np.stack([np.ascontiguousarray(A.T), np.ascontiguousarray(expect.T)]))
    else:
        both = torch.empty((2, n, n), dtype=tdt)
    if dist is not None:
        both = both.cuda()
        dist.broadcast(both, src=0)
        both = both.cpu()
    A = both[0].numpy().T
    expect = both[1].numpy().T
    loc = np.asfortranarray(O.scatter_block_cyclic(A, nb, (P, Q), src)[(myrow, mycol)])
    exp_loc = O.scatter_block_cyclic(expect, nb, (P, Q), src)[(myrow, mycol)]
    orig = loc.copy(order="F")
    info = pkg.cholesky_factorization(ctx, "L", loc, nb, n=n, isrc=src[0], jsrc=src[1])
    nt = -(-n // nb)
    gi = np.concatenate([np.arange(g * nb, min(n, (g + 1) * nb)) for g in range(nt) if O.rank_global_tile(g, P, src[0]) == myrow]
                        or [np.zeros(0, int)])
    gj = np.concatenate([np.arange(g * nb, min(n, (g + 1) * nb)) for g in range(nt) if O.rank_global_tile(g, Q, src[1]) == mycol]
                        or [np.zeros(0, int)])
    mask = gi[:, None] >= gj[None, :]
    tol = O.cholesky_tolerance(n, dt)
    e_, v_ = np.where(mask, exp_loc, 0), np.where(mask, loc, 0)
    ok, _, msg = O.check_near(e_, v_, tol, tol)
    diff = np.abs(e_ - v_)
    amax = np.maximum(np.abs(e_), np.abs(v_))
    with np.errstate(divide="ignore", invalid="ignore"):
        rel = np.where(amax > 0, diff / amax, 0.0)
    worst = float(np.minimum(diff, rel).max() / tol) if diff.size else 0.0  # < 1 <=> every element passes CHECK_MATRIX_NEAR
    untouched = bool(np.array_equal(np.where(mask, 0, loc), np.where(mask, 0, orig)))
    res = pkg.check_cholesky(ctx, "L", orig, loc, nb, n=n, isrc=src[0], jsrc=src[1])
    bad = 0 if (ok and untouched and info == 0) else 1
    worst_all = float(worst)
    if dist is not None:
        t = torch.tensor([float(bad), worst_all], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        bad, worst_all = int(t[0].item()), t[1].item()
    if not ok:
        log(f"[bench] rank {rank} oracle parity FAILED: {msg}")
    return {"n": n, "nb": nb, "grid": [P, Q], "source_rank": list(src), "dtype": dt.name, "info": int(info),
            "elementwise_vs_oracle_ok_all_ranks": bad == 0, "max_error_over_tolerance": worst_all,
            "tolerance": float(tol), "tolerance_rule": "4 (n+1) c eps, |d| or |d|/max(|e|,|v|) (test_cholesky.cpp:76-77)",
            "unreferenced_triangle_untouched": untouched, "grid_residual_max_diff_over_max_a": res,
            "residual_gate_eps_n": float(np.finfo(dt.type(0).real.dtype).eps * n), "seconds": time.perf_counter() - t0}


def next_rows(pkg, ctx, torch, O, n: int, nb: int):
    """SURVEY 8(f) rows 1-3 in the driver-visible line (1 GPU, fp64): the consumers of the factor through the C ABI at a
    size that takes a fraction of a second — device time of the whole call (CUDA events inside the library), a residual,
    and an element-wise oracle verdict at n = 1024 with the reference's tolerances. Never part of the timed POTRF region."""
    out = {}
    dt = np.float64
    b = np.zeros((n, n), dtype=dt, order="F")
    pkg.set_random_hermitian_positive_definite(ctx, b, n, nb)
    fac = b.copy(order="F")
    assert pkg.cholesky_factorization(ctx, "L", fac, nb) == 0
    d_b = torch.from_numpy(b).cuda()  # (symmetric: row- and column-major coincide)
    d_fac = torch.from_numpy(np.ascontiguousarray(fac.T)).cuda()  # memory = column-major factor
    eye = torch.eye(n, dtype=torch.float64, device="cuda")
    # -- inverse from the Cholesky factor
    ms = []
    for _ in range(2):
        w = d_fac.clone()
        torch.cuda.synchronize()
        pkg.inverse_device(ctx, 3, "L", "N", w.data_ptr(), dt, n, nb, n)
        ms.append(pkg.last_solver_device_ms(ctx))
    low = torch.tril(w.T)
    res = ((low + torch.tril(low, -1).T) @ d_b - eye).abs().max().item()
    out["inverse_from_cholesky_factor"] = {"api": "dlaf_b200_inverse_device_d (dlaf_inverse_from_cholesky_factor_d on device memory)",
                                           "n": n, "nb": nb, "ms_device": min(ms), "value": 2 * n ** 3 / 3 / (min(ms) * 1e-3) / 1e9,
                                           "unit": "GFLOP/s", "flops_model": "2 n^3 / 3", "max_abs_invA_A_minus_I": res,
                                           "guard_fallback_steps": pkg.last_inverse_guard_steps(ctx), "launches": pkg.last_solver_launch_count(ctx)}
    # -- generalized -> standard: A = B with the diagonal shifted (Hermitian, not a multiple of B)
    d_a = d_b.contiguous().clone()  # row-major copy of a symmetric matrix: its memory is also the column-major matrix
    d_a.diagonal().sub_(float(n))
    ms = []
    for _ in range(2):
        w = d_a.clone()
        torch.cuda.synchronize()
        pkg.generalized_to_standard_device(ctx, "L", w.data_ptr(), d_fac.data_ptr(), dt, n, nb, n)
        ms.append(pkg.last_solver_device_ms(ctx))
    low = torch.tril(w.T)
    lmat = torch.tril(d_fac.T)
    res = torch.tril(lmat @ (low + torch.tril(low, -1).T) @ lmat.T - d_a).abs().max().item() / d_a.abs().max().item()
    out["generalized_to_standard"] = {"api": "dlaf_b200_generalized_to_standard_device_d", "n": n, "nb": nb, "ms_device": min(ms),
                                      "value": float(n) ** 3 / (min(ms) * 1e-3) / 1e9, "unit": "GFLOP/s", "flops_model": "n^3",
                                      "max_LCLh_minus_A_over_max_A": res, "guard_fallback_steps": pkg.last_inverse_guard_steps(ctx),
                                      "launches": pkg.last_solver_launch_count(ctx)}
    del w, low, lmat, d_a, d_b, eye
    # -- triangular solver (host-buffer entry; the device time of the sweep is reported by the library)
    nrhs = n // 2
    rng = np.random.default_rng(1)
    rhs = np.asfortranarray(rng.uniform(-1, 1, (n, nrhs)))
    lo = np.asfortranarray(np.tril(fac))
    ms = []
    for _ in range(2):
        x = rhs.copy(order="F")
        pkg.triangular_solver(ctx, "L", "L", "N", "N", 1.0, lo, x, nb, nb)
        ms.append(pkg.last_solver_device_ms(ctx))
    d_l, d_x, d_r = (torch.from_numpy(np.ascontiguousarray(v)).cuda() for v in (lo, x, rhs))
    res = (d_l @ d_x - d_r).abs().max().item() / (np.abs(x).max() * np.abs(lo).max() * n)
    out["triangular_solver"] = {"api": "dlaf_b200_triangular_solver_d (Left, Lower, NoTrans; host buffers, device time of the sweep)",
                                "n": n, "nrhs": nrhs, "nb": nb, "ms_device": min(ms), "value": float(n) * n * nrhs / (min(ms) * 1e-3) / 1e9,
                                "unit": "GFLOP/s", "flops_model": "n^2 nrhs", "residual_over_n_maxA_maxX": res,
                                "launches": pkg.last_solver_launch_count(ctx)}
    del d_l, d_x, d_r, d_fac
    torch.cuda.empty_cache()
    # -- element-wise oracle verdicts at n = 1024 (reference tolerances)
    m, mb = 1024, 256
    spd = O.set_random_hermitian_positive_definite(m, mb, dt)
    f = spd.copy(order="F")
    assert O.cholesky_local("L", f, mb, 8) == 0
    par = {}
    ref = f.copy(order="F")
    O.inverse_from_cholesky_factor("L", ref, mb)
    got = f.copy(order="F")
    pkg.inverse_from_cholesky_factor(ctx, "L", got, mb)
    sc = float(np.abs(np.tril(ref)).max())
    par["inverse_from_cholesky_factor"] = bool(O.check_near(np.tril(ref) / sc, np.tril(got) / sc, O.inverse_tolerance(m, dt),
                                                            O.inverse_tolerance(m, dt))[0])
    a2 = np.asfortranarray(spd - m * np.eye(m))
    ref = a2.copy(order="F")
    O.generalized_to_standard("L", ref, f, mb)
    got = a2.copy(order="F")
    pkg.generalized_to_standard(ctx, "L", got, f, mb)
    par["generalized_to_standard"] = bool(O.check_near(np.tril(ref), np.tril(got), 0.0,
                                                       O.gen_to_std_tolerance(m, dt) * max(1.0, float(np.abs(np.tril(ref)).max())))[0])
    r2 = np.asfortranarray(rng.uniform(-1, 1, (m, 512)))
    ref = r2.copy(order="F")
    lo2 = np.asfortranarray(np.tril(f))
    O.triangular_solver("L", "L", "N", "N", 1.0, lo2, ref, mb, 128)
    got = r2.copy(order="F")
    pkg.triangular_solver(ctx, "L", "L", "N", "N", 1.0, lo2, got, mb, 128)
    tol = O.triangular_tolerance(m, dt) * max(1.0, float(np.abs(ref).max()))
    par["triangular_solver"] = bool(O.check_near(ref, got, tol, tol)[0])
    out["elementwise_vs_oracle_n1024"] = par
    return out


def triangle_bytes(n: int, nb: int, P: int, Q: int, vr: int, vc: int, itemsize: int) -> int:
    nt = -(-n // nb)
    total = 0
    for gj in range(vc, nt, Q):
        width = min(nb, n - gj * nb)
        rows = sum(min(nb, n - gi * nb) for gi in range(vr, nt, P) if gi >= gj)
        total += rows * width * itemsize
    return total


def dump_outputs(out_dir, torch, dist, d_work, n, nb, P, Q, myrow, mycol, ld, rank):
    """Writes the factor the last timed step left in d_work (this rank's column-major local part, source rank (0, 0)) as
    DIR/factor_diagonal.npy (all n diagonal entries) and DIR/factor_lower_sample.npy (DUMP_SAMPLES entries (i, j), i >= j,
    drawn from DUMP_SEED, so the positions depend on n only). Every global entry is owned by exactly one rank: each rank
    fills the ones it holds into a zero vector and a sum over the ranks assembles the sample on rank 0."""
    rng = np.random.default_rng(DUMP_SEED)
    i, j = rng.integers(0, n, DUMP_SAMPLES), rng.integers(0, n, DUMP_SAMPLES)
    diag = np.arange(n)
    arrays = {}
    for name, (rows, cols) in (("factor_diagonal", (diag, diag)),
                               ("factor_lower_sample", (np.maximum(i, j), np.minimum(i, j)))):
        mine = ((rows // nb) % P == myrow) & ((cols // nb) % Q == mycol)
        lrow = (rows // nb) // P * nb + rows % nb
        lcol = (cols // nb) // Q * nb + cols % nb
        flat = torch.from_numpy((lcol * ld + lrow)[mine]).cuda()
        vals = torch.zeros(len(rows), dtype=d_work.dtype, device=d_work.device)
        vals[torch.from_numpy(mine).cuda()] = d_work.reshape(-1)[flat]
        if dist is not None:
            dist.all_reduce(vals)
        v = vals.cpu().numpy()
        arrays[name] = np.stack([v.real, v.imag], axis=-1) if np.iscomplexobj(v) else v
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        for name, v in arrays.items():
            np.save(os.path.join(out_dir, f"{name}.npy"), v)
        log(f"[bench] wrote {', '.join(f'{k}.npy {v.shape}' for k, v in arrays.items())} to {out_dir}")


def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        log(f"[bench] WORLD_SIZE={world} but --gpus {args.gpus}: launch with torchrun --nproc-per-node {args.gpus}")
        args.gpus = world
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local_rank)
    os.environ["DLAF_B200_DEVICE"] = str(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    pkg = ge.load_package()
    pkg.lib()  # fails loudly if the CUDA library has not been built (no fallback)
    pkg.initialize()
    P, Q = (args.grid_rows, args.grid_cols) if args.grid_rows and args.grid_cols else GRIDS.get(world, (1, world))
    assert P * Q == world, f"grid {P}x{Q} does not match {world} ranks"
    comm = pkg.comm_create_from_torch() if world > 1 else None
    ctx = pkg.create_grid(comm, P, Q, "C")  # ColumnMajor like the miniapp (miniapp_cholesky.cpp:113)
    _, _, myrow, mycol = pkg.grid_info(ctx)
    n, nb = args.n, args.nb
    desc0 = pkg.descriptor(n, nb, 1)
    lr, lc = pkg.local_shape(ctx, desc0)
    ld = lr
    dtype = pkg.TYPES[args.type]
    tdt = {"s": torch.float32, "d": torch.float64, "c": torch.complex64, "z": torch.complex128}[args.type]
    itemsize = np.dtype(dtype).itemsize
    eps = float(np.finfo(np.dtype(dtype).type(0).real.dtype).eps)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    # ---- synthetic input: the miniapp's generator, into pinned host memory (column-major lr x lc)
    t0 = time.perf_counter()
    h_ref_t = torch.empty((lc, lr), dtype=tdt, pin_memory=True)
    h_ref = h_ref_t.numpy().T  # (lr, lc) Fortran-ordered view
    pkg.set_random_hermitian_positive_definite(ctx, h_ref, n, nb)
    log(f"[bench] rank {rank}: generated local {lr}x{lc} in {time.perf_counter() - t0:.1f}s")
    d_ref = h_ref_t.cuda()
    d_work = torch.empty_like(d_ref)
    stream = torch.cuda.current_stream()
    pkg.set_profiling(ctx, True)
    flops = pkg.total_ops(dtype, n)

    # ---- device-resident steps (the miniapp's timed region)
    W, K = args.warmup, args.steps
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    prof_ms = prof_fl = 0.0
    prof_n = 0
    chain = None
    launches = 0
    for i in range(W):
        d_work.copy_(d_ref)
        barrier()
        pkg.cholesky_factorization_device(ctx, "L", d_work.data_ptr(), dtype, n, nb, ld, stream.cuda_stream)
        assert pkg.wait(ctx, stream.cuda_stream) == 0
    sampler = ClockSampler(local_rank)
    barrier()
    wall0 = time.perf_counter()
    with sampler:
        for i in range(K):
            d_work.copy_(d_ref)  # restore the input (not part of the step); matrix >> L2, so every step starts cold
            barrier()
            ev[i][0].record(stream)
            pkg.cholesky_factorization_device(ctx, "L", d_work.data_ptr(), dtype, n, nb, ld, stream.cuda_stream)
            ev[i][1].record(stream)
            info = pkg.wait(ctx, stream.cuda_stream)
            assert info == 0, f"info {info}"
            chain = pkg.read_chain_profile(ctx)
            ms, fl, cnt = pkg.read_profile(ctx)
            prof_ms += ms
            prof_fl += fl
            prof_n += cnt
            launches += pkg.last_launch_count(ctx)
        barrier()
    wall = time.perf_counter() - wall0
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = allmax(sum(step_ms))
    ms_per_step = total_ms / K
    value = flops / (ms_per_step * 1e-3) / 1e9
    clocks = sampler.summary()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, torch, dist if world > 1 else None, d_work, n, nb, P, Q, myrow, mycol, ld, rank)

    # ---- correctness of the timed result, for EVERY world size: the product's own distributed result check (the
    # miniapp's check_cholesky on the GPU grid, engine_check.cu: native GEMMs, independent of the int8 engine), and on one
    # GPU additionally an independent torch fp64 checker.
    residual = residual_torch = None
    if not args.no_check:
        residual = pkg.check_cholesky_device(ctx, "L", d_ref.data_ptr(), d_work.data_ptr(), dtype, n, nb, ld,
                                             stream.cuda_stream)
        if world == 1 and args.type == "d":
            try:
                residual_torch = residual_check_torch(torch, d_ref.view(n, n), d_work.view(n, n), n)
            except Exception as e:  # pragma: no cover
                log(f"[bench] torch residual check skipped: {e}")
        assert residual <= 100 * eps * n, f"residual {residual} above the miniapp's ERROR gate"

    # ---- precision evidence in the same run (checker): the timed result of the int8-digit engine next to the native
    # fp64 (DMMA) engine on the same input — residuals of both and the largest difference between the two factors.
    accuracy = None
    if not args.no_check and world == 1 and args.type == "d" and os.environ.get("DLAF_B200_D_BULK", "ozaki") == "ozaki":
        prev = os.environ.get("DLAF_B200_D_BULK")
        ctx2 = None
        try:
            os.environ["DLAF_B200_D_BULK"] = "dmma"
            ctx2 = pkg.create_grid(None, 1, 1, "C")  # fresh context -> fresh engine that reads the switch
            d_nat = d_ref.clone()
            pkg.cholesky_factorization_device(ctx2, "L", d_nat.data_ptr(), dtype, n, nb, ld, stream.cuda_stream)
            assert pkg.wait(ctx2, stream.cuda_stream) == 0
            res_nat = residual_check_torch(torch, d_ref.view(n, n), d_nat.view(n, n), n)
            max_diff = max_l = 0.0
            for j0 in range(0, n, 4096):  # [col, row] views: the lower triangle of L is the upper triangle of the view
                j1 = min(n, j0 + 4096)
                a_, b_ = torch.triu(d_work.view(n, n)[j0:j1, j0:]), torch.triu(d_nat.view(n, n)[j0:j1, j0:])
                max_diff = max(max_diff, (a_ - b_).abs().max().item())
                max_l = max(max_l, b_.abs().max().item())
                del a_, b_
            accuracy = {"residual_int8_digit_engine": residual_torch, "residual_native_fp64_engine": res_nat,
                        "max_abs_diff_between_the_two_factors": max_diff, "max_abs_factor_entry": max_l,
                        "diff_in_ulps_of_max_entry": max_diff / (max_l * float(np.finfo(np.float64).eps)),
                        "gate_eps_n": float(np.finfo(np.float64).eps * n)}
            del d_nat
        except Exception as e:  # pragma: no cover
            log(f"[bench] native-engine comparison skipped: {e!r}")
        finally:
            if ctx2 is not None:
                try:
                    pkg.free_grid(ctx2)
                except Exception:
                    pass
            if prev is None:
                os.environ.pop("DLAF_B200_D_BULK", None)
            else:
                os.environ["DLAF_B200_D_BULK"] = prev

    # ---- roofline of the dominant kernel (bulk trailing update on stream L)
    # fp64 engine (DLAF_B200_D_BULK): "ozaki" (default) = exact int8 digit products on tcgen05, 36 int8 MACs per fp64 MAC,
    # bounded by the int8 tensor pipe; "dmma" = native fp64 DMMA, bounded by the fp64 tensor pipe.
    engine = os.environ.get("DLAF_B200_D_BULK", "ozaki")
    peak64 = pkg.measure_fp64_tensor_peak_tflops()
    achieved64 = (prof_fl / (prof_ms * 1e-3) / 1e12) if prof_ms > 0 else None
    cap_file = "r02_ncu_ozaki_bulk.json" if engine == "ozaki" else "r01_ncu_gemm_bulk_final.json"
    if args.type != "d":
        engine = {"s": "tf32x3", "c": "simt", "z": "zdmma"}[args.type]
    traffic, traffic_note = None, None
    try:  # DRAM bytes of the dominant kernel from the committed ncu --set full capture (one launch)
        with open(os.path.join(ROOT, "profiles", cap_file)) as f:
            cap = json.load(f)
        traffic = cap["dram_bytes_read"] + cap["dram_bytes_write"]
        traffic_note = (f"ncu capture of ONE launch: {cap['launch']}; algorithmic bytes of that launch "
                        f"{cap['algorithmic_bytes']}; {cap.get('note', '')}")
    except Exception:
        pass
    if engine == "ozaki":
        peak8_issue = pkg.measure_int8_tensor_peak_tops()
        mp = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                mp = json.load(f)
        except Exception:
            pass
        # int8 dense tensor rate = 2 x the bf16 rate on tcgen05 (nominal 4.5 vs 2.25 POP/s): the denominator is 2 x the
        # driver-measured cuBLAS bf16 throughput — the SUSTAINED figure, because this kernel is timed inside a long step
        bf16_s, bf16_b = mp.get("bf16_tflops_sustained"), mp.get("bf16_tflops")
        peak8 = 2.0 * bf16_s if bf16_s else (2.0 * bf16_b if bf16_b else 2.0 * 1400.0)
        peak_src = ("2 x MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if bf16_s else
                    ("2 x MEASURED_PEAKS.json bf16_tflops (of measured, burst)" if bf16_b else "2 x 1400 (of fallback, sustained)"))
        pairs = pkg.ozaki_pairs()
        achieved8 = achieved64 * pairs if achieved64 else None
        roofline = {
            "kernel": f"gemm_ozaki_i8_kernel<64> (bulk trailing update, stream L): fp64 C -= A B^T as {pairs} exact int8 tcgen05 digit-plane products",
            "bound": "tensor", "achieved": achieved8, "peak": peak8, "unit": "TFLOP/s",
            "frac": (achieved8 / peak8) if achieved8 else None,
            "unit_note": f"int8 tensor-core tera-ops/s (1 MAC = 2 ops); algorithmic ops per launch = {pairs} x the fp64 flops of "
                         "the update (7 balanced radix-256 digits, digit pairs t + u <= 6; round 1 used 36)",
            "int8_macs_per_fp64_mac": pairs,
            "guard_fallback_steps_last_run": pkg.guard_fallback_steps(ctx),
            "fp64_equivalent_tflops": achieved64, "fp64_tensor_peak_tflops": peak64,
            "frac_of_fp64_tensor_roofline": (achieved64 / peak64) if achieved64 else None,
            "traffic": traffic, "traffic_note": traffic_note,
            "peak_source": peak_src + "; other denominators for context: 2 x bf16 burst = %s, this GPU's tcgen05.mma.kind::i8 issue-rate "
                           "microbenchmark (all-ones data, no power cap) = %.0f, nominal 4500. The MMA phase of this kernel is bound by "
                           "shared-memory operand reads (~98 B/clk/SM: 96 KB per k-step in 986 clk vs 896 at the pipe's rate, "
                           "profiles/r02_ozaki_i8_v5_*.log), the epilogue (7 x 64 TMEM columns drained at ~3.3k clk per tile) is exposed because "
                           "the accumulators fill TMEM. fp64 tensor (DMMA) peak measured by microbenchmark." % (
                               (2.0 * bf16_b) if bf16_b else None, peak8_issue),
            "peak_int8_issue_rate_microbenchmark": peak8_issue,
        }
    elif engine == "tf32x3":
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except Exception:
            pass
        peak_tf32 = peaks.get("bf16_tflops", 2250.0) / 2.0  # tf32 dense = half the bf16 rate on tcgen05
        ach = achieved64 * 3.0 if achieved64 else None
        roofline = {
            "kernel": "gemm_tf32x3_kernel (bulk trailing update, stream L): fp32 C -= A B^T as 3 tcgen05 kind::tf32 MMAs (hi*hi, hi*lo, lo*hi)",
            "bound": "tensor", "achieved": ach, "peak": peak_tf32, "unit": "TFLOP/s", "frac": (ach / peak_tf32) if ach else None,
            "fp32_equivalent_tflops": achieved64, "traffic": None,
            "peak_source": "MEASURED_PEAKS.json bf16_tflops / 2 (tf32 runs at half the bf16 rate); nominal fallback 1125",
        }
    else:
        roofline = {
            "kernel": {"dmma": "gemm_nt_f64_kernel<GemmCfg<64,64,16,3,4,2,2>>", "zdmma": "gemm_nt_z_kernel (complex128 on DMMA)",
                       "simt": "gemm_nt_simt_kernel<float2>"}.get(engine, engine) + " (bulk trailing update, stream L)",
            "bound": "tensor" if engine != "simt" else "fp32 FMA pipe",
            "achieved": achieved64, "peak": peak64 if engine != "simt" else None, "unit": "TFLOP/s",
            "frac": (achieved64 / peak64) if (achieved64 and engine != "simt") else None,
            "traffic": traffic if engine == "dmma" else None, "traffic_note": traffic_note if engine == "dmma" else None,
            "peak_source": "measured now on this GPU: DMMA.8x8x4 issue-rate microbenchmark (dlaf_b200_measure_fp64_tensor_peak_tflops); "
                           "MEASURED_PEAKS.json holds no fp64 figure (bf16 cuBLAS + HBM copy only); nominal B200 fp64 = 40 TFLOP/s",
        }
    roofline.update({
        "engine": engine, "launches_timed": prof_n, "critical_path_ms_last_step": chain,
        "kernel_ms_per_step": prof_ms / K if K else None,
        "kernel_share_of_step": (prof_ms / K) / ms_per_step if K else None,
        "whole_potrf_frac_of_fp64_tensor_peak": value / 1e3 / (peak64 * world),
    })
    del d_work

    # ---- end to end through the reference-facing C ABI with HOST buffers (H2D + D2H inside), E steps on pinned
    # memory plus the same call on PAGEABLE memory (what a ScaLAPACK caller passes)
    E = args.e2e_steps if args.e2e_steps >= 0 else K
    e2e = None
    if E > 0:
        h_work_t = torch.empty((lc, lr), dtype=tdt, pin_memory=True)
        h_work = h_work_t.numpy().T
        tchar = args.type

        def e2e_run(buf_t, buf, reps):
            times = []
            for i in range(1 + reps):
                buf_t.copy_(h_ref_t)
                barrier()
                t0 = time.perf_counter()
                info = pkg.cholesky_factorization(ctx, "L", buf, nb, n=n)
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                assert info == 0
                if i >= 1:
                    times.append(dt)
            return allmax(sum(times) / len(times))

        e2e_s = e2e_run(h_work_t, h_work, E)
        tb = triangle_bytes(n, nb, P, Q, myrow, mycol, itemsize)
        e2e = {"value": flops / e2e_s / 1e9, "unit": "GFLOP/s", "ms_per_step": e2e_s * 1e3,
               "h2d_bytes_per_step": tb, "d2h_bytes_per_step": tb, "steps": E,
               "api": f"dlaf_cholesky_factorization_{tchar} (pinned host local matrix, referenced triangle only)"}
        if not args.no_check:
            # the e2e result itself is checked on the grid (host flavour of the distributed check)
            e2e["residual"] = pkg.check_cholesky(ctx, "L", h_ref, h_work, nb, n=n)
        try:
            p_work_t = torch.empty((lc, lr), dtype=tdt)  # ordinary (pageable) host memory
            p_s = e2e_run(p_work_t, p_work_t.numpy().T, min(E, 2))
            e2e["pageable_host"] = {"value": flops / p_s / 1e9, "unit": "GFLOP/s", "ms_per_step": p_s * 1e3,
                                    "steps": min(E, 2)}
            del p_work_t
        except Exception as e:  # pragma: no cover
            log(f"[bench] pageable e2e skipped: {e!r}")

    # ---- element-wise parity with the oracle, in the driver-visible line for EVERY world size: a smaller case
    # (--parity-n, nb as benchmarked) with a NON-ZERO source rank on grids (test/unit/factorization/test_cholesky.cpp:85),
    # factorised through the host C ABI, compared with the reference algorithm's factor at the reference's unit-test
    # tolerance (test_cholesky.cpp:76-77). The oracle runs on rank 0 only; its factor travels over torch.distributed.
    parity = None
    if not args.no_check and args.parity_n > 0:
        parity = oracle_parity(pkg, ctx, torch, dist if world > 1 else None, rank, world, P, Q, myrow, mycol,
                               args.parity_n, nb, dtype)

    # ---- CPU baseline: the reference algorithm on this box's host cores, bounded sample. Runs in a child
    # process (the reference arm of this script) so that a host BLAS problem cannot take the bench down.
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.type == "d":
        cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "0",
               "--n", str(n), "--nb", str(nb)]
        if args.cpu_sample_n:
            cmd += ["--cpu-sample-n", str(args.cpu_sample_n)]
        try:
            env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
            cpu = json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
        except Exception as e:  # pragma: no cover
            cpu = {"value": None, "unit": "GFLOP/s", "cores": None, "kind": "port", "sample": f"failed: {e!r}"}

    # ---- vendor-library GPU reference on the same box, same run (SURVEY 8d): monolithic cusolverDnDpotrf, the
    # routine the reference's GPU backend calls per tile. Measurement aid (tools/cusolver_potrf_ref), never on the
    # product path; absent binary -> null.
    gpu_ref = None
    exe = os.path.join(ROOT, "tools", "cusolver_potrf_ref")
    if rank == 0 and world == 1 and not args.no_gpu_reference and os.path.exists(exe) and args.type == "d":
        try:
            del d_ref
            torch.cuda.empty_cache()
            r = subprocess.run([exe, str(n)], capture_output=True, text=True, timeout=300)
            for ln in r.stdout.splitlines():
                if " best:" in ln:
                    tok = ln.split()
                    gpu_ref = {"kind": "cusolverDnDpotrf (monolithic, device-resident, lower)", "ms": float(tok[3]),
                               "value": float(tok[5]), "unit": "GFLOP/s", "n": n}
        except Exception as e:  # pragma: no cover
            log(f"[bench] cusolver reference skipped: {e}")

    # ---- the algorithms that consume the factor (SURVEY 8f rows 1-3), short, after everything that is timed for POTRF
    # Runs in a child process (this script, --impl next-rows): nothing it does can take the POTRF line down.
    nxt = None
    if rank == 0 and world == 1 and args.next_n > 0 and args.type == "d" and not args.no_check:
        try:
            torch.cuda.empty_cache()
            env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "next-rows", "--next-n", str(args.next_n),
                                "--nb", str(nb if nb <= 512 else 512)], capture_output=True, text=True, timeout=600, env=env)
            nxt = json.loads(r.stdout.strip().splitlines()[-1])
        except Exception as e:  # pragma: no cover
            log(f"[bench] next rows skipped: {e!r}")
            nxt = {"skipped": repr(e)[:200]}

    if rank == 0:
        line = {
            "metric": METRIC if (args.type, n, nb) == ("d", 32768, 512) else f"POTRF GFLOP/s ({args.type}, N={n}, nb={nb})",
            "value": value, "unit": "GFLOP/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": {"s": "f32", "d": "f64", "c": "c64", "z": "c128"}[args.type], "data": "synthetic",
            "dtype_note": (("fp64 in, fp64 out; panels (POTRF/TRSM) in native fp64 DMMA; trailing update = exact int8 digit products "
                            "(7 balanced radix-256 digits of a 55-bit row mantissa, int32 accumulation, exact recombination; error model "
                            "and data-dependent native-fp64 fallback: dla-future_b200/csrc/gemm_ozaki.h)")
                           if os.environ.get("DLAF_B200_D_BULK", "ozaki") == "ozaki" else "native fp64 (DMMA)") if args.type == "d"
            else {"s": "fp32 in/out; trailing update 3xTF32 on tcgen05", "c": "complex64, SIMT", "z": "complex128, DMMA"}[args.type],
            "config": {"workload": f"{ {'s': 'fp32', 'd': 'fp64', 'c': 'complex64', 'z': 'complex128'}[args.type] } POTRF N={n} nb={nb} uplo=L, grid {P}x{Q} (ColumnMajor), device-resident, in place",
                       "input": "set_random_hermitian_positive_definite (miniapp generator), restored before every step",
                       "l2": "matrix (%.1f GB per GPU) is larger than L2; every step starts from a fresh copy" % (lr * lc * itemsize / 1e9),
                       "timing": "CUDA events on the launching stream per step, summed over K steps, max over ranks",
                       "wall_s_incl_restore": wall},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
            "gpu_library_reference": gpu_ref,
            "accuracy_vs_native_fp64_engine": accuracy,
            "residual_max_diff_over_max_a": residual,
            "residual_checker": "the product's distributed check_cholesky on the GPU grid (miniapp_cholesky.cpp:408-446), every world size",
            "residual_torch_checker": residual_torch,
            "residual_gate_eps_n": eps * n,
            "oracle_parity": parity,
            "next_rows": nxt,
            "step_ms": step_ms,
        }
        print(json.dumps(line), flush=True)
    pkg.free_grid(ctx)
    if world > 1:
        dist.destroy_process_group()


def run_next_rows(args):
    import torch

    pkg = ge.load_package()
    pkg.initialize()
    ctx = pkg.create_grid(None, 1, 1, "C")
    out = next_rows(pkg, ctx, torch, ge.load_oracle(), args.next_n, args.nb)
    print(json.dumps(out), flush=True)
    pkg.free_grid(ctx)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference_arm(a)
    elif a.impl == "next-rows":
        run_next_rows(a)
    else:
        run_ours(a)
