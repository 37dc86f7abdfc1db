"""GPU tests of the triangular multiplication (dlaf_b200_triangular_multiplication_*, trmm_engine.cu) through the C ABI,
mirroring test/unit/multiplication/test_multiplication_triangular.cpp: the reference's closed forms for every side / uplo /
op / diag combination and size of its table, random products against the oracle's tile loops (tests/trmm_oracle.py) on
every update engine, the device flavour, the int8 digit guard, round trips with the solver and the Cholesky factor, and
the distributed sweep on 2, 4 and 8 GPUs."""
import itertools
import os
import subprocess
import sys

import numpy as np
import pytest

import trmm_oracle

pytestmark = pytest.mark.gpu

TYPES = ["s", "d", "c", "z"]
HERE = os.path.dirname(os.path.abspath(__file__))


def _alpha(oracle, dt):
    return oracle.TRIANGULAR_TEST_ALPHA if np.dtype(dt).kind == "c" else oracle.TRIANGULAR_TEST_ALPHA.real


def _random_problem(oracle, dt, side, uplo, m, n, mb, nb, seed=3):
    """the Cholesky factor of the miniapp's matrix scaled to O(1) entries, -9.9 in its unreferenced triangle; random B"""
    rng = np.random.default_rng(seed)
    na, ba = (m, mb) if side == "L" else (n, nb)
    spd = oracle.set_random_hermitian_positive_definite(na, ba, dt)
    assert oracle.cholesky_local(uplo, spd, ba) == 0
    tri = np.tril if uplo == "L" else np.triu
    other = np.triu(np.full((na, na), -9.9), 1) if uplo == "L" else np.tril(np.full((na, na), -9.9), -1)
    a = np.asfortranarray((tri(spd) / np.sqrt(na) + other).astype(dt))
    b = rng.uniform(-1, 1, (m, n))
    if np.dtype(dt).kind == "c":
        b = b + 1j * rng.uniform(-1, 1, (m, n))
    return a, np.asfortranarray(b.astype(dt))


def _check_against_oracle(pkg, oracle, grid11, t, m, n, mb, nb, side, uplo, op, diag="N"):
    dt = pkg.TYPES[t]
    a, b = _random_problem(oracle, dt, side, uplo, m, n, mb, nb)
    alpha = _alpha(oracle, dt)
    ref = b.copy(order="F")
    trmm_oracle.triangular_multiplication(side, uplo, op, diag, alpha, a, ref, mb, nb)
    out = b.copy(order="F")
    pkg.triangular_multiplication(grid11, side, uplo, op, diag, alpha, a, out, mb, nb)
    tol = trmm_oracle.tolerance(max(m, n), dt) * max(1.0, float(np.abs(ref).max()))
    ok, _, msg = oracle.check_near(ref, out, tol, tol)
    assert ok, f"{t} {side}{uplo}{op}{diag} m={m} n={n} mb={mb} nb={nb}: {msg}"
    return out


@pytest.mark.parametrize("t", TYPES)
def test_closed_forms_all_combinations(pkg, oracle, grid11, t):
    dt = pkg.TYPES[t]
    alpha = _alpha(oracle, dt)
    for side, uplo, op, diag in itertools.product("LR", "LU", "NTC", "NU"):
        for m, n, mb, nb in oracle.TRIANGULAR_TEST_SIZES:
            a, b, expected = trmm_oracle.golden(oracle, side, uplo, op, diag, alpha, m, n, dt)
            a0 = a.copy(order="F")
            pkg.triangular_multiplication(grid11, side, uplo, op, diag, alpha, a, b, mb, nb)
            tol = trmm_oracle.tolerance(m, dt)
            ok, _, msg = oracle.check_near(expected, b, tol, tol)
            assert ok, f"{t} {side}{uplo}{op}{diag} m={m} n={n} mb={mb} nb={nb}: {msg}"
            assert np.array_equal(a, a0), "the triangular matrix is read-only"
    assert pkg.last_solver_launch_count(grid11) > 0


@pytest.mark.parametrize("t,m,n,mb,nb", [("d", 1536, 1024, 512, 512), ("d", 700, 300, 100, 64), ("s", 640, 512, 128, 128),
                                         ("z", 512, 384, 64, 64), ("c", 300, 200, 96, 64), ("d", 1024, 768, 256, 128),
                                         ("z", 384, 600, 96, 64)])
@pytest.mark.parametrize("side,uplo,op", [("L", "L", "N"), ("L", "L", "C"), ("L", "U", "T"), ("L", "U", "N"), ("R", "L", "N"),
                                          ("R", "L", "C"), ("R", "U", "T"), ("R", "U", "N")])
def test_random_products_match_oracle(pkg, oracle, grid11, t, m, n, mb, nb, side, uplo, op):
    _check_against_oracle(pkg, oracle, grid11, t, m, n, mb, nb, side, uplo, op)


@pytest.mark.parametrize("t", ["d", "z"])
def test_device_flavour_equals_host_flavour(pkg, oracle, grid11, t):
    import torch

    dt = pkg.TYPES[t]
    m, n, mb, nb = 768, 640, 256, 128
    for side, uplo, op in [("L", "L", "N"), ("R", "U", "C")]:
        a, b = _random_problem(oracle, dt, side, uplo, m, n, mb, nb)
        host = b.copy(order="F")
        pkg.triangular_multiplication(grid11, side, uplo, op, "N", 1.5, a, host, mb, nb)
        # column-major device copies: the transpose of a contiguous row-major tensor
        da = torch.from_numpy(np.ascontiguousarray(a.T)).cuda()
        db = torch.from_numpy(np.ascontiguousarray(b.T)).cuda()
        torch.cuda.synchronize()
        pkg.triangular_multiplication_device(grid11, side, uplo, op, "N", 1.5, da.data_ptr(), db.data_ptr(), dt, m, n, mb, nb,
                                             a.shape[0], m, stream=torch.cuda.current_stream().cuda_stream)
        dev = db.cpu().numpy().T
        assert np.array_equal(dev, host)
        assert np.array_equal(da.cpu().numpy().T, a)


def test_native_fp64_engine_matches_oracle(pkg, oracle, grid11, monkeypatch):
    """DLAF_B200_D_BULK=dmma (native fp64 products) and the default int8 digit engine both meet the tolerance."""
    for side, uplo, op in [("L", "L", "N"), ("R", "U", "C")]:
        default = _check_against_oracle(pkg, oracle, grid11, "d", 1024, 1024, 512, 512, side, uplo, op)
        monkeypatch.setenv("DLAF_B200_D_BULK", "dmma")
        native = _check_against_oracle(pkg, oracle, grid11, "d", 1024, 1024, 512, 512, side, uplo, op)
        monkeypatch.delenv("DLAF_B200_D_BULK")
        assert not np.array_equal(default, native), "the two engines round differently"


def test_guard_on_rows_spanning_many_binades(pkg, oracle, grid11):
    """Rows of Y that span more than 40 binades: the int8 digit guard sends those steps to the native kernel, and the
    result still meets the tolerance componentwise (against |op(A)| |B|, the bound of a native product)."""
    m, n, nb = 1024, 768, 256
    a, b = _random_problem(oracle, np.float64, "R", "L", m, n, nb, nb)
    rng = np.random.default_rng(7)
    b = np.asfortranarray(b * np.exp2(-rng.integers(0, 60, size=b.shape)))
    ref = b.copy(order="F")
    trmm_oracle.triangular_multiplication("R", "L", "N", "N", 1.0, a, ref, nb, nb)
    out = b.copy(order="F")
    pkg.triangular_multiplication(grid11, "R", "L", "N", "N", 1.0, a, out, nb, nb)
    assert pkg.last_inverse_guard_steps(grid11) > 0
    bound = np.abs(b) @ np.abs(np.tril(a))
    assert (np.abs(out - ref) <= trmm_oracle.tolerance(n, np.float64) * bound).all()


@pytest.mark.parametrize("t", TYPES)
def test_multiplication_then_solve_restores_b(pkg, oracle, grid11, t):
    dt = pkg.TYPES[t]
    m, n, mb, nb = 512, 384, 128, 128
    for side, uplo, op in [("L", "L", "N"), ("L", "U", "C"), ("R", "L", "T"), ("R", "U", "N")]:
        a, b = _random_problem(oracle, dt, side, uplo, m, n, mb, nb)
        na = m if side == "L" else n
        a = np.asfortranarray((a * np.sqrt(na)).astype(dt))  # the factor itself: well conditioned
        x = b.copy(order="F")
        pkg.triangular_multiplication(grid11, side, uplo, op, "N", 2.0, a, x, mb, nb)
        pkg.triangular_solver(grid11, side, uplo, op, "N", 1.0, a, x, mb, nb)
        eps = np.finfo(np.dtype(dt).type(0).real.dtype).eps
        assert np.abs(x - 2.0 * b).max() <= 200 * na * eps * np.abs(b).max()


def test_apply_cholesky_factor_end_to_end(pkg, oracle, grid11):
    """L (L^H X) with the factor of cholesky_factorization equals A X (fp64, config-sized tiles)."""
    n, nb, nrhs = 2048, 512, 256
    a = oracle.set_random_hermitian_positive_definite(n, nb, np.float64)
    f = a.copy(order="F")
    assert pkg.cholesky_factorization(grid11, "L", f, nb) == 0
    rng = np.random.default_rng(9)
    x = np.asfortranarray(rng.uniform(-1, 1, (n, nrhs)))
    y = x.copy(order="F")
    pkg.triangular_multiplication(grid11, "L", "L", "C", "N", 1.0, f, y, nb, 128)
    pkg.triangular_multiplication(grid11, "L", "L", "N", "N", 1.0, f, y, nb, 128)
    ax = a @ x
    assert np.abs(y - ax).max() <= 50 * n * np.finfo(np.float64).eps * np.abs(a).max() * np.abs(x).max()


@pytest.mark.parametrize("t", TYPES)
def test_zero_alpha_and_empty(pkg, grid11, t):
    dt = pkg.TYPES[t]
    a = np.asfortranarray(np.full((300, 300), np.nan).astype(dt))
    b = np.asfortranarray(np.full((300, 200), np.nan).astype(dt))
    pkg.triangular_multiplication(grid11, "L", "L", "N", "N", 0.0, a, b, 128, 128)
    assert (b == 0).all()
    b = np.asfortranarray(np.full((200, 300), np.nan).astype(dt))
    pkg.triangular_multiplication(grid11, "R", "U", "C", "U", 0.0, a, b, 64, 100)
    assert (b == 0).all()
    for m, n in [(0, 5), (5, 0), (0, 0)]:
        aa = np.zeros((max(1, m), max(1, m)), dtype=dt, order="F")
        bb = np.asfortranarray(np.ones((max(1, m), max(1, n)), dtype=dt))
        pkg.triangular_multiplication(grid11, "L", "L", "N", "N", 1.0, aa, bb, 4, 4, m=m, n=n)
        assert (bb == 1).all()


def _ngpus():
    try:
        import torch

        return torch.cuda.device_count()
    except Exception:
        return 0


def _launch(nproc, grid, order, port):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(HERE, "trmm_dist_worker.py"), "--grid", grid, "--order", order]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1800, env=dict(os.environ, MASTER_ADDR="127.0.0.1"))
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    assert "total failures 0" in r.stdout, r.stdout[-2000:]


@pytest.mark.parametrize("grid,order,nproc", [("2x1", "R", 2), ("1x2", "C", 2), ("2x2", "C", 4), ("1x4", "R", 4), ("2x4", "C", 8),
                                              ("3x2", "R", 8)])
def test_distributed_multiplication(grid, order, nproc):
    if _ngpus() < nproc:
        pytest.skip(f"needs {nproc} GPUs")
    _launch(nproc, grid, order, 29641)
