"""CPU checks of the triangular-multiplication oracle (tests/trmm_oracle.py) against the reference's closed forms, and of
the closed forms themselves: every side / uplo / op / diag combination, size of the reference's table and element type."""
import itertools

import numpy as np
import pytest

import trmm_oracle

TYPES = ["s", "d", "c", "z"]
COMBOS = list(itertools.product("LR", "LU", "NTC", "NU"))


def _alpha(oracle, dt):
    return oracle.TRIANGULAR_TEST_ALPHA if np.dtype(dt).kind == "c" else oracle.TRIANGULAR_TEST_ALPHA.real


@pytest.mark.parametrize("t", TYPES)
def test_oracle_reproduces_closed_forms(oracle, t):
    dt = oracle.DTYPES[t]
    alpha = _alpha(oracle, dt)
    for side, uplo, op, diag in COMBOS:
        for m, n, mb, nb in oracle.TRIANGULAR_TEST_SIZES:
            a, b_in, expected = trmm_oracle.golden(oracle, side, uplo, op, diag, alpha, m, n, dt)
            a0 = a.copy()
            b = b_in.copy(order="F")
            trmm_oracle.triangular_multiplication(side, uplo, op, diag, alpha, a, b, mb, nb)
            tol = trmm_oracle.tolerance(m, dt)
            ok, _, msg = oracle.check_near(expected, b, tol, tol)
            assert ok, f"{t} {side}{uplo}{op}{diag} m={m} n={n} mb={mb} nb={nb}: {msg}"
            assert np.array_equal(a, a0)


@pytest.mark.parametrize("side,uplo,op,diag", COMBOS)
def test_golden_triple_is_the_product(oracle, side, uplo, op, diag):
    """Plain numpy: B_expected = alpha op(A) B_in (Left) / alpha B_in op(A) (Right) with the referenced triangle of A."""
    alpha = oracle.TRIANGULAR_TEST_ALPHA
    for m, n, _, _ in oracle.TRIANGULAR_TEST_SIZES:
        a, b_in, expected = trmm_oracle.golden(oracle, side, uplo, op, diag, alpha, m, n, np.complex128)
        t = np.tril(a) if uplo == "L" else np.triu(a)
        if diag == "U":
            t = t - np.diag(np.diag(t)) + np.eye(t.shape[0])
        opa = {"N": t, "T": t.T, "C": t.conj().T}[op]
        prod = alpha * (opa @ b_in if side == "L" else b_in @ opa)
        assert np.allclose(prod, expected, rtol=1e-12, atol=1e-12 * max(1.0, np.abs(expected).max(initial=0)))


@pytest.mark.parametrize("t,m,n,mb,nb", [("d", 130, 70, 32, 16), ("z", 50, 90, 16, 24), ("s", 64, 33, 16, 8)])
@pytest.mark.parametrize("side,uplo,op,diag", [("L", "L", "N", "N"), ("L", "U", "C", "U"), ("R", "L", "T", "N"), ("R", "U", "C", "N")])
def test_oracle_random_against_dense_product(oracle, t, m, n, mb, nb, side, uplo, op, diag):
    """Random data with ragged tiles: the tile loops equal the dense product (the unreferenced triangle holds garbage)."""
    dt = oracle.DTYPES[t]
    rng = np.random.default_rng(5)
    na = m if side == "L" else n
    a = rng.uniform(-1, 1, (na, na)) + (1j * rng.uniform(-1, 1, (na, na)) if np.dtype(dt).kind == "c" else 0)
    b = rng.uniform(-1, 1, (m, n)) + (1j * rng.uniform(-1, 1, (m, n)) if np.dtype(dt).kind == "c" else 0)
    a, b = np.asfortranarray(a.astype(dt)), np.asfortranarray(b.astype(dt))
    alpha = _alpha(oracle, dt)
    tri = np.tril(a) if uplo == "L" else np.triu(a)
    if diag == "U":
        tri = tri - np.diag(np.diag(tri)) + np.eye(na, dtype=dt)
    opa = {"N": tri, "T": tri.T, "C": tri.conj().T}[op].astype(np.complex128)
    ref = alpha * (opa @ b if side == "L" else b @ opa)
    out = b.copy(order="F")
    trmm_oracle.triangular_multiplication(side, uplo, op, diag, alpha, a, out, mb, nb)
    eps = np.finfo(np.dtype(dt).type(0).real.dtype).eps
    assert np.abs(out - ref).max() <= 10 * na * eps * max(1.0, np.abs(ref).max())
