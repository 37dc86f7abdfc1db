"""The schedule of the triangular multiplication (trmm_engine.cu, tri_sweep.cuh) modelled on simulated P x Q grids
(tests/trmm_schedule_model.py) against the reference's closed forms: every side / uplo / op / diag combination and size of
its table, the reference's distributed source rank (P-1, min(1, Q-1)), padded tiles like the kernels'."""
import itertools

import numpy as np
import pytest

import trmm_oracle
import trmm_schedule_model as model

GRIDS = [(1, 1), (2, 1), (1, 2), (2, 2), (3, 2)]


@pytest.mark.parametrize("P,Q", GRIDS)
@pytest.mark.parametrize("t", ["d", "z"])
def test_schedule_model_closed_forms(oracle, P, Q, t):
    dt = oracle.DTYPES[t]
    alpha = oracle.TRIANGULAR_TEST_ALPHA if t == "z" else oracle.TRIANGULAR_TEST_ALPHA.real
    g = 8  # small granularity: tiles are padded, as on the GPU (128 / 64), but the model stays cheap
    for side, uplo, op, diag in itertools.product("LR", "LU", "NTC", "NU"):
        for m, n, mb, nb in oracle.TRIANGULAR_TEST_SIZES:
            a, b_in, expected = trmm_oracle.golden(oracle, side, uplo, op, diag, alpha, m, n, dt)
            out = model.run(side, uplo, op, diag, alpha, a, b_in, mb, nb, P, Q, g)
            tol = trmm_oracle.tolerance(m, dt)
            ok, _, msg = oracle.check_near(expected, out, tol, tol)
            assert ok, f"{P}x{Q} {side}{uplo}{op}{diag} m={m} n={n} mb={mb} nb={nb}: {msg}"


@pytest.mark.parametrize("P,Q", [(2, 2), (3, 2)])
def test_schedule_model_random_against_oracle(oracle, P, Q):
    rng = np.random.default_rng(11)
    for side, uplo, op in itertools.product("LR", "LU", "NC"):
        m, n, mb, nb = 37, 29, 6, 5
        na = m if side == "L" else n
        a = np.asfortranarray(rng.uniform(-1, 1, (na, na)) + 1j * rng.uniform(-1, 1, (na, na)))
        b = np.asfortranarray(rng.uniform(-1, 1, (m, n)) + 1j * rng.uniform(-1, 1, (m, n)))
        ref = b.copy(order="F")
        trmm_oracle.triangular_multiplication(side, uplo, op, "N", 0.5 - 2j, a, ref, mb, nb)
        out = model.run(side, uplo, op, "N", 0.5 - 2j, a, b, mb, nb, P, Q, 4)
        assert np.abs(out - ref).max() < 1e-12 * na * np.abs(ref).max()
