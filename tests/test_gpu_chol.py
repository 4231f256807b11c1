"""The one-CTA Cholesky (csrc/chol.cuh) on its own, through api.chol_probe: the factor L of an SPD matrix A and the
carried rows X L^-T against NumPy, at every m mod 8 (partial last diagonal tile, carried rows inside it, pure
carried tile rows), at the state sizes the filter runs (180 window pivots, 202 = 30-clone state, 210 = hybrid), and
bit for bit across two runs."""
import numpy as np
import pytest

from orcvio_b200 import api

pytestmark = pytest.mark.gpu

MS = list(range(8, 18)) + [64, 180, 202, 210]
NXS = [0, 1, 7, 17, 22]


def _problem(m, nx):
    rng = np.random.default_rng(1000 * m + nx)
    B = rng.standard_normal((m, m))
    A = B @ B.T / m + np.eye(m)            # eigenvalues in about [1, 5]: well conditioned
    X = rng.standard_normal((nx, m)) if nx else None
    return A, X


@pytest.mark.parametrize("nx", NXS)
@pytest.mark.parametrize("m", MS)
def test_chol_probe_matches_numpy(m, nx):
    A, X = _problem(m, nx)
    L, Xs, _, _ = api.chol_probe(A, X, reps=1)
    Lr = np.linalg.cholesky(A)
    assert np.array_equal(np.triu(L, 1), np.zeros((m, m)))
    assert np.abs(L - Lr).max() <= 1e-12 * np.abs(Lr).max()
    if nx:
        Xr = np.linalg.solve(Lr, X.T).T
        assert np.abs(Xs - Xr).max() <= 1e-12 * np.abs(Xr).max()
    L2, Xs2, _, _ = api.chol_probe(A, X, reps=1)
    assert L.tobytes() == L2.tobytes()
    if nx:
        assert Xs.tobytes() == Xs2.tobytes()
