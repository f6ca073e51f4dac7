"""The reflection sign of the Umeyama / Kabsch solve in oracle.umeyama and template.umeyama (CPU only).

The sign is det U det V of Sxy = U diag(s) V^T.  It equals sign det Sxy when Sxy has full rank; for a planar shape
(Sxy of rank 2, det Sxy = +-0 or rounding noise) only det U det V makes U diag(1, 1, d) V^T a rotation.  The device's
solve (update.cu procrustes_solve_dev) takes the same rule and is checked in test_update_phase_gpu.py."""
import numpy as np
import pytest

from gingr_b200.rotation import euler_to_matrix


def _solvers():
    from gingr_b200 import template
    from oracle import oracle
    return [("oracle", oracle.umeyama), ("template", template.umeyama)]


def _planted(seed):
    rng = np.random.default_rng(seed)
    e = (rng.uniform(-np.pi, np.pi), rng.uniform(-1.3, 1.3), rng.uniform(-np.pi, np.pi))
    return np.asarray(euler_to_matrix(*e), dtype=float), rng.normal(size=3)


@pytest.mark.parametrize("similarity", [False, True], ids=["rigid", "similarity"])
@pytest.mark.parametrize("which", [0, 1], ids=["oracle", "template"])
def test_planar_inputs_recover_the_planted_rotation(which, similarity):
    _, solve = _solvers()[which]
    for seed in range(200):
        rng = np.random.default_rng(1000 + seed)
        X = np.column_stack([rng.uniform(-0.5, 0.5, 50), rng.uniform(-1.2, 1.2, 50), np.zeros(50)])
        if seed % 2:
            X = X[:, [0, 2, 1]]   # the plane y = 0
        R, t = _planted(seed)
        c = 1.7 if similarity else 1.0
        Y = c * X @ R.T + t
        Rg, tg, cg = solve(X, Y, similarity)
        assert abs(np.linalg.det(Rg) - 1.0) < 1e-12
        assert np.max(np.abs(Rg - R)) < 1e-9, seed
        assert np.max(np.abs(tg - t)) < 1e-9 and abs(cg - c) < 1e-9


@pytest.mark.parametrize("which", [0, 1], ids=["oracle", "template"])
def test_collinear_inputs_reach_the_optimum(which):
    """Rank 1: the rotation is not unique, but tr(R^T Sxy) must reach s_0, its maximum over rotations."""
    _, solve = _solvers()[which]
    for seed in range(50):
        rng = np.random.default_rng(2000 + seed)
        X = np.outer(rng.uniform(-1, 1, 40), rng.normal(size=3))
        R, t = _planted(seed)
        Y = X @ R.T + t + 1e-3 * rng.normal(size=X.shape)
        Rg, _, _ = solve(X, Y, False)
        Sxy = (Y - Y.mean(0)).T @ (X - X.mean(0)) / len(X)
        s = np.linalg.svd(Sxy, compute_uv=False)
        assert abs(np.linalg.det(Rg) - 1.0) < 1e-12
        assert s[1] < 1e-12 * s[0]
        assert np.trace(Rg.T @ Sxy) >= s[0] * (1.0 - 1e-12), seed


@pytest.mark.parametrize("which", [0, 1], ids=["oracle", "template"])
def test_full_rank_sign_is_sign_det(which):
    """Full rank, proper and mirrored: the rule gives the sign det Sxy result."""
    _, solve = _solvers()[which]
    for seed in range(50):
        rng = np.random.default_rng(3000 + seed)
        X = rng.normal(size=(30, 3))
        R, t = _planted(seed)
        mirror = np.diag([1.0, 1.0, -1.0]) if seed % 2 else np.eye(3)
        Y = X @ (R @ mirror).T + t
        Rg, _, _ = solve(X, Y, False)
        Sxy = (Y - Y.mean(0)).T @ (X - X.mean(0)) / len(X)
        U, s, Vt = np.linalg.svd(Sxy)
        J = np.diag([1.0, 1.0, -1.0 if np.linalg.det(Sxy) < 0 else 1.0])
        assert np.max(np.abs(Rg - U @ J @ Vt)) < 1e-9
