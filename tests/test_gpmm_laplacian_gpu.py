"""The inverse-Laplacian GPMM built on the device (gingr_gpmm_inverse_laplacian) against oracle/laplacian.py: the
kernel entry by entry at full rank, the truncated models through their Nystrom form, the largest allowed template, and
the model in the registration, posterior, instance, download and cache paths.

Tolerance at full rank.  The device forms A = L + gamma I (or L + P) exactly (small integers and gamma), factorises it
(backward error ~ n u |A|), reads the identity rows out as L_A^-T and forms Y Y^T: the forward error of A^-1 is then
about n u kappa(A) |A^-1|.  The pivoted Cholesky of Ks (x) I3 at relTol 0 and the Jacobi rotations add a backward error
of ~ n u |Ks|, and numpy's SVD-based pinv has the same kappa-proportional error as the device.  Hence
    max |C - Ks (x) I3| <= 16 M u kappa(A) max |Ks|,
with kappa(A) = lambda_max(A) / lambda_min(A) computed from the eigenvalues of A (for gamma = 0, A = L + P, whose
eigenvalue on each component's constant vector is 1).

Truncated models.  Late in the factorisation a vertex whose neighbours are all pivots is decoupled from the rest, with
residual scaling / A_ii: vertices of equal degree tie exactly and rounding picks among them, differently on the device
and in numpy.  The pivot sets may then differ, but the trace history, and with it the rank, does not (a decoupled pivot
removes only its own residual).  What is checked in every case is therefore the defining property of the pivoted
Cholesky: the covariance of coordinate d is the Nystrom approximation Ks[:, S] Ks[S, S]^-1 Ks[S, :] of its pivot set S
(the points whose variance it reproduces exactly), with |S| summed over d equal to the rank of the reference, and the
total variance equal to the reference's.  Where the reference's pivot values are separated from the runner-up by far
more than rounding at every step the model uses (margin > 1e-6: the capped cases and the random meshes away from the
late decoupled stage), the pivot order is well defined, and the variances and the covariance must also match the
reference entry by entry, within the full-rank bound above."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

U = 2.0 ** -53


def _lap():
    from oracle import laplacian
    return laplacian


def _mesh(kind):
    from gingr_b200 import synthetic
    if kind == "icosphere":
        return synthetic.icosphere(3)                        # 642 vertices
    if kind == "patch":
        return synthetic.random_patch(300, 3)
    if kind == "two":
        a, ta = synthetic.random_sphere_mesh(250, 1)
        b, tb = synthetic.random_sphere_mesh(90, 2)
        return np.vstack([a, b + [300.0, 0.0, 0.0]]), np.vstack([ta, tb + 250])
    if kind == "isolated":                                   # a sphere plus one vertex in no triangle
        a, ta = synthetic.random_sphere_mesh(200, 4)
        return np.vstack([a, [[0.0, 0.0, 0.0]]]), ta
    raise ValueError(kind)


def _kappa(M, tri, gamma):
    lap = _lap()
    A = lap.graph_laplacian(M, tri) + (gamma * np.eye(M) if gamma > 0.0 else lap.projector(M, tri))
    ev = np.linalg.eigvalsh(A)
    return ev[-1] / ev[0]


def _nystrom_check(Ks, basis, var, rank):
    C = (basis * var) @ basis.T
    kmax = np.max(np.abs(Ks))
    taken = 0
    for d in range(3):
        for e in range(3):
            if e != d:
                assert np.max(np.abs(C[d::3, e::3])) <= 1e-10 * kmax
        Cd = C[d::3, d::3]
        # (a vertex with a zero kernel row -- isolated, gamma = 0 -- is never a pivot)
        S = np.flatnonzero((np.abs(np.diag(Ks) - np.diag(Cd)) <= 1e-9 * kmax) & (np.diag(Ks) > 1e-9 * kmax))
        ny = Ks[:, S] @ np.linalg.solve(Ks[np.ix_(S, S)], Ks[S, :])
        assert np.max(np.abs(Cd - ny)) <= 1e-8 * kmax
        taken += len(S)
    assert taken == rank


@pytest.mark.parametrize("kind", ["icosphere", "patch", "two", "isolated"])
@pytest.mark.parametrize("gamma", [0.0, 1e-3, 1.0])
@pytest.mark.parametrize("tol,cap", [(0.01, 0), (0.1, 0), (0.0, 301), (0.05, 200)])
def test_laplacian_gpmm_matches_the_oracle(ctx, kind, gamma, tol, cap):
    from gingr_b200 import api
    lap = _lap()
    ref, tri = _mesh(kind)
    M = len(ref)
    scaling = 20.0
    Ks = lap.inverse_laplacian_kernel_matrix(M, tri, scaling, gamma)
    rank, kd, Ls, margin = lap.triples_cholesky(Ks, tol, cap or None, with_margin=True)
    dm = api.Model.inverseLaplacian(ctx, ref, tri, scaling, gamma, tol, cap)
    assert dm.rank == rank
    gref, mean, basis, var = dm.download()
    assert np.array_equal(gref, ref) and np.all(mean == 0.0)
    assert np.all(np.diff(var) <= 0.0)
    assert np.max(np.abs(basis.T @ basis - np.eye(dm.rank))) < 1e-10
    assert abs(var.sum() - sum(np.sum(Ls[:, :k] ** 2) for k in kd)) <= 1e-9 * var.sum()
    _nystrom_check(Ks, basis, var, rank)
    if margin > 1e-6:
        rel = max(1e-9, 16 * M * U * _kappa(M, tri, gamma))
        lit = lap.triples_covariance(kd, Ls)
        ovar = np.sort(np.concatenate([np.linalg.svd(Ls[:, :k], compute_uv=False) ** 2 for k in kd]))[::-1]
        assert np.max(np.abs(var - ovar)) <= rel * ovar[0]
        assert np.max(np.abs((basis * var) @ basis.T - lit)) <= rel * np.max(np.abs(lit))
    dm.close()


def test_the_entrywise_comparison_covers_the_untied_cases():
    """The cases of test_laplacian_gpmm_matches_the_oracle whose pivot order is well defined are compared entry by entry;
    these are all capped cases on the random meshes and the gamma = 1e-3 models of the open patch."""
    lap = _lap()
    for kind in ("patch", "two", "isolated"):
        ref, tri = _mesh(kind)
        for gamma in (0.0, 1e-3, 1.0):
            Ks = lap.inverse_laplacian_kernel_matrix(len(ref), tri, 20.0, gamma)
            for tol, cap in ((0.0, 301), (0.05, 200)):
                assert lap.triples_cholesky(Ks, tol, cap, with_margin=True)[3] > 1e-6
    ref, tri = _mesh("patch")
    Ks = lap.inverse_laplacian_kernel_matrix(len(ref), tri, 20.0, 1e-3)
    assert all(lap.triples_cholesky(Ks, tol, None, with_margin=True)[3] > 1e-6 for tol in (0.01, 0.1))


@pytest.mark.parametrize("kind", ["icosphere", "patch", "two", "isolated"])
@pytest.mark.parametrize("gamma", [0.0, 1e-3, 1.0])
def test_full_rank_model_is_the_kernel(ctx, kind, gamma):
    """relTol 0: rank 3M for gamma > 0, 3 (M - #components) for gamma = 0 (there relTol 1e-12: the residual of the null
    space is rounding, ~u |Ks| per entry, far below 1e-12 tr Ks, and the smallest real pivot far above it)."""
    from gingr_b200 import api
    lap = _lap()
    ref, tri = _mesh(kind)
    M = len(ref)
    Ks = lap.inverse_laplacian_kernel_matrix(M, tri, 5.0, gamma)
    ncomp = lap.components(M, tri).max() + 1
    dm = api.Model.inverseLaplacian(ctx, ref, tri, 5.0, gamma, 0.0 if gamma > 0.0 else 1e-12)
    assert dm.rank == (3 * M if gamma > 0.0 else 3 * (M - ncomp))
    _, _, basis, var = dm.download()
    C = (basis * var) @ basis.T
    bound = 16 * M * U * _kappa(M, tri, gamma) * np.max(np.abs(Ks))
    assert np.max(np.abs(C - np.kron(Ks, np.eye(3)))) <= bound
    dm.close()


def test_largest_template_with_a_rank_cap(ctx):
    """M = 6000 (the limit), capped at 301 columns: rank, total variance and the covariance rows of 400 vertices
    against the scalar oracle on the same mesh (Ks by the inverse: gamma > 0, where pinv is the inverse)."""
    from gingr_b200 import api, synthetic
    lap = _lap()
    ref, tri = synthetic.random_patch(6000, 7)
    M = len(ref)
    L = np.zeros((M, M))
    e = np.concatenate([tri[:, [0, 1]], tri[:, [1, 2]], tri[:, [2, 0]]])
    L[e[:, 0], e[:, 1]] = L[e[:, 1], e[:, 0]] = -1.0
    L[np.diag_indices(M)] = -L.sum(axis=1)
    Ks = 10.0 * np.linalg.inv(L + 1.0 * np.eye(M))
    rank, kd, Ls = lap.triples_cholesky(Ks, 0.01, 301)
    dm = api.Model.inverseLaplacian(ctx, ref, tri, 10.0, 1.0, 0.01, 301)
    assert dm.rank == rank == 301
    _, _, basis, var = dm.download()
    assert abs(var.sum() - sum(np.sum(Ls[:, :k] ** 2) for k in kd)) <= 1e-9 * var.sum()
    rows = np.random.default_rng(0).choice(M, 400, replace=False)
    for d in range(3):
        F = Ls[:, :kd[d]]
        Cd = (basis[3 * rows + d] * var) @ basis[d::3].T
        assert np.max(np.abs(Cd - F[rows] @ F.T)) <= 1e-9 * np.max(np.abs(Ks))
    dm.close()


@pytest.mark.parametrize("algorithm", ["cpd", "icp"])
def test_registrations_with_a_laplacian_model_match_the_oracle(ctx, oracle, algorithm):
    from gingr_b200 import api, synthetic
    ref, tri = synthetic.icosphere(3)
    tv, tt = synthetic.sphere_mesh(700)
    target = synthetic.make_target(tv, 0)
    dm = api.Model.inverseLaplacian(ctx, ref, tri, 20.0, 0.0, 0.01)
    assert dm.rank <= 9472
    gref, mean, basis, var = dm.download()
    om = oracle.Gpmm(gref, mean, np.ascontiguousarray(basis), var, tri)
    dt = api.Target(ctx, target, tt)
    if algorithm == "cpd":
        reg = api.CpdRegistration(ctx, dm, dt, api.CpdConfiguration(maxIterations=6, w=0.05))
        oalgo = oracle.CpdAlgorithm(oracle.CpdConfig(max_iterations=6, w=0.05), literal=False)
    else:
        reg = api.IcpRegistration(ctx, dm, dt, api.IcpConfiguration(maxIterations=6, initialSigma=2.0, endSigma=0.5))
        oalgo = oracle.IcpAlgorithm(oracle.IcpConfig(max_iterations=6, initial_sigma=2.0, end_sigma=0.5))
    out = reg.run(reg.initializeState(globalTransformation=api.RIGID_TRANSFORMS))
    ofinal = oracle.run(oalgo, oracle.initial_state(om, target, tt, global_transformation=oracle.RIGID_TRANSFORMS))
    diag = float(np.linalg.norm(ref.max(0) - ref.min(0)))
    assert np.max(np.abs(out.fit - ofinal.fit)) < 1e-6 * diag
    assert abs(out.sigma2 - ofinal.sigma2) <= 1e-6 * max(ofinal.sigma2, 1e-12)
    reg.close(); dt.close(); dm.close()


def test_instance_posterior_and_round_trip(ctx):
    from gingr_b200 import api
    ref, tri = _mesh("patch")
    dm = api.Model.inverseLaplacian(ctx, ref, tri, 20.0, 1e-3, 0.02)
    gref, mean, basis, var = dm.download()
    alpha = np.random.default_rng(1).normal(size=dm.rank)
    fit = dm.instance(api.ModelFittingParameters(scale=1.0, translation=np.zeros(3), euler=(0.0, 0.0, 0.0), shape=alpha))
    expect = ref + (basis @ (np.sqrt(var) * alpha)).reshape(-1, 3)
    assert np.max(np.abs(fit - expect)) <= 1e-9 * np.max(np.abs(expect))
    um = api.Model(ctx, gref, mean, basis, var, tri)
    for x, y in zip(um.download(), (gref, mean, basis, var)):
        assert np.array_equal(x, y)
    pid = np.arange(0, len(ref), 5, dtype=np.int32)
    pm = api.posterior_model(ctx, dm, np.eye(3), np.zeros(3), pid, ref[pid] + [0.0, 0.0, 1.0], np.full(len(pid), 0.5))
    _, pmean, pbasis, pvar = pm.download()
    assert pm.rank == dm.rank and np.all(np.isfinite(pmean)) and np.all(np.diff(pvar) <= 0.0)
    assert np.max(np.abs(pbasis.T @ pbasis - np.eye(pm.rank))) < 1e-9
    assert pvar.sum() < var.sum()
    pm.close(); um.close(); dm.close()


def test_model_cache_with_the_laplacian_kernel(ctx, tmp_path):
    import os
    from gingr_b200 import api, io
    ref, tri = _mesh("patch")
    k = api.InvLapKernel(scaling=20.0, gamma=0.0)
    a = io.load_or_create_model(ctx, str(tmp_path), "patch", ref, tri, k, relativeTolerance=0.05)
    path = os.path.join(str(tmp_path), "patch_dec-full_InvLap_20.0_0.0.h5.json")
    assert os.path.isfile(path)
    stamp = os.stat(path).st_mtime_ns
    b = io.load_or_create_model(ctx, str(tmp_path), "patch", ref, tri, k, relativeTolerance=0.05)
    assert os.stat(path).st_mtime_ns == stamp and a.rank == b.rank
    for x, y in zip(a.download(), b.download()):
        assert np.array_equal(x, y)
    a.close(); b.close()


def test_laplacian_gpmm_argument_errors(ctx):
    from gingr_b200 import api
    from gingr_b200._native import GINGR_ERR_ARG, GINGR_ERR_UNSUPPORTED
    ref, tri = _mesh("patch")
    bad = [dict(tri=np.zeros((0, 3), np.int32)), dict(tri=None), dict(tri=np.vstack([tri, [[0, 1, len(ref)]]])),
           dict(tri=np.vstack([tri, [[-1, 1, 2]]])), dict(scaling=0.0), dict(scaling=-1.0), dict(scaling=np.inf),
           dict(scaling=np.nan), dict(gamma=-1e-9), dict(gamma=np.inf), dict(gamma=np.nan), dict(tol=-0.1),
           dict(tol=np.nan), dict(cap=-1)]
    for b in bad:
        a = dict(tri=tri, scaling=1.0, gamma=0.0, tol=0.01, cap=0)
        a.update(b)
        with pytest.raises(api.GingrError) as e:
            api.Model.inverseLaplacian(ctx, ref, a["tri"], a["scaling"], a["gamma"], a["tol"], a["cap"])
        assert e.value.code == GINGR_ERR_ARG, b
    from gingr_b200 import synthetic
    big, btri = synthetic.random_patch(6001, 5)
    with pytest.raises(api.GingrError) as e:
        api.Model.inverseLaplacian(ctx, big, btri, 1.0, 1.0, 0.01, 30)
    assert e.value.code == GINGR_ERR_UNSUPPORTED
    with pytest.raises(FloatingPointError):                  # (L + 1e-6 I)^-1 has entries ~1 / (M gamma): overflows
        api.Model.inverseLaplacian(ctx, ref, tri, 1e308, 1e-6)
