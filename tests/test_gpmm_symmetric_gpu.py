"""The mirror-symmetric GPMM built on the device (gingr_gpmm_gaussian_symmetric) against the literal 3M x 3M
approximateGPCholesky of scalismo's symmetrised kernel (oracle/symmetric.py), with the tolerances of
tests/test_gpmm_gpu.py; mirror symmetry of the built covariance; the trace criterion at scale; and the model in the
registration, posterior and cache paths."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

S = np.array([-1.0, 1.0, 1.0])


def _cloud(kind, n, seed=0):
    rng = np.random.default_rng(seed)
    from gingr_b200 import synthetic
    p = synthetic.fibonacci_sphere(n) + 0.5 * rng.normal(size=(n, 3))
    if kind == "plane":
        p[: n // 5, 0] = 0.0
    elif kind == "mirrored":
        h = p[p[:, 0] > 1.0][: (n - 3) // 2]
        p = np.vstack([h, h * S, rng.normal(size=(3, 3)) * [0.0, 60.0, 60.0]])
    elif kind == "far":
        p[:, 0] = np.abs(p[:, 0]) + 1e4
    return p


def _sym():
    from oracle import symmetric
    return symmetric


CASES = [("generic", 60, [70.0, 25.0], [50.0, 10.0], 0.01, 0), ("generic", 150, [70.0], [50.0], 0.01, 0),
         ("plane", 150, [60.0], [30.0], 0.12, 0), ("plane", 150, [60.0], [30.0], 0.16, 0),
         ("plane", 120, [40.0], [20.0], 0.001, 50), ("mirrored", 150, [70.0], [50.0], 0.05, 0),
         ("mirrored", 120, [60.0, 20.0], [30.0, 10.0], 0.1, 0), ("far", 120, [60.0], [30.0], 0.1, 0),
         ("generic", 90, [500.0], [5.0], 0.3, 0), ("plane", 100, [50.0], [30.0], 0.0, 7),
         ("plane", 100, [50.0], [30.0], 0.0, 20), ("generic", 100, [50.0], [30.0], 0.0, 31)]


@pytest.mark.parametrize("kind,M,sig,sc,tol,cap", CASES)
def test_symmetric_gpmm_matches_literal_construction(ctx, kind, M, sig, sc, tol, cap):
    from gingr_b200 import api
    ref = _cloud(kind, M)
    om, L = _sym().approximate_gp_cholesky_symmetric(ref, sig, sc, tol, cap or None)
    dm = api.Model.gaussianSymmetric(ctx, ref, None, sig, sc, tol, cap)
    assert dm.rank == om.rank
    gref, mean, basis, var = dm.download()
    assert np.array_equal(gref, ref) and np.all(mean == 0.0)
    assert np.max(np.abs(var - om.variance)) <= 1e-9 * om.variance[0]
    assert np.all(np.diff(var) <= 0.0)
    assert np.max(np.abs(basis.T @ basis - np.eye(dm.rank))) < 1e-10
    lit = L @ L.T
    assert np.max(np.abs((basis * var) @ basis.T - lit)) <= 1e-9 * np.max(np.abs(lit))
    on = np.flatnonzero(ref[:, 0] == 0.0)
    assert np.all(basis[3 * on, :] == 0.0)          # points on the plane stay on it, exactly
    dm.close()


def test_symmetric_model_is_mirror_symmetric(ctx):
    """K - C is PSD with trace <= relTol tr K, so max |P C P^T - C| <= 2 relTol tr K for the mirror operator P."""
    from gingr_b200 import api
    ref = _cloud("mirrored", 200, 3)
    M, tol, sig, sc = len(ref), 0.02, [60.0], [40.0]
    dm = api.Model.gaussianSymmetric(ctx, ref, None, sig, sc, tol)
    _, _, basis, var = dm.download()
    C = (basis * var) @ basis.T
    img = ref * S
    pi = np.array([int(np.argmin(np.sum((ref - img[i]) ** 2, axis=1))) for i in range(M)])
    assert all(np.array_equal(ref[pi[i]], img[i]) for i in range(M))
    P = np.zeros((3 * M, 3 * M))
    for i in range(M):
        for d in range(3):
            P[3 * pi[i] + d, 3 * i + d] = S[d]
    trK = float(np.trace(_sym().symmetric_gaussian_kernel_matrix(ref, sig, sc)))
    assert np.max(np.abs(P @ C @ P.T - C)) <= 2.0 * tol * trK
    dm.close()


def test_symmetric_gpmm_at_scale_meets_the_trace_criterion(ctx):
    from gingr_b200 import api, synthetic
    M = 20000
    ref = synthetic.fibonacci_sphere(M) + 0.5 * np.random.default_rng(0).normal(size=(M, 3))
    sig, sc, tol = 70.0, 50.0, 0.01
    dm = api.Model.gaussianSymmetric(ctx, ref, None, [sig], [sc], tol)
    _, _, basis, var = dm.download()
    e = sc * np.exp(-4.0 * ref[:, 0] ** 2 / (sig * sig))
    trK = float(np.sum(3.0 * sc + e))
    assert trK - var.sum() <= tol * trK * (1 + 1e-9)
    assert 30 <= dm.rank <= 6000
    assert np.max(np.abs(basis.T @ basis - np.eye(dm.rank))) < 1e-9
    diag_cov = np.einsum("ij,j,ij->i", basis, var, basis)
    kdiag = np.repeat(sc, 3 * M) + np.repeat(e, 3) * np.tile(S, M)
    assert np.all(diag_cov <= kdiag * (1 + 1e-9) + 1e-12 * sc)
    dm.close()


def test_symmetric_model_registers_like_the_uploaded_one(ctx, oracle):
    from gingr_b200 import api, synthetic
    ref = _cloud("generic", 300)
    tv, tt = synthetic.sphere_mesh(350)
    target = synthetic.make_target(tv, 0)
    dm = api.Model.gaussianSymmetric(ctx, ref, None, [70.0], [50.0], 0.01)
    gref, mean, basis, var = dm.download()
    um = api.Model(ctx, gref, mean, basis, var)
    dt = api.Target(ctx, target, tt)
    outs = []
    for model in (dm, um):
        reg = api.CpdRegistration(ctx, model, dt, api.CpdConfiguration(maxIterations=12, w=0.05))
        outs.append(reg.run(reg.initializeState(globalTransformation=api.RIGID_TRANSFORMS)))
        reg.close()
    diag = float(np.linalg.norm(ref.max(0) - ref.min(0)))
    assert np.max(np.abs(outs[0].fit - outs[1].fit)) < 1e-6 * diag
    assert abs(outs[0].sigma2 - outs[1].sigma2) <= 1e-6 * outs[1].sigma2
    om = oracle.Gpmm(gref, mean, np.ascontiguousarray(basis), var, None)
    oalgo = oracle.CpdAlgorithm(oracle.CpdConfig(max_iterations=12, w=0.05), literal=False)
    ofinal = oracle.run(oalgo, oracle.initial_state(om, target, tt, global_transformation=oracle.RIGID_TRANSFORMS))
    assert np.max(np.abs(outs[0].fit - ofinal.fit)) < 1e-6 * diag
    dm.close(); um.close(); dt.close()


def test_posterior_model_of_a_symmetric_model(ctx):
    from gingr_b200 import api
    ref = _cloud("plane", 200, 1)
    dm = api.Model.gaussianSymmetric(ctx, ref, None, [60.0], [10.0], 0.02)
    pid = np.arange(0, 200, 4, dtype=np.int32)
    pm = api.posterior_model(ctx, dm, np.eye(3), np.zeros(3), pid, ref[pid] + [0.0, 1.0, 0.0], np.full(len(pid), 0.5))
    _, mean, basis, var = pm.download()
    prior_var = dm.download()[3]
    assert pm.rank == dm.rank and np.all(np.isfinite(mean)) and np.all(np.diff(var) <= 0.0)
    assert np.max(np.abs(basis.T @ basis - np.eye(pm.rank))) < 1e-9
    assert var.sum() < prior_var.sum()
    assert np.all(mean[3 * np.flatnonzero(ref[:, 0] == 0.0)] == 0.0)     # the plane's x rows stay zero
    pm.close(); dm.close()


def test_model_cache_with_the_symmetric_kernel(ctx, tmp_path):
    import os
    from gingr_b200 import api, io
    ref = _cloud("plane", 90)
    k = api.GaussSymKernel(scaling=50.0, sigma=70.0)
    a = io.load_or_create_model(ctx, str(tmp_path), "blob", ref, None, k, relativeTolerance=0.05)
    path = os.path.join(str(tmp_path), "blob_dec-full_GaussSym_50.0_70.0.h5.json")
    assert os.path.isfile(path)
    stamp = os.stat(path).st_mtime_ns
    b = io.load_or_create_model(ctx, str(tmp_path), "blob", ref, None, k, relativeTolerance=0.05)
    assert os.stat(path).st_mtime_ns == stamp and a.rank == b.rank
    for x, y in zip(a.download(), b.download()):
        assert np.array_equal(x, y)
    a.close(); b.close()


def test_symmetric_gpmm_argument_errors(ctx):
    from gingr_b200 import api
    ref = _cloud("generic", 30)
    with pytest.raises(api.GingrError):
        api.Model.gaussianSymmetric(ctx, ref, None, [0.0], [1.0])
    with pytest.raises(api.GingrError):
        api.Model.gaussianSymmetric(ctx, ref, None, [1.0] * 9, [1.0] * 9)
    with pytest.raises(api.GingrError):
        api.Model.gaussianSymmetric(ctx, ref, None, [10.0], [1.0], relativeTolerance=1.5)
    with pytest.raises(api.GingrError):
        api.Model.gaussianSymmetric(ctx, ref, None, [10.0], [-1.0])
