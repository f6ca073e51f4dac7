"""The GP posterior as a device model (gingr_model_posterior, gingr_registration_posterior_model) against scalismo's
definition restated with the oracle: model.transform(R, t).posterior(obs) has reference R ref + t, mean
posed.mean + posed.basis (D c), basis posed.basis U and variance s with svd(D Minv D) = U diag(s) U^T
(oracle.posterior_model for the registration-level form).  Tolerances: variances 1e-9 of the largest, covariances 1e-9
of the largest prior variance, mean and reference 1e-9 of the bounding-box diagonal; the basis is compared up to sign
where an eigenvalue is simple and through its covariance elsewhere."""
import dataclasses

import numpy as np
import pytest

from test_posterior_model_host import _reference_posterior
from test_update_gpu import _compare, _problem, _to_api_state

pytestmark = pytest.mark.gpu


def _gpmm(oracle, M, r, seed=0, orthonormal=True):
    from gingr_b200 import synthetic
    ref, tri = synthetic.sphere_mesh(M)
    _, basis, var = synthetic.make_gpmm(ref, r, seed, orthonormal=orthonormal)
    mean = np.random.default_rng(seed + 7).normal(scale=0.5, size=3 * M)
    return oracle.Gpmm(ref, mean, basis, var, tri)


def _upload(ctx, m):
    from gingr_b200 import api
    return api.Model(ctx, m.ref, m.mean, m.basis, m.variance, m.tri)


def _as_oracle(oracle, dm):
    ref, mean, basis, var = dm.download()
    return oracle.Gpmm(ref, mean, np.ascontiguousarray(basis), var, dm.triangles)


def _diag(m):
    return float(np.linalg.norm(m.ref.max(0) - m.ref.min(0)))


def _check_against(got, want, lam_max, diag, full_cov=True):
    s_max = float(np.max(want.variance))
    assert np.max(np.abs(got.variance - want.variance)) <= 1e-9 * s_max
    assert np.all(np.diff(got.variance) <= 0.0)
    assert np.max(np.abs(got.ref - want.ref)) <= 1e-9 * diag
    assert np.max(np.abs(got.mean - want.mean)) <= 1e-9 * diag
    if full_cov:
        Kg = (got.basis * got.variance) @ got.basis.T
        Kw = (want.basis * want.variance) @ want.basis.T
        assert np.max(np.abs(Kg - Kw)) <= 1e-9 * lam_max
    # eigenvectors up to sign where the eigenvalue is simple (relative gap to both neighbours)
    s = want.variance
    gap = np.minimum(np.abs(np.diff(s, prepend=np.inf)), np.abs(np.diff(s, append=-np.inf)))
    simple = np.nonzero(gap > 1e-3 * s_max)[0]
    for j in simple:
        a, b = got.basis[:, j], want.basis[:, j]
        sg = 1.0 if a @ b >= 0 else -1.0
        assert np.max(np.abs(a - sg * b)) <= 1e-6 * max(np.max(np.abs(b)), 1e-300), j


def _observations(m, R, t, kind, rng):
    M, r = m.M, m.rank
    posed = m.transform(R, t)
    if kind == "iso":
        obs = posed.instance(rng.normal(size=r)) + rng.normal(scale=0.3, size=(M, 3))
        pids = rng.permutation(M)[: max(3, (3 * M) // 4)].astype(np.int32)
        var = rng.uniform(0.05, 5.0, size=M)[pids]
        return pids, obs[pids], var, np.eye(3)[None] * var[:, None, None]
    n = max(6, M // 3)
    pids = rng.integers(0, M, size=n).astype(np.int32)
    pids[1] = pids[0]                                               # one vertex observed twice
    obs = posed.instance(rng.normal(size=r))[pids] + rng.normal(scale=0.5, size=(n, 3))
    A = rng.normal(size=(n, 3, 3))
    cov = A @ np.transpose(A, (0, 2, 1)) + 0.1 * np.eye(3)
    return pids, obs, cov, cov


@pytest.mark.parametrize("M,r", [(60, 12), (300, 130), (1000, 257)])
@pytest.mark.parametrize("kind", ["iso", "full"])
@pytest.mark.parametrize("posed", [False, True])
def test_kernel_level_matches_scalismo_posterior(ctx, oracle, M, r, kind, posed):
    from gingr_b200 import api
    m = _gpmm(oracle, M, r, seed=M + r)
    dm = _upload(ctx, m)
    rng = np.random.default_rng(M)
    R, t = (oracle.euler_to_matrix(0.2, -0.1, 0.3), np.array([3.0, -2.0, 1.0])) if posed else (np.eye(3), np.zeros(3))
    pids, pts, noise, cov = _observations(m, R, t, kind, rng)
    pm = api.posterior_model(ctx, dm, R, t, pids, pts, noise)
    got = _as_oracle(oracle, pm)
    want = _reference_posterior(oracle, m, R, t, pids, pts, cov)
    _check_against(got, want, float(m.variance.max()), _diag(m), full_cov=M <= 300)
    assert np.max(np.abs(got.basis.T @ got.basis - np.eye(r))) <= 1e-12
    assert np.array_equal(pm.reference, got.ref) and pm.rank == r and pm.M == M


def test_kronecker_model_degenerate_eigenspaces(ctx, oracle):
    """A Ks (x) I3 model (device-built GPMM) with isotropic noise: the eigenvalues come in triples, so the basis is
    compared through the projectors onto each eigenvalue cluster (and the covariance)."""
    from gingr_b200 import api, synthetic
    ref, tri = synthetic.sphere_mesh(200)
    dm = api.Model.gaussianMixture(ctx, ref, tri, [60.0], [10.0], relativeTolerance=0.02)
    m = _as_oracle(oracle, dm)
    rng = np.random.default_rng(9)
    pids = np.arange(0, m.M, 2, dtype=np.int32)
    pts = m.instance(rng.normal(size=m.rank))[pids] + rng.normal(scale=0.2, size=(len(pids), 3))
    var = np.full(len(pids), 0.5)
    R, t = oracle.euler_to_matrix(0.1, 0.2, -0.3), np.array([1.0, 2.0, 3.0])
    got = _as_oracle(oracle, api.posterior_model(ctx, dm, R, t, pids, pts, var))
    want = _reference_posterior(oracle, m, R, t, pids, pts, np.eye(3)[None] * var[:, None, None])
    _check_against(got, want, float(m.variance.max()), _diag(m))
    s = want.variance
    starts = [0] + [j for j in range(1, len(s)) if s[j - 1] - s[j] > 1e-6 * s[0]] + [len(s)]
    for a, b in zip(starts[:-1], starts[1:]):
        Pg = got.basis[:, a:b] @ got.basis[:, a:b].T
        Pw = want.basis[:, a:b] @ want.basis[:, a:b].T
        assert np.max(np.abs(Pg - Pw)) <= 1e-6, (a, b)


@pytest.mark.parametrize("which", ["non_orthonormal", "new_reference"])
def test_non_orthonormal_bases(ctx, oracle, which):
    from gingr_b200 import api, synthetic
    if which == "non_orthonormal":
        m = _gpmm(oracle, 300, 90, seed=2, orthonormal=False)
        dm = _upload(ctx, m)
    else:
        base = _gpmm(oracle, 400, 90, seed=3)
        new_ref, new_tri = synthetic.sphere_mesh(250, radius=99.0)
        dm = _upload(ctx, base).newReference(new_ref, new_tri)
        m = base.new_reference(new_ref, new_tri)
    rng = np.random.default_rng(5)
    R, t = oracle.euler_to_matrix(-0.2, 0.1, 0.05), np.array([0.5, -1.0, 2.0])
    pids, pts, noise, cov = _observations(m, R, t, "iso", rng)
    got = _as_oracle(oracle, api.posterior_model(ctx, dm, R, t, pids, pts, noise))
    want = _reference_posterior(oracle, m, R, t, pids, pts, cov)
    _check_against(got, want, float(m.variance.max()), _diag(m))


def test_no_observations_give_the_posed_prior(ctx, oracle):
    from gingr_b200 import api
    m = _gpmm(oracle, 120, 30, seed=4)
    dm = _upload(ctx, m)
    R, t = oracle.euler_to_matrix(0.3, 0.0, -0.2), np.array([1.0, 1.0, -1.0])
    got = _as_oracle(oracle, api.posterior_model(ctx, dm, R, t, np.zeros(0, np.int32), np.zeros((0, 3)), np.zeros(0)))
    posed = m.transform(R, t)
    assert np.max(np.abs(got.variance - m.variance)) <= 1e-12 * m.variance.max()
    Kg = (got.basis * got.variance) @ got.basis.T
    Kw = (posed.basis * posed.variance) @ posed.basis.T
    assert np.max(np.abs(Kg - Kw)) <= 1e-9 * m.variance.max()
    assert np.max(np.abs(got.mean - posed.mean)) <= 1e-9 * _diag(m)
    assert np.max(np.abs(got.ref - posed.ref)) <= 1e-9 * _diag(m)


def test_zero_variances_keep_their_unit_vectors(ctx, oracle):
    from gingr_b200 import api
    m = _gpmm(oracle, 150, 40, seed=6)
    m.variance[[3, 17]] = 0.0
    dm = _upload(ctx, m)
    rng = np.random.default_rng(6)
    R, t = oracle.euler_to_matrix(0.1, -0.2, 0.3), np.array([2.0, 0.0, 1.0])
    pids, pts, noise, cov = _observations(m, R, t, "iso", rng)
    got = _as_oracle(oracle, api.posterior_model(ctx, dm, R, t, pids, pts, noise))
    want = _reference_posterior(oracle, m, R, t, pids, pts, cov)
    posed = m.transform(R, t)
    assert np.all(got.variance[-2:] == 0.0) and np.all(got.variance[:-2] > 0.0)
    assert np.max(np.abs(got.basis[:, -2:] - posed.basis[:, [3, 17]])) <= 1e-14 * np.max(np.abs(posed.basis))
    _check_against(dataclasses.replace(got, basis=got.basis[:, :-2], variance=got.variance[:-2]),
                   dataclasses.replace(want, basis=want.basis[:, :-2], variance=want.variance[:-2]),
                   float(m.variance.max()), _diag(m))


def test_non_finite_noise_raises_without_a_handle(ctx, oracle):
    from gingr_b200 import api
    m = _gpmm(oracle, 60, 12)
    dm = _upload(ctx, m)
    pids = np.arange(10, dtype=np.int32)
    noise = np.ones(10)
    noise[4] = np.nan
    with pytest.raises(FloatingPointError):
        api.posterior_model(ctx, dm, np.eye(3), np.zeros(3), pids, m.ref[pids], noise)
    with pytest.raises(ValueError):
        api.posterior_model(ctx, dm, np.eye(3), np.zeros(3), pids, m.ref[pids], np.ones(9))


def test_two_calls_are_bit_identical(ctx, oracle):
    from gingr_b200 import api
    m = _gpmm(oracle, 300, 130, seed=8)
    dm = _upload(ctx, m)
    rng = np.random.default_rng(8)
    R, t = oracle.euler_to_matrix(0.2, 0.1, 0.0), np.array([1.0, 0.0, 0.0])
    pids, pts, noise, _ = _observations(m, R, t, "iso", rng)
    a = api.posterior_model(ctx, dm, R, t, pids, pts, noise).download()
    b = api.posterior_model(ctx, dm, R, t, pids, pts, noise).download()
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


def test_the_new_model_is_a_first_class_handle(ctx, oracle):
    """Three CPD updates on the posterior model against the oracle on its download, instance(), and a round trip."""
    from gingr_b200 import api
    m, target, tt = _problem(oracle, 150, 180, 24, seed=11)
    dm = _upload(ctx, m)
    rng = np.random.default_rng(11)
    R, t = oracle.euler_to_matrix(0.05, 0.02, -0.03), np.array([0.5, 0.5, -0.5])
    pids, pts, noise, _ = _observations(m, R, t, "iso", rng)
    pm = api.posterior_model(ctx, dm, R, t, pids, pts, noise)
    om = _as_oracle(oracle, pm)
    diag = _diag(om)
    dt = api.Target(ctx, target, tt)
    reg = api.CpdRegistration(ctx, pm, dt, api.CpdConfiguration(maxIterations=10, w=0.05))
    oalgo = oracle.CpdAlgorithm(oracle.CpdConfig(max_iterations=10, w=0.05), literal=False)
    ost = oalgo.initialize(oracle.initial_state(om, target, tt, global_transformation=oracle.RIGID_TRANSFORMS))
    for _ in range(3):
        gst = reg.propose(_to_api_state(ost, api))
        ost = oracle.propose(oalgo, ost)
        _compare(gst, ost, diag)
    reg.close()
    p = api.ModelFittingParameters(1.2, np.array([1.0, -2.0, 0.5]), (0.1, -0.2, 0.05), rng.normal(size=om.rank))
    fit = pm.instance(p)
    ofit = oracle.model_instance_shape_pose_scale(om, oracle.Params(p.scale, p.translation, p.euler, p.shape))
    assert np.max(np.abs(fit - ofit)) <= 1e-9 * diag
    back = _as_oracle(oracle, api.Model(ctx, om.ref, om.mean, om.basis, om.variance, om.tri))
    assert np.array_equal(back.ref, om.ref) and np.array_equal(back.mean, om.mean) and np.array_equal(back.basis, om.basis)
    assert np.max(np.abs(back.variance - om.variance)) <= 1e-15 * om.variance.max()


def _registration(ctx, oracle, algo, landmarks=False):
    from gingr_b200 import api
    m, target, tt = _problem(oracle, 150, 180, 20, seed=13)
    dm = _upload(ctx, m)
    dt = api.Target(ctx, target, tt)
    lm = None
    if algo == "icp":
        reg = api.IcpRegistration(ctx, dm, dt, api.IcpConfiguration(maxIterations=40, initialSigma=2.0, endSigma=0.5))
        oalgo = oracle.IcpAlgorithm(oracle.IcpConfig(max_iterations=40, initial_sigma=2.0, end_sigma=0.5))
    else:
        reg = api.CpdRegistration(ctx, dm, dt, api.CpdConfiguration(maxIterations=40, w=0.1))
        oalgo = oracle.CpdAlgorithm(oracle.CpdConfig(max_iterations=40, w=0.1), literal=False)
    if landmarks:
        rng = np.random.default_rng(4)
        lm_pid = np.array([3, 40, 77, 111], dtype=np.int32)
        lm_pts = m.ref[lm_pid] + rng.normal(scale=2.0, size=(4, 3)) + 5.0
        A = rng.normal(size=(4, 3, 3))
        lm_cov = A @ np.transpose(A, (0, 2, 1)) + np.eye(3)
        reg.setLandmarks(lm_pid, lm_pts, lm_cov)
        lm = oracle.Landmarks(lm_pid, lm_pts, lm_cov)
    ost = oalgo.initialize(oracle.initial_state(m, target, tt, global_transformation=oracle.RIGID_TRANSFORMS, landmarks=lm))
    for _ in range(2):
        ost = oracle.propose(oalgo, ost)
    return reg, oalgo, ost, m, (dm, dt)


@pytest.mark.parametrize("algo,landmarks", [("cpd", False), ("icp", False), ("cpd", True)])
def test_registration_level_matches_oracle(ctx, oracle, algo, landmarks):
    from gingr_b200 import api
    reg, oalgo, ost, m, keep = _registration(ctx, oracle, algo, landmarks)
    st = _to_api_state(ost, api)
    before = reg.update(st)
    n0 = ctx.launch_count
    again = reg.update(st)
    launches = ctx.launch_count - n0
    got = _as_oracle(oracle, reg.computePosterior(st))
    want = oracle.posterior_model(oalgo, ost)
    s_max = float(want.variance.max())
    diag = _diag(m)
    assert np.max(np.abs(got.variance - want.variance)) <= 1e-6 * s_max
    assert np.max(np.abs(got.ref - want.ref)) <= 1e-9 * diag
    assert np.max(np.abs(got.mean - want.mean)) <= 1e-6 * diag
    Kg = (got.basis * got.variance) @ got.basis.T
    Kw = (want.basis * want.variance) @ want.basis.T
    assert np.max(np.abs(Kg - Kw)) <= 1e-6 * float(m.variance.max())
    # the registration is left as it was: the next update is the same, bit for bit and launch for launch
    n1 = ctx.launch_count
    after = reg.update(st)
    assert ctx.launch_count - n1 == launches
    for a, b in ((before, again), (before, after)):
        assert np.array_equal(a.fit, b.fit) and np.array_equal(a.modelParameters.shape, b.modelParameters.shape)
        assert a.sigma2 == b.sigma2 and tuple(a.modelParameters.euler) == tuple(b.modelParameters.euler)
    reg.close()


def test_at_scale_against_the_device_posterior_entries(ctx):
    """C4 model size (M = 20 000, r = 2000, 3/4 of the vertices observed): per-vertex covariance blocks of the new model
    against gingr_posterior_covariance, its mean against gingr_posterior_mean, orthonormality of its basis."""
    from gingr_b200 import api, synthetic
    M, r = 20000, 2000
    ref = synthetic.fibonacci_sphere(M)
    _, basis, var = synthetic.make_gpmm(ref, r, 1)
    rng = np.random.default_rng(0)
    mean = rng.normal(scale=0.5, size=3 * M)
    dm = api.Model(ctx, ref, mean, basis, var)
    R, t = synthetic.euler_matrix(0.1, -0.2, 0.05), np.array([1.0, 2.0, -3.0])
    pids = rng.permutation(M)[: (3 * M) // 4].astype(np.int32)
    pts = (ref[pids] + rng.normal(scale=2.0, size=(len(pids), 3))) @ R.T + t
    noise = rng.uniform(0.5, 4.0, size=len(pids))
    pm = api.posterior_model(ctx, dm, R, t, pids, pts, noise)
    gref, gmean, gbasis, gvar = pm.download()
    cov = api.posterior_covariance(ctx, dm, R, t, pids, pts, noise)
    _, mesh = api.posterior_mean(ctx, dm, R, t, pids, pts, noise)
    B = gbasis.reshape(M, 3, r)
    blocks = np.einsum("iak,k,ibk->iab", B, gvar, B)
    assert np.max(np.abs(blocks - cov)) <= 1e-9 * var.max()
    diag = float(np.linalg.norm(ref.max(0) - ref.min(0)))
    assert np.max(np.abs(gref + gmean.reshape(M, 3) - mesh)) <= 1e-9 * diag
    G = gbasis.T @ gbasis
    assert np.max(np.abs(G - np.eye(r))) <= 1e-12
    assert np.all(np.diff(gvar) <= 0.0) and gvar[-1] > 0.0
