"""The BCPD configuration of GingrAlgorithm on the device (GINGR_ALGO_BCPD) against the oracle's literal restatement
(oracle/bcpd.py): coefficients, fit and sigma2 to 1e-6 relative as for CPD, the per-vertex mixing weights alpha and
posterior variances Sigma to 1e-9 relative; the device digamma against scipy; the iteration's E-step against
gingr_bcpd_estep; graph replay against kernel-by-kernel runs and batched against solo registrations, bit for bit; the
refused calls; the launch count of the CPD iteration.

Mistakes the tests are aimed at: s^2 instead of s in the row factor (the oracle comparison and the E-step identity, from
the second iteration on, where s != 1 under similarity transforms and Sigma != prior), an off-by-one in the digamma
recurrence (psi(x) + 1/x: the digamma bound and alpha), the variance rows of the wrong vertex (Sigma against the
oracle), sigma2bar left out of the sigma2 hook (sigma2), alpha / Sigma advanced on a failed iteration (the
flexibility-error case)."""
import os
import subprocess
import sys
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


# The synthetic spheres and the femur are shrunk by this factor: at their own size the outlier term c = w / N of BCPD's E-step
# (BCPD.scala:170-181, kept literally) outweighs every Gaussian at the initial sigma2, Nhat is tiny, and the sigma2 hook's
# sigma2 sigma2bar / (3 Nhat) makes sigma2 grow without bound when w > 0.
SHRINK = 20.0


def _problem(oracle, M, N, r, seed):
    from gingr_b200 import synthetic
    ref, tri = synthetic.sphere_mesh(M)
    mean, basis, var = synthetic.make_gpmm(ref, r, seed + 1)
    tv, tt = synthetic.sphere_mesh(N)
    target = synthetic.make_target(tv, seed)
    k = SHRINK
    return oracle.Gpmm(ref / k, mean / k, basis, var / (k * k), tri), target / k, tt


def _to_api_state(ost, api):
    p = ost.params
    return api.GeneralRegistrationState(
        api.ModelFittingParameters(p.scale, np.asarray(p.translation, float), tuple(p.euler), p.shape.copy()),
        ost.fit.copy(), ost.sigma2, ost.global_transformation, ost.step_length, "", ost.iteration, ost.status)


def _rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / max(float(np.max(np.abs(b))), 1e-300))


def _compare(gst, ost, diag, tol=1e-6):
    a_scale = max(np.max(np.abs(ost.params.shape)), 1e-12)
    assert gst.status == ost.status and gst.iteration == ost.iteration
    assert np.max(np.abs(gst.modelParameters.shape - ost.params.shape)) < tol * a_scale
    assert np.max(np.abs(gst.fit - ost.fit)) < tol * diag
    assert abs(gst.sigma2 - ost.sigma2) <= tol * abs(ost.sigma2)
    assert abs(gst.modelParameters.scale - ost.params.scale) < tol


def _run_pair(ctx, oracle, m, target, tt, gtc, w, kappa, iters, landmarks=None, initial_sigma=None):
    """Device and oracle side by side; the oracle's pose / shape / sigma2 are handed to the device every iteration (no
    drift of those), alpha and Sigma stay on each side and are compared after every update."""
    from gingr_b200 import api
    from oracle import bcpd
    diag = np.linalg.norm(m.ref.max(0) - m.ref.min(0))
    dm = api.Model(ctx, m.ref, m.mean, m.basis, m.variance, m.tri)
    dt = api.Target(ctx, target, tt)
    reg = api.BcpdRegistration(ctx, dm, dt, api.BcpdConfiguration(w=w, kappa=kappa, initialSigma=initial_sigma))
    algo = bcpd.BcpdAlgorithm(bcpd.BcpdConfig(w=w, kappa=kappa, initial_sigma=initial_sigma))
    lms = None
    if landmarks is not None:
        pid, pts, cov = landmarks
        reg.setLandmarks(pid, pts, cov)
        lms = oracle.Landmarks(np.asarray(pid, np.int32), pts, cov)
    ost = algo.initialize(oracle.initial_state(m, target, tt, global_transformation=gtc, landmarks=lms))
    gst = reg.initializeState(globalTransformation=gtc)
    assert abs(gst.sigma2 - ost.sigma2) <= 1e-12 * ost.sigma2
    a, s = reg.bcpdState()
    assert np.all(a == 1.0 / m.M) and _rel(s, algo.Sigma) < 1e-12
    for _ in range(iters):
        gst = reg.propose(_to_api_state(ost, api))
        ost = bcpd.propose(algo, ost)
        _compare(gst, ost, diag)
        a, s = reg.bcpdState()
        assert _rel(a, algo.alpha) < 1e-9, _rel(a, algo.alpha)
        assert _rel(s, algo.Sigma) < 1e-9, _rel(s, algo.Sigma)
    reg.close()
    dt.close()
    dm.close()
    return gst, ost


@pytest.mark.parametrize("gt,w,kappa,lm", [("rigid", 0.0, 1.0, False), ("similarity", 0.1, 10.0, False),
                                           ("none", 0.1, 1.0, True), ("similarity", 0.0, 10.0, True),
                                           ("rigid", 0.1, 10.0, True), ("none", 0.0, 1.0, False)])
def test_bcpd_iterations_match_oracle_on_spheres(ctx, oracle, gt, w, kappa, lm):
    gtc = {"none": oracle.NO_TRANSFORMS, "rigid": oracle.RIGID_TRANSFORMS, "similarity": oracle.SIMILARITY_TRANSFORMS}[gt]
    m, target, tt = _problem(oracle, 120, 150, 40, seed=3)
    landmarks = None
    if lm:
        rng = np.random.default_rng(4)
        pid = np.array([3, 40, 77, 111], dtype=np.int32)
        pts = m.ref[pid] + rng.normal(scale=2.0, size=(4, 3)) + 5.0
        A = rng.normal(size=(4, 3, 3))
        cov = A @ np.transpose(A, (0, 2, 1)) + np.eye(3)
        landmarks = (pid, pts, cov)
    _run_pair(ctx, oracle, m, target, tt, gtc, w, kappa, 6, landmarks)


def test_bcpd_iterations_match_oracle_on_the_femur(ctx, oracle):
    sys.path.insert(0, os.path.join(HERE, "golden"))
    import make_golden
    gold = np.load(os.path.join(HERE, "golden", "femur_golden.npz"))
    sub_r, sub_t = gold["ref_v"][::16], gold["tgt_v"][::16]
    mean, basis, var = make_golden.femur_gpmm(sub_r)
    k = SHRINK
    m = oracle.Gpmm(sub_r / k, mean / k, basis, var / (k * k), None)
    sub_t = sub_t / k
    lm_pid, _ = oracle.nearest_vertex(gold["lm_ref"], sub_r)
    landmarks = (lm_pid.astype(np.int32), gold["lm_tgt"] / k, np.tile(np.eye(3) / (k * k), (6, 1, 1)))
    _run_pair(ctx, oracle, m, sub_t, None, oracle.SIMILARITY_TRANSFORMS, 0.1, 1.0, 8, landmarks)


def test_flexibility_error_leaves_alpha_and_sigma(ctx, oracle):
    """An iteration whose posterior fails (a non-finite sigma2 makes every nu NaN) keeps the BCPD state."""
    from gingr_b200 import api
    m, target, tt = _problem(oracle, 100, 100, 30, seed=6)
    dm = api.Model(ctx, m.ref, m.mean, m.basis, m.variance, m.tri)
    dt = api.Target(ctx, target, tt)
    reg = api.BcpdRegistration(ctx, dm, dt, api.BcpdConfiguration())
    st = reg.propose(reg.initializeState())
    a0, s0 = reg.bcpdState()
    bad = reg.update(api.GeneralRegistrationState(st.modelParameters, st.fit, float("nan"), st.globalTransformation,
                                                  st.stepLength, "", st.iteration, st.status))
    assert bad.status == api.STATUS_MODEL_FLEXIBILITY_ERROR
    a1, s1 = reg.bcpdState()
    assert np.array_equal(a0, a1) and np.array_equal(s0, s1)
    reg.close()


def test_state_is_the_prior_from_creation(ctx, oracle):
    """Without gingr_initialize_state the registration already holds alpha = 1 / M and the prior variances, so an update of
    a state the caller built runs like any other."""
    from gingr_b200 import api
    from oracle import bcpd
    m, target, tt = _problem(oracle, 100, 120, 30, seed=12)
    dm = api.Model(ctx, m.ref, m.mean, m.basis, m.variance, m.tri)
    dt = api.Target(ctx, target, tt)
    reg = api.BcpdRegistration(ctx, dm, dt, api.BcpdConfiguration())
    a, s = reg.bcpdState()
    assert np.all(a == 1.0 / m.M) and _rel(s, bcpd.prior_variance(m)) < 1e-12
    pars = api.ModelFittingParameters(1.0, np.zeros(3), (0.0, 0.0, 0.0), np.zeros(m.rank))
    st = reg.update(api.GeneralRegistrationState(pars, np.zeros((m.M, 3)), 16.0, api.RIGID_TRANSFORMS))
    assert st.status == api.STATUS_NONE and np.all(np.isfinite(st.fit)) and st.sigma2 != 16.0
    a1, s1 = reg.bcpdState()
    assert not np.array_equal(a1, a) and np.all(np.isfinite(a1)) and np.all(s1 > 0.0)
    reg.close()


def test_device_digamma_within_a_few_ulp_of_scipy(ctx):
    """psi on [1e-3, 1e8].  Error bound of the device algorithm: the recurrence adds n <= 6 terms 1/(x + k), each with one
    rounding in x + k and one in the division, and the series (|terms| <= ln x + 1) is evaluated with about 4 roundings
    plus < 1 ulp of truncation; so |psi_dev - psi| <= 8 eps (sum_k 1/(x + k) + |psi(x + n)|), a few ulp of the largest
    magnitude in the sum (near the root of psi at 1.4616 the cancellation makes a relative bound meaningless)."""
    from scipy.special import digamma
    lib = ctx._lib
    lib.gingr_debug_digamma.restype = ctypes.c_int32
    lib.gingr_debug_digamma.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_double),
                                        ctypes.POINTER(ctypes.c_double)]
    rng = np.random.default_rng(0)
    x = np.concatenate([np.logspace(-3, 8, 20000), rng.uniform(1e-3, 20.0, 20000), [1.4616321449683622, 6.0, 5.999999999, 1.0]])
    out = np.empty_like(x)
    ctx.check(lib.gingr_debug_digamma(ctx.handle, len(x), x.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                      out.ctypes.data_as(ctypes.POINTER(ctypes.c_double))))
    n = np.maximum(np.ceil(6.0 - x), 0.0)
    terms = np.array([np.sum(1.0 / (xi + np.arange(int(ni)))) for xi, ni in zip(x, n)])
    bound = 8.0 * np.finfo(float).eps * (terms + np.abs(digamma(x + n)))
    err = np.abs(out - digamma(x))
    assert np.all(err <= bound), (x[np.argmax(err / bound)], float(np.max(err / bound)))


def test_iteration_estep_equals_gingr_bcpd_estep(ctx, oracle):
    """The observation weights of the first iteration, as obs_kernel forms them from nu, are the ones gingr_bcpd_estep's nu
    gives for the same fit, Sigma, alpha, sigma2, s and w: bit for bit."""
    from gingr_b200 import api
    m, target, tt = _problem(oracle, 300, 400, 40, seed=8)
    dm = api.Model(ctx, m.ref, m.mean, m.basis, m.variance, m.tri)
    dt = api.Target(ctx, target, tt)
    cfg = api.BcpdConfiguration(w=0.1, lambda_=2.0)
    reg = api.BcpdRegistration(ctx, dm, dt, cfg)
    st = reg.initializeState(globalTransformation=api.SIMILARITY_TRANSFORMS)
    st = reg.propose(st)   # s != 1 and Sigma != prior from here on
    st = reg.propose(st)
    alpha, sigma = reg.bcpdState()
    nu, nup, _, xhat = api.bcpd_estep(ctx, dt, st.fit, sigma, alpha, st.sigma2, st.modelParameters.scale, cfg.w)
    lib = ctx._lib
    f = lib.gingr_debug_posterior_system
    f.restype = ctypes.c_int32
    dp = ctypes.POINTER(ctypes.c_double)
    f.argtypes = [ctypes.c_void_p, ctypes.POINTER(api.GingrState), dp, ctypes.c_int32, dp, dp, dp]
    pod, a = st.to_pod()
    r = m.rank
    sys_ = np.empty((r + 1) * r)
    wrow = np.empty(3 * m.M)
    u = np.empty(3 * m.M)
    ctx.check(f(reg.handle, ctypes.byref(pod), a.ctypes.data_as(dp), 0, sys_.ctypes.data_as(dp), wrow.ctypes.data_as(dp),
                u.ctypes.data_as(dp)))
    var = st.sigma2 * cfg.lambda_ * (1.0 / nu)
    wt = 1.0 / var
    assert np.array_equal(wrow.reshape(-1, 3)[:, 0], wt)
    # the observation points: u = wt R^T (xhat - (R (ref + mean) + t)) with gingr_bcpd_estep's xhat = PX / nu (the rotation
    # is formed on the device from the same Euler angles, hence a tolerance instead of bit equality)
    p = st.modelParameters
    R = oracle.euler_to_matrix(*p.euler)
    base = m.ref + m.mean.reshape(-1, 3)
    u_exp = wt[:, None] * ((xhat - (base @ R.T + np.asarray(p.translation))) @ R)
    assert np.max(np.abs(u.reshape(-1, 3) - u_exp)) <= 1e-11 * np.max(np.abs(u_exp))
    # nu' through sXX: the sigma2 this iteration commits, from gingr_bcpd_estep's nu, nu', xhat on the same inputs
    fit = st.fit
    nhat = nu.sum()
    sxx = nup @ (target * target).sum(1)
    sxy = ((nu[:, None] * xhat) * fit).sum()
    syy = nu @ (fit * fit).sum(1)
    s2_exp = (sxx - 2.0 * sxy + syy + st.sigma2 * (nu @ sigma) / nhat) / (3.0 * nhat)
    nxt = reg.update(st)
    assert nxt.status == api.STATUS_NONE
    assert abs(nxt.sigma2 - s2_exp) <= 1e-9 * abs(s2_exp), (nxt.sigma2, s2_exp)
    reg.close()


_REPLAY = r"""
import sys, numpy as np
sys.path.insert(0, {root!r})
from gingr_b200 import api, synthetic
ref, tri = synthetic.sphere_mesh(200)
mean, basis, var = synthetic.make_gpmm(ref, 40, 2)
tv, tt = synthetic.sphere_mesh(260)
k = {shrink!r}
ctx = api.Context(0)
dm = api.Model(ctx, ref / k, mean / k, basis, var / (k * k), tri)
dt = api.Target(ctx, synthetic.make_target(tv, 1) / k, tt)
reg = api.BcpdRegistration(ctx, dm, dt, api.BcpdConfiguration(w=0.1, kappa=10.0))
reg.initializeState(globalTransformation=api.SIMILARITY_TRANSFORMS)
reg.updateChain(4)
st = reg.downloadState()
a, s = reg.bcpdState()
np.savez({out!r}, fit=st.fit, alpha=st.modelParameters.shape, sigma2=st.sigma2, ba=a, bs=s)
"""


def test_graph_replay_equals_kernel_by_kernel(tmp_path):
    outs = []
    for graph in ("2", "0"):
        out = str(tmp_path / f"g{graph}.npz")
        env = dict(os.environ, GINGR_CUDA_GRAPH=graph)
        subprocess.run([sys.executable, "-c", _REPLAY.format(root=ROOT, out=out, shrink=SHRINK)], check=True, env=env, timeout=300)
        outs.append(np.load(out))
    for k in ("fit", "alpha", "sigma2", "ba", "bs"):
        assert np.array_equal(outs[0][k], outs[1][k]), k


def test_batched_registrations_equal_solo_ones(ctx, oracle):
    from gingr_b200 import api
    m, target, tt = _problem(oracle, 150, 180, 30, seed=9)
    dm = api.Model(ctx, m.ref, m.mean, m.basis, m.variance, m.tri)
    dt = api.Target(ctx, target, tt)
    cfgs = [api.BcpdConfiguration(w=0.1, kappa=1.0), api.BcpdConfiguration(w=0.0, kappa=10.0)]
    batch = [api.BcpdRegistration(ctx, dm, dt, c) for c in cfgs]
    solo = [api.BcpdRegistration(ctx, dm, dt, c) for c in cfgs]
    for reg in batch + solo:
        reg.initializeState(globalTransformation=api.RIGID_TRANSFORMS)
    api.update_batch(batch, 3)
    for reg in solo:
        reg.updateChain(3)
    for b, s in zip(batch, solo):
        sb, ss = b.downloadState(), s.downloadState()
        assert np.array_equal(sb.fit, ss.fit) and sb.sigma2 == ss.sigma2 and sb.iteration == ss.iteration == 3
        ab, bb = b.bcpdState()
        as_, bs = s.bcpdState()
        assert np.array_equal(ab, as_) and np.array_equal(bb, bs)
    for reg in batch + solo:
        reg.close()


def test_refused_calls(ctx, oracle):
    from gingr_b200 import api, _native as nat
    m, target, tt = _problem(oracle, 80, 90, 20, seed=10)
    dm = api.Model(ctx, m.ref, m.mean, m.basis, m.variance, m.tri)
    dt = api.Target(ctx, target, tt)
    reg = api.BcpdRegistration(ctx, dm, dt)
    st = reg.initializeState()
    calls = [lambda: reg.update(st, probabilistic=True, seed=1), lambda: reg.updateChainSampled(2, 1),
             lambda: api.update_batch([reg, api.BcpdRegistration(ctx, dm, dt)], 1, probabilistic=True, seed=1),
             lambda: reg.configureProbabilistic(api.ProbabilisticSettings())]
    for call in calls:
        with pytest.raises(nat.GingrError) as e:
            call()
        assert e.value.code == nat.GINGR_ERR_UNSUPPORTED
    with pytest.raises(nat.GingrError) as e:   # kappa must be positive
        ctx.check(ctx._lib.gingr_registration_set_bcpd(reg.handle, 0.0))
    assert e.value.code == nat.GINGR_ERR_ARG
    reg.close()


# Kernel launches of one CPD iteration of the problem below, as counted before the BCPD flavour existed.
CPD_ITERATION_LAUNCHES = 29


def test_cpd_iteration_keeps_its_launch_count(ctx, oracle):
    """The CPD iteration launches what it launched before the BCPD flavour existed; the BCPD iteration is the CPD one with
    its own prepare / observation / sigma2 kernels in the same places and two launches more (the variance rows, the next
    BCPD state)."""
    from gingr_b200 import api
    m, target, tt = _problem(oracle, 200, 240, 40, seed=11)
    dm = api.Model(ctx, m.ref, m.mean, m.basis, m.variance, m.tri)
    dt = api.Target(ctx, target, tt)
    counts = []
    for reg in (api.CpdRegistration(ctx, dm, dt, api.CpdConfiguration(w=0.1)),
                api.BcpdRegistration(ctx, dm, dt, api.BcpdConfiguration(w=0.1))):
        reg.initializeState()
        reg.updateChain(1)      # captures the graph
        ctx.synchronize()
        l0 = ctx.launch_count
        reg.updateChain(3)
        ctx.synchronize()
        counts.append((ctx.launch_count - l0) // 3)
        reg.close()
    assert counts[0] == CPD_ITERATION_LAUNCHES, counts
    assert counts[1] == counts[0] + 2, counts
