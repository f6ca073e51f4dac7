"""Ranks above 64 x the SM count (9472 on a B200), up to 18 000, the largest rank the device builders produce.

Above 9472 the two back substitutions (chol.cu, chol_df.cu) run more 64-row blocks than the GPU has SMs: their CTAs take
their blocks by atomic ticket, so the spin waits hold whatever the grid size.  Above 12 800 the two-vector instance pass
of the iteration runs as two one-vector passes.  The cases here:
  * gingr_spd_solve just above the old ceiling and at a ragged last block, against LAPACK; at n = 18 000 through the
    residual, sampled rows of L L^T - A, and two runs in a row that must give the same bits (the ticket and the flags
    reset themselves);
  * CPD at rank 9600 against oracle.fast, and the iteration's fit against s (R (ref + mean + Phi D alpha) + t) formed on
    the host (the two-vector instance pass);
  * CPD, ICP and BCPD at rank 9600: captured graphs against kernel-by-kernel runs, and batched registrations and MH chains
    against solo ones, bit for bit; a chain of MH steps in one call against single steps;
  * an inverse-Laplacian model of 6000 vertices at rank >= 17 000: a CPD run, its fit (the one-vector instance pass), the
    posterior mean against its system Mx c = rhs formed on the host (a matvec), and posterior_covariance against
    Q Mx^-1 Q^T at sampled vertices;
  * the registration's posterior model at rank 9600 against the system gingr_debug_posterior_system returns.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M_9600, R_9600 = 3300, 9600          # 3M = 9900 >= r; 150 blocks of 64 rows against 148 SMs


def _spd(n, seed, k=64, cond=1e3):
    """Dense SPD with a spread spectrum: a rank-k Gram plus a diagonal, cheap to form at n = 18 000."""
    rng = np.random.default_rng(seed)
    Q = rng.normal(size=(n, k))
    A = Q @ Q.T / k
    A[np.diag_indices(n)] += rng.uniform(1.0, cond, size=n) / cond * (np.trace(A) / n)
    return A


@pytest.mark.parametrize("n", [9473, 9536, 9600, 12801])
def test_spd_solve_matches_lapack_above_the_sm_count(ctx, n):
    from gingr_b200 import api
    A = _spd(n, n)
    B = np.random.default_rng(n + 1).normal(size=(1, n))
    out = api.spd_solve(ctx, A, B)
    L = np.linalg.cholesky(A)
    assert np.max(np.abs(out["L"] - L)) < 1e-12 * np.abs(L).max()
    Y = np.linalg.solve(L, B.T).T
    assert np.max(np.abs(out["Y"] - Y)) < 1e-11 * max(1.0, np.abs(Y).max())
    x = np.linalg.solve(A, B[0])
    assert np.max(np.abs(out["x"] - x)) < 1e-10 * max(1.0, np.abs(x).max())


def test_spd_solve_rank_18000_residual_and_repeatability(ctx):
    from gingr_b200 import api
    n = 18000
    A = _spd(n, 5)
    b = np.random.default_rng(6).normal(size=(1, n))
    o1 = api.spd_solve(ctx, A, b)
    o2 = api.spd_solve(ctx, A, b)
    assert np.array_equal(o1["L"], o2["L"]) and np.array_equal(o1["x"], o2["x"])
    x, L = o1["x"], o1["L"]
    assert np.all(np.isfinite(x))
    assert np.linalg.norm(A @ x - b[0]) <= 1e-10 * np.linalg.norm(b[0])
    rows = np.random.default_rng(7).choice(n, size=48, replace=False)
    rows[:2] = (0, n - 1)
    assert np.max(np.abs(L[rows] @ L.T - A[rows])) < 1e-12 * np.abs(A).max()


def _problem(oracle, M, N, r, seed, orthonormal=True):
    from gingr_b200 import synthetic
    ref, tri = synthetic.sphere_mesh(M)
    mean, basis, var = synthetic.make_gpmm(ref, r, seed + 1, orthonormal=orthonormal)
    tv, tt = synthetic.sphere_mesh(N)
    target = synthetic.make_target(tv, seed)
    return oracle.Gpmm(ref, mean, basis, var, tri), target, tt


def _to_api_state(ost, api):
    p = ost.params
    return api.GeneralRegistrationState(
        api.ModelFittingParameters(p.scale, np.asarray(p.translation, float), tuple(p.euler), p.shape.copy()),
        ost.fit.copy(), ost.sigma2, ost.global_transformation, ost.step_length, "", ost.iteration, ost.status)


def _host_fit(oracle, ref, mean, basis, var, st):
    """s (R (ref + mean + Phi D alpha) + t) of a state, in float64 on the host."""
    p = st.modelParameters
    R = oracle.euler_to_matrix(*p.euler)
    x = ref + mean.reshape(-1, 3) + (basis @ (np.sqrt(var) * p.shape)).reshape(-1, 3)
    return p.scale * (x @ R.T + np.asarray(p.translation))


def test_cpd_rank_9600_matches_fast_oracle_and_its_fit(ctx, oracle):
    from gingr_b200 import api
    from oracle import fast
    m, target, tt = _problem(oracle, M_9600, 3000, R_9600, seed=0)
    diag = float(np.linalg.norm(m.ref.max(0) - m.ref.min(0)))
    dm = api.Model(ctx, m.ref, m.mean, m.basis, m.variance, m.tri)
    dt = api.Target(ctx, target, tt)
    reg = api.CpdRegistration(ctx, dm, dt, api.CpdConfiguration(w=0.1))
    algo = oracle.CpdAlgorithm(oracle.CpdConfig(w=0.1))
    fm = fast.FastCpdModel(m)
    ost = algo.initialize(oracle.initial_state(m, target, tt, global_transformation=oracle.RIGID_TRANSFORMS))
    for _ in range(2):
        gst = reg.propose(_to_api_state(ost, api))
        ost = fast.propose(fm, algo, ost)
        a_scale = max(np.max(np.abs(ost.params.shape)), 1e-12)
        assert gst.status == ost.status and gst.iteration == ost.iteration
        assert np.max(np.abs(gst.modelParameters.shape - ost.params.shape)) < 1e-6 * a_scale
        assert np.max(np.abs(gst.fit - ost.fit)) < 1e-6 * diag
        assert abs(gst.sigma2 - ost.sigma2) <= 1e-6 * abs(ost.sigma2)
        assert np.max(np.abs(gst.fit - _host_fit(oracle, m.ref, m.mean, m.basis, m.variance, gst))) < 1e-9 * diag
    reg.close()


_REPLAY = r"""
import sys, numpy as np
sys.path.insert(0, {root!r})
from gingr_b200 import api, synthetic
ref, tri = synthetic.sphere_mesh({M})
mean, basis, var = synthetic.make_gpmm(ref, {r}, 2, orthonormal=False)
tv, tt = synthetic.sphere_mesh(3000)
ctx = api.Context(0)
dm = api.Model(ctx, ref, mean, basis, var, tri)
dt = api.Target(ctx, synthetic.make_target(tv, 1), tt)
out = {{}}
regs = {{"cpd": api.CpdRegistration(ctx, dm, dt, api.CpdConfiguration(w=0.1)),
        "icp": api.IcpRegistration(ctx, dm, dt, api.IcpConfiguration(initialSigma=2.0, endSigma=0.5)),
        "bcpd": api.BcpdRegistration(ctx, dm, dt, api.BcpdConfiguration(w=0.1))}}
for name, reg in regs.items():
    reg.initializeState(globalTransformation=api.RIGID_TRANSFORMS)
    reg.updateChain(2)
    st = reg.downloadState()
    out[name + "_fit"], out[name + "_alpha"], out[name + "_sigma2"] = st.fit, st.modelParameters.shape, st.sigma2
    reg.close()
np.savez({out!r}, **out)
"""


def test_graph_replay_equals_kernel_by_kernel_at_rank_9600(tmp_path):
    outs = []
    for graph in ("2", "0"):
        out = str(tmp_path / f"g{graph}.npz")
        env = dict(os.environ, GINGR_CUDA_GRAPH=graph)
        subprocess.run([sys.executable, "-c", _REPLAY.format(root=ROOT, out=out, M=M_9600, r=R_9600)], check=True, env=env,
                       timeout=600)
        outs.append(np.load(out))
    for k in outs[0].files:
        assert np.all(np.isfinite(outs[0][k])), k
        assert np.array_equal(outs[0][k], outs[1][k]), k


@pytest.fixture(scope="module")
def model_9600(ctx, oracle):
    from gingr_b200 import api
    m, target, tt = _problem(oracle, M_9600, 3000, R_9600, seed=3, orthonormal=False)
    dm = api.Model(ctx, m.ref, m.mean, m.basis, m.variance, m.tri)
    dt = api.Target(ctx, target, tt)
    yield m, dm, dt
    dm.close()
    dt.close()


def test_batched_updates_equal_solo_ones_at_rank_9600(ctx, model_9600):
    from gingr_b200 import api
    _, dm, dt = model_9600
    cfgs = [api.CpdConfiguration(w=0.1), api.CpdConfiguration(w=0.0)]
    batch = [api.CpdRegistration(ctx, dm, dt, c) for c in cfgs]
    solo = [api.CpdRegistration(ctx, dm, dt, c) for c in cfgs]
    for reg in batch + solo:
        reg.initializeState(globalTransformation=api.RIGID_TRANSFORMS)
    api.update_batch(batch, 2)
    for reg in solo:
        reg.updateChain(2)
    for b, s in zip(batch, solo):
        sb, ss = b.downloadState(), s.downloadState()
        assert np.all(np.isfinite(sb.fit)) and sb.iteration == ss.iteration == 2
        assert np.array_equal(sb.fit, ss.fit) and np.array_equal(sb.modelParameters.shape, ss.modelParameters.shape)
        assert sb.sigma2 == ss.sigma2
    for reg in batch + solo:
        reg.close()


def test_mh_chain_equals_single_steps_and_batch_at_rank_9600(ctx, model_9600):
    from gingr_b200 import api
    _, dm, dt = model_9600
    gs = api.ProbabilisticSettings(uncertainty=1.5, randomMixture=0.5)

    def chain():
        reg = api.IcpRegistration(ctx, dm, dt, api.IcpConfiguration(maxIterations=40, initialSigma=2.0, endSigma=0.5))
        reg.configureProbabilistic(gs)
        reg.initializeState(globalTransformation=api.RIGID_TRANSFORMS)
        return reg
    a, b = chain(), chain()
    for _ in range(3):
        a.mcmcChain(1, 77)
    b.mcmcChain(3, 77)
    sa, sb = a.downloadState(), b.downloadState()
    assert np.all(np.isfinite(sa.fit))
    assert np.array_equal(sa.fit, sb.fit) and np.array_equal(sa.modelParameters.shape, sb.modelParameters.shape)
    assert np.array_equal(a.mcmcStats()[1], b.mcmcStats()[1])
    a.close()
    b.close()
    # batched chains: chain k of the batch == a solo chain with seed + k
    chains = [chain() for _ in range(2)]
    api.mcmc_batch(chains, 2, seed=100)
    ctx.synchronize()
    for k, c in enumerate(chains):
        solo = chain()
        solo.mcmcChain(2, 100 + k)
        s1, s2 = c.downloadState(), solo.downloadState()
        assert np.array_equal(s1.fit, s2.fit) and np.array_equal(c.mcmcStats()[1], solo.mcmcStats()[1])
        solo.close()
    for c in chains:
        c.close()


def _observations(M, n, seed, ref, mean, basis, var):
    rng = np.random.default_rng(seed)
    pids = np.sort(rng.choice(M, size=n, replace=False)).astype(np.int32)
    truth = ref + mean.reshape(-1, 3) + (basis @ (np.sqrt(var) * rng.normal(size=var.shape[0]))).reshape(-1, 3)
    pts = truth[pids] + rng.normal(scale=0.3, size=(n, 3))
    noise = rng.uniform(0.5, 2.0, size=n)
    return pids, pts, noise


def _host_system(pids, pts, noise, ref, mean, basis, var):
    """Mx = I + Q_o^T W Q_o and rhs = Q_o^T W (y - ref - mean) at the identity pose, Q_o the observed rows of Phi D."""
    rows = (3 * pids[:, None] + np.arange(3)[None, :]).reshape(-1)
    Qo = basis[rows] * np.sqrt(var)[None, :]
    w = np.repeat(1.0 / noise, 3)
    Mx = Qo.T @ (Qo * w[:, None])
    Mx[np.diag_indices_from(Mx)] += 1.0
    rhs = Qo.T @ (w * (pts - ref[pids] - mean.reshape(-1, 3)[pids]).reshape(-1))
    return Mx, rhs


def test_inverse_laplacian_rank_above_17000(ctx):
    """6000 vertices, gamma > 0, relativeTolerance 0: the builders' largest rank."""
    import scipy.linalg as sla
    from gingr_b200 import api, synthetic
    from oracle import oracle
    M = 6000
    ref, tri = synthetic.sphere_mesh(M)
    dm = api.Model.inverseLaplacian(ctx, ref, tri, 100.0, 1.0, 0.0)
    assert dm.rank >= 17000
    ref_d, mean, basis, var = dm.download()
    basis = np.ascontiguousarray(basis)
    diag = float(np.linalg.norm(ref.max(0) - ref.min(0)))
    # a short CPD run ends finite, and its fit is the instance of its coefficients (one-vector instance pass)
    tv, tt = synthetic.sphere_mesh(5000)
    dt = api.Target(ctx, synthetic.make_target(tv, 4), tt)
    reg = api.CpdRegistration(ctx, dm, dt, api.CpdConfiguration(maxIterations=4, w=0.1))
    fin = reg.run(reg.initializeState(globalTransformation=api.RIGID_TRANSFORMS))
    assert fin.iteration >= 1 and np.isfinite(fin.sigma2)
    assert np.all(np.isfinite(fin.fit)) and np.all(np.isfinite(fin.modelParameters.shape))
    assert np.max(np.abs(fin.fit - _host_fit(oracle, ref_d, mean, basis, var, fin))) < 1e-9 * diag
    reg.close()
    dt.close()
    # posterior mean: the device's coefficients solve the host's system
    pids, pts, noise = _observations(M, 600, 5, ref_d, mean, basis, var)
    eye, zero = np.eye(3), np.zeros(3)
    c, _ = api.posterior_mean(ctx, dm, eye, zero, pids, pts, noise)
    Mx, rhs = _host_system(pids, pts, noise, ref_d, mean, basis, var)
    assert np.linalg.norm(Mx @ c - rhs) <= 1e-9 * np.linalg.norm(rhs)
    # posterior covariance at sampled vertices: Q_v Mx^-1 Q_v^T
    cov = api.posterior_covariance(ctx, dm, eye, zero, pids, pts, noise)
    assert np.all(np.isfinite(cov))
    vs = np.random.default_rng(8).choice(M, size=24, replace=False)
    vs[:2] = (pids[0], M - 1)
    Qv = basis[(3 * vs[:, None] + np.arange(3)[None, :]).reshape(-1)] * np.sqrt(var)[None, :]
    del basis
    fac = sla.cho_factor(Mx, lower=True, overwrite_a=True, check_finite=False)
    full = Qv @ sla.cho_solve(fac, Qv.T, check_finite=False)
    blocks = np.stack([full[3 * k:3 * k + 3, 3 * k:3 * k + 3] for k in range(len(vs))])
    assert np.max(np.abs(cov[vs] - blocks)) < 1e-9 * np.abs(blocks).max()
    dm.close()


def test_registration_posterior_model_matches_its_system_at_rank_9600(ctx, model_9600):
    """gingr_registration_posterior_model at the identity pose: mean - model mean = Q Mx^-1 rhs and the covariance blocks
    Q_v Mx^-1 Q_v^T at sampled vertices, with Mx and rhs the system gingr_debug_posterior_system returns at that state."""
    import ctypes

    import scipy.linalg as sla
    from gingr_b200 import api, _native as nat
    m, dm, dt = model_9600
    r = dm.rank
    reg = api.CpdRegistration(ctx, dm, dt, api.CpdConfiguration(w=0.1))
    st = reg.initializeState(globalTransformation=api.NO_TRANSFORMS)
    hook = ctx._lib.gingr_debug_posterior_system
    hook.argtypes = [ctypes.c_void_p, ctypes.POINTER(nat.GingrState), nat.dp, ctypes.c_int32, nat.dp, nat.dp, nat.dp]
    hook.restype = ctypes.c_int32
    pod, alpha = st.to_pod()
    system = np.full((r + 1, r), np.nan)
    assert ctx.check(hook(reg.handle, ctypes.byref(pod), nat.as_dp(alpha), 0, nat.as_dp(system), None, None)) == 0
    pm = reg.computePosterior(st)
    _, pmean, pb, pv = pm.download()
    pm.close()
    reg.close()
    fac = sla.cho_factor(system[:r], lower=True, check_finite=False)
    Q = m.basis * np.sqrt(m.variance)[None, :]
    dmean = Q @ sla.cho_solve(fac, system[r], check_finite=False)
    assert np.max(np.abs((pmean - m.mean) - dmean)) < 1e-8 * np.abs(dmean).max()
    vs = np.random.default_rng(10).choice(m.M, size=32, replace=False)
    rows = (3 * vs[:, None] + np.arange(3)[None, :]).reshape(-1)
    Qv = Q[rows]
    want = Qv @ sla.cho_solve(fac, Qv.T, check_finite=False)
    got = (pb[rows] * pv[None, :]) @ pb[rows].T
    blocks = lambda F: np.stack([F[3 * k:3 * k + 3, 3 * k:3 * k + 3] for k in range(len(vs))])
    assert np.max(np.abs(blocks(got) - blocks(want))) < 1e-8 * np.abs(blocks(want)).max()
