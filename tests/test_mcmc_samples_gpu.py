"""Posterior variance maps from Metropolis-Hastings chains collected on the device (gingr_mcmc_collect /
gingr_mcmc_samples, mcmc.cuh) against the logged run that helper.py reduces on the host (LogHelper.samplesFromLog,
PosteriorHelper.computeDistanceMapFromMeshes*), and the properties of the collection: independent of how a chain's steps
are split over calls or graphs, read-only for the chain, batched, reset with the chain, stopped at an error state."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

from test_update_gpu import _problem

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GS = dict(uncertainty=1.5, randomMixture=0.5)


def _builder(ctx, oracle, algo="icp", M=100, N=110, r=10, seed=2, with_tri=True):
    from gingr_b200 import api
    m, target, tt = _problem(oracle, M, N, r, seed)
    dm = api.Model(ctx, m.ref, m.mean, m.basis, m.variance, m.tri if with_tri else None)
    dt = api.Target(ctx, target, tt)

    def make(collection=None, step_length=1.0, status=api.STATUS_NONE, init=True):
        if algo == "icp":
            reg = api.IcpRegistration(ctx, dm, dt, api.IcpConfiguration(maxIterations=40, initialSigma=2.0, endSigma=0.5))
        else:
            reg = api.CpdRegistration(ctx, dm, dt, api.CpdConfiguration(maxIterations=40, w=0.1))
        reg.configureProbabilistic(api.ProbabilisticSettings(**GS))
        if collection is not None:
            reg.collectSamples(collection)
        if init:
            pars = api.ModelFittingParameters(1.0, np.zeros(3), (0.0, 0.0, 0.0), np.zeros(dm.rank))
            reg.initializeState(general=api.GeneralRegistrationState(pars, np.zeros((dm.M, 3)), globalTransformation=api.RIGID_TRANSFORMS,
                                                                     stepLength=step_length, status=status))
        return reg
    diag = float(np.linalg.norm(m.ref.max(0) - m.ref.min(0)))
    return make, dm, dt, m, diag


def _same(a, b):
    assert a.count == b.count
    for x, y in ((a.mean, b.mean), (a.cov, b.cov), (a.normal, b.normal)):
        assert np.array_equal(x, y, equal_nan=True)


def _close(a, b, tol):
    assert a.count == b.count
    for x, y in ((a.mean, b.mean), (a.cov, b.cov), (a.normal, b.normal)):
        assert np.max(np.abs(x - y)) <= tol * np.max(np.abs(y))


@pytest.mark.parametrize("algo", ["icp", "cpd"])
@pytest.mark.parametrize("burn,every,total", [(5, 3, 50), (0, 1, 100)])
def test_collected_statistics_equal_the_logged_chain_reduced_on_the_host(ctx, oracle, algo, burn, every, total):
    from gingr_b200 import api, helper, io
    make, dm, dt, m, diag = _builder(ctx, oracle, algo)
    reg = make(init=False)
    st0 = reg.initializeState(globalTransformation=api.RIGID_TRANSFORMS)
    logger = io.JSONStateLogger()
    reg.runProbabilistic(st0, api.ProbabilisticSettings(**GS), seed=11, iterations=60, acceptRejectLogger=logger,
                         sampleCollection=api.SampleCollection(burnIn=burn, takeEveryN=every, total=total))
    st = api.sample_statistics([reg])
    recs = helper.samples_from_log(logger.log, takeEveryN=every, total=total, burnIn=burn)
    assert st.count == len(recs) == len(range(burn, min(61, total), every))
    shapes = helper.log_samples_to_shapes(dm, [r for r, _ in recs])
    x = np.stack(shapes)
    assert len({r for _, r in recs}) > 3                        # the chain moved: several distinct states
    assert np.max(np.abs(st.mean - x.mean(0))) <= 1e-12 * diag
    cov = np.stack([np.cov(x[:, k, :].T, ddof=1) for k in range(dm.M)])
    assert np.max(np.abs(st.cov - cov)) <= 1e-9 * np.max(np.abs(cov))
    for got, want in ((st.distanceMapTotal(), helper.distance_map_total(shapes)),
                      (st.distanceMapNormal(), helper.distance_map_normal(shapes, m.tri)),
                      (st.distanceMapNormal(m.ref, m.tri, sumNormals=False),
                       helper.distance_map_normal(shapes, m.tri, reference=m.ref, sumNormals=False))):
        assert np.max(np.abs(got - want)) <= 1e-9 * np.max(want)
    reg.close()


_SPLIT = r"""
import sys, numpy as np
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
from gingr_b200 import api
from oracle import oracle as o
from test_mcmc_samples_gpu import _builder
o.build()
ctx = api.Context(0)
make, dm, dt, m, diag = _builder(ctx, o)
out = {{}}
for name, parts in (("split", (7, 13)), ("whole", (20,))):
    reg = make(api.SampleCollection(burnIn=2, takeEveryN=3, total=100))
    for k in parts:
        reg.mcmcChain(k, 21)
    st = api.sample_statistics([reg])
    out.update({{name + "_n": st.count, name + "_mean": st.mean, name + "_cov": st.cov, name + "_normal": st.normal}})
np.savez({out!r}, **out)
"""


def test_statistics_do_not_depend_on_how_the_steps_are_split_or_replayed(tmp_path):
    res = []
    for graph in (None, "0"):
        out = str(tmp_path / f"g{graph}.npz")
        env = dict(os.environ)
        if graph is not None:
            env["GINGR_CUDA_GRAPH"] = graph
        script = _SPLIT.format(root=ROOT, tests=os.path.join(ROOT, "tests"), out=out)
        subprocess.run([sys.executable, "-c", script], check=True, env=env, timeout=600)
        res.append(np.load(out))
    assert int(res[0]["whole_n"]) == 7                         # states 2, 5, ..., 20
    for r in res:
        for k in ("n", "mean", "cov", "normal"):
            assert np.array_equal(r["split_" + k], res[0]["whole_" + k]), k


def test_collection_is_read_only_for_the_chain_and_costs_one_launch_per_step(ctx, oracle):
    from gingr_b200 import api
    make, dm, dt, m, diag = _builder(ctx, oracle)
    on, off = make(api.SampleCollection(takeEveryN=1)), make()
    launches = []
    for reg in (on, off):
        reg.mcmcChain(1, 33)
        ctx.synchronize()
        l0 = ctx.launch_count
        reg.mcmcChain(11, 33)
        ctx.synchronize()
        launches.append(ctx.launch_count - l0)
    assert launches[0] - launches[1] == 11, launches
    a, b = on.downloadState(), off.downloadState()
    assert np.array_equal(a.fit, b.fit) and np.array_equal(a.modelParameters.shape, b.modelParameters.shape)
    assert a.sigma2 == b.sigma2 and a.iteration == b.iteration and a.status == b.status
    (va, ca), (vb, cb) = on.mcmcStats(), off.mcmcStats()
    assert np.array_equal(va, vb) and np.array_equal(ca, cb) and ca[3] > 0
    ba, bb = on.mcmcBest(), off.mcmcBest()
    assert np.array_equal(ba.fit, bb.fit) and np.array_equal(ba.modelParameters.shape, bb.modelParameters.shape)
    assert api.sample_statistics([on]).count == 13
    on.close(); off.close()


def test_batched_chains_collect_in_the_batched_sequence_and_pool_like_merge(ctx, oracle):
    from gingr_b200 import api
    make, dm, dt, m, diag = _builder(ctx, oracle, seed=3)
    coll = api.SampleCollection(burnIn=1, takeEveryN=2, total=100)
    n, iters = 48, 6
    chains = [make(coll) for _ in range(n)]
    api.mcmc_batch(chains, 1, seed=500)
    ctx.synchronize()
    l0 = ctx.launch_count
    api.mcmc_batch(chains, iters - 1, seed=500)
    ctx.synchronize()
    per_step = (ctx.launch_count - l0) / (iters - 1)
    assert per_step < 100, f"{per_step} launches per MH step of {n} chains: the batched sequence did not run"
    per_chain = [api.sample_statistics([c]) for c in chains]
    assert all(s.count == 3 for s in per_chain)                # states 1, 3, 5
    for k in (0, 1, 7, n - 1):
        solo = make(coll)
        solo.mcmcChain(iters, 500 + k)
        _close(per_chain[k], api.sample_statistics([solo]), 1e-9)
        solo.close()
    pooled = api.sample_statistics(chains)
    assert pooled.count == 3 * n
    _close(pooled, functools.reduce(lambda a, b: a.merge(b), per_chain), 1e-12)
    assert np.all(pooled.distanceMapTotal() > 0.0)
    for c in chains:
        c.close()


def test_accumulators_restart_with_the_chain_and_with_a_new_rule(ctx, oracle):
    from gingr_b200 import api
    make, dm, dt, m, diag = _builder(ctx, oracle)
    coll = api.SampleCollection(takeEveryN=1)
    a = make(coll)
    st0 = a.initializeState(globalTransformation=api.RIGID_TRANSFORMS)
    a.mcmcChain(6, 5)
    a.initializeState(general=st0)                               # a new chain starts: statistics from zero
    a.mcmcChain(6, 9)
    b = make(coll)
    b.mcmcChain(6, 9)
    _same(api.sample_statistics([a]), api.sample_statistics([b]))
    # a new rule in the middle of a chain: the states after it only (the step count goes on)
    c = make(coll)
    c.mcmcChain(4, 13)
    c.collectSamples(api.SampleCollection(burnIn=0, takeEveryN=1))
    c.mcmcChain(6, 13)
    d = make(api.SampleCollection(burnIn=5, takeEveryN=1))
    d.mcmcChain(10, 13)
    sc = api.sample_statistics([c])
    assert sc.count == 6
    _same(sc, api.sample_statistics([d]))
    # gingr_mcmc_configure discards the rule with the rest of the chain
    c.configureProbabilistic(api.ProbabilisticSettings(**GS))
    with pytest.raises(api.GingrError) as e:
        api.sample_statistics([c])
    assert e.value.code == api.nat.GINGR_ERR_ARG
    for r in (a, b, c, d):
        r.close()


def test_a_chain_at_a_model_flexibility_error_collects_that_state_and_nothing_after(ctx, oracle):
    """The error state is built numerically: a chain whose start state carries ModelFlexibilityError.  The MH decision
    rejects every proposal from it, so states 1, 2, ... repeat it; the logged run stops there and the device collects
    state 0 only.  The same chain without the error status collects every state."""
    from gingr_b200 import api
    make, dm, dt, m, diag = _builder(ctx, oracle)
    coll = api.SampleCollection(takeEveryN=1)
    bad, good = make(coll, status=api.STATUS_MODEL_FLEXIBILITY_ERROR), make(coll)
    fit0 = bad.downloadState().fit
    bad.mcmcChain(10, 3)
    good.mcmcChain(10, 3)
    sb, sg = api.sample_statistics([bad]), api.sample_statistics([good])
    assert sb.count == 1 and sg.count == 11
    assert bad.mcmcStats()[1][3] == 0 and bad.downloadState().status == api.STATUS_MODEL_FLEXIBILITY_ERROR
    assert np.max(np.abs(sb.mean - fit0)) <= 1e-12 * diag and np.all(np.isnan(sb.cov))
    bad.close(); good.close()


def test_argument_errors(ctx, oracle):
    from gingr_b200 import api, _native as nat
    import ctypes
    make, dm, dt, m, diag = _builder(ctx, oracle)
    lib = ctx._lib

    def samples(regs, cov=False, normal=False):
        arr = (ctypes.c_void_p * len(regs))(*[r.handle for r in regs])
        mean = np.empty((dm.M, 3))
        c9, n3 = np.empty((dm.M, 9)), np.empty((dm.M, 3))
        return lib.gingr_mcmc_samples(arr, len(regs), None, nat.as_dp(mean), nat.as_dp(c9) if cov else None,
                                      nat.as_dp(n3) if normal else None)

    raw = api.IcpRegistration(ctx, dm, dt, api.IcpConfiguration(initialSigma=2.0, endSigma=0.5))
    assert lib.gingr_mcmc_collect(raw.handle, 0, 1, 10) == nat.GINGR_ERR_ARG       # not configured
    reg = make()
    for args in ((-1, 1, 10), (0, -1, 10), (0, 1, -1)):
        assert lib.gingr_mcmc_collect(reg.handle, *args) == nat.GINGR_ERR_ARG
    reg.mcmcChain(2, 1)
    assert samples([reg]) == nat.GINGR_ERR_ARG                                       # collection off
    reg.collectSamples(api.SampleCollection(takeEveryN=0))
    assert samples([reg]) == nat.GINGR_ERR_ARG
    one = make(api.SampleCollection(takeEveryN=1, total=1))
    one.mcmcChain(3, 1)
    assert samples([one]) == nat.GINGR_OK and samples([one], cov=True) == nat.GINGR_ERR_ARG   # one sample
    s1 = api.sample_statistics([one])
    assert s1.count == 1 and np.all(np.isnan(s1.cov))
    two = make(api.SampleCollection(takeEveryN=1))
    two.mcmcChain(3, 1)
    assert samples([two], cov=True, normal=True) == nat.GINGR_OK
    # another model on the same ctx, and another ctx
    make2, dm2, dt2, _, _ = _builder(ctx, oracle, algo="cpd", with_tri=False)
    other = make2(api.SampleCollection(takeEveryN=1))
    other.mcmcChain(3, 1)
    assert samples([two, other]) == nat.GINGR_ERR_ARG
    assert samples([other], normal=True) == nat.GINGR_ERR_ARG                     # no model triangles
    assert api.sample_statistics([other]).normal is None
    ctx2 = api.Context(0)
    make3, dm3, dt3, _, _ = _builder(ctx2, oracle)
    far = make3(api.SampleCollection(takeEveryN=1))
    far.mcmcChain(3, 1)
    assert samples([two, far]) == nat.GINGR_ERR_ARG
    for r in (raw, reg, one, two, other, far, dm3, dt3):   # everything of ctx2 goes before ctx2
        r.close()
    ctx2.close()
