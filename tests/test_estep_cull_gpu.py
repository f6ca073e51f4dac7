"""Tile-pair culling of the CPD E-step: at sizes where the library culls, the results match the dense sweeps (culling forced
off with GINGR_ESTEP_CULL=0) and the oracle, culling really happens, a non-finite column turns it off, and the k-d orders
of the fit and the target do not show through in the outputs."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _sphere(n, seed, radius=100.0, noise=1.0):
    rng = np.random.default_rng(seed)
    p = rng.normal(size=(n, 3))
    p *= radius / np.linalg.norm(p, axis=1, keepdims=True)
    return p + noise * rng.normal(size=(n, 3))


@pytest.fixture(scope="module")
def big():
    return _sphere(20000, 1), _sphere(40000, 2)


def _estep(ctx, monkeypatch, fit, target, sigma2, w, cull):
    from gingr_b200 import api
    monkeypatch.setenv("GINGR_ESTEP_CULL", cull)
    t = api.Target(ctx, target)
    try:
        return api.cpd_estep(ctx, t, fit, sigma2, w)
    finally:
        t.close()


def _close(a, b, rtol):
    a, b = np.asarray(a), np.asarray(b)
    assert np.array_equal(np.isnan(a), np.isnan(b))
    ok = ~np.isnan(b)
    np.testing.assert_allclose(a[ok], b[ok], rtol=rtol, atol=rtol * float(np.max(np.abs(b[ok]), initial=0.0)))


@pytest.mark.parametrize("sigma2", [10.0, 25.0, 100.0])
@pytest.mark.parametrize("w", [0.1, 0.0])
def test_culled_estep_matches_dense(ctx, monkeypatch, big, sigma2, w):
    fit, tgt = big
    auto = _estep(ctx, monkeypatch, fit, tgt, sigma2, w, "")
    dense = _estep(ctx, monkeypatch, fit, tgt, sigma2, w, "0")
    for x, y in zip(auto, dense):
        _close(x, y, 1e-12)


@pytest.mark.parametrize("sigma2", [10.0, 100.0])
def test_forced_cull_matches_oracle(ctx, oracle, monkeypatch, sigma2):
    fit, tgt = _sphere(1500, 3), _sphere(4000, 4)
    P1, Pt1, PX = _estep(ctx, monkeypatch, fit, tgt, sigma2, 0.1, "1")
    P = oracle.cpd_P(fit, tgt, sigma2, 0.1)
    r1, rt1, rx = oracle.P_reductions(P, tgt)
    np.testing.assert_allclose(P1, r1, rtol=1e-9, atol=1e-300)
    np.testing.assert_allclose(Pt1, rt1, rtol=1e-9, atol=1e-300)
    np.testing.assert_allclose(PX, rx, rtol=1e-9, atol=1e-9 * float(np.abs(rx).max()))


def test_shuffled_input_order_gives_the_same_result(ctx, monkeypatch, big):
    fit, tgt = big
    rng = np.random.default_rng(5)
    pf, pt = rng.permutation(len(fit)), rng.permutation(len(tgt))
    a = _estep(ctx, monkeypatch, fit, tgt, 25.0, 0.1, "")
    b = _estep(ctx, monkeypatch, fit[pf], tgt[pt], 25.0, 0.1, "")
    _close(b[0], a[0][pf], 1e-13)
    _close(b[1], a[1][pt], 1e-13)
    _close(b[2], a[2][pf], 1e-13)


def test_nonfinite_column_turns_culling_off(ctx, monkeypatch, big):
    """w = 0 and a target point far from every model point: its column sum underflows to 0, w_j = 1/0, and the dense
    sums give NaN for every P1_i and PX_i (0 * inf), as the reference does.  Culling would have dropped that column."""
    fit, tgt = big
    tgt = np.vstack([tgt, [[1.0e4, 0.0, 0.0]]])
    auto = _estep(ctx, monkeypatch, fit, tgt, 10.0, 0.0, "")
    dense = _estep(ctx, monkeypatch, fit, tgt, 10.0, 0.0, "0")
    assert np.all(np.isnan(auto[0])) and np.all(np.isnan(auto[2]))
    assert np.isnan(auto[1][-1])
    for x, y in zip(auto, dense):
        _close(x, y, 1e-12)


def test_culling_happens_in_a_registration(ctx, monkeypatch):
    """The live tile-pair fractions of the profile fall below 1 once sigma2 is small, and are 1 with culling off."""
    from gingr_b200 import api, synthetic
    M, N = 20000, 100000
    ref = synthetic.fibonacci_sphere(M)
    tv = synthetic.make_target(synthetic.fibonacci_sphere(N), 0)
    mean, basis, var = synthetic.make_gpmm(ref, 32, 1, orthonormal=False)
    model = api.Model(ctx, ref, mean, basis, var)
    tgt = api.Target(ctx, tv)
    live = {}
    for cull in ("", "0"):
        monkeypatch.setenv("GINGR_ESTEP_CULL", cull)
        reg = api.CpdRegistration(ctx, model, tgt, api.CpdConfiguration(maxIterations=10 ** 6, w=0.1, initialSigma=25.0))
        reg.initializeState(globalTransformation=api.RIGID_TRANSFORMS)
        reg.setProfiling(True)
        reg.updateChain(2)
        ms, it = reg.getProfile()
        live[cull] = (ms[6] / it, ms[7] / it)
        reg.close()
    model.close(); tgt.close()
    assert live["0"] == (1.0, 1.0)
    assert 0.0 < live[""][0] < 0.9 and 0.0 < live[""][1] < 0.9, live
