"""The posterior system of an iteration, entry by entry, on every code path of the DMMA Gram (gram.cu).

An iteration forms  Mx = I + D (Phi^T W Phi + LM) D  and  rhs = D (Phi^T W q + landmark terms)  (W = diag(wrow),
u = W q, D = diag(sqrt(lambda)), LM = sum_l Phi_l^T A_l Phi_l with A_l = R^T C_l^-1 R).  gingr_debug_posterior_system
(exported, not in gingr_cuda.h) runs the registration's posterior phase at a given state and returns the kept raw
system: both triangles of Mx as the MH chain reads them, the rhs, and the wrow / u that obs_kernel wrote.

Gram paths (`_paths` mirrors them on the host; every case asserts the one it means to hit), rp = r rounded up to 8:
  corner     rp < 64: one tile, its 64 x 64 corner cut into 16 x 32 warp pieces
  fused rhs  no landmarks and rp % 128 != 0: the residual rides along as column rp of the A panel and comes out as row
             rp of the last tile row; rp % 128 == 64 puts that row on the first row of the second warp row (idle rule)
  gemvT      otherwise the rhs is a pass of its own over Phi
  schedule   T tiles on n CTAs: full rounds, then rem = T mod n tiles whose chunks [0, K1) go to rem main CTAs and
             [K1, K) are cut into n - rem tail ranges, which may cross from one tile into the next

Tier 1: bit-exact at any size.  The basis holds integers |Phi| <= 8, the variances are powers of 4 (sqrt(lambda) a
power of 2), reference, mean and target lie on the 2^-10 grid, the pose is the identity, alpha = 0 and sigma2 a power
of 2, and the observations come from point-cloud ICP, so that every closest point is a target vertex and every
residual a multiple of 2^-10.  Weights are cnt / sigma2 with integer cnt (1 forward; the number of target points
folded onto the vertex reversed; 0 at landmark ids).  Every product Phi_ka w_k Phi_kb is then a multiple of
1 / sigma2, every product Phi_kb w_k q_k a multiple of 2^-10 / sigma2, and every partial sum of them stays below
3M 64 cnt_max / sigma2 < 2^30 / sigma2: all of them are exact in float64, in ANY summation order, and so are the
power-of-two scalings by D and the added identity.  The device's Mx (and the forward rhs) must therefore equal a float64
product of the same inputs bit for bit, whatever its order.  Landmarks at the identity pose with diagonal power-of-two
covariances keep A_l (the host's cofactor inverse, then R^T C^-1 R) and their rhs exact as well.  Reversed, the
residual is the mean of several target points and not dyadic: there Mx is exact and the rhs is held to the tier-2 bound.

Tier 2: 80-bit, bounded.  Orthonormal bases with decaying variances, rotated and translated poses, alpha != 0: CPD with
weights from ~1e-100 to ~1e10, forward and reversed ICP, landmarks with full covariances.  The reference is formed in
numpy longdouble from the device's own wrow and u, so the E-step's and the closest-point error do not enter.  With
u = 2^-53 and gamma_n = n u / (1 - n u):
  Mx    each Gram term Phi_ka (Phi_kb w_k) carries 2 roundings and is summed with the others in some order, a landmark
        term sum_de Phi_la,d A_de Phi_lb,e 9 terms with 3 roundings each; then two scalings by D and the identity:
          |Mx - Mx_ref|_ab <= gamma_n d_a d_b (|Phi|^T W |Phi| + LMabs)_ab + u |Mx_ref|_ab,   n = rows + 9 L + 8
        plus, for landmarks, the error of A_l itself: the host's 3 x 3 cofactor inverse of C_l is accurate to about
        kappa(C_l) u relative to max|C_l^-1| and the rotation adds a few roundings, so
          + 16 kappa(C_l) u d_a d_b (|Phi_l|^T (max|A_l| 1 1^T) |Phi_l|)_ab   (every case has kappa(C_l) <= 10).
  rhs   the same form over |Phi|^T |u| with n = rows + 8: the fused path multiplies q_k by fl(w_k Phi_kb) where the
        reference has fl(w_k q_k) = u_k, one rounding more than the product itself.  Landmark rhs terms are formed from
        p_l - (R b_l + t) and carry roundings relative to |p_l| + |R||b_l| + |t|, not to the residual.
Wiring of the returned vectors:
  ICP   wrow is exactly cnt / sigma2 and 0 at landmark ids; forward, u is w R^T (cp - (R (ref + mean) + t)) with the
        bit-exact closest points of api.icp_closest, to 16 u w (|cp| + |R||b| + |t|).
  CPD   wrow is P1 / (sigma2 lambda) with P1 within the E-step's entry bound (test_estep_paths_gpu.py):
        4 ((2 x_max + 8) 1.2e-16 + 4 u (|x|^2 + |y|^2)_max / (2 sigma2) + (M + N) u) relative, plus 3 u for the two
        divisions of the weight.
"""
import ctypes
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

L = np.longdouble
U = 2.0 ** -53
BT, BK = 128, 32


def _need_longdouble():
    if np.finfo(np.longdouble).eps >= np.finfo(np.float64).eps:
        pytest.skip("no extended precision on this platform")


def _grid(a):
    return np.round(np.asarray(a, dtype=float) * 1024.0) / 1024.0


def _gamma(n):
    return n * U / (1.0 - n * U)


@functools.lru_cache(maxsize=None)
def _num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------------------------------------
# host mirror of the Gram's path choices (gram.cu GramPlan::build, gram_rhs_fusable, gram_ws_kernel)
# ---------------------------------------------------------------------------------------------
def _schedule(rows, r, ncta):
    nt = -(-r // BT)
    ntiles = nt * (nt + 1) // 2
    K = max(1, -(-rows // BK))
    n = ncta
    rem = ntiles % n
    out = dict(ntiles=ntiles, more_tiles=ntiles > n, rem=rem, K1=None, crossing=False)
    if rem:
        K1 = K * rem // n
        ov, pieces = 0.75, float(rem) / (n - rem) + 1.0
        best_t, best_k = 1e300, K1
        for k in range(max(0, K1 - 2), min(K, K1 + 8) + 1):
            t_main = k + ov if k > 0 else 0.0
            t_tail = float(rem) * (K - k) / (n - rem) + (ov * pieces if K - k > 0 else 0.0)
            t = max(t_main, t_tail)
            if t < best_t:
                best_t, best_k = t, k
        tail, ntail = K - best_k, n - rem
        total = rem * tail
        for j in range(ntail):
            u0, u1 = total * j // ntail, total * (j + 1) // ntail
            if u1 > u0 and u0 // tail != (u1 - 1) // tail:
                out["crossing"] = True
        out["K1"] = best_k
    return out


def _paths(rows, r, any_lm=False, max_cta=0):
    rp = (r + 7) // 8 * 8
    ncta = min(_num_sms(), max_cta) if max_cta > 0 else _num_sms()
    fused = not any_lm and rp % BT != 0
    p = dict(corner=rp < 64, fused=fused, rhs_on_warp_row=fused and rp % BT == 64, gemvT=not fused)
    p.update(_schedule(rows, r, ncta))
    return p


# ---------------------------------------------------------------------------------------------
# the hook
# ---------------------------------------------------------------------------------------------
def _hook(ctx):
    from gingr_b200 import _native as nat
    f = ctx._lib.gingr_debug_posterior_system
    f.argtypes = [ctypes.c_void_p, ctypes.POINTER(nat.GingrState), nat.dp, ctypes.c_int32, nat.dp, nat.dp, nat.dp]
    f.restype = ctypes.c_int32
    return f


def _system(reg, state, max_cta=0):
    """(Mx [r, r], rhs [r], wrow [3M], u [3M], code) of the posterior phase at `state`."""
    from gingr_b200 import _native as nat
    r, M = reg.model.rank, reg.model.M
    pod, alpha = state.to_pod()
    sys = np.full((r + 1, r), np.nan)
    wrow, u = np.full(3 * M, np.nan), np.full(3 * M, np.nan)
    code = reg.ctx.check(_hook(reg.ctx)(reg.handle, ctypes.byref(pod), nat.as_dp(alpha), int(max_cta), nat.as_dp(sys),
                                        nat.as_dp(wrow), nat.as_dp(u)))
    return sys[:r], sys[r], wrow, u, code


def _state(r, sigma2, translation=(0.0, 0.0, 0.0), euler=(0.0, 0.0, 0.0), alpha=None):
    from gingr_b200 import api
    shape = np.zeros(r) if alpha is None else np.asarray(alpha, dtype=float)
    pars = api.ModelFittingParameters(1.0, np.asarray(translation, dtype=float), tuple(euler), shape)
    return api.GeneralRegistrationState(pars, np.zeros((1, 3)), sigma2=sigma2)


def _exact_equal(what, got, ref):
    bad = ~(got == ref)
    assert not bad.any(), (f"{what}: {int(bad.sum())} of {bad.size} entries differ, first at {np.argwhere(bad)[0].tolist()}: "
                           f"{got[tuple(np.argwhere(bad)[0])]!r} vs {ref[tuple(np.argwhere(bad)[0])]!r}")


def _check(what, got, ref, lim):
    """|got - ref| <= lim entry by entry in longdouble; returns the worst err / lim."""
    got = np.asarray(got, dtype=float).astype(L)
    err = np.abs(got - ref)
    bad = ~(err <= lim)
    assert not bad.any(), (f"{what}: {int(bad.sum())} of {bad.size} entries out of bound, first at "
                           f"{np.argwhere(bad)[0].tolist()}, worst err/bound "
                           f"{float(np.max(err / np.where(lim > 0, lim, L(1)))):.3g}")
    return float(np.max(err / np.where(lim > 0, lim, L(1))))


# ---------------------------------------------------------------------------------------------
# tier 1: dyadic problems
# ---------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _dyadic(M, r, seed, sl_exp=(-2, 0)):
    """ref, mean, target on the 2^-10 grid, integer basis |Phi| <= 8, sqrt(lambda) = 2^e with e in sl_exp."""
    rng = np.random.default_rng(seed)
    ref = _grid(rng.uniform(-16.0, 16.0, (M, 3)))
    mean = _grid(rng.uniform(-0.25, 0.25, (M, 3)))
    base = ref + mean
    tgt = _grid(np.vstack([base[rng.integers(0, M, M + M // 2)] + rng.normal(scale=0.4, size=(M + M // 2, 3)),
                           rng.uniform(-16.0, 16.0, (max(4, M // 8), 3))]))
    phi = rng.integers(-8, 9, (3 * M, r)).astype(float)
    e = rng.integers(sl_exp[0], sl_exp[1] + 1, r)
    return ref, mean, tgt, phi, 4.0 ** e.astype(float)


def _exact_product(a, b):
    """a^T b in float64: exact for the dyadic inputs above whatever the order, so the GPU does the large ones."""
    if a.shape[0] * a.shape[1] * b.shape[1] < 2e9:
        return a.T @ b
    import torch
    ta, tb = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
    return (ta.T @ tb).cpu().numpy()


class _Icp:
    """A point-cloud ICP registration of a dyadic problem (closed by the caller)."""

    def __init__(self, ctx, M, r, seed=0, reverse=False, sigma2=2.0, landmarks=0, sl_exp=(-2, 0)):
        from gingr_b200 import api
        self.ref, self.mean, self.tgt_pts, self.phi, self.var = _dyadic(M, r, seed, sl_exp)
        self.M, self.r, self.sigma2 = M, r, sigma2
        self.model = api.Model(ctx, self.ref, self.mean.reshape(-1), self.phi, self.var)
        self.target = api.Target(ctx, self.tgt_pts)
        cfg = api.IcpConfiguration(initialSigma=sigma2, endSigma=sigma2 / 2, reverseCorrespondenceDirection=reverse,
                                   correspondenceMethod=api.POINTCLOUD_CLOSEST_POINT)
        self.reg = api.IcpRegistration(ctx, self.model, self.target, cfg)
        self.ctx, self.reverse = ctx, reverse
        self.lm_pid = np.zeros(0, dtype=np.int32)
        if landmarks:
            rng = np.random.default_rng(seed + 1000)
            self.lm_pid = rng.choice(M, landmarks, replace=False).astype(np.int32)
            self.lm_pts = _grid(self.ref[self.lm_pid] + self.mean[self.lm_pid] + rng.uniform(-1, 1, (landmarks, 3)))
            self.lm_cov = np.stack([np.diag(2.0 ** rng.integers(-2, 3, 3).astype(float)) for _ in range(landmarks)])
            self.reg.setLandmarks(self.lm_pid, self.lm_pts, self.lm_cov)

    def close(self):
        for h in (self.reg, self.target, self.model):
            h.close()

    def counts(self, t):
        from gingr_b200 import api
        fit = self.ref + self.mean + np.asarray(t)
        if self.reverse:
            tid, w, _ = api.icp_closest_reversal(self.ctx, self.target, fit, None, api.POINTCLOUD_CLOSEST_POINT)
            cnt = np.bincount(tid[w == 1], minlength=self.M).astype(float)
            return cnt, None
        _, cp, w, _ = api.icp_closest(self.ctx, self.target, fit, None, api.POINTCLOUD_CLOSEST_POINT)
        return w.astype(float), cp - fit

    def reference(self, t=(0.0, 0.0, 0.0)):
        """(wrow, Mx, rhs) in float64 (rhs None when it is not dyadic); exact for the dyadic inputs."""
        cnt, q = self.counts(t)
        cnt[self.lm_pid] = 0.0
        wrow = np.repeat(cnt / self.sigma2, 3)
        d = np.sqrt(self.var)
        G = _exact_product(self.phi * wrow[:, None], self.phi)
        b = None if q is None else _exact_product(self.phi, (wrow * q.reshape(-1))[:, None])[:, 0]
        for l, p in enumerate(self.lm_pid):
            rows = self.phi[3 * p:3 * p + 3]
            A = np.linalg.inv(self.lm_cov[l])
            G = G + rows.T @ A @ rows
            if b is not None:
                b = b + rows.T @ (A @ (self.lm_pts[l] - (self.ref[p] + self.mean[p] + np.asarray(t))))
        Mx = d[:, None] * G * d[None, :] + np.eye(self.r)
        return wrow, Mx, None if b is None else d * b


def _check_exact(case, t=(0.0, 0.0, 0.0), max_cta=0):
    Mx, rhs, wrow, u, code = _system(case.reg, _state(case.r, case.sigma2, translation=t), max_cta)
    assert code == 0
    w_ref, Mx_ref, rhs_ref = case.reference(t)
    _exact_equal("wrow", wrow, w_ref)
    _exact_equal("Mx", Mx, Mx_ref)
    if rhs_ref is not None:
        _exact_equal("rhs", rhs, rhs_ref)
    else:
        _need_longdouble()
        ref = _rhs_ref(case.phi, u, case.var)
        _check("rhs", rhs, ref, _rhs_bound(case.phi, u, case.var, ref))
    return Mx, rhs


# ranks by path: corner, rhs row on the warp boundary, one general tile, tile multiples (gemvT), multi-tile fused
RANKS = [(1, 40), (9, 40), (56, 30), (57, 40), (64, 50), (185, 90), (65, 40), (120, 50), (121, 60), (128, 50),
         (256, 100), (2304, 800), (9472, 3158), (129, 60), (257, 100), (2290, 800), (9400, 3140)]


@pytest.mark.parametrize("r,M", RANKS, ids=[f"r{r}" for r, _ in RANKS])
def test_exact_system_by_rank(ctx, r, M):
    p = _paths(3 * M, r)
    assert p["corner"] == (r <= 56)
    assert p["rhs_on_warp_row"] == (r in (57, 64, 185))
    assert p["gemvT"] == (r in (121, 128, 256, 2304, 9472))
    assert p["more_tiles"] == (r >= 2290)
    case = _Icp(ctx, M, r, seed=r, sl_exp=(-4, -3) if r > 2000 else (-2, 0))
    try:
        _check_exact(case)
    finally:
        case.close()


# rows: one chunk (3M < 32), an exact multiple of 32, ragged, fewer rows than the rank (rank-deficient Gram)
ROWS = [(130, 7), (130, 32), (130, 37), (130, 20), (40, 5), (40, 64), (40, 11), (300, 96)]


@pytest.mark.parametrize("r,M", ROWS, ids=[f"r{r}-rows{3 * m}" for r, m in ROWS])
def test_exact_system_by_rows(ctx, r, M):
    case = _Icp(ctx, M, r, seed=1000 + M, sl_exp=(-4, -2))
    try:
        _check_exact(case)
    finally:
        case.close()


def test_rows_cases_cover_every_kind():
    rows = [3 * m for _, m in ROWS]
    assert any(x < 32 for x in rows) and any(x % 32 == 0 for x in rows)
    assert any(x % 32 and x > 32 for x in rows) and any(3 * m < r for r, m in ROWS)


# CTA caps on ranks whose schedules give rem = 0, K1 = 0 and tail ranges that cross tiles; reversed ICP, so that the
# weights differ from row to row
CAPS = [0, 1, 2, 3, 7, 37, 147]
CAP_RANKS = [(257, 200), (640, 300), (129, 150)]


@pytest.mark.parametrize("max_cta", CAPS)
@pytest.mark.parametrize("r,M", CAP_RANKS, ids=[f"r{r}" for r, _ in CAP_RANKS])
def test_exact_system_with_cta_caps(ctx, r, M, max_cta):
    case = _Icp(ctx, M, r, seed=7 + r, reverse=True)
    try:
        Mx0, _ = _check_exact(case, max_cta=max_cta)
        Mx1, _ = _check_exact(case)   # the plan of the registration is back
        _exact_equal("Mx after the capped call", Mx1, Mx0)
    finally:
        case.close()


def test_cta_cap_cases_cover_the_schedule_splits():
    kinds = [_paths(3 * M, r, max_cta=c) for r, M in CAP_RANKS for c in CAPS]
    assert any(k["rem"] == 0 and k["ntiles"] > 1 for k in kinds)
    assert any(k["K1"] == 0 for k in kinds)
    assert any(k["K1"] is not None and k["K1"] > 0 for k in kinds)
    assert any(k["crossing"] for k in kinds)
    assert any(k["more_tiles"] for k in kinds)


@pytest.mark.parametrize("r,M", [(57, 40), (130, 60), (257, 120), (2290, 800)], ids=lambda v: str(v))
def test_exact_system_reversed(ctx, r, M):
    """Reversed ICP: weights cnt / sigma2 with integer cnt >= 0 per vertex; Mx exact, rhs bounded."""
    case = _Icp(ctx, M, r, seed=40 + r, reverse=True, sl_exp=(-4, -3) if r > 2000 else (-2, 0))
    try:
        cnt, _ = case.counts((0.0, 0.0, 0.0))
        assert len(np.unique(cnt)) >= 3
        _check_exact(case)
    finally:
        case.close()


@pytest.mark.parametrize("r,M,nl", [(40, 40, 4), (130, 60, 7), (256, 100, 3)], ids=["r40", "r130", "r256"])
def test_exact_system_with_landmarks(ctx, r, M, nl):
    """Landmarks (weights 0 at their ids, blocks added by the finish, rhs by gemvT + landmark kernel), all exact."""
    case = _Icp(ctx, M, r, seed=90 + r, landmarks=nl)
    try:
        p = _paths(3 * M, r, any_lm=True)
        assert p["gemvT"]
        _check_exact(case, t=(1.0, -2.0, 0.5))
    finally:
        case.close()


@pytest.mark.parametrize("n", [2, 8, 64])
def test_batched_chains_exact(ctx, n):
    """One update_batch step on n chains (capped Gram schedules for n > 2): the hook on each chain reproduces the exact
    system of its start state, and every chain's new state is bit-identical to a solo registration's."""
    from gingr_b200 import api
    r, M = 300, 160
    cap = max(1, 2 * _num_sms() // n)
    assert _paths(3 * M, r, max_cta=cap)["ntiles"] == 6
    case = _Icp(ctx, M, r, seed=5)
    chains, starts = [], []
    cfg = case.reg.config
    try:
        for k in range(n):
            c = api.IcpRegistration(ctx, case.model, case.target, cfg)
            chains.append(c)
            starts.append(c.initializeState(translation=(float(k % 5) - 2.0, 0.5 * (k % 3), 0.0)))
        api.update_batch(chains, 1)
        got = [c.downloadState() for c in chains]
        for k in (0, n // 2, n - 1):
            solo = api.IcpRegistration(ctx, case.model, case.target, cfg)
            try:
                want = solo.update(starts[k])
            finally:
                solo.close()
            g, w = got[k], want
            _exact_equal("fit", g.fit, w.fit)
            _exact_equal("alpha", g.modelParameters.shape, w.modelParameters.shape)
            _exact_equal("translation", g.modelParameters.translation, w.modelParameters.translation)
            assert tuple(g.modelParameters.euler) == tuple(w.modelParameters.euler) and g.sigma2 == w.sigma2
            t = tuple(starts[k].modelParameters.translation)
            Mx, rhs, wrow, _, code = _system(chains[k], starts[k])
            w_ref, Mx_ref, rhs_ref = case.reference(t)
            _exact_equal("batched wrow", wrow, w_ref)
            _exact_equal("batched Mx", Mx, Mx_ref)
            _exact_equal("batched rhs", rhs, rhs_ref)
    finally:
        for c in chains:
            c.close()
        case.close()


def test_hook_leaves_updates_unchanged(ctx):
    """Updates after hook calls (one of them with a CTA cap) are bit-identical to those of a registration that never
    made them, with the same launch count."""
    case = _Icp(ctx, 300, 257, seed=11, reverse=True)
    from gingr_b200 import api
    other = api.IcpRegistration(ctx, case.model, case.target, case.reg.config)
    try:
        st = _state(case.r, case.sigma2, translation=(0.25, 0.0, -0.5))
        outs = []
        for reg, calls in ((case.reg, (0, 7, 0)), (other, ())):
            for c in calls:
                _system(reg, st, c)
            l0 = ctx.launch_count
            s1 = reg.update(st)
            s2 = reg.update(s1)
            outs.append((s1, s2, ctx.launch_count - l0))
        (a1, a2, la), (b1, b2, lb) = outs
        assert la == lb
        for x, y in ((a1, b1), (a2, b2)):
            _exact_equal("fit", x.fit, y.fit)
            _exact_equal("alpha", x.modelParameters.shape, y.modelParameters.shape)
            assert x.sigma2 == y.sigma2 and tuple(x.modelParameters.euler) == tuple(y.modelParameters.euler)
    finally:
        other.close()
        case.close()


# ---------------------------------------------------------------------------------------------
# tier 2: realistic registrations against longdouble references from the device's wrow and u
# ---------------------------------------------------------------------------------------------
def _gram_ref(phi, wrow, var, lm=()):
    """Mx_ref, the bound matrix of the module docstring."""
    P = phi.astype(L)
    d = np.sqrt(var.astype(L))
    G = (P * wrow.astype(L)[:, None]).T @ P
    A_abs = (np.abs(phi) * np.abs(wrow)[:, None]).T @ np.abs(phi)
    extra = np.zeros_like(A_abs)
    for rows, A, kappa in lm:
        Rl = rows.astype(L)
        G = G + Rl.T @ A @ Rl
        A_abs = A_abs + np.abs(rows).T @ np.abs(A.astype(float)) @ np.abs(rows)
        extra = extra + 16.0 * kappa * U * float(np.max(np.abs(A.astype(float)))) * (np.abs(rows).sum(0)[:, None] *
                                                                                   np.abs(rows).sum(0)[None, :])
    Mx = d[:, None] * G * d[None, :] + np.eye(len(var), dtype=L)
    n = phi.shape[0] + 9 * len(lm) + 8
    df = np.sqrt(var)
    lim = (_gamma(n) * A_abs + extra) * df[:, None] * df[None, :]
    return Mx, lim.astype(L) + L(U) * np.abs(Mx)


def _rhs_ref(phi, u, var):
    return np.sqrt(var.astype(L)) * (phi.astype(L).T @ u.astype(L))


def _rhs_bound(phi, u, var, ref, extra=0.0):
    lim = _gamma(phi.shape[0] + 8) * np.sqrt(var) * (np.abs(phi).T @ np.abs(u)) + extra
    return lim.astype(L) + L(U) * np.abs(ref)


def _rotation(euler):
    from gingr_b200.rotation import euler_to_matrix
    return np.asarray(euler_to_matrix(*euler), dtype=float)


@functools.lru_cache(maxsize=None)
def _smooth(M, r, seed, far=0):
    """Points on a shell of radius ~10 (the last `far` on a sphere of radius 3 at x = 30), an orthonormal smooth basis,
    variances 4 * 0.99^k."""
    from gingr_b200 import synthetic
    rng = np.random.default_rng(seed)
    ref = rng.normal(size=(M, 3))
    ref = 10.0 * ref / np.linalg.norm(ref, axis=1, keepdims=True) * rng.uniform(0.9, 1.1, (M, 1))
    if far:
        ref[M - far:] = ref[M - far:] * 0.3 + (30.0, 0.0, 0.0)
    mean, basis, var = synthetic.make_gpmm(ref, r, seed, lambda0=4.0, decay=0.99, kernel_sigma=6.0)
    mean = 0.05 * rng.normal(size=3 * M)
    return ref, mean, basis, var


POSE = dict(euler=(0.3, -0.2, 0.45), translation=(1.5, -0.75, 2.0))


def _tier2_state(r, sigma2, seed):
    rng = np.random.default_rng(seed)
    return _state(r, sigma2, alpha=0.3 * rng.normal(size=r), **POSE)


def _device_fit(reg, st):
    """The fit of `st` as the device evaluates it (initializeState), so that the host's searches see the same points."""
    return reg.initializeState(general=st).fit


def _check_system(phi, var, Mx, rhs, wrow, u, lm=(), lm_q=()):
    """Mx and rhs against the longdouble reference; lm = [(Phi_l rows, A_l, kappa_l)], lm_q = [(q_l, bound of q_l)] with
    q_l = R^T (p_l - (R b_l + t)) the landmark residual."""
    _need_longdouble()
    Mx_ref, lim = _gram_ref(phi, wrow, var, lm)
    worst = _check("Mx", Mx, Mx_ref, lim)
    _exact_equal("Mx symmetry", Mx, Mx.T)
    d = np.sqrt(var.astype(L))
    ref = _rhs_ref(phi, u, var)
    extra = np.zeros(len(var))
    for (rows, A, _kappa), (q, qerr) in zip(lm, lm_q):
        ref = ref + d * (rows.astype(L).T @ (A @ q))
        extra = extra + np.sqrt(var) * (np.abs(rows).T @ (np.abs(A.astype(float)) @ qerr))
    return max(worst, _check("rhs", rhs, ref, _rhs_bound(phi, u, var, ref, extra)))


def _cpd_p1(fit, tgt, sigma2, w):
    """longdouble P1 of CPD at `fit` and the E-step's relative bound on it."""
    f, t = fit.astype(L), tgt.astype(L)
    x = ((t[None, :, :] - f[:, None, :]) ** 2).sum(-1) / (L(2) * L(sigma2))
    K = np.exp(-x)
    c = (L(2) * L(np.pi) * L(sigma2)) ** (L(3) / L(2)) * L(w) / (L(1) - L(w)) * L(len(fit)) / L(len(tgt))
    P1 = (K / (K.sum(0) + c)[None, :]).sum(1)
    live = x[x < 1085.0 * np.log(2.0)]
    xmax = float(live.max())
    expanded = 4.0 * U * (float(np.max((fit * fit).sum(1))) + float(np.max((tgt * tgt).sum(1)))) / (2.0 * sigma2)
    tol = 4.0 * ((2.0 * xmax + 8.0) * 1.2e-16 + expanded + (len(fit) + len(tgt)) * U) + 3.0 * U
    return P1, tol


@pytest.mark.parametrize("r,M", [(50, 600), (130, 900)], ids=["r50", "r130"])
def test_cpd_system_bounded(ctx, r, M):
    """CPD at sigma2 = 0.01, lambda = 1e-7, w = 0.1: weights P1 / (sigma2 lambda) from ~1e-100 (a cluster of model points
    whose targets sit 2.25 further out, so no target is nearer than ~2.2) to ~1e10 (targets 0.03 from their points)."""
    from gingr_b200 import api
    nfar = M // 10
    ref, mean, phi, var = _smooth(M, r, r, far=nfar)
    sigma2, lam, w = 0.01, 1e-7, 0.1
    model = api.Model(ctx, ref, mean, phi, var)
    st = _tier2_state(r, sigma2, r)
    fit_target = api.Target(ctx, ref[:4])
    reg0 = api.CpdRegistration(ctx, model, fit_target, api.CpdConfiguration(initialSigma=sigma2))
    fit = _device_fit(reg0, st)
    reg0.close()
    fit_target.close()
    rng = np.random.default_rng(r)
    near, far = fit[:M - nfar], fit[M - nfar:]
    tgt = near[rng.integers(0, len(near), M)] + rng.normal(scale=0.03, size=(M, 3))
    c = far.mean(0)
    out = far - c
    tgt = np.vstack([tgt, c + out * (1.0 + 2.25 / np.linalg.norm(out, axis=1, keepdims=True))])
    target = api.Target(ctx, tgt)
    reg = api.CpdRegistration(ctx, model, target, api.CpdConfiguration(initialSigma=sigma2, w=w, lambda_=lam))
    try:
        Mx, rhs, wrow, u, code = _system(reg, st)
        assert code == 0
        _need_longdouble()
        P1, tol = _cpd_p1(fit, tgt, sigma2, w)
        w_ref = np.repeat(P1 / (L(sigma2) * L(lam)), 3)
        _check("wrow", wrow, w_ref, L(tol) * w_ref)
        assert wrow.min() < 1e-90 and wrow.max() > 1e9, (wrow.min(), wrow.max())
        _check_system(phi, var, Mx, rhs, wrow, u)
    finally:
        for h in (reg, target, model):
            h.close()


@pytest.mark.parametrize("reverse", [False, True], ids=["forward", "reversed"])
@pytest.mark.parametrize("r,M", [(64, 500), (256, 1200), (700, 1200)], ids=["r64", "r256", "r700"])
def test_icp_system_bounded(ctx, r, M, reverse):
    from gingr_b200 import api
    ref, mean, phi, var = _smooth(M, r, r + 1)
    sigma2 = 0.7
    rng = np.random.default_rng(r)
    st = _tier2_state(r, sigma2, r + 1)
    model = api.Model(ctx, ref, mean, phi, var)
    R, t = _rotation(POSE["euler"]), np.asarray(POSE["translation"])
    tgt = (ref + mean.reshape(-1, 3))[rng.integers(0, M, M)] @ R.T + t + rng.normal(scale=0.2, size=(M, 3))
    target = api.Target(ctx, tgt)
    cfg = api.IcpConfiguration(initialSigma=sigma2, reverseCorrespondenceDirection=reverse,
                               correspondenceMethod=api.POINTCLOUD_CLOSEST_POINT)
    reg = api.IcpRegistration(ctx, model, target, cfg)
    try:
        fit = _device_fit(reg, st)
        Mx, rhs, wrow, u, code = _system(reg, st)
        assert code == 0
        b = ref + mean.reshape(-1, 3)
        if reverse:
            tid, w01, _ = api.icp_closest_reversal(ctx, target, fit, None, api.POINTCLOUD_CLOSEST_POINT)
            cnt = np.bincount(tid[w01 == 1], minlength=M).astype(float)
        else:
            _, cp, w01, _ = api.icp_closest(ctx, target, fit, None, api.POINTCLOUD_CLOSEST_POINT)
            cnt = w01.astype(float)
        _exact_equal("wrow", wrow, np.repeat(cnt / sigma2, 3))
        if not reverse:
            _need_longdouble()
            RL, tL = R.astype(L), t.astype(L)
            res = cp.astype(L) - (b.astype(L) @ RL.T + tL)
            u_ref = (np.repeat(cnt / sigma2, 3).astype(L) * (res @ RL).reshape(-1))
            mag = np.abs(cp).max(1) + (np.abs(b) @ np.abs(R).T).max(1) + np.abs(t).max()
            _check("u", u, u_ref, L(16.0 * U) * np.repeat(cnt / sigma2 * mag, 3).astype(L))
        _check_system(phi, var, Mx, rhs, wrow, u)
    finally:
        for h in (reg, target, model):
            h.close()


def test_landmark_system_bounded(ctx):
    """Forward ICP with 6 landmarks of full covariance (kappa <= 10) under a rotated pose: weights 0 at landmark ids,
    the finish's landmark blocks and the landmark rhs bounded."""
    from gingr_b200 import api
    r, M, nl = 130, 700, 6
    ref, mean, phi, var = _smooth(M, r, 3)
    sigma2 = 0.5
    rng = np.random.default_rng(3)
    R, t = _rotation(POSE["euler"]), np.asarray(POSE["translation"])
    b = ref + mean.reshape(-1, 3)
    tgt = b[rng.integers(0, M, M)] @ R.T + t + rng.normal(scale=0.2, size=(M, 3))
    pid = rng.choice(M, nl, replace=False).astype(np.int32)
    pts = b[pid] @ R.T + t + rng.normal(scale=0.3, size=(nl, 3))
    covs, kappas = [], []
    for _ in range(nl):
        Q, _r = np.linalg.qr(rng.normal(size=(3, 3)))
        ev = np.array([1.0, rng.uniform(1.0, 9.0), 9.5]) * 0.2
        covs.append(Q @ np.diag(ev) @ Q.T)
        kappas.append(float(np.linalg.cond(covs[-1])))
    assert max(kappas) <= 10.0
    model = api.Model(ctx, ref, mean, phi, var)
    target = api.Target(ctx, tgt)
    cfg = api.IcpConfiguration(initialSigma=sigma2, useLandmarkCorrespondence=True,
                               correspondenceMethod=api.POINTCLOUD_CLOSEST_POINT)
    reg = api.IcpRegistration(ctx, model, target, cfg)
    reg.setLandmarks(pid, pts, np.stack(covs))
    st = _tier2_state(r, sigma2, 3)
    try:
        fit = _device_fit(reg, st)
        Mx, rhs, wrow, u, code = _system(reg, st)
        assert code == 0
        _, _, w01, _ = api.icp_closest(ctx, target, fit, None, api.POINTCLOUD_CLOSEST_POINT)
        cnt = w01.astype(float)
        cnt[pid] = 0.0
        _exact_equal("wrow", wrow, np.repeat(cnt / sigma2, 3))
        _need_longdouble()
        RL, tL = R.astype(L), t.astype(L)
        lm, qs = [], []
        for l, p in enumerate(pid):
            C = np.asarray(covs[l], dtype=L)
            # the float64 inverse and one Newton step X <- X (2I - C X): C^-1 to longdouble accuracy
            X = np.linalg.inv(covs[l]).astype(L)
            X = X @ (L(2) * np.eye(3, dtype=L) - C @ X)
            A = RL.T @ X @ RL
            q = (pts[l].astype(L) - (RL @ b[p].astype(L) + tL)) @ RL
            # q's roundings are relative to |p| + |R||b| + |t|; A's error (16 kappa u max|A|) is moved onto q
            mag = np.abs(pts[l]).max() + (np.abs(R) @ np.abs(b[p])).max() + np.abs(t).max()
            qerr = (16.0 * U * mag + 16.0 * kappas[l] * U * float(np.abs(q).max())) * np.ones(3)
            lm.append((phi[3 * p:3 * p + 3], A, kappas[l]))
            qs.append((q, qerr))
        _check_system(phi, var, Mx, rhs, wrow, u, lm=lm, lm_q=qs)
    finally:
        for h in (reg, target, model):
            h.close()
