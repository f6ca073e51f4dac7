"""Every code path of the CPD / BCPD E-step (estep.cu) against an 80-bit reference, entry by entry.

The E-step chooses its arithmetic per launch from the inputs:
  expanded   -k|x - y|^2 = -k|x|^2 - k|y|^2 + 2k x.y        while 64 log2(e) d2max / (2 sigma2) < 2^22  (estep_expand_ok;
             CPD both sweeps, BCPD sweep B only: sweep A has a row factor)
  SAFE       difference form, one range compare              while 256 log2(e) d2max / (2 sigma2) < 2^31 - 2^20
                                                             (estep_safe_range)
  clamped    difference form, full range check               otherwise
with d2max = 3 (max|fit| + max|target|)^2 (d2_bound, capi.cu).  On top of that it may cull tile pairs
(GINGR_ESTEP_CULL) and split either sweep's streamed dimension over several CTAs (GINGR_ESTEP_SPLITS_A / _B).
`_paths` mirrors the two predicates on the host and every case asserts the path it means to hit.

Reference.  P1, Pt1, PX (CPD.scala:54-75) and nu, nu', Nhat, xhat (BCPD.scala:167-209, as oracle.bcpd_estep restates
them) in numpy longdouble straight from the definitions, together with the column sums and the condition sums
S_i = sum_j P_ij |x_j|.  Coordinates are multiples of 2^-10 and translations are integers, so a translated copy has
exactly the same pair distances: P1 and Pt1 are unchanged, PX gains P1_i t and S_i grows by at most |t| P1_i.  One
reference therefore checks every translation of its geometry.

Entry-wise bounds (u = 2^-53).  Each kernel value K_ij = exp(-x), x = d^2 / (2 sigma2), carries a relative error of
  difference paths   delta(x) = (2x + 8) 1.2e-16     (d^2 is exact on the grid; the bound of the kernel accuracy test
                                                      in test_estep_gpu.py: the scaled argument is rounded once)
  expanded path      delta(x) + 4u (|x|^2 + |y|^2) / (2 sigma2)   (cancellation of the expanded square, estep.cu)
delta_max is taken over the pairs whose K the kernel can represent (x < 1085 ln 2): the others are exactly 0 there and
below 2^-1085 in the reference.  Column sums add M positive terms (relative error <= delta_max + M u), the
denominator, its reciprocal and Pt1 add a few roundings, and each row sum adds N positive terms K_ij w_j whose own
error is that of K_ij plus that of w_j.  To first order every P1 / Pt1 / nu / nu' entry is therefore within
2 delta_max + (M + N + 3) u of itself and every PX entry within the same factor times S_i (each term of PX is a term of
P1 times x_j).  The tests allow c = 4 times (delta_max + (M + N) u): twice the first-order count, which leaves room
for the few roundings of the scalar c, of the BCPD row factors and of the reference's own 80-bit sums, while a single
wrong term of relative size 1e-12 still fails.  Culling drops at most 2^-60 of any sum, far below u.  No case has an
entry whose only terms are subnormal (test_gradual_underflow_band covers those).
"""
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

L = np.longdouble
U = 2.0 ** -53
C_BOUND = 4.0
LOG2E = 1.4426950408889634074
X_REPRESENTABLE = 1085.0 * np.log(2.0)   # the kernel keeps K = 2^64-biased values down to 2^-1085
CHUNK = 1 << 18                          # pairs per longdouble block
MAX_SPLITS = "1000000"                   # clamped by the planner to ceil(M / 128), ceil(N / 128)


def _need_longdouble():
    if np.finfo(np.longdouble).eps >= np.finfo(np.float64).eps:
        pytest.skip("no extended precision on this platform")


def _grid(a):
    return np.round(np.asarray(a, dtype=float) * 1024.0) / 1024.0


# ---------------------------------------------------------------------------------------------
# host mirror of the path predicates (capi.cu d2_bound, estep.cu estep_expand_ok / estep_safe_range)
# ---------------------------------------------------------------------------------------------
def _d2_bound(fit, tgt):
    s = float(np.max(np.abs(fit))) + float(np.max(np.abs(tgt)))
    return 3.0 * s * s


def _expand_ratio(fit, tgt, sigma2):
    return _d2_bound(fit, tgt) * (64.0 * LOG2E / (2.0 * sigma2)) / 4194304.0


def _safe_ratio(fit, tgt, sigma2):
    return _d2_bound(fit, tgt) * (256.0 * LOG2E / (2.0 * sigma2)) / 2146435072.0


def _paths(fit, tgt, sigma2, rowf=False):
    """(sweep A, sweep B) arithmetic of one launch: 'expanded', 'safe' or 'clamped'."""
    d2max = _d2_bound(fit, tgt)
    ok = sigma2 > 0.0 and d2max > 0.0
    expand = ok and d2max * (64.0 * LOG2E / (2.0 * sigma2)) < 4194304.0
    safe = ok and d2max * (256.0 * LOG2E / (2.0 * sigma2)) < 2146435072.0
    diff = "safe" if safe else "clamped"
    return ("expanded" if expand and not rowf else diff), ("expanded" if expand else diff)


def _shift_for(fit, tgt, sigma2, which, ratio):
    """Integer t such that translating both clouds by (t, t, t) puts the launch at `ratio` times the `which` switch."""
    per_d2 = (64.0 * LOG2E / (2.0 * sigma2)) / 4194304.0 if which == "expand" else \
        (256.0 * LOG2E / (2.0 * sigma2)) / 2146435072.0
    s = np.sqrt(ratio / per_d2 / 3.0)
    t = float(round((s - fit.max() - tgt.max()) / 2.0))
    assert t > max(-fit.min(), -tgt.min())
    return t


def _kd_tiles(pts, big, small):
    """Index sets of the aligned `small`-point runs of estep.cu's kd_order (which points share a tile; the order
    inside a tile is not needed)."""
    out = []
    todo = [np.arange(len(pts))]
    while todo:
        idx = todo.pop()
        n = len(idx)
        g = big if n > big else small
        if n <= g:
            out.append(idx)
            continue
        sub = pts[idx]
        ax = int(np.argmax(sub.max(0) - sub.min(0)))
        order = idx[np.lexsort((idx, sub[:, ax]))]
        mid = -(-n // g) // 2 * g
        todo += [order[mid:], order[:mid]]
    return out


# ---------------------------------------------------------------------------------------------
# 80-bit references
# ---------------------------------------------------------------------------------------------
def _kernel_matrix(fit, tgt, sigma2):
    """K [M, N] in longdouble and the largest x = d^2 / (2 sigma2) the kernel can represent."""
    f, t = fit.astype(L), tgt.astype(L)
    M, N = len(f), len(t)
    k = L(1) / (L(2) * L(sigma2))
    K = np.empty((M, N), dtype=L)
    xmax = 0.0
    rows = max(1, CHUNK // N)
    for i0 in range(0, M, rows):
        d2 = ((t[None, :, :] - f[i0:i0 + rows, None, :]) ** 2).sum(-1)
        x = d2 * k
        K[i0:i0 + rows] = np.exp(-x)
        live = x[x < X_REPRESENTABLE]
        if live.size:
            xmax = max(xmax, float(live.max()))
    return K, xmax


def _reductions(K, rowf, a, c, tgt):
    """P = rowf_i K_ij / (a sum_i rowf_i K_ij + c) and its reductions."""
    t = tgt.astype(L)
    FK = K * rowf[:, None]
    colsum = FK.sum(0)
    wj = L(1) / (a * colsum + c)
    P = FK * wj[None, :]
    return dict(P1=P.sum(1), Pt1=colsum * wj, PX=P @ t, S=P @ np.sqrt((t * t).sum(1)), colsum=colsum)


@functools.lru_cache(maxsize=None)
def _cpd_ref(name, sigma2, w):
    _need_longdouble()
    fit, tgt = GEOMETRIES[name]()
    K, xmax = _kernel_matrix(fit, tgt, sigma2)
    M, N = len(fit), len(tgt)
    c = (L(2) * L(np.pi) * L(sigma2)) ** (L(3) / L(2)) * L(w) / (L(1) - L(w)) * L(M) / L(N)
    r = _reductions(K, np.ones(M, dtype=L), L(1), c, tgt)
    r["xmax"] = xmax
    return r


@functools.lru_cache(maxsize=None)
def _bcpd_ref(name, sigma2, s, w):
    _need_longdouble()
    y, x = GEOMETRIES[name]()
    sig, al = _bcpd_factors(len(y))
    K, xmax = _kernel_matrix(y, x, sigma2)
    M, N = len(y), len(x)
    norm = (L(2) * L(np.pi) * L(sigma2)) ** (-L(3) / L(2))
    rowf = (L(1) - L(w)) * norm * np.exp(-L(s) / (L(2) * L(sigma2)) * (L(3) * sig.astype(L))) * al.astype(L)
    r = _reductions(K, rowf, L(1) - L(w), L(w) / L(N), x)
    r["xmax"] = xmax
    return r


def _bcpd_factors(M):
    rng = np.random.default_rng(77)
    return rng.uniform(0.1, 1.0, M), rng.uniform(0.5, 1.5, M) / M


# ---------------------------------------------------------------------------------------------
# geometries (all coordinates on the 2^-10 grid)
# ---------------------------------------------------------------------------------------------
def _cube_cloud():
    rng = np.random.default_rng(1)
    fit = _grid(rng.uniform(-8.0, 8.0, (513, 3)))
    tgt = _grid(fit[rng.integers(0, 513, 1537)] + rng.normal(scale=1.5, size=(1537, 3)))
    return fit, tgt


def _cube_cloud_far_row():
    """The cube cloud with its last model point moved 8064 along x: every pair of that row has a scaled exponent
    of about 3e9, beyond the 2^31 - 2^20 the SAFE form handles, so only the full range check makes its K 0."""
    fit, tgt = _cube_cloud()
    fit = fit.copy()
    fit[-1] = (8064.0, 0.0, 0.0)
    return fit, tgt


def _clusters(M, N, n, spacing=48.0, seed=3):
    """n clusters of side 8 (targets: a model point + uniform noise of +-1) spaced along x; model and target sizes
    split as evenly as possible."""
    rng = np.random.default_rng(seed)
    fit, tgt = [], []
    for c, (m, k) in enumerate(zip(np.array_split(np.arange(M), n), np.array_split(np.arange(N), n))):
        centre = np.array([c * spacing, 0.0, 0.0])
        f = rng.uniform(-4.0, 4.0, (len(m), 3)) + centre
        fit.append(f)
        tgt.append(f[rng.integers(0, len(m), len(k))] + rng.uniform(-1.0, 1.0, (len(k), 3)))
    return _grid(np.vstack(fit)), _grid(np.vstack(tgt))


def _far_targets(mixed):
    """Model clusters B (x ~ 0) and C (x ~ 80), 512 points each.  640 targets near B, a far group at x ~ 30 whose
    nearest model points are B's at distance 27.5 .. 33 (column sums ~ 1e-210 at sigma2 = 0.75, so w_j ~ 1e210 with
    w = 0), and targets near C.  mixed: 32 far points that share one 64-column tile with the 32 lowest-x C targets, so
    that tile's w_min is ~ 1 and its w_max ~ 1e210; otherwise 64 far points with whole tiles of their own."""
    rng = np.random.default_rng(11 if mixed else 12)
    B = rng.uniform(-2.0, 2.0, (512, 3))
    C = rng.uniform(-2.0, 2.0, (512, 3)) + (80.0, 0.0, 0.0)
    nb, nf, nc = 640, (32 if mixed else 64), 641
    tb = B[rng.integers(0, 512, nb)] + rng.uniform(-0.5, 0.5, (nb, 3))
    tf = rng.uniform(-0.5, 0.5, (nf, 3)) + (30.0, 0.0, 0.0)
    tc = C[rng.integers(0, 512, nc)] + rng.uniform(-0.5, 0.5, (nc, 3))
    return _grid(np.vstack([B, C])), _grid(np.vstack([tb, tf, tc]))


def _planar():
    rng = np.random.default_rng(21)
    f = np.zeros((513, 3)); f[:, :2] = rng.uniform(0.0, 64.0, (513, 2))
    t = np.zeros((1535, 3)); t[:, :2] = f[rng.integers(0, 513, 1535), :2] + rng.normal(scale=0.7, size=(1535, 2))
    return _grid(f), _grid(t)


def _collinear():
    rng = np.random.default_rng(22)
    f = np.zeros((511, 3)); f[:, 0] = rng.uniform(0.0, 512.0, 511)
    t = np.zeros((1537, 3)); t[:, 0] = f[rng.integers(0, 511, 1537), 0] + rng.normal(scale=1.0, size=1537)
    return _grid(f), _grid(t)


def _repeated():
    """257 copies of one target point (whole 64-column tiles of a single point) and 33 copies of one model point
    next to it, in a cube of side 32."""
    rng = np.random.default_rng(23)
    p = np.array([5.0, 7.0, 3.0])
    f = np.vstack([rng.uniform(0.0, 32.0, (480, 3)), np.tile(p + 0.25, (33, 1))])
    t = np.vstack([f[rng.integers(0, 513, 1280)] + rng.normal(scale=0.5, size=(1280, 3)), np.tile(p, (257, 1))])
    return _grid(f), _grid(t)


def _anisotropic():
    """1000 : 1 : 1e-3 boxes (z is 0 or 2^-10)."""
    rng = np.random.default_rng(24)
    ext = np.array([1000.0, 1.0, 0.0])
    f = rng.uniform(0.0, 1.0, (2049, 3)) * ext
    f[:, 2] = rng.integers(0, 2, 2049) / 1024.0
    t = f[rng.integers(0, 2049, 1537)] + rng.normal(scale=[1.0, 0.1, 0.0], size=(1537, 3))
    t[:, 2] = rng.integers(0, 2, 1537) / 1024.0
    return _grid(f), _grid(t)


def _small(M, N):
    def make():
        rng = np.random.default_rng(M * 7919 + N)
        fit = _grid(rng.uniform(0.0, 24.0, (M, 3)))
        return fit, _grid(fit[rng.integers(0, M, N)] + rng.normal(scale=1.0, size=(N, 3)))
    return make


GEOMETRIES = {
    "cube": _cube_cloud,
    "cube_far_row": _cube_cloud_far_row,
    "clusters3_aligned": lambda: _clusters(1536, 2304, 3),
    "clusters3_ragged": lambda: _clusters(2049, 1537, 3),
    "clusters2_ragged": lambda: _clusters(511, 3073, 2),
    "far_alone": lambda: _far_targets(False),
    "far_mixed": lambda: _far_targets(True),
    "planar": _planar,
    "collinear": _collinear,
    "repeated": _repeated,
    "anisotropic": _anisotropic,
}
for _m, _n in [(31, 63), (33, 65), (31, 257), (33, 255), (513, 63), (2049, 65)]:
    GEOMETRIES[f"small_{_m}x{_n}"] = _small(_m, _n)


# ---------------------------------------------------------------------------------------------
# running and checking
# ---------------------------------------------------------------------------------------------
def _env(monkeypatch, cull, splits=None):
    monkeypatch.setenv("GINGR_ESTEP_CULL", cull)
    if splits is None:
        monkeypatch.delenv("GINGR_ESTEP_SPLITS_A", raising=False)
        monkeypatch.delenv("GINGR_ESTEP_SPLITS_B", raising=False)
    else:
        monkeypatch.setenv("GINGR_ESTEP_SPLITS_A", splits)
        monkeypatch.setenv("GINGR_ESTEP_SPLITS_B", splits)


def _cpd(ctx, fit, tgt, sigma2, w):
    from gingr_b200 import api
    t = api.Target(ctx, tgt)
    try:
        return api.cpd_estep(ctx, t, fit, sigma2, w)
    finally:
        t.close()


def _check(what, got, ref, lim):
    """|got - ref| <= lim entry by entry (an entry with lim = 0 must be exact); returns the worst err / lim."""
    got = np.asarray(got, dtype=float).astype(L)
    ref, lim = np.broadcast_arrays(ref, lim)
    assert np.all((ref == 0) | (np.abs(ref) > 2.0 ** -1000)), f"{what}: reference entry in the subnormal range"
    err = np.abs(got - ref)
    bad = ~(err <= lim)
    ratio = err / np.where(lim > 0, lim, L(1))
    assert not bad.any(), (f"{what}: {int(bad.sum())} of {bad.size} entries out of bound, first at "
                           f"{np.argwhere(bad)[0].tolist()}, worst err/bound {float(np.max(ratio)):.3g}")
    return float(np.max(ratio))


def _tol(ref, M, N, expanded_term=0.0):
    return L(C_BOUND * ((2.0 * ref["xmax"] + 8.0) * 1.2e-16 + expanded_term + (M + N) * U))


def _expanded_term(fit, tgt, sigma2):
    return 4.0 * U * (float(np.max((fit * fit).sum(1))) + float(np.max((tgt * tgt).sum(1)))) / (2.0 * sigma2)


def _check_cpd(got, ref, tol, shift=0.0):
    P1, Pt1, PX = got
    rPX = ref["PX"] + ref["P1"][:, None] * L(shift)
    S = ref["S"] + L(abs(shift) * np.sqrt(3.0)) * ref["P1"]
    return max(_check("P1", P1, ref["P1"], tol * ref["P1"]),
               _check("Pt1", Pt1, ref["Pt1"], tol * ref["Pt1"]),
               _check("PX", PX, rPX, tol * S[:, None]))


def _cpd_case(ctx, monkeypatch, name, sigma2, w, cull, want, splits=None):
    """One kernel-level CPD E-step of a named geometry, checked entry by entry; `want` is the path it must take."""
    fit, tgt = GEOMETRIES[name]()
    ref = _cpd_ref(name, sigma2, w)
    assert _paths(fit, tgt, sigma2) == (want, want)
    _env(monkeypatch, cull, splits)
    got = _cpd(ctx, fit, tgt, sigma2, w)
    extra = _expanded_term(fit, tgt, sigma2) if want == "expanded" else 0.0
    return _check_cpd(got, ref, _tol(ref, len(fit), len(tgt), extra))


# ---------------------------------------------------------------------------------------------
# arithmetic paths
# ---------------------------------------------------------------------------------------------
SIGMA2_CUBE = 4.0
TRANSLATIONS = [("expand", 0.9, "expanded"), ("expand", 1.1, "safe"), ("expand", 16.0, "safe"),
                ("safe", 0.9, "safe"), ("safe", 1.1, "clamped")]


@pytest.mark.parametrize("cull", ["0", "1"])
@pytest.mark.parametrize("w", [0.0, 0.1])
@pytest.mark.parametrize("which,ratio,path", TRANSLATIONS, ids=[f"{p}-{r}x{s}" for s, r, p in TRANSLATIONS])
def test_cpd_paths_near_their_switches(ctx, monkeypatch, which, ratio, path, w, cull):
    """One cube cloud, translated so that d2max sits just below / above each switch and far past the expanded one.
    The expanded path is held to its own bound; the difference paths to delta(x) alone, which the expanded form
    misses by far at 16x its switch."""
    fit0, tgt0 = GEOMETRIES["cube"]()
    ref = _cpd_ref("cube", SIGMA2_CUBE, w)
    t = _shift_for(fit0, tgt0, SIGMA2_CUBE, which, ratio)
    fit, tgt = fit0 + t, tgt0 + t
    got_ratio = (_expand_ratio if which == "expand" else _safe_ratio)(fit, tgt, SIGMA2_CUBE)
    assert abs(got_ratio / ratio - 1.0) < 0.02, got_ratio
    assert _paths(fit, tgt, SIGMA2_CUBE) == (path, path)
    _env(monkeypatch, cull)
    got = _cpd(ctx, fit, tgt, SIGMA2_CUBE, w)
    extra = _expanded_term(fit, tgt, SIGMA2_CUBE) if path == "expanded" else 0.0
    _check_cpd(got, ref, _tol(ref, len(fit), len(tgt), extra), shift=t)


@pytest.mark.parametrize("cull", ["0", "1"])
@pytest.mark.parametrize("w", [0.0, 0.1])
def test_cpd_clamped_path_with_a_far_model_point(ctx, monkeypatch, w, cull):
    """A model point 8064 away: its pairs leave the range of the SAFE form, their K must come out exactly 0 (so its P1
    and PX are exactly 0) and every other entry must be untouched."""
    fit, tgt = GEOMETRIES["cube_far_row"]()
    d2 = ((tgt - fit[-1]) ** 2).sum(1)
    scaled = d2 * (256.0 * LOG2E / (2.0 * SIGMA2_CUBE))
    assert scaled.min() > 2.0 ** 31 + 2.0 ** 20 and scaled.max() < 2.0 ** 32
    _cpd_case(ctx, monkeypatch, "cube_far_row", SIGMA2_CUBE, w, cull, "clamped")
    assert _cpd_ref("cube_far_row", SIGMA2_CUBE, w)["P1"][-1] == 0


# ---------------------------------------------------------------------------------------------
# BCPD: sweep A in the difference form (row factors), sweep B expanded when allowed
# ---------------------------------------------------------------------------------------------
BCPD_ARGS = (SIGMA2_CUBE, 1.1, 0.2)   # sigma2, s, w


def _check_bcpd(got, ref, tol, shift=0.0):
    nu, nup, nhat, xhat = got
    N = len(nup)
    r = max(_check("nu", nu, ref["P1"], tol * ref["P1"]),
            _check("nu'", nup, ref["Pt1"], tol * ref["Pt1"]))
    rnhat = ref["Pt1"].sum()
    r = max(r, _check("Nhat", nhat, rnhat, (tol + L(N * U)) * rnhat))
    live = ref["P1"] > 0
    inv = np.where(live, L(1) / np.where(live, ref["P1"], L(1)), L(0))
    rx = (ref["PX"] + ref["P1"][:, None] * L(shift)) * inv[:, None]
    S = (ref["S"] + L(abs(shift) * np.sqrt(3.0)) * ref["P1"]) * inv
    return max(r, _check("xhat", xhat, rx, (L(2) * tol + L(U)) * S[:, None]))


@pytest.mark.parametrize("case", ["expanded-B", "clamped"])
def test_bcpd_paths(ctx, monkeypatch, case):
    from gingr_b200 import api
    name = "cube" if case == "expanded-B" else "cube_far_row"
    y0, x0 = GEOMETRIES[name]()
    sigma2, s, w = BCPD_ARGS
    ref = _bcpd_ref(name, sigma2, s, w)
    t = _shift_for(y0, x0, sigma2, "expand", 0.9) if case == "expanded-B" else 0.0
    y, x = y0 + t, x0 + t
    want = ("safe", "expanded") if case == "expanded-B" else ("clamped", "clamped")
    assert _paths(y, x, sigma2, rowf=True) == want
    sig, al = _bcpd_factors(len(y))
    _env(monkeypatch, "")
    tg = api.Target(ctx, x)
    try:
        got = api.bcpd_estep(ctx, tg, y, sig, al, sigma2, s, w)
    finally:
        tg.close()
    extra = _expanded_term(y, x, sigma2) if want[1] == "expanded" else 0.0
    _check_bcpd(got, ref, _tol(ref, len(y), len(x), extra), shift=t)
    if case == "clamped":
        assert got[0][-1] == 0 and np.all(got[3][-1] == 0)


# ---------------------------------------------------------------------------------------------
# culling: splits, ragged shapes, clusters, far w = 0 columns, degenerate boxes
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("splits", ["1", "3", MAX_SPLITS])
def test_forced_splits_on_a_culled_geometry(ctx, monkeypatch, splits):
    """Three clusters 48 apart at sigma2 = 4: column block 2 (cluster 3's targets) keeps only cluster 3's 16 model
    sub-tiles, so with the largest split count most of its CTAs get empty ranges."""
    _cpd_case(ctx, monkeypatch, "clusters3_aligned", 4.0, 0.1, "1", "expanded", splits)


@pytest.mark.parametrize("name,w", [("clusters3_ragged", 0.1), ("clusters3_ragged", 0.0), ("clusters2_ragged", 0.1)])
def test_culled_clusters(ctx, monkeypatch, name, w):
    """Cluster gaps of 38 against the rule's sqrt(2 sigma2 (ln M + 60 ln 2 + 1)) = 20 (plus the within-cluster U_C
    term): cross-cluster tile pairs are culled, their K (~ e^-180) are not 0 in FP64, and dropping them must not show."""
    _cpd_case(ctx, monkeypatch, name, 4.0, w, "1", "expanded")


@pytest.mark.parametrize("mixed", [False, True], ids=["alone", "mixed-tile"])
@pytest.mark.parametrize("cull", ["0", "1"])
def test_far_target_columns_with_huge_weights(ctx, monkeypatch, mixed, cull):
    """w = 0 and a far target group: w_j ~ 1e210 for its columns, which give the nearest model points P_ij ~ 1.
    Sweep B's rule must use the tile's largest w_j: with the smallest, the mixed tile would be culled for cluster B's
    rows and those P_ij lost."""
    name = "far_mixed" if mixed else "far_alone"
    fit, tgt = GEOMETRIES[name]()
    far = np.abs(tgt[:, 0] - 30.0) < 1.0
    tiles = _kd_tiles(tgt, 1536, 64)
    kinds = {(bool(far[tl].any()), bool((~far[tl]).any())) for tl in tiles}
    assert ((True, True) in kinds) == mixed, kinds                    # a tile holds far and near columns
    assert ((True, False) in kinds) != mixed, kinds                   # far columns fill tiles of their own
    ref = _cpd_ref(name, 0.75, 0.0)
    wj = 1.0 / ref["colsum"][far].astype(float)
    assert np.all(np.isfinite(wj)) and wj.min() > 1e180
    _cpd_case(ctx, monkeypatch, name, 0.75, 0.0, cull, "safe")


@pytest.mark.parametrize("name,sigma2,path", [("planar", 2.0, "expanded"), ("collinear", 4.0, "safe"),
                                              ("repeated", 1.0, "expanded"), ("anisotropic", 16.0, "safe")])
def test_culled_degenerate_boxes(ctx, monkeypatch, name, sigma2, path):
    """Boxes of zero thickness (planar, collinear, 1000 : 1 : 1e-3) or of a single point (tiles of one repeated
    point)."""
    _cpd_case(ctx, monkeypatch, name, sigma2, 0.1, "1", path)


@pytest.mark.parametrize("name", [n for n in GEOMETRIES if n.startswith("small_")])
@pytest.mark.parametrize("splits", [None, MAX_SPLITS], ids=["planned", "max-splits"])
def test_ragged_small_shapes_culled(ctx, monkeypatch, name, splits):
    """Both dimensions one past / short of a sub-tile, target tile or column block."""
    _cpd_case(ctx, monkeypatch, name, 1.0, 0.1, "1", "expanded", splits)


# ---------------------------------------------------------------------------------------------
# registration with culling against the dense E-step
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sphere_problem(ctx):
    from gingr_b200 import api, synthetic
    M, N = 20000, 100000
    ref = synthetic.fibonacci_sphere(M)
    tv = synthetic.make_target(synthetic.fibonacci_sphere(N), 0)
    mean, basis, var = synthetic.make_gpmm(ref, 32, 1, orthonormal=False)
    model = api.Model(ctx, ref, mean, basis, var)
    tgt = api.Target(ctx, tv)
    yield model, tgt
    model.close()
    tgt.close()


def _rotation(axis, degrees):
    a = np.asarray(axis, dtype=float) / np.linalg.norm(axis)
    th = np.deg2rad(degrees)
    A = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + np.sin(th) * A + (1 - np.cos(th)) * A @ A


# Measured on an NVIDIA B200 (1000 W limit), culled against dense after 5 iterations: at most 1.5e-13 (sigma2), 5.2e-14
# (alpha), 1.0e-15 (fit / diagonal), 8.9e-16 (pose); live fractions 0.27 / 0.34 (identity) and 0.27 / 0.39 (turned).
REG_TOL = 1e-11


@pytest.mark.parametrize("turn", [0.0, 90.0], ids=["identity", "turned-90"])
def test_registration_with_culling_matches_dense(ctx, monkeypatch, sphere_problem, turn):
    """Five CPD iterations at M = 20 000, N = 100 000 with culling on (live fractions < 0.9 asserted) and off.  The
    turned start rotates the fit 90 degrees about (1, 1, 1), so its sub-tile boxes are no longer the tight boxes of
    the reference's k-d tiles."""
    from gingr_b200 import api
    model, tgt = sphere_problem
    R = _rotation((1.0, 1.0, 1.0), turn)
    out = {}
    for cull in ("1", "0"):
        _env(monkeypatch, cull)
        reg = api.CpdRegistration(ctx, model, tgt, api.CpdConfiguration(maxIterations=10 ** 6, w=0.1, initialSigma=25.0))
        try:
            reg.initializeState(globalTransformation=api.RIGID_TRANSFORMS, rotation=R)
            reg.setProfiling(True)
            reg.updateChain(5)
            ms, it = reg.getProfile()
            out[cull] = (reg.downloadState(), ms[6] / it, ms[7] / it)
        finally:
            reg.close()
    (a, la, lb), (d, da, db) = out["1"], out["0"]
    assert (da, db) == (1.0, 1.0)
    assert 0.0 < la < 0.9 and 0.0 < lb < 0.9, (la, lb)
    diag = float(np.linalg.norm(d.fit.max(0) - d.fit.min(0)))
    pa, pd = a.modelParameters, d.modelParameters
    diffs = {
        "fit": float(np.max(np.abs(a.fit - d.fit))) / diag,
        "alpha": float(np.max(np.abs(pa.shape - pd.shape))) / float(np.max(np.abs(pd.shape))),
        "sigma2": abs(a.sigma2 - d.sigma2) / d.sigma2,
        "translation": float(np.max(np.abs(pa.translation - pd.translation))) / diag,
        "euler": float(np.max(np.abs(np.subtract(pa.euler, pd.euler)))),
    }
    print(f"registration turn={turn}: live A {la:.3f} B {lb:.3f}, culled vs dense {diffs}")
    assert a.status == d.status
    assert all(v < REG_TOL for v in diffs.values()), diffs
