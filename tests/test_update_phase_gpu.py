"""The iteration's update phase (update.cu enqueue_update_phase), stage by stage, against extended-precision references.

gingr_debug_update_phase (exported, not in gingr_cuda.h) runs the posterior phase at a given state, copies the factor L
and z = L^-1 rhs out, runs the update phase as an iteration does and returns what every stage wrote: c, S c, alpha*,
alpha_c, q, alpha_new, both instances, newshape, the coefficient residual u, the Procrustes sums, the state block, the
committed alpha and the refreshed fit, and the model constants S and W0.  Every reference below is built from the
device's own input to that stage, so errors do not compound and a failure names one kernel.  References are numpy
longdouble; the 3 x 3 SVD, asin / atan2 of the Euler conversion and euler_to_matrix are mpmath at 40 digits.

Bounds, with u = 2^-53 and gamma_n = n u / (1 - n u):
  back substitution  per 64-row block k, acc_k = z'_k - sum_{i>k} L_ik^T c_i from the device's L, z' and c, and
        |L_kk^T c_k - acc_k| <= gamma_{r+2} (|L|^T |c|)_k + 64 u kappa(L_kk) (|acc_k| + (|L_kk|^T |c_k|))_max:
        the first term is the accumulation and the triangular product, the second the kernels that multiply by an
        inverted diagonal block (Z L_kk - I is of the order 64 u kappa(L_kk)).  Mx = I + D Phi^T W Phi D of these cases
        has kappa(L_kk) of a few units.
  S c, W0 (S c), W0 q   each entry a dot product of length r:  gamma_r (|A| |x|).
  W0 itself   the model's regression constant (S + 1e-5 I)^-1: ||(S + 1e-5 I) W0 x - x|| <= 4 r u kappa ||x|| for two
        probe vectors x (ranks <= 2000, where kappa is an eigenvalue ratio the host can afford).
  combine     alpha_c = alpha + (alpha* - alpha) step: two roundings, or one with either FMA contraction:
        2 u (|alpha| + |alpha* - alpha| step).
  instances   per row, Phi (sqrt(lambda) alpha): gamma_{r+1} (|Phi| |D alpha|), the staging product included.
  Procrustes  X = (ref + mean) + inst_a, Y = R ((ref + mean) + inst_b) + t with the state's R and t:
        newshape = Y to gamma_8 (|R| |b| + |t|) per point; the means to gamma_{M+8} times the mean of the same magnitudes;
        the centred sums from the device's means to gamma_{M+8} sum (|x| + |mu_x|)_a (|y| + |mu_y|)_b.
  R1, t, scale   from an mpmath Kabsch / Umeyama solve of the device's sums and means, Sxy = U diag(s) V^T,
        d = det U det V, R = U diag(1, 1, d) V^T, then the Euler round trip R1 = euler(angles(R)):
          always  tr(R1^T Sxy) >= tr(R1_ref^T Sxy) - 1e-13 sum s_i (outside the gimbal band R1_ref = R and the right side
                  is the optimum s_0 + s_1 + d s_2 over proper rotations);  R1 is orthonormal and det R1 = +1;
          where s_1 + s_2 > 1e-3 s_0 (R unique and well conditioned)  R1 entry-wise to 64 u (s_0 / (s_1 + s_2)) / cos(theta)
                  (the round trip divides by cos(theta)), t to the matching magnitudes, scale to 16 u.
  Euler       NEW_EULER = mpmath angles(R1) with the 1e-4 band on |R1_20|, to 16 u (1 + |angle|);
        R2 = mpmath euler(NEW_EULER) to 8 u.  The band is on |R_20| = |sin theta|: theta = pi/2 - delta lies inside it
        for delta < 0.01414, so the cases put theta at pi/2 - 5e-5 and pi/2 - 0.005 (inside; the second outside a 1e-6
        band) and at pi/2 - 0.03 (outside).
  u           R1^T (newshape - (R1 b + t)):  8 u |R1|^T (|newshape| + |R1| |b| + |t|).
  q           D Phi^T u:  gamma_{3M+16} D (|Phi|^T |u|) (split partial sums and their reduction included).
  commit      alpha is bit-equal to alpha_new and the pose fields to NEW_*; after a failed posterior the state is unchanged,
        status and retry counter as GingrAlgorithm.scala:193-210.
  fit         s (R2 ((ref + mean) + Phi D alpha) + t): the instance bound carried through the pose, plus 8 u of the
        magnitudes.
  sample      z' - z equals oracle.standard_normals(r, seed, iteration) to u |z'| + 16 u (|n| + 8): the device's log, sin
        and cos against host libm.

Paths (`_paths` mirrors the host's choices; every case asserts the ones it means to hit):
  back substitution   r <= 64 chol_backsolve_small_kernel; otherwise chol_backsolve_z_kernel (fresh factor) or the
                      ticket-ordered chol_backsolve_kernel (kept factor, the MH chain); r = 9600 has 150 blocks > 148 SMs
  matvec              dense_matvec_kernel below r = 512, dense_matvec2_kernel from 512 (odd r: a tail column)
  instances           gemv_rows_kernel<2>; above r = 12 800 two <1> passes
  Procrustes          ceil(M / 256) blocks summed by 32 lanes: more than 32 blocks reuse lanes
  gemvT               rows 3M split in rows_per_cta (a multiple of 4, 16..512): many splits, a ragged last one
"""
import ctypes
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

L = np.longdouble
U = 2.0 ** -53
DS = dict(SCALE=0, T=1, EULER=4, SIGMA2=10, STEP=11, R=12, NEW_SCALE=24, NEW_T=25, NEW_EULER=28, R1=31, R2=40,
          NEW_SIGMA2=50, MUX=56, MUY=59, COUNT=80)
IS = dict(GT=0, ITER=1, STATUS=2, RETRY=6, COUNT=16)
SIMILARITY, RIGID, NO_T = 0, 1, 2   # GINGR_*_TRANSFORMS


def _need_longdouble():
    if np.finfo(np.longdouble).eps >= np.finfo(np.float64).eps:
        pytest.skip("no extended precision on this platform")


def _gamma(n):
    return n * U / (1.0 - n * U)


@functools.lru_cache(maxsize=None)
def _num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------------------------------------
# host mirror of the path choices (chol.cu chol_backsolve_enqueue, vecops.cu)
# ---------------------------------------------------------------------------------------------
def _gemvT_rows_per_cta(rows, sms):
    want = -(-max(rows, 1) // (2 * sms))
    return max(16, min(512, (want + 3) // 4 * 4))


def _paths(M, r, kept_factor=0, sms=None):
    sms = sms or _num_sms()
    nb = -(-r // 64)
    rows = 3 * M
    rpc = _gemvT_rows_per_cta(rows, sms)
    splits = max(1, -(-rows // rpc))
    pblocks = -(-max(M, 1) // 256)
    return dict(backsolve="small" if nb == 1 else ("ticket" if kept_factor else "z"), blocks_over_sms=nb > sms,
                matvec2=r >= 512, odd_tail=r >= 512 and r % 2 == 1, split_instances=2 * r * 8 > 200 * 1024,
                pad=r % 8 != 0, pro_blocks=pblocks, lanes_reused=pblocks > 32, gt_splits=splits,
                gt_last_ragged=(rows - (splits - 1) * rpc) % 4 != 0)


# ---------------------------------------------------------------------------------------------
# the hook
# ---------------------------------------------------------------------------------------------
def _hook(ctx):
    from gingr_b200 import _native as nat
    f = ctx._lib.gingr_debug_update_phase
    ip = ctypes.POINTER(ctypes.c_int32)
    f.argtypes = ([ctypes.c_void_p, ctypes.POINTER(nat.GingrState), nat.dp, ctypes.c_int32, ctypes.c_uint64, ctypes.c_int32]
                  + [nat.dp] * 10 + [ip, nat.dp, nat.dp, nat.dp, nat.dp])
    f.restype = ctypes.c_int32
    return f


def _run(reg, state, probabilistic=0, seed=0, kept_factor=0):
    from gingr_b200 import _native as nat
    r, M = reg.model.rank, reg.model.M
    pod, alpha = state.to_pod()
    o = dict(L=np.full((r, r), np.nan), z=np.full(r, np.nan), z2=np.full(r, np.nan), vec=np.full((6, r), np.nan),
             inst_a=np.full(3 * M, np.nan), inst_b=np.full(3 * M, np.nan), newshape=np.full(3 * M, np.nan),
             u=np.full(3 * M, np.nan), pro_sums=np.full(10, np.nan), ds=np.full(DS["COUNT"], np.nan),
             is_=np.zeros(IS["COUNT"], dtype=np.int32), alpha=np.full(r, np.nan), fit=np.full(3 * M, np.nan),
             S=np.full((r, r), np.nan), W0=np.full((r, r), np.nan))
    d = nat.as_dp
    code = reg.ctx.check(_hook(reg.ctx)(reg.handle, ctypes.byref(pod), d(alpha), int(probabilistic), int(seed), int(kept_factor),
                                        d(o["L"]), d(o["z"]), d(o["z2"]), d(o["vec"]), d(o["inst_a"]), d(o["inst_b"]),
                                        d(o["newshape"]), d(o["u"]), d(o["pro_sums"]), d(o["ds"]),
                                        o["is_"].ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), d(o["alpha"]), d(o["fit"]),
                                        d(o["S"]), d(o["W0"])))
    assert code == 0
    o["L"] = np.tril(o["L"])
    return o


def _check(what, got, ref, lim):
    """|got - ref| <= lim entry by entry in longdouble."""
    got = np.asarray(got, dtype=float).astype(L)
    ref = np.asarray(ref).astype(L)
    lim = np.broadcast_to(np.asarray(lim).astype(L), ref.shape)
    err = np.abs(got - ref)
    bad = ~(err <= lim)
    assert not bad.any(), (f"{what}: {int(bad.sum())} of {bad.size} entries out of bound, first at "
                           f"{np.argwhere(bad)[0].tolist()}: {float(got[tuple(np.argwhere(bad)[0])])!r} vs "
                           f"{float(ref[tuple(np.argwhere(bad)[0])])!r}, worst err/bound "
                           f"{float(np.max(err / np.where(lim > 0, lim, L(1)))):.3g}")


def _exact(what, got, ref):
    got, ref = np.asarray(got), np.asarray(ref)
    bad = ~(got == ref)
    assert not bad.any(), f"{what}: {int(bad.sum())} of {bad.size} entries differ, first at {np.argwhere(bad)[0].tolist()}"


def _ldot(A, x, chunk=2048):
    """A x in longdouble, A float64 [n, k] converted by row chunks."""
    x = np.asarray(x).astype(L)
    return np.concatenate([A[i:i + chunk].astype(L) @ x for i in range(0, A.shape[0], chunk)])


def _ldotT(A, x, chunk=2048):
    """A^T x in longdouble."""
    x = np.asarray(x).astype(L)
    out = np.zeros(A.shape[1], dtype=L)
    for i in range(0, A.shape[0], chunk):
        out += A[i:i + chunk].astype(L).T @ x[i:i + chunk]
    return out


# ---------------------------------------------------------------------------------------------
# problems
# ---------------------------------------------------------------------------------------------
def _shape(kind, M, rng):
    if kind == "shell":
        p = rng.normal(size=(M, 3))
        return p / np.linalg.norm(p, axis=1, keepdims=True) * rng.uniform(0.8, 1.2, (M, 1)) * np.array([1.0, 0.8, 0.6])
    if kind == "flat":   # a patch in z = 0, longer along y than along x
        return np.column_stack([rng.uniform(-0.5, 0.5, M), rng.uniform(-1.2, 1.2, M), np.zeros(M)])
    if kind == "line":   # on the x axis
        return np.column_stack([rng.uniform(-1.0, 1.0, M), np.zeros(M), np.zeros(M)])
    if kind == "cap":    # the shell lifted to z >= 0.3: no mirror symmetry in z
        p = _shape("shell", M, rng)
        p[:, 2] = np.abs(p[:, 2]) + 0.3
        return p
    if kind == "octahedron":
        return np.vstack([np.eye(3), -np.eye(3)])
    raise ValueError(kind)


@functools.lru_cache(maxsize=4)
def _model_data(kind, M, r, seed, zero_mean=False, zero_z=False, mirror_mode=False):
    """ref [M, 3], mean [3M], basis [3M, r] with unit columns, variances 0.3 / (1 + k / 50) (sqrt(lambda) not a power of 2)."""
    rng = np.random.default_rng(seed)
    ref = _shape(kind, M, rng)
    mean = np.zeros(3 * M) if zero_mean else 0.02 * rng.normal(size=3 * M)
    phi = rng.standard_normal((3 * M, r))
    if zero_z:
        phi[2::3] = 0.0
    if mirror_mode:   # mode 0 moves every point along z by its own z: alpha_0 ~ -2 / sqrt(lambda_0) mirrors the shape
        phi[:, 0] = 0.0
        phi[2::3, 0] = ref[:, 2]
    phi /= np.linalg.norm(phi, axis=0, keepdims=True)
    var = 0.3 / (1.0 + np.arange(r) / 50.0)
    return ref, mean, phi, var


class _Case:
    """A registration of one model (closed by the caller)."""

    def __init__(self, ctx, kind, M, r, seed=0, algo="icp", zero_mean=False, zero_z=False, mirror=False, pose=None,
                 sigma2=0.5, target_alpha=None):
        from gingr_b200 import api
        from gingr_b200.rotation import euler_to_matrix
        self.ref, self.mean, self.phi, self.var = _model_data(kind, M, r, seed, zero_mean, zero_z, mirror)
        self.M, self.r, self.sigma2 = M, r, sigma2
        rng = np.random.default_rng(seed + 1)
        pose = pose or dict(euler=(0.3, -0.2, 0.45), translation=(0.15, -0.1, 0.2))
        R = np.asarray(euler_to_matrix(*pose["euler"]), dtype=float)
        b = self.ref + self.mean.reshape(-1, 3)
        if mirror:
            tgt = b * np.array([1.0, 1.0, -1.0])
        else:
            a = 0.3 * rng.normal(size=r) if target_alpha is None else target_alpha
            tgt = b + (self.phi @ (np.sqrt(self.var) * a)).reshape(-1, 3)
        tgt = tgt @ R.T + np.asarray(pose["translation"]) + 0.003 * rng.normal(size=tgt.shape)
        self.model = api.Model(ctx, self.ref, self.mean, self.phi, self.var)
        self.target = api.Target(ctx, tgt)
        if algo == "cpd":
            cfg = api.CpdConfiguration(initialSigma=sigma2, w=0.1)
            self.reg = api.CpdRegistration(ctx, self.model, self.target, cfg)
        else:
            cfg = api.IcpConfiguration(initialSigma=sigma2, endSigma=sigma2 / 2, correspondenceMethod=api.POINTCLOUD_CLOSEST_POINT)
            self.reg = api.IcpRegistration(ctx, self.model, self.target, cfg)
        self.ctx = ctx

    def state(self, euler=(0.3, -0.2, 0.45), translation=(0.15, -0.1, 0.2), alpha=None, scale=1.0, gt=RIGID, step=1.0,
              iteration=1, sigma2=None):
        from gingr_b200 import api
        a = np.zeros(self.r) if alpha is None else np.asarray(alpha, dtype=float)
        pars = api.ModelFittingParameters(scale, np.asarray(translation, dtype=float), tuple(euler), a)
        return api.GeneralRegistrationState(pars, np.zeros((self.M, 3)), sigma2=self.sigma2 if sigma2 is None else sigma2,
                                            globalTransformation=gt, stepLength=step, iteration=iteration)

    def close(self):
        for h in (self.reg, self.target, self.model):
            h.close()


# ---------------------------------------------------------------------------------------------
# mpmath rotations
# ---------------------------------------------------------------------------------------------
def _mp():
    import mpmath
    mpmath.mp.dps = 40
    return mpmath


def _mp_euler_to_matrix(e):
    mp = _mp()
    phi, theta, psi = (mp.mpf(float(v)) for v in e)
    cph, sph, cth, sth, cps, sps = mp.cos(phi), mp.sin(phi), mp.cos(theta), mp.sin(theta), mp.cos(psi), mp.sin(psi)
    return mp.matrix([[cth * cph, sps * sth * cph - cps * sph, sps * sph + cps * sth * cph],
                      [cth * sph, cps * cph + sps * sth * sph, cps * sth * sph - sps * cph],
                      [-sth, sps * cth, cps * cth]])


def _mp_matrix_to_euler(R):
    """update.cu matrix_to_euler_dev (RotationSpace3D.rotMatrixToEulerAngles), band 1e-4 on |R_20|."""
    mp = _mp()
    if abs(abs(R[2, 0]) - 1) > mp.mpf("0.0001"):
        theta = mp.asin(-R[2, 0])
        ct = mp.cos(theta)
        return [mp.atan2(R[1, 0] / ct, R[0, 0] / ct), theta, mp.atan2(R[2, 1] / ct, R[2, 2] / ct)]
    if abs(R[2, 0] + 1) < mp.mpf("0.0001"):
        return [mp.mpf(0), mp.pi / 2, mp.atan2(R[0, 1], R[0, 2])]
    return [mp.mpf(0), -mp.pi / 2, mp.atan2(-R[0, 1], -R[0, 2])]


def _to_mp(a):
    mp = _mp()
    return mp.matrix([[mp.mpf(float(v)) for v in row] for row in np.asarray(a, dtype=float).reshape(3, 3)])


def _np(m):
    return np.array([[float(m[i, j]) for j in range(m.cols)] for i in range(m.rows)])


def _kabsch(Sxy):
    """(R, s, d): R = U diag(1, 1, d) V^T with d = det U det V, the proper rotation maximising tr(R^T Sxy)."""
    mp = _mp()
    A = _to_mp(Sxy)
    Um, s, Vt = mp.svd_r(A)
    d = 1 if mp.det(Um) * mp.det(Vt) > 0 else -1
    R = Um * mp.diag([1, 1, d]) * Vt
    return R, [s[0], s[1], s[2]], d


# ---------------------------------------------------------------------------------------------
# the stage checks
# ---------------------------------------------------------------------------------------------
def _check_backsolve(o):
    Lf, c = o["L"], o["vec"][0]
    z2 = o["z2"]
    r = len(c)
    absLc = np.abs(Lf).T @ np.abs(c)
    cl = c.astype(L)
    for k0 in range(0, r, 64):
        k1 = min(r, k0 + 64)
        Lkk = Lf[k0:k1, k0:k1]
        acc = z2[k0:k1].astype(L)
        if k1 < r:
            acc = acc - Lf[k1:, k0:k1].astype(L).T @ cl[k1:]
        res = Lkk.astype(L).T @ cl[k0:k1] - acc
        Z = np.linalg.inv(Lkk)
        kappa = float(np.linalg.norm(Lkk, np.inf) * np.linalg.norm(Z, np.inf))
        mag = float(np.max(np.abs(acc.astype(float)) + np.abs(Lkk).T @ np.abs(c[k0:k1])))
        lim = _gamma(r + 2) * absLc[k0:k1] + 64.0 * U * kappa * mag
        _check(f"back substitution block {k0 // 64}", res, np.zeros(k1 - k0), lim)


def _check_matvec(what, A, x, y):
    ref = _ldot(A, x)
    _check(what, y, ref, _gamma(len(x)) * (np.abs(A) @ np.abs(x)))


def _check_w0(S, W0, seed=0):
    r = S.shape[0]
    B = S + 1e-5 * np.eye(r)
    ev = np.linalg.eigvalsh(B)
    kappa = float(ev[-1] / ev[0])
    rng = np.random.default_rng(seed)
    for _ in range(2):
        x = rng.normal(size=r)
        y = _ldot(W0, x)
        res = _ldot(B, y.astype(float)) + _ldot(B, (y - y.astype(float).astype(L)).astype(float)) - x.astype(L)
        nrm = float(np.sqrt(np.sum(res.astype(float) ** 2)))
        assert nrm <= 4.0 * r * U * kappa * float(np.linalg.norm(x)), (nrm, kappa)


def _check_stages(case, st, o, probabilistic=False, seed=0):
    """Every stage from the device's own input to it; returns (Sxy, s, d, R) of the Procrustes solve (R before the
    Euler round trip, mpmath)."""
    _need_longdouble()
    r, M = case.r, case.M
    phi, sl = case.phi, np.sqrt(case.var)
    ds, is_ = o["ds"], o["is_"]
    c, Sc, astar, ac, q, anew = o["vec"]
    alpha = np.asarray(st.modelParameters.shape, dtype=float)
    # sample, back substitution, regression products
    if probabilistic:
        from oracle import oracle
        n = oracle.standard_normals(r, seed, st.iteration)
        _check("posterior sample", o["z2"].astype(L) - o["z"].astype(L), n, U * np.abs(o["z2"]) + 16.0 * U * (np.abs(n) + 8.0))
    else:
        _exact("z without a sample", o["z2"], o["z"])
    _check_backsolve(o)
    _check_matvec("S c", o["S"], c, Sc)
    _check_matvec("alpha* = W0 (S c)", o["W0"], Sc, astar)
    step = float(ds[DS["STEP"]])
    _check("combine", ac, alpha.astype(L) + (astar.astype(L) - alpha.astype(L)) * L(step),
           2.0 * U * (np.abs(alpha) + np.abs(astar - alpha) * abs(step)))
    # instances
    for name, v, inst in (("instance(alpha)", alpha, o["inst_a"]), ("instance(alpha_c)", ac, o["inst_b"])):
        _check(name, inst, _ldot(phi, sl * v), _gamma(r + 1) * (np.abs(phi) @ np.abs(sl * v)))
    # Procrustes sums, from the device's instances and the state pose
    b = (case.ref.reshape(-1) + case.mean).reshape(-1, 3)
    bl = case.ref.reshape(-1, 3).astype(L) + case.mean.reshape(-1, 3).astype(L)
    # the state's pose: DS_R is left as the posterior phase set it, DS_T holds the committed translation by now
    R, t = ds[DS["R"]:DS["R"] + 9].reshape(3, 3), np.asarray(st.modelParameters.translation, dtype=float)
    X = bl + o["inst_a"].reshape(-1, 3).astype(L)
    Bb = bl + o["inst_b"].reshape(-1, 3).astype(L)
    Y = Bb @ R.T.astype(L) + t.astype(L)
    magX = np.abs(b) + np.abs(o["inst_a"].reshape(-1, 3))
    magY = (np.abs(b) + np.abs(o["inst_b"].reshape(-1, 3))) @ np.abs(R).T + np.abs(t)
    _check("newshape", o["newshape"].reshape(-1, 3), Y, _gamma(8) * magY)
    mux, muy = ds[DS["MUX"]:DS["MUX"] + 3], ds[DS["MUY"]:DS["MUY"] + 3]
    _check("mean of X", mux, X.mean(0), _gamma(M + 8) * magX.mean(0))
    _check("mean of Y", muy, Y.mean(0), _gamma(M + 8) * magY.mean(0))
    xc, yc = X - mux.astype(L), Y - muy.astype(L)
    ax, ay = magX + np.abs(mux), magY + np.abs(muy)
    sums = o["pro_sums"]
    _check("sum |x - mux|^2", sums[0], np.sum(xc * xc), _gamma(M + 8) * np.sum(ax * ax))
    _check("Sxy sums", sums[1:10].reshape(3, 3), yc.T @ xc, _gamma(M + 8) * (ay.T @ ax))
    # the solve, from the device's sums and means
    mp = _mp()
    gt = int(is_[IS["GT"]])
    R1 = ds[DS["R1"]:DS["R1"] + 9].reshape(3, 3)
    t1, c1 = ds[DS["NEW_T"]:DS["NEW_T"] + 3], float(ds[DS["NEW_SCALE"]])
    Sxy = sums[1:10].reshape(3, 3) / M
    Rk, s, d = _kabsch(Sxy)
    if gt == NO_T:
        _exact("R1 without transforms", R1, np.eye(3))
        _exact("t without transforms", t1, np.zeros(3))
        assert c1 == 1.0
    else:
        R1_ref = _mp_euler_to_matrix([float(v) for v in _mp_matrix_to_euler(Rk)])
        ssum = float(s[0] + s[1] + s[2])
        got = float(mp.fsum(_to_mp(R1)[i, j] * _to_mp(Sxy)[i, j] for i in range(3) for j in range(3)))
        want = float(mp.fsum(R1_ref[i, j] * _to_mp(Sxy)[i, j] for i in range(3) for j in range(3)))
        assert got >= want - 1e-13 * ssum, f"tr(R1^T Sxy) = {got!r} short of {want!r} (s = {[float(v) for v in s]}, d = {d})"
        _check("R1^T R1", R1.T.astype(L) @ R1.astype(L), np.eye(3), 8.0 * U)
        assert abs(float(np.linalg.det(R1)) - 1.0) < 1e-14
        scale_ref = (s[0] + s[1] + d * s[2]) / (mp.mpf(float(sums[0])) / M) if gt == SIMILARITY else mp.mpf(1)
        if gt == RIGID:
            assert c1 == 1.0
        else:
            assert abs(c1 - float(scale_ref)) <= 16.0 * U * abs(float(scale_ref)) * ssum / float(s[0] + s[1] + d * s[2])
        if float(s[1] + s[2]) > 1e-3 * float(s[0]):
            ct = max(abs(float(mp.cos(mp.asin(-Rk[2, 0])))), 1e-3)
            dR = 64.0 * U * float(s[0] / (s[1] + s[2])) / ct
            _check("R1", R1, _np(R1_ref), dR + 8.0 * U)
            Rn = _np(Rk)
            t_ref = [mp.mpf(float(muy[i])) - scale_ref * mp.fsum(Rk[i, j] * mp.mpf(float(mux[j])) for j in range(3)) for i in range(3)]
            lim = (np.abs(muy) + c1 * (np.abs(Rn) @ np.abs(mux))) * 8.0 * U + c1 * (dR * ct + 16.0 * U) * np.abs(mux).sum()
            _check("t", t1, np.array([L(str(v)) for v in t_ref]), lim)
    # Euler round trips from the device's R1 and NEW_EULER
    e2 = ds[DS["NEW_EULER"]:DS["NEW_EULER"] + 3]
    e_ref = _mp_matrix_to_euler(_to_mp(R1))
    _check("NEW_EULER", e2, np.array([L(str(v)) for v in e_ref]), 16.0 * U * (1.0 + np.abs(e2)))
    # coefficient residual and q
    u = o["u"].reshape(-1, 3)
    ns = o["newshape"].reshape(-1, 3)
    res = ns.astype(L) - (bl @ R1.T.astype(L) + t1.astype(L))
    mag = np.abs(ns) + np.abs(b) @ np.abs(R1).T + np.abs(t1)
    _check("coefficient residual u", u, res @ R1.astype(L), 8.0 * U * (mag @ np.abs(R1)))
    _check("q = D Phi^T u", q, sl.astype(L) * _ldotT(phi, o["u"]), _gamma(3 * M + 16) * sl * (np.abs(phi).T @ np.abs(o["u"])))
    _check_matvec("alpha_new = W0 q", o["W0"], q, anew)
    return Sxy, s, d, Rk


def _check_commit_and_fit(case, st, o):
    ds, is_ = o["ds"], o["is_"]
    _exact("committed alpha", o["alpha"], o["vec"][5])
    assert ds[DS["SCALE"]] == ds[DS["NEW_SCALE"]]
    _exact("committed t", ds[DS["T"]:DS["T"] + 3], ds[DS["NEW_T"]:DS["NEW_T"] + 3])
    _exact("committed Euler angles", ds[DS["EULER"]:DS["EULER"] + 3], ds[DS["NEW_EULER"]:DS["NEW_EULER"] + 3])
    assert ds[DS["SIGMA2"]] == ds[DS["NEW_SIGMA2"]]
    assert is_[IS["STATUS"]] == st.status and is_[IS["RETRY"]] == 10
    R2 = ds[DS["R2"]:DS["R2"] + 9].reshape(3, 3)
    _check("R2", R2, _np(_mp_euler_to_matrix(ds[DS["EULER"]:DS["EULER"] + 3])).astype(L), 8.0 * U)
    _check_fit(case, o, R2, ds[DS["T"]:DS["T"] + 3], float(ds[DS["SCALE"]]))


def _check_fit(case, o, R2, t, s):
    sl = np.sqrt(case.var)
    v = sl * o["alpha"]
    inst = _ldot(case.phi, v).reshape(-1, 3)
    ib = (_gamma(case.r + 1) * (np.abs(case.phi) @ np.abs(v))).reshape(-1, 3)
    b = case.ref + case.mean.reshape(-1, 3)
    x = case.ref.astype(L) + case.mean.reshape(-1, 3).astype(L) + inst
    ref = (x @ R2.T.astype(L) + t.astype(L)) * L(s)
    mag = (np.abs(b) + np.abs(inst.astype(float))) @ np.abs(R2).T + np.abs(t)
    _check("fit", o["fit"].reshape(-1, 3), ref, abs(s) * (ib @ np.abs(R2).T + 8.0 * U * mag))


def _check_production(case, st, o, probabilistic=False, seed=0):
    """The hook's committed state and fit are those of gingr_update from the same input, bit for bit."""
    out = case.reg.update(st, probabilistic, seed)
    ds = o["ds"]
    _exact("alpha vs gingr_update", out.modelParameters.shape, o["alpha"])
    _exact("fit vs gingr_update", out.fit.reshape(-1), o["fit"])
    _exact("t vs gingr_update", np.asarray(out.modelParameters.translation), ds[DS["T"]:DS["T"] + 3])
    _exact("Euler angles vs gingr_update", np.asarray(out.modelParameters.euler), ds[DS["EULER"]:DS["EULER"] + 3])
    assert out.modelParameters.scale == ds[DS["SCALE"]] and out.sigma2 == ds[DS["SIGMA2"]]


def _full(case, st, probabilistic=0, seed=0, kept_factor=0, production=True, w0=None):
    o = _run(case.reg, st, probabilistic, seed, kept_factor)
    out = _check_stages(case, st, o, bool(probabilistic), seed)
    _check_commit_and_fit(case, st, o)
    if w0 if w0 is not None else case.r <= 2000:
        _check_w0(o["S"], o["W0"])
    if production and not kept_factor:
        _check_production(case, st, o, bool(probabilistic), seed)
    return o, out


# ---------------------------------------------------------------------------------------------
# ranks and rows
# ---------------------------------------------------------------------------------------------
RANKS = [(1, 40, 0), (7, 20, 0), (64, 255, 0), (65, 256, 0), (65, 256, 1), (127, 257, 1), (511, 300, 0), (512, 400, 1),
         (513, 8449, 0), (2000, 700, 0), (2000, 700, 1)]


@pytest.mark.parametrize("r,M,kept", RANKS, ids=[f"r{r}-M{M}-kept{k}" for r, M, k in RANKS])
def test_update_phase_by_rank(ctx, r, M, kept):
    p = _paths(M, r, kept)
    assert p["backsolve"] == ("small" if r <= 64 else ("ticket" if kept else "z"))
    assert p["matvec2"] == (r >= 512) and p["odd_tail"] == (r == 513)
    case = _Case(ctx, "shell", M, r, seed=r + M)
    try:
        rng = np.random.default_rng(r)
        st = case.state(alpha=0.4 * rng.normal(size=r), step=0.5 if r % 2 else 1.0)
        _full(case, st, kept_factor=kept)
    finally:
        case.close()


def test_rank_and_row_cases_cover_every_path():
    sms = 148
    kinds = [_paths(M, r, k, sms) for r, M, k in RANKS]
    assert {k["backsolve"] for k in kinds} == {"small", "z", "ticket"}
    assert any(k["odd_tail"] for k in kinds) and any(k["matvec2"] and not k["odd_tail"] for k in kinds)
    assert any(r % 8 == 1 for r, _, _ in RANKS) and any(r % 8 == 7 for r, _, _ in RANKS)
    assert any(M < 32 for _, M, _ in RANKS) and {255, 256, 257} <= {M for _, M, _ in RANKS}
    assert any(k["lanes_reused"] and k["pro_blocks"] % 32 for k in kinds)
    assert any(k["gt_splits"] > 16 and k["gt_last_ragged"] for k in kinds)
    big = [_paths(M_9600, 9600, k, sms) for k in (0, 1)] + [_paths(M_12801, 12801, 0, sms)]
    assert all(k["blocks_over_sms"] for k in big[:2]) and big[2]["split_instances"]
    assert not _paths(400, 12800, 0, sms)["split_instances"]


M_9600, M_12801 = 3300, 4400


@pytest.mark.parametrize("kept", [0, 1])
def test_update_phase_rank_9600(ctx, kept):
    """150 blocks of 64 rows on 148 SMs, for the workspace and the ticket-ordered back substitution."""
    assert _paths(M_9600, 9600, kept)["blocks_over_sms"]
    case = _Case(ctx, "shell", M_9600, 9600, seed=96)
    try:
        st = case.state(alpha=0.3 * np.random.default_rng(96).normal(size=9600))
        _full(case, st, kept_factor=kept, production=kept == 0)
    finally:
        case.close()


def test_update_phase_rank_12801(ctx):
    """Two one-vector instance passes (2 r doubles exceed the shared memory of the two-vector pass)."""
    assert _paths(M_12801, 12801)["split_instances"]
    case = _Case(ctx, "shell", M_12801, 12801, seed=128)
    try:
        st = case.state(alpha=0.3 * np.random.default_rng(128).normal(size=12801), step=0.5)
        _full(case, st)
    finally:
        case.close()


# ---------------------------------------------------------------------------------------------
# poses and transformations
# ---------------------------------------------------------------------------------------------
H = np.pi / 2
POSES = {
    "general": dict(euler=(0.3, -0.2, 0.45), translation=(0.15, -0.1, 0.2)),
    "gimbal-deep+": dict(euler=(0.4, H - 5e-5, -0.3), translation=(0.1, 0.0, -0.1)),
    "gimbal-deep-": dict(euler=(-0.2, -(H - 5e-5), 0.6), translation=(0.1, 0.0, -0.1)),
    "gimbal-band+": dict(euler=(0.4, H - 0.005, -0.3), translation=(0.1, 0.0, -0.1)),
    "gimbal-band-": dict(euler=(-0.2, -(H - 0.005), 0.6), translation=(0.1, 0.0, -0.1)),
    "gimbal-out+": dict(euler=(0.4, H - 0.03, -0.3), translation=(0.1, 0.0, -0.1)),
    "gimbal-out-": dict(euler=(-0.2, -(H - 0.03), 0.6), translation=(0.1, 0.0, -0.1)),
    "half-turn": dict(euler=(np.pi, 0.0, 0.0), translation=(0.0, 0.2, 0.0)),
    "far": dict(euler=(0.7, 0.5, -1.1), translation=(1e4, -6e3, 8e3)),
}


@pytest.mark.parametrize("gt", [RIGID, SIMILARITY, NO_T], ids=["rigid", "similarity", "none"])
@pytest.mark.parametrize("pose", list(POSES))
def test_update_phase_poses(ctx, pose, gt):
    """Step 0 keeps alpha_c = alpha, so the Procrustes rotation is the state's own (theta where the case puts it); the
    similarity cases start from scale 1.7."""
    pz = POSES[pose]
    r, M = 40, 300
    case = _Case(ctx, "shell", M, r, seed=7, pose=pz)
    try:
        rng = np.random.default_rng(11)
        st = case.state(alpha=0.3 * rng.normal(size=r), step=0.0 if pose.startswith("gimbal") else 0.5,
                        scale=1.7 if gt == SIMILARITY else 1.0, gt=gt, **pz)
        o, (Sxy, s, d, Rk) = _full(case, st)
        if gt != NO_T and pose.startswith("gimbal"):
            band = abs(abs(float(Rk[2, 0])) - 1.0)
            assert (band < 1e-6) == ("deep" in pose) and (band < 1e-4) == ("out" not in pose), band
    finally:
        case.close()


def test_combine_with_steps(ctx):
    """Step lengths 1, 0.5 and 0.3 from alpha != 0."""
    r, M = 90, 400
    case = _Case(ctx, "shell", M, r, seed=3)
    try:
        a = 0.5 * np.random.default_rng(3).normal(size=r)
        for step in (1.0, 0.5, 0.3):
            _full(case, case.state(alpha=a, step=step))
    finally:
        case.close()


# ---------------------------------------------------------------------------------------------
# shapes
# ---------------------------------------------------------------------------------------------
FLAT_POSES = [dict(euler=(0.4, -0.3, 0.7), translation=(0.2, -0.1, 0.3)),
              dict(euler=(-1.1, 0.6, 2.0), translation=(-0.3, 0.5, 0.1))]


@pytest.mark.parametrize("k", [0, 1])
@pytest.mark.parametrize("gt", [RIGID, SIMILARITY], ids=["rigid", "similarity"])
@pytest.mark.parametrize("algo", ["cpd", "icp"])
def test_flat_patch_at_alpha_zero(ctx, algo, gt, k):
    """A flat reference with mean 0 at alpha = 0: X is exactly planar, Sxy has a zero column and det Sxy = +-0.  The
    rotation must still be the proper one that maximises tr(R^T Sxy)."""
    pz = FLAT_POSES[k]
    r, M = 30, 400
    case = _Case(ctx, "flat", M, r, seed=20 + k, algo=algo, zero_mean=True, pose=pz, sigma2=0.05 if algo == "cpd" else 0.5)
    try:
        st = case.state(gt=gt, **pz)
        o, (Sxy, s, d, _) = _full(case, st)
        assert np.all(Sxy[:, 2] == 0.0) and float(s[2]) == 0.0
    finally:
        case.close()


def test_model_with_zero_z_rows(ctx):
    """Basis rows of z all zero on a flat reference: X is planar at every alpha."""
    r, M = 50, 500
    pz = FLAT_POSES[0]
    case = _Case(ctx, "flat", M, r, seed=31, zero_mean=True, zero_z=True, pose=pz)
    try:
        st = case.state(alpha=0.5 * np.random.default_rng(31).normal(size=r), **pz)
        o, (Sxy, s, d, _) = _full(case, st)
        assert np.all(Sxy[:, 2] == 0.0)
        o2 = _run(case.reg, case.state(alpha=o["alpha"], gt=SIMILARITY, **pz))
        _check_stages(case, case.state(alpha=o["alpha"], gt=SIMILARITY, **pz), o2)
    finally:
        case.close()


def test_octahedron(ctx):
    """Six vertices of an octahedron: equal singular values."""
    r, M = 5, 6
    case = _Case(ctx, "octahedron", M, r, seed=41, zero_mean=True, target_alpha=np.zeros(5))
    try:
        _full(case, case.state(step=0.0))
        _full(case, case.state(step=0.0, gt=SIMILARITY, scale=1.3))
    finally:
        case.close()


def test_mirrored_target(ctx):
    """The target is the shape mirrored in z and the model can follow it (mode 0 moves every point along z by its own z,
    observations weigh 100): newshape is nearly the mirror image of X, det Sxy < 0 and d = -1."""
    r, M = 20, 300
    case = _Case(ctx, "cap", M, r, seed=51, zero_mean=True, mirror=True, pose=dict(euler=(0.0, 0.0, 0.0), translation=(0.0, 0.0, 0.0)),
                 sigma2=0.01)
    try:
        o, (Sxy, s, d, _) = _full(case, case.state(euler=(0.0, 0.0, 0.0), translation=(0.0, 0.0, 0.0)))
        assert np.linalg.det(Sxy) < 0 and d == -1
    finally:
        case.close()


@pytest.mark.parametrize("gt", [RIGID, SIMILARITY], ids=["rigid", "similarity"])
def test_collinear_shape(ctx, gt):
    """Points on a line: Sxy has rank 1 and the rotation is not unique; it must reach the optimum all the same."""
    r, M = 12, 200
    pz = FLAT_POSES[1]
    case = _Case(ctx, "line", M, r, seed=61, zero_mean=True, pose=pz)
    try:
        o, (Sxy, s, d, _) = _full(case, case.state(gt=gt, **pz))
        assert np.all(Sxy[:, 1:] == 0.0)
    finally:
        case.close()


# ---------------------------------------------------------------------------------------------
# modes and failures
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("r,M,kept", [(40, 300, 0), (200, 500, 0), (200, 500, 1), (513, 600, 1)],
                         ids=["r40", "r200", "r200-kept", "r513-kept"])
def test_probabilistic(ctx, r, M, kept):
    case = _Case(ctx, "shell", M, r, seed=71 + r)
    try:
        st = case.state(alpha=0.2 * np.random.default_rng(r).normal(size=r), iteration=3)
        _full(case, st, probabilistic=1, seed=0x1234567890ABCDEF, kept_factor=kept)
    finally:
        case.close()


@pytest.mark.parametrize("probabilistic", [0, 1])
def test_failed_posterior_keeps_the_state(ctx, probabilistic):
    """CPD at a non-finite sigma2 fails its posterior: alpha, pose and sigma2 stay, the deterministic update reports
    ModelFlexibilityError and the probabilistic one spends a retry (GingrAlgorithm.scala:193-208)."""
    from gingr_b200 import api
    r, M = 30, 200
    case = _Case(ctx, "shell", M, r, seed=81, algo="cpd", sigma2=0.05)
    try:
        a = 0.3 * np.random.default_rng(81).normal(size=r)
        st = case.state(alpha=a, iteration=2, sigma2=float("nan"))
        o = _run(case.reg, st, probabilistic)
        ds, is_ = o["ds"], o["is_"]
        _exact("alpha after a failed posterior", o["alpha"], a)
        _exact("t after a failed posterior", ds[DS["T"]:DS["T"] + 3], np.asarray(st.modelParameters.translation))
        _exact("Euler angles after a failed posterior", ds[DS["EULER"]:DS["EULER"] + 3], np.asarray(st.modelParameters.euler))
        assert ds[DS["SCALE"]] == 1.0 and np.isnan(ds[DS["SIGMA2"]])
        if probabilistic:
            assert is_[IS["STATUS"]] == st.status and is_[IS["RETRY"]] == 9
        else:
            assert is_[IS["STATUS"]] == api.STATUS_MODEL_FLEXIBILITY_ERROR and is_[IS["RETRY"]] == 10
    finally:
        case.close()


def test_hook_leaves_updates_unchanged(ctx):
    """Updates after hook calls are bit-identical to those of a registration that never made them, with the same launch
    count."""
    from gingr_b200 import api
    case = _Case(ctx, "shell", 300, 100, seed=91)
    other = api.IcpRegistration(ctx, case.model, case.target, case.reg.config)
    try:
        st = case.state(alpha=0.2 * np.random.default_rng(91).normal(size=100))
        outs = []
        for reg, calls in ((case.reg, (0, 1)), (other, ())):
            for kept in calls:
                _run(reg, st, 0, 0, kept)
            l0 = ctx.launch_count
            s1 = reg.update(st)
            s2 = reg.update(s1)
            outs.append((s1, s2, ctx.launch_count - l0))
        (a1, a2, la), (b1, b2, lb) = outs
        assert la == lb
        for x, y in ((a1, b1), (a2, b2)):
            _exact("fit", x.fit, y.fit)
            _exact("alpha", x.modelParameters.shape, y.modelParameters.shape)
            assert x.sigma2 == y.sigma2 and tuple(x.modelParameters.euler) == tuple(y.modelParameters.euler)
    finally:
        other.close()
        case.close()
