"""Host-side mirror of GiNGR's registration API over libgingr_cuda.so.

Names and argument meaning follow the reference (paths relative to
/root/reference/src/main/scala/gingr/):
  CpdConfiguration / IcpConfiguration      registration/config/CPD.scala:105-115, ICP.scala:54-66
  GeneralRegistrationState, ModelFittingParameters   api/GeneralRegistrationState.scala:28-41,
                                                     api/ModelFittingParameters.scala:31-74
  CpdRegistration / IcpRegistration (GingrAlgorithm) registration/config/CPD.scala:117-160,
                                                     ICP.scala:84-110, api/GingrAlgorithm.scala:65-303
Everything numeric happens in the CUDA library; this module only marshals arrays.  No CPU fallback.
"""
from __future__ import annotations

import ctypes
import dataclasses
from dataclasses import dataclass, field
from typing import Callable, Optional, Sequence, Tuple

import numpy as np

from . import _native as nat
from ._native import (ALGO_BCPD, ALGO_CPD, ALGO_ICP, NO_TRANSFORMS, POINTCLOUD_CLOSEST_POINT, RIGID_TRANSFORMS,
                      SIMILARITY_TRANSFORMS, STATUS_CONVERGED, STATUS_MAX_ITERATION,
                      STATUS_MODEL_FLEXIBILITY_ERROR, STATUS_NONE, TRIANGULAR_CLOSEST_POINT,
                      ALONG_NORMAL_CLOSEST_POINT, EVAL_MODEL_TO_TARGET, EVAL_SYMMETRIC, EVAL_TARGET_TO_MODEL,
                      GingrConfig, GingrError, GingrMcmcSettings, GingrState)


class Context:
    """One CUDA device + stream (gingr_ctx).  Single-threaded, like a GingrAlgorithm instance."""

    def __init__(self, device: int = 0):
        self._lib = nat.load()
        h = ctypes.c_void_p()
        nat.check(self._lib.gingr_ctx_create(int(device), ctypes.byref(h)))
        self.handle = h
        self.device = device
        self.nranks, self.rank = 1, 0

    def close(self):
        if getattr(self, "handle", None):
            self._lib.gingr_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, code):
        return nat.check(code, self.handle)

    @property
    def stream(self) -> int:
        return int(self._lib.gingr_ctx_stream(self.handle) or 0)

    def synchronize(self):
        self.check(self._lib.gingr_ctx_synchronize(self.handle))

    @property
    def launch_count(self) -> int:
        return int(self._lib.gingr_ctx_launch_count(self.handle))

    @staticmethod
    def unique_id() -> bytes:
        buf = (ctypes.c_char * 128)()
        nat.check(nat.load().gingr_comm_unique_id(ctypes.byref(buf)))
        return bytes(buf.raw)

    def comm_init(self, nranks: int, rank: int, uid: bytes):
        buf = (ctypes.c_char * 128).from_buffer_copy(uid)
        self.check(self._lib.gingr_comm_init(self.handle, int(nranks), int(rank), ctypes.byref(buf)))
        self.nranks, self.rank = nranks, rank


class Target:
    """Target TriangleMesh (or point set) resident on the device (gingr_target)."""

    def __init__(self, ctx: Context, points, triangles=None):
        self.ctx = ctx
        pts = nat.f64(points).reshape(-1, 3)
        tri = None if triangles is None else nat.i32(triangles).reshape(-1, 3)
        self.N = pts.shape[0]
        self.T = 0 if tri is None else tri.shape[0]
        h = ctypes.c_void_p()
        ctx.check(ctx._lib.gingr_target_upload(ctx.handle, self.N, nat.as_dp(pts), nat.as_ip(tri), self.T,
                                               ctypes.byref(h)))
        self.handle = h
        self.points = pts
        self.triangles = tri

    def close(self):
        if getattr(self, "handle", None):
            self.ctx._lib.gingr_target_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Model:
    """scalismo PointDistributionModel on the device (gingr_model): reference points, meanVector,
    basisMatrix [3M, r] (row 3*pid+d), variance [r], optional reference triangles."""

    def __init__(self, ctx: Context, ref_points, mean, basis, variance, triangles=None):
        self.ctx = ctx
        ref = nat.f64(ref_points).reshape(-1, 3)
        self.M = ref.shape[0]
        mean = nat.f64(mean).reshape(-1)
        var = nat.f64(variance).reshape(-1)
        self.rank = var.shape[0]
        basis = np.asarray(basis, dtype=np.float64)
        if mean.shape != (3 * self.M,) or basis.shape != (3 * self.M, self.rank):
            raise ValueError(f"model arrays: mean must be [3M], basis [3M, r]; got {mean.shape}, {basis.shape} for M = {self.M}, r = {self.rank}")
        basis_f = np.asfortranarray(basis)   # Breeze column-major layout; ld = 3M
        tri = None if triangles is None else nat.i32(triangles).reshape(-1, 3)
        self.T = 0 if tri is None else tri.shape[0]
        h = ctypes.c_void_p()
        ctx.check(ctx._lib.gingr_model_upload(ctx.handle, self.M, self.rank, nat.as_dp(ref), nat.as_dp(mean),
                                              basis_f.ctypes.data_as(nat.dp), 3 * self.M, nat.as_dp(var),
                                              nat.as_ip(tri), self.T, ctypes.byref(h)))
        self.handle = h
        self.triangles = tri
        self.reference = ref.copy()      # host copy of model.reference.pointSet (landmark look-up, file export)

    @staticmethod
    def gaussianMixture(ctx: Context, ref_points, triangles, sigmas, scalings, relativeTolerance: float = 0.01,
                        maxRank: int = 0) -> "Model":
        """GPMMTriangleMesh3D(reference, relativeTolerance).GaussianMixture(pars) (api/gpmm/GPMMHelper.scala:117-121;
        .Gaussian(sigma, scaling) is the one-kernel case, :100-103) built on the device."""
        return Model._build_gpmm(ctx, "gingr_gpmm_gaussian_mixture", ref_points, triangles, sigmas, scalings, relativeTolerance, maxRank)

    @staticmethod
    def gaussianSymmetric(ctx: Context, ref_points, triangles, sigmas, scalings, relativeTolerance: float = 0.01,
                          maxRank: int = 0) -> "Model":
        """The mirror-symmetric Gaussian (mixture) model about the plane x = 0, built on the device: scalismo's
        symmetrised kernel K(x, y) = diag(k(x, y) - k(Sx, y), k(x, y) + k(Sx, y), k(x, y) + k(Sx, y)), S = diag(-1, 1, 1),
        k = sum_q scaling_q exp(-|x - y|^2 / sigma_q^2).  Left and right halves deform as mirror images; the caller centres
        the template on the plane x = 0.  Arguments and stopping rule as gaussianMixture."""
        return Model._build_gpmm(ctx, "gingr_gpmm_gaussian_symmetric", ref_points, triangles, sigmas, scalings, relativeTolerance, maxRank)

    @staticmethod
    def inverseLaplacian(ctx: Context, ref_points, triangles, scaling: float, gamma: float, relativeTolerance: float = 0.01,
                         maxRank: int = 0) -> "Model":
        """The inverse-Laplacian model (the model chooser's look-up kernel, api/gpmm LaplacianHelper.scala:26-55 with
        MatrixHelper.pinv :23-26), built on the device: vertices close on the triangle graph move together, vertices merely
        close in space (fingers, the lips of a jaw) do not.  This project's reading of the kernel: L = D - A, the graph
        Laplacian of the triangle edges with unit weights; Ks = scaling (L + gamma I)^-1, or scaling pinv(L) for gamma = 0;
        K = Ks (x) I3; then approximateGPCholesky with the stopping rule of gaussianMixture.  Needs triangles and at most 6000
        vertices.  The models are nearly full rank (about 0.97-0.99 of 3M at relativeTolerance 0.01); registrations,
        posteriors and solves take every rank the builders produce, up to 18 000 (tested up to that rank), so maxRank is
        only needed to trade accuracy for time.  With gamma = 0 the kernel has rank
        3 (M - #components); at relativeTolerance 0 the factorisation would go on to take noise columns from the
        rounding-level residual of the null space, so a full-rank gamma = 0 model wants a small positive tolerance (1e-12
        suffices).  Raises FloatingPointError when L + gamma I is not numerically positive definite."""
        ref = nat.f64(ref_points).reshape(-1, 3)
        tri = None if triangles is None else nat.i32(triangles).reshape(-1, 3)
        h = ctypes.c_void_p()
        rank = ctypes.c_int32()
        code = ctx.check(ctx._lib.gingr_gpmm_inverse_laplacian(ctx.handle, ref.shape[0], nat.as_dp(ref), nat.as_ip(tri),
                                                               0 if tri is None else tri.shape[0], float(scaling), float(gamma),
                                                               float(relativeTolerance), int(maxRank), ctypes.byref(h),
                                                               ctypes.byref(rank)))
        if code == nat.GINGR_MODEL_FLEXIBILITY:
            raise FloatingPointError("inverseLaplacian: L + gamma I is not numerically positive definite (ModelFlexibilityError)")
        m = Model.__new__(Model)
        m.ctx, m.M, m.rank, m.T, m.handle, m.triangles = ctx, ref.shape[0], int(rank.value), tri.shape[0], h, tri
        m.reference = ref.copy()
        return m

    @staticmethod
    def _build_gpmm(ctx: Context, entry: str, ref_points, triangles, sigmas, scalings, relativeTolerance, maxRank) -> "Model":
        """A model from one of the device GPMM builders, which share their arguments."""
        ref = nat.f64(ref_points).reshape(-1, 3)
        tri = None if triangles is None else nat.i32(triangles).reshape(-1, 3)
        sg, sc = nat.f64(np.atleast_1d(sigmas)), nat.f64(np.atleast_1d(scalings))
        if sg.shape != sc.shape or sg.ndim != 1:
            raise ValueError(f"{entry}: one scaling per sigma")
        build = getattr(ctx._lib, entry)
        h = ctypes.c_void_p()
        rank = ctypes.c_int32()
        ctx.check(build(ctx.handle, ref.shape[0], nat.as_dp(ref), nat.as_ip(tri), 0 if tri is None else tri.shape[0], len(sg),
                        nat.as_dp(sg), nat.as_dp(sc), float(relativeTolerance), int(maxRank), ctypes.byref(h), ctypes.byref(rank)))
        m = Model.__new__(Model)
        m.ctx, m.M, m.rank, m.T, m.handle, m.triangles = ctx, ref.shape[0], int(rank.value), 0 if tri is None else tri.shape[0], h, tri
        m.reference = ref.copy()
        return m

    @staticmethod
    def automaticGaussian(ctx: Context, ref_points, triangles, relativeTolerance: float = 0.01, maxRank: int = 0) -> "Model":
        """GPMMTriangleMesh3D(reference, relativeTolerance).AutomaticGaussian() (api/gpmm/GPMMHelper.scala:119-129): the
        two-kernel mixture (maxDist/4, maxDist/8) + (maxDist/8, maxDist/16) with maxDist the largest point distance."""
        d = maximum_point_distance(ref_points)
        return Model.gaussianMixture(ctx, ref_points, triangles, [d / 4.0, d / 8.0], [d / 8.0, d / 16.0], relativeTolerance, maxRank)

    @staticmethod
    def automaticGPMMfromTemplate(ctx: Context, ref_points, triangles, relativeTolerance: float = 0.1, maxRank: int = 0) -> "Model":
        """GPMMHelper.automaticGPMMfromTemplate (api/registration/utils/GPMMHelper.scala:38-68): three Gaussian kernels from
        the largest point distance d and the smallest nearest-neighbour distance e: (sigma, scaling) = (d/4, d/8),
        (d/8, d/16), (5e, 5e/2); relativeTolerance 0.1."""
        d = maximum_point_distance(ref_points)
        e = minimum_point_distance(ref_points)
        sig = [d / 4.0, d / 8.0, e * 5.0]
        return Model.gaussianMixture(ctx, ref_points, triangles, sig, [v / 2.0 for v in sig], relativeTolerance, maxRank)

    def download(self):
        """(reference points [M, 3], meanVector [3M], basisMatrix [3M, r], variance [r]) as scalismo stores them."""
        ref = np.empty((self.M, 3))
        mean = np.empty(3 * self.M)
        basis = np.empty((3 * self.M, self.rank), order="F")
        var = np.empty(self.rank)
        self.ctx.check(self.ctx._lib.gingr_model_download(self.ctx.handle, self.handle, None, None, nat.as_dp(ref), nat.as_dp(mean),
                                                          basis.ctypes.data_as(nat.dp), 3 * self.M, nat.as_dp(var)))
        return ref, mean, basis, var

    @staticmethod
    def _from_handle(ctx: Context, h, M: int, rank: int, triangles) -> "Model":
        """A model the library built: its host copy of the reference points is read back from the device."""
        m = Model.__new__(Model)
        m.ctx, m.M, m.rank, m.handle, m.triangles = ctx, M, rank, h, triangles
        m.T = 0 if triangles is None else triangles.shape[0]
        m.reference = np.empty((M, 3))
        ctx.check(ctx._lib.gingr_model_download(ctx.handle, h, None, None, nat.as_dp(m.reference), None, None, 0, None))
        return m

    def newReference(self, ref_points, triangles=None) -> "Model":
        """model.newReference(newRef, NearestNeighborInterpolator()) (SimpleRegistrator.scala:90-92) on the device: the
        new model's rows are gathered from the resident basis at the nearest old reference points."""
        ref = nat.f64(ref_points).reshape(-1, 3)
        tri = None if triangles is None else nat.i32(triangles).reshape(-1, 3)
        h = ctypes.c_void_p()
        self.ctx.check(self.ctx._lib.gingr_model_new_reference(self.ctx.handle, self.handle, ref.shape[0], nat.as_dp(ref),
                                                               nat.as_ip(tri), 0 if tri is None else tri.shape[0],
                                                               ctypes.byref(h)))
        m = Model.__new__(Model)
        m.ctx, m.M, m.rank, m.T, m.handle, m.triangles = self.ctx, ref.shape[0], self.rank, 0 if tri is None else tri.shape[0], h, tri
        m.reference = ref.copy()
        return m

    def instance(self, parameters: "ModelFittingParameters") -> np.ndarray:
        """ModelFittingParameters.modelInstanceShapePoseScale(model, parameters) (ModelFittingParameters.scala:130-143)."""
        st = GingrState()
        st.scale = float(parameters.scale)
        for d in range(3):
            st.translation[d] = float(parameters.translation[d])
            st.euler[d] = float(parameters.euler[d])
            st.center[d] = float(parameters.center[d])
        st.rank = self.rank
        alpha = nat.f64(parameters.shape)
        if alpha.shape != (self.rank,):
            raise ValueError(f"shape coefficients have shape {alpha.shape}, the model has rank {self.rank}")
        fit = np.empty((self.M, 3))
        self.ctx.check(self.ctx._lib.gingr_model_instance(self.ctx.handle, self.handle, ctypes.byref(st), nat.as_dp(alpha),
                                                          nat.as_dp(fit)))
        return fit

    def close(self):
        if getattr(self, "handle", None):
            self.ctx._lib.gingr_model_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---------------------------------------------------------------------------------------------
# kernel-level operators
# ---------------------------------------------------------------------------------------------
def _max_pair_distance(a: np.ndarray, b: np.ndarray) -> float:
    best = 0.0
    step = max(1, (1 << 22) // max(1, b.shape[0]))
    for i0 in range(0, a.shape[0], step):
        d = a[i0:i0 + step, None, :] - b[None, :, :]
        best = max(best, float(np.sqrt(d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1] + d[..., 2] * d[..., 2]).max()))
    return best


def maximum_point_distance(points, brute_force_limit: int = 2048) -> float:
    """PointSetHelper.maximumPointDistance (api/gpmm/GPMMHelper.scala:76-81): max over all pairs of (p1 - p2).norm, the
    reference's O(M^2) loop ("TODO: compute faster for large pointsets").  The maximum is attained between two vertices
    of the convex hull, so above brute_force_limit points only hull vertices are paired; the distances themselves are
    formed exactly as EuclideanVector3D.norm does (sqrt(x*x + y*y + z*z) of the component differences), so the value is
    the reference's bit for bit.  Host side (once per model construction)."""
    p = np.ascontiguousarray(np.asarray(points, dtype=np.float64).reshape(-1, 3))
    if p.shape[0] > brute_force_limit:
        try:
            from scipy.spatial import ConvexHull, QhullError
            try:
                p = p[ConvexHull(p).vertices]
            except QhullError:      # degenerate (flat) point sets: pair everything
                pass
        except ImportError:
            pass
    return _max_pair_distance(p, p)


def minimum_point_distance(points) -> float:
    """PointSetHelper.minimumPointDistance (api/gpmm/GPMMHelper.scala:83-85, registration/utils/GPMMHelper.scala:35-37): the
    smallest distance from a point to its nearest OTHER point (0 when the set holds duplicates).  Neighbour candidates come
    from a KD-tree; the distances are re-formed as EuclideanVector3D.norm does, so the value is the brute-force one."""
    p = np.ascontiguousarray(np.asarray(points, dtype=np.float64).reshape(-1, 3))
    n = p.shape[0]
    if n < 2:
        raise ValueError("minimum point distance needs two points")
    try:
        from scipy.spatial import cKDTree
        k = min(4, n)
        _, nb = cKDTree(p).query(p, k=k)                         # self + the next k - 1 candidates
        nb = nb[:, 1:] if k > 1 else nb
        d = p[:, None, :] - p[nb]
        cand = np.sqrt(d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1] + d[..., 2] * d[..., 2])
        return float(cand.min())
    except ImportError:
        best = np.inf
        for i0 in range(0, n, 1024):
            d = p[i0:i0 + 1024, None, :] - p[None, :, :]
            dist = np.sqrt(d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1] + d[..., 2] * d[..., 2])
            dist[np.arange(dist.shape[0]), np.arange(i0, i0 + dist.shape[0])] = np.inf
            best = min(best, float(dist.min()))
        return best


def cpd_estep(ctx: Context, target: Target, fit, sigma2: float, w: float):
    """P1[M], Pt1[N_local], PX[M,3] of CpdRegistrationState.P (CPD.scala:54-75) without forming P."""
    fit = nat.f64(fit).reshape(-1, 3)
    M = fit.shape[0]
    n_local = _local_count(target.N, ctx)
    P1, Pt1, PX = np.empty(M), np.empty(n_local), np.empty((M, 3))
    ctx.check(ctx._lib.gingr_cpd_estep(ctx.handle, target.handle, M, nat.as_dp(fit), float(sigma2), float(w),
                                       nat.as_dp(P1), nat.as_dp(Pt1), nat.as_dp(PX)))
    return P1, Pt1, PX


def bcpd_estep(ctx: Context, target: Target, y, sigma_mm, alpha, sigma2: float, s: float, w: float):
    """nu, nu', Nhat, xhat of BCPD.computeP + reductions (BCPD.scala:167-184, :200-209)."""
    y = nat.f64(y).reshape(-1, 3)
    M = y.shape[0]
    sm, al = nat.f64(sigma_mm), nat.f64(alpha)
    n_local = _local_count(target.N, ctx)
    nu, nup, xhat = np.empty(M), np.empty(n_local), np.empty((M, 3))
    nhat = ctypes.c_double()
    ctx.check(ctx._lib.gingr_bcpd_estep(ctx.handle, target.handle, M, nat.as_dp(y), nat.as_dp(sm), nat.as_dp(al),
                                        float(sigma2), float(s), float(w), nat.as_dp(nu), nat.as_dp(nup),
                                        ctypes.byref(nhat), nat.as_dp(xhat)))
    return nu, nup, float(nhat.value), xhat


def cpd_initial_sigma2(ctx: Context, target: Target, points) -> float:
    """computeInitialSigma2 (CPD.scala:81-90)."""
    pts = nat.f64(points).reshape(-1, 3)
    out = ctypes.c_double()
    ctx.check(ctx._lib.gingr_cpd_initial_sigma2(ctx.handle, target.handle, pts.shape[0], nat.as_dp(pts),
                                                ctypes.byref(out)))
    return float(out.value)


def icp_closest(ctx: Context, target: Target, template_points, template_triangles, method: int):
    """closestPointCorrespondence (ClosestPointRegistrator.scala:74-96, :133-160):
    returns idx[M] (nearest target vertex), cp[M,3], w[M] in {0,1}, mean distance."""
    tpl = nat.f64(template_points).reshape(-1, 3)
    M = tpl.shape[0]
    tri = None if template_triangles is None else nat.i32(template_triangles).reshape(-1, 3)
    T = 0 if tri is None else tri.shape[0]
    idx = np.empty(M, dtype=np.int32)
    cp = np.empty((M, 3))
    w = np.empty(M, dtype=np.uint8)
    md = ctypes.c_double()
    ctx.check(ctx._lib.gingr_icp_closest(ctx.handle, target.handle, M, nat.as_dp(tpl), nat.as_ip(tri), T, int(method),
                                         nat.as_ip(idx), nat.as_dp(cp), nat.as_bp(w), ctypes.byref(md)))
    return idx, cp, w, float(md.value)


def icp_closest_reversal(ctx: Context, target: Target, template_points, template_triangles, method: int):
    """closestPointCorrespondenceReversal (ClosestPointRegistrator.scala:34-45): per TARGET vertex j the template
    vertex id its correspondence maps back to and the 0/1 weight; the observation is (tpl_id[j], target[j], w[j])."""
    tpl = nat.f64(template_points).reshape(-1, 3)
    M = tpl.shape[0]
    tri = None if template_triangles is None else nat.i32(template_triangles).reshape(-1, 3)
    T = 0 if tri is None else tri.shape[0]
    tid = np.empty(target.N, dtype=np.int32)
    w = np.empty(target.N, dtype=np.uint8)
    md = ctypes.c_double()
    ctx.check(ctx._lib.gingr_icp_closest_reversal(ctx.handle, target.handle, M, nat.as_dp(tpl), nat.as_ip(tri), T,
                                                  int(method), nat.as_ip(tid), nat.as_bp(w), ctypes.byref(md)))
    return tid, w, float(md.value)


def posterior_mean(ctx: Context, model: Model, R, t, pids, points, noise):
    """model.transform(R, t).posterior(obs).mean -> (coefficients[r], mean mesh points[M,3]).
    noise: [n] isotropic variances or [n,3,3] covariances.  (GingrAlgorithm.scala:297-301, SURVEY A3)"""
    R = nat.f64(R).reshape(3, 3)
    t = nat.f64(t).reshape(3)
    pids = nat.i32(pids)
    pts = nat.f64(points).reshape(-1, 3)
    noise = nat.f64(noise)
    kind = 0 if noise.ndim == 1 else 1
    n = pids.shape[0]
    if pids.ndim != 1 or pts.shape[0] != n:
        raise ValueError(f"{n} point ids but {pts.shape[0]} points")
    if noise.shape not in ((n,), (n, 3, 3)):
        raise ValueError(f"noise must have shape ({n},) or ({n}, 3, 3), got {noise.shape}")
    c = np.empty(model.rank)
    mesh = np.empty((model.M, 3))
    code = ctx.check(ctx._lib.gingr_posterior_mean(ctx.handle, model.handle, nat.as_dp(R), nat.as_dp(t),
                                                   pids.shape[0], nat.as_ip(pids), nat.as_dp(pts), kind,
                                                   nat.as_dp(noise), nat.as_dp(c), nat.as_dp(mesh)))
    if code == nat.GINGR_MODEL_FLEXIBILITY:
        raise FloatingPointError("posterior failed (ModelFlexibilityError)")
    return c, mesh


def posterior_covariance(ctx: Context, model: Model, R, t, pids, points, noise) -> np.ndarray:
    """Covariance of model.transform(R, t).posterior(obs) at the mesh points -> [M, 3, 3]
    (GingrAlgorithm.scala:300; the quantity helper/PosteriorHelper.scala:26-80 colour-maps).  Arguments as posterior_mean."""
    R = nat.f64(R).reshape(3, 3)
    t = nat.f64(t).reshape(3)
    pids = nat.i32(pids)
    pts = nat.f64(points).reshape(-1, 3)
    noise = nat.f64(noise)
    n = pids.shape[0]
    if pids.ndim != 1 or pts.shape[0] != n:
        raise ValueError(f"{n} point ids but {pts.shape[0]} points")
    if noise.shape not in ((n,), (n, 3, 3)):
        raise ValueError(f"noise must have shape ({n},) or ({n}, 3, 3), got {noise.shape}")
    cov = np.empty((model.M, 3, 3))
    code = ctx.check(ctx._lib.gingr_posterior_covariance(ctx.handle, model.handle, nat.as_dp(R), nat.as_dp(t), n, nat.as_ip(pids),
                                                         nat.as_dp(pts), 0 if noise.ndim == 1 else 1, nat.as_dp(noise), nat.as_dp(cov)))
    if code == nat.GINGR_MODEL_FLEXIBILITY:
        raise FloatingPointError("posterior failed (ModelFlexibilityError)")
    return cov


def posterior_model(ctx: Context, model: Model, R, t, pids, points, noise) -> Model:
    """model.transform(R, t).posterior(obs) as a new device model (scalismo PointDistributionModel.posterior, SURVEY A3;
    GingrAlgorithm.scala:299-300): reference R ref + t, mean R (mean + basis D c), basis (I (x) R) basis U, variance s
    (descending) with U diag(s) U^T = D Mx^-1 D.  Arguments as posterior_mean; raises FloatingPointError where the
    posterior fails (ModelFlexibilityError)."""
    R = nat.f64(R).reshape(3, 3)
    t = nat.f64(t).reshape(3)
    pids = nat.i32(pids)
    pts = nat.f64(points).reshape(-1, 3)
    noise = nat.f64(noise)
    n = pids.shape[0]
    if pids.ndim != 1 or pts.shape[0] != n:
        raise ValueError(f"{n} point ids but {pts.shape[0]} points")
    if noise.shape not in ((n,), (n, 3, 3)):
        raise ValueError(f"noise must have shape ({n},) or ({n}, 3, 3), got {noise.shape}")
    h = ctypes.c_void_p()
    code = ctx.check(ctx._lib.gingr_model_posterior(ctx.handle, model.handle, nat.as_dp(R), nat.as_dp(t), n, nat.as_ip(pids),
                                                    nat.as_dp(pts), 0 if noise.ndim == 1 else 1, nat.as_dp(noise), ctypes.byref(h)))
    if code == nat.GINGR_MODEL_FLEXIBILITY:
        raise FloatingPointError("posterior failed (ModelFlexibilityError)")
    return Model._from_handle(ctx, h, model.M, model.rank, model.triangles)


def posterior_model_profile(ctx: Context):
    """Device times (ms) of the last posterior model built on ctx: dict(system, jacobi, gemm, constants, total, sweeps)."""
    ms = np.zeros(5)
    sweeps = ctypes.c_int32()
    ctx.check(ctx._lib.gingr_posterior_model_profile(ctx.handle, nat.as_dp(ms), ctypes.byref(sweeps)))
    return dict(system=float(ms[0]), jacobi=float(ms[1]), gemm=float(ms[2]), constants=float(ms[3]), total=float(ms[4]),
                sweeps=int(sweeps.value))


def spd_solve(ctx: Context, A, B=None, reps: int = 1):
    """The on-device r x r Cholesky solve of the regression (scalismo: Minv = pinv(Mx); c = Minv * rhs; SURVEY A3).
    A: [n, n] symmetric positive definite; B: [nrhs, n] right-hand sides as rows (or None).
    -> dict(L=[n, n] lower factor, Y=[nrhs, n] rows L^-1 b_q, x=[n] A^-1 b_0 (None without B), ms=device time of one
    factorisation + back substitution).  Raises FloatingPointError when A is not positive definite."""
    A = nat.f64(A)
    n = A.shape[0]
    if A.shape != (n, n):
        raise ValueError(f"A must be square, got {A.shape}")
    nrhs = 0
    if B is not None:
        B = nat.f64(B).reshape(-1, n)
        nrhs = B.shape[0]
    L = np.empty((n, n))
    Y = np.empty((nrhs, n))
    x = np.empty(n) if nrhs else None
    ms = ctypes.c_double()
    code = ctx.check(ctx._lib.gingr_spd_solve(ctx.handle, n, nat.as_dp(A), nrhs, nat.as_dp(B), nat.as_dp(L), nat.as_dp(Y),
                                              nat.as_dp(x), int(reps), ctypes.byref(ms)))
    if code == nat.GINGR_MODEL_FLEXIBILITY:
        raise FloatingPointError("matrix not positive definite (ModelFlexibilityError)")
    return dict(L=L, Y=Y, x=x, ms=float(ms.value))


def coefficients(ctx: Context, model: Model, R, t, mesh_points):
    """model.transform(R, t).coefficients(mesh) (GingrAlgorithm.scala:215, :236)."""
    R = nat.f64(R).reshape(3, 3)
    t = nat.f64(t).reshape(3)
    mesh = nat.f64(mesh_points).reshape(-1, 3)
    if mesh.shape[0] != model.M:
        raise ValueError(f"mesh has {mesh.shape[0]} points, the model has {model.M}")
    c = np.empty(model.rank)
    code = ctx.check(ctx._lib.gingr_coefficients(ctx.handle, model.handle, nat.as_dp(R), nat.as_dp(t),
                                                 nat.as_dp(mesh), nat.as_dp(c)))
    if code == nat.GINGR_MODEL_FLEXIBILITY:
        raise FloatingPointError("coefficients failed (ModelFlexibilityError)")
    return c


def _local_count(n: int, ctx: Context) -> int:
    base, rem = divmod(n, ctx.nranks)
    return base + (1 if ctx.rank < rem else 0)


def shard_range(n: int, nranks: int, rank: int) -> Tuple[int, int]:
    """[begin, begin+count) of n items owned by `rank` -- the partition libgingr_cuda uses for target
    points (E-step) and GPMM points (Gram / fit evaluation)."""
    base, rem = divmod(n, nranks)
    begin = rank * base + min(rank, rem)
    return begin, base + (1 if rank < rem else 0)


# ---------------------------------------------------------------------------------------------
# state / configuration records
# ---------------------------------------------------------------------------------------------
@dataclass
class ModelFittingParameters:
    """api/ModelFittingParameters.scala:57-74: scale, pose (translation, Euler rotation), shape."""
    scale: float
    translation: np.ndarray
    euler: Tuple[float, float, float]
    shape: np.ndarray
    center: np.ndarray = field(default_factory=lambda: np.zeros(3))


@dataclass
class GeneralRegistrationState:
    """Numeric part of api/GeneralRegistrationState.scala:28-41 (model/target live in device handles)."""
    modelParameters: ModelFittingParameters
    fit: np.ndarray
    sigma2: float = 1.0
    globalTransformation: int = RIGID_TRANSFORMS
    stepLength: float = 1.0
    generatedBy: str = ""
    iteration: int = 0
    status: int = STATUS_NONE

    def statusText(self) -> str:
        """The sentence printStatus() prints (GeneralRegistrationState.scala:104-114)."""
        n = self.iteration + 1
        return {STATUS_NONE: "Initial state - no iterations performed!",
                STATUS_CONVERGED: f"Fitting converged after {n} accepted iterations!",
                STATUS_MAX_ITERATION: f"Fitting finished the MaxIterations with ({n}) accepted iterations!",
                STATUS_MODEL_FLEXIBILITY_ERROR: f"Model not flexible enough to compute posterior model - finished after {n} accepted iterations!",
                }[self.status]

    def printStatus(self) -> None:
        print(self.statusText())

    def to_pod(self) -> Tuple[GingrState, np.ndarray]:
        p = self.modelParameters
        st = GingrState()
        st.scale = float(p.scale)
        st.translation[:] = [float(v) for v in p.translation]
        st.euler[:] = [float(v) for v in p.euler]
        st.center[:] = [float(v) for v in p.center]
        st.sigma2 = float(self.sigma2)
        st.step_length = float(self.stepLength)
        st.global_transformation = int(self.globalTransformation)
        st.iteration = int(self.iteration)
        st.status = int(self.status)
        alpha = nat.f64(p.shape).copy()
        st.rank = alpha.shape[0]
        return st, alpha

    @staticmethod
    def from_pod(st: GingrState, alpha: np.ndarray, fit: np.ndarray, generatedBy: str = "") -> "GeneralRegistrationState":
        p = ModelFittingParameters(st.scale, np.array(list(st.translation)), tuple(st.euler), alpha.copy(),
                                   np.array(list(st.center)))
        return GeneralRegistrationState(p, fit, st.sigma2, st.global_transformation, st.step_length, generatedBy,
                                        st.iteration, st.status)


@dataclass
class CpdConfiguration:
    """registration/config/CPD.scala:105-115"""
    maxIterations: int = 100
    threshold: float = 1e-10
    converged: Callable = lambda last, cur, thr: abs(last.sigma2 - cur.sigma2) < thr
    useLandmarkCorrespondence: bool = True
    initialSigma: Optional[float] = None
    w: float = 0.0
    lambda_: float = 1.0

    def to_pod(self) -> GingrConfig:
        c = GingrConfig()
        c.algorithm = ALGO_CPD
        c.max_iterations = self.maxIterations
        c.threshold = self.threshold
        c.use_landmark_correspondence = int(self.useLandmarkCorrespondence)
        c.has_initial_sigma = int(self.initialSigma is not None)
        c.initial_sigma = float(self.initialSigma or 0.0)
        c.w = self.w
        c.lambda_ = self.lambda_
        return c


@dataclass
class IcpConfiguration:
    """registration/config/ICP.scala:54-66"""
    maxIterations: int = 100
    threshold: float = 1e-10
    converged: Callable = lambda last, cur, thr: False
    useLandmarkCorrespondence: bool = True
    initialSigma: float = 100.0
    endSigma: float = 1.0
    reverseCorrespondenceDirection: bool = False
    correspondenceMethod: int = TRIANGULAR_CLOSEST_POINT

    @property
    def sigmaStep(self) -> float:
        return (self.initialSigma - self.endSigma) / float(self.maxIterations)

    def to_pod(self) -> GingrConfig:
        c = GingrConfig()
        c.algorithm = ALGO_ICP
        c.max_iterations = self.maxIterations
        c.threshold = self.threshold
        c.use_landmark_correspondence = int(self.useLandmarkCorrespondence)
        c.has_initial_sigma = 1
        c.initial_sigma = float(self.initialSigma)
        c.end_sigma = float(self.endSigma)
        c.reverse_correspondence_direction = int(self.reverseCorrespondenceDirection)
        c.correspondence_method = int(self.correspondenceMethod)
        return c


@dataclass
class BcpdConfiguration:
    """The BCPD configuration of GingrAlgorithm (include/gingr_cuda.h GINGR_ALGO_BCPD; this project's reading of
    other/algorithms/cpd/BCPD.scala on GiNGR's hooks).  Every field but `kappa` means what it means for CPD; `kappa` is the
    Dirichlet concentration of the mixing-weight update alpha_m = exp(psi(kappa + nu_m) - psi(kappa M + Nhat)).

    Scale: the E-step's outlier term is w / N, literally as in BCPD.scala, against Gaussians of height (2 pi sigma2)^-3/2.
    With w > 0 on data whose initial sigma2 is large (coordinates of hundreds of units) it outweighs every Gaussian, Nhat
    becomes tiny and sigma2 grows without bound; use w = 0 there, or scale the coordinates down."""
    maxIterations: int = 100
    threshold: float = 1e-10
    converged: Callable = lambda last, cur, thr: abs(last.sigma2 - cur.sigma2) < thr
    useLandmarkCorrespondence: bool = True
    initialSigma: Optional[float] = None
    w: float = 0.0
    lambda_: float = 1.0
    kappa: float = 1.0

    def to_pod(self) -> GingrConfig:
        c = CpdConfiguration(self.maxIterations, self.threshold, self.converged, self.useLandmarkCorrespondence,
                             self.initialSigma, self.w, self.lambda_).to_pod()
        c.algorithm = ALGO_BCPD
        return c


class GingrAlgorithm:
    """api/GingrAlgorithm.scala:65-303 with `update` (:192-254) executed on the device."""
    name = "Gingr"

    def __init__(self, ctx: Context, model: Model, target: Target, config):
        self.ctx, self.model, self.target, self.config = ctx, model, target, config
        pod = config.to_pod()
        h = ctypes.c_void_p()
        ctx.check(ctx._lib.gingr_registration_create(ctx.handle, model.handle, target.handle, ctypes.byref(pod),
                                                     ctypes.byref(h)))
        self.handle = h

    def close(self):
        if getattr(self, "handle", None):
            self.ctx._lib.gingr_registration_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def setLandmarks(self, pids, points, cov=None):
        """GeneralRegistrationState.landmarkCorrespondences (GeneralRegistrationState.scala:43-62),
        resolved by the caller: reference vertex ids, target landmark points, 3x3 covariances (I3 default)."""
        pids = nat.i32(pids)
        pts = nat.f64(points).reshape(-1, 3)
        L = pids.shape[0]
        cov = np.tile(np.eye(3), (L, 1, 1)) if cov is None else nat.f64(cov).reshape(L, 3, 3)
        cov = nat.f64(cov)
        self.ctx.check(self.ctx._lib.gingr_registration_set_landmarks(self.handle, L, nat.as_ip(pids), nat.as_dp(pts),
                                                                      nat.as_dp(cov)))

    def initializeState(self, globalTransformation: int = RIGID_TRANSFORMS, rotation=None, translation=None,
                        general: Optional[GeneralRegistrationState] = None) -> GeneralRegistrationState:
        """GeneralRegistrationState.apply (:136-178) + initializeState (CPD.scala:92-103 / ICP.scala:74-86)."""
        if general is None:
            from .rotation import matrix_to_euler
            euler = (0.0, 0.0, 0.0) if rotation is None else matrix_to_euler(np.asarray(rotation, dtype=float))
            t = np.zeros(3) if translation is None else np.asarray(translation, dtype=float)
            pars = ModelFittingParameters(1.0, t, euler, np.zeros(self.model.rank))
            general = GeneralRegistrationState(pars, np.zeros((self.model.M, 3)),
                                               globalTransformation=globalTransformation)
        st, alpha = general.to_pod()
        fit = np.empty((self.model.M, 3))
        self.ctx.check(self.ctx._lib.gingr_initialize_state(self.handle, ctypes.byref(st), nat.as_dp(alpha),
                                                            nat.as_dp(fit)))
        return GeneralRegistrationState.from_pod(st, alpha, fit, general.generatedBy)

    def update(self, current: GeneralRegistrationState, probabilistic: bool = False, seed: int = 0,
               with_fit: bool = True) -> GeneralRegistrationState:
        """GingrAlgorithm.update (:192-254).  The returned state's `fit` is already the refreshed fit of
        GingrGeneratorWrapper.propose (the reference leaves the old fit in place until `propose`)."""
        st, alpha = current.to_pod()
        out = GingrState()
        alpha_out = np.empty_like(alpha)
        fit = np.empty((self.model.M, 3)) if with_fit else None
        self.ctx.check(self.ctx._lib.gingr_update(self.handle, ctypes.byref(st), nat.as_dp(alpha), int(probabilistic),
                                                  int(seed), ctypes.byref(out), nat.as_dp(alpha_out), nat.as_dp(fit)))
        return GeneralRegistrationState.from_pod(out, alpha_out, fit if with_fit else current.fit, current.generatedBy)

    def propose(self, current: GeneralRegistrationState, probabilistic: bool = False,
                seed: int = 0) -> GeneralRegistrationState:
        """GingrGeneratorWrapper.propose (GingrGeneratorWrapper.scala:28-39) around the deterministic
        wrapper (GeneratorWrapperDeterministic.scala:28-34) or, with probabilistic=True, the informed proposal of
        GeneratorWrapperStochastic.gingrPropose (GeneratorWrapperStochastic.scala:34-40): update, refresh fit,
        iteration += 1."""
        ns = self.update(current, probabilistic, seed)
        return dataclasses.replace(ns, generatedBy="Stochastic" if probabilistic else "Deterministic",
                                   iteration=ns.iteration + 1)

    def run(self, initialState: GeneralRegistrationState, callBackLogger=None) -> GeneralRegistrationState:
        """Deterministic GingrAlgorithm.run (:115-175): the chain yields the initial state first, so
        maxIterations - 1 proposals are made; stops on converged(last, cur) or ModelFlexibilityError."""
        st = initialState
        last = None
        final = STATUS_MAX_ITERATION
        for k in range(self.config.maxIterations):
            if k > 0:
                st = self.propose(st)
            if callBackLogger is not None:
                callBackLogger(st)
            converged = last is not None and self.config.converged(last, st, self.config.threshold)
            error = st.status == STATUS_MODEL_FLEXIBILITY_ERROR
            last = st
            if converged:
                final = STATUS_CONVERGED
                break
            if error:
                break
        if st.status == STATUS_NONE:
            st = dataclasses.replace(st, status=final)
        return st

    def computePosterior(self, current: GeneralRegistrationState) -> Model:
        """GingrAlgorithm.computePosterior(current) (:281-302): the posterior model of the configuration's correspondences
        and uncertainties (and landmarks) at `current`.  Raises FloatingPointError where the posterior fails.  The device-resident
        state is replaced; the next update uploads its own."""
        st, alpha = current.to_pod()
        h = ctypes.c_void_p()
        code = self.ctx.check(self.ctx._lib.gingr_registration_posterior_model(self.handle, ctypes.byref(st), nat.as_dp(alpha),
                                                                               ctypes.byref(h)))
        if code == nat.GINGR_MODEL_FLEXIBILITY:
            raise FloatingPointError("posterior failed (ModelFlexibilityError)")
        return Model._from_handle(self.ctx, h, self.model.M, self.model.rank, self.model.triangles)

    # device-resident chaining (throughput runs)
    def updateChain(self, iters: int):
        self.ctx.check(self.ctx._lib.gingr_update_chain(self.handle, int(iters)))

    def updateChainSampled(self, iters: int, seed: int):
        self.ctx.check(self.ctx._lib.gingr_update_chain_sampled(self.handle, int(iters), int(seed)))

    def downloadState(self) -> GeneralRegistrationState:
        st = GingrState()
        alpha = np.empty(self.model.rank)
        fit = np.empty((self.model.M, 3))
        self.ctx.check(self.ctx._lib.gingr_state_download(self.handle, ctypes.byref(st), nat.as_dp(alpha),
                                                          nat.as_dp(fit)))
        return GeneralRegistrationState.from_pod(st, alpha, fit)

    # ---- probabilistic registration (GingrAlgorithm.run with ProbabilisticSettings, :115-190) --------------------
    def configureProbabilistic(self, settings: "ProbabilisticSettings"):
        """Attach ProbabilisticSettings(IndependentPoints(...), randomMixture) to the registration."""
        pod = settings.to_pod()
        mids = None if settings.modelPointIds is None else nat.i32(settings.modelPointIds)
        tids = None if settings.targetPointIds is None else nat.i32(settings.targetPointIds)
        self.ctx.check(self.ctx._lib.gingr_mcmc_configure(self.handle, ctypes.byref(pod), nat.as_ip(mids),
                                                          0 if mids is None else len(mids), nat.as_ip(tids),
                                                          0 if tids is None else len(tids)))
        self.probabilisticSettings = settings

    def logValue(self, state: GeneralRegistrationState):
        """(Prior, Distance) log values of the evaluators (Evaluator.scala:43-60); their sum is the product evaluator."""
        st, alpha = state.to_pod()
        out = np.zeros(2)
        self.ctx.check(self.ctx._lib.gingr_evaluate_log_value(self.handle, ctypes.byref(st), nat.as_dp(alpha), nat.as_dp(out)))
        return float(out[0]), float(out[1])

    def logTransitionProbability(self, frm: GeneralRegistrationState, to: GeneralRegistrationState) -> float:
        """GeneratorWrapperStochastic.logTransitionProbability (GeneratorWrapperStochastic.scala:42-63)."""
        sf, af = frm.to_pod()
        stt, at = to.to_pod()
        out = np.zeros(1)
        self.ctx.check(self.ctx._lib.gingr_log_transition_probability(self.handle, ctypes.byref(sf), nat.as_dp(af),
                                                                      ctypes.byref(stt), nat.as_dp(at), nat.as_dp(out)))
        return float(out[0])

    def mcmcChain(self, iters: int, seed: int):
        """`iters` Metropolis-Hastings steps from the device-resident state, on the device (gingr_mcmc_chain)."""
        self.ctx.check(self.ctx._lib.gingr_mcmc_chain(self.handle, int(iters), int(seed)))

    def mcmcStats(self):
        values = np.zeros(16)
        counts = np.zeros(32, dtype=np.int32)
        self.ctx.check(self.ctx._lib.gingr_mcmc_stats(self.handle, nat.as_dp(values), nat.as_ip(counts)))
        return values, counts

    def mcmcBest(self) -> GeneralRegistrationState:
        st = GingrState()
        alpha = np.empty(self.model.rank)
        fit = np.empty((self.model.M, 3))
        self.ctx.check(self.ctx._lib.gingr_mcmc_best(self.handle, ctypes.byref(st), nat.as_dp(alpha), nat.as_dp(fit)))
        return GeneralRegistrationState.from_pod(st, alpha, fit)

    def collectSamples(self, collection: Optional["SampleCollection"]):
        """Collect the chain's states on the device by the rule of LogHelper.samplesFromLog (LogHelper.scala:29-43), for
        the posterior variance maps (sample_statistics).  None switches collection off.  Set it after
        configureProbabilistic, which discards it; the accumulators restart with every fresh chain."""
        c = SampleCollection(takeEveryN=0) if collection is None else collection
        self.ctx.check(self.ctx._lib.gingr_mcmc_collect(self.handle, int(c.burnIn), int(c.takeEveryN), int(c.total)))

    def generatorNames(self, settings: "ProbabilisticSettings"):
        """generatedBy of the ten leaves of generatorCombined (GingrAlgorithm.scala:177-190, sampling/Generator.scala:31-83),
        in the order of the device's leaf index (mcmcStats counts[1])."""
        r, t, sh = settings.rotationSdev, settings.translationSdev, settings.shapeSteps
        return ([self.name] + [f"Rotation{a}-{float(v)!r}" for a, v in zip(("Yaw", "Pitch", "Roll"), r)] +
                [f"Translation{a}-{float(v)!r}" for a, v in zip("XYZ", t)] + [f"RandomShape-{float(v)!r}" for v in sh])

    def runProbabilistic(self, initialState: GeneralRegistrationState, settings: "ProbabilisticSettings", seed: int = 0,
                         iterations: Optional[int] = None, acceptRejectLogger=None, callBackLogger=None,
                         sampleCollection: Optional["SampleCollection"] = None) -> GeneralRegistrationState:
        """GingrAlgorithm.run with probabilisticSettings (:115-175): maxIterations - 1 MH steps, returns the best sample
        (:160-163) with status MaxIteration unless the chain ended in ModelFlexibilityError.

        Without loggers the whole chain runs on the device in one call.  With an acceptRejectLogger (io.JSONStateLogger:
        accept(state, values) / reject(state, values)) or a callBackLogger (callable(state), ChainStateLogger.logState)
        the same chain -- same seed, same draws, same decisions -- is advanced one step per call and read back after
        each step, as scalismo's logged iterator does (:126-134).  A rejected proposal is logged with its generator name
        and log values; its scale (the only parameter jsonLogFormat keeps for a rejected sample) is the current
        state's, which differs from the proposal's only for a rejected informed SimilarityTransforms step.

        sampleCollection: collect the chain's states on the device (collectSamples); read them with sample_statistics."""
        self.configureProbabilistic(settings)
        if sampleCollection is not None:
            self.collectSamples(sampleCollection)
        logged = acceptRejectLogger is not None or callBackLogger is not None
        # the evaluators depend on the parameters only; evaluated BEFORE initializeState because gingr_evaluate_log_value
        # replaces the device-resident state the chain starts from
        lp0 = dict(zip(("Prior", "Distance"), self.logValue(initialState))) if acceptRejectLogger is not None else None
        st, alpha = initialState.to_pod()
        fit = np.empty((self.model.M, 3))
        self.ctx.check(self.ctx._lib.gingr_initialize_state(self.handle, ctypes.byref(st), nat.as_dp(alpha), nat.as_dp(fit)))
        steps = max((self.config.maxIterations - 1) if iterations is None else int(iterations), 0)
        if not logged:
            self.mcmcChain(steps, seed)
        else:
            names = self.generatorNames(settings)
            current = dataclasses.replace(GeneralRegistrationState.from_pod(st, alpha, fit), generatedBy=initialState.generatedBy)
            if acceptRejectLogger is not None:                         # :126 the initial state is logged as accepted
                acceptRejectLogger.accept(current, lp0)
            if callBackLogger is not None:
                callBackLogger(current)
            for _ in range(steps):
                self.mcmcChain(1, seed)
                values, counts = self.mcmcStats()
                lp = {"Prior": float(values[2]), "Distance": float(values[3])}
                name = names[int(counts[1])]
                if counts[2]:
                    current = dataclasses.replace(self.downloadState(), generatedBy=name)
                    if acceptRejectLogger is not None:
                        acceptRejectLogger.accept(current, lp)
                elif acceptRejectLogger is not None:
                    acceptRejectLogger.reject(dataclasses.replace(current, generatedBy=name), lp)
                if callBackLogger is not None:
                    callBackLogger(current)
                if current.status == STATUS_MODEL_FLEXIBILITY_ERROR:   # :150-153 the chain stops at an error state
                    break
        best = self.mcmcBest()
        if best.status == STATUS_NONE:
            best = dataclasses.replace(best, status=STATUS_MAX_ITERATION)
        return best

    def setProfiling(self, enable: bool):
        self.ctx.check(self.ctx._lib.gingr_registration_set_profiling(self.handle, int(enable)))

    def getProfile(self):
        """(ms[8] summed over `iterations`, iterations) since the last call; see include/gingr_cuda.h."""
        ms = np.zeros(8)
        it = ctypes.c_int32()
        self.ctx.check(self.ctx._lib.gingr_registration_get_profile(self.handle, nat.as_dp(ms), ctypes.byref(it)))
        return ms, int(it.value)


def update_batch(chains: Sequence[GingrAlgorithm], iters: int, probabilistic: bool = False, seed: int = 0):
    """`iters` update+propose steps of every chain (independent registrations on one ctx; gingr_update_batch).
    Each chain must hold a device-resident state (initializeState / update); read results with downloadState().
    All chains advance through one batched kernel sequence per iteration (one launch per kernel of the iteration, chain =
    blockIdx.z) when the iteration is batch-aware -- CPD and the ICP flavours on the scans are; the uniform-grid searches of
    large meshes replay per-chain graphs."""
    ctx = chains[0].ctx
    arr = (ctypes.c_void_p * len(chains))(*[c.handle for c in chains])
    ctx.check(ctx._lib.gingr_update_batch(arr, len(chains), int(iters), int(probabilistic), int(seed)))


def chain_range(n_chains: int, nranks: int, rank: int) -> Tuple[int, int]:
    """(first, count) of the chains rank `rank` runs when n_chains independent chains are divided over nranks processes
    (SURVEY.md 8e: replicas only, no collective).  Chain k always uses seed + k, whichever rank runs it, so the division
    does not change any chain."""
    return shard_range(n_chains, nranks, rank)


def mcmc_batch(chains: Sequence[GingrAlgorithm], iters: int, seed: int = 0):
    """`iters` MH steps of every chain (independent chains on one ctx; gingr_mcmc_batch); chain k uses seed + k.  One batched
    kernel sequence per MH step serves all chains (csrc/batch.cuh); the chains are the chains solo runs with the same seeds
    produce, up to the summation order of a chain's Gram partials when many chains share the GPU."""
    ctx = chains[0].ctx
    arr = (ctypes.c_void_p * len(chains))(*[c.handle for c in chains])
    ctx.check(ctx._lib.gingr_mcmc_batch(arr, len(chains), int(iters), int(seed)))


@dataclass(frozen=True)
class SampleCollection:
    """Which chain states are collected (LogHelper.samplesFromLog, LogHelper.scala:29-43, with its defaults): state i (0 =
    the start state, i >= 1 = the state after the i-th MH step) when i >= burnIn, (i - burnIn) % takeEveryN == 0 and
    i < total, unless state i - 1 ended the chain with a ModelFlexibilityError.  takeEveryN = 0: no collection."""
    burnIn: int = 0
    takeEveryN: int = 50
    total: int = 100


@dataclass
class SampleStatistics:
    """Per-vertex statistics of collected chain states (gingr_mcmc_samples): count, mean fit [M, 3], covariance [M, 3, 3]
    (1 / (count - 1) normalisation; NaN below 2 samples), mean of the sample's unit vertex normals [M, 3] (None without
    model triangles).  The maps of PosteriorHelper (PosteriorHelper.scala:31-79) are closed forms of these."""
    count: int
    mean: np.ndarray
    cov: np.ndarray
    normal: Optional[np.ndarray]

    def distanceMapTotal(self) -> np.ndarray:
        """PosteriorHelper.computeDistanceMapFromMeshesTotal (:31-53): the trace of the per-vertex covariance."""
        return np.trace(self.cov, axis1=1, axis2=2).copy()

    def distanceMapNormal(self, reference=None, triangles=None, sumNormals: bool = True) -> np.ndarray:
        """PosteriorHelper.computeDistanceMapFromMeshesNormal (:55-79): nu^T cov nu with nu the mean of the sample normals
        (sumNormals, not renormalised) or the unit vertex normal of the reference mesh (reference points and triangles)."""
        if sumNormals:
            if self.normal is None:
                raise ValueError("no sample normals: the model has no triangles")
            nu = self.normal
        else:
            if reference is None or triangles is None:
                raise ValueError("sumNormals = False needs the reference points and triangles")
            from .helper import vertex_normals
            nu = vertex_normals(reference, triangles)
        return np.einsum("mi,mij,mj->m", nu, self.cov, nu)

    def merge(self, other: "SampleStatistics") -> "SampleStatistics":
        """The statistics of both sample sets (Chan et al.'s pairwise update, the formula gingr_mcmc_samples pools chains
        with), e.g. of chains divided over GPUs or processes (chain_range)."""
        na, nb = int(self.count), int(other.count)
        if nb == 0:
            return self
        if na == 0:
            return other
        n = na + nb
        zero = np.zeros((self.mean.shape[0], 3, 3))
        sa = self.cov * float(na - 1) if na > 1 else zero      # one sample: no scatter
        sb = other.cov * float(nb - 1) if nb > 1 else zero
        d = other.mean - self.mean
        mean = self.mean + d * (float(nb) / float(n))
        scatter = (sa + sb) + d[:, :, None] * d[:, None, :] * (float(na) * float(nb) / float(n))
        normal = None
        if self.normal is not None and other.normal is not None:
            normal = (self.normal * float(na) + other.normal * float(nb)) / float(n)
        return SampleStatistics(n, mean, scatter / float(n - 1), normal)


def sample_statistics(chains: Sequence[GingrAlgorithm]) -> SampleStatistics:
    """The collected statistics of the chains (collectSamples), pooled on the device in the order of `chains`; the chains
    share one ctx and one model."""
    ctx, model = chains[0].ctx, chains[0].model
    arr = (ctypes.c_void_p * len(chains))(*[c.handle for c in chains])
    count = ctypes.c_int64()
    ctx.check(ctx._lib.gingr_mcmc_samples(arr, len(chains), ctypes.byref(count), None, None, None))
    n = int(count.value)
    mean = np.empty((model.M, 3))
    cov = np.full((model.M, 3, 3), np.nan)
    normal = np.empty((model.M, 3)) if model.T > 0 else None
    ctx.check(ctx._lib.gingr_mcmc_samples(arr, len(chains), None, nat.as_dp(mean), nat.as_dp(cov) if n >= 2 else None,
                                          nat.as_dp(normal)))
    return SampleStatistics(n, mean, cov, normal)


@dataclass
class ProbabilisticSettings:
    """ProbabilisticSettings(IndependentPoints(state, uncertainty, mode, evaluatedPoints), randomMixture)
    (GingrAlgorithm.scala:40-50, sampling/Evaluator.scala:43-60) with the proposal widths of Generator.DefaultRandom
    (sampling/Generator.scala:27-83).  modelPointIds / targetPointIds stand in for the decimation of
    numberOfPointsForComparison (None: all points)."""
    uncertainty: float = 1.0
    mode: int = EVAL_MODEL_TO_TARGET
    randomMixture: float = 0.5
    modelPointIds: Optional[np.ndarray] = None
    targetPointIds: Optional[np.ndarray] = None
    rotationSdev: Tuple[float, float, float] = (0.01, 0.01, 0.01)      # yaw, pitch, roll
    translationSdev: Tuple[float, float, float] = (0.1, 0.1, 0.1)
    shapeSteps: Tuple[float, float, float] = (1.0, 0.1, 0.01)

    def to_pod(self) -> GingrMcmcSettings:
        p = GingrMcmcSettings()
        p.random_mixture = float(self.randomMixture)
        p.uncertainty = float(self.uncertainty)
        p.evaluation_mode = int(self.mode)
        for k in range(3):
            p.rot_sdev[k] = float(self.rotationSdev[k])
            p.trans_sdev[k] = float(self.translationSdev[k])
            p.shape_sdev[k] = float(self.shapeSteps[k])
        return p


def _scala_double(x: float) -> str:
    """Double.toString as the JVM prints it for the magnitudes kernel parameters take (1e-3 <= |x| < 1e7: plain decimal
    with at least one fraction digit, which is Python's repr)."""
    return repr(float(x))


@dataclass(frozen=True)
class GaussKernel:
    """simple/SimpleModels.scala:37-40."""
    scaling: float
    sigma: float
    name = "Gauss"

    @property
    def printpars(self) -> str:
        return _scala_double(self.scaling) + "_" + _scala_double(self.sigma)


@dataclass(frozen=True)
class GaussSymKernel:
    """The mirror-symmetric Gaussian kernel about x = 0 (Model.gaussianSymmetric) with one (scaling, sigma).  The
    reference's own name for this selector is not known here: the name "GaussSym", and with it the cache file name
    <name>_dec-<d>_GaussSym_<scaling>_<sigma>.h5.json, are this project's."""
    scaling: float
    sigma: float
    name = "GaussSym"

    @property
    def printpars(self) -> str:
        return _scala_double(self.scaling) + "_" + _scala_double(self.sigma)


@dataclass(frozen=True)
class InvLapKernel:
    """The inverse-Laplacian look-up kernel (Model.inverseLaplacian) with its (scaling, gamma).  The name "InvLap", and
    with it the cache file name <name>_dec-<d>_InvLap_<scaling>_<gamma>.h5.json, are this project's."""
    scaling: float
    gamma: float
    name = "InvLap"

    @property
    def printpars(self) -> str:
        return _scala_double(self.scaling) + "_" + _scala_double(self.gamma)


@dataclass(frozen=True)
class GaussMixKernel:
    """simple/SimpleModels.scala:41-44 (AutomaticGaussian)."""
    name = "GaussMix"
    printpars = ""


class SimpleTriangleModels3D:
    """simple/SimpleModels.scala:54-77 for the Gaussian families (the kernels the demos load: femur Gauss(50, 70), bunny
    Gauss(20, 40), DemoDatasetLoader.scala:113-114, :146-147), the mirror-symmetric Gaussian kernel (GaussSymKernel) and
    the inverse-Laplacian look-up kernel (InvLapKernel).  The dot-product kernels are not on the path SURVEY.md 8 scopes
    and are refused rather than approximated."""

    @staticmethod
    def create(ctx: Context, reference_points, triangles, kernelSelect, relativeTolerance: float = 0.01) -> Model:
        if isinstance(kernelSelect, GaussKernel):
            return Model.gaussianMixture(ctx, reference_points, triangles, [kernelSelect.sigma], [kernelSelect.scaling],
                                         relativeTolerance)
        if isinstance(kernelSelect, GaussSymKernel):
            return Model.gaussianSymmetric(ctx, reference_points, triangles, [kernelSelect.sigma], [kernelSelect.scaling],
                                           relativeTolerance)
        if isinstance(kernelSelect, InvLapKernel):
            return Model.inverseLaplacian(ctx, reference_points, triangles, kernelSelect.scaling, kernelSelect.gamma,
                                          relativeTolerance)
        if isinstance(kernelSelect, GaussMixKernel):
            return Model.automaticGaussian(ctx, reference_points, triangles, relativeTolerance)
        raise NotImplementedError(f"kernel {type(kernelSelect).__name__} is outside the device GPMM builder (Gaussian families, "
                                  "their mirror-symmetric form and the inverse Laplacian only)")


class SimpleRegistrator:
    """Host mirror of api/registration/SimpleRegistrator.scala:34-158 over device handles: run / runDecimated with the
    hand-over of (pose, scale, shape) between resolution levels (examples/DemoMultiResolution.scala:39-47).  The
    decimated reference and target meshes are the caller's, or come from gingr_b200.decimate when point counts are given
    (scalismo's quadric `decimate` lives in scalismo; SURVEY.md 8c states the substitution); the re-referenced model is
    built on the device from the resident basis (Model.newReference)."""

    def __init__(self, ctx: Context, algorithm, config, model: Model, target: Target, evaluatorUncertainty: float = 1.0,
                 evaluationMode: int = EVAL_MODEL_TO_TARGET, logFileFittingParameters: Optional[str] = None,
                 initialModelParameterTransform=None, modelLandmarks=None, targetLandmarks=None,
                 evaluatedPoints: Optional[int] = None):
        """initialModelParameterTransform: (rotation matrix [3, 3], translation [3]) of the TranslationAfterRotation the
        initial pose is taken from (GeneralRegistrationState.scala:143-157); modelLandmarks / targetLandmarks: io.Landmark
        lists, matched by id on the reference of the model a run uses (:43-62, :111-122); evaluatedPoints: the evaluator's
        numberOfPointsForComparison (IndependentPointDistanceEvaluator.scala:39-47)."""
        self.ctx, self.algorithm, self.config, self.model, self.target = ctx, algorithm, config, model, target
        self.evaluatorUncertainty, self.evaluationMode = evaluatorUncertainty, evaluationMode
        self.logFileFittingParameters = logFileFittingParameters
        self.initialModelParameterTransform = initialModelParameterTransform
        self.modelLandmarks, self.targetLandmarks = modelLandmarks, targetLandmarks
        self.evaluatedPoints = evaluatedPoints
        self.jsonLogger = None       # the JSONStateLogger of the last logged probabilistic run (:139)

    def _evaluated_point_ids(self, model: Model, target: Target):
        """The evaluator's point subsets for evaluatedPoints = n.  Kept from the reference: the MODEL ids are those of the
        decimated instance used as ids of the full mesh, i.e. simply the first n ids (IndependentPointDistanceEvaluator
        .scala:46-47, :50).  Substituted: the target points are about n target vertices spread evenly over the target
        (one per occupied cell of a uniform grid, decimate.decimate_points) instead of the vertices of scalismo's quadric
        decimation (SURVEY.md 8c)."""
        if self.evaluatedPoints is None:
            return None, None
        from .decimate import decimate_points
        n = int(self.evaluatedPoints)
        mids = np.arange(min(n, model.M), dtype=np.int32)
        tids = decimate_points(target.points, n).astype(np.int32)
        return mids, tids

    def _run(self, model: Model, target: Target, generalState, globalTransformation, probabilistic, randomMixture, callback,
             seed):
        reg = self.algorithm(self.ctx, model, target, self.config)
        try:
            if self.modelLandmarks and self.targetLandmarks:
                from .io import landmark_correspondences
                pids, pts, covs = landmark_correspondences(self.modelLandmarks, self.targetLandmarks, model.reference)
                if len(pids):
                    reg.setLandmarks(pids, pts, covs)
            if generalState is not None:
                # combineStates (:76-82): clearIteration, status None, then initializeState recomputes sigma2 from the config.
                # The state keeps ITS OWN globalTransformation: the reference ignores the call argument whenever a
                # generalState is given (:93-95, :135-137)
                g = dataclasses.replace(generalState, iteration=0, status=STATUS_NONE)
                st = reg.initializeState(general=g)
            elif self.initialModelParameterTransform is not None:
                rot, trans = self.initialModelParameterTransform
                st = reg.initializeState(globalTransformation=globalTransformation, rotation=rot, translation=trans)
            else:
                st = reg.initializeState(globalTransformation=globalTransformation)
            if probabilistic:
                mids, tids = self._evaluated_point_ids(model, target)
                settings = ProbabilisticSettings(uncertainty=self.evaluatorUncertainty, mode=self.evaluationMode,
                                                 randomMixture=randomMixture, modelPointIds=mids, targetPointIds=tids)
                # The reference always attaches a JSONStateLogger here (:139-145).  The log costs one host round trip per
                # MH step, so it is kept only when somebody reads it: a log file or a callback was asked for; otherwise
                # the whole chain stays on the device.
                if self.logFileFittingParameters is not None or callback is not None:
                    from .io import JSONStateLogger
                    self.jsonLogger = JSONStateLogger(path=self.logFileFittingParameters)
                    final = reg.runProbabilistic(st, settings, seed=seed, acceptRejectLogger=self.jsonLogger, callBackLogger=callback)
                    if self.logFileFittingParameters is not None:
                        self.jsonLogger.write()                                                    # writeLog (:150)
                else:
                    final = reg.runProbabilistic(st, settings, seed=seed)
            else:
                final = reg.run(st, callback)
        finally:
            reg.close()
        # "Final registration with full resolution meshes" (:152-157): the fit is re-evaluated on the full model
        return dataclasses.replace(final, fit=self.model.instance(final.modelParameters))

    def run(self, generalState=None, globalTransformation: int = RIGID_TRANSFORMS, probabilistic: bool = False,
            randomMixture: float = 0.5, callback=None, seed: int = 0) -> GeneralRegistrationState:
        return self._run(self.model, self.target, generalState, globalTransformation, probabilistic, randomMixture, callback, seed)

    def runDecimated(self, decimatedReference, decimatedTarget, generalState=None,
                     globalTransformation: int = RIGID_TRANSFORMS, probabilistic: bool = False, randomMixture: float = 0.5,
                     callback=None, seed: int = 0) -> GeneralRegistrationState:
        """decimateState + run (:58-70, :84-106).  decimatedReference / decimatedTarget: either the number of points, as in
        the reference (runDecimated(modelPoints, targetPoints, ...)) -- the meshes are then decimated by
        gingr_b200.decimate (shortest-edge collapse, the stated stand-in for scalismo's quadric decimate) -- or the
        (points, triangles) of meshes the caller decimated."""
        if isinstance(decimatedReference, (int, np.integer)):
            from .decimate import decimate
            decimatedReference = decimate(self.model.reference, self.model.triangles, int(decimatedReference))
        if isinstance(decimatedTarget, (int, np.integer)):
            from .decimate import decimate
            decimatedTarget = decimate(self.target.points, self.target.triangles, int(decimatedTarget))
        dm = self.model.newReference(*decimatedReference)
        dt = Target(self.ctx, *decimatedTarget)
        try:
            return self._run(dm, dt, generalState, globalTransformation, probabilistic, randomMixture, callback, seed)
        finally:
            dm.close()
            dt.close()


class GingrInterface:
    """simple/GingrInterface.scala:20-64: the model / target / landmarks / evaluator options once, then .CPD(config) or
    .ICP(config) -> SimpleRegistrator."""

    def __init__(self, ctx: Context, model: Model, target: Target, initialModelParameterTransform=None, modelLandmarks=None,
                 targetLandmarks=None, evaluatorUncertainty: float = 1.0, evaluatedPoints: Optional[int] = None,
                 evaluationMode: int = EVAL_MODEL_TO_TARGET, logFileFittingParameters: Optional[str] = None):
        self.ctx, self.model, self.target = ctx, model, target
        self._options = dict(evaluatorUncertainty=evaluatorUncertainty, evaluationMode=evaluationMode,
                             logFileFittingParameters=logFileFittingParameters,
                             initialModelParameterTransform=initialModelParameterTransform, modelLandmarks=modelLandmarks,
                             targetLandmarks=targetLandmarks, evaluatedPoints=evaluatedPoints)

    def CPD(self, config: Optional["CpdConfiguration"] = None) -> "SimpleRegistrator":
        return SimpleRegistrator(self.ctx, CpdRegistration, config or CpdConfiguration(), self.model, self.target, **self._options)

    def ICP(self, config: Optional["IcpConfiguration"] = None) -> "SimpleRegistrator":
        return SimpleRegistrator(self.ctx, IcpRegistration, config or IcpConfiguration(), self.model, self.target, **self._options)


class CpdRegistration(GingrAlgorithm):
    """registration/config/CPD.scala:117-160"""
    name = "CPD"

    def __init__(self, ctx, model, target, config: Optional[CpdConfiguration] = None):
        super().__init__(ctx, model, target, config or CpdConfiguration())


class IcpRegistration(GingrAlgorithm):
    """registration/config/ICP.scala:84-110"""
    name = "ICP"

    def __init__(self, ctx, model, target, config: Optional[IcpConfiguration] = None):
        super().__init__(ctx, model, target, config or IcpConfiguration())


class BcpdRegistration(GingrAlgorithm):
    """GingrAlgorithm with BCPD correspondences (BcpdConfiguration).  Besides the GeneralRegistrationState the registration
    keeps per-vertex mixing weights and posterior variances on the device: creation and initializeState set them to 1 / M
    and the prior variance, every committed update advances them (bcpdState() reads them back).  Deterministic updates on one GPU
    only: the probabilistic calls raise GingrError with GINGR_ERR_UNSUPPORTED."""
    name = "BCPD"

    def __init__(self, ctx, model, target, config: Optional[BcpdConfiguration] = None):
        super().__init__(ctx, model, target, config or BcpdConfiguration())
        self.ctx.check(self.ctx._lib.gingr_registration_set_bcpd(self.handle, float(self.config.kappa)))

    def bcpdState(self) -> Tuple[np.ndarray, np.ndarray]:
        """(alpha[M], Sigma[M]): the mixing weights and per-vertex posterior variances the next update's E-step uses."""
        alpha, sigma = np.empty(self.model.M), np.empty(self.model.M)
        self.ctx.check(self.ctx._lib.gingr_bcpd_state_download(self.handle, nat.as_dp(alpha), nat.as_dp(sigma)))
        return alpha, sigma
