"""
oracle.py -- CPU restatement (numpy + the C loops in gingr_oracle.c) of GiNGR's per-iteration
hot path `GingrAlgorithm.update` and the functions it calls.

THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / `--impl reference` legs may import it.  Nothing under gingr_b200/
imports it and the product has no CPU fallback.

PARITY UNPINNED.  The reference (unibas-gravis/GiNGR, Scala 3) has no tests that pin numbers
(src/test/scala/DummyTest.scala.scala:1-3), cannot be compiled here (no JVM/sbt, and its
arithmetic lives in the un-vendored dependency `ch.unibas.cs.gravis::scalismo:1.0-RC1`
(build.sbt:40) + Breeze).  This file restates the reference's own Scala sources line by line
(citations are relative to /root/reference/src/main/scala/gingr/) and restates scalismo's
published algorithms where the reference calls into them; such lines are tagged
[scalismo-recalled] (see SURVEY.md Appendix A).

Conventions: points are float64 arrays [n,3]; GPMM basis is [3M, r] with row 3*pid+d
(Breeze column-major on the JVM; numpy layout is irrelevant to the arithmetic).
"""
from __future__ import annotations

import ctypes
import dataclasses
import math
import os
import subprocess
from dataclasses import dataclass, field
from typing import Optional, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "libgingr_oracle.so")
_lib = None

c_dp = ctypes.POINTER(ctypes.c_double)
c_ip = ctypes.POINTER(ctypes.c_int32)
c_bp = ctypes.POINTER(ctypes.c_uint8)


def build(force: bool = False) -> str:
    """Compile gingr_oracle.c -> oracle/_build/libgingr_oracle.so (gcc, OpenMP, no FMA contraction)."""
    src = os.path.join(_HERE, "gingr_oracle.c")
    if (not force) and os.path.exists(_LIB_PATH) and os.path.getmtime(_LIB_PATH) >= os.path.getmtime(src):
        return _LIB_PATH
    os.makedirs(os.path.dirname(_LIB_PATH), exist_ok=True)
    cmd = ["gcc", "-O2", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC",
           "-fvisibility=hidden", "-o", _LIB_PATH, src, "-lm"]
    subprocess.check_call(cmd)
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        _lib = ctypes.CDLL(_LIB_PATH)
        _lib.oracle_cpd_initial_sigma2.restype = ctypes.c_double
        _lib.oracle_num_threads.restype = ctypes.c_int
    return _lib


def _d(a):
    return a.ctypes.data_as(c_dp)


def _i(a):
    return a.ctypes.data_as(c_ip)


def _c(a, dtype=np.float64):
    return np.ascontiguousarray(a, dtype=dtype)


def num_threads() -> int:
    return int(lib().oracle_num_threads())


def set_num_threads(n: int) -> None:
    lib().oracle_set_num_threads(int(n))


# ---------------------------------------------------------------------------------------------
# K1: CPD / BCPD E-step
# ---------------------------------------------------------------------------------------------
def cpd_P(fit, target, sigma2, w):
    """CpdRegistrationState.P, literal, materialised M x N.  registration/config/CPD.scala:54-75"""
    fit, target = _c(fit), _c(target)
    M, N = fit.shape[0], target.shape[0]
    P = np.empty((M, N))
    lib().oracle_cpd_P(M, N, _d(fit), _d(target), ctypes.c_double(sigma2), ctypes.c_double(w), _d(P))
    return P


def P_reductions(P, target):
    """P1 = sum(P,Axis._1), Pt1 = sum(P,Axis._0), PX = P*X.  CPD.scala:36, :139-145"""
    P, target = _c(P), _c(target)
    M, N = P.shape
    P1, Pt1, PX = np.empty(M), np.empty(N), np.empty((M, 3))
    lib().oracle_P_reductions(M, N, _d(P), _d(target), _d(P1), _d(Pt1), _d(PX))
    return P1, Pt1, PX


def cpd_correspondence(P, fit, target):
    """CPDCorrespondence.estimate, literal.  CPD.scala:32-49"""
    P, fit, target = _c(P), _c(fit), _c(target)
    M, N = P.shape
    td = np.empty((M, 3))
    lib().oracle_cpd_correspondence(M, N, _d(P), _d(fit), _d(target), _d(td))
    return td


def cpd_estep(fit, target, sigma2, w, fast=False):
    """Streaming E-step (P never stored): P1[M], Pt1[N], PX[M,3].  Same formulas as cpd_P."""
    fit, target = _c(fit), _c(target)
    M, N = fit.shape[0], target.shape[0]
    P1, Pt1, PX = np.empty(M), np.empty(N), np.empty((M, 3))
    if fast:
        lib().oracle_cpd_estep_fast(M, N, _d(fit), _d(target), ctypes.c_double(sigma2), ctypes.c_double(w),
                                    _d(P1), _d(Pt1), _d(PX))
    else:
        lib().oracle_cpd_estep_stream(M, N, _d(fit), _d(target), ctypes.c_double(sigma2), ctypes.c_double(w),
                                      _d(P1), _d(Pt1), _d(PX), None)
    return P1, Pt1, PX


def cpd_initial_sigma2(reference_pts, target):
    """computeInitialSigma2.  CPD.scala:81-90 (over model.mean points, CPD.scala:95)"""
    a, b = _c(reference_pts), _c(target)
    return float(lib().oracle_cpd_initial_sigma2(a.shape[0], b.shape[0], _d(a), _d(b)))


def cpd_sigma2_update(P1, Pt1, PX, target, TY):
    """CpdRegistration.updateSigma2.  CPD.scala:133-147
    xPx = Pt1 . rowsum(X*X) ; yPy = P1 . rowsum(TY*TY) ; trPXY = sum(TY * (P X)) ; /(Np*3)"""
    X = np.asarray(target)
    Np = float(np.sum(P1))
    xPx = float(np.dot(Pt1, np.sum(X * X, axis=1)))
    yPy = float(np.dot(P1, np.sum(TY * TY, axis=1)))
    trPXY = float(np.sum(TY * PX))
    return (xPx - 2 * trPXY + yPy) / (Np * 3.0)


def bcpd_P(y, x, sigma_mm, alpha, sigma2, s, w):
    """BCPD.computeP literal (quirks kept).  other/algorithms/cpd/BCPD.scala:167-184"""
    y, x, sigma_mm, alpha = _c(y), _c(x), _c(sigma_mm), _c(alpha)
    M, N = y.shape[0], x.shape[0]
    P = np.empty((M, N))
    lib().oracle_bcpd_P(M, N, _d(y), _d(x), _d(sigma_mm), _d(alpha), ctypes.c_double(sigma2), ctypes.c_double(s),
                        ctypes.c_double(w), _d(P))
    return P


def bcpd_estep(y, x, sigma_mm, alpha, sigma2, s, w):
    """BCPD.Iteration's P-reductions.  BCPD.scala:200-209: nu = P 1, nu' = P^T 1, Nhat = sum nu',
    xhat = pinv(diag(nu (x) 1_3)) (P (x) I_3) X  (= (P X)_m / nu_m, 0 where nu_m == 0)."""
    P = bcpd_P(y, x, sigma_mm, alpha, sigma2, s, w)
    nu, nup, PX = P_reductions(P, x)
    nhat = float(np.sum(nup))
    inv = np.where(nu != 0.0, 1.0 / np.where(nu != 0.0, nu, 1.0), 0.0)
    return nu, nup, nhat, PX * inv[:, None]


# ---------------------------------------------------------------------------------------------
# K2: closest point
# ---------------------------------------------------------------------------------------------
def nearest_vertex(queries, points):
    """findClosestPoint: O(MN) FP64 scan, ties -> lowest index.  ClosestPointRegistrator.scala:141"""
    q, p = _c(queries), _c(points)
    idx = np.empty(q.shape[0], dtype=np.int32)
    d2 = np.empty(q.shape[0])
    lib().oracle_nearest_vertex(q.shape[0], _d(q), p.shape[0], _d(p), _i(idx), _d(d2))
    return idx, d2


def closest_on_surface(queries, verts, tri):
    """closestPointOnSurface [scalismo-recalled A6]: exact nearest point over all triangles."""
    q, v, t = _c(queries), _c(verts), _c(tri, np.int32)
    cp = np.empty((q.shape[0], 3))
    d2 = np.empty(q.shape[0])
    ti = np.empty(q.shape[0], dtype=np.int32)
    lib().oracle_closest_on_surface(q.shape[0], _d(q), v.shape[0], _d(v), t.shape[0], _i(t), _d(cp), _d(d2), _i(ti))
    return cp, d2, ti


def vertex_normals(verts, tri):
    """mesh.vertexNormals [scalismo-recalled A6]"""
    v, t = _c(verts), _c(tri, np.int32)
    n = np.empty_like(v)
    lib().oracle_vertex_normals(v.shape[0], _d(v), t.shape[0], _i(t), _d(n))
    return n


def boundary_vertices(n_verts, tri):
    """mesh.operations.pointIsOnBoundary for every vertex [scalismo-recalled A6]"""
    t = _c(tri, np.int32)
    out = np.zeros(n_verts, dtype=np.uint8)
    lib().oracle_boundary_vertices(int(n_verts), t.shape[0], _i(t), out.ctypes.data_as(c_bp))
    return out.astype(bool)


def line_mesh_min_dist(p, direction, verts, tri, skip_incident=True):
    """min distance from p to intersections != p of the infinite line p + s*dir with the mesh.
    skip_incident: query i is vertex i of the mesh; triangles incident to it are skipped."""
    p, d, v, t = _c(p), _c(direction), _c(verts), _c(tri, np.int32)
    out = np.empty(p.shape[0])
    lib().oracle_line_mesh_min_dist(p.shape[0], _d(p), _d(d), v.shape[0], _d(v), t.shape[0], _i(t),
                                    int(bool(skip_incident)), _d(out))
    return out


def line_mesh_nearest(p, direction, verts, tri):
    """nearest intersection != p of the infinite line p + s*dir with a mesh (the along-normal flavour):
    (distance, hit point); distance = inf and hit = p when the line misses the mesh."""
    p, d, v, t = _c(p), _c(direction), _c(verts), _c(tri, np.int32)
    dist = np.empty(p.shape[0])
    hit = np.empty_like(p)
    lib().oracle_line_mesh_nearest(p.shape[0], _d(p), _d(d), v.shape[0], _d(v), t.shape[0], _i(t), _d(dist), _d(hit))
    return dist, hit


METHOD_TRIANGULAR, METHOD_ALONG_NORMAL, METHOD_POINTCLOUD = 0, 1, 2


def closest_point_correspondence(method, template_v, template_tri, target_v, target_tri):
    """closestPointCorrespondence of the three flavours -> (cp[M,3], w[M], mean distance).
    ClosestPointRegistrator.scala:74-96 (triangular), :98-131 (along normal), :133-160 (point cloud)."""
    template_v, target_v = _c(template_v), _c(target_v)
    M = template_v.shape[0]
    if method == METHOD_POINTCLOUD:
        idx, d2 = nearest_vertex(template_v, target_v)  # :141
        return target_v[idx].copy(), np.ones(M), float(np.sum(np.sqrt(d2)) / M), idx
    tgt_boundary = boundary_vertices(target_v.shape[0], target_tri)
    n_tpl = vertex_normals(template_v, template_tri)
    n_tgt = vertex_normals(target_v, target_tri)
    if method == METHOD_TRIANGULAR:
        cp, d2, _ = closest_on_surface(template_v, target_v, target_tri)  # :82
        idx, _ = nearest_vertex(cp, target_v)  # :83
        w = np.ones(M)
        w[tgt_boundary[idx]] = 0.0  # :85
        nt = n_tgt[idx]
        opp = (n_tpl[:, 0] * nt[:, 0] + n_tpl[:, 1] * nt[:, 1] + n_tpl[:, 2] * nt[:, 2]) < 0  # :86-88
        w[opp] = 0.0
        v = template_v - cp  # :63-64
        md = line_mesh_min_dist(template_v, v, template_v, template_tri)  # :65-70
        vnorm = np.sqrt(v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1] + v[:, 2] * v[:, 2])
        w[md < vnorm] = 0.0  # :71, :89
        return cp, w, float(np.sum(np.sqrt(d2)) / M), idx
    # ClosestPointAlongNormalTriangleMesh3D  :98-131
    dist, hit = line_mesh_nearest(template_v, n_tpl, target_v, target_tri)        # :105-110
    has = np.isfinite(dist)
    idx, _ = nearest_vertex(hit, target_v)                                         # :113
    w = np.ones(M)
    w[tgt_boundary[idx]] = 0.0                                                     # :115
    nt = n_tgt[idx]
    opp = (n_tpl[:, 0] * nt[:, 0] + n_tpl[:, 1] * nt[:, 1] + n_tpl[:, 2] * nt[:, 2]) < 0   # :116-122
    w[opp] = 0.0
    v = template_v - hit
    md = line_mesh_min_dist(template_v, v, template_v, template_tri)               # :123
    vnorm = np.sqrt(v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1] + v[:, 2] * v[:, 2])
    w[md < vnorm] = 0.0
    w[~has] = 0.0                                                                  # :127 (p, 0.0)
    cp = np.where(has[:, None], hit, template_v)
    return cp, w, float(np.sum(np.where(has, dist, 0.0)) / M), idx                 # :128


def icp_correspondence(method, reverse, fit_v, fit_tri, target_v, target_tri):
    """ICPCorrespondence.estimate -> (pids[n], points[n,3]) with only w == 1 kept.  ICP.scala:37-51"""
    if not reverse:
        cp, w, _, _ = closest_point_correspondence(method, fit_v, fit_tri, target_v, target_tri)
        keep = w == 1.0
        return np.nonzero(keep)[0].astype(np.int32), cp[keep]
    # closestPointCorrespondenceReversal  ClosestPointRegistrator.scala:34-45
    cp, w, _, _ = closest_point_correspondence(method, target_v, target_tri, fit_v, fit_tri)
    tid, _ = nearest_vertex(cp, fit_v)  # template.pointSet.findClosestPoint(p).id
    keep = w == 1.0
    return tid[keep].astype(np.int32), _c(target_v)[keep]


# ---------------------------------------------------------------------------------------------
# scalismo pieces on the path [scalismo-recalled], SURVEY.md Appendix A
# ---------------------------------------------------------------------------------------------
def euler_to_matrix(phi, theta, psi):
    """scalismo Rotation(phi, theta, psi, center): R = Rz(phi) Ry(theta) Rx(psi)  [scalismo-recalled A4]"""
    cph, sph = math.cos(phi), math.sin(phi)
    cth, sth = math.cos(theta), math.sin(theta)
    cps, sps = math.cos(psi), math.sin(psi)
    return np.array([
        [cth * cph, sps * sth * cph - cps * sph, sps * sph + cps * sth * cph],
        [cth * sph, cps * cph + sps * sth * sph, cps * sth * sph - sps * cph],
        [-sth, sps * cth, cps * cth],
    ])


def matrix_to_euler(R):
    """RotationSpace3D.rotMatrixToEulerAngles (Slabaugh)  [scalismo-recalled A4];
    used at GeneralRegistrationState.scala:83-87, :143."""
    if abs(abs(R[2, 0]) - 1) > 0.0001:
        theta = math.asin(-R[2, 0])
        ct = math.cos(theta)
        psi = math.atan2(R[2, 1] / ct, R[2, 2] / ct)
        phi = math.atan2(R[1, 0] / ct, R[0, 0] / ct)
        return phi, theta, psi
    phi = 0.0
    if abs(R[2, 0] + 1) < 0.0001:
        theta = math.pi / 2.0
        psi = phi + math.atan2(R[0, 1], R[0, 2])
    else:
        theta = -math.pi / 2.0
        psi = -phi + math.atan2(-R[0, 1], -R[0, 2])
    return phi, theta, psi


def breeze_pinv(A):
    """breeze.linalg.pinv: SVD, reciprocal of every non-zero singular value, no tolerance cut."""
    U, s, Vt = np.linalg.svd(A)
    si = np.where(s == 0.0, 0.0, 1.0 / np.where(s == 0.0, 1.0, s))
    return (Vt.T * si) @ U.T


def umeyama(X, Y, similarity):
    """LandmarkRegistration.{rigid,similarity}3DLandmarkRegistration about center = origin
    [scalismo-recalled A4]; called from GingrAlgorithm.scala:260-279.  x -> c R x + t."""
    n = X.shape[0]
    mu_x = X.mean(axis=0)
    mu_y = Y.mean(axis=0)
    Xc, Yc = X - mu_x, Y - mu_y
    sigma2_x = float(np.sum(Xc * Xc) / n)
    Sxy = (Yc.T @ Xc) / n
    U, D, Vt = np.linalg.svd(Sxy)
    # The reflection sign is det U det V (Kabsch / Umeyama), where the scalismo rule reads sign det Sxy.  The two agree
    # whenever Sxy has full rank.  At rank 2 (planar shapes) det Sxy is +-0 or rounding noise and the literal rule's result
    # depends on the SVD's sign conventions: half the time U V^T is a reflection.  det U det V makes it a rotation always.
    S = np.eye(3)
    if np.linalg.det(U) * np.linalg.det(Vt) < 0:
        S[2, 2] = -1.0
    R = U @ S @ Vt
    c = float(np.trace(np.diag(D) @ S) / sigma2_x) if similarity else 1.0
    t = mu_y - c * (R @ mu_x)
    # the rotation is returned as Euler angles and rebuilt from them
    R = euler_to_matrix(*matrix_to_euler(R))
    return R, t, c


# ---------------------------------------------------------------------------------------------
# GPMM (scalismo PointDistributionModel / DiscreteLowRankGaussianProcess) [scalismo-recalled A1-A3]
# ---------------------------------------------------------------------------------------------
@dataclass
class Gpmm:
    ref: np.ndarray          # [M,3]  reference mesh points
    mean: np.ndarray         # [3M]   meanVector
    basis: np.ndarray        # [3M,r] basisMatrix
    variance: np.ndarray     # [r]    lambda
    tri: Optional[np.ndarray] = None  # [T,3] int32 triangles of the reference mesh

    @property
    def M(self):
        return self.ref.shape[0]

    @property
    def rank(self):
        return self.variance.shape[0]

    def instance(self, alpha):
        """instance(alpha) = ref + reshape(mean + basis (sqrt(lambda) * alpha))   [A1]"""
        return self.ref + (self.mean + self.basis @ (np.sqrt(self.variance) * alpha)).reshape(-1, 3)

    def transform(self, R, t):
        """PointDistributionModel.transform(rigid), rotation centre = origin   [A2]
        ref' = R ref + t ; mean'_i = R mean_i ; basis'_{i,k} = R basis_{i,k} ; lambda unchanged."""
        ref = self.ref @ R.T + t
        mean = (self.mean.reshape(-1, 3) @ R.T).reshape(-1)
        B = self.basis.reshape(self.M, 3, self.rank)
        basis = np.einsum("ab,mbk->mak", R, B).reshape(3 * self.M, self.rank)
        return Gpmm(ref, mean, basis, self.variance, self.tri)

    def new_reference(self, new_ref, new_tri=None) -> "Gpmm":
        """model.newReference(newRef, NearestNeighborInterpolator()) [scalismo-recalled A7]: mean deformation and basis
        rows of the nearest old reference point (lowest index on ties).  SimpleRegistrator.scala:90-92"""
        idx, _ = nearest_vertex(new_ref, self.ref)
        rows = (3 * idx.astype(np.int64)[:, None] + np.arange(3)[None, :]).reshape(-1)
        return Gpmm(_c(new_ref), self.mean[rows].copy(), self.basis[rows, :].copy(), self.variance, new_tri)

    def _regression(self, pids, values, cov_inv):
        """genericRegressionComputations  [A3].  values = y_i (displacements), cov_inv[n,3,3]."""
        pids = np.asarray(pids, dtype=np.int64)
        rows = (3 * pids[:, None] + np.arange(3)[None, :]).reshape(-1)
        Q = self.basis[rows, :] * np.sqrt(self.variance)[None, :]
        m = self.mean[rows]
        n = pids.shape[0]
        QtL = np.einsum("nak,nab->kbn", Q.reshape(n, 3, -1), cov_inv).transpose(0, 2, 1).reshape(self.rank, 3 * n)
        Mx = QtL @ Q + np.eye(self.rank)
        self._last_Mx = Mx   # kept for posterior sampling (test infrastructure convenience)
        Minv = breeze_pinv(Mx)
        y = np.asarray(values).reshape(-1)
        return Minv, QtL, y, m

    def posterior_coefficients(self, pids, points, cov):
        """coefficient vector of PointDistributionModel.posterior(obs)'s mean  [A3].
        cov: [n,3,3] observation covariances.  Raises on non-finite input like breeze inv/svd."""
        cov = np.asarray(cov)
        if not np.all(np.isfinite(cov)):
            raise FloatingPointError("non-finite observation covariance")
        cov_inv = np.linalg.inv(cov)
        values = np.asarray(points) - self.ref[np.asarray(pids)]
        Minv, QtL, y, m = self._regression(pids, values, cov_inv)
        if not (np.all(np.isfinite(Minv)) and np.all(np.isfinite(QtL))):
            raise FloatingPointError("non-finite regression")
        c = (Minv @ QtL) @ (y - m)
        return c, Minv

    def coefficients(self, mesh_pts):
        """PointDistributionModel.coefficients(mesh): all M points, noise 1e-5 I3  [A3]"""
        M = self.M
        cov_inv = np.broadcast_to(np.eye(3) / 1e-5, (M, 3, 3))
        values = np.asarray(mesh_pts) - self.ref
        Minv, QtL, y, m = self._regression(np.arange(M), values, cov_inv)
        c = (Minv @ QtL) @ (y - m)
        if not np.all(np.isfinite(c)):
            raise FloatingPointError("non-finite coefficients")
        return c


# ---------------------------------------------------------------------------------------------
# State / config records (layout of api/GeneralRegistrationState.scala:28-41,
# api/ModelFittingParameters.scala:31-74)
# ---------------------------------------------------------------------------------------------
STATUS_NONE, STATUS_MAX_ITERATION, STATUS_CONVERGED, STATUS_MODEL_FLEXIBILITY_ERROR = 0, 1, 2, 3  # FittingStatuses.scala:20-23
SIMILARITY_TRANSFORMS, RIGID_TRANSFORMS, NO_TRANSFORMS = 0, 1, 2  # GlobalTranformationType.scala:20-24


@dataclass
class Params:
    """ModelFittingParameters: scale, pose (translation, Euler rotation about centre), shape."""
    scale: float
    translation: np.ndarray
    euler: Tuple[float, float, float]
    shape: np.ndarray

    def rotation_matrix(self):
        return euler_to_matrix(*self.euler)


@dataclass
class Landmarks:
    """GeneralRegistrationState.landmarkCorrespondences (GeneralRegistrationState.scala:43-62):
    (closest reference vertex id, target landmark point, model landmark covariance or I3)."""
    pids: np.ndarray   # [L] int
    points: np.ndarray  # [L,3]
    cov: np.ndarray    # [L,3,3]


@dataclass
class State:
    model: Gpmm
    params: Params
    target: np.ndarray                 # [N,3]
    target_tri: Optional[np.ndarray]
    fit: np.ndarray                    # [M,3]
    sigma2: float = 1.0
    global_transformation: int = RIGID_TRANSFORMS
    step_length: float = 1.0
    iteration: int = 0
    status: int = STATUS_NONE
    landmarks: Optional[Landmarks] = None


def model_instance_shape_pose_scale(model: Gpmm, p: Params):
    """ModelFittingParameters.modelInstanceShapePoseScale: s * (R instance(alpha) + t).
    ModelFittingParameters.scala:130-143"""
    return (model.instance(p.shape) @ p.rotation_matrix().T + p.translation) * p.scale


def initial_state(model: Gpmm, target, target_tri=None, global_transformation=RIGID_TRANSFORMS,
                  R0=None, t0=None, landmarks=None) -> State:
    """GeneralRegistrationState.apply.  GeneralRegistrationState.scala:136-178"""
    if R0 is not None:
        euler = matrix_to_euler(np.asarray(R0))
        t = np.asarray(t0, dtype=float)
    else:
        euler, t = (0.0, 0.0, 0.0), np.zeros(3)
    p = Params(1.0, t, euler, np.zeros(model.rank))
    fit = model_instance_shape_pose_scale(model, p)
    return State(model, p, _c(target), target_tri, fit, global_transformation=global_transformation,
                 landmarks=landmarks)


@dataclass
class CpdConfig:
    """CpdConfiguration.  CPD.scala:105-115"""
    max_iterations: int = 100
    threshold: float = 1e-10
    use_landmark_correspondence: bool = True
    initial_sigma: Optional[float] = None
    w: float = 0.0
    lam: float = 1.0

    def converged(self, last: State, cur: State):
        return abs(last.sigma2 - cur.sigma2) < self.threshold


@dataclass
class IcpConfig:
    """IcpConfiguration.  ICP.scala:54-66"""
    max_iterations: int = 100
    threshold: float = 1e-10
    use_landmark_correspondence: bool = True
    initial_sigma: float = 100.0
    end_sigma: float = 1.0
    reverse: bool = False
    method: int = METHOD_TRIANGULAR

    @property
    def sigma_step(self):
        return (self.initial_sigma - self.end_sigma) / float(self.max_iterations)

    def converged(self, last, cur):
        return False


class CpdAlgorithm:
    """CpdRegistration + CpdRegistrationState + CPDCorrespondence.  CPD.scala:30-160"""
    name = "CPD"

    def __init__(self, config: CpdConfig, literal: bool = True):
        self.config = config
        self.literal = literal   # literal = materialise P like the reference; else streaming E-step

    def initialize(self, general: State) -> State:
        """CpdRegistrationState.apply.  CPD.scala:92-103"""
        s2 = self.config.initial_sigma
        if s2 is None:
            mean_pts = general.model.instance(np.zeros(general.model.rank))  # model.mean
            s2 = cpd_initial_sigma2(mean_pts, general.target)
        return dataclasses.replace(general, sigma2=float(s2))

    def estep(self, st: State):
        if self.literal:
            P = cpd_P(st.fit, st.target, st.sigma2, self.config.w)
            P1, Pt1, PX = P_reductions(P, st.target)
            td = cpd_correspondence(P, st.fit, st.target)
        else:
            P1, Pt1, PX = cpd_estep(st.fit, st.target, st.sigma2, self.config.w, fast=True)
            td = PX / P1[:, None]
        return P1, Pt1, PX, td

    def observations(self, st: State):
        """getCorrespondence + getUncertainty for every pid.  CPD.scala:32-49, :120-128"""
        P1, Pt1, PX, td = self.estep(st)
        with np.errstate(divide="ignore"):
            var = st.sigma2 * self.config.lam * (1.0 / P1)   # eye(3) * sigma2 * lambda * P1inv(id)
        cov = np.eye(3)[None, :, :] * var[:, None, None]
        st._estep = (P1, Pt1, PX)
        return np.arange(st.model.M, dtype=np.int32), td, cov

    def update_sigma2(self, st: State) -> float:
        """CPD.scala:133-147 -- P and fit are those of the *pre-update* state (SURVEY 3.2 step 7)."""
        P1, Pt1, PX = st._estep
        return cpd_sigma2_update(P1, Pt1, PX, st.target, st.fit)


class IcpAlgorithm:
    """IcpRegistration + ICPCorrespondence.  ICP.scala:37-110"""
    name = "ICP"

    def __init__(self, config: IcpConfig):
        self.config = config

    def initialize(self, general: State) -> State:
        """IcpRegistrationState.apply: sigma2 = config.initialSigma.  ICP.scala:74-86"""
        return dataclasses.replace(general, sigma2=float(self.config.initial_sigma))

    def observations(self, st: State):
        pids, pts = icp_correspondence(self.config.method, self.config.reverse, st.fit, st.model.tri, st.target,
                                       st.target_tri)
        cov = np.eye(3)[None, :, :] * np.full(len(pids), st.sigma2)[:, None, None]   # ICP.scala:90-92
        return pids, pts, cov

    def update_sigma2(self, st: State) -> float:
        """ICP.scala:96-99"""
        return max(st.sigma2 - self.config.sigma_step, self.config.end_sigma)


def compute_posterior_coefficients(algo, st: State):
    """GingrAlgorithm.computePosterior.  api/GingrAlgorithm.scala:281-302.
    Returns (posed model, coefficient vector c of the posterior mean, Minv)."""
    pids, pts, cov = algo.observations(st)
    if algo.config.use_landmark_correspondence and st.landmarks is not None and len(st.landmarks.pids) > 0:
        lm = st.landmarks
        keep = ~np.isin(pids, lm.pids)                                    # :289-293
        pids = np.concatenate([pids[keep], lm.pids.astype(pids.dtype)])   # :294
        pts = np.concatenate([pts[keep], lm.points])
        cov = np.concatenate([cov[keep], lm.cov])
    posed = st.model.transform(st.params.rotation_matrix(), st.params.translation)  # :299
    c, Minv = posed.posterior_coefficients(pids, pts, cov)                # :300
    return posed, c, Minv


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (Salmon et al. 2011), vectorised over numpy uint64 arrays holding 32-bit words."""
    M0, M1, W0, W1, MASK = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85, 0xFFFFFFFF
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & MASK for c in (c0, c1, c2, c3))
    k0, k1 = np.uint64(k0 & MASK), np.uint64(k1 & MASK)
    for _ in range(10):
        p0, p1 = np.uint64(M0) * c0, np.uint64(M1) * c2
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & np.uint64(MASK), p1 >> np.uint64(32), p1 & np.uint64(MASK)
        c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
        k0, k1 = (k0 + np.uint64(W0)) & np.uint64(MASK), (k1 + np.uint64(W1)) & np.uint64(MASK)
    return c0, c1, c2, c3


def standard_normals(r: int, seed: int, iteration: int):
    """z[r] ~ N(0, 1): the stream gingr_update(probabilistic) uses (include/gingr_cuda.h): Philox4x32-10 with
    key = seed, counter = (pair index, iteration, 0, 0), 53-bit uniforms, Box-Muller."""
    npair = (r + 1) // 2
    p = np.arange(npair, dtype=np.uint64)
    zero = np.zeros(npair, dtype=np.uint64)
    x0, x1, x2, x3 = philox4x32_10(p, zero + np.uint64(iteration & 0xFFFFFFFF), zero, zero, seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    u1 = ((x0 >> np.uint64(5)).astype(np.float64) * 67108864.0 + (x1 >> np.uint64(6)).astype(np.float64) + 0.5) / 9007199254740992.0
    u2 = ((x2 >> np.uint64(5)).astype(np.float64) * 67108864.0 + (x3 >> np.uint64(6)).astype(np.float64) + 0.5) / 9007199254740992.0
    rad = np.sqrt(-2.0 * np.log(u1))
    ang = 6.283185307179586476925 * u2
    z = np.empty(2 * npair)
    z[0::2] = rad * np.cos(ang)
    z[1::2] = rad * np.sin(ang)
    return z[:r]


RETRY_COUNTER_INIT = 10  # GingrAlgorithm.scala:69-70


def update(algo, st: State, probabilistic: bool = False, seed: int = 0, counter: Optional[int] = None) -> State:
    """GingrAlgorithm.update, literal.  api/GingrAlgorithm.scala:192-254.  `counter`: second word of the Philox counter
    of the posterior-sample stream (default: the state's iteration; the MH chain passes its step index)."""
    try:
        with np.errstate(all="ignore"):
            posed, c_post, Minv = compute_posterior_coefficients(algo, st)
        if not np.all(np.isfinite(c_post)):
            raise FloatingPointError("posterior not finite")
    except (FloatingPointError, np.linalg.LinAlgError, ValueError):
        if st.iteration > 0:                                              # :195-205
            if probabilistic and getattr(algo, "retry_counter", RETRY_COUNTER_INIT) != 0:
                algo.retry_counter = getattr(algo, "retry_counter", RETRY_COUNTER_INIT) - 1   # :200-201
                return st
            return dataclasses.replace(st, status=STATUS_MODEL_FLEXIBILITY_ERROR)
        return st                                                         # :206-208
    algo.retry_counter = min(RETRY_COUNTER_INIT, getattr(algo, "retry_counter", RETRY_COUNTER_INIT) + 1)   # :210
    if probabilistic:
        # posterior.sample() :211 [scalismo-recalled A3]: coefficients ~ N(c, Minv).  scalismo draws them as
        # D^-1 U_s sqrt(s) z from svd(D Minv D); the same law is c + L^-T z with Mx = L L^T, which is the form
        # (and the z stream) libgingr_cuda documents -- identical distribution, different individual draws.
        L = np.linalg.cholesky(posed._last_Mx)
        z = standard_normals(st.model.rank, seed, st.iteration if counter is None else counter)
        c_post = c_post + np.linalg.solve(L.T, z)
    shapeproposal = posed.instance(c_post)                                # posterior.mean | sample  :211
    transformed_init = posed                                              # :212 (same transform)
    try:
        new_coeffs = transformed_init.coefficients(shapeproposal)         # :214-216
    except (FloatingPointError, np.linalg.LinAlgError):
        return dataclasses.replace(st, status=STATUS_MODEL_FLEXIBILITY_ERROR)
    cur = st.params.shape
    combined = cur + (new_coeffs - cur) * st.step_length                  # :218-220
    newshape = transformed_init.instance(combined)                        # :222
    current_fit_no_transform = st.model.instance(cur)                     # :224
    if st.global_transformation == SIMILARITY_TRANSFORMS:                 # :227-231
        R, t, s = umeyama(current_fit_no_transform, newshape, True)
    elif st.global_transformation == RIGID_TRANSFORMS:
        R, t, s = umeyama(current_fit_no_transform, newshape, False)
    else:
        R, t, s = np.eye(3), np.zeros(3), 1.0
    transformed = st.model.transform(R, t)                                # :232-234
    try:
        alpha = transformed.coefficients(newshape)                        # :235-237
    except (FloatingPointError, np.linalg.LinAlgError):
        return dataclasses.replace(st, status=STATUS_MODEL_FLEXIBILITY_ERROR)
    euler = matrix_to_euler(R)                                            # updateRotation :83-87
    params = Params(float(s), np.asarray(t, dtype=float), euler, alpha)   # :239-243
    new_state = dataclasses.replace(st, params=params)
    new_state._estep = getattr(st, "_estep", None)
    sigma2 = algo.update_sigma2(new_state)                                # :245-246 (fit/P still pre-update)
    return dataclasses.replace(new_state, sigma2=float(sigma2))


def propose(algo, st: State, probabilistic: bool = False, seed: int = 0, counter: Optional[int] = None) -> State:
    """GingrGeneratorWrapper.propose: update, refresh fit, iteration += 1.
    api/sampling/generators/GingrGeneratorWrapper.scala:28-39"""
    ns = update(algo, st, probabilistic, seed, counter)
    fit = model_instance_shape_pose_scale(ns.model, ns.params)
    return dataclasses.replace(ns, fit=fit, iteration=ns.iteration + 1)


def run(algo, initial: State, callback=None) -> State:
    """Deterministic GingrAlgorithm.run: the MH iterator yields the initial state first, so
    .take(maxIterations) performs maxIterations-1 proposals (always accepted); stops when
    converged(last, cur) or on ModelFlexibilityError.  api/GingrAlgorithm.scala:115-175"""
    st = algo.initialize(initial)
    last = None
    final_status = STATUS_MAX_ITERATION
    for k in range(algo.config.max_iterations):
        if k > 0:
            st = propose(algo, st)
        if callback is not None:
            callback(st)
        converged = last is not None and algo.config.converged(last, st)
        error = st.status == STATUS_MODEL_FLEXIBILITY_ERROR
        last = st
        if converged:
            final_status = STATUS_CONVERGED
            break
        if error:
            break
    if st.status == STATUS_NONE:
        st = dataclasses.replace(st, status=final_status)
    return st


# ---------------------------------------------------------------------------------------------
# Probabilistic registration: evaluators, proposal mixture, Metropolis-Hastings (api/sampling/*,
# GingrAlgorithm.scala:115-190).  Literal restatement; scalismo / Breeze behaviour tagged [scalismo-recalled].
# ---------------------------------------------------------------------------------------------
EVAL_MODEL_TO_TARGET, EVAL_TARGET_TO_MODEL, EVAL_SYMMETRIC = 0, 1, 2   # IndependentPointDistanceEvaluator.scala:26-32
LEAF_NAMES = ("informed", "rot_yaw", "rot_pitch", "rot_roll", "trans_x", "trans_y", "trans_z", "shape_0", "shape_1", "shape_2")


@dataclass
class McmcSettings:
    """ProbabilisticSettings(IndependentPoints(state, uncertainty, mode, evaluatedPoints), randomMixture) and the
    widths of Generator.DefaultRandom.  GingrAlgorithm.scala:40-50, sampling/Evaluator.scala:43-60, Generator.scala:27-83"""
    uncertainty: float = 1.0
    mode: int = EVAL_MODEL_TO_TARGET
    random_mixture: float = 0.5
    model_ids: Optional[np.ndarray] = None     # stand-in for decimate(numberOfPointsForComparison)
    target_ids: Optional[np.ndarray] = None
    rot_sdev: Tuple[float, float, float] = (0.01, 0.01, 0.01)     # yaw (psi), pitch (theta), roll (phi)
    trans_sdev: Tuple[float, float, float] = (0.1, 0.1, 0.1)
    shape_steps: Tuple[float, float, float] = (1.0, 0.1, 0.01)


def gaussian_logpdf(x, mu, sd):
    """Breeze Gaussian(mu, sd).logPdf / scalismo GaussianEvaluator.logDensity  [scalismo-recalled]"""
    return -((x - mu) ** 2) / (2.0 * sd * sd) - np.log(sd * np.sqrt(2.0 * np.pi))


def model_evaluator(alpha):
    """ModelEvaluator.logValue: MultivariateNormalDistribution(0, I_r).logpdf(alpha).  ModelEvaluator.scala:25-32"""
    a = np.asarray(alpha, dtype=float)
    return float(-0.5 * (a @ a) - 0.5 * a.shape[0] * np.log(2.0 * np.pi))


def distance_evaluator(settings: McmcSettings, st: State):
    """IndependentPointDistanceEvaluator.computeLogValue.  IndependentPointDistanceEvaluator.scala:54-78"""
    def m2t():
        pts = st.fit if settings.model_ids is None else st.fit[np.asarray(settings.model_ids)]
        _, d2, _ = closest_on_surface(pts, st.target, st.target_tri)
        return float(np.sum(gaussian_logpdf(np.sqrt(d2), 0.0, settings.uncertainty)))

    def t2m():
        pts = st.target if settings.target_ids is None else st.target[np.asarray(settings.target_ids)]
        _, d2, _ = closest_on_surface(pts, st.fit, st.model.tri)
        return float(np.sum(gaussian_logpdf(np.sqrt(d2), 0.0, settings.uncertainty)))
    if settings.mode == EVAL_MODEL_TO_TARGET:
        return m2t()
    if settings.mode == EVAL_TARGET_TO_MODEL:
        return t2m()
    return 0.5 * m2t() + 0.5 * t2m()


def log_value(settings: McmcSettings, st: State):
    """EvaluatorWrapper(probabilistic = true): ProductEvaluator(Prior, Distance) -> (prior, distance); the log value
    is their sum.  sampling/Evaluator.scala:25-28, :49-59"""
    return model_evaluator(st.params.shape), distance_evaluator(settings, st)


def posterior_model(algo, st: State) -> Gpmm:
    """cashedPosterior(state): model.transform(rigid).posterior(obs) as a full PointDistributionModel [A3]:
    mean' + Phi' (sqrt(lambda) c), basis Phi' U_s, variance s with svd(D Minv D).  GingrAlgorithm.scala:281-302"""
    posed, c, Minv = compute_posterior_coefficients(algo, st)
    if not np.all(np.isfinite(c)):
        raise FloatingPointError("posterior not finite")
    D = np.sqrt(st.model.variance)
    Sigma = D[:, None] * Minv * D[None, :]
    U, s, _ = np.linalg.svd(Sigma)
    return Gpmm(posed.ref, posed.mean + posed.basis @ (D * c), posed.basis @ U, s, posed.tri)


def log_transition_informed(algo, frm: State, to: State) -> float:
    """GeneratorWrapperStochastic.logTransitionProbability.  GeneratorWrapperStochastic.scala:42-63"""
    try:
        with np.errstate(all="ignore"):
            posterior = posterior_model(algo, frm)
    except (FloatingPointError, np.linalg.LinAlgError, ValueError):
        return -np.inf                                                    # :44-45
    if frm.step_length != 1.0:                                            # :47-51
        comp = frm.params.shape + (to.params.shape - frm.params.shape) / frm.step_length
        to_mesh = frm.model.instance(comp)
    else:
        to_mesh = frm.fit
    try:
        with np.errstate(all="ignore"):
            projected = posterior.coefficients(to_mesh)                   # :53
        v = float(-0.5 * (projected @ projected) - 0.5 * projected.shape[0] * np.log(2.0 * np.pi))   # gp.logpdf [A1]
        return v if np.isfinite(v) else -np.inf
    except (FloatingPointError, np.linalg.LinAlgError, ValueError):
        return -np.inf                                                    # :57-60


def leaf_weights(rho: float):
    """Flattened weights of MixtureProposal(rho *: DefaultRandom + (1 - rho) *: informed).  Generator.scala:31-83,
    GingrAlgorithm.scala:184-187 (scalismo normalises the weights of every mixture)."""
    w = np.zeros(10)
    w[0] = 1.0 - rho
    w[1:4] = rho * 0.5 * 0.5 / 3.0
    w[4:7] = rho * 0.5 * 0.5 / 3.0
    w[7:10] = rho * 0.5 / 3.0
    return w


_EULER_SLOT = {1: 2, 2: 1, 3: 0}   # YawAxis -> psi, PitchAxis -> theta, RollAxis -> phi (RandomPoseUpdateProposal.scala:40-44)


def mixture_log_transition(settings: McmcSettings, a: State, b: State, t_informed: float) -> float:
    """MixtureProposal.logTransitionProbability(a, b) = log sum_k w_k exp(t_k) [scalismo-recalled A5] with the random
    leaves of RandomPoseUpdateProposal.scala:47-63, :96-107 and RandomShapeUpdateProposal.scala:42-50."""
    w = leaf_weights(settings.random_mixture)
    pa, pb = a.params, b.params
    scale_eq = pa.scale == pb.scale
    trans_eq = bool(np.all(np.asarray(pa.translation) == np.asarray(pb.translation)))
    rot_eq = tuple(pa.euler) == tuple(pb.euler)
    shape_eq = bool(np.all(pa.shape == pb.shape))
    with np.errstate(all="ignore"):
        s = w[0] * np.exp(t_informed)
        for k in range(3):
            if scale_eq and trans_eq and shape_eq:
                slot = _EULER_SLOT[1 + k]
                s += w[1 + k] * np.exp(gaussian_logpdf(pb.euler[slot] - pa.euler[slot], 0.0, settings.rot_sdev[k]))
            if scale_eq and rot_eq and shape_eq:
                s += w[4 + k] * np.exp(gaussian_logpdf(pb.translation[k] - pa.translation[k], 0.0, settings.trans_sdev[k]))
            if scale_eq and rot_eq and trans_eq:
                sd = settings.shape_steps[k]
                ss = float(np.sum((pb.shape - pa.shape) ** 2))
                s += w[7 + k] * np.exp(-ss / (2.0 * sd * sd) - len(pa.shape) * np.log(sd * np.sqrt(2.0 * np.pi)))
        return float(np.log(s))


def _u53(a, b):
    return ((int(a) >> 5) * 67108864.0 + (int(b) >> 6) + 0.5) / 9007199254740992.0


def mcmc_uniforms(seed: int, step: int):
    """(u_choice, u_accept) of MH step `step`: Philox counter (0, step, 1, 0)  (gingr_b200/csrc/mcmc.cuh)."""
    x = philox4x32_10(np.array([0]), np.array([step]), np.array([1]), np.array([0]), seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    return _u53(x[0][0], x[1][0]), _u53(x[2][0], x[3][0])


def mcmc_normals(n: int, seed: int, step: int):
    """Perturbation normals of the random proposals: Philox counter (pair, step, 2, 0), Box-Muller."""
    npair = (n + 1) // 2
    p = np.arange(npair, dtype=np.uint64)
    zero = np.zeros(npair, dtype=np.uint64)
    x0, x1, x2, x3 = philox4x32_10(p, zero + np.uint64(step), zero + np.uint64(2), zero, seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    u1 = ((x0 >> np.uint64(5)).astype(np.float64) * 67108864.0 + (x1 >> np.uint64(6)).astype(np.float64) + 0.5) / 9007199254740992.0
    u2 = ((x2 >> np.uint64(5)).astype(np.float64) * 67108864.0 + (x3 >> np.uint64(6)).astype(np.float64) + 0.5) / 9007199254740992.0
    rad = np.sqrt(-2.0 * np.log(u1))
    ang = 6.283185307179586476925 * u2
    z = np.empty(2 * npair)
    z[0::2] = rad * np.cos(ang)
    z[1::2] = rad * np.sin(ang)
    return z[:n]


def random_proposal(settings: McmcSettings, cur: State, leaf: int, seed: int, step: int) -> State:
    """gingrPropose of the random generators + GingrGeneratorWrapper.propose (fit refresh, iteration + 1).
    RandomPoseUpdateProposal.scala:37-47, :80-94; RandomShapeUpdateProposal.scala:32-40; GingrGeneratorWrapper.scala:28-39"""
    p = cur.params
    euler, trans, shape = list(p.euler), np.array(p.translation, dtype=float), p.shape.copy()
    if 1 <= leaf <= 3:
        euler[_EULER_SLOT[leaf]] += settings.rot_sdev[leaf - 1] * mcmc_normals(1, seed, step)[0]
    elif 4 <= leaf <= 6:
        trans[leaf - 4] += settings.trans_sdev[leaf - 4] * mcmc_normals(1, seed, step)[0]
    else:
        shape = shape + settings.shape_steps[leaf - 7] * mcmc_normals(len(shape), seed, step)
    params = Params(p.scale, trans, tuple(euler), shape)
    ns = dataclasses.replace(cur, params=params)
    return dataclasses.replace(ns, fit=model_instance_shape_pose_scale(ns.model, params), iteration=cur.iteration + 1)


def mcmc_step(algo, settings: McmcSettings, cur: State, lp_cur, step: int, seed: int):
    """One step of scalismo MetropolisHastings [A5] with generatorCombined (GingrAlgorithm.scala:177-190).
    Returns (state, (prior, distance) of it, info dict)."""
    u_choice, u_accept = mcmc_uniforms(seed, step)
    w = leaf_weights(settings.random_mixture)
    leaf, acc = len(w) - 1, 0.0
    for k in range(len(w)):
        acc += w[k]
        if u_choice < acc:
            leaf = k
            break
    if w[leaf] <= 0.0:
        leaf = 0
    if leaf == 0:
        prop = propose(algo, cur, True, seed, counter=step)               # GeneratorWrapperStochastic.gingrPropose
    else:
        prop = random_proposal(settings, cur, leaf, seed, step)
    t_fw = log_transition_informed(algo, cur, prop)
    t_bw = log_transition_informed(algo, prop, cur)
    fw = mixture_log_transition(settings, cur, prop, t_fw)
    bw = mixture_log_transition(settings, prop, cur, t_bw)
    lp_prop = log_value(settings, prop)
    info = {"leaf": leaf, "t_fw": t_fw, "t_bw": t_bw, "fw": fw, "bw": bw, "lp_prop": lp_prop, "u_accept": u_accept}
    if cur.status == STATUS_MODEL_FLEXIBILITY_ERROR:
        info["accept"] = False
        return cur, lp_cur, info
    if np.isnan(fw) or np.isnan(bw):
        info["accept"] = False                                            # scalismo throws; the chain keeps its state here
        return cur, lp_cur, info
    ratio = -np.inf if (np.isneginf(fw) or np.isneginf(bw)) else fw - bw
    with np.errstate(all="ignore"):
        a = (lp_prop[0] + lp_prop[1]) - (lp_cur[0] + lp_cur[1]) - ratio
        accept = bool(a > 0.0 or u_accept < np.exp(a))
    info["a"] = a
    info["accept"] = accept
    return (prop, lp_prop, info) if accept else (cur, lp_cur, info)


# ---------------------------------------------------------------------------------------------
# GPMM construction (api/gpmm/GPMMHelper.scala:39-54, :99-129; scalismo approximateGPCholesky [scalismo-recalled A7])
# ---------------------------------------------------------------------------------------------
def gaussian_mixture_kernel_matrix(pts, sigmas, scalings):
    """Scalar kernel sum_q scaling_q exp(-|x - y|^2 / sigma_q^2)  (scalismo GaussianKernel: sigma^2, not 2 sigma^2)."""
    p = _c(pts)
    d2 = ((p[:, None, :] - p[None, :, :]) ** 2).sum(-1)
    return sum(sc * np.exp(-d2 / (sg * sg)) for sg, sc in zip(np.atleast_1d(sigmas), np.atleast_1d(scalings)))


def pivoted_cholesky(K, rel_tol, max_rank=None):
    """scalismo PivotedCholesky.computeApproximateCholesky with RelativeTolerance, literal: columns are added while the
    residual trace exceeds rel_tol * trace(K); the pivot is the first maximal residual diagonal."""
    n = K.shape[0]
    d = np.diag(K).astype(float).copy()
    tol = rel_tol * d.sum()
    cap = n if not max_rank else min(n, max_rank)
    cols = []
    done = np.zeros(n, dtype=bool)
    tr = d.sum()
    while len(cols) < cap and tr > tol:
        dm = np.where(done, -np.inf, d)
        p = int(np.argmax(dm))
        if not dm[p] > 0.0:
            cols.append(np.zeros(n))
            done[p] = True
        else:
            piv = np.sqrt(dm[p])
            col = K[:, p].astype(float).copy()
            for c in cols:
                col -= c * c[p]
            col /= piv
            col[done] = 0.0
            col[p] = piv
            done[p] = True
            d = d - col * col
            cols.append(col)
        tr = float(d[~done].sum())
    return np.stack(cols, axis=1) if cols else np.zeros((n, 0))


def approximate_gp_cholesky(ref, sigmas, scalings, rel_tol=0.01, max_rank=None) -> "Gpmm":
    """LowRankGaussianProcess.approximateGPCholesky for DiagonalKernel(scalar Gaussian mixture, 3), LITERAL: the
    3M x 3M matrix K = Ks (x) I3 (row 3 i + d), pivoted Cholesky L, (V, s) = svd(L^T L), basis = L V s^-1/2, variance = s."""
    Ks = gaussian_mixture_kernel_matrix(ref, sigmas, scalings)
    K = np.kron(Ks, np.eye(3))
    L = pivoted_cholesky(K, rel_tol, max_rank)
    V, s, _ = np.linalg.svd(L.T @ L)
    basis = L @ V / np.sqrt(s)[None, :]
    return Gpmm(_c(ref), np.zeros(3 * len(ref)), basis, s, None), L


def approximate_gp_cholesky_structured(ref, sigmas, scalings, rel_tol=0.01, max_rank=None):
    """The same through the scalar M x M factorisation (what gingr_b200/csrc/gpmm.cuh does): returns (rank, L L^T as the
    per-dimension scalar factors) -- dims < rank % 3 use one more scalar column."""
    Ks = gaussian_mixture_kernel_matrix(ref, sigmas, scalings)
    M = Ks.shape[0]
    full_cap = 3 * M if not max_rank else min(3 * M, max_rank)
    Ls = pivoted_cholesky(Ks, 0.0, min(M, (full_cap + 2) // 3))
    # scalar traces T(k) before step k
    T = [float(np.trace(Ks) - np.sum(Ls[:, :k] ** 2)) for k in range(Ls.shape[1] + 1)]
    # residual of already chosen pivots is exactly zero in exact arithmetic; mirror the device (sum over not-done rows)
    tol = rel_tol * 3.0 * T[0]
    rank = None
    for kk in range(Ls.shape[1]):
        for c in range(3):
            tr = 3.0 * T[kk] - c * (T[kk] - T[kk + 1])
            if not tr > tol or 3 * kk + c >= full_cap:
                rank = 3 * kk + c
                break
        if rank is not None:
            break
    if rank is None:
        rank = min(3 * Ls.shape[1], full_cap)
    return rank, Ls
