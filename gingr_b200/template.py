"""TemplateRegistration (api/registration/config/Template.scala:24-59): the reference's extension point for a user-defined
GiNGR algorithm -- a `getCorrespondence` closure (state -> CorrespondencePairs) and a `getUncertainty` closure (point id,
state -> observation covariance) plugged into the unchanged `GingrAlgorithm.update` (api/GingrAlgorithm.scala:192-254).

The closures are host code by construction (arbitrary user logic), so here one iteration is the reference's statement
sequence with every GPMM operation on the device through the kernel-level entry points -- posterior mean
(gingr_posterior_mean: weighted Gram on the FP64 tensor pipe, Cholesky solve, mean evaluation), both `coefficients` calls
(gingr_coefficients) and both instances (gingr_model_instance) -- and only the O(M) Procrustes reduction and the scalar
bookkeeping in numpy.  The built-in CPD / ICP algorithms do NOT take this route: their whole iteration is device resident
(gingr_update).  Deterministic proposals only (posterior.mean); the probabilistic machinery belongs to the built-ins."""
from __future__ import annotations

import dataclasses
from dataclasses import dataclass
from typing import Callable, Optional, Tuple

import numpy as np

from . import api
from .rotation import euler_to_matrix, matrix_to_euler


def umeyama(X: np.ndarray, Y: np.ndarray, similarity: bool, euler_round_trip: bool = True) -> Tuple[np.ndarray, np.ndarray, float]:
    """scalismo LandmarkRegistration.{rigid, similarity}3DLandmarkRegistration about the origin, as called from
    GingrAlgorithm.scala:260-279 [scalismo-recalled, SURVEY A4]: x -> s R x + t minimising the squared residual; with
    euler_round_trip the rotation goes through its Euler angles and back, as the state stores it
    (GeneralRegistrationState.scala:83-87)."""
    n = X.shape[0]
    mx, my = X.mean(axis=0), Y.mean(axis=0)
    Xc, Yc = X - mx, Y - my
    var_x = float(np.sum(Xc * Xc) / n)
    S = (Yc.T @ Xc) / n
    U, D, Vt = np.linalg.svd(S)
    J = np.eye(3)
    if np.linalg.det(U) * np.linalg.det(Vt) < 0:   # sign det S at full rank; also a rotation for planar shapes (rank 2)
        J[2, 2] = -1.0
    R = U @ J @ Vt
    s = float(np.trace(np.diag(D) @ J) / var_x) if similarity else 1.0
    t = my - s * (R @ mx)
    if euler_round_trip:
        R = euler_to_matrix(*matrix_to_euler(R))
    return R, t, s


def _never_converged(last, current, threshold) -> bool:
    return False


@dataclass
class TemplateConfiguration:
    """Template.scala:24-29 (maxIterations = 1, threshold = 1e-5, converged = never, useLandmarkCorrespondence = true)."""
    maxIterations: int = 1
    threshold: float = 1e-5
    converged: Callable = _never_converged
    useLandmarkCorrespondence: bool = True


class TemplateRegistration:
    """Template.scala:44-59.  getCorrespondence(state) -> (pids [n] int, points [n, 3]) -- CorrespondencePairs
    (CorrespondencePairs.scala:23); default: no pairs.  getUncertainty(pids, state) -> [n] isotropic variances or
    [n, 3, 3] covariances for those ids (vectorised form of the per-id closure; default: identity covariance).
    updateSigma2(state) -> float (GingrAlgorithm.scala:256-258; default: unchanged)."""
    name = "Template"

    def __init__(self, ctx: "api.Context", model: "api.Model", target=None, config: Optional[TemplateConfiguration] = None,
                 getCorrespondence: Optional[Callable] = None, getUncertainty: Optional[Callable] = None,
                 updateSigma2: Optional[Callable] = None):
        self.ctx, self.model, self.target = ctx, model, target
        self.config = config or TemplateConfiguration()
        self.getCorrespondence = getCorrespondence or (lambda state: (np.zeros(0, np.int32), np.zeros((0, 3))))
        self.getUncertainty = getUncertainty or (lambda pids, state: np.ones(len(pids)))
        self.updateSigma2 = updateSigma2 or (lambda state: state.sigma2)
        self._landmarks = None

    def close(self):
        pass

    def setLandmarks(self, pids, points, cov=None):
        """GeneralRegistrationState.landmarkCorrespondences (GeneralRegistrationState.scala:43-62), resolved by the caller."""
        pids = np.asarray(pids, dtype=np.int32).reshape(-1)
        pts = np.asarray(points, dtype=np.float64).reshape(-1, 3)
        cov = np.tile(np.eye(3), (len(pids), 1, 1)) if cov is None else np.asarray(cov, dtype=np.float64).reshape(-1, 3, 3)
        if not (len(pids) == len(pts) == len(cov)):
            raise ValueError("landmarks: one point and one covariance per id")
        self._landmarks = (pids, pts, cov)

    # ---- state ------------------------------------------------------------------------------------
    def initializeState(self, globalTransformation: int = api.RIGID_TRANSFORMS, rotation=None, translation=None,
                        general: Optional["api.GeneralRegistrationState"] = None) -> "api.GeneralRegistrationState":
        """GeneralRegistrationState.apply (:136-178) + TemplateRegistration.initializeState (Template.scala:53-58): no sigma2
        initialisation, the fit is the model instance at the state's parameters."""
        if general is None:
            euler = (0.0, 0.0, 0.0) if rotation is None else matrix_to_euler(np.asarray(rotation, dtype=float))
            t = np.zeros(3) if translation is None else np.asarray(translation, dtype=float)
            pars = api.ModelFittingParameters(1.0, t, euler, np.zeros(self.model.rank))
            general = api.GeneralRegistrationState(pars, np.zeros((self.model.M, 3)), globalTransformation=globalTransformation)
        return dataclasses.replace(general, fit=self.model.instance(general.modelParameters))

    def _observations(self, state):
        """computePosterior's observation list (GingrAlgorithm.scala:281-296): correspondences with their uncertainties,
        minus those at landmark ids, plus the landmark observations."""
        pids, pts = self.getCorrespondence(state)
        pids = np.asarray(pids, dtype=np.int32).reshape(-1)
        pts = np.asarray(pts, dtype=np.float64).reshape(-1, 3)
        if len(pids) != len(pts):
            raise ValueError("getCorrespondence: one point per id")
        noise = np.asarray(self.getUncertainty(pids, state), dtype=np.float64)
        if noise.shape not in ((len(pids),), (len(pids), 3, 3)):
            raise ValueError("getUncertainty: [n] variances or [n, 3, 3] covariances")
        if self.config.useLandmarkCorrespondence and self._landmarks is not None and len(self._landmarks[0]):
            lp, lpts, lcov = self._landmarks
            keep = ~np.isin(pids, lp)
            if noise.ndim == 1:
                noise = noise[:, None, None] * np.eye(3)[None]
            pids = np.concatenate([pids[keep], lp])
            pts = np.concatenate([pts[keep], lpts])
            noise = np.concatenate([noise[keep], lcov])
        return pids, pts, noise

    # ---- one iteration ---------------------------------------------------------------------------------
    def update(self, current: "api.GeneralRegistrationState") -> "api.GeneralRegistrationState":
        """GingrAlgorithm.update(current, probabilistic = false) (:192-254)."""
        p = current.modelParameters
        R0, t0 = euler_to_matrix(*p.euler), np.asarray(p.translation, dtype=np.float64)
        failed = dataclasses.replace(current, status=api.STATUS_MODEL_FLEXIBILITY_ERROR)
        try:
            pids, pts, noise = self._observations(current)
            if len(pids) == 0 or not np.all(np.isfinite(noise)):
                raise FloatingPointError("no usable observations")
            _, shapeproposal = api.posterior_mean(self.ctx, self.model, R0, t0, pids, pts, noise)          # :193, :211
        except FloatingPointError:
            return failed if current.iteration > 0 else current                                             # :194-208
        try:
            new_coefficients = api.coefficients(self.ctx, self.model, R0, t0, shapeproposal)               # :214-216
        except FloatingPointError:
            return failed
        cur = np.asarray(p.shape, dtype=np.float64)
        combined = cur + (new_coefficients - cur) * current.stepLength                                      # :218-220
        newshape = self.model.instance(api.ModelFittingParameters(1.0, t0, tuple(p.euler), combined))      # :222
        no_transform = self.model.instance(api.ModelFittingParameters(1.0, np.zeros(3), (0.0, 0.0, 0.0), cur))   # :224
        if current.globalTransformation == api.SIMILARITY_TRANSFORMS:                                      # :227-231
            R, t, s = umeyama(no_transform, newshape, True)
        elif current.globalTransformation == api.RIGID_TRANSFORMS:
            R, t, s = umeyama(no_transform, newshape, False)
        else:
            R, t, s = np.eye(3), np.zeros(3), 1.0
        try:
            alpha = api.coefficients(self.ctx, self.model, R, t, newshape)                                  # :232-237
        except FloatingPointError:
            return failed
        pars = api.ModelFittingParameters(float(s), np.asarray(t, dtype=np.float64), matrix_to_euler(R), alpha)   # :239-243
        new_state = dataclasses.replace(current, modelParameters=pars)
        return dataclasses.replace(new_state, sigma2=float(self.updateSigma2(new_state)))                   # :245-246

    def propose(self, current: "api.GeneralRegistrationState") -> "api.GeneralRegistrationState":
        """GingrGeneratorWrapper.propose (GingrGeneratorWrapper.scala:28-39): update, refreshed fit, iteration + 1."""
        ns = self.update(current)
        return dataclasses.replace(ns, fit=self.model.instance(ns.modelParameters), iteration=ns.iteration + 1,
                                   generatedBy="Deterministic")

    def run(self, initialState: "api.GeneralRegistrationState", callBackLogger=None) -> "api.GeneralRegistrationState":
        """Deterministic GingrAlgorithm.run (:115-175); same loop as api.GingrAlgorithm.run."""
        st, last, final = initialState, None, api.STATUS_MAX_ITERATION
        for k in range(self.config.maxIterations):
            if k > 0:
                st = self.propose(st)
            if callBackLogger is not None:
                callBackLogger(st)
            converged = last is not None and self.config.converged(last, st, self.config.threshold)
            error = st.status == api.STATUS_MODEL_FLEXIBILITY_ERROR
            last = st
            if converged:
                final = api.STATUS_CONVERGED
                break
            if error:
                break
        if st.status == api.STATUS_NONE:
            st = dataclasses.replace(st, status=final)
        return st
