"""The BCPD configuration of GingrAlgorithm (GINGR_ALGO_BCPD, gingr_b200/csrc/update.cu) for the tests: a literal restatement
of this project's reading of the textbook BCPD (other/algorithms/cpd/BCPD.scala) on GiNGR's three hooks, beside
oracle.CpdAlgorithm.

    E-step        P materialised with BCPD.computeP's formula (oracle.bcpd_P, quirks kept: s, not s^2, in the exponent and
                  (1 - w) applied twice), from the pre-update fit, Sigma, alpha, the state's sigma2 and scale
    observations  xhat_m with noise sigma2 lambda / nu_m I3 (CPD.scala:125 with P1 -> nu)
    sigma2 hook   (sXX - 2 sXY + sYY + sigma2 sigma2bar) / (3 Nhat), sigma2bar = sum nu_m Sigma_m / Nhat
    next state    alpha_m = exp(psi(kappa + nu_m) - psi(kappa M + Nhat)) (scipy.special.digamma) and
                  Sigma_m = tr(cov_m) / 3 of the iteration's dense posterior covariance Q Minv Q^T, committed with the state

The per-registration state (alpha, Sigma) lives on the algorithm object, as it lives next to the device state block."""
import dataclasses

import numpy as np
from scipy.special import digamma

from . import oracle as o


@dataclasses.dataclass
class BcpdConfig(o.CpdConfig):
    kappa: float = 1.0


def prior_variance(model: o.Gpmm) -> np.ndarray:
    """Sigma_m = tr(Phi_m Lambda Phi_m^T) / 3: the posterior variance without observations."""
    Q = model.basis * np.sqrt(model.variance)[None, :]
    return (Q * Q).sum(1).reshape(-1, 3).sum(1) / 3.0


def posterior_vertex_variance(model: o.Gpmm, Minv: np.ndarray) -> np.ndarray:
    """Sigma_m = tr(cov_m) / 3 with cov_m = Q_m Minv Q_m^T (Q = Phi D), by the trace formula: sum over the three rows
    q of vertex m of q Minv q^T."""
    Q = model.basis * np.sqrt(model.variance)[None, :]
    return ((Q @ Minv) * Q).sum(1).reshape(-1, 3).sum(1) / 3.0


def sigma2_terms(P, target, fit):
    """(sXX, sXY, sYY, Nhat) on a materialised P: sXX = sum_n nu'_n |x_n|^2, sXY = sum_m (P X)_m . fit_m,
    sYY = sum_m nu_m |fit_m|^2, Nhat = sum nu'."""
    X, Y = np.asarray(target), np.asarray(fit)
    nu, nup = P.sum(1), P.sum(0)
    return (float(nup @ (X * X).sum(1)), float(((P @ X) * Y).sum()), float(nu @ (Y * Y).sum(1)), float(nup.sum()))


class BcpdAlgorithm:
    name = "BCPD"

    def __init__(self, config: BcpdConfig):
        self.config = config
        self.alpha = None
        self.Sigma = None

    def initialize(self, general: o.State) -> o.State:
        """CPD's initializeState for sigma2; alpha = 1 / M, Sigma = the prior variance."""
        M = general.model.M
        self.alpha = np.full(M, 1.0 / M)
        self.Sigma = prior_variance(general.model)
        return o.CpdAlgorithm(self.config).initialize(general)

    def estep(self, st: o.State):
        P = o.bcpd_P(st.fit, st.target, self.Sigma, self.alpha, st.sigma2, st.params.scale, self.config.w)
        nu, nup, PX = o.P_reductions(P, st.target)
        return P, nu, nup, PX

    def observations(self, st: o.State):
        P, nu, nup, PX = self.estep(st)
        with np.errstate(divide="ignore", invalid="ignore"):
            xhat = PX / nu[:, None]
            var = st.sigma2 * self.config.lam * (1.0 / nu)
        cov = np.eye(3)[None, :, :] * var[:, None, None]
        st._estep = (P, nu, nup, PX)
        return np.arange(st.model.M, dtype=np.int32), xhat, cov

    def update_sigma2(self, st: o.State) -> float:
        """On the pre-update fit, with the Sigma the E-step used; sC = sigma2 sigma2bar kept literally."""
        P, nu, nup, PX = st._estep
        sXX, sXY, sYY, nhat = sigma2_terms(P, st.target, st.fit)
        s2bar = float(nu @ self.Sigma) / nhat
        return (sXX - 2.0 * sXY + sYY + st.sigma2 * s2bar) / (3.0 * nhat)


def update(algo: BcpdAlgorithm, st: o.State) -> o.State:
    """One deterministic update; alpha and Sigma advance only when the iteration commits its new state."""
    new = o.update(algo, st)
    if new.params is st.params:   # posterior or coefficients failure: the state, alpha and Sigma stay
        return new
    with np.errstate(all="ignore"):
        posed, c, Minv = o.compute_posterior_coefficients(algo, st)
    P, nu, nup, PX = st._estep
    nhat = float(nup.sum())
    kappa, M = algo.config.kappa, st.model.M
    algo.alpha = np.exp(digamma(kappa + nu) - digamma(kappa * M + nhat))
    algo.Sigma = posterior_vertex_variance(st.model, Minv)
    return new


def propose(algo: BcpdAlgorithm, st: o.State) -> o.State:
    ns = update(algo, st)
    fit = o.model_instance_shape_pose_scale(ns.model, ns.params)
    return dataclasses.replace(ns, fit=fit, iteration=ns.iteration + 1)
