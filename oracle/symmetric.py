"""The mirror-symmetric Gaussian kernel about x = 0 (gingr_gpmm_gaussian_symmetric) for the tests: the literal 3M x 3M
construction, and a numpy restatement of the device's per-block merge (gingr_b200/csrc/gpmm.cuh, gpmm_build).

scalismo's symmetrised kernel with S = diag(-1, 1, 1), k the scalar Gaussian mixture and k_m(x, y) = k(S x, y):
    K(x, y) = DiagonalKernel(k, 3) + DiagonalKernel(-k_m, k_m, k_m)
            = diag(k(x, y) - k(S x, y), k(x, y) + k(S x, y), k(x, y) + k(S x, y))."""
import numpy as np

from .oracle import Gpmm, _c, pivoted_cholesky

MIRROR = np.array([-1.0, 1.0, 1.0])


def _mixture(a, b, sigmas, scalings):
    d2 = ((a[:, None, :] - b[None, :, :]) ** 2).sum(-1)
    return sum(sc * np.exp(-d2 / (sg * sg)) for sg, sc in zip(np.atleast_1d(sigmas), np.atleast_1d(scalings)))


def symmetric_gaussian_kernel_matrix(ref, sigmas, scalings):
    """The literal 3M x 3M matrix (row 3 i + d): the 3 x 3 kernel K(x_i, x_j) = k(x_i, x_j) I + k(S x_i, x_j) diag(-1, 1, 1)
    placed at block (i, j)."""
    p = _c(ref)
    k = _mixture(p, p, sigmas, scalings)
    km = _mixture(p * MIRROR, p, sigmas, scalings)
    return np.kron(k, np.eye(3)) + np.kron(km, np.diag(MIRROR))


def approximate_gp_cholesky_symmetric(ref, sigmas, scalings, rel_tol=0.01, max_rank=None):
    """approximateGPCholesky for the symmetric kernel, LITERAL: pivoted Cholesky L of the 3M x 3M matrix, (V, s) =
    svd(L^T L), basis = L V s^-1/2, variance = s.  -> (Gpmm, L)."""
    K = symmetric_gaussian_kernel_matrix(ref, sigmas, scalings)
    L = pivoted_cholesky(K, rel_tol, max_rank)
    V, s, _ = np.linalg.svd(L.T @ L)
    basis = L @ V / np.sqrt(s)[None, :]
    return Gpmm(_c(ref), np.zeros(3 * len(ref)), basis, s, None), L


def _scalar_history(B):
    """The device's scalar pivoted Cholesky of a block to the end: factor, pivot points, pivot values and T(k), the residual
    trace over the points not yet chosen before step k (k = 0..M)."""
    M = B.shape[0]
    d = np.diag(B).copy()
    done = np.zeros(M, dtype=bool)
    L = np.zeros((M, M))
    piv, dpiv, T = [], [], []
    for k in range(M):
        dm = np.where(done, -np.inf, d)
        p = int(np.argmax(dm))            # first maximal
        piv.append(p); dpiv.append(float(dm[p])); T.append(float(d[~done].sum()))
        if dm[p] > 0.0:
            col = (B[:, p] - L[:, :k] @ L[p, :k]) / np.sqrt(dm[p])
            col[done] = 0.0
            col[p] = np.sqrt(dm[p])
            d = d - col * col
            L[:, k] = col
        done[p] = True
    T.append(0.0)
    return L, piv, dpiv, T


def merged_cholesky_symmetric(ref, sigmas, scalings, rel_tol=0.01, max_rank=None):
    """The device's construction restated: scalar factorisations of K- = k - k_m (coordinate 0) and K+ = k + k_m
    (coordinates 1 and 2), merged in the literal order -- at each step the coordinate whose next pivot value is largest,
    ties to the lowest index 3 i + d -- until trace <= rel_tol * trace(K) or max_rank columns.
    -> (rank, columns taken per coordinate [3], factors [K-, K+], 3M x 3M covariance of the taken columns)."""
    p = _c(ref)
    M = len(p)
    k = _mixture(p, p, sigmas, scalings)
    km = _mixture(p * MIRROR, p, sigmas, scalings)
    hist = [_scalar_history(k - km), _scalar_history(k + km)]
    g = (0, 1, 1)
    full_cap = 3 * M if not max_rank else min(3 * M, max_rank)
    tol = rel_tol * (hist[0][3][0] + 2.0 * hist[1][3][0])
    kd = [0, 0, 0]
    cols = 0
    while cols < full_cap:
        if not sum(hist[g[d]][3][kd[d]] for d in range(3)) > tol:
            break
        cand = [(-hist[g[d]][2][kd[d]], 3 * hist[g[d]][1][kd[d]] + d, d) for d in range(3) if kd[d] < M]
        if not cand:
            break
        d = min(cand)[2]
        kd[d] += 1
        cols += 1
    cov = np.zeros((3 * M, 3 * M))
    for d in range(3):
        Lf = hist[g[d]][0][:, :kd[d]]
        cov[d::3, d::3] = Lf @ Lf.T
    return cols, kd, [hist[0][0], hist[1][0]], cov
