"""The inverse-Laplacian kernel (gingr_gpmm_inverse_laplacian) for the tests: the literal construction, and a numpy
restatement of the device's scalar factorisation taken in triples (gingr_b200/csrc/gpmm.cuh, gpmm_build).

This project's reading of the reference's look-up kernel (LaplacianHelper.scala:26-55, MatrixHelper.pinv :23-26):
    L  = D - A, the combinatorial graph Laplacian of the triangle edges: unit weights, each undirected edge counted
         once however many triangles share it, self-edges of degenerate triangles ignored;
    Ks = scaling pinv(L + gamma I)   (the inverse for gamma > 0);
    K  = Ks (x) I3 (row 3 i + d), then scalismo's approximateGPCholesky; the mean is zero."""
import numpy as np

from .oracle import Gpmm, _c, pivoted_cholesky

# numpy.linalg.pinv's cut of small singular values, relative to the largest: the zero eigenvalues of L (one per
# component) come out of the SVD at the rounding level (~1e-15 of |L|), the smallest non-zero ones of a graph Laplacian
# on at most 6000 vertices lie far above 1e-10 of |L|
PINV_RCOND = 1e-10


def graph_laplacian(M, tri):
    """L = D - A from loops over the triangles."""
    A = np.zeros((M, M))
    for t in np.asarray(tri).reshape(-1, 3):
        for e in range(3):
            a, b = int(t[e]), int(t[(e + 1) % 3])
            if a != b:
                A[a, b] = 1.0
                A[b, a] = 1.0
    return np.diag(A.sum(axis=1)) - A


def components(M, tri):
    """Connected components of the edge graph (a vertex in no triangle is its own) -> label per vertex, numbered in
    order of the first vertex."""
    label = -np.ones(M, dtype=int)
    L = graph_laplacian(M, tri)
    n = 0
    for s in range(M):
        if label[s] >= 0:
            continue
        stack = [s]
        label[s] = n
        while stack:
            v = stack.pop()
            for w in np.nonzero(L[v] < 0.0)[0]:
                if label[w] < 0:
                    label[w] = n
                    stack.append(w)
        n += 1
    return label


def projector(M, tri):
    """P = sum_c 1_c 1_c^T / |c| over the components."""
    lab = components(M, tri)
    same = lab[:, None] == lab[None, :]
    size = np.bincount(lab)
    return same / size[lab][:, None]


def inverse_laplacian_kernel_matrix(M, tri, scaling, gamma):
    """Ks = scaling pinv(L + gamma I) through the SVD (numpy.linalg.pinv), the reference's route."""
    return scaling * np.linalg.pinv(graph_laplacian(M, tri) + gamma * np.eye(M), rcond=PINV_RCOND)


def approximate_gp_cholesky_laplacian(M, ref, tri, scaling, gamma, rel_tol=0.01, max_rank=None):
    """approximateGPCholesky for Ks (x) I3, LITERAL: pivoted Cholesky L of the 3M x 3M matrix, (V, s) = svd(L^T L),
    basis = L V s^-1/2, variance = s.  -> (Gpmm, L)."""
    K = np.kron(inverse_laplacian_kernel_matrix(M, tri, scaling, gamma), np.eye(3))
    L = pivoted_cholesky(K, rel_tol, max_rank)
    V, s, _ = np.linalg.svd(L.T @ L)
    basis = L @ V / np.sqrt(s)[None, :]
    return Gpmm(_c(ref), np.zeros(3 * M), basis, s, None), L


def triples_cholesky(Ks, rel_tol=0.01, max_rank=None, with_margin=False):
    """The device's construction restated: the scalar pivoted Cholesky of Ks, taken in triples -- a pivot (p, d) leaves
    the residuals of (p, d') untouched, so the literal order is (p, 0), (p, 1), (p, 2) and, after c columns of triple k,
    the residual trace is 3 T(k) - c (T(k) - T(k + 1)) with T the scalar traces over the points not yet chosen.
    -> (rank, columns per coordinate [3], scalar factor; coordinate d uses its first kd[d] columns), and with
    with_margin the smallest relative gap (best - runner-up) / best between the pivot value and the next one over the
    steps whose columns the model uses: where it is far above rounding, every correct implementation picks the same
    pivots."""
    M = Ks.shape[0]
    full_cap = 3 * M if not max_rank else min(3 * M, max_rank)
    d = np.diag(Ks).copy()
    done = np.zeros(M, dtype=bool)
    Ls = np.zeros((M, 0))
    T = [float(d.sum())]
    tol = rel_tol * 3.0 * T[0]
    rank = 0
    gaps = []
    while rank < full_cap:
        k = rank // 3
        c = rank % 3
        if Ls.shape[1] == k:                      # the scalar step k, then T(k + 1)
            if k >= M:
                break
            dm = np.where(done, -np.inf, d)
            p = int(np.argmax(dm))
            second = np.max(np.where(np.arange(M) == p, -np.inf, dm)) if M > 1 else -np.inf
            gaps.append((dm[p] - second) / dm[p] if dm[p] > 0.0 and np.isfinite(second) else np.inf)
            col = np.zeros(M)
            if dm[p] > 0.0:
                piv = np.sqrt(dm[p])
                col = (Ks[:, p] - Ls @ Ls[p]) / piv
                col[done] = 0.0
                col[p] = piv
                d = d - col * col
            done[p] = True
            Ls = np.hstack([Ls, col[:, None]])
            T.append(float(d[~done].sum()))
        tr = 3.0 * T[k] - c * (T[k] - T[k + 1])
        if not tr > tol:
            break
        rank += 1
    kd = [rank // 3 + (1 if dd < rank % 3 else 0) for dd in range(3)]
    if with_margin:
        return rank, kd, Ls, min(gaps[:max(kd)], default=np.inf)
    return rank, kd, Ls


def triples_covariance(kd, Ls):
    """The 3M x 3M covariance of the columns triples_cholesky took."""
    M = Ls.shape[0]
    cov = np.zeros((3 * M, 3 * M))
    for dd in range(3):
        F = Ls[:, :kd[dd]]
        cov[dd::3, dd::3] = F @ F.T
    return cov
