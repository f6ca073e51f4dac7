"""Seeded synthetic inputs of the shapes named in BASELINE.json / SURVEY.md 8(d): Fibonacci-sphere meshes,
smoothly displaced targets and low-rank GPMMs.  There is no network for datasets; bench.py and the tests
use these generators (and the two femur STL fixtures under tests/golden where present)."""
from __future__ import annotations

import numpy as np


def fibonacci_sphere(n: int, radius: float = 100.0) -> np.ndarray:
    """n quasi-uniform points on a sphere."""
    i = np.arange(n) + 0.5
    phi = np.arccos(1 - 2 * i / n)
    theta = np.pi * (1 + 5 ** 0.5) * i
    return radius * np.stack([np.cos(theta) * np.sin(phi), np.sin(theta) * np.sin(phi), np.cos(phi)], axis=1)


def sphere_mesh(n: int, radius: float = 100.0):
    """Fibonacci sphere with its convex-hull triangulation (closed, consistently outward oriented)."""
    from scipy.spatial import ConvexHull
    pts = fibonacci_sphere(n, radius)
    hull = ConvexHull(pts)
    tri = hull.simplices.astype(np.int32)
    a, b, c = pts[tri[:, 0]], pts[tri[:, 1]], pts[tri[:, 2]]
    flip = np.einsum("ij,ij->i", np.cross(b - a, c - a), a + b + c) < 0
    tri[flip] = tri[flip][:, [0, 2, 1]]
    return pts, tri


def icosphere(subdivisions: int, radius: float = 100.0):
    """Icosahedron with every triangle split in four, `subdivisions` times: 10 4^s + 2 vertices (642 for s = 3)."""
    t = (1.0 + 5.0 ** 0.5) / 2.0
    verts = [(-1, t, 0), (1, t, 0), (-1, -t, 0), (1, -t, 0), (0, -1, t), (0, 1, t), (0, -1, -t), (0, 1, -t), (t, 0, -1),
             (t, 0, 1), (-t, 0, -1), (-t, 0, 1)]
    tri = [(0, 11, 5), (0, 5, 1), (0, 1, 7), (0, 7, 10), (0, 10, 11), (1, 5, 9), (5, 11, 4), (11, 10, 2), (10, 7, 6), (7, 1, 8),
           (3, 9, 4), (3, 4, 2), (3, 2, 6), (3, 6, 8), (3, 8, 9), (4, 9, 5), (2, 4, 11), (6, 2, 10), (8, 6, 7), (9, 8, 1)]
    v = [np.asarray(p, float) / np.linalg.norm(p) for p in verts]
    for _ in range(subdivisions):
        mid, nxt = {}, []

        def m(a, b):
            k = (min(a, b), max(a, b))
            if k not in mid:
                p = v[a] + v[b]
                v.append(p / np.linalg.norm(p))
                mid[k] = len(v) - 1
            return mid[k]
        for a, b, c in tri:
            ab, bc, ca = m(a, b), m(b, c), m(c, a)
            nxt += [(a, ab, ca), (b, bc, ab), (c, ca, bc), (ab, bc, ca)]
        tri = nxt
    return radius * np.array(v), np.array(tri, dtype=np.int32)


def grid_patch(n: int, spacing: float = 1.0):
    """Open n x n vertex grid in the plane z = 0, two triangles per cell (a surface with a boundary)."""
    y, x = np.mgrid[0:n, 0:n]
    pts = spacing * np.stack([x.ravel(), y.ravel(), np.zeros(n * n)], axis=1).astype(float)
    i = (np.arange(n - 1)[:, None] * n + np.arange(n - 1)[None, :]).ravel()
    tri = np.concatenate([np.stack([i, i + 1, i + n + 1], 1), np.stack([i, i + n + 1, i + n], 1)]).astype(np.int32)
    return pts, tri


def random_sphere_mesh(n: int, seed: int, radius: float = 100.0):
    """Convex hull of n random points on a sphere: a closed mesh whose graph has no symmetry (unlike the icosphere's,
    where pivot values of a graph kernel tie exactly)."""
    from scipy.spatial import ConvexHull
    p = np.random.default_rng(seed).normal(size=(n, 3))
    p = radius * p / np.linalg.norm(p, axis=1)[:, None]
    return p, ConvexHull(p).simplices.astype(np.int32)


def random_patch(n: int, seed: int, size: float = 100.0):
    """Delaunay triangulation of n random points in a square in the plane z = 0: an open mesh without symmetry."""
    from scipy.spatial import Delaunay
    q = np.random.default_rng(seed).uniform(0.0, size, size=(n, 2))
    return np.hstack([q, np.zeros((n, 1))]), Delaunay(q).simplices.astype(np.int32)


def euler_matrix(phi, theta, psi):
    from .rotation import euler_to_matrix
    return euler_to_matrix(phi, theta, psi)


def smooth_displacement(points: np.ndarray, rng: np.random.Generator, n_waves: int = 8, amp: float = 3.0,
                        wavelength: float = 50.0) -> np.ndarray:
    """sum_k a_k sin(w_k . p + phi_k),  a_k ~ N(0, amp^2) per axis, |w_k| ~ 1/wavelength."""
    out = np.zeros_like(points)
    for _ in range(n_waves):
        w = rng.normal(size=3)
        w *= (1.0 / wavelength) / np.linalg.norm(w)
        a = rng.normal(scale=amp, size=3)
        ph = rng.uniform(0, 2 * np.pi)
        out += np.sin(points @ w + ph)[:, None] * a[None, :]
    return out


def make_target(points: np.ndarray, seed: int, t=(5.0, 5.0, 5.0), euler=(0.05, 0.05, 0.05)) -> np.ndarray:
    rng = np.random.default_rng(seed)
    R = euler_matrix(*euler)
    return (points + smooth_displacement(points, rng)) @ R.T + np.asarray(t)


def make_gpmm(ref: np.ndarray, rank: int, seed: int, lambda0: float = 100.0, decay: float = 0.995,
              kernel_sigma: float = 60.0, orthonormal: bool = True):
    """(mean = 0, basis [3M, r], variance [r]).  Basis columns: smooth vector fields built from Gaussian-kernel
    features at `rank` random centres (Nystrom style), QR-orthonormalised; for large M a seeded Gaussian matrix
    is used before QR.  variance_k = lambda0 * decay^k."""
    rng = np.random.default_rng(seed)
    M = ref.shape[0]
    r = int(rank)
    if M <= 20000 and r <= 600:
        nc = max(1, (r + 2) // 3)
        centres = ref[rng.choice(M, size=min(nc, M), replace=nc > M)]
        d2 = ((ref[:, None, :] - centres[None, :, :]) ** 2).sum(-1)
        feat = np.exp(-d2 / (2 * kernel_sigma ** 2))                      # [M, nc]
        B = np.zeros((3 * M, 3 * feat.shape[1]))
        for d in range(3):
            B[d::3, d::3] = feat
        B = B[:, :r] if B.shape[1] >= r else np.concatenate([B, rng.normal(size=(3 * M, r - B.shape[1]))], axis=1)
        B = B + 1e-3 * rng.normal(size=B.shape)
    else:
        B = rng.normal(size=(3 * M, r))
    if orthonormal:
        B, _ = np.linalg.qr(B)
    else:
        B /= np.linalg.norm(B, axis=0, keepdims=True)
    variance = lambda0 * decay ** np.arange(r)
    return np.zeros(3 * M), np.ascontiguousarray(B), variance


def workload(name: str, seed: int = 0):
    """Named workloads (SURVEY.md 8d).  Returns dict(ref, tri, mean, basis, variance, target, target_tri)."""
    sizes = {
        "c1": (100, 100, 50), "c2": (100, 100, 50), "c3a": (100, 100, 50), "c3b": (500, 500, 100),
        "c3c": (1000, 1000, 100), "c4": (20000, 200000, 2000), "c4_small": (4000, 20000, 500),
    }
    M, N, r = sizes[name]
    ref, tri = sphere_mesh(M)
    tgt_pts, tgt_tri = sphere_mesh(N) if N <= 50000 else (fibonacci_sphere(N), None)
    target = make_target(tgt_pts, seed)
    mean, basis, variance = make_gpmm(ref, r, seed + 1)
    return dict(ref=ref, tri=tri, mean=mean, basis=basis, variance=variance, target=target, target_tri=tgt_tri)
