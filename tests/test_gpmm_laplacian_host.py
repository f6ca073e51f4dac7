"""CPU tests of the inverse-Laplacian GPMM construction (gingr_gpmm_inverse_laplacian): the projector formula the device
uses for the pseudo-inverse, the scalar factorisation taken in triples against the literal 3M x 3M pivoted Cholesky of
Ks (x) I3 (oracle/laplacian.py), the graph Laplacian's indifference to duplicated, degenerate and reordered triangles, and
the Python and C++ mirrors of the new factory."""
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lap():
    from oracle import laplacian
    return laplacian


def _mesh(kind):
    """(M, triangles) of the test meshes: one component, several, an isolated vertex, an open patch, and meshes with
    duplicated and degenerate triangles.  The random meshes have no graph symmetry: on the icosphere or the grid, pivot
    values tie exactly and rounding orders them, differently in differently ordered sums."""
    from gingr_b200 import synthetic
    if kind == "icosphere":
        v, t = synthetic.icosphere(2)
        return len(v), t
    if kind == "grid":
        return 81, synthetic.grid_patch(9)[1]
    if kind == "duplicates":
        v, t = synthetic.icosphere(2)
        return len(v), np.vstack([t, t[:40], t[5:9, ::-1], [[3, 3, 7], [9, 9, 9], [11, 2, 11]]])
    if kind == "sphere":
        return 160, synthetic.random_sphere_mesh(160, 0)[1]
    two = np.vstack([synthetic.random_sphere_mesh(150, 1)[1], synthetic.random_sphere_mesh(50, 2)[1] + 150])
    if kind == "two":
        return 200, two
    if kind == "three_and_isolated":           # two spheres, a tree of degenerate triangles and an isolated last vertex
        tree = 200 + np.array([[0, 1, 1], [1, 2, 2], [2, 3, 3], [4, 1, 4], [4, 5, 5], [5, 6, 6], [6, 7, 7]])
        return 209, np.vstack([two, tree])
    if kind == "patch":
        return 100, synthetic.random_patch(100, 3)[1]
    raise ValueError(kind)


@pytest.mark.parametrize("kind", ["icosphere", "grid", "duplicates", "two", "three_and_isolated", "patch"])
def test_projector_formula_is_the_pseudo_inverse(lap, kind):
    M, tri = _mesh(kind)
    L = lap.graph_laplacian(M, tri)
    P = lap.projector(M, tri)
    ncomp = lap.components(M, tri).max() + 1
    assert np.allclose(P @ P, P) and np.allclose(L @ P, 0.0)
    assert np.linalg.matrix_rank(L) == M - ncomp
    proj = np.linalg.inv(L + P) - P
    pinv = np.linalg.pinv(L, rcond=lap.PINV_RCOND)
    assert np.max(np.abs(proj - pinv)) <= 1e-12 * np.max(np.abs(pinv))


def test_components_count_isolated_vertices_and_lone_triangles(lap):
    M, tri = _mesh("three_and_isolated")
    lab = lap.components(M, tri)
    assert lab.max() + 1 == 4 and lab[-1] == 3 and len(set(lab[-9:-1])) == 1


def test_laplacian_ignores_duplicates_degenerate_triangles_and_order(lap):
    M, tri = _mesh("icosphere")
    L = lap.graph_laplacian(M, tri)
    _, dup = _mesh("duplicates")
    assert np.array_equal(lap.graph_laplacian(M, dup[:-3]), L)
    perm = np.random.default_rng(0).permutation(len(tri))
    assert np.array_equal(lap.graph_laplacian(M, tri[perm][:, [1, 2, 0]]), L)
    assert np.array_equal(np.diag(L)[:12], np.full(12, 5.0)) and np.all(np.diag(L)[12:] == 6.0)   # icosahedron corners


def _check(lap, M, tri, scaling, gamma, tol, cap):
    Ks = lap.inverse_laplacian_kernel_matrix(M, tri, scaling, gamma)
    rank, kd, Ls = lap.triples_cholesky(Ks, tol, cap)
    cov = lap.triples_covariance(kd, Ls)
    _, L = lap.approximate_gp_cholesky_laplacian(M, np.zeros((M, 3)), tri, scaling, gamma, tol, cap)
    lit = L @ L.T
    assert rank == L.shape[1] == sum(kd)
    assert np.max(np.abs(cov - lit)) <= 1e-10 * np.max(np.abs(lit))
    return rank


# Late in the factorisation a vertex whose neighbours are all pivots is decoupled, with residual scaling / (L + gamma I)_ii:
# vertices of equal degree then tie exactly, and rounding orders them.  The tree and the isolated vertex of
# "three_and_isolated" tie in this way early, so the entry-wise comparison runs on the meshes where it is well posed
# (tests/test_gpmm_laplacian_gpu.py checks the device through the Nystrom form instead, which holds for any tie order).
@pytest.mark.parametrize("kind", ["sphere", "two", "patch"])
@pytest.mark.parametrize("gamma", [0.0, 1e-3, 1.0])
@pytest.mark.parametrize("tol,cap", [(0.01, None), (0.1, None), (0.3, None), (0.0, 100), (0.0, 101), (0.0, 102)])
def test_triples_equal_the_literal_factorisation(lap, kind, gamma, tol, cap):
    M, tri = _mesh(kind)
    rank = _check(lap, M, tri, 2.0, gamma, tol, cap)
    assert rank <= (cap or 3 * M)


def test_rel_tol_sweep_gives_every_rank_residue(lap):
    M, tri = _mesh("two")
    seen = {_check(lap, M, tri, 1.0, 0.5, tol, None) % 3 for tol in (0.2, 0.21, 0.22, 0.23, 0.24, 0.25)}
    assert seen == {0, 1, 2}


@pytest.mark.parametrize("gamma,expect", [(0.0, "null"), (1e-3, "full"), (1.0, "full")])
def test_full_factorisation_reproduces_the_kernel(lap, gamma, expect):
    M, tri = _mesh("three_and_isolated")
    Ks = lap.inverse_laplacian_kernel_matrix(M, tri, 3.0, gamma)
    ncomp = lap.components(M, tri).max() + 1
    rank, kd, Ls = lap.triples_cholesky(Ks, 0.0 if gamma > 0.0 else 1e-12)
    cov = lap.triples_covariance(kd, Ls)
    assert rank == (3 * M if expect == "full" else 3 * (M - ncomp))
    assert np.max(np.abs(cov - np.kron(Ks, np.eye(3)))) <= 1e-11 * np.max(np.abs(Ks))


def test_python_mirror_exposes_the_factory_and_the_kernel_select(monkeypatch):
    from gingr_b200 import api, io
    k = api.InvLapKernel(scaling=50.0, gamma=0.0)
    assert k.name == "InvLap" and k.printpars == "50.0_0.0"
    assert io.model_file_name("hand", 2000, k.name, k.printpars) == "hand_dec-2000_InvLap_50.0_0.0.h5.json"
    seen = {}
    monkeypatch.setattr(api.Model, "inverseLaplacian",
                        staticmethod(lambda ctx, ref, tri, sc, g, tol, cap=0: seen.update(sc=sc, g=g, tol=tol)))
    api.SimpleTriangleModels3D.create(None, np.zeros((4, 3)), np.zeros((1, 3), np.int32), api.InvLapKernel(2.0, 0.5), 0.02)
    assert seen == {"sc": 2.0, "g": 0.5, "tol": 0.02}
    with pytest.raises(NotImplementedError):
        api.SimpleTriangleModels3D.create(None, np.zeros((4, 3)), None, object())
    from gingr_b200 import _native as nat
    from ctypes import c_double, c_int32, c_void_p
    assert nat.SIGNATURES["gingr_gpmm_inverse_laplacian"] == (c_int32, [c_void_p, c_int32, nat.dp, nat.ip, c_int32, c_double,
                                                                       c_double, c_double, c_int32, nat.vpp, nat.ip])


def test_cpp_mirror_declares_the_factory(tmp_path):
    import shutil
    import subprocess
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    src = tmp_path / "lap.cpp"
    src.write_text(r'''
#include "gingr.hpp"
int main() {
  gingr::Model (*f)(const gingr::Context&, int, const double*, const int32_t*, int, double, double, double, int) =
      &gingr::Model::inverseLaplacian;
  return f == nullptr;
}
''')
    p = subprocess.run(["g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-I" + os.path.join(ROOT, "include"),
                        str(src)], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
