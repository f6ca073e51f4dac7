"""CPU tests of the mirror-symmetric GPMM construction (gingr_gpmm_gaussian_symmetric): the device's two-block merge,
restated in numpy (oracle/symmetric.py), gives the rank and covariance of the literal 3M x 3M pivoted Cholesky of
scalismo's symmetrised kernel; the kernel matrix itself; and the Python and C++ mirrors of the new factory."""
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def sym():
    from oracle import symmetric
    return symmetric


def _cloud(kind, n, seed):
    rng = np.random.default_rng(seed)
    p = rng.normal(size=(n, 3)) * 40.0
    if kind == "plane":                      # a fifth of the points exactly on x = 0
        p[: n // 5, 0] = 0.0
    elif kind == "mirrored":                 # every point's image is in the set, plus three points on the plane
        h = p[: n // 2]
        p = np.vstack([h, h * [-1.0, 1.0, 1.0], rng.normal(size=(3, 3)) * [0.0, 40.0, 40.0]])
    elif kind == "far":                      # e_i = exp(-4 x^2 / sigma^2) underflows: K- and K+ are both k
        p[:, 0] = np.abs(p[:, 0]) + 1e4
    return p


def _check(sym, ref, sig, sc, tol, cap):
    _, L = sym.approximate_gp_cholesky_symmetric(ref, sig, sc, tol, cap)
    rank, kd, _, cov = sym.merged_cholesky_symmetric(ref, sig, sc, tol, cap)
    lit = L @ L.T
    assert rank == L.shape[1] == sum(kd)
    assert np.max(np.abs(cov - lit)) <= 1e-10 * np.max(np.abs(lit))
    return rank, kd


@pytest.mark.parametrize("kind", ["generic", "plane", "mirrored", "far"])
@pytest.mark.parametrize("sig,sc", [([60.0], [50.0]), ([60.0, 20.0], [50.0, 10.0])])
@pytest.mark.parametrize("tol,cap", [(0.1, None), (0.03, None), (0.01, 20), (0.3, None), (0.05, 31)])
def test_merge_equals_the_literal_factorisation(sym, kind, sig, sc, tol, cap):
    # on mirrored sets K+ / K- lose rank: the tolerances stay well above the rounding floor, below which the literal
    # algorithm's own pivots are noise
    ref = _cloud(kind, 45, 7)
    _check(sym, ref, sig, sc, tol, cap)


def test_far_points_tie_the_blocks_and_the_index_rule_decides(sym):
    ref = _cloud("far", 40, 3)
    M = len(ref)
    K = sym.symmetric_gaussian_kernel_matrix(ref, [60.0], [50.0])
    assert np.array_equal(K[0::3, 0::3], K[1::3, 1::3])          # k_m underflows to exactly 0
    rank, kd = _check(sym, ref, [60.0], [50.0], 0.2, None)
    # equal blocks: the literal sequence takes whole triples (p, 0), (p, 1), (p, 2)
    assert max(kd) - min(kd) <= 1 and kd == sorted(kd, reverse=True)
    assert 0 < rank < 3 * M


@pytest.mark.parametrize("cap", [1, 2, 3, 4, 5, 7, 8, 13, 20])
def test_caps_cut_between_coordinates_and_blocks(sym, cap):
    ref = _cloud("plane", 40, 11)
    rank, kd = _check(sym, ref, [50.0], [30.0], 0.0, cap)
    assert rank == cap


def test_caps_leave_coordinates_one_and_two_apart_and_split_the_blocks(sym):
    ref = _cloud("generic", 40, 5)
    seen = set()
    for cap in range(1, 25):
        _, kd = _check(sym, ref, [50.0], [30.0], 0.0, cap)
        assert kd[1] - kd[2] in (0, 1)
        seen.add(kd[1] - kd[2])
    assert seen == {0, 1}


def test_rel_tol_sweep_gives_every_rank_residue(sym):
    ref = _cloud("plane", 40, 2)
    residues = set()
    for tol in np.linspace(0.02, 0.5, 30):
        rank, _ = _check(sym, ref, [60.0], [30.0], float(tol), None)
        residues.add(rank % 3)
    assert residues == {0, 1, 2}


def test_kernel_matrix_entries_symmetry_and_mirror_invariance(sym):
    ref = _cloud("mirrored", 30, 4)
    M = len(ref)
    sig, sc = [50.0, 15.0], [20.0, 5.0]
    K = sym.symmetric_gaussian_kernel_matrix(ref, sig, sc)

    def k(x, y):
        return sum(s * np.exp(-np.sum((x - y) ** 2) / (g * g)) for g, s in zip(sig, sc))

    S = np.array([-1.0, 1.0, 1.0])
    for i, j in [(0, 1), (3, 17), (5, 5), (M - 1, 2)]:
        for d in range(3):
            want = k(ref[i], ref[j]) + S[d] * k(S * ref[i], ref[j])
            assert abs(K[3 * i + d, 3 * j + d] - want) <= 1e-13 * sum(sc)
            for e in range(3):
                if e != d:
                    assert K[3 * i + d, 3 * j + e] == 0.0
    assert np.max(np.abs(K - K.T)) <= 1e-13 * sum(sc)
    assert np.linalg.eigvalsh(K).min() >= -1e-9 * sum(sc)
    # the diagonal: s - e_i for x, s + e_i for y and z
    e = sum(s * np.exp(-4.0 * ref[:, 0] ** 2 / (g * g)) for g, s in zip(sig, sc))
    assert np.max(np.abs(np.diag(K)[0::3] - (sum(sc) - e))) <= 1e-13 * sum(sc)
    assert np.max(np.abs(np.diag(K)[1::3] - (sum(sc) + e))) <= 1e-13 * sum(sc)
    # P K P^T = K for the mirror permutation-reflection P of a symmetric set
    P = _mirror_operator(ref)
    assert np.max(np.abs(P @ K @ P.T - K)) <= 1e-12 * sum(sc)
    # points on the plane: their x rows and columns vanish
    on = np.flatnonzero(ref[:, 0] == 0.0)
    assert on.size == 3 and np.all(K[3 * on, :] == 0.0)


def _mirror_operator(ref):
    """P[3 pi(i) + d, 3 i + d] = S_d with pi(i) the index of the mirror image of point i."""
    M = len(ref)
    img = ref * [-1.0, 1.0, 1.0]
    pi = [int(np.argmin(np.sum((ref - img[i]) ** 2, axis=1))) for i in range(M)]
    assert all(np.array_equal(ref[pi[i]], img[i]) for i in range(M))
    P = np.zeros((3 * M, 3 * M))
    for i in range(M):
        for d, s in enumerate((-1.0, 1.0, 1.0)):
            P[3 * pi[i] + d, 3 * i + d] = s
    return P


def test_python_mirror_exposes_the_factory_and_the_kernel_select(monkeypatch):
    from gingr_b200 import api, io
    k = api.GaussSymKernel(scaling=50.0, sigma=70.0)
    assert k.name == "GaussSym" and k.printpars == "50.0_70.0"
    assert io.model_file_name("skull", None, k.name, k.printpars) == "skull_dec-full_GaussSym_50.0_70.0.h5.json"
    with pytest.raises(ValueError):
        api.Model.gaussianSymmetric(None, np.zeros((4, 3)), None, [1.0, 2.0], [1.0])
    seen = {}
    monkeypatch.setattr(api.Model, "gaussianSymmetric",
                        staticmethod(lambda ctx, ref, tri, sig, sc, tol, cap=0: seen.update(sig=sig, sc=sc, tol=tol)))
    api.SimpleTriangleModels3D.create(None, np.zeros((4, 3)), None, k, 0.02)
    assert seen == {"sig": [70.0], "sc": [50.0], "tol": 0.02}
    with pytest.raises(NotImplementedError):
        api.SimpleTriangleModels3D.create(None, np.zeros((4, 3)), None, object())
    from gingr_b200 import _native as nat
    assert nat.SIGNATURES["gingr_gpmm_gaussian_symmetric"] == nat.SIGNATURES["gingr_gpmm_gaussian_mixture"]


def test_cpp_mirror_declares_the_factory(tmp_path):
    import shutil
    import subprocess
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    src = tmp_path / "sym.cpp"
    src.write_text(r'''
#include "gingr.hpp"
int main() {
  gingr::Model (*f)(const gingr::Context&, int, const double*, const int32_t*, int, const std::vector<double>&,
                    const std::vector<double>&, double, int) = &gingr::Model::gaussianSymmetric;
  return f == nullptr;
}
''')
    p = subprocess.run(["g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-I" + os.path.join(ROOT, "include"),
                        str(src)], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
