"""CPU tests of the device sample collection (gingr_mcmc_collect / gingr_mcmc_samples, mcmc.cuh): the Welford update of
mcmc_collect_kernel and the Chan pooling of mcmc_samples_pool_kernel restated in numpy against two-pass statistics, the
maps of api.SampleStatistics against helper's maps, and the agreement of the C, C++, Python and Scala surfaces."""
import ctypes
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROW, COL = (0, 0, 0, 1, 1, 2), (0, 1, 2, 1, 2, 2)


def _welford(xs):
    """mcmc_collect_kernel, one vertex set at a time: (count, mean [M, 3], scatter [M, 6])."""
    M = xs[0].shape[0]
    mean, sc, n = np.zeros((M, 3)), np.zeros((M, 6)), 0
    for x in xs:
        n += 1
        d = x - mean
        mean = mean + d / float(n)
        e = x - mean
        for q in range(6):
            sc[:, q] = sc[:, q] + d[:, ROW[q]] * e[:, COL[q]]
    return n, mean, sc


def _chan(parts):
    """mcmc_samples_pool_kernel: pairwise pooling in the order of `parts`."""
    na, mu, S = 0, None, None
    for nb, mb, Sb in parts:
        if nb == 0:
            continue
        if na == 0:
            na, mu, S = nb, mb.copy(), Sb.copy()
            continue
        nn = na + nb
        f, w = float(nb) / float(nn), (float(na) * float(nb)) / float(nn)
        d = mb - mu
        mu = mu + d * f
        for q in range(6):
            S[:, q] = (S[:, q] + Sb[:, q]) + (d[:, ROW[q]] * d[:, COL[q]]) * w
        na = nn
    return na, mu, S


def _full(S):
    C = np.empty((S.shape[0], 3, 3))
    for q in range(6):
        C[:, ROW[q], COL[q]] = C[:, COL[q], ROW[q]] = S[:, q]
    return C


def _two_pass(xs):
    x = np.stack(xs)
    mean = x.mean(0)
    d = x - mean
    return mean, np.einsum("nmi,nmj->mij", d, d)


def test_welford_and_chan_pooling_equal_two_pass_statistics():
    rng = np.random.default_rng(4)
    M = 50
    centre = rng.normal(size=(M, 3)) * 100.0          # large offset: the one-pass form must not lose the small spread
    xs = [centre + rng.normal(size=(M, 3)) * rng.uniform(0.01, 2.0, (M, 1)) for _ in range(37)]
    n, mean, S = _welford(xs)
    tm, tS = _two_pass(xs)
    assert n == 37
    assert np.max(np.abs(mean - tm)) <= 1e-12 * np.max(np.abs(tm))
    assert np.max(np.abs(_full(S) - tS)) <= 1e-10 * np.max(np.abs(tS))
    # unequal counts, an empty chain in the middle, pooled in order
    cuts = [0, 1, 1, 9, 30, 37]
    parts = [_welford(xs[a:b]) if b > a else (0, np.zeros((M, 3)), np.zeros((M, 6))) for a, b in zip(cuts[:-1], cuts[1:])]
    pn, pm, pS = _chan(parts)
    assert pn == 37
    assert np.max(np.abs(pm - tm)) <= 1e-12 * np.max(np.abs(tm))
    assert np.max(np.abs(_full(pS) - tS)) <= 1e-10 * np.max(np.abs(tS))
    # one chain pools to itself, bit for bit
    one = _chan([parts[3]])
    assert one[0] == parts[3][0] and np.array_equal(one[1], parts[3][1]) and np.array_equal(one[2], parts[3][2])


def _stats(api, helper, xs, tri):
    n, mean, S = _welford(xs)
    normal = sum(helper.vertex_normals(x, tri) for x in xs) / float(n)
    return api.SampleStatistics(n, mean, _full(S) / float(n - 1), normal)


def test_maps_from_statistics_equal_the_helper_maps():
    from gingr_b200 import api, helper, synthetic
    ref, tri = synthetic.sphere_mesh(120)
    rng = np.random.default_rng(8)
    xs = [ref * rng.uniform(0.9, 1.1) + rng.normal(size=ref.shape) * 0.05 for _ in range(23)]
    st = _stats(api, helper, xs, tri)
    want = helper.distance_map_total(xs)
    assert np.max(np.abs(st.distanceMapTotal() - want)) <= 1e-12 * np.max(want)
    want = helper.distance_map_normal(xs, tri)
    assert np.max(np.abs(st.distanceMapNormal() - want)) <= 1e-12 * np.max(want)
    want = helper.distance_map_normal(xs, tri, reference=ref, sumNormals=False)
    assert np.max(np.abs(st.distanceMapNormal(ref, tri, sumNormals=False) - want)) <= 1e-12 * np.max(want)
    # merge of unequal halves (one of them a single sample) = the statistics of all samples
    for cut in (1, 9):
        if cut == 1:   # gingr_mcmc_samples leaves the covariance of a single sample undefined
            a = api.SampleStatistics(1, xs[0].copy(), np.full((ref.shape[0], 3, 3), np.nan), helper.vertex_normals(xs[0], tri))
        else:
            a = _stats(api, helper, xs[:cut], tri)
        m = a.merge(_stats(api, helper, xs[cut:], tri))
        assert m.count == st.count
        for got, want in ((m.mean, st.mean), (m.cov, st.cov), (m.normal, st.normal)):
            assert np.max(np.abs(got - want)) <= 1e-12 * np.max(np.abs(want))
    empty = api.SampleStatistics(0, np.zeros_like(ref), np.zeros((ref.shape[0], 3, 3)), np.zeros_like(ref))
    assert empty.merge(st) is st and st.merge(empty) is st


def _header_protos():
    h = open(os.path.join(ROOT, "include", "gingr_cuda.h")).read()
    h = re.sub(r"/\*.*?\*/", "", h, flags=re.S)
    return {m.group(1): " ".join(m.group(2).split())
            for m in re.finditer(r"GINGR_API\s+int32_t\s+(gingr_\w+)\s*\(([^;]*?)\)\s*;", h)}


def test_sample_prototypes_agree_across_c_python_cpp_and_scala():
    from gingr_b200 import _native as nat
    protos = _header_protos()
    assert protos["gingr_mcmc_collect"] == "gingr_registration* reg, int32_t burn_in, int32_t take_every_n, int32_t total"
    assert protos["gingr_mcmc_samples"] == ("gingr_registration** regs, int32_t n, int64_t* count, double* mean , "
                                            "double* cov , double* normal")
    assert nat.SIGNATURES["gingr_mcmc_collect"] == (ctypes.c_int32, [ctypes.c_void_p] + [ctypes.c_int32] * 3)
    assert nat.SIGNATURES["gingr_mcmc_samples"] == (ctypes.c_int32, [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int32,
                                                                     ctypes.POINTER(ctypes.c_int64), nat.dp, nat.dp, nat.dp])
    shim = open(os.path.join(ROOT, "scala", "gingr", "api", "registration", "cuda", "GingrCudaNative.scala")).read()
    assert re.search(r'fn\("gingr_mcmc_collect",\s*JAVA_INT,\s*ADDRESS,\s*JAVA_INT,\s*JAVA_INT,\s*JAVA_INT\)', shim)
    assert re.search(r'fn\("gingr_mcmc_samples",\s*JAVA_INT,\s*ADDRESS,\s*JAVA_INT(,\s*ADDRESS){4}\)', shim)
    hpp = open(os.path.join(ROOT, "include", "gingr.hpp")).read()
    assert "gingr_mcmc_collect(h_, c.burnIn, c.takeEveryN, c.total)" in hpp
    assert re.search(r"gingr_mcmc_samples\(regs, 1, &s\.count,", hpp)


def test_sample_collection_defaults_are_those_of_samples_from_log():
    import inspect
    from gingr_b200 import api, helper
    c = api.SampleCollection()
    sig = inspect.signature(helper.samples_from_log).parameters
    assert (c.burnIn, c.takeEveryN, c.total) == (sig["burnIn"].default, sig["takeEveryN"].default, sig["total"].default)


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="no cuobjdump")
def test_collect_kernel_has_its_batched_twin_in_the_library():
    from gingr_b200 import build
    lib = build.LIB if os.path.exists(build.LIB) else build.build()
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    names = re.findall(r"Function : (\S+)", out)
    assert any("mcmc_collect_kernel_batched" in n for n in names)
    assert any("mcmc_collect_kernel" in n and "batched" not in n for n in names)
    assert any("mcmc_samples_pool_kernel" in n for n in names)
