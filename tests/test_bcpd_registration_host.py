"""CPU tests of the BCPD configuration of GingrAlgorithm (GINGR_ALGO_BCPD): the oracle's formulas against their literal
definitions (the per-vertex variance against the dense 3M x 3M posterior covariance, the sigma2 terms against the double
sum over a materialised P), and the agreement of the C, C++, Python and Scala surfaces of the new calls."""
import ctypes
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bc(oracle):
    from oracle import bcpd
    return bcpd


def _model(oracle, M=40, r=12, seed=3):
    rng = np.random.default_rng(seed)
    ref = rng.normal(size=(M, 3)) * 10.0
    basis, _ = np.linalg.qr(rng.normal(size=(3 * M, r)))
    return oracle.Gpmm(ref, rng.normal(size=3 * M) * 0.1, basis, np.sort(rng.uniform(1.0, 9.0, r))[::-1].copy())


def test_vertex_variance_is_the_diagonal_of_the_dense_posterior_covariance(oracle, bc):
    model = _model(oracle)
    rng = np.random.default_rng(5)
    M = model.M
    R = oracle.euler_to_matrix(0.3, -0.2, 0.5)
    posed = model.transform(R, np.array([1.0, 2.0, -3.0]))
    pids = np.arange(M)
    var = rng.uniform(0.5, 4.0, M)
    cov = np.eye(3)[None] * var[:, None, None]
    pts = posed.instance(np.zeros(model.rank)) + rng.normal(size=(M, 3))
    _, Minv = posed.posterior_coefficients(pids, pts, cov)
    Q = posed.basis * np.sqrt(posed.variance)[None, :]
    dense = Q @ Minv @ Q.T                                             # 3M x 3M posterior covariance
    lit = np.array([np.trace(dense[3 * m:3 * m + 3, 3 * m:3 * m + 3]) / 3.0 for m in range(M)])
    assert np.max(np.abs(bc.posterior_vertex_variance(model, Minv) - lit)) <= 1e-13 * np.max(lit)
    # no observations: the prior variance, tr(Phi_m Lambda Phi_m^T) / 3
    prior = Q @ Q.T
    lit0 = np.array([np.trace(prior[3 * m:3 * m + 3, 3 * m:3 * m + 3]) / 3.0 for m in range(M)])
    assert np.max(np.abs(bc.prior_variance(model) - lit0)) <= 1e-13 * np.max(lit0)
    assert np.max(np.abs(bc.posterior_vertex_variance(model, np.eye(model.rank)) - lit0)) <= 1e-13 * np.max(lit0)


def test_sigma2_terms_equal_the_literal_double_sum(oracle, bc):
    rng = np.random.default_rng(11)
    M, N = 30, 45
    fit = rng.normal(size=(M, 3)) * 3.0
    x = rng.normal(size=(N, 3)) * 3.0
    P = oracle.bcpd_P(fit, x, rng.uniform(0.0, 0.5, M), rng.dirichlet(np.ones(M)), 4.0, 1.3, 0.1)
    sXX, sXY, sYY, nhat = bc.sigma2_terms(P, x, fit)
    lit = sum(P[m, n] * float(np.sum((x[n] - fit[m]) ** 2)) for m in range(M) for n in range(N))
    assert abs((sXX - 2.0 * sXY + sYY) - lit) <= 1e-12 * lit
    assert abs(nhat - P.sum()) <= 1e-13 * nhat


def _header_protos():
    h = open(os.path.join(ROOT, "include", "gingr_cuda.h")).read()
    h = re.sub(r"/\*.*?\*/", "", h, flags=re.S)
    return {m.group(1): " ".join(m.group(2).split())
            for m in re.finditer(r"GINGR_API\s+int32_t\s+(gingr_\w+)\s*\(([^;]*?)\)\s*;", h)}


def test_bcpd_prototypes_agree_across_c_python_and_scala():
    from gingr_b200 import _native as nat
    protos = _header_protos()
    assert protos["gingr_registration_set_bcpd"] == "gingr_registration* reg, double kappa"
    assert protos["gingr_bcpd_state_download"] == "gingr_registration* reg, double* alpha , double* sigma"
    assert nat.SIGNATURES["gingr_registration_set_bcpd"] == (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_double])
    assert nat.SIGNATURES["gingr_bcpd_state_download"] == (ctypes.c_int32, [ctypes.c_void_p, nat.dp, nat.dp])
    shim = open(os.path.join(ROOT, "scala", "gingr", "api", "registration", "cuda", "GingrCudaNative.scala")).read()
    assert re.search(r'fn\("gingr_registration_set_bcpd",\s*JAVA_INT,\s*ADDRESS,\s*JAVA_DOUBLE\)', shim)
    assert re.search(r'fn\("gingr_bcpd_state_download",\s*JAVA_INT,\s*ADDRESS,\s*ADDRESS,\s*ADDRESS\)', shim)


def test_algorithm_routing_and_config_size():
    from gingr_b200 import _native as nat, api
    h = open(os.path.join(ROOT, "include", "gingr_cuda.h")).read()
    assert re.search(r"#define GINGR_ALGO_BCPD 2\b", h)
    assert (nat.ALGO_CPD, nat.ALGO_ICP, nat.ALGO_BCPD) == (0, 1, 2)
    assert ctypes.sizeof(nat.GingrConfig) == 64
    c = api.BcpdConfiguration(maxIterations=7, initialSigma=2.5, w=0.1, lambda_=3.0, kappa=10.0).to_pod()
    assert c.algorithm == nat.ALGO_BCPD and c.max_iterations == 7 and c.w == 0.1 and c.lambda_ == 3.0
    assert c.has_initial_sigma == 1 and c.initial_sigma == 2.5
    d = api.BcpdConfiguration()
    cpd = api.CpdConfiguration()
    assert (d.maxIterations, d.threshold, d.useLandmarkCorrespondence, d.initialSigma, d.w, d.lambda_, d.kappa) == \
        (cpd.maxIterations, cpd.threshold, cpd.useLandmarkCorrespondence, cpd.initialSigma, cpd.w, cpd.lambda_, 1.0)
    assert issubclass(api.BcpdRegistration, api.GingrAlgorithm) and api.BcpdRegistration.name == "BCPD"


def test_cpp_bcpd_configuration_matches_the_python_mirror(tmp_path):
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    src = tmp_path / "t.cpp"
    src.write_text('#include "gingr.hpp"\n#include <cstdio>\n'
                   "int main() { gingr::BcpdConfiguration c; c.w = 0.1; c.kappa = 10.0; gingr_config p = c.toPod();\n"
                   '  std::printf("%d %d %.17g %.17g %d %zu\\n", p.algorithm, p.max_iterations, p.w, p.lambda, p.has_initial_sigma,\n'
                   "              sizeof(gingr_config));\n"
                   "  static_assert(std::is_same_v<gingr::BcpdRegistration, gingr::GingrAlgorithm<gingr::BcpdConfiguration>>);\n"
                   "  return 0; }\n")
    exe = tmp_path / "t"
    subprocess.run(["g++", "-std=c++17", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    assert out == ["2", "100", "0.10000000000000001", "1", "0", "64"]
