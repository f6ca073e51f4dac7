"""Host-only checks behind the posterior model (gingr_model_posterior): scalismo's low-rank posterior model, as the GPU
tests restate it from the oracle's regression, equals dense Gaussian conditioning of the 3M x 3M prior covariance; the
registration-level oracle (oracle.posterior_model) is the same formula; and the basis product of the library runs on the
FP64 tensor pipe (SASS DMMA.8x8x4, no DFMA, no local-memory spill).  No GPU."""
import collections
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "gingr_b200", "lib", "libgingr_cuda.so")


def _reference_posterior(oracle, m, R, t, pids, pts, cov):
    """model.transform(R, t).posterior(obs) as a model: reference and mean of the posed model plus basis (D c),
    basis posed.basis U, variance s with svd(D Minv D) = U diag(s) U^T (the formula of oracle.posterior_model)."""
    posed = m.transform(R, t)
    c, Minv = posed.posterior_coefficients(pids, pts, cov)
    D = np.sqrt(m.variance)
    U, s, _ = np.linalg.svd(D[:, None] * Minv * D[None, :])
    return oracle.Gpmm(posed.ref, posed.mean + posed.basis @ (D * c), posed.basis @ U, s, posed.tri)


def _small_model(oracle, M=40, r=15, seed=0, orthonormal=True):
    from gingr_b200 import synthetic
    ref, tri = synthetic.sphere_mesh(M)
    _, basis, var = synthetic.make_gpmm(ref, r, seed, orthonormal=orthonormal)
    mean = np.random.default_rng(seed + 1).normal(scale=0.5, size=3 * M)
    return oracle.Gpmm(ref, mean, basis, var, tri)


@pytest.mark.parametrize("kind", ["iso", "full"])
@pytest.mark.parametrize("orthonormal", [True, False])
def test_low_rank_posterior_model_is_dense_gaussian_conditioning(oracle, kind, orthonormal):
    m = _small_model(oracle, orthonormal=orthonormal)
    M = m.M
    rng = np.random.default_rng(3)
    R, t = oracle.euler_to_matrix(0.3, -0.2, 0.1), np.array([1.0, -2.0, 0.5])
    posed = m.transform(R, t)
    pids = np.array([0, 4, 4, 9, 13, 21, 30, 39], dtype=np.int32)
    n = len(pids)
    pts = posed.instance(rng.normal(size=m.rank))[pids] + rng.normal(scale=0.3, size=(n, 3))
    if kind == "iso":
        cov = np.eye(3)[None] * rng.uniform(0.1, 2.0, size=n)[:, None, None]
    else:
        A = rng.normal(size=(n, 3, 3))
        cov = A @ np.transpose(A, (0, 2, 1)) + 0.2 * np.eye(3)
    got = _reference_posterior(oracle, m, R, t, pids, pts, cov)
    # dense: f ~ N(mu, K) over the 3M coordinates of the posed model, y = f[obs rows] + eps, eps ~ N(0, blockdiag(cov))
    mu = (posed.ref.reshape(-1) + posed.mean)
    K = (posed.basis * posed.variance) @ posed.basis.T
    rows = (3 * pids[:, None] + np.arange(3)[None, :]).reshape(-1)
    S = K[np.ix_(rows, rows)]
    for k in range(n):
        S[3 * k:3 * k + 3, 3 * k:3 * k + 3] += cov[k]
    G = np.linalg.solve(S, K[rows, :]).T                          # K[:, o] S^-1
    mean_dense = mu + G @ (pts.reshape(-1) - mu[rows])
    cov_dense = K - G @ K[rows, :]
    scale = float(np.max(np.abs(K)))
    assert np.max(np.abs(got.ref.reshape(-1) + got.mean - mean_dense)) <= 1e-9 * np.max(np.abs(mu))
    assert np.max(np.abs((got.basis * got.variance) @ got.basis.T - cov_dense)) <= 1e-9 * scale
    assert np.all(np.diff(got.variance) <= 1e-12 * got.variance[0])


def test_registration_level_oracle_is_the_same_formula(oracle):
    from gingr_b200 import synthetic
    m = _small_model(oracle, M=50, r=12, seed=2)
    tv, tt = synthetic.sphere_mesh(60)
    target = synthetic.make_target(tv, 1)
    algo = oracle.CpdAlgorithm(oracle.CpdConfig(max_iterations=5, w=0.1))
    st = algo.initialize(oracle.initial_state(m, target, tt, global_transformation=oracle.RIGID_TRANSFORMS,
                                              R0=oracle.euler_to_matrix(0.05, 0.0, -0.02), t0=[1.0, 0.0, 0.5]))
    pids, pts, cov = algo.observations(st)
    want = _reference_posterior(oracle, m, st.params.rotation_matrix(), st.params.translation, pids, pts, cov)
    got = oracle.posterior_model(algo, st)
    for a, b in ((got.ref, want.ref), (got.mean, want.mean), (got.basis, want.basis), (got.variance, want.variance)):
        assert np.max(np.abs(a - b)) <= 1e-12 * max(float(np.max(np.abs(b))), 1.0)


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="no cuobjdump")
def test_basis_product_runs_on_the_fp64_tensor_pipe():
    if not os.path.exists(LIB):
        from gingr_b200 import build
        build.build()
    out = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
    blocks = [b for b in re.split(r"\n\s*Function : ", out)[1:] if "basis_rotate_kernel" in b.split("\n", 1)[0]]
    assert len(blocks) == 1
    ops = collections.Counter(re.findall(r"^\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_]*(?:\.[A-Z0-9_x]+)*)",
                                         blocks[0], flags=re.M))

    def count(prefix):
        return sum(v for k, v in ops.items() if k == prefix or k.startswith(prefix + "."))

    assert any(k.startswith("DMMA.8x8x4") for k in ops) and count("DMMA") >= 96
    assert count("DFMA") == 0
    assert count("LDL") == 0 and count("STL") == 0
