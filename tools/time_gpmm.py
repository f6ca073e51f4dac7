"""GPMM construction on the device (gingr_gpmm_gaussian_mixture, or gingr_gpmm_gaussian_symmetric with kernel
"symmetric"): wall time incl. the host syncs of the batch / sweep checks.
usage: python tools/time_gpmm.py [M] [sigma] [scaling] [relTol] [gaussian|symmetric]"""
import json, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from gingr_b200 import api, synthetic
M = int(sys.argv[1]) if len(sys.argv) > 1 else 100000
sigma = float(sys.argv[2]) if len(sys.argv) > 2 else 70.0
scaling = float(sys.argv[3]) if len(sys.argv) > 3 else 50.0
tol = float(sys.argv[4]) if len(sys.argv) > 4 else 0.01
kernel = sys.argv[5] if len(sys.argv) > 5 else "gaussian"
build = {"gaussian": api.Model.gaussianMixture, "symmetric": api.Model.gaussianSymmetric}[kernel]
ref = synthetic.fibonacci_sphere(M)
ctx = api.Context(0)
build(ctx, ref[:2000], None, [sigma], [scaling], tol).close()     # warm-up (module load)
ctx.synchronize()
l0 = ctx.launch_count
t0 = time.perf_counter()
m = build(ctx, ref, None, [sigma], [scaling], tol)
ctx.synchronize()
dt = time.perf_counter() - t0
_, _, basis, var = m.download()
# trace(K) = sum_i 3 s for the Gaussian kernel, sum_i (3 s + e_i) with e_i = s exp(-4 x_i0^2 / sigma^2) for the symmetric one
tr = 3.0 * M * scaling + (float(np.sum(scaling * np.exp(-4.0 * ref[:, 0] ** 2 / sigma ** 2))) if kernel == "symmetric" else 0.0)
print(json.dumps({"kernel": kernel, "M": M, "sigma": sigma, "scaling": scaling, "rel_tol": tol, "rank": m.rank, "seconds": dt,
                  "launches": ctx.launch_count - l0, "residual_trace_fraction": float((tr - var.sum()) / tr),
                  "orthonormality_error": float(np.max(np.abs(basis.T @ basis - np.eye(m.rank))))}))
