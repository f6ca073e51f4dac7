"""Cholesky + back substitution of the r x r posterior matrix alone (profile slot 3) on a small registration whose
iteration is dominated by it.   usage: python tools/time_chol.py [r] [iters]"""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from gingr_b200 import api, synthetic
r = int(sys.argv[1]) if len(sys.argv) > 1 else 2000
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 10
M, N = max(700, r + 100), 1000
ref = synthetic.fibonacci_sphere(M)
mean, basis, var = synthetic.make_gpmm(ref, r, 1, orthonormal=False)
target = synthetic.make_target(synthetic.fibonacci_sphere(N), 0)
ctx = api.Context(0)
model = api.Model(ctx, ref, mean, basis, var)
tgt = api.Target(ctx, target)
reg = api.CpdRegistration(ctx, model, tgt, api.CpdConfiguration(maxIterations=10 ** 6, w=0.1))
reg.initializeState(globalTransformation=api.RIGID_TRANSFORMS)
reg.updateChain(3)
ctx.synchronize()
reg.setProfiling(True)
reg.updateChain(iters)
ms, it = reg.getProfile()
st = reg.downloadState()
assert np.all(np.isfinite(st.fit)) and st.status != api.STATUS_MODEL_FLEXIBILITY_ERROR
print(json.dumps({"rank": r, "iters": it, "cholesky_backsolve_ms": ms[3] / it, "iteration_ms": ms[4] / it,
                  "alpha_checksum": float(np.sum(st.modelParameters.shape)), "sigma2": st.sigma2}))
