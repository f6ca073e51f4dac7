"""n independent deterministic CPD registrations (M = N = 200, rank 50) through gingr_update_batch.
usage: python tools/time_cpd_batch.py [n] [iters]"""
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from gingr_b200 import api, synthetic

n = int(sys.argv[1]) if len(sys.argv) > 1 else 256
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 20
M, N, r = 200, 200, 50
ctx = api.Context(0)
ref, tri = synthetic.sphere_mesh(M)
mean, basis, var = synthetic.make_gpmm(ref, r, 1)
tv, tt = synthetic.sphere_mesh(N)
model = api.Model(ctx, ref, mean, basis, var, tri)
tgt = api.Target(ctx, synthetic.make_target(tv, 0), tt)
chains = [api.CpdRegistration(ctx, model, tgt, api.CpdConfiguration(maxIterations=10 ** 6, w=0.1)) for _ in range(n)]
for c in chains:
    c.initializeState(globalTransformation=api.RIGID_TRANSFORMS)
api.update_batch(chains, 3)
ctx.synchronize()
l0 = ctx.launch_count
t0 = time.perf_counter()
api.update_batch(chains, iters)
ctx.synchronize()
dt = time.perf_counter() - t0
print(json.dumps({"workload": f"{n} CPD registrations M=N={M} rank={r}",
                  "chain_iterations_per_s": n * iters / dt, "ms_per_iteration_of_all_chains": dt / iters * 1e3,
                  "launches_per_iteration": (ctx.launch_count - l0) / iters,
                  "finite": bool(np.all(np.isfinite(chains[-1].downloadState().fit)))}))
