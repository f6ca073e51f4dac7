"""GPMM construction on the device (gingr_gpmm_gaussian_mixture, gingr_gpmm_gaussian_symmetric with kernel "symmetric",
gingr_gpmm_inverse_laplacian with kernel "laplacian"): wall time incl. the host syncs of the batch / sweep checks.
usage: python tools/time_gpmm.py [M] [sigma] [scaling] [relTol] [gaussian|symmetric]
       python tools/time_gpmm.py laplacian [M] [gamma] [scaling] [relTol] [runs]
The laplacian form builds on an icosphere (M = 642, 2562, ...) or else the hull of M random points on a sphere, and
reports the best and spread of `runs` wall times, then per-phase device times from torch.profiler runs of their own.
The phases follow the build in device order: assembly + inverse (everything before the first pivoted-Cholesky kernel:
Laplacian, data-flow Cholesky, transpose, Gram), pivoted Cholesky, Jacobi, and assembly + constants (everything from the
basis assembly on: topology and the regression constants, which use the Gram and Cholesky kernels too)."""
import json, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from gingr_b200 import api, synthetic


def laplacian(argv):
    M = int(argv[0]) if len(argv) > 0 else 642
    gamma = float(argv[1]) if len(argv) > 1 else 0.0
    scaling = float(argv[2]) if len(argv) > 2 else 1.0
    tol = float(argv[3]) if len(argv) > 3 else 0.01
    runs = int(argv[4]) if len(argv) > 4 else 3
    s = {162: 2, 642: 3, 2562: 4, 10242: 5}.get(M)
    ref, tri = synthetic.icosphere(s) if s else synthetic.random_sphere_mesh(M, 0)
    ctx = api.Context(0)
    api.Model.inverseLaplacian(ctx, ref[:42], synthetic.icosphere(1)[1], scaling, gamma, tol).close()   # module load
    ctx.synchronize()
    wall, launches = [], []
    for _ in range(runs):
        l0 = ctx.launch_count
        t0 = time.perf_counter()
        m = api.Model.inverseLaplacian(ctx, ref, tri, scaling, gamma, tol)
        ctx.synchronize()
        wall.append(time.perf_counter() - t0)
        launches.append(ctx.launch_count - l0)
        rank = m.rank
        m.close()
    import torch
    from torch.profiler import ProfilerActivity, profile
    # the kernels that open a phase; every device event belongs to the phase of the last such kernel before it
    opens = [("pivoted_cholesky", ("gpmm_init_diag", "gpmm_argmax", "gpmm_column")),
             ("jacobi", ("gpmm_jacobi", "gpmm_colnorm")),
             ("assembly_constants", ("gpmm_assemble",))]
    phases = []
    for _ in range(runs):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            m = api.Model.inverseLaplacian(ctx, ref, tri, scaling, gamma, tol)
            ctx.synchronize()
        m.close()
        ms = {"assembly_inverse": 0.0, "pivoted_cholesky": 0.0, "jacobi": 0.0, "assembly_constants": 0.0}
        phase = "assembly_inverse"
        events = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        for e in sorted(events, key=lambda e: e.time_range.start):
            phase = next((p for p, keys in opens if any(k in e.name for k in keys)), phase)
            ms[phase] += e.device_time / 1000.0
        phases.append(ms)
    out = {"kernel": "laplacian", "M": M, "T": int(len(tri)), "gamma": gamma, "scaling": scaling, "rel_tol": tol, "rank": rank,
           "launches": launches[0], "seconds_best": min(wall), "seconds_runs": wall,
           "phase_ms_best": {k: min(p[k] for p in phases) for k in phases[0]},
           "phase_ms_runs": phases}
    print(json.dumps(out))


if len(sys.argv) > 1 and sys.argv[1] == "laplacian":
    laplacian(sys.argv[2:])
    sys.exit(0)

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
