"""Per-iteration E-step cost of the seeded C4 chain (bench.py inputs: M = 20 000, N = 200 000, rank 2000, w = 0.1), with the
tile-pair culling of the E-step as the library chooses it and once forced off (GINGR_ESTEP_CULL=0).  Per iteration it prints
the sigma2 going into the iteration, the live fraction of the tile pairs of each sweep (counted on the device by the cull
kernels) and the sweep times (CUDA events; each bracket includes that sweep's cull kernels).
usage: python tools/time_estep_cull.py [iterations] [--out FILE.json]"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from gingr_b200 import api


def run(ctx, inputs, iters, cull):
    if cull is None:
        os.environ.pop("GINGR_ESTEP_CULL", None)
    else:
        os.environ["GINGR_ESTEP_CULL"] = "1" if cull else "0"
    ref, mean, basis, var, target = inputs
    model = api.Model(ctx, ref, mean, basis, var)
    tgt = api.Target(ctx, target)
    reg = api.CpdRegistration(ctx, model, tgt, api.CpdConfiguration(maxIterations=10 ** 6, w=bench.W_OUTLIER))
    reg.initializeState(globalTransformation=api.RIGID_TRANSFORMS)
    reg.setProfiling(True)
    rows = []
    for it in range(iters):
        sigma2 = reg.downloadState().sigma2
        reg.updateChain(1)
        ms, n = reg.getProfile()
        rows.append({"iter": it, "sigma2": sigma2, "live_a": ms[6] / n, "live_b": ms[7] / n,
                     "sweep_a_ms": ms[0] / n, "sweep_b_ms": ms[1] / n, "iteration_ms": ms[4] / n})
    reg.close(); model.close(); tgt.close()
    os.environ.pop("GINGR_ESTEP_CULL", None)
    return rows


def main():
    iters = int(sys.argv[1]) if len(sys.argv) > 1 and not sys.argv[1].startswith("-") else 24
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    ctx = api.Context(0)
    inputs = bench.make_inputs("c4")
    run(ctx, inputs, 2, None)   # warm-up: module load, graph capture
    res = {"auto": run(ctx, inputs, iters, None), "dense": run(ctx, inputs, iters, False)}
    print(f"{'it':>3} {'sigma2':>9} {'live A':>7} {'live B':>7} {'A ms':>7} {'B ms':>7} {'A dense':>8} {'B dense':>8}")
    for a, d in zip(res["auto"], res["dense"]):
        print(f"{a['iter']:3d} {a['sigma2']:9.2f} {a['live_a']:7.3f} {a['live_b']:7.3f} {a['sweep_a_ms']:7.3f} {a['sweep_b_ms']:7.3f}"
              f" {d['sweep_a_ms']:8.3f} {d['sweep_b_ms']:8.3f}")
    if out:
        with open(out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
