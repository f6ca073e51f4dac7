"""Phase times of the posterior model (gingr_model_posterior) at two sizes: a C4-size synthetic model (M = 20 000,
r = 2000, 3/4 of the vertices observed) and a GPMM built on the device at M = 100 000.  Per phase (CUDA events, from
gingr_posterior_model_profile): observations + system + factorisation, Jacobi (with its sweep count), the basis product on
DMMA (TFLOP/s over the 2 * 3M * r^2 flop it does, and that rate over the DMMA peak of FP64_PEAKS.json), mean / reference /
regression constants, and the whole call.  The card's name and power limit are read in the same run.
usage: python tools/time_posterior_model.py [--out FILE.json]"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

from gingr_b200 import api, synthetic


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def observations(model, frac, seed):
    rng = np.random.default_rng(seed)
    M = model.M
    pids = rng.permutation(M)[: int(frac * M)].astype(np.int32)
    pts = model.reference[pids] + rng.normal(scale=2.0, size=(len(pids), 3))
    return pids, pts, rng.uniform(0.5, 4.0, size=len(pids))


def measure(ctx, model, reps, peak):
    pids, pts, noise = observations(model, 0.75, 1)
    R, t = synthetic.euler_matrix(0.1, -0.05, 0.02), np.array([1.0, -2.0, 0.5])
    api.posterior_model(ctx, model, R, t, pids, pts, noise).close()        # warm-up: module load, every shape once
    runs = []
    for _ in range(reps):
        pm = api.posterior_model(ctx, model, R, t, pids, pts, noise)
        pm.close()
        runs.append(api.posterior_model_profile(ctx))
    best = min(runs, key=lambda p: p["total"])
    flop = 2.0 * 3 * model.M * model.rank * model.rank
    tflops = flop / (best["gemm"] * 1e-3) / 1e12
    return {"M": model.M, "r": model.rank, "observed": len(pids), "reps": reps, "best_ms": best,
            "all_total_ms": [p["total"] for p in runs], "gemm_tflops": tflops, "gemm_share_of_dmma_peak": tflops / peak}


def main():
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    with open(os.path.join(ROOT, "FP64_PEAKS.json")) as f:
        peak = json.load(f)["microbench"]["dmma_tflops_sustained"]
    ctx = api.Context(0)
    res = {"card": card(), "dmma_peak_tflops": peak}
    ref = synthetic.fibonacci_sphere(20000)
    _, basis, var = synthetic.make_gpmm(ref, 2000, 1)
    c4 = api.Model(ctx, ref, np.zeros(3 * 20000), basis, var)
    del basis
    res["c4_synthetic"] = measure(ctx, c4, 3, peak)
    c4.close()
    ref = synthetic.fibonacci_sphere(100000)
    big = api.Model.gaussianMixture(ctx, ref, None, [30.0], [50.0], 0.01, maxRank=1500)
    res["gpmm_100k"] = measure(ctx, big, 2, peak)
    big.close()
    print(json.dumps(res, indent=1))
    if out:
        with open(out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
