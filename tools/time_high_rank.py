"""One CPD iteration per phase at ranks around and above 64 x the SM count (9472 on a B200), up to 18 000, the largest rank
the device builders produce.  For each r in --ranks: M = ceil(r / 3) template points (the smallest M with 3M >= r),
N = 4M target points on a sphere, a seeded column-normalised Gaussian basis, w = 0.1, RigidTransforms.  Per phase (CUDA
events of gingr_registration_get_profile, best of `reps` single-iteration chains after one warm-up iteration): E-step
sweeps A / B, Gram, Cholesky + back substitution, whole iteration.  The card's name and power limit are read in the same
run.

--c4 instead times the C4 workload of bench.py (M = 20 000, N = 200 000, r = 2000) and reports every rep's Cholesky +
back-substitution phase; with --root DIR the package is imported from another source tree (for instance a build of the
parent commit), so that two builds can be alternated in one session.
usage: python tools/time_high_rank.py [--ranks 2000,9472,...] [--reps K] [--out FILE.json]
       python tools/time_high_rank.py --c4 [--root DIR] [--reps K] [--out FILE.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PHASES = ("estep_sweep_a", "estep_sweep_b", "gram", "cholesky_backsolve", "iteration")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def measure(api, reg, reps):
    reg.initializeState(globalTransformation=api.RIGID_TRANSFORMS)
    reg.updateChain(1)                      # warm-up: capture, module load
    reg.setProfiling(True)
    runs = []
    for _ in range(reps):
        reg.updateChain(1)
        ms, it = reg.getProfile()
        runs.append([float(v) for v in ms[:5] / max(it, 1)])
    reg.setProfiling(False)
    return runs


def one_rank(api, synthetic, np, ctx, r, reps):
    M = -(-r // 3)
    N = 4 * M
    ref = synthetic.fibonacci_sphere(M)
    target = synthetic.make_target(synthetic.fibonacci_sphere(N), 0)
    mean, basis, var = synthetic.make_gpmm(ref, r, 1, orthonormal=False)
    model = api.Model(ctx, ref, mean, basis, var)
    del basis
    tgt = api.Target(ctx, target)
    reg = api.CpdRegistration(ctx, model, tgt, api.CpdConfiguration(w=0.1))
    t0 = time.perf_counter()
    runs = measure(api, reg, reps)
    wall = time.perf_counter() - t0
    st = reg.downloadState()
    reg.close()
    tgt.close()
    model.close()
    best = min(runs, key=lambda v: v[4])
    return {"r": r, "M": M, "N": N, "blocks_of_64": -(-r // 64), "best_ms": dict(zip(PHASES, best)),
            "iteration_ms_all": [v[4] for v in runs], "wall_s_warmup_and_reps": wall,
            "finite": bool(np.all(np.isfinite(st.fit)) and np.isfinite(st.sigma2))}


def c4(api, synthetic, ctx, reps):
    M, N, R = 20000, 200000, 2000
    ref = synthetic.fibonacci_sphere(M)
    target = synthetic.make_target(synthetic.fibonacci_sphere(N), 0)
    mean, basis, var = synthetic.make_gpmm(ref, R, 1, orthonormal=False)   # as bench.py at C4
    model = api.Model(ctx, ref, mean, basis, var)
    tgt = api.Target(ctx, target)
    reg = api.CpdRegistration(ctx, model, tgt, api.CpdConfiguration(w=0.1))
    runs = measure(api, reg, reps)
    reg.close()
    return {"M": M, "N": N, "r": R, "cholesky_backsolve_ms_all": [v[3] for v in runs],
            "iteration_ms_all": [v[4] for v in runs]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ranks", default="2000,9472,9536,12808,18000")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--c4", action="store_true")
    ap.add_argument("--root", default=ROOT)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.root))
    import numpy as np

    from gingr_b200 import api, synthetic
    ctx = api.Context(0)
    out = {"card": card(), "reps": args.reps, "root": os.path.abspath(args.root),
           "method": "per-phase CUDA events of gingr_registration_get_profile over single-iteration chains after one warm-up"}
    if args.c4:
        out["c4"] = c4(api, synthetic, ctx, args.reps)
    else:
        out["ranks"] = [one_rank(api, synthetic, np, ctx, int(r), args.reps) for r in args.ranks.split(",")]
    print(json.dumps(out, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
