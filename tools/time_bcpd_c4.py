"""One BCPD update (GINGR_ALGO_BCPD) at the C4 size -- M = 20 000, N = 200 000, r = 2000, w = 0.1, RigidTransforms -- beside
the CPD update of bench.py's workload on the same model and target in the same run.  Per phase (CUDA events of
gingr_registration_get_profile, best of `reps` single-iteration chains): E-step sweeps A / B, Gram, Cholesky + back
substitution (for BCPD with the 3M rows of Q riding through the factorisation), whole iteration.  Reported beside them:
the factorisation difference (the solve of the variance rows), the whole-iteration difference, and what of it lies outside
the E-step, Gram and factorisation events (filling the variance rows, reducing them to Sigma, the small kernels).  The
card's name and power limit are read in the same run.
usage: python tools/time_bcpd_c4.py [--reps K] [--out FILE.json]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

from gingr_b200 import api, synthetic

M, N, R, W = 20000, 200000, 2000, 0.1
PHASES = ("estep_sweep_a", "estep_sweep_b", "gram", "cholesky_backsolve", "iteration")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def measure(reg, reps):
    reg.initializeState(globalTransformation=api.RIGID_TRANSFORMS)
    reg.updateChain(1)                      # warm-up: capture, module load
    reg.setProfiling(True)
    runs = []
    for _ in range(reps):
        reg.updateChain(1)
        ms, it = reg.getProfile()
        runs.append(ms[:5] / max(it, 1))
    reg.setProfiling(False)
    best = min(runs, key=lambda v: v[4])
    st = reg.downloadState()
    return {k: float(v) for k, v in zip(PHASES, best)}, st


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ref = synthetic.fibonacci_sphere(M)
    target = synthetic.make_target(synthetic.fibonacci_sphere(N), 0)
    mean, basis, var = synthetic.make_gpmm(ref, R, 1, orthonormal=False)   # as bench.py at C4
    ctx = api.Context(0)
    model = api.Model(ctx, ref, mean, basis, var)
    tgt = api.Target(ctx, target)
    out = {"card": card(), "M": M, "N": N, "r": R, "w": W, "reps": args.reps,
           "method": "best of reps single-iteration chains, per-phase CUDA events"}
    cpd = api.CpdRegistration(ctx, model, tgt, api.CpdConfiguration(w=W))
    out["cpd_ms"], _ = measure(cpd, args.reps)
    cpd.close()
    bcpd = api.BcpdRegistration(ctx, model, tgt, api.BcpdConfiguration(w=W))
    out["bcpd_ms"], st = measure(bcpd, args.reps)
    alpha, sigma = bcpd.bcpdState()
    bcpd.close()
    out["bcpd_state_after_warmup_and_reps"] = {"iteration": st.iteration, "status": st.status, "sigma2": st.sigma2,
                                               "alpha_sum": float(alpha.sum()), "sigma_mean": float(sigma.mean()),
                                               "finite": bool(np.all(np.isfinite(alpha)) and np.all(np.isfinite(sigma)))}
    b, c = out["bcpd_ms"], out["cpd_ms"]
    # The two registrations are measured separately, so differences of their phases carry the run-to-run spread of both.
    # factorisation: the 3M rows of Q solved against L with the system (3M r^2 flop, about one Gram-sized product)
    out["factorisation_extra_ms"] = b["cholesky_backsolve"] - c["cholesky_backsolve"]
    out["iteration_extra_ms"] = b["iteration"] - c["iteration"]
    # the rest of the whole-iteration difference: bcpd_var_rows_kernel (writes the 3M x rp rows, ~1 GB at C4) and
    # bcpd_state_kernel (reads them back), which lie outside the factorisation events, plus the E-step difference (BCPD
    # sweeps are not culled) and the small kernels
    out["estep_extra_ms"] = (b["estep_sweep_a"] + b["estep_sweep_b"]) - (c["estep_sweep_a"] + c["estep_sweep_b"])
    out["rows_fill_state_and_rest_ms"] = out["iteration_extra_ms"] - out["factorisation_extra_ms"] - out["estep_extra_ms"] - \
        (b["gram"] - c["gram"])
    out["variance_rows_bytes"] = 3 * M * R * 8
    out["variance_rows_solve_flop"] = 3 * M * R * R
    fx = out["factorisation_extra_ms"]
    out["variance_rows_solve_tflops"] = 3 * M * R * R / (fx * 1e-3) / 1e12 if fx > 0.0 else None
    print(json.dumps(out, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
