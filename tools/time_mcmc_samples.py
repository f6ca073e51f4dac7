"""Cost of collecting Metropolis-Hastings samples on the device (gingr_mcmc_collect / gingr_mcmc_samples).

1. The C5 workload of bench_secondary.c5_mcmc (1024 ICP chains, M = N = 100, rank 50, randomMixture 0.5) under
   gingr_mcmc_batch: MH steps/s with collection off, with takeEveryN = 1 and with takeEveryN = 50, and launches per batched
   step.  The variants alternate on the same chains; after each switch one untimed batched step rebuilds the batched
   graph, then `--steps` steps are timed with a host clock around work that ends in a device synchronise.
2. One chain of `--chain-steps` steps at the same size: the logged runProbabilistic (one host round trip per step, a
   JSON record per state) reduced on the host by helper (samples_from_log, log_samples_to_shapes, distance_map_total /
   _normal) against device collection + sample_statistics, wall time for the same two maps; variants alternate after one
   warm-up run each.  The maps of the two paths are compared.

The card's name, power limit and maximum SM clock are read in the same run.
usage: python tools/time_mcmc_samples.py [--reps K] [--steps S] [--chain-steps S] [--out FILE.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BURN_IN, EVERY = 100, 10          # the thinning of the single-chain comparison


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def problem(api, synthetic, ctx):
    M, N, r = 100, 100, 50
    ref, tri = synthetic.sphere_mesh(M)
    mean, basis, var = synthetic.make_gpmm(ref, r, 1)
    tv, tt = synthetic.sphere_mesh(N)
    model = api.Model(ctx, ref, mean, basis, var, tri)
    tgt = api.Target(ctx, synthetic.make_target(tv, 0), tt)
    return model, tgt, ref, tri


def c5(api, np, ctx, model, tgt, reps, steps, n_chains=1024):
    cfg = api.IcpConfiguration(maxIterations=10 ** 6, initialSigma=1.0, endSigma=1.0)
    settings = api.ProbabilisticSettings(uncertainty=1.0, randomMixture=0.5)
    chains = []
    for _ in range(n_chains):
        c = api.IcpRegistration(ctx, model, tgt, cfg)
        c.configureProbabilistic(settings)
        c.initializeState(globalTransformation=api.RIGID_TRANSFORMS)
        chains.append(c)
    variants = {"off": None, "takeEveryN_1": api.SampleCollection(burnIn=0, takeEveryN=1, total=2 ** 31 - 1),
                "takeEveryN_50": api.SampleCollection(burnIn=0, takeEveryN=50, total=2 ** 31 - 1)}
    out = {k: {"seconds": [], "steps_per_s": [], "launches_per_batched_step": None} for k in variants}
    api.mcmc_batch(chains, 3, seed=0)      # warm-up: priming, module load
    ctx.synchronize()
    for _ in range(reps):
        for name, coll in variants.items():
            for c in chains:
                c.collectSamples(coll)
            api.mcmc_batch(chains, 1, seed=0)   # rebuilds the batched graph for this variant (untimed)
            ctx.synchronize()
            l0 = ctx.launch_count
            t0 = time.perf_counter()
            api.mcmc_batch(chains, steps, seed=0)
            ctx.synchronize()
            dt = time.perf_counter() - t0
            out[name]["seconds"].append(dt)
            out[name]["steps_per_s"].append(n_chains * steps / dt)
            out[name]["launches_per_batched_step"] = (ctx.launch_count - l0) / steps
    st = api.sample_statistics(chains)       # last variant: takeEveryN = 50
    out["pooled_count_last_variant"] = st.count
    out["finite"] = bool(np.all(np.isfinite(st.distanceMapTotal())))
    for c in chains:
        c.close()
    for name in variants:
        v = out[name]["steps_per_s"]
        out[name]["median_steps_per_s"] = sorted(v)[len(v) // 2]
    off = out["off"]["median_steps_per_s"]
    for name in ("takeEveryN_1", "takeEveryN_50"):
        out[name]["median_rate_vs_off"] = out[name]["median_steps_per_s"] / off
    return out


def single_chain(api, helper, io, np, ctx, model, tgt, ref, tri, reps, steps):
    cfg = api.IcpConfiguration(maxIterations=10 ** 6, initialSigma=1.0, endSigma=1.0)
    settings = api.ProbabilisticSettings(uncertainty=1.0, randomMixture=0.5)
    coll = api.SampleCollection(burnIn=BURN_IN, takeEveryN=EVERY, total=steps + 1)
    reg = api.IcpRegistration(ctx, model, tgt, cfg)
    st0 = reg.initializeState(globalTransformation=api.RIGID_TRANSFORMS)

    def logged():
        log = io.JSONStateLogger()
        reg.runProbabilistic(st0, settings, seed=7, iterations=steps, acceptRejectLogger=log)
        recs = helper.samples_from_log(log.log, takeEveryN=EVERY, total=steps + 1, burnIn=BURN_IN)
        shapes = helper.log_samples_to_shapes(model, [r for r, _ in recs])
        return len(shapes), helper.distance_map_total(shapes), helper.distance_map_normal(shapes, tri)

    def device():
        reg.runProbabilistic(st0, settings, seed=7, iterations=steps, sampleCollection=coll)
        s = api.sample_statistics([reg])
        return s.count, s.distanceMapTotal(), s.distanceMapNormal()

    res = {"logged": {"seconds": []}, "device": {"seconds": []}}
    maps = {}
    for name, fn in (("logged", logged), ("device", device)):
        maps[name] = fn()                     # warm-up
    for _ in range(reps):
        for name, fn in (("logged", logged), ("device", device)):
            ctx.synchronize()
            t0 = time.perf_counter()
            maps[name] = fn()
            res[name]["seconds"].append(time.perf_counter() - t0)
    reg.close()
    for name in res:
        v = res[name]["seconds"]
        res[name]["median_seconds"] = sorted(v)[len(v) // 2]
    res["speedup_median"] = res["logged"]["median_seconds"] / res["device"]["median_seconds"]
    (nl, tl, ml), (nd, td, md) = maps["logged"], maps["device"]
    res["samples"] = {"logged": nl, "device": nd}
    res["max_rel_diff_total_map"] = float(np.max(np.abs(tl - td)) / np.max(tl))
    res["max_rel_diff_normal_map"] = float(np.max(np.abs(ml - md)) / np.max(ml))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--chain-steps", type=int, default=1000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    import numpy as np
    from gingr_b200 import api, helper, io, synthetic
    ctx = api.Context(0)
    model, tgt, ref, tri = problem(api, synthetic, ctx)
    out = {"gpu": card(), "workload": "1024 ICP chains, M = N = 100, rank 50, randomMixture 0.5 (bench_secondary.c5_mcmc)",
           "c5_batched": c5(api, np, ctx, model, tgt, a.reps, a.steps),
           "single_chain": dict(single_chain(api, helper, io, np, ctx, model, tgt, ref, tri, a.reps, a.chain_steps),
                                steps=a.chain_steps, burnIn=BURN_IN, takeEveryN=EVERY),
           "gpu_after": card()}
    model.close()
    tgt.close()
    ctx.close()
    text = json.dumps(out, indent=2)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
