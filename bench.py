#!/usr/bin/env python
"""bench.py -- GiNGR update() iterations/s on the BASELINE.json workload (C4: CPD, M = 20 000 moving points,
N = 200 000 target points, rank-2000 GPMM, w = 0.1), synthetic seeded inputs (SURVEY.md 8d).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload c4|c4_small|c3c|c1] [--dump-outputs DIR]

One "step" = one GingrAlgorithm.update + fit refresh (GingrGeneratorWrapper.propose) of ONE registration.
With N > 1 (torchrun, one rank per GPU) the same registration is sharded over the ranks -- target points in the
E-step, basis rows in the Gram / fit passes -- and the partial sums are all-reduced with NCCL inside the
library, so scaling is STRONG (total work fixed).  Prints one JSON line (rank 0).

  value   iterations/s with model/target/state resident in HBM: K iterations chained on the device
          (gingr_update_chain), CUDA events on the library's stream, max over ranks.
  e2e     the same through the reference-facing call gingr_update with HOST state in / out (state + alpha H2D,
          state + alpha + fit D2H every step).
  roofline  dominant kernel, timed live with CUDA events recorded around it on the library's stream, in an
            event-instrumented pass of the same chain right after the timed one (the timed chain replays the captured
            iteration graph, which cannot carry per-iteration events).
  parity    the first iterations of the seeded chain re-played and compared with the cached oracle values
            (tests/golden/c4_chain_oracle.npz, oracle/fast.py); the run fails if any exceeds 1e-6.
  cpu_baseline  the CPU oracle (port of the reference path, NOT the JVM) on this box's cores: ONE real update() of the
            same workload (bounded sample = 1 iteration), N = 1 only.
  secondary the other named configurations of BASELINE.json (C1, C3, C5) and the ICP iteration at 200k points with the K2
            roofline (bench_secondary.py).

--dump-outputs DIR writes the state the timed path computed in its last step (fit, shape coefficients, sigma2, scale,
translation, Euler angles, iteration count) as DIR/<name>.npy in float64.  The inputs are seeded, so two builds run
with the same arguments can be compared output for output.

--impl reference times the CPU port as the main line (the JVM reference cannot run here: no JVM, scalismo /
Breeze jars absent; DESIGN.md): real update() iterations of the oracle (oracle/fast.py: the algorithmic-minimum form,
pinned to the literal restatement by tests/test_oracle_fast.py) on the SAME workload, all host cores, --steps / --warmup
honoured, wall clock -- no sampling, no extrapolation.
"""
from __future__ import annotations

import os
import sys

# The CPU legs use every host core.  torchrun exports OMP_NUM_THREADS=1 to its workers, which would silently turn the
# reference arm into a one-core run: undo that BEFORE numpy / OpenBLAS / libgomp read the environment.
_CPU_CORES = os.cpu_count() or 1
if "--impl" in sys.argv and "reference" in sys.argv:
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(_CPU_CORES)

import argparse
import json
import statistics
import subprocess
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (M, N, r, description)
    "c4": (20000, 200000, 2000, "CPD M=20000 N=200000 rank=2000 w=0.1 RigidTransforms (BASELINE configs[3], 200k-point CPD)"),
    "c4_small": (4000, 20000, 500, "CPD M=4000 N=20000 rank=500 w=0.1 (reduced C4, smoke only)"),
    "c3c": (1000, 1000, 100, "CPD M=N=1000 rank=100 (DemoMultiResolution size)"),
    "c1": (100, 100, 50, "CPD M=N=100 rank=50 (DemoCPD size)"),
}
W_OUTLIER = 0.1
FLOP_PER_PAIR = 71.0   # SURVEY.md 8(d): two sweeps, exp counted as 22 flop


_INPUT_CACHE = {}


def make_inputs(name: str, seed: int = 0):
    if (name, seed) not in _INPUT_CACHE:
        _INPUT_CACHE[(name, seed)] = _make_inputs(name, seed)
    return _INPUT_CACHE[(name, seed)]


def _make_inputs(name: str, seed: int = 0):
    from gingr_b200 import synthetic
    M, N, r, _ = WORKLOADS[name]
    ref = synthetic.fibonacci_sphere(M)
    target = synthetic.make_target(synthetic.fibonacci_sphere(N), seed)
    mean, basis, var = synthetic.make_gpmm(ref, r, seed + 1, orthonormal=(M <= 20000 and r <= 600))
    return ref, mean, basis, var, target


def load_peaks():
    peaks = {}
    for fn in ("MEASURED_PEAKS.json", "FP64_PEAKS.json"):
        p = os.path.join(ROOT, fn)
        if os.path.exists(p):
            with open(p) as f:
                peaks[fn] = json.load(f)
    return peaks


def dump_outputs(out_dir: str, scale, translation, euler, shape, fit, sigma2, iteration):
    """The registration state a caller receives after the last timed step, one float64 .npy file per field.  `iteration`
    is the number of updates behind the state (warm-up included), so dumps of runs with different warm-up agree on which
    step they describe."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"scale": scale, "translation": translation, "euler": euler, "shape": shape, "fit": fit, "sigma2": sigma2,
              "iteration": iteration}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        fd, self.path = tempfile.mkstemp(suffix=".csv")
        os.close(fd)
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            hi = [s for s in sm if s >= 0.5 * max(sm)]   # samples under load
            out["sm_mhz"] = statistics.median(hi)
            out["sm_max_mhz"] = max(mx)
        out["reasons"] = sorted(reasons)
        return out


# ---------------------------------------------------------------------------------------------------
# CPU port (oracle) timing -- only the cpu_baseline / --impl reference legs touch oracle/
# ---------------------------------------------------------------------------------------------------
def _use_all_cores():
    """All host cores for the C oracle (OpenMP) and for numpy / scipy BLAS, whatever the environment said at start-up."""
    from oracle import oracle
    oracle.build()
    oracle.set_num_threads(_CPU_CORES)
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=_CPU_CORES)
    except Exception:
        pass
    return oracle.num_threads()


def cpu_oracle_chain(name: str, warmup: int, steps: int, initial_sigma2=None, budget_s: float = 1e9):
    """Real update() iterations of the CPU port on the workload `name`: -> (seconds per timed iteration (list), cores,
    description, final state).  Model constants (Q^T Q and its factor: once per model, like the model upload on the GPU
    side) and the initial state are built outside the timed iterations.  Stops early only if budget_s is exceeded."""
    from oracle import fast, oracle
    cores = _use_all_cores()
    M, N, r, _ = WORKLOADS[name]
    ref, mean, basis, var, target = make_inputs(name)
    om = oracle.Gpmm(ref, mean, basis, var, None)
    fm = fast.FastCpdModel(om)
    algo = oracle.CpdAlgorithm(oracle.CpdConfig(w=W_OUTLIER, initial_sigma=initial_sigma2), literal=False)
    st = algo.initialize(oracle.initial_state(om, target, None, global_transformation=oracle.RIGID_TRANSFORMS))
    t_start = time.perf_counter()
    secs = []
    for k in range(warmup + steps):
        t0 = time.perf_counter()
        st = fast.propose(fm, algo, st)
        dt = time.perf_counter() - t0
        if st.status == oracle.STATUS_MODEL_FLEXIBILITY_ERROR:
            raise SystemExit("bench.py: the CPU port reported ModelFlexibilityError")
        if k >= warmup:
            secs.append(dt)
        if time.perf_counter() - t_start > budget_s and len(secs) >= 1:
            break
    note = (f"{len(secs)} real update() + fit refresh of the CPU port (oracle/fast.py: C/OpenMP streaming E-step, BLAS dsyrk Gram, "
            f"Cholesky, 5 basis passes) on the full workload M={M} N={N} rank={r}, {cores} threads, wall clock per iteration; "
            "no sampling, no extrapolation")
    return secs, cores, note, st


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    name = args.workload
    M, N, r, desc = WORKLOADS[name]
    secs, cores, note, st = cpu_oracle_chain(name, args.warmup, args.steps, budget_s=args.ref_budget_s)
    if args.dump_outputs:
        p = st.params
        dump_outputs(args.dump_outputs, p.scale, p.translation, p.euler, p.shape, st.fit, st.sigma2, st.iteration)
    sec = statistics.mean(secs)
    v = 1.0 / sec
    line = {
        "impl": "reference", "metric": "GiNGR update() iterations/s", "value": v, "unit": "iterations/s",
        "n_gpus": args.gpus, "steps": len(secs), "warmup": args.warmup, "ms_per_step": 1e3 * sec,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc, "M": M, "N": N, "rank": r, "w": W_OUTLIER, "algorithm": "CPD",
                   "note": "CPU port of the reference path (no JVM in this image), every iteration a real update() on the full workload"},
        "cpu_baseline": {"value": v, "unit": "iterations/s", "cores": cores, "kind": "port", "sample": note},
        "e2e": {"value": v, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "final_sigma2": st.sigma2,
        "seconds_per_iteration": {"min": min(secs), "max": max(secs)},
    }
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------------
# parity of the timed configuration against the cached oracle chain
# ---------------------------------------------------------------------------------------------------
GOLDEN_C4 = os.path.join(ROOT, "tests", "golden", "c4_chain_oracle.npz")
PARITY_TOL = 1e-6


def chain_parity(reg, api, ref, iterations=None):
    """Re-play the first iterations of the seeded C4 chain from the initial state and compare every component with the
    cached oracle values (tests/golden/make_c4_golden.py): coefficients relative to max |alpha|, fit relative to the mesh
    diagonal, sigma2 relative.  Returns the parity record (all ranks hold the full state after an iteration)."""
    g = np.load(GOLDEN_C4)
    n_it = g["alpha"].shape[0] if iterations is None else min(iterations, g["alpha"].shape[0])
    diag = float(np.linalg.norm(ref.max(0) - ref.min(0)))
    st = reg.initializeState(globalTransformation=api.RIGID_TRANSFORMS)
    rec = {"against": "tests/golden/c4_chain_oracle.npz (oracle/fast.py, generated by tests/golden/make_c4_golden.py)",
           "iterations": int(n_it), "tolerance": PARITY_TOL,
           "sigma2_initial_rel_err": abs(st.sigma2 - float(g["sigma2"][0])) / float(g["sigma2"][0])}
    worst = rec["sigma2_initial_rel_err"]
    e_a = e_f = e_s = e_t = 0.0
    for k in range(n_it):
        st = reg.propose(st)
        if st.status == api.STATUS_MODEL_FLEXIBILITY_ERROR:
            raise SystemExit("bench.py: ModelFlexibilityError while re-playing the golden chain")
        a = g["alpha"][k]
        e_a = max(e_a, float(np.max(np.abs(st.modelParameters.shape - a)) / max(np.max(np.abs(a)), 1e-300)))
        e_f = max(e_f, float(np.max(np.abs(st.fit[g["fit_idx"]] - g["fit_sub"][k])) / diag),
                  float(np.max(np.abs(st.fit.sum(axis=0) - g["fit_sum"][k])) / (diag * st.fit.shape[0])))
        e_s = max(e_s, abs(st.sigma2 - float(g["sigma2"][k + 1])) / float(g["sigma2"][k + 1]))
        e_t = max(e_t, float(np.max(np.abs(st.modelParameters.translation - g["translation"][k])) / diag),
                  float(np.max(np.abs(np.array(st.modelParameters.euler) - g["euler"][k]))))
    rec.update({"alpha_rel_err": e_a, "fit_rel_err": e_f, "sigma2_rel_err": e_s, "pose_err": e_t})
    worst = max(worst, e_a, e_f, e_s, e_t)
    rec["max_rel_err"] = worst
    rec["ok"] = bool(worst < PARITY_TOL)
    return rec


# ---------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from gingr_b200 import api

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU path (use --impl reference for the CPU port)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    name = args.workload
    M, N, r, desc = WORKLOADS[name]
    ref, mean, basis, var, target = make_inputs(name)

    ctx = api.Context(local_rank)
    if world > 1:
        uid = [api.Context.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(world, rank, uid[0])
    model = api.Model(ctx, ref, mean, basis, var)
    tgt = api.Target(ctx, target)
    reg = api.CpdRegistration(ctx, model, tgt, api.CpdConfiguration(maxIterations=10 ** 6, w=W_OUTLIER))
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local_rank))

    def barrier():
        ctx.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    # ---- device-resident chain: `value` ---------------------------------------------------------------
    # The timed region replays the captured iteration graph (the product path).  The per-kernel times of the
    # roofline come from a second, event-instrumented pass of the same chain right after it (events cannot live
    # inside the replayed graph); its total is reported as phases_ms.iteration next to ms_per_step.
    parity = None
    if name == "c4" and os.path.exists(GOLDEN_C4):
        parity = chain_parity(reg, api, ref)
        if not parity["ok"]:
            raise SystemExit(f"bench.py: parity against the cached oracle chain FAILED: {json.dumps(parity)}")
    state0 = reg.initializeState(globalTransformation=api.RIGID_TRANSFORMS)
    reg.updateChain(max(args.warmup, 3))
    barrier()
    l0 = ctx.launch_count
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    reg.updateChain(args.steps)
    e1.record(stream)
    barrier()
    launches = ctx.launch_count - l0
    ms_chain = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        st = reg.downloadState()
        p = st.modelParameters
        dump_outputs(args.dump_outputs, p.scale, p.translation, p.euler, p.shape, st.fit, st.sigma2, st.iteration)
    reg.setProfiling(True)
    barrier()
    reg.updateChain(args.steps)
    barrier()
    clocks = sampler.stop()
    prof_ms, prof_it = reg.getProfile()
    reg.setProfiling(False)
    final = reg.downloadState()
    if not np.all(np.isfinite(final.fit)) or final.status == api.STATUS_MODEL_FLEXIBILITY_ERROR:
        raise SystemExit("bench.py: registration diverged / ModelFlexibilityError inside the timed region")

    # ---- host in / host out through gingr_update: `e2e` -------------------------------------------------
    st = reg.initializeState(globalTransformation=api.RIGID_TRANSFORMS)
    for _ in range(max(args.warmup, 3)):
        st = reg.propose(st)
    barrier()
    t0 = time.perf_counter()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record(stream)
    for _ in range(args.steps):
        st = reg.propose(st)
    e3.record(stream)
    barrier()
    ms_e2e = max(e2.elapsed_time(e3), 0.0)
    wall_e2e = (time.perf_counter() - t0) * 1e3
    ms_e2e = max(ms_e2e, wall_e2e if world == 1 else ms_e2e)

    if world > 1:
        t = torch.tensor([ms_chain, ms_e2e], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_chain, ms_e2e = float(t[0]), float(t[1])

    # ---- secondary entries: the other named configurations (short; C5 on every rank, the rest at N = 1) -------------
    secondary = None
    if name == "c4" and not args.no_secondary:
        import bench_secondary as bs
        reg.close()
        reg = None
        model.close()
        secondary = {}
        barrier()
        # independent chains need a context that is not part of a communicator (gingr_mcmc_configure: replicas only)
        ctx5 = api.Context(local_rank) if world > 1 else ctx
        c5 = bs.c5_mcmc(ctx5, world, rank)
        if ctx5 is not ctx:
            ctx5.close()
        agg = torch.tensor([float(c5["chains"] * c5["steps"]), float(c5["accepted"]), float(c5["launches"])], dtype=torch.float64, device="cuda")
        tmax = torch.tensor([c5["seconds"]], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(agg)
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        secondary["c5_mcmc"] = {
            "workload": "1024 independent Metropolis-Hastings chains of the C1 size (ICP proposal + random pose / shape proposals, "
                        "evaluators, accept / reject on the device), divided among the GPUs (replicas, no collective)",
            "gpus": world, "chains": 1024, "mh_steps_per_chain": c5["steps"], "chain_steps_per_s": float(agg[0]) / float(tmax[0]),
            "chain_steps_per_s_per_gpu": float(agg[0]) / float(tmax[0]) / world, "acceptance_rate": float(agg[1]) / (1024 * (c5["steps"] + 3)),
            "launches_per_chain_step": float(agg[2]) / float(agg[0]),
            "launches_per_mh_step_per_gpu": float(agg[2]) / world / c5["steps"],
            "path": "one batched kernel sequence per MH step for all chains of a GPU (blockIdx.z = chain, gingr_b200/csrc/batch.cuh)",
            "finite": c5["finite"]}
        if world == 1:
            secondary["c5_update_batch"] = bs.c5_update_batch(ctx)
            secondary["c1_icp"] = bs.c1_icp(ctx)
            secondary["c3_multiresolution"] = bs.c3_pipeline(ctx)
            secondary["icp_200k"] = bs.icp_200k(ctx, ROOT)

    if rank == 0:
        peaks = load_peaks()
        fp = peaks.get("FP64_PEAKS.json", {})
        mb = fp.get("microbench", {})
        dfma_peak = mb.get("dfma_tflops_sustained") or mb.get("dfma_tflops") or 33.7
        dmma_peak = fp.get("cublas_dgemm_tflops_sustained") and max(fp.get("cublas_dgemm_tflops_sustained"), mb.get("dmma_tflops_sustained", 0)) or 37.0
        it = max(prof_it, 1)
        n_local = api.shard_range(N, world, 0)[1]
        m_local = api.shard_range(M, world, 0)[1]
        t_a, t_b, t_g, t_c, t_it = (prof_ms[k] / it for k in (0, 1, 2, 3, 4))
        estep_flop = FLOP_PER_PAIR * M * n_local
        gram_flop = 3.0 * m_local * r * (r + 1)
        estep_tf = estep_flop / ((t_a + t_b) * 1e-3) / 1e12 if (t_a + t_b) > 0 else 0.0
        gram_tf = gram_flop / (t_g * 1e-3) / 1e12 if t_g > 0 else 0.0
        # DRAM bytes per launch from the committed ncu --set full capture of this workload (profiles/ncu_traffic.json);
        # only valid for the configuration it was captured on (C4, 1 GPU)
        traffic = {}
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if name == "c4" and world == 1 and os.path.exists(tpath):
            with open(tpath) as f:
                traffic = {k: v["dram_bytes"] for k, v in json.load(f)["kernels"].items()}
        tr_estep = (traffic.get("estep_colsum_kernel", 0) + traffic.get("estep_rowsum_kernel", 0)) or None
        rl_estep = {"kernel": "estep_colsum_kernel+estep_rowsum_kernel (K1)", "bound": "fp64", "achieved": estep_tf,
                    "peak": dfma_peak, "unit": "TFLOP/s", "frac": estep_tf / dfma_peak, "traffic": tr_estep,
                    "ms": t_a + t_b, "algorithmic_flop": estep_flop,
                    "algorithmic_bytes": 24.0 * (M + n_local) + 8.0 * (4 * M + n_local),
                    "peak_source": "FP64_PEAKS.json dfma_tflops_sustained (measured, tools/fp64_peaks.cu)",
                    "note": "achieved = SURVEY 8(d) ALGORITHMIC count (71 flop per pair, exp = 22) / time; the kernels issue 14 + 17 "
                            "FP64 instructions per pair (expanded-distance path, table-driven 2^x), ncu FP64 pipe active 78-79 % "
                            "(profiles/r02_ncu_top_kernels.md)"}
        rl_gram = {"kernel": "gram_ws_kernel (K3, DMMA.8x8x4, warp-specialised, cp.async.bulk)", "bound": "tensor",
                   "achieved": gram_tf, "peak": dmma_peak, "unit": "TFLOP/s", "frac": gram_tf / dmma_peak,
                   "traffic": traffic.get("gram_ws_kernel"), "ms": t_g, "algorithmic_flop": gram_flop,
                   "algorithmic_bytes": 8.0 * 3 * m_local * r,
                   "peak_source": "FP64_PEAKS.json max(cuBLAS DGEMM sustained, DMMA issue peak) (measured)"}
        dominant = rl_estep if (t_a + t_b) >= t_g else rl_gram
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            try:
                secs, cores, note, _ = cpu_oracle_chain(name, 0, 1, initial_sigma2=state0.sigma2)
                cpu = {"value": 1.0 / secs[0], "unit": "iterations/s", "cores": cores, "kind": "port", "sample": note}
            except Exception as ex:  # the oracle is test infrastructure: its absence must not fail the bench
                cpu = {"value": None, "unit": "iterations/s", "cores": 0, "kind": "port", "sample": f"unavailable: {ex}"}
        h2d = 112 + 8 * r
        d2h = 112 + 8 * r + 24 * M
        line = {
            "metric": "GiNGR update() iterations/s", "value": args.steps / (ms_chain * 1e-3), "unit": "iterations/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_chain / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": desc, "M": M, "N": N, "rank": r, "w": W_OUTLIER, "algorithm": "CPD",
                       "sharding": f"targets/{world} (E-step), basis rows/{world} (Gram, fit); NCCL all-reduce" if world > 1 else "single GPU",
                       "timed_path": "captured CUDA graph of the iteration, replayed K times on the device",
                       "l2": "inputs larger than L2 (basis 8*3M*r bytes = %.0f MB re-read every step)" % (8.0 * 3 * M * r / 1e6)},
            "clocks": clocks,
            "e2e": {"value": args.steps / (ms_e2e * 1e-3), "unit": "iterations/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches),
            "roofline": dominant,
            "rooflines": [rl_estep, rl_gram],
            "phases_ms": {"estep_sweepA": t_a, "estep_sweepB": t_b, "gram": t_g, "cholesky_backsolve": t_c,
                          "iteration": t_it},
            "cpu_baseline": cpu,
            "final_sigma2": final.sigma2,
            "parity": parity,
            "secondary": secondary,
        }
        print(json.dumps(line))
    if reg is not None:
        reg.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the C1 / C3 / C5 / ICP-200k entries")
    ap.add_argument("--ref-budget-s", type=float, default=900.0,
                    help="--impl reference: stop after this many seconds of iterations (the completed count is reported)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the state computed by the last timed step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
