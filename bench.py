#!/usr/bin/env python
"""
bench.py -- headline benchmark of the HMC hot path (BASELINE.json: leapfrog-steps*chains/sec fp64, Neal's funnel).

One "step" = one pass of the hot path over one batch: ITERS HMC iterations (nSteps=5 leapfrog steps each) for CHAINS
chains of the 10-dim Neal's funnel, sampling phase, every sample written out.  Metric = leapfrog steps x chains per
second = CHAINS*ITERS*5 / time.

  value     : device-resident (chain state + sample buffer in HBM), timed with CUDA events on the sampler's stream.
  e2e       : the same work through the public one-call API (rn_sample over the C ABI) with HOST buffers: seeds
              host->device and every sample device->host inside the timed region.
  roofline  : compulsory-traffic HBM accounting of SURVEY.md 8(d) (B_step = [8(2(2n+1)+n)+32]/L bytes per leapfrog
              step) against MEASURED_PEAKS.json; plus an fp64 view (emitter op counts vs a DFMA peak measured here),
              because this path is FP64-pipe bound, not HBM bound.
  cpu_baseline / --impl reference : the CPU oracle (C++ restatement of the reference's LeapFrog + DataFunction
              interpreter; the JVM reference cannot run here) on the box's host cores, bounded sample.

Multi-GPU (torchrun): chains are sharded over ranks, no data-path collective, weak scaling (CHAINS per GPU fixed).

--dump-outputs DIR writes the draws of the last timed step (a seeded sample of them, see dump_outputs) so that two builds
can be compared output for output: the seeds, and therefore the inputs, are the same in every run with the same arguments.
The bench writes nothing into the source tree: kernels compiled at run time are cached in a temporary directory.
"""
import argparse
import atexit
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only; no __pycache__ in it either way

import numpy as np  # noqa: E402

N_DIM = 10
N_STEPS = 5
STEP_SIZE = 0.1
METRIC = "leapfrog_steps_x_chains_per_sec"
DUMP_LAST_DRAW_BYTES = 16_000_000  # --dump-outputs writes less than 64 MB in all
DUMP_SAMPLES_BYTES = 47_000_000


def bytes_per_leapfrog_step(n, L):
    """SURVEY.md 8(d): read+write the params array, write one sample, RNG state r/w, per HMC iteration of L steps."""
    return (8.0 * (2 * (2 * n + 1) + n) + 32.0) / L


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region: NVML every ~5 ms (nvidia-smi every 200 ms when the
    NVML binding is missing)."""
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index = index
        self.sm, self.max_sm, self.reasons = [], None, set()
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run_nvml(self):
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        self.max_sm = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        while not self._stop.is_set():
            self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                else nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            for nm, b in bits.items():
                if r & b:
                    self.reasons.add(nm)
            self._stop.wait(0.005)

    def _run_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                r = [x.strip() for x in out.split(",")]
                self.sm.append(float(r[0]))
                self.max_sm = float(r[1])
                for k, nm in enumerate(self.NAMES):
                    if r[2 + k].lower().startswith("active"):
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop.wait(0.2)

    def _run(self):
        try:
            self._run_nvml()
        except Exception:
            self._run_smi()

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=5)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_sm,
                "reasons": [n for n in self.NAMES if n in self.reasons], "samples": len(self.sm)}


def ncu_capture(math):
    """dram__bytes_{read,write}.sum, fp64-pipe activity ... of ONE rn_k_iter launch at the default workload, from the most
    recent `ncu --set full` capture of this kernel (scripts/ncu_summary.py writes profiles/ncu_funnel_<math>.json from the
    .ncu-rep; the capture cannot run inside a timed bench).  None when no capture of the current kernel is committed."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_funnel_%s.json" % math)))
    except Exception:
        return None


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


CPU_NOTE = ("C++ restatement of the reference's LeapFrog/HMC (oracle/) over the model's DataFunction COMPILED to straight-line "
            "C++ (g++ -O2 -ffp-contract=off; bit-identical to the oracle's interpreter, tests/test_oracle_compiled.py) -- the "
            "stand-in for the JVM `asm` path after JIT compilation, which cannot run in this image; one chain per host "
            "thread, threads pinned, cores = affinity mask capped by the cgroup CPU quota")


def _oracle_arm():
    """the CPU arm's model, config and core count (shared by --impl reference and the cpu_baseline leg)"""
    from oracle.rainier_py.binding import OracleModel, default_config, lib
    rir = open(os.path.join(ROOT, "rainier_b200", "models", "funnel10.rir"), "rb").read()
    om = OracleModel(rir, []).compile_density()
    L = lib()
    cores = L.rno_hardware_threads()
    L.rno_set_threads(cores)
    L.rno_set_pinning(1)
    return om, default_config(), cores, L.rno_machine_threads()


def run_reference(args):
    """--impl reference: the CPU oracle (stand-in for the JVM `asm` path, which cannot run here) on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from rainier_b200 import abi
    om, cfg, cores, machine = _oracle_arm()
    cfg.sampler, cfg.n_steps = abi.RN_SAMPLER_HMC, N_STEPS
    cfg.step_size_tuner, cfg.static_step_size = abi.RN_STEP_STATIC, STEP_SIZE
    cfg.mass_tuner = abi.RN_MASS_IDENTITY
    cfg.warmup_iterations = 0
    chains = cores * 4
    # size the per-step sample so that warmup+steps finish in a few minutes: calibrate on a short run
    cfg.iterations = 2000
    t = time.perf_counter()
    om.sample(cfg, seeds=np.arange(chains) + 1000)
    dt = time.perf_counter() - t
    rate0 = chains * cfg.iterations * N_STEPS / dt
    target_s = 4.0
    cfg.iterations = max(100, int(rate0 * target_s / (chains * N_STEPS)))
    for _ in range(args.warmup):
        om.sample(cfg, seeds=np.arange(chains) + 1000)
    t = time.perf_counter()
    for k in range(args.steps):
        om.sample(cfg, seeds=np.arange(chains) + 1000 + k)
    dt = time.perf_counter() - t
    value = args.steps * chains * cfg.iterations * N_STEPS / dt
    sample = "%d chains x %d HMC iterations x %d leapfrog steps per step, one chain per thread" % (chains, cfg.iterations, N_STEPS)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "leapfrog-steps*chains/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "neals_funnel_10d_hmc_nsteps5", "sampler": "HMC(nSteps=5)", "step_size": STEP_SIZE,
                   "chains": chains, "iterations_per_step": cfg.iterations},
        "cpu_baseline": {"value": value, "unit": "leapfrog-steps*chains/s", "cores": cores, "machine_threads": machine,
                         "per_core": value / cores, "kind": "port", "sample": sample, "note": CPU_NOTE},
        "e2e": {"value": value, "unit": "leapfrog-steps*chains/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def cpu_baseline_leg():
    from rainier_b200 import abi
    om, cfg, cores, machine = _oracle_arm()
    cfg.sampler, cfg.n_steps = abi.RN_SAMPLER_HMC, N_STEPS
    cfg.step_size_tuner, cfg.static_step_size = abi.RN_STEP_STATIC, STEP_SIZE
    cfg.mass_tuner = abi.RN_MASS_IDENTITY
    cfg.warmup_iterations = 0
    chains = cores * 4
    cfg.iterations = 2000
    t = time.perf_counter()
    om.sample(cfg, seeds=np.arange(chains) + 1000)
    dt = time.perf_counter() - t
    rate0 = chains * cfg.iterations * N_STEPS / dt
    cfg.iterations = max(100, int(rate0 * 12.0 / (chains * N_STEPS)))
    t = time.perf_counter()
    om.sample(cfg, seeds=np.arange(chains) + 1000)
    dt = time.perf_counter() - t
    value = chains * cfg.iterations * N_STEPS / dt
    return {"value": value, "unit": "leapfrog-steps*chains/s", "cores": cores, "machine_threads": machine, "per_core": value / cores,
            "kind": "port", "note": CPU_NOTE,
            "sample": "%d chains x %d HMC iterations x %d leapfrog steps (%.1f s), one chain per host thread" % (
                chains, cfg.iterations, N_STEPS, dt)}



def _load_npz_model(name):
    """RIR + columns of a BASELINE configuration from build/models/<name>.npz -- written by __graft_entry__.build() with the
    Python stand-in of the reference's Scala front end (the product side of the bench never imports oracle/)."""
    f = os.path.join(ROOT, "build", "models", name + ".npz")
    if not os.path.exists(f):
        return None
    z = np.load(f)
    return z["rir"].tobytes(), [z["c%d" % i] for i in range(int(z["ncols"]))]


def extra_configs(args, torch, dist, api, abi, rank, local_rank, world):
    """BASELINE.json configs[2..4] next to the headline (device-resident, device-timed, max over ranks):
      cfg3  logistic regression 50 x 100k, 2048 chains on ONE GPU (each rank runs the full config; value = one rank's rate)
      cfg4  eight schools, DefaultConfig (EHMC + DualAvg + diagonal mass), 8192 chains SHARDED over the ranks, warmup with
            the pooled mass-matrix statistics all-reduced over NCCL through the product's own communicator (rn_comm)
      cfg5  Poisson GLM 1000 groups / 1M rows, 4096 chains SHARDED over the ranks (strong scaling)"""
    out = {}
    dev = torch.device("cuda", local_rank)

    def device_rate(model, cfg, chains, iters, reps, seed0):
        s = api.CudaSampler(model, cfg, seeds=np.arange(chains, dtype=np.int64) + seed0)
        s.warmup(-1)
        stream = torch.cuda.ExternalStream(s.stream, device=dev)
        s.run(iters)
        s.sync()
        st0 = sum(x.leapfrogSteps for x in s.stats()[0])
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            s.run(iters)
        e1.record(stream)
        s.sync()
        torch.cuda.synchronize()
        stats = s.stats()[0]
        steps = float(sum(x.leapfrogSteps for x in stats) - st0)
        acc = float(np.mean([x.accepted / max(1, x.iterations) for x in stats]))
        s.close()
        t = torch.tensor([e0.elapsed_time(e1) * 1e-3], dtype=torch.float64, device=dev)
        n = torch.tensor([steps, acc], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(n, op=dist.ReduceOp.SUM)
        return float(n[0]) / float(t[0]), float(t[0]), float(n[1]) / world

    def static(eps, iters):
        return api.make_config(iterations=iters, warmupIterations=0, sampler=api.HMCSampler(N_STEPS), stepSizeTuner=api.StaticStepSize(eps),
                               massMatrixTuner=api.IdentityMassMatrixTuner(), launchIterations=iters)

    # ---- cfg4: the one collective of the design ----
    try:
        rir = open(os.path.join(ROOT, "rainier_b200", "models", "eight_schools.rir"), "rb").read()
        model = api.CudaModel(rir, [], device=local_rank)
        total = 8192
        per = total // world
        seeds = np.arange(total, dtype=np.int64)[rank * per:(rank + 1) * per] + 1
        comm = api.Comm.from_torch_distributed(local_rank) if world > 1 else None
        res = {}
        if comm is not None:  # NCCL sets its channels up inside the first collective (~0.2 s): not a warmup's cost
            w = api.CudaSampler(model, api.SamplerConfig(iterations=1, warmupIterations=500, adaptation=abi.RN_ADAPT_POOLED), seeds=seeds)
            w.set_comm(comm)
            w.warmup(-1)
            w.sync()
            w.close()
        for mode in ("pooled", "per_chain"):
            cfg = api.SamplerConfig(iterations=500, warmupIterations=500, adaptation=abi.RN_ADAPT_POOLED if mode == "pooled" else 0)
            s = api.CudaSampler(model, cfg, seeds=seeds)
            if mode == "pooled" and comm is not None:
                s.set_comm(comm)
            stream = torch.cuda.ExternalStream(s.stream, device=dev)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            ev[0].record(stream)
            s.warmup(-1)
            ev[1].record(stream)
            s.run(500)
            ev[2].record(stream)
            s.sync()
            torch.cuda.synchronize()
            st, mass = s.stats()
            calls, us = s.comm_stats()
            steps = float(sum(x.leapfrogSteps for x in st))
            t = torch.tensor([ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), us], dtype=torch.float64, device=dev)
            n = torch.tensor([steps], dtype=torch.float64, device=dev)
            same = torch.tensor(np.asarray(mass[0], dtype=np.float64), device=dev)
            lo, hi = same.clone(), same.clone()
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dist.all_reduce(n, op=dist.ReduceOp.SUM)
                dist.all_reduce(lo, op=dist.ReduceOp.MIN)
                dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            res[mode] = {"warmup_ms": float(t[0]), "sampling_ms": float(t[1]), "sampling_steps_x_chains_per_s": float(n[0]) / (float(t[1]) * 1e-3),
                         "allreduce_calls": calls, "allreduce_us_total": float(t[2]),
                         "mass_matrix_identical_on_all_ranks": bool(torch.equal(lo, hi)) if mode == "pooled" else None}
            s.close()
        if comm is not None:
            comm.close()
        model.close()
        out["cfg4_eight_schools_8192_chains"] = dict(res, chains_total=total, chains_per_gpu=per, scaling="strong",
                                                     config="DefaultConfig: EHMC(1024) + DualAvg(0.8) + DiagonalMassMatrixTuner; 500 warmup + 500 sampling iterations",
                                                     collective="ncclAllReduce(sum, f64, 2n+1 = 21 doubles) per mass-matrix window through rn_comm (NCCL over NVLink)")
    except Exception as e:  # a side measurement must not take the headline down
        out["cfg4_eight_schools_8192_chains"] = {"error": str(e)[:300]}

    # ---- cfg5: 4096 chains sharded ----
    try:
        mm = _load_npz_model("cfg5_primal")
        if mm is None:
            out["cfg5_poisson_glm_4096_chains"] = {"unavailable": "build/models/cfg5_primal.npz not built"}
        else:
            model = api.CudaModel(mm[0], mm[1], device=local_rank)
            total = 4096
            per = total // world
            # the step size comes from 30 warmup iterations of DualAvg(0.8) (a fixed guess from a random start is rejected
            # every time on a posterior this narrow); the timed part is the sampling phase with that adapted step
            cfg5 = api.make_config(iterations=2, warmupIterations=30, sampler=api.HMCSampler(N_STEPS), stepSizeTuner=api.DualAvgTuner(0.8),
                                   massMatrixTuner=api.IdentityMassMatrixTuner(), launchIterations=2)
            rate, secs, acc = device_rate(model, cfg5, per, 2, 1, 1000 + rank * per)
            out["cfg5_poisson_glm_4096_chains"] = {"steps_x_chains_per_s": rate, "seconds": secs, "accept_rate": acc, "chains_total": total,
                                                   "chains_per_gpu": per, "scaling": "strong", "rows": 1000000, "groups": 1000,
                                                   "config": "HMC(nSteps=5), step size from 30 DualAvg(0.8) warmup iterations, primal RIR + adjoint gradient (Lookup -> scatter)"}
            model.close()
    except Exception as e:
        out["cfg5_poisson_glm_4096_chains"] = {"error": str(e)[:300]}

    # ---- cfg3: 2048 chains on one GPU ----
    try:
        mm = _load_npz_model("cfg3_primal")
        if mm is None:
            out["cfg3_logreg_2048_chains"] = {"unavailable": "build/models/cfg3_primal.npz not built"}
        else:
            model = api.CudaModel(mm[0], mm[1], device=local_rank)
            cfg = static(0.01, 2)
            rate, secs, acc = device_rate(model, cfg, 2048, 2, 1, 1000)
            src = model.emit_source(cfg)
            out["cfg3_logreg_2048_chains"] = {"steps_x_chains_per_s_per_gpu": rate / world, "seconds": secs, "accept_rate": acc, "chains_per_gpu": 2048,
                                              "rows": 100000, "covariates": 50, "config": "HMC(nSteps=5), static step 0.01, primal RIR + adjoint gradient",
                                              "kernel": "chain-batched DMMA (mma.sync.m8n8k4.f64)" if "rn_dmma(z" in src else "rows across lanes"}
            model.close()
    except Exception as e:
        out["cfg3_logreg_2048_chains"] = {"error": str(e)[:300]}
    return out


def _seeded_chains(total, k):
    """all chains when k covers them, else a fixed, seeded choice of k of them (ascending)"""
    if k >= total:
        return np.arange(total)
    return np.sort(np.random.default_rng(0).choice(total, k, replace=False))


def dump_outputs(out_dir, d_samples):
    """The draws the last timed step returned to its caller (d_samples: [iterations][n][chains] fp64 on the device), as
      last_draw.npy  [n][chains]          the final position of every chain (a seeded sample beyond 16 MB)
      samples.npy    [iterations][n][k]   every draw of a seeded sample of k chains (at most 47 MB; the last
                                          iterations only if one chain's draws alone exceed that)"""
    import torch
    iters, n, chains = d_samples.shape
    os.makedirs(out_dir, exist_ok=True)
    pick = torch.from_numpy(_seeded_chains(chains, DUMP_LAST_DRAW_BYTES // (8 * n))).to(d_samples.device)
    np.save(os.path.join(out_dir, "last_draw.npy"), d_samples[-1].index_select(1, pick).cpu().numpy())
    it = min(iters, DUMP_SAMPLES_BYTES // (8 * n))
    pick = torch.from_numpy(_seeded_chains(chains, DUMP_SAMPLES_BYTES // (8 * n * it))).to(d_samples.device)
    np.save(os.path.join(out_dir, "samples.npy"), d_samples[iters - it:].index_select(2, pick).cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--chains", type=int, default=151552,
                    help="chains per GPU; default = 148 SMs x 4 resident CTAs x 128 threads x 2 waves")
    ap.add_argument("--iters", type=int, default=100, help="HMC iterations per step")
    ap.add_argument("--math", default="parity", choices=["parity", "fast"])
    ap.add_argument("--grad", default="auto", choices=["auto", "symbolic", "adjoint"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the cfg3/cfg4/cfg5 side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the draws of the last timed step to DIR/*.npy (rank 0's chains when sharded)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    from rainier_b200 import abi, api

    if "RN_KERNEL_CACHE" not in os.environ and os.path.isdir(os.path.join(ROOT, "build", "kcache")):
        # NVRTC of the 1000-parameter model: ~35 s otherwise.  A temporary copy of build()'s cubins takes the kernels
        # compiled at run time, so that the tree stays as build() left it
        kcache = tempfile.mkdtemp(prefix="rn_kcache_")
        atexit.register(shutil.rmtree, kcache, True)
        shutil.copytree(os.path.join(ROOT, "build", "kcache"), kcache, dirs_exist_ok=True)
        os.environ["RN_KERNEL_CACHE"] = kcache
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    C_, I_ = args.chains, args.iters
    rir = open(os.path.join(ROOT, "rainier_b200", "models", "funnel10.rir"), "rb").read()
    model = api.CudaModel(rir, [], device=local_rank)
    cfg = api.make_config(iterations=I_, warmupIterations=0, sampler=api.HMCSampler(N_STEPS),
                          stepSizeTuner=api.StaticStepSize(STEP_SIZE), massMatrixTuner=api.IdentityMassMatrixTuner(),
                          mathMode=abi.RN_MATH_FAST if args.math == "fast" else abi.RN_MATH_PARITY,
                          gradientMode={"auto": 0, "symbolic": 1, "adjoint": 2}[args.grad], launchIterations=I_)
    seeds = np.arange(C_, dtype=np.int64) + 1000 + rank * C_  # chain c of the job: ScalaRNG(1000 + c)

    # ---------------- device-resident leg ("value") ----------------
    smp = api.CudaSampler(model, cfg, seeds=seeds)
    smp.warmup(-1)  # LeapFrog.initialize (no warmup iterations configured)
    stream = torch.cuda.ExternalStream(smp.stream, device=torch.device("cuda", local_rank))
    d_samples = torch.empty((I_, N_DIM, C_), dtype=torch.float64, device="cuda")
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device="cuda")  # > 126 MB L2
    for _ in range(args.warmup):
        smp.run(I_, d_samples.data_ptr())
    smp.sync()
    launches0 = smp.launches
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    with ClockSampler(local_rank) as clocks:
        for k in range(args.steps):
            with torch.cuda.stream(stream):
                flush.zero_()  # L2 flush between timed steps (outside the per-step events)
                ev[k][0].record(stream)
            smp.run(I_, d_samples.data_ptr())
            ev[k][1].record(stream)
        smp.sync()
        torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = sum(a.elapsed_time(b) for a, b in ev)
    launches = smp.launches - launches0
    stats, _ = smp.stats()
    acc = float(np.mean([s.accepted / max(1, s.iterations) for s in stats[:4096]]))
    t_total = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_total, op=dist.ReduceOp.MAX)
    ms_max = float(t_total.item())
    total_steps = float(world) * C_ * I_ * N_STEPS * args.steps
    value = total_steps / (ms_max * 1e-3)
    smp.close()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_samples)

    # ---------------- end-to-end leg: public one-call API (rn_sample over the C ABI), HOST buffers ----------------
    # every step: seeds host->device, all samples device->host.  Headline = page-locked caller buffer (rn_host_alloc,
    # what the JNI shim hands the JVM as a direct ByteBuffer); also reported for a pageable caller buffer.
    e2e_cfg, keep = api.lower_config(cfg)
    import ctypes as CT
    seeds_pin = api.PinnedBuffer((C_,), device=local_rank, dtype=np.int64)  # inputs come from page-locked memory too
    seeds_pin.array[:] = seeds
    seeds_host = seeds_pin.array
    pin = api.PinnedBuffer((C_, I_, N_DIM), device=local_rank)
    pageable = np.empty((C_, I_, N_DIM))

    def e2e_leg(buf, n_rep):
        """every call timed on its own (host clock around the blocking rn_sample); the value is computed from the MEDIAN
        call -- the box is a shared host and a single call that collides with another tenant's PCIe/CPU traffic would
        otherwise decide the number (min/mean/max are reported next to it)"""
        def step():
            rc = api.lib().rn_sample(model.h, CT.byref(e2e_cfg), seeds_host.ctypes.data, C_, buf.ctypes.data, None, None)
            if rc != 0:
                raise RuntimeError(api.lib().rn_last_error().decode())
        for _ in range(3):  # warm: page-faults the host buffer, pins the staging ring, grows the device scratch pool
            step()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        times = []
        for _ in range(n_rep):
            t0 = time.perf_counter()
            step()
            times.append(time.perf_counter() - t0)
        t = torch.tensor([float(np.median(times)), min(times), float(np.mean(times)), max(times)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        med, lo, mean, hi = (float(x) for x in t.tolist())
        units = float(world) * C_ * I_ * N_STEPS
        return units / med, {"median": med * 1e3, "min": lo * 1e3, "mean": mean * 1e3, "max": hi * 1e3}

    n_e2e = args.steps
    # supplementary: the same call returning only Trace.diagnostics (rHat / ESS reduced on the device, rn_config.diagnostics
    # with samples == NULL) -- what the path does when the caller needs summaries rather than 1.2 GB of draws
    diag_cfg, keep2 = api.lower_config(cfg)
    diag_out = np.empty((N_DIM, 2))
    diag_cfg.diagnostics = diag_out.ctypes.data_as(CT.POINTER(CT.c_double))

    def diag_step():
        rc = api.lib().rn_sample(model.h, CT.byref(diag_cfg), seeds_host.ctypes.data, C_, None, None, None)
        if rc != 0:
            raise RuntimeError(api.lib().rn_last_error().decode())
    for _ in range(2):
        diag_step()
    tt = []
    for _ in range(n_e2e):
        t0 = time.perf_counter()
        diag_step()
        tt.append(time.perf_counter() - t0)
    diag_ms = float(np.median(tt)) * 1e3
    e2e_value, e2e_ms = e2e_leg(pin.array, n_e2e)
    e2e_pageable, e2e_pageable_ms = e2e_leg(pageable, n_e2e)
    pin.close()
    seeds_pin.close()

    extras = None if args.no_configs else extra_configs(args, torch, dist, api, abi, rank, local_rank, world)
    if rank == 0:
        peaks, peak_kind = measured_peaks()
        cap = ncu_capture(args.math)
        have_cap = bool(cap) and (C_, I_) == (151552, 100)
        bps = bytes_per_leapfrog_step(N_DIM, N_STEPS)
        per_gpu_rate = value / world
        achieved = per_gpu_rate * bps / 1e9
        counts = model.op_counts(cfg)
        evals_per_step = (N_STEPS + 1) / N_STEPS  # l+1 density evaluations per takeSteps(l)
        flops_step = counts["flops_invariant"] * evals_per_step + 6.0 * N_DIM  # + integrator updates
        line = {
            "metric": METRIC, "value": value, "unit": "leapfrog-steps*chains/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "neals_funnel_10d_hmc_nsteps5", "sampler": "HMC(nSteps=5)", "step_size": STEP_SIZE,
                       "chains_per_gpu": C_, "iterations_per_step": I_, "math": args.math, "gradient": args.grad,
                       "parallelism": "chains sharded over %d GPU(s), no data-path collective" % world,
                       "l2": "state %.0f MB < L2; L2 flushed (256 MB write) between timed steps; sample stream %.0f MB/step" % (
                           C_ * (3 * N_DIM + 8) * 8 / 1e6, C_ * I_ * N_DIM * 8 / 1e6),
                       "accept_rate": acc},
            "gpu_launches": int(launches),
            "clocks": clocks.summary(),
            "e2e": {"value": e2e_value, "unit": "leapfrog-steps*chains/s", "h2d_bytes_per_step": int(C_ * 8),
                    "d2h_bytes_per_step": int(C_ * I_ * N_DIM * 8),
                    "api": "rn_sample (C ABI), host buffers: seeds in, [chains][iterations][n] samples out (page-locked, rn_host_alloc)",
                    "steps": n_e2e, "ms_per_call": e2e_ms, "statistic": "median call (max over ranks)",
                    "pageable_caller_buffer_value": e2e_pageable, "pageable_ms_per_call": e2e_pageable_ms,
                    "diagnostics_only": {"value": C_ * I_ * N_STEPS / (diag_ms * 1e-3), "ms_per_call": diag_ms, "d2h_bytes_per_step": N_DIM * 16,
                                         "max_rhat": float(np.max(diag_out[:, 0])), "min_ess": float(np.min(diag_out[:, 1])),
                                         "note": "per rank; same rn_sample call with samples=NULL, rn_config.diagnostics set"}},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": achieved / peaks["hbm_gbs"],
                         "traffic": cap["dram_bytes"] if have_cap else None,
                         "traffic_unit": "bytes per rn_k_iter launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)",
                         "traffic_source": cap["source"] if have_cap else None,
                         # the same fraction computed from the bytes that actually crossed the HBM interface (state is L2-resident
                         # across the 100 iterations of a launch, so this is well below the compulsory-traffic figure)
                         "measured_traffic_frac": (cap["dram_bytes"] / (ms_max / args.steps * 1e-3) / 1e9 / peaks["hbm_gbs"]) if have_cap else None,
                         "algorithmic_bytes_per_launch": bps * C_ * I_ * N_STEPS, "peak_source": peak_kind,
                         "bytes_per_leapfrog_step": bps,
                         "note": "compulsory-traffic accounting (SURVEY.md 8d); the kernel is bound by the FP64 pipe / instruction issue, see fp64"},
            "fp64": {"flops_per_leapfrog_step": flops_step, "special_per_leapfrog_step": counts["special_invariant"] * evals_per_step,
                     "achieved_tflops": per_gpu_rate * flops_step / 1e12,
                     "ncu_fp64_pipe_active_pct": cap.get("fp64_pipe_active_pct") if have_cap else None,
                     "ncu_issue_active_pct": cap.get("issue_active_pct") if have_cap else None,
                     "ncu_source": cap["source"] if have_cap else None},
        }
        try:  # the end-to-end call is bound by the device->host link, not by the kernel: say how close to it the call runs
            gbs = C_ * I_ * N_DIM * 8 / (float(e2e_ms["median"]) * 1e-3) / 1e9
            line["e2e"]["pcie"] = {"achieved_gbs": gbs, "measured_d2h_gbs": 56.7, "frac": gbs / 56.7,
                                   "source": "profiles/r1_pcie_probe.txt (page-locked cuMemcpyDtoH on a B200 box of this pool)",
                                   "note": "per rank; whole rn_sample call (create, kernels, drain, stats) over the sample bytes"}
        except Exception:
            pass
        if extras is not None:
            line["configs"] = extras
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline_leg()
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
