#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 batched-chain backend.

Metric (BASELINE.json): Lotka-Volterra two-level delayed-acceptance chain-steps/s
(and ESS/s), weak-scaled: 65,536 chains per GPU (= C5's 524,288 chains at 8 GPUs).

  python bench.py --gpus 1 --steps K --warmup W            # our arm
  python bench.py --impl reference --steps K --warmup W    # CPU arm (oracle port, all host threads)
  torchrun ... bench.py --gpus N ...                        # one rank per GPU, NCCL
  python bench.py ... --dump-outputs DIR                    # also write the timed path's final chain state as .npy

A "step" is one pass of the hot path over the whole ensemble: one yg_run launch
of `--transitions` (default 300) Metropolis-Hastings transitions of every chain, so that the
default 20 timed steps span about 2 s.  Rank 0 prints ONE JSON line.

  --scaling strong     C5's literal reading: 524,288 chains in total, sharded over the N GPUs
                       (default: weak, 65,536 chains per GPU)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import bench_problems as bp     # noqa: E402

CHAINS_PER_GPU = 65536
STRONG_TOTAL_CHAINS = 524288
METRIC = "LV two-level delayed-acceptance chain-steps/s"
UNIT = "chain-steps/s"


def workload_config(args, n_gpus):
    strong = getattr(args, "scaling", "weak") == "strong"
    return {
        "workload": "C5 example_inference_lotkaVolterra_twoLevel: LV RK4 forward (Nc=64 coarse / Nf=512 fine, "
                    "nData=10 design points, T=10), Gaussian likelihood (var 0.04), prior N(0,1.4 I), "
                    "base proposal 0.1 I, sub-chain J=3, theta0 = truth + 0.05 N(0,I)",
        "chains_per_gpu": args.chains,
        "total_chains": args.chains * n_gpus,
        "transitions_per_step": args.transitions,
        "parallelism": f"chains sharded, {n_gpus} x {args.chains}, no data-path collective"
                       + (" (strong scaling: 524,288 chains in total)" if strong else ""),
        "l2": "L2 flushed (512 MiB write) between timed iterations; the per-chain state (4 MiB) is smaller than L2",
    }


# --------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md "clocks line")
# --------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, pw = [], [], set(), []
        for (t, line) in self.rows:
            if t < t0 - 0.05 or t > t1 + 0.05:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------
# DRAM traffic of the dominant kernel: read at run time from the committed ncu capture
# --------------------------------------------------------------------------------------
_UNIT = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}


def ncu_traffic_per_launch(chains, kernel="lv_mh_kernel"):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel`, from the newest committed
    `ncu --set full` summary under profiles/ whose capture ran this ensemble size (the summary's header row
    'chains_per_gpu' names it).  Returns (bytes or None, source)."""
    import csv
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_%s_ncu_full.csv" % kernel)), reverse=True):
        try:
            rows = {r[0]: r for r in csv.reader(open(path)) if r}
            if "chains_per_gpu" in rows and int(float(rows["chains_per_gpu"][2])) != int(chains):
                continue
            if "chains_per_gpu" not in rows and int(chains) != CHAINS_PER_GPU:
                continue
            tot = 0.0
            for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                r = rows[key]
                vals = [float(x) for x in r[2:] if x not in ("", "nan", "-nan")]      # a cut-short launch reads nan
                tot += _UNIT[r[1]] * sum(vals) / len(vals)
            return tot, "ncu dram__bytes_read.sum + dram__bytes_write.sum per launch, %s (parsed at run time)" % os.path.relpath(path, ROOT)
        except Exception:
            continue
    return None, "no committed ncu capture of %s at %d chains" % (kernel, chains)


# --------------------------------------------------------------------------------------
# CPU arm: the oracle port (C, OpenMP) on the host cores
# --------------------------------------------------------------------------------------
def cpu_chain_steps_per_s(meta, arrays, target_seconds, seed=11):
    """Times oracle/yagre_oracle.c (yo_run_philox) on all host threads over a bounded sample
    of the same workload: chains x transitions grown until about target_seconds of work."""
    from oracle import cport
    pb = cport.Problem(meta, arrays)
    # every host core this process may use (torchrun exports OMP_NUM_THREADS=1: ask explicitly)
    threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    n_chains, n_tr = max(8 * threads, 64), 20
    th0 = bp.lv_initial_states(n_chains)
    t = time.perf_counter()
    cport.run_philox(pb, th0, seed, n_tr, store=False, n_threads=threads)
    dt = time.perf_counter() - t
    rate = n_chains * n_tr / dt
    n_tr = int(max(20, min(20000, target_seconds * rate / n_chains)))
    t = time.perf_counter()
    r = cport.run_philox(pb, th0, seed, n_tr, store=False, n_threads=threads)
    dt = time.perf_counter() - t
    return dict(value=n_chains * n_tr / dt, seconds=dt, threads=threads, chains=n_chains, transitions=n_tr,
                accept=float(r["n_accept"].sum()) / (n_chains * n_tr))


def cpu_ess_per_s(meta, arrays, steps, burnin, target_seconds, rate_hint, seed=13):
    """ESS/s of the CPU port on the example's sampling run (`steps` transitions, burn-in discarded; ESS per chain =
    (N - burnIn) // IAT_max, example_inference_lotkaVolterra_twoLevel.py:117-118,132; the oracle's IAT is pinned to
    the reference's integrated_autocorrelation).  Chains sized for about target_seconds of sampling."""
    from oracle import cport
    pb = cport.Problem(meta, arrays)
    threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    n_chains = int(max(threads, min(8 * threads, target_seconds * rate_hint / steps)))
    n_chains = max(threads, (n_chains // threads) * threads)
    th0 = bp.lv_initial_states(n_chains)
    t = time.perf_counter()
    r = cport.run_philox(pb, th0, seed, steps, store=True, n_threads=threads)
    dt = time.perf_counter() - t
    ess, iats = 0, []
    for c in range(n_chains):
        iat = max(cport.iat(r["traj"][c, burnin:], "max"), 1)
        iats.append(iat)
        ess += (steps - burnin) // iat
    return dict(ess_per_s=ess / dt, ensemble_ess=float(ess), mean_iat_max=float(np.mean(iats)), chains=n_chains,
                chain_length=steps, burn_in=burnin, sampling_s=dt, threads=threads)


def python_reference_timing():
    """The pure-Python reference's own numbers (oracle/time_reference.py, run in the build container: the
    reference cannot travel to the GPU box).  Reported beside the C port, never as the ratio's denominator."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02_reference_python_timing.json")))
        return {"measured_in": "build container (%d cores), NOT on this box" % d["host"]["cores"],
                "rk4_plugin": {k: d["rk4_plugin"][k] for k in ("chain_steps_per_s", "chain_steps_per_s_per_core", "ess_per_s", "processes")},
                "as_shipped_solve_ivp": {k: d["as_shipped_solve_ivp"][k] for k in ("chain_steps_per_s", "chain_steps_per_s_per_core", "ess_per_s", "processes")},
                "source": "profiles/r02_reference_python_timing.json (oracle/time_reference.py)"}
    except Exception:
        return None


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    meta, arrays = bp.lv_problem(True)
    cfg = workload_config(args, args.gpus)
    times, units, info = [], [], None
    for i in range(args.warmup + args.steps):
        info = cpu_chain_steps_per_s(meta, arrays, args.cpu_seconds / max(args.steps, 1), seed=11 + i)
        if i >= args.warmup:
            times.append(info["seconds"]); units.append(info["chains"] * info["transitions"])
    value = sum(units) / sum(times)
    sample = (f"{info['chains']} chains x {info['transitions']} transitions per step, same problem/noise keying, "
              f"oracle/yagre_oracle.c (C restatement of the reference step, -O2 -ffp-contract=off, OpenMP)")
    ess = None
    if not args.no_ess:
        ess = cpu_ess_per_s(meta, arrays, args.ess_steps, args.ess_burnin, min(args.cpu_seconds, 10.0), value)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": info["threads"], "kind": "port", "sample": sample,
                         "ess_per_s": ess and ess["ess_per_s"], "ess": ess, "python_reference": python_reference_timing()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "ess": ess and {"ess_per_s": ess["ess_per_s"], "cores": ess["threads"], "ensemble_ess": ess["ensemble_ess"],
                        "mean_iat_max": ess["mean_iat_max"], "chain_length": ess["chain_length"], "burn_in": ess["burn_in"]},
        "cores": info["threads"],
        "gpu_launches": 0,
        "note": "the reference is pure Python (~40 chain-steps/s/core with an RK4 plugin, BASELINE.md); "
                "it cannot travel to the GPU box, so this arm times the C port of the same algorithm",
    }
    emit(line)


# --------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------
def run_gpu_arm(args):
    import torch
    import torch.distributed as dist
    from yagre_mcmc_b200.ensemble import ChainEnsemble, LoweredProblem, fp64_peak_tflops, iat_ess, rk4_loop_steps_per_s

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
    dev = torch.device("cuda", local)
    n_gpus = world

    meta, arrays = bp.lv_problem(True)
    pb = LoweredProblem(meta, arrays)
    if args.scaling == "strong":            # C5's literal reading: 524,288 chains in total over the N GPUs
        args.chains = STRONG_TOTAL_CHAINS // world
    nc, S = args.chains, args.transitions
    offset = rank * nc
    ens = ChainEnsemble(pb, nc, device=local, seed=args.seed, chain_offset=offset)
    th0 = bp.lv_initial_states(nc, chain_offset=offset)
    ens.set_state(th0)
    ens.run(args.burnin, samples=False)                       # burn-in so the timed steps are in stationarity
    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)
    pooled = None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def one_step(timed):
        nonlocal pooled
        flush.fill_(1)                                        # L2 flush between iterations
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ens.run(S, samples=False)
        if world > 1:                                         # pooled moments / R-hat statistics: the only collective
            pooled = ens.pooled_stats()
            dist.all_reduce(pooled)
        e1.record()
        return (e0, e1)

    for _ in range(args.warmup):
        one_step(False)
    barrier()
    c0 = ens.counters()
    l0 = ens.last_launch()["launches"]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    barrier()
    t0 = time.time()
    evs = [one_step(True) for _ in range(args.steps)]
    barrier()
    t1 = time.time()
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    ms = [a.elapsed_time(b) for (a, b) in evs]
    total_ms = float(sum(ms))
    c1 = ens.counters()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: v.double().cpu().numpy() for k, v in ens.state().items() if torch.is_tensor(v)},
                     f"_rank{rank}" if world > 1 else "")
    launches = ens.last_launch()["launches"] - l0
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    evals = torch.tensor([c1["coarse_evals"] - c0["coarse_evals"], c1["fine_evals"] - c0["fine_evals"],
                          c1["accepted"] - c0["accepted"], launches], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(evals)
    total_ms_max = float(t.item())
    coarse_ev, fine_ev, n_acc, launches_all = [float(x) for x in evals.tolist()]
    units = float(nc) * n_gpus * S * args.steps
    value = units / (total_ms_max * 1e-3)

    # ---- roofline of the dominant kernel (lv_mh_kernel): FP64 pipe ---------------------------------
    flops = bp.lv_flops_per_eval(meta["n_data"], meta["Nc"]) * coarse_ev + \
        bp.lv_flops_per_eval(meta["n_data"], meta["Nf"]) * fine_ev
    peak = fp64_peak_tflops(local, 30.0)
    achieved = flops / n_gpus / (total_ms_max * 1e-3) / 1e12          # per GPU
    # RK4 steps per second of one GPU against (a) the instructions the kernel issues for them and (b) the bare
    # integrator loop measured live: the stage-point RK4 step (lv_model.cuh) executes the 58 textbook flop of a
    # step in 20 FP64-pipe instructions, six of which take 1.5 issue slots (three vector-register sources)
    rk4_rate = flops / bp.LV_FLOP_PER_RK4_STEP / n_gpus / (total_ms_max * 1e-3)
    loop_rate = rk4_loop_steps_per_s(local, 30.0)
    traffic, traffic_src = ncu_traffic_per_launch(nc)
    roofline = {"bound": "fp64", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                # the two fractions that say how busy the pipe is, beside the algorithmic one (VERDICT r1 weak item 3)
                "frac_executed": rk4_rate * 40e-12 / peak, "frac_issue_slots": rk4_rate * 46e-12 / peak,
                "frac_of_bare_rk4_loop": rk4_rate / loop_rate,
                "frac_note": "frac counts SURVEY 8d's algorithmic (textbook) 58 flop per RK4 step; the kernel issues 20 FP64 "
                             "instructions (40 flop slots, 23 issue slots) for them, so frac can exceed 1: frac_executed = issued "
                             "FP64 instructions x 2 / peak, frac_issue_slots weights the six three-register-source instructions "
                             "1.5x, frac_of_bare_rk4_loop = RK4 steps/s of the whole MH kernel / of nothing but lv_integrate",
                "executed": {"fp64_instr_per_rk4_step": 20, "issue_slots_per_rk4_step": 23,
                             "tflops": rk4_rate * 40e-12, "frac": rk4_rate * 40e-12 / peak,
                             "slot_frac": rk4_rate * 46e-12 / peak},
                "rk4_loop": {"steps_per_s": rk4_rate, "bare_loop_steps_per_s": loop_rate, "frac": rk4_rate / loop_rate,
                             "note": "whole MH kernel against nothing but lv_integrate (1024 threads per SM; the bare loop is flat from 512 up)"},
                # dram__bytes_read.sum + dram__bytes_write.sum per launch, parsed at run time from the committed
                # `ncu --set full` capture of this kernel at this ensemble size (null when no capture matches)
                "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": 96.0 * args.chains,
                "kernel": "lv_mh_kernel<true>", "launch_ms": total_ms_max / args.steps,
                "algorithmic_flop_per_launch": flops / n_gpus / args.steps,
                "peak_source": "yg_fp64_peak: DFMA micro-benchmarks (pure chains / two-source 30-instruction mix) measured "
                               "live on this GPU, best of variants; MEASURED_PEAKS.json has no fp64 entry",
                "forward_evals_per_transition": {"coarse": coarse_ev / units, "fine": fine_ev / units}}

    # ---- end to end through the public API: host theta0 in, host trajectory out ---------------------
    e2e = None
    if not args.no_e2e:
        # Every step: H2D of the step's initial states (pinned), yg_set_state + yg_run with samples, D2H of the
        # step's trajectory and accept counts (pinned).  The D2H of step i runs on a copy stream while step i+1
        # computes (two output buffers); the timed region spans the first H2D to the last D2H.
        n_e2e = max(5, args.steps // 2)
        host_in = torch.from_numpy(th0).pin_memory()
        host_out = [torch.empty((S, 2, nc), dtype=torch.float64).pin_memory() for _ in range(2)]
        host_acc = [torch.empty((nc,), dtype=torch.int64).pin_memory() for _ in range(2)]
        dev_out = [torch.empty((S, 2, nc), dtype=torch.float64, device=dev) for _ in range(2)]
        dev_acc = [torch.empty((nc,), dtype=torch.int64, device=dev) for _ in range(2)]
        copied = [None, None]
        main, side = torch.cuda.current_stream(dev), torch.cuda.Stream(dev)

        def e2e_step(i):
            b = i % 2
            flush.fill_(1)
            if copied[b] is not None:
                main.wait_event(copied[b])                              # buffer b was read out two steps ago
            ens.set_state(host_in.to(dev, non_blocking=True))           # H2D + log-posterior of the start state
            ens.run(S, samples_out=dev_out[b])
            dev_acc[b].copy_(ens.accept_counts())
            done = torch.cuda.Event()
            done.record(main)
            side.wait_event(done)
            with torch.cuda.stream(side):
                host_out[b].copy_(dev_out[b], non_blocking=True)        # D2H trajectory
                host_acc[b].copy_(dev_acc[b], non_blocking=True)        # D2H acceptance counts
                copied[b] = torch.cuda.Event()
                copied[b].record(side)

        for i in range(2):
            e2e_step(i)
        torch.cuda.synchronize(dev)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(main)
        for i in range(n_e2e):
            e2e_step(i)
        fin = torch.cuda.Event()
        fin.record(side)
        main.wait_event(fin)
        e1.record(main)
        torch.cuda.synchronize(dev)
        et = torch.tensor([e0.elapsed_time(e1) / n_e2e], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(et, op=dist.ReduceOp.MAX)
        e2e = {"value": float(nc) * n_gpus * S / (float(et.item()) * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": int(host_in.numel() * 8), "d2h_bytes_per_step": int(host_out[0].numel() * 8 + nc * 8),
               "ms_per_step": float(et.item()), "steps": n_e2e,
               "path": "ChainEnsemble.set_state(pinned host theta0) + run(S, samples) + trajectory and accept counts to "
                       "pinned host; the D2H of a step overlaps the next step's kernels on a copy stream"}

    # ---- ESS/s: the sampling run of the example (5,000 steps, burn-in 100), IAT on the device -------------------
    # Three arms through the same handle type: the example's fixed proposal (0.1 I); the pooled proposal covariance
    # (burn-in -> all-reduce pooled moments -> restart from the last states: the reference's burn-in restart idiom,
    # example_inference_linearModel_twoLevel.py:228,236); per-chain adaptive Metropolis on the coarse proposal.
    ess = None
    if not args.no_ess:
        from yagre_mcmc_b200.parallel import pooled_diagnostics, pooled_proposal_covariance, split_rhat

        def timed_run(e, n, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = e.run(n, **kw)
            e1.record()
            torch.cuda.synchronize(dev)
            return out, e0.elapsed_time(e1)

        def ess_of(e, pre_ms, label):
            """Sampling run of the example on ensemble e (state already set); pre_ms = device time already spent on
            burn-in / pooling for this arm, charged to the ESS/s denominator."""
            # the trajectory buffer (5.2 GB at the default sizes) is allocated once, outside the timed region
            out, run_ms = timed_run(e, args.ess_steps, samples_out=ess_buf)
            e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e2.record()
            iat, ess_c = iat_ess(out["samples"][args.ess_burnin:], "max")
            e3.record()
            torch.cuda.synchronize(dev)
            tt = torch.tensor([run_ms + pre_ms, e2.elapsed_time(e3)], dtype=torch.float64, device=dev)
            ss = torch.tensor([float(ess_c.sum().item()), float(iat.double().sum().item()),
                               float((ess_c == 0).sum().item())], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                dist.all_reduce(ss)
            pd_ = pooled_diagnostics(e)
            srh = split_rhat(out["samples"][args.ess_burnin:])
            del out
            return {"ess_per_s": float(ss[0].item()) / (float(tt[0].item()) * 1e-3), "ensemble_ess": float(ss[0].item()),
                    "mean_iat_max": float(ss[1].item()) / (nc * n_gpus), "degenerate_chains": int(ss[2].item()),
                    "chain_length": args.ess_steps, "burn_in": args.ess_burnin, "sampling_ms": float(tt[0].item()),
                    "iat_kernel_ms": float(tt[1].item()), "proposal": label,
                    "chain_steps_per_s": float(nc) * n_gpus * args.ess_steps / (float(tt[0].item()) * 1e-3),
                    "diagnostics": {"n_chains": pd_["n_chains"], "pooled_mean": [float(x) for x in pd_["mean"]],
                                    "pooled_variance": [float(x) for x in np.diag(pd_["covariance"])],
                                    "acceptance_rate": float(pd_["acceptance_rate"]), "rhat": [float(x) for x in pd_["rhat"]],
                                    "split_rhat": [float(x) for x in srh],
                                    "collective": "all_reduce(sum) of %d doubles (NCCL)" % (3 + 2 * 2 + 2 * 4) if world > 1 else "single rank"}}

        ess_buf = torch.empty((args.ess_steps, 2, nc), dtype=torch.float64, device=dev)
        ens.set_state(th0)
        torch.cuda.synchronize(dev)
        barrier()
        ess = ess_of(ens, 0.0, "fixed 0.1 I (example_inference_lotkaVolterra_twoLevel.py:95-96)")
        ess["definition"] = ("per chain (N - burnIn) // IAT_max (example_inference_lotkaVolterra_twoLevel.py:117-118,132), "
                             "summed over chains / sampling wall time (burn-in and, for the pooled arm, the pooling run included)")
        # pooled proposal covariance: burn-in, pool over ALL chains of ALL ranks, restart from the last states
        ens.set_state(th0)
        barrier()
        _, burn_ms = timed_run(ens, args.pool_burnin, samples=False)
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        pooled_info = pooled_proposal_covariance(ens)
        last = ens.state()["theta"].t().contiguous()
        ens.set_state(last)
        p1.record()
        torch.cuda.synchronize(dev)
        ess["pooled"] = ess_of(ens, burn_ms + p0.elapsed_time(p1),
                               "pooled: chol(2.4^2/d Sigma_pooled) after %d burn-in transitions" % args.pool_burnin)
        ess["pooled"]["prop_L"] = [[float(x) for x in row] for row in pooled_info["prop_L"]]
        ess["pooled"]["pool_burnin"] = args.pool_burnin
        ens.set_proposal_factor(arrays["prop_L"])                    # back to the example's proposal
        # per-chain adaptive Metropolis on the coarse proposal (reference interface chain/adaptive.py:37-64)
        ens_am = ChainEnsemble(pb, nc, device=local, seed=args.seed + 1, chain_offset=offset,
                               adaptive=dict(idle=50, collection=300, eps=1e-8, refresh=10))
        ens_am.set_state(th0)
        barrier()
        _, burn_ms = timed_run(ens_am, args.pool_burnin, samples=False)
        last = ens_am.state()["theta"].t().contiguous()
        ens_am.set_state(last, keep_adaptation=True)
        ess["adaptive"] = ess_of(ens_am, burn_ms, "per-chain adaptive Metropolis (idle 50, collection 300, refresh 10 coarse "
                                                  "proposals) after %d burn-in transitions" % args.pool_burnin)
        ens_am.close()
        # tuned arm (profiles/r02_ess_sweep.txt): the sub-chain length is a user parameter like the proposal; J = 8
        # coarse steps with the pooled proposal covariance make almost every fine step an independent draw
        # (IAT_max -> 1) -- fewer chain-steps/s, more than twice the ESS/s of the example's J = 3 / 0.1 I
        meta_t, arrays_t = bp.lv_problem(True, J=args.tuned_j)
        ens_t = ChainEnsemble(LoweredProblem(meta_t, arrays_t), nc, device=local, seed=args.seed + 2, chain_offset=offset)
        ens_t.set_state(th0)
        barrier()
        _, burn_ms = timed_run(ens_t, args.pool_burnin, samples=False)
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        pooled_t = pooled_proposal_covariance(ens_t)
        last = ens_t.state()["theta"].t().contiguous()
        ens_t.set_state(last)
        p1.record()
        torch.cuda.synchronize(dev)
        ess["tuned"] = ess_of(ens_t, burn_ms + p0.elapsed_time(p1),
                              "sub-chain length J = %d (the example uses 3) + pooled proposal covariance chol(2.4^2/d Sigma_pooled) "
                              "after %d burn-in transitions" % (args.tuned_j, args.pool_burnin))
        ess["tuned"]["sub_chain_length"] = args.tuned_j
        ess["tuned"]["prop_L"] = [[float(x) for x in row] for row in pooled_t["prop_L"]]
        ess["tuned"]["over_example"] = ess["tuned"]["ess_per_s"] / ess["ess_per_s"]
        ens_t.close()
        del ess_buf

    # ---- the other BASELINE.json configs, briefly (rank 0, N = 1): parity-tested elsewhere, timed here ----
    others = None
    hbm_peak = None
    try:
        hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        pass
    if n_gpus == 1 and not args.no_configs:
        others = measure_other_configs(local, peak, value, hbm_peak or 6650.0)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    cpu = None
    if n_gpus == 1 and not args.no_cpu:
        info = cpu_chain_steps_per_s(meta, arrays, args.cpu_seconds)
        cess = None if args.no_ess else cpu_ess_per_s(meta, arrays, args.ess_steps, args.ess_burnin,
                                                      min(args.cpu_seconds, 10.0), info["value"])
        cpu = {"value": info["value"], "unit": UNIT, "cores": info["threads"], "kind": "port",
               "sample": f"{info['chains']} chains x {info['transitions']} transitions of the same workload "
                         f"({info['seconds']:.1f} s), oracle/yagre_oracle.c with OpenMP over chains",
               "accept_rate": info["accept"], "ess_per_s": cess and cess["ess_per_s"], "ess": cess,
               "python_reference": python_reference_timing()}

    # sample write-back roofline (secondary bound): bytes of the e2e/ESS path per chain-step = 8 d
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms_max / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": workload_config(args, n_gpus),
        "accept_rate": n_acc / units,
        "roofline": roofline,
        "roofline_hbm": {"bound": "hbm", "achieved": (ess and 16.0 * nc * args.ess_steps / (ess["sampling_ms"] * 1e-3) / 1e9),
                         "peak": hbm_peak or 6650.0, "unit": "GB/s",
                         "peak_source": "MEASURED_PEAKS.json" if hbm_peak else "fallback",
                         "note": "sample write-back (16 B per stored chain-step) during the ESS sampling run; far from "
                                 "the bound by design: the path is FP64-compute bound"},
        "cpu_baseline": cpu,
        # every GPU/CPU ratio a reader forms from this line is against THIS many host threads (VERDICT r1 weak item 8)
        "cpu_cores": cpu and cpu["cores"],
        "e2e": e2e,
        "ess": ess,
        "other_configs": others,
        "gpu_launches": int(launches_all),
        "clocks": clocks,
        "launch": ens.last_launch(),
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def measure_other_configs(device, fp64_peak, main_value, hbm_peak_gbs):
    """Device-timed chain-steps/s of C2, C3, C4, the adaptive / full-size / long-grid variants of C5 and the GEMM-sized
    linear model (state resident in HBM, 3 timed launches after a warm-up launch each).  Secondary numbers: the
    headline stays the C5 line."""
    import torch
    from yagre_mcmc_b200.ensemble import ChainEnsemble, LoweredProblem, fp64_tensor_peak_tflops

    def timed(ens, steps, reps=3, **kw):
        ens.run(steps, samples=False)
        torch.cuda.synchronize()
        c0 = ens.counters()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            ens.run(steps, **kw) if kw else ens.run(steps, samples=False)
        e1.record()
        torch.cuda.synchronize()
        c1 = ens.counters()
        ms = e0.elapsed_time(e1)
        return ms, {k: c1[k] - c0[k] for k in ("transitions", "accepted", "coarse_evals", "fine_evals")}

    def lv_entry(meta, ms, c, kernel):
        fl = bp.lv_flops_per_eval(meta["n_data"], meta["Nc"]) * c["coarse_evals"] if meta["levels"] == 2 else 0.0
        fl += bp.lv_flops_per_eval(meta["n_data"], meta["Nf"]) * c["fine_evals"]
        rk4 = fl / bp.LV_FLOP_PER_RK4_STEP / ms * 1e3
        return {"chain_steps_per_s": c["transitions"] / ms * 1e3, "accept_rate": c["accepted"] / c["transitions"],
                "fp64_tflops": fl / ms * 1e-9, "frac_of_fp64_peak": fl / ms * 1e-9 / fp64_peak,
                "frac_executed": rk4 * 40e-12 / fp64_peak, "kernel": kernel}

    # static per-step instruction counts of the one-chain-per-thread kernels, from the committed ncu capture
    try:
        gi = json.load(open(os.path.join(ROOT, "profiles", "r02_generic_instr.json")))
    except Exception:
        gi = {}

    def small_entry(name, ms, c, d, stored_ms, stored_steps, n_chains, kernel):
        """FP64-issue and HBM write-back fractions of a cheap-target kernel (SURVEY 8d: both bounds reported)."""
        e = {"chain_steps_per_s": c["transitions"] / ms * 1e3, "accept_rate": c["accepted"] / c["transitions"], "kernel": kernel}
        g = gi.get(name)
        if g:
            per_step = g["fp64_warp_inst_per_launch"] * 32.0 / g["chain_steps_per_launch"]     # thread-level, full warps
            e["roofline_fp64_issue"] = {
                "fp64_inst_per_chain_step": per_step, "achieved_tflops_issued": per_step * 2.0 * e["chain_steps_per_s"] * 1e-12,
                "peak": fp64_peak, "frac": per_step * 2.0 * e["chain_steps_per_s"] * 1e-12 / fp64_peak,
                "ncu_pipe_fp64_cycles_active_pct": g.get("pipe_fp64_cycles_active_pct"),
                "ncu_issue_active_pct": g.get("issue_active_pct"), "ncu_warps_active_pct": g.get("warps_active_pct"),
                "source": "instruction count: ncu sm__inst_executed_pipe_fp64.sum of profiles/r02_generic_instr.json; rate: this run"}
        stored_rate = n_chains * stored_steps / stored_ms * 1e3
        e["roofline_hbm_writeback"] = {"bytes_per_stored_chain_step": 8 * d, "chain_steps_per_s_with_samples": stored_rate,
                                       "achieved_gbs": 8.0 * d * stored_rate * 1e-9, "peak": hbm_peak_gbs,
                                       "frac": 8.0 * d * stored_rate * 1e-9 / hbm_peak_gbs}
        e["bound"] = ("latency: neither bound is approached at this ensemble size (one chain per thread, %d chains = %d warps "
                      "on %d sub-partitions)" % (n_chains, n_chains // 32, 148 * 4))
        return e

    out = {}
    # C4: LV single level, 65,536 chains
    meta, arrays = bp.lv_problem(False)
    ens = ChainEnsemble(LoweredProblem(meta, arrays), 65536, device=device, seed=5)
    ens.set_state(bp.lv_initial_states(65536))
    ms, c = timed(ens, 20)
    out["C4_lv_single_level_65536"] = lv_entry(meta, ms, c, "lv_mh_kernel<false>")
    ens.close()
    # C4 / C5 with per-chain adaptive Metropolis (VERDICT r1 item 1: within 2 % of the non-adaptive lines)
    ens = ChainEnsemble(LoweredProblem(meta, arrays), 65536, device=device, seed=5,
                        adaptive=dict(idle=50, collection=300, eps=1e-8, refresh=10))
    ens.set_state(bp.lv_initial_states(65536))
    ens.run(400, samples=False)
    ms, c = timed(ens, 20)
    out["C4_lv_single_level_adaptive_65536"] = lv_entry(meta, ms, c, "lv_mh_kernel<false>, per-chain adaptive Metropolis")
    ens.close()
    # ESS/s of C4 (example_inference_lotkaVolterra_singleLevel.py: 0.15 I proposal, acceptance 0.11) against the same
    # chains with the per-chain adaptive proposal: 16,384 chains x 2,000 transitions, burn-in 400 (adaptation included
    # in the time), IAT on the device
    from yagre_mcmc_b200.ensemble import iat_ess
    c4 = {}
    for label, ad in (("fixed_0.15I", None), ("adaptive", dict(idle=50, collection=300, eps=1e-8, refresh=10))):
        ens = ChainEnsemble(LoweredProblem(meta, arrays), 16384, device=device, seed=6, adaptive=ad)
        ens.set_state(bp.lv_initial_states(16384))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        smp = ens.run(2000, samples=True)["samples"]
        e1.record()
        torch.cuda.synchronize()
        iat, ess_c = iat_ess(smp[400:], "max")
        c4[label] = {"ess_per_s": float(ess_c.sum().item()) / (e0.elapsed_time(e1) * 1e-3), "mean_iat_max": float(iat.double().mean().item()),
                     "degenerate_chains": int((ess_c == 0).sum().item()),
                     "chain_steps_per_s": 16384 * 2000 / (e0.elapsed_time(e1) * 1e-3)}
        del smp
        ens.close()
    c4["adaptive_over_fixed"] = c4["adaptive"]["ess_per_s"] / c4["fixed_0.15I"]["ess_per_s"]
    out["C4_ess_16384x2000"] = c4
    meta, arrays = bp.lv_problem(True)
    ens = ChainEnsemble(LoweredProblem(meta, arrays), 65536, device=device, seed=5)
    ens.set_state(bp.lv_initial_states(65536))
    ens.run(150, samples=False)
    ms0, c0 = timed(ens, 50)
    ens.close()
    for label, ad in (("refresh10", dict(idle=50, collection=300, eps=1e-8, refresh=10)),
                      ("refresh1", dict(idle=50, collection=300, eps=1e-8, refresh=1))):
        ens = ChainEnsemble(LoweredProblem(meta, arrays), 65536, device=device, seed=5, adaptive=ad)
        ens.set_state(bp.lv_initial_states(65536))
        ens.run(150, samples=False)                      # past idle + collection (counted in coarse proposals)
        ms, c = timed(ens, 50)
        e = lv_entry(meta, ms, c, "lv_mh_kernel<true>, per-chain adaptive coarse proposal (%s)" % label)
        # time per forward evaluation performed (the adapted proposal changes acceptance, hence the work per step)
        e["ms_per_1e9_rk4_steps"] = ms / ((c["coarse_evals"] * meta["Nc"] + c["fine_evals"] * meta["Nf"]) * meta["n_data"] * 1e-9)
        e["same_for_fixed_proposal"] = ms0 / ((c0["coarse_evals"] * meta["Nc"] + c0["fine_evals"] * meta["Nf"]) * meta["n_data"] * 1e-9)
        e["rk4_rate_vs_fixed_proposal"] = e["same_for_fixed_proposal"] / e["ms_per_1e9_rk4_steps"]
        out["C5_lv_two_level_adaptive_%s_65536" % label] = e
        ens.close()
    # C5 at its literal size on ONE GPU: 524,288 chains (BASELINE.json configs[4]; strong-scaling base line)
    ens = ChainEnsemble(LoweredProblem(meta, arrays), 524288, device=device, seed=5)
    ens.set_state(bp.lv_initial_states(524288))
    ms, c = timed(ens, 50)
    out["C5_524288_one_gpu"] = lv_entry(meta, ms, c, "lv_mh_kernel<true>")
    out["C5_524288_one_gpu"]["vs_65536_chains"] = out["C5_524288_one_gpu"]["chain_steps_per_s"] / main_value
    ens.close()
    # C5 with the finer fine level SURVEY 8d asks to report as well: Nf = 1024
    meta, arrays = bp.lv_problem(True, Nf=1024)
    ens = ChainEnsemble(LoweredProblem(meta, arrays), 65536, device=device, seed=5)
    ens.set_state(bp.lv_initial_states(65536))
    ms, c = timed(ens, 20)
    out["C5_lv_two_level_Nf1024_65536"] = lv_entry(meta, ms, c, "lv_mh_kernel<true>")
    ens.close()
    # long observation grid (VERDICT r1 weak item 7): 256 design points per forward evaluation
    meta, arrays = bp.lv_problem(True, n_data=256)
    ens = ChainEnsemble(LoweredProblem(meta, arrays), 16384, device=device, seed=5)
    ens.set_state(bp.lv_initial_states(16384))
    ms, c = timed(ens, 10)
    out["C5_lv_two_level_ndata256_16384"] = lv_entry(meta, ms, c, "lv_mh_kernel<true>")
    out["C5_lv_two_level_ndata256_16384"]["launch"] = ens.last_launch()
    ens.close()
    # C3: linear two level (J = 5), 16,384 chains -- a few hundred FP64 instructions per step, latency bound
    meta, arrays = bp.linear_problem(True)
    ens = ChainEnsemble(LoweredProblem(meta, arrays), 16384, device=device, seed=5)
    ens.set_state(np.zeros((16384, 2)))
    ms, c = timed(ens, 5000)
    buf = torch.empty((5000, 2, 16384), dtype=torch.float64, device="cuda")
    sms, _ = timed(ens, 5000, reps=1, samples_out=buf)
    out["C3_linear_two_level_16384"] = small_entry("C3", ms, c, 2, sms, 5000, 16384,
                                                   "generic_mh_kernel<2,2,true> (warp-specialised: producer / consumer warps)")
    ens.close()
    # C3 with the adaptive error model of the same example (example_inference_linearModel_twoLevel.py:180-250,
    # chain/method/aem.py): per-chain error-model moments and the LRU(3) cache of the coarse likelihood in the step loop
    ens = ChainEnsemble(LoweredProblem(meta, arrays), 16384, device=device, seed=5, aem=dict(min_data=8, heuristic=True))
    ens.set_state(np.zeros((16384, 2)))
    ms, c = timed(ens, 5000)
    out["C3_linear_two_level_aem_16384"] = {
        "chain_steps_per_s": c["transitions"] / ms * 1e3, "accept_rate": c["accepted"] / c["transitions"],
        "coarse_evals_per_step": c["coarse_evals"] / c["transitions"], "fine_evals_per_step": c["fine_evals"] / c["transitions"],
        "kernel": "aem_mh_kernel (adaptive error model, min_data 8, noise-scaling heuristic)",
        "vs_plain_two_level": (c["transitions"] / ms * 1e3) / out["C3_linear_two_level_16384"]["chain_steps_per_s"]}
    ens.close()
    # ESS/s of C3 with and without the adaptive error model (SURVEY 8f rank 1: the error model lifts the acceptance of
    # the example and cuts its IAT): 16,384 chains x 20,000 transitions thinned by 4, burn-in 1,000, IAT on the device
    c3 = {}
    for label, aem in (("two_level", None), ("two_level_aem", dict(min_data=8, heuristic=True))):
        ens = ChainEnsemble(LoweredProblem(meta, arrays), 16384, device=device, seed=6, aem=aem)
        ens.set_state(np.zeros((16384, 2)))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        smp = ens.run(20000, thin=4, samples=True)["samples"]
        e1.record()
        torch.cuda.synchronize()
        iat, ess_c = iat_ess(smp[250:], "max")            # in units of stored (every 4th) states
        c3[label] = {"ess_per_s": float(ess_c.sum().item()) / (e0.elapsed_time(e1) * 1e-3),
                     "mean_iat_max_transitions": 4.0 * float(iat.double().mean().item()),
                     "degenerate_chains": int((ess_c == 0).sum().item()),
                     "chain_steps_per_s": 16384 * 20000 / (e0.elapsed_time(e1) * 1e-3)}
        del smp
        ens.close()
    c3["aem_over_plain"] = c3["two_level_aem"]["ess_per_s"] / c3["two_level"]["ess_per_s"]
    out["C3_ess_16384x20000"] = c3
    # C2: 2-D Gaussian target, per-chain adaptive Metropolis, 4,096 chains
    meta, arrays = bp.gauss2d_problem()
    ens = ChainEnsemble(LoweredProblem(meta, arrays), 4096, device=device, seed=5,
                        adaptive=dict(idle=5000, collection=5000, eps=1e-4))
    ens.set_state(np.tile([-8.0, -7.0], (4096, 1)))
    ens.run(12000, samples=False)
    ms, c = timed(ens, 5000)
    buf = torch.empty((5000, 2, 4096), dtype=torch.float64, device="cuda")
    sms, _ = timed(ens, 5000, reps=1, samples_out=buf)
    out["C2_gauss2d_adaptive_4096"] = small_entry("C2", ms, c, 2, sms, 5000, 4096,
                                                  "generic_mh_kernel<2,2,false> (adaptive; warp-specialised: producer / consumer warps)")
    ens.close()
    del buf
    # GEMM-sized linear model (SURVEY 8d variant): d = 64, dataDim = 256, 65,536 chains, FP64 tensor path
    tpeak = fp64_tensor_peak_tflops(device, 20.0)
    for (d_, dd_, two, J_, key) in ((64, 256, False, 1, "linear_d64_x256_65536"), (32, 96, True, 3, "linear_d32_x96_two_level_65536")):
        meta, arrays = bp.big_linear_problem(d_, dd_, 1, two_level=two, J=J_)
        mean, _ = bp.linear_gaussian_posterior(arrays, meta["levels"] - 1)
        for welford in (True, False):
            ens = ChainEnsemble(LoweredProblem(meta, arrays), 65536, device=device, seed=5, welford=welford)
            ens.set_state(np.tile(mean, (65536, 1)))
            ms, c = timed(ens, 50)
            fl = bp.big_linear_flops_per_eval(d_, dd_) * (c["coarse_evals"] + c["fine_evals"])
            e = {"chain_steps_per_s": c["transitions"] / ms * 1e3, "accept_rate": c["accepted"] / c["transitions"],
                 "fp64_tflops": fl / ms * 1e-9, "dmma_peak_tflops": tpeak, "frac_of_dmma_peak": fl / ms * 1e-9 / tpeak,
                 "kernel": "linear_dmma_mh_kernel",
                 "diagnostics": "FullDiagnostics (Welford moments of every chain maintained in L2)" if welford else
                                "AcceptanceRateDiagnostics (the default of the reference's builders, chain/builder.py:14-16)"}
            out[key if welford else key + "_acceptance_diagnostics"] = e
            ens.close()
    return out


DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def dump_outputs(out_dir, arrays, suffix=""):
    """Writes the chain state the timed steps leave behind (ChainEnsemble.state(): theta [d, n], logpost [levels, n],
    n_accept [n], Welford w_mean [d, n] and w_m2; chains on the last axis) as out_dir/<name><suffix>.npy in float64,
    so that two builds can be compared output for output.  Above DUMP_LIMIT_BYTES in all, a fixed seeded sample of
    the chains is written instead, and its chain indices as chain_index.npy."""
    n = arrays["theta"].shape[-1]
    per_chain = 8 * sum(a.size // n for a in arrays.values())
    if n * per_chain > DUMP_LIMIT_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n, DUMP_LIMIT_BYTES // (per_chain + 8), replace=False))
        arrays = {k: a[..., keep] for k, a in arrays.items()}
        arrays["chain_index"] = keep
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + suffix + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


_JSON_OUT = None


def protect_stdout():
    """stdout carries exactly ONE JSON line.  Libraries (NCCL's version banner, for one) write to file descriptor 1
    directly, so fd 1 is pointed at stderr for the whole run and the JSON line goes to a private copy of the
    original stdout."""
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line):
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


def main():
    protect_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--chains", type=int, default=CHAINS_PER_GPU, help="chains per GPU")
    ap.add_argument("--transitions", type=int, default=300, help="MH transitions of every chain per bench step "
                    "(300 x 65,536 chains = about 0.1 s per step: the default 20 timed steps span 2 s)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --chains per GPU; strong: 524,288 chains in total (BASELINE.json configs[4])")
    ap.add_argument("--pool-burnin", type=int, default=500, help="burn-in transitions before the proposal covariance is pooled")
    ap.add_argument("--tuned-j", type=int, default=8, help="sub-chain length of the tuned ESS arm (profiles/r02_ess_sweep.txt)")
    ap.add_argument("--burnin", type=int, default=100)
    ap.add_argument("--seed", type=int, default=20261018)
    ap.add_argument("--ess-steps", type=int, default=5000)
    ap.add_argument("--ess-burnin", type=int, default=100)
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-ess", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the brief timing of the other BASELINE.json configs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the chain state they computed "
                    "(theta, log-posterior, accept counts, Welford moments) as DIR/<name>.npy, float64, at most 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm (the CPU arm sizes its sample from the measured rate)")
    if args.warmup < 3:
        args.warmup = 3 if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
