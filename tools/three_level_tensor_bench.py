"""MLDA with two surrogates on the FP64 tensor path (linear_dmma_kernel.cu, three levels) on the GPU.

    python tools/three_level_tensor_bench.py [--out profiles] [--ab PARENT_LIB] [--rounds 3]

writes three_level_tensor.json and three_level_tensor.md to --out.

1. Rates at 65,536 chains (AcceptanceRateDiagnostics, as the builders default to), device events around 1,000
   transitions after 20 of warm-up: chain-steps/s; algorithmic TFLOP/s = 2 d rows per evaluation that the coarse / mid /
   fine counters report, rows = data_dim of the level evaluated; the fraction of the FP64 tensor peak
   (yg_fp64_tensor_peak) measured in the same run.  Shapes: three-level 64 x 256 and 32 x 96 (J = 3,
   bench_problems.big_linear_three_level_problem), each with its two-level equivalent in the same process: the same
   problem without the middle level (the sub-chain on level 0, the screen on the target).
2. --ab: the single- and two-level 64 x 256 workloads (bench_problems.big_linear_problem, J = 3) with this tree's
   library and with PARENT_LIB (a build of the parent commit), alternating, one process per round and library.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench_problems as bp                                                      # noqa: E402

NC, WARMUP, STEPS = 65536, 20, 1000

SHAPES = [
    # name, d, data_dims, levels kept
    ("three_64x256_J3", 64, (256, 256, 256), (0, 1, 2)),
    ("two_64x256_J3", 64, (256, 256, 256), (0, 2)),
    ("three_32x96_J3", 32, (96, 96, 96), (0, 1, 2)),
    ("two_32x96_J3", 32, (96, 96, 96), (0, 2)),
]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "sm_clock_max": clock}


def keep_levels(meta, arrays, keep):
    """The problem restricted to the levels `keep` (renumbered from 0)."""
    out = {"prop_L": arrays["prop_L"]}
    for new, old in enumerate(keep):
        out.update({f"L{new}_{k[3:]}": v for k, v in arrays.items() if k.startswith(f"L{old}_")})
    return dict(meta, levels=len(keep), J=meta["J"] if len(keep) > 1 else 1), out


def timed(meta, arrays, start):
    """(seconds, counter deltas, launch) of STEPS transitions after WARMUP."""
    from yagre_mcmc_b200.ensemble import ChainEnsemble, LoweredProblem
    ens = ChainEnsemble(LoweredProblem(meta, arrays), NC, seed=5, welford=False)
    ens.set_state(np.tile(start, (NC, 1)))
    ens.run(WARMUP, samples=False)
    torch.cuda.synchronize()
    c0 = ens.counters()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ens.run(STEPS, samples=False)
    e1.record()
    e1.synchronize()
    s = e0.elapsed_time(e1) * 1e-3
    c1 = ens.counters()
    ev = {k: c1[k] - c0[k] for k in ("transitions", "accepted", "coarse_evals", "mid_evals", "fine_evals",
                                     "coarse_accepted")}
    launch = ens.last_launch()
    ens.close()
    torch.cuda.empty_cache()
    return s, ev, launch


def rate(name, d, dims, keep, tpeak):
    meta, arrays = bp.big_linear_three_level_problem(d, dims, 1, J=3)
    mean, _ = bp.linear_gaussian_posterior(arrays, 2)              # start every chain at the target's mean
    meta, arrays = keep_levels(meta, arrays, keep)
    s, ev, launch = timed(meta, arrays, mean)
    rows = [dims[l] for l in keep]
    by_level = [ev["coarse_evals"], ev["mid_evals"], ev["fine_evals"]] if len(keep) == 3 else \
        [ev["coarse_evals"], ev["fine_evals"]]
    flop = sum(bp.big_linear_flops_per_eval(d, r) * n for r, n in zip(rows, by_level))
    out = dict(name=name, d=d, data_dims=rows, levels=len(keep), J=meta["J"], chains=NC, steps=STEPS, seconds=s,
               counters=ev, launch=launch, chain_steps_per_s=ev["transitions"] / s, tflops=flop / s / 1e12,
               frac_of_fp64_peak=flop / s / 1e12 / tpeak, accept_rate=ev["accepted"] / ev["transitions"])
    print(json.dumps(out), flush=True)
    return out


def ab_child():
    """One round of the A/B comparison in this process (the library of YAGRE_B200_LIB)."""
    res = {}
    for name, two in (("single_64x256", False), ("two_64x256_J3", True)):
        meta, arrays = bp.big_linear_problem(64, 256, 1, two_level=two, J=3)
        mean, _ = bp.linear_gaussian_posterior(arrays, meta["levels"] - 1)
        s, ev, launch = timed(meta, arrays, mean)
        res[name] = dict(chain_steps_per_s=ev["transitions"] / s, counters=ev, launch=launch)
    print("AB " + json.dumps(res), flush=True)


def ab(parent_lib, rounds):
    libs = {"this": os.path.join(ROOT, "yagre_mcmc_b200", "libyagre_b200.so"), "parent": os.path.abspath(parent_lib)}
    runs = []
    for r in range(rounds):
        for tag in (("this", "parent") if r % 2 == 0 else ("parent", "this")):
            env = dict(os.environ, YAGRE_B200_LIB=libs[tag])
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--ab-child"], env=env, capture_output=True,
                               text=True, check=True)
            line = [ln for ln in p.stdout.splitlines() if ln.startswith("AB ")][-1]
            runs.append(dict(round=r, lib=tag, **json.loads(line[3:])))
            print(json.dumps(runs[-1]), flush=True)
    summary = {}
    for w in ("single_64x256", "two_64x256_J3"):
        v = {tag: [x[w]["chain_steps_per_s"] for x in runs if x["lib"] == tag] for tag in libs}
        same = all(x[w]["counters"] == runs[0][w]["counters"] for x in runs)
        summary[w] = dict(this=v["this"], parent=v["parent"], counters_identical=same,
                          ratio_of_medians=float(np.median(v["this"]) / np.median(v["parent"])))
    return dict(runs=runs, summary=summary)


def write_md(path, res):
    g = res["gpu"]
    lines = ["# MLDA with two surrogates on the FP64 tensor path", "",
             f"Measured on {g['name']} at a power limit of {g['power_limit']} (max SM clock {g['sm_clock_max']}); "
             f"FP64 tensor peak measured in the same run: {res['fp64_tensor_peak_tflops']:.1f} TFLOP/s.  "
             f"{NC} chains, AcceptanceRateDiagnostics, CUDA events around {STEPS} transitions after {WARMUP} of "
             "warm-up.  TFLOP/s counts 2 d rows per evaluation the coarse / mid / fine counters report.  Produced by "
             "tools/three_level_tensor_bench.py.", "",
             "| shape | levels | warps | smem (B) | chain-steps/s | TFLOP/s | of FP64 peak | accept | coarse / mid / fine evals per transition |",
             "|---|---|---|---|---|---|---|---|---|"]
    for r in res["rates"]:
        c, t = r["counters"], r["counters"]["transitions"]
        lines.append(f"| {r['name']} | {r['levels']} | {r['launch']['block'] // 32} | {r['launch']['smem']} | "
                     f"{r['chain_steps_per_s']:.3e} | {r['tflops']:.2f} | {r['frac_of_fp64_peak']:.2f} | "
                     f"{r['accept_rate']:.2f} | {c['coarse_evals'] / t:.2f} / {c['mid_evals'] / t:.2f} / "
                     f"{c['fine_evals'] / t:.2f} |")
    if "ab" in res:
        lines += ["", "## One- and two-level 64 x 256: this tree against the parent commit", "",
                  "Alternating processes, one per round and library; chain-steps/s.", "",
                  "| workload | this tree | parent | ratio of medians | counters identical |", "|---|---|---|---|---|"]
        for w, s in res["ab"]["summary"].items():
            lines.append(f"| {w} | {', '.join(f'{x:.4e}' for x in s['this'])} | "
                         f"{', '.join(f'{x:.4e}' for x in s['parent'])} | {s['ratio_of_medians']:.4f} | "
                         f"{s['counters_identical']} |")
    open(path, "w").write("\n".join(lines) + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--ab", default=None, help="library of the parent commit for the A/B comparison")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--ab-child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    if args.ab_child:
        return ab_child()
    from yagre_mcmc_b200.ensemble import fp64_tensor_peak_tflops
    res = dict(gpu=gpu_info(), fp64_tensor_peak_tflops=fp64_tensor_peak_tflops(0, 50.0))
    res["rates"] = [rate(*s, res["fp64_tensor_peak_tflops"]) for s in SHAPES]
    if args.ab:
        res["ab"] = ab(args.ab, args.rounds)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "three_level_tensor.json"), "w") as f:
        json.dump(res, f, indent=1)
    write_md(os.path.join(args.out, "three_level_tensor.md"), res)


if __name__ == "__main__":
    main()
