"""The tensor path with operands streamed from L2 (smem_plan.h: big_tensor_plan) on the GPU.

    python tools/streamed_operand_bench.py [--out profiles] [--sweep LIB ...]

writes streamed_operand.json and streamed_operand.md to --out.

1. Rates at 65,536 chains (AcceptanceRateDiagnostics, as the builders default to), device events around 1,000
   transitions after 20 of warm-up: chain-steps/s; algorithmic TFLOP/s = 2 d rows per evaluation the counters report
   (coarse and fine), rows = data_dim (+ d for a dense prior); the fraction of the FP64 tensor peak measured in the same
   run.
2. L2 read bandwidth: tools/probe_l2_read.cu, compiled into a temporary directory (every SM reads one 128-KiB buffer).
3. The streamed evaluations' least time against the launch time: their flop over the FP64 peak, and their A-operand
   bytes (0.5 B per flop: one 8-byte element serves 8 chains x 2 flop) over the measured L2 bandwidth.
4. Prefetch depth: --sweep takes dev builds of the library (make -C yagre_mcmc_b200/csrc stream_depth DEPTH=n: level
   1's G of every two-level problem streamed, YG_STREAM_DEPTH = n) and measures two-level 64 x 256 and 64 x 128 with
   each, in a process of its own.  64 x 128 fits shared memory with 12 warps, so against the default build it compares
   the streamed instance with the resident one at the same warps: what L2 latency, the larger step loop and the spills
   cost, if anything.
5. ptxas registers / spills and SASS size of the KQ = 16 instances (linear_dmma_kernel.cu compiled into a temporary
   directory with the library's flags).
6. ESS/s of two-level 64 x 256 at 4,096 chains, isotropic factor against the pooled dense factor
   (tools/pooled_samples_bench.py's ess_run: burn-in, pooling over the thinned burn-in, 10,000 unthinned steps).
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench_problems as bp                                                      # noqa: E402
from yagre_mcmc_b200.ensemble import ChainEnsemble, LoweredProblem, fp64_tensor_peak_tflops   # noqa: E402

NC, WARMUP, STEPS = 65536, 20, 1000

SHAPES = [
    # name, d, data_dim, two level, dense factor, dense prior, operands streamed
    ("two_64x256_J3", 64, 256, True, False, False, "G1"),
    ("two_64x256_J3_pooled_dense_factor", 64, 256, True, True, False, "G1"),
    ("two_64x176_J3", 64, 176, True, False, False, "none (largest resident)"),
    ("two_64x128_J3", 64, 128, True, False, False, "none"),
    ("two_64x192_J3", 64, 192, True, False, False, "G1"),
    ("single_64x256_dense_prior_dense_factor", 64, 256, False, True, True, "Ld"),
]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "sm_clock_max": clock}


def problem(d, dd, two, dense_L, dense_prior):
    meta, arrays = bp.big_linear_problem(d, dd, 1, two_level=two, J=3)
    arrays = dict(arrays)
    mean, cov = bp.linear_gaussian_posterior(arrays, meta["levels"] - 1)
    if dense_prior:
        A = np.random.default_rng(5).standard_normal((d, d))
        pc = 2.0 * (A @ A.T / d + 0.5 * np.eye(d))
        prec = np.linalg.inv(pc)
        for l in range(meta["levels"]):
            arrays[f"L{l}_prior_prec"] = 0.5 * (prec + prec.T)
        mean, cov = bp.linear_gaussian_posterior(arrays, meta["levels"] - 1)
    if dense_L:                                                # the pooled factor: 2.4^2 / d of the posterior covariance
        arrays["prop_L"] = np.linalg.cholesky(2.4 ** 2 / d * cov)
    return meta, arrays, mean


def rate(name, d, dd, two, dense_L, dense_prior, streamed, tpeak, l2_tbs=None):
    meta, arrays, mean = problem(d, dd, two, dense_L, dense_prior)
    rows = dd + (d if dense_prior else 0)
    ens = ChainEnsemble(LoweredProblem(meta, arrays), NC, seed=5, welford=False)
    ens.set_state(np.tile(mean, (NC, 1)))
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
    ev = {k: c1[k] - c0[k] for k in ("transitions", "accepted", "coarse_evals", "fine_evals", "coarse_accepted")}
    fpe = bp.big_linear_flops_per_eval(d, rows)
    flop = fpe * (ev["coarse_evals"] + ev["fine_evals"])
    # the streamed evaluations: level 1's G once per counted fine evaluation; the dense factor J times per transition
    # (d (d + 1) flop of the triangle per proposal and chain)
    s_flop = 0.0
    if "G1" in streamed:
        s_flop += fpe * ev["fine_evals"]
    if "Ld" in streamed:
        s_flop += d * (d + 1) * ev["transitions"] * meta["J"]
    t_fp, t_l2 = s_flop / (tpeak * 1e12), 0.5 * s_flop / (l2_tbs * 1e12) if l2_tbs else 0.0
    out = dict(name=name, d=d, data_dim=dd, rows=rows, levels=meta["levels"], J=meta["J"], dense_factor=dense_L,
               dense_prior=dense_prior, streamed=streamed, chains=NC, steps=STEPS, seconds=s, counters=ev,
               launch=ens.last_launch(), chain_steps_per_s=ev["transitions"] / s, tflops=flop / s / 1e12,
               frac_of_fp64_peak=flop / s / 1e12 / tpeak, streamed_flop=s_flop,
               streamed_fp64_bound_frac=t_fp / s, streamed_l2_bound_frac=t_l2 / s)
    ens.close()
    torch.cuda.empty_cache()
    print(json.dumps(out), flush=True)
    return out


def l2_probe():
    nvcc = shutil.which("nvcc") or os.path.join(os.environ.get("CUDA_HOME") or "/usr/local/cuda", "bin", "nvcc")
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "probe_l2_read")
        subprocess.run([nvcc, "-O3", "-gencode", "arch=compute_100a,code=sm_100a",
                        os.path.join(ROOT, "tools", "probe_l2_read.cu"), "-o", exe], check=True)
        return json.loads(subprocess.run([exe], capture_output=True, text=True, check=True).stdout)


def compile_report():
    """ptxas -v and SASS of linear_dmma_kernel.cu with the library's flags: per KQ = 16 instance registers, spill bytes,
    SASS instructions, local loads / stores and DMMAs."""
    import re
    nvcc = shutil.which("nvcc") or os.path.join(os.environ.get("CUDA_HOME") or "/usr/local/cuda", "bin", "nvcc")
    src = os.path.join(ROOT, "yagre_mcmc_b200", "csrc", "linear_dmma_kernel.cu")
    with tempfile.TemporaryDirectory() as tmp:
        obj = os.path.join(tmp, "k.o")
        log = subprocess.run([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xptxas", "-v",
                              "-c", src, "-o", obj], capture_output=True, text=True, check=True).stderr
        sass = subprocess.run([os.path.join(os.path.dirname(nvcc), "cuobjdump"), "-sass", obj],
                              capture_output=True, text=True, check=True).stdout
    out, cur = {}, None
    for line in log.splitlines():
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            cur = m.group(1) if "linear_dmma_mh_kernelILi16E" in m.group(1) else None
            if cur:
                out[cur] = {}
        elif cur and "spill stores" in line:
            out[cur]["spill_store_bytes"], out[cur]["spill_load_bytes"] = map(int, re.findall(r"(\d+) bytes spill", line))
        elif cur and "Used" in line and "registers" in line:
            out[cur]["registers"] = int(re.search(r"Used (\d+) registers", line).group(1))
    cur = None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1) if m.group(1) in out else None
            if cur:
                out[cur].update(sass_instructions=0, ldl=0, stl=0, dmma=0)
            continue
        if cur and re.search(r"/\*[0-9a-f]{4,}\*/\s+\S", line):
            o = out[cur]
            o["sass_instructions"] += 1
            o["ldl"] += " LDL" in line
            o["stl"] += " STL" in line
            o["dmma"] += " DMMA" in line

    def name(k):
        t, f, st = re.search(r"ILi16ELb(\d)ELb(\d)ELb(\d)E", k).groups()
        return f"<16, two={t == '1'}, free_noise={f == '1'}, streamed={st == '1'}>"
    return {name(k): v for k, v in sorted(out.items())}


def sweep(libs):
    """Each library in a process of its own: the rates of two-level 64 x 256 and 64 x 128."""
    rows = []
    for lib in libs:
        env = dict(os.environ, YAGRE_B200_LIB=os.path.abspath(lib))
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--only", "two_64x256_J3,two_64x128_J3"],
                           env=env, capture_output=True, text=True, check=True)
        for line in r.stdout.splitlines():
            if line.startswith("{"):
                row = json.loads(line)
                row["library"] = os.path.basename(lib)
                rows.append(row)
    return rows


def ess_compare():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from pooled_samples_bench import ess_run
    meta, arrays = bp.big_linear_problem(64, 256, 1, two_level=True, J=3)
    mean, _ = bp.linear_gaussian_posterior(arrays, 1)
    iso, _ = ess_run(meta, arrays, mean, False, 2000, 1, 10000)
    dense, _ = ess_run(meta, arrays, mean, True, 2000, 10, 10000)
    return dict(isotropic=iso, pooled_dense=dense, ess_per_s_ratio=dense["ess_per_s"] / iso["ess_per_s"])


def markdown(res):
    g = res["gpu"]
    lines = ["# Tensor path with operands streamed from L2", "",
             f"Measured on {g['name']}, power limit {g['power_limit']}, max SM clock {g['sm_clock_max']}; FP64 tensor "
             f"peak measured in the same run: {res['fp64_tensor_peak_tflops']:.1f} TFLOP/s; L2 read bandwidth "
             f"(tools/probe_l2_read.cu, 128 KiB read by every SM): {res['l2']['tb_per_s']:.2f} TB/s.  "
             f"{NC:,} chains, {STEPS} transitions after {WARMUP} of warm-up, device events; AcceptanceRateDiagnostics.  "
             "Produced by tools/streamed_operand_bench.py.", "",
             "## Rates", "",
             "| shape | streamed | block | smem B | chain-steps/s | TFLOP/s | of FP64 peak | coarse / fine evals | "
             "streamed: FP64 bound | streamed: L2 bound |",
             "|---|---|---|---|---|---|---|---|---|---|"]
    for r in res["rates"]:
        c = r["counters"]
        lines.append(f"| {r['name']} | {r['streamed']} | {r['launch']['block']} | {r['launch']['smem']} | "
                     f"{r['chain_steps_per_s']:.3g} | {r['tflops']:.2f} | {r['frac_of_fp64_peak']:.2f} | "
                     f"{c['coarse_evals']:,} / {c['fine_evals']:,} | {r['streamed_fp64_bound_frac']:.3f} | "
                     f"{r['streamed_l2_bound_frac']:.3f} |")
    lines += ["", "TFLOP/s: 2 d rows per counted evaluation over the launch time.  The last two columns: the least time "
              "of the streamed evaluations (flop over the FP64 peak; A-operand bytes, 0.5 B per flop, over the L2 "
              "bandwidth) as a fraction of the launch time.", "",
              "## Prefetch depth (dev builds that stream level 1's G of every two-level problem)", "",
              "| library | shape | block | smem B | chain-steps/s | TFLOP/s |", "|---|---|---|---|---|---|"]
    for r in res["sweep"]:
        lines.append(f"| {r['library']} | {r['name']} | {r['launch']['block']} | {r['launch']['smem']} | "
                     f"{r['chain_steps_per_s']:.4g} | {r['tflops']:.2f} |")
    lines += ["", "## Registers, spills and SASS of the KQ = 16 instances (this build, default depth)", "",
              "| instance | registers | spill stores / loads B | SASS instructions | STL / LDL | DMMA |",
              "|---|---|---|---|---|---|"]
    for k, v in res["compile"].items():
        lines.append(f"| {k} | {v['registers']} | {v['spill_store_bytes']} / {v['spill_load_bytes']} | "
                     f"{v['sass_instructions']} | {v['stl']} / {v['ldl']} | {v['dmma']} |")
    e = res.get("ess")
    lines += ["", "## ESS/s, two-level 64 x 256, J = 3, 4,096 chains", ""]
    if e:
        lines += ["| factor | block | accept | IAT_max median | ESS/s |", "|---|---|---|---|---|"]
        for f in ("isotropic", "pooled_dense"):
            r = e[f]
            lines.append(f"| {f} | {r['launch']['block']} | {r['accept_rate']:.3f} | {r['iat_max_median']:.0f} | "
                         f"{r['ess_per_s']:.3g} |")
        lines.append(f"| ratio | | | | {e['ess_per_s_ratio']:.2f} |")
    else:
        lines.append("Not measured.")
    return "\n".join(lines) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--sweep", nargs="*", default=[], help="dev builds of the library to compare (see 4. above)")
    ap.add_argument("--only", help="comma-separated shapes: print their rates as JSON lines and write nothing")
    ap.add_argument("--no-ess", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU")
    if args.only:
        tpeak = fp64_tensor_peak_tflops(0, 5.0)
        for s in SHAPES:
            if s[0] in args.only.split(","):
                rate(*s, tpeak)
        return
    res = dict(gpu=gpu_info(), fp64_tensor_peak_tflops=fp64_tensor_peak_tflops(0, 20.0))
    res["l2"] = l2_probe()
    print(json.dumps(res), flush=True)
    res["rates"] = [rate(*s, res["fp64_tensor_peak_tflops"], res["l2"]["tb_per_s"]) for s in SHAPES]
    res["sweep"] = sweep(args.sweep)
    res["compile"] = compile_report()
    print(json.dumps(res["compile"]), flush=True)
    res["ess"] = None if args.no_ess else ess_compare()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "streamed_operand.json"), "w") as f:
        json.dump(res, f, indent=1)
    with open(os.path.join(args.out, "streamed_operand.md"), "w") as f:
        f.write(markdown(res))


if __name__ == "__main__":
    main()
