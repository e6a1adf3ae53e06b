"""Pooled statistics from stored samples (yg_pooled_samples) on the GPU: kernel time against torch, and the effect of
the pooled dense proposal factor on the tensor-path linear models.

    python tools/pooled_samples_bench.py [--out profiles]

writes pooled_samples.json and pooled_samples.md to --out.

1. Kernel time, CUDA events around back-to-back calls after warm-up, 65,536 chains, d in {8, 16, 32, 64}, n_samples in
   {1, 40, 300}.  Every call reads a different copy of the buffer, with at least 512 MB of copies, so no call finds its
   input in the 126 MB L2.  Bytes: one read of the buffer; flop: the symmetric product, d (d + 1) per sample vector
   (the kernel's DMMA tiles issue 20 / 32 of the full 2 d^2 at d = 64).  The least time is the larger of bytes over
   7.7 TB/s (HBM3e, data sheet) and flop over the FP64 tensor peak measured in the same run.  The same statistics with
   torch (per-chain mean, centred copy, matmul) are timed on the same inputs.
2. Sampling, 64 x 256 single level and 32 x 96 two-level (J = 3), isotropic factor of bench_problems against the pooled
   dense factor: chain-steps/s at 65,536 chains (50 transitions, AcceptanceRateDiagnostics as the builders default to),
   and from 4,096 chains started at the posterior mean: burn-in, pooling over a thinned burn-in trajectory, then an
   unthinned series whose per-chain IAT_max (yg_iat_ess) gives the ESS; ESS/s charges burn-in, pooling and production.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench_problems as bp                                                      # noqa: E402
from yagre_mcmc_b200 import _lib                                                 # noqa: E402
from yagre_mcmc_b200.ensemble import (ChainEnsemble, LoweredProblem, fp64_tensor_peak_tflops, iat_ess,  # noqa: E402
                                      pooled_sample_stats)
from yagre_mcmc_b200.parallel import moments_from_stats, proposal_factor_from_covariance   # noqa: E402

HBM_TBS = 7.7
L2_ROTATE_BYTES = 512 << 20


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "sm_clock_max": clock}


def events_ms(fn, reps):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        fn(i)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def torch_stats(x):
    ns, d, nc = x.shape
    m = x.mean(dim=0)                                                            # [d, nc]
    y = x - m                                                                    # centred copy
    Y = y.permute(1, 0, 2).reshape(d, ns * nc)
    m2 = Y @ Y.T
    var = (y * y).sum(dim=0).sum(dim=1) / (ns - 1) if ns > 1 else torch.zeros(d, dtype=x.dtype, device=x.device)
    return torch.cat([torch.tensor([nc, ns, 0.0], dtype=x.dtype, device=x.device), m.sum(dim=1), (m @ m.T).reshape(-1),
                      m2.reshape(-1), var])


def block_rel_diff(a, b, d):
    """max |a - b| / max |b| over each block of the vector, worst block."""
    worst, o = 0.0, 3
    for n in (d, d * d, d * d, d):
        ref = np.abs(b[o:o + n]).max()
        if ref > 0:
            worst = max(worst, float(np.abs(a[o:o + n] - b[o:o + n]).max() / ref))
        o += n
    return worst


def kernel_times(tpeak):
    import ctypes as C
    lib = _lib.load()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rows = []
    nc = 65536
    for d in (8, 16, 32, 64):
        for ns in (1, 40, 300):
            size = ns * d * nc * 8
            copies = max(1, -(-L2_ROTATE_BYTES // size))
            g = torch.Generator(device="cuda").manual_seed(d * 1000 + ns)
            bufs = [torch.randn(ns, d, nc, dtype=torch.float64, device="cuda", generator=g) + 3.0
                    for _ in range(copies)]
            ws = torch.empty(int(lib.yg_pooled_samples_workspace_len(d, nc)), dtype=torch.float64, device="cuda")
            out = torch.empty(int(lib.yg_pooled_len(d)), dtype=torch.float64, device="cuda")

            def call(i):
                _lib.check(lib.yg_pooled_samples(C.c_void_p(bufs[i % copies].data_ptr()), ns, d, nc,
                                                 C.c_void_p(ws.data_ptr()), ws.numel(), C.c_void_p(out.data_ptr()), st))
            reps = max(10, min(200, int(2e10 / max(size, 1))), copies)
            events_ms(call, max(3, copies))                                      # warm-up
            ms = events_ms(call, reps)
            v = pooled_sample_stats(bufs[0]).cpu().numpy()
            tv = torch_stats(bufs[0])
            torch_reps = max(3, min(20, reps // 4))
            events_ms(lambda i: torch_stats(bufs[i % copies]), 2)
            tms = events_ms(lambda i: torch_stats(bufs[i % copies]), torch_reps)
            flop = d * (d + 1) * ns * nc
            t_hbm, t_fp = size / (HBM_TBS * 1e12) * 1e3, flop / (tpeak * 1e12) * 1e3
            rows.append(dict(d=d, n_samples=ns, n_chains=nc, buffer_bytes=size, copies_rotated=copies, reps=reps,
                             kernel_ms=ms, torch_ms=tms, speedup_vs_torch=tms / ms,
                             hbm_tb_per_s=size / (ms * 1e-3) / 1e12, fp64_tflops=flop / (ms * 1e-3) / 1e12,
                             bound="HBM" if t_hbm >= t_fp else "FP64", least_time_ms=max(t_hbm, t_fp),
                             frac_of_bound=max(t_hbm, t_fp) / ms,
                             max_block_rel_diff_vs_torch=block_rel_diff(v, tv.cpu().numpy(), d)))
            print(json.dumps(rows[-1]), flush=True)
            del bufs, tv
            torch.cuda.empty_cache()
    return rows


def rate(meta, arrays, L, mean):
    a = dict(arrays)
    if L is not None:
        a["prop_L"] = L
    ens = ChainEnsemble(LoweredProblem(meta, a), 65536, seed=5, welford=False)
    ens.set_state(np.tile(mean, (65536, 1)))
    ens.run(10, samples=False)
    torch.cuda.synchronize()
    c0 = ens.counters()
    t0 = time.perf_counter()
    ens.run(50, samples=False)
    torch.cuda.synchronize()
    t = time.perf_counter() - t0
    c1 = ens.counters()
    out = dict(chain_steps_per_s=(c1["transitions"] - c0["transitions"]) / t,
               accept_rate=(c1["accepted"] - c0["accepted"]) / (c1["transitions"] - c0["transitions"]),
               launch=ens.last_launch())
    ens.close()
    return out


def ess_run(meta, arrays, mean, pool, burn, thin_burn, prod):
    """4,096 chains from the posterior mean: burn-in (stored thinned when pooling), optional pooling, production."""
    nc = 4096
    ens = ChainEnsemble(LoweredProblem(meta, arrays), nc, seed=9, welford=False)
    ens.set_state(np.tile(mean, (nc, 1)))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    burn_s = ens.run(burn, thin=thin_burn, samples=pool)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    L = None
    if pool:
        v = pooled_sample_stats(burn_s["samples"])
        cov = moments_from_stats(v, meta["dim"])["covariance"]
        L = proposal_factor_from_covariance(cov)
        ens.rebuild_proposal_factor(L)
        ens.set_state(ens.state()["theta"].t().contiguous())
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    c0 = ens.counters()
    s = ens.run(prod, samples=True)["samples"]
    torch.cuda.synchronize()
    t3 = time.perf_counter()
    c1 = ens.counters()
    iat, ess = iat_ess(s, "max")
    iat, ess = iat.cpu().numpy(), ess.cpu().numpy()
    res = dict(burn_in=burn, production=prod, chains=nc, burn_s=t1 - t0, pool_s=t2 - t1, prod_s=t3 - t2,
               accept_rate=(c1["accepted"] - c0["accepted"]) / (c1["transitions"] - c0["transitions"]),
               iat_max_median=float(np.median(iat)), iat_max_p90=float(np.percentile(iat, 90)),
               window_closed_fraction=float((5 * iat < prod).mean()), ess_total=int(ess.sum()),
               ess_per_s=float(ess.sum() / (t3 - t0)), launch=ens.last_launch())
    ens.close()
    del s
    torch.cuda.empty_cache()
    return res, L


def sampling():
    out = {}
    for d, dd, two, J, key in ((64, 256, False, 1, "linear_d64_x256"), (32, 96, True, 3, "linear_d32_x96_two_level")):
        meta, arrays = bp.big_linear_problem(d, dd, 1, two_level=two, J=J)
        mean, cov = bp.linear_gaussian_posterior(arrays, meta["levels"] - 1)
        iso_ess, _ = ess_run(meta, arrays, mean, False, 2000, 1, 10000)
        dense_ess, L = ess_run(meta, arrays, mean, True, 2000, 10, 10000)
        out[key] = dict(posterior_condition_number=float(np.linalg.cond(cov)),
                        isotropic=dict(rate_65536=rate(meta, arrays, None, mean), ess_4096=iso_ess),
                        pooled_dense=dict(rate_65536=rate(meta, arrays, L, mean), ess_4096=dense_ess))
        out[key]["ess_per_s_ratio"] = dense_ess["ess_per_s"] / iso_ess["ess_per_s"]
        print(key, json.dumps(out[key]), flush=True)
    return out


def markdown(res):
    g = res["gpu"]
    lines = [f"# Pooled statistics from stored samples (yg_pooled_samples)", "",
             f"Measured on {g['name']}, power limit {g['power_limit']}, max SM clock {g['sm_clock_max']}; "
             f"FP64 tensor peak measured in the same run: {res['fp64_tensor_peak_tflops']:.1f} TFLOP/s; HBM bound: "
             f"{HBM_TBS} TB/s (data sheet, not measured).  Produced by tools/pooled_samples_bench.py.", "",
             "## Kernel time, 65,536 chains (buffers rotated past L2)", "",
             "| d | samples | MB | kernel ms | TB/s | TFLOP/s | bound | of bound | torch ms | speed-up | max rel diff |",
             "|---|---|---|---|---|---|---|---|---|---|---|"]
    for r in res["kernel"]:
        lines.append(f"| {r['d']} | {r['n_samples']} | {r['buffer_bytes'] / 1e6:.0f} | {r['kernel_ms']:.3f} | "
                     f"{r['hbm_tb_per_s']:.2f} | {r['fp64_tflops']:.2f} | {r['bound']} | {r['frac_of_bound']:.2f} | "
                     f"{r['torch_ms']:.3f} | {r['speedup_vs_torch']:.1f} | {r['max_block_rel_diff_vs_torch']:.1e} |")
    lines += ["", "## Sampling: isotropic factor against the pooled dense factor", "",
              "| model | factor | chain-steps/s (65,536) | block | accept | IAT_max median (4,096) | ESS/s |",
              "|---|---|---|---|---|---|---|"]
    for key, v in res["sampling"].items():
        for f in ("isotropic", "pooled_dense"):
            r, e = v[f]["rate_65536"], v[f]["ess_4096"]
            lines.append(f"| {key} | {f} | {r['chain_steps_per_s']:.3g} | {r['launch']['block']} | {e['accept_rate']:.3f} | "
                         f"{e['iat_max_median']:.0f} | {e['ess_per_s']:.3g} |")
        lines.append(f"| {key} | ESS/s ratio | | | | | {v['ess_per_s_ratio']:.2f} |")
    return "\n".join(lines) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU")
    res = dict(gpu=gpu_info(), fp64_tensor_peak_tflops=fp64_tensor_peak_tflops(0, 20.0), hbm_tb_per_s_datasheet=HBM_TBS)
    res["kernel"] = kernel_times(res["fp64_tensor_peak_tflops"])
    res["sampling"] = sampling()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "pooled_samples.json"), "w") as f:
        json.dump(res, f, indent=1)
    with open(os.path.join(args.out, "pooled_samples.md"), "w") as f:
        f.write(markdown(res))


if __name__ == "__main__":
    main()
