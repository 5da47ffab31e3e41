#!/usr/bin/env python
"""Task-5 part-2 pilot-density study (`Task 5/Task5_part2.m:46-321`): ``part2.sweep_lib`` (one ``ofdm_sweep_part2`` call)
against the composed driver ``part2.sweep`` on the same arguments, alternated in one process; a check that both give
identical per-run NMSE arrays, NMSE and BER; a per-stage split of both from torch.profiler; and the bytes and flops of the
two new kernels from the shapes.  Prints one JSON line per workload.

    python tools/bench_part2_sweep.py [--runs 100,4096] [--profiles EPA,ETU] [--precision f32] [--reps 2]

Workloads: the script's 57 combs (`:13-17`) x 100 runs (its monteCarloRuns) and x 4,096 runs, SNR 20 dB, 16QAM, Nfft 4096,
N_carrier 1024, FP32.  Times are host clocks around calls that end in a device synchronise, after one warm-up of each path."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import ofdm_b200 as G  # noqa: E402
from ofdm_b200 import part2  # noqa: E402
from bench_mse_sweep import card  # noqa: E402

NFFT, NC, S, TG, SNR, FS = 4096, 1024, 14, 512, 20.0, 4e7


def kernel_ms(fn):
    """Device time per kernel name (ms) of one call of fn, from torch.profiler, and the number of kernel launches."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out, n = {}, 0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0.0)
        if t > 0:
            key = e.key.split("(")[0].split("<")[0][:48]
            out[key] = round(out.get(key, 0.0) + t / 1e3, 3)
            n += e.count
    return dict(sorted(out.items(), key=lambda kv: -kv[1])[:14]), n


def shapes(ctx, combs, runs, profile, seed):
    """Bytes and flops of part2_front_end_kernel + part2_decide_kernel over the whole call, from the shapes.  The FIR runs the
    NON-ZERO taps only (nnz per run, counted on the runs' own impulse responses: at 40 MHz a path whose delay is a whole
    number of samples gives a single non-zero tap through the windowed sinc).  Complex MAC = 8 flops, radix-4 FFT ~
    5 N log2 N, per data carrier and estimator a complex division (~11) and 16 squared distances (~64).  HBM bytes: the
    estimates read (4 x N_carrier/Nfft complex per symbol, the decide kernel's only large input), the impulse responses and
    y; the noisy stream (516 KB per point) is L2-resident.  Returns (flops, of them FIR flops, bytes, mean nnz, h_len)."""
    _, D, _ = ctx.tdl_info(profile, FS)
    off, _, _ = part2.lib_layout(combs)
    esz = 16 if ctx.f64 else 8
    flops = byts = fir_flops = 0
    nnz_all = []
    for k in range(len(combs)):
        h = ctx.tdl_channel(profile, FS, runs, seed=seed, first_stream_id=k * 1_000_003)
        nnz = (h != 0).sum(dim=1).double()
        nnz_all.append(nnz)
        Np = int(off[k + 1] - off[k])
        Nd = NC - Np
        fir = float(nnz.sum()) * NFFT * 8
        fft = 5 * NFFT * 12
        fir_flops += (1 + S) * fir
        flops += (1 + S) * fir + runs * ((1 + S) * fft + S * 4 * Nd * 75)
        byts += runs * esz * (D * (1 + S) + Np + S * Nd * 4)
    return flops, fir_flops, byts, float(torch.cat(nnz_all).mean()), D


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", default="100,4096")
    ap.add_argument("--profiles", default="EPA,ETU")
    ap.add_argument("--precision", default="f32", choices=["f32", "f64"])
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--seed", type=int, default=1)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_part2_sweep: no CUDA device (the library has no CPU path)")
    ctx = G.Context(0, a.precision)
    name, power = card()
    combs, _ = part2.part2_combs()
    bits = np.random.default_rng(a.seed).integers(0, 2, S * NC * 4).astype(np.uint8)
    for profile in a.profiles.split(","):
        for runs in [int(x) for x in a.runs.split(",")]:
            kw = dict(profile=profile, fs_hz=FS, snr_db=SNR, seed=a.seed)
            captured = {}

            def run_fn(*args, **k):
                out = part2.run_point(*args, **k)
                captured[(k["point_id"], k["first_run"])] = out[0]
                return out

            lib = lambda: part2.sweep_lib(ctx, combs, runs, bits, **kw)                       # noqa: E731
            comp = lambda: part2.sweep(ctx, combs, runs, lambda n: bits[:n], run_fn=run_fn, **kw)   # noqa: E731
            lib(), comp()                                                                     # warm-up of both paths
            t_lib, t_comp = [], []
            for _ in range(a.reps):
                for f, acc in ((lib, t_lib), (comp, t_comp)):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    res = f()
                    torch.cuda.synchronize()
                    acc.append(time.perf_counter() - t0)
                    if f is lib:
                        NMSE, BER, per, counts, _ = res
                    else:
                        N2, B2 = res
            comp_per = np.stack([captured[(k, 0)].T for k in range(len(combs))])
            same = bool(np.array_equal(per, comp_per) and np.array_equal(NMSE, N2) and np.array_equal(BER, B2))
            sub = combs[:: max(1, len(combs) // 4)][:4]                                       # profiled on four points
            lib_k, lib_n = kernel_ms(lambda: part2.sweep_lib(ctx, sub, runs, bits, **kw))
            comp_k, comp_n = kernel_ms(lambda: part2.sweep(ctx, sub, runs, lambda n: bits[:n], **kw))
            fused = sum(v for k, v in lib_k.items() if k.startswith("void part2_") or k.startswith("part2_"))
            flops, fir_flops, byts, nnz, D = shapes(ctx, sub, runs, profile, a.seed)
            print(json.dumps({
                "workload": f"Task5_part2 pilot-density study: {len(combs)} combs x {runs} runs, {profile}, {SNR:g} dB, {a.precision}",
                "gpu": name, "power_limit_and_max_sm_clock": power,
                "lib_seconds": [round(t, 4) for t in t_lib], "composed_seconds": [round(t, 4) for t in t_comp],
                "speedup_median": round(float(np.median(t_comp) / np.median(t_lib)), 2),
                "runs_per_s_lib": round(len(combs) * runs / float(np.median(t_lib)), 1),
                "identical_per_run_nmse_and_ber": same,
                "nmse_mean_over_points": [float(x) for x in NMSE.mean(axis=1)], "ber_mean_over_points": [float(x) for x in BER.mean(axis=1)],
                "profiled_points": [int(c) for c in sub],
                "lib_kernel_ms": lib_k, "lib_kernel_launches": lib_n,
                "composed_kernel_ms": comp_k, "composed_kernel_launches": comp_n,
                "fading_taps_nonzero_mean": round(nnz, 2), "fading_h_len": D,
                "fused_kernels_ms": round(fused, 3), "fused_kernels_gflop": round(flops / 1e9, 2),
                "fused_kernels_fir_gflop": round(fir_flops / 1e9, 2), "fused_kernels_hbm_mb": round(byts / 1e6, 1),
                "fused_kernels_tflops_achieved": round(flops / (fused * 1e-3) / 1e12, 2) if fused else None,
                "fused_kernels_hbm_bound_ms": round(byts / 7.7e12 * 1e3, 4)}))
            sys.stdout.flush()


if __name__ == "__main__":
    main()
