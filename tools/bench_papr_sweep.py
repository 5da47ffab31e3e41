#!/usr/bin/env python
"""Task-2 PAPR study (`Task 2/Main_model_Task_2.m:72-82`) through ``ofdm_sweep_papr``: whole-call time against the same
tiles through the composed exported calls (ofdm_payload_bernoulli -> ofdm_tx_chain_p -> ofdm_window_papr -> binning on the
device with torch.bincount -> ofdm_papr), the two alternated in one process, medians reported; a check that both give the
same histogram (exactly) and per-stream PAPR (within 1e-4 dB in FP32); a torch.profiler kernel split of one call of each
path, taken after the timed runs with the profiler off during them; and the algorithmic bytes: the TX chain writes every
stream once and the statistics read it once (8 B per complex64 sample each way), so the statistics kernel's bytes/s is
that read over its profiled time.  Prints one JSON line per layout.

    python tools/bench_papr_sweep.py [--streams-per-point 8192] [--repeats 5] [--layouts task2,task5]

Layouts, FP32, points (plain, scrambled) x Bernoulli p = 0.05:
  task2: params_task4(percent=1, scale=2.0, alternate=True): Nfft 1024, T_Guard 128, 50 symbols, 79,000-bit streams
         (the Task-2 script's layout, `Task 2/Main_model_Task_2.m:14,58`), L = 57,600 samples;
  task5: params_task5(comb=4): Nfft 4096, T_Guard 512, 14 symbols, L = 64,512 samples."""
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
import ofdm_b200 as G  # noqa: E402
from ofdm_b200 import sweep  # noqa: E402
from oracle import chains as OC  # noqa: E402

HBM_TBPS = 7.7     # one B200, HGX data sheet
LAYOUTS = {"task2": lambda: OC.params_task4(percent=1, scale=2.0, alternate=True), "task5": lambda: OC.params_task5(comb=4)}


def card():
    """Name, power limit and maximum SM clock of the GPU this process runs on, read now."""
    name = torch.cuda.get_device_name()
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "not available"
    return name, out


def link(ctx, p, scramble=True):
    return ctx.link_params(p.Nfft, p.T_Guard, p.N_carrier, p.N_symb, p.Amount_ODFM_SpF, p.Constellation, p.dataCarriers, p.pilotCarriers,
                           p.pilotValues, scramble=scramble)


def composed(ctx, lps, p, points, spp, tile, seed, bin_db, n_bins, hist, papr):
    """The study as exported calls per tile, as a user composes it without ofdm_sweep_papr."""
    for (k, j0, n) in sweep.tiles(len(points), spp, tile):
        scr, pone = points[k]
        bits = ctx.payload_bernoulli(n, p.stream_bits, pone, seed=seed, first_stream_id=j0)
        tx, _ = ctx.tx_chain(lps[scr], bits, n, want_power=True)
        tx = tx.reshape(n, -1)
        w = ctx.window_papr(tx, p.Nfft)
        q = torch.nan_to_num(torch.floor(w.double() / bin_db), nan=0.0).clamp_(0, n_bins - 1).long()
        hist[k] += torch.bincount(q.reshape(-1), minlength=n_bins)
        del w, q
        papr[k, j0:j0 + n] = ctx.papr(tx)


def kernel_ms(fn):
    """Kernel times of one call of fn from torch.profiler, by kernel name."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0.0)
        if t > 0:
            key = e.key.split("(")[0][:70]
            out[key] = round(out.get(key, 0.0) + t / 1e3, 4)
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def run_layout(ctx, name, spp, repeats, seed, bin_db, n_bins):
    p = LAYOUTS[name]()
    lp = link(ctx, p)
    lps = {0: link(ctx, p, scramble=False), 1: lp}
    points = [(0, 0.05), (1, 0.05)]
    tile = min(8192, spp)
    L = p.N_symb * (p.Nfft + p.T_Guard)
    hist_c = torch.zeros((2, n_bins), dtype=torch.int64, device=ctx.device)
    papr_c = torch.zeros((2, spp), dtype=torch.float64, device=ctx.device)
    runs = {
        "ofdm_sweep_papr": lambda: sweep.papr_sweep_local(ctx, lp, points, spp, seed=seed, bin_db=bin_db, n_bins=n_bins),
        "composed exported calls": lambda: composed(ctx, lps, p, points, spp, tile, seed, bin_db, n_bins, hist_c.zero_(), papr_c.zero_()),
    }
    for fn in runs.values():                   # warm-up: modules loaded, pools in place
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in runs}
    for _ in range(repeats):                   # alternated in one process
        for k, fn in runs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            times[k].append(time.perf_counter() - t0)
    med = {k: float(np.median(v)) for k, v in times.items()}

    hist, papr = sweep.papr_sweep_local(ctx, lp, points, spp, seed=seed, bin_db=bin_db, n_bins=n_bins)
    composed(ctx, lps, p, points, spp, tile, seed, bin_db, n_bins, hist_c.zero_(), papr_c.zero_())
    torch.cuda.synchronize()
    hist_equal = bool(torch.equal(hist, hist_c))
    papr_dev = float((papr - papr_c).abs().max())
    counts_ok = bool((hist.sum(dim=1) == spp * (L - p.Nfft + 1)).all())
    ex = sweep.papr_exceedance(hist.cpu().numpy(), bin_db, 0.02)

    split_call = kernel_ms(runs["ofdm_sweep_papr"])
    split_comp = kernel_ms(runs["composed exported calls"])
    streams = 2 * spp
    sig = streams * L * 8                      # complex64 stream bytes: written once by the TX chain, read once by the statistics
    stats_ms = sum(v for k, v in split_call.items() if "papr_stats_kernel" in k)
    stats_gbps = sig / (stats_ms / 1e3) / 1e9 if stats_ms > 0 else None
    return {
        "bench": "papr_sweep", "layout": name, "Nfft": p.Nfft, "L": L, "stream_bits": p.stream_bits, "points": points,
        "streams_per_point": spp, "tile": tile, "repeats": repeats, "bin_db": bin_db, "n_bins": n_bins,
        "median_s": {k: round(v, 4) for k, v in med.items()}, "all_s": {k: [round(x, 4) for x in v] for k, v in times.items()},
        "streams_per_s_call": round(streams / med["ofdm_sweep_papr"]),
        "composed_over_call": round(med["composed exported calls"] / med["ofdm_sweep_papr"], 3),
        "identity": {"hist_equal": hist_equal, "papr_max_abs_diff_db": papr_dev, "hist_counts_ok": counts_ok},
        "exceeded_with_p_0.02_db": [round(float(x), 3) for x in ex],
        "algorithmic_bytes": {"tx_write_per_stream": L * 8, "stats_read_per_stream": L * 8, "each_way_per_8192_tile_GB": round(8192 * L * 8 / 1e9, 3)},
        "stats_kernel_ms": round(stats_ms, 3), "stats_kernel_GBps": round(stats_gbps, 1) if stats_gbps else None,
        "stats_kernel_share_of_7.7TBps": round(stats_gbps / (HBM_TBPS * 1e3), 3) if stats_gbps else None,
        "kernel_ms_call": split_call, "kernel_ms_composed": split_comp,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams-per-point", type=int, default=8192)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--layouts", default="task2,task5")
    ap.add_argument("--bin-db", type=float, default=0.01)
    ap.add_argument("--n-bins", type=int, default=4000)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_papr_sweep: no CUDA device (the library has no CPU path)")
    ctx = G.Context(0, "f32")
    name, power = card()
    for lay in a.layouts.split(","):
        out = run_layout(ctx, lay, a.streams_per_point, a.repeats, a.seed, a.bin_db, a.n_bins)
        out["gpu"], out["power_limit_and_max_sm_clock"] = name, power
        print(json.dumps(out), flush=True)
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
