#!/usr/bin/env python
"""Task-4 sync sweep (`Task 4/Main_model_Task_4.m:95-110,277-374`) through ``ofdm_sweep_sync``: whole-call time against
(a) the same tiles through the composed exported calls (payload, DeScrambler, ofdm_draw_sto_cfo, ofdm_tx_chain_p,
ofdm_channel_t4_p, ofdm_rx_chain_t4_ex with every estimate output and H, ofdm_mse) and (b) ``ofdm_sweep_ber``'s Task-4 chain
at the same shape and seed, the three alternated in one process; a check that the composed calls give the same records and
counters; a torch.profiler kernel split of one tile; and the algorithmic bytes of the call.  Prints one JSON line.

    python tools/bench_sync_sweep.py [--streams-per-point 8192] [--snr-step 2] [--tile 0] [--repeats 5]

Default: params_task4 (Nfft 1024, N_carrier 400, 68 pilots, Nd 332, S 50, 16QAM), the 3-tap channel of `:252-264`, STO and
CFO drawn as the BER sweep draws them, every receiver stage on, SNR 0:2:30 = 16 points x 8,192 streams, FP32."""
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

TAPS4 = [[0, 1], [4, .6], [10, .3]]


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


def true_response(p):
    h = np.zeros(11)
    for d, a in TAPS4:
        h[int(d)] = a
    return h, np.fft.fft(h, p.Nfft)[:p.N_carrier]


def composed(ctx, lp, lp_tx, p, snrs, spp, tile, seed, Ht_dev, h_dev, rec=None, counts=None):
    """The sweep as exported calls per tile (as a user composes it today); fills rec (n_snr, 9, spp) fields 0-5, 7, 8 and
    counts (n_snr, 4) on the device when given.  The H error is ofdm_mse of the FP32 estimate against the FP32 true response."""
    words = p.stream_bits // 32
    for (i, s0, n) in sweep.tiles(len(snrs), spp, tile):
        g0 = i * spp + s0
        sbits = torch.empty(n * words, dtype=torch.int32, device=ctx.device)
        ctx._chk(ctx.lib.ofdm_payload_bits(ctx.h, ctx.p(sbits), n, words, seed, g0))
        bits = ctx.scramble(sbits, n * p.Amount_OFDM_Frames, p.frame_bits, descramble=True)
        sto = torch.empty(n, dtype=torch.int32, device=ctx.device)
        cfo = torch.empty(n, dtype=torch.float64, device=ctx.device)
        ctx._chk(ctx.lib.ofdm_draw_sto_cfo(ctx.h, n, seed, g0, p.Nfft + p.T_Guard, 30, ctx.p(sto), ctx.p(cfo)))
        tx, psum = ctx.tx_chain(lp_tx, sbits, n, want_power=True)
        rx = ctx.channel_t4(tx.reshape(n, -1), float(snrs[i]), sto, cfo, p.Nfft, h_dev, seed=seed, first_stream_id=g0, power_sum=psum)
        del tx
        out = ctx.rx_chain_t4_fused(lp, rx.reshape(n, p.N_symb, -1), tx_bits_dev=bits, want_bits=False, want_H=True)
        herr = ctx.mse(Ht_dev.expand(n, -1).contiguous(), out["H"], p.N_carrier)
        if rec is not None:
            r = rec[i, :, s0:s0 + n]
            r[0], r[1], r[2], r[3], r[4], r[5], r[7], r[8] = (out["TgPosition"], out["FreqOffset"], out["IFO"], out["tau"], out["phase_shift"], herr,
                                                              sto, cfo)
            counts[i, 0] += out["counts"][0]
            counts[i, 1] += out["counts"][1]
            counts[i, 2] += out["fail"].sum()
            counts[i, 3] += (out["IFO"] == -1).sum()


def sync_kernel_ms(ctx, lp, snr, n, seed):
    """Kernel times of ONE tile of ofdm_sweep_sync (one point of n streams) from torch.profiler, by kernel name."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sweep.sync_sweep_local(ctx, lp, [snr], n, TAPS4, seed=seed, tile=n)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0.0)
        if t > 0:
            out[e.key.split("(")[0].split("<")[0][:60]] = round(t / 1e3, 4)
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def algorithmic_bytes(p):
    """HBM bytes per stream the sync call needs at minimum, by stage (one read / write of every array it cannot avoid)."""
    L = p.stream_len * 8                       # complex64 samples
    bins = p.N_symb * (len(p.dataCarriers) + len(p.pilotCarriers)) * 8
    payload = p.stream_bits // 8
    return {"payload + DeScrambler": 3 * payload, "TX chain (write)": L + payload, "channel (read tx, write rx)": 2 * L,
            "AutoCorrFunction (read rx)": L, "IFO search (read one symbol)": p.Nfft * 8, "symbol FFTs (read rx, write bins)": L + bins,
            "post / statistics (read bins, payload; write record)": bins + payload + 9 * 8}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams-per-point", type=int, default=8192)
    ap.add_argument("--snr-step", type=float, default=2.0)
    ap.add_argument("--tile", type=int, default=0, help="streams per work item (0 = the library default, 8192)")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--seed", type=int, default=1)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sync_sweep: no CUDA device (the library has no CPU path)")
    ctx = G.Context(0, "f32")
    p = OC.params_task4()
    lp, lp_tx = link(ctx, p), link(ctx, p, scramble=False)
    snrs = np.arange(0.0, 30.0 + 1e-9, a.snr_step)
    spp = a.streams_per_point
    tile = a.tile or 8192
    h, Ht = true_response(p)
    h_dev = ctx.cplx(h.astype(np.complex128))
    Ht_dev = ctx.cplx(Ht)
    name, power = card()

    runs = {
        "ofdm_sweep_sync": lambda: sweep.sync_sweep_local(ctx, lp, snrs, spp, TAPS4, seed=a.seed, tile=a.tile),
        "ofdm_sweep_ber (Task-4 chain)": lambda: sweep.sweep_local(ctx, lp, snrs, spp, TAPS4, "task4", seed=a.seed, tile=a.tile),
        "composed exported calls": lambda: composed(ctx, lp, lp_tx, p, snrs, spp, tile, a.seed, Ht_dev, h_dev),
    }
    for fn in runs.values():                   # warm-up: modules loaded, plans and pools in place
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in runs}
    for _ in range(a.repeats):                 # alternated in one process
        for k, fn in runs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            times[k].append(time.perf_counter() - t0)
    med = {k: float(np.median(v)) for k, v in times.items()}

    # identity: the library call against the composed calls
    rec, cnt = sweep.sync_sweep_local(ctx, lp, snrs, spp, TAPS4, seed=a.seed, tile=a.tile)
    crec = torch.zeros_like(rec)
    ccnt = torch.zeros_like(cnt)
    composed(ctx, lp, lp_tx, p, snrs, spp, tile, a.seed, Ht_dev, h_dev, crec, ccnt)
    torch.cuda.synchronize()
    r, c = rec.cpu().numpy(), crec.cpu().numpy()
    est_equal = all(np.array_equal(r[:, f], c[:, f], equal_nan=True) for f in (0, 1, 2, 3, 4, 7, 8))
    counts_equal = bool(torch.equal(cnt, ccnt))
    # the library's H error is against the double response; the composed FP32 ofdm_mse against the rounded one
    ok = ~np.isnan(c[:, 5])
    herr_rel = float(np.max(np.abs(r[:, 5][ok] - c[:, 5][ok]) / c[:, 5][ok])) if ok.any() else 0.0
    nan_equal = bool(np.array_equal(np.isnan(r[:, 5]), np.isnan(c[:, 5])))

    streams = len(snrs) * spp
    by = algorithmic_bytes(p)
    tot = sum(by.values()) * streams
    out = {
        "bench": "sync_sweep", "gpu": name, "power_limit_and_max_sm_clock": power, "shape": "params_task4, 3 taps, drawn STO/CFO, all stages on",
        "snr_points": len(snrs), "streams_per_point": spp, "tile": tile, "repeats": a.repeats,
        "median_s": {k: round(v, 4) for k, v in med.items()}, "all_s": {k: [round(x, 4) for x in v] for k, v in times.items()},
        "sync_over_ber": round(med["ofdm_sweep_sync"] / med["ofdm_sweep_ber (Task-4 chain)"], 4),
        "composed_over_sync": round(med["composed exported calls"] / med["ofdm_sweep_sync"], 3),
        "streams_per_s_sync": round(streams / med["ofdm_sweep_sync"]),
        "identity": {"estimates_bit_equal": est_equal, "counters_equal": counts_equal, "h_err_nan_cells_equal": nan_equal,
                     "h_err_max_rel_vs_fp32_ofdm_mse": herr_rel},
        "algorithmic_bytes_per_stream": by, "algorithmic_GBps_sync": round(tot / med["ofdm_sweep_sync"] / 1e9, 1),
        "kernel_ms_one_tile": sync_kernel_ms(ctx, lp, 10.0, min(spp, tile), a.seed),
    }
    print(json.dumps(out))


if __name__ == "__main__":
    main()
