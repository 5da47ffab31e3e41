#!/usr/bin/env python
"""Task-3 BER/MER study (`Task 3/Main_model_Task_3.m:192-268`) through ``ofdm_sweep_mer``: the whole figure (BPSK, QPSK, 8PSK
and 16QAM over 0:0.5:30 dB) as ONE call, against (a) the same streams through ``ofdm_sweep_sync`` with every receiver stage
off, one call per constellation, and (b) the same streams through the composed exported calls per tile (ofdm_payload_bits,
bit packing, DeScrambler, ofdm_tx_chain_p, ofdm_channel_t4_p, ofdm_rx_chain_t4_ex(0, 0, 0)), all three in one process with
a check that their {errors, bits} counters are identical (the sync arm numbers the streams of each constellation from 0, so
it is compared with ofdm_sweep_mer called once per constellation); then a torch.profiler run of one 16QAM tile for the receiver
kernel's time and its bytes/s.  Prints one JSON line.

    python tools/bench_mer_sweep.py [--streams-per-point 8192] [--repeats 2]

Receiver bytes are counted from shapes: per stream the 8 * S * Nfft bytes of samples it transforms (the cyclic prefix is
not read), the S * Nd * bps / 8 bytes of transmitted bits it compares with, and its 16 bytes of MER sums."""
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

NAMES = ("BPSK", "QPSK", "8PSK", "16QAM")
SNRS = [0.5 * i for i in range(61)]
SCALE = 4.0 / 3.0                                   # Task 3's pilots: 4/3 * max|constellation|


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


def timed(ctx, fn):
    ctx.sync()
    t0 = time.perf_counter()
    out = fn()
    ctx.sync()
    return time.perf_counter() - t0, out


def arm_mer(ctx, lp, spp):
    cons = [c for c in NAMES for _ in SNRS]
    res = sweep.mer_sweep(ctx, lp, cons, SNRS * len(NAMES), spp, seed=1, pilot_scale=SCALE)
    return res["counts"][:, :2]


def mer_per_constellation(ctx, lp, spp):
    """The sync arm's streams through ofdm_sweep_mer (one call per constellation, g numbered from 0 in each)."""
    return np.concatenate([sweep.mer_sweep(ctx, lp, c, SNRS, spp, seed=1, pilot_scale=SCALE)["counts"][:, :2] for c in NAMES])


def arm_sync(ctx, spp):
    out = []
    for c in NAMES:                                  # one call per constellation: its own pilots, g numbered from 0
        p = OC.params_task4(alternate=False, Constellation=c)
        r = sweep.sync_sweep(ctx, link(ctx, p), SNRS, spp, seed=1, sto=0, cfo=0.0, time_desync=False, freq_desync=False, mp_desync=False)
        out.append(r["counts"][:, :2])
    return np.concatenate(out)


def arm_composed(ctx, spp, tile=8192):
    """The one-call figure's streams (g = point * spp + j over the 4 x 61 points) through the exported calls."""
    out = []
    shifts = torch.arange(32, device=ctx.device, dtype=torch.int64)
    one = ctx.cplx(np.ones(1, dtype=np.complex128))
    for ci, c in enumerate(NAMES):
        p = OC.params_task4(alternate=False, Constellation=c)
        lp, lp_tx = link(ctx, p), link(ctx, p, scramble=False)
        words = -(-p.stream_bits // 32)
        counts = torch.zeros((len(SNRS), 4), dtype=torch.int64, device=ctx.device)
        for (i, s0, n) in sweep.tiles(len(SNRS), spp, tile):
            g0 = (ci * len(SNRS) + i) * spp + s0
            raw = torch.empty(n * words, dtype=torch.int32, device=ctx.device)
            ctx._chk(ctx.lib.ofdm_payload_bits(ctx.h, ctx.p(raw), n, words, 1, g0))
            bits = ((raw.view(n, words).to(torch.int64)[..., None] >> shifts) & 1).reshape(n, -1)[:, :p.stream_bits].reshape(-1)
            pad = (-bits.numel()) % 32
            bits = torch.cat([bits, bits.new_zeros(pad)]).view(-1, 32)
            sbits = ((bits << shifts).sum(dim=1) & 0xFFFFFFFF).to(torch.int64)
            sbits = torch.where(sbits >= 2 ** 31, sbits - 2 ** 32, sbits).to(torch.int32)      # packed s, the library's bit layout
            pbits = ctx.scramble(sbits, n * p.Amount_OFDM_Frames, p.frame_bits, descramble=True)
            tx, psum = ctx.tx_chain(lp_tx, sbits, n, want_power=True)
            sto = torch.zeros(n, dtype=torch.int32, device=ctx.device)
            cfo = torch.zeros(n, dtype=torch.float64, device=ctx.device)
            rx = ctx.channel_t4(tx.reshape(n, -1), SNRS[i], sto, cfo, p.Nfft, one, seed=1, first_stream_id=g0, power_sum=psum)
            r = ctx.rx_chain_t4_fused(lp, rx.reshape(n, p.N_symb, -1), tx_bits_dev=pbits, time_desync=False, freq_desync=False, mp_desync=False,
                                      want_bits=False)
            counts[i, :2] += r["counts"][:2]
        ctx.sync()
        out.append(counts[:, :2].cpu().numpy())
    return np.concatenate(out)


def receiver_kernel(ctx, lp, p, n):
    """torch.profiler over one 16QAM call of n streams: (receiver kernel ms, whole-call kernels ms)."""
    from torch.profiler import ProfilerActivity, profile
    sweep.mer_sweep(ctx, lp, "16QAM", [10.0], n, pilot_scale=SCALE)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sweep.mer_sweep(ctx, lp, "16QAM", [10.0], n, pilot_scale=SCALE)
        ctx.sync()
    rx_us = tot_us = 0.0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
        if e.key.startswith("void rx_t3_kernel") or "rx_t3_kernel" in e.key:
            rx_us += t
        tot_us += t if "kernel" in e.key or e.key.startswith("void ") else 0.0
    return rx_us / 1e3, tot_us / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams-per-point", type=int, default=8192)
    ap.add_argument("--repeats", type=int, default=2)
    a = ap.parse_args()
    spp = a.streams_per_point
    ctx = G.default_context("f32")
    p = OC.params_task4(alternate=False)
    lp = link(ctx, p)
    name, power = card()
    arm_mer(ctx, lp, 64), arm_sync(ctx, 64), arm_composed(ctx, 64)          # warm-up of every shape the timed calls use
    t = {"mer": [], "sync": [], "composed": []}
    counters = {}
    for _ in range(a.repeats):                       # alternated, so that a slow spell of the shared host hits every arm
        for arm, fn in (("mer", lambda: arm_mer(ctx, lp, spp)), ("sync", lambda: arm_sync(ctx, spp)), ("composed", lambda: arm_composed(ctx, spp))):
            s, c = timed(ctx, fn)
            t[arm].append(s)
            counters[arm] = c
    same = bool(np.array_equal(counters["mer"], counters["composed"]) and np.array_equal(mer_per_constellation(ctx, lp, spp), counters["sync"]))
    n_streams = len(NAMES) * len(SNRS) * spp
    n_prof = min(spp, 8192)
    rx_ms, tot_ms = receiver_kernel(ctx, lp, p, n_prof)
    rx_bytes = n_prof * (8 * p.N_symb * p.Nfft + p.stream_bits // 8 + 16)
    print(json.dumps({
        "bench": "mer_sweep", "gpu": name, "power_limit_and_max_sm_clock": power,
        "shape": f"params_task4 (Nfft 1024, N_carrier 400, Nd 332, S 50), pilots 4/3 max|c|, 4 constellations x {len(SNRS)} SNR x {spp} streams",
        "streams": n_streams, "counters_identical": same,
        "mer_call_s": min(t["mer"]), "sync_per_constellation_s": min(t["sync"]), "composed_s": min(t["composed"]),
        "mer_streams_per_s": n_streams / min(t["mer"]), "sync_streams_per_s": n_streams / min(t["sync"]),
        "composed_streams_per_s": n_streams / min(t["composed"]),
        "all_times_s": t,
        "receiver_kernel": {"streams": n_prof, "ms": rx_ms, "bytes": rx_bytes, "GB_per_s": rx_bytes / (rx_ms * 1e-3) / 1e9 if rx_ms else None,
                            "all_kernels_of_call_ms": tot_ms},
        "ber_16qam_at_10dB": float(counters["mer"][3 * len(SNRS) + 20, 0] / counters["mer"][3 * len(SNRS) + 20, 1]),
    }))
    if not same:
        sys.exit("counters differ between the arms")


if __name__ == "__main__":
    main()
