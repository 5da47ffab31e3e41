#!/usr/bin/env python
"""Channel-estimation MSE-vs-SNR sweep (`Task 5/Main_model_Task_5.m:303-346`) through ``ofdm_sweep_mse``: whole-call time,
a per-stage split of one tile, and a check that the same tiles pushed through the composed exported calls give identical
per-stream arrays.  Prints one JSON line (on rank 0).

    python tools/bench_mse_sweep.py [--streams-per-point 4096] [--tile 0] [--snr-step 0.5] [--comb 1] [--gpus N]

Default: the script's main configuration (Nfft 4096, N_carrier 1024, comb 1 = pilots only, pilots 4/3 of the 16QAM
maximum, the six taps of `:112-119`), SNR 0:0.5:30 = 61 points x 4,096 streams, FP32.  --gpus N > 1 re-runs the script
under torch.distributed.run with one process per GPU (the stage split and the check run on rank 0 only)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ofdm_b200 as G  # noqa: E402
from ofdm_b200 import layouts, sweep  # noqa: E402

TAPS = layouts.TAPS_TASK5


def card():
    """Name and power limit of the GPU this process runs on, read now."""
    name = torch.cuda.get_device_name()
    try:
        idx = torch.cuda.current_device()
        out = subprocess.run(["nvidia-smi", "-i", str(idx), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "not available"
    return name, out


class Stages:
    """CUDA events around named stages, summed per name."""

    def __init__(self):
        self.ev = []

    def run(self, name, fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        self.ev.append((name, a, b))
        return out

    def ms(self):
        torch.cuda.synchronize()
        res = {}
        for name, a, b in self.ev:
            res[name] = res.get(name, 0.0) + a.elapsed_time(b)
        return res


def composed_tile(ctx, lp, snr, g0, n, seed, tie_eps, Ldict, st):
    """One tile of the sweep as exported calls (what ofdm_sweep_mse fuses or chains internally): (per_stream [4, n], near)."""
    pc, pv = lp.pilotCarriers, lp.pilotValues
    S, Nfft, Tg, Nc, K = lp.S, lp.Nfft, lp.Tg, lp.N_carrier, len(TAPS)
    h, Htrue = ctx.mp_channel_resp(TAPS, Nfft)
    h_dev = ctx.cplx(h)

    def front():
        if lp.Nd == 0:
            tx = ctx.modulate(ctx.map_carriers(None, 1, S, Nfft, [], pc, pv), Tg).expand(n, -1, -1).contiguous()
            psum = None
        else:
            words = lp.stream_bits // 32
            bits = torch.empty(n * words, dtype=torch.int32, device=ctx.device)
            ctx._chk(ctx.lib.ofdm_payload_bits(ctx.h, ctx.p(bits), n, words, seed, g0))
            tx, psum = ctx.tx_chain(lp, bits, n, want_power=True)
        rx = ctx.channel_t5(tx, snr_db=float(snr), h_dev=h_dev, seed=seed, first_stream_id=g0, power_sum=psum)
        del tx
        Y = ctx.demodulate(rx, Nfft, Tg)
        return Y, ctx.pilot_ls(Y, pv, pc)

    Y, y = st.run("front end: TX, channel, demodulate, pilot_ls (composed)", front)
    H_ls, hls = st.run("LS + ifft", lambda: (lambda H: (H, ctx.fft(H, inverse=True)))(ctx.ls_ce(Y, pv, pc, Nc)))
    H_mm = st.run("MMSE", lambda: ctx.mmse_ce(Y, pv, pc, Nc, hls, float(snr)))
    del Y
    H_mp = st.run("MP", lambda: ctx.mp(y, Nfft, K, Ldict=Ldict, pilot_loc=pc)[0])
    H_omp, _, _, _, near = st.run("OMP", lambda: ctx.omp(y, Nfft, K, Ldict=Ldict, pilot_loc=pc, tie_eps=tie_eps))
    ref = Htrue[None].expand(n, -1).contiguous()
    per = st.run("MSE x 4", lambda: torch.stack([ctx.mse(ref, H, Nc) for H in (H_ls, H_mm, H_mp, H_omp)]))
    return per.cpu().numpy(), int((near != 0).sum().item())


def fused_kernel_ms(ctx, lp, snr, n, seed, tie_eps, Ldict):
    """Kernel times of ONE fused tile (ofdm_sweep_mse with one point of n streams), from torch.profiler, by kernel name."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sweep.mse_sweep_local(ctx, lp, [snr], n, TAPS, Ldict, seed=seed, tile=n, tie_eps=tie_eps)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0.0)
        if t > 0:
            out[e.key.split("(")[0].split("<")[0][:60]] = round(t / 1e3, 4)
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams-per-point", type=int, default=4096)
    ap.add_argument("--tile", type=int, default=0, help="streams per work item (0 = the library default, 8192)")
    ap.add_argument("--snr-step", type=float, default=0.5)
    ap.add_argument("--comb", type=int, default=1)
    ap.add_argument("--precision", default="f32", choices=["f32", "f64"])
    ap.add_argument("--tie-eps", type=float, default=1e-4)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--gpus", type=int, default=1)
    a = ap.parse_args()
    if a.gpus > 1 and "RANK" not in os.environ:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", str(a.gpus), "--master-addr", "127.0.0.1", os.path.abspath(__file__)]
        sys.exit(subprocess.run(cmd + sys.argv[1:]).returncode)
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    if not torch.cuda.is_available():
        raise SystemExit("bench_mse_sweep: no CUDA device (the library has no CPU path)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = G.Context(local, a.precision)
    lp = layouts.task5_link(ctx, comb=a.comb, scale=4.0 / 3.0, alternate=False, scramble=False)
    Ldict = -(-lp.N_carrier // a.comb)
    snrs = np.arange(0.0, 30.0 + 1e-9, a.snr_step)
    spp = a.streams_per_point
    name, power = card()
    # warm-up over two points at the timed tile size: kernels loaded, plans and the pool's buffers in place
    sweep.mse_sweep(ctx, lp, snrs[:2], spp, TAPS, Ldict, seed=a.seed + 1, rank=rank, world=world, tile=a.tile, tie_eps=a.tie_eps)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    per, cnt = sweep.mse_sweep_local(ctx, lp, snrs, spp, TAPS, Ldict, seed=a.seed, rank=rank, world=world, tile=a.tile, tie_eps=a.tie_eps)
    e1.record()
    torch.cuda.synchronize()
    dt = torch.tensor([e0.elapsed_time(e1) * 1e-3], dtype=torch.float64, device=ctx.device)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    mean, per_h, counts = sweep.reduce_mse(per, cnt)
    if rank == 0:
        # the same tiles (first tile of three points) through the composed exported calls, each stage between events
        tile = min(a.tile or 8192, spp)
        check, near_ok = [], True
        for i in sorted({0, len(snrs) // 2, len(snrs) - 1}):
            st = Stages()
            want, near = composed_tile(ctx, lp, snrs[i], i * spp, tile, a.seed, a.tie_eps, Ldict, st)
            check.append(bool(np.array_equal(per_h[i, :, :tile], want)))
            near_ok &= (tile < spp) or near == int(counts[i, 1])
            stages = st.ms()                            # the last point's: every stage already warm
        kern = fused_kernel_ms(ctx, lp, float(snrs[0]), tile, a.seed, a.tie_eps, Ldict)
        total = len(snrs) * spp
        print(json.dumps({
            "workload": "MSE-vs-SNR sweep (Main_model_Task_5.m:303-346): comb %d, %s, SNR 0:%g:30 (%d points) x %d streams, LS/MMSE/MP/OMP"
                        % (a.comb, a.precision, a.snr_step, len(snrs), spp),
            "gpu": name, "power_limit_and_max_sm_clock": power, "n_gpus": world, "tile": a.tile or 8192,
            "seconds": float(dt.item()), "streams": total, "streams_per_s": total / float(dt.item()),
            "mean_mse_at_snr": {str(float(snrs[i])): [float(x) for x in mean[i]] for i in range(0, len(snrs), 10)},
            "omp_near_tie_frames": int(counts[:, 1].sum()),
            "stage_ms_one_tile_composed": {k: round(v, 3) for k, v in stages.items()}, "stage_tile_streams": tile,
            "fused_kernel_ms_one_tile": kern,
            "composed_equals_fused": bool(all(check) and near_ok)}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
