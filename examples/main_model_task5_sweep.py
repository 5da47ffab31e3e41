#!/usr/bin/env python
"""`Task 5/Main_model_Task_5.m:303-346` (channel-estimation half): the MSE of the LS / MMSE / MP / OMP estimates against
the true frequency response over SNR 0:0.5:30 dB, averaged over many noise realisations per point, as one library call
per rank (``ofdm_sweep_mse``).  Main configuration of the script: Nfft 4096, N_carrier 1024, comb 1 (pilots only,
`:24-33`), pilot amplitude 4/3 of the 16QAM maximum, the six taps of `:112-119`.  Plotting is left out.

    python examples/main_model_task5_sweep.py [--streams 1024] [--precision f32|f64]
    python -m torch.distributed.run --nproc_per_node 8 examples/main_model_task5_sweep.py      # one share per GPU
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def run(streams=1024, precision="f32", snrs=None, seed=1, rank=0, world=1, device=0):
    import ofdm_b200 as G
    from ofdm_b200 import layouts, sweep
    ctx = G.Context(device, precision)
    # `Main_model_Task_5.m:6-46`: comb 1 puts a pilot on every carrier of N_carrier, amplitude 4/3 of the 16QAM maximum
    lp = layouts.task5_link(ctx, comb=1, scale=4.0 / 3.0, alternate=False, scramble=False)
    snrs = np.arange(0, 30.5, 0.5) if snrs is None else np.asarray(snrs, dtype=np.float64)
    return snrs, sweep.mse_sweep(ctx, lp, snrs, streams, layouts.TAPS_TASK5, seed=seed, rank=rank, world=world, tie_eps=1e-4)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=1024, help="noise realisations per SNR point")
    ap.add_argument("--precision", default="f32", choices=["f32", "f64"])
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
        dist.init_process_group("nccl")
    snrs, (mean, _, counts) = run(args.streams, args.precision, rank=rank, world=world, device=int(os.environ.get("LOCAL_RANK", 0)))
    if rank == 0:
        print("SNR(dB)   MSE_LS      MSE_MMSE    MSE_MP      MSE_OMP     OMP near-tie frames")
        for s, m, c in zip(snrs, mean, counts):
            print("%6.1f  %.4e  %.4e  %.4e  %.4e  %d / %d" % (s, m[0], m[1], m[2], m[3], c[1], c[0]))
    if world > 1:
        dist.destroy_process_group()
