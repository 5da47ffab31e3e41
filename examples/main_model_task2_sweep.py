#!/usr/bin/env python
"""Task 2's PAPR study (`Task 2/Main_model_Task_2.m:72-82`, `Task 2/README.md:54,69-71`) as library calls (``ofdm_sweep_papr``):
the PAPR of the transmitted signal without and with the scrambler, for a balanced and a strongly biased Bernoulli payload over
many streams, and for the image payload of the script when a TIFF is given.  Task-2 layout: Nfft 1024, 400 carriers, 1 %
pilots at amplitude 2 alternating in sign, 50 symbols of 16QAM (79,000 payload bits per stream).

    python examples/main_model_task2_sweep.py [image.tiff] [--streams 4096]
    python -m torch.distributed.run --nproc_per_node 8 examples/main_model_task2_sweep.py      # one share per GPU

Columns: mean stream PAPR (calculatePAPR) and the window PAPR (calculate_window_PAPR) exceeded with probability 0.02, 1e-3 and
1e-5, read from a histogram of 0.01 dB bins.  The image rows transmit the image's first 79,000 bits once, as the script does;
their 0.02 figures are pin P7 (21.878 / 10.911 dB on the float64 oracle; the README reads about 22 / 10)."""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

PROBS = (0.02, 1e-3, 1e-5)
BIN_DB, N_BINS = 0.01, 4000


def run(image=None, streams=4096, seed=1, rank=0, world=1, device=0):
    import ofdm_b200 as G
    from ofdm_b200 import sweep
    from oracle import chains as OC
    ctx = G.Context(device, "f32")
    p = OC.params_task4(percent=1, scale=2.0, alternate=True)
    lp = ctx.link_params(p.Nfft, p.T_Guard, p.N_carrier, p.N_symb, p.Amount_ODFM_SpF, p.Constellation, p.dataCarriers, p.pilotCarriers,
                         p.pilotValues)
    rows = []
    for pone in (0.5, 0.05):
        res = sweep.papr_sweep(ctx, lp, [(0, pone), (1, pone)], streams, seed=seed, rank=rank, world=world, bin_db=BIN_DB, n_bins=N_BINS)
        for k, name in enumerate(("plain", "scrambled")):
            rows.append((f"Bernoulli p={pone}", name, streams, res["papr_mean"][k], [sweep.papr_exceedance(res["hist"][k], BIN_DB, q) for q in PROBS]))
    if image:
        from ofdm_b200 import realisations
        bits = realisations.file_reader(image, p.stream_bits)
        res = sweep.papr_sweep(ctx, lp, [(0, None), (1, None)], 1, rank=rank, world=world, bin_db=BIN_DB, n_bins=N_BINS, pool=bits, pool_stride=0)
        for k, name in enumerate(("plain", "scrambled")):
            rows.append((os.path.basename(image), name, 1, res["papr_mean"][k], [sweep.papr_exceedance(res["hist"][k], BIN_DB, q) for q in PROBS]))
    return rows


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("image", nargs="?", help="TIFF payload, read as file_reader.m does")
    ap.add_argument("--streams", type=int, default=4096, help="streams per Bernoulli point")
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
        dist.init_process_group("nccl")
    rows = run(args.image, args.streams, rank=rank, world=world, device=int(os.environ.get("LOCAL_RANK", 0)))
    if rank == 0:
        print("payload                signal      streams   mean PAPR(dB)   window PAPR exceeded with p = " + " / ".join(f"{q:g}" for q in PROBS))
        for src, name, n, mean, ex in rows:
            print(f"{src:<22} {name:<11} {n:>7}   {mean:13.3f}   " + " / ".join(f"{x:6.2f}" for x in ex))
    if world > 1:
        dist.destroy_process_group()
