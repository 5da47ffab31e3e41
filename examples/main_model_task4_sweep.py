#!/usr/bin/env python
"""The two link-quality results of `Task 4/README.md` as one library call per rank each (``ofdm_sweep_sync``), plus the
BER / MER table of the Task-4 chain with randomly drawn impairments:

  1. channel-estimate error over SNR at pilot step 4 (`Task 4/graphs/nmse(snr).png`, `README.md:189-193`): 25 % pilots,
     Noise then the 3-tap channel, no STO / CFO, the receiver without its sync stages;
  2. CFO-estimator error and failure rate over SNR at STO 150, CFO 0.24, no multipath (`README.md:111-121`);
  3. BER, MER and detector failures with Time_Delay = randi([0, Nfft + T_Guard]) and Freq_Shift = randi([0, 30]) + rand - 0.5
     over the 3-tap channel (`Main_model_Task_4.m:95-110,252-264,374`).

    python examples/main_model_task4_sweep.py [--streams 4096]
    python -m torch.distributed.run --nproc_per_node 8 examples/main_model_task4_sweep.py      # one share per GPU
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

TAPS4 = [[0, 1], [4, .6], [10, .3]]                         # `Main_model_Task_4.m:252-264`
FIGURE = {0.0: 5.5e-3, 10.0: 4e-4, 15.0: 1e-4}              # read off `Task 4/graphs/nmse(snr).png`


def run(streams=4096, seed=1, rank=0, world=1, device=0):
    import ofdm_b200 as G
    from ofdm_b200 import sweep
    from oracle import chains as OC
    ctx = G.Context(device, "f32")

    def link(p):
        return ctx.link_params(p.Nfft, p.T_Guard, p.N_carrier, p.N_symb, p.Amount_ODFM_SpF, p.Constellation, p.dataCarriers, p.pilotCarriers,
                               p.pilotValues)

    snrs = np.arange(0.0, 30.0 + 1e-9, 2.5)
    kw = dict(seed=seed, rank=rank, world=world)
    nmse = sweep.sync_sweep(ctx, link(OC.params_task4(percent=25)), snrs, streams, TAPS4, sto=0, cfo=0.0, time_desync=False, freq_desync=False, **kw)
    cfo = sweep.sync_sweep(ctx, link(OC.params_task4()), snrs, streams, None, sto=150, cfo=0.24, mp_desync=False, **kw)
    ber = sweep.sync_sweep(ctx, link(OC.params_task4()), snrs, streams, TAPS4, **kw)
    return snrs, nmse, cfo, ber


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=4096, help="streams per SNR point")
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
        dist.init_process_group("nccl")
    snrs, nmse, cfo, ber = run(args.streams, rank=rank, world=world, device=int(os.environ.get("LOCAL_RANK", 0)))
    if rank == 0:
        print("1. Channel estimate at pilot step 4 (101 pilots), 3-tap channel, no STO/CFO")
        print("SNR(dB)   mean|H_est-H|^2  NMSE (/mean|H|^2)  figure   NaN cells")
        for s, m, n, k in zip(snrs, nmse["h_err_mean"], nmse["nmse"], nmse["h_err_nan"]):
            print("%6.1f   %.3e        %.3e          %-8s %d" % (s, m, n, "%.1e" % FIGURE[s] if s in FIGURE else "", k))
        print("\n2. CFO estimator at STO 150, CFO 0.24, no multipath (error = FreqOffset + max(IFO,0) - CFO)")
        print("SNR(dB)   detector failures  mean error   RMS error   |error| <= 0.02   timing residual (min..max)")
        for i, s in enumerate(snrs):
            print("%6.1f   %8.4f           %+.4f     %.4f      %.4f            %d..%d" % (
                s, cfo["fail_rate"][i], cfo["cfo_err_mean"][i], cfo["cfo_err_rms"][i], cfo["cfo_within"][i], cfo["timing_min"][i], cfo["timing_max"][i]))
        print("\n3. Drawn STO / CFO, 3-tap channel, all receiver stages")
        print("SNR(dB)   BER        mean MER(dB)  detector failures  IFO misses")
        for i, s in enumerate(snrs):
            print("%6.1f   %.4e   %7.2f       %.4f             %.4f" % (s, ber["ber"][i], ber["mer_db"][i], ber["fail_rate"][i], ber["ifo_miss_rate"][i]))
    if world > 1:
        dist.destroy_process_group()
