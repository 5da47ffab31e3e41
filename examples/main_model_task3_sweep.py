"""Task 3 on the GPU in one library call per study (`Task 3/Main_model_Task_3.m:192-268`, `Task 3/README.md:53-60`):

  1. the BER-vs-SNR figure: BPSK, QPSK, 8PSK and 16QAM over 0:0.5:30 dB, 4 x 61 = 244 points in ONE ofdm_sweep_mer call;
  2. the MER print at 25 dB (16QAM, `README.md:53-55`);
  3. what uncorrected impairments do to the Task-3 receiver, which has no synchroniser or equaliser: STO 5, CFO 0.1 and the
     Task-4 three-tap channel, each alone and together, noise-free and at 20 dB.

    python examples/main_model_task3_sweep.py [--streams N] [--seed S]

Task 3's pilots are one real value, 4/3 * max|constellation| (`Main_model_Task_3.m:57-59`).  Prints tables only."""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ofdm_b200 as G  # noqa: E402
from ofdm_b200 import sweep  # noqa: E402
from oracle import chains as OC  # noqa: E402

NAMES = ("BPSK", "QPSK", "8PSK", "16QAM")
TAPS4 = [[0, 1], [4, .6], [10, .3]]            # `Task 4/Main_model_Task_4.m:252-264`


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=2048, help="streams per point")
    ap.add_argument("--seed", type=int, default=1)
    a = ap.parse_args()
    ctx = G.default_context("f32")
    p = OC.params_task4(alternate=False)
    lp = ctx.link_params(p.Nfft, p.T_Guard, p.N_carrier, p.N_symb, p.Amount_ODFM_SpF, p.Constellation, p.dataCarriers, p.pilotCarriers,
                         p.pilotValues)
    snrs = [0.5 * i for i in range(61)]
    fig = sweep.mer_sweep(ctx, lp, [c for c in NAMES for _ in snrs], snrs * len(NAMES), a.streams, seed=a.seed, pilot_scale=4.0 / 3.0)
    ber = fig["ber"].reshape(len(NAMES), len(snrs))
    print(f"BER over SNR, {a.streams} streams of {p.N_symb} symbols per point (one ofdm_sweep_mer call, 244 points)")
    print(f"{'SNR dB':>7} " + " ".join(f"{c:>11}" for c in NAMES))
    for i, s in enumerate(snrs):
        print(f"{s:7.1f} " + " ".join(f"{ber[k, i]:11.3e}" for k in range(len(NAMES))))

    p2 = OC.params_task4(percent=0.25, alternate=False)          # the README's run had (almost) no pilots: Np = 2
    lp2 = ctx.link_params(p2.Nfft, p2.T_Guard, p2.N_carrier, p2.N_symb, p2.Amount_ODFM_SpF, p2.Constellation, p2.dataCarriers,
                          p2.pilotCarriers, p2.pilotValues)
    m = sweep.mer_sweep(ctx, lp2, "16QAM", [25.0], a.streams, seed=a.seed, pilot_scale=4.0 / 3.0)
    print(f"\nSNR=25 dB; MER={m['mer_db'][0]:.4f} dB; BER={m['ber'][0]:.3g}   (README: MER=29.0341 dB; BER=0)")

    cases = [("none", 0, 0.0, None), ("STO 5", 5, 0.0, None), ("CFO 0.1", 0, 0.1, None), ("3-tap channel", 0, 0.0, TAPS4),
             ("all three", 5, 0.1, TAPS4)]
    print("\nUncorrected impairments, 16QAM / QPSK: BER and MER (dB)")
    print(f"{'impairment':>14} {'SNR':>5} {'BER 16QAM':>10} {'MER 16QAM':>10} {'BER QPSK':>10} {'MER QPSK':>9}")
    for name, sto, cfo, taps in cases:
        r = sweep.mer_sweep(ctx, lp, ["16QAM", "16QAM", "QPSK", "QPSK"], [np.inf, 20.0, np.inf, 20.0], a.streams, taps, seed=a.seed,
                            pilot_scale=4.0 / 3.0, sto=sto, cfo=cfo)
        for j, snr in enumerate(("inf", "20")):
            print(f"{name:>14} {snr:>5} {r['ber'][j]:10.3e} {r['mer_db'][j]:10.2f} {r['ber'][2 + j]:10.3e} {r['mer_db'][2 + j]:9.2f}")


if __name__ == "__main__":
    main()
