#!/usr/bin/env python
"""Task-5 part 2 (`Task 5/Task5_part2.m:46-321`) in one library call: the NMSE and BER of the LS, MMSE, MP and OMP channel
estimates for the script's 57 pilot combs (`:13-17`) x 100 static EPA fading runs at 20 dB (`ofdm_sweep_part2`).

    python examples/task5_part2_sweep.py [image.tiff]

With a TIFF path the payload is read from the image as `file_reader.m:4-11` does; otherwise it is seeded random bits."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ofdm_b200 as G  # noqa: E402
from ofdm_b200 import part2  # noqa: E402


def main():
    ctx = G.Context(0, "f32")
    combs, amounts = part2.part2_combs()
    need = 2 * 7 * 1020 * 4                                   # the longest stream: comb 256, four pilots
    if len(sys.argv) > 1:
        from ofdm_b200 import realisations
        bits = np.asarray(realisations.file_reader(sys.argv[1], need), dtype=np.uint8)
    else:
        bits = np.random.default_rng(1).integers(0, 2, need).astype(np.uint8)
    NMSE, BER, _, counts, runs = part2.sweep_lib(ctx, combs, 100, bits, profile="EPA", fs_hz=4e7, snr_db=20.0, seed=1)
    print(f"{'comb':>5} {'pilots':>6} | " + " ".join(f"NMSE {e:<5}" for e in part2.ESTIMATORS) + " | "
          + " ".join(f"BER {e:<6}" for e in part2.ESTIMATORS))
    for k, (c, a) in enumerate(zip(combs, amounts)):
        print(f"{c:>5} {a:>6} | " + " ".join(f"{x:10.3e}" for x in NMSE[:, k]) + " | " + " ".join(f"{x:10.3e}" for x in BER[:, k]))
    print(f"{int(runs[:, 0].sum())} runs; OMP runs with a near-tie: {int(runs[:, 1].sum())}")


if __name__ == "__main__":
    main()
