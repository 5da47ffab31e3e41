"""Pin P7 (DESIGN §2): the windowed-PAPR CCDF of Task 2 (`Task 2/README.md:69-71`), beside P4 (the whole-signal PAPR,
tests/test_reference_pins.py::test_P4_task2_papr).  The README reads the value that the window PAPR exceeds with probability
0.02 off calculateCCDF's curve: about 22 dB plain and about 10 dB scrambled.  The experiment is `Task 2/Main_model_Task_2.m:72-82`
on the eagle payload in the Task-2 layout (params_task4(percent=1, scale=2.0, alternate=True)): calculate_window_PAPR(tx, Nfft),
then the smallest ecdf support point whose CCDF is <= 0.02.  On the float64 oracle that is 21.878 dB plain and 10.911 dB
scrambled; tests/test_gpu_sweep_papr.py reads the same figure from ofdm_sweep_papr's histogram."""
import numpy as np

import oracle as O
from oracle import chains as OC

import reference_pins as RP

P7_README = {"plain": 22.0, "scrambled": 10.0}          # `Task 2/README.md:69-71`, read off the CCDF figure
P7_TOL = 1.5                                            # as P4: the figure is read by eye
P7_ORACLE = {"plain": 21.878, "scrambled": 10.911}      # regression values of the oracle
P7_PROB = 0.02


def window_papr_exceeded(tx, Nfft, prob=P7_PROB):
    x, c = O.calculateCCDF(O.calculate_window_PAPR(tx, Nfft))
    return x[np.argmax(c <= prob)]


def test_P7_task2_window_papr_ccdf():
    p = OC.params_task4(percent=1, scale=2.0, alternate=True)
    bits = RP.eagle_bits(p.stream_bits)
    for name, scr in (("plain", False), ("scrambled", True)):
        v = window_papr_exceeded(OC.tx_chain(p, bits, scramble=scr, fast=True)[0], p.Nfft)
        assert abs(v - P7_README[name]) < P7_TOL, (name, v)
        assert abs(v - P7_ORACLE[name]) < 0.01, (name, v)
