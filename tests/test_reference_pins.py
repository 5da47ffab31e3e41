"""The oracle against the numbers the reference itself holds (see `tests/reference_pins.py` for what each pins and which
experiment definitions are inferred).  CPU only; the same pins run on the CUDA path in `test_gpu_reference_pins.py`."""
import hashlib
import json
import os

import numpy as np
import pytest
from scipy.interpolate import interp1d

import oracle as O
from oracle import chains as OC

import reference_pins as RP


def test_payload_fixture_is_the_pinned_payload(tmp_path):
    d = json.load(open(os.path.join(RP.HERE, "golden", "eagle_bits_digest.json")))
    raw = open(os.path.join(RP.HERE, "golden", "eagle_bits.bin"), "rb").read()
    assert hashlib.sha256(raw).hexdigest() == d["sha256_of_packbits"]
    b = RP.eagle_bits(129600)
    assert b.size == d["n_bits"] and int(b.sum()) == d["n_ones"] and "".join(map(str, b[:64])) == d["first_64"]
    path = RP.write_eagle_tiff(tmp_path / "eagle.tiff")
    assert np.array_equal(b, OC.read_payload_bits(path, 129600))


def _task3_ber(cname, snr, seeds):
    """One point of `Task 3/Main_model_Task_3.m:192-268`."""
    p = OC.params_task4(alternate=False, Constellation=cname)          # Task 3 passes the scalar amplitude: all +a (:57-59)
    bits = RP.eagle_bits(p.stream_bits)
    tx, _, _ = OC.tx_chain(p, bits, fast=True)
    out = []
    for seed in seeds:
        rx, _ = O.Noise(snr, tx, rng=np.random.default_rng(seed))
        Y = O.OFDM_demodulator(rx.reshape((p.Nfft + p.T_Guard, p.N_symb), order="F"), p.T_Guard)
        raw = O.demapping(-1, O.get_payload(Y, p.dataCarriers).ravel(order="F"), cname)
        out.append(float(np.mean(OC.scramble_frames(p, raw, descramble=True, fast=True) != bits)))
    return float(np.mean(out))


@pytest.mark.parametrize("cname", list(RP.BER_SNR_FIGURE))
def test_P1_ber_snr_curve_of_task3_figure(cname):
    for snr, fig in RP.BER_SNR_FIGURE[cname].items():
        ber = _task3_ber(cname, snr, seeds=range(8))
        assert abs(ber / fig - 1) < RP.ber_tolerance(fig, cname), (cname, snr, ber, fig)


def _mer_awgn(percent, seeds):
    p = OC.params_task4(percent=percent, alternate=False)
    tx, _, _ = OC.tx_chain(p, RP.eagle_bits(p.stream_bits), fast=True)
    mers = []
    for seed in seeds:
        rx, _ = O.Noise(25, tx, rng=np.random.default_rng(seed))
        Y = O.OFDM_demodulator(rx.reshape((p.Nfft + p.T_Guard, p.N_symb), order="F"), p.T_Guard)
        mers.append(O.MER_func(O.get_payload(Y, p.dataCarriers).ravel(order="F"), "16QAM"))
    a2 = (4 / 3) ** 2 * 1.8
    analytic = 25 + 10 * np.log10(p.Nfft / (len(p.dataCarriers) + len(p.pilotCarriers) * a2))
    return float(np.mean(mers)), analytic, len(p.pilotCarriers)


def test_P2_mer_at_25dB_awgn():
    mer, analytic, Np = _mer_awgn(0.25, range(6))
    assert Np == 2
    assert abs(analytic - RP.MER_AWGN_25DB) < 0.01            # 29.035 vs the README's 29.0341
    assert abs(mer - RP.MER_AWGN_25DB) < 0.08                 # single-run sigma 0.02 dB + payload-dependent 0.03 dB
    mer15, analytic15, _ = _mer_awgn(15, range(3))            # the committed script: 27.8 dB, same relation
    assert abs(mer15 - analytic15) < 0.15 and abs(mer15 - 27.8) < 0.1


def task4_mer_experiment(percent=50):
    """Noise-free 3-tap experiment of `Task 4/README.md:179-183` on the oracle.  Returns MER per interpolation method over
    the data carriers inside the uniform pilot run, and over all data carriers."""
    p = OC.params_task4(percent=percent)
    bits = RP.eagle_bits(p.stream_bits)
    tx, _, _ = OC.tx_chain(p, bits, fast=True)
    rx = OC.impair_task4(p, tx, taps=RP.TAPS_T4)
    Y = O.OFDM_demodulator(rx.reshape((p.Nfft + p.T_Guard, p.N_symb), order="F"), p.T_Guard)
    allc = np.arange(1, p.Nfft + 1)
    H_spline, Hp = O.estimate_channel(Y, allc, p.pilotCarriers, p.pilotValues)
    pc = p.pilotCarriers.astype(np.float64)
    H_lin = interp1d(pc, Hp, kind="linear", bounds_error=False, fill_value=np.nan)(allc)
    H_cub = np.full(p.Nfft, np.nan, dtype=complex)
    last_uniform = int(pc[-2])
    H_cub[:last_uniform] = RP.keys_cubic(pc[:-1], Hp[:-1], np.arange(1.0, last_uniform + 1))
    inner = p.dataCarriers[p.dataCarriers < last_uniform]

    def mer(H, rows):
        eq = O.equalize_signal(Y, H, p.N_carrier)
        return O.MER_func(eq[rows - 1, :].ravel(order="F"), p.Constellation)

    return {"linear": mer(H_lin, inner), "cubic": mer(H_cub, inner), "spline": mer(H_spline, inner),
            "linear_all": mer(H_lin, p.dataCarriers), "spline_all": mer(H_spline, p.dataCarriers)}


def test_P3_task4_mer_table():
    r = task4_mer_experiment(50)
    assert abs(r["linear"] - RP.MER_TABLE_T4["linear"]) < 0.5          # 59.8
    assert abs(r["spline"] - RP.MER_TABLE_T4["spline"]) < 0.5          # 130.1
    assert abs(r["cubic"] - RP.MER_TABLE_T4["cubic"]) < 1.5            # 106.9 (end treatment of the author's run unknown)
    assert abs(r["linear_all"] - 59.75) < 0.05 and abs(r["spline_all"] - 123.15) < 0.1
    r15 = task4_mer_experiment(15)                                     # the committed script's pilots: regression values
    assert abs(r15["linear_all"] - 42.74) < 0.05 and abs(r15["spline_all"] - 94.25) < 0.1


def test_P4_task2_papr():
    p = OC.params_task4(percent=1, scale=2.0, alternate=True)          # `Task 2/Main_model_Task_2.m:14,58` + v1 mapper
    bits = RP.eagle_bits(p.stream_bits)
    plain = O.calculatePAPR(OC.tx_chain(p, bits, scramble=False)[0])
    scr = O.calculatePAPR(OC.tx_chain(p, bits, scramble=True, fast=True)[0])
    assert abs(plain - RP.PAPR_T2["plain"]) < 1.5 and abs(scr - RP.PAPR_T2["scrambled"]) < 1.5
    assert abs(plain - 22.483) < 0.01 and abs(scr - 11.199) < 0.01     # regression values of the oracle
