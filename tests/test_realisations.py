"""Realisation import/export (SURVEY 8f rank 2): the MAT-file codec against SciPy's (checker only), the committed
golden realisation against the oracle, and the payload reader against the pinned reference payload."""
import hashlib
import json
import os

import numpy as np
import pytest

import ofdm_b200  # noqa: F401
from ofdm_b200 import realisations as R
from oracle import chains as OC

import reference_pins as RP

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_mat5_round_trip_and_scipy_interop(tmp_path):
    scipy_io = pytest.importorskip("scipy.io")
    rng = np.random.default_rng(0)
    a = {"x": rng.standard_normal((5, 3)), "z": rng.standard_normal((7, 2)) + 1j * rng.standard_normal((7, 2)), "s": 3.5, "name": "16QAM",
         "i": np.arange(9, dtype=np.int32).reshape(3, 3), "b": np.array([[True, False, True]]), "f": rng.standard_normal(4).astype(np.float32)}
    R.savemat5(tmp_path / "ours.mat", a)
    back = R.loadmat5(tmp_path / "ours.mat")
    theirs = scipy_io.loadmat(tmp_path / "ours.mat")                      # SciPy reads what we write ...
    for k in ("x", "z", "i", "f"):
        assert np.array_equal(np.asarray(back[k]).reshape(np.asarray(theirs[k]).shape), theirs[k]) and np.array_equal(np.squeeze(theirs[k]), np.squeeze(a[k]))
    assert back["name"] == "16QAM" and theirs["name"][0] == "16QAM" and back["s"][0, 0] == 3.5 and back["b"].dtype == bool
    for comp in (False, True):                                           # ... and we read what SciPy (= MATLAB's save -v6 / -v7 layout) writes
        scipy_io.savemat(tmp_path / "theirs.mat", a, do_compression=comp)
        r = R.loadmat5(tmp_path / "theirs.mat")
        for k in ("x", "z", "i", "f"):
            assert np.array_equal(np.squeeze(r[k]), np.squeeze(a[k])) and r[k].dtype == np.asarray(a[k]).dtype
        assert r["name"] == "16QAM" and np.array_equal(r["b"], a["b"])
    # integer-valued doubles stored narrow (MATLAB does this on save): class double comes back
    scipy_io.savemat(tmp_path / "n.mat", {"bits": np.array([[0, 1, 1, 0]], dtype=np.uint8)})
    assert R.loadmat5(tmp_path / "n.mat")["bits"].dtype == np.uint8
    with pytest.raises(ValueError):
        (tmp_path / "bad.mat").write_bytes(b"\x89HDF\r\n" + b"\0" * 200)
        R.loadmat5(tmp_path / "bad.mat")


def test_export_import_realisation(tmp_path):
    rng = np.random.default_rng(1)
    bits = rng.integers(0, 2, 1000).astype(np.uint8)
    normals = rng.standard_normal((300, 2))
    R.export_realisation(tmp_path / "r.mat", input_bits=bits, noise_normals=normals, channel_taps=[[0, 1], [4, .6]], Time_Delay=37, Freq_Shift=7.24, SNR_dB=25,
                         h_t=np.array([1 + 1j, 0.5j]), ref_tau=1.0)
    d = R.import_realisation(tmp_path / "r.mat")
    assert np.array_equal(d["input_bits"], bits) and d["input_bits"].dtype == np.uint8 and np.array_equal(d["noise_normals"], normals)
    assert d["Time_Delay"] == 37.0 and d["Freq_Shift"] == 7.24 and d["SNR_dB"] == 25.0 and np.array_equal(d["channel_taps"], [[0, 1], [4, .6]])
    assert np.array_equal(d["h_t"].ravel(), [1 + 1j, 0.5j])
    with pytest.raises(KeyError):
        R.export_realisation(tmp_path / "x.mat", bogus=1)
    with pytest.raises(ValueError):
        R.export_realisation(tmp_path / "x.mat", noise_normals=np.zeros((2, 300)))


def _golden():
    import importlib.util
    spec = importlib.util.spec_from_file_location("mkfix", os.path.join(GOLD, "make_realisation_fixture.py"))
    mk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mk)
    return mk, R.import_realisation(os.path.join(GOLD, "realisation_small.mat"))


def test_oracle_reproduces_the_golden_realisation():
    """The committed fixture pins the oracle: same inputs -> the stored stream, estimate, bits and error count."""
    mk, g = _golden()
    p = mk.small_params()
    tx, _, _ = OC.tx_chain(p, g["input_bits"])
    rx = OC.channel_task5(p, tx, g["SNR_dB"], g["channel_taps"], normals=g["noise_normals"].T)
    ref = OC.rx_chain_task5(p, rx, g["input_bits"])
    assert np.allclose(tx, g["ref_tx"].ravel(), rtol=0, atol=1e-13) and np.allclose(rx, g["ref_rx"].ravel(), rtol=0, atol=1e-13)
    assert np.allclose(ref["H"], g["ref_H_LS"].ravel(), rtol=1e-12, atol=1e-13)
    assert np.array_equal(ref["bits"], g["ref_bits"].ravel().astype(np.uint8)) and ref["errors"] == int(g["ref_errors"].ravel()[0]) > 0


def test_payload_reader_and_display_pic(tmp_path):
    # a synthetic 8-bit TIFF (two strips) through the baseline reader and the Otsu threshold
    import struct
    rng = np.random.default_rng(3)
    img = np.where(rng.random((20, 12)) < 0.4, rng.integers(150, 256, (20, 12)), rng.integers(0, 90, (20, 12))).astype(np.uint8)
    data = img.tobytes()
    ifd_off = 8 + len(data)
    entries = [(256, 4, 1, 12), (257, 4, 1, 20), (258, 3, 1, 8), (259, 3, 1, 1), (262, 3, 1, 1), (277, 3, 1, 1), (278, 4, 1, 10),
               (273, 4, 2, ifd_off + 2 + 9 * 12 + 4), (279, 4, 2, ifd_off + 2 + 9 * 12 + 4 + 8)]
    ifd = struct.pack("<H", len(entries)) + b"".join(struct.pack("<HHII", *e) for e in entries) + struct.pack("<I", 0)
    extra = struct.pack("<II", 8, 8 + 120) + struct.pack("<II", 120, 120)
    (tmp_path / "t.tiff").write_bytes(b"II*\0" + struct.pack("<I", ifd_off) + data + ifd + extra)
    assert np.array_equal(R.read_tiff_gray8(tmp_path / "t.tiff"), img)
    bits = R.file_reader(tmp_path / "t.tiff", 100)
    assert bits.shape == (100,) and np.array_equal(bits, (img > 120).ravel(order="F")[:100].astype(np.uint8))   # bimodal image: any threshold in the gap
    with pytest.raises(IndexError):
        R.file_reader(tmp_path / "t.tiff", 241)
    pic = R.display_pic(bits, side=12)
    assert pic.shape == (12, 12) and pic.dtype == np.uint8 and np.array_equal((pic.ravel(order="F")[:100] // 255), bits) and not pic.ravel(order="F")[100:].any()


def test_file_reader_on_the_reference_payload(tmp_path):
    d = json.load(open(os.path.join(GOLD, "eagle_bits_digest.json")))
    eagle = RP.write_eagle_tiff(tmp_path / "eagle.tiff")
    bits = R.file_reader(eagle, d["n_bits"])
    assert int(bits.sum()) == d["n_ones"] and "".join(map(str, bits[:64])) == d["first_64"]
    assert hashlib.sha256(np.packbits(bits).tobytes()).hexdigest() == d["sha256_of_packbits"]
    assert np.array_equal(bits, OC.read_payload_bits(eagle, d["n_bits"]))
