"""Multi-rank path of the sync sweep on CPU: world sizes 2 and 3 over `gloo` run the host logic of ``sweep.sync_sweep``
(share rule, disjoint per-stream records, one all_reduce each of the float64 records and the int64 counters, the host
statistics) with a stand-in compute -- the product has no CPU compute path.  Every rank must hold exactly the world-1
result, NaN cells included."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from ofdm_b200 import sweep

SNRS = [0.0, 5.0, 10.0, 15.0]
SPP, TILE, SL = 31, 8, 1152     # ragged: four tiles per point, the last one of 7 streams


def fake_compute(i, snr_db, s0, n):
    """A record per stream keyed by the global stream id only (as the Philox-keyed GPU path is): detector fallbacks and NaN
    channel errors at the low points, IFO misses, varied exponents so that any re-association would show."""
    g = i * SPP + s0 + np.arange(n)
    frac = ((g * 2654435761) % 1000003) / 1000003.0
    fail = (snr_db < 5) & (g % 3 != 0)
    tg = np.where(fail, 65.0, 1000.0 + (g % 13))
    ifo = np.where(g % 11 == 0, -1.0, 0.0)
    cfo = (g % 31) + frac - 0.5
    fo = cfo - np.maximum(ifo, 0) + (frac - 0.5) * 10.0 ** (-snr_db / 20.0 - 1)
    herr = np.where(fail & (g % 2 == 0), np.nan, (1.0 + frac) * 10.0 ** (-snr_db / 10.0 - 2))
    rec = np.stack([tg, fo, ifo, frac * 1e-3, frac - 0.5, herr, snr_db + 5 * frac, (g * 7) % 1153, cfo])
    errs = int(np.sum((g * 40503) % 1000))
    return rec, (errs, 66400 * n, int(fail.sum()), int((ifo == -1).sum()))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        res = sweep.run_sync_sweep(SNRS, SPP, TILE, fake_compute, rank, world, h_power=1.41, sym_len=SL)
        np.savez(os.path.join(out_dir, f"res{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


def test_world1_statistics():
    res = sweep.run_sync_sweep(SNRS, SPP, TILE, fake_compute, 0, 1, h_power=1.41, sym_len=SL)
    rec = res["rec"]
    assert rec.shape == (len(SNRS), 9, SPP) and res["counts"].shape == (len(SNRS), 4)
    for i in range(len(SNRS)):
        r, c = fake_compute(i, SNRS[i], 0, SPP)                 # the whole point as one tile: the same cells
        assert np.array_equal(rec[i], r, equal_nan=True) and np.array_equal(res["counts"][i], c)
        herr = r[5]
        assert res["h_err_nan"][i] == np.isnan(herr).sum()
        assert np.isclose(res["h_err_mean"][i], np.nanmean(herr)) and np.isclose(res["nmse"][i], np.nanmean(herr) / 1.41)
        e = r[1] + np.maximum(r[2], 0) - r[8]
        assert np.isclose(res["cfo_err_rms"][i], np.sqrt(np.mean(e ** 2)))
        assert res["timing_max"][i] == np.max((r[7] + r[0]) % SL)
        assert res["fail_rate"][i] == c[2] / SPP and res["ifo_miss_rate"][i] == c[3] / SPP
    assert res["h_err_nan"][0] > 0 and res["h_err_nan"][-1] == 0


def test_share_rule_matches_library():
    """sweep.share / sweep.tiles against ofdm_sweep_share, which needs no device (skipped without the built library)."""
    from ofdm_b200 import _cabi
    try:
        lib = _cabi.load()
    except (RuntimeError, OSError) as e:
        pytest.skip(f"library not built: {e}")
    for total in (0, 1, 7, 124, 4096 * 61 + 3):
        for world in (1, 2, 3, 7):
            for rank in range(world):
                first, count = C.c_int64(), C.c_int64()
                assert lib.ofdm_sweep_share(total, rank, world, C.byref(first), C.byref(count)) == 0
                assert sweep.share(total, rank, world) == (first.value, count.value)


@pytest.mark.parametrize("world", [2, 3])
def test_sync_sweep_independent_of_rank_count(tmp_path, world):
    one = sweep.run_sync_sweep(SNRS, SPP, TILE, fake_compute, 0, 1, h_power=1.41, sym_len=SL)
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        got = np.load(tmp_path / f"res{r}.npz")
        assert set(got.files) == set(one)
        for k in one:                                           # bit-identical on every rank, NaN cells included
            assert np.array_equal(got[k], one[k], equal_nan=np.asarray(one[k]).dtype.kind == "f"), k
