"""Multi-rank path of the Task-3 MER study on CPU: world sizes 2 and 3 over `gloo` run the host logic of ``sweep.mer_sweep``
(share rule, disjoint per-stream MER sums, one all_reduce each of the float64 sums and the int64 counters, the host
statistics) with a stand-in compute -- the product has no CPU compute path.  Points of different constellations carry
different bits per stream, and the tiles are ragged.  Every rank must hold exactly the world-1 result."""
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from ofdm_b200 import sweep

POINTS = [("BPSK", 0.0), ("QPSK", 5.0), ("8PSK", 10.0), ("16QAM", 15.0), ("16QAM", np.inf)]
BPS = {"BPSK": 1, "QPSK": 2, "8PSK": 3, "16QAM": 4}
SPP, TILE = 29, 8               # ragged: four tiles per point, the last one of 5 streams
STREAM_SYMBOLS = 50 * 332


def fake_compute(k, point, s0, n):
    """MER sums per stream keyed by the global stream id only (as the Philox-keyed GPU path is), with varied exponents so
    that any re-association of the sums would show; counters that depend on the point's bits per stream."""
    cname, snr = point
    g = k * SPP + s0 + np.arange(n)
    frac = ((g * 2654435761) % 1000003) / 1000003.0
    f0 = STREAM_SYMBOLS * (1.0 + frac * 1e-3)
    f1 = f0 * 10.0 ** (-(min(snr, 120.0) + 3 * frac) / 10.0)
    bits = STREAM_SYMBOLS * BPS[cname] * n
    errs = 0 if snr > 100 else int(np.sum((g * 40503) % 997))
    return np.stack([f0, f1]), (errs, bits, int(np.sum(g % 5 == 0)))


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
        res = sweep.run_mer_sweep(POINTS, SPP, TILE, fake_compute, rank, world)
        np.savez(os.path.join(out_dir, f"res{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


def test_world1_statistics_against_numpy():
    res = sweep.run_mer_sweep(POINTS, SPP, TILE, fake_compute, 0, 1)
    assert res["mer"].shape == (len(POINTS), 2, SPP) and res["counts"].shape == (len(POINTS), 3)
    for k, pt in enumerate(POINTS):
        m, c = fake_compute(k, pt, 0, SPP)                      # the whole point as one tile: the same cells
        assert np.array_equal(res["mer"][k], m) and np.array_equal(res["counts"][k], c)
        assert res["counts"][k, 1] == SPP * STREAM_SYMBOLS * BPS[pt[0]]
        assert res["ber"][k] == c[0] / c[1] and res["near"][k] == c[2]
        s0 = s1 = 0.0
        for j in range(SPP):                                    # the pooled MER sums in stream order
            s0 += m[0, j]
            s1 += m[1, j]
        assert res["mer_db"][k] == 10 * np.log10(s0 / s1)
        per = 10 * np.log10(m[0] / m[1])
        assert np.array_equal(res["per_stream_db"][k], per)
        assert np.isclose(res["mer_stream_db"][k], per.mean(), rtol=1e-12)
    assert res["ber"][-1] == 0


def test_mer_params_per_point_fields():
    mp_ = sweep.mer_params(["BPSK", "16QAM"], [3.0, 9.0], 17, [[0, 1], [4, .6]], seed=5, rank=1, world=2, tile=3, pilot_scale=4 / 3,
                           sto=[0, 5], cfo=0.1, near_eps=1e-3)
    assert mp_.n_points == 2 and [mp_.constellation_host[i] for i in range(2)] == [1, 4]
    assert [mp_.nsto_host[i] for i in range(2)] == [0, 5] and [mp_.cfo_host[i] for i in range(2)] == [0.1, 0.1]
    assert mp_.n_taps == 2 and mp_.streams_per_point == 17 and (mp_.rank, mp_.world, mp_.tile_streams) == (1, 2, 3)
    assert bool(mp_.nsto_host) and not bool(sweep.mer_params("QPSK", [1.0], 4).nsto_host)   # NULL: STO 0 at every point
    with pytest.raises(ValueError):
        sweep.mer_params(["BPSK"], [1.0, 2.0], 4)


@pytest.mark.parametrize("world", [2, 3])
def test_mer_sweep_independent_of_rank_count(tmp_path, world):
    one = sweep.run_mer_sweep(POINTS, SPP, TILE, fake_compute, 0, 1)
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        got = np.load(tmp_path / f"res{r}.npz")
        assert set(got.files) == set(one)
        for k in one:                                           # bit-identical on every rank
            assert np.array_equal(got[k], one[k]), k
