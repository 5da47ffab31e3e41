"""Multi-rank path of the PAPR study on CPU: world sizes 2 and 3 over `gloo` run the host logic of ``sweep.papr_sweep``
(share rule, tiles, the integer histogram and the disjoint per-stream PAPR cells, one all_reduce each) with a stand-in
compute -- the product has no CPU compute path.  Every rank must hold exactly the world-1 result.  The CCDF and the
exceedance read from a histogram are checked against numpy on synthetic values."""
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from ofdm_b200 import sweep

POINTS = [(0, 0.05), (1, 0.05), (0, 0.5), (1, 0.5)]
SPP, TILE, NB, BIN = 29, 8, 700, 0.05     # ragged: four tiles per point, the last one of 5 streams
WINDOWS = 40                              # stand-in windows per stream


def _values(k, g):
    """Stand-in window PAPR values of the streams with global ids g (keyed by g only, as the Philox-keyed GPU path is);
    some land in the overflow bin."""
    frac = ((g[:, None] * 2654435761 + np.arange(WINDOWS) * 40503) % 1000003) / 1000003.0
    return 4.0 + 35.0 * frac ** (1 + k)


def fake_compute(k, point, s0, n):
    g = k * SPP + s0 + np.arange(n)
    v = _values(k, g)
    b = np.minimum(np.floor(v / BIN), NB - 1).astype(np.int64)
    return np.bincount(b.ravel(), minlength=NB), v.max(axis=1) - v.mean(axis=1)


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
        res = sweep.run_papr_sweep(POINTS, SPP, TILE, fake_compute, rank, world, n_bins=NB, bin_db=BIN)
        np.savez(os.path.join(out_dir, f"res{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


def test_world1_and_tiles():
    res = sweep.run_papr_sweep(POINTS, SPP, TILE, fake_compute, 0, 1, n_bins=NB, bin_db=BIN)
    assert res["hist"].shape == (len(POINTS), NB) and res["papr"].shape == (len(POINTS), SPP)
    for k in range(len(POINTS)):
        h, p = fake_compute(k, POINTS[k], 0, SPP)              # the whole point as one tile
        assert np.array_equal(res["hist"][k], h) and np.array_equal(res["papr"][k], p)
        assert res["hist"][k].sum() == SPP * WINDOWS and res["papr_mean"][k] == p.mean()
    assert np.array_equal(res["edges"], np.arange(NB) * BIN)
    assert res["hist"][:, -1].sum() > 0                        # the overflow bin is used
    for tile in (1, 5, 100):
        other = sweep.run_papr_sweep(POINTS, SPP, tile, fake_compute, 0, 1, n_bins=NB, bin_db=BIN)
        assert all(np.array_equal(other[key], res[key]) for key in res), tile


def test_ccdf_and_exceedance_match_numpy():
    rng = np.random.default_rng(7)
    v = np.concatenate([rng.gamma(4.0, 2.0, 50000), [100.0, 250.0]])      # two values far above the last edge
    nb, bw = 2000, 0.025
    b = np.minimum(np.floor(v / bw), nb - 1).astype(np.int64)
    h = np.bincount(b, minlength=nb)
    c = sweep.papr_ccdf(h)
    edges = np.arange(nb) * bw
    # the CCDF at an edge is the fraction of values at or above it, except that the last bin holds everything above
    want = np.array([np.mean(b >= i) for i in range(nb)])
    assert np.allclose(c, want, rtol=0, atol=1e-15)
    assert np.allclose(c[:-1], [np.mean(v >= e) for e in edges[:-1]], rtol=0, atol=1e-15)
    assert c[-1] == np.mean(v >= edges[-1]) and c[0] == 1.0
    for prob in (0.5, 0.02, 1e-3, 1e-4):
        ex = sweep.papr_exceedance(h, bw, prob)
        i = int(round(ex / bw))
        assert c[i] <= prob and (i == 0 or c[i - 1] > prob)
        # against the ecdf reading (the smallest value whose CCDF is <= prob): at most one bin above it
        xs = np.sort(v)
        ccdf = 1.0 - np.arange(1, v.size + 1) / v.size
        ref = xs[np.argmax(ccdf <= prob)]
        if ref < edges[-1]:
            assert ref < ex <= ref + bw + 1e-12, (prob, ex, ref)
    assert sweep.papr_exceedance(h, bw, 1e-9) == nb * bw                 # never reached inside the histogram
    two = np.stack([h, h[::-1]])
    assert np.array_equal(sweep.papr_exceedance(two, bw, 0.02), [sweep.papr_exceedance(h, bw, 0.02), sweep.papr_exceedance(h[::-1], bw, 0.02)])


@pytest.mark.parametrize("world", [2, 3])
def test_papr_sweep_independent_of_rank_count(tmp_path, world):
    one = sweep.run_papr_sweep(POINTS, SPP, TILE, fake_compute, 0, 1, n_bins=NB, bin_db=BIN)
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        got = np.load(tmp_path / f"res{r}.npz")
        assert set(got.files) == set(one)
        for k in one:
            assert np.array_equal(got[k], one[k]), k
