"""Multi-rank path of the MSE sweep on CPU: world sizes 2 and 3 over `gloo` run the host logic of ``sweep.mse_sweep``
(share rule, disjoint per-stream cells, one all_reduce each of the float64 array and the int64 counters, host mean) with a
stand-in compute -- the product has no CPU compute path.  Every rank must hold exactly the world-1 result."""
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from ofdm_b200 import sweep

SNRS = [0.0, 7.5, 15.0, 30.0]
SPP, TILE = 29, 8         # ragged: four tiles per point, the last one of 5 streams


def fake_compute(i, snr_db, s0, n):
    """Float per-stream values keyed by the global stream id only (as the Philox-keyed GPU path is), with varied exponents
    so that any re-association in the reduction would show."""
    g = i * SPP + s0 + np.arange(n)
    frac = ((g * 2654435761) % 1000003) / 1000003.0
    m = np.stack([(1.0 + frac) * 10.0 ** (-snr_db / 10.0 - e) for e in range(4)])
    return m, (n, int(np.sum(g % 7 == 0)))


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
        mean, per, counts = sweep.run_mse_sweep(SNRS, SPP, TILE, fake_compute, rank, world)
        np.save(os.path.join(out_dir, f"mean{rank}.npy"), mean)
        np.save(os.path.join(out_dir, f"per{rank}.npy"), per)
        np.save(os.path.join(out_dir, f"counts{rank}.npy"), counts)
    finally:
        dist.destroy_process_group()


def test_world1_fills_every_cell_once():
    mean, per, counts = sweep.run_mse_sweep(SNRS, SPP, TILE, fake_compute, 0, 1)
    assert per.shape == (len(SNRS), 4, SPP) and mean.shape == (len(SNRS), 4) and counts.shape == (len(SNRS), 2)
    assert np.all(per > 0)
    for i in range(len(SNRS)):
        m, c = fake_compute(i, SNRS[i], 0, SPP)                 # the whole point as one tile: the same cells
        assert np.array_equal(per[i], m) and counts[i, 0] == SPP and counts[i, 1] == c[1]
    assert np.array_equal(mean, per.mean(axis=2))


@pytest.mark.parametrize("world", [2, 3])
def test_mse_sweep_independent_of_rank_count(tmp_path, world):
    mean1, per1, counts1 = sweep.run_mse_sweep(SNRS, SPP, TILE, fake_compute, 0, 1)
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        assert np.array_equal(np.load(tmp_path / f"per{r}.npy"), per1)          # bit-identical on every rank
        assert np.array_equal(np.load(tmp_path / f"mean{r}.npy"), mean1)
        assert np.array_equal(np.load(tmp_path / f"counts{r}.npy"), counts1)
