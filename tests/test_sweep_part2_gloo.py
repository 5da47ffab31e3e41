"""Host logic of ``part2.sweep_lib`` on CPU: the layout, Ldict and pilot pattern it hands to ``ofdm_sweep_part2`` are those of
the composed driver, the share rule is the library's, and at world sizes 2 and 3 over `gloo` the reduction (disjoint per-run
cells, one all_reduce each of the per-run array, the counts and the runs) matches world 1 bit for bit -- with a stand-in
compute, since the product has no CPU compute path."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import ofdm_b200  # noqa: F401
from ofdm_b200 import part2, sweep

N_POINTS, RUNS, TILE = 5, 23, 6          # ragged: four tiles per point, the last one of 5 runs


def run_part2_sweep(n_points, mc_runs, tile, compute, rank=0, world=1):
    """The host side of ``part2.sweep_lib`` around a stand-in ``compute(point, first_run, n_runs) -> (nmse[4, n_runs],
    counts[4, 3], runs[2])`` for one tile: this rank's tiles (``sweep.tiles``, the tiling of ofdm_sweep_part2), disjoint
    per-run cells, then ``part2.reduce_part2``."""
    per = torch.zeros((n_points, 4, mc_runs), dtype=torch.float64)
    counts = torch.zeros((n_points, 4, 3), dtype=torch.int64)
    runs = torch.zeros((n_points, 2), dtype=torch.int64)
    for (k, r0, n) in sweep.tiles(n_points, mc_runs, tile, rank, world):
        m, c, r = compute(k, r0, n)
        per[k, :, r0:r0 + n] = torch.as_tensor(np.asarray(m, dtype=np.float64))
        counts[k] += torch.as_tensor(np.asarray(c, dtype=np.int64))
        runs[k] += torch.as_tensor(np.asarray(r, dtype=np.int64))
    return part2.reduce_part2(per, counts, runs)


def fake_compute(k, r0, n):
    """Per-run values keyed by the global item only (as the Philox-keyed GPU path is), with varied exponents so that any
    re-association in the reduction would show; integer counters summed per point."""
    g = k * RUNS + r0 + np.arange(n)
    frac = ((g * 2654435761) % 1000003) / 1000003.0
    m = np.stack([(1.0 + frac) * 10.0 ** (-k - e) for e in range(4)])
    c = np.array([[int(np.sum((g * 7 + e) % 5)), n * 1000, int(np.sum(g % (e + 2) == 0))] for e in range(4)])
    return m, c, (n, int(np.sum(g % 7 == 0)))


def test_layout_matches_the_composed_driver():
    combs, _ = part2.part2_combs()
    off, car, ldict = part2.lib_layout(combs)
    assert off[0] == 0 and off.size == 58 and ldict.size == 57
    for k, comb in enumerate(combs):
        pc, dc = part2.layout(1024, comb=int(comb))
        assert np.array_equal(car[off[k]:off[k + 1]], pc)
        assert ldict[k] == -(-4096 // int(comb))
        assert np.array_equal(np.setdiff1d(np.arange(1, 1025), car[off[k]:off[k + 1]]), dc)
    rng = np.random.default_rng(4)
    masks = [np.sort(rng.permutation(1024)[:64]) + 1, np.sort(rng.permutation(1024)[:200]) + 1]
    off, car, ldict = part2.lib_layout([0, 0], reg_pilot=False, random_masks=masks)
    for k in range(2):
        assert np.array_equal(car[off[k]:off[k + 1]], part2.layout(1024, pilotCarriers=masks[k])[0])
    assert np.array_equal(ldict, [4096, 4096])


@pytest.mark.parametrize("Np", [4, 256, 255])
def test_pilot_pattern_is_the_composed_pilot_grid(Np):
    amp = 2.0 * 3 * np.sqrt(2) / np.sqrt(10)
    pat = part2.pilot_pattern(amp)
    pv = part2.pilot_values(Np, 14, amp)
    assert pat.dtype == np.complex128 and pat[1].imag != 0            # the exp(1i*pi) residue is kept
    for q in range(Np):
        assert np.all(pv[q] == pat[q % 2])


def test_share_rule_is_the_librarys():
    from ofdm_b200 import _cabi
    lib = _cabi.load()
    first, count = C.c_int64(), C.c_int64()
    for total in (1, 57, 5700, 57 * 4096 + 3):
        for world in (1, 2, 3, 8):
            for rank in range(world):
                assert lib.ofdm_sweep_share(total, rank, world, C.byref(first), C.byref(count)) == 0
                assert (first.value, count.value) == sweep.share(total, rank, world)


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
        for name, a in zip(("nmse", "ber", "per", "counts", "runs"), run_part2_sweep(N_POINTS, RUNS, TILE, fake_compute, rank, world)):
            np.save(os.path.join(out_dir, f"{name}{rank}.npy"), a)
    finally:
        dist.destroy_process_group()


def test_world1_fills_every_cell_once():
    NMSE, BER, per, counts, runs = run_part2_sweep(N_POINTS, RUNS, TILE, fake_compute)
    assert NMSE.shape == (4, N_POINTS) and BER.shape == (4, N_POINTS) and per.shape == (N_POINTS, 4, RUNS)
    assert np.all(per > 0) and np.all(runs[:, 0] == RUNS)
    for k in range(N_POINTS):
        m, c, r = fake_compute(k, 0, RUNS)                             # the whole point as one tile: the same cells and sums
        assert np.array_equal(per[k], m) and np.array_equal(counts[k], c) and runs[k, 1] == r[1]
    assert np.allclose(NMSE, per.mean(axis=2).T, rtol=1e-15, atol=0)
    assert np.array_equal(BER, (counts[:, :, 0] / counts[:, :, 1]).T)


@pytest.mark.parametrize("world", [2, 3])
def test_part2_lib_reduction_independent_of_rank_count(tmp_path, world):
    want = run_part2_sweep(N_POINTS, RUNS, TILE, fake_compute)
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        for name, a in zip(("nmse", "ber", "per", "counts", "runs"), want):
            assert np.array_equal(np.load(tmp_path / f"{name}{r}.npy"), a), (name, r)
