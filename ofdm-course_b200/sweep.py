"""Monte-Carlo BER-vs-SNR and channel-estimation MSE-vs-SNR sweeps sharded over ranks (SURVEY 8e; loop shape of
`Task 3/Main_model_Task_3.m:192-268`, `Task 5/Main_model_Task_5.m:303-346`, and the Task-4 impaired channel
`Task 4/Main_model_Task_4.m:95-110,277-366` swept over SNR).

The compute is ONE C-ABI call per rank, ``ofdm_sweep_ber`` (csrc/sweep.cu): global stream g = snr_index *
streams_per_point + j; rank r of R takes the contiguous share [T r / R, T (r+1) / R) of the T = n_snr * streams_per_point
streams (equal to within one stream for any R) -- **no data-path collective**; the only exchange is one
``all_reduce(SUM)`` of the int64 counters at the end (NCCL on GPUs; the same host logic runs over ``gloo`` in the CPU
tests with a stand-in compute function).  Payload bits, noise, STO and CFO draws are Philox streams keyed by g, so the
counters do not depend on the number of ranks.

``mse_sweep`` is the channel-estimation half of `Task 5/Main_model_Task_5.m:303-346` (LS / MMSE / MP / OMP MSE per stream,
``ofdm_sweep_mse`` in csrc/sweep_mse.cu) on the same share rule; its per-stream float64 array is summed over the ranks,
which is exact because every cell is written by exactly one rank.

``sync_sweep`` is Task 4's own study (``ofdm_sweep_sync`` in csrc/sweep_sync.cu): the synchroniser's estimates, the
channel-estimate error and the MER of every stream of the Task-4 chain, one record per stream, reduced the same way.

``papr_sweep`` is Task 2's study (``ofdm_sweep_papr`` in csrc/sweep_papr.cu): the PAPR of every transmitted stream and an
integer histogram of the PAPR of all its Nfft-sample windows, plain against scrambled, one all-reduce each.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from . import _cabi
from .part2 import ESTIMATORS  # noqa: F401  (order of the estimator axis: LS, MMSE, MP, OMP)

CHAINS = {"task5": 0, "task4": 1}


def share(total_streams, rank, world):
    """(first, count) of the contiguous share of the global stream range -- the rule of ``ofdm_sweep_share``."""
    lo, hi = total_streams * rank // world, total_streams * (rank + 1) // world
    return lo, hi - lo


def tiles(n_snr, streams_per_point, tile, rank=0, world=1):
    """The work items of one rank: (snr_index, first_stream_within_point, n_streams), never straddling an SNR point."""
    first, count = share(n_snr * streams_per_point, rank, world)
    out, g, end = [], first, first + count
    while g < end:
        i = g // streams_per_point
        n = min(tile, end - g, (i + 1) * streams_per_point - g)
        out.append((i, g - i * streams_per_point, n))
        g += n
    return out


def all_reduce_sum(*tensors):
    """Sum each tensor in place over all ranks (no-op without an initialised process group of more than one rank)."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        for t in tensors:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)


def reduce_counts(counts, device=None):
    """Sum an int64 counter tensor over all ranks (no-op without an initialised process group)."""
    t = counts if isinstance(counts, torch.Tensor) else torch.as_tensor(np.asarray(counts), dtype=torch.int64)
    if device is not None:
        t = t.to(device)
    all_reduce_sum(t)
    return t


def run_sweep(snrs_db, streams_per_point, tile, compute, rank=0, world=1, device=None, n_counters=4):
    """Generic host driver (used with a stand-in ``compute`` in the gloo tests).
    ``compute(snr_index, snr_db, first_stream, n_streams) -> n_counters ints`` processes one tile on this rank; returns an
    int64 array (n_snr, n_counters) identical on every rank."""
    snrs_db = list(snrs_db)
    local = np.zeros((len(snrs_db), n_counters), dtype=np.int64)
    for (i, s0, n) in tiles(len(snrs_db), streams_per_point, tile, rank, world):
        local[i] += np.asarray(compute(i, snrs_db[i], s0, n), dtype=np.int64)
    return reduce_counts(torch.from_numpy(local), device).cpu().numpy()


def sweep_local(ctx, lp, snrs_db, streams_per_point, taps=None, chain="task5", seed=1, rank=0, world=1, tile=0, near_eps=0.0,
                sto_max=None, cfo_int_max=30, counts=None):
    """This rank's share of the sweep through ``ofdm_sweep_ber``; returns the device counters (n_snr, 4) int64
    {errors, bits, near-boundary symbols, detector failures} WITHOUT synchronising (everything is stream-ordered)."""
    snr = np.ascontiguousarray(np.asarray(snrs_db, dtype=np.float64))
    sp = _cabi.SweepParams()
    sp.chain = CHAINS[chain]
    sp.n_snr = snr.size
    sp.snr_db_host = snr.ctypes.data_as(_cabi.pdbl)
    sp.streams_per_point = int(streams_per_point)
    sp.tile_streams = int(tile)
    sp.rank, sp.world = int(rank), int(world)
    sp.seed = int(seed)
    t = None
    if taps is not None:
        t = np.ascontiguousarray(np.asarray(taps, dtype=np.float64).reshape(-1, 2))
        sp.taps_host = t.ctypes.data_as(_cabi.pdbl)
        sp.n_taps = t.shape[0]
    sp.near_eps = float(near_eps)
    sp.sto_max = int(lp.Nfft + lp.Tg if sto_max is None else sto_max)
    sp.cfo_int_max = int(cfo_int_max)
    if counts is None:
        counts = torch.zeros((snr.size, 4), dtype=torch.int64, device=ctx.device)
    ctx._chk(ctx.lib.ofdm_sweep_ber(ctx.h, C.byref(lp), C.byref(sp), ctx.p(counts)))
    return counts


def ber_sweep(ctx, lp, snrs_db, streams_per_point, taps=None, chain="task5", seed=1, rank=0, world=1, tile=0, near_eps=0.0, **kw):
    """Whole sweep: this rank's share on its GPU, then the closing all-reduce.  Returns (n_snr, 4) int64 on the host,
    identical on every rank and for every world size."""
    acc = sweep_local(ctx, lp, snrs_db, streams_per_point, taps, chain, seed, rank, world, tile, near_eps, **kw)
    if world > 1:
        reduce_counts(acc)                      # NCCL all-reduce on the device tensor, ordered after the sweep's stream work
    ctx.sync()
    return acc.cpu().numpy()


def reduce_mse(per_stream, counts):
    """Sum the per-stream MSE array (n_snr, 4, streams_per_point) float64 and the counters (n_snr, 2) int64 over all ranks
    (no-op without an initialised process group) and take the mean over the streams of each point on the host.
    Returns (mean[n_snr, 4], per_stream, counts) as NumPy arrays, identical on every rank."""
    all_reduce_sum(per_stream, counts)                        # exact: every cell is non-zero on one rank only
    per = per_stream.cpu().numpy()
    return per.mean(axis=2), per, counts.cpu().numpy()


def run_mse_sweep(snrs_db, streams_per_point, tile, compute, rank=0, world=1):
    """Generic host driver of the MSE sweep (used with a stand-in ``compute`` in the gloo tests).
    ``compute(snr_index, snr_db, first_stream, n_streams) -> (mse[4, n_streams], (streams, near_ties))`` processes one tile
    on this rank; the result is that of :func:`reduce_mse`."""
    snrs_db = list(snrs_db)
    per = torch.zeros((len(snrs_db), 4, int(streams_per_point)), dtype=torch.float64)
    counts = torch.zeros((len(snrs_db), 2), dtype=torch.int64)
    for (i, s0, n) in tiles(len(snrs_db), streams_per_point, tile, rank, world):
        m, c = compute(i, snrs_db[i], s0, n)
        per[i, :, s0:s0 + n] = torch.as_tensor(np.asarray(m, dtype=np.float64))
        counts[i] += torch.as_tensor(np.asarray(c, dtype=np.int64))
    return reduce_mse(per, counts)


def mse_sweep_local(ctx, lp, snrs_db, streams_per_point, taps, Ldict=None, seed=1, rank=0, world=1, tile=0, tie_eps=0.0, per_stream=None, counts=None):
    """This rank's share of the MSE sweep through ``ofdm_sweep_mse``, WITHOUT synchronising: writes its cells of
    ``per_stream`` (n_snr, 4, streams_per_point) float64 and adds to ``counts`` (n_snr, 2) int64 {streams, OMP frames with a
    near-tie}; both are zero-initialised device tensors when not given.  ``Ldict`` defaults to the script's
    ceil(N_carrier / comb) (`Main_model_Task_5.m:182-190`)."""
    snr = np.ascontiguousarray(np.asarray(snrs_db, dtype=np.float64))
    pc = np.asarray(lp.pilotCarriers)
    if Ldict is None:
        Ldict = -(-int(lp.N_carrier) // int(pc[1] - pc[0]))
    sp = _cabi.SweepParams()
    sp.chain = CHAINS["task5"]
    sp.n_snr = snr.size
    sp.snr_db_host = snr.ctypes.data_as(_cabi.pdbl)
    sp.streams_per_point = int(streams_per_point)
    sp.tile_streams = int(tile)
    sp.rank, sp.world = int(rank), int(world)
    sp.seed = int(seed)
    t = np.ascontiguousarray(np.asarray(taps, dtype=np.float64).reshape(-1, 2))
    sp.taps_host = t.ctypes.data_as(_cabi.pdbl)
    sp.n_taps = t.shape[0]
    sp.near_eps = float(tie_eps)
    if per_stream is None:
        per_stream = torch.zeros((snr.size, 4, int(streams_per_point)), dtype=torch.float64, device=ctx.device)
    if counts is None:
        counts = torch.zeros((snr.size, 2), dtype=torch.int64, device=ctx.device)
    ctx._chk(ctx.lib.ofdm_sweep_mse(ctx.h, C.byref(lp), C.byref(sp), int(Ldict), ctx.p(per_stream), ctx.p(counts)))
    return per_stream, counts


def mse_sweep(ctx, lp, snrs_db, streams_per_point, taps, Ldict=None, seed=1, rank=0, world=1, tile=0, tie_eps=0.0):
    """Whole MSE-vs-SNR sweep: this rank's call, then one all-reduce each of the per-stream array and the counters.
    Returns (mean[n_snr, 4], per_stream[n_snr, 4, streams_per_point], counts[n_snr, 2]) on the host, estimators in the
    order LS, MMSE, MP, OMP; identical on every rank and for every world size and tile."""
    per, cnt = mse_sweep_local(ctx, lp, snrs_db, streams_per_point, taps, Ldict, seed, rank, world, tile, tie_eps)
    ctx.sync()
    return reduce_mse(per, cnt)                 # NCCL all-reduce on the device tensors when world > 1


SYNC_FIELDS = ("TgPosition", "FreqOffset", "IFO", "tau", "phase_shift", "h_err", "mer_db", "nsto", "cfo")


def channel_power(taps, Nfft, N_carrier):
    """mean |H(k)|^2 over k = 1..N_carrier of H = fft(h, Nfft) (`get_MP_channel_resp.m:2-19`, later rows overwrite); 1 without
    multipath.  The denominator of the NMSE that :func:`reduce_sync` reports."""
    if taps is None or len(taps) == 0:
        return 1.0
    t = np.asarray(taps, dtype=np.float64).reshape(-1, 2)
    h = np.zeros(int(t[:, 0].max()) + 1)
    for d, a in t:
        h[int(d)] = a
    H = np.fft.fft(h, int(Nfft))[:int(N_carrier)]
    return float(np.mean(np.abs(H) ** 2))


def reduce_sync(rec, counts, h_power=1.0, sym_len=1152, cfo_tol=0.02):
    """Sum the per-stream records (n_snr, 9, streams_per_point) float64 and the counters (n_snr, 4) int64 over all ranks -- one
    all-reduce each, exact because every record cell is written by one rank (no-op without an initialised process group) --
    then form the per-point statistics on the host.  Returns a dict of NumPy arrays over the SNR points, identical on every
    rank:
      ber, fail_rate (guard-interval detector fell back to TgPosition 65), ifo_miss_rate (IFO = -1);
      cfo_err_mean / cfo_err_rms / cfo_within: the CFO error FreqOffset + max(IFO, 0) - cfo, and the fraction of streams with
      |error| <= cfo_tol;
      timing_mean / timing_std / timing_min / timing_max: the residual (nsto + TgPosition) mod sym_len;
      h_err_mean over the non-NaN cells, h_err_nan (NaN cells), nmse = h_err_mean / h_power;
      mer_db: mean of the finite per-stream MER values in dB;
    plus ``rec`` and ``counts`` themselves."""
    all_reduce_sum(rec, counts)
    r = rec.cpu().numpy()
    c = counts.cpu().numpy()
    n = r.shape[2]
    tg, fo, ifo, herr, mer, nsto, cfo = (r[:, SYNC_FIELDS.index(f), :] for f in ("TgPosition", "FreqOffset", "IFO", "h_err", "mer_db", "nsto", "cfo"))
    e = fo + np.maximum(ifo, 0) - cfo
    t = np.mod(nsto + tg, sym_len)
    ok = ~np.isnan(herr)
    n_ok = ok.sum(axis=1)
    h_mean = np.where(n_ok > 0, np.where(ok, herr, 0.0).sum(axis=1) / np.maximum(n_ok, 1), np.nan)
    fin = np.isfinite(mer)
    mer_db = np.where(fin.sum(axis=1) > 0, np.where(fin, mer, 0.0).sum(axis=1) / np.maximum(fin.sum(axis=1), 1), np.nan)
    return {
        "ber": c[:, 0] / np.maximum(c[:, 1], 1), "fail_rate": c[:, 2] / n, "ifo_miss_rate": c[:, 3] / n,
        "cfo_err_mean": e.mean(axis=1), "cfo_err_rms": np.sqrt(np.mean(e ** 2, axis=1)), "cfo_within": np.mean(np.abs(e) <= cfo_tol, axis=1),
        "timing_mean": t.mean(axis=1), "timing_std": t.std(axis=1), "timing_min": t.min(axis=1), "timing_max": t.max(axis=1),
        "h_err_mean": h_mean, "h_err_nan": (~ok).sum(axis=1), "nmse": h_mean / h_power, "mer_db": mer_db,
        "rec": r, "counts": c,
    }


def run_sync_sweep(snrs_db, streams_per_point, tile, compute, rank=0, world=1, **reduce_kw):
    """Generic host driver of the sync sweep (used with a stand-in ``compute`` in the gloo tests).
    ``compute(snr_index, snr_db, first_stream, n_streams) -> (rec[9, n_streams], counts[4])`` processes one tile on this rank;
    the result is that of :func:`reduce_sync`."""
    snrs_db = list(snrs_db)
    rec = torch.zeros((len(snrs_db), 9, int(streams_per_point)), dtype=torch.float64)
    counts = torch.zeros((len(snrs_db), 4), dtype=torch.int64)
    for (i, s0, n) in tiles(len(snrs_db), streams_per_point, tile, rank, world):
        r, c = compute(i, snrs_db[i], s0, n)
        rec[i, :, s0:s0 + n] = torch.as_tensor(np.asarray(r, dtype=np.float64))
        counts[i] += torch.as_tensor(np.asarray(c, dtype=np.int64))
    return reduce_sync(rec, counts, **reduce_kw)


def sync_sweep_local(ctx, lp, snrs_db, streams_per_point, taps=None, seed=1, rank=0, world=1, tile=0, sto=None, cfo=None, sto_max=None,
                     cfo_int_max=30, time_desync=True, freq_desync=True, mp_desync=True, rec=None, counts=None):
    """This rank's share of the sync sweep through ``ofdm_sweep_sync``, WITHOUT synchronising: writes its cells of ``rec``
    (n_snr, 9, streams_per_point) float64, fields :data:`SYNC_FIELDS`, and adds to ``counts`` (n_snr, 4) int64 {bit errors,
    bits, detector failures, IFO misses}; both are zero-initialised device tensors when not given.  With ``sto`` and ``cfo``
    every stream gets that STO / CFO; otherwise they are drawn as :func:`sweep_local` draws them (``sto_max`` defaults to
    Nfft + Tg)."""
    snr = np.ascontiguousarray(np.asarray(snrs_db, dtype=np.float64))
    sp = _cabi.SyncParams()
    sp.n_snr = snr.size
    sp.snr_db_host = snr.ctypes.data_as(_cabi.pdbl)
    sp.streams_per_point = int(streams_per_point)
    sp.tile_streams = int(tile)
    sp.rank, sp.world = int(rank), int(world)
    sp.seed = int(seed)
    t = None
    if taps is not None and len(taps):
        t = np.ascontiguousarray(np.asarray(taps, dtype=np.float64).reshape(-1, 2))
        sp.taps_host = t.ctypes.data_as(_cabi.pdbl)
        sp.n_taps = t.shape[0]
    fixed = sto is not None or cfo is not None
    sp.sto_mode = 1 if fixed else 0
    sp.sto_fixed = int(sto or 0)
    sp.cfo_fixed = float(cfo or 0.0)
    sp.sto_max = int(lp.Nfft + lp.Tg if sto_max is None else sto_max)
    sp.cfo_int_max = int(cfo_int_max)
    sp.time_desync, sp.freq_desync, sp.mp_desync = int(bool(time_desync)), int(bool(freq_desync)), int(bool(mp_desync))
    if rec is None:
        rec = torch.zeros((snr.size, 9, int(streams_per_point)), dtype=torch.float64, device=ctx.device)
    if counts is None:
        counts = torch.zeros((snr.size, 4), dtype=torch.int64, device=ctx.device)
    ctx._chk(ctx.lib.ofdm_sweep_sync(ctx.h, C.byref(lp), C.byref(sp), ctx.p(rec), ctx.p(counts)))
    return rec, counts


def sync_sweep(ctx, lp, snrs_db, streams_per_point, taps=None, seed=1, rank=0, world=1, tile=0, cfo_tol=0.02, **kw):
    """Whole sync sweep: this rank's call, then one all-reduce each of the records and the counters, and the per-point
    statistics of :func:`reduce_sync` (NMSE against mean |H|^2 of ``taps``); identical on every rank and for every world
    size and tile."""
    rec, cnt = sync_sweep_local(ctx, lp, snrs_db, streams_per_point, taps, seed, rank, world, tile, **kw)
    ctx.sync()
    return reduce_sync(rec, cnt, h_power=channel_power(taps, lp.Nfft, lp.N_carrier), sym_len=lp.Nfft + lp.Tg, cfo_tol=cfo_tol)


def papr_sweep_local(ctx, lp, points, streams_per_point, seed=1, rank=0, world=1, tile=0, bin_db=0.01, n_bins=4000, pool=None, pool_stride=0,
                     hist=None, papr=None):
    """This rank's share of the PAPR study through ``ofdm_sweep_papr``, WITHOUT synchronising.  ``points``: a list of
    ``(scramble, p_one)``; ``p_one`` is P(bit = 1) of the Philox payload and is ignored when ``pool`` (0/1 payload bits, e.g.
    ``realisations.file_reader``) is given: stream j then transmits pool bits (j * pool_stride + i) mod len(pool).  Writes
    its cells of ``papr`` (n_points, streams_per_point) float64 and adds to ``hist`` (n_points, n_bins) int64, window
    PAPR v in bin min(floor(v / bin_db), n_bins - 1); both are zero-initialised device tensors when not given."""
    pts = [(int(bool(s)), p) for s, p in points]
    scr = np.ascontiguousarray(np.array([s for s, _ in pts], dtype=np.int32))
    pone = np.ascontiguousarray(np.array([0.5 if p is None else float(p) for _, p in pts], dtype=np.float64))
    pp = _cabi.PaprParams()
    pp.n_points = len(pts)
    pp.scramble_host = scr.ctypes.data_as(_cabi.pi32)
    pp.p_one_host = pone.ctypes.data_as(_cabi.pdbl)
    words = None
    if pool is not None:
        bits = np.asarray(pool).ravel()
        words = np.ascontiguousarray(np.packbits(bits.astype(np.uint8), bitorder="little"))
        words = np.concatenate([words, np.zeros((-words.size) % 4, dtype=np.uint8)]).view(np.uint32)
        pp.pool_host = words.ctypes.data_as(C.POINTER(C.c_uint32))
        pp.pool_bits = int(bits.size)
        pp.pool_stride = int(pool_stride)
    pp.streams_per_point = int(streams_per_point)
    pp.tile_streams = int(tile)
    pp.rank, pp.world = int(rank), int(world)
    pp.seed = int(seed)
    pp.bin_db = float(bin_db)
    pp.n_bins = int(n_bins)
    if hist is None:
        hist = torch.zeros((len(pts), int(n_bins)), dtype=torch.int64, device=ctx.device)
    if papr is None:
        papr = torch.zeros((len(pts), int(streams_per_point)), dtype=torch.float64, device=ctx.device)
    ctx._chk(ctx.lib.ofdm_sweep_papr(ctx.h, C.byref(lp), C.byref(pp), ctx.p(papr), ctx.p(hist)))
    return hist, papr


def papr_ccdf(hist):
    """CCDF at the bin edges b * bin_db of an (n_points, n_bins) or (n_bins,) histogram: the fraction of windows whose bin is
    >= b, i.e. P(PAPR >= b * bin_db) (exact at the edges; the last bin holds everything above its edge)."""
    h = np.asarray(hist, dtype=np.int64)
    tail = np.cumsum(h[..., ::-1], axis=-1)[..., ::-1]
    return tail / np.maximum(tail[..., :1], 1)


def papr_exceedance(hist, bin_db, prob):
    """The smallest bin edge whose CCDF is <= prob -- the PAPR "exceeded with probability prob" that `Task 2/README.md:69-71`
    reads off calculateCCDF's curve, to within one bin above it.  One value per point of an (n_points, n_bins) histogram."""
    c = papr_ccdf(hist)
    below = c <= prob
    idx = np.where(below.any(axis=-1), below.argmax(axis=-1), c.shape[-1])
    return idx * float(bin_db)


def reduce_papr(hist, papr, bin_db=0.01):
    """Sum the histogram (n_points, n_bins) int64 and the per-stream PAPR (n_points, streams_per_point) float64 over all
    ranks -- one all-reduce each, exact because the histogram is integer and every PAPR cell is written by one rank (no-op
    without an initialised process group).  Returns a dict of NumPy arrays, identical on every rank: ``hist``, ``edges``
    (b * bin_db), ``ccdf`` at the edges (:func:`papr_ccdf`), ``papr`` and its mean per point ``papr_mean``."""
    all_reduce_sum(hist, papr)
    h = hist.cpu().numpy()
    p = papr.cpu().numpy()
    return {"hist": h, "edges": np.arange(h.shape[-1]) * float(bin_db), "ccdf": papr_ccdf(h), "papr": p, "papr_mean": p.mean(axis=-1)}


def run_papr_sweep(points, streams_per_point, tile, compute, rank=0, world=1, n_bins=4000, bin_db=0.01):
    """Generic host driver of the PAPR study (used with a stand-in ``compute`` in the gloo tests).
    ``compute(point_index, point, first_stream, n_streams) -> (hist[n_bins], papr[n_streams])`` processes one tile on this
    rank; the result is that of :func:`reduce_papr`."""
    points = list(points)
    hist = torch.zeros((len(points), int(n_bins)), dtype=torch.int64)
    papr = torch.zeros((len(points), int(streams_per_point)), dtype=torch.float64)
    for (k, s0, n) in tiles(len(points), streams_per_point, tile, rank, world):
        h, p = compute(k, points[k], s0, n)
        hist[k] += torch.as_tensor(np.asarray(h, dtype=np.int64))
        papr[k, s0:s0 + n] = torch.as_tensor(np.asarray(p, dtype=np.float64))
    return reduce_papr(hist, papr, bin_db)


def papr_sweep(ctx, lp, points, streams_per_point, seed=1, rank=0, world=1, tile=0, bin_db=0.01, n_bins=4000, pool=None, pool_stride=0):
    """Whole PAPR study: this rank's call (:func:`papr_sweep_local`), then :func:`reduce_papr`; identical on every rank and
    for every world size and tile."""
    hist, papr = papr_sweep_local(ctx, lp, points, streams_per_point, seed, rank, world, tile, bin_db, n_bins, pool, pool_stride)
    ctx.sync()
    return reduce_papr(hist, papr, bin_db)
