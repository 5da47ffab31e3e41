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

``mer_sweep`` is Task 3's study (``ofdm_sweep_mer`` in csrc/sweep_mer.cu): the BER and MER of the receiver without
synchroniser or estimator, over points that each have their own constellation and SNR, one all-reduce each of the per-stream
MER sums and the counters.

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


def sweep_params(lp, snrs_db, streams_per_point, taps=None, chain="task5", seed=1, rank=0, world=1, tile=0, near_eps=0.0,
                 sto_max=None, cfo_int_max=30):
    """The ``ofdm_sweep_params`` of :func:`sweep_local`'s arguments (its host arrays are kept alive on the returned object)."""
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
    sp._keep = (snr, t)
    return sp


def sweep_local(ctx, lp, snrs_db, streams_per_point, taps=None, chain="task5", seed=1, rank=0, world=1, tile=0, near_eps=0.0,
                sto_max=None, cfo_int_max=30, counts=None):
    """This rank's share of the sweep through ``ofdm_sweep_ber``; returns the device counters (n_snr, 4) int64
    {errors, bits, near-boundary symbols, detector failures} WITHOUT synchronising (everything is stream-ordered)."""
    sp = sweep_params(lp, snrs_db, streams_per_point, taps, chain, seed, rank, world, tile, near_eps, sto_max, cfo_int_max)
    if counts is None:
        counts = torch.zeros((sp.n_snr, 4), dtype=torch.int64, device=ctx.device)
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


def mse_params(lp, snrs_db, streams_per_point, taps, Ldict=None, seed=1, rank=0, world=1, tile=0, tie_eps=0.0):
    """(``ofdm_sweep_params``, Ldict) of :func:`mse_sweep_local`'s arguments (host arrays kept alive on the params)."""
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
    sp._keep = (snr, t)
    return sp, int(Ldict)


def mse_sweep_local(ctx, lp, snrs_db, streams_per_point, taps, Ldict=None, seed=1, rank=0, world=1, tile=0, tie_eps=0.0, per_stream=None, counts=None):
    """This rank's share of the MSE sweep through ``ofdm_sweep_mse``, WITHOUT synchronising: writes its cells of
    ``per_stream`` (n_snr, 4, streams_per_point) float64 and adds to ``counts`` (n_snr, 2) int64 {streams, OMP frames with a
    near-tie}; both are zero-initialised device tensors when not given.  ``Ldict`` defaults to the script's
    ceil(N_carrier / comb) (`Main_model_Task_5.m:182-190`)."""
    sp, Ldict = mse_params(lp, snrs_db, streams_per_point, taps, Ldict, seed, rank, world, tile, tie_eps)
    if per_stream is None:
        per_stream = torch.zeros((sp.n_snr, 4, int(streams_per_point)), dtype=torch.float64, device=ctx.device)
    if counts is None:
        counts = torch.zeros((sp.n_snr, 2), dtype=torch.int64, device=ctx.device)
    ctx._chk(ctx.lib.ofdm_sweep_mse(ctx.h, C.byref(lp), C.byref(sp), Ldict, ctx.p(per_stream), ctx.p(counts)))
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


def sync_params(lp, snrs_db, streams_per_point, taps=None, seed=1, rank=0, world=1, tile=0, sto=None, cfo=None, sto_max=None,
                cfo_int_max=30, time_desync=True, freq_desync=True, mp_desync=True):
    """The ``ofdm_sync_params`` of :func:`sync_sweep_local`'s arguments (host arrays kept alive on the returned object)."""
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
    sp._keep = (snr, t)
    return sp


def sync_sweep_local(ctx, lp, snrs_db, streams_per_point, taps=None, seed=1, rank=0, world=1, tile=0, sto=None, cfo=None, sto_max=None,
                     cfo_int_max=30, time_desync=True, freq_desync=True, mp_desync=True, rec=None, counts=None):
    """This rank's share of the sync sweep through ``ofdm_sweep_sync``, WITHOUT synchronising: writes its cells of ``rec``
    (n_snr, 9, streams_per_point) float64, fields :data:`SYNC_FIELDS`, and adds to ``counts`` (n_snr, 4) int64 {bit errors,
    bits, detector failures, IFO misses}; both are zero-initialised device tensors when not given.  With ``sto`` and ``cfo``
    every stream gets that STO / CFO; otherwise they are drawn as :func:`sweep_local` draws them (``sto_max`` defaults to
    Nfft + Tg)."""
    sp = sync_params(lp, snrs_db, streams_per_point, taps, seed, rank, world, tile, sto, cfo, sto_max, cfo_int_max, time_desync, freq_desync,
                     mp_desync)
    if rec is None:
        rec = torch.zeros((sp.n_snr, 9, int(streams_per_point)), dtype=torch.float64, device=ctx.device)
    if counts is None:
        counts = torch.zeros((sp.n_snr, 4), dtype=torch.int64, device=ctx.device)
    ctx._chk(ctx.lib.ofdm_sweep_sync(ctx.h, C.byref(lp), C.byref(sp), ctx.p(rec), ctx.p(counts)))
    return rec, counts


def sync_sweep(ctx, lp, snrs_db, streams_per_point, taps=None, seed=1, rank=0, world=1, tile=0, cfo_tol=0.02, **kw):
    """Whole sync sweep: this rank's call, then one all-reduce each of the records and the counters, and the per-point
    statistics of :func:`reduce_sync` (NMSE against mean |H|^2 of ``taps``); identical on every rank and for every world
    size and tile."""
    rec, cnt = sync_sweep_local(ctx, lp, snrs_db, streams_per_point, taps, seed, rank, world, tile, **kw)
    ctx.sync()
    return reduce_sync(rec, cnt, h_power=channel_power(taps, lp.Nfft, lp.N_carrier), sym_len=lp.Nfft + lp.Tg, cfo_tol=cfo_tol)


MER_FIELDS = ("ideal_power", "error_power")


def reduce_mer(mer, counts):
    """Sum the per-stream MER sums (n_points, 2, streams_per_point) float64 -- field 0 the sum of |ideal|^2, field 1 the sum
    of |ideal - rx|^2 over the stream's data symbols -- and the counters (n_points, 3) int64 {bit errors, bits, near-boundary
    symbols} over all ranks: one all-reduce each, exact because every MER cell is written by one rank (no-op without an
    initialised process group).  Returns a dict of NumPy arrays over the points, identical on every rank:
      ber; mer_db, the pooled MER_func 10 log10(sum f0 / sum f1) with both sums taken in stream order; mer_stream_db, the
      mean of the finite per-stream MER values in dB (``per_stream_db``); near, the near-boundary symbol count;
    plus ``mer`` and ``counts`` themselves."""
    all_reduce_sum(mer, counts)
    m = mer.cpu().numpy()
    c = counts.cpu().numpy()
    pooled = np.cumsum(m, axis=2)[:, :, -1]
    with np.errstate(divide="ignore", invalid="ignore"):
        per_db = 10 * np.log10(m[:, 0, :] / m[:, 1, :])
        mer_db = 10 * np.log10(pooled[:, 0] / pooled[:, 1])
    fin = np.isfinite(per_db)
    n_fin = fin.sum(axis=1)
    mean_db = np.where(n_fin > 0, np.where(fin, per_db, 0.0).sum(axis=1) / np.maximum(n_fin, 1), np.nan)
    return {"ber": c[:, 0] / np.maximum(c[:, 1], 1), "mer_db": mer_db, "mer_stream_db": mean_db, "near": c[:, 2],
            "per_stream_db": per_db, "mer": m, "counts": c}


def run_mer_sweep(points, streams_per_point, tile, compute, rank=0, world=1):
    """Generic host driver of the MER study (used with a stand-in ``compute`` in the gloo tests).
    ``compute(point_index, point, first_stream, n_streams) -> (mer[2, n_streams], counts[3])`` processes one tile on this
    rank; the result is that of :func:`reduce_mer`."""
    points = list(points)
    mer = torch.zeros((len(points), 2, int(streams_per_point)), dtype=torch.float64)
    counts = torch.zeros((len(points), 3), dtype=torch.int64)
    for (k, s0, n) in tiles(len(points), streams_per_point, tile, rank, world):
        m, c = compute(k, points[k], s0, n)
        mer[k, :, s0:s0 + n] = torch.as_tensor(np.asarray(m, dtype=np.float64))
        counts[k] += torch.as_tensor(np.asarray(c, dtype=np.int64))
    return reduce_mer(mer, counts)


def _per_point(v, n, dtype):
    """None, a scalar or n values, as a contiguous array of n (None stays None)."""
    if v is None:
        return None
    a = np.asarray(v, dtype=dtype)
    return np.ascontiguousarray(np.full(n, a, dtype=dtype) if a.ndim == 0 else a.reshape(n))


def mer_params(constellations, snrs_db, streams_per_point, taps=None, seed=1, rank=0, world=1, tile=0, pilot_scale=0.0, sto=None, cfo=None,
               near_eps=0.0):
    """The ``ofdm_mer_params`` of :func:`mer_sweep_local`'s arguments (host arrays kept alive on the returned object)."""
    from .link import CONSTELLATIONS
    snr = np.ascontiguousarray(np.asarray(snrs_db, dtype=np.float64).ravel())
    n = snr.size
    names = [constellations] * n if isinstance(constellations, str) else list(constellations)
    if len(names) != n:
        raise ValueError(f"{len(names)} constellations for {n} SNR points")
    cons = np.ascontiguousarray(np.array([CONSTELLATIONS[str(c)] if str(c) in CONSTELLATIONS else int(c) for c in names], dtype=np.int32))
    mp = _cabi.MerParams()
    mp.n_points = n
    mp.constellation_host = cons.ctypes.data_as(_cabi.pi32)
    mp.snr_db_host = snr.ctypes.data_as(_cabi.pdbl)
    mp.pilot_scale = float(pilot_scale)
    nsto, cf = _per_point(sto, n, np.int32), _per_point(cfo, n, np.float64)
    if nsto is not None:
        mp.nsto_host = nsto.ctypes.data_as(_cabi.pi32)
    if cf is not None:
        mp.cfo_host = cf.ctypes.data_as(_cabi.pdbl)
    t = None
    if taps is not None and len(taps):
        t = np.ascontiguousarray(np.asarray(taps, dtype=np.float64).reshape(-1, 2))
        mp.taps_host = t.ctypes.data_as(_cabi.pdbl)
        mp.n_taps = t.shape[0]
    mp.streams_per_point = int(streams_per_point)
    mp.tile_streams = int(tile)
    mp.rank, mp.world = int(rank), int(world)
    mp.seed = int(seed)
    mp.near_eps = float(near_eps)
    mp._keep = (snr, cons, nsto, cf, t)
    return mp


def mer_sweep_local(ctx, lp, constellations, snrs_db, streams_per_point, taps=None, seed=1, rank=0, world=1, tile=0, pilot_scale=0.0, sto=None,
                    cfo=None, near_eps=0.0, mer=None, counts=None):
    """This rank's share of the Task-3 study through ``ofdm_sweep_mer``, WITHOUT synchronising.  Point k is
    (``constellations[k]``, ``snrs_db[k]``; a single name applies to every point), with the fixed STO / CFO ``sto`` / ``cfo``
    (None, one value, or one per point; not corrected by the receiver).  ``pilot_scale`` > 0 makes every pilot of point k the
    real value pilot_scale * max|constellation| (Task 3's scalar pilots); 0 keeps ``lp``'s pilots.  Writes its cells of ``mer``
    (n_points, 2, streams_per_point) float64, fields :data:`MER_FIELDS`, and adds to ``counts`` (n_points, 3) int64 {bit errors,
    bits, near-boundary symbols}; both are zero-initialised device tensors when not given."""
    mp = mer_params(constellations, snrs_db, streams_per_point, taps, seed, rank, world, tile, pilot_scale, sto, cfo, near_eps)
    if mer is None:
        mer = torch.zeros((mp.n_points, 2, int(streams_per_point)), dtype=torch.float64, device=ctx.device)
    if counts is None:
        counts = torch.zeros((mp.n_points, 3), dtype=torch.int64, device=ctx.device)
    ctx._chk(ctx.lib.ofdm_sweep_mer(ctx.h, C.byref(lp), C.byref(mp), ctx.p(mer), ctx.p(counts)))
    return mer, counts


def mer_sweep(ctx, lp, constellations, snrs_db, streams_per_point, taps=None, seed=1, rank=0, world=1, tile=0, **kw):
    """Whole Task-3 study: this rank's call, then :func:`reduce_mer` (one all-reduce each of the per-stream MER sums and the
    counters); identical on every rank and for every world size and tile."""
    mer, cnt = mer_sweep_local(ctx, lp, constellations, snrs_db, streams_per_point, taps, seed, rank, world, tile, **kw)
    ctx.sync()
    return reduce_mer(mer, cnt)


def papr_params(points, streams_per_point, seed=1, rank=0, world=1, tile=0, bin_db=0.01, n_bins=4000, pool=None, pool_stride=0):
    """The ``ofdm_papr_params`` of :func:`papr_sweep_local`'s arguments (host arrays kept alive on the returned object)."""
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
    pp._keep = (scr, pone, words)
    return pp


def papr_sweep_local(ctx, lp, points, streams_per_point, seed=1, rank=0, world=1, tile=0, bin_db=0.01, n_bins=4000, pool=None, pool_stride=0,
                     hist=None, papr=None):
    """This rank's share of the PAPR study through ``ofdm_sweep_papr``, WITHOUT synchronising.  ``points``: a list of
    ``(scramble, p_one)``; ``p_one`` is P(bit = 1) of the Philox payload and is ignored when ``pool`` (0/1 payload bits, e.g.
    ``realisations.file_reader``) is given: stream j then transmits pool bits (j * pool_stride + i) mod len(pool).  Writes
    its cells of ``papr`` (n_points, streams_per_point) float64 and adds to ``hist`` (n_points, n_bins) int64, window
    PAPR v in bin min(floor(v / bin_db), n_bins - 1); both are zero-initialised device tensors when not given."""
    pp = papr_params(points, streams_per_point, seed, rank, world, tile, bin_db, n_bins, pool, pool_stride)
    if hist is None:
        hist = torch.zeros((pp.n_points, int(n_bins)), dtype=torch.int64, device=ctx.device)
    if papr is None:
        papr = torch.zeros((pp.n_points, int(streams_per_point)), dtype=torch.float64, device=ctx.device)
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


class Group:
    """Several GPUs of this process as ONE ``ofdm_group`` (include/ofdm_b200.h): each method runs a sweep's shares on all
    members at once, one host thread per member inside the library, and returns the assembled host arrays as NumPy --
    bit-identical to the single-context call with world 1, without ``torch.distributed``.  ``devices``: CUDA ordinals
    (0-based, repeats allowed); member i is rank i.  The methods take the arguments of the matching ``*_sweep_local``
    function without rank / world / output tensors."""

    def __init__(self, devices, precision="f32"):
        from .link import OfdmError
        self.lib = _cabi.load()
        ids = np.ascontiguousarray(np.asarray(list(devices), dtype=np.int32))
        h = C.c_void_p()
        rc = self.lib.ofdm_group_create(C.byref(h), ids.ctypes.data_as(_cabi.pi32), int(ids.size), 1 if precision in ("f64", 1, "double") else 0)
        if rc != 0:
            err = OfdmError(f"status {rc}: ofdm_group_create failed for devices {ids.tolist()}")
            err.status = rc
            raise err
        self.h = h
        self.devices = tuple(int(d) for d in ids)

    def close(self):
        if getattr(self, "h", None):
            self.lib.ofdm_group_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _chk(self, rc):
        if rc != 0:
            from .link import OfdmError
            err = OfdmError(f"status {rc}: {self.lib.ofdm_group_last_error(self.h).decode()}")
            err.status = rc
            raise err

    def sweep_ber(self, lp, snrs_db, streams_per_point, taps=None, chain="task5", seed=1, tile=0, near_eps=0.0, sto_max=None, cfo_int_max=30):
        """Counters (n_snr, 4) int64 of :func:`sweep_local`."""
        sp = sweep_params(lp, snrs_db, streams_per_point, taps, chain, seed, 0, 1, tile, near_eps, sto_max, cfo_int_max)
        counts = np.zeros((sp.n_snr, 4), dtype=np.int64)
        self._chk(self.lib.ofdm_group_sweep_ber(self.h, C.byref(lp), C.byref(sp), counts.ctypes.data))
        return counts

    def sweep_mse(self, lp, snrs_db, streams_per_point, taps, Ldict=None, seed=1, tile=0, tie_eps=0.0):
        """(per_stream (n_snr, 4, streams_per_point) float64, counts (n_snr, 2) int64) of :func:`mse_sweep_local`."""
        sp, Ldict = mse_params(lp, snrs_db, streams_per_point, taps, Ldict, seed, 0, 1, tile, tie_eps)
        per = np.zeros((sp.n_snr, 4, int(streams_per_point)), dtype=np.float64)
        counts = np.zeros((sp.n_snr, 2), dtype=np.int64)
        self._chk(self.lib.ofdm_group_sweep_mse(self.h, C.byref(lp), C.byref(sp), Ldict, per.ctypes.data, counts.ctypes.data))
        return per, counts

    def sweep_sync(self, lp, snrs_db, streams_per_point, taps=None, seed=1, tile=0, **kw):
        """(rec (n_snr, 9, streams_per_point) float64, counts (n_snr, 4) int64) of :func:`sync_sweep_local`."""
        sp = sync_params(lp, snrs_db, streams_per_point, taps, seed, 0, 1, tile, **kw)
        rec = np.zeros((sp.n_snr, 9, int(streams_per_point)), dtype=np.float64)
        counts = np.zeros((sp.n_snr, 4), dtype=np.int64)
        self._chk(self.lib.ofdm_group_sweep_sync(self.h, C.byref(lp), C.byref(sp), rec.ctypes.data, counts.ctypes.data))
        return rec, counts

    def sweep_papr(self, lp, points, streams_per_point, seed=1, tile=0, bin_db=0.01, n_bins=4000, pool=None, pool_stride=0):
        """(hist (n_points, n_bins) int64, papr (n_points, streams_per_point) float64) of :func:`papr_sweep_local`."""
        pp = papr_params(points, streams_per_point, seed, 0, 1, tile, bin_db, n_bins, pool, pool_stride)
        hist = np.zeros((pp.n_points, int(n_bins)), dtype=np.int64)
        papr = np.zeros((pp.n_points, int(streams_per_point)), dtype=np.float64)
        self._chk(self.lib.ofdm_group_sweep_papr(self.h, C.byref(lp), C.byref(pp), papr.ctypes.data, hist.ctypes.data))
        return hist, papr

    def sweep_mer(self, lp, constellations, snrs_db, streams_per_point, taps=None, seed=1, tile=0, **kw):
        """(mer (n_points, 2, streams_per_point) float64, counts (n_points, 3) int64) of :func:`mer_sweep_local`."""
        mp = mer_params(constellations, snrs_db, streams_per_point, taps, seed, 0, 1, tile, **kw)
        mer = np.zeros((mp.n_points, 2, int(streams_per_point)), dtype=np.float64)
        counts = np.zeros((mp.n_points, 3), dtype=np.int64)
        self._chk(self.lib.ofdm_group_sweep_mer(self.h, C.byref(lp), C.byref(mp), mer.ctypes.data, counts.ctypes.data))
        return mer, counts

    def sweep_part2(self, combs, mc_runs, payload_bits, *, tile=0, **kw):
        """(per_run (n_points, 4, mc_runs) float64, counts (n_points, 4, 3) int64, runs (n_points, 2) int64) of
        ``part2.sweep_lib_local``; keywords as ``part2.lib_params``."""
        from .part2 import lib_params
        lp, pp = lib_params(combs, mc_runs, payload_bits, tile=tile, **kw)
        per = np.zeros((pp.n_points, 4, int(mc_runs)), dtype=np.float64)
        counts = np.zeros((pp.n_points, 4, 3), dtype=np.int64)
        runs = np.zeros((pp.n_points, 2), dtype=np.int64)
        self._chk(self.lib.ofdm_group_sweep_part2(self.h, C.byref(lp), C.byref(pp), per.ctypes.data, counts.ctypes.data, runs.ctypes.data))
        return per, counts, runs
