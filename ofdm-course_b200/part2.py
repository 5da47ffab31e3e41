"""Task 5 part 2 on the GPU: pilot-comb sweep x Monte-Carlo channel realisations x {LS, MMSE, MP, OMP}
(`Task 5/Task5_part2.m:46-321`, SURVEY 8f rank 1).

One sweep point (a pilot layout) is one batch: the layout's TX stream is built and noised ONCE
(`Task5_part2.m:128-132` -- every Monte-Carlo run filters the same noisy stream), the `monteCarloRuns` channel
realisations are the batch axis, and every stage is a C-ABI call: ofdm_tx_chain, ofdm_add_noise,
ofdm_tdl_channel (stand-in for lteFadingChannel), ofdm_apply_fir, ofdm_demodulate, ofdm_ls_ce, ofdm_mmse_ce,
ofdm_pilot_ls, ofdm_mp, ofdm_omp, ofdm_fft, ofdm_mse, ofdm_equalize, ofdm_get_payload, ofdm_demap,
ofdm_ber_count.  Points x run-blocks are dealt round-robin to the ranks; every (point, run, estimator) cell is
written by exactly one rank, so the closing all_reduce(SUM) is exact and independent of the rank count.

``sweep_lib`` runs the same experiment as ONE C-ABI call per rank, ``ofdm_sweep_part2`` (csrc/sweep_part2.cu), with the keys
of ``run_point``: its per-run NMSE and per-point error counts equal those of ``sweep`` bit for bit.  Ranks take the contiguous
share of the (point, run) items that ``ofdm_sweep_share`` gives, as the other library sweeps do.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

ESTIMATORS = ("LS", "MMSE", "MP", "OMP")


def part2_combs(N_carrier=1024, lo=4, hi=256):
    """`combs = 4:1:256` de-duplicated by the pilot count floor(N_carrier/comb) (`Task5_part2.m:13-17`)."""
    combs = np.arange(lo, hi + 1)
    amounts = N_carrier // combs
    _, ia = np.unique(amounts, return_index=True)
    combs = combs[np.sort(ia)]
    return combs, N_carrier // combs


def layout(N_carrier, comb=None, pilotCarriers=None):
    """1-based pilot / data carriers of a sweep point (`Task5_part2.m:50-80`)."""
    allc = np.arange(1, N_carrier + 1)
    pc = allc[::comb] if pilotCarriers is None else np.sort(np.asarray(pilotCarriers, dtype=np.int64))
    return pc, allc[~np.isin(allc, pc)]


def pilot_values(Np, N_symb, amp):
    """Alternating +amp, -amp (`Task5_part2.m:86-91`: exp(1i*pi) and the ctranspose are kept)."""
    pv = np.full(Np, amp * np.exp(1j * 0), dtype=np.complex128)
    pv[1::2] = amp * np.exp(1j * np.pi)
    return np.tile(np.conj(pv)[:, None], (1, N_symb))


def run_point(ctx, pc, dc, bits, n_runs, *, profile="EPA", fs_hz=4e7, snr_db=20.0, seed=1, point_id=0, first_run=0,
              Ldict=None, h_dev=None, Nfft=4096, N_carrier=1024, frames=2, spf=7, constellation="16QAM", noise_normals=None):
    """`n_runs` Monte-Carlo runs of one pilot layout.  bits: the layout's payload (uint8 0/1, stream_bits long).
    h_dev: imported impulse responses (n_runs x D) instead of the device generator.  Returns
    (nmse float64[n_runs, 4], errors int64[4], bits_per_run, extras)."""
    from . import link as G
    S = frames * spf
    Tg = Nfft // 8
    d, bps = G.constellation_func(constellation)
    amp = 2.0 * float(np.max(np.abs(d)))
    pv = pilot_values(len(pc), S, amp)
    lp = ctx.link_params(Nfft, Tg, N_carrier, S, spf, constellation, dc, pc, pv, scramble=False)
    bits = np.asarray(bits, dtype=np.uint8).ravel()
    assert bits.size == lp.stream_bits
    tx = ctx.tx_chain(lp, ctx.bits(bits), 1).reshape(1, -1)
    # AWGN once per layout, before the channel (`Task5_part2.m:132`); keyed by the point, not by the run
    txn, _ = ctx.add_noise(tx, snr_db, normals_dev=noise_normals, seed=seed, first_stream_id=point_id)
    n_paths, _, _ = ctx.tdl_info(profile, fs_hz)
    if h_dev is None:
        h_dev = ctx.tdl_channel(profile, fs_hz, n_runs, seed=seed, first_stream_id=point_id * 1_000_003 + first_run)
    D = h_dev.shape[-1]
    rx = ctx.apply_fir(txn.expand(n_runs, -1).contiguous(), h_dev, per_stream=True)
    Y = ctx.demodulate(rx.reshape(n_runs, S, Nfft + Tg), Nfft, Tg)
    h_full = torch.zeros((n_runs, Nfft), dtype=h_dev.dtype, device=h_dev.device)
    h_full[:, :D] = h_dev
    H_f = ctx.fft(h_full)                                        # `H_f = fft(h_t)`, :155
    H = {}
    H["LS"] = ctx.ls_ce(Y, pv, pc, N_carrier)
    H["MMSE"] = ctx.mmse_ce(Y, pv, pc, N_carrier, h_full[:, :N_carrier].contiguous(), snr_db)   # true CIR, :176-177
    y = ctx.pilot_ls(Y, pv, pc)
    if Ldict is None:
        Ldict = Nfft
    H["MP"] = ctx.mp(y, Nfft, n_paths, Ldict=Ldict, pilot_loc=pc)[0]
    H["OMP"] = ctx.omp(y, Nfft, n_paths, Ldict=Ldict, pilot_loc=pc)[0]
    nmse = torch.stack([ctx.mse(H_f, H[k], N_carrier) for k in ESTIMATORS], dim=1)
    ref_bits = ctx.bits(np.tile(bits, n_runs))
    errors = np.zeros(4, dtype=np.int64)
    for j, k in enumerate(ESTIMATORS):
        eq = ctx.equalize(Y, H[k], N_carrier)
        iq = ctx.get_payload(eq, dc)
        out_bits = ctx.demap(iq.reshape(-1), constellation)
        out_bits = out_bits[0] if isinstance(out_bits, tuple) else out_bits
        errors[j] = int(ctx.ber_count(ref_bits, out_bits, n_runs * bits.size)[0].item())
    return nmse.cpu().numpy(), errors, bits.size, {"H": H, "H_f": H_f, "h": h_dev, "Y": Y}


def sweep(ctx, combs, mc_runs, payload, *, block=None, rank=0, world=1, reg_pilot=True, random_masks=None, run_fn=None, **kw):
    """The whole experiment: returns (NMSE[4, n_points], BER[4, n_points]) identical on every rank.
    payload(n_bits) -> uint8 bits (the reference reads them from eagle.tiff, `file_reader.m:4-11`).
    run_fn: stand-in for run_point (CPU tests of the sharding logic only)."""
    N_carrier = kw.get("N_carrier", 1024)
    Nfft = kw.get("Nfft", 4096)
    block = block or mc_runs
    n_pts = len(combs)
    nm = torch.zeros((n_pts, mc_runs, 4), dtype=torch.float64)
    er = torch.zeros((n_pts, 4), dtype=torch.int64)
    nb = torch.zeros(n_pts, dtype=torch.int64)
    items = [(k, r0) for k in range(n_pts) for r0 in range(0, mc_runs, block)]
    for (k, r0) in items[rank::world]:
        comb = int(combs[k])
        if reg_pilot:
            pc, dc = layout(N_carrier, comb=comb)
            Ldict = -(-Nfft // comb)                              # F(:,1:ceil(Nfft/comb)), :183-185
        else:
            pc, dc = layout(N_carrier, pilotCarriers=random_masks[k])
            Ldict = Nfft
        n = min(block, mc_runs - r0)
        spb = 2 * 7 * len(dc) * 4
        nmse, errs, bits_run, _ = (run_fn or run_point)(ctx, pc, dc, payload(spb), n, point_id=k, first_run=r0, Ldict=Ldict, **kw)
        nm[k, r0:r0 + n] = torch.from_numpy(nmse)
        er[k] += torch.from_numpy(errs)
        nb[k] += n * bits_run
    from .sweep import all_reduce_sum                            # sweep imports this module
    if dist.is_available() and dist.is_initialized() and dist.get_backend() == "nccl":
        nm, er, nb = nm.to(ctx.device), er.to(ctx.device), nb.to(ctx.device)
    all_reduce_sum(nm, er, nb)
    nm, er, nb = nm.cpu(), er.cpu(), nb.cpu()
    NMSE = nm.mean(dim=1).numpy().T                               # mean over the Monte-Carlo runs, :311-314
    BER = (er.double() / nb.double()[:, None]).numpy().T          # equal run sizes: mean of per-run BERs, :305-308
    return NMSE, BER


def lib_layout(combs, N_carrier=1024, Nfft=4096, reg_pilot=True, random_masks=None):
    """The pilot layouts of ``sweep`` in the form ``ofdm_sweep_part2`` takes: (offsets int32[n_points + 1], 1-based pilot
    carriers int32 concatenated over the points, Ldict int32[n_points]) with the layout and Ldict rules of ``sweep``."""
    n_pts = len(combs)
    pcs, ldict = [], []
    for k in range(n_pts):
        if reg_pilot:
            comb = int(combs[k])
            pc, _ = layout(N_carrier, comb=comb)
            ldict.append(-(-Nfft // comb))
        else:
            pc, _ = layout(N_carrier, pilotCarriers=random_masks[k])
            ldict.append(Nfft)
        pcs.append(pc)
    offsets = np.concatenate([[0], np.cumsum([len(pc) for pc in pcs])]).astype(np.int32)
    return offsets, np.concatenate(pcs).astype(np.int32), np.asarray(ldict, dtype=np.int32)


def pilot_pattern(amp):
    """The two pilot values of ``pilot_values`` (pilot q carries pattern[q % 2] in every symbol), as the exact doubles."""
    return pilot_values(2, 1, amp)[:, 0]


def reduce_part2(per_run, counts, runs):
    """Sum the per-run NMSE (n_points, 4, mc_runs) float64, the counts (n_points, 4, 3) and the runs (n_points, 2) int64 over
    all ranks (no-op without an initialised process group), then form ``sweep``'s results with its own arithmetic.
    Returns (NMSE[4, n_points], BER[4, n_points], per_run, counts, runs) as NumPy arrays, identical on every rank."""
    from .sweep import all_reduce_sum                            # sweep imports this module
    all_reduce_sum(per_run, counts, runs)                        # exact: every NMSE cell is non-zero on one rank only
    per, cnt, rn = per_run.cpu().numpy(), counts.cpu().numpy(), runs.cpu().numpy()
    nm = torch.from_numpy(np.ascontiguousarray(per.transpose(0, 2, 1)))      # the (point, run, estimator) layout of sweep
    er = torch.from_numpy(np.ascontiguousarray(cnt[:, :, 0]))
    nb = torch.from_numpy(np.ascontiguousarray(cnt[:, 0, 1]))
    NMSE = nm.mean(dim=1).numpy().T
    BER = (er.double() / nb.double()[:, None]).numpy().T
    return NMSE, BER, per, cnt, rn


def lib_params(combs, mc_runs, payload_bits, *, tile=0, rank=0, world=1, reg_pilot=True, random_masks=None, profile="EPA", fs_hz=4e7,
               snr_db=20.0, seed=1, near_eps=0.0, tie_eps=0.0, Nfft=4096, N_carrier=1024, frames=2, spf=7, constellation="16QAM"):
    """(``ofdm_link_params``, ``ofdm_part2_params``) of :func:`sweep_lib_local`'s arguments (host arrays kept alive on the
    part-2 params)."""
    from . import _cabi
    from . import link as G
    offsets, carriers, ldict = lib_layout(combs, N_carrier, Nfft, reg_pilot, random_masks)
    n_pts = ldict.size
    d, _ = G.constellation_func(constellation)
    pattern = np.ascontiguousarray(pilot_pattern(2.0 * float(np.max(np.abs(d)))))
    bits = np.asarray(payload_bits, dtype=np.uint8).ravel()
    words = G.pack_bits(bits)
    lp = _cabi.LinkParams()
    lp.Nfft, lp.Tg, lp.N_carrier, lp.S, lp.SpF = int(Nfft), int(Nfft) // 8, int(N_carrier), int(frames * spf), int(spf)
    lp.constellation = G.CONSTELLATIONS[str(constellation)]
    pp = _cabi.Part2Params()
    pp.n_points = n_pts
    pp.pilot_offsets_host = offsets.ctypes.data_as(_cabi.pi32)
    pp.pilot_carriers_host = carriers.ctypes.data_as(_cabi.pi32)
    pp.ldict_host = ldict.ctypes.data_as(_cabi.pi32)
    pp.pilot_pattern_host = pattern.ctypes.data_as(_cabi.pdbl)
    pp.payload_host = words.ctypes.data_as(C.POINTER(C.c_uint32))
    pp.payload_bits = bits.size
    pp.profile = G.TDL_PROFILES[str(profile).upper()]
    pp.fs_hz, pp.snr_db = float(fs_hz), float(snr_db)
    pp.mc_runs, pp.tile_runs = int(mc_runs), int(tile)
    pp.rank, pp.world, pp.seed = int(rank), int(world), int(seed)
    pp.near_eps, pp.tie_eps = float(near_eps), float(tie_eps)
    pp._keep = (offsets, carriers, ldict, pattern, words)
    return lp, pp


def sweep_lib_local(ctx, combs, mc_runs, payload_bits, *, tile=0, rank=0, world=1, per_run=None, counts=None, runs=None, **kw):
    """This rank's share of the experiment through ``ofdm_sweep_part2``, WITHOUT synchronising: writes its cells of ``per_run``
    (n_points, 4, mc_runs) float64 and adds to ``counts`` (n_points, 4, 3) and ``runs`` (n_points, 2) int64; all three are
    zero-initialised device tensors when not given.  ``payload_bits``: uint8 0/1, at least the longest stream of any point.
    The other keywords are those of :func:`lib_params`."""
    lp, pp = lib_params(combs, mc_runs, payload_bits, tile=tile, rank=rank, world=world, **kw)
    n_pts = pp.n_points
    if per_run is None:
        per_run = torch.zeros((n_pts, 4, int(mc_runs)), dtype=torch.float64, device=ctx.device)
    if counts is None:
        counts = torch.zeros((n_pts, 4, 3), dtype=torch.int64, device=ctx.device)
    if runs is None:
        runs = torch.zeros((n_pts, 2), dtype=torch.int64, device=ctx.device)
    ctx._chk(ctx.lib.ofdm_sweep_part2(ctx.h, C.byref(lp), C.byref(pp), ctx.p(per_run), ctx.p(counts), ctx.p(runs)))
    return per_run, counts, runs


def sweep_lib(ctx, combs, mc_runs, payload_bits, *, tile=0, rank=0, world=1, reg_pilot=True, random_masks=None, **kw):
    """The whole experiment as one library call per rank, then one all-reduce each of the per-run array, the counts and the
    runs.  Takes ``sweep``'s layout arguments; ``payload_bits`` are the bits ``sweep``'s ``payload`` would return (point k sends
    the first S * Nd_k * bps of them).  Returns (NMSE[4, n_points], BER[4, n_points], per_run[n_points, 4, mc_runs],
    counts[n_points, 4, 3] {errors, bits, near-boundary symbols}, runs[n_points, 2] {runs, OMP runs with a near-tie}),
    estimators in the order LS, MMSE, MP, OMP; identical on every rank and for every world size and tile."""
    per, cnt, rn = sweep_lib_local(ctx, combs, mc_runs, payload_bits, tile=tile, rank=rank, world=world, reg_pilot=reg_pilot,
                                   random_masks=random_masks, **kw)
    ctx.sync()
    return reduce_part2(per, cnt, rn)             # NCCL all-reduce on the device tensors when world > 1
