#!/usr/bin/env python
"""bench.py -- OFDM symbols/s through the full Task-5 RX chain (SURVEY 8d, workload M1).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--streams B] [--dump-outputs DIR]

One "step" = one pass of the fused RX chain (OFDM_demodulator -> LS_CE -> equalize_signal ->
get_payload -> demapping -> DeScrambler -> BER count) over a batch of B synthetic streams of 14 OFDM
symbols (Nfft 4096, CP 512, 1024 carriers, comb-4 pilots, 16QAM, 6-tap multipath + AWGN 20 dB)
that is already resident in HBM.  `value` is device-timed whole-job throughput; `e2e` is the same
chain through the host-buffer C-ABI entry (pinned host memory, H2D + D2H inside the timed region).
`--impl reference` times the CPU restatement of the reference (oracle/, NumPy float64 -- MATLAB and
Octave do not exist on the box) on all host cores.  Prints ONE JSON line on rank 0.

`--dump-outputs DIR` writes, after the timed steps, what the last timed step returned to its caller (rank 0's):
DIR/bits.npy (decided bits, 0/1), DIR/H.npy (LS channel estimate, real and imaginary parts) and DIR/counts.npy (errors,
bits, near-boundary decisions of one step).  The inputs are seeded, so two builds run with the same arguments can be
compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

TAPS5 = [[0, 1], [4, .8], [10, .6], [15, .4], [21, .2], [25, .1]]
A_M1 = 34121.0           # algorithmic bytes per OFDM symbol (SURVEY 8d / DESIGN.md): 8*4096 + 768 + 8192/14
SNR_DB = 20.0
METRIC = "OFDM symbols/s, full Task-5 RX chain"
WORKLOAD = "M1: Task-5 RX chain, Nfft 4096, CP 512, Nc 1024, comb 4 (Np 256, Nd 768), 16QAM, 14 symbols/stream, 6-tap + AWGN 20 dB"


# --------------------------------------------------------------------------------------------
def cpu_chain_worker(args):
    """One bounded sample of the workload through the oracle on one host process: `n_streams` distinct streams,
    passed through the RX chain repeatedly until `target_s` seconds of chain time have been spent."""
    seed, n_streams, target_s = args
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    import oracle as O
    from oracle import chains as OC
    p = OC.params_task5(comb=4)
    rng = np.random.default_rng(seed)
    rxs, bits = [], []
    for _ in range(n_streams):                         # untimed: build the inputs
        b = rng.integers(0, 2, p.stream_bits).astype(np.uint8)
        tx, _, _ = OC.tx_chain(p, b, fast=True)
        rxs.append(OC.channel_task5(p, tx, SNR_DB, TAPS5, rng=rng))
        bits.append(b)
    t0 = time.perf_counter()
    errs, passes = 0, 0
    while True:
        for r, b in zip(rxs, bits):
            errs += OC.rx_chain_task5(p, r, b, fast=True)["errors"]
        passes += 1
        if time.perf_counter() - t0 >= target_s:
            break
    return time.perf_counter() - t0, passes * n_streams * p.N_symb, errs, passes


def cpu_baseline(n_proc, streams_per_proc, seed=1234, target_s=10.0):
    """Oracle throughput on `n_proc` host processes (every worker runs for about `target_s` seconds of RX-chain time;
    symbols of all workers / the slowest worker's time)."""
    import multiprocessing as mp
    ctxm = mp.get_context("spawn")
    t0 = time.perf_counter()
    if n_proc == 1:
        res = [cpu_chain_worker((seed, streams_per_proc, target_s))]
    else:
        with ctxm.Pool(n_proc) as pool:
            res = pool.map(cpu_chain_worker, [(seed + i, streams_per_proc, target_s) for i in range(n_proc)])
    wall = max(r[0] for r in res)
    syms = sum(r[1] for r in res)
    return syms / wall, syms, wall, time.perf_counter() - t0


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples = []
        self.stop_flag = False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        sm, mx, reasons = [], [], set()
        for s in self.samples:
            try:
                sm.append(float(s[1])); mx.append(float(s[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture, if any."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(path):
        try:
            return json.load(open(path))
        except Exception:
            return None
    return None


DUMP_STREAMS = 128      # --dump-outputs sample: 128 x 43,008 bits as float32 + 128 x 1,024 complex carriers = 23.1 MB


def dump_outputs(out_dir, B, words, out_bits, H, counts, steps):
    """Write what the last timed step returned: decided bits and channel estimate of a fixed, seeded sample of streams,
    and one step's counters (every timed step decodes the same input, so the accumulated counters are `steps` times one
    step's).  Runs after the last timed event, so the copies are not timed."""
    import torch
    from ofdm_b200 import unpack_bits
    idx = np.sort(np.random.default_rng(0).choice(B, min(B, DUMP_STREAMS), replace=False))
    sel = torch.from_numpy(idx).to(H.device)
    w = out_bits.view(B, words).index_select(0, sel).cpu().numpy()
    bits = unpack_bits(w.view(np.uint32), w.size * 32).reshape(len(idx), words * 32).astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "bits.npy"), bits)
    np.save(os.path.join(out_dir, "H.npy"), torch.view_as_real(H.index_select(0, sel)).cpu().numpy())
    np.save(os.path.join(out_dir, "counts.npy"), counts.cpu().numpy().astype(np.float64) / steps)


# --------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    if rank != 0:
        return
    n_proc = os.cpu_count() or 1
    per_proc = args.ref_streams
    vals = []
    for _ in range(args.warmup):
        pass  # the oracle has no warm-up state worth timing; keep the run short
    for _ in range(args.steps):
        v, syms, wall, _ = cpu_baseline(n_proc, per_proc, target_s=args.cpu_seconds)
        vals.append((v, syms, wall))
    v = float(np.median([x[0] for x in vals]))
    line = {"metric": METRIC, "value": v, "unit": "symbols/s", "n_gpus": args.gpus, "steps": len(vals), "warmup": 0,
            "ms_per_step": 1e3 * float(np.median([x[2] for x in vals])), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference",
            "config": {"workload": WORKLOAD, "note": "NumPy float64 restatement of the reference (oracle/), MATLAB/Octave absent"},
            "cpu_baseline": {"value": v, "unit": "symbols/s", "cores": n_proc, "kind": "port",
                             "sample": f"{n_proc} processes x {per_proc} distinct streams x 14 symbols, repeated for ~{args.cpu_seconds:g} s of RX-chain time per step"},
            "e2e": {"value": v, "unit": "symbols/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def numa_place(local_rank, world):
    """Before any pinned allocation: split the visible cores evenly over the local ranks (so the copy-issuing threads of
    different ranks do not share cores) and prefer the GPU's own NUMA node for this process's pages, when the container
    lets us.  Returns what was done, for the record."""
    info = {}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local_rank)],
                             capture_output=True, text=True, timeout=10).stdout.strip()
        bdf = out.lower()
        if bdf.startswith("00000000:"):
            bdf = "0000:" + bdf.split(":", 1)[1]
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        info["gpu_numa_node"] = node
    except Exception:
        node = -1
    try:
        cpus = sorted(os.sched_getaffinity(0))
        if node >= 0:
            try:
                def expand(txt):
                    out = []
                    for part in txt.strip().split(","):
                        a, _, b = part.partition("-")
                        out += list(range(int(a), int(b or a) + 1))
                    return out
                local = [c for c in expand(open(f"/sys/devices/system/node/node{node}/cpulist").read()) if c in cpus]
                if len(local) >= 2:
                    cpus = local
                    info["cores_on_gpu_node"] = len(local)
            except Exception:
                pass
        if world > 1 and len(cpus) >= 2 * world:
            per = len(cpus) // world
            mine = cpus[(local_rank % world) * per:(local_rank % world + 1) * per]
            os.sched_setaffinity(0, mine)
            info["cores"] = f"{mine[0]}-{mine[-1]}"
    except Exception:
        pass
    if node >= 0:
        try:   # set_mempolicy(MPOL_PREFERRED = 1, nodemask, maxnode): pinned buffers land next to the GPU
            import ctypes
            libc = ctypes.CDLL(None, use_errno=True)
            mask = ctypes.c_ulong(1 << node)
            rc = libc.syscall(238, 1, ctypes.byref(mask), ctypes.c_ulong(64))
            info["mempolicy_preferred_node"] = node if rc == 0 else f"refused (errno {ctypes.get_errno()})"
        except Exception:
            pass
    return info


def run_gpu(args, rank, world, local_rank):
    import hashlib
    import torch
    import torch.distributed as dist
    numa = numa_place(local_rank, world)
    import ofdm_b200 as G
    from ofdm_b200 import layouts, sweep

    torch.cuda.set_device(local_rank)
    ctx = G.Context(local_rank, "f32")
    lp = layouts.task5_link(ctx, comb=4)         # M1 shape: the package's own layout helpers (no oracle in this arm)

    class _P:                                    # the handful of sizes the rest of this function reads
        Nfft, T_Guard, N_carrier, N_symb, stream_bits = lp.Nfft, lp.Tg, lp.N_carrier, lp.S, lp.stream_bits
    p = _P
    B = args.streams
    S = p.N_symb
    words = p.stream_bits // 32
    dev = ctx.device
    # ---- synthetic inputs, generated on the device in chunks (TX chain + Task-5 channel)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1000 + rank)
    tx_bits = torch.randint(-2**31, 2**31 - 1, (B * words,), dtype=torch.int32, device=dev, generator=gen)
    rx = torch.empty((B, S, p.Nfft + p.T_Guard), dtype=torch.complex64, device=dev)
    h_dev = ctx.cplx(ctx.mp_channel_resp(TAPS5, p.Nfft)[0])
    chunk = min(B, 2048)
    for c0 in range(0, B, chunk):
        nb = min(chunk, B - c0)
        tx = ctx.tx_chain(lp, tx_bits[c0 * words:(c0 + nb) * words], nb)
        ctx.channel_t5(tx, snr_db=SNR_DB, h_dev=h_dev, seed=42, first_stream_id=rank * B + c0, out=rx[c0:c0 + nb].reshape(nb, -1))
        del tx
    out_bits = torch.empty(B * words, dtype=torch.int32, device=dev)
    H = torch.empty((B, p.N_carrier), dtype=torch.complex64, device=dev)
    counts = torch.zeros(3, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()

    def step(eps=args.near_eps):
        ctx.rx_chain_t5(lp, rx, B, tx_bits_dev=tx_bits, out_bits=out_bits, H=H, counts=counts, near_eps=eps)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    counts.zero_()
    l0 = ctx.launches
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    ev[0].record()
    for i in range(args.steps):
        step()
        ev[i + 1].record()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, B, words, out_bits, H, counts, args.steps)
    if world > 1:
        dist.all_reduce(counts)             # the chain's only collective: int64 error / bit counters
    barrier()
    launches = ctx.launches - l0
    cnt = counts.cpu().numpy()              # counters of exactly the timed steps
    total_ms = ev[0].elapsed_time(ev[-1])
    kernel_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    # keep the GPU busy a little longer so the clock sampler sees load even for very short runs
    t_end = time.time() + 1.0
    while rank == 0 and time.time() < t_end and len(sampler.samples) < 8:
        step()
        torch.cuda.synchronize()
    sampler.stop_flag = True
    syms_per_step = B * S
    value = world * syms_per_step * args.steps / (total_ms * 1e-3)
    # the same kernel without the near-boundary counter (NEAR = false instantiation), for the cost of the counting
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    step(0.0)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(max(3, args.steps // 4)):
        step(0.0)
    e1.record()
    torch.cuda.synchronize()
    near_off_ms = e0.elapsed_time(e1) / max(3, args.steps // 4)

    # ---- e2e: host buffers through the C-ABI host entry (H2D of rx + tx bits, D2H of bits + H + counters)
    Be = min(B, args.e2e_streams)
    rx_h = torch.empty((Be, S, p.Nfft + p.T_Guard), dtype=torch.complex64).pin_memory()
    rx_h.copy_(rx[:Be])
    tb_h = torch.empty(Be * words, dtype=torch.int32).pin_memory()
    tb_h.copy_(tx_bits[:Be * words])
    ob_h = torch.empty(Be * words, dtype=torch.int32).pin_memory()
    H_h = torch.empty((Be, p.N_carrier), dtype=torch.complex64).pin_memory()
    torch.cuda.synchronize()
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        ctx.rx_chain_t5_host(lp, rx_h, Be, tb_h, ob_h, H_h, chunk=args.e2e_chunk)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        c_host = ctx.rx_chain_t5_host(lp, rx_h, Be, tb_h, ob_h, H_h, chunk=args.e2e_chunk, near_eps=args.near_eps)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_val = world * Be * S * e2e_steps / e2e_s
    h2d = Be * S * p.Nfft * 8 + tb_h.numel() * 4      # the host entry leaves the cyclic prefix on the host (strided H2D copy)
    d2h = ob_h.numel() * 4 + H_h.numel() * 8 + 24
    # host-side ceiling of the same transfer: a plain pinned H2D copy of the step's input bytes, all ranks at once
    stage = torch.empty(h2d // 8, dtype=torch.complex64, device=dev)
    src = rx_h.reshape(-1)[:stage.numel()]
    stage.copy_(src, non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(3):
        stage.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    cp_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([cp_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        cp_s = float(t.item())
    h2d_ceiling_gbs = world * 3 * stage.numel() * 8 / cp_s / 1e9
    del stage, rx_h, tb_h, ob_h, H_h

    # ---- M5 (BASELINE config 5): the full TX -> channel -> RX BER-vs-SNR sweep, STRONG scaling (fixed total work), one
    # ofdm_sweep_ber call per rank + the path's only collective (int64 all-reduce).  Reported beside the headline.
    m5 = {}
    del rx, out_bits, H
    torch.cuda.empty_cache()
    snrs = np.arange(0.0, 30.0 + 1e-9, 0.5)
    for chain, spp, taps, A_sym in (("task5", args.m5_streams, layouts.TAPS_TASK5, 144713.0), ("task4", args.m5_streams_t4, layouts.TAPS_TASK4, None)):
        if spp <= 0:
            continue
        lps = lp if chain == "task5" else layouts.task4_link(ctx)
        # The Task-4 leg costs more at low SNR (streams whose detector fails in the prefix take the full-length autocorrelation
        # re-scan), so its points are handed over in low / high interleaved order (0, 30, 0.5, 29.5, ...): every contiguous rank
        # share then holds the same mix.  `order` maps list position -> SNR index; the record is reported in SNR order.
        order = np.arange(len(snrs))
        if chain == "task4":
            order = np.array([k // 2 if k % 2 == 0 else len(snrs) - 1 - k // 2 for k in range(len(snrs))])
        snr_list = snrs[order]
        sweep.ber_sweep(ctx, lps, snr_list[:2], args.m5_tile * world, taps, chain, seed=7, rank=rank, world=world, tile=args.m5_tile)   # warm the pool
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launches
        e0.record()
        acc = sweep.sweep_local(ctx, lps, snr_list, spp, taps, chain, seed=7, rank=rank, world=world, tile=args.m5_tile, near_eps=args.near_eps)
        if world > 1:
            dist.all_reduce(acc)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        res = np.empty_like(acc.cpu().numpy())
        res[order] = acc.cpu().numpy()                        # back to SNR order
        syms = len(snrs) * spp * lps.S
        ber = res[:, 0] / np.maximum(res[:, 1], 1)
        rec = {"workload": f"SNR 0:0.5:30 (61 points{', handed over low/high interleaved' if chain == 'task4' else ''}) x {spp} streams x {lps.S} symbols, {chain} chain, tile {args.m5_tile} streams",
               "scaling": "strong", "symbols": int(syms), "ms": ms, "symbols_per_s": syms / ms * 1e3,
               "kernels_this_rank": int(ctx.launches - l0), "counters_sha1": hashlib.sha1(res.tobytes()).hexdigest(),
               "ber_at_0_10_20_30_dB": [float(ber[i]) for i in (0, 20, 40, 60)], "near_boundary": int(res[:, 2].sum()),
               "detector_failures": int(res[:, 3].sum())}
        if A_sym:
            pk = load_peaks()[0]
            rec["algorithmic_bytes_per_symbol"] = A_sym      # 36,864 TX write + 73,728 channel read+write + 34,121 RX
            rec["hbm_frac_per_gpu"] = A_sym * syms / (ms * 1e-3) / 1e9 / world / pk
        m5[chain] = rec

    if rank != 0:
        return
    peak, peak_src = load_peaks()
    k_ms = float(np.mean(kernel_ms))
    achieved = A_M1 * syms_per_step / (k_ms * 1e-3) / 1e9
    traffic = load_traffic()
    line = {
        "metric": METRIC, "value": value, "unit": "symbols/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "streams_per_gpu": B, "symbols_per_step_per_gpu": syms_per_step,
                   "input_bytes_per_gpu": int(B * S * (p.Nfft + p.T_Guard) * 8), "l2_policy": "inputs (33.8 GB at the default batch) larger than L2; no flush needed",
                   "noise": "Philox4x32-10 keyed by global stream id", "e2e_streams": Be, "e2e_chunk_streams": args.e2e_chunk,
                   "ber": float(cnt[0]) / max(float(cnt[1]), 1.0),
                   "near_eps": args.near_eps, "near_boundary_symbols_per_step": int(cnt[2]) // max(args.steps, 1) // world,
                   "data_symbols_per_step": int(cnt[1]) // 4 // max(args.steps, 1) // world,
                   "ms_per_step_without_near_counter": near_off_ms},
        "clocks": sampler.summary(),
        "e2e": {"value": e2e_val, "unit": "symbols/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "h2d_gbs": world * h2d * e2e_steps / e2e_s / 1e9, "plain_pinned_h2d_copy_gbs_all_ranks": h2d_ceiling_gbs,
                "streams": Be, "why_not_headline_batch": "pinning 33.8 GB per rank takes longer than the measurement; the rate is set by the host link, not by the batch",
                "numa": numa},
        "m5": m5,
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": ((traffic or {}).get("dram_bytes_per_symbol") or 0) * syms_per_step or None, "peak_source": peak_src,
                     "traffic_source": (traffic or {}).get("source"),
                     "kernel": "rx4096_kernel<NEAR=%s>" % ("true" if args.near_eps > 0 else "false"), "algorithmic_bytes_per_symbol": A_M1, "kernel_ms": k_ms},
    }
    if world == 1 and not args.no_cpu:
        n_proc = os.cpu_count() or 1
        v, syms, wall, tot = cpu_baseline(n_proc, args.ref_streams, target_s=args.cpu_seconds)
        line["cpu_baseline"] = {"value": v, "unit": "symbols/s", "cores": n_proc, "kind": "port",
                                "sample": f"{n_proc} processes x {args.ref_streams} distinct streams x 14 symbols of the same workload, repeated: "
                                          f"{syms} symbols in {wall:.1f} s of RX-chain time per process (NumPy float64 oracle, vectorised descrambler)"}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--streams", type=int, default=65536, help="streams per GPU per step (M1: 65,536 = 917,504 symbols)")
    ap.add_argument("--e2e-streams", type=int, default=8192)
    ap.add_argument("--m5-streams", type=int, default=8192, help="streams per SNR point of the Task-5 sweep record (0 = skip)")
    ap.add_argument("--m5-streams-t4", type=int, default=8192, help="streams per SNR point of the Task-4 (STO/CFO) sweep record (0 = skip)")
    ap.add_argument("--m5-tile", type=int, default=8192)
    ap.add_argument("--e2e-chunk", type=int, default=512)
    ap.add_argument("--ref-streams", type=int, default=200, help="distinct streams per host process in the CPU sample")
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="RX-chain time per host process in the CPU sample")
    ap.add_argument("--near-eps", type=float, default=1e-4,
                    help="squared-distance margin below which a decision counts as 'within epsilon of a boundary' (0 = counter off)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy (GPU path)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; the reference arm has none to write")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_gpu(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
