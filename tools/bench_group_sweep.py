#!/usr/bin/env python
"""ofdm_group_sweep_ber on bench.py's M5 workload, in ONE process, at 1, 2, 4 and 8 members on distinct GPUs (as many as
the box has), beside bench.py's own torch.distributed figure on the same box.

    python tools/bench_group_sweep.py [--out profiles/<name>.json] [--no-distributed]

Workload (bench.py's M5 record): SNR 0:0.5:30 (61 points) x 8,192 streams x 14 symbols, Task-5 chain (Nfft 4096, comb 4,
16QAM, the channel of `Task 5/Main_model_Task_5.m:112-119`) and Task-4 chain with the SNR points handed over low / high
interleaved, seed 7, tile 8,192, near_eps 1e-4.  Each group size is warmed up with one call first; the timed call is a host
clock around ofdm_group_sweep_ber, which returns synchronised (thread start, the sweep on every member, the D2H of the
counters).  The counters must be identical for every group size (counters_sha1, in SNR order as bench.py hashes them)."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ofdm_b200 as G  # noqa: E402
from ofdm_b200 import layouts  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return [line.strip() for line in q.stdout.splitlines() if line.strip()] or [q.stderr.strip()]


def distributed_bench(n):
    """bench.py --gpus n under torch.distributed.run: its JSON result line (m5 records), run from a scratch directory"""
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
               "--master-port", "29531", os.path.join(ROOT, "bench.py"), "--gpus", str(n), "--steps", "5", "--warmup", "2", "--no-cpu"]
        r = subprocess.run(cmd, capture_output=True, text=True, cwd=tmp)
    shown = " ".join(["python"] + cmd[1:9] + ["bench.py"] + cmd[10:])
    for line in reversed(r.stdout.splitlines()):
        if line.startswith("{"):
            res = json.loads(line)
            return {"command": shown, "m5": res.get("m5")}
    return {"command": shown, "error": (r.stderr or r.stdout)[-2000:]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams-per-point", type=int, default=8192)
    ap.add_argument("--tile", type=int, default=8192)
    ap.add_argument("--out", help="also write the JSON record here")
    ap.add_argument("--no-distributed", action="store_true", help="skip the torch.distributed bench.py run")
    a = ap.parse_args()
    n_gpus = torch.cuda.device_count()
    if n_gpus == 0:
        raise SystemExit("no CUDA device: this benchmark measures GPUs")
    sizes = [n for n in (1, 2, 4, 8) if n <= n_gpus]
    ctx = G.Context(0, "f32")                     # only for the link parameters' host arrays
    snrs = np.arange(0.0, 30.0 + 1e-9, 0.5)
    out = {"gpus": gpu_info(), "n_gpus_visible": n_gpus, "workloads": {}}
    groups = {n: G.Group(range(n)) for n in sizes}
    for chain in ("task5", "task4"):
        lp, taps = (layouts.task5_link(ctx, comb=4), layouts.TAPS_TASK5) if chain == "task5" else (layouts.task4_link(ctx), layouts.TAPS_TASK4)
        order = np.arange(len(snrs))
        if chain == "task4":
            order = np.array([k // 2 if k % 2 == 0 else len(snrs) - 1 - k // 2 for k in range(len(snrs))])
        snr_list = snrs[order]
        syms = len(snrs) * a.streams_per_point * lp.S
        runs = []
        for n in sizes:
            g = groups[n]
            g.sweep_ber(lp, snr_list[:2], a.tile * n, taps, chain, seed=7, tile=a.tile)      # warm-up: pools, modules
            t0 = time.perf_counter()
            acc = g.sweep_ber(lp, snr_list, a.streams_per_point, taps, chain, seed=7, tile=a.tile, near_eps=1e-4)
            dt = time.perf_counter() - t0
            res = np.empty_like(acc)
            res[order] = acc
            runs.append({"members": n, "devices": list(range(n)), "seconds": dt, "symbols_per_s": syms / dt,
                         "counters_sha1": hashlib.sha1(res.tobytes()).hexdigest()})
        for r in runs:
            r["scaling_vs_1"] = r["symbols_per_s"] / runs[0]["symbols_per_s"]
            r["efficiency"] = r["scaling_vs_1"] / r["members"]
        out["workloads"][chain] = {
            "workload": f"SNR 0:0.5:30 (61 points{', handed over low/high interleaved' if chain == 'task4' else ''}) x {a.streams_per_point} "
                        f"streams x {lp.S} symbols, {chain} chain, tile {a.tile}, one process, ofdm_group_sweep_ber",
            "symbols": syms, "runs": runs, "counters_identical": len({r["counters_sha1"] for r in runs}) == 1}
    for g in groups.values():
        g.close()
    ctx.close()
    if not a.no_distributed:
        out["torch_distributed_bench"] = distributed_bench(sizes[-1])
    txt = json.dumps(out)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
