"""Which CUDA kernels a call launched, read from the CUDA activity of `torch.profiler`, and a per-module registry of what the
cases of a test module saw.  Shared by the kernel-variant matrices (`test_gpu_fast4096_variants.py`,
`test_gpu_fast1024_variants.py`); `parse_kernel` is checked on the CPU in `test_kernel_witness_cpu.py`.

Also `t4_phase_bounds`, the interval the Task-4 phase estimate may take, which both matrices use for the M2 receiver."""
import re

import numpy as np

import oracle as O


def _targ(x):
    x = re.sub(r"^\((?:unsigned\s+)?(?:int|long|short|char|bool)\)\s*", "", x.strip())
    if x in ("true", "false"):
        return x == "true"
    m = re.fullmatch(r"(-?(?:0x[0-9a-fA-F]+|\d+))[uUlL]*", x)
    return int(m.group(1), 0) if m else x


def parse_kernel(name):
    """'void rx4096_kernel<true, false, (int)257, true>(Fast4096Params, ...)' -> ('rx4096_kernel', (True, False, 257, True));
    None for activity that is not a kernel (memsets, copies)."""
    s = name.strip()
    if s.startswith("void "):
        s = s[5:]
    m = re.match(r"[A-Za-z_][\w:]*", s)
    if not m:
        return None
    ident, i, args = m.group(0).split("::")[-1], m.end(), ()
    if i < len(s) and s[i] == "<":
        depth, parts, cur = 0, [], ""
        for j in range(i, len(s)):
            ch = s[j]
            if ch in "<(":
                depth += 1
                if depth == 1 and ch == "<":
                    continue
            elif ch in ">)":
                depth -= 1
                if depth == 0:
                    break
            if ch == "," and depth == 1:
                parts.append(cur)
                cur = ""
            else:
                cur += ch
        parts.append(cur)
        args, i = tuple(_targ(x) for x in parts), j + 1
    if i >= len(s) or s[i] != "(":
        return None
    return ident, args


def witness(fn):
    """Run fn() under torch.profiler (CUDA activity only); returns (fn's result, parsed kernels in launch order) -- kernels is
    None when the profiler recorded no CUDA activity (no CUPTI on this box)."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA]
    if not names:
        return out, None
    return out, [k for k in map(parse_kernel, names) if k is not None]


class Registry:
    """What the cases of one test module launched: seen[(kernel, template arguments)] = ids of the cases that launched it,
    ran = ids of the matrix cases that ran in this session, available = False once a profiled call recorded no CUDA activity
    at all (None before any)."""

    def __init__(self):
        self.seen = {}
        self.ran = set()
        self.available = None

    def record(self, kernels, case):
        """Adds one profiled call's kernels; False when the profiler saw nothing, so the caller skips its kernel asserts."""
        if kernels is None:
            self.available = False
            return False
        if self.available is None:
            self.available = True
        for k in kernels:
            self.seen.setdefault(k, set()).add(case)
        return True


def t4_phase_bounds(p, rx, ref, time_desync=True, freq_desync=True):
    """Interval of fine_sync's phase_shift (`fine_sync.m:47-52`, the mean of the pilot angles above 1e-3) over the signs of exact
    zeros.  The pilots of a symbol that add_STO zero-filled give tx * conj(rx) = +-0 +-0j, whose angle is 0, +pi or -pi depending
    only on the signs of the zeros (the order of the arithmetic, not its accuracy): such a pilot is left out of the mean or
    counted at +pi or -pi, and each one moves the mean by about pi / n.  Returns (lo, hi) over every choice; the oracle's own value
    is one of them.  `ref` is OC.rx_chain_task4's result on the same stream with the same stages on."""
    x = np.asarray(rx, dtype=np.complex128).ravel()
    # the oracle's receiver up to fine_sync (OC.rx_chain_task4), with its own integer and frequency estimates
    if time_desync:
        x = O.add_STO(O.add_STO(x, ref["TgPosition"]), -(p.Nfft + p.T_Guard))
    if freq_desync:
        x = O.add_CFO(x, -ref["FreqOffset"], p.Nfft)
        if ref["IFO"] >= 0:                                                           # IFO = -1: no bin above 0.77, none removed
            x, _ = O.remove_IFO(x, p.Nfft)
    Y = O.OFDM_demodulator(x.reshape((p.Nfft + p.T_Guard, p.N_symb), order="F"), p.T_Guard)
    pc = np.asarray(p.pilotCarriers)
    rxp = Y[pc - 1, :]
    if time_desync:
        rxp = rxp * np.exp(2j * np.pi * ref["tau"] * (pc - 1))[:, None]            # `fine_sync.m:39-42`
    prod = p.pilotValues.ravel(order="F") * np.conj(rxp.ravel(order="F"))
    zero = prod == 0
    a = np.angle(prod[~zero])
    a = a[np.abs(a) > 1e-3]
    z = int(zero.sum())
    means = [(a.sum() + np.pi * (kp - km)) / (a.size + kp + km) for kp in range(z + 1) for km in range(z + 1 - kp)]
    return min(means), max(means)
