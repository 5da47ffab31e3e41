"""Host-side mirror of the reference's function boundary, on top of the C ABI.

Two layers:

* :class:`Context` -- thin, batched, device-resident wrappers (torch CUDA tensors in/out), one
  method per C entry point of ``include/ofdm_b200.h``.
* module-level functions with the **reference's names, argument order and return shapes**
  (``Scrambler``, ``mapping``, ``OFDM_demodulator``, ``LS_CE`` ...): host NumPy arrays in and out,
  1-based index vectors, column-major matrices -- what the MATLAB wrappers in ``matlab/`` do through
  the MEX gateway, written in Python because neither MATLAB nor Octave exists in the build image.

PyTorch is used for device memory and streams only.  Nothing here computes on the CPU and nothing
imports ``oracle``; without the CUDA library the import of ``_cabi`` raises.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _cabi

CONSTELLATIONS = {"BPSK": 1, "QPSK": 2, "8PSK": 3, "16QAM": 4}
TDL_PROFILES = {"EPA": 0, "EVA": 1, "ETU": 2}
DEFAULT_REGISTER = np.array([1, 0, 0, 1, 0, 1, 0, 1, 0, 0, 0, 0, 0, 0, 0], dtype=np.uint8)


class OfdmError(RuntimeError):
    pass


def _i32(a):
    a = np.ascontiguousarray(np.asarray(a).ravel(), dtype=np.int32)
    return a, a.ctypes.data_as(_cabi.pi32)


def _f64c(a):
    """complex host array -> interleaved doubles"""
    a = np.ascontiguousarray(np.asarray(a, dtype=np.complex128))
    return a, a.ctypes.data_as(_cabi.pdbl)


def pack_bits(bits):
    """0/1 array -> packed uint32 words, LSB-first (the device bit layout)."""
    b = np.asarray(bits).ravel().astype(np.uint8)
    by = np.packbits(b, bitorder="little")
    pad = (-by.size) % 4
    if pad:
        by = np.concatenate([by, np.zeros(pad, dtype=np.uint8)])
    return by.view(np.uint32).copy()


def unpack_bits(words, n_bits):
    w = np.ascontiguousarray(np.asarray(words, dtype=np.uint32))
    return np.unpackbits(w.view(np.uint8), bitorder="little")[:n_bits]


class Context:
    """One context per GPU (``ofdm_ctx``).  ``precision``: 'f32' (default) or 'f64'."""

    def __init__(self, device=0, precision="f32"):
        self.lib = _cabi.load()
        if not torch.cuda.is_available():
            raise OfdmError("no CUDA device: ofdm_b200 has no CPU fallback")
        self.device = torch.device("cuda", device)
        self.f64 = precision in ("f64", 1, "double")
        h = C.c_void_p()
        rc = self.lib.ofdm_ctx_create(C.byref(h), device, 1 if self.f64 else 0)
        if rc != 0:
            raise OfdmError(f"ofdm_ctx_create failed with status {rc} (no sm_100 device?)")
        self.h = h
        self.cdtype = torch.complex128 if self.f64 else torch.complex64
        self.rdtype = torch.float64 if self.f64 else torch.float32
        with torch.cuda.device(self.device):
            self._stream = torch.cuda.current_stream()
            self._chk(self.lib.ofdm_ctx_set_stream(self.h, C.c_void_p(self._stream.cuda_stream or 1)))  # 0 -> cudaStreamLegacy

    def close(self):
        if getattr(self, "h", None):
            self.lib.ofdm_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---------------------------------------------------------------- helpers
    def _chk(self, rc):
        if rc != 0:
            raise OfdmError(f"status {rc}: {self.lib.ofdm_last_error(self.h).decode()}")

    def use_current_stream(self):
        s = torch.cuda.current_stream(self.device)
        self._stream = s
        self._chk(self.lib.ofdm_ctx_set_stream(self.h, C.c_void_p(s.cuda_stream or 1)))

    def sync(self):
        self._chk(self.lib.ofdm_sync(self.h))

    @property
    def launches(self):
        return int(self.lib.ofdm_launch_count(self.h))

    def cplx(self, a):
        """host/any array -> contiguous complex device tensor of the context's type"""
        if isinstance(a, torch.Tensor):
            return a.to(self.device, self.cdtype).contiguous()
        return torch.from_numpy(np.ascontiguousarray(np.asarray(a, dtype=np.complex128))).to(self.device).to(self.cdtype).contiguous()

    def real(self, a, dtype=torch.float64):
        if isinstance(a, torch.Tensor):
            return a.to(self.device, dtype).contiguous()
        return torch.from_numpy(np.ascontiguousarray(np.asarray(a))).to(self.device).to(dtype).contiguous()

    def bits(self, bits):
        """0/1 host array -> packed int32 device tensor"""
        return torch.from_numpy(pack_bits(bits).view(np.int32)).to(self.device)

    def empty_c(self, *shape):
        return torch.empty(shape, dtype=self.cdtype, device=self.device)

    def zeros_words(self, n_bits):
        return torch.zeros((n_bits + 31) // 32, dtype=torch.int32, device=self.device)

    @staticmethod
    def p(t):
        return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)

    def host_bits(self, words, n_bits):
        return unpack_bits(words.cpu().numpy().view(np.uint32), n_bits)

    def link_params(self, Nfft, Tg, N_carrier, S, SpF, constellation, dataCarriers, pilotCarriers, pilotValues,
                    Register=DEFAULT_REGISTER, scramble=True):
        """Build an ``ofdm_link_params`` (keeps the host arrays alive on the returned object)."""
        lp = _cabi.LinkParams()
        keep = []
        d, dp = _i32(dataCarriers)
        pc, pp = _i32(pilotCarriers)
        pv = np.asarray(pilotValues, dtype=np.complex128)
        if pv.ndim == 1:
            pv = np.tile(pv[:, None], (1, S))
        pv, pvp = _f64c(np.asfortranarray(pv).ravel(order="F"))
        reg = np.ascontiguousarray(np.asarray(Register, dtype=np.uint8))
        keep += [d, pc, pv, reg]
        lp.Nfft, lp.Tg, lp.N_carrier, lp.S, lp.SpF = int(Nfft), int(Tg), int(N_carrier), int(S), int(SpF)
        lp.constellation = CONSTELLATIONS[str(constellation)]
        lp.Nd, lp.Np = d.size, pc.size
        lp.data_carriers_host, lp.pilot_carriers_host, lp.pilot_vals_host = dp, pp, pvp
        lp.reg0_host = reg.ctypes.data_as(_cabi.pu8)
        lp.scramble = 1 if scramble else 0
        lp._keep = keep
        lp.dataCarriers, lp.pilotCarriers, lp.pilotValues = d, pc, pv.reshape(S, pc.size).T.copy()   # (Np, S)
        lp.Register, lp.constellation_name = reg, str(constellation)
        lp.bps = {1: 1, 2: 2, 3: 3, 4: 4}[lp.constellation]
        lp.frame_bits = lp.SpF * lp.Nd * lp.bps
        lp.stream_bits = lp.S * lp.Nd * lp.bps
        lp.stream_len = lp.S * (lp.Nfft + lp.Tg)
        return lp

    # ---------------------------------------------------------------- a1/a2
    def scramble(self, bits_dev, n_frames, frame_bits, Register=DEFAULT_REGISTER, descramble=False, want_regs=False):
        out = torch.empty_like(bits_dev)
        reg = np.ascontiguousarray(np.asarray(Register, dtype=np.uint8))
        regs = torch.empty((n_frames, 15), dtype=torch.uint8, device=self.device) if want_regs else None
        fn = self.lib.ofdm_descramble if descramble else self.lib.ofdm_scramble
        self._chk(fn(self.h, self.p(bits_dev), self.p(out), n_frames, frame_bits, reg.ctypes.data_as(_cabi.pu8), self.p(regs)))
        return (out, regs) if want_regs else out

    # ---------------------------------------------------------------- a4/a5
    def map(self, bits_dev, n_bits, constellation):
        cid = CONSTELLATIONS[str(constellation)]
        bps = {1: 1, 2: 2, 3: 3, 4: 4}[cid]
        n_sym = (n_bits + bps - 1) // bps
        iq = self.empty_c(n_sym)
        pad = C.c_int(0)
        self._chk(self.lib.ofdm_map(self.h, self.p(bits_dev), n_bits, cid, self.p(iq), C.byref(pad)))
        return iq, pad.value

    def demap(self, iq_dev, constellation, near_eps=0.0, want_near=False):
        cid = CONSTELLATIONS[str(constellation)]
        bps = {1: 1, 2: 2, 3: 3, 4: 4}[cid]
        n_sym = iq_dev.numel()
        out = self.zeros_words(n_sym * bps)
        near = torch.zeros(1, dtype=torch.int64, device=self.device) if want_near else None
        self._chk(self.lib.ofdm_demap(self.h, self.p(iq_dev), n_sym, cid, self.p(out), float(near_eps), self.p(near)))
        return (out, int(near.item())) if want_near else out

    # ---------------------------------------------------------------- a6-a9
    def map_carriers(self, qam_dev, B, S, Nfft, dataCarriers, pilotCarriers, pilotValues, pilot_mode=0):
        d, dp = _i32(dataCarriers)
        pc, pp = _i32(pilotCarriers)
        if pilot_mode == 0:
            pv = np.asarray(pilotValues, dtype=np.complex128).reshape(pc.size, -1)
            pv, pvp = _f64c(pv.ravel(order="F"))
        elif pilot_mode == 1:
            pv, pvp = _f64c(np.array([pilotValues]))
        else:
            pv = np.array([float(pilotValues)], dtype=np.float64)
            pvp = pv.ctypes.data_as(_cabi.pdbl)
        grid = self.empty_c(B, S, Nfft)
        self._chk(self.lib.ofdm_map_carriers(self.h, self.p(qam_dev), B, S, Nfft, dp, d.size, pp, pc.size, pvp, pilot_mode, self.p(grid)))
        return grid

    def modulate(self, grid_dev, Tg):
        B, S, Nfft = grid_dev.shape
        out = self.empty_c(B, S, Nfft + Tg)
        self._chk(self.lib.ofdm_modulate(self.h, self.p(grid_dev), B, S, Nfft, Tg, self.p(out)))
        return out

    def demodulate(self, time_dev, Nfft, Tg):
        B, S, _ = time_dev.shape
        out = self.empty_c(B, S, Nfft)
        self._chk(self.lib.ofdm_demodulate(self.h, self.p(time_dev), B, S, Nfft, Tg, self.p(out)))
        return out

    def get_payload(self, grid_dev, dataCarriers):
        B, S, Nfft = grid_dev.shape
        d, dp = _i32(dataCarriers)
        out = self.empty_c(B, S, d.size)
        self._chk(self.lib.ofdm_get_payload(self.h, self.p(grid_dev), B, S, Nfft, dp, d.size, self.p(out)))
        return out

    def fft(self, x_dev, inverse=False):
        N = x_dev.shape[-1]
        out = torch.empty_like(x_dev)
        self._chk(self.lib.ofdm_fft(self.h, self.p(x_dev), self.p(out), x_dev.numel() // N, N, 1 if inverse else 0))
        return out

    # ---------------------------------------------------------------- a10-a13
    def add_sto(self, x_dev, nsto):
        B, L = x_dev.shape
        n = nsto.to(self.device, torch.int32).contiguous() if isinstance(nsto, torch.Tensor) else \
            self.real(np.broadcast_to(np.asarray(nsto), (B,)).copy(), torch.int32)
        out = torch.empty_like(x_dev)
        self._chk(self.lib.ofdm_add_sto(self.h, self.p(x_dev), B, L, self.p(n), self.p(out)))
        return out

    def add_cfo(self, x_dev, cfo, Nfft):
        B, L = x_dev.shape
        c = cfo.to(self.device, torch.float64).contiguous() if isinstance(cfo, torch.Tensor) else \
            self.real(np.broadcast_to(np.asarray(cfo, dtype=np.float64), (B,)).copy())
        out = torch.empty_like(x_dev)
        self._chk(self.lib.ofdm_add_cfo(self.h, self.p(x_dev), B, L, self.p(c), Nfft, self.p(out)))
        return out

    def add_noise(self, x_dev, snr_db, normals_dev=None, seed=0, first_stream_id=0):
        B, L = x_dev.shape
        s = self.real(np.broadcast_to(np.asarray(snr_db, dtype=np.float64), (B,)).copy())
        out = torch.empty_like(x_dev)
        nvar = torch.empty(B, dtype=torch.float64, device=self.device)
        self._chk(self.lib.ofdm_add_noise(self.h, self.p(x_dev), B, L, self.p(s), self.p(normals_dev), seed, first_stream_id, self.p(out), self.p(nvar)))
        return out, nvar

    def mp_channel_resp(self, channel_taps, Nfft):
        taps = np.ascontiguousarray(np.asarray(channel_taps, dtype=np.float64).reshape(-1, 2))
        cap = int(taps[:, 0].max()) + 1
        h = np.zeros(cap, dtype=np.float64)
        hl = C.c_int(0)
        H = self.empty_c(Nfft)
        self._chk(self.lib.ofdm_mp_channel_resp(self.h, taps.ctypes.data_as(_cabi.pdbl), taps.shape[0], Nfft, h.ctypes.data_as(_cabi.pdbl), cap,
                                                C.byref(hl), self.p(H)))
        return h[: hl.value], H

    def apply_fir(self, x_dev, h_dev, per_stream=False):
        B, L = x_dev.shape
        D = h_dev.shape[-1]
        out = torch.empty_like(x_dev)
        self._chk(self.lib.ofdm_apply_fir(self.h, self.p(x_dev), B, L, self.p(h_dev), D, 1 if per_stream else 0, self.p(out)))
        return out

    def tdl_info(self, profile, fs_hz):
        """(n_paths, h_len, delays in samples) of the EPA / EVA / ETU tapped-delay-line model at `fs_hz`."""
        n, hl = C.c_int(0), C.c_int(0)
        d = np.zeros(9, dtype=np.float64)
        rc = self.lib.ofdm_tdl_info(TDL_PROFILES[str(profile).upper()], float(fs_hz), C.byref(n), C.byref(hl), d.ctypes.data_as(_cabi.pdbl))
        if rc != 0:
            raise OfdmError(f"status {rc}: unknown delay profile {profile!r} or sampling rate")
        return n.value, hl.value, d[: n.value]

    def tdl_channel(self, profile, fs_hz, B, seed=0, first_stream_id=0, want_gains=False):
        """Static fading realisations standing in for lteFadingChannel (`Task5_part2.m:152-154`): h (B x h_len)."""
        n, hl, _ = self.tdl_info(profile, fs_hz)
        h = self.empty_c(B, hl)
        g = self.empty_c(B, n) if want_gains else None
        self._chk(self.lib.ofdm_tdl_channel(self.h, TDL_PROFILES[str(profile).upper()], float(fs_hz), B, seed, first_stream_id, hl, self.p(h), self.p(g)))
        return (h, g) if want_gains else h

    def mse(self, a_dev, b_dev, n):
        """Per-stream mean |a - b|^2 over the first n entries of each row (`Task5_part2.m:200-203`)."""
        B = a_dev.shape[0]
        out = torch.empty(B, dtype=torch.float64, device=self.device)
        self._chk(self.lib.ofdm_mse(self.h, self.p(a_dev), a_dev.shape[-1], self.p(b_dev), b_dev.shape[-1], B, n, self.p(out)))
        return out

    # ---------------------------------------------------------------- a14-a16
    def cp_autocorr(self, rx_dev, W, Nfft, want_autocorr=False):
        B, L = rx_dev.shape
        ac = self.empty_c(B, L - W - Nfft) if want_autocorr else None
        tg = torch.empty(B, dtype=torch.int32, device=self.device)
        fo = torch.empty(B, dtype=torch.float64, device=self.device)
        fail = torch.empty(B, dtype=torch.int32, device=self.device)
        self._chk(self.lib.ofdm_cp_autocorr(self.h, self.p(rx_dev), B, L, W, Nfft, self.p(ac), self.p(tg), self.p(fo), self.p(fail)))
        return ac, tg, fo, fail

    def remove_ifo(self, rx_dev, Nfft):
        B, L = rx_dev.shape
        out = torch.empty_like(rx_dev)
        ifo = torch.empty(B, dtype=torch.int32, device=self.device)
        self._chk(self.lib.ofdm_remove_ifo(self.h, self.p(rx_dev), B, L, Nfft, self.p(out), self.p(ifo)))
        return out, ifo

    def fine_sync(self, grid_dev, pilotCarriers, pilotValues, time_desync, freq_desync):
        B, S, Nfft = grid_dev.shape
        pc, pp = _i32(pilotCarriers)
        pv, pvp = _f64c(np.asarray(pilotValues, dtype=np.complex128).reshape(pc.size, -1).ravel(order="F"))
        out = torch.empty_like(grid_dev)
        tau = torch.empty(B, dtype=torch.float64, device=self.device)
        ph = torch.empty(B, dtype=torch.float64, device=self.device)
        self._chk(self.lib.ofdm_fine_sync(self.h, self.p(grid_dev), B, S, Nfft, pp, pc.size, pvp, int(bool(time_desync)), int(bool(freq_desync)),
                                          self.p(out), self.p(tau), self.p(ph)))
        return out, tau, ph

    # ---------------------------------------------------------------- a17-a21
    def estimate_channel(self, grid_dev, allCarriers, pilotCarriers, pilotValues):
        B, S, Nfft = grid_dev.shape
        ac, ap = _i32(allCarriers)
        pc, pp = _i32(pilotCarriers)
        pv, pvp = _f64c(np.asarray(pilotValues, dtype=np.complex128).reshape(pc.size, -1).ravel(order="F"))
        H = self.empty_c(B, ac.size)
        Hp = self.empty_c(B, pc.size)
        self._chk(self.lib.ofdm_estimate_channel(self.h, self.p(grid_dev), B, S, Nfft, ap, ac.size, pp, pc.size, pvp, self.p(H), self.p(Hp)))
        return H, Hp

    def ls_ce(self, grid_dev, Xp, pilot_loc, N_carrier):
        B, S, Nfft = grid_dev.shape
        pc, pp = _i32(pilot_loc)
        pv, pvp = _f64c(np.asarray(Xp, dtype=np.complex128).ravel(order="F")[: pc.size])
        H = self.empty_c(B, N_carrier)
        self._chk(self.lib.ofdm_ls_ce(self.h, self.p(grid_dev), B, S, Nfft, pp, pc.size, pvp, N_carrier, self.p(H)))
        return H

    def mmse_ce(self, grid_dev, Xp, pilot_loc, N_carrier, h_dev, snr_db):
        B, S, Nfft = grid_dev.shape
        pc, pp = _i32(pilot_loc)
        pv, pvp = _f64c(np.asarray(Xp, dtype=np.complex128).reshape(pc.size, -1)[:, 0])
        snr = self.real(np.broadcast_to(np.asarray(snr_db, dtype=np.float64), (B,)).copy())
        H = self.empty_c(B, N_carrier)
        self._chk(self.lib.ofdm_mmse_ce(self.h, self.p(grid_dev), B, S, Nfft, pp, pc.size, pvp, N_carrier, self.p(h_dev), h_dev.shape[-1], self.p(snr), self.p(H)))
        return H

    def mmse_ce_shared(self, grid_dev, Xp, pilot_loc, N_carrier, h_dev, snr_db):
        """MMSE_CE with ONE impulse response ``h_dev`` (1-D) and ONE SNR for the whole batch (``ofdm_mmse_ce_shared``)."""
        B, S, Nfft = grid_dev.shape
        pc, pp = _i32(pilot_loc)
        pv, pvp = _f64c(np.asarray(Xp, dtype=np.complex128).reshape(pc.size, -1)[:, 0])
        H = self.empty_c(B, N_carrier)
        self._chk(self.lib.ofdm_mmse_ce_shared(self.h, self.p(grid_dev), B, S, Nfft, pp, pc.size, pvp, N_carrier, self.p(h_dev), h_dev.numel(),
                                               float(snr_db), self.p(H)))
        return H

    def interpolate(self, Hp_dev, pilot_loc, N, method):
        B = Hp_dev.shape[0]
        pc, pp = _i32(pilot_loc)
        H = self.empty_c(B, N)
        m = 0 if str(method)[0].lower() == "l" else 1
        self._chk(self.lib.ofdm_interpolate(self.h, self.p(Hp_dev), B, pp, pc.size, N, m, self.p(H)))
        return H

    def equalize(self, grid_dev, H_dev, N_carrier):
        B, S, Nfft = grid_dev.shape
        out = torch.empty_like(grid_dev)
        self._chk(self.lib.ofdm_equalize(self.h, self.p(grid_dev), B, S, Nfft, self.p(H_dev), H_dev.shape[-1], N_carrier, self.p(out)))
        return out

    def pilot_ls(self, grid_dev, Xp, pilot_loc):
        """`Y = RX(pilotCarriers,1)./pilotValues(:,1)` (`Main_model_Task_5.m:191`): B x Np."""
        B, S, Nfft = grid_dev.shape
        pc, pp = _i32(pilot_loc)
        pv, pvp = _f64c(np.asarray(Xp, dtype=np.complex128).reshape(pc.size, -1)[:, 0])
        y = self.empty_c(B, pc.size)
        self._chk(self.lib.ofdm_pilot_ls(self.h, self.p(grid_dev), B, S, Nfft, pp, pc.size, pvp, self.p(y)))
        return y

    # ---------------------------------------------------------------- a22/a23
    def _pursuit(self, omp, y_dev, Nfft, K, A_dev=None, Ldict=None, pilot_loc=None, tie_eps=None):
        B, Np = y_dev.shape
        if A_dev is not None:
            Ldict = A_dev.numel() // Np
        H = self.empty_c(B, Nfft)
        h = self.empty_c(B, Nfft)
        idx = torch.zeros((B, K), dtype=torch.int32, device=self.device)
        keep, pp = _i32(pilot_loc) if pilot_loc is not None else (None, None)  # noqa: F841 (keeps the array alive)
        if omp:
            iters = torch.zeros(B, dtype=torch.int32, device=self.device)
            if tie_eps is not None:
                near = torch.zeros(B, dtype=torch.int32, device=self.device)
                self._chk(self.lib.ofdm_omp_ex(self.h, self.p(y_dev), B, Np, self.p(A_dev), Ldict, pp, Nfft, K, self.p(H), self.p(h), self.p(idx), self.p(iters),
                                               self.p(near), float(tie_eps)))
                return H, h, idx, iters, near
            self._chk(self.lib.ofdm_omp(self.h, self.p(y_dev), B, Np, self.p(A_dev), Ldict, pp, Nfft, K, self.p(H), self.p(h), self.p(idx), self.p(iters)))
            return H, h, idx, iters
        self._chk(self.lib.ofdm_mp(self.h, self.p(y_dev), B, Np, self.p(A_dev), Ldict, pp, Nfft, K, self.p(H), self.p(h), self.p(idx)))
        return H, h, idx

    def omp(self, y_dev, Nfft, K, A_dev=None, Ldict=None, pilot_loc=None, tie_eps=None):
        """``tie_eps``: also return per-frame near-tie counts (iterations whose top-2 |A^H r|^2 margin is below tie_eps)."""
        return self._pursuit(True, y_dev, Nfft, K, A_dev, Ldict, pilot_loc, tie_eps)

    def mp(self, y_dev, Nfft, K, A_dev=None, Ldict=None, pilot_loc=None):
        return self._pursuit(False, y_dev, Nfft, K, A_dev, Ldict, pilot_loc)

    # ---------------------------------------------------------------- a24/a25
    def ber_count(self, tx_dev, rx_dev, n_bits, counts=None):
        if counts is None:
            counts = torch.zeros(2, dtype=torch.int64, device=self.device)
        self._chk(self.lib.ofdm_ber_count(self.h, self.p(tx_dev), self.p(rx_dev), n_bits, self.p(counts)))
        return counts

    def mer(self, iq_dev, constellation, sums=None):
        if sums is None:
            sums = torch.zeros(2, dtype=torch.float64, device=self.device)
        self._chk(self.lib.ofdm_mer(self.h, self.p(iq_dev), iq_dev.numel(), CONSTELLATIONS[str(constellation)], self.p(sums)))
        return sums

    # ---------------------------------------------------------------- PAPR / CCDF
    def papr(self, x_dev):
        """`calculatePAPR.m:2-11` per stream (x_dev: B x L) -> B doubles (dB)."""
        B, L = x_dev.shape
        out = torch.empty(B, dtype=torch.float64, device=self.device)
        self._chk(self.lib.ofdm_papr(self.h, self.p(x_dev), B, L, self.p(out)))
        return out

    def window_papr(self, x_dev, Nfft):
        """`calculate_window_PAPR.m:2-15` per stream -> B x (L - Nfft + 1)."""
        B, L = x_dev.shape
        out = torch.empty((B, L - Nfft + 1), dtype=self.rdtype, device=self.device)
        self._chk(self.lib.ofdm_window_papr(self.h, self.p(x_dev), B, L, int(Nfft), self.p(out)))
        return out

    def ccdf(self, values_dev):
        """`calculateCCDF.m:2-6`: (PAPR_ccdf, CCDF) with ecdf's leading duplicate of the minimum."""
        v = values_dev.reshape(-1).contiguous()
        n = v.numel()
        xs = torch.empty(n + 1, dtype=v.dtype, device=self.device)
        cc = torch.empty(n + 1, dtype=v.dtype, device=self.device)
        cnt = torch.zeros(1, dtype=torch.int64, device=self.device)
        self._chk(self.lib.ofdm_ccdf(self.h, self.p(v), n, self.p(xs), self.p(cc), self.p(cnt)))
        k = int(cnt.item())
        return xs[:k], cc[:k]

    def payload_bernoulli(self, n_streams, stream_bits, p_one, seed=1, first_stream_id=0):
        """The Bernoulli payload of ``ofdm_sweep_papr``: streams first_stream_id .. + n_streams - 1 of stream_bits bits as one
        contiguous packed bitstream (int32 words, the input of :meth:`tx_chain`)."""
        out = torch.empty(((int(n_streams) * int(stream_bits) + 31) // 32,), dtype=torch.int32, device=self.device)
        self._chk(self.lib.ofdm_payload_bernoulli(self.h, self.p(out), int(n_streams), int(stream_bits), float(p_one), int(seed), int(first_stream_id)))
        return out

    # ---------------------------------------------------------------- fused chains
    def tx_chain(self, lp, bits_dev, B, want_power=False):
        """TX chain; with ``want_power`` also returns sum |x|^2 per stream (float64, B) for ``channel_t5(power_sum=...)``."""
        out = self.empty_c(B, lp.S, lp.Nfft + lp.Tg)
        if not want_power:
            self._chk(self.lib.ofdm_tx_chain(self.h, C.byref(lp), self.p(bits_dev), B, self.p(out)))
            return out
        psum = torch.empty(B, dtype=torch.float64, device=self.device)
        self._chk(self.lib.ofdm_tx_chain_p(self.h, C.byref(lp), self.p(bits_dev), B, self.p(out), self.p(psum)))
        return out, psum

    def channel_t5(self, tx_dev, snr_db=None, h_dev=None, normals_dev=None, seed=0, first_stream_id=0, out=None, power_sum=None):
        x = tx_dev.reshape(tx_dev.shape[0], -1)
        B, L = x.shape
        if snr_db is None:
            s = None
        elif np.ndim(snr_db) == 0 and not isinstance(snr_db, torch.Tensor):
            s = torch.full((B,), float(snr_db), dtype=torch.float64, device=self.device)      # filled on the device: no host copy, no implicit sync
        else:
            s = self.real(np.broadcast_to(np.asarray(snr_db, dtype=np.float64), (B,)).copy())
        if out is None:
            out = torch.empty_like(x)
        D = h_dev.shape[-1] if h_dev is not None else 0
        self._chk(self.lib.ofdm_channel_t5_p(self.h, self.p(x), B, L, self.p(s), self.p(power_sum), self.p(normals_dev), seed, first_stream_id, self.p(h_dev), D,
                                             self.p(out)))
        return out.reshape(tx_dev.shape)

    def channel_t4(self, tx_dev, snr_db, nsto, cfo, Nfft, h_dev, normals_dev=None, seed=0, first_stream_id=0, out=None, power_sum=None):
        """Task-4 channel in one pass: Noise -> add_STO -> add_CFO -> multipath (`Task 4/Main_model_Task_4.m:95,103,110,263-264`);
        the same bits as add_noise / add_sto / add_cfo / apply_fir called in turn."""
        x = tx_dev.reshape(tx_dev.shape[0], -1)
        B, L = x.shape
        if np.ndim(snr_db) == 0 and not isinstance(snr_db, torch.Tensor):
            s = torch.full((B,), float(snr_db), dtype=torch.float64, device=self.device)
        else:
            s = self.real(np.broadcast_to(np.asarray(snr_db, dtype=np.float64), (B,)).copy())
        n = nsto if isinstance(nsto, torch.Tensor) else torch.as_tensor(np.broadcast_to(np.asarray(nsto, dtype=np.int32), (B,)).copy(), device=self.device)
        c = cfo if isinstance(cfo, torch.Tensor) else self.real(np.broadcast_to(np.asarray(cfo, dtype=np.float64), (B,)).copy())
        if out is None:
            out = torch.empty_like(x)
        self._chk(self.lib.ofdm_channel_t4_p(self.h, self.p(x), B, L, self.p(s), self.p(power_sum), self.p(normals_dev), seed, first_stream_id, self.p(n), self.p(c),
                                             Nfft, self.p(h_dev), h_dev.shape[-1], self.p(out)))
        return out.reshape(tx_dev.shape)

    def rx_chain_t5(self, lp, rx_dev, B, tx_bits_dev=None, want_bits=True, want_H=True, counts=None, near_eps=0.0, want_err_per_stream=False,
                    out_bits=None, H=None):
        if want_bits and out_bits is None:
            out_bits = self.zeros_words(B * lp.stream_bits)
        if want_H and H is None:
            H = self.empty_c(B, lp.N_carrier)
        if counts is None:
            counts = torch.zeros(3, dtype=torch.int64, device=self.device)
        eps = torch.zeros(B, dtype=torch.int32, device=self.device) if want_err_per_stream else None
        self._chk(self.lib.ofdm_rx_chain_t5(self.h, C.byref(lp), self.p(rx_dev), B, self.p(tx_bits_dev), self.p(out_bits) if want_bits else None,
                                            self.p(H) if want_H else None, self.p(counts), self.p(eps), float(near_eps)))
        return {"bits": out_bits, "H": H, "counts": counts, "err_per_stream": eps}

    def rx_chain_t4(self, lp, rx_dev, tx_bits_dev=None, time_desync=True, freq_desync=True, mp_desync=True, near_eps=0.0):
        """Task-4 sync + CE chain on B device-resident streams, the calls of `Task 4/Main_model_Task_4.m:277-366` in
        order: AutoCorrFunction -> add_STO x2 -> add_CFO -> remove_IFO -> OFDM_demodulator -> fine_sync ->
        estimate_channel -> equalize_signal -> get_payload -> demapping -> DeScrambler -> BER count."""
        B = rx_dev.shape[0]
        x = rx_dev.reshape(B, -1)
        info = {}
        if time_desync or freq_desync:
            _, tg, fo, fail = self.cp_autocorr(x, lp.Tg, lp.Nfft)
            info.update(TgPosition=tg, FreqOffset=fo, fail=fail)
            if time_desync:
                x = self.add_sto(x, tg)
                x = self.add_sto(x, -(lp.Nfft + lp.Tg))
        if freq_desync:
            x = self.add_cfo(x, -info["FreqOffset"], lp.Nfft)
            x, ifo = self.remove_ifo(x, lp.Nfft)
            info.update(IFO=ifo)
        grid = self.demodulate(x.reshape(B, lp.S, lp.Nfft + lp.Tg), lp.Nfft, lp.Tg)
        if time_desync or freq_desync:
            grid, tau, ph = self.fine_sync(grid, lp.pilotCarriers, lp.pilotValues, time_desync, freq_desync)
            info.update(tau=tau, phase_shift=ph)
        if mp_desync:
            H, _ = self.estimate_channel(grid, np.arange(1, lp.Nfft + 1), lp.pilotCarriers, lp.pilotValues)
            grid = self.equalize(grid, H, lp.N_carrier)
            info.update(H=H)
        iq = self.get_payload(grid, lp.dataCarriers)
        near = None
        if near_eps > 0:
            raw, near = self.demap(iq.reshape(-1), lp.constellation_name, near_eps, want_near=True)
        else:
            raw = self.demap(iq.reshape(-1), lp.constellation_name)
        frames = lp.S // lp.SpF
        bits = self.scramble(raw, B * frames, lp.frame_bits, lp.Register, descramble=True) if lp.scramble else raw
        info.update(bits=bits, rx_iq=iq, near=near)
        if tx_bits_dev is not None:
            info["counts"] = self.ber_count(tx_bits_dev, bits, B * lp.stream_bits)
        return info

    def rx_chain_t4_fused(self, lp, rx_dev, tx_bits_dev=None, time_desync=True, freq_desync=True, mp_desync=True, near_eps=0.0, want_bits=True,
                          want_H=False):
        """Same chain as :meth:`rx_chain_t4` through the fused C entry ``ofdm_rx_chain_t4`` (FP32 contexts)."""
        B = rx_dev.shape[0]
        dev = self.device
        out_bits = self.zeros_words(B * lp.stream_bits) if want_bits else None
        counts = torch.zeros(3, dtype=torch.int64, device=dev)
        tg = torch.zeros(B, dtype=torch.int32, device=dev)
        fo = torch.zeros(B, dtype=torch.float64, device=dev)
        ifo = torch.zeros(B, dtype=torch.int32, device=dev)
        tau = torch.zeros(B, dtype=torch.float64, device=dev)
        ph = torch.zeros(B, dtype=torch.float64, device=dev)
        H = self.empty_c(B, lp.N_carrier) if want_H else None
        fail = torch.zeros(B, dtype=torch.int32, device=dev)
        self._chk(self.lib.ofdm_rx_chain_t4_ex(self.h, C.byref(lp), self.p(rx_dev), B, int(bool(time_desync)), int(bool(freq_desync)), int(bool(mp_desync)),
                                               self.p(tx_bits_dev), self.p(out_bits), self.p(counts), self.p(tg), self.p(fo), self.p(ifo), self.p(tau),
                                               self.p(ph), self.p(H), float(near_eps), self.p(fail)))
        return {"bits": out_bits, "counts": counts, "TgPosition": tg, "FreqOffset": fo, "IFO": ifo, "tau": tau, "phase_shift": ph, "H": H,
                "near": counts[2], "fail": fail}

    def rx_chain_t5_host(self, lp, rx_host, B, tx_bits_host=None, out_bits_host=None, H_host=None, chunk=2048, near_eps=0.0):
        """Host buffers in, host buffers out (torch CPU tensors, ideally pinned).  Returns counts (3 int64:
        errors, bits, symbols within ``near_eps`` of a decision boundary)."""
        counts = np.zeros(3, dtype=np.int64)
        hp = lambda t: C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)
        self._chk(self.lib.ofdm_rx_chain_t5_host_eps(self.h, C.byref(lp), hp(rx_host), B, hp(tx_bits_host), hp(out_bits_host), hp(H_host),
                                                     counts.ctypes.data_as(C.c_void_p), chunk, float(near_eps)))
        return counts


# ======================================================================================
# Reference-named API (host arrays, one stream per call as in MATLAB)
# ======================================================================================
_default = {}


def default_context(precision="f32"):
    key = "f64" if precision in ("f64", 1, "double") else "f32"
    if key not in _default:
        _default[key] = Context(0, key)
    return _default[key]


def _ctx(precision):
    return default_context(precision)


def constellation_func(Constellation):
    """`Task 5/constellation_func.m:4-29` -> (Dictionary, Bit_depth_Dict); table from the library."""
    lib = _cabi.load()
    tab = np.zeros(32, dtype=np.float64)
    bps = C.c_int(0)
    rc = lib.ofdm_constellation(CONSTELLATIONS[str(Constellation)], tab.ctypes.data_as(_cabi.pdbl), C.byref(bps))
    if rc:
        raise OfdmError("unknown constellation")
    n = 1 << bps.value
    return tab[0:2 * n:2] + 1j * tab[1:2 * n:2], bps.value


def Scrambler(Register, sequence, precision="f32"):
    """`Task 5/Scrambler.m:1` -> [sc_sequence, Register]"""
    c = _ctx(precision)
    seq = np.asarray(sequence).ravel()
    out, regs = c.scramble(c.bits(seq), 1, seq.size, Register, want_regs=True)
    return c.host_bits(out, seq.size), regs.cpu().numpy()[0]


def DeScrambler(Register, sequence, precision="f32"):
    """`Task 5/DeScrambler.m:1` -> [dsc_sequence, Register]"""
    c = _ctx(precision)
    seq = np.asarray(sequence).ravel()
    out, regs = c.scramble(c.bits(seq), 1, seq.size, Register, descramble=True, want_regs=True)
    return c.host_bits(out, seq.size), regs.cpu().numpy()[0]


def mapping(bits, constellation, precision="f32"):
    """`Task 5/mapping.m:1` -> [IQ, pad]"""
    c = _ctx(precision)
    b = np.asarray(bits).ravel()
    iq, pad = c.map(c.bits(b), b.size, constellation)
    return iq.cpu().numpy(), pad


def demapping(pad, IQ, Constellation, precision="f32"):
    """`Task 5/demapping.m:1` -> de_bits (1 x N)"""
    c = _ctx(precision)
    iq = c.cplx(np.asarray(IQ).ravel())
    _, bps = constellation_func(Constellation)
    words = c.demap(iq, Constellation)
    bits = c.host_bits(words, iq.numel() * bps)
    return bits[: bits.size - pad] if pad != -1 else bits


def _grid_to_dev(c, X):
    """(Nfft, S) column-major host matrix -> device (1, S, Nfft)"""
    X = np.asarray(X)
    return c.cplx(np.ascontiguousarray(X.T))[None]


def _grid_to_host(t):
    return t[0].cpu().numpy().T.copy()


def OFDM_map_carriers(QAM_payload, N_symb, Nfft, dataCarriers, pilotCarriers, pilotValues, precision="f32"):
    """`Task 5/OFDM_map_carriers.m:2` (v2; a scalar ``pilotValues`` broadcasts as in MATLAB)."""
    c = _ctx(precision)
    q = c.cplx(np.asarray(QAM_payload).ravel())
    mode = 1 if np.ndim(pilotValues) == 0 else 0
    return _grid_to_host(c.map_carriers(q, 1, N_symb, Nfft, dataCarriers, pilotCarriers, pilotValues, mode))


def OFDM_map_carriers_v1(QAM_payload, N_symb, Nfft, dataCarriers, pilotCarriers, amp_pilots, precision="f32"):
    """`Task 1/OFDM_map_carriers.m:2` (v1: alternating +a / a*exp(i*pi) pilots, 50 symbols)."""
    if N_symb != 50:
        raise OfdmError("Task-1 OFDM_map_carriers hard-codes repmat(...,1,50)")
    c = _ctx(precision)
    q = c.cplx(np.asarray(QAM_payload).ravel())
    return _grid_to_host(c.map_carriers(q, 1, N_symb, Nfft, dataCarriers, pilotCarriers, amp_pilots, 2))


def OFDM_modulator(OFDM_symbols, T_guard, precision="f32"):
    """`Task 5/OFDM_modulator.m:2`"""
    c = _ctx(precision)
    return _grid_to_host(c.modulate(_grid_to_dev(c, OFDM_symbols), int(T_guard)))


def OFDM_demodulator(OFDM_time_guarded, T_guard, precision="f32"):
    """`Task 5/OFDM_demodulator.m:2`"""
    c = _ctx(precision)
    X = np.asarray(OFDM_time_guarded)
    return _grid_to_host(c.demodulate(_grid_to_dev(c, X), X.shape[0] - int(T_guard), int(T_guard)))


def get_payload(RX_OFDM_symbols, dataCarriers, precision="f32"):
    """`Task 5/get_payload.m:2`"""
    c = _ctx(precision)
    return _grid_to_host(c.get_payload(_grid_to_dev(c, RX_OFDM_symbols), dataCarriers))


def add_STO(y, nSTO, precision="f32"):
    """`Task 5/add_STO.m:1`"""
    c = _ctx(precision)
    return c.add_sto(c.cplx(np.asarray(y).ravel())[None], int(nSTO))[0].cpu().numpy()


def add_CFO(y, CFO, Nfft, precision="f32"):
    """`Task 5/add_CFO.m:1`"""
    c = _ctx(precision)
    return c.add_cfo(c.cplx(np.asarray(y).ravel())[None], float(CFO), int(Nfft))[0].cpu().numpy()


def Noise(SNR, IQ_TX, normals=None, seed=0, precision="f32"):
    """`Task 5/Noise.m:1` -> [IQ_RX, N_var].  ``normals`` (2, L) imports a shared realisation (real block,
    imaginary block); without it the library draws Philox normals from ``seed``."""
    c = _ctx(precision)
    x = c.cplx(np.asarray(IQ_TX).ravel())[None]
    nd = c.real(np.asarray(normals)[None], c.rdtype) if normals is not None else None
    out, nvar = c.add_noise(x, float(SNR), nd, seed)
    return out[0].cpu().numpy(), float(nvar[0].item())


def get_MP_channel_resp(channel_taps, Nfft, precision="f32"):
    """`Task 5/get_MP_channel_resp.m:2` -> [impulse_response, frequency_response]"""
    c = _ctx(precision)
    h, H = c.mp_channel_resp(channel_taps, int(Nfft))
    return h, H.cpu().numpy()


def apply_channel(x, h, precision="f32"):
    """``conv(x, h.', 'full')`` truncated to ``length(x)`` (`Task 5/Main_model_Task_5.m:126-127`)."""
    c = _ctx(precision)
    return c.apply_fir(c.cplx(np.asarray(x).ravel())[None], c.cplx(np.asarray(h).ravel()))[0].cpu().numpy()


def AutoCorrFunction(RxSignal, WidthWindow, Nfft, precision="f32"):
    """`Task 5/AutoCorrFunction.m:1` -> [AutoCorr, TgPosition, FreqOffset]"""
    c = _ctx(precision)
    ac, tg, fo, _ = c.cp_autocorr(c.cplx(np.asarray(RxSignal).ravel())[None], int(WidthWindow), int(Nfft), want_autocorr=True)
    return ac[0].cpu().numpy(), int(tg[0].item()), float(fo[0].item())


def remove_IFO(rx_signal, Nfft, precision="f32"):
    """`Task 5/remove_IFO.m:1` -> [fixed_rx_signal, IFO]; raises like MATLAB when no bin exceeds 0.77."""
    c = _ctx(precision)
    out, ifo = c.remove_ifo(c.cplx(np.asarray(rx_signal).ravel())[None], int(Nfft))
    k = int(ifo[0].item())
    if k < 0:
        raise IndexError("remove_IFO: no spectrum bin above 0.77 (inds(1) on empty)")
    return out[0].cpu().numpy(), k


def fine_sync(rx_signal, pilotCarriers, pilotValues, time_desync, freq_desync, return_estimates=False, precision="f32"):
    """`Task 4/fine_sync.m:1`"""
    c = _ctx(precision)
    out, tau, ph = c.fine_sync(_grid_to_dev(c, rx_signal), pilotCarriers, pilotValues, time_desync, freq_desync)
    res = _grid_to_host(out)
    return (res, float(tau[0].item()), float(ph[0].item())) if return_estimates else res


def estimate_channel(rx_signal, allCarriers, pilotCarriers, pilotValues, precision="f32"):
    """`Task 5/estimate_channel.m:1` -> [H_est, Hest_at_pilots]"""
    c = _ctx(precision)
    H, Hp = c.estimate_channel(_grid_to_dev(c, rx_signal), allCarriers, pilotCarriers, pilotValues)
    return H[0].cpu().numpy(), Hp[0].cpu().numpy()


def LS_CE(Y, Xp, pilot_loc, N_carrier, precision="f32"):
    """`Task 5/LS_CE.m:1`"""
    c = _ctx(precision)
    return c.ls_ce(_grid_to_dev(c, Y), Xp, pilot_loc, int(N_carrier))[0].cpu().numpy()


def MMSE_CE(Y, Xp, pilot_loc, Nfft, N_carrier, h, SNR, precision="f32"):
    """`Task 5/MMSE_CE.m:1`"""
    c = _ctx(precision)
    return c.mmse_ce(_grid_to_dev(c, Y), Xp, pilot_loc, int(N_carrier), c.cplx(np.asarray(h).ravel())[None], float(SNR))[0].cpu().numpy()


def interpolate(H, pilot_loc, Nfft, method, precision="f32"):
    """`Task 5/interpolate.m:1`"""
    c = _ctx(precision)
    return c.interpolate(c.cplx(np.asarray(H).ravel())[None], pilot_loc, int(Nfft), method)[0].cpu().numpy()


def equalize_signal(OFDM_demod, Hest, N_carrier, precision="f32"):
    """`Task 5/equalize_signal.m:1`"""
    c = _ctx(precision)
    return _grid_to_host(c.equalize(_grid_to_dev(c, OFDM_demod), c.cplx(np.asarray(Hest).ravel())[None], int(N_carrier)))


def OMP_estimate(Y, sensing_matrix, Nfft, dominant_taps, SNR_dB=None, precision="f32"):
    """`Task 5/OMP_estimate.m:2` -> [H_OMP, h_impulse_est, index]; ``sensing_matrix`` (Np, Ldict) dense."""
    c = _ctx(precision)
    A = np.asarray(sensing_matrix)
    H, h, idx, it = c.omp(c.cplx(np.asarray(Y).ravel())[None], int(Nfft), int(dominant_taps), A_dev=c.cplx(np.asfortranarray(A).ravel(order="F")))
    n = int(it[0].item())
    return H[0].cpu().numpy(), h[0].cpu().numpy(), idx[0, :n].cpu().numpy().astype(np.int64)


def MP_estimate(Y, sensing_matrix, Nfft, dominant_taps, precision="f32"):
    """`Task 5/MP_estimate.m:2` -> [H_MP, h_impulse_est]"""
    c = _ctx(precision)
    A = np.asarray(sensing_matrix)
    H, h, _ = c.mp(c.cplx(np.asarray(Y).ravel())[None], int(Nfft), int(dominant_taps), A_dev=c.cplx(np.asfortranarray(A).ravel(order="F")))
    return H[0].cpu().numpy(), h[0].cpu().numpy()


def BER_func(Bit_Tx, Bit_Rx, precision="f32"):
    """`Task 5/BER_func.m:1`"""
    c = _ctx(precision)
    tx = np.asarray(Bit_Tx).ravel()
    cnt = c.ber_count(c.bits(tx), c.bits(np.asarray(Bit_Rx).ravel()), tx.size).cpu().numpy()
    return float(cnt[0]) / float(cnt[1])


def MER_func(IQ_RX, Constellation, precision="f32"):
    """`Task 5/MER_func.m:1`"""
    c = _ctx(precision)
    s = c.mer(c.cplx(np.asarray(IQ_RX).ravel()), Constellation).cpu().numpy()
    return 10 * np.log10(s[0] / s[1])


def calculatePAPR(OFDM_signal, precision="f32"):
    """`Task 5/calculatePAPR.m:2` -> PAPR in dB"""
    c = _ctx(precision)
    return float(c.papr(c.cplx(np.asarray(OFDM_signal).ravel())[None])[0].item())


def calculate_window_PAPR(Tx_OFDM_Signal, Nfft, precision="f32"):
    """`Task 5/calculate_window_PAPR.m:2` -> PAPRs (1 x L-Nfft+1)"""
    c = _ctx(precision)
    return c.window_papr(c.cplx(np.asarray(Tx_OFDM_Signal).ravel())[None], int(Nfft)).cpu().numpy().astype(np.float64)


def calculateCCDF(PAPR_values, precision="f32"):
    """`Task 5/calculateCCDF.m:2` -> (PAPR_ccdf, CCDF), column vectors as MATLAB's ecdf returns them"""
    c = _ctx(precision)
    xs, cc = c.ccdf(c.real(np.asarray(PAPR_values, dtype=np.float64).ravel(), c.rdtype))
    return xs.cpu().numpy().astype(np.float64)[:, None], cc.cpu().numpy().astype(np.float64)[:, None]
