"""ctypes binding of the C ABI in ``include/ofdm_b200.h`` (one Python callable per exported symbol).

There is no CPU fallback: importing this module without the built CUDA library raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# OFDM_B200_LIB selects another build of the same library (kernel A/B experiments, tools/ab_variants.sh)
LIB_PATH = os.environ.get("OFDM_B200_LIB") or os.path.join(_HERE, "lib", "libofdm_b200.so")

vp, i32, i64, u64, dbl = C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_double
pi32 = C.POINTER(C.c_int32)
pdbl = C.POINTER(C.c_double)
pu8 = C.POINTER(C.c_uint8)


class LinkParams(C.Structure):
    """``ofdm_link_params`` of include/ofdm_b200.h."""
    _fields_ = [("Nfft", C.c_int32), ("Tg", C.c_int32), ("N_carrier", C.c_int32), ("S", C.c_int32), ("SpF", C.c_int32),
                ("constellation", C.c_int32), ("Nd", C.c_int32), ("Np", C.c_int32),
                ("data_carriers_host", pi32), ("pilot_carriers_host", pi32), ("pilot_vals_host", pdbl),
                ("reg0_host", pu8), ("scramble", C.c_int32)]


class SweepParams(C.Structure):
    """``ofdm_sweep_params`` of include/ofdm_b200.h."""
    _fields_ = [("chain", C.c_int32), ("n_snr", C.c_int32), ("snr_db_host", pdbl), ("streams_per_point", C.c_int64),
                ("tile_streams", C.c_int64), ("rank", C.c_int32), ("world", C.c_int32), ("seed", C.c_uint64),
                ("taps_host", pdbl), ("n_taps", C.c_int32), ("near_eps", C.c_double), ("sto_max", C.c_int32),
                ("cfo_int_max", C.c_int32)]


class Part2Params(C.Structure):
    """``ofdm_part2_params`` of include/ofdm_b200.h."""
    _fields_ = [("n_points", C.c_int32), ("pilot_offsets_host", pi32), ("pilot_carriers_host", pi32), ("ldict_host", pi32),
                ("pilot_pattern_host", pdbl), ("payload_host", C.POINTER(C.c_uint32)), ("payload_bits", C.c_int64),
                ("profile", C.c_int32), ("fs_hz", C.c_double), ("snr_db", C.c_double), ("mc_runs", C.c_int64),
                ("tile_runs", C.c_int64), ("rank", C.c_int32), ("world", C.c_int32), ("seed", C.c_uint64),
                ("near_eps", C.c_double), ("tie_eps", C.c_double)]


class SyncParams(C.Structure):
    """``ofdm_sync_params`` of include/ofdm_b200.h."""
    _fields_ = [("n_snr", C.c_int32), ("snr_db_host", pdbl), ("streams_per_point", C.c_int64), ("tile_streams", C.c_int64),
                ("rank", C.c_int32), ("world", C.c_int32), ("seed", C.c_uint64), ("taps_host", pdbl), ("n_taps", C.c_int32),
                ("sto_mode", C.c_int32), ("sto_max", C.c_int32), ("cfo_int_max", C.c_int32), ("sto_fixed", C.c_int32),
                ("cfo_fixed", C.c_double), ("time_desync", C.c_int32), ("freq_desync", C.c_int32), ("mp_desync", C.c_int32)]


class PaprParams(C.Structure):
    """``ofdm_papr_params`` of include/ofdm_b200.h."""
    _fields_ = [("n_points", C.c_int32), ("scramble_host", pi32), ("p_one_host", pdbl), ("pool_host", C.POINTER(C.c_uint32)),
                ("pool_bits", C.c_int64), ("pool_stride", C.c_int64), ("streams_per_point", C.c_int64), ("tile_streams", C.c_int64),
                ("rank", C.c_int32), ("world", C.c_int32), ("seed", C.c_uint64), ("bin_db", C.c_double), ("n_bins", C.c_int32)]


class MerParams(C.Structure):
    """``ofdm_mer_params`` of include/ofdm_b200.h."""
    _fields_ = [("n_points", C.c_int32), ("constellation_host", pi32), ("snr_db_host", pdbl), ("pilot_scale", C.c_double),
                ("nsto_host", pi32), ("cfo_host", pdbl), ("taps_host", pdbl), ("n_taps", C.c_int32),
                ("streams_per_point", C.c_int64), ("tile_streams", C.c_int64), ("rank", C.c_int32), ("world", C.c_int32),
                ("seed", C.c_uint64), ("near_eps", C.c_double)]


# name -> (restype, argtypes); every symbol declared in include/ofdm_b200.h
SIGNATURES = {
    "ofdm_ctx_create": (i32, [C.POINTER(vp), i32, i32]),
    "ofdm_ctx_destroy": (None, [vp]),
    "ofdm_last_error": (C.c_char_p, [vp]),
    "ofdm_ctx_set_stream": (i32, [vp, vp]),
    "ofdm_sync": (i32, [vp]),
    "ofdm_precision": (i32, [vp]),
    "ofdm_malloc": (i32, [vp, C.POINTER(vp), C.c_size_t]),
    "ofdm_free": (i32, [vp, vp]),
    "ofdm_memset": (i32, [vp, vp, i32, C.c_size_t]),
    "ofdm_h2d": (i32, [vp, vp, vp, C.c_size_t]),
    "ofdm_d2h": (i32, [vp, vp, vp, C.c_size_t]),
    "ofdm_host_alloc": (i32, [C.POINTER(vp), C.c_size_t]),
    "ofdm_host_free": (i32, [vp]),
    "ofdm_launch_count": (i64, [vp]),
    "ofdm_version": (C.c_char_p, []),
    "ofdm_scramble": (i32, [vp, vp, vp, i64, i64, pu8, vp]),
    "ofdm_descramble": (i32, [vp, vp, vp, i64, i64, pu8, vp]),
    "ofdm_constellation": (i32, [i32, pdbl, C.POINTER(i32)]),
    "ofdm_map": (i32, [vp, vp, i64, i32, vp, C.POINTER(i32)]),
    "ofdm_demap": (i32, [vp, vp, i64, i32, vp, dbl, vp]),
    "ofdm_map_carriers": (i32, [vp, vp, i64, i32, i32, pi32, i32, pi32, i32, pdbl, i32, vp]),
    "ofdm_modulate": (i32, [vp, vp, i64, i32, i32, i32, vp]),
    "ofdm_demodulate": (i32, [vp, vp, i64, i32, i32, i32, vp]),
    "ofdm_get_payload": (i32, [vp, vp, i64, i32, i32, pi32, i32, vp]),
    "ofdm_fft": (i32, [vp, vp, vp, i64, i32, i32]),
    "ofdm_add_sto": (i32, [vp, vp, i64, i64, vp, vp]),
    "ofdm_add_cfo": (i32, [vp, vp, i64, i64, vp, i32, vp]),
    "ofdm_add_noise": (i32, [vp, vp, i64, i64, vp, vp, u64, i64, vp, vp]),
    "ofdm_mp_channel_resp": (i32, [vp, pdbl, i32, i32, pdbl, i32, C.POINTER(i32), vp]),
    "ofdm_apply_fir": (i32, [vp, vp, i64, i64, vp, i32, i32, vp]),
    "ofdm_tdl_info": (i32, [i32, dbl, C.POINTER(i32), C.POINTER(i32), pdbl]),
    "ofdm_tdl_channel": (i32, [vp, i32, dbl, i64, u64, i64, i32, vp, vp]),
    "ofdm_mse": (i32, [vp, vp, i64, vp, i64, i64, i32, vp]),
    "ofdm_cp_autocorr": (i32, [vp, vp, i64, i64, i32, i32, vp, vp, vp, vp]),
    "ofdm_remove_ifo": (i32, [vp, vp, i64, i64, i32, vp, vp]),
    "ofdm_fine_sync": (i32, [vp, vp, i64, i32, i32, pi32, i32, pdbl, i32, i32, vp, vp, vp]),
    "ofdm_estimate_channel": (i32, [vp, vp, i64, i32, i32, pi32, i32, pi32, i32, pdbl, vp, vp]),
    "ofdm_ls_ce": (i32, [vp, vp, i64, i32, i32, pi32, i32, pdbl, i32, vp]),
    "ofdm_mmse_ce": (i32, [vp, vp, i64, i32, i32, pi32, i32, pdbl, i32, vp, i32, vp, vp]),
    "ofdm_mmse_ce_shared": (i32, [vp, vp, i64, i32, i32, pi32, i32, pdbl, i32, vp, i32, dbl, vp]),
    "ofdm_interpolate": (i32, [vp, vp, i64, pi32, i32, i32, i32, vp]),
    "ofdm_equalize": (i32, [vp, vp, i64, i32, i32, vp, i32, i32, vp]),
    "ofdm_pilot_ls": (i32, [vp, vp, i64, i32, i32, pi32, i32, pdbl, vp]),
    "ofdm_omp": (i32, [vp, vp, i64, i32, vp, i32, pi32, i32, i32, vp, vp, vp, vp]),
    "ofdm_omp_ex": (i32, [vp, vp, i64, i32, vp, i32, pi32, i32, i32, vp, vp, vp, vp, vp, dbl]),
    "ofdm_mp": (i32, [vp, vp, i64, i32, vp, i32, pi32, i32, i32, vp, vp, vp]),
    "ofdm_ber_count": (i32, [vp, vp, vp, i64, vp]),
    "ofdm_mer": (i32, [vp, vp, i64, i32, vp]),
    "ofdm_papr": (i32, [vp, vp, i64, i64, vp]),
    "ofdm_window_papr": (i32, [vp, vp, i64, i64, i32, vp]),
    "ofdm_ccdf": (i32, [vp, vp, i64, vp, vp, vp]),
    "ofdm_tx_chain": (i32, [vp, C.POINTER(LinkParams), vp, i64, vp]),
    "ofdm_tx_chain_p": (i32, [vp, C.POINTER(LinkParams), vp, i64, vp, vp]),
    "ofdm_channel_t5_p": (i32, [vp, vp, i64, i64, vp, vp, vp, u64, i64, vp, i32, vp]),
    "ofdm_channel_t5": (i32, [vp, vp, i64, i64, vp, vp, u64, i64, vp, i32, vp]),
    "ofdm_channel_t4_p": (i32, [vp, vp, i64, i64, vp, vp, vp, u64, i64, vp, vp, i32, vp, i32, vp]),
    "ofdm_rx_chain_t5": (i32, [vp, C.POINTER(LinkParams), vp, i64, vp, vp, vp, vp, vp, dbl]),
    "ofdm_rx_chain_t5_host": (i32, [vp, C.POINTER(LinkParams), vp, i64, vp, vp, vp, vp, i64]),
    "ofdm_rx_chain_t5_host_eps": (i32, [vp, C.POINTER(LinkParams), vp, i64, vp, vp, vp, vp, i64, dbl]),
    "ofdm_rx_chain_t4": (i32, [vp, C.POINTER(LinkParams), vp, i64, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, dbl]),
    "ofdm_sweep_ber": (i32, [vp, C.POINTER(LinkParams), C.POINTER(SweepParams), vp]),
    "ofdm_sweep_mse": (i32, [vp, C.POINTER(LinkParams), C.POINTER(SweepParams), i32, vp, vp]),
    "ofdm_sweep_part2": (i32, [vp, C.POINTER(LinkParams), C.POINTER(Part2Params), vp, vp, vp]),
    "ofdm_sweep_sync": (i32, [vp, C.POINTER(LinkParams), C.POINTER(SyncParams), vp, vp]),
    "ofdm_sweep_papr": (i32, [vp, C.POINTER(LinkParams), C.POINTER(PaprParams), vp, vp]),
    "ofdm_sweep_mer": (i32, [vp, C.POINTER(LinkParams), C.POINTER(MerParams), vp, vp]),
    "ofdm_sweep_share": (i32, [i64, i32, i32, C.POINTER(i64), C.POINTER(i64)]),
    "ofdm_payload_bits": (i32, [vp, vp, i64, i64, u64, i64]),
    "ofdm_draw_sto_cfo": (i32, [vp, i64, u64, i64, i32, i32, vp, vp]),
    "ofdm_payload_bernoulli": (i32, [vp, vp, i64, i64, dbl, u64, i64]),
    "ofdm_rx_chain_t4_ex": (i32, [vp, C.POINTER(LinkParams), vp, i64, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, dbl, vp]),
    "ofdm_group_create": (i32, [C.POINTER(vp), pi32, i32, i32]),
    "ofdm_group_destroy": (None, [vp]),
    "ofdm_group_last_error": (C.c_char_p, [vp]),
    "ofdm_group_size": (i32, [vp]),
    "ofdm_group_sweep_ber": (i32, [vp, C.POINTER(LinkParams), C.POINTER(SweepParams), vp]),
    "ofdm_group_sweep_mse": (i32, [vp, C.POINTER(LinkParams), C.POINTER(SweepParams), i32, vp, vp]),
    "ofdm_group_sweep_sync": (i32, [vp, C.POINTER(LinkParams), C.POINTER(SyncParams), vp, vp]),
    "ofdm_group_sweep_papr": (i32, [vp, C.POINTER(LinkParams), C.POINTER(PaprParams), vp, vp]),
    "ofdm_group_sweep_mer": (i32, [vp, C.POINTER(LinkParams), C.POINTER(MerParams), vp, vp]),
    "ofdm_group_sweep_part2": (i32, [vp, C.POINTER(LinkParams), C.POINTER(Part2Params), vp, vp, vp]),
}

_lib = None


def load():
    """Load ``lib/libofdm_b200.so`` (built by ``make`` / ``__graft_entry__.build()``).  Raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback for this package)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
