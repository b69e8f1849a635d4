"""ctypes binding of libqdsp_b200.so (the C ABI declared in include/qdsp_b200.h).

The shared library is built in-tree by ``qdsp_b200/csrc/Makefile`` (``__graft_entry__.build()``).
There is no CPU fallback: if the library is missing, or no CUDA device is usable, every compute
entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
import re
from functools import lru_cache

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libqdsp_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(HERE), "include", "qdsp_b200.h")

F32, CF32 = 0, 1
CS16, CS8, CU8 = 2, 3, 4    # integer IQ: interleaved (re, im) int16 / int8 / uint8 pairs

_f, _d, _i, _u, _ll, _ull = C.c_float, C.c_double, C.c_int, C.c_uint, C.c_longlong, C.c_ulonglong
_vp, _sz = C.c_void_p, C.c_size_t
_fp, _ip, _llp = C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_longlong)

# name -> (restype, argtypes); must cover every symbol declared in include/qdsp_b200.h
SIGNATURES = {
    "qdsp_abi_version": (_i, []),
    "qdsp_last_error": (C.c_char_p, []),
    "qdsp_device_count": (_i, []),
    "qdsp_set_device": (_i, [_i]),
    "qdsp_get_device": (_i, []),
    "qdsp_malloc_device": (_vp, [_sz]),
    "qdsp_free_device": (None, [_vp]),
    "qdsp_malloc_pinned": (_vp, [_sz]),
    "qdsp_free_pinned": (None, [_vp]),
    "qdsp_memset_device": (_i, [_vp, _i, _sz, _vp]),
    "qdsp_copy_h2d": (_i, [_vp, _vp, _sz, _vp]),
    "qdsp_copy_d2h": (_i, [_vp, _vp, _sz, _vp]),
    "qdsp_copy_d2d": (_i, [_vp, _vp, _sz, _vp]),
    "qdsp_copy_peer": (_i, [_vp, _i, _vp, _i, _sz, _vp]),
    "qdsp_enable_peer_access": (_i, [_i, _i]),
    "qdsp_ipc_export": (_i, [_vp, _vp]),
    "qdsp_ipc_open": (_vp, [_vp]),
    "qdsp_ipc_close": (_i, [_vp]),
    "qdsp_stream_create": (_vp, []),
    "qdsp_stream_destroy": (None, [_vp]),
    "qdsp_stream_sync": (_i, [_vp]),
    "qdsp_launch_count": (_ll, []),
    "qdsp_event_create": (_vp, []),
    "qdsp_event_destroy": (None, [_vp]),
    "qdsp_event_record": (_i, [_vp, _vp]),
    "qdsp_stream_wait_event": (_i, [_vp, _vp]),
    "qdsp_event_sync": (_i, [_vp]),
    "qdsp_iq_convert_process": (_ll, [_i, _f, _f, _vp, _vp, _ll, _vp]),
    "qdsp_blackman_tap_count": (_i, [_f, _f, _f]),
    "qdsp_blackman_taps": (None, [_f, _f, _f, _fp, _i, _f]),
    "qdsp_blackman_bandpass_taps": (None, [_f, _f, _f, _f, _fp, _i, _f]),
    "qdsp_rrc_taps": (None, [_i, _f, _f, _f, _fp]),
    "qdsp_rates_to_ratio": (None, [_f, _f, _ip, _ip]),
    "qdsp_vfo_design": (_i, [_f, _f, _f, _fp, _i, _ip, _ip]),
    "qdsp_resamp_schedule": (_i, [_i, _i, _i, _ip, _ip]),
    "qdsp_fir_create": (_vp, [_i, _fp, _i]),
    "qdsp_fir_destroy": (None, [_vp]),
    "qdsp_fir_set_taps": (_i, [_vp, _fp, _i]),
    "qdsp_fir_process": (_ll, [_vp, _vp, _vp, _ll, _vp]),
    "qdsp_fir_history_len": (_i, [_vp]),
    "qdsp_fir_get_history": (_i, [_vp, _vp]),
    "qdsp_fir_set_history": (_i, [_vp, _vp]),
    "qdsp_fir_import_tail": (_i, [_vp, _vp, _i, _vp]),
    "qdsp_fir_process_halo": (_ll, [_vp, _vp, _vp, _vp, _ll, _vp]),
    "qdsp_fir_reset": (_i, [_vp]),
    "qdsp_fir_set_variant": (_i, [_vp, _i]),
    "qdsp_resamp_create": (_vp, [_i, _fp, _i, _i, _i]),
    "qdsp_resamp_destroy": (None, [_vp]),
    "qdsp_resamp_set_taps": (_i, [_vp, _fp, _i]),
    "qdsp_resamp_taps_per_phase": (_i, [_vp]),
    "qdsp_resamp_out_count": (_ll, [_vp, _ll]),
    "qdsp_resamp_process": (_ll, [_vp, _vp, _vp, _ll, _ip, _i, _i, _ip, _vp]),
    "qdsp_resamp_schedule_device": (_ll, [_vp, _ll, _ip, _i, _i, _vp, _vp, _vp]),
    "qdsp_resamp_history_len": (_i, [_vp]),
    "qdsp_resamp_get_history": (_i, [_vp, _vp]),
    "qdsp_resamp_set_history": (_i, [_vp, _vp]),
    "qdsp_resamp_reset": (_i, [_vp]),
    "qdsp_resamp_set_variant": (_i, [_vp, _i]),
    "qdsp_power_decim_process": (_ll, [_u, _vp, _vp, _ll, _vp]),
    "qdsp_xlator_create": (_vp, [_f, _f]),
    "qdsp_xlator_destroy": (None, [_vp]),
    "qdsp_xlator_set_frequency": (_i, [_vp, _f, _f]),
    "qdsp_xlator_get_phase_delta": (None, [_vp, _fp, _fp]),
    "qdsp_xlator_get_phase": (None, [_vp, _fp, _fp]),
    "qdsp_xlator_set_phase": (None, [_vp, _f, _f]),
    "qdsp_xlator_process": (_ll, [_vp, _vp, _vp, _ll, _vp]),
    "qdsp_fmdemod_create": (_vp, [_f, _f, _i]),
    "qdsp_fmdemod_destroy": (None, [_vp]),
    "qdsp_fmdemod_get_phase": (_f, [_vp]),
    "qdsp_fmdemod_set_phase": (_i, [_vp, _f]),
    "qdsp_fmdemod_process": (_ll, [_vp, _vp, _vp, _ll, _vp]),
    "qdsp_stereofm_create": (_vp, [_f, _f]),
    "qdsp_stereofm_destroy": (None, [_vp]),
    "qdsp_stereofm_process": (_ll, [_vp, _vp, _vp, _ll, _ip, _i, _i, _vp]),
    "qdsp_stereo_matrix_process": (_ll, [_vp, _vp, _vp, _ll, _vp]),
    "qdsp_vfofm_create": (_vp, [_f, _f, _f, _f, _f]),
    "qdsp_vfofm_destroy": (None, [_vp]),
    "qdsp_vfofm_design": (_i, [_vp, _ip, _ip, _ip]),
    "qdsp_vfofm_set_offset": (_i, [_vp, _f]),
    "qdsp_vfofm_get_phase": (None, [_vp, _fp, _fp]),
    "qdsp_vfofm_set_phase": (_i, [_vp, _f, _f]),
    "qdsp_vfofm_out_count": (_ll, [_vp, _ll, _ip, _i, _i]),
    "qdsp_vfofm_process": (_ll, [_vp, _vp, _vp, _vp, _ll, _ip, _i, _i, _ip, _vp]),
    "qdsp_vfofm_process_host": (_ll, [_vp, _vp, _vp, _ll, _i, _vp]),
    "qdsp_vfofm_process_replay": (_ll, [_vp, _vp, _vp, _vp, _ll, _ip, _i, _i, _fp, _ll, _vp]),
    "qdsp_vfofm_reset": (_i, [_vp]),
    "qdsp_vfofm_set_variant": (_i, [_vp, _i]),
    "qdsp_vfofm_set_input_format": (_i, [_vp, _i, _f, _f]),
    "qdsp_vfofm_seek": (_i, [_vp, _ll]),
    "qdsp_vfofm_import_tail": (_i, [_vp, _vp, _i, _vp]),
    "qdsp_vfofm_history_len": (_i, [_vp]),
    "qdsp_vfofm_enable_timing": (_i, [_vp, _i]),
    "qdsp_vfofm_enable_timing_ring": (_i, [_vp, _i]),
    "qdsp_vfofm_kernel_ms_mean": (_d, [_vp, _ip]),
    "qdsp_vfofm_kernel_ms": (_d, [_vp]),
    "qdsp_channelizer_create": (_vp, [_i, _fp, _f, _f, _f, _f]),
    "qdsp_channelizer_destroy": (None, [_vp]),
    "qdsp_channelizer_design": (_i, [_vp, _ip, _ip, _ip]),
    "qdsp_channelizer_process": (_ll, [_vp, _vp, _vp, _ll, _ll, _ip, _i, _i, _vp]),
    "qdsp_channelizer_process_iq": (_ll, [_vp, _vp, _vp, _vp, _ll, _ll, _ip, _i, _i, _vp]),
    "qdsp_channelizer_reset": (_i, [_vp]),
    "qdsp_channelizer_set_variant": (_i, [_vp, _i]),
    "qdsp_channelizer_set_input_format": (_i, [_vp, _i, _f, _f]),
    "qdsp_channelizer_seek": (_i, [_vp, _ll]),
    "qdsp_channelizer_set_offsets": (_i, [_vp, _fp]),
    "qdsp_channelizer_fft_form": (_i, [_vp]),
    "qdsp_scatter_rows": (_ll, [_vp, _ll, _vp, _i, _ll, _i, _vp]),
    "qdsp_spectrum_create": (_vp, [_i, _fp, _i, _i]),
    "qdsp_spectrum_destroy": (None, [_vp]),
    "qdsp_spectrum_out_rows": (_ll, [_vp, _ll]),
    "qdsp_spectrum_process": (_ll, [_vp, _vp, _vp, _ll, _vp]),
    "qdsp_spectrum_reset": (_i, [_vp]),
    "qdsp_spectrum_set_input_format": (_i, [_vp, _i, _f, _f]),
    "qdsp_deemp_create": (_vp, [_f, _f]),
    "qdsp_deemp_destroy": (None, [_vp]),
    "qdsp_deemp_process": (_ll, [_vp, _vp, _vp, _ll, _vp]),
    "qdsp_deemp_set_params": (_i, [_vp, _f, _f]),
    "qdsp_deemp_get_state": (_i, [_vp, _fp, _fp]),
    "qdsp_deemp_set_state": (_i, [_vp, _f, _f]),
    "qdsp_agc_create": (_vp, [_f, _f]),
    "qdsp_agc_destroy": (None, [_vp]),
    "qdsp_agc_process": (_ll, [_vp, _vp, _vp, _ll, _ip, _i, _i, _vp]),
    "qdsp_agc_set_params": (_i, [_vp, _f, _f]),
    "qdsp_agc_get_state": (_i, [_vp, _fp]),
    "qdsp_agc_set_state": (_i, [_vp, _f]),
    "qdsp_cagc_create": (_vp, [_f, _f, _f]),
    "qdsp_cagc_destroy": (None, [_vp]),
    "qdsp_cagc_process": (_ll, [_vp, _vp, _vp, _ll, _vp]),
    "qdsp_cagc_set_params": (_i, [_vp, _f, _f, _f]),
    "qdsp_cagc_get_state": (_i, [_vp, _fp]),
    "qdsp_cagc_set_state": (_i, [_vp, _f]),
    "qdsp_ffagc_create": (_vp, [_i]),
    "qdsp_ffagc_destroy": (None, [_vp]),
    "qdsp_ffagc_process": (_ll, [_vp, _vp, _vp, _ll, _vp]),
    "qdsp_costas_create": (_vp, [_i, _f]),
    "qdsp_costas_destroy": (None, [_vp]),
    "qdsp_costas_process": (_ll, [_vp, _vp, _vp, _ll, _vp]),
    "qdsp_costas_get_state": (_i, [_vp, _fp]),
    "qdsp_costas_set_state": (_i, [_vp, _fp]),
    "qdsp_costas_set_chunking": (_i, [_vp, _i, _i]),
    "qdsp_costas_last_residual": (_f, [_vp]),
    "qdsp_math_process": (_ll, [_i, _i, _vp, _vp, _vp, _ll, _vp]),
    "qdsp_layout_process": (_ll, [_i, _vp, _vp, _vp, _vp, _ll, _vp]),
    "qdsp_volume_level": (_f, [_f]),
    "qdsp_volume_process": (_ll, [_i, _f, _i, _vp, _vp, _ll, _vp]),
    "qdsp_threshold_process": (_ll, [_vp, _vp, _ll, _vp]),
    "qdsp_delayimag_create": (_vp, []),
    "qdsp_delayimag_destroy": (None, [_vp]),
    "qdsp_delayimag_process": (_ll, [_vp, _vp, _vp, _ll, _vp]),
    "qdsp_delayimag_get_state": (_i, [_vp, _fp]),
    "qdsp_delayimag_set_state": (_i, [_vp, _f]),
    "qdsp_amdemod_create": (_vp, []),
    "qdsp_amdemod_destroy": (None, [_vp]),
    "qdsp_amdemod_process": (_ll, [_vp, _vp, _vp, _ll, _ip, _i, _i, _vp]),
    "qdsp_squelch_create": (_vp, [_f]),
    "qdsp_squelch_destroy": (None, [_vp]),
    "qdsp_squelch_set_level": (None, [_vp, _f]),
    "qdsp_squelch_get_level": (_f, [_vp]),
    "qdsp_squelch_process": (_ll, [_vp, _vp, _vp, _ll, _ip, _i, _i, _vp]),
    "qdsp_ssbdemod_create": (_vp, [_f, _f, _i]),
    "qdsp_ssbdemod_destroy": (None, [_vp]),
    "qdsp_ssbdemod_configure": (_i, [_vp, _f, _f, _i]),
    "qdsp_ssbdemod_get_phase_delta": (None, [_vp, _fp, _fp]),
    "qdsp_ssbdemod_get_phase": (None, [_vp, _fp, _fp]),
    "qdsp_ssbdemod_set_phase": (None, [_vp, _f, _f]),
    "qdsp_ssbdemod_process": (_ll, [_vp, _vp, _vp, _ll, _vp]),
    "qdsp_mm_create": (_vp, [_i, _f, _f, _f, _f, _fp]),
    "qdsp_mm_destroy": (None, [_vp]),
    "qdsp_mm_set_omega": (_i, [_vp, _f, _f]),
    "qdsp_mm_set_gains": (_i, [_vp, _f, _f]),
    "qdsp_mm_set_omega_rel_limit": (_i, [_vp, _f]),
    "qdsp_mm_max_out": (_ll, [_vp, _ll]),
    "qdsp_mm_process": (_ll, [_vp, _vp, _vp, _ll, _ip, _i, _i, _ip, _vp]),
    "qdsp_mm_get_state": (_i, [_vp, _fp]),
    "qdsp_mm_set_state": (_i, [_vp, _fp]),
    "qdsp_sinesource_create": (_vp, [_f, _f]),
    "qdsp_sinesource_destroy": (None, [_vp]),
    "qdsp_sinesource_configure": (_i, [_vp, _f, _f]),
    "qdsp_sinesource_get_phase": (None, [_vp, _fp, _fp]),
    "qdsp_sinesource_set_phase": (None, [_vp, _f, _f]),
    "qdsp_sinesource_process": (_ll, [_vp, _vp, _ll, _vp]),
    "qdsp_synth_uniform_cf32": (_i, [_vp, _ull, _ll, _ll, _vp]),
    "qdsp_synth_fm_cf32": (_i, [_vp, _ll, _ll, _ll, _ll, _ll, _d, _d, _d, _ull, _vp]),
    "qdsp_synth_comb_cf32": (_i, [_vp, _ll, _ll, _ll, _i, _ll, _d, _d, _d, _ull, _vp]),
    "qdsp_synth_qpsk_cf32": (_i, [_vp, _ll, _ll, _ull, _i, _d, _d, _d, _ll, _vp]),
    "qdsp_measure_fp32_peak": (_d, [_i, _i]),
}


class QdspError(RuntimeError):
    pass


def header_symbols() -> list[str]:
    """Every function name declared in include/qdsp_b200.h (used by the symbol-export test)."""
    with open(HEADER_PATH) as f:
        text = f.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(qdsp_[a-z0-9_]+)\s*\(", text)))


@lru_cache(maxsize=None)
def load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise QdspError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C qdsp_b200/csrc`). qdsp_b200 has no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


def last_error() -> str:
    return load().qdsp_last_error().decode(errors="replace")


def check(rc, what: str = "qdsp call"):
    """Raise on the C ABI's -1 / NULL error convention."""
    if rc is None or (isinstance(rc, int) and rc < 0):
        raise QdspError(f"{what} failed: {last_error()}")
    return rc


def require_device() -> int:
    n = load().qdsp_device_count()
    if n <= 0:
        raise QdspError("no CUDA device: qdsp_b200 runs only on B200 (sm_100a) and has no CPU fallback")
    return n
