"""ctypes binding of include/gsmcal.h (the same symbols a MEX gateway binds)."""
from __future__ import annotations

import ctypes as C
import os

from .build import LIB

c_i64 = C.c_int64
c_dp = C.POINTER(C.c_double)
c_u8p = C.POINTER(C.c_uint8)
c_ip = C.POINTER(C.c_int)
c_i64p = C.POINTER(C.c_int64)


class StreamResult(C.Structure):
    _fields_ = [("n_coarse", C.c_int32), ("n_fcch", C.c_int32), ("n_pos_info", C.c_int32), ("flags", C.c_int32),
                ("r_len", C.c_int64 * 3), ("sampling_ppm", C.c_double * 2), ("carrier_ppm", C.c_double * 2),
                ("total_sampling_ppm", C.c_double), ("total_carrier_ppm", C.c_double)]


class DemodResult(C.Structure):
    _fields_ = [("n_sch", C.c_int32), ("n_sch_ok", C.c_int32), ("n_fcch", C.c_int32), ("flags", C.c_int32),
                ("fcch_mean_freq", C.c_double), ("fcch_carrier_ppm", C.c_double)]


class BcchResult(C.Structure):
    _fields_ = [("carrier_ppm", C.c_double), ("nts_idx", C.c_int32), ("flags", C.c_int32), ("corr_abs", C.c_double * 32)]


class SchTimingResult(C.Structure):
    _fields_ = [("n_sch", C.c_int32), ("n_fit", C.c_int32), ("flags", C.c_int32), ("reserved", C.c_int32),
                ("t0", C.c_double), ("fit_ppm", C.c_double), ("rms", C.c_double)]


class SchDecodeResult(C.Structure):
    _fields_ = [("n_sch", C.c_int32), ("n_crc_ok", C.c_int32), ("n_agree", C.c_int32), ("flags", C.c_int32), ("bsic", C.c_int32),
                ("fn_first", C.c_int32), ("frame_clock_start", C.c_double)]


class CarrierFitResult(C.Structure):
    _fields_ = [("n_fcch", C.c_int32), ("n_fit", C.c_int32), ("flags", C.c_int32), ("reserved", C.c_int32),
                ("t_mean", C.c_double), ("freq_hz", C.c_double), ("drift_hz_per_s", C.c_double), ("rms_hz", C.c_double),
                ("residual_ppm", C.c_double), ("carrier_fit_ppm", C.c_double), ("drift_ppm_per_s", C.c_double)]


class SysinfoResult(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("n_blocks", "n_fire_ok", "n_si3", "n_si3_agree", "flags", "si_mask", "mcc", "mnc", "mnc_digits",
                                         "lac", "ci", "reserved")]


# the leading arguments of gsmcal_calibrate_batch and its variants: raw, raw_mem, n_iq, D, carrier_freq, tpl, coef, n_taps, osr,
# coarse_dr, results, coarse_pos, coarse_snr, fcch_pos, pos_info, cuda_stream
_BATCH = [C.c_void_p, C.c_int, c_i64, c_i64, C.c_double, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 6

# every symbol include/gsmcal.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "gsmcal_abi_version": (C.c_int, []),
    "gsmcal_last_error": (C.c_char_p, []),
    "gsmcal_device_count": (C.c_int, []),
    "gsmcal_set_device": (C.c_int, [C.c_int]),
    "gsmcal_release": (None, []),
    "gsmcal_raw2iq_u8": (C.c_int, [C.c_void_p, c_i64, c_i64, C.c_void_p]),
    "gsmcal_raw2iq_f64": (C.c_int, [C.c_void_p, c_i64, c_i64, C.c_void_p]),
    "gsmcal_fir1": (C.c_int, [C.c_int, C.c_double, C.c_void_p]),
    "gsmcal_fir_filter": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, c_i64, c_i64, C.c_int, C.c_void_p]),
    "gsmcal_raw2iq_fir_u8": (C.c_int, [C.c_void_p, c_i64, c_i64, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "gsmcal_chn_filter_8x_4x": (C.c_int, [C.c_void_p, c_i64, c_i64, C.c_void_p]),
    "gsmcal_chn_filter_4x": (C.c_int, [C.c_void_p, c_i64, c_i64, C.c_void_p]),
    "gsmcal_chn_filter_taps": (C.c_int, [C.c_int, C.c_void_p, c_ip]),
    "gsmcal_band_power_u8": (C.c_int, [C.c_void_p, c_i64, c_i64, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "gsmcal_diversity_power_u8": (C.c_int, [C.c_void_p, c_i64, c_i64, c_i64, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "gsmcal_move_fft_snr_runtime_avg": (C.c_int, [C.c_void_p, c_i64, C.c_int, C.c_int, C.c_double, c_ip, c_dp, c_dp, c_dp]),
    "gsmcal_move_fft_snr_trace": (C.c_int, [C.c_void_p, c_i64, C.c_int, C.c_void_p]),
    "gsmcal_specific_fft_snr_fix_avg": (C.c_int, [C.c_void_p, c_i64, c_i64, c_i64, C.c_int, C.c_double, C.c_double, c_ip, c_dp, c_dp]),
    "gsmcal_FCCH_coarse_position": (C.c_int, [C.c_void_p, c_i64, C.c_int, C.c_void_p, C.c_void_p, c_i64, c_i64p]),
    "gsmcal_max_bursts": (c_i64, [c_i64, C.c_int]),
    "gsmcal_FCCH_fine_correction": (C.c_int, [C.c_void_p, c_i64, C.c_void_p, c_i64, C.c_int, C.c_double, C.c_void_p, c_i64, c_i64p,
                                              C.c_void_p, c_i64, c_i64p, c_dp, c_dp]),
    "gsmcal_SCH_training_sequence_gen": (C.c_int, [C.c_int, C.c_void_p]),
    "gsmcal_SCH_corr_rate_correction": (C.c_int, [C.c_void_p, c_i64, C.c_void_p, c_i64, C.c_void_p, C.c_int, C.c_void_p, c_i64, c_i64p,
                                                  C.c_void_p, c_i64, c_i64p, c_dp]),
    "gsmcal_carrier_correct_post_SCH": (C.c_int, [C.c_void_p, c_i64, C.c_void_p, c_i64, C.c_int, C.c_double, C.c_void_p, c_i64, c_i64p, c_dp]),
    "gsmcal_total_ppm_calculation": (C.c_int, [C.c_void_p, c_i64, c_dp]),
    "gsmcal_normal_training_sequence_gen": (C.c_int, [C.c_int, C.c_void_p]),
    "gsmcal_FCCH_demod": (C.c_int, [C.c_void_p, c_i64, C.c_void_p, c_i64, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, c_i64,
                                    C.POINTER(c_i64), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "gsmcal_BCCH_demod": (C.c_int, [C.c_void_p, c_i64, C.c_void_p, c_i64, C.c_void_p, C.c_int, C.c_double,
                                    C.POINTER(C.c_double), C.POINTER(C.c_int), C.c_void_p]),
    "gsmcal_SCH_demod": (C.c_int, [C.c_void_p, c_i64, C.c_void_p, c_i64, C.c_void_p, C.c_int, c_i64, C.POINTER(c_i64),
                                   C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsmcal_calibrate_batch": (C.c_int, _BATCH),
    "gsmcal_calibrate_batch_r": (C.c_int, _BATCH + [C.c_void_p, C.c_int, c_i64]),
    "gsmcal_calibrate_demod_batch": (C.c_int, _BATCH + [C.c_void_p] * 8),
    "gsmcal_calibrate_demod_bcch_batch": (C.c_int, _BATCH + [C.c_void_p] * 10),
    "gsmcal_calibrate_sch_decode_batch": (C.c_int, _BATCH + [C.c_void_p] * 15),
    "gsmcal_calibrate_sch_timing_batch": (C.c_int, _BATCH + [C.c_void_p] * 3),
    "gsmcal_calibrate_carrier_fit_batch": (C.c_int, _BATCH + [C.c_void_p] * 4),
    "gsmcal_calibrate_cell_batch": (C.c_int, _BATCH + [C.c_void_p] * 13),
    "gsmcal_calibrate_sysinfo_batch": (C.c_int, _BATCH + [C.c_void_p] * 23),
    "gsmcal_calibrate_batch_submit": (C.c_int, [C.c_int, C.c_void_p, c_i64, c_i64, C.c_double, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsmcal_calibrate_batch_collect": (C.c_int, [C.c_int]),
    "gsmcal_calibrate_batch_cancel": (C.c_int, [C.c_int]),
    "gsmcal_last_batch_stage_ms": (C.c_int, [C.c_void_p, C.c_int]),
    "gsmcal_fcch_scan": (C.c_int, [C.c_void_p, C.c_int, c_i64, c_i64, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsmcal_debug_set": (C.c_int, [C.c_int, C.c_int]),
    "gsmcal_debug_get": (c_i64, [C.c_int]),
    "gsmcal_launch_count": (c_i64, [C.c_int]),
    "gsmcal_fp64_peak": (C.c_int, [c_dp, C.c_void_p]),
    "gsmcal_stage_launch": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, c_i64, c_i64, C.c_void_p, C.c_int, C.c_void_p]),
}

_lib = None


class GsmcalError(RuntimeError):
    def __init__(self, code, text):
        super().__init__(f"gsmcal error {code}: {text}")
        self.code = code


def lib() -> C.CDLL:
    """Loads the in-tree libgsmcal.so; raises if it has not been built (there is no fallback implementation)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB):
            raise ImportError(f"{LIB} is missing - run __graft_entry__.build() (nvcc) first; there is no CPU fallback")
        _lib = C.CDLL(LIB)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(_lib, name)
            fn.restype = res
            fn.argtypes = args
    return _lib


def check(rc: int):
    if rc != 0:
        raise GsmcalError(rc, lib().gsmcal_last_error().decode())
