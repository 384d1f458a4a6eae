"""Host-side mirror of the reference's MATLAB function interface, on top of the C ABI (include/gsmcal.h).

Same names, argument meaning and sentinel behaviour as the .m files (SURVEY.md Appendix A); arrays are
NumPy, streams are columns, positions are 1-based doubles.  Python stand-ins for MATLAB shapes:
`array([-1.])` for the scalar -1 and `None` for `r = -1`.  Nothing here computes on the CPU: every call
goes through libgsmcal.so and raises if the library or a CUDA device is missing.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from ._lib import (BcchResult, CarrierFitResult, DemodResult, GsmcalError, SchDecodeResult, SchTimingResult, StreamResult,  # noqa: F401
                   SysinfoResult, check, lib)

SYMBOL_RATE = (1625.0 / 6.0) * 1e3


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _cols(a, dtype):
    """MATLAB matrix (rows x cols) -> C-contiguous [cols][rows] buffer == column-major storage."""
    a = np.asarray(a)
    if a.ndim == 1:
        a = a[:, None]
    return np.ascontiguousarray(a.T.astype(dtype, copy=False)), a.shape[0], a.shape[1]


def device_count() -> int:
    return lib().gsmcal_device_count()


def set_device(i: int):
    check(lib().gsmcal_set_device(int(i)))


def launch_count(reset: bool = False) -> int:
    return int(lib().gsmcal_launch_count(1 if reset else 0))


# ---- K1 raw2iq.m:5-8 -------------------------------------------------------------------------------
def raw2iq(a) -> np.ndarray:
    a = np.asarray(a)
    if a.dtype == np.uint8:
        buf, rows, cols = _cols(a, np.uint8)
        fn = lib().gsmcal_raw2iq_u8
    else:
        buf, rows, cols = _cols(a, np.float64)
        fn = lib().gsmcal_raw2iq_f64
    n = rows // 2
    out = np.empty((cols, n), dtype=np.complex128)
    check(fn(_ptr(buf), n, cols, _ptr(out)))
    return out.T


# ---- K2 ----------------------------------------------------------------------------------------------
def fir1(order: int, wn: float) -> np.ndarray:
    coef = np.empty(order + 1)
    check(lib().gsmcal_fir1(int(order), float(wn), _ptr(coef)))
    return coef


def fir_filter(coef, s, decim: int = 1) -> np.ndarray:
    """filter(coef,1,s) then s(1:decim:end,:)  (gsm_sync_demod.m:110,117)."""
    coef = np.ascontiguousarray(coef, dtype=np.float64)
    s = np.asarray(s)
    one_d = s.ndim == 1
    buf, n, cols = _cols(s, np.complex128)
    n_out = (n + decim - 1) // decim
    out = np.empty((cols, n_out), dtype=np.complex128)
    check(lib().gsmcal_fir_filter(_ptr(coef), len(coef), _ptr(buf), n, cols, int(decim), _ptr(out)))
    return out[0] if one_d else out.T


def raw2iq_fir(a_u8, coef, decim: int = 1) -> np.ndarray:
    coef = np.ascontiguousarray(coef, dtype=np.float64)
    buf, rows, cols = _cols(a_u8, np.uint8)
    n = rows // 2
    n_out = (n + decim - 1) // decim
    out = np.empty((cols, n_out), dtype=np.complex128)
    check(lib().gsmcal_raw2iq_fir_u8(_ptr(buf), n, cols, _ptr(coef), len(coef), int(decim), _ptr(out)))
    return out.T


def chn_filter_taps(which: int) -> np.ndarray:
    coef = np.empty(64)
    n = C.c_int(0)
    check(lib().gsmcal_chn_filter_taps(int(which), _ptr(coef), C.byref(n)))
    return coef[:n.value].copy()


def chn_filter_8x_4x(s) -> np.ndarray:
    s = np.asarray(s)
    one_d = s.ndim == 1
    buf, n, cols = _cols(s, np.complex128)
    out = np.empty((cols, (n + 1) // 2), dtype=np.complex128)
    check(lib().gsmcal_chn_filter_8x_4x(_ptr(buf), n, cols, _ptr(out)))
    return out[0] if one_d else out.T


def chn_filter_4x(s) -> np.ndarray:
    s = np.asarray(s)
    one_d = s.ndim == 1
    buf, n, cols = _cols(s, np.complex128)
    out = np.empty((cols, n), dtype=np.complex128)
    check(lib().gsmcal_chn_filter_4x(_ptr(buf), n, cols, _ptr(out)))
    return out[0] if one_d else out.T


def band_power(a_u8, coef=None, decim: int = 1) -> np.ndarray:
    """mean(abs(r(1:decim:end,:)).^2,1): scan_band_power_spectrum.m:80-85 / multi_rtl_sdr_split_scanner.m:154-156."""
    buf, rows, cols = _cols(a_u8, np.uint8)
    out = np.empty(cols)
    if coef is None:
        check(lib().gsmcal_band_power_u8(_ptr(buf), rows // 2, cols, None, 0, int(decim), _ptr(out)))
    else:
        coef = np.ascontiguousarray(coef, dtype=np.float64)
        check(lib().gsmcal_band_power_u8(_ptr(buf), rows // 2, cols, _ptr(coef), len(coef), int(decim), _ptr(out)))
    return out


# ---- K3 ----------------------------------------------------------------------------------------------
def _stream(s):
    return np.ascontiguousarray(np.asarray(s).reshape(-1), dtype=np.complex128)


def move_fft_snr_runtime_avg(s, mv_len: int, fft_len: int, th: float):
    s = _stream(s)
    flag = C.c_int(0)
    idx, avg, snr = C.c_double(), C.c_double(), C.c_double()
    check(lib().gsmcal_move_fft_snr_runtime_avg(_ptr(s), len(s), int(mv_len), int(fft_len), float(th),
                                                C.byref(flag), C.byref(idx), C.byref(avg), C.byref(snr)))
    return bool(flag.value), idx.value, avg.value, snr.value


def move_fft_snr_trace(s, fft_len: int) -> np.ndarray:
    s = _stream(s)
    out = np.empty(len(s) - fft_len + 1)
    check(lib().gsmcal_move_fft_snr_trace(_ptr(s), len(s), int(fft_len), _ptr(out)))
    return out


def specific_fft_snr_fix_avg(s, target_set, fft_len: int, th: float, avg_snr: float):
    s = _stream(s)
    flag = C.c_int(0)
    idx, snr = C.c_double(), C.c_double()
    check(lib().gsmcal_specific_fft_snr_fix_avg(_ptr(s), len(s), int(target_set[0]), int(target_set[1]), int(fft_len),
                                                float(th), float(avg_snr), C.byref(flag), C.byref(idx), C.byref(snr)))
    return bool(flag.value), idx.value, snr.value


# ---- K4 ----------------------------------------------------------------------------------------------
def FCCH_coarse_position(s, decimation_ratio: int):
    s = _stream(s)
    cap = int(lib().gsmcal_max_bursts(len(s), int(decimation_ratio)))
    pos, snr = np.empty(cap), np.empty(cap)
    n = C.c_int64(0)
    check(lib().gsmcal_FCCH_coarse_position(_ptr(s), len(s), int(decimation_ratio), _ptr(pos), _ptr(snr), cap, C.byref(n)))
    if n.value < 0:
        return np.array([-1.0]), np.array([-1.0])
    return pos[:n.value].copy(), snr[:n.value].copy()


# ---- K5-K8 --------------------------------------------------------------------------------------------
def FCCH_fine_correction(s, base_position, oversampling_ratio: int, carrier_freq: float):
    s = _stream(s)
    base = np.ascontiguousarray(np.asarray(base_position, dtype=np.float64).reshape(-1))
    pos = np.empty(max(len(base), 1))
    r = np.empty(len(s), dtype=np.complex128)
    n_pos, r_len = C.c_int64(0), C.c_int64(0)
    sppm, cppm = C.c_double(), C.c_double()
    check(lib().gsmcal_FCCH_fine_correction(_ptr(s), len(s), _ptr(base), len(base), int(oversampling_ratio), float(carrier_freq),
                                            _ptr(pos), len(pos), C.byref(n_pos), _ptr(r), len(r), C.byref(r_len),
                                            C.byref(sppm), C.byref(cppm)))
    fcch_pos = np.array([-1.0]) if n_pos.value < 0 else pos[:n_pos.value].copy()
    r_out = None if r_len.value < 0 else r[:r_len.value]
    return fcch_pos, r_out, sppm.value, cppm.value


def gsm_SCH_training_sequence_gen(oversampling_ratio: int) -> np.ndarray:
    out = np.empty(64 * oversampling_ratio, dtype=np.complex128)
    check(lib().gsmcal_SCH_training_sequence_gen(int(oversampling_ratio), _ptr(out)))
    return out


def SCH_corr_rate_correction(s, FCCH_pos, sch_training_sequence, oversampling_ratio: int):
    fpos = np.ascontiguousarray(np.asarray(FCCH_pos, dtype=np.float64).reshape(-1))
    tpl = _stream(sch_training_sequence)
    if tpl.size != 64 * oversampling_ratio:
        raise ValueError("sch_training_sequence must hold 64*oversampling_ratio samples")
    s = _stream(s if s is not None else [-1.0])
    rows_cap = max(6 * len(fpos), 1)
    pinfo = np.empty(2 * rows_cap)
    r = np.empty(len(s), dtype=np.complex128)
    n_rows, r_len = C.c_int64(0), C.c_int64(0)
    sppm = C.c_double()
    check(lib().gsmcal_SCH_corr_rate_correction(_ptr(s), len(s), _ptr(fpos), len(fpos), _ptr(tpl), int(oversampling_ratio),
                                                _ptr(pinfo), rows_cap, C.byref(n_rows), _ptr(r), len(r), C.byref(r_len), C.byref(sppm)))
    if n_rows.value < 0:
        pos_info = np.array([[-1.0, -1.0]])
    else:
        nr = n_rows.value
        pos_info = np.stack([pinfo[:nr], pinfo[nr:2 * nr]], axis=1)
    r_out = None if r_len.value < 0 else r[:r_len.value]
    return pos_info, r_out, sppm.value


def carrier_correct_post_SCH(s, pos_info, oversampling_ratio: int, carrier_freq: float):
    pinfo = np.asarray(pos_info, dtype=np.float64).reshape(-1, 2)
    flat = np.ascontiguousarray(np.concatenate([pinfo[:, 0], pinfo[:, 1]]))
    s = _stream(s if s is not None else [-1.0])
    r = np.empty(len(s), dtype=np.complex128)
    r_len = C.c_int64(0)
    cppm = C.c_double()
    check(lib().gsmcal_carrier_correct_post_SCH(_ptr(s), len(s), _ptr(flat), pinfo.shape[0], int(oversampling_ratio), float(carrier_freq),
                                                _ptr(r), len(r), C.byref(r_len), C.byref(cppm)))
    return (None if r_len.value < 0 else r[:r_len.value]), cppm.value


def total_ppm_calculation(ppm_in) -> float:
    p = np.ascontiguousarray(np.asarray(ppm_in, dtype=np.float64).reshape(-1))
    out = C.c_double()
    check(lib().gsmcal_total_ppm_calculation(_ptr(p), len(p), C.byref(out)))
    return out.value


# ---- SURVEY 8(f) rows 2 and 4: FCCH_demod.m, BCCH_demod.m, SCH_demod.m, gsm_normal_training_sequence_gen.m -------------
def _pinfo(pos_info):
    pinfo = np.asarray(pos_info, dtype=np.float64).reshape(-1, 2)
    return pinfo, np.ascontiguousarray(np.concatenate([pinfo[:, 0], pinfo[:, 1]]))


def gsm_normal_training_sequence_gen(oversampling_ratio: int) -> np.ndarray:
    """(26*osr) x 8 complex128, one normal training sequence per column."""
    out = np.empty((8, 26 * int(oversampling_ratio)), dtype=np.complex128)
    check(lib().gsmcal_normal_training_sequence_gen(int(oversampling_ratio), _ptr(out)))
    return out.T


def FCCH_demod(s, pos_info, oversampling_ratio: int, carrier_freq: float):
    """What FCCH_demod.m displays: dict(freq, mean_freq, carrier_ppm, snr, max_idx); None on the `pos_info==-1` path."""
    pinfo, flat = _pinfo(pos_info)
    s = _stream(s if s is not None else [-1.0])
    cap = max(1, pinfo.shape[0])
    freq, snr, idx = np.empty(cap), np.empty(cap), np.empty(cap)
    n, mf, cp = C.c_int64(0), C.c_double(), C.c_double()
    check(lib().gsmcal_FCCH_demod(_ptr(s), len(s), _ptr(flat), pinfo.shape[0], int(oversampling_ratio), float(carrier_freq),
                                  _ptr(freq), _ptr(snr), _ptr(idx), cap, C.byref(n), C.byref(mf), C.byref(cp)))
    if n.value < 0:
        return None
    k = n.value
    return dict(freq=freq[:k], mean_freq=mf.value, carrier_ppm=cp.value, snr=snr[:k], max_idx=idx[:k])


def BCCH_demod(s, pos_info, normal_training_sequence, oversampling_ratio: int, carrier_freq: float):
    """(carrier_ppm, normal_training_sequence_idx, |corr_val| 8 x 4 or None); (-1, -1, None) on the early returns."""
    pinfo, flat = _pinfo(pos_info)
    s = _stream(s if s is not None else [-1.0])
    nts = np.ascontiguousarray(np.asarray(normal_training_sequence, dtype=np.complex128).T)     # column-major (26*osr) x 8
    mag = np.full((4, 8), np.nan)
    cp, idx = C.c_double(), C.c_int()
    check(lib().gsmcal_BCCH_demod(_ptr(s), len(s), _ptr(flat), pinfo.shape[0], _ptr(nts), int(oversampling_ratio), float(carrier_freq),
                                  C.byref(cp), C.byref(idx), _ptr(mag)))
    return cp.value, idx.value, (None if np.isnan(mag).all() else mag.T.copy())


def SCH_demod(s, pos_info, training_sequence, oversampling_ratio: int):
    """dict(demod_bits [H x 148], bits_to_decoder [H x 148], corr_val [H x 85]); None on the `pos_info==-1` path."""
    pinfo, flat = _pinfo(pos_info)
    s = _stream(s if s is not None else [-1.0])
    tpl = _stream(training_sequence)
    cap = max(1, pinfo.shape[0])
    bits, dec, corr = np.zeros((cap, 148), dtype=np.uint8), np.zeros((cap, 148), dtype=np.uint8), np.zeros((cap, 85))
    n = C.c_int64(0)
    check(lib().gsmcal_SCH_demod(_ptr(s), len(s), _ptr(flat), pinfo.shape[0], _ptr(tpl), int(oversampling_ratio), cap, C.byref(n),
                                 _ptr(bits), _ptr(dec), _ptr(corr)))
    if n.value < 0:
        return None
    k = n.value
    return dict(demod_bits=bits[:k].astype(np.int64), bits_to_decoder=dec[:k].astype(np.int64), corr_val=corr[:k])


# ---- batched pipeline ---------------------------------------------------------------------------------
def max_bursts(n_iq: int, osr: int = 8, coarse_dr: int = 8) -> int:
    dec = osr * coarse_dr
    return int(lib().gsmcal_max_bursts((n_iq + dec - 1) // dec, coarse_dr))


def _unpack_results(res, D, cap, coarse_pos, coarse_snr, fcch_pos, pos_info):
    out = []
    for d in range(D):
        r = res[d]
        item = dict(
            coarse_pos=np.array([-1.0]) if r.n_coarse < 0 else coarse_pos[d, :r.n_coarse].copy(),
            coarse_snr=np.array([-1.0]) if r.n_coarse < 0 else coarse_snr[d, :r.n_coarse].copy(),
            fcch_pos=np.array([-1.0]) if r.n_fcch < 0 else fcch_pos[d, :r.n_fcch].copy(),
            pos_info=np.array([[-1.0, -1.0]]) if r.n_pos_info < 0 else pos_info[d, :r.n_pos_info, :].copy(),
            sampling_ppm=(r.sampling_ppm[0], r.sampling_ppm[1]),
            carrier_ppm=(r.carrier_ppm[0], r.carrier_ppm[1]),
            total_sampling_ppm=r.total_sampling_ppm, total_carrier_ppm=r.total_carrier_ppm,
            r_len=tuple(r.r_len), flags=r.flags)
        out.append(item)
    return out


def _batch_args(raw, carrier_freq, sch_training_sequence, coef, osr, coarse_dr, device_ptr, n_iq, n_streams, cuda_stream, details):
    """The 16 leading arguments of gsmcal_calibrate_batch and its variants, for `raw` ([D, 2N] uint8 on the host, or one row) or, with
    device_ptr, a capture of n_streams x n_iq resident in HBM.  Returns (args, keep, D, n_iq, cap, res, arrays): keep holds the host
    arrays args point into, res the D result records, arrays (coarse_pos, coarse_snr, fcch_pos, pos_info), or None without details."""
    tpl = _stream(sch_training_sequence)
    coef = np.ascontiguousarray(coef, dtype=np.float64)
    if device_ptr is None:
        raw = np.ascontiguousarray(raw, dtype=np.uint8)
        if raw.ndim == 1:
            raw = raw[None, :]
        D, n_iq = raw.shape[0], raw.shape[1] // 2
        ptr, mem = _ptr(raw), 0
    else:
        D, ptr, mem = int(n_streams), C.c_void_p(int(device_ptr)), 1
    cap = max_bursts(n_iq, osr, coarse_dr)
    res = (StreamResult * D)()
    arrays = (np.empty((D, cap)), np.empty((D, cap)), np.empty((D, cap)), np.empty((D, 6 * cap, 2))) if details else None
    args = [ptr, mem, int(n_iq), D, float(carrier_freq), _ptr(tpl), _ptr(coef), len(coef), int(osr), int(coarse_dr), C.cast(res, C.c_void_p),
            *([_ptr(a) for a in arrays] if details else [None] * 4), C.c_void_p(cuda_stream)]
    return args, (raw, tpl, coef), D, n_iq, cap, res, arrays


def calibrate_batch(raw, carrier_freq: float, sch_training_sequence, coef, osr: int = 8, coarse_dr: int = 8,
                    device_ptr: int | None = None, n_iq: int | None = None, n_streams: int | None = None,
                    cuda_stream: int = 0, details: bool = True, r_correct=None, r_device_ptr: int | None = None,
                    sch_timing: bool = False, carrier_fit: bool = False, sch_decode: bool = False, sysinfo: bool = False):
    """gsm_sync_demod.m:107-124 for every row of `raw` ([D, 2N] uint8, row d == dongle d's fread column).

    `raw` is a host NumPy array, or pass device_ptr/n_iq/n_streams for a capture already resident in HBM.
    Returns a list of per-stream dicts with the same keys as the function-by-function chain.

    sch_timing=True (osr 8, not with r_correct / r_device_ptr, implies details) also times every SCH burst of pos_info to a fraction
    of a sample on r_correct and fits a line through the burst times (gsmcal_calibrate_sch_timing_batch, include/gsmcal.h); each dict
    gains timing: dict(t0, fit_ppm, rms, n_fit, flags, tau, x): t0 the raw-capture time (0-based samples) of the first fitted burst's
    training start, fit_ppm the sample clock error of the fit, rms its residual (samples), flags TIMING_* bits, and per SCH row tau (time
    in r_correct, 1-based) and x (time in the uint8 capture, 0-based), NaN where excluded; tau and x are None when the step did not
    run (TIMING_NO_POS_INFO / TIMING_NO_R_CORRECT).

    carrier_fit=True (osr 8, not with r_correct / r_device_ptr or sch_timing, implies details) also estimates the tone of every FCCH
    burst of pos_info on r_correct from the periodogram maximum of its interior and fits a line through the tones over capture time
    (gsmcal_calibrate_carrier_fit_batch, include/gsmcal.h); each dict gains carrier: dict(carrier_fit_ppm, drift_ppm_per_s, t_mean,
    freq_hz, drift_hz_per_s, rms_hz, residual_ppm, n_fit, flags, f, t, row_flags): carrier_fit_ppm the dongle's carrier error at t_mean
    (seconds of capture time), drift_ppm_per_s its drift, freq_hz / drift_hz_per_s / rms_hz the line through the tones in r_correct's
    frame, residual_ppm what total_carrier_ppm left, flags CARRIER_* bits, and per FCCH row f (Hz), t (s) and row_flags, f and t NaN
    where excluded; f, t and row_flags are None when the step did not run (CARRIER_NO_POS_INFO / CARRIER_NO_R_CORRECT).

    sch_decode=True (only with carrier_fit=True) then demodulates every SCH burst of pos_info on r_correct with the fitted residual
    removed and decodes it (gsmcal_calibrate_cell_batch, include/gsmcal.h); each dict also gains
      cell: calibrate_demod_batch(..., sch_decode=True)'s cell dict plus df, the residual removed from each SCH row (Hz; NaN without a
            fit, where flags has SCHDEC_UNCORRECTED and the rows are demodulated as calibrate_demod_batch does);
      sch:  dict(demod_bits [n x 148], corr_val [n x 85], sch_ok [n] bool) of the corrected rows, n = SCH rows of pos_info.
    cell's per-row arrays and sch are None where SCH_demod did not run.  frame_clock_offsets takes these results as they are.

    sysinfo=True (only with carrier_fit=True and sch_decode=True) then decodes every BCCH block of pos_info with the training sequence of
    the cell's BCC (gsmcal_calibrate_sysinfo_batch, include/gsmcal.h); each dict also gains
      sysinfo: dict(n_blocks, n_fire_ok, n_si3, n_si3_agree, flags, si_mask, mcc, mnc, mnc_digits, lac, ci, cgi, fn, tc, block_flags,
               hamming, payload, lag, row_flags, steal): flags SI_* bits, si_mask SI_HAS_* bits, the SI3 fields (-1 without an SI3) and
               cgi = (mcc, mnc, mnc_digits, lac, ci) or None; per block fn, tc, block_flags, hamming [n] and payload [n x 23] uint8; per
               BCCH row lag, row_flags, steal [n x 4] (lag -128 where the row was not correlated).  The arrays are None when n_blocks < 0."""
    if (sch_timing or carrier_fit) and (r_correct is not None or r_device_ptr is not None):
        raise ValueError("sch_timing / carrier_fit do not combine with r_correct / r_device_ptr")
    if sch_timing and carrier_fit:
        raise ValueError("sch_timing and carrier_fit are separate calls")
    if sch_decode and (sch_timing or not carrier_fit):
        raise ValueError("calibrate_batch decodes SCH bursts only with carrier_fit=True and without sch_timing")
    if sysinfo and not (carrier_fit and sch_decode):
        raise ValueError("calibrate_batch decodes BCCH blocks only with carrier_fit=True and sch_decode=True")
    details = details or sch_timing or carrier_fit
    args, keep, D, n_iq, cap, res, arrays = _batch_args(raw, carrier_freq, sch_training_sequence, coef, osr, coarse_dr, device_ptr, n_iq,
                                                        n_streams, cuda_stream, details)
    if sch_timing:
        tm = (SchTimingResult * D)()
        tau, x = np.empty((D, cap)), np.empty((D, cap))
        check(lib().gsmcal_calibrate_sch_timing_batch(*args, C.cast(tm, C.c_void_p), _ptr(tau), _ptr(x)))
    elif carrier_fit:
        cf = (CarrierFitResult * D)()
        f, t, rf = np.empty((D, cap)), np.empty((D, cap)), np.empty((D, cap), dtype=np.uint8)
        cf_args = [C.cast(cf, C.c_void_p), _ptr(f), _ptr(t), _ptr(rf)]
        if sch_decode:
            sd = (SchDecodeResult * D)()
            sch_ok, bits, corr = np.zeros((D, cap), dtype=np.uint8), np.zeros((D, cap, 148), dtype=np.uint8), np.zeros((D, cap, 85))
            df, fn, bsic = np.empty((D, cap)), np.empty((D, cap), dtype=np.int32), np.empty((D, cap), dtype=np.int32)
            ham, rfl = np.empty((D, cap), dtype=np.uint8), np.empty((D, cap), dtype=np.uint8)
            cell_args = [C.cast(sd, C.c_void_p), _ptr(sch_ok), _ptr(bits), _ptr(corr), _ptr(df), _ptr(fn), _ptr(bsic), _ptr(ham), _ptr(rfl)]
            if sysinfo:
                nts = np.ascontiguousarray(gsm_normal_training_sequence_gen(osr).T)          # column-major (26*osr) x 8
                si = (SysinfoResult * D)()
                lag, brf, steal = (np.empty((D, cap, 4), dtype=t) for t in (np.int8, np.uint8, np.uint8))
                bfn, btc, bfl = np.empty((D, cap), dtype=np.int32), np.empty((D, cap), dtype=np.uint8), np.empty((D, cap), dtype=np.uint8)
                bham, pay = np.empty((D, cap), dtype=np.uint16), np.empty((D, cap, 23), dtype=np.uint8)
                check(lib().gsmcal_calibrate_sysinfo_batch(*args, *cf_args, *cell_args, _ptr(nts), C.cast(si, C.c_void_p), _ptr(lag), _ptr(brf),
                                                           _ptr(steal), _ptr(bfn), _ptr(btc), _ptr(bfl), _ptr(bham), _ptr(pay)))
            else:
                check(lib().gsmcal_calibrate_cell_batch(*args, *cf_args, *cell_args))
        else:
            check(lib().gsmcal_calibrate_carrier_fit_batch(*args, *cf_args))
    elif r_correct is None and r_device_ptr is None:
        check(lib().gsmcal_calibrate_batch(*args))
    else:
        # r_correct: a [D, n_iq] complex128 host array to fill, or r_device_ptr: a device buffer of D * n_iq complex128
        if r_device_ptr is not None:
            rp, rmem = C.c_void_p(int(r_device_ptr)), 1
        else:
            assert r_correct.dtype == np.complex128 and r_correct.flags.c_contiguous and r_correct.shape == (D, n_iq)
            rp, rmem = _ptr(r_correct), 0
        check(lib().gsmcal_calibrate_batch_r(*args, rp, rmem, int(n_iq)))
    if not details:
        return res
    out = _unpack_results(res, D, cap, *arrays)
    if sch_timing:
        for d, item in enumerate(out):
            t = tm[d]
            n = t.n_sch
            item["timing"] = dict(t0=t.t0, fit_ppm=t.fit_ppm, rms=t.rms, n_fit=t.n_fit, flags=t.flags,
                                  tau=None if n < 0 else tau[d, :n].copy(), x=None if n < 0 else x[d, :n].copy())
    if carrier_fit:
        for d, item in enumerate(out):
            c = cf[d]
            n = c.n_fcch
            item["carrier"] = dict(carrier_fit_ppm=c.carrier_fit_ppm, drift_ppm_per_s=c.drift_ppm_per_s, t_mean=c.t_mean, freq_hz=c.freq_hz,
                                   drift_hz_per_s=c.drift_hz_per_s, rms_hz=c.rms_hz, residual_ppm=c.residual_ppm, n_fit=c.n_fit,
                                   flags=c.flags, f=None if n < 0 else f[d, :n].copy(), t=None if n < 0 else t[d, :n].copy(),
                                   row_flags=None if n < 0 else rf[d, :n].astype(np.int64))
    if sch_decode:
        for d, item in enumerate(out):
            item["cell"] = _cell_dict(sd[d], d, fn, bsic, ham, rfl)
            n = sd[d].n_sch
            item["cell"]["df"] = None if n < 0 else df[d, :n].copy()
            item["sch"] = None if n < 0 else dict(demod_bits=bits[d, :n].astype(np.int64), corr_val=corr[d, :n].copy(),
                                                  sch_ok=sch_ok[d, :n].astype(bool))
    if sysinfo:
        for d, item in enumerate(out):
            r, n = si[d], si[d].n_blocks
            rows = lambda a: None if n < 0 else a[d, :n].astype(np.int64)          # noqa: E731
            item["sysinfo"] = dict(n_blocks=n, n_fire_ok=r.n_fire_ok, n_si3=r.n_si3, n_si3_agree=r.n_si3_agree, flags=r.flags,
                                   si_mask=r.si_mask, mcc=r.mcc, mnc=r.mnc, mnc_digits=r.mnc_digits, lac=r.lac, ci=r.ci,
                                   cgi=None if r.flags & SI_NO_SI3 or n < 0 else (r.mcc, r.mnc, r.mnc_digits, r.lac, r.ci),
                                   fn=rows(bfn), tc=rows(btc), block_flags=rows(bfl), hamming=rows(bham),
                                   payload=None if n < 0 else pay[d, :n].copy(), lag=rows(lag), row_flags=rows(brf), steal=rows(steal))
    return out


def _cell_dict(c, d, fn, bsic, ham, rfl):
    """the cell dict of stream d from its gsmcal_sch_decode_result and the per-row arrays"""
    n = c.n_sch
    rows = lambda a: None if n < 0 else a[d, :n].astype(np.int64)          # noqa: E731
    return dict(bsic=c.bsic, ncc=c.bsic >> 3 if c.bsic >= 0 else -1, bcc=c.bsic & 7 if c.bsic >= 0 else -1, fn_first=c.fn_first,
                frame_clock_start=c.frame_clock_start, n_crc_ok=c.n_crc_ok, n_agree=c.n_agree, flags=c.flags, fn=rows(fn),
                bsic_rows=rows(bsic), hamming=rows(ham), row_flags=rows(rfl))


TIMING_NO_POS_INFO, TIMING_NO_R_CORRECT, TIMING_RANGE, TIMING_EDGE, TIMING_FEW = 1, 2, 4, 8, 16
CARRIER_NO_POS_INFO, CARRIER_NO_R_CORRECT, CARRIER_RANGE, CARRIER_EDGE, CARRIER_NOCONV, CARRIER_FEW = 1, 2, 4, 8, 16, 32
DEMOD_NO_POS_INFO, DEMOD_NO_R_CORRECT, DEMOD_SCH_RANGE, DEMOD_FCCH_RANGE = 1, 2, 4, 8
BCCH_NO_POS_INFO, BCCH_FEW_BCCH, BCCH_FCCH_RANGE, BCCH_TRAIN_RANGE = 1, 2, 4, 8
SCHDEC_NO_POS_INFO, SCHDEC_NO_R_CORRECT, SCHDEC_NONE, SCHDEC_DISAGREE = 1, 2, 4, 8
SCHDEC_ROW_WINDOW, SCHDEC_ROW_ALIGN, SCHDEC_ROW_CRC, SCHDEC_ROW_FIELD = 1, 2, 4, 8
SCHDEC_UNCORRECTED = 16                            # calibrate_batch(..., carrier_fit=True, sch_decode=True): no fit, rows not corrected
SI_NO_POS_INFO, SI_NO_R_CORRECT, SI_NO_CELL, SI_UNCORRECTED, SI_NO_SI3, SI_SI3_DISAGREE = 1, 2, 4, 8, 16, 32
SI_ROW_RANGE, SI_ROW_EDGE = 1, 2
SI_BLK_FN, SI_BLK_ROW, SI_BLK_FIRE, SI_BLK_SHORT = 1, 2, 4, 8
SI_HAS = {0x19: 1, 0x1A: 2, 0x02: 4, 0x03: 8, 0x07: 16, 0x1B: 32, 0x1C: 64, 0x00: 128}     # message type -> si_mask bit
SI_HAS_OTHER = 256
FN_MOD = 2715648                                   # TDMA frames in a hyperframe


def calibrate_demod_batch(raw, carrier_freq: float, sch_training_sequence, coef, osr: int = 8, coarse_dr: int = 8,
                          device_ptr: int | None = None, n_iq: int | None = None, n_streams: int | None = None, cuda_stream: int = 0,
                          normal_training_sequence=None, sch_decode: bool = False):
    """calibrate_batch followed by SCH_demod / FCCH_demod on every stream's r_correct (gsm_sync_demod.m:144-145), which is never
    materialised.  Same inputs as calibrate_batch.  Each per-stream dict holds calibrate_batch's keys plus
      sch:  dict(demod_bits [n x 148], bits_to_decoder [n x 148], corr_val [n x 85], sch_ok [n] bool), n = SCH rows of pos_info;
            a row whose equaliser window leaves r_correct has sch_ok False and zeros;
      fcch: dict(freq, mean_freq, carrier_ppm, snr, max_idx) as FCCH_demod returns it; NaN for a window outside r_correct, and
            mean_freq / carrier_ppm NaN unless every window lies inside;
      demod_flags: DEMOD_* bits.
    sch and fcch are None where the demodulators do not run: pos_info == -1 (DEMOD_NO_POS_INFO) or r_correct == -1
    (DEMOD_NO_R_CORRECT).
    With normal_training_sequence ((26*osr) x 8, gsm_normal_training_sequence_gen) BCCH_demod (gsm_sync_demod.m:146) runs as well and
    each dict gains
      bcch: dict(carrier_ppm, nts_idx, corr_abs, flags): carrier_ppm of r_correct (== fcch carrier_ppm), nts_idx 1..8 or -1, corr_abs
            abs(corr_val) 8 x 4 (NaN columns for training windows outside r_correct, BCCH_TRAIN_RANGE), flags BCCH_* bits; carrier_ppm,
            nts_idx, corr_abs are (-1, -1, None) for BCCH_NO_POS_INFO / BCCH_FEW_BCCH as BCCH_demod returns them, (NaN, -1, None) for
            BCCH_FCCH_RANGE (no FCCH mean to correct with).
    sch_decode=True also decodes every SCH burst (gsmcal_calibrate_sch_decode_batch, definition in include/gsmcal.h) and each dict gains
      cell: dict(bsic, ncc, bcc, fn_first, frame_clock_start, n_crc_ok, n_agree, flags, fn, bsic_rows, hamming, row_flags): the cell's
            BSIC (ncc = bsic >> 3, bcc = bsic & 7; -1 without a winner), the TDMA frame number of the first SCH row of pos_info, the GSM
            time of capture sample 0 in nominal samples since FN 0 (NaN without a winner), the rows that decoded and that voted for the
            winner, flags SCHDEC_* bits, and per SCH row fn, bsic_rows (-1 where not decoded), hamming and row_flags (SCHDEC_ROW_*);
            the per-row arrays are None where SCH_demod did not run.  A winner with n_agree 1 may be a false CRC pass (about 1 in 1024
            rows of noise passes the 10-bit CRC)."""
    args, keep, D, n_iq, cap, res, arrays = _batch_args(raw, carrier_freq, sch_training_sequence, coef, osr, coarse_dr, device_ptr, n_iq,
                                                        n_streams, cuda_stream, True)
    dem = (DemodResult * D)()
    sch_ok = np.zeros((D, cap), dtype=np.uint8)
    bits, dec = np.zeros((D, cap, 148), dtype=np.uint8), np.zeros((D, cap, 148), dtype=np.uint8)
    corr = np.zeros((D, cap, 85))
    freq, snr, idx = np.empty((D, cap)), np.empty((D, cap)), np.empty((D, cap))
    args += [C.cast(dem, C.c_void_p), _ptr(sch_ok), _ptr(bits), _ptr(dec), _ptr(corr), _ptr(freq), _ptr(snr), _ptr(idx)]
    nts_args = [None, None]
    if normal_training_sequence is not None:
        nts_m = np.asarray(normal_training_sequence)
        if nts_m.shape != (26 * int(osr), 8):
            raise ValueError("normal_training_sequence must be (26*osr) x 8")
        nts = np.ascontiguousarray(nts_m.T, dtype=np.complex128)                # column-major (26*osr) x 8
        bc = (BcchResult * D)()
        nts_args = [_ptr(nts), C.cast(bc, C.c_void_p)]
    if sch_decode:
        sd = (SchDecodeResult * D)()
        fn, bsic = np.empty((D, cap), dtype=np.int32), np.empty((D, cap), dtype=np.int32)
        ham, rfl = np.empty((D, cap), dtype=np.uint8), np.empty((D, cap), dtype=np.uint8)
        check(lib().gsmcal_calibrate_sch_decode_batch(*args, *nts_args, C.cast(sd, C.c_void_p), _ptr(fn), _ptr(bsic), _ptr(ham), _ptr(rfl)))
    elif normal_training_sequence is None:
        check(lib().gsmcal_calibrate_demod_batch(*args))
    else:
        check(lib().gsmcal_calibrate_demod_bcch_batch(*args, *nts_args))
    out = _unpack_results(res, D, cap, *arrays)
    for d, item in enumerate(out):
        r = dem[d]
        item["demod_flags"] = r.flags
        ns, nf = r.n_sch, r.n_fcch
        item["sch"] = None if ns < 0 else dict(demod_bits=bits[d, :ns].astype(np.int64), bits_to_decoder=dec[d, :ns].astype(np.int64),
                                               corr_val=corr[d, :ns].copy(), sch_ok=sch_ok[d, :ns].astype(bool))
        item["fcch"] = None if nf < 0 else dict(freq=freq[d, :nf].copy(), mean_freq=r.fcch_mean_freq, carrier_ppm=r.fcch_carrier_ppm,
                                                snr=snr[d, :nf].copy(), max_idx=idx[d, :nf].copy())
        if normal_training_sequence is not None:
            b = bc[d]
            none = b.flags & (BCCH_NO_POS_INFO | BCCH_FEW_BCCH | BCCH_FCCH_RANGE)
            item["bcch"] = dict(carrier_ppm=b.carrier_ppm, nts_idx=b.nts_idx, flags=b.flags,
                                corr_abs=None if none else np.array(b.corr_abs).reshape(4, 8).T.copy())
        if sch_decode:
            item["cell"] = _cell_dict(sd[d], d, fn, bsic, ham, rfl)
    return out


def frame_clock_offsets(results, ref: int = 0, osr: int = 8) -> np.ndarray:
    """Capture-start offsets on the cell's frame clock, from calibrate_demod_batch(..., sch_decode=True) or calibrate_batch(...,
    carrier_fit=True, sch_decode=True) results: for every stream that
    decoded the same BSIC as stream `ref` (both with a winner), frame_clock_start[d] - frame_clock_start[ref] wrapped into (-H/2, H/2],
    H = one hyperframe = 2,715,648 * 1250 * osr nominal samples; NaN for every other stream.  Positive: stream d started later."""
    h = float(FN_MOD * 1250 * int(osr))
    cells = [r["cell"] for r in results]
    c0 = cells[ref]
    out = np.full(len(cells), np.nan)
    if c0["bsic"] < 0:
        return out
    for d, c in enumerate(cells):
        if c["bsic"] == c0["bsic"] and c["n_agree"] > 0:
            v = (c["frame_clock_start"] - c0["frame_clock_start"]) % h                # exact: integer-valued doubles below 2^53
            out[d] = v - h if v > h / 2 else v
    return out


class PendingBatch:
    """A batch submitted with calibrate_batch_submit: owns the output arrays until collect() fills them."""

    def __init__(self, slot, D, cap, res, arrays, keep):
        self.slot, self.D, self.cap, self.res, self.arrays, self._keep = slot, D, cap, res, arrays, keep
        self._open = True

    def cancel(self):
        """Give the slot back without results (the library never writes this object's arrays after that)."""
        if self._open:
            self._open = False
            check(lib().gsmcal_calibrate_batch_cancel(self.slot))

    def __del__(self):                       # a dropped PendingBatch must not leave its slot busy with dangling pointers
        try:
            self.cancel()
        except Exception:
            pass

    def collect(self, details: bool | None = None):
        if not self._open:
            raise GsmcalError(-1, "this batch was already collected or cancelled")
        check(lib().gsmcal_calibrate_batch_collect(self.slot))
        self._open = False
        if self.arrays is None or details is False:
            return self.res
        return _unpack_results(self.res, self.D, self.cap, *self.arrays)


def calibrate_batch_submit(slot: int, device_ptr: int, n_iq: int, n_streams: int, carrier_freq: float, sch_training_sequence, coef,
                           osr: int = 8, coarse_dr: int = 8, cuda_stream: int = 0, details: bool = False) -> PendingBatch:
    """Enqueue gsm_sync_demod.m:107-124 for a capture resident in HBM and return at once; `.collect()` waits for the results.
    Up to 4 slots may be in flight: the front of batch k+1 overlaps the FP64-bound stages of batch k on the device."""
    args, keep, D, n_iq, cap, res, arrays = _batch_args(None, carrier_freq, sch_training_sequence, coef, osr, coarse_dr, device_ptr, n_iq,
                                                        n_streams, cuda_stream, details)
    check(lib().gsmcal_calibrate_batch_submit(int(slot), args[0], *args[2:]))             # no raw_mem: the capture is on the device
    return PendingBatch(int(slot), D, cap, res, arrays, keep)


STAGE_NAMES = ("colsum_u8", "coarse", "fine_peak", "fine_tone", "sch", "post", "demod")


def last_batch_stage_ms() -> dict:
    ms = np.zeros(8)
    n = lib().gsmcal_last_batch_stage_ms(_ptr(ms), 8)
    return {STAGE_NAMES[i]: float(ms[i]) for i in range(n)}


def fcch_scan(raw, coef, osr: int = 8, coarse_dr: int = 8):
    """Per-channel FCCH detection of multi_rtl_sdr_gsm_FCCH_scanner.m:132-135,163-186.  raw: [n_chan, 2N] uint8."""
    raw = np.ascontiguousarray(raw, dtype=np.uint8)
    coef = np.ascontiguousarray(coef, dtype=np.float64)
    n_chan, n_iq = raw.shape[0], raw.shape[1] // 2
    cap = max_bursts(n_iq, osr, coarse_dr)
    snr, num_hit = np.empty(n_chan), np.empty(n_chan)
    pos = np.empty((n_chan, cap))
    npos = np.empty(n_chan, dtype=np.int32)
    check(lib().gsmcal_fcch_scan(_ptr(raw), 0, n_iq, n_chan, _ptr(coef), len(coef), int(osr), int(coarse_dr),
                                 _ptr(snr), _ptr(num_hit), _ptr(pos), _ptr(npos), None))
    positions = [np.array([-1.0]) if npos[i] < 0 else pos[i, :npos[i]].copy() for i in range(n_chan)]
    return snr, num_hit, positions


def diversity_power_spectrum(s_all_u8, coef, decim: int):
    """multi_rtl_sdr_diversity_scanner.m:150-176: every dongle scans the same band; per-dongle mean power after
    raw2iq -> filter -> r(1:decim:end), then the incoherent mean across dongles - one library call, the combination runs on the
    device.  s_all_u8: [2N, n_freq, n_dongle] uint8.  Returns (power_spectrum [n_dongle, n_freq], power_spectrum_combine [n_freq]),
    linear units."""
    s_all_u8 = np.asarray(s_all_u8, dtype=np.uint8)
    rows, n_freq, n_dongle = s_all_u8.shape
    buf = np.ascontiguousarray(np.transpose(s_all_u8, (2, 1, 0)))            # column-major 2N x n_freq x n_dongle == C order [dongle][freq][2N]
    coef = np.ascontiguousarray(coef, dtype=np.float64)
    per = np.empty((n_freq, n_dongle))                                        # column-major n_dongle x n_freq
    combine = np.empty(n_freq)
    check(lib().gsmcal_diversity_power_u8(_ptr(buf), rows // 2, n_freq, n_dongle, _ptr(coef), len(coef), int(decim), _ptr(per), _ptr(combine)))
    return per.T.copy(), combine
