"""fp64 restatement of gsmcal_calibrate_carrier_fit_batch (include/gsmcal.h): the carrier frequency of every FCCH burst of pos_info
from the periodogram maximum of its interior on r_correct, and the least-squares line through those frequencies over capture time.
Test infrastructure, like oracle/: the GPU results are compared against it and the synthetic truth checks run on it."""
from __future__ import annotations

import math

import numpy as np

OSR = 8
SYMBOL_RATE = (1625.0 / 6.0) * 1e3
FS = SYMBOL_RATE * OSR
F_NOM = SYMBOL_RATE / 4.0             # the FCCH tone, fs/32 at osr 8
OFF = 16 * OSR                        # the window starts 16 symbols into the burst
W = 116 * OSR                         # and covers 116 symbols: 928 samples
HALF = (W - 1) / 2.0                  # m = n - HALF, n = 0..W-1
GRID_K = 14                           # coarse grid: delta_k = k*FS/(4W), k = -14..14 (583.7 Hz steps, +-8172 Hz)
NEWTON = 5                            # Newton steps on P'(delta) = 0
TOL_HZ = 1e-4                         # |last step| above this: NOCONV
HZ_PER_RAD = FS / (2.0 * math.pi)     # omega (rad/sample) -> Hz

NO_POS_INFO, NO_R_CORRECT, RANGE, EDGE, NOCONV, FEW = 1, 2, 4, 8, 16, 32

TWIDDLE = np.exp(-1j * np.pi * np.arange(32) / 16.0)     # exp(-i*pi*n/16), n mod 32


def total_ppm2(a: float, b: float) -> float:
    """total_ppm_calculation([a, b]) (total_ppm_calculation.m:5-21)"""
    if a == math.inf and b == math.inf:
        return math.inf
    acc = 1.0
    acc = acc * (1.0 + a * 1e-6)
    acc = acc * (1.0 + b * 1e-6)
    return (acc - 1.0) * 1e6


def periodogram(y: np.ndarray, omega: float) -> float:
    """P = |sum y[n] exp(-i*omega*m)|^2 (re^2 + im^2), m = n - (W-1)/2"""
    m = np.arange(len(y)) - (len(y) - 1) / 2.0
    s = np.sum(y * np.exp(-1j * omega * m))
    return s.real * s.real + s.imag * s.imag


def tone_estimate(x: np.ndarray) -> dict:
    """One window of W samples (r_correct from p + 16*osr on): the nominal tone removed, the first maximum of the periodogram on the
    29-point grid, NEWTON Newton steps from it.  Returns f (Hz, NaN where excluded), the row flag, the grid index k* and the last step
    (Hz)."""
    x = np.asarray(x, dtype=np.complex128).reshape(-1)
    assert len(x) == W
    n = np.arange(W)
    m = n - HALF
    y = x * TWIDDLE[n % 32]
    ks = np.arange(-GRID_K, GRID_K + 1)
    s = np.exp(-1j * np.pi * np.outer(ks, m) / (2.0 * W)) @ y
    p = s.real * s.real + s.imag * s.imag
    i = int(np.argmax(p))                                       # first maximum
    k = int(ks[i])
    out = dict(k=k, f=math.nan, flag=0, last_step_hz=math.nan)
    if abs(k) == GRID_K:
        out["flag"] = EDGE
        return out
    omega = math.pi * k / (2.0 * W)
    step = 0.0
    for _ in range(NEWTON):
        v = y * np.exp(-1j * omega * m)
        s0, s1, s2 = np.sum(v), np.sum(m * v), np.sum(m * m * v)
        num = (s0.conjugate() * s1).imag                         # P'/2
        den = abs(s1) ** 2 - (s0.conjugate() * s2).real           # P''/2
        step = -num / den
        omega = omega + step
    out["last_step_hz"] = abs(step) * HZ_PER_RAD
    if not abs(step) * HZ_PER_RAD <= TOL_HZ:
        out["flag"] = NOCONV
        return out
    out["f"] = F_NOM + omega * HZ_PER_RAD
    return out


def row_time(p: float, e1: float, e2: float) -> float:
    """capture time (s) of the window centre: tau_c = p + 16*osr + (W-1)/2 in r_correct, x_c = ((tau_c - 1)(1+e2))(1+e1) raw samples"""
    tau_c = p + OFF + HALF
    return (((tau_c - 1.0) * (1.0 + e2)) * (1.0 + e1)) / FS


def fit_line(t, f):
    """f = a + b*(t - t_bar), every sum in row order: returns t_bar, a, b, rms"""
    n = len(t)
    st = sf = 0.0
    for ti, fi in zip(t, f):
        st += ti
        sf += fi
    t_bar, a = st / n, sf / n
    stt = stf = 0.0
    for ti, fi in zip(t, f):
        dt = ti - t_bar
        stt += dt * dt
        stf += dt * (fi - a)
    b = stf / stt
    ss = 0.0
    for ti, fi in zip(t, f):
        e = (fi - a) - b * (ti - t_bar)
        ss += e * e
    return t_bar, a, b, math.sqrt(ss / n)


def carrier_fit(r_correct, pos_info, e1: float, e2: float, total_carrier_ppm: float, carrier_freq: float) -> dict:
    """Every FCCH row (type 0) of pos_info, in order: f (Hz in r_correct's frame), t (s of capture time), the row's flag; then the
    fit.  r_correct: calibrate_stream's r_final (r(j) = r_correct[j-1]); e1, e2 = sampling_ppm[0], [1] * 1e-6."""
    r = np.asarray(r_correct).reshape(-1)
    pinfo = np.asarray(pos_info, dtype=np.float64).reshape(-1, 2)
    pos = pinfo[pinfo[:, 1] == 0, 0]
    n = len(pos)
    f, t = np.full(n, np.nan), np.full(n, np.nan)
    row_flag, k = np.zeros(n, dtype=np.int64), np.zeros(n, dtype=np.int64)
    for i, p in enumerate(pos):
        if not (p == math.floor(p) and p >= 1 and p + 148 * OSR - 1 <= len(r)):       # FCCH_demod's window check
            row_flag[i] = RANGE
            continue
        j0 = int(p) - 1 + OFF
        est = tone_estimate(r[j0:j0 + W])
        row_flag[i], k[i] = est["flag"], est["k"]
        if est["flag"] == 0:
            f[i] = est["f"]
            t[i] = row_time(p, e1, e2)
    flags = 0
    for v in row_flag:
        flags |= int(v)
    used = np.isfinite(f)
    n_fit = int(used.sum())
    out = dict(f=f, t=t, row_flag=row_flag, k=k, n_fcch=n, n_fit=n_fit, flags=flags, t_mean=math.nan, freq_hz=math.nan,
               drift_hz_per_s=math.nan, rms_hz=math.nan, residual_ppm=math.nan, carrier_fit_ppm=math.nan, drift_ppm_per_s=math.nan)
    if n_fit < 3:
        out["flags"] |= FEW
        return out
    t_bar, a, b, rms = fit_line([float(v) for v in t[used]], [float(v) for v in f[used]])
    residual = 1e6 * (a - F_NOM) / carrier_freq
    out.update(t_mean=t_bar, freq_hz=a, drift_hz_per_s=b, rms_hz=rms, residual_ppm=residual,
               carrier_fit_ppm=total_ppm2(total_carrier_ppm, residual), drift_ppm_per_s=1e6 * b / carrier_freq)
    return out


def carrier_reference(cal: dict, carrier_freq: float) -> dict:
    """the record of one stream from oracle.calibrate_stream's outputs: the sentinels (pos_info == -1, r_correct == -1), then
    carrier_fit on r_final"""
    pinfo = np.asarray(cal["pos_info"], dtype=np.float64).reshape(-1, 2)
    nan = dict(n_fcch=-1, n_fit=0, t_mean=math.nan, freq_hz=math.nan, drift_hz_per_s=math.nan, rms_hz=math.nan,
               residual_ppm=math.nan, carrier_fit_ppm=math.nan, drift_ppm_per_s=math.nan, f=None, t=None, row_flag=None)
    if pinfo.size > 0 and np.all(pinfo == -1):
        return dict(nan, flags=NO_POS_INFO)
    if cal["r_final"] is None:
        return dict(nan, flags=NO_R_CORRECT)
    e1, e2 = cal["sampling_ppm"][0] * 1e-6, cal["sampling_ppm"][1] * 1e-6
    return carrier_fit(cal["r_final"], pinfo, e1, e2, cal["total_carrier_ppm"], carrier_freq)
