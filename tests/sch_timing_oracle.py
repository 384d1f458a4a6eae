"""fp64 restatement of gsmcal_calibrate_sch_timing_batch (include/gsmcal.h): sub-sample timing of every SCH burst of pos_info on
r_correct and the least-squares line through the burst times in raw-capture samples.  Test infrastructure, like oracle/: the GPU
results are compared against it and the synthetic truth checks run on it."""
from __future__ import annotations

import math

import numpy as np

OSR = 8
L = 64 * OSR                  # template samples
PRE = 42 * OSR                # training start behind the SCH row's position
LAG_LO, LAG_HI = -8 * OSR, 3 * OSR     # SCH_corr_rate_correction.m:36,45-48: 89 lags
N_LAG = LAG_HI - LAG_LO + 1

NO_POS_INFO, NO_R_CORRECT, RANGE, EDGE, FEW = 1, 2, 4, 8, 16


def parabola_delta(ym: float, y0: float, yp: float) -> float:
    """vertex offset of the parabola through (-1, ym), (0, y0), (1, yp); 0 when the three points are collinear"""
    den = ym - 2.0 * y0 + yp
    return 0.0 if den == 0.0 else 0.5 * (ym - yp) / den


def correlate(r: np.ndarray, g: int, template: np.ndarray) -> np.ndarray:
    """c(l) = |sum_{n<512} conj(t_n) r(g+l+n)|^2, l = -64..24, r 1-based (r[0] is r(1)); abs first, then square"""
    s0 = g + LAG_LO - 1
    win = np.lib.stride_tricks.sliding_window_view(r[s0:s0 + N_LAG + L - 1], L)
    return np.abs(win @ np.conj(np.asarray(template).reshape(-1))) ** 2


def fit_line(m, x):
    """b = sum (m-mean m)(x-mean x) / sum (m-mean m)^2, a = mean x - b mean m, rms of x - a - b m; every sum in order"""
    n = len(m)
    sm = sx = 0.0
    for mi, xi in zip(m, x):
        sm += mi
        sx += xi
    m_bar, x_bar = sm / n, sx / n
    sxy = smm = 0.0
    for mi, xi in zip(m, x):
        dm, dx = mi - m_bar, xi - x_bar
        sxy += dm * dx
        smm += dm * dm
    b = sxy / smm
    a = x_bar - b * m_bar
    ss = 0.0
    for mi, xi in zip(m, x):
        e = xi - a - b * mi
        ss += e * e
    return a, b, math.sqrt(ss / n)


def sch_fine_timing(r_correct, pos_info, template, osr: int, e1: float, e2: float) -> dict:
    """Every SCH row (type 1) of pos_info, in order: tau (time in r_correct, 1-based), x (raw-capture time, 0-based), l* (the lag of
    the first maximum), the row's flag (0, RANGE or EDGE) and the relative gap between its two largest |corr|^2; then the fit.
    r_correct: the stream of calibrate_stream's r_final (r(j) = r_correct[j-1]); e1, e2 = sampling_ppm[0], [1] * 1e-6."""
    assert osr == OSR
    r = np.asarray(r_correct).reshape(-1)
    pinfo = np.asarray(pos_info, dtype=np.float64).reshape(-1, 2)
    pos = pinfo[pinfo[:, 1] == 1, 0]
    n = len(pos)
    tau, x = np.full(n, np.nan), np.full(n, np.nan)
    lstar, row_flag, gap = np.full(n, -10 ** 6), np.zeros(n, dtype=np.int64), np.full(n, np.nan)
    for i, p in enumerate(pos):
        g = p + PRE
        if not (p == math.floor(p) and g + LAG_LO >= 1 and g + LAG_HI + L - 1 <= len(r)):
            row_flag[i] = RANGE
            continue
        c = correlate(r, int(g), template)
        k = int(np.argmax(c))                                   # first maximum
        srt = np.sort(c)
        gap[i] = (srt[-1] - srt[-2]) / srt[-1]
        lstar[i] = k + LAG_LO
        if k == 0 or k == N_LAG - 1:
            row_flag[i] = EDGE
            continue
        tau[i] = (g + (k + LAG_LO)) + parabola_delta(float(c[k - 1]), float(c[k]), float(c[k + 1]))
    for i in range(n):
        x[i] = ((tau[i] - 1.0) * (1.0 + e2)) * (1.0 + e1)
    flags = 0
    for f in row_flag:
        flags |= int(f)
    fit = np.isfinite(x)
    n_fit = int(fit.sum())
    out = dict(tau=tau, x=x, lstar=lstar, row_flag=row_flag, gap=gap, n_sch=n, n_fit=n_fit, flags=flags,
               t0=math.nan, fit_ppm=math.nan, rms=math.nan)
    if n_fit < 3:
        out["flags"] |= FEW
        return out
    p_first = pos[fit][0]
    a, b, rms = fit_line([float(p - p_first) for p in pos[fit]], [float(v) for v in x[fit]])
    out.update(t0=a, fit_ppm=(b - 1.0) * 1e6, rms=rms)
    return out


def timing_reference(cal: dict, template, osr: int = OSR) -> dict:
    """the record of one stream from oracle.calibrate_stream's outputs: the sentinels (pos_info == -1, r_correct == -1), then
    sch_fine_timing on r_final with e1, e2 from the stream's sampling_ppm"""
    pinfo = np.asarray(cal["pos_info"], dtype=np.float64).reshape(-1, 2)
    if pinfo.size > 0 and np.all(pinfo == -1):
        return dict(n_sch=-1, n_fit=0, flags=NO_POS_INFO, t0=math.nan, fit_ppm=math.nan, rms=math.nan, tau=None, x=None)
    if cal["r_final"] is None:
        return dict(n_sch=-1, n_fit=0, flags=NO_R_CORRECT, t0=math.nan, fit_ppm=math.nan, rms=math.nan, tau=None, x=None)
    e1, e2 = cal["sampling_ppm"][0] * 1e-6, cal["sampling_ppm"][1] * 1e-6
    return sch_fine_timing(cal["r_final"], pinfo, template, osr, e1, e2)
