"""fp64 restatement of gsmcal_calibrate_cell_batch (include/gsmcal.h): the carrier fit of carrier_fit_oracle, then SCH_demod of every SCH row
of pos_info on r_correct with the fitted residual removed from its equaliser window, then the SCH decoding of sch_decode_oracle.  The
FDE / MLSE body is oracle.SCH_demod's own, run on the rotated window.  Test infrastructure, like oracle/."""
from __future__ import annotations

import math

import numpy as np

import carrier_fit_oracle as CF
import gsmcal_oracle as oracle
import sch_decode_oracle as S

OSR = 8
FS = CF.FS
F_NOM = CF.F_NOM
EX = 8                                # SCH_demod.m's ex_len: the window starts 8 symbols before the burst
N = 194 * OSR                         # the equaliser window, SCH_demod.m:79-81
UNCORRECTED = 16                      # decode-record flag: no carrier fit, df = 0


def row_time(p: float, e1: float, e2: float) -> float:
    """capture time (s) of the training centre r(p + 74*osr), mapped as the carrier fit's step 5"""
    return (((p + 74 * OSR - 1.0) * (1.0 + e2)) * (1.0 + e1)) / FS


def row_residual(p: float, e1: float, e2: float, carrier: dict) -> float:
    """df_i (Hz, r_correct's frame) of the SCH row at p: the fitted line at its training centre"""
    return (carrier["freq_hz"] - F_NOM) + carrier["drift_hz_per_s"] * (row_time(p, e1, e2) - carrier["t_mean"])


def demod_window(x, template, df: float) -> dict:
    """SCH_demod.m:83-110 on one equaliser window x (194*osr samples of r_correct from p - 8*osr) after exp(-i*2*pi*df*n/fs)"""
    x = np.asarray(x, dtype=np.complex128).reshape(-1)
    assert len(x) == N
    if df != 0.0:
        x = x * np.exp(-1j * 2.0 * np.pi * df * np.arange(N) / FS)
    got = oracle.SCH_demod(x, np.array([[EX * OSR + 1.0, 1.0]]), template, OSR)       # the window is the whole stream: sp = 1
    return {k: v[0] for k, v in got.items()}


def cell_sync(r_correct, pos_info, e1: float, e2: float, carrier: dict, template) -> dict:
    """Every SCH row (type 1) of pos_info, in order: df, demod_bits, bits_to_decoder, corr_val, sch_ok; then the decode.  carrier: the
    stream's carrier-fit record (carrier_fit_oracle.carrier_fit's keys, or the GPU's); without a fit (CARRIER_FEW) every df is 0 and
    reported as NaN, and the record gets UNCORRECTED."""
    r = np.asarray(r_correct).reshape(-1)
    pinfo = np.asarray(pos_info, dtype=np.float64).reshape(-1, 2)
    pos = pinfo[pinfo[:, 1] == 1, 0]
    n = len(pos)
    fitted = not (carrier["flags"] & CF.FEW)
    out = dict(df=np.full(n, np.nan), demod_bits=np.zeros((n, 148), dtype=np.int64), bits_to_decoder=np.zeros((n, 148), dtype=np.int64),
               corr_val=np.zeros((n, 85)), sch_ok=np.zeros(n, dtype=bool))
    for i, p in enumerate(pos):
        df = row_residual(p, e1, e2, carrier) if fitted else 0.0
        if fitted:
            out["df"][i] = df
        sp = int(p) - EX * OSR
        if not (p == math.floor(p) and sp >= 1 and sp + N - 1 <= len(r)):
            continue
        got = demod_window(r[sp - 1:sp - 1 + N], template, df)
        out["sch_ok"][i] = True
        for k in ("demod_bits", "bits_to_decoder", "corr_val"):
            out[k][i] = got[k]
    rec, rows = S.decode_stream(out["demod_bits"], out["corr_val"], out["sch_ok"], pos, OSR)
    if not fitted:
        rec["flags"] |= UNCORRECTED
    return dict(out, rec=rec, rows=rows)


def cell_reference(cal: dict, carrier_freq: float, template) -> dict:
    """one stream from oracle.calibrate_stream's outputs: the carrier fit, then cell_sync on r_final; the sentinels (pos_info == -1,
    r_correct == -1) as sch_decode_oracle.decode_stream gives them"""
    carrier = CF.carrier_reference(cal, carrier_freq)
    if carrier["flags"] & (CF.NO_POS_INFO | CF.NO_R_CORRECT):
        rec, rows = S.decode_stream(None, None, None, None, OSR, carrier["flags"])
        return dict(carrier=carrier, rec=rec, rows=rows, df=None)
    e1, e2 = cal["sampling_ppm"][0] * 1e-6, cal["sampling_ppm"][1] * 1e-6
    return dict(cell_sync(cal["r_final"], cal["pos_info"], e1, e2, carrier, template), carrier=carrier)
