"""NumPy restatement of the BCCH decoding of gsmcal_calibrate_sysinfo_batch (definition: include/gsmcal.h), written independently of
the kernels and of the synthetic generator's encoder: the block list, each burst's lag search and one-tap equaliser in front of the
oracle's GMSK MLSE, the burst bits, the deinterleaver, the 228-step Viterbi with its tie rule, the Fire check, the payload, the SI mask
and the SI3 vote.  It runs behind cell_sync_oracle (the carrier fit and the SCH decoding).  Test infrastructure, like oracle/."""
from __future__ import annotations

import math

import numpy as np

import carrier_fit_oracle as CF
import cell_sync_oracle as CS
import gsmcal_oracle as oracle

OSR = 8
FS = CF.FS
F = 1250 * OSR
N = 194 * OSR
NY = N + 159
LAG0, NLAG = 64, 160
FN_MOD = 2715648
NO_POS_INFO, NO_R_CORRECT, NO_CELL, UNCORRECTED, NO_SI3, SI3_DISAGREE = 1, 2, 4, 8, 16, 32
ROW_RANGE, ROW_EDGE = 1, 2
BLK_FN, BLK_ROW, BLK_FIRE, BLK_SHORT = 1, 2, 4, 8
HAS = {0x19: 1, 0x1A: 2, 0x02: 4, 0x03: 8, 0x07: 16, 0x1B: 32, 0x1C: 64, 0x00: 128}
HAS_OTHER = 256
G40 = [40, 26, 23, 17, 3, 0]                           # exponents of the Fire generator
NO_LAG = -128


def blocks_of(pos_info):
    """[rows of block b]: the type-2 rows directly behind each type-1 row, pos_info order (a type-1 row with none is no block)"""
    out, cur, after_sch = [], None, False
    for p, t in np.asarray(pos_info, dtype=np.float64).reshape(-1, 2):
        if t == 2 and after_sch:
            if cur is None:
                cur = []
                out.append(cur)
            if len(cur) < 4:
                cur.append(float(p))
            continue
        after_sch, cur = t == 1, None
    return out


def burst(r, p, df, t, tsc_bits):
    """one BCCH row at p: (lag, row flag, steal (b60, b87), i(0..113) or None); t the 208-sample training waveform of the TSC"""
    s0 = p - 128                                       # g - 64 - 69*osr, g = p + 61*osr
    if not (p == math.floor(p) and s0 >= 1 and s0 + NY - 1 <= len(r)):
        return NO_LAG, ROW_RANGE, (0, 0), None
    s0 = int(s0)
    y = r[s0 - 1:s0 - 1 + NY] * np.exp(-1j * 2.0 * np.pi * df * np.arange(NY) / FS)
    c = np.array([np.dot(np.conj(t), y[li + 69 * OSR:li + 69 * OSR + 208]) for li in range(NLAG)])
    pw = c.real ** 2 + c.imag ** 2
    li = int(np.argmax(pw))                            # first maximum
    lag = li - LAG0
    flag = ROW_EDGE if lag in (-LAG0, NLAG - 1 - LAG0) else 0
    h = c[li] / float(np.sum(t.real ** 2 + t.imag ** 2))
    w = np.conj(h) / (h.real ** 2 + h.imag ** 2)
    x = y[li:li + N] * w
    m = oracle.gmsk_viterbi_demod(x, OSR, 30)[38:186]
    b = {61 + j: int(tsc_bits[j]) for j in range(26)}
    for i in range(60, -1, -1):
        b[i] = b[i + 1] ^ (1 - int(m[i + 1]))
    for i in range(87, 148):
        b[i] = b[i - 1] ^ (1 - int(m[i]))
    ib = np.array([b[i] for i in range(3, 60)] + [b[i] for i in range(88, 145)], dtype=np.int64)
    return lag, flag, (b[60], b[87]), ib


def deinterleave(ib):
    """c(k) = i_(k mod 4)(2*((49k) mod 57) + ((k mod 8) div 4)), k = 0..455; ib [4][114]"""
    return np.array([ib[k % 4][2 * ((49 * k) % 57) + ((k % 8) // 4)] for k in range(456)], dtype=np.int64)


def viterbi(c):
    """(u(0..227), hamming): sch_decode_oracle's decoder over 228 steps (states = the last four inputs, a tie keeps the predecessor whose
    dropped bit is 0, from and back to the all-zero state)"""
    inf = 10 ** 6
    metric = [0] + [inf] * 15                          # state s = u(k) | u(k-1) << 1 | u(k-2) << 2 | u(k-3) << 3
    hist = []
    for k in range(228):
        c0, c1 = int(c[2 * k]), int(c[2 * k + 1])
        nm, dec = [0] * 16, [0] * 16
        for s in range(16):
            u, prev = s & 1, s >> 1
            best = None
            for dropped in (0, 1):
                pv = prev | (dropped << 3)
                u1, u3, u4 = pv & 1, (pv >> 2) & 1, dropped
                cand = metric[pv] + int((u ^ u3 ^ u4) != c0) + int((u ^ u1 ^ u3 ^ u4) != c1)
                if best is None or cand < best:
                    best, dec[s] = cand, dropped
            nm[s] = best
        metric = nm
        hist.append(dec)
    u, s = [0] * 228, 0
    for k in range(227, -1, -1):
        u[k] = s & 1
        s = (s >> 1) | (hist[k][s] << 3)
    return np.array(u, dtype=np.int64), metric[0]


def fire_ok(u):
    """d(0)D^223 + ... + p(39) divided by g(D) leaves 1 + D + ... + D^39"""
    r = [int(x) for x in u[:224]]
    for i in range(184):
        if r[i]:
            for e in G40:
                r[i + 40 - e] ^= 1
    return all(r[184:224])


def payload(u):
    return bytes(sum(int(u[8 * m + q]) << q for q in range(8)) for m in range(23))


def si3_fields(pay):
    """(mcc, mnc, mnc_digits, lac, ci) of an SI3 payload (octets 3..9; nibbles as they are)"""
    ci = (pay[3] << 8) | pay[4]
    mcc = 100 * (pay[5] & 15) + 10 * (pay[5] >> 4) + (pay[6] & 15)
    d3, m1, m2 = pay[6] >> 4, pay[7] & 15, pay[7] >> 4
    mnc, nd = (10 * m1 + m2, 2) if d3 == 15 else (100 * m1 + 10 * m2 + d3, 3)
    return mcc, mnc, nd, (pay[8] << 8) | pay[9], ci


def decode_block(ib):
    """(hamming, fire passed, payload) of a block's four rows of coded bits"""
    u, ham = viterbi(deinterleave(ib))
    return ham, fire_ok(u), payload(u[:184])


def sysinfo_stream(r, pos_info, e1, e2, carrier, rec, nts):
    """the record, per-block and per-row outputs of one stream whose SCH decoding record is rec (cell_sync_oracle's) and whose carrier
    record is carrier; nts the (26*osr) x 8 normal training waveforms"""
    r = np.asarray(r).reshape(-1)
    blocks = blocks_of(pos_info)
    n = len(blocks)
    cell = rec["bsic"] >= 0
    fitted = not (carrier["flags"] & CF.FEW)
    out = dict(n_blocks=n, n_fire_ok=0, n_si3=0, n_si3_agree=0, flags=0, si_mask=0, mcc=-1, mnc=-1, mnc_digits=-1, lac=-1, ci=-1)
    blk = dict(fn=np.full(n, -1, dtype=np.int64), tc=np.full(n, 255, dtype=np.int64), block_flags=np.zeros(n, dtype=np.int64),
               hamming=np.zeros(n, dtype=np.int64), payload=np.zeros((n, 23), dtype=np.uint8))
    rows = dict(lag=np.full((n, 4), NO_LAG, dtype=np.int64), row_flags=np.zeros((n, 4), dtype=np.int64), steal=np.zeros((n, 4), dtype=np.int64))
    if not cell:
        out["flags"] |= NO_CELL
    if not fitted:
        out["flags"] |= UNCORRECTED
    pinfo = np.asarray(pos_info, dtype=np.float64).reshape(-1, 2)
    p_first = pinfo[pinfo[:, 1] == 1, 0][0] if cell else 0.0
    si3 = []
    for b, rws in enumerate(blocks):
        if not cell:
            continue
        tsc = rec["bsic"] & 7
        t, tb = np.asarray(nts)[:, tsc], oracle.NORMAL_TRAINING_BITS[tsc]
        fn = (rec["fn_first"] + int(rws[0] - p_first) // F) % FN_MOD
        blk["fn"][b], blk["tc"][b] = fn, (fn // 51) % 8
        fl = (BLK_SHORT if len(rws) < 4 else 0) | (BLK_FN if fn % 51 != 2 else 0)
        ib = []
        for k, p in enumerate(rws):
            df = CS.row_residual(p, e1, e2, carrier) if fitted else 0.0
            lag, rf, st, bits = burst(r, p, df, t, tb)
            rows["lag"][b, k], rows["row_flags"][b, k], rows["steal"][b, k] = lag, rf, st[0] | (st[1] << 1)
            fl |= BLK_ROW if rf else 0
            ib.append(bits)
        if not fl:
            ham, ok, pay = decode_block(ib)
            blk["hamming"][b] = ham
            blk["payload"][b] = np.frombuffer(pay, dtype=np.uint8)
            if not ok:
                fl |= BLK_FIRE
            else:
                out["n_fire_ok"] += 1
                bit = HAS.get(pay[2], HAS_OTHER) if pay[1] == 0x06 else HAS_OTHER
                out["si_mask"] |= bit
                if bit == 32:
                    si3.append((b, pay[3:10]))
        blk["block_flags"][b] = fl
    out["n_si3"] = len(si3)
    if not si3:
        out["flags"] |= NO_SI3
    else:
        votes = {}
        for b, key in si3:
            cnt, first = votes.get(key, (0, b))
            votes[key] = (cnt + 1, first)
        key, (cnt, _) = max(votes.items(), key=lambda kv: (kv[1][0], -kv[1][1]))
        out["n_si3_agree"] = cnt
        if cnt < len(si3):
            out["flags"] |= SI3_DISAGREE
        out["mcc"], out["mnc"], out["mnc_digits"], out["lac"], out["ci"] = si3_fields(bytes(3) + key)
    return out, blk, rows


def sysinfo_reference(cal: dict, carrier_freq: float, template, nts) -> dict:
    """one stream from oracle.calibrate_stream's outputs: cell_sync_oracle's carrier fit and SCH decoding, then the BCCH decoding on
    r_final; the sentinels as the decoding call gives them (n_blocks = -1)"""
    cs = CS.cell_reference(cal, carrier_freq, template)
    if cs["rows"] is None:
        flags = NO_POS_INFO if cs["rec"]["flags"] & 1 else NO_R_CORRECT
        rec = dict(n_blocks=-1, n_fire_ok=0, n_si3=0, n_si3_agree=0, flags=flags, si_mask=0, mcc=-1, mnc=-1, mnc_digits=-1, lac=-1, ci=-1)
        return dict(cs, si=rec, blocks=None, bcch_rows=None)
    e1, e2 = cal["sampling_ppm"][0] * 1e-6, cal["sampling_ppm"][1] * 1e-6
    si, blk, rows = sysinfo_stream(cal["r_final"], cal["pos_info"], e1, e2, cs["carrier"], cs["rec"], nts)
    return dict(cs, si=si, blocks=blk, bcch_rows=rows)
