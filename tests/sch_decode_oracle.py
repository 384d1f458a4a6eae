"""NumPy restatement of the SCH channel decoding of gsmcal_calibrate_sch_decode_batch (definition: include/gsmcal.h), written
independently of the kernel and of the synthetic generator's encoder: burst bits from the demodulated symbols, the 16-state
hard-decision Viterbi with its tie rule, the CRC, the fields, the per-stream vote and the frame clock."""
import math

import numpy as np

import gsmcal_oracle as oracle

WINDOW, ALIGN, CRC, FIELD = 1, 2, 4, 8                  # row flags
NO_POS_INFO, NO_R_CORRECT, NONE, DISAGREE = 1, 2, 4, 8  # stream flags
FN_MOD = 2715648
G = (1, 0, 1, 0, 1, 1, 1, 0, 1, 0, 1)                   # g(D) coefficients of D^10 .. D^0
T = np.asarray(oracle.SCH_TRAINING_BITS, dtype=np.int64)


def coded_bits(m, k):
    """the 78 coded bits e of a burst whose 148 demodulated symbols are m (m_i = 1 where b_i == b_(i-1)), training at k"""
    m = np.asarray(m, dtype=np.int64)
    b = {k + j: int(T[j]) for j in range(64)}
    for i in range(k - 1, k - 40, -1):
        b[i] = b[i + 1] ^ (1 - int(m[i + 1]))
    for i in range(k + 64, k + 103):
        b[i] = b[i - 1] ^ (1 - int(m[i]))
    return np.array([b[i] for i in range(k - 39, k)] + [b[i] for i in range(k + 64, k + 103)], dtype=np.int64)


def conv_encode(u):
    """c(2k) = u(k)+u(k-3)+u(k-4), c(2k+1) = u(k)+u(k-1)+u(k-3)+u(k-4) (mod 2), k = 0..38"""
    u = list(u)
    at = lambda i: u[i] if i >= 0 else 0               # noqa: E731
    out = []
    for k in range(len(u)):
        out += [at(k) ^ at(k - 3) ^ at(k - 4), at(k) ^ at(k - 1) ^ at(k - 3) ^ at(k - 4)]
    return np.array(out, dtype=np.int64)


def viterbi(e):
    """(u(0..38), hamming): states are the last four inputs (u(k), u(k-1), u(k-2), u(k-3)); a state keeps the predecessor with the
    smaller metric, on a tie the one whose dropped (oldest) bit is 0; start and end in the all-zero state"""
    e = np.asarray(e, dtype=np.int64)
    inf = 10 ** 6
    metric = {s: (0 if s == (0, 0, 0, 0) else inf) for s in _states()}
    path = {s: [] for s in _states()}
    for k in range(39):
        nm, np_ = {}, {}
        for s in _states():
            u = s[0]
            best = None
            for dropped in (0, 1):
                prev = s[1:] + (dropped,)
                c0 = u ^ prev[2] ^ prev[3]
                c1 = u ^ prev[0] ^ prev[2] ^ prev[3]
                cand = metric[prev] + int(c0 != e[2 * k]) + int(c1 != e[2 * k + 1])
                if best is None or cand < best:
                    best, bp = cand, prev
            nm[s], np_[s] = best, path[bp] + [u]
        metric, path = nm, np_
    return np.array(path[(0, 0, 0, 0)], dtype=np.int64), metric[(0, 0, 0, 0)]


def _states():
    return [((s >> 3) & 1, (s >> 2) & 1, (s >> 1) & 1, s & 1) for s in range(16)]


def crc_ok(u):
    """d(0)D^34 + ... + p(9) divided by g(D) leaves 1 + D + ... + D^9"""
    r = [int(x) for x in u[:35]]
    for i in range(25):
        if r[i]:
            for j in range(11):
                r[i + j] ^= G[j]
    return all(r[25:35])


def parity(d):
    """the p(0..9) that make crc_ok(d + p) true"""
    r = [int(x) for x in d] + [0] * 10
    for i in range(25):
        if r[i]:
            for j in range(11):
                r[i + j] ^= G[j]
    return [1 - x for x in r[25:]]


def pack(bsic, t1, t2, t3p):
    """d(0..24), TS 44.018 9.1.30 in OsmocomBB's order"""
    b = lambda v, i: (v >> i) & 1                      # noqa: E731
    return ([b(t1, 9), b(t1, 10)] + [b(bsic, i) for i in range(6)] + [b(t1, i) for i in range(1, 9)] + [b(t3p, 1), b(t3p, 2)]
            + [b(t2, i) for i in range(5)] + [b(t1, 0), b(t3p, 0)])


def unpack(d):
    d = [int(x) for x in d]
    bsic = sum(d[2 + i] << i for i in range(6))
    t1 = (d[0] << 9) | (d[1] << 10) | sum(d[8 + i] << (1 + i) for i in range(8)) | d[23]
    t3p = (d[16] << 1) | (d[17] << 2) | d[24]
    t2 = sum(d[18 + i] << i for i in range(5))
    return bsic, t1, t2, t3p


def fn_of(t1, t2, t3p):
    t3 = 10 * t3p + 1
    return 51 * ((t3 - t2) % 26) + t3 + 1326 * t1


def fields_of(fn):
    return fn // 1326, fn % 26, ((fn % 51) - 1) // 10


def encode(bsic, fn):
    d = pack(bsic, *fields_of(fn))
    return conv_encode(d + parity(d) + [0, 0, 0, 0])


def decode_row(m, corr, ok):
    """(fn, bsic, hamming, row_flags) of one SCH row"""
    if not ok:
        return -1, -1, 0, WINDOW
    k = int(np.argmax(np.asarray(corr)))
    if k < 39 or k > 45:
        return -1, -1, 0, ALIGN
    u, ham = viterbi(coded_bits(m, k))
    if not crc_ok(u):
        return -1, -1, ham, CRC
    bsic, t1, t2, t3p = unpack(u[:25])
    if t2 > 25 or t3p > 4:
        return -1, -1, ham, FIELD
    return fn_of(t1, t2, t3p), bsic, ham, 0


def decode_stream(demod_bits, corr_val, sch_ok, sch_pos, osr=8, demod_flags=0):
    """the per-stream record and the per-row outputs; demod_bits [n x 148], corr_val [n x 85], sch_ok [n], sch_pos [n]
    (None when SCH_demod did not run: demod_flags NO_POS_INFO / NO_R_CORRECT)"""
    rec = dict(n_sch=-1, n_crc_ok=0, n_agree=0, flags=0, bsic=-1, fn_first=-1, frame_clock_start=math.nan)
    if demod_flags & (NO_POS_INFO | NO_R_CORRECT):
        rec["flags"] = NO_POS_INFO if demod_flags & NO_POS_INFO else NO_R_CORRECT
        return rec, None
    n = len(sch_ok)
    rows = [decode_row(demod_bits[i], corr_val[i], bool(sch_ok[i])) for i in range(n)]
    fn = np.array([r[0] for r in rows], dtype=np.int64)
    rec["n_sch"] = n
    frame = 1250 * osr
    votes = {}
    for i, r in enumerate(rows):
        if r[3] == 0:
            f = (sch_pos[i] - sch_pos[0]) / frame
            assert f == int(f)
            key = ((int(r[0]) - int(f)) % FN_MOD, int(r[1]))
            cnt, first = votes.get(key, (0, i))
            votes[key] = (cnt + 1, first)
    rec["n_crc_ok"] = sum(v[0] for v in votes.values())
    if not votes:
        rec["flags"] = NONE
    else:
        key, (cnt, _) = max(votes.items(), key=lambda kv: (kv[1][0], -kv[1][1]))
        rec.update(n_agree=cnt, fn_first=key[0], bsic=key[1],
                   frame_clock_start=float((key[0] * frame - (int(sch_pos[0]) - 1)) % (FN_MOD * frame)))
        if cnt < rec["n_crc_ok"]:
            rec["flags"] = DISAGREE
    per_row = dict(fn=fn, bsic=np.array([r[1] for r in rows], dtype=np.int64), hamming=np.array([r[2] for r in rows], dtype=np.int64),
                   row_flags=np.array([r[3] for r in rows], dtype=np.int64))
    return rec, per_row


def decode_demod(item, osr=8):
    """decode_stream on what calibrate_demod_batch (or the oracle's sync_demod_stream) returns for one stream"""
    s = item["sch"]
    if s is None:
        return decode_stream(None, None, None, None, osr, item["demod_flags"])
    pinfo = np.asarray(item["pos_info"]).reshape(-1, 2)
    pos = pinfo[pinfo[:, 1] == 1, 0]
    return decode_stream(s["demod_bits"], s["corr_val"], s["sch_ok"], pos, osr, item["demod_flags"])
