"""Synthetic GSM C0 (BCCH carrier) capture generator - the stand-in for rtl_tcp's uint8 I,Q stream.

The reference has no recorded captures (SURVEY.md section 4), so tests and bench.py use this seeded
generator: repeating 51-multiframe with FCCH in TS0 of frames 0,10,20,30,40 and SCH in frames
1,11,21,31,41 (64-bit extended training sequence of gsm_SCH_training_sequence_gen.m:17-19 at bit 42),
random bursts elsewhere, GMSK BT 0.3 / L=4 / h=0.5 at 8 samples per symbol and 1250 samples per slot,
sampling-clock error applied by exact re-timing of the continuous phase, carrier error, AWGN, DC, and
round+clip to uint8 around 127.5 - the wire format `fread(tcp, n, 'uint8')` sees (gsm_sync_demod.m:96).

Written with torch so the same code runs on the CPU (tests, fixtures) and on the GPU (bench.py, where
1024 x 21.7 M samples would take far too long on the host).  torch here is data plumbing only.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np
import torch

SYMBOL_RATE = (1625.0 / 6.0) * 1e3
SLOT = 1250                 # samples per slot at 8x
SYM_PER_SLOT = 156          # impulses per slot (148 burst bits + 8 guard bits; the quarter bit is 2 samples of hold)
FRAME = 8 * SLOT
MULTIFRAME = 51 * FRAME

SCH_TRAINING_BITS = (1, 0, 1, 1, 1, 0, 0, 1, 0, 1, 1, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 1, 0,
                     0, 0, 0, 0, 0, 1, 1, 1, 1, 0, 0, 1, 0, 1, 1, 0, 1, 0, 1, 0, 0, 0,
                     1, 0, 1, 0, 1, 1, 1, 0, 1, 1, 0, 0, 0, 0, 1, 1, 0, 1, 1)

_SIGMA = math.sqrt(math.log(2.0)) / (2.0 * math.pi * 0.3)


def _big_f(u: torch.Tensor) -> torch.Tensor:
    return u * 0.5 * torch.erfc(-u / math.sqrt(2.0)) + torch.exp(-0.5 * u * u) / math.sqrt(2.0 * math.pi)


def _big_g(t: torch.Tensor) -> torch.Tensor:
    return (_SIGMA / 2.0) * (_big_f((t + 0.5) / _SIGMA) - _big_f((t - 0.5) / _SIGMA))


def gmsk_q(tau: torch.Tensor) -> torch.Tensor:
    """Integrated, L=4-truncated GMSK frequency pulse; tau in symbols; q(<=0)=0, q(>=4)=1."""
    tau = tau.clamp(0.0, 4.0)
    c = torch.tensor([-2.0, 2.0], dtype=tau.dtype, device=tau.device)
    g = _big_g(c)
    return (_big_g(tau - 2.0) - g[0]) / (g[1] - g[0])


@dataclass
class StreamSpec:
    """Impairments of one synthetic dongle stream."""
    seed: int
    n_samples: int
    sampling_ppm: float = 0.0       # receiver clock fast by this much -> burst spacing grows by (1+e)
    carrier_ppm: float = 0.0        # of carrier_freq
    carrier_freq: float = 957.4e6   # gsm_sync_demod.m:14
    snr_db: float = 20.0
    phase0: float = 0.0
    start_offset: float = 0.0       # nominal samples into the multiframe at receiver sample 0
    amplitude: float = 40.0
    dc: complex = 127.4 + 127.6j
    drop_fcch: tuple = field(default_factory=tuple)   # indices (0-based, in order of appearance) of FCCH bursts to replace by data
    noise_only: bool = False
    tsc: int | None = None          # normal training sequence code (0..7) put at bits 61..86 of every normal burst; None = random bits
    bsic: int | None = None         # 0..63: every SCH burst carries the coded (BSIC, FN) of TS 45.003 4.7; None = random coded bits
    fn0: int = 0                    # TDMA frame number of slot 0's frame (a multiple of 51, below FN_MOD)


def random_spec(seed: int, n_samples: int, carrier_freq: float = 957.4e6) -> StreamSpec:
    """The impairment distribution of SURVEY.md section 8(d), narrowed to the range the reference chain locks on."""
    rng = np.random.default_rng(seed)
    return StreamSpec(seed=seed, n_samples=n_samples,
                      sampling_ppm=float(rng.uniform(-40.0, 35.0)),
                      carrier_ppm=float(rng.uniform(-25.0, 25.0)),
                      carrier_freq=carrier_freq,
                      snr_db=float(rng.uniform(15.0, 25.0)),
                      phase0=float(rng.uniform(0.0, 2.0 * math.pi)),
                      start_offset=float(rng.integers(0, MULTIFRAME)))


NORMAL_TRAINING_BITS = (      # gsm_normal_training_sequence_gen.m:17-24
    (0, 0, 1, 0, 0, 1, 0, 1, 1, 1, 0, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 1, 0, 1, 1, 1),
    (0, 0, 1, 0, 1, 1, 0, 1, 1, 1, 0, 1, 1, 1, 1, 0, 0, 0, 1, 0, 1, 1, 0, 1, 1, 1),
    (0, 1, 0, 0, 0, 0, 1, 1, 1, 0, 1, 1, 1, 0, 1, 0, 0, 1, 0, 0, 0, 0, 1, 1, 1, 0),
    (0, 1, 0, 0, 0, 1, 1, 1, 1, 0, 1, 1, 0, 1, 0, 0, 0, 1, 0, 0, 0, 1, 1, 1, 1, 0),
    (0, 0, 0, 1, 1, 0, 1, 0, 1, 1, 1, 0, 0, 1, 0, 0, 0, 0, 0, 1, 1, 0, 1, 0, 1, 1),
    (0, 1, 0, 0, 1, 1, 1, 0, 1, 0, 1, 1, 0, 0, 0, 0, 0, 1, 0, 0, 1, 1, 1, 0, 1, 0),
    (1, 0, 1, 0, 0, 1, 1, 1, 1, 1, 0, 1, 1, 0, 0, 0, 1, 0, 1, 0, 0, 1, 1, 1, 1, 1),
    (1, 1, 1, 0, 1, 1, 1, 1, 0, 0, 0, 1, 0, 0, 1, 0, 1, 1, 1, 0, 1, 1, 1, 1, 0, 0))


FN_MOD = 26 * 51 * 2048     # TDMA frames in a hyperframe (TS 45.002 3.3.2.2)


def sch_fields(fn: int):
    """(T1, T2, T3') of an SCH frame number (FN mod 51 in 1, 11, 21, 31, 41)"""
    t3 = fn % 51
    assert t3 % 10 == 1 and t3 <= 41, "not an SCH frame"
    return fn // 1326, fn % 26, (t3 - 1) // 10


def sch_encode(bsic: int, fn: int) -> np.ndarray:
    """The 78 coded bits of an SCH burst (TS 45.003 4.7): the 25 information bits packed as TS 44.018 9.1.30 (OsmocomBB's order),
    the 10 parity bits that leave the remainder 1 + D + ... + D^9 modulo D^10 + D^8 + D^6 + D^5 + D^4 + D^2 + 1, four tail bits, and the
    rate-1/2 code G0 = 1 + D^3 + D^4, G1 = 1 + D + D^3 + D^4.  Parity with a live cell is unverified (no recorded capture)."""
    t1, t2, t3p = sch_fields(fn)
    bit = lambda v, i: (v >> i) & 1                                      # noqa: E731
    d = [bit(t1, 9), bit(t1, 10)] + [bit(bsic, i) for i in range(6)] + [bit(t1, i) for i in range(1, 9)]
    d += [bit(t3p, 1), bit(t3p, 2)] + [bit(t2, i) for i in range(5)] + [bit(t1, 0), bit(t3p, 0)]
    rem = 0
    for b in d + [0] * 10:                                              # d(D) * D^10 mod g(D)
        rem = (rem << 1) | b
        if rem & 0x400:
            rem ^= 0x575
    u = d + [((rem ^ 0x3FF) >> (9 - i)) & 1 for i in range(10)] + [0, 0, 0, 0]
    c = []
    for k in range(39):
        v = lambda j: u[k - j] if k >= j else 0                         # noqa: E731
        c += [v(0) ^ v(3) ^ v(4), v(0) ^ v(1) ^ v(3) ^ v(4)]
    return np.array(c, dtype=np.int64)


def _slot_bits(n_slots: int, gen: torch.Generator, device, drop_fcch=(), tsc=None) -> torch.Tensor:
    """[n_slots, 156] bits: TS0 of frames 0/10/20/30/40 (mod 51) FCCH, 1/11/21/31/41 SCH, else random."""
    bits = torch.randint(0, 2, (n_slots, SYM_PER_SLOT), generator=gen, device=device, dtype=torch.int64)
    bits[:, 0:3] = 0
    bits[:, 145:148] = 0
    bits[:, 148:156] = 1
    if tsc is not None:
        bits[:, 61:87] = torch.tensor(NORMAL_TRAINING_BITS[int(tsc)], device=device, dtype=torch.int64)
    slot = torch.arange(n_slots, device=device)
    frame = (slot // 8) % 51
    ts0 = (slot % 8) == 0
    is_fcch = ts0 & (frame % 10 == 0) & (frame <= 40)
    is_sch = ts0 & (frame % 10 == 1) & (frame <= 41)
    fcch_slots = torch.nonzero(is_fcch).flatten()
    if len(drop_fcch):
        keep = torch.ones(len(fcch_slots), dtype=torch.bool, device=device)
        for d in drop_fcch:
            if d < len(keep):
                keep[d] = False
        fcch_slots = fcch_slots[keep]
    bits[fcch_slots, 0:148] = 0
    ts = torch.tensor(SCH_TRAINING_BITS, device=device, dtype=torch.int64)
    bits[is_sch, 42:106] = ts
    return bits


def stream_bits(spec: StreamSpec, gen: torch.Generator | None = None, device="cpu") -> torch.Tensor:
    """[n_slots, 156] burst bits of the stream (what generate_stream modulates); gen: the stream's generator, seeded here when None.
    With spec.bsic set, the coded SCH bits are written over bits 3..41 and 106..144 of every SCH burst after the random draws, so the
    generator's later draws (the noise) and every other bit are those of bsic=None."""
    dev = torch.device(device)
    if gen is None:
        gen = torch.Generator(device=dev)
        gen.manual_seed(int(spec.seed))
    inv = 1.0 / (1.0 + spec.sampling_ppm * 1e-6)
    t_end = spec.start_offset + spec.n_samples * inv
    n_slots = int(t_end // SLOT) + 3
    bits = _slot_bits(n_slots, gen, dev, spec.drop_fcch, spec.tsc)
    if spec.bsic is not None:
        assert 0 <= spec.bsic < 64 and spec.fn0 % 51 == 0 and 0 <= spec.fn0 < FN_MOD
        for s in range(0, n_slots, 8):
            if (s // 8) % 51 % 10 == 1 and (s // 8) % 51 <= 41:
                c = torch.from_numpy(sch_encode(spec.bsic, (spec.fn0 + s // 8) % FN_MOD)).to(dev)
                bits[s, 3:42] = c[:39]
                bits[s, 106:145] = c[39:]
    return bits


def true_frame_clock_start(spec: StreamSpec) -> float:
    """GSM time of receiver sample 0 in nominal 8x samples since FN 0 (the quantity gsmcal_sch_decode_result.frame_clock_start measures)"""
    return spec.fn0 * FRAME + spec.start_offset


def generate_stream(spec: StreamSpec, device="cpu", out: torch.Tensor | None = None) -> torch.Tensor:
    """Returns 2*n_samples uint8 (I,Q interleaved).  `out` may be a preallocated uint8 view to fill."""
    dev = torch.device(device)
    n = spec.n_samples
    gen = torch.Generator(device=dev)
    gen.manual_seed(int(spec.seed))
    f64 = torch.float64
    inv = 1.0 / (1.0 + spec.sampling_ppm * 1e-6)
    bits = stream_bits(spec, gen, dev).flatten()
    prev = torch.cat([torch.ones(1, dtype=torch.int64, device=dev), bits[:-1]])
    a = (1 - 2 * (bits ^ prev)).to(torch.int64)                 # +1 where a bit equals its predecessor
    psum = torch.cumsum(a, 0)                                   # P[m] = sum_{i<=m} a_i

    result = out if out is not None else torch.empty(2 * n, dtype=torch.uint8, device=dev)
    noise_sigma = spec.amplitude / math.sqrt(2.0) * 10.0 ** (-spec.snr_db / 20.0)
    w_off = 2.0 * math.pi * (spec.carrier_ppm * 1e-6 * spec.carrier_freq) / (SYMBOL_RATE * 8)
    chunk = 1 << 22
    for c0 in range(0, n, chunk):
        c1 = min(n, c0 + chunk)
        idx = torch.arange(c0, c1, device=dev, dtype=f64)
        t = spec.start_offset + idx * inv                        # nominal time in samples
        slot = torch.floor(t / SLOT)
        w = t - slot * SLOT
        k = torch.clamp(torch.floor(w / 8.0), max=SYM_PER_SLOT - 1)
        g = (slot * SYM_PER_SLOT + k).to(torch.int64)
        gm4 = g - 4
        base = torch.where(gm4 >= 0, psum[gm4.clamp(min=0)], torch.zeros_like(gm4))
        phase = (base % 4).to(f64)                               # whole quarter turns, exact
        for j in range(4):
            gj = g - j
            valid = gj >= 0
            gjc = gj.clamp(min=0)
            tj = (gjc // SYM_PER_SLOT).to(f64) * SLOT + (gjc % SYM_PER_SLOT).to(f64) * 8.0
            phase = phase + torch.where(valid, a[gjc].to(f64) * gmsk_q((t - tj) / 8.0), torch.zeros_like(t))
        theta = (math.pi / 2.0) * phase + (idx * w_off + spec.phase0)
        amp = 0.0 if spec.noise_only else spec.amplitude
        re = amp * torch.cos(theta) + noise_sigma * torch.randn(c1 - c0, generator=gen, device=dev, dtype=f64)
        im = amp * torch.sin(theta) + noise_sigma * torch.randn(c1 - c0, generator=gen, device=dev, dtype=f64)
        re = torch.clamp(torch.round(re + spec.dc.real), 0, 255).to(torch.uint8)
        im = torch.clamp(torch.round(im + spec.dc.imag), 0, 255).to(torch.uint8)
        result[2 * c0:2 * c1:2] = re
        result[2 * c0 + 1:2 * c1:2] = im
    return result


def generate_batch(specs, device="cpu") -> torch.Tensor:
    """[D, 2N] uint8, one row per stream (== one column of the reference's 2N x D matrix)."""
    n = specs[0].n_samples
    out = torch.empty((len(specs), 2 * n), dtype=torch.uint8, device=device)
    for d, sp in enumerate(specs):
        assert sp.n_samples == n
        generate_stream(sp, device, out[d])
    return out


def true_fcch_starts(spec: StreamSpec) -> np.ndarray:
    """1-based receiver sample index of every FCCH burst start inside the capture (sanity checks only)."""
    scale = 1.0 + spec.sampling_ppm * 1e-6
    res = []
    t_end = spec.start_offset + spec.n_samples / scale
    mf0 = int(spec.start_offset // MULTIFRAME)
    m = mf0
    while m * MULTIFRAME < t_end:
        for f in (0, 10, 20, 30, 40):
            t = m * MULTIFRAME + f * FRAME
            nidx = (t - spec.start_offset) * scale
            if 0 <= nidx < spec.n_samples:
                res.append(nidx + 1)
        m += 1
    return np.array(res)
