"""sch_corr_kernel's fp32 screen (osr 8): every lag is correlated in fp32, the lags that cannot hold the maximum are ruled out with the
bound eps of DESIGN.md section 4, and the few that can are evaluated in fp64 in the tiled correlation's operation order.
CPU: a NumPy emulation of the screen in the kernel's order on random and adversarial windows, |screen - fp64| <= eps for every lag.
GPU: the screen (debug key 24 = 0) against the fp64 correlation of every lag (= 1) and the forced fallback (= 2): identical outputs on
the captures, on the Appendix-A SCH paths, on a noise-only stream, on a planted near-tie and through the drop-in."""
import math
import os
import re

import numpy as np
import pytest

import gsmcal_oracle as oracle
from gsmcal import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KERNELS = os.path.join(ROOT, "multi-rtl-sdr-calibration_b200", "csrc", "gsmcal_kernels.cuh")
FS = oracle.SYMBOL_RATE * 8
CARRIER = 957.4e6
N_SYNC = 1020000
L, N_LAG, N_SMP, NSL = 512, 89, 600, 16
U = 2.0 ** -24


def _kernel_const(name):
    m = re.search(r"#define\s+%s\s+([0-9.eE+-]+)" % name, open(KERNELS).read())
    return float(m.group(1))


EPS_K, EPS_ABS, E_MAX = _kernel_const("SCH_EPS_K"), _kernel_const("SCH_EPS_ABS"), _kernel_const("SCH_E_MAX")


# ---- CPU: the screen's bound -----------------------------------------------------------------------------------------------------
def _fmaf(a, b, c):
    # fp32 FMA: the product of two floats is exact in float64; the sum is rounded to float64, then to float32 (at most one ulp of double
    # rounding more than the hardware FMA, far inside the bound's slack)
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def screen_corr(win, tpl):
    """The kernel's fp32 screen: lane j owns template samples [16j, 16j+16), a 32-FMA chain per component, the fold by 16 and 8, then
    the row sums ((r0+r1)+(r2+r3)) + ((r4+r5)+(r6+r7)).  Returns complex128 [N_LAG]."""
    wf = np.stack([win.real, win.imag], -1).astype(np.float32)            # [N_SMP, 2]
    tf = np.stack([tpl.real, tpl.imag], -1).astype(np.float32)
    lags = np.arange(N_LAG)[:, None, None]
    idx = lags + NSL * np.arange(32)[None, :, None] + np.arange(NSL)[None, None, :]        # [lag, lane, n]
    w = wf[idx]                                                          # [lag, lane, n, 2]
    t = tf[(NSL * np.arange(32)[:, None] + np.arange(NSL)[None, :])]     # [lane, n, 2]
    ar = np.zeros((N_LAG, 32), np.float32)
    ai = np.zeros((N_LAG, 32), np.float32)
    for n in range(NSL):
        wx, wy, tx, ty = w[:, :, n, 0], w[:, :, n, 1], t[None, :, n, 0], t[None, :, n, 1]
        ar = _fmaf(wx, tx, _fmaf(wy, ty, ar))
        ai = _fmaf(wy, tx, _fmaf(-wx, ty, ai))

    def fold(a):
        a = (a[:, :16] + a[:, 16:]).astype(np.float32)
        a = (a[:, :8] + a[:, 8:16]).astype(np.float32)
        s0 = ((a[:, 0] + a[:, 1]) + (a[:, 2] + a[:, 3])).astype(np.float32)
        s1 = ((a[:, 4] + a[:, 5]) + (a[:, 6] + a[:, 7])).astype(np.float32)
        return (s0 + s1).astype(np.float32).astype(np.float64)
    return fold(ar) + 1j * fold(ai)


def exact_corr(win, tpl):
    idx = np.arange(N_LAG)[:, None] + np.arange(L)[None, :]
    return np.array([sum(v) for v in (win[idx] * np.conj(tpl)[None, :]).astype(np.clongdouble)], dtype=np.complex128)


def screen_eps(win, tpl):
    e_w = float(np.sum(np.abs(win) ** 2)) * (1 + 1e-12)
    e_t = float(np.sum(np.abs(tpl) ** 2)) * (1 + 1e-12)
    if not (e_w <= E_MAX and e_t <= E_MAX):
        return None
    return EPS_K * U * math.sqrt(e_w * e_t) * (1 + 1e-12) + EPS_ABS * (1 + math.sqrt(L * e_t) + math.sqrt(L * e_w))


def _windows():
    rng = np.random.default_rng(7)
    tpl = oracle.gsm_SCH_training_sequence_gen(8)
    cn = lambda n, s=1.0: s * (rng.standard_normal(n) + 1j * rng.standard_normal(n))      # noqa: E731
    out = [("noise", cn(N_SMP)), ("zero", np.zeros(N_SMP, complex))]
    w = cn(N_SMP, 1e-3)
    w[64:64 + L] += tpl                                                  # a burst at lag 64
    out.append(("burst", w))
    out.append(("dynamic_range", cn(N_SMP) * 10.0 ** rng.uniform(-30, 12, N_SMP)))
    spike = np.zeros(N_SMP, complex)
    spike[300] = 3e15 + 1e15j
    spike[10] = 1e-25
    out.append(("spike", spike))
    out.append(("tiny", cn(N_SMP, 1e-36)))                               # fp32 subnormal / underflow territory
    out.append(("large", cn(N_SMP, 1e15)))
    near = np.zeros(N_SMP, complex)
    near[64:64 + L] += 0.5 * tpl
    near[65:65 + L] += 0.5 * tpl
    out.append(("tie", near))
    return tpl, out


def test_screen_constants_match_the_derivation():
    # sqrt(2) * (37 + 2 + 2) u (lane chains of 32 FMAs, fold 2, rows 3; two input roundings) rounded up with room to spare
    assert EPS_K >= math.sqrt(2) * 41 * 1.01
    assert EPS_ABS == 2.0 ** -100 and E_MAX == 2.0 ** 120


@pytest.mark.parametrize("case", range(8))
def test_screen_error_within_eps(case):
    tpl, wins = _windows()
    name, win = wins[case]
    eps = screen_eps(win, tpl)
    assert eps is not None and math.isfinite(eps), name
    err = np.abs(screen_corr(win, tpl) - exact_corr(win, tpl))
    assert np.all(err <= eps), (name, float(np.max(err)), eps)


def test_screen_bound_refuses_overflow():
    tpl, _ = _windows()
    assert screen_eps(np.full(N_SMP, 1e60 + 0j), tpl) is None
    assert screen_eps(np.full(N_SMP, np.nan + 0j), tpl) is None
    assert screen_eps(np.full(N_SMP, np.inf + 0j), tpl) is None


def test_zero_window_leaves_every_lag_a_candidate():
    # M = max(|c| - eps) = -eps < 0, so every lag passes (|c| + eps)(1 + 1e-9) >= M (1 - 1e-9): 89 > 8 candidates -> the fp64 fallback
    tpl, _ = _windows()
    win = np.zeros(N_SMP, complex)
    eps = screen_eps(win, tpl)
    a = np.abs(screen_corr(win, tpl))
    m = np.max(a - eps)
    assert np.count_nonzero((a + eps) * (1 + 1e-9) >= m * (1 - 1e-9)) == N_LAG


# ---- GPU -------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def coef47():
    return oracle.fir1(46, 200e3 / FS)


@pytest.fixture(scope="module")
def tpl():
    return oracle.gsm_SCH_training_sequence_gen(8)


@pytest.fixture(scope="module")
def captures():
    specs = [synth.random_spec(seed, N_SYNC) for seed in (1, 2, 3, 4, 5)]
    return specs, synth.generate_batch(specs).numpy()


def _lib():
    from gsmcal._lib import lib
    return lib()


def _stats():
    g = _lib().gsmcal_debug_get
    return dict(screened=g(120), fallback=g(121), hist=[g(121 + c) for c in range(1, 9)])


def _run_modes(fn, modes=(0, 1, 2)):
    out, stats = {}, {}
    try:
        for m in modes:
            assert _lib().gsmcal_debug_set(24, m) == 0
            out[m] = fn()
            stats[m] = _stats()
    finally:
        _lib().gsmcal_debug_set(24, 0)
    return out, stats


def _same_batch(a, b):
    for sa, sb in zip(a, b):
        for k in ("coarse_pos", "coarse_snr", "fcch_pos", "pos_info"):
            assert np.array_equal(sa[k], sb[k]), k
        for k in ("sampling_ppm", "carrier_ppm", "total_sampling_ppm", "total_carrier_ppm", "flags", "r_len"):
            assert np.array_equal(np.asarray(sa[k]), np.asarray(sb[k])), k


@pytest.mark.gpu
def test_debug_key_24_rejects_other_values(gpu):
    assert _lib().gsmcal_debug_set(24, 3) != 0
    assert _lib().gsmcal_debug_set(24, -1) != 0
    assert _lib().gsmcal_debug_set(24, 0) == 0


@pytest.mark.gpu
def test_batch_identical_across_modes(gpu, captures, coef47, tpl):
    _, raw = captures
    out, stats = _run_modes(lambda: gpu.calibrate_batch(raw, CARRIER, tpl, coef47))
    _same_batch(out[0], out[1])
    _same_batch(out[0], out[2])
    assert stats[0]["screened"] > 0 and stats[0]["screened"] == sum(stats[0]["hist"])
    assert stats[1]["screened"] == 0 and stats[1]["fallback"] > 0
    assert stats[2]["screened"] == 0 and stats[2]["fallback"] == stats[0]["screened"] + stats[0]["fallback"]


@pytest.mark.gpu
def test_device_resident_submit_identical_across_modes(gpu, captures, coef47, tpl):
    import torch
    _, raw = captures
    dev = torch.from_numpy(raw).cuda()
    n_iq, D = raw.shape[1] // 2, raw.shape[0]
    out, stats = _run_modes(lambda: gpu.calibrate_batch(None, CARRIER, tpl, coef47, device_ptr=dev.data_ptr(), n_iq=n_iq, n_streams=D),
                            modes=(0, 1))
    _same_batch(out[0], out[1])
    assert stats[0]["screened"] > 0


def _planted(tpl, shift=0, frac=None, n_burst=6, noise=0.0, seed=3):
    """SCH templates on a 10-frame FCCH grid; shift moves every template by whole samples off lag 64 (-64 -> lag 0, +24 -> lag 88);
    frac = (a, b) plants a * tpl[n] + b * tpl[n - 1]: two neighbouring lags within ~|a - b| of each other."""
    fcch = 2001.0 + 10000.0 * np.arange(n_burst)
    n = int(fcch[-1]) + 10336 + 2 * 512 + 20000
    rng = np.random.default_rng(seed)
    s = noise * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    for p in fcch:
        a = int(p) + 10336 - 1 + shift
        if frac is None:
            s[a:a + 512] += tpl
        else:
            s[a:a + 512] += frac[0] * tpl
            s[a + 1:a + 513] += frac[1] * tpl
    return s, fcch


def _same_dropin(a, b):
    assert np.array_equal(a[0], b[0])
    assert (a[1] is None) == (b[1] is None) and (a[1] is None or np.array_equal(a[1], b[1]))
    assert a[2] == b[2] or (math.isnan(a[2]) and math.isnan(b[2]))


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["chain", "edge_abort", "spurious", "lag0", "lag88", "noise_only", "near_tie", "zero"])
def test_dropin_identical_across_modes(gpu, captures, coef47, tpl, case):
    if case in ("chain", "edge_abort", "spurious"):
        _, raw = captures
        r = oracle.fir_filter(coef47, oracle.raw2iq(raw[0])[:, 0])
        coarse, _ = oracle.FCCH_coarse_position(r[::64], 8)
        fpos, r1, _, _ = oracle.FCCH_fine_correction(r, coarse, 8, CARRIER)
        s, fcch = r1, fpos - {"chain": 0, "edge_abort": 41, "spurious": 200}[case]
    elif case == "lag0":
        s, fcch = _planted(tpl, shift=-64, noise=1e-3)
    elif case == "lag88":
        s, fcch = _planted(tpl, shift=24, noise=1e-3)
    elif case == "noise_only":
        s, fcch = _planted(tpl, noise=1.0)
        s = s - _planted(tpl)[0]                                         # the same noise without the templates
    elif case == "near_tie":
        s, fcch = _planted(tpl, frac=(0.5 + 5e-8, 0.5 - 5e-8))
    else:
        s, fcch = np.zeros(200000, complex), 2001.0 + 10000.0 * np.arange(6)
    out, stats = _run_modes(lambda: gpu.SCH_corr_rate_correction(s, fcch, tpl, 8))
    _same_dropin(out[0], out[1])
    _same_dropin(out[0], out[2])
    if case in ("lag0", "lag88"):
        ref = oracle.SCH_corr_rate_correction(s, fcch, tpl, 8)
        assert np.array_equal(out[0][0], ref[0])
    if case == "near_tie":
        assert sum(stats[0]["hist"][1:]) > 0                              # the screen kept both neighbours and chose in fp64
    if case == "zero":
        assert stats[0]["screened"] == 0 and stats[0]["fallback"] > 0     # 89 candidates: the fp64 fallback
