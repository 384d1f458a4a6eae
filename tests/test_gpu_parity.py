"""Parity of the CUDA hot path (through the C ABI) against the CPU oracle on identical inputs.

Bars (BASELINE.json north_star): burst indices / pos_info / hit_idx / raw2iq bit-exact; ppm within 1e-3 ppm;
floating-point streams within the relative tolerance written in each test.
"""
import json
import math
import os

import numpy as np
import pytest

import gsmcal_oracle as oracle
from gsmcal import synth

pytestmark = pytest.mark.gpu

FS = oracle.SYMBOL_RATE * 8
CARRIER = 957.4e6
N_SYNC = 1020000                       # gsm_sync_demod.m:23-29
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def rel_err(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


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


@pytest.fixture(scope="module")
def oracle_chain(captures, coef47, tpl):
    """Oracle intermediates for seed 1, shared by the per-function tests."""
    _, raw = captures
    r = oracle.fir_filter(coef47, oracle.raw2iq(raw[0])[:, 0])
    coarse, coarse_snr = oracle.FCCH_coarse_position(r[::64], 8)
    fpos, r1, sppm1, cppm1 = oracle.FCCH_fine_correction(r, coarse, 8, CARRIER)
    pinfo, r2, sppm2 = oracle.SCH_corr_rate_correction(r1, fpos, tpl, 8)
    r3, cppm2 = oracle.carrier_correct_post_SCH(r2, pinfo, 8, CARRIER)
    return dict(r=r, coarse=coarse, coarse_snr=coarse_snr, fpos=fpos, r1=r1, sppm1=sppm1, cppm1=cppm1,
                pinfo=pinfo, r2=r2, sppm2=sppm2, r3=r3, cppm2=cppm2)


# ---- K1 ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_iq,cols", [(1, 1), (7, 3), (4096, 2), (100003, 5), (1020000, 2)])
def test_raw2iq_u8_bit_exact(gpu, n_iq, cols):
    rng = np.random.default_rng(n_iq)
    a = rng.integers(0, 256, size=(2 * n_iq, cols), dtype=np.uint8)
    got = gpu.raw2iq(a)
    ref = oracle.raw2iq(a)
    assert got.shape == ref.shape
    assert np.array_equal(got, ref)


def test_raw2iq_double_input_bit_exact(gpu):
    rng = np.random.default_rng(3)
    a = rng.integers(0, 256, size=(2 * 5001, 2)).astype(np.float64)      # what fread(...,'uint8') returns
    assert np.array_equal(gpu.raw2iq(a), oracle.raw2iq(a))


def test_raw2iq_extremes(gpu):
    for v in (0, 255):
        a = np.full((2 * 1000, 1), v, dtype=np.uint8)
        assert np.array_equal(gpu.raw2iq(a), oracle.raw2iq(a))


# ---- K2 ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("order,decim", [(46, 1), (30, 1), (63, 1), (127, 1), (46, 64), (30, 64), (63, 20), (46, 2), (46, 3)])
def test_fir_filter_matches_lfilter(gpu, order, decim):
    rng = np.random.default_rng(order * 100 + decim)
    n = 50021
    s = rng.standard_normal((n, 2)) * 40 + 1j * rng.standard_normal((n, 2)) * 40
    coef = oracle.fir1(order, 0.09)
    got = gpu.fir_filter(coef, s, decim)
    ref = oracle.fir_filter(coef, s, decim)
    assert got.shape == ref.shape
    assert rel_err(got, ref) < 1e-14            # same nesting order as direct-form-II-transposed, FMA instead of mul+add


def test_fir_short_input_startup_transient(gpu):
    coef = oracle.fir1(46, 0.09)
    s = (np.arange(10) + 1j * np.arange(10)).astype(np.complex128)       # shorter than the filter
    assert rel_err(gpu.fir_filter(coef, s), oracle.fir_filter(coef, s)) < 1e-14


def test_fir1_matches_firwin(gpu):
    for order, wn in ((46, 200e3 / FS), (30, 200e3 / FS), (63, 0.05 / 2.048), (127, 0.01)):
        assert np.max(np.abs(gpu.fir1(order, wn) - oracle.fir1(order, wn))) < 2e-16


def test_fused_raw2iq_fir(gpu, captures, coef47):
    _, raw = captures
    a = raw[:2, :2 * 200000].T.copy()
    ref = oracle.fir_filter(coef47, oracle.raw2iq(a))
    assert rel_err(gpu.raw2iq_fir(a, coef47, 1), ref) < 1e-14
    assert rel_err(gpu.raw2iq_fir(a, coef47, 64), ref[::64]) < 1e-14


def test_chn_filters_with_fda_taps(gpu):
    with open(os.path.join(GOLDEN, "chn_filter_taps.json")) as f:
        g = json.load(f)
    num8 = np.array([float.fromhex(h) for h in g["Num_8x"]["hex"]])
    num4 = np.array([float.fromhex(h) for h in g["Num_4x"]["hex"]])
    assert np.array_equal(gpu.chn_filter_taps(8), num8)
    assert np.array_equal(gpu.chn_filter_taps(4), num4)
    rng = np.random.default_rng(7)
    s = rng.standard_normal((20001, 2)) + 1j * rng.standard_normal((20001, 2))
    assert rel_err(gpu.chn_filter_8x_4x(s), oracle.chn_filter_8x_4x(s, num8)) < 1e-14
    assert rel_err(gpu.chn_filter_4x(s), oracle.chn_filter_4x(s, num4)) < 1e-14


def test_band_power_scanners(gpu):
    rng = np.random.default_rng(11)
    a = np.clip(np.round(rng.standard_normal((2 * 12288, 4)) * 20 + 127.5), 0, 255).astype(np.uint8)
    assert rel_err(gpu.band_power(a), oracle.band_power(a)) < 1e-12                 # scan_band_power_spectrum.m
    a = np.clip(np.round(rng.standard_normal((2 * 204800, 3)) * 20 + 127.5), 0, 255).astype(np.uint8)
    coef = oracle.fir1(63, 0.05 / 2.048)
    assert rel_err(gpu.band_power(a, coef, 20), oracle.band_power(a, coef, 20)) < 1e-12   # split scanner


# ---- K3 / K4 ---------------------------------------------------------------------------------------
def test_move_fft_snr_runtime_avg(gpu, oracle_chain):
    s = oracle_chain["r"][::64][:3594]
    ref = oracle.move_fft_snr_runtime_avg(s, 160, 16, 10)
    got = gpu.move_fft_snr_runtime_avg(s, 160, 16, 10)
    assert got[0] == ref[0] and got[1] == ref[1]
    assert abs(got[2] - ref[2]) < 1e-9 and abs(got[3] - ref[3]) < 1e-9
    _, trace = oracle.move_fft_snr_runtime_avg(s, 160, 16, 10, return_trace=True)
    assert np.max(np.abs(gpu.move_fft_snr_trace(s, 16) - trace)) < 1e-9


def test_move_fft_no_hit_sentinel(gpu):
    rng = np.random.default_rng(5)
    s = rng.standard_normal(2000) + 1j * rng.standard_normal(2000)
    assert gpu.move_fft_snr_runtime_avg(s, 160, 16, 10) == oracle.move_fft_snr_runtime_avg(s, 160, 16, 10) == (False, -1.0, math.inf, math.inf)


def test_specific_fft_snr_fix_avg(gpu, oracle_chain):
    s = oracle_chain["r"][::64]
    p = int((oracle_chain["coarse"][1] - 1) / 8 + 1)
    for avg in (0.0, 30.0):
        ref = oracle.specific_fft_snr_fix_avg(s, (p - 5, p + 5), 16, 10, avg)
        got = gpu.specific_fft_snr_fix_avg(s, (p - 5, p + 5), 16, 10, avg)
        assert got[0] == ref[0] and got[1] == ref[1]
        if ref[0]:
            assert abs(got[2] - ref[2]) < 1e-9
        else:
            assert got[2] == math.inf


def test_fcch_coarse_position(gpu, oracle_chain):
    pos, snr = gpu.FCCH_coarse_position(oracle_chain["r"][::64], 8)
    assert np.array_equal(pos, oracle_chain["coarse"])
    assert np.max(np.abs(snr - oracle_chain["coarse_snr"])) < 1e-9


def test_fcch_coarse_noise_only_sentinel(gpu):
    rng = np.random.default_rng(9)
    s = rng.standard_normal(16000) + 1j * rng.standard_normal(16000)
    pos, snr = gpu.FCCH_coarse_position(s, 8)
    ref = oracle.FCCH_coarse_position(s, 8)
    assert np.array_equal(pos, ref[0]) and np.array_equal(snr, ref[1]) and pos[0] == -1


# ---- K5-K8 -----------------------------------------------------------------------------------------
def test_fcch_fine_correction(gpu, oracle_chain):
    fpos, r1, sppm, cppm = gpu.FCCH_fine_correction(oracle_chain["r"], oracle_chain["coarse"], 8, CARRIER)
    assert np.array_equal(fpos, oracle_chain["fpos"])
    assert sppm == oracle_chain["sppm1"]                      # integer differences -> identical fp64
    assert abs(cppm - oracle_chain["cppm1"]) < 1e-3
    assert len(r1) == len(oracle_chain["r1"])
    assert rel_err(r1, oracle_chain["r1"]) < 1e-8             # derotation phase: n*dphi reaches 1e5..1e6 rad


def test_fcch_fine_fewer_than_5_hits_sentinel(gpu, oracle_chain):
    fpos, r1, sppm, cppm = gpu.FCCH_fine_correction(oracle_chain["r"], oracle_chain["coarse"][:4], 8, CARRIER)
    assert np.array_equal(fpos, [-1.0]) and r1 is None and sppm == math.inf and cppm == math.inf


def test_fcch_fine_runout_keeps_first_round_positions(gpu, oracle_chain):
    # truncate the stream so only 3 coarse hits survive the run-out check: FCCH_pos = first-round positions, r = -1
    n_cut = int(oracle_chain["coarse"][3] * 8)
    s = oracle_chain["r"][:n_cut]
    ref = oracle.FCCH_fine_correction(s, oracle_chain["coarse"], 8, CARRIER)
    got = gpu.FCCH_fine_correction(s, oracle_chain["coarse"], 8, CARRIER)
    assert len(ref[0]) < 5 and np.array_equal(got[0], ref[0]) and got[1] is None and ref[1] is None
    assert got[2] == math.inf and got[3] == math.inf


def test_fcch_fine_bad_spacing_returns_s(gpu, oracle_chain):
    base = oracle_chain["coarse"].copy()
    base[2] += 700                                             # > 4000 ppm of 10 frames: spacing classification fails
    ref = oracle.FCCH_fine_correction(oracle_chain["r"], base, 8, CARRIER)
    got = gpu.FCCH_fine_correction(oracle_chain["r"], base, 8, CARRIER)
    assert np.array_equal(ref[0], [-1.0]) and np.array_equal(got[0], [-1.0])
    assert np.array_equal(got[1], oracle_chain["r"]) and got[2] == math.inf


# ---- K9-K10 ----------------------------------------------------------------------------------------
def test_sch_template_generator(gpu, tpl):
    assert np.max(np.abs(gpu.gsm_SCH_training_sequence_gen(8) - tpl)) < 1e-12
    assert np.max(np.abs(gpu.gsm_SCH_training_sequence_gen(4) - oracle.gsm_SCH_training_sequence_gen(4))) < 1e-12


def test_sch_corr_rate_correction(gpu, oracle_chain, tpl):
    pinfo, r2, sppm = gpu.SCH_corr_rate_correction(oracle_chain["r1"], oracle_chain["fpos"], tpl, 8)
    assert np.array_equal(pinfo, oracle_chain["pinfo"])
    assert sppm == oracle_chain["sppm2"]
    assert rel_err(r2, oracle_chain["r2"]) < 1e-13


def test_sch_sentinels(gpu, oracle_chain, tpl):
    r1, fpos = oracle_chain["r1"], oracle_chain["fpos"]
    got = gpu.SCH_corr_rate_correction(r1, fpos[:4], tpl, 8)
    assert np.array_equal(got[0], [[-1.0, -1.0]]) and got[1] is None and got[2] == math.inf
    # shifted FCCH positions push the correlation peak to the window edge -> pos_info=[-1,-1]
    ref = oracle.SCH_corr_rate_correction(r1, fpos - 41, tpl, 8)
    got = gpu.SCH_corr_rate_correction(r1, fpos - 41, tpl, 8)
    assert ref[0].shape == (1, 2) and np.array_equal(got[0], ref[0]) and got[1] is None and ref[1] is None
    # positions 200 samples off: peaks are spurious, the spacing test fails -> pos_info=-ones(3H,2), r=s
    ref = oracle.SCH_corr_rate_correction(r1, fpos - 200, tpl, 8)
    got = gpu.SCH_corr_rate_correction(r1, fpos - 200, tpl, 8)
    assert np.array_equal(got[0], ref[0]) and (got[1] is None) == (ref[1] is None)
    # stream cut so fewer than 5 SCH fit: pos_info = -ones(3H,2)
    n_cut = int(fpos[4] + 5000)
    ref = oracle.SCH_corr_rate_correction(r1[:n_cut], fpos, tpl, 8)
    got = gpu.SCH_corr_rate_correction(r1[:n_cut], fpos, tpl, 8)
    assert ref[0].shape == (3 * len(fpos), 2) and np.array_equal(got[0], ref[0]) and got[1] is None and ref[1] is None


def test_carrier_correct_post_sch(gpu, oracle_chain):
    r3, cppm = gpu.carrier_correct_post_SCH(oracle_chain["r2"], oracle_chain["pinfo"], 8, CARRIER)
    assert abs(cppm - oracle_chain["cppm2"]) < 1e-3
    assert rel_err(r3, oracle_chain["r3"]) < 1e-8
    for bad in (np.array([[-1.0, -1.0]]), -np.ones((30, 2)), oracle_chain["pinfo"][:3]):
        r, c = gpu.carrier_correct_post_SCH(oracle_chain["r2"], bad, 8, CARRIER)
        rr, cc = oracle.carrier_correct_post_SCH(oracle_chain["r2"], bad, 8, CARRIER)
        assert r is None and rr is None and c == math.inf and cc == math.inf


def test_total_ppm_calculation(gpu):
    for v in ([-35.0, 1.2], [math.inf, math.inf], [3.0, math.inf], [0.0, 0.0]):
        assert gpu.total_ppm_calculation(v) == oracle.total_ppm_calculation(v)


# ---- batched pipeline ------------------------------------------------------------------------------
def _check_stream(got, ref):
    assert np.array_equal(got["coarse_pos"], ref["coarse_pos"])
    assert np.array_equal(got["fcch_pos"], ref["fcch_pos"])
    assert np.array_equal(got["pos_info"], ref["pos_info"])
    for k in ("sampling_ppm", "carrier_ppm"):
        for a, b in zip(got[k], ref[k]):
            assert (a == b) if math.isinf(b) else abs(a - b) < 1e-3
    for k in ("total_sampling_ppm", "total_carrier_ppm"):
        assert (got[k] == ref[k]) if math.isinf(ref[k]) else abs(got[k] - ref[k]) < 1e-3


def test_calibrate_batch_matches_function_chain(gpu, captures, coef47, tpl):
    _, raw = captures
    got = gpu.calibrate_batch(raw, CARRIER, tpl, coef47)
    for d in range(raw.shape[0]):
        _check_stream(got[d], oracle.calibrate_stream(raw[d], CARRIER, tpl, coef47))


def test_osr8_fast_path_equals_round1_kernels(gpu, captures, coef47, tpl):
    """fine_core8_kernel + filtered-window cache (tier 2 and both tone stages read it) against the generic tier-1 kernel that
    re-filters in every stage (debug key 9): every output identical, ppm included (the cached samples are the same bits)."""
    from gsmcal._lib import lib
    _, raw = captures
    new = gpu.calibrate_batch(raw, CARRIER, tpl, coef47)
    lib().gsmcal_debug_set(9, 1)
    try:
        old = gpu.calibrate_batch(raw, CARRIER, tpl, coef47)
    finally:
        lib().gsmcal_debug_set(9, 0)
    for d, (a, b) in enumerate(zip(new, old)):
        for k in ("coarse_pos", "coarse_snr", "fcch_pos", "pos_info"):
            assert np.array_equal(a[k], b[k]), k
        assert a["sampling_ppm"] == b["sampling_ppm"] and a["flags"] & ~32 == b["flags"] & ~32
        assert np.allclose(a["carrier_ppm"], b["carrier_ppm"], rtol=0, atol=1e-9)
        if d < 2:
            _check_stream(a, oracle.calibrate_stream(raw[d], CARRIER, tpl, coef47))


def test_tone8_equals_generic_tone_estimator(gpu, captures, coef47, tpl):
    """tone8_kernel (cache-fed, Horner band DFT, certified gate) against tone_est_kernel for every burst (debug key 11); also with
    fewer tier-1 passes (key 10) so that more bursts reach the 64-bin band kernel"""
    from gsmcal._lib import lib
    _, raw = captures
    new = gpu.calibrate_batch(raw, CARRIER, tpl, coef47)
    outs = []
    for key, val, back in ((11, 1, 0), (10, 1, 8)):
        lib().gsmcal_debug_set(key, val)
        try:
            outs.append(gpu.calibrate_batch(raw, CARRIER, tpl, coef47))
        finally:
            lib().gsmcal_debug_set(key, back)
    for old in outs:
        for a, b in zip(new, old):
            for k in ("coarse_pos", "fcch_pos", "pos_info"):
                assert np.array_equal(a[k], b[k]), k
            assert a["sampling_ppm"] == b["sampling_ppm"]
            assert np.allclose(a["carrier_ppm"], b["carrier_ppm"], rtol=0, atol=1e-9)


def test_osr8_fast_path_other_tap_counts(gpu, captures, tpl):
    """the 48- and 64-tap instantiations of the fast path (zero-padded on the old side) and a filter too long for it (generic path)"""
    _, raw = captures
    for order in (30, 47, 63, 70):
        coef = oracle.fir1(order, 200e3 / FS)
        got = gpu.calibrate_batch(raw[:2], CARRIER, tpl, coef)
        for d in range(2):
            _check_stream(got[d], oracle.calibrate_stream(raw[d], CARRIER, tpl, coef))


def test_calibrate_batch_matches_golden(gpu, captures, coef47, tpl):
    _, raw = captures
    with open(os.path.join(GOLDEN, "pipeline_golden.json")) as f:
        g = json.load(f)["cases"]
    got = gpu.calibrate_batch(raw, CARRIER, tpl, coef47)
    for d, seed in enumerate((1, 2, 3, 4, 5)):
        c = g[str(seed)]
        assert np.array_equal(got[d]["fcch_pos"], c["fcch_pos"])
        assert np.array_equal(got[d]["pos_info"], np.array(c["pos_info"]))
        assert abs(got[d]["total_sampling_ppm"] - c["total_sampling_ppm"]) < 1e-3
        assert abs(got[d]["total_carrier_ppm"] - c["total_carrier_ppm"]) < 1e-3


def test_calibrate_batch_negative_fixtures(gpu, coef47, tpl):
    n = N_SYNC
    specs = [
        synth.StreamSpec(seed=21, n_samples=n, noise_only=True),                                  # coarse -1
        synth.StreamSpec(seed=22, n_samples=n, snr_db=0.0, sampling_ppm=5, carrier_ppm=3),        # weak: sentinel chain
        synth.StreamSpec(seed=23, n_samples=n, sampling_ppm=-12, carrier_ppm=8, drop_fcch=(2,)),  # dropped FCCH: chain stops early
        synth.StreamSpec(seed=24, n_samples=n, sampling_ppm=10, carrier_ppm=-20, start_offset=123456.0),
    ]
    raw = synth.generate_batch(specs).numpy()
    got = gpu.calibrate_batch(raw, CARRIER, tpl, coef47)
    for d in range(len(specs)):
        _check_stream(got[d], oracle.calibrate_stream(raw[d], CARRIER, tpl, coef47))
    assert got[0]["coarse_pos"][0] == -1 and math.isinf(got[0]["total_sampling_ppm"])


def test_fcch_scan_channels(gpu):
    n = 640000                                      # multi_rtl_sdr_gsm_FCCH_scanner.m:39-49
    coef = oracle.fir1(30, 200e3 / FS)
    specs = [synth.StreamSpec(seed=31, n_samples=n, sampling_ppm=7, carrier_ppm=-4, start_offset=4000.0),
             synth.StreamSpec(seed=32, n_samples=n, noise_only=True),
             synth.StreamSpec(seed=33, n_samples=n, sampling_ppm=-20, carrier_ppm=15, snr_db=12, start_offset=250000.0)]
    raw = synth.generate_batch(specs).numpy()
    snr, num_hit, positions = gpu.fcch_scan(raw, coef)
    for c in range(len(specs)):
        rs, rn, rp, _ = oracle.fcch_scan_channel(raw[c], coef)
        assert np.array_equal(positions[c], rp)
        assert num_hit[c] == rn and abs(snr[c] - rs) < 1e-9


def test_device_resident_batch_equals_host_batch(gpu, captures, coef47, tpl):
    torch = pytest.importorskip("torch")
    _, raw = captures
    dev = torch.from_numpy(raw[:2].copy()).cuda()
    torch.cuda.synchronize()
    a = gpu.calibrate_batch(None, CARRIER, tpl, coef47, device_ptr=dev.data_ptr(), n_iq=raw.shape[1] // 2, n_streams=2)
    b = gpu.calibrate_batch(raw[:2], CARRIER, tpl, coef47)
    for x, y in zip(a, b):
        assert np.array_equal(x["pos_info"], y["pos_info"]) and x["total_carrier_ppm"] == y["total_carrier_ppm"]


def test_band_limited_fine_search_equals_all_bin_search(gpu, captures, coef47, tpl):
    """The certified 64-bin sliding DFT must return exactly what the all-bin search returns (it falls back when unsure)."""
    from gsmcal._lib import lib
    _, raw = captures
    fast = gpu.calibrate_batch(raw, CARRIER, tpl, coef47)
    lib().gsmcal_debug_set(0, 1)
    try:
        full = gpu.calibrate_batch(raw, CARRIER, tpl, coef47)
    finally:
        lib().gsmcal_debug_set(0, 0)
    n_fallback = 0
    for a, b in zip(fast, full):
        assert np.array_equal(a["fcch_pos"], b["fcch_pos"]) and np.array_equal(a["pos_info"], b["pos_info"])
        assert a["sampling_ppm"] == b["sampling_ppm"]
        n_fallback += 1 if (a["flags"] & 32) else 0
    assert n_fallback <= 1, "the band certificate should hold for clean captures"


# ---- BASELINE full-size streams (10 s, 21 666 667 IQ) and size-independent properties ----------------------------
N_10S = 21666667


@pytest.fixture(scope="module")
def captures_10s():
    torch = pytest.importorskip("torch")
    specs = [synth.random_spec(seed, N_10S) for seed in (101, 102)]
    raw = synth.generate_batch(specs, device="cuda")
    torch.cuda.synchronize()
    return specs, raw


def test_full_size_streams_match_oracle(gpu, captures_10s, coef47, tpl):
    specs, raw = captures_10s
    got = gpu.calibrate_batch(None, CARRIER, tpl, coef47, device_ptr=raw.data_ptr(), n_iq=N_10S, n_streams=raw.shape[0])
    host = raw.cpu().numpy()
    for d in range(raw.shape[0]):
        ref = oracle.calibrate_stream(host[d], CARRIER, tpl, coef47)
        _check_stream(got[d], ref)
        assert len(got[d]["fcch_pos"]) > 200 and got[d]["pos_info"].shape[0] > 550
        # sanity against the injected impairments (not parity): 10 s gives 0.05 ppm resolution on the sampling clock
        assert abs(got[d]["total_sampling_ppm"] - specs[d].sampling_ppm) < 0.2
        assert abs(got[d]["total_carrier_ppm"] - specs[d].carrier_ppm) < 1.6


def test_full_size_staggered_submit_collect_equals_synchronous_call(gpu, coef47, tpl):
    """BASELINE-size rows (43 333 334 bytes: every row starts 6 bytes further from a 16-byte boundary, so the TMA-ring column sums peel
    heads and tails), two batches of four streams in flight with the library defaults (staggered, two stream groups per batch)."""
    torch = pytest.importorskip("torch")
    specs = [synth.random_spec(seed, N_10S) for seed in (201, 202, 203, 204, 205)]
    raw = synth.generate_batch(specs, device="cuda")
    torch.cuda.synchronize()
    st = torch.cuda.current_stream().cuda_stream
    row = raw.shape[1]
    ref_a = gpu.calibrate_batch(None, CARRIER, tpl, coef47, device_ptr=raw.data_ptr(), n_iq=N_10S, n_streams=4, cuda_stream=st)
    ref_b = gpu.calibrate_batch(None, CARRIER, tpl, coef47, device_ptr=raw.data_ptr() + row, n_iq=N_10S, n_streams=4, cuda_stream=st)
    pend = [gpu.calibrate_batch_submit(0, raw.data_ptr(), N_10S, 4, CARRIER, tpl, coef47, cuda_stream=st, details=True),
            gpu.calibrate_batch_submit(1, raw.data_ptr() + row, N_10S, 4, CARRIER, tpl, coef47, cuda_stream=st, details=True)]
    got = [pend[0].collect()]
    pend.append(gpu.calibrate_batch_submit(0, raw.data_ptr(), N_10S, 4, CARRIER, tpl, coef47, cuda_stream=st, details=True))
    got += [pend[1].collect(), pend[2].collect()]
    for g, ref in zip(got, (ref_a, ref_b, ref_a)):
        for x, y in zip(g, ref):
            for k in ("coarse_pos", "coarse_snr", "fcch_pos", "pos_info"):
                np.testing.assert_array_equal(x[k], y[k])
            assert x["sampling_ppm"] == y["sampling_ppm"] and x["carrier_ppm"] == y["carrier_ppm"] and x["flags"] == y["flags"]
            assert x["total_sampling_ppm"] == y["total_sampling_ppm"] and x["total_carrier_ppm"] == y["total_carrier_ppm"]
    assert sum(1 for x in got[0] if len(x["fcch_pos"]) > 200) >= 3            # the streams do lock: the comparison is not about sentinels


def test_full_size_structural_properties(gpu, captures_10s, coef47, tpl):
    specs, raw = captures_10s
    got = gpu.calibrate_batch(None, CARRIER, tpl, coef47, device_ptr=raw.data_ptr(), n_iq=N_10S, n_streams=raw.shape[0])
    again = gpu.calibrate_batch(None, CARRIER, tpl, coef47, device_ptr=raw.data_ptr(), n_iq=N_10S, n_streams=raw.shape[0])
    for a, b in zip(got, again):                                  # deterministic: integer atomics only
        assert np.array_equal(a["pos_info"], b["pos_info"]) and a["carrier_ppm"] == b["carrier_ppm"]
    for r in got:
        d = np.diff(r["fcch_pos"])
        assert set(d.tolist()) <= {100000.0, 110000.0}            # FCCH_pos is rebuilt on the ideal 10/11-frame grid
        assert np.all(np.diff(r["coarse_pos"]) > 0)
        p = r["pos_info"]
        assert np.all(np.diff(p[:, 0]) > 0)                       # bursts in time order
        assert set(p[:, 1].tolist()) == {0.0, 1.0, 2.0}
        f = p[p[:, 1] == 0, 0]
        s = p[p[:, 1] == 1, 0]
        assert np.all(s[:len(f)] - f[:len(s)] == 10000)           # SCH one frame after its FCCH (SCH_corr_rate_correction.m:146-151)
        b = p[p[:, 1] == 2, 0]
        assert len(b) % 4 == 0 or len(b) >= 4


def test_batch_is_stream_independent(gpu, captures, coef47, tpl):
    """Permuting / duplicating streams permutes / duplicates the results: no cross-stream state."""
    _, raw = captures
    base = gpu.calibrate_batch(raw, CARRIER, tpl, coef47)
    perm = [3, 0, 0, 4, 1, 2, 2]
    got = gpu.calibrate_batch(raw[perm], CARRIER, tpl, coef47)
    for i, src in enumerate(perm):
        assert np.array_equal(got[i]["pos_info"], base[src]["pos_info"])
        assert got[i]["sampling_ppm"] == base[src]["sampling_ppm"] and got[i]["carrier_ppm"] == base[src]["carrier_ppm"]
    one = gpu.calibrate_batch(raw[2:3], CARRIER, tpl, coef47)     # D = 1
    assert np.array_equal(one[0]["pos_info"], base[2]["pos_info"])


@pytest.mark.parametrize("n_iq", [230016, 230017, 400001])
def test_short_and_odd_length_captures(gpu, coef47, tpl, n_iq):
    """23 frames is the minimum FCCH_coarse_position accepts (s(1:3594)); such captures end on the '<5 hits' sentinels."""
    specs = [synth.random_spec(7, n_iq), synth.random_spec(8, n_iq)]
    raw = synth.generate_batch(specs).numpy()
    got = gpu.calibrate_batch(raw, CARRIER, tpl, coef47)
    for d in range(2):
        _check_stream(got[d], oracle.calibrate_stream(raw[d], CARRIER, tpl, coef47))


def test_capture_shorter_than_23_frames_is_a_range_error(gpu, coef47, tpl):
    raw = np.zeros((1, 2 * 200000), dtype=np.uint8)
    with pytest.raises(gpu.GsmcalError) as e:
        gpu.calibrate_batch(raw, CARRIER, tpl, coef47)
    assert e.value.code == -4
    with pytest.raises(IndexError):
        oracle.calibrate_stream(raw[0] + 1, CARRIER, tpl, coef47)


def test_other_filter_lengths_through_the_batch(gpu, captures, tpl):
    _, raw = captures
    for order in (30, 63):
        coef = oracle.fir1(order, 200e3 / FS)
        got = gpu.calibrate_batch(raw[:2], CARRIER, tpl, coef)
        for d in range(2):
            _check_stream(got[d], oracle.calibrate_stream(raw[d], CARRIER, tpl, coef))


def test_tier3_multiblock_search_equals_all_bin_search(gpu, captures, coef47, tpl):
    """Force every burst that reaches tier 2 to fail its certificate: tier 3 (19 band blocks per burst + combine, and the
    single-block all-bin kernel once more than FALL_GRID bursts are listed) must reproduce the all-bin result."""
    from gsmcal._lib import lib
    _, raw = captures
    lib().gsmcal_debug_set(0, 1)
    try:
        full = gpu.calibrate_batch(raw, CARRIER, tpl, coef47)
    finally:
        lib().gsmcal_debug_set(0, 0)
    lib().gsmcal_debug_set(4, 1)
    try:
        for groups, limit in ((1, 256), (2, 256), (1, 0)):       # limit 0: the work list goes to the single-block all-bin kernel
            lib().gsmcal_debug_set(3, groups)
            lib().gsmcal_debug_set(5, limit)
            t3 = gpu.calibrate_batch(raw, CARRIER, tpl, coef47)
            assert lib().gsmcal_debug_get(1) > 0
            for a, b in zip(t3, full):
                assert np.array_equal(a["fcch_pos"], b["fcch_pos"]) and np.array_equal(a["pos_info"], b["pos_info"])
                assert a["sampling_ppm"] == b["sampling_ppm"]
                # the forced all-bin path estimates the tone with tone_est_kernel, the tiers with tone8_kernel (same statements, other summation order)
                assert np.allclose(a["carrier_ppm"], b["carrier_ppm"], rtol=0, atol=1e-9)
    finally:
        lib().gsmcal_debug_set(4, 0)
        lib().gsmcal_debug_set(5, 256)
        lib().gsmcal_debug_set(3, 4)


def test_drop_in_chain_at_4x_oversampling(gpu, captures, tpl):
    """The reference functions take oversampling_ratio as an argument; run the per-function chain at 4 samples/symbol on
    the stream chn_filter_8x_4x produces (chn_filter_8x_4x.m: 60-tap equiripple filter, keep every 2nd sample)."""
    _, raw = captures
    with open(os.path.join(GOLDEN, "chn_filter_taps.json")) as f:
        num8 = np.array([float.fromhex(h) for h in json.load(f)["Num_8x"]["hex"]])
    b = oracle.raw2iq(raw[3])[:, 0]
    s4_ref = oracle.chn_filter_8x_4x(b, num8)
    s4 = gpu.chn_filter_8x_4x(gpu.raw2iq(raw[3])[:, 0])
    assert rel_err(s4, s4_ref) < 1e-14
    coarse_ref = oracle.FCCH_coarse_position(s4_ref[::32], 8)
    coarse = gpu.FCCH_coarse_position(s4_ref[::32], 8)
    assert np.array_equal(coarse[0], coarse_ref[0]) and len(coarse[0]) >= 5
    ref = oracle.FCCH_fine_correction(s4_ref, coarse_ref[0], 4, CARRIER)
    got = gpu.FCCH_fine_correction(s4_ref, coarse_ref[0], 4, CARRIER)
    assert np.array_equal(got[0], ref[0]) and got[2] == ref[2] and abs(got[3] - ref[3]) < 1e-3
    assert rel_err(got[1], ref[1]) < 1e-8
    tpl4 = oracle.gsm_SCH_training_sequence_gen(4)
    ref_s = oracle.SCH_corr_rate_correction(ref[1], ref[0], tpl4, 4)
    got_s = gpu.SCH_corr_rate_correction(ref[1], ref[0], tpl4, 4)
    assert np.array_equal(got_s[0], ref_s[0]) and got_s[2] == ref_s[2]
    if ref_s[1] is not None:
        ref_c = oracle.carrier_correct_post_SCH(ref_s[1], ref_s[0], 4, CARRIER)
        got_c = gpu.carrier_correct_post_SCH(ref_s[1], ref_s[0], 4, CARRIER)
        assert (ref_c[0] is None) == (got_c[0] is None)
        assert (got_c[1] == ref_c[1]) if math.isinf(ref_c[1]) else abs(got_c[1] - ref_c[1]) < 1e-3


# ---- BASELINE configs 2 and 4 at the reference's own sizes -----------------------------------------------------------
def test_config2_fcch_scanner_all_126_frequencies(gpu):
    """multi_rtl_sdr_gsm_FCCH_scanner.m: 935:0.2:960 MHz = 126 points, 640 000 IQ each, fir1(30), /64, coarse + acceptance."""
    torch = pytest.importorskip("torch")
    n, n_freq = 640000, 126
    coef = oracle.fir1(30, 200e3 / FS)
    carriers = {5: 11.0, 17: -23.0, 40: 3.5, 41: 30.0, 77: -8.0, 90: 0.0, 101: 19.0, 102: -31.0, 120: 7.0, 125: -2.0, 60: 14.0, 33: -17.0}
    specs = []
    for c in range(n_freq):
        if c in carriers:
            specs.append(synth.StreamSpec(seed=500 + c, n_samples=n, sampling_ppm=carriers[c], carrier_ppm=-carriers[c] / 2,
                                          snr_db=12.0 + (c % 10), start_offset=float((c * 7919) % synth.MULTIFRAME)))
        else:
            specs.append(synth.StreamSpec(seed=500 + c, n_samples=n, noise_only=True))
    raw = synth.generate_batch(specs, device="cuda").cpu().numpy()
    snr, num_hit, positions = gpu.fcch_scan(raw, coef)
    n_found = 0
    for c in range(n_freq):
        rs, rn, rp, _ = oracle.fcch_scan_channel(raw[c], coef)
        assert np.array_equal(positions[c], rp), f"channel {c}"
        assert num_hit[c] == rn and abs(snr[c] - rs) < 1e-9
        n_found += rn > 0
    assert n_found >= 10 and all(num_hit[c] == 0 for c in range(n_freq) if c not in carriers)


def test_config4_band_power_scans_at_reference_sizes(gpu):
    rng = np.random.default_rng(44)
    # scan_band_power_spectrum.m:14-20,48: 251 frequencies x 2 dongles x 3 datagrams of 8192 bytes (12 288 IQ)
    a = np.clip(np.round(rng.standard_normal((2 * 12288, 502)) * rng.uniform(3, 40, size=502) + 127.5), 0, 255).astype(np.uint8)
    got, ref = gpu.band_power(a), oracle.band_power(a)
    assert rel_err(got, ref) < 1e-12
    assert np.max(np.abs(10 * np.log10(got) - 10 * np.log10(ref))) < 1e-10
    # multi_rtl_sdr_split_scanner.m:40-57,71,154-156: 204 800 IQ per frequency at 2.048 MS/s, fir1(63, RBW/fs), /20 (64 of the 501 points)
    a = np.clip(np.round(rng.standard_normal((2 * 204800, 64)) * rng.uniform(3, 40, size=64) + 127.5), 0, 255).astype(np.uint8)
    coef = oracle.fir1(63, 0.05 / 2.048)
    assert rel_err(gpu.band_power(a, coef, 20), oracle.band_power(a, coef, 20)) < 1e-12


def test_randomised_impairment_sweep(gpu, coef47, tpl):
    """32 streams with wide random impairments (SNR 4-25 dB, amplitude 8-60 LSB, +-45 ppm clock, +-28 ppm carrier): every
    outcome - full lock, SNR-gate failure, short chains, no FCCH - must equal the oracle's (tests/stress_parity.py is the long form)."""
    rng = np.random.default_rng(7)
    specs = [synth.StreamSpec(seed=3000 + i, n_samples=N_SYNC, sampling_ppm=float(rng.uniform(-45, 45)), carrier_ppm=float(rng.uniform(-28, 28)),
                              snr_db=float(rng.uniform(4, 25)), phase0=float(rng.uniform(0, 6.28)),
                              start_offset=float(rng.integers(0, synth.MULTIFRAME)), amplitude=float(rng.uniform(8, 60))) for i in range(32)]
    raw = synth.generate_batch(specs, device="cuda").cpu().numpy()
    got = gpu.calibrate_batch(raw, CARRIER, tpl, coef47)
    outcomes = set()
    for d in range(len(specs)):
        ref = oracle.calibrate_stream(raw[d], CARRIER, tpl, coef47)
        _check_stream(got[d], ref)
        outcomes.add((ref["fcch_pos"][0] == -1, ref["pos_info"].shape[0] > 1))
    assert len(outcomes) >= 2


def test_diversity_scanner_combine(gpu):
    """multi_rtl_sdr_diversity_scanner.m:150-176: per-dongle power spectra and their incoherent mean."""
    rng = np.random.default_rng(5)
    s_all = np.clip(np.round(rng.standard_normal((2 * 20480, 12, 3)) * rng.uniform(3, 40, size=(1, 12, 3)) + 127.5), 0, 255).astype(np.uint8)
    coef = oracle.fir1(63, 0.05 / 2.048)
    per, comb = gpu.diversity_power_spectrum(s_all, coef, 20)
    ref = np.stack([oracle.band_power(s_all[:, :, i], coef, 20) for i in range(3)], axis=0)
    assert rel_err(per, ref) < 1e-12 and rel_err(comb, ref.mean(axis=0)) < 1e-12


def test_split_and_diversity_scanners_at_the_reference_size(gpu):
    """multi_rtl_sdr_split_scanner.m:40-57,154-156 at its own size (501 frequencies x 204,800 IQ at 2.048 MS/s, fir1(63, 0.05/2.048), /20)
    and the diversity scanner's device-side combination over 2 dongles at the same size (multi_rtl_sdr_diversity_scanner.m:150-176).
    The oracle filters 1002 columns of 204,800 samples: the slow part of this test is the CPU."""
    rng = np.random.default_rng(17)
    s_all = np.clip(np.round(rng.standard_normal((2 * 204800, 501, 2)) * rng.uniform(3, 40, size=(1, 501, 2)) + 127.5), 0, 255).astype(np.uint8)
    coef = oracle.fir1(63, 0.05 / 2.048)
    ref = np.stack([np.concatenate([oracle.band_power(s_all[:, f0:f0 + 64, i], coef, 20) for f0 in range(0, 501, 64)]) for i in range(2)], axis=0)
    assert rel_err(gpu.band_power(s_all[:, :, 0], coef, 20), ref[0]) < 1e-12               # split scanner: 501 frequencies, one dongle's share
    per, comb = gpu.diversity_power_spectrum(s_all, coef, 20)
    assert per.shape == (2, 501) and comb.shape == (501,)
    assert rel_err(per, ref) < 1e-12 and rel_err(comb, ref.sum(axis=0) / 2) < 1e-12


def test_submit_cancel_gives_the_slot_back(gpu, captures, coef47, tpl):
    import torch
    _, raw = captures
    a = torch.from_numpy(raw[:2].copy()).cuda()
    torch.cuda.synchronize()
    n_iq = raw.shape[1] // 2
    p = gpu.calibrate_batch_submit(0, a.data_ptr(), n_iq, 2, CARRIER, tpl, coef47)
    with pytest.raises(gpu.GsmcalError):                              # the slot is busy until collected or cancelled
        gpu.calibrate_batch_submit(0, a.data_ptr(), n_iq, 2, CARRIER, tpl, coef47)
    p.cancel()
    with pytest.raises(gpu.GsmcalError):
        p.collect()
    q = gpu.calibrate_batch_submit(0, a.data_ptr(), n_iq, 2, CARRIER, tpl, coef47, details=True)
    del p                                                             # a dropped, cancelled handle must not touch the slot again
    got = q.collect()
    _check_stream(got[0], oracle.calibrate_stream(raw[0], CARRIER, tpl, coef47))
    r = gpu.calibrate_batch_submit(1, a.data_ptr(), n_iq, 2, CARRIER, tpl, coef47)
    del r                                                             # dropped without collect: __del__ cancels, the slot is free again
    gpu.calibrate_batch_submit(1, a.data_ptr(), n_iq, 2, CARRIER, tpl, coef47).collect()


def test_second_device_after_the_first(gpu, captures, coef47, tpl):
    """per-device state (kernel attributes, stage events, twiddles, workspaces): device 1 used after device 0 in one process.
    Fewer than 8 streams takes the single-group path that records the stage events."""
    if gpu.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    _, raw = captures
    a = gpu.calibrate_batch(raw[:2], CARRIER, tpl, coef47)
    gpu.set_device(1)
    try:
        b = gpu.calibrate_batch(raw[:2], CARRIER, tpl, coef47)
        r = oracle.fir_filter(coef47, oracle.raw2iq(raw[0])[:, 0])
        pinfo = a[0]["pos_info"]
        d1 = gpu.FCCH_demod(r, pinfo, 8, CARRIER)                    # opts into > 48 KB of dynamic shared memory on device 1
        s1 = gpu.SCH_demod(r, pinfo, tpl, 8)
    finally:
        gpu.set_device(0)
    d0 = gpu.FCCH_demod(r, pinfo, 8, CARRIER)
    for x, y in zip(a, b):
        assert np.array_equal(x["pos_info"], y["pos_info"]) and x["total_carrier_ppm"] == y["total_carrier_ppm"]
    assert np.array_equal(d0["max_idx"], d1["max_idx"]) and s1 is not None


# ---- submit / collect: several batches in flight give the results of the synchronous call ---------------------------------------
def test_submit_collect_matches_synchronous_call(gpu, captures, coef47, tpl):
    import torch
    _, raw = captures
    a = torch.from_numpy(raw[:3].copy()).cuda()
    b = torch.from_numpy(raw[2:5].copy()).cuda()
    torch.cuda.synchronize()
    st = torch.cuda.current_stream().cuda_stream
    ref_a = gpu.calibrate_batch(None, CARRIER, tpl, coef47, device_ptr=a.data_ptr(), n_iq=N_SYNC, n_streams=3, cuda_stream=st)
    ref_b = gpu.calibrate_batch(None, CARRIER, tpl, coef47, device_ptr=b.data_ptr(), n_iq=N_SYNC, n_streams=3, cuda_stream=st)
    pend = [gpu.calibrate_batch_submit(0, a.data_ptr(), N_SYNC, 3, CARRIER, tpl, coef47, cuda_stream=st, details=True),
            gpu.calibrate_batch_submit(1, b.data_ptr(), N_SYNC, 3, CARRIER, tpl, coef47, cuda_stream=st, details=True),
            gpu.calibrate_batch_submit(2, a.data_ptr(), N_SYNC, 3, CARRIER, tpl, coef47, cuda_stream=st, details=True)]
    from gsmcal._lib import GsmcalError
    with pytest.raises(GsmcalError):                       # a slot holds one batch at a time
        gpu.calibrate_batch_submit(1, b.data_ptr(), N_SYNC, 3, CARRIER, tpl, coef47, cuda_stream=st)
    got = [p.collect() for p in pend]
    for g, ref in zip(got, (ref_a, ref_b, ref_a)):
        for x, y in zip(g, ref):
            for k in ("coarse_pos", "coarse_snr", "fcch_pos", "pos_info"):
                np.testing.assert_array_equal(x[k], y[k])
            assert x["sampling_ppm"] == y["sampling_ppm"] and x["carrier_ppm"] == y["carrier_ppm"] and x["flags"] == y["flags"]
    with pytest.raises(GsmcalError):
        pend[0].collect()                                  # nothing pending in the slot any more
    # slots are reusable, and the synchronous call still works in between
    again = gpu.calibrate_batch_submit(0, b.data_ptr(), N_SYNC, 3, CARRIER, tpl, coef47, cuda_stream=st, details=True).collect()
    assert [x["pos_info"].tolist() for x in again] == [y["pos_info"].tolist() for y in ref_b]


@pytest.mark.parametrize("stages,blocks", [(7, 1), (2, 3), (24, 1), (3, 2), (1, 1)])
def test_submit_collect_trickle_column_sums_and_staggered_batches(gpu, captures, coef47, tpl, stages, blocks):
    """debug keys 17-18: column sums by the TMA-ring kernel at several ring sizes (ragged stream starts: 2*N_RAG is not a multiple of 16),
    FP64 stages gated behind the previous batch - same records as the synchronous call, bit for bit.  (The default is 2 stages x 3
    blocks per SM.)"""
    import torch
    from gsmcal._lib import lib
    _, raw = captures
    N_RAG = N_SYNC - 3                                             # stream d starts 10*d bytes past a 16-byte boundary
    a = torch.from_numpy(np.ascontiguousarray(raw[:3, :2 * N_RAG])).cuda()
    b = torch.from_numpy(np.ascontiguousarray(raw[1:6, :2 * N_RAG])).cuda()
    torch.cuda.synchronize()
    st = torch.cuda.current_stream().cuda_stream
    ref_a = gpu.calibrate_batch(None, CARRIER, tpl, coef47, device_ptr=a.data_ptr(), n_iq=N_RAG, n_streams=3, cuda_stream=st)
    ref_b = gpu.calibrate_batch(None, CARRIER, tpl, coef47, device_ptr=b.data_ptr(), n_iq=N_RAG, n_streams=5, cuda_stream=st)
    for key, val in ((17, stages), (18, blocks)):
        assert lib().gsmcal_debug_set(key, val) == 0
    try:
        pend = [gpu.calibrate_batch_submit(0, a.data_ptr(), N_RAG, 3, CARRIER, tpl, coef47, cuda_stream=st, details=True),
                gpu.calibrate_batch_submit(1, b.data_ptr(), N_RAG, 5, CARRIER, tpl, coef47, cuda_stream=st, details=True)]
        got = [pend[0].collect()]
        pend.append(gpu.calibrate_batch_submit(0, b.data_ptr(), N_RAG, 5, CARRIER, tpl, coef47, cuda_stream=st, details=True))
        got += [pend[1].collect(), pend[2].collect()]
    finally:
        for key, val in ((17, 2), (18, 3)):                                       # the library defaults
            lib().gsmcal_debug_set(key, val)
    for g, ref in zip(got, (ref_a, ref_b, ref_b)):
        assert len(g) == len(ref)
        for x, y in zip(g, ref):
            for k in ("coarse_pos", "coarse_snr", "fcch_pos", "pos_info"):
                np.testing.assert_array_equal(x[k], y[k])
            assert x["sampling_ppm"] == y["sampling_ppm"] and x["carrier_ppm"] == y["carrier_ppm"] and x["flags"] == y["flags"]


# ---- SURVEY Appendix A: deliberate fixtures through the DROP-IN entry points, each asserting the branch it took ----------------
def _same_fine(got, ref, r_tol):
    assert np.array_equal(got[0], ref[0])
    assert (got[1] is None) == (ref[1] is None)
    if ref[1] is not None:
        assert len(got[1]) == len(ref[1]) and rel_err(got[1], ref[1]) < r_tol
    assert (got[2] == ref[2]) if math.isinf(ref[2]) else got[2] == ref[2]
    assert (got[3] == ref[3]) if math.isinf(ref[3]) else abs(got[3] - ref[3]) < 1e-3


def test_appendix_a_fine_overrun_returns_four_positions(gpu):
    import appendix_a_fixtures as fx
    args, took = fx.fine_overrun_drops_to_four()                     # FCCH_fine_correction.m:135-137,142
    ref, got = oracle.FCCH_fine_correction(*args), gpu.FCCH_fine_correction(*args)
    assert took(ref) and took(got)
    _same_fine(got, ref, 1e-13)                                      # r is resampled only on this path


def test_appendix_a_fine_snr_gate_return(gpu):
    import appendix_a_fixtures as fx
    args, took = fx.fine_snr_gate_return()                           # FCCH_fine_correction.m:192-196
    ref, got = oracle.FCCH_fine_correction(*args), gpu.FCCH_fine_correction(*args)
    assert took(ref) and took(got)
    _same_fine(got, ref, 1e-8)                                       # r is resampled and derotated


def test_appendix_a_sch_paths(gpu, tpl):
    import appendix_a_fixtures as fx
    args, took, _ = fx.sch_e_zero_skips_interp1(tpl)                 # SCH_corr_rate_correction.m:120-128
    ref, got = oracle.SCH_corr_rate_correction(*args), gpu.SCH_corr_rate_correction(*args)
    assert took(ref) and took(got) and np.array_equal(got[0], ref[0]) and got[2] == ref[2] == 0.0
    for build in (fx.sch_last_slot_does_not_fit, fx.sch_bcch_rows_run_out):      # :153-159, :167-178
        args, took = build(tpl)
        ref, got = oracle.SCH_corr_rate_correction(*args), gpu.SCH_corr_rate_correction(*args)
        assert took(ref) and took(got)
        assert np.array_equal(got[0], ref[0]) and got[2] == ref[2] and np.array_equal(got[1], ref[1])


def test_planted_known_answers_through_the_c_abi(gpu, tpl):
    """hand-derived answers (no oracle involved): templates planted on the ideal grid -> pos_info rows by the rules of
    SCH_corr_rate_correction.m:138-181; tones planted at known starts -> FCCH_pos, 0 ppm sampling error, the planted carrier offset"""
    osr, frame = 8, 10000
    for gaps, flagged in (((10, 10, 10, 11, 10, 10), {5}), ((10, 10, 10, 10, 11, 10), {1, 6}), ((10, 10, 10, 10, 10), set())):
        fcch = np.cumsum([2001] + [g * frame for g in gaps]).astype(np.float64)
        n = int(fcch[-1]) + 10336 + 512 + 5 * frame
        s = np.zeros(n, dtype=np.complex128)
        for p in fcch:
            s[int(p) + 10336 - 1:int(p) + 10336 - 1 + 512] = tpl
        pos_info, r, ppm = gpu.SCH_corr_rate_correction(s, fcch, tpl, osr)
        rows = []
        for i, p in enumerate(fcch, 1):
            rows += [[p, 0.0], [p + 10000, 1.0]] + ([[p + 10000 + k * frame, 2.0] for k in (1, 2, 3, 4)] if i in flagged else [])
        assert pos_info.tolist() == rows and ppm == 0.0 and np.array_equal(r, s)
    f_off = 2500.0
    rg = np.random.default_rng(5)
    starts = np.cumsum([30001] + [g * frame for g in (10, 10, 11, 10, 10)])
    n = int(starts[-1]) + 3 * frame
    s = 1e-3 * (rg.standard_normal(n) + 1j * rg.standard_normal(n))
    for p in starts:
        s[p - 1:p - 1 + 1184] += np.exp(2j * np.pi * (oracle.SYMBOL_RATE / 4 + f_off) * (p - 1 + np.arange(1184)) / FS)
    base = np.round((starts - 1) / osr) + 1 + np.array([3, -7, 0, 11, -20, 5])
    fpos, r, sppm, cppm = gpu.FCCH_fine_correction(s, base, osr, CARRIER)
    assert fpos.tolist() == starts.astype(float).tolist() and sppm == 0.0 and abs(cppm - 1e6 * f_off / CARRIER) < 1e-3


def test_pageable_host_buffers_go_through_the_staging_ring(gpu, captures, coef47, tpl):
    """NumPy arrays are pageable (like an mxArray): transfers above 32 MB use the library's pinned staging ring, both directions;
    results are the bytes a plain cudaMemcpy delivers (debug key 12 switches the ring off)."""
    from gsmcal._lib import lib
    rng = np.random.default_rng(3)
    n = 3_000_001                                                   # 48 MB of complex128 per column, odd length
    s = rng.standard_normal((n, 2)) + 1j * rng.standard_normal((n, 2))
    coef = oracle.fir1(46, 0.09)
    before = int(lib().gsmcal_debug_get(30))
    got = gpu.fir_filter(coef, s)
    moved = int(lib().gsmcal_debug_get(30)) - before
    assert moved >= 2 * s.nbytes                                    # in and out went through the ring
    lib().gsmcal_debug_set(12, 1)
    try:
        plain = gpu.fir_filter(coef, s)
        assert int(lib().gsmcal_debug_get(30)) - before == moved
    finally:
        lib().gsmcal_debug_set(12, 0)
    assert np.array_equal(got, plain)
    assert rel_err(got[:50000], oracle.fir_filter(coef, s[:50000])) < 1e-14
    a = rng.integers(0, 256, size=(2 * 20_000_003, 1), dtype=np.uint8)      # 40 MB uint8 -> 320 MB complex128 back
    assert np.array_equal(gpu.raw2iq(a), oracle.raw2iq(a))


def test_calibrate_batch_r_materialises_r_correct(gpu, captures, coef47, tpl):
    """gsmcal_calibrate_batch_r: the corrected stream gsm_sync_demod.m:120 hands to SCH_demod, written in one fused pass from the uint8
    capture (filter -> interp1(e1) -> derotate -> interp1(e2) -> derotate), against the oracle's function-by-function r_final; rows of
    streams whose chain did not complete (r = -1) are left untouched."""
    _, raw = captures
    specs = [synth.StreamSpec(seed=21, n_samples=N_SYNC, noise_only=True)]
    raw4 = np.concatenate([raw[:3], synth.generate_batch(specs).numpy()], axis=0)
    D, n_iq = raw4.shape[0], raw4.shape[1] // 2
    r = np.full((D, n_iq), 7.0 + 7.0j, dtype=np.complex128)
    got = gpu.calibrate_batch(raw4, CARRIER, tpl, coef47, r_correct=r)
    for d in range(D):
        ref = oracle.calibrate_stream(raw4[d], CARRIER, tpl, coef47)
        _check_stream(got[d], ref)
        if ref["r_final"] is None:
            assert got[d]["r_len"][2] == -1 and np.all(r[d] == 7.0 + 7.0j)
        else:
            n = got[d]["r_len"][2]
            assert n == len(ref["r_final"])
            assert rel_err(r[d, :n], ref["r_final"]) < 1e-8          # two derotations with n*dphi up to 1e5..1e6 rad
            assert np.all(r[d, n:] == 7.0 + 7.0j)
    assert got[3]["r_len"][2] == -1


def test_bench_workload_streams_match_the_oracle(gpu, coef47, tpl):
    """32 of bench.py's own 10 s streams (BASELINE config 5, seeds = stream indices) - half of them streams that do NOT fully calibrate
    in the timed run (SCH spacing failures, short chains, the SCH edge abort, the SNR-gate stream) - through the batched pipeline and
    through oracle.calibrate_stream on a process pool; bench.py's own comparison code, so the bench line's `oracle_agreement` is tested."""
    import sys
    torch = pytest.importorskip("torch")
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    n_iq = bench.N_IQ_10S
    failing = [48, 59, 94, 100, 122, 126, 179, 183, 218, 224, 300, 307, 309, 319, 332, 336]      # non-calibrating in profiles/r2*_bench*.json
    seeds = sorted(set(failing + list(range(0, 1024, 64))))
    raw = torch.empty((len(seeds), 2 * n_iq), dtype=torch.uint8, device="cuda")
    for i, sd in enumerate(seeds):
        synth.generate_stream(synth.random_spec(sd, n_iq), "cuda", raw[i])
    torch.cuda.synchronize()
    res = gpu.calibrate_batch(None, CARRIER, tpl, coef47, device_ptr=raw.data_ptr(), n_iq=n_iq, n_streams=len(seeds), details=False)
    rep = bench.oracle_agreement(gpu, raw, res, n_iq, tpl, coef47, len(seeds), os.cpu_count() or 4)
    assert rep["oracle_agrees"] == f"{len(seeds)}/{len(seeds)}", rep
    assert len(rep["checked_streams"]) == len(seeds)
    hist = rep["outcome_histogram_rank0"]
    assert hist.get("calibrated", 0) >= 8 and sum(v for k, v in hist.items() if k != "calibrated") >= 8, hist
