"""CPU tests of the oracle itself: MATLAB-semantics known answers, the reference's only golden data (the FIR
numerators inside the .fda sessions), and the committed pipeline fixtures (oracle drift guard)."""
import hashlib
import json
import math
import os

import numpy as np
import pytest
import scipy.linalg

import gsmcal_oracle as oracle
from gsmcal import synth

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
FS = oracle.SYMBOL_RATE * 8


def test_matlab_round_half_away_from_zero():
    assert oracle.mround(12500 / 8) == 1563 and round(12500 / 8) == 1562        # FCCH_coarse_position.m:35
    assert oracle.mround(13750 / 8) == 1719                                      # FCCH_coarse_position.m:36
    assert oracle.mround(-2.5) == -3 and oracle.mround(2.5) == 3 and oracle.mround(0.49999) == 0


def test_fda_numerators_golden():
    with open(os.path.join(GOLDEN, "chn_filter_taps.json")) as f:
        g = json.load(f)
    for key, n, b0, mid, total, sha in (("Num_8x", 60, -8.3045994016978379e-04, 1.3251507266392798e-01, 0.99423319989488024, "e2af20c654d63a5d"),
                                        ("Num_4x", 30, -2.1523104568354720e-03, 2.5886862810293920e-01, 0.99424850511591401, "b2f1c92d5f526927")):
        b = np.array([float.fromhex(h) for h in g[key]["hex"]])
        assert len(b) == n and b[0] == b0 and b[n // 2 - 1] == mid and b[n // 2] == mid
        assert np.array_equal(b, b[::-1])                                        # linear phase
        assert abs(b.sum() - total) < 1e-15
        assert hashlib.sha256(b.astype("<f8").tobytes()).hexdigest().startswith(sha)


def test_raw2iq_known_answer():
    a = np.array([[1, 10], [2, 20], [3, 30], [4, 40], [8, 50], [9, 60]], dtype=np.uint8)      # 3 IQ pairs x 2 dongles
    b = oracle.raw2iq(a)
    assert np.array_equal(b[:, 0], np.array([1 + 2j, 3 + 4j, 8 + 9j]) - (4 + 5j))
    assert np.array_equal(b[:, 1], np.array([10 + 20j, 30 + 40j, 50 + 60j]) - (30 + 40j))
    assert abs(b.sum()) == 0


def test_toeplitz_construction_is_sliding_windows():
    """FCCH_fine_correction.m:48-49 / SCH_corr_rate_correction.m:50-51: column b of the matrix is s(sp+b-1 : sp+b-1+L-1)."""
    rng = np.random.default_rng(0)
    s = rng.standard_normal(40) + 1j * rng.standard_normal(40)
    sp, length, L = 3, 7, 12                                  # 1-based start, windows, window length
    ep = sp + length - 1
    col = s[sp - 1:ep + L - 1]
    row = np.concatenate([[s[sp - 1]], np.zeros(length - 1)])
    m = scipy.linalg.toeplitz(col, row)[length - 1:, ::-1]
    win = np.lib.stride_tricks.sliding_window_view(s[sp - 1:sp - 1 + length + L - 1], L)
    assert np.array_equal(m, win.T)


def test_interp1_matches_numpy_interp():
    rng = np.random.default_rng(1)
    v = rng.standard_normal(1000) + 1j * rng.standard_normal(1000)
    for e in (35e-6, -20e-6, 1e-3):
        max_len = int(math.floor(len(v) / (1 + e))) if e >= 0 else len(v)
        got = oracle.interp1_uniform(v, e, max_len)
        xq = np.minimum(np.arange(max_len) * (1 + e), len(v) - 1)
        ref = np.interp(xq, np.arange(len(v)), v.real) + 1j * np.interp(xq, np.arange(len(v)), v.imag)
        assert np.max(np.abs(got - ref)) < 1e-12


def test_fir1_is_unity_gain_hamming_sinc():
    h = oracle.fir1(46, 200e3 / FS)
    assert len(h) == 47 and abs(h.sum() - 1) < 1e-15 and np.allclose(h, h[::-1], atol=0, rtol=1e-14)
    x = np.zeros(100, complex); x[0] = 1
    assert np.allclose(oracle.fir_filter(h, x)[:47], h)       # zero initial state, transient kept
    assert len(oracle.fir_filter(h, np.ones(129, complex), 64)) == 3


def test_moving_fft_detects_a_tone_burst_and_honours_the_999_warmup():
    rng = np.random.default_rng(2)
    n = 1200
    s = 0.3 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    s[600:640] += 3 * np.exp(2j * np.pi * 0.25 * np.arange(40))
    hit, idx, avg, snr = oracle.move_fft_snr_runtime_avg(s, 160, 16, 10)
    assert hit and 585 <= idx <= 610 and snr - avg > 10
    early = s.copy(); early[:1200] = 0.3 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    early[20:60] += 3 * np.exp(2j * np.pi * 0.25 * np.arange(40))          # inside the 999-seeded FIFO: suppressed
    assert oracle.move_fft_snr_runtime_avg(early[:150], 160, 16, 10) == (False, -1.0, math.inf, math.inf)
    f, i, sn = oracle.specific_fft_snr_fix_avg(s, (595, 605), 16, 10, avg)
    assert f and 595 <= i <= 605


def test_tone_estimator_is_unbiased_on_a_pure_tone():
    n = np.arange(4000)
    f = oracle.SYMBOL_RATE / 4 + 1234.5
    r = np.exp(2j * np.pi * f * n / FS)
    fo, _, _ = oracle.tone_freq_estimate(r, [101, 1500], 1184, FS)
    assert np.max(np.abs(fo - f)) < 1e-6


def test_spacing_classification_thresholds():
    pos = np.array([1, 100001, 200003, 310003, 410003], dtype=float)
    ok, a, b, exp, d10, d11 = oracle.classify_spacing(pos, 8, 400)
    assert ok and list(a) == [True, True, False, True] and list(b) == [False, False, True, False] and exp == 410000
    pos[2] += 40                                                             # |diff-100000| = 42 >= floor(40) -> unclassified
    assert not oracle.classify_spacing(pos, 8, 400)[0]
    assert oracle.classify_spacing(pos, 8, 4000)[0]


def test_total_ppm_calculation():
    assert oracle.total_ppm_calculation([math.inf, math.inf]) == math.inf
    assert oracle.total_ppm_calculation([5.0, math.inf]) == math.inf
    assert abs(oracle.total_ppm_calculation([-35.0, 1.0]) - ((1 - 35e-6) * (1 + 1e-6) - 1) * 1e6) < 1e-12


def test_sch_template_properties():
    t = oracle.gsm_SCH_training_sequence_gen(8)
    assert t.shape == (512,) and np.allclose(np.abs(t), 1)
    d = oracle.differential_encode(oracle.SCH_TRAINING_BITS)
    assert d[0] == 0 and d[1] == 0 and d[3] == 1                              # bits 1,0,1,1 against a leading 0
    # a run of equal differential symbols is a tone at +fs_sym/4: pi/2 per symbol once the L=4 pulses overlap fully
    ph = np.unwrap(np.angle(oracle.gmsk_modulate(np.ones(20, dtype=np.int64), 8)))
    assert np.allclose(np.diff(ph[8 * 4::8]), np.pi / 2, atol=1e-12)
    assert abs(oracle.gmsk_q(np.float64(4.0)) - 1) < 1e-15 and oracle.gmsk_q(np.float64(0.0)) == 0 and abs(oracle.gmsk_q(np.float64(2.0)) - 0.5) < 1e-12


def test_fcch_of_the_generator_is_a_quarter_symbol_rate_tone():
    sp = synth.StreamSpec(seed=5, n_samples=30000, snr_db=60.0, start_offset=0.0)
    raw = synth.generate_stream(sp).numpy()
    b = oracle.raw2iq(raw)[:, 0]
    seg = b[100:1100]                                                        # inside the first FCCH burst
    rot = np.angle(np.mean(seg[1:] / seg[:-1]))                              # CW_check.m:6
    assert abs(rot * FS / (2 * np.pi) - oracle.SYMBOL_RATE / 4) < 300
    resid = np.angle(seg[1:] / seg[:-1]) - rot                               # CW_check.m:8: no lost samples
    assert np.max(np.abs(resid)) < 0.2


@pytest.mark.parametrize("seed", ["1", "4"])
def test_oracle_reproduces_committed_pipeline_fixture(seed):
    with open(os.path.join(GOLDEN, "pipeline_golden.json")) as f:
        g = json.load(f)
    c = g["cases"][seed]
    spec = synth.random_spec(int(seed), g["n_samples"])
    raw = synth.generate_stream(spec).numpy()
    assert hashlib.sha256(raw.tobytes()).hexdigest() == c["raw_sha256"], "synthetic generator drifted"
    res = oracle.calibrate_stream(raw, spec.carrier_freq, oracle.gsm_SCH_training_sequence_gen(8), oracle.fir1(46, 200e3 / FS))
    assert res["coarse_pos"].tolist() == c["coarse_pos"] and res["fcch_pos"].tolist() == c["fcch_pos"]
    assert res["pos_info"].tolist() == c["pos_info"]
    assert [float(x).hex() for x in res["sampling_ppm"]] == c["sampling_ppm"]
    assert abs(res["total_carrier_ppm"] - c["total_carrier_ppm"]) < 1e-9
    # sanity against the injected truth (not parity): the estimator is biased by about -1 ppm (SURVEY Appendix B)
    assert abs(res["total_sampling_ppm"] - spec.sampling_ppm) < 1.2
    assert abs(res["total_carrier_ppm"] - spec.carrier_ppm) < 1.6
    types = res["pos_info"][:, 1]
    assert set(types.tolist()) <= {0.0, 1.0, 2.0} and (types == 0).sum() >= 5


def test_oracle_sentinel_paths():
    rng = np.random.default_rng(3)
    noise = rng.standard_normal(20000) + 1j * rng.standard_normal(20000)
    pos, snr = oracle.FCCH_coarse_position(noise, 8)
    assert pos.tolist() == [-1.0] and snr.tolist() == [-1.0]
    f = oracle.FCCH_fine_correction(noise, pos, 8, 957.4e6)
    assert f[0].tolist() == [-1.0] and f[1] is None and f[2] == math.inf and f[3] == math.inf
    s = oracle.SCH_corr_rate_correction(np.array([-1.0]), f[0], np.ones(512, complex), 8)
    assert s[0].tolist() == [[-1.0, -1.0]] and s[1] is None and s[2] == math.inf
    c = oracle.carrier_correct_post_SCH(np.array([-1.0]), s[0], 8, 957.4e6)
    assert c == (None, math.inf)
    with pytest.raises(IndexError):
        oracle.FCCH_coarse_position(noise[:3000], 8)          # s(1:3594) would raise in MATLAB


# ---- SURVEY 8(f) rows 2 and 4: demodulator family -------------------------------------------------------------------
def test_normal_training_sequences_follow_the_reference_table():
    nts = oracle.gsm_normal_training_sequence_gen(8)
    assert nts.shape == (208, 8) and np.allclose(np.abs(nts), 1.0)
    assert oracle.NORMAL_TRAINING_BITS.shape == (8, 26)
    assert oracle.NORMAL_TRAINING_BITS[0].tolist() == [0, 0, 1, 0, 0, 1, 0, 1, 1, 1, 0, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 1, 0, 1, 1, 1]
    for q in range(8):                                # column q: differential encoding against a leading 0, own modulator state
        ref = oracle.gmsk_modulate(oracle.differential_encode(oracle.NORMAL_TRAINING_BITS[q]), 8)
        assert np.array_equal(nts[:, q], ref)
    gram = np.abs(nts.conj().T @ nts) / 208           # the eight sequences are mutually distinguishable
    assert np.all(gram[~np.eye(8, dtype=bool)] < 0.8)


@pytest.mark.parametrize("osr,noise", [(8, 0.0), (8, 0.25), (4, 0.2), (1, 0.1)])
def test_gmsk_viterbi_inverts_the_modulator(osr, noise):
    rng = np.random.default_rng(osr)
    bits = rng.integers(0, 2, 160)
    x = oracle.gmsk_modulate(bits, osr)
    x = x + noise * (rng.standard_normal(len(x)) + 1j * rng.standard_normal(len(x)))
    out = oracle.gmsk_viterbi_demod(x, osr, 30)
    assert out[:30].tolist() == [0] * 30              # TracebackDepth delay
    assert np.array_equal(out[30:], bits[:130])


def test_fcch_demod_on_a_pure_tone():
    osr, n = 8, 6000
    f = oracle.SYMBOL_RATE / 4 + 1234.5
    s = np.exp(2j * np.pi * f * np.arange(n) / FS + 0.3j)
    pinfo = np.array([[101.0, 0.0], [2001.0, 0.0], [3000.0, 1.0]])
    d = oracle.FCCH_demod(s, pinfo, osr, 957.4e6)
    assert len(d["freq"]) == 2 and np.max(np.abs(d["freq"] - f)) < 1e-6
    assert abs(d["carrier_ppm"] - 1e6 * 1234.5 / 957.4e6) < 1e-9
    assert d["max_idx"].tolist() == [round(f * 1184 / FS)] * 2 and np.all(d["snr"] > 5)
    assert oracle.FCCH_demod(s, np.array([[-1.0, -1.0]]), osr, 957.4e6) is None


def test_sch_demod_finds_the_training_sequence():
    osr = 4
    rng = np.random.default_rng(11)
    bits = rng.integers(0, 2, 148 + 90)
    b0 = 30
    bits[b0 + 42:b0 + 42 + 64] = oracle.SCH_TRAINING_BITS
    prev = np.concatenate([[1], bits[:-1]])
    tx = oracle.gmsk_modulate((bits == prev).astype(np.int64), osr) * np.exp(0.7j)
    tx = tx + 0.02 * (rng.standard_normal(len(tx)) + 1j * rng.standard_normal(len(tx)))
    d = oracle.SCH_demod(tx, np.array([[b0 * osr + 1.0, 1.0]]), oracle.gsm_SCH_training_sequence_gen(osr), osr)
    assert d["demod_bits"].shape == (1, 148) and d["corr_val"].shape == (1, 85)
    assert d["corr_val"][0].argmax() == 42 and d["corr_val"][0].max() == 64
    sent = (bits == prev).astype(np.int64)[b0:b0 + 148]
    assert np.mean(d["demod_bits"][0] == sent) > 0.97
    # bits_to_decoder = abs(diff([0 ~demod_bits])) (:97): its running XOR gives ~demod_bits back
    assert np.array_equal(np.cumsum(d["bits_to_decoder"][0]) % 2, 1 - d["demod_bits"][0])
    with pytest.raises(IndexError):
        oracle.SCH_demod(tx, np.array([[len(tx) - 100.0, 1.0]]), oracle.gsm_SCH_training_sequence_gen(osr), osr)


def test_bcch_demod_identifies_the_training_sequence_code():
    import dataclasses
    spec = dataclasses.replace(synth.random_spec(2, 1020000), tsc=5)
    raw = synth.generate_stream(spec).numpy()
    res = oracle.calibrate_stream(raw, spec.carrier_freq, oracle.gsm_SCH_training_sequence_gen(8), oracle.fir1(46, 200e3 / FS))
    nts = oracle.gsm_normal_training_sequence_gen(8)
    ppm, idx, mag = oracle.BCCH_demod(res["r_final"], res["pos_info"], nts, 8, spec.carrier_freq)
    assert idx == 6 and mag.shape == (8, 4) and abs(ppm) < 1e-6      # r_final is already carrier-corrected
    assert oracle.BCCH_demod(res["r_final"], np.array([[-1.0, -1.0]]), nts, 8, spec.carrier_freq) == (-1.0, -1, None)


# ---- the reference's own manual checks, as assertions (SURVEY section 4) ---------------------------------------------------------
def test_diff_gmsk_mod_demod_script():
    """test_diff_GMSK_mod_demod.m:16-45: 13 bits -> differential encoding against a leading 1 -> GMSK -> Viterbi demodulation with
    TracebackDepth 5 -> the script displays the differences (all zero when the chain is consistent)."""
    s_bit = np.array([0, 1, 0, 1, 1, 0, 1, 0, 1, 1, 0, 1, 1])
    gmsk_s_bit = 1 - np.abs(np.diff(np.concatenate([[1], s_bit])))            # :19
    s = oracle.gmsk_modulate(gmsk_s_bit, 8)                                   # :21
    gmsk_r_bit = oracle.gmsk_viterbi_demod(s, 8, 5)[5:]                       # :34-35
    assert np.array_equal(gmsk_r_bit, gmsk_s_bit[:len(gmsk_r_bit)])           # :37
    r_bit = 1 - gmsk_r_bit                                                    # :39-43: running XOR from 0
    r_bit = np.cumsum(r_bit) % 2
    # the script encodes against a leading 1 but decodes from 0, so its last display is the complement pattern of s_bit
    assert np.array_equal(1 - r_bit, s_bit[:len(r_bit)]) or np.array_equal(r_bit, s_bit[:len(r_bit)])


def test_online_reestimation_after_correction_is_zero():
    """The commented 'test on line' blocks (FCCH_fine_correction.m:167-183, carrier_correct_post_SCH.m:131-153): re-running the
    tone estimator on the corrected stream must give the target fs_sym/4."""
    spec = synth.random_spec(3, 1020000)
    raw = synth.generate_stream(spec).numpy()
    r = oracle.fir_filter(oracle.fir1(46, 200e3 / FS), oracle.raw2iq(raw)[:, 0])
    pos, _ = oracle.FCCH_coarse_position(r[::64], 8)
    fpos, r1, _, cppm1 = oracle.FCCH_fine_correction(r, pos, 8, spec.carrier_freq)
    fo, _, _ = oracle.tone_freq_estimate(r1, fpos, 1184, FS)
    assert abs(oracle.matlab_mean(fo) - oracle.SYMBOL_RATE / 4) < 1e-6 and abs(cppm1) > 1e-3
    pinfo, r2, _ = oracle.SCH_corr_rate_correction(r1, fpos, oracle.gsm_SCH_training_sequence_gen(8), 8)
    r3, _ = oracle.carrier_correct_post_SCH(r2, pinfo, 8, spec.carrier_freq)
    fo3, _, _ = oracle.tone_freq_estimate(r3, pinfo[pinfo[:, 1] == 0, 0], 1184, FS)
    assert abs(oracle.matlab_mean(fo3) - oracle.SYMBOL_RATE / 4) < 1e-6


# ---- fixtures lifted from / generated with the reference tree (oracle/make_golden.py) ---------------------------------------------
def test_training_bit_tables_match_the_reference_literals():
    """tests/golden/training_bits.json is PARSED from gsm_SCH_training_sequence_gen.m:17-19 and
    gsm_normal_training_sequence_gen.m:17-24; every hand-typed copy of the tables must equal it."""
    with open(os.path.join(GOLDEN, "training_bits.json")) as f:
        g = json.load(f)
    sch, nts = g["sch_extended_training_sequence"]["bits"], g["normal_training_sequences"]["bits"]
    assert oracle.SCH_TRAINING_BITS.tolist() == sch and list(synth.SCH_TRAINING_BITS) == sch
    assert oracle.NORMAL_TRAINING_BITS.tolist() == nts and [list(r) for r in synth.NORMAL_TRAINING_BITS] == nts


def test_library_training_sequences_use_the_reference_bits(built_lib):
    """The two generators are host code (no GPU needed): their embedded bit tables must be the reference's."""
    import gsmcal
    with open(os.path.join(GOLDEN, "training_bits.json")) as f:
        g = json.load(f)
    sch = np.array(g["sch_extended_training_sequence"]["bits"])
    ref = oracle.gmsk_modulate(oracle.differential_encode(sch), 8)
    assert np.max(np.abs(gsmcal.gsm_SCH_training_sequence_gen(8) - ref)) < 1e-12
    nts = gsmcal.gsm_normal_training_sequence_gen(8)
    for q, bits in enumerate(g["normal_training_sequences"]["bits"]):
        ref = oracle.gmsk_modulate(oracle.differential_encode(np.array(bits)), 8)
        assert np.max(np.abs(nts[:, q] - ref)) < 1e-12


def test_oracle_reproduces_committed_demod_fixture():
    import dataclasses
    with open(os.path.join(GOLDEN, "demod_golden.json")) as f:
        g = json.load(f)
    c = g["cases"]["2"]
    spec = dataclasses.replace(synth.random_spec(2, g["n_samples"]), tsc=c["tsc"])
    raw = synth.generate_stream(spec).numpy()
    assert hashlib.sha256(raw.tobytes()).hexdigest() == c["raw_sha256"], "synthetic generator drifted"
    tpl = oracle.gsm_SCH_training_sequence_gen(8)
    res = oracle.calibrate_stream(raw, spec.carrier_freq, tpl, oracle.fir1(46, 200e3 / FS))
    r3, pinfo = res["r_final"], res["pos_info"]
    keep = np.array([not (t == 1 and p - 64 + 1552 - 1 > len(r3)) for p, t in pinfo])
    sd = oracle.SCH_demod(r3, pinfo[keep], tpl, 8)
    assert ["".join(str(int(b)) for b in row) for row in sd["demod_bits"]] == c["sch_demod_bits"]
    assert sd["corr_val"].argmax(axis=1).tolist() == c["sch_corr_argmax"] and sd["corr_val"].max(axis=1).tolist() == c["sch_corr_peak"]
    fd = oracle.FCCH_demod(r3, pinfo, 8, spec.carrier_freq)
    assert fd["max_idx"].tolist() == c["fcch_max_idx"]
    assert np.max(np.abs(fd["freq"] - np.array(c["fcch_freq"]))) < 1e-6 and np.max(np.abs(fd["snr"] - np.array(c["fcch_snr"]))) < 1e-9
    ppm, idx, _ = oracle.BCCH_demod(r3, pinfo, oracle.gsm_normal_training_sequence_gen(8), 8, spec.carrier_freq)
    assert idx == c["bcch_idx"] == c["tsc"] + 1 and abs(ppm - c["bcch_carrier_ppm"]) < 1e-9


def test_algorithm_constants_match_the_reference_source():
    """tests/golden/reference_constants.json is extracted by regular expressions from the defining lines of the .m files."""
    with open(os.path.join(GOLDEN, "reference_constants.json")) as f:
        g = json.load(f)
    for k, v in oracle.CONSTANTS.items():
        assert float(v) == g[k]["value"], (k, v, g[k])
    assert g["min_bursts_sch"]["value"] == oracle.CONSTANTS["min_bursts"] and g["len_fcch_cw"]["value"] == oracle.LEN_FCCH_CW


@pytest.mark.parametrize("gaps,flagged", [((10, 10, 10, 11, 10, 10), {5}), ((10, 10, 10, 10, 11, 10), {1, 6}), ((10, 10, 10, 10, 10), set())])
def test_pos_info_rows_known_answer(gaps, flagged):
    """K10 by hand (SCH_corr_rate_correction.m:138-181): templates planted exactly where the burst format puts them, so the peak is
    the centre lag, e = 0, and every row of pos_info can be written down: per SCH i the FCCH row (SCH-10336, 0), the SCH row
    (SCH-336, 1), and four BCCH rows (+k*10000, 2) after the SCH bursts flagged by the 11-frame gaps (b_idx+1 and b_idx-4)."""
    osr, frame = 8, 10000
    ts = oracle.gsm_SCH_training_sequence_gen(osr)
    fcch = np.cumsum([2001] + [g * frame for g in gaps]).astype(np.float64)
    n = int(fcch[-1]) + 10336 + 512 + 5 * frame
    s = np.zeros(n, dtype=np.complex128)
    for p in fcch:
        t0 = int(p) + 10336                              # training_sp (1-based)
        s[t0 - 1:t0 - 1 + 512] = ts
    pos_info, r, ppm = oracle.SCH_corr_rate_correction(s, fcch, ts, osr)
    assert ppm == 0.0 and np.array_equal(r, s)           # e == 0: no interp1 (:120)
    rows = []
    for i, p in enumerate(fcch, 1):
        sch = p + 10336
        rows.append([sch - 10336, 0.0])
        rows.append([sch - 336, 1.0])
        if i in flagged:
            rows += [[sch - 336 + k * frame, 2.0] for k in (1, 2, 3, 4)]
    assert pos_info.tolist() == rows


def test_fine_correction_known_answer_on_planted_tones():
    """K5-K8 by hand (FCCH_fine_correction.m:32-165): six 1184-sample tones planted 10/11 frames apart in weak noise.  The window
    that covers a tone completely has the largest max-bin power, so FCCH_pos are the planted starts; the spacing is nominal, so
    e = 0 and the regridded positions (:127-133) equal the found ones; the carrier error follows from the tone frequency."""
    osr, frame, n_tone = 8, 10000, 1184
    f_tone = oracle.SYMBOL_RATE / 4 + 2500.0
    rng = np.random.default_rng(5)
    starts = np.cumsum([30001] + [g * frame for g in (10, 10, 11, 10, 10)])
    n = int(starts[-1]) + 3 * frame
    s = 1e-3 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    for p in starts:
        k = np.arange(n_tone)
        s[p - 1:p - 1 + n_tone] += np.exp(2j * np.pi * f_tone * (p - 1 + k) / FS)
    base = np.round((starts - 1) / osr) + 1 + np.array([3, -7, 0, 11, -20, 5])          # coarse guesses, within +-64 symbols
    fpos, r, sppm, cppm = oracle.FCCH_fine_correction(s, base, osr, 957.4e6)
    assert fpos.tolist() == starts.astype(float).tolist()
    assert sppm == 0.0 and len(r) == n
    assert abs(cppm - 1e6 * 2500.0 / 957.4e6) < 1e-3                                   # the 1e-3 noise floor moves the estimate by ~0.03 Hz
    # r = s .* exp(1i*n*comp) (:163-165): the tone sits on fs_sym/4 afterwards
    fo, _, _ = oracle.tone_freq_estimate(r, fpos, n_tone, FS)
    assert abs(oracle.matlab_mean(fo) - oracle.SYMBOL_RATE / 4) < 1e-6 and np.max(np.abs(fo - oracle.SYMBOL_RATE / 4)) < 2.0   # mean exact, bursts within noise


# ---- SURVEY Appendix A paths that random captures rarely reach: the deliberate fixtures do drive the oracle there -------------
def test_appendix_a_fixtures_take_their_branches():
    import appendix_a_fixtures as fx
    tpl = oracle.gsm_SCH_training_sequence_gen(8)
    args, took = fx.fine_overrun_drops_to_four()
    assert took(oracle.FCCH_fine_correction(*args))                 # FCCH_fine_correction.m:135-137,142
    args, took = fx.fine_snr_gate_return()
    info = {}
    res = oracle.FCCH_fine_correction(*args, info)
    assert took(res) and np.min(info["fine_gate_snr"]) < 5.0 - 3.0  # :192-196, well below the 5 dB gate
    args, took, _ = fx.sch_e_zero_skips_interp1(tpl)
    assert took(oracle.SCH_corr_rate_correction(*args))             # SCH_corr_rate_correction.m:120-128
    args, took = fx.sch_last_slot_does_not_fit(tpl)
    assert took(oracle.SCH_corr_rate_correction(*args))             # :153-159
    args, took = fx.sch_bcch_rows_run_out(tpl)
    assert took(oracle.SCH_corr_rate_correction(*args))             # :167-178
