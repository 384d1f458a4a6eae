"""gsmcal_calibrate_cell_batch: the carrier fit, then SCH_demod of every SCH burst with the fitted residual removed, then SCH decoding.
CPU: the flag and its export, argument checks without a launch, the MEX gateway against the stub, known answers of the restatement in
cell_sync_oracle.py and its accuracy on the oracle chain at the reference's 0.47 s.  GPU: parity with the restatement on the GPU's own
r_correct and carrier records and with the oracle chain, byte-identical outputs and launches of the existing calls, drifting 10 s
streams, two dongles aligned at 0.47 s, stream independence and device input, the stage timing, the MEX gateway end
to end and the rtl_tcp ingest."""
import ctypes as C
import dataclasses
import math
import os
import subprocess

import numpy as np
import pytest

import carrier_fit_oracle as CF
import cell_sync_oracle as CS
import gsmcal_oracle as oracle
import sch_decode_oracle as S
from gsmcal import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MEX = os.path.join(ROOT, "multi-rtl-sdr-calibration_b200", "mex")
FS = oracle.SYMBOL_RATE * 8
CARRIER = 957.4e6
N_SYNC = 1020000                       # gsm_sync_demod.m's 102 frames, 0.47 s
N_10S = 21666667
# Seeds that decode every SCH row in a 40-seed oracle run at 0.47 s (DESIGN.md 6b): random_spec(seed, N_SYNC), bsic = seed % 64,
# fn0 = 51 * (seed * 7919 % 50000).  frame_clock_start - truth is -23 samples on all of them: the 47-tap channel filter's group delay.
SEEDS = (1, 11, 28)
FILTER_DELAY = -23.0
PAIR_SEED = 72                         # the second dongle of the sch-decode tests' pair, on seed 11's cell


def _cell_spec(seed, n=N_SYNC):
    return dataclasses.replace(synth.random_spec(seed, n), bsic=seed % 64, fn0=51 * (seed * 7919 % 50000))


def _vp(a):
    return a.ctypes.data_as(C.c_void_p)


# ---- CPU: ABI ------------------------------------------------------------------------------------------------------------------
def test_uncorrected_flag_and_export(built_lib):
    from gsmcal import _lib, api
    hdr = open(os.path.join(ROOT, "include", "gsmcal.h")).read()
    assert hdr.split("#define GSMCAL_SCHDEC_UNCORRECTED")[1].split()[0] == "16"
    assert api.SCHDEC_UNCORRECTED == 16 == CS.UNCORRECTED
    assert all(api.SCHDEC_UNCORRECTED & v == 0 for v in (api.SCHDEC_NO_POS_INFO, api.SCHDEC_NO_R_CORRECT, api.SCHDEC_NONE, api.SCHDEC_DISAGREE))
    assert "gsmcal_calibrate_cell_batch" in _lib.SIGNATURES
    out = subprocess.run(["nm", "-D", "--defined-only", built_lib], capture_output=True, text=True).stdout
    assert " T gsmcal_calibrate_cell_batch" in out


def _call(raw, n_iq, D, osr=8, carrier=True, dec=True):
    from gsmcal._lib import CarrierFitResult, SchDecodeResult, StreamResult, lib
    tpl = np.ones(64 * max(osr, 1), dtype=np.complex128)
    coef = oracle.fir1(46, 200e3 / FS)
    n = max(D, 1)
    res, cf, sd = (StreamResult * n)(), (CarrierFitResult * n)(), (SchDecodeResult * n)()
    return lib().gsmcal_calibrate_cell_batch(_vp(raw), 0, n_iq, D, CARRIER, _vp(tpl), _vp(coef), len(coef), osr, 8, C.cast(res, C.c_void_p),
                                             None, None, None, None, None, C.cast(cf, C.c_void_p) if carrier else None, None, None, None,
                                             C.cast(sd, C.c_void_p) if dec else None, *[None] * 8)


def test_cell_batch_argument_errors_launch_nothing(built_lib):
    import gsmcal
    from gsmcal import api
    from gsmcal._lib import lib
    raw = np.zeros((1, 2 * 300000), dtype=np.uint8)
    n0 = api.launch_count()
    for osr in (0, 9, 1, 4):
        assert _call(raw, 300000, 1, osr=osr) == -1
    assert b"oversampling_ratio must be 8" in lib().gsmcal_last_error()
    assert _call(raw, 300000, 1, carrier=False) == -1
    assert _call(raw, 300000, 1, dec=False) == -1
    assert b"null carrier or dec" in lib().gsmcal_last_error()
    assert _call(raw, 300000, 0) == -1
    assert _call(raw, 1000, 1) == -4                       # shorter than the 23 frames of the coarse search: GSMCAL_ERR_RANGE
    tpl, coef = np.ones(512, complex), oracle.fir1(46, 0.09)
    for kw in (dict(sch_decode=True), dict(sch_decode=True, sch_timing=True), dict(sch_decode=True, carrier_fit=True, sch_timing=True)):
        with pytest.raises(ValueError):
            gsmcal.calibrate_batch(raw, CARRIER, tpl, coef, **kw)
    assert api.launch_count() == n0


def test_cell_batch_needs_a_device(built_lib):
    import gsmcal
    if gsmcal.device_count() > 0:
        pytest.skip("a CUDA device is present")
    raw = np.zeros((1, 2 * 300000), dtype=np.uint8)
    assert _call(raw, 300000, 1) == -2
    with pytest.raises(gsmcal.GsmcalError) as e:
        gsmcal.calibrate_batch(raw, CARRIER, np.ones(512, complex), oracle.fir1(46, 0.09), carrier_fit=True, sch_decode=True)
    assert e.value.code == -2


def _gateway(tmp_path, built_lib, body, name="h"):
    src = tmp_path / f"{name}.c"
    src.write_text(body)
    exe = tmp_path / name
    libdir = os.path.dirname(built_lib)
    subprocess.run(["gcc", "-std=c11", "-Wno-unused-function", "-DGSMCAL_MEX_gsm_calibrate_cell_batch", f"-I{MEX}/stub", f"-I{ROOT}/include",
                    str(src), os.path.join(MEX, "gsmcal_mex.c"), f"-L{libdir}", "-lgsmcal", f"-Wl,-rpath,{libdir}", "-lm", "-o", str(exe)], check=True)
    return exe


def test_cell_gateway_compiles_against_stub(tmp_path):
    obj = tmp_path / "g.o"
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Wno-unused-function", "-c", "-DGSMCAL_MEX_gsm_calibrate_cell_batch", f"-I{MEX}/stub",
                    f"-I{ROOT}/include", os.path.join(MEX, "gsmcal_mex.c"), "-o", str(obj)], check=True)
    sym = subprocess.run(["nm", str(obj)], capture_output=True, text=True).stdout
    assert " T mexFunction" in sym and " U gsmcal_calibrate_cell_batch" in sym and " U gsmcal_calibrate_carrier_fit_batch" not in sym
    assert "gsm_calibrate_cell_batch" in open(os.path.join(MEX, "Makefile.mex")).read()


@pytest.mark.parametrize("nlhs,nrhs", [(7, 4), (6, 3), (6, 5)])
def test_cell_gateway_usage_errors(built_lib, tmp_path, nlhs, nrhs):
    exe = _gateway(tmp_path, built_lib, r'''#include "mex.h"
int main(void) {
    size_t dims[2] = {600000, 1};
    mxArray *raw = mxCreateNumericArray(2, dims, mxUINT8_CLASS, mxREAL);
    mxArray *t = mxCreateDoubleMatrix(512, 1, mxCOMPLEX), *c = mxCreateDoubleMatrix(1, 47, mxREAL);
    mxArray *out[7]; const mxArray *rhs[5] = {raw, mxCreateDoubleScalar(957.4e6), t, c, c};
    mexFunction(%d, out, %d, rhs);
    return 0;
}
''' % (nlhs, nrhs))
    p = subprocess.run([str(exe)], capture_output=True, text=True)
    assert p.returncode == 3 and "gsmcal:nargin" in p.stderr


# ---- CPU: known answers of the restatement ------------------------------------------------------------------------------------
def _burst_capture(df_hz, bsic=45, fn0=51 * 2000, seed=5):
    """a clean capture whose SCH bursts carry (bsic, fn) and a carrier offset of df_hz; returns (r, 1-based positions of its SCH bursts,
    the spec).  No channel filter: the burst starts exactly on its slot."""
    spec = synth.StreamSpec(seed=seed, n_samples=300000, bsic=bsic, fn0=fn0, snr_db=40.0, carrier_ppm=df_hz / CARRIER * 1e6)
    raw = synth.generate_stream(spec).numpy()
    r = oracle.raw2iq(raw)[:, 0]
    r = r - np.mean(r)
    frames = [f for f in range(spec.n_samples // synth.FRAME - 1) if f % 51 % 10 == 1 and f % 51 <= 41]
    return r, np.array([f * synth.FRAME + 1.0 for f in frames]), spec


def test_zero_residual_is_sch_demod():
    tpl = oracle.gsm_SCH_training_sequence_gen(8)
    r, pos, _ = _burst_capture(800.0)
    pinfo = np.stack([pos, np.ones_like(pos)], 1)
    out = CS.cell_sync(r, pinfo, 0.0, 0.0, dict(flags=CF.FEW), tpl)
    ref = oracle.SCH_demod(r, pinfo, tpl, 8)
    for k in ("demod_bits", "bits_to_decoder", "corr_val"):
        np.testing.assert_array_equal(out[k], ref[k])
    assert np.all(np.isnan(out["df"])) and out["rec"]["flags"] & CS.UNCORRECTED


def test_constant_phase_cancels_in_the_equaliser():
    tpl = oracle.gsm_SCH_training_sequence_gen(8)
    r, pos, _ = _burst_capture(1000.0)
    sp = int(pos[0]) - 8 * 8
    x = r[sp - 1:sp - 1 + CS.N]
    a = CS.demod_window(x, tpl, 1000.0)
    for phi in (0.7, -2.9):
        b = CS.demod_window(x * np.exp(1j * phi), tpl, 1000.0)
        for k in ("demod_bits", "bits_to_decoder", "corr_val"):
            np.testing.assert_array_equal(a[k], b[k])


def test_planted_offset_fails_uncorrected_and_decodes_corrected():
    tpl = oracle.gsm_SCH_training_sequence_gen(8)
    r, pos, spec = _burst_capture(1000.0)
    sp = int(pos[1]) - 8 * 8
    x = r[sp - 1:sp - 1 + CS.N]
    raw_row = CS.demod_window(x, tpl, 0.0)
    fixed = CS.demod_window(x, tpl, 1000.0)
    fn = spec.fn0 + int(pos[1] - 1) // synth.FRAME
    assert S.decode_row(raw_row["demod_bits"], raw_row["corr_val"], True)[3] != 0
    assert S.decode_row(fixed["demod_bits"], fixed["corr_val"], True) == (fn, 45, 0, 0)


def test_row_time_and_residual_follow_the_carrier_fit():
    e1, e2 = -14e-6, 3e-6
    p = 402353.0
    assert CS.row_time(p, e1, e2) == CF.row_time(p + 74 * 8 - CF.OFF - CF.HALF, e1, e2)
    car = dict(freq_hz=CF.F_NOM + 1000.0, drift_hz_per_s=50.0, t_mean=CS.row_time(p, e1, e2))
    assert CS.row_residual(p, e1, e2, car) == 1000.0
    later = CS.row_residual(p + 10 * 10000, e1, e2, car)
    assert abs(later - (1000.0 + 50.0 * 10 * 10000 * (1 + e1) * (1 + e2) / FS)) < 1e-9


@pytest.fixture(scope="module")
def coef():
    return oracle.fir1(46, 200e3 / FS)


@pytest.fixture(scope="module")
def tpl():
    return oracle.gsm_SCH_training_sequence_gen(8)


@pytest.fixture(scope="module")
def oracle_chain(coef, tpl):
    """the oracle chain and the restatement on SEEDS at 0.47 s"""
    specs = [_cell_spec(s) for s in SEEDS]
    raw = synth.generate_batch(specs).numpy()
    cals = [oracle.calibrate_stream(raw[d], CARRIER, tpl, coef) for d in range(len(specs))]
    return specs, raw, cals, [CS.cell_reference(c, CARRIER, tpl) for c in cals]


def test_restatement_decodes_short_captures(oracle_chain):
    specs, _, _, refs = oracle_chain
    for s, ref in zip(specs, refs):
        rec = ref["rec"]
        assert rec["bsic"] == s.bsic and rec["flags"] == 0
        assert rec["n_agree"] >= rec["n_sch"] - 1 and rec["n_sch"] >= 9
        assert rec["frame_clock_start"] - synth.true_frame_clock_start(s) == FILTER_DELAY
        assert np.all(np.abs(ref["df"] - 1000.0) < 60.0)                # the about +1 kHz total_carrier_ppm leaves
        assert np.median(ref["rows"]["hamming"]) <= 2


# ---- GPU -----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def batch(gpu, coef, tpl):
    """_specs()'s mix (random coded bits, a noise-only stream, one without r_correct) and streams that carry a cell"""
    from test_gpu_demod_batch import _specs
    specs = _specs() + [_cell_spec(s) for s in SEEDS + (38, 3, 4)]
    raw = synth.generate_batch(specs).numpy()
    got = gpu.calibrate_batch(raw, CARRIER, tpl, coef, carrier_fit=True, sch_decode=True)
    return specs, raw, got


def _r_correct(gpu, raw, coef, tpl):
    D, n_iq = raw.shape[0], raw.shape[1] // 2
    r = np.zeros((D, n_iq), dtype=np.complex128)
    res = gpu.calibrate_batch(raw, CARRIER, tpl, coef, r_correct=r)
    return r, res


def _check_rows(g, ref):
    """the GPU's cell / sch entries against cell_sync's output for one stream"""
    c, s = g["cell"], g["sch"]
    for k in ("n_crc_ok", "n_agree", "flags", "bsic", "fn_first"):
        assert c[k] == ref["rec"][k], k
    assert np.float64(c["frame_clock_start"]).tobytes() == np.float64(ref["rec"]["frame_clock_start"]).tobytes()
    np.testing.assert_array_equal(s["sch_ok"], ref["sch_ok"])
    for k in ("demod_bits", "corr_val"):
        np.testing.assert_array_equal(s[k], ref[k])
    for a, b in (("fn", "fn"), ("bsic_rows", "bsic"), ("hamming", "hamming"), ("row_flags", "row_flags")):
        np.testing.assert_array_equal(c[a], ref["rows"][b])
    assert np.array_equal(np.isnan(c["df"]), np.isnan(ref["df"]))
    ok = ~np.isnan(ref["df"])
    if ok.any():
        assert np.max(np.abs(c["df"][ok] - ref["df"][ok])) < 1e-9


def _restate(g, r_row, tpl):
    """cell_sync on the GPU's own r_correct and carrier record of one stream"""
    car = dict(g["carrier"])
    e1, e2 = g["sampling_ppm"][0] * 1e-6, g["sampling_ppm"][1] * 1e-6
    return CS.cell_sync(r_row[:g["r_len"][2]], g["pos_info"], e1, e2, car, tpl)


@pytest.mark.gpu
def test_cell_matches_the_restatement_on_the_gpus_carrier_records(gpu, batch, coef, tpl):
    specs, raw, got = batch
    r, _ = _r_correct(gpu, raw, coef, tpl)
    ran = 0
    for d, g in enumerate(got):
        if g["cell"]["fn"] is None:
            assert g["sch"] is None and g["cell"]["df"] is None
            assert g["cell"]["flags"] in (S.NO_POS_INFO, S.NO_R_CORRECT) and g["cell"]["flags"] == g["carrier"]["flags"]
            continue
        _check_rows(g, _restate(g, r[d], tpl))
        ran += 1
    assert ran >= 8
    flags = [g["cell"]["flags"] for g in got]
    assert S.NO_POS_INFO in flags and S.NO_R_CORRECT in flags


@pytest.mark.gpu
def test_cell_matches_the_oracle_chain(batch, coef, tpl):
    specs, raw, got = batch
    for d in [i for i, s in enumerate(specs) if s.bsic is not None][:2]:
        ref = CS.cell_reference(oracle.calibrate_stream(raw[d], CARRIER, tpl, coef), CARRIER, tpl)
        _check_rows(got[d], ref)


@pytest.mark.gpu
def test_cell_recovers_every_synthetic_cell(batch):
    specs, _, got = batch
    n = 0
    for s, g in zip(specs, got):
        if s.bsic is None:
            continue
        c = g["cell"]
        assert c["bsic"] == s.bsic and c["flags"] == 0 and c["n_agree"] >= len(c["fn"]) - 1
        assert c["frame_clock_start"] - synth.true_frame_clock_start(s) == FILTER_DELAY
        n += 1
    assert n == 6


def _raw_outputs(raw, mode):
    """every output of gsmcal_calibrate_batch ('batch'), _carrier_fit_batch ('carrier'), _sch_decode_batch ('decode') or _cell_batch
    ('cell') as bytes, with the launch count"""
    from gsmcal import api
    from gsmcal._lib import CarrierFitResult, DemodResult, SchDecodeResult, StreamResult, lib
    coef = oracle.fir1(46, 200e3 / FS)
    tpl = oracle.gsm_SCH_training_sequence_gen(8)
    D, n_iq = raw.shape[0], raw.shape[1] // 2
    cap = api.max_bursts(n_iq)
    res, cf, sd, dem = (StreamResult * D)(), (CarrierFitResult * D)(), (SchDecodeResult * D)(), (DemodResult * D)()
    arrs = [np.full((D, cap), 7.0), np.full((D, cap), 7.0), np.full((D, cap), 7.0), np.full((D, 6 * cap, 2), 7.0)]
    args = [_vp(raw), 0, n_iq, D, CARRIER, _vp(tpl), _vp(coef), len(coef), 8, 8, C.cast(res, C.c_void_p)] + [_vp(a) for a in arrs] + [None]
    cfr = [np.full((D, cap), 7.0), np.full((D, cap), 7.0), np.full((D, cap), 7, np.uint8)]
    dec = [np.full((D, cap), 7, np.int32), np.full((D, cap), 7, np.int32), np.full((D, cap), 7, np.uint8), np.full((D, cap), 7, np.uint8)]
    rows = [np.zeros((D, cap), np.uint8), np.zeros((D, cap, 148), np.uint8), np.zeros((D, cap, 148), np.uint8), np.zeros((D, cap, 85))]
    n0 = api.launch_count()
    if mode == "batch":
        assert lib().gsmcal_calibrate_batch(*args) == 0
    elif mode == "carrier":
        assert lib().gsmcal_calibrate_carrier_fit_batch(*args, C.cast(cf, C.c_void_p), *[_vp(a) for a in cfr]) == 0
    elif mode == "decode":
        assert lib().gsmcal_calibrate_sch_decode_batch(*args, C.cast(dem, C.c_void_p), *[_vp(a) for a in rows], None, None, None, None, None,
                                                       C.cast(sd, C.c_void_p), *[_vp(a) for a in dec]) == 0
    else:
        df = np.full((D, cap), 7.0)
        assert lib().gsmcal_calibrate_cell_batch(*args, C.cast(cf, C.c_void_p), *[_vp(a) for a in cfr], C.cast(sd, C.c_void_p), _vp(rows[0]),
                                                 _vp(rows[1]), _vp(rows[3]), _vp(df), *[_vp(a) for a in dec]) == 0
    n = api.launch_count() - n0
    return dict(batch=(bytes(res), [a.tobytes() for a in arrs]), carrier=(bytes(cf), [a.tobytes() for a in cfr]),
                decode=(bytes(sd), [a.tobytes() for a in dec])), n


@pytest.mark.gpu
def test_existing_calls_unchanged_and_carrier_records_identical(gpu, batch):
    raw = batch[1]
    plain, n_plain = _raw_outputs(raw, "batch")
    car, n_car = _raw_outputs(raw, "carrier")
    cell, n_cell = _raw_outputs(raw, "cell")
    dec, n_dec = _raw_outputs(raw, "decode")
    again, n_again = _raw_outputs(raw, "batch")
    assert plain["batch"] == car["batch"] == cell["batch"] == dec["batch"] == again["batch"]
    assert cell["carrier"] == car["carrier"]                                 # the carrier fit, byte for byte
    assert n_plain == n_again and n_car == n_plain + 3
    assert n_cell == n_car + 3                     # one stream group: fft(template) in the set-up, SCH_demod less df, SCH decoding
    assert cell["decode"] != dec["decode"]                                   # the correction changes what decodes


@pytest.mark.gpu
def test_drifting_full_length_streams_decode_every_row(gpu, coef, tpl):
    torch = pytest.importorskip("torch")
    specs = [dataclasses.replace(_cell_spec(101, N_10S), carrier_drift_ppm_per_s=0.02),
             dataclasses.replace(_cell_spec(132, N_10S), bsic=101 % 64, carrier_drift_ppm_per_s=-0.02)]
    raw = synth.generate_batch(specs, device="cuda")
    torch.cuda.synchronize()
    got = gpu.calibrate_batch(None, CARRIER, tpl, coef, device_ptr=raw.data_ptr(), n_iq=N_10S, n_streams=2, carrier_fit=True, sch_decode=True)
    for s, g in zip(specs, got):
        c = g["cell"]
        assert len(c["fn"]) > 150 and c["flags"] == 0 and c["bsic"] == s.bsic
        assert c["n_agree"] >= np.sum(c["row_flags"] != S.WINDOW) - 2
        assert abs(c["frame_clock_start"] - synth.true_frame_clock_start(s) - FILTER_DELAY) <= 1.0
        car = g["carrier"]
        b, t = car["drift_hz_per_s"], car["t"][np.isfinite(car["t"])]
        assert abs(b - s.carrier_drift_ppm_per_s * CARRIER * 1e-6) < 5 * car["rms_hz"] / math.sqrt(np.sum((t - car["t_mean"]) ** 2)) + 0.01
        span = c["df"][-1] - c["df"][0]                                   # the drift term: b over the SCH rows' time span
        assert abs(span / b - (g["pos_info"][g["pos_info"][:, 1] == 1, 0][-1] - g["pos_info"][g["pos_info"][:, 1] == 1, 0][0]) / FS) < 0.01
    want = synth.true_frame_clock_start(specs[1]) - synth.true_frame_clock_start(specs[0])
    assert abs(gpu.frame_clock_offsets(got)[1] - want) <= 1.0


@pytest.mark.gpu
def test_two_short_captures_align_on_one_cell(gpu, coef, tpl):
    """seed 11 and seed 72 on seed 11's cell, 3 multiframes + 12,345 samples apart, at 0.47 s: every row decodes on both"""
    a = _cell_spec(11)
    b = dataclasses.replace(_cell_spec(PAIR_SEED), bsic=a.bsic, fn0=a.fn0 + 153, start_offset=a.start_offset + 12345)
    other = _cell_spec(28)
    raw = synth.generate_batch([a, b, other]).numpy()
    got = gpu.calibrate_batch(raw, CARRIER, tpl, coef, carrier_fit=True, sch_decode=True)
    old = gpu.calibrate_demod_batch(raw, CARRIER, tpl, coef, sch_decode=True)
    for g, o in zip(got, old):
        assert g["cell"]["n_agree"] >= len(g["cell"]["fn"]) - 1 and g["cell"]["n_agree"] > o["cell"]["n_agree"]
    off = gpu.frame_clock_offsets(got)
    assert off[0] == 0.0 and abs(off[1] - (153 * 10000 + 12345)) <= 1.0 and math.isnan(off[2])


def _cell_bytes(item):
    c = item["cell"]
    return (tuple(c[k] for k in ("bsic", "fn_first", "n_crc_ok", "n_agree", "flags")), np.float64(c["frame_clock_start"]).tobytes(),
            None if c["fn"] is None else tuple(c[k].tobytes() for k in ("fn", "bsic_rows", "hamming", "row_flags", "df")),
            None if item["sch"] is None else tuple(item["sch"][k].tobytes() for k in ("demod_bits", "corr_val", "sch_ok")))


@pytest.mark.gpu
def test_cell_stream_independence_and_device_input(gpu, batch, coef, tpl):
    torch = pytest.importorskip("torch")
    _, raw, got = batch
    D = raw.shape[0]
    alone = gpu.calibrate_batch(raw[-4:-3], CARRIER, tpl, coef, carrier_fit=True, sch_decode=True)[0]
    assert _cell_bytes(alone) == _cell_bytes(got[D - 4])
    perm = np.random.default_rng(7).permutation(D)
    big = np.concatenate([raw[perm], raw[perm[::-1]]])                                 # 2D streams: several stream groups
    shuffled = gpu.calibrate_batch(big, CARRIER, tpl, coef, carrier_fit=True, sch_decode=True)
    for i, d in enumerate(perm):
        assert _cell_bytes(shuffled[i]) == _cell_bytes(got[d])
        assert _cell_bytes(shuffled[2 * D - 1 - i]) == _cell_bytes(got[d])
    dev = torch.from_numpy(raw.copy()).cuda()
    torch.cuda.synchronize()
    on_dev = gpu.calibrate_batch(None, CARRIER, tpl, coef, device_ptr=dev.data_ptr(), n_iq=raw.shape[1] // 2, n_streams=D, carrier_fit=True,
                                 sch_decode=True)
    for a, b in zip(on_dev, got):
        assert _cell_bytes(a) == _cell_bytes(b)


@pytest.mark.gpu
def test_cell_stage_is_reported(gpu, batch, coef, tpl):
    from gsmcal._lib import lib
    raw = batch[1]
    lib().gsmcal_debug_set(3, 1)
    try:
        gpu.calibrate_batch(raw[:4], CARRIER, tpl, coef, carrier_fit=True, sch_decode=True)
        ms = gpu.api.last_batch_stage_ms()
        assert len(ms) == 7 and list(ms.values())[6] > 0
    finally:
        lib().gsmcal_debug_set(3, 4)


@pytest.mark.gpu
def test_mex_gsm_calibrate_cell_batch(gpu, built_lib, tmp_path, batch, tpl):
    specs, raw, got = batch
    pick = [4, 7] + [i for i, s in enumerate(specs) if s.bsic is not None][:2]       # noise only, no r_correct, two cells
    a = np.ascontiguousarray(raw[pick].T)                                              # 2N x D uint8
    (tmp_path / "raw.bin").write_bytes(a.tobytes(order="F"))
    coef = oracle.fir1(46, 200e3 / FS)
    fmt = lambda v: ",".join("%r" % x for x in np.asarray(v).ravel(order="F").tolist())     # noqa: E731
    exe = _gateway(tmp_path, built_lib, r'''#include "mex.h"
#include "gsmcal.h"
static const double tre[] = {%s}, tim[] = {%s}, cf[] = {%s};
static double f1(const mxArray *s, size_t d, const char *k) { return mxGetPr(mxGetField(s, d, k))[0]; }
int main(int argc, char **argv) {
    size_t rows = %d, D = %d;
    size_t dims[2] = {rows, D};
    mxArray *raw = mxCreateNumericArray(2, dims, mxUINT8_CLASS, mxREAL);
    FILE *f = fopen(argv[1], "rb"); if (fread(mxGetData(raw), 1, rows * D, f) != rows * D) return 5; fclose(f);
    mxArray *t = mxCreateDoubleMatrix(512, 1, mxCOMPLEX), *c = mxCreateDoubleMatrix(1, 47, mxREAL);
    for (int i = 0; i < 512; ++i) { mxGetPr(t)[i] = tre[i]; mxGetPi(t)[i] = tim[i]; }
    for (int i = 0; i < 47; ++i) mxGetPr(c)[i] = cf[i];
    mxArray *out[6]; const mxArray *rhs[4] = {raw, mxCreateDoubleScalar(%r), t, c};
    mexFunction(6, out, 4, rhs);
    for (size_t d = 0; d < D; ++d) {
        printf("%%.17g %%.17g %%.17g %%.17g %%.17g %%.17g %%.17g", f1(out[4], d, "carrier_fit_ppm"), f1(out[4], d, "flags"), f1(out[5], d, "bsic"),
               f1(out[5], d, "fn_first"), f1(out[5], d, "n_agree"), f1(out[5], d, "flags"), f1(out[5], d, "frame_clock_start"));
        mxArray *fa = mxGetField(out[5], d, "fn");
        printf(" %%zu", mxGetN(fa));
        const char *k[] = {"fn", "bsic_rows", "hamming", "row_flags", "df"};
        for (int j = 0; j < 5; ++j) for (size_t i = 0; i < mxGetN(fa); ++i) printf(" %%.17g", mxGetPr(mxGetField(out[5], d, k[j]))[i]);
        printf("\n");
    }
    return 0;
}
''' % (fmt(np.asarray(tpl).real), fmt(np.asarray(tpl).imag), fmt(coef), a.shape[0], len(pick), CARRIER))
    lines = subprocess.run([str(exe), str(tmp_path / "raw.bin")], capture_output=True, text=True, check=True).stdout.strip().split("\n")
    assert len(lines) == len(pick)
    for line, d in zip(lines, pick):
        v = [float(x) for x in line.split()]
        c, cr = got[d]["cell"], got[d]["carrier"]
        assert np.float64(v[0]).tobytes() == np.float64(cr["carrier_fit_ppm"]).tobytes() and int(v[1]) == cr["flags"]
        assert [int(x) for x in v[2:6]] == [c["bsic"], c["fn_first"], c["n_agree"], c["flags"]]
        assert np.float64(v[6]).tobytes() == np.float64(c["frame_clock_start"]).tobytes()
        n = int(v[7])
        assert n == (0 if c["fn"] is None else len(c["fn"]))
        if n:
            per = np.array(v[8:]).reshape(5, n)
            for j, k in enumerate(("fn", "bsic_rows", "hamming", "row_flags")):
                np.testing.assert_array_equal(per[j], c[k])
            np.testing.assert_array_equal(per[4], c["df"])


@pytest.mark.gpu
def test_ingest_forwards_cell_sync(gpu):
    from gsmcal import ingest
    from gsmcal.rtl_tcp_replay import ReplayDongle
    N = N_SYNC
    specs = [_cell_spec(seed, 2 * N + 8) for seed in SEEDS]
    raw = synth.generate_batch(specs).numpy()
    srvs = [ReplayDongle(raw[d]) for d in range(len(specs))]
    try:
        res = ingest.calibrate_from_dongles([(s.host, s.port) for s in srvs], N, CARRIER, n_captures=1, carrier_fit=True, sch_decode=True)[0]
    finally:
        for s in srvs:
            s.close()
    direct_in = np.stack([s.expected(2 * N - 12, 2 * N) for s in srvs])
    direct = gpu.calibrate_batch(direct_in, CARRIER, gpu.gsm_SCH_training_sequence_gen(8), gpu.fir1(46, 200e3 / FS), carrier_fit=True,
                                 sch_decode=True)
    assert len(res) == len(direct) == len(specs)
    for a, b, s in zip(res, direct, specs):
        assert _cell_bytes(a) == _cell_bytes(b)
        assert a["carrier"]["carrier_fit_ppm"] == b["carrier"]["carrier_fit_ppm"]
        assert a["cell"]["bsic"] == s.bsic
