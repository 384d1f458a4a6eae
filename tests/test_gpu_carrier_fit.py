"""gsmcal_calibrate_carrier_fit_batch: gsmcal_calibrate_batch followed by the tone of every FCCH burst from the periodogram maximum of
its interior on r_correct and a least-squares line through the tones over capture time.  CPU: record layout and flags, export,
argument checks without a launch, the MEX gateway against the stub, known answers of the restatement in carrier_fit_oracle.py, its
accuracy against the synthetic truth and the generator's carrier drift.  GPU: parity with the oracle chain followed by
carrier_fit_oracle.carrier_reference, every calibrate_batch output byte-identical, drifting full-length streams, stream independence,
host against device input, the stage timing, the MEX gateway end to end and the rtl_tcp ingest."""
import ctypes as C
import dataclasses
import math
import os
import subprocess

import numpy as np
import pytest
from scipy.signal import lfilter

import carrier_fit_oracle as CF
import gsmcal_oracle as oracle
from gsmcal import synth
from test_gpu_demod_batch import _specs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MEX = os.path.join(ROOT, "multi-rtl-sdr-calibration_b200", "mex")
FS = oracle.SYMBOL_RATE * 8
CARRIER = 957.4e6
N_SYNC = 1020000
N_10S = 21666667
# An oracle run over random_spec(seed, 1020000) for seeds 1..40 (the default 0.47 s capture; every seed fits 9 or 10 FCCH bursts, all
# flags 0) gave |carrier_fit_ppm - injected ppm| at most 0.00302 ppm (median 0.00093, 95th percentile 0.00219), against
# total_carrier_ppm - injected ppm between -1.963 and -1.052 ppm (median -1.069).  The fit residual RMS was 0.90..6.9 Hz.
ACCURACY_PPM = 0.005


# ---- CPU: ABI ------------------------------------------------------------------------------------------------------------------
def test_carrier_result_layout():
    from gsmcal import api
    from gsmcal._lib import CarrierFitResult
    assert C.sizeof(CarrierFitResult) == 72
    names = ("n_fcch", "n_fit", "flags", "reserved", "t_mean", "freq_hz", "drift_hz_per_s", "rms_hz", "residual_ppm", "carrier_fit_ppm",
             "drift_ppm_per_s")
    assert [getattr(CarrierFitResult, f).offset for f in names] == [0, 4, 8, 12, 16, 24, 32, 40, 48, 56, 64]
    hdr = open(os.path.join(ROOT, "include", "gsmcal.h")).read()
    for name, v in (("NO_POS_INFO", 1), ("NO_R_CORRECT", 2), ("RANGE", 4), ("EDGE", 8), ("NOCONV", 16), ("FEW", 32)):
        assert hdr.split(f"#define GSMCAL_CARRIER_{name}")[1].split()[0] == str(v)
        assert getattr(api, f"CARRIER_{name}") == v == getattr(CF, name)


def test_carrier_fit_batch_symbol_exported(built_lib):
    from gsmcal import _lib
    assert "gsmcal_calibrate_carrier_fit_batch" in _lib.SIGNATURES
    out = subprocess.run(["nm", "-D", "--defined-only", built_lib], capture_output=True, text=True).stdout
    assert " T gsmcal_calibrate_carrier_fit_batch" in out


def _call(raw, n_iq, D, osr=8, carrier=True):
    from gsmcal._lib import CarrierFitResult, StreamResult, lib
    tpl = np.ones(64 * max(osr, 1), dtype=np.complex128)
    coef = oracle.fir1(46, 200e3 / FS)
    res, cf = (StreamResult * max(D, 1))(), (CarrierFitResult * max(D, 1))()
    vp = lambda a: a.ctypes.data_as(C.c_void_p)                                       # noqa: E731
    return lib().gsmcal_calibrate_carrier_fit_batch(vp(raw), 0, n_iq, D, CARRIER, vp(tpl), vp(coef), len(coef), osr, 8,
                                                    C.cast(res, C.c_void_p), None, None, None, None, None,
                                                    C.cast(cf, C.c_void_p) if carrier else None, None, None, None)


def test_carrier_fit_argument_errors_launch_nothing(built_lib):
    import gsmcal
    from gsmcal import api
    from gsmcal._lib import lib
    raw = np.zeros((1, 2 * 300000), dtype=np.uint8)
    n0 = api.launch_count()
    assert _call(raw, 300000, 1, carrier=False) == -1
    for osr in (0, 1, 4, 9):
        assert _call(raw, 300000, 1, osr=osr) == -1
        assert b"oversampling_ratio must be 8" in lib().gsmcal_last_error()
    assert _call(raw, 300000, 0) == -1
    assert _call(raw, 1000, 1) == -4                       # shorter than the 23 frames of the coarse search: GSMCAL_ERR_RANGE
    tpl, coef = np.ones(512, complex), oracle.fir1(46, 0.09)
    with pytest.raises(ValueError):
        gsmcal.calibrate_batch(raw, CARRIER, tpl, coef, sch_timing=True, carrier_fit=True)
    with pytest.raises(ValueError):
        gsmcal.calibrate_batch(raw, CARRIER, tpl, coef, r_correct=np.zeros((1, 300000), complex), carrier_fit=True)
    assert api.launch_count() == n0


def test_carrier_fit_batch_needs_a_device(built_lib):
    import gsmcal
    if gsmcal.device_count() > 0:
        pytest.skip("a CUDA device is present")
    raw = np.zeros((1, 2 * 300000), dtype=np.uint8)
    assert _call(raw, 300000, 1) == -2
    with pytest.raises(gsmcal.GsmcalError) as e:
        gsmcal.calibrate_batch(raw, CARRIER, np.ones(512, complex), oracle.fir1(46, 0.09), carrier_fit=True)
    assert e.value.code == -2


@pytest.mark.parametrize("interleaved", [0, 1])
def test_carrier_gateway_compiles_against_stub(tmp_path, interleaved):
    obj = tmp_path / "g.o"
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Wno-unused-function", "-c", "-DGSMCAL_MEX_gsm_calibrate_carrier_batch",
                    f"-DMX_HAS_INTERLEAVED_COMPLEX={interleaved}", f"-I{MEX}/stub", f"-I{ROOT}/include", os.path.join(MEX, "gsmcal_mex.c"),
                    "-o", str(obj)], check=True)
    sym = subprocess.run(["nm", str(obj)], capture_output=True, text=True).stdout
    assert " T mexFunction" in sym and " U gsmcal_calibrate_carrier_fit_batch" in sym
    assert "gsm_calibrate_carrier_batch" in open(os.path.join(MEX, "Makefile.mex")).read()


@pytest.mark.parametrize("nlhs,nrhs", [(6, 4), (5, 3), (5, 5)])
def test_carrier_gateway_usage_errors(built_lib, tmp_path, nlhs, nrhs):
    src = tmp_path / "h.c"
    src.write_text(r'''#include "mex.h"
int main(void) {
    size_t dims[2] = {600000, 1};
    mxArray *raw = mxCreateNumericArray(2, dims, mxUINT8_CLASS, mxREAL);
    mxArray *t = mxCreateDoubleMatrix(512, 1, mxCOMPLEX), *c = mxCreateDoubleMatrix(1, 47, mxREAL);
    mxArray *out[6]; const mxArray *rhs[5] = {raw, mxCreateDoubleScalar(957.4e6), t, c, c};
    mexFunction(%d, out, %d, rhs);
    return 0;
}
''' % (nlhs, nrhs))
    exe = tmp_path / "h"
    libdir = os.path.dirname(built_lib)
    subprocess.run(["gcc", "-std=c11", "-Wno-unused-function", "-DGSMCAL_MEX_gsm_calibrate_carrier_batch", f"-I{MEX}/stub", f"-I{ROOT}/include",
                    str(src), os.path.join(MEX, "gsmcal_mex.c"), f"-L{libdir}", "-lgsmcal", f"-Wl,-rpath,{libdir}", "-lm", "-o", str(exe)], check=True)
    p = subprocess.run([str(exe)], capture_output=True, text=True)
    assert p.returncode == 3 and "gsmcal:nargin" in p.stderr


# ---- CPU: known answers of the restatement ------------------------------------------------------------------------------------
def _tone(delta, phase=0.3, amp=1.0):
    n = np.arange(CF.W)
    return amp * np.exp(1j * (2 * np.pi * (CF.F_NOM + delta) * n / FS + phase))


@pytest.mark.parametrize("delta", [-6000.0, -1234.567, -0.25, 0.0, 291.8, 1041.7, 7700.0])
def test_pure_tone_is_recovered(delta):
    out = CF.tone_estimate(_tone(delta))
    assert out["flag"] == 0
    assert abs(out["f"] - (CF.F_NOM + delta)) < 1e-6
    assert out["last_step_hz"] < 1e-6


def test_periodogram_is_unbiased_in_filtered_noise_and_lag1_is_not():
    """tones plus complex white noise through the 47-tap channel filter (20 dB in the filter's band): the noise autocorrelation at lag 1
    is real and positive, so the lag-1 phase increment angle(sum x(n+1) conj(x(n))) is pulled towards 0 Hz; the periodogram maximum
    is not.  Over 64 windows per tone its mean error stays inside 5 standard errors of 0, while the lag-1 mean is off by > 100 Hz."""
    coef = oracle.fir1(46, 200e3 / FS)
    rg = np.random.default_rng(11)
    sigma = 0.1 / math.sqrt(np.sum(coef ** 2))               # noise power 0.01 after the filter, tone power 1
    for delta in (-1500.0, 350.0, 1041.7):
        e_pg, e_l1 = [], []
        for _ in range(64):
            w = sigma / math.sqrt(2) * (rg.standard_normal(CF.W + 200) + 1j * rg.standard_normal(CF.W + 200))
            x = _tone(delta, phase=rg.uniform(0, 2 * np.pi)) + lfilter(coef, 1.0, w)[200:]
            est = CF.tone_estimate(x)
            assert est["flag"] == 0
            e_pg.append(est["f"] - (CF.F_NOM + delta))
            e_l1.append(np.angle(np.sum(x[1:] * np.conj(x[:-1]))) * FS / (2 * np.pi) - (CF.F_NOM + delta))
        e_pg, e_l1 = np.array(e_pg), np.array(e_l1)
        assert abs(e_pg.mean()) < 5 * e_pg.std() / math.sqrt(len(e_pg)) + 1e-3, delta
        assert e_pg.std() < 10.0
        assert e_l1.mean() < -100.0, delta


def test_fit_recovers_a_planted_line():
    t = [0.0, 0.5, 1.0, 2.5]                              # every product and sum of the fit is exact: the line comes back bit for bit
    a0, b0 = 67700.5, 2.0
    t_bar, a, b, rms = CF.fit_line(t, [a0 + b0 * (v - 1.0) for v in t])
    assert (t_bar, a, b, rms) == (1.0, a0, b0, 0.0)


def _planted_stream(tones, pos, n=110000):
    """r with a pure tone f_i in the interior window of each FCCH row p_i (zeros elsewhere)"""
    r = np.zeros(n, complex)
    for p, f in zip(pos, tones):
        j0 = int(p) - 1 + CF.OFF
        r[j0:j0 + CF.W] = np.exp(2j * np.pi * f * np.arange(CF.W) / FS)
    return r


def test_carrier_fit_of_planted_tones():
    """tones on a planted line over the rows' capture times: the fit, its ppm figures and the row times as include/gsmcal.h states"""
    e1, e2 = 12e-6, -3e-6
    pos = np.array([1000.0 + 20000.0 * i for i in range(5)])
    t = np.array([CF.row_time(p, e1, e2) for p in pos])
    f0, slope = CF.F_NOM + 812.5, 300.0
    r = _planted_stream(f0 + slope * (t - t.mean()), pos)
    pinfo = np.column_stack([pos, np.zeros(5)])
    out = CF.carrier_fit(r, pinfo, e1, e2, -4.5, CARRIER)
    assert out["flags"] == 0 and out["n_fit"] == 5 and list(out["row_flag"]) == [0] * 5
    assert np.array_equal(out["t"], t)
    assert t[0] == ((((1000.0 + 128 + 463.5) - 1.0) * (1.0 + e2)) * (1.0 + e1)) / FS
    assert abs(out["t_mean"] - t.mean()) < 1e-15
    assert abs(out["freq_hz"] - f0) < 1e-6 and abs(out["drift_hz_per_s"] - slope) < 1e-4 and out["rms_hz"] < 1e-6
    assert out["residual_ppm"] == 1e6 * (out["freq_hz"] - CF.F_NOM) / CARRIER
    assert out["carrier_fit_ppm"] == oracle.total_ppm_calculation([-4.5, out["residual_ppm"]])
    assert out["drift_ppm_per_s"] == 1e6 * out["drift_hz_per_s"] / CARRIER


def test_rows_and_flags_of_the_restatement():
    """EDGE for a tone outside the grid, RANGE for an FCCH window that leaves r, FEW below three used rows, NaN where excluded"""
    pos = np.array([1000.0, 21000.0, 41000.0, 109000.0])
    r = _planted_stream([CF.F_NOM + 100.0, CF.F_NOM + 9000.0, CF.F_NOM - 20.0], pos[:3])
    pinfo = np.array([[pos[0], 0.0], [500.0, 1.0], [pos[1], 0.0], [pos[2], 0.0], [pos[3], 0.0], [90000.0, 2.0]])
    out = CF.carrier_fit(r, pinfo, 0.0, 0.0, 1.0, CARRIER)
    assert out["n_fcch"] == 4 and out["n_fit"] == 2
    assert list(out["row_flag"]) == [0, CF.EDGE, 0, CF.RANGE]
    assert out["k"][1] == CF.GRID_K
    assert out["flags"] == CF.EDGE | CF.RANGE | CF.FEW
    assert all(math.isnan(out[k]) for k in ("t_mean", "freq_hz", "drift_hz_per_s", "rms_hz", "carrier_fit_ppm", "drift_ppm_per_s"))
    assert np.isnan(out["f"][[1, 3]]).all() and np.isnan(out["t"][[1, 3]]).all()
    assert abs(out["f"][0] - (CF.F_NOM + 100.0)) < 1e-6 and abs(out["f"][2] - (CF.F_NOM - 20.0)) < 1e-6


# ---- CPU: the restatement against the synthetic truth ---------------------------------------------------------------------------
SEEDS = range(1, 9)


@pytest.fixture(scope="module")
def truth_runs():
    tpl = oracle.gsm_SCH_training_sequence_gen(8)
    coef = oracle.fir1(46, 200e3 / FS)
    out = []
    for seed in SEEDS:
        spec = synth.random_spec(seed, N_SYNC)
        raw = synth.generate_batch([spec]).numpy()[0]
        cal = oracle.calibrate_stream(raw, CARRIER, tpl, coef)
        out.append((spec, cal, CF.carrier_reference(cal, CARRIER)))
    return out


def test_carrier_fit_ppm_is_within_bound_of_the_injected_ppm(truth_runs):
    for spec, cal, r in truth_runs:
        assert r["flags"] == 0 and r["n_fit"] >= 9, spec.seed
        assert abs(r["carrier_fit_ppm"] - spec.carrier_ppm) < ACCURACY_PPM, spec.seed
        assert r["rms_hz"] < 10.0


def test_total_carrier_ppm_is_off_by_more_than_1_ppm(truth_runs):
    """what the feature fixes: the reference's estimate on the same captures"""
    for spec, cal, _ in truth_runs:
        assert cal["total_carrier_ppm"] - spec.carrier_ppm < -1.0, spec.seed


# ---- CPU: the generator's carrier drift ---------------------------------------------------------------------------------------
def test_zero_drift_is_byte_identical():
    spec = synth.random_spec(4, 200000)
    a = synth.generate_stream(spec).numpy()
    b = synth.generate_stream(dataclasses.replace(spec, carrier_drift_ppm_per_s=0.0)).numpy()
    assert a.tobytes() == b.tobytes()
    assert synth.true_carrier_ppm(spec, 3.0) == spec.carrier_ppm


def test_drifting_spec_phase_increments_rise_at_the_injected_rate():
    """CW_check.m:6 style: the mean phase increment angle(u(n+1)/u(n)) over each FCCH burst of the unfiltered capture (60 dB, so the
    uint8 rounding is the only noise) rises at drift * 1e-6 * carrier_freq Hz per second"""
    drift = 4.0
    spec = synth.StreamSpec(seed=9, n_samples=N_SYNC, carrier_ppm=2.0, carrier_drift_ppm_per_s=drift, snr_db=60.0, start_offset=777.0)
    raw = synth.generate_stream(spec).numpy().astype(np.float64)
    u = (raw[0::2] - 127.5) + 1j * (raw[1::2] - 127.5)
    t, f = [], []
    for s in synth.true_fcch_starts(spec):
        j = int(round(s)) - 1 + CF.OFF
        if j + CF.W >= len(u):
            continue
        x = u[j:j + CF.W]
        f.append(np.angle(np.mean(x[1:] / x[:-1])) * FS / (2 * np.pi))
        t.append((j + (CF.W - 1) / 2) / FS)
    t, f = np.array(t), np.array(f)
    assert len(t) >= 9
    slope = np.polyfit(t, f, 1)[0]
    want = drift * 1e-6 * CARRIER
    assert abs(slope - want) < 0.02 * want
    f_truth = CF.F_NOM + synth.true_carrier_ppm(spec, t) * 1e-6 * CARRIER
    assert np.max(np.abs(f - f_truth)) < 30.0


# ---- GPU -----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def coef():
    return oracle.fir1(46, 200e3 / FS)


@pytest.fixture(scope="module")
def tpl():
    return oracle.gsm_SCH_training_sequence_gen(8)


FIT_KEYS = ("t_mean", "freq_hz", "drift_hz_per_s", "rms_hz", "residual_ppm", "carrier_fit_ppm", "drift_ppm_per_s")


def _check_carrier(item, r):
    """GPU record against the restatement: flags, counts and row flags exact; f within 1e-6 Hz; t exactly the stated arithmetic on the
    stream's pos_info and sampling_ppm; the fit within the spread those f differences allow"""
    g = item["carrier"]
    assert g["flags"] == r["flags"] and g["n_fit"] == r["n_fit"]
    if r["f"] is None:
        assert g["f"] is None and g["t"] is None and g["row_flags"] is None
        assert all(math.isnan(g[k]) for k in FIT_KEYS)
        return
    assert np.array_equal(g["row_flags"], r["row_flag"])
    assert np.array_equal(np.isnan(g["f"]), np.isnan(r["f"])) and np.array_equal(np.isnan(g["t"]), np.isnan(r["t"]))
    ok = np.isfinite(r["f"])
    assert np.max(np.abs(g["f"][ok] - r["f"][ok]), initial=0.0) < 1e-6
    pinfo = item["pos_info"]
    pos = pinfo[pinfo[:, 1] == 0, 0]
    e1, e2 = item["sampling_ppm"][0] * 1e-6, item["sampling_ppm"][1] * 1e-6
    want_t = np.array([CF.row_time(p, e1, e2) if o else np.nan for p, o in zip(pos, ok)])
    assert g["t"][ok].tobytes() == want_t[ok].tobytes()
    if r["flags"] & CF.FEW:
        assert all(math.isnan(g[k]) for k in FIT_KEYS)
        return
    assert abs(g["t_mean"] - r["t_mean"]) < 1e-12 and abs(g["freq_hz"] - r["freq_hz"]) < 1e-6
    assert abs(g["drift_hz_per_s"] - r["drift_hz_per_s"]) < 1e-4 and abs(g["rms_hz"] - r["rms_hz"]) < 1e-5
    assert abs(g["carrier_fit_ppm"] - r["carrier_fit_ppm"]) < 1e-8 and abs(g["residual_ppm"] - r["residual_ppm"]) < 1e-9
    assert abs(g["drift_ppm_per_s"] - r["drift_ppm_per_s"]) < 1e-9


@pytest.fixture(scope="module")
def batch(gpu, coef, tpl):
    specs = _specs()                    # normal streams, a noise-only stream (pos_info == -1), one without r_correct
    raw = synth.generate_batch(specs).numpy()
    got = gpu.calibrate_batch(raw, CARRIER, tpl, coef, carrier_fit=True)
    cal = [oracle.calibrate_stream(raw[d], CARRIER, tpl, coef) for d in range(len(specs))]
    ref = [CF.carrier_reference(c, CARRIER) for c in cal]
    return raw, got, ref, cal, specs


@pytest.mark.gpu
def test_carrier_fit_batch_matches_oracle(batch):
    raw, got, ref, cal, specs = batch
    for g, r, c in zip(got, ref, cal):
        assert np.array_equal(g["pos_info"], c["pos_info"])
        _check_carrier(g, r)
    flags = [r["flags"] for r in ref]
    assert CF.NO_POS_INFO in flags and CF.NO_R_CORRECT in flags and sum(f == 0 for f in flags) >= 4
    for g, s in zip(got, specs):
        if g["carrier"]["flags"] == 0 and s.snr_db >= 15:
            assert abs(g["carrier"]["carrier_fit_ppm"] - s.carrier_ppm) < ACCURACY_PPM


def _raw_call(raw, carrier):
    """every output of gsmcal_calibrate_batch (carrier False) or gsmcal_calibrate_carrier_fit_batch, as bytes"""
    from gsmcal import api
    from gsmcal._lib import CarrierFitResult, StreamResult, lib
    coef = oracle.fir1(46, 200e3 / FS)
    tpl = oracle.gsm_SCH_training_sequence_gen(8)
    D, n_iq = raw.shape[0], raw.shape[1] // 2
    cap = api.max_bursts(n_iq)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)                                       # noqa: E731
    res = (StreamResult * D)()
    cal = [np.full((D, cap), 7.0), np.full((D, cap), 7.0), np.full((D, cap), 7.0), np.full((D, 6 * cap, 2), 7.0)]
    args = [vp(raw), 0, n_iq, D, CARRIER, vp(tpl), vp(coef), len(coef), 8, 8, C.cast(res, C.c_void_p)] + [vp(a) for a in cal] + [None]
    n0 = api.launch_count()
    if carrier:
        cf = (CarrierFitResult * D)()
        assert lib().gsmcal_calibrate_carrier_fit_batch(*args, C.cast(cf, C.c_void_p), None, None, None) == 0
    else:
        assert lib().gsmcal_calibrate_batch(*args) == 0
    return (bytes(res), [a.tobytes() for a in cal]), api.launch_count() - n0


@pytest.mark.gpu
def test_calibrate_batch_outputs_and_launches_unchanged(gpu, batch):
    raw = batch[0]
    plain, n_plain = _raw_call(raw, False)
    fitted, n_fitted = _raw_call(raw, True)
    again, n_again = _raw_call(raw, False)
    assert plain == fitted == again
    assert n_plain == n_again and n_fitted == n_plain + 3                             # one stream group: three more kernels


def _carrier_bytes(item):
    c = item["carrier"]
    return (np.array([c[k] for k in FIT_KEYS]).tobytes(), c["n_fit"], c["flags"],
            None if c["f"] is None else (c["f"].tobytes(), c["t"].tobytes(), c["row_flags"].tobytes()))


@pytest.mark.gpu
def test_carrier_stream_independence_and_device_input(gpu, batch, coef, tpl):
    torch = pytest.importorskip("torch")
    raw, got = batch[0], batch[1]
    D = raw.shape[0]
    alone = gpu.calibrate_batch(raw[1:2], CARRIER, tpl, coef, carrier_fit=True)[0]
    assert _carrier_bytes(alone) == _carrier_bytes(got[1])
    perm = np.random.default_rng(7).permutation(D)
    big = np.concatenate([raw[perm], raw[perm[::-1]]])                                 # 2D streams: several stream groups
    shuffled = gpu.calibrate_batch(big, CARRIER, tpl, coef, carrier_fit=True)
    for i, d in enumerate(perm):
        assert _carrier_bytes(shuffled[i]) == _carrier_bytes(got[d])
        assert _carrier_bytes(shuffled[2 * D - 1 - i]) == _carrier_bytes(got[d])
    dev = torch.from_numpy(raw.copy()).cuda()
    torch.cuda.synchronize()
    on_dev = gpu.calibrate_batch(None, CARRIER, tpl, coef, device_ptr=dev.data_ptr(), n_iq=raw.shape[1] // 2, n_streams=D, carrier_fit=True)
    for a, b in zip(on_dev, got):
        assert _carrier_bytes(a) == _carrier_bytes(b)


@pytest.mark.gpu
def test_carrier_stage_is_reported(gpu, batch, coef, tpl):
    from gsmcal._lib import lib
    raw = batch[0]
    lib().gsmcal_debug_set(3, 1)
    try:
        gpu.calibrate_batch(raw[:4], CARRIER, tpl, coef, carrier_fit=True)
        ms = gpu.api.last_batch_stage_ms()
        assert len(ms) == 7 and list(ms.values())[6] > 0
    finally:
        lib().gsmcal_debug_set(3, 4)


@pytest.mark.gpu
@pytest.mark.parametrize("drift", [0.02, -0.02])
def test_drifting_full_length_stream(gpu, coef, tpl, drift):
    """a 10 s device-resident capture whose carrier drifts by `drift` ppm/s: the fitted drift within 5 standard errors of the injected
    one (the standard error from the fit's own row scatter: rms / sqrt(sum (t - t_mean)^2)), carrier_fit_ppm within the accuracy bound
    of the truth at t_mean"""
    torch = pytest.importorskip("torch")
    spec = dataclasses.replace(synth.random_spec(101 if drift > 0 else 132, N_10S), carrier_drift_ppm_per_s=drift)
    raw = synth.generate_batch([spec], device="cuda")
    torch.cuda.synchronize()
    c = gpu.calibrate_batch(None, CARRIER, tpl, coef, device_ptr=raw.data_ptr(), n_iq=N_10S, n_streams=1, carrier_fit=True)[0]["carrier"]
    assert c["flags"] == 0 and c["n_fit"] > 150
    t = c["t"][np.isfinite(c["t"])]
    se = c["rms_hz"] / math.sqrt(np.sum((t - c["t_mean"]) ** 2)) * 1e6 / CARRIER
    assert abs(c["drift_ppm_per_s"] - drift) < 5 * se + 1e-5
    assert abs(c["carrier_fit_ppm"] - synth.true_carrier_ppm(spec, c["t_mean"])) < ACCURACY_PPM


@pytest.mark.gpu
def test_mex_gsm_calibrate_carrier_batch(gpu, built_lib, tmp_path, batch, tpl):
    raw, got = batch[0], batch[1]
    pick = [0, 1, 4, 7]                                                                # flags 0, 0, 1 (noise only), 2 (dropped FCCH)
    a = np.ascontiguousarray(raw[pick].T)                                              # 2N x D uint8
    (tmp_path / "raw.bin").write_bytes(a.tobytes(order="F"))
    coef = oracle.fir1(46, 200e3 / FS)
    fmt = lambda v: ",".join("%r" % x for x in np.asarray(v).ravel(order="F").tolist())     # noqa: E731
    src = tmp_path / "h.c"
    src.write_text(r'''#include "mex.h"
#include "gsmcal.h"
static const double tre[] = {%s}, tim[] = {%s}, cf[] = {%s};
static const char *keys[] = {"t_mean", "freq_hz", "drift_hz_per_s", "rms_hz", "residual_ppm", "carrier_fit_ppm", "drift_ppm_per_s"};
int main(int argc, char **argv) {
    size_t rows = %d, D = %d;
    size_t dims[2] = {rows, D};
    mxArray *raw = mxCreateNumericArray(2, dims, mxUINT8_CLASS, mxREAL);
    FILE *f = fopen(argv[1], "rb"); if (fread(mxGetData(raw), 1, rows * D, f) != rows * D) return 5; fclose(f);
    mxArray *t = mxCreateDoubleMatrix(512, 1, mxCOMPLEX), *c = mxCreateDoubleMatrix(1, 47, mxREAL);
    for (int i = 0; i < 512; ++i) { mxGetPr(t)[i] = tre[i]; mxGetPi(t)[i] = tim[i]; }
    for (int i = 0; i < 47; ++i) mxGetPr(c)[i] = cf[i];
    mxArray *out[5]; const mxArray *rhs[4] = {raw, mxCreateDoubleScalar(%r), t, c};
    mexFunction(5, out, 4, rhs);
    for (size_t d = 0; d < D; ++d) {
        mxArray *fa = mxGetField(out[4], d, "f"), *ta = mxGetField(out[4], d, "t"), *ra = mxGetField(out[4], d, "row_flags");
        printf("%%g %%g", mxGetPr(mxGetField(out[4], d, "flags"))[0], mxGetPr(mxGetField(out[4], d, "n_fit"))[0]);
        for (int k = 0; k < 7; ++k) printf(" %%.17g", mxGetPr(mxGetField(out[4], d, keys[k]))[0]);
        printf(" %%zu", mxGetN(fa));
        for (size_t i = 0; i < mxGetN(fa); ++i) printf(" %%.17g %%.17g %%g", mxGetPr(fa)[i], mxGetPr(ta)[i], mxGetPr(ra)[i]);
        printf("\n");
    }
    return 0;
}
''' % (fmt(np.asarray(tpl).real), fmt(np.asarray(tpl).imag), fmt(coef), a.shape[0], len(pick), CARRIER))
    exe = tmp_path / "h"
    libdir = os.path.dirname(built_lib)
    subprocess.run(["gcc", "-std=c11", "-Wno-unused-function", "-DGSMCAL_MEX_gsm_calibrate_carrier_batch", f"-I{MEX}/stub", f"-I{ROOT}/include",
                    str(src), os.path.join(MEX, "gsmcal_mex.c"), f"-L{libdir}", "-lgsmcal", f"-Wl,-rpath,{libdir}", "-lm", "-o", str(exe)], check=True)
    lines = subprocess.run([str(exe), str(tmp_path / "raw.bin")], capture_output=True, text=True, check=True).stdout.strip().split("\n")
    assert len(lines) == len(pick)
    seen = set()
    for line, d in zip(lines, pick):
        v = [float(s) for s in line.split()]
        c = got[d]["carrier"]
        assert int(v[0]) == c["flags"] and int(v[1]) == c["n_fit"]
        assert np.array(v[2:9]).tobytes() == np.array([c[k] for k in FIT_KEYS]).tobytes()
        n = int(v[9])
        assert n == (0 if c["f"] is None else len(c["f"]))
        if n:
            ftr = np.array(v[10:]).reshape(n, 3)
            assert ftr[:, 0].tobytes() == c["f"].tobytes() and ftr[:, 1].tobytes() == c["t"].tobytes()
            assert np.array_equal(ftr[:, 2].astype(np.int64), c["row_flags"])
        seen.add(c["flags"] & 3)
    assert seen == {0, 1, 2}


@pytest.mark.gpu
def test_ingest_calibrate_with_carrier_fit_equals_direct(gpu):
    import torch
    from gsmcal import ingest
    from gsmcal.rtl_tcp_replay import ReplayDongle
    N = N_SYNC
    specs = [synth.random_spec(seed, 2 * N + 8) for seed in (1, 2, 3)]
    raw = synth.generate_batch(specs, device="cuda").cpu().numpy()
    srvs = [ReplayDongle(raw[d]) for d in range(len(specs))]
    try:
        res = ingest.calibrate_from_dongles([(s.host, s.port) for s in srvs], N, CARRIER, n_captures=1, carrier_fit=True)[0]
    finally:
        for s in srvs:
            s.close()
    direct_in = np.stack([s.expected(2 * N - 12, 2 * N) for s in srvs])
    direct = gpu.calibrate_batch(direct_in, CARRIER, gpu.gsm_SCH_training_sequence_gen(8), gpu.fir1(46, 200e3 / FS), carrier_fit=True)
    assert len(res) == len(direct) == 3
    for a, b in zip(res, direct):
        np.testing.assert_array_equal(a["pos_info"], b["pos_info"])
        assert _carrier_bytes(a) == _carrier_bytes(b)
    assert sum(r["carrier"]["flags"] & CF.FEW == 0 for r in res) >= 2
    torch.cuda.synchronize()
