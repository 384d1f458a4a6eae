"""gsmcal_calibrate_sch_timing_batch: gsmcal_calibrate_batch followed by sub-sample timing of every SCH burst on r_correct and a
least-squares clock fit per stream.  CPU: record layout and flags, export, argument checks without a launch, the MEX gateway against
the stub, known answers of the restatement in sch_timing_oracle.py and its accuracy against the synthetic truth.  GPU: parity with the
oracle chain followed by sch_timing_oracle.sch_fine_timing, every calibrate_batch output byte-identical, relative timing of shifted
captures, host against device input, full-length streams, the stage timing, the MEX gateway end to end and the rtl_tcp ingest."""
import ctypes as C
import dataclasses
import math
import os
import subprocess

import numpy as np
import pytest

import gsmcal_oracle as oracle
import sch_timing_oracle as T
from gsmcal import synth
from test_gpu_demod_batch import _specs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MEX = os.path.join(ROOT, "multi-rtl-sdr-calibration_b200", "mex")
FS = oracle.SYMBOL_RATE * 8
CARRIER = 957.4e6
N_SYNC = 1020000
N_10S = 21666667


# ---- CPU: ABI ------------------------------------------------------------------------------------------------------------------
def test_timing_result_layout():
    from gsmcal import api
    from gsmcal._lib import SchTimingResult
    assert C.sizeof(SchTimingResult) == 40
    assert [getattr(SchTimingResult, f).offset for f in ("n_sch", "n_fit", "flags", "reserved", "t0", "fit_ppm", "rms")] == [0, 4, 8, 12, 16, 24, 32]
    hdr = open(os.path.join(ROOT, "include", "gsmcal.h")).read()
    for name, v in (("NO_POS_INFO", 1), ("NO_R_CORRECT", 2), ("RANGE", 4), ("EDGE", 8), ("FEW", 16)):
        assert hdr.split(f"#define GSMCAL_TIMING_{name}")[1].split()[0] == str(v)
        assert getattr(api, f"TIMING_{name}") == v == getattr(T, name)


def test_timing_batch_symbol_exported(built_lib):
    from gsmcal import _lib
    assert "gsmcal_calibrate_sch_timing_batch" in _lib.SIGNATURES
    out = subprocess.run(["nm", "-D", "--defined-only", built_lib], capture_output=True, text=True).stdout
    assert " T gsmcal_calibrate_sch_timing_batch" in out


def _call(raw, n_iq, D, osr=8, timing=True):
    from gsmcal._lib import SchTimingResult, StreamResult, lib
    tpl = np.ones(64 * max(osr, 1), dtype=np.complex128)
    coef = oracle.fir1(46, 200e3 / FS)
    res, tm = (StreamResult * max(D, 1))(), (SchTimingResult * max(D, 1))()
    vp = lambda a: a.ctypes.data_as(C.c_void_p)                                       # noqa: E731
    return lib().gsmcal_calibrate_sch_timing_batch(vp(raw), 0, n_iq, D, CARRIER, vp(tpl), vp(coef), len(coef), osr, 8,
                                                   C.cast(res, C.c_void_p), None, None, None, None, None,
                                                   C.cast(tm, C.c_void_p) if timing else None, None, None)


def test_timing_batch_argument_errors_launch_nothing(built_lib):
    from gsmcal import api
    from gsmcal._lib import lib
    raw = np.zeros((1, 2 * 300000), dtype=np.uint8)
    n0 = api.launch_count()
    assert _call(raw, 300000, 1, timing=False) == -1
    for osr in (0, 1, 4, 9):
        assert _call(raw, 300000, 1, osr=osr) == -1
        assert b"oversampling_ratio must be 8" in lib().gsmcal_last_error()
    assert _call(raw, 300000, 0) == -1
    assert _call(raw, 1000, 1) == -4                       # shorter than the 23 frames of the coarse search: GSMCAL_ERR_RANGE
    assert api.launch_count() == n0


def test_timing_batch_needs_a_device(built_lib):
    import gsmcal
    if gsmcal.device_count() > 0:
        pytest.skip("a CUDA device is present")
    raw = np.zeros((1, 2 * 300000), dtype=np.uint8)
    assert _call(raw, 300000, 1) == -2
    with pytest.raises(gsmcal.GsmcalError) as e:
        gsmcal.calibrate_batch(raw, CARRIER, np.ones(512, complex), oracle.fir1(46, 0.09), sch_timing=True)
    assert e.value.code == -2


def test_timing_python_rejects_r_correct():
    import gsmcal
    with pytest.raises(ValueError):
        gsmcal.calibrate_batch(np.zeros((1, 600000), np.uint8), CARRIER, np.ones(512, complex), oracle.fir1(46, 0.09),
                               r_correct=np.zeros((1, 300000), complex), sch_timing=True)


def test_timing_gateway_compiles_against_stub(tmp_path):
    obj = tmp_path / "g.o"
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Wno-unused-function", "-c", "-DGSMCAL_MEX_gsm_calibrate_batch", f"-I{MEX}/stub",
                    f"-I{ROOT}/include", os.path.join(MEX, "gsmcal_mex.c"), "-o", str(obj)], check=True)
    sym = subprocess.run(["nm", str(obj)], capture_output=True, text=True).stdout
    assert " T mexFunction" in sym and " U gsmcal_calibrate_sch_timing_batch" in sym and " U gsmcal_calibrate_batch" in sym


@pytest.mark.parametrize("nlhs,nrhs", [(6, 4), (5, 3), (5, 5)])
def test_timing_gateway_usage_errors(built_lib, tmp_path, nlhs, nrhs):
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
    subprocess.run(["gcc", "-std=c11", "-Wno-unused-function", "-DGSMCAL_MEX_gsm_calibrate_batch", f"-I{MEX}/stub", f"-I{ROOT}/include", str(src),
                    os.path.join(MEX, "gsmcal_mex.c"), f"-L{libdir}", "-lgsmcal", f"-Wl,-rpath,{libdir}", "-lm", "-o", str(exe)], check=True)
    p = subprocess.run([str(exe)], capture_output=True, text=True)
    assert p.returncode == 3 and "gsmcal:nargin" in p.stderr


# ---- CPU: known answers of the restatement ------------------------------------------------------------------------------------
def test_parabola_vertex_of_a_planted_quadratic():
    for v, a, c in ((0.3125, -2.0, 7.0), (-0.25, -0.5, 1.0), (0.0, -3.0, 2.0), (0.4375, -1.0, 100.0)):
        y = [a * (k - v) ** 2 + c for k in (-1, 0, 1)]
        assert T.parabola_delta(*y) == v
    assert T.parabola_delta(1.0, 1.0, 1.0) == 0.0


def _planted(shift, n=4000, g=1500, seed=3):
    """the SCH template at training start g + shift (fractional) by band-limited (periodic sinc) interpolation, in weak noise"""
    t = oracle.gsm_SCH_training_sequence_gen(8)
    x = np.zeros(n, complex)
    x[g - 1:g - 1 + T.L] = t
    f = np.fft.fftfreq(n)
    r = np.fft.ifft(np.fft.fft(x) * np.exp(-2j * np.pi * f * shift))
    rg = np.random.default_rng(seed)
    return r + 1e-3 * (rg.standard_normal(n) + 1j * rg.standard_normal(n)), t


@pytest.mark.parametrize("shift", [0.0, 0.21, -0.37, 0.5, 3.81, -6.6])
def test_fractional_shift_is_recovered(shift):
    g = 1500
    r, t = _planted(shift)
    p = g - T.PRE
    out = T.sch_fine_timing(r, np.array([[p, 1.0]]), t, 8, 0.0, 0.0)
    assert out["row_flag"][0] == 0
    assert abs(out["tau"][0] - (g + shift)) < 0.02
    assert out["x"][0] == out["tau"][0] - 1.0


def test_fit_recovers_a_planted_line():
    m = [0.0, 1024.0, 2048.0, 5120.0]                     # every product and sum of the fit is exact: b and a come back bit for bit
    a0, b0 = 1234.5, 1.0 + 2.0 ** -10
    a, b, rms = T.fit_line(m, [a0 + b0 * v for v in m])
    assert a == a0 and b == b0 and rms == 0.0


def test_rows_and_flags_of_the_restatement():
    """RANGE for a window outside r, EDGE for a maximum on the last lag, FEW below three fitted rows, NaN where excluded"""
    g = 1500
    r, t = _planted(0.0)
    pinfo = np.array([[g - T.PRE, 1.0], [g - T.PRE - 26, 1.0], [3900.0, 1.0], [77.0, 0.0]])
    out = T.sch_fine_timing(r, pinfo, t, 8, 1e-5, -2e-6)
    assert out["n_sch"] == 3 and out["n_fit"] == 1
    assert list(out["row_flag"]) == [0, T.EDGE, T.RANGE]
    assert out["lstar"][0] == 0 and out["lstar"][1] == T.LAG_HI
    assert out["flags"] == T.EDGE | T.RANGE | T.FEW and math.isnan(out["fit_ppm"])
    assert out["x"][0] == ((out["tau"][0] - 1.0) * (1.0 - 2e-6)) * (1.0 + 1e-5)
    assert np.isnan(out["tau"][1:]).all() and np.isnan(out["x"][1:]).all()


# ---- CPU: the restatement against the synthetic truth ---------------------------------------------------------------------------
# An oracle run over random_spec(seed, 1020000) for seeds 1..40 (the default 0.47 s capture of gsm_sync_demod.m; all 40 reach a fit
# over 9 or 10 SCH bursts) gave |fit_ppm - injected ppm| at most 0.383 ppm (median 0.059, 95th percentile 0.135), against at most
# 1.099 ppm (median 0.311) for total_sampling_ppm, whose lattice step is 1.087 ppm.  The fit residual RMS was 0.035..0.095 samples,
# except 0.539 on seed 24.  fit_ppm was closer to the truth than total_sampling_ppm on 37 of the 40 seeds, and on all 14 where the two
# differ by more than half a lattice step (no seed had them a whole step apart).  The seeds here are the first eight (RMS at most
# 0.095, four of them more than half a step apart).
SEEDS = range(1, 9)
HALF_STEP = 0.5 * 1.087


@pytest.fixture(scope="module")
def truth_runs():
    tpl = oracle.gsm_SCH_training_sequence_gen(8)
    coef = oracle.fir1(46, 200e3 / FS)
    out = []
    for seed in SEEDS:
        spec = synth.random_spec(seed, N_SYNC)
        raw = synth.generate_batch([spec]).numpy()[0]
        cal = oracle.calibrate_stream(raw, CARRIER, tpl, coef)
        out.append((spec, cal, T.timing_reference(cal, tpl)))
    return out


def test_fit_ppm_is_within_bound_of_the_injected_ppm(truth_runs):
    for spec, cal, t in truth_runs:
        assert t["flags"] == 0 and t["n_fit"] >= 9
        assert abs(t["fit_ppm"] - spec.sampling_ppm) < 0.5, spec.seed
        assert t["rms"] < 0.15


def test_fit_ppm_beats_the_lattice(truth_runs):
    better = [abs(t["fit_ppm"] - s.sampling_ppm) < abs(c["total_sampling_ppm"] - s.sampling_ppm)
              for s, c, t in truth_runs if abs(t["fit_ppm"] - c["total_sampling_ppm"]) > HALF_STEP]
    assert len(better) >= 3 and all(better)
    worst_fit = max(abs(t["fit_ppm"] - s.sampling_ppm) for s, _, t in truth_runs)
    worst_chain = max(abs(c["total_sampling_ppm"] - s.sampling_ppm) for s, c, _ in truth_runs)
    assert worst_fit < worst_chain


# ---- GPU -----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def coef():
    return oracle.fir1(46, 200e3 / FS)


@pytest.fixture(scope="module")
def tpl():
    return oracle.gsm_SCH_training_sequence_gen(8)


def _check_timing(g, r):
    """GPU record against the restatement: flags and counts exact, l* exact where the oracle's top two are apart by more than
    1e-9 relative, tau and x within 1e-6 samples, fit_ppm within 1e-6 ppm, t0 within 1e-6 samples"""
    assert g["flags"] == r["flags"] and g["n_fit"] == r["n_fit"]
    if r["tau"] is None:
        assert g["tau"] is None and g["x"] is None
        return
    assert len(g["tau"]) == r["n_sch"]
    sep = r["gap"] > 1e-9
    assert np.array_equal(np.isnan(g["tau"][sep]), np.isnan(r["tau"][sep]))
    ok = sep & np.isfinite(r["tau"])
    g_l = np.floor(g["tau"][ok] - (np.asarray(r["tau"][ok]) - r["lstar"][ok]) + 0.5)      # the lag the GPU's tau sits at
    assert np.array_equal(g_l, r["lstar"][ok].astype(float))
    assert np.max(np.abs(g["tau"][ok] - r["tau"][ok]), initial=0.0) < 1e-6
    assert np.max(np.abs(g["x"][ok] - r["x"][ok]), initial=0.0) < 1e-6
    if r["flags"] & T.FEW:
        assert math.isnan(g["fit_ppm"]) and math.isnan(g["t0"]) and math.isnan(g["rms"])
    elif sep.all():
        assert abs(g["fit_ppm"] - r["fit_ppm"]) < 1e-6 and abs(g["t0"] - r["t0"]) < 1e-6 and abs(g["rms"] - r["rms"]) < 1e-6


@pytest.fixture(scope="module")
def batch(gpu, coef, tpl):
    specs = _specs()                    # normal streams, a noise-only stream (pos_info == -1), one without r_correct
    raw = synth.generate_batch(specs).numpy()
    got = gpu.calibrate_batch(raw, CARRIER, tpl, coef, sch_timing=True)
    cal = [oracle.calibrate_stream(raw[d], CARRIER, tpl, coef) for d in range(len(specs))]
    ref = [T.timing_reference(c, tpl) for c in cal]
    return raw, got, ref, cal


@pytest.mark.gpu
def test_timing_batch_matches_oracle(batch):
    raw, got, ref, cal = batch
    for g, r, c in zip(got, ref, cal):
        assert np.array_equal(g["pos_info"], c["pos_info"])
        _check_timing(g["timing"], r)
    flags = [r["flags"] for r in ref]
    assert T.NO_POS_INFO in flags and T.NO_R_CORRECT in flags and sum(f == 0 for f in flags) >= 4


def _raw_call(raw, timing):
    """every output of gsmcal_calibrate_batch (timing False) or gsmcal_calibrate_sch_timing_batch, as bytes"""
    from gsmcal import api
    from gsmcal._lib import SchTimingResult, StreamResult, lib
    coef = oracle.fir1(46, 200e3 / FS)
    tpl = oracle.gsm_SCH_training_sequence_gen(8)
    D, n_iq = raw.shape[0], raw.shape[1] // 2
    cap = api.max_bursts(n_iq)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)                                       # noqa: E731
    res = (StreamResult * D)()
    cal = [np.full((D, cap), 7.0), np.full((D, cap), 7.0), np.full((D, cap), 7.0), np.full((D, 6 * cap, 2), 7.0)]
    args = [vp(raw), 0, n_iq, D, CARRIER, vp(tpl), vp(coef), len(coef), 8, 8, C.cast(res, C.c_void_p)] + [vp(a) for a in cal] + [None]
    n0 = api.launch_count()
    if timing:
        tm = (SchTimingResult * D)()
        assert lib().gsmcal_calibrate_sch_timing_batch(*args, C.cast(tm, C.c_void_p), None, None) == 0
    else:
        assert lib().gsmcal_calibrate_batch(*args) == 0
    return (bytes(res), [a.tobytes() for a in cal]), api.launch_count() - n0


@pytest.mark.gpu
def test_calibrate_batch_outputs_and_launches_unchanged(gpu, batch):
    raw = batch[0]
    plain, n_plain = _raw_call(raw, False)
    timed, n_timed = _raw_call(raw, True)
    again, n_again = _raw_call(raw, False)
    assert plain == timed == again
    assert n_plain == n_again and n_timed == n_plain + 3                              # one stream group: three more kernels


@pytest.mark.gpu
@pytest.mark.parametrize("delta", [0.37, 3.81, -0.6])
def test_relative_timing_of_shifted_captures(gpu, coef, tpl, delta):
    """two captures of one signal whose start differs by delta nominal samples: t0 differs by -delta*(1 + ppm*1e-6) up to the
    estimation error, which the oracle on the same inputs bounds"""
    base = synth.random_spec(3, N_SYNC)
    specs = [base, dataclasses.replace(base, start_offset=base.start_offset + delta)]
    raw = synth.generate_batch(specs).numpy()
    got = gpu.calibrate_batch(raw, CARRIER, tpl, coef, sch_timing=True)
    ref = [T.timing_reference(oracle.calibrate_stream(raw[d], CARRIER, tpl, coef), tpl) for d in range(2)]
    for g, r in zip(got, ref):
        _check_timing(g["timing"], r)
    # the same bursts head both fits (the integer pos_info grids of the two captures may differ by a few samples)
    assert got[0]["timing"]["flags"] == got[1]["timing"]["flags"] == 0 and len(got[0]["timing"]["tau"]) == len(got[1]["timing"]["tau"])
    assert abs(got[0]["pos_info"][0, 0] - got[1]["pos_info"][0, 0]) < 16
    want = -delta * (1.0 + base.sampling_ppm * 1e-6)
    err_ref = abs((ref[1]["t0"] - ref[0]["t0"]) - want)
    err_gpu = abs((got[1]["timing"]["t0"] - got[0]["timing"]["t0"]) - want)
    assert err_gpu <= err_ref + 1e-5 and err_gpu < 0.7


def _timing_bytes(item):
    t = item["timing"]
    return (np.array([t["t0"], t["fit_ppm"], t["rms"]]).tobytes(), t["n_fit"], t["flags"],
            None if t["tau"] is None else (t["tau"].tobytes(), t["x"].tobytes()))


@pytest.mark.gpu
def test_timing_stream_independence_and_device_input(gpu, batch, coef, tpl):
    torch = pytest.importorskip("torch")
    raw, got, _, _ = batch
    D = raw.shape[0]
    alone = gpu.calibrate_batch(raw[1:2], CARRIER, tpl, coef, sch_timing=True)[0]
    assert _timing_bytes(alone) == _timing_bytes(got[1])
    perm = np.random.default_rng(7).permutation(D)
    big = np.concatenate([raw[perm], raw[perm[::-1]]])                                 # 2D streams: several stream groups
    shuffled = gpu.calibrate_batch(big, CARRIER, tpl, coef, sch_timing=True)
    for i, d in enumerate(perm):
        assert _timing_bytes(shuffled[i]) == _timing_bytes(got[d])
        assert _timing_bytes(shuffled[2 * D - 1 - i]) == _timing_bytes(got[d])
    dev = torch.from_numpy(raw.copy()).cuda()
    torch.cuda.synchronize()
    on_dev = gpu.calibrate_batch(None, CARRIER, tpl, coef, device_ptr=dev.data_ptr(), n_iq=raw.shape[1] // 2, n_streams=D, sch_timing=True)
    for a, b in zip(on_dev, got):
        assert _timing_bytes(a) == _timing_bytes(b)


@pytest.mark.gpu
def test_timing_stage_is_reported(gpu, batch, coef, tpl):
    from gsmcal._lib import lib
    raw = batch[0]
    lib().gsmcal_debug_set(3, 1)
    try:
        gpu.calibrate_batch(raw[:4], CARRIER, tpl, coef, sch_timing=True)
        ms = gpu.api.last_batch_stage_ms()
        assert len(ms) == 7 and list(ms.values())[6] > 0
    finally:
        lib().gsmcal_debug_set(3, 4)


@pytest.mark.gpu
def test_timing_full_length_streams_match_oracle(gpu, coef, tpl):
    torch = pytest.importorskip("torch")
    specs = [synth.random_spec(seed, N_10S) for seed in (101, 132)]
    raw = synth.generate_batch(specs, device="cuda")
    torch.cuda.synchronize()
    got = gpu.calibrate_batch(None, CARRIER, tpl, coef, device_ptr=raw.data_ptr(), n_iq=N_10S, n_streams=2, sch_timing=True)
    host = raw.cpu().numpy()
    for d in range(2):
        ref = T.timing_reference(oracle.calibrate_stream(host[d], CARRIER, tpl, coef), tpl)
        assert ref["flags"] & T.FEW == 0 and ref["n_fit"] > 100
        _check_timing(got[d]["timing"], ref)
        assert abs(got[d]["timing"]["fit_ppm"] - specs[d].sampling_ppm) < 0.1


@pytest.mark.gpu
def test_mex_gsm_calibrate_batch_timing(gpu, built_lib, tmp_path, batch, tpl):
    raw, got, _, _ = batch
    pick = [0, 1, 4, 7]                                                                # flags 0, 0, 1 (noise only), 2 (dropped FCCH)
    a = np.ascontiguousarray(raw[pick].T)                                              # 2N x D uint8
    (tmp_path / "raw.bin").write_bytes(a.tobytes(order="F"))
    coef = oracle.fir1(46, 200e3 / FS)
    fmt = lambda v: ",".join("%r" % x for x in np.asarray(v).ravel(order="F").tolist())     # noqa: E731
    src = tmp_path / "h.c"
    src.write_text(r'''#include "mex.h"
#include "gsmcal.h"
static const double tre[] = {%s}, tim[] = {%s}, cf[] = {%s};
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
        mxArray *ta = mxGetField(out[4], d, "tau"), *xa = mxGetField(out[4], d, "x");
        printf("%%g %%g %%.17g %%.17g %%.17g %%zu", mxGetPr(mxGetField(out[4], d, "flags"))[0], mxGetPr(mxGetField(out[4], d, "n_fit"))[0],
               mxGetPr(mxGetField(out[4], d, "t0"))[0], mxGetPr(mxGetField(out[4], d, "fit_ppm"))[0], mxGetPr(mxGetField(out[4], d, "rms"))[0], mxGetN(ta));
        for (size_t i = 0; i < mxGetN(ta); ++i) printf(" %%.17g %%.17g", mxGetPr(ta)[i], mxGetPr(xa)[i]);
        printf("\n");
    }
    return 0;
}
''' % (fmt(np.asarray(tpl).real), fmt(np.asarray(tpl).imag), fmt(coef), a.shape[0], len(pick), CARRIER))
    exe = tmp_path / "h"
    libdir = os.path.dirname(built_lib)
    subprocess.run(["gcc", "-std=c11", "-Wno-unused-function", "-DGSMCAL_MEX_gsm_calibrate_batch", f"-I{MEX}/stub", f"-I{ROOT}/include", str(src),
                    os.path.join(MEX, "gsmcal_mex.c"), f"-L{libdir}", "-lgsmcal", f"-Wl,-rpath,{libdir}", "-lm", "-o", str(exe)], check=True)
    lines = subprocess.run([str(exe), str(tmp_path / "raw.bin")], capture_output=True, text=True, check=True).stdout.strip().split("\n")
    assert len(lines) == len(pick)
    seen = set()
    for line, d in zip(lines, pick):
        v = [float(s) for s in line.split()]
        t = got[d]["timing"]
        assert int(v[0]) == t["flags"] and int(v[1]) == t["n_fit"]
        assert np.array(v[2:5]).tobytes() == np.array([t["t0"], t["fit_ppm"], t["rms"]]).tobytes()
        n = int(v[5])
        assert n == (0 if t["tau"] is None else len(t["tau"]))
        if n:
            tx = np.array(v[6:]).reshape(n, 2)
            assert tx[:, 0].tobytes() == t["tau"].tobytes() and tx[:, 1].tobytes() == t["x"].tobytes()
        seen.add(t["flags"] & 3)
    assert seen == {0, 1, 2}


@pytest.mark.gpu
def test_ingest_calibrate_with_timing_equals_direct(gpu):
    import torch
    from gsmcal import ingest
    from gsmcal.rtl_tcp_replay import ReplayDongle
    N = N_SYNC
    specs = [synth.random_spec(seed, 2 * N + 8) for seed in (1, 2, 3)]
    raw = synth.generate_batch(specs, device="cuda").cpu().numpy()
    srvs = [ReplayDongle(raw[d]) for d in range(len(specs))]
    try:
        res = ingest.calibrate_from_dongles([(s.host, s.port) for s in srvs], N, CARRIER, n_captures=1, sch_timing=True)[0]
    finally:
        for s in srvs:
            s.close()
    direct_in = np.stack([s.expected(2 * N - 12, 2 * N) for s in srvs])
    direct = gpu.calibrate_batch(direct_in, CARRIER, gpu.gsm_SCH_training_sequence_gen(8), gpu.fir1(46, 200e3 / FS), sch_timing=True)
    assert len(res) == len(direct) == 3
    for a, b in zip(res, direct):
        np.testing.assert_array_equal(a["pos_info"], b["pos_info"])
        assert _timing_bytes(a) == _timing_bytes(b)
    assert sum(r["timing"]["flags"] & T.FEW == 0 for r in res) >= 2
    torch.cuda.synchronize()
