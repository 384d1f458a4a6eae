"""gsmcal_calibrate_demod_batch: the batched pipeline followed by SCH_demod / FCCH_demod on every stream's r_correct, evaluated from the
uint8 capture.  CPU: record layout, export, argument checks, the MEX gateway against the stub.  GPU: parity with sync_demod_stream below
(the oracle chain, then the oracle's demodulators; bits, bits_to_decoder, corr_val, max_idx exact; freq 1e-6 Hz; snr 1e-9 dB; mean 1e-6 Hz;
ppm 1e-9),
calibration outputs unchanged, the drop-in demodulators on calibrate_batch_r's r_correct, stream independence, full-length streams and
the MEX gateway end to end."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

import gsmcal_oracle as oracle
from gsmcal import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MEX = os.path.join(ROOT, "multi-rtl-sdr-calibration_b200", "mex")
FS = oracle.SYMBOL_RATE * 8
CARRIER = 957.4e6
N_SYNC = 1020000
N_10S = 21666667


# ---- CPU -----------------------------------------------------------------------------------------------------------------------
def test_demod_result_layout():
    from gsmcal._lib import DemodResult
    assert C.sizeof(DemodResult) == 32
    assert [getattr(DemodResult, f).offset for f in ("n_sch", "n_sch_ok", "n_fcch", "flags", "fcch_mean_freq", "fcch_carrier_ppm")] == [0, 4, 8, 12, 16, 24]
    hdr = open(os.path.join(ROOT, "include", "gsmcal.h")).read()
    for name, v in (("NO_POS_INFO", 1), ("NO_R_CORRECT", 2), ("SCH_RANGE", 4), ("FCCH_RANGE", 8)):
        assert f"#define GSMCAL_DEMOD_{name}" in hdr and hdr.split(f"#define GSMCAL_DEMOD_{name}")[1].split()[0] == str(v)


def test_demod_batch_symbol_exported(built_lib):
    from gsmcal import _lib
    assert "gsmcal_calibrate_demod_batch" in _lib.SIGNATURES
    assert hasattr(_lib.lib(), "gsmcal_calibrate_demod_batch")
    out = subprocess.run(["nm", "-D", "--defined-only", built_lib], capture_output=True, text=True).stdout
    assert " T gsmcal_calibrate_demod_batch" in out


def _call(raw, n_iq, D, osr=8, demod=True, tpl_len=None):
    from gsmcal._lib import DemodResult, StreamResult, lib
    tpl = np.ones(64 * osr if tpl_len is None else tpl_len, dtype=np.complex128)
    coef = oracle.fir1(46, 200e3 / FS)
    res, dem = (StreamResult * max(D, 1))(), (DemodResult * max(D, 1))()
    vp = lambda a: a.ctypes.data_as(C.c_void_p)                                       # noqa: E731
    return lib().gsmcal_calibrate_demod_batch(vp(raw) if raw is not None else None, 0, n_iq, D, CARRIER, vp(tpl), vp(coef), len(coef), osr, 8,
                                              C.cast(res, C.c_void_p), None, None, None, None, None,
                                              C.cast(dem, C.c_void_p) if demod else None, None, None, None, None, None, None, None)


def test_demod_batch_bad_arguments(built_lib):
    raw = np.zeros((1, 2 * 300000), dtype=np.uint8)
    assert _call(raw, 300000, 1, demod=False) == -1
    assert _call(raw, 300000, 1, osr=0) == -1
    assert _call(raw, 300000, 1, osr=9) == -1
    assert _call(None, 300000, 1) == -1
    assert _call(raw, 300000, 0) == -1
    assert _call(raw, 1000, 1) == -4                                                   # shorter than 23 frames


def test_demod_batch_needs_a_device(built_lib):
    import gsmcal
    if gsmcal.device_count() > 0:
        pytest.skip("a CUDA device is present")
    raw = np.zeros((1, 2 * 300000), dtype=np.uint8)
    assert _call(raw, 300000, 1) == -2
    with pytest.raises(gsmcal.GsmcalError) as e:
        gsmcal.calibrate_demod_batch(raw, CARRIER, np.ones(512, complex), oracle.fir1(46, 0.09))
    assert e.value.code == -2


def test_demod_gateway_compiles_against_stub(tmp_path):
    obj = tmp_path / "g.o"
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Wno-unused-function", "-c", "-DGSMCAL_MEX_gsm_calibrate_demod_batch", f"-I{MEX}/stub",
                    f"-I{ROOT}/include", os.path.join(MEX, "gsmcal_mex.c"), "-o", str(obj)], check=True)
    sym = subprocess.run(["nm", str(obj)], capture_output=True, text=True).stdout
    assert " T mexFunction" in sym and " U gsmcal_calibrate_demod_batch" in sym


# ---- GPU -----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def coef():
    return oracle.fir1(46, 200e3 / FS)


@pytest.fixture(scope="module")
def tpl():
    return oracle.gsm_SCH_training_sequence_gen(8)


def sync_demod_stream(raw_u8, carrier_freq, template, coef, osr=8):
    """Reference of one stream: oracle.calibrate_stream, then oracle.SCH_demod / oracle.FCCH_demod on r_final (gsm_sync_demod.m:144-145),
    with the rules of the batched call: pos_info == -1 -> flags 1, r_final == -1 -> flags 2 (sch = fcch = None); an SCH row whose
    equaliser window leaves r_final has sch_ok False and zero bits / correlations (flags 4); an FCCH window outside r_final gives NaN
    for that row and for mean_freq / carrier_ppm (flags 8)."""
    res = oracle.calibrate_stream(raw_u8, carrier_freq, template, coef, osr)
    pinfo, r = np.asarray(res["pos_info"], dtype=np.float64).reshape(-1, 2), res["r_final"]
    sch = fcch = None
    if pinfo.size > 0 and np.all(pinfo == -1):
        flags = 1
    elif r is None:
        flags = 2
    else:
        flags, n = 0, len(r)
        srows = pinfo[pinfo[:, 1] == 1]
        s_ok = np.array([p - 8 * osr >= 1 and p - 8 * osr + 194 * osr - 1 <= n for p in srows[:, 0]], dtype=bool)
        sch = dict(demod_bits=np.zeros((len(srows), 148), dtype=np.int64), bits_to_decoder=np.zeros((len(srows), 148), dtype=np.int64),
                   corr_val=np.zeros((len(srows), 85)), sch_ok=s_ok)
        if s_ok.any():
            got = oracle.SCH_demod(r, srows[s_ok], template, osr)
            for k in ("demod_bits", "bits_to_decoder", "corr_val"):
                sch[k][s_ok] = got[k]
        if not s_ok.all():
            flags |= 4
        frows = pinfo[pinfo[:, 1] == 0]
        f_ok = np.array([p >= 1 and p + 148 * osr - 1 <= n for p in frows[:, 0]], dtype=bool)
        nan = np.full(len(frows), np.nan)
        fcch = dict(freq=nan.copy(), mean_freq=math.nan, carrier_ppm=math.nan, snr=nan.copy(), max_idx=nan.copy())
        if f_ok.any():
            got = oracle.FCCH_demod(r, frows[f_ok], osr, carrier_freq)
            for k in ("freq", "snr", "max_idx"):
                fcch[k][f_ok] = got[k]
            if f_ok.all():
                fcch["mean_freq"], fcch["carrier_ppm"] = got["mean_freq"], got["carrier_ppm"]
        if not f_ok.all():
            flags |= 8
    return dict(res, sch=sch, fcch=fcch, demod_flags=flags)


def _specs():
    """seeds with a normal training sequence code and with random bits, a noise-only stream, weak / offset chains, and streams with
    one FCCH burst dropped that reaches pos_info with fewer than four BCCH rows (no r_correct)"""
    import dataclasses
    out = [synth.random_spec(1, N_SYNC), synth.random_spec(2, N_SYNC), synth.random_spec(3, N_SYNC), synth.random_spec(5, N_SYNC)]
    out[0] = dataclasses.replace(out[0], tsc=0)
    out[1] = dataclasses.replace(out[1], tsc=5)
    out += [synth.StreamSpec(seed=21, n_samples=N_SYNC, noise_only=True),
            synth.StreamSpec(seed=22, n_samples=N_SYNC, snr_db=0.0, sampling_ppm=5, carrier_ppm=3),
            synth.StreamSpec(seed=24, n_samples=N_SYNC, sampling_ppm=10, carrier_ppm=-20, start_offset=123456.0)]
    out.append(synth.StreamSpec(seed=264, n_samples=N_SYNC, start_offset=492899.0, sampling_ppm=-0.9354346474586492,
                                carrier_ppm=-6.129562661063993, drop_fcch=(10,)))
    return out


@pytest.fixture(scope="module")
def batch(gpu, coef, tpl):
    specs = _specs()
    raw = synth.generate_batch(specs).numpy()
    got = gpu.calibrate_demod_batch(raw, CARRIER, tpl, coef)
    ref = [sync_demod_stream(raw[d], CARRIER, tpl, coef) for d in range(len(specs))]
    return raw, got, ref


def _check_demod(g, r):
    assert g["demod_flags"] == r["demod_flags"]
    for key in ("sch", "fcch"):
        assert (g[key] is None) == (r[key] is None)
    if r["sch"] is not None:
        gs, rs = g["sch"], r["sch"]
        np.testing.assert_array_equal(gs["sch_ok"], rs["sch_ok"])
        for k in ("demod_bits", "bits_to_decoder", "corr_val"):
            np.testing.assert_array_equal(gs[k], rs[k])
    if r["fcch"] is not None:
        gf, rf = g["fcch"], r["fcch"]
        np.testing.assert_array_equal(gf["max_idx"], rf["max_idx"])
        assert np.array_equal(np.isnan(gf["freq"]), np.isnan(rf["freq"]))
        ok = ~np.isnan(rf["freq"])
        if ok.any():
            assert np.max(np.abs(gf["freq"][ok] - rf["freq"][ok])) < 1e-6
            assert np.max(np.abs(gf["snr"][ok] - rf["snr"][ok])) < 1e-9
        if math.isnan(rf["mean_freq"]):
            assert math.isnan(gf["mean_freq"]) and math.isnan(gf["carrier_ppm"])
        else:
            assert abs(gf["mean_freq"] - rf["mean_freq"]) < 1e-6 and abs(gf["carrier_ppm"] - rf["carrier_ppm"]) < 1e-9


@pytest.mark.gpu
def test_demod_batch_matches_oracle(batch):
    raw, got, ref = batch
    assert len(got) >= 8
    for g, r in zip(got, ref):
        assert np.array_equal(g["pos_info"], r["pos_info"])
        _check_demod(g, r)
    flags = [r["demod_flags"] for r in ref]
    assert any(f & 1 for f in flags), "no stream without pos_info"
    assert any(f & 2 for f in flags), "no stream with pos_info but no r_correct"
    assert any(f == 0 for f in flags), "no stream demodulated in full"
    assert any(r["fcch"] is not None and np.isfinite(r["fcch"]["mean_freq"]) for r in ref)


@pytest.mark.gpu
def test_calibration_outputs_unchanged(gpu, batch, coef, tpl):
    from gsmcal._lib import DemodResult, StreamResult, lib
    raw = batch[0]
    D, n_iq = raw.shape[0], raw.shape[1] // 2
    cap = gpu.max_bursts(n_iq)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)                                       # noqa: E731
    outs = []
    for demod in (False, True):
        res = (StreamResult * D)()
        arr = [np.full((D, cap), 7.0), np.full((D, cap), 7.0), np.full((D, cap), 7.0), np.full((D, 6 * cap, 2), 7.0)]
        common = [vp(raw), 0, n_iq, D, CARRIER, vp(tpl), vp(coef), len(coef), 8, 8, C.cast(res, C.c_void_p)] + [vp(a) for a in arr] + [None]
        if demod:
            dem = (DemodResult * D)()
            rc = lib().gsmcal_calibrate_demod_batch(*common, C.cast(dem, C.c_void_p), None, None, None, None, None, None, None)
        else:
            rc = lib().gsmcal_calibrate_batch(*common)
        assert rc == 0
        outs.append((bytes(res), [a.tobytes() for a in arr]))
    assert outs[0] == outs[1]


@pytest.mark.gpu
def test_drop_in_demodulators_on_materialised_r_correct(gpu, batch, coef, tpl):
    raw, got, _ = batch
    D, n_iq = raw.shape[0], raw.shape[1] // 2
    r_correct = np.zeros((D, n_iq), dtype=np.complex128)
    cal = gpu.calibrate_batch(raw, CARRIER, tpl, coef, r_correct=r_correct)
    n_checked = 0
    for d in range(D):
        g, n3 = got[d], cal[d]["r_len"][2]
        if g["sch"] is None or n3 < 0:
            continue
        r3, pinfo = r_correct[d, :n3], cal[d]["pos_info"]
        srows = pinfo[pinfo[:, 1] == 1][g["sch"]["sch_ok"]]
        if len(srows):
            s = gpu.SCH_demod(r3, srows, tpl, 8)
            np.testing.assert_array_equal(g["sch"]["demod_bits"][g["sch"]["sch_ok"]], s["demod_bits"])
            np.testing.assert_array_equal(g["sch"]["corr_val"][g["sch"]["sch_ok"]], s["corr_val"])
            n_checked += 1
        fok = ~np.isnan(g["fcch"]["freq"])
        if fok.any():
            f = gpu.FCCH_demod(r3, pinfo[pinfo[:, 1] == 0][fok], 8, CARRIER)
            assert np.max(np.abs(g["fcch"]["freq"][fok] - f["freq"])) < 1e-6
            np.testing.assert_array_equal(g["fcch"]["max_idx"][fok], f["max_idx"])
    assert n_checked >= 2


def _same(a, b):
    assert a["demod_flags"] == b["demod_flags"]
    for key in ("sch", "fcch"):
        assert (a[key] is None) == (b[key] is None)
        if a[key] is not None:
            for k in a[key]:
                np.testing.assert_array_equal(a[key][k], b[key][k])


@pytest.mark.gpu
def test_stream_independence_and_device_input(gpu, batch, coef, tpl):
    torch = pytest.importorskip("torch")
    raw, got, _ = batch
    D = raw.shape[0]
    alone = gpu.calibrate_demod_batch(raw[2:3], CARRIER, tpl, coef)[0]
    _same(alone, got[2])
    perm = np.random.default_rng(3).permutation(D)
    big = np.concatenate([raw[perm], raw[perm[::-1]]])                                 # 2D streams: several stream groups
    shuffled = gpu.calibrate_demod_batch(big, CARRIER, tpl, coef)
    for i, d in enumerate(perm):
        _same(shuffled[i], got[d])
        _same(shuffled[2 * D - 1 - i], got[d])
    dev = torch.from_numpy(raw.copy()).cuda()
    torch.cuda.synchronize()
    on_dev = gpu.calibrate_demod_batch(None, CARRIER, tpl, coef, device_ptr=dev.data_ptr(), n_iq=raw.shape[1] // 2, n_streams=D)
    for a, b in zip(on_dev, got):
        _same(a, b)


@pytest.mark.gpu
def test_stage_timing_reports_demod(gpu, batch, coef, tpl):
    from gsmcal._lib import lib
    raw = batch[0]
    lib().gsmcal_debug_set(3, 1)
    try:
        gpu.calibrate_demod_batch(raw[:4], CARRIER, tpl, coef)
        ms = gpu.api.last_batch_stage_ms()
        assert list(ms) == list(gpu.api.STAGE_NAMES) and ms["demod"] > 0
        gpu.calibrate_batch(raw[:4], CARRIER, tpl, coef)
        assert len(gpu.api.last_batch_stage_ms()) == 6
    finally:
        lib().gsmcal_debug_set(3, 4)


@pytest.mark.gpu
def test_full_length_streams_match_oracle(gpu, coef, tpl):
    torch = pytest.importorskip("torch")
    # seed 132: the last SCH row's equaliser window runs past the end of r_correct (sch_ok = 0, GSMCAL_DEMOD_SCH_RANGE)
    specs = [synth.random_spec(seed, N_10S) for seed in (101, 132)]
    raw = synth.generate_batch(specs, device="cuda")
    torch.cuda.synchronize()
    got = gpu.calibrate_demod_batch(None, CARRIER, tpl, coef, device_ptr=raw.data_ptr(), n_iq=N_10S, n_streams=2)
    host = raw.cpu().numpy()
    refs = [sync_demod_stream(host[d], CARRIER, tpl, coef) for d in range(2)]
    for d in range(2):
        assert refs[d]["demod_flags"] in (0, 4) and len(refs[d]["sch"]["sch_ok"]) > 100
        _check_demod(got[d], refs[d])
    assert refs[0]["demod_flags"] == 0 and refs[1]["demod_flags"] == 4
    bad = ~got[1]["sch"]["sch_ok"]
    assert bad.sum() >= 1 and not got[1]["sch"]["demod_bits"][bad].any() and not got[1]["sch"]["corr_val"][bad].any()


@pytest.mark.gpu
def test_mex_gsm_calibrate_demod_batch(gpu, built_lib, tmp_path, batch, coef, tpl):
    raw, got, _ = batch
    a = np.ascontiguousarray(raw[:3].T)                                                # 2N x D uint8
    (tmp_path / "raw.bin").write_bytes(a.tobytes(order="F"))
    src = tmp_path / "h.c"
    tp = ",".join("%r" % v for v in np.asarray(tpl).real.tolist())
    ti = ",".join("%r" % v for v in np.asarray(tpl).imag.tolist())
    cf = ",".join("%r" % v for v in coef.tolist())
    src.write_text(r'''#include "mex.h"
#include "gsmcal.h"
static const double tre[] = {%s}, tim[] = {%s}, cf[] = {%s};
int main(int argc, char **argv) {
    size_t rows = %d, D = 3;
    size_t dims[2] = {rows, D};
    mxArray *raw = mxCreateNumericArray(2, dims, mxUINT8_CLASS, mxREAL);
    FILE *f = fopen(argv[1], "rb"); if (fread(mxGetData(raw), 1, rows * D, f) != rows * D) return 5; fclose(f);
    mxArray *t = mxCreateDoubleMatrix(512, 1, mxCOMPLEX), *c = mxCreateDoubleMatrix(1, 47, mxREAL);
    for (int i = 0; i < 512; ++i) { mxGetPr(t)[i] = tre[i]; mxGetPi(t)[i] = tim[i]; }
    for (int i = 0; i < 47; ++i) mxGetPr(c)[i] = cf[i];
    mxArray *out[6]; const mxArray *rhs[4] = {raw, mxCreateDoubleScalar(%r), t, c};
    mexFunction(6, out, 4, rhs);
    for (size_t d = 0; d < D; ++d) {
        mxArray *b = mxGetField(out[4], d, "demod_bits"), *ok = mxGetField(out[4], d, "sch_ok"), *fr = mxGetField(out[5], d, "freq");
        printf("D %%zu %%g %%zu %%zu %%.17g\n", d, mxGetPr(mxGetField(out[4], d, "flags"))[0], mxGetN(b), mxGetN(fr), mxGetPr(mxGetField(out[5], d, "mean_freq"))[0]);
        for (size_t i = 0; i < 148 * mxGetN(b); ++i) printf("%%d", (int)mxGetPr(b)[i]);
        printf("\n");
        for (size_t i = 0; i < mxGetN(ok); ++i) printf("%%d", (int)mxGetPr(ok)[i]);
        printf("\n");
    }
    return 0;
}
''' % (tp, ti, cf, a.shape[0], CARRIER))
    exe = tmp_path / "h"
    libdir = os.path.dirname(built_lib)
    subprocess.run(["gcc", "-std=c11", "-Wno-unused-function", "-DGSMCAL_MEX_gsm_calibrate_demod_batch", f"-I{MEX}/stub", f"-I{ROOT}/include", str(src),
                    os.path.join(MEX, "gsmcal_mex.c"), f"-L{libdir}", "-lgsmcal", f"-Wl,-rpath,{libdir}", "-lm", "-o", str(exe)], check=True)
    lines = subprocess.run([str(exe), str(tmp_path / "raw.bin")], capture_output=True, text=True, check=True).stdout.split("\n")
    for d in range(3):
        head, bits, ok = lines[3 * d].split(), lines[3 * d + 1], lines[3 * d + 2]
        g = got[d]
        assert int(float(head[2])) == g["demod_flags"]
        n_sch = 0 if g["sch"] is None else len(g["sch"]["sch_ok"])
        n_fcch = 0 if g["fcch"] is None else len(g["fcch"]["freq"])
        assert int(head[3]) == n_sch and int(head[4]) == n_fcch
        if n_sch:
            assert bits == "".join(str(int(v)) for v in g["sch"]["demod_bits"].ravel())
            assert ok == "".join(str(int(v)) for v in g["sch"]["sch_ok"])
        if g["fcch"] is not None and np.isfinite(g["fcch"]["mean_freq"]):
            assert abs(float(head[5]) - g["fcch"]["mean_freq"]) < 1e-9
