"""gsmcal_calibrate_demod_bcch_batch: gsmcal_calibrate_demod_batch followed by BCCH_demod (gsm_sync_demod.m:146) on every stream's
r_correct, evaluated from the uint8 capture.  CPU: record layout and flags, export, argument checks, the MEX gateway against the stub.
GPU: parity with the oracle chain followed by oracle.BCCH_demod (flags equal, carrier ppm 1e-9, |corr| 1e-8 relative to the burst's
largest magnitude, nts_idx equal where the oracle's top two are apart), the carrier ppm equal to FCCH_demod's, every other output
byte-identical to gsmcal_calibrate_demod_batch, the drop-in on calibrate_batch_r's r_correct, stream independence, full-length streams,
the stage timing, the MEX gateway end to end and the rtl_tcp ingest."""
import ctypes as C
import dataclasses
import math
import os
import subprocess

import numpy as np
import pytest

import gsmcal_oracle as oracle
from gsmcal import synth
from test_gpu_demod_batch import _specs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MEX = os.path.join(ROOT, "multi-rtl-sdr-calibration_b200", "mex")
FS = oracle.SYMBOL_RATE * 8
CARRIER = 957.4e6
N_10S = 21666667


# ---- CPU -----------------------------------------------------------------------------------------------------------------------
def test_bcch_result_layout():
    from gsmcal._lib import BcchResult
    assert C.sizeof(BcchResult) == 272
    assert [getattr(BcchResult, f).offset for f in ("carrier_ppm", "nts_idx", "flags", "corr_abs")] == [0, 8, 12, 16]
    hdr = open(os.path.join(ROOT, "include", "gsmcal.h")).read()
    for name, v in (("NO_POS_INFO", 1), ("FEW_BCCH", 2), ("FCCH_RANGE", 4), ("TRAIN_RANGE", 8)):
        assert f"#define GSMCAL_BCCH_{name}" in hdr and hdr.split(f"#define GSMCAL_BCCH_{name}")[1].split()[0] == str(v)


def test_bcch_batch_symbol_exported(built_lib):
    from gsmcal import _lib
    assert "gsmcal_calibrate_demod_bcch_batch" in _lib.SIGNATURES
    assert hasattr(_lib.lib(), "gsmcal_calibrate_demod_bcch_batch")
    out = subprocess.run(["nm", "-D", "--defined-only", built_lib], capture_output=True, text=True).stdout
    assert " T gsmcal_calibrate_demod_bcch_batch" in out


def _call(raw, n_iq, D, osr=8, nts=True, bcch=True):
    from gsmcal._lib import BcchResult, DemodResult, StreamResult, lib
    tpl = np.ones(64 * osr, dtype=np.complex128)
    seq = np.ones((8, 26 * max(osr, 1)), dtype=np.complex128)
    coef = oracle.fir1(46, 200e3 / FS)
    res, dem, bc = (StreamResult * max(D, 1))(), (DemodResult * max(D, 1))(), (BcchResult * max(D, 1))()
    vp = lambda a: a.ctypes.data_as(C.c_void_p)                                       # noqa: E731
    return lib().gsmcal_calibrate_demod_bcch_batch(vp(raw), 0, n_iq, D, CARRIER, vp(tpl), vp(coef), len(coef), osr, 8,
                                                   C.cast(res, C.c_void_p), None, None, None, None, None,
                                                   C.cast(dem, C.c_void_p), None, None, None, None, None, None, None,
                                                   vp(seq) if nts else None, C.cast(bc, C.c_void_p) if bcch else None)


def test_bcch_batch_bad_arguments(built_lib):
    raw = np.zeros((1, 2 * 300000), dtype=np.uint8)
    assert _call(raw, 300000, 1, nts=False) == -1
    assert _call(raw, 300000, 1, bcch=False) == -1
    assert _call(raw, 300000, 1, osr=0) == -1
    assert _call(raw, 300000, 1, osr=9) == -1


def test_bcch_batch_needs_a_device(built_lib):
    import gsmcal
    if gsmcal.device_count() > 0:
        pytest.skip("a CUDA device is present")
    raw = np.zeros((1, 2 * 300000), dtype=np.uint8)
    assert _call(raw, 300000, 1) == -2
    with pytest.raises(gsmcal.GsmcalError) as e:
        gsmcal.calibrate_demod_batch(raw, CARRIER, np.ones(512, complex), oracle.fir1(46, 0.09),
                                     normal_training_sequence=np.ones((208, 8), complex))
    assert e.value.code == -2


def test_bcch_gateway_compiles_against_stub(tmp_path):
    obj = tmp_path / "g.o"
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Wno-unused-function", "-c", "-DGSMCAL_MEX_gsm_calibrate_demod_batch", f"-I{MEX}/stub",
                    f"-I{ROOT}/include", os.path.join(MEX, "gsmcal_mex.c"), "-o", str(obj)], check=True)
    sym = subprocess.run(["nm", str(obj)], capture_output=True, text=True).stdout
    assert " T mexFunction" in sym and " U gsmcal_calibrate_demod_bcch_batch" in sym and " U gsmcal_calibrate_demod_batch" in sym


def test_bcch_gateway_needs_the_fifth_input_for_seven_outputs(built_lib, tmp_path):
    src = tmp_path / "h.c"
    src.write_text(r'''#include "mex.h"
int main(void) {
    size_t dims[2] = {600000, 1};
    mxArray *raw = mxCreateNumericArray(2, dims, mxUINT8_CLASS, mxREAL);
    mxArray *t = mxCreateDoubleMatrix(512, 1, mxCOMPLEX), *c = mxCreateDoubleMatrix(1, 47, mxREAL);
    mxArray *out[7]; const mxArray *rhs[4] = {raw, mxCreateDoubleScalar(957.4e6), t, c};
    mexFunction(7, out, 4, rhs);
    return 0;
}
''')
    exe = tmp_path / "h"
    libdir = os.path.dirname(built_lib)
    subprocess.run(["gcc", "-std=c11", "-Wno-unused-function", "-DGSMCAL_MEX_gsm_calibrate_demod_batch", f"-I{MEX}/stub", f"-I{ROOT}/include", str(src),
                    os.path.join(MEX, "gsmcal_mex.c"), f"-L{libdir}", "-lgsmcal", f"-Wl,-rpath,{libdir}", "-lm", "-o", str(exe)], check=True)
    p = subprocess.run([str(exe)], capture_output=True, text=True)
    assert p.returncode == 3 and "gsmcal:nargin" in p.stderr


# ---- GPU -----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def coef():
    return oracle.fir1(46, 200e3 / FS)


@pytest.fixture(scope="module")
def tpl():
    return oracle.gsm_SCH_training_sequence_gen(8)


@pytest.fixture(scope="module")
def nts():
    return oracle.gsm_normal_training_sequence_gen(8)


def bcch_reference(res, nts, osr=8):
    """Reference of one stream's BCCH record from oracle.calibrate_stream's outputs: the sentinels of gsmcal_calibrate_demod_bcch_batch
    in their order, then oracle.BCCH_demod(r_final, ...); a training window outside r_final gets a NaN column and nts_idx -1."""
    pinfo, r = np.asarray(res["pos_info"], dtype=np.float64).reshape(-1, 2), res["r_final"]
    if pinfo.size > 0 and np.all(pinfo == -1):
        return dict(flags=1, carrier_ppm=-1.0, nts_idx=-1, corr_abs=None)
    bpos = pinfo[pinfo[:, 1] == 2, 0]
    if len(bpos) < 4:
        return dict(flags=2, carrier_ppm=-1.0, nts_idx=-1, corr_abs=None)
    assert r is not None                          # carrier_correct_post_SCH fails after a valid pos_info only with < 4 BCCH rows
    n, L = len(r), 26 * osr
    fpos = pinfo[pinfo[:, 1] == 0, 0]
    if len(fpos) == 0 or not all(p >= 1 and p + 148 * osr - 1 <= n for p in fpos):
        return dict(flags=4, carrier_ppm=math.nan, nts_idx=-1, corr_abs=None)
    ok = [p + 61 * osr >= 1 and p + 61 * osr + L - 1 <= n for p in bpos[:4]]
    if all(ok):
        cp, idx, mag = oracle.BCCH_demod(r, pinfo, nts, osr, CARRIER)
        return dict(flags=0, carrier_ppm=cp, nts_idx=idx, corr_abs=mag)
    rb, cp = oracle.carrier_correct_post_SCH(r, pinfo, osr, CARRIER)
    mag = np.full((8, 4), np.nan)
    for b, p in enumerate(bpos[:4]):
        if ok[b]:
            s0 = int(p) + 61 * osr - 1
            mag[:, b] = np.abs(np.asarray(nts).conj().T @ rb[s0:s0 + L])
    return dict(flags=8, carrier_ppm=cp, nts_idx=-1, corr_abs=mag)


def _separated(mag):
    """the oracle's first maximum of every column is ahead of the runner-up by more than 1e-9 relative"""
    s = -np.sort(-mag, axis=0)
    return bool(np.all((s[0] - s[1]) > 1e-9 * s[0]))


def _check_bcch(g, r):
    assert g["flags"] == r["flags"]
    if r["flags"] in (1, 2):
        assert g["carrier_ppm"] == -1.0 and g["nts_idx"] == -1 and g["corr_abs"] is None
        return
    if r["flags"] == 4:
        assert math.isnan(g["carrier_ppm"]) and g["nts_idx"] == -1 and g["corr_abs"] is None
        return
    assert abs(g["carrier_ppm"] - r["carrier_ppm"]) < 1e-9
    ga, ra = g["corr_abs"], r["corr_abs"]
    assert ga.shape == (8, 4)
    assert np.array_equal(np.isnan(ga), np.isnan(ra))
    for b in range(4):
        if not np.isnan(ra[:, b]).any():
            assert np.max(np.abs(ga[:, b] - ra[:, b])) <= 1e-8 * np.max(ra[:, b])
    if r["flags"] == 8:
        assert g["nts_idx"] == -1
    elif _separated(ra):
        assert g["nts_idx"] == r["nts_idx"]


@pytest.fixture(scope="module")
def batch(gpu, coef, tpl, nts):
    specs = _specs()
    raw = synth.generate_batch(specs).numpy()
    got = gpu.calibrate_demod_batch(raw, CARRIER, tpl, coef, normal_training_sequence=gpu.gsm_normal_training_sequence_gen(8))
    cal = [oracle.calibrate_stream(raw[d], CARRIER, tpl, coef) for d in range(len(specs))]
    ref = [bcch_reference(c, nts) for c in cal]
    return raw, got, ref, cal


@pytest.mark.gpu
def test_bcch_batch_matches_oracle(batch):
    raw, got, ref, cal = batch
    assert len(got) >= 8
    for g, r, c in zip(got, ref, cal):
        assert np.array_equal(g["pos_info"], c["pos_info"])
        _check_bcch(g["bcch"], r)
        if g["demod_flags"] & 2:
            assert g["bcch"]["flags"] == 2
    assert got[0]["bcch"]["nts_idx"] == 1 and got[1]["bcch"]["nts_idx"] == 6         # tsc 0 and tsc 5
    flags = [r["flags"] for r in ref]
    assert 0 in flags and 1 in flags and 2 in flags


@pytest.mark.gpu
def test_bcch_carrier_ppm_is_fcch_demod_carrier_ppm(batch):
    got = batch[1]
    n = 0
    for g in got:
        if g["bcch"]["flags"] == 0:
            assert np.float64(g["bcch"]["carrier_ppm"]).tobytes() == np.float64(g["fcch"]["carrier_ppm"]).tobytes()
            n += 1
    assert n >= 2


def _raw_call(raw, nts=None):
    """every output of gsmcal_calibrate_demod_batch (nts None) or gsmcal_calibrate_demod_bcch_batch, as bytes; per-row demod outputs
    only for the rows the demod record says exist"""
    from gsmcal import api
    from gsmcal._lib import BcchResult, DemodResult, StreamResult, lib
    coef = oracle.fir1(46, 200e3 / FS)
    tpl = oracle.gsm_SCH_training_sequence_gen(8)
    D, n_iq = raw.shape[0], raw.shape[1] // 2
    cap = api.max_bursts(n_iq)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)                                       # noqa: E731
    res, dem = (StreamResult * D)(), (DemodResult * D)()
    cal = [np.full((D, cap), 7.0), np.full((D, cap), 7.0), np.full((D, cap), 7.0), np.full((D, 6 * cap, 2), 7.0)]
    ok, bits, dec = np.full((D, cap), 7, np.uint8), np.full((D, cap, 148), 7, np.uint8), np.full((D, cap, 148), 7, np.uint8)
    corr, freq, snr, idx = np.full((D, cap, 85), 7.0), np.full((D, cap), 7.0), np.full((D, cap), 7.0), np.full((D, cap), 7.0)
    args = [vp(raw), 0, n_iq, D, CARRIER, vp(tpl), vp(coef), len(coef), 8, 8, C.cast(res, C.c_void_p)] + [vp(a) for a in cal] + [None]
    args += [C.cast(dem, C.c_void_p)] + [vp(a) for a in (ok, bits, dec, corr, freq, snr, idx)]
    bc = None
    if nts is None:
        rc = lib().gsmcal_calibrate_demod_batch(*args)
    else:
        bc = (BcchResult * D)()
        rc = lib().gsmcal_calibrate_demod_bcch_batch(*args, vp(np.ascontiguousarray(nts.T)), C.cast(bc, C.c_void_p))
    assert rc == 0
    rows = []
    for d in range(D):
        ns, nf = max(dem[d].n_sch, 0), max(dem[d].n_fcch, 0)
        rows.append(b"".join(a[d, :ns].tobytes() for a in (ok, bits, dec, corr)) + b"".join(a[d, :nf].tobytes() for a in (freq, snr, idx)))
    return (bytes(res), [a.tobytes() for a in cal], bytes(dem), rows), bc


@pytest.mark.gpu
def test_other_outputs_unchanged(gpu, batch, nts):
    raw = batch[0]
    plain, _ = _raw_call(raw)
    with_bcch, bc = _raw_call(raw, np.asarray(nts, dtype=np.complex128))
    assert plain == with_bcch
    assert any(bc[d].flags == 0 for d in range(raw.shape[0]))


@pytest.mark.gpu
def test_drop_in_bcch_demod_on_materialised_r_correct(gpu, batch, coef, tpl):
    raw, got, _, _ = batch
    D, n_iq = raw.shape[0], raw.shape[1] // 2
    r_correct = np.zeros((D, n_iq), dtype=np.complex128)
    cal = gpu.calibrate_batch(raw, CARRIER, tpl, coef, r_correct=r_correct)
    seq = gpu.gsm_normal_training_sequence_gen(8)
    n_checked = 0
    for d in range(D):
        g = got[d]["bcch"]
        if g["flags"] != 0:
            continue
        n3 = cal[d]["r_len"][2]
        cp, idx, mag = gpu.BCCH_demod(r_correct[d, :n3], cal[d]["pos_info"], seq, 8, CARRIER)
        assert abs(g["carrier_ppm"] - cp) < 1e-9
        for b in range(4):
            assert np.max(np.abs(g["corr_abs"][:, b] - mag[:, b])) <= 1e-8 * np.max(mag[:, b])
        if _separated(mag):
            assert g["nts_idx"] == idx
        n_checked += 1
    assert n_checked >= 2


def _bcch_bytes(item):
    b = item["bcch"]
    return (np.float64(b["carrier_ppm"]).tobytes(), b["nts_idx"], b["flags"], None if b["corr_abs"] is None else b["corr_abs"].tobytes())


@pytest.mark.gpu
def test_bcch_stream_independence_and_device_input(gpu, batch, coef, tpl):
    torch = pytest.importorskip("torch")
    raw, got, _, _ = batch
    D = raw.shape[0]
    seq = gpu.gsm_normal_training_sequence_gen(8)
    alone = gpu.calibrate_demod_batch(raw[1:2], CARRIER, tpl, coef, normal_training_sequence=seq)[0]
    assert _bcch_bytes(alone) == _bcch_bytes(got[1])
    perm = np.random.default_rng(5).permutation(D)
    big = np.concatenate([raw[perm], raw[perm[::-1]]])                                 # 2D streams: several stream groups
    shuffled = gpu.calibrate_demod_batch(big, CARRIER, tpl, coef, normal_training_sequence=seq)
    for i, d in enumerate(perm):
        assert _bcch_bytes(shuffled[i]) == _bcch_bytes(got[d])
        assert _bcch_bytes(shuffled[2 * D - 1 - i]) == _bcch_bytes(got[d])
    dev = torch.from_numpy(raw.copy()).cuda()
    torch.cuda.synchronize()
    on_dev = gpu.calibrate_demod_batch(None, CARRIER, tpl, coef, device_ptr=dev.data_ptr(), n_iq=raw.shape[1] // 2, n_streams=D,
                                       normal_training_sequence=seq)
    for a, b in zip(on_dev, got):
        assert _bcch_bytes(a) == _bcch_bytes(b)


@pytest.mark.gpu
def test_bcch_stage_timing_reports_demod(gpu, batch, coef, tpl):
    from gsmcal._lib import lib
    raw = batch[0]
    lib().gsmcal_debug_set(3, 1)
    try:
        gpu.calibrate_demod_batch(raw[:4], CARRIER, tpl, coef, normal_training_sequence=gpu.gsm_normal_training_sequence_gen(8))
        ms = gpu.api.last_batch_stage_ms()
        assert list(ms) == list(gpu.api.STAGE_NAMES) and len(ms) == 7 and ms["demod"] > 0
    finally:
        lib().gsmcal_debug_set(3, 4)


@pytest.mark.gpu
def test_bcch_full_length_streams_match_oracle(gpu, coef, tpl, nts):
    torch = pytest.importorskip("torch")
    tscs = (3, 6)
    specs = [dataclasses.replace(synth.random_spec(seed, N_10S), tsc=t) for seed, t in zip((101, 132), tscs)]
    raw = synth.generate_batch(specs, device="cuda")
    torch.cuda.synchronize()
    got = gpu.calibrate_demod_batch(None, CARRIER, tpl, coef, device_ptr=raw.data_ptr(), n_iq=N_10S, n_streams=2,
                                    normal_training_sequence=gpu.gsm_normal_training_sequence_gen(8))
    host = raw.cpu().numpy()
    for d in range(2):
        ref = bcch_reference(oracle.calibrate_stream(host[d], CARRIER, tpl, coef), nts)
        assert ref["flags"] == 0
        _check_bcch(got[d]["bcch"], ref)
        assert got[d]["bcch"]["nts_idx"] == tscs[d] + 1


@pytest.mark.gpu
def test_mex_gsm_calibrate_demod_batch_bcch(gpu, built_lib, tmp_path, batch, tpl):
    raw, got, _, _ = batch
    pick = [0, 1, 4, 7]                                                                # flags 0, 0, 1 (noise only), 2 (dropped FCCH)
    a = np.ascontiguousarray(raw[pick].T)                                              # 2N x D uint8
    (tmp_path / "raw.bin").write_bytes(a.tobytes(order="F"))
    seq = gpu.gsm_normal_training_sequence_gen(8)                                     # (208, 8)
    coef = oracle.fir1(46, 200e3 / FS)
    fmt = lambda v: ",".join("%r" % x for x in np.asarray(v).ravel(order="F").tolist())     # noqa: E731
    src = tmp_path / "h.c"
    src.write_text(r'''#include "mex.h"
#include "gsmcal.h"
static const double tre[] = {%s}, tim[] = {%s}, nre[] = {%s}, nim[] = {%s}, cf[] = {%s};
int main(int argc, char **argv) {
    size_t rows = %d, D = %d;
    size_t dims[2] = {rows, D};
    mxArray *raw = mxCreateNumericArray(2, dims, mxUINT8_CLASS, mxREAL);
    FILE *f = fopen(argv[1], "rb"); if (fread(mxGetData(raw), 1, rows * D, f) != rows * D) return 5; fclose(f);
    mxArray *t = mxCreateDoubleMatrix(512, 1, mxCOMPLEX), *c = mxCreateDoubleMatrix(1, 47, mxREAL), *n = mxCreateDoubleMatrix(208, 8, mxCOMPLEX);
    for (int i = 0; i < 512; ++i) { mxGetPr(t)[i] = tre[i]; mxGetPi(t)[i] = tim[i]; }
    for (int i = 0; i < 8 * 208; ++i) { mxGetPr(n)[i] = nre[i]; mxGetPi(n)[i] = nim[i]; }
    for (int i = 0; i < 47; ++i) mxGetPr(c)[i] = cf[i];
    mxArray *out[7]; const mxArray *rhs[5] = {raw, mxCreateDoubleScalar(%r), t, c, n};
    mexFunction(7, out, 5, rhs);
    for (size_t d = 0; d < D; ++d) {
        mxArray *ca = mxGetField(out[6], d, "corr_abs");
        printf("%%g %%g %%.17g %%zu %%zu", mxGetPr(mxGetField(out[6], d, "flags"))[0], mxGetPr(mxGetField(out[6], d, "idx"))[0],
               mxGetPr(mxGetField(out[6], d, "carrier_ppm"))[0], mxGetM(ca), mxGetN(ca));
        for (int i = 0; i < 32; ++i) printf(" %%.17g", mxGetPr(ca)[i]);
        printf("\n");
    }
    return 0;
}
''' % (fmt(np.asarray(tpl).real), fmt(np.asarray(tpl).imag), fmt(seq.real), fmt(seq.imag), fmt(coef), a.shape[0], len(pick), CARRIER))
    exe = tmp_path / "h"
    libdir = os.path.dirname(built_lib)
    subprocess.run(["gcc", "-std=c11", "-Wno-unused-function", "-DGSMCAL_MEX_gsm_calibrate_demod_batch", f"-I{MEX}/stub", f"-I{ROOT}/include", str(src),
                    os.path.join(MEX, "gsmcal_mex.c"), f"-L{libdir}", "-lgsmcal", f"-Wl,-rpath,{libdir}", "-lm", "-o", str(exe)], check=True)
    lines = subprocess.run([str(exe), str(tmp_path / "raw.bin")], capture_output=True, text=True, check=True).stdout.strip().split("\n")
    assert len(lines) == len(pick)
    seen = set()
    for line, d in zip(lines, pick):
        v = line.split()
        b = got[d]["bcch"]
        assert int(float(v[0])) == b["flags"] and int(float(v[1])) == b["nts_idx"] and v[3:5] == ["8", "4"]
        assert np.float64(float(v[2])).tobytes() == np.float64(b["carrier_ppm"]).tobytes()
        mag = np.array([float(x) for x in v[5:]]).reshape(4, 8).T
        if b["corr_abs"] is None:
            assert np.isnan(mag).all()
        else:
            np.testing.assert_array_equal(mag, b["corr_abs"])
        seen.add(b["flags"])
    assert seen == {0, 1, 2}


@pytest.mark.gpu
def test_ingest_calibrate_demod_equals_direct(gpu):
    import torch
    from gsmcal import ingest
    from gsmcal.rtl_tcp_replay import ReplayDongle
    N = 1_020_000                                 # gsm_sync_demod.m:23-29
    tscs = (2, 7, 4)
    specs = [dataclasses.replace(synth.random_spec(seed, 2 * N + 8), tsc=t) for seed, t in zip((1, 2, 3), tscs)]
    raw = synth.generate_batch(specs, device="cuda").cpu().numpy()
    srvs = [ReplayDongle(raw[d]) for d in range(len(specs))]
    try:
        res = ingest.calibrate_from_dongles([(s.host, s.port) for s in srvs], N, CARRIER, n_captures=1, demod=True)[0]
    finally:
        for s in srvs:
            s.close()
    direct_in = np.stack([s.expected(2 * N - 12, 2 * N) for s in srvs])
    direct = gpu.calibrate_demod_batch(direct_in, CARRIER, gpu.gsm_SCH_training_sequence_gen(8), gpu.fir1(46, 200e3 / FS),
                                       normal_training_sequence=gpu.gsm_normal_training_sequence_gen(8))
    assert len(res) == len(direct) == 3
    for a, b in zip(res, direct):
        np.testing.assert_array_equal(a["pos_info"], b["pos_info"])
        assert a["demod_flags"] == b["demod_flags"]
        assert _bcch_bytes(a) == _bcch_bytes(b)
    assert sum(r["bcch"]["nts_idx"] == t + 1 for r, t in zip(res, tscs)) >= 2
    torch.cuda.synchronize()
