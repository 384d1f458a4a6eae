"""gsmcal_calibrate_sysinfo_batch: the cell call, then every BCCH block of pos_info decoded to its System Information and, from SI3, the
cell's CGI.  CPU: the record and its flags, argument checks without a launch, the pieces of the restatement in bcch_decode_oracle.py
(interleaver, Fire code, Viterbi, SI3 parse), a decode of the generator's own noise-free bursts and the accuracy on the oracle chain at
0.47 s.  GPU: parity with the restatement on the GPU's own r_correct, byte-identical outputs and launches of the cell call, stream
independence and device input, drifting 10 s streams, two dongles on one cell, the stage timing and the rtl_tcp ingest."""
import ctypes as C
import dataclasses
import os
import subprocess

import numpy as np
import pytest

import bcch_decode_oracle as B
import cell_sync_oracle as CS
import gsmcal_oracle as oracle
from gsmcal import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MEX = os.path.join(ROOT, "multi-rtl-sdr-calibration_b200", "mex")
FS = oracle.SYMBOL_RATE * 8
CARRIER = 957.4e6
N_SYNC = 1020000                       # gsm_sync_demod.m's 102 frames, 0.47 s
N_10S = 21666667
SEEDS = (1, 11, 28)                    # every SCH row decodes at 0.47 s (test_gpu_cell_sync.py)
EARLY_SEED = 24                        # pos_info locked about 57 samples early (DESIGN.md 6b)
CS_FILTER_DELAY = -23.0                # the channel filter's group delay: pos_info sits 23 samples behind the burst


def _cgi(seed):
    """(ci, mcc, mnc, lac, mnc_digits) of seed's synthetic cell: 2- and 3-digit MNCs alternate"""
    return 0x1000 + seed, 262 + seed % 3, seed % 100, 0x2000 + 7 * seed, 2 + seed % 2


def _si(seed):
    """SI3 on the even TCs, SI4 on the odd ones: every 0.47 s capture (two or three blocks) holds an SI3 and an SI4"""
    ci, mcc, mnc, lac, nd = _cgi(seed)
    si3, si4 = synth.si3_message(ci, mcc, mnc, lac, nd), synth.si4_message(mcc, mnc, lac, nd)
    return tuple(si3 if tc % 2 == 0 else si4 for tc in range(8))


def _spec(seed, n=N_SYNC, cell_seed=None):
    cs = seed if cell_seed is None else cell_seed
    bsic = cs % 64
    return dataclasses.replace(synth.random_spec(seed, n), bsic=bsic, tsc=bsic & 7, fn0=51 * (cs * 7919 % 50000), sysinfo=_si(cs))


def _vp(a):
    return a.ctypes.data_as(C.c_void_p)


# ---- CPU: ABI ------------------------------------------------------------------------------------------------------------------
def test_record_flags_and_export(built_lib):
    from gsmcal import _lib, api
    assert C.sizeof(_lib.SysinfoResult) == 48
    hdr = open(os.path.join(ROOT, "include", "gsmcal.h")).read()
    assert "} gsmcal_sysinfo_result;       /* 48 bytes */" in hdr
    val = lambda n: int(hdr.split("#define GSMCAL_SI_" + n)[1].split()[0])      # noqa: E731
    assert [val(n) for n in ("NO_POS_INFO", "NO_R_CORRECT", "NO_CELL", "UNCORRECTED", "NO_SI3", "SI3_DISAGREE")] == \
        [api.SI_NO_POS_INFO, api.SI_NO_R_CORRECT, api.SI_NO_CELL, api.SI_UNCORRECTED, api.SI_NO_SI3, api.SI_SI3_DISAGREE] == [1, 2, 4, 8, 16, 32]
    assert [val(n) for n in ("BLK_FN", "BLK_ROW", "BLK_FIRE", "BLK_SHORT")] == [B.BLK_FN, B.BLK_ROW, B.BLK_FIRE, B.BLK_SHORT]
    assert [val(n) for n in ("ROW_RANGE", "ROW_EDGE")] == [B.ROW_RANGE, B.ROW_EDGE]
    has = {"SI1": 0x19, "SI2": 0x1A, "SI2BIS": 0x02, "SI2TER": 0x03, "SI2QUATER": 0x07, "SI3": 0x1B, "SI4": 0x1C, "SI13": 0x00}
    assert {val("HAS_" + k): v for k, v in has.items()} == {b: t for t, b in api.SI_HAS.items()} == {b: t for t, b in B.HAS.items()}
    assert val("HAS_OTHER") == api.SI_HAS_OTHER == B.HAS_OTHER
    out = subprocess.run(["nm", "-D", "--defined-only", built_lib], capture_output=True, text=True).stdout
    assert " T gsmcal_calibrate_sysinfo_batch" in out


def _call(raw, n_iq, D, osr=8, nts=True, si=True, carrier=True, dec=True):
    from gsmcal._lib import CarrierFitResult, SchDecodeResult, StreamResult, SysinfoResult, lib
    tpl = np.ones(64 * max(osr, 1), dtype=np.complex128)
    coef = oracle.fir1(46, 200e3 / FS)
    n = max(D, 1)
    res, cf, sd, s = (StreamResult * n)(), (CarrierFitResult * n)(), (SchDecodeResult * n)(), (SysinfoResult * n)()
    t = np.ones((8, 26 * 8), dtype=np.complex128)
    return lib().gsmcal_calibrate_sysinfo_batch(_vp(raw), 0, n_iq, D, CARRIER, _vp(tpl), _vp(coef), len(coef), osr, 8, C.cast(res, C.c_void_p),
                                                None, None, None, None, None, C.cast(cf, C.c_void_p) if carrier else None, None, None, None,
                                                C.cast(sd, C.c_void_p) if dec else None, *[None] * 8, _vp(t) if nts else None,
                                                C.cast(s, C.c_void_p) if si else None, *[None] * 8)


def test_sysinfo_argument_errors_launch_nothing(built_lib):
    import gsmcal
    from gsmcal import api
    from gsmcal._lib import lib
    raw = np.zeros((1, 2 * 300000), dtype=np.uint8)
    n0 = api.launch_count()
    for osr in (0, 9, 1, 4):
        assert _call(raw, 300000, 1, osr=osr) == -1
    assert b"oversampling_ratio must be 8" in lib().gsmcal_last_error()
    for kw in (dict(nts=False), dict(si=False), dict(carrier=False), dict(dec=False)):
        assert _call(raw, 300000, 1, **kw) == -1
        assert b"calibrate_sysinfo_batch: null" in lib().gsmcal_last_error()
    assert _call(raw, 300000, 0) == -1
    tpl, coef = np.ones(512, complex), oracle.fir1(46, 0.09)
    for kw in (dict(sysinfo=True), dict(sysinfo=True, carrier_fit=True), dict(sysinfo=True, sch_decode=True),
               dict(sysinfo=True, carrier_fit=True, sch_decode=True, sch_timing=True)):
        with pytest.raises(ValueError):
            gsmcal.calibrate_batch(raw, CARRIER, tpl, coef, **kw)
    assert api.launch_count() == n0


def test_sysinfo_needs_a_device(built_lib):
    import gsmcal
    if gsmcal.device_count() > 0:
        pytest.skip("a CUDA device is present")
    raw = np.zeros((1, 2 * 300000), dtype=np.uint8)
    assert _call(raw, 300000, 1) == -2


def test_sysinfo_gateway_compiles_against_stub(tmp_path):
    obj = tmp_path / "g.o"
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Wno-unused-function", "-c", "-DGSMCAL_MEX_gsm_calibrate_sysinfo_batch", f"-I{MEX}/stub",
                    f"-I{ROOT}/include", os.path.join(MEX, "gsmcal_mex.c"), "-o", str(obj)], check=True)
    sym = subprocess.run(["nm", str(obj)], capture_output=True, text=True).stdout
    assert " T mexFunction" in sym and " U gsmcal_calibrate_sysinfo_batch" in sym and " U gsmcal_calibrate_cell_batch" not in sym
    assert "gsm_calibrate_sysinfo_batch" in open(os.path.join(MEX, "Makefile.mex")).read()


@pytest.mark.parametrize("nlhs,nrhs,nts_rows,err", [(8, 5, 208, "nargin"), (7, 4, 208, "nargin"), (7, 5, 207, "size")])
def test_sysinfo_gateway_usage_errors(built_lib, tmp_path, nlhs, nrhs, nts_rows, err):
    src = tmp_path / "h.c"
    src.write_text(r'''#include "mex.h"
int main(void) {
    size_t dims[2] = {600000, 1};
    mxArray *raw = mxCreateNumericArray(2, dims, mxUINT8_CLASS, mxREAL);
    mxArray *t = mxCreateDoubleMatrix(512, 1, mxCOMPLEX), *c = mxCreateDoubleMatrix(1, 47, mxREAL), *n = mxCreateDoubleMatrix(%d, 8, mxCOMPLEX);
    mxArray *out[8]; const mxArray *rhs[5] = {raw, mxCreateDoubleScalar(957.4e6), t, c, n};
    mexFunction(%d, out, %d, rhs);
    return 0;
}
''' % (nts_rows, nlhs, nrhs))
    exe = tmp_path / "h"
    libdir = os.path.dirname(built_lib)
    subprocess.run(["gcc", "-std=c11", "-Wno-unused-function", "-DGSMCAL_MEX_gsm_calibrate_sysinfo_batch", f"-I{MEX}/stub", f"-I{ROOT}/include",
                    str(src), os.path.join(MEX, "gsmcal_mex.c"), f"-L{libdir}", "-lgsmcal", f"-Wl,-rpath,{libdir}", "-lm", "-o", str(exe)], check=True)
    p = subprocess.run([str(exe)], capture_output=True, text=True)
    assert p.returncode == 3 and "gsmcal:" + err in p.stderr


# ---- CPU: the pieces of the restatement --------------------------------------------------------------------------------------
def test_interleaver_is_a_permutation():
    seen = {(k % 4, 2 * ((49 * k) % 57) + ((k % 8) // 4)) for k in range(456)}
    assert len(seen) == 456 and all(0 <= j < 114 for _, j in seen)
    ib = np.arange(456).reshape(4, 114)                       # distinct labels survive the round trip through the generator's mapping
    c = B.deinterleave(ib)
    assert sorted(c.tolist()) == list(range(456))


def _u(msg):
    """u(0..227) of a message: data, parity (from the generator's encoder, decoded back by the restatement) and tail"""
    u, ham = B.viterbi(B.deinterleave(synth.bcch_encode(msg)))
    assert ham == 0
    return u


def test_fire_round_trip_and_detection():
    msg = synth.si3_message(0xBEEF, 901, 70, 0x1234, 3)
    u = _u(msg)
    assert B.fire_ok(u) and B.payload(u) == msg and not u[224:].any()
    for i in range(224):                                       # every single-bit error
        v = u.copy(); v[i] ^= 1
        assert not B.fire_ok(v)
    rng = np.random.default_rng(3)
    for _ in range(200):                                       # bursts of at most 12 bits (first and last flipped)
        n = int(rng.integers(2, 13)); s = int(rng.integers(0, 224 - n + 1))
        v = u.copy(); v[s] ^= 1; v[s + n - 1] ^= 1
        v[s + 1:s + n - 1] ^= rng.integers(0, 2, n - 2)
        assert not B.fire_ok(v)


def test_viterbi_corrects_spread_errors_and_keeps_the_tie_rule():
    msg = synth.si4_message(234, 15, 0x0101)
    c = B.deinterleave(synth.bcch_encode(msg))
    bad = c.copy()
    for k in (5, 120, 240, 333, 450):
        bad[k] ^= 1
    u, ham = B.viterbi(bad)
    assert ham == 5 and B.payload(u) == msg and B.fire_ok(u)
    # one coded pair (1, 1) at step 0 from state 0: input 1 costs 0, input 0 costs 2 -> no tie; (1, 0): both inputs cost 1 from state 0,
    # and the survivors into states 0 and 1 differ only in the dropped bit, which the rule keeps at 0: an all-zero decision remains
    c2 = np.zeros(456, dtype=np.int64); c2[0] = 1
    u2, ham2 = B.viterbi(c2)
    assert ham2 == 1 and not u2.any()


@pytest.mark.parametrize("mnc,nd", [(1, 2), (1, 3), (260, 3), (99, 2)])
def test_si3_parse(mnc, nd):
    msg = synth.si3_message(0x0A0B, 310, mnc, 0xFFFE, nd)
    assert msg[1] == 0x06 and msg[2] == 0x1B and len(msg) == 23
    assert B.si3_fields(msg) == (310, mnc, nd, 0xFFFE, 0x0A0B)
    assert (msg[6] >> 4 == 0xF) == (nd == 2)


def test_decodes_the_generators_noise_free_bursts():
    """clean bursts on their slots: the restatement's burst step with the true TSC and no carrier finds lag 0 and every block's message"""
    spec = dataclasses.replace(_spec(5, n=51 * 10000 * 2), snr_db=60.0, sampling_ppm=0.0, carrier_ppm=0.0, start_offset=0.0, phase0=0.3)
    r = oracle.raw2iq(synth.generate_stream(spec).numpy())[:, 0]
    r = r - np.mean(r)
    t = oracle.gsm_normal_training_sequence_gen(8)[:, spec.tsc]
    for mf in range(2):
        ib = []
        for k in range(4):
            p = (mf * 51 + 2 + k) * 10000 + 1.0
            lag, fl, st, bits = B.burst(r, p, 0.0, t, oracle.NORMAL_TRAINING_BITS[spec.tsc])
            assert (lag, fl, st) == (0, 0, (1, 1))
            ib.append(bits)
        ham, ok, pay = B.decode_block(ib)
        assert ok and ham == 0 and pay == spec.sysinfo[(spec.fn0 // 51 + mf) % 8]


def test_generator_without_sysinfo_is_unchanged():
    a = dataclasses.replace(synth.random_spec(7, 200000), bsic=7, tsc=7)
    b = dataclasses.replace(a, sysinfo=_si(7))
    ra, rb = synth.stream_bits(a), synth.stream_bits(b)
    frame = (np.arange(ra.shape[0]) // 8) % 51
    other = ~((np.arange(ra.shape[0]) % 8 == 0) & (frame >= 2) & (frame <= 5))
    assert np.array_equal(ra.numpy()[other], rb.numpy()[other]) and not np.array_equal(ra.numpy(), rb.numpy())
    assert np.array_equal(synth.generate_stream(a).numpy(), synth.generate_stream(dataclasses.replace(synth.random_spec(7, 200000), bsic=7,
                                                                                                        tsc=7)).numpy())


# ---- CPU: accuracy on the oracle chain at 0.47 s --------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def coef():
    return oracle.fir1(46, 200e3 / FS)


@pytest.fixture(scope="module")
def tpl():
    return oracle.gsm_SCH_training_sequence_gen(8)


@pytest.fixture(scope="module")
def nts():
    return oracle.gsm_normal_training_sequence_gen(8)


@pytest.fixture(scope="module")
def oracle_chain(coef, tpl, nts):
    specs = [_spec(s) for s in SEEDS]
    raw = synth.generate_batch(specs).numpy()
    cals = [oracle.calibrate_stream(raw[d], CARRIER, tpl, coef) for d in range(len(specs))]
    return specs, raw, cals, [B.sysinfo_reference(c, CARRIER, tpl, nts) for c in cals]


def test_restatement_decodes_every_block(oracle_chain):
    specs, _, _, refs = oracle_chain
    for s, ref in zip(specs, refs):
        si, blk = ref["si"], ref["blocks"]
        full = blk["block_flags"] & B.BLK_SHORT == 0
        assert si["n_blocks"] >= 2 and np.all(blk["block_flags"][full] == 0) and si["n_fire_ok"] == int(full.sum())
        for b in np.nonzero(full)[0]:
            assert bytes(blk["payload"][b]) == s.sysinfo[blk["tc"][b]]
            assert blk["tc"][b] == (blk["fn"][b] // 51) % 8 and blk["fn"][b] % 51 == 2
        ci, mcc, mnc, lac, nd = _cgi(s.seed)
        assert (si["mcc"], si["mnc"], si["mnc_digits"], si["lac"], si["ci"]) == (mcc, mnc, nd, lac, ci)
        assert si["flags"] == 0 and si["si_mask"] == 32 | 64
        assert np.all(np.abs(ref["bcch_rows"]["lag"][full]) <= 1) and np.all(ref["bcch_rows"]["steal"][full] == 3)


def test_lag_search_recovers_the_early_pos_info(coef, tpl, nts):
    """seed 24's pos_info points about 57 samples early, into the previous slot, and its SCH rows do not decode.  With the true BSIC and
    frame number (the truth mapped through the capture's frame timing), its BCCH bursts are found at l* in +55..+70 and decode."""
    s = _spec(EARLY_SEED)
    cal = oracle.calibrate_stream(synth.generate_stream(s).numpy(), CARRIER, tpl, coef)
    cs = CS.cell_reference(cal, CARRIER, tpl)
    assert cs["rec"]["bsic"] == -1
    pinfo = cal["pos_info"]
    p_first = pinfo[pinfo[:, 1] == 1, 0][0]
    frame = round((p_first - 1 + s.start_offset + CS_FILTER_DELAY) / 10000)
    rec = dict(cs["rec"], bsic=s.bsic, fn_first=(s.fn0 + frame) % B.FN_MOD)
    e1, e2 = cal["sampling_ppm"][0] * 1e-6, cal["sampling_ppm"][1] * 1e-6
    si, blk, rows = B.sysinfo_stream(cal["r_final"], pinfo, e1, e2, cs["carrier"], rec, nts)
    full = blk["block_flags"] & B.BLK_SHORT == 0
    assert full.sum() >= 2
    assert np.all((rows["lag"][full] >= 55) & (rows["lag"][full] <= 70))
    assert np.all(blk["block_flags"][full] == 0)
    for b in np.nonzero(full)[0]:
        assert bytes(blk["payload"][b]) == s.sysinfo[blk["tc"][b]]


# ---- GPU -----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def batch(gpu, coef, tpl):
    """_specs()'s mix (random bits, noise only, no r_correct) and streams with a cell and its System Information"""
    from test_gpu_demod_batch import _specs
    specs = _specs() + [_spec(s) for s in SEEDS + (38, 3, EARLY_SEED)]
    raw = synth.generate_batch(specs).numpy()
    return specs, raw, gpu.calibrate_batch(raw, CARRIER, tpl, coef, carrier_fit=True, sch_decode=True, sysinfo=True)


def _check(g, ref):
    si = g["sysinfo"]
    for k in ("n_blocks", "n_fire_ok", "n_si3", "n_si3_agree", "flags", "si_mask", "mcc", "mnc", "mnc_digits", "lac", "ci"):
        assert si[k] == ref["si"][k], k
    if ref["blocks"] is None:
        assert si["fn"] is None
        return
    for k in ("fn", "tc", "block_flags", "hamming"):
        np.testing.assert_array_equal(si[k if k != "block_flags" else "block_flags"], ref["blocks"][k], err_msg=k)
    np.testing.assert_array_equal(si["payload"], ref["blocks"]["payload"])
    for k in ("lag", "row_flags", "steal"):
        have = ref["blocks"]["fn"] >= 0                         # rows of streams without a cell are not correlated
        np.testing.assert_array_equal(si[k][have], ref["bcch_rows"][k][have], err_msg=k)


@pytest.mark.gpu
def test_sysinfo_matches_the_restatement_on_the_gpus_r_correct(gpu, batch, coef, tpl, nts):
    specs, raw, got = batch
    D, n_iq = raw.shape[0], raw.shape[1] // 2
    r = np.zeros((D, n_iq), dtype=np.complex128)
    gpu.calibrate_batch(raw, CARRIER, tpl, coef, r_correct=r)
    ran = 0
    for d, g in enumerate(got):
        if g["sysinfo"]["n_blocks"] < 0:
            assert g["sysinfo"]["flags"] in (B.NO_POS_INFO, B.NO_R_CORRECT)
            continue
        e1, e2 = g["sampling_ppm"][0] * 1e-6, g["sampling_ppm"][1] * 1e-6
        rec = dict(bsic=g["cell"]["bsic"], fn_first=g["cell"]["fn_first"])
        si, blk, rows = B.sysinfo_stream(r[d, :g["r_len"][2]], g["pos_info"], e1, e2, dict(g["carrier"]), rec, nts)
        _check(g, dict(si=si, blocks=blk, bcch_rows=rows))
        ran += 1
    assert ran >= 8


@pytest.mark.gpu
def test_sysinfo_matches_the_oracle_chain_and_the_truth(batch, coef, tpl, nts):
    specs, raw, got = batch
    cells = [d for d, s in enumerate(specs) if s.sysinfo is not None and s.seed != EARLY_SEED]
    for d in cells[:2]:
        _check(got[d], B.sysinfo_reference(oracle.calibrate_stream(raw[d], CARRIER, tpl, coef), CARRIER, tpl, nts))
    right = 0
    for d in cells:                     # a 0.47 s capture holds two or three blocks: some decode only an SI4 (seed 38: its last row leaves r_correct)
        ci, mcc, mnc, lac, nd = _cgi(specs[d].seed)
        si = got[d]["sysinfo"]
        assert si["cgi"] == (mcc, mnc, nd, lac, ci) and si["flags"] == 0 or si["flags"] == B.NO_SI3 and si["n_si3"] == 0 and si["si_mask"] == 64
        right += si["cgi"] is not None
    assert right >= 4
    early = got[[s.seed for s in specs].index(EARLY_SEED)]["sysinfo"]
    assert early["flags"] & B.NO_CELL


def _outputs(raw, mode):
    """every output of gsmcal_calibrate_cell_batch ('cell') or _sysinfo_batch ('sysinfo') as bytes, with the launch count"""
    from gsmcal import api
    from gsmcal._lib import CarrierFitResult, SchDecodeResult, StreamResult, SysinfoResult, lib
    coef = oracle.fir1(46, 200e3 / FS)
    tpl = oracle.gsm_SCH_training_sequence_gen(8)
    D, n_iq = raw.shape[0], raw.shape[1] // 2
    cap = api.max_bursts(n_iq)
    res, cf, sd, si = (StreamResult * D)(), (CarrierFitResult * D)(), (SchDecodeResult * D)(), (SysinfoResult * D)()
    arrs = [np.full((D, cap), 7.0), np.full((D, cap), 7.0), np.full((D, cap), 7.0), np.full((D, 6 * cap, 2), 7.0)]
    args = [_vp(raw), 0, n_iq, D, CARRIER, _vp(tpl), _vp(coef), len(coef), 8, 8, C.cast(res, C.c_void_p)] + [_vp(a) for a in arrs] + [None]
    cfr = [np.full((D, cap), 7.0), np.full((D, cap), 7.0), np.full((D, cap), 7, np.uint8)]
    cell = [np.zeros((D, cap), np.uint8), np.zeros((D, cap, 148), np.uint8), np.zeros((D, cap, 85)), np.full((D, cap), 7.0),
            np.full((D, cap), 7, np.int32), np.full((D, cap), 7, np.int32), np.full((D, cap), 7, np.uint8), np.full((D, cap), 7, np.uint8)]
    cell_args = [C.cast(cf, C.c_void_p), *[_vp(a) for a in cfr], C.cast(sd, C.c_void_p), *[_vp(a) for a in cell]]
    n0 = api.launch_count()
    if mode == "cell":
        assert lib().gsmcal_calibrate_cell_batch(*args, *cell_args) == 0
    else:
        nts = np.ascontiguousarray(oracle.gsm_normal_training_sequence_gen(8).T)
        assert lib().gsmcal_calibrate_sysinfo_batch(*args, *cell_args, _vp(nts), C.cast(si, C.c_void_p), *[None] * 8) == 0
    n = api.launch_count() - n0
    return (bytes(res), [a.tobytes() for a in arrs], bytes(cf), [a.tobytes() for a in cfr], bytes(sd), [a.tobytes() for a in cell]), n


@pytest.mark.gpu
def test_cell_call_unchanged_by_the_sysinfo_stage(gpu, batch):
    raw = batch[1]
    cell, n_cell = _outputs(raw, "cell")
    si, n_si = _outputs(raw, "sysinfo")
    again, n_again = _outputs(raw, "cell")
    assert cell == si == again
    assert n_cell == n_again and n_si == n_cell + 3               # one stream group: block list, BCCH bursts, block decoding


def _si_bytes(item):
    s = item["sysinfo"]
    return (tuple(s[k] for k in ("n_blocks", "n_fire_ok", "n_si3", "n_si3_agree", "flags", "si_mask", "mcc", "mnc", "mnc_digits", "lac", "ci")),
            None if s["fn"] is None else tuple(s[k].tobytes() for k in ("fn", "tc", "block_flags", "hamming", "payload", "lag", "row_flags",
                                                                           "steal")))


@pytest.mark.gpu
def test_sysinfo_stream_independence_and_device_input(gpu, batch, coef, tpl):
    torch = pytest.importorskip("torch")
    _, raw, got = batch
    D = raw.shape[0]
    kw = dict(carrier_fit=True, sch_decode=True, sysinfo=True)
    alone = gpu.calibrate_batch(raw[-3:-2], CARRIER, tpl, coef, **kw)[0]
    assert _si_bytes(alone) == _si_bytes(got[D - 3])
    perm = np.random.default_rng(9).permutation(D)
    big = np.concatenate([raw[perm], raw[perm[::-1]]])                                 # 2D streams: several stream groups
    shuffled = gpu.calibrate_batch(big, CARRIER, tpl, coef, **kw)
    for i, d in enumerate(perm):
        assert _si_bytes(shuffled[i]) == _si_bytes(got[d]) == _si_bytes(shuffled[2 * D - 1 - i])
    dev = torch.from_numpy(raw.copy()).cuda()
    torch.cuda.synchronize()
    on_dev = gpu.calibrate_batch(None, CARRIER, tpl, coef, device_ptr=dev.data_ptr(), n_iq=raw.shape[1] // 2, n_streams=D, **kw)
    for a, b in zip(on_dev, got):
        assert _si_bytes(a) == _si_bytes(b)


@pytest.mark.gpu
def test_drifting_full_length_streams_report_their_cgi(gpu, coef, tpl):
    torch = pytest.importorskip("torch")
    specs = [dataclasses.replace(_spec(101, N_10S), carrier_drift_ppm_per_s=0.02),
             dataclasses.replace(_spec(132, N_10S), carrier_drift_ppm_per_s=-0.02)]
    raw = synth.generate_batch(specs, device="cuda")
    torch.cuda.synchronize()
    got = gpu.calibrate_batch(None, CARRIER, tpl, coef, device_ptr=raw.data_ptr(), n_iq=N_10S, n_streams=2, carrier_fit=True, sch_decode=True,
                              sysinfo=True)
    for s, g in zip(specs, got):
        si = g["sysinfo"]
        ci, mcc, mnc, lac, nd = _cgi(s.seed)
        assert si["n_blocks"] >= 40 and si["cgi"] == (mcc, mnc, nd, lac, ci) and si["flags"] == 0
        full = si["block_flags"] & B.BLK_SHORT == 0
        assert si["n_fire_ok"] >= full.sum() - 1 and si["si_mask"] == 32 | 64
        ok = si["block_flags"] == 0
        assert all(bytes(si["payload"][b]) == s.sysinfo[si["tc"][b]] for b in np.nonzero(ok)[0])


@pytest.mark.gpu
def test_two_dongles_on_one_cell_report_the_same_cgi(gpu, coef, tpl):
    """seeds 11 and 72 on seed 11's cell, and seed 28's cell given seed 11's BSIC: the BSIC cannot tell the third from the first two,
    the CGI does"""
    a = _spec(11)
    b = dataclasses.replace(_spec(72, cell_seed=11), fn0=a.fn0 + 153, start_offset=a.start_offset + 12345)
    c = dataclasses.replace(_spec(28), bsic=a.bsic, tsc=a.bsic & 7)
    raw = synth.generate_batch([a, b, c]).numpy()
    got = gpu.calibrate_batch(raw, CARRIER, tpl, coef, carrier_fit=True, sch_decode=True, sysinfo=True)
    assert [g["cell"]["bsic"] for g in got] == [a.bsic] * 3
    cgi = [g["sysinfo"]["cgi"] for g in got]
    assert cgi[0] == cgi[1] != cgi[2] and None not in cgi


@pytest.mark.gpu
def test_sysinfo_stage_is_reported(gpu, batch, coef, tpl):
    from gsmcal._lib import lib
    raw = batch[1]
    lib().gsmcal_debug_set(3, 1)
    try:
        gpu.calibrate_batch(raw[:4], CARRIER, tpl, coef, carrier_fit=True, sch_decode=True, sysinfo=True)
        ms = gpu.api.last_batch_stage_ms()
        assert len(ms) == 7 and list(ms.values())[6] > 0
    finally:
        lib().gsmcal_debug_set(3, 4)


@pytest.mark.gpu
def test_ingest_forwards_sysinfo(gpu):
    from gsmcal import ingest
    from gsmcal.rtl_tcp_replay import ReplayDongle
    N = N_SYNC
    specs = [_spec(seed, 2 * N + 8) for seed in SEEDS]
    raw = synth.generate_batch(specs).numpy()
    srvs = [ReplayDongle(raw[d]) for d in range(len(specs))]
    try:
        res = ingest.calibrate_from_dongles([(s.host, s.port) for s in srvs], N, CARRIER, n_captures=1, carrier_fit=True, sch_decode=True,
                                            sysinfo=True)[0]
    finally:
        for s in srvs:
            s.close()
    direct_in = np.stack([s.expected(2 * N - 12, 2 * N) for s in srvs])
    direct = gpu.calibrate_batch(direct_in, CARRIER, gpu.gsm_SCH_training_sequence_gen(8), gpu.fir1(46, 200e3 / FS), carrier_fit=True,
                                 sch_decode=True, sysinfo=True)
    for a, b in zip(res, direct):
        assert _si_bytes(a) == _si_bytes(b)
