"""Pins the oracle to a run of the reference itself - WHEN such a run exists.

oracle/export_fixtures.py writes the inputs, oracle/run_reference.m runs the unmodified reference function files on them under GNU
Octave / MATLAB and saves out_<case>.mat next to them.  Neither runtime exists in the build image, so normally this test only
checks that the recipe is complete and consistent (inputs export and reload, the .m file calls functions the reference defines,
in gsm_sync_demod.m's order) and SKIPS the comparison; with tests/golden/reference_run/out_*.mat present it asserts
oracle == reference at the north-star tolerances and the "parity unpinned" cap can be lifted.
"""
import json
import math
import os
import re

import numpy as np
import pytest
import scipy.io

import gsmcal_oracle as oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RUN = os.path.join(ROOT, "tests", "golden", "reference_run")
FS = oracle.SYMBOL_RATE * 8


def _load(path):
    return scipy.io.loadmat(path, squeeze_me=True)


def _vec(x):
    return np.atleast_1d(np.asarray(x, dtype=np.complex128 if np.iscomplexobj(x) else np.float64)).reshape(-1)


def test_recipe_exports_and_reloads(tmp_path):
    import sys
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import export_fixtures
    m = export_fixtures.main(str(tmp_path), n=200000)          # short captures: CPU-suite budget
    names = [c["name"] for c in m["cases"]]
    assert {"seed1", "noise_only", "dropped_fcch", "fine_overrun", "fine_snr_gate", "sch_e_zero", "sch_bcch_runout"} <= set(names)
    a = _load(os.path.join(tmp_path, "case_seed1.mat"))
    assert a["raw"].dtype == np.uint8 and a["raw"].size == 400000 and a["coef"].size == 47 and a["tpl"].size == 512
    assert np.array_equal(_vec(a["coef"]), oracle.fir1(46, 200e3 / FS))
    num = _load(os.path.join(tmp_path, "gsm_chn_filter_8x.mat"))["Num"]
    assert num.size == 60 and abs(float(np.sum(num)) - 0.99423319989488024) < 1e-15          # SURVEY 8c checksum
    assert os.path.exists(os.path.join(tmp_path, "run_reference.m"))


def test_run_reference_m_calls_the_reference_functions_in_script_order():
    src = open(os.path.join(ROOT, "oracle", "run_reference.m")).read()
    order = ["raw2iq(", "filter(in.coef", "FCCH_coarse_position(", "FCCH_fine_correction(", "SCH_corr_rate_correction(",
             "carrier_correct_post_SCH(", "total_ppm_calculation("]
    pos = [src.index(k) for k in order]
    assert pos == sorted(pos)                                   # gsm_sync_demod.m:107-124
    with open(os.path.join(ROOT, "tests", "golden", "reference_functions.json")) as f:
        defined = json.load(f)["functions"]                     # the reference's function files, with their defining lines
    for fn in ("raw2iq", "FCCH_coarse_position", "move_fft_snr_runtime_avg", "FCCH_fine_correction", "SCH_corr_rate_correction",
               "carrier_correct_post_SCH", "total_ppm_calculation", "chn_filter_8x_4x", "chn_filter_4x"):
        assert re.search(r"\b%s\(" % fn, src), fn              # the script calls it ...
        assert defined[fn].startswith(fn + ".m:"), fn           # ... and the reference defines it ...
        assert not re.search(r"^\s*function\b.*\b%s\s*\(" % fn, src, re.M), fn                       # ... not the script itself
        assert not any(os.path.exists(os.path.join(d, fn + ".m")) for d in (os.path.join(ROOT, "oracle"), RUN)), fn   # nor a .m of ours


def _have_run():
    return os.path.exists(os.path.join(RUN, "manifest.json")) and any(f.startswith("out_") for f in os.listdir(RUN))


@pytest.mark.skipif(not _have_run(), reason="no reference run present: python oracle/export_fixtures.py, then run_reference.m under Octave/MATLAB")
def test_oracle_equals_reference_run():
    with open(os.path.join(RUN, "manifest.json")) as f:
        man = json.load(f)
    checked = 0
    for c in man["cases"]:
        out_path = os.path.join(RUN, f"out_{c['name']}.mat")
        if not os.path.exists(out_path):
            continue
        ref = _load(out_path)
        stride = int(ref["stride"])
        if c["kind"] == "capture":
            a = _load(os.path.join(RUN, f"case_{c['name']}.mat"))
            raw, coef, tpl = _vec(a["raw"]).astype(np.uint8), _vec(a["coef"]), _vec(a["tpl"])
            r0 = oracle.raw2iq(raw)[:, 0]
            assert np.array_equal(r0[:4096], _vec(ref["r0_head"]))                      # raw2iq bit-exact
            r = oracle.fir_filter(coef, r0)
            assert np.max(np.abs(r[::stride] - _vec(ref["r_s"]))) <= 1e-12 * np.max(np.abs(r))
            info = {}
            got = oracle.calibrate_stream(raw, float(a["carrier_freq"]), tpl, coef, info=info)
            assert np.array_equal(got["coarse_pos"], _vec(ref["position"]))
            assert np.allclose(got["coarse_snr"], _vec(ref["snr"]), rtol=0, atol=1e-9)
            assert np.array_equal(got["fcch_pos"], _vec(ref["FCCH_pos"]))
            assert np.array_equal(got["pos_info"].reshape(-1, 2), np.asarray(ref["pos_info"], dtype=np.float64).reshape(-1, 2))
            for g, k in ((got["sampling_ppm"][0], "sppm1"), (got["sampling_ppm"][1], "sppm2"), (got["carrier_ppm"][0], "cppm1"),
                         (got["carrier_ppm"][1], "cppm2"), (got["total_sampling_ppm"], "total_sampling_ppm"), (got["total_carrier_ppm"], "total_carrier_ppm")):
                rv = float(ref[k])
                assert (g == rv) if math.isinf(rv) else abs(g - rv) < 1e-3, k
            r3 = got["r_final"]
            if int(ref["r3_len"]) > 1:
                assert r3 is not None and len(r3) == int(ref["r3_len"])
                assert np.max(np.abs(r3[::stride] - _vec(ref["r3_s"]))) <= 1e-9 * np.max(np.abs(r3))
            else:
                assert r3 is None
            with open(os.path.join(ROOT, "tests", "golden", "chn_filter_taps.json")) as f:
                g = json.load(f)
            num8 = np.array([float.fromhex(h) for h in g["Num_8x"]["hex"]])
            num4 = np.array([float.fromhex(h) for h in g["Num_4x"]["hex"]])
            assert np.max(np.abs(oracle.chn_filter_8x_4x(r0[:20000], num8) - _vec(ref["chn8"]))) < 1e-12 * np.max(np.abs(r0))
            assert np.max(np.abs(oracle.chn_filter_4x(r0[:20000], num4) - _vec(ref["chn4"]))) < 1e-12 * np.max(np.abs(r0))
        elif c["kind"] == "planted_fine":
            a = _load(os.path.join(RUN, f"planted_{c['name']}.mat"))
            fpos, r1, sppm, cppm = oracle.FCCH_fine_correction(_vec(a["s"]), _vec(a["base_position"]), int(a["osr"]), float(a["carrier_freq"]))
            assert np.array_equal(fpos, _vec(ref["FCCH_pos"]))
            for g, k in ((sppm, "sppm1"), (cppm, "cppm1")):
                rv = float(ref[k])
                assert (g == rv) if math.isinf(rv) else abs(g - rv) < 1e-3
            assert (r1 is None and int(ref["r1_len"]) == 1) or len(r1) == int(ref["r1_len"])
        else:
            a = _load(os.path.join(RUN, f"planted_{c['name']}.mat"))
            pinfo, r2, sppm = oracle.SCH_corr_rate_correction(_vec(a["s"]), _vec(a["FCCH_pos"]), _vec(a["tpl"]), int(a["osr"]))
            assert np.array_equal(pinfo.reshape(-1, 2), np.asarray(ref["pos_info"], dtype=np.float64).reshape(-1, 2))
            rv = float(ref["sppm2"])
            assert (sppm == rv) if math.isinf(rv) else abs(sppm - rv) < 1e-3
        checked += 1
    assert checked > 0
