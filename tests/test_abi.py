"""CPU checks of the drop-in boundary: the C-ABI library builds for sm_100a, loads, exports every symbol that
include/gsmcal.h declares, its host-only entry points agree with the oracle, and compute calls fail loudly
(no CPU fallback) when there is no CUDA device."""
import ctypes as C
import json
import math
import os
import re
import subprocess

import numpy as np
import pytest

import gsmcal_oracle as oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FS = oracle.SYMBOL_RATE * 8


def declared_symbols():
    with open(os.path.join(ROOT, "include", "gsmcal.h")) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    return sorted(set(re.findall(r"\b(gsmcal_[A-Za-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(built_lib):
    from gsmcal import _lib
    lib = _lib.lib()
    names = declared_symbols()
    assert len(names) >= 28
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/gsmcal.h but not exported"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature"
    out = subprocess.run(["nm", "-D", "--defined-only", built_lib], capture_output=True, text=True).stdout
    exported = set(re.findall(r"\bT (gsmcal_\w+)", out))
    assert set(names) <= exported
    assert lib.gsmcal_abi_version() == 1


def test_library_is_sm100a_native_code(built_lib):
    out = subprocess.run(["cuobjdump", "-lelf", built_lib], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_result_record_layout():
    from gsmcal._lib import StreamResult
    assert C.sizeof(StreamResult) == 88


def test_host_only_entry_points_match_oracle(built_lib):
    import gsmcal
    for order, wn in ((46, 200e3 / FS), (30, 200e3 / FS), (63, 0.05 / 2.048), (127, 0.02)):
        assert np.max(np.abs(gsmcal.fir1(order, wn) - oracle.fir1(order, wn))) < 2e-16
    with open(os.path.join(ROOT, "tests", "golden", "chn_filter_taps.json")) as f:
        g = json.load(f)
    assert gsmcal.chn_filter_taps(8).tolist() == [float.fromhex(h) for h in g["Num_8x"]["hex"]]
    assert gsmcal.chn_filter_taps(4).tolist() == [float.fromhex(h) for h in g["Num_4x"]["hex"]]
    for v in ([-35.0, 1.2], [math.inf, math.inf], [3.0, math.inf], [0.0], []):
        assert gsmcal.total_ppm_calculation(v) == oracle.total_ppm_calculation(v)
    for osr in (4, 8):
        assert np.max(np.abs(gsmcal.gsm_SCH_training_sequence_gen(osr) - oracle.gsm_SCH_training_sequence_gen(osr))) < 1e-12
    assert gsmcal.max_bursts(21666667) == math.ceil(math.ceil(21666667 / 64) / 1562.5) + 2


def test_sentinels_need_no_device(built_lib):
    """The '<5 hits' early returns of the reference are decided before any GPU work (FCCH_fine_correction.m:12-15 ...)."""
    import gsmcal
    s = np.zeros(100, dtype=np.complex128)
    f = gsmcal.FCCH_fine_correction(s, [-1.0], 8, 957.4e6)
    assert f[0].tolist() == [-1.0] and f[1] is None and f[2] == math.inf and f[3] == math.inf
    p = gsmcal.SCH_corr_rate_correction(s, [-1.0], np.ones(512, complex), 8)
    assert p[0].tolist() == [[-1.0, -1.0]] and p[1] is None and p[2] == math.inf
    c = gsmcal.carrier_correct_post_SCH(s, [[-1.0, -1.0]], 8, 957.4e6)
    assert c == (None, math.inf)
    assert gsmcal.carrier_correct_post_SCH(s, [[10.0, 0.0]] + [[20.0 + k, 2.0] for k in range(3)], 8, 957.4e6) == (None, math.inf)   # < 4 BCCH rows
    assert gsmcal.specific_fft_snr_fix_avg(s, (5, 4), 16, 10.0, 1.0) == (False, -1.0, math.inf)                                 # empty target set


def test_host_decided_range_errors_need_no_device(built_lib):
    """Every window the drop-ins can check on the host is checked before any device work: the reference's index errors come out as
    GSMCAL_ERR_RANGE with the same text on a machine without a GPU (not as GSMCAL_ERR_CUDA), and launch nothing on one with a GPU."""
    import gsmcal
    s = np.zeros(20000, dtype=np.complex128)
    tpl, nts = np.ones(512, complex), np.ones((208, 8), complex)
    bcch = [[3000.0 + k * 1250, 2.0] for k in range(4)]
    cases = [
        ("base_position(1)=10 puts the search window before the first sample",
         lambda: gsmcal.FCCH_fine_correction(np.zeros(80000, complex), [10.0, 2000.0, 3000.0, 4000.0, 5000.0], 8, 957.4e6)),
        ("FCCH_pos(1) puts the search window before the first sample",
         lambda: gsmcal.SCH_corr_rate_correction(s, [-20000.0, 1.0, 2.0, 3.0, 4.0], tpl, 8)),
        ("carrier_correct_post_SCH: FCCH window outside the stream",
         lambda: gsmcal.carrier_correct_post_SCH(s, [[19000.0, 0.0]] + bcch, 8, 957.4e6)),
        ("FCCH_demod: no FCCH rows", lambda: gsmcal.FCCH_demod(s, bcch, 8, 957.4e6)),
        ("SCH_demod: equaliser window of the SCH burst at 19900 outside the stream", lambda: gsmcal.SCH_demod(s, [[19900.0, 1.0]], tpl, 8)),
        ("BCCH_demod: training window of BCCH burst 4 outside the stream",
         lambda: gsmcal.BCCH_demod(s, [[1001.0, 0.0]] + bcch[:3] + [[19900.0, 2.0]], nts, 8, 957.4e6)),
        ("specific_fft_snr_fix_avg: window outside the stream", lambda: gsmcal.specific_fft_snr_fix_avg(s, (0, 100), 64, 10.0, 1.0)),
        ("FCCH_coarse_position: stream shorter than 23 frames", lambda: gsmcal.FCCH_coarse_position(s[:1000], 8)),
    ]
    launches = gsmcal.launch_count()
    for text, call in cases:
        with pytest.raises(gsmcal.GsmcalError) as e:
            call()
        assert e.value.code == -4 and text in str(e.value), str(e.value)
    assert gsmcal.launch_count() == launches


def test_compute_fails_loudly_without_a_gpu(built_lib):
    import gsmcal
    if gsmcal.device_count() > 0:
        pytest.skip("a CUDA device is present")
    a = np.zeros((64, 1), dtype=np.uint8)
    with pytest.raises(gsmcal.GsmcalError) as e:
        gsmcal.raw2iq(a)
    assert e.value.code == -2 and "no CPU fallback" in str(e.value)
    with pytest.raises(gsmcal.GsmcalError):
        gsmcal.calibrate_batch(np.zeros((1, 2 * 300000), dtype=np.uint8), 957.4e6, np.ones(512, complex), gsmcal.fir1(46, 0.09))


def test_bad_arguments_are_rejected(built_lib):
    import gsmcal
    with pytest.raises(gsmcal.GsmcalError):
        gsmcal.fir1(200, 0.1)
    with pytest.raises(gsmcal.GsmcalError):
        gsmcal.chn_filter_taps(5)
    with pytest.raises(ValueError):
        gsmcal.SCH_corr_rate_correction(np.zeros(10, complex), np.arange(5.0), np.ones(100, complex), 8)


def test_demod_family_sentinels_and_loud_failure(built_lib):
    """SURVEY 8(f) rows 2/4: the `pos_info==-1` returns are decided on the host; real work without a GPU is an error, not a fallback."""
    import gsmcal
    s = np.zeros(20000, dtype=np.complex128)
    m1 = np.array([[-1.0, -1.0]])
    assert gsmcal.FCCH_demod(s, m1, 8, 957.4e6) is None
    assert gsmcal.SCH_demod(s, m1, np.ones(512, complex), 8) is None
    assert gsmcal.BCCH_demod(s, m1, np.ones((208, 8), complex), 8, 957.4e6) == (-1.0, -1, None)
    assert gsmcal.gsm_normal_training_sequence_gen(8).shape == (208, 8)
    if gsmcal.device_count() > 0:
        pytest.skip("a CUDA device is present")
    rows = np.array([[1001.0, 0.0], [1001.0 + 10336 - 336, 1.0]] + [[3000.0 + k * 1250, 2.0] for k in range(4)])
    for call in (lambda: gsmcal.FCCH_demod(s, rows, 8, 957.4e6),
                 lambda: gsmcal.SCH_demod(s, rows, np.ones(512, complex), 8),
                 lambda: gsmcal.BCCH_demod(s, rows, np.ones((208, 8), complex), 8, 957.4e6),
                 lambda: gsmcal.calibrate_batch_submit(0, 0x1000, 300000, 1, 957.4e6, np.ones(512, complex), gsmcal.fir1(46, 0.09))):
        with pytest.raises(gsmcal.GsmcalError) as e:
            call()
        assert e.value.code == -2


def test_debug_set_accepts_exactly_the_documented_keys():
    """gsmcal_debug_set's keys are the tuning surface the profiles/ scripts use: the library accepts exactly the keys listed here, and each
    must be described in the comment above its declaration (include/gsmcal.h)."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(root, "multi-rtl-sdr-calibration_b200", "csrc", "gsmcal_api.cu")).read()
    body = src[src.index("int gsmcal_debug_set(int key, int value)"):]
    body = body[:body.index("\n}\n")]
    keys = sorted({int(k) for k in re.findall(r"key == (\d+)", body)})
    assert keys == [0, 3, 4, 5, 6, 8, 9, 10, 11, 12, 13, 14, 17, 18, 24]
    hdr = open(os.path.join(root, "include", "gsmcal.h")).read()
    doc = hdr[hdr.index("test / tuning hooks"):hdr.index("int gsmcal_debug_set")]
    documented = {int(k) for k in re.findall(r"(?:key |; |, |\* )(\d+)(?:,| =)", doc)}
    missing = [k for k in keys if k not in documented]
    assert not missing, f"debug keys without a line in include/gsmcal.h: {missing}"


def test_debug_set_rejects_removed_and_unknown_keys(built_lib):
    """Keys of the removed overlap experiments (7, 15, 16, 19, 21, 22, 23) and keys that never existed are argument errors; no device
    is needed to reject them."""
    from gsmcal import _lib
    lib = _lib.lib()
    for key in (7, 15, 16, 19, 21, 22, 23, 99):
        assert lib.gsmcal_debug_set(key, 1) == -1, key
        assert "unknown key" in lib.gsmcal_last_error().decode()
