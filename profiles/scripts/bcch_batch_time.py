"""Time gsmcal_calibrate_demod_bcch_batch against gsmcal_calibrate_demod_batch on the workload of demod_batch_time.py (1024 synthetic 10 s
streams, seeds 0.., generated on the GPU and resident in HBM: 44 GB, far above L2), with the normal training sequence code of stream d
set to d % 8, and write profiles/bcch_batch_1gpu.json.

Alternates the two calls (host clock ending in the call's own stream synchronise), then one run with a single stream group (debug key
3 = 1) for the stage breakdown, then one torch.profiler run for the per-kernel CUDA times of the demod stage.  Also reports how many
streams identify their own training sequence code (nts_idx == tsc + 1), and the card's name and power limit read in the same call."""
import argparse
import ctypes as C
import dataclasses
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (os.path.join(ROOT, "multi-rtl-sdr-calibration_b200"), os.path.join(ROOT, "oracle")):
    sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import gsmcal  # noqa: E402
from gsmcal import synth  # noqa: E402
from gsmcal._lib import BcchResult, DemodResult, StreamResult, lib  # noqa: E402

N_IQ_10S = 21666667
FS = gsmcal.api.SYMBOL_RATE * 8


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=1024)
    ap.add_argument("--n-iq", type=int, default=N_IQ_10S)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bcch_batch_1gpu.json"))
    a = ap.parse_args()
    if gsmcal.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    D, n_iq = a.streams, a.n_iq
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    raw = torch.empty((D, 2 * n_iq), dtype=torch.uint8, device="cuda")
    tsc = [d % 8 for d in range(D)]
    for d in range(D):
        synth.generate_stream(dataclasses.replace(synth.random_spec(d, n_iq), tsc=tsc[d]), "cuda", raw[d])
    torch.cuda.synchronize()
    coef = gsmcal.fir1(46, 200e3 / FS)
    tpl = gsmcal.gsm_SCH_training_sequence_gen(8)
    nts = np.ascontiguousarray(gsmcal.gsm_normal_training_sequence_gen(8).T)    # column-major (26*8) x 8
    L = lib()
    res, dem, bc = (StreamResult * D)(), (DemodResult * D)(), (BcchResult * D)()
    vp = lambda x: x.ctypes.data_as(C.c_void_p)                       # noqa: E731
    args = [C.c_void_p(raw.data_ptr()), 1, n_iq, D, 957.4e6, vp(tpl), vp(coef), len(coef), 8, 8, C.cast(res, C.c_void_p), None, None, None, None, None,
            C.cast(dem, C.c_void_p), None, None, None, None, None, None, None]

    def demod():
        rc = L.gsmcal_calibrate_demod_batch(*args)
        assert rc == 0, L.gsmcal_last_error()

    def bcch():
        rc = L.gsmcal_calibrate_demod_bcch_batch(*args, vp(nts), C.cast(bc, C.c_void_p))
        assert rc == 0, L.gsmcal_last_error()

    for f in (demod, bcch, demod, bcch):
        f()
    t_dem, t_bc = [], []
    for _ in range(a.reps):
        for f, acc in ((demod, t_dem), (bcch, t_bc)):
            t0 = time.perf_counter(); f(); torch.cuda.synchronize(); acc.append((time.perf_counter() - t0) * 1e3)
    flags, hit, missed = {}, 0, []
    for d in range(D):
        flags[bc[d].flags] = flags.get(bc[d].flags, 0) + 1
        hit += int(bc[d].nts_idx == tsc[d] + 1)
        if bc[d].flags == 0 and bc[d].nts_idx != tsc[d] + 1:
            missed.append(dict(seed=d, tsc=tsc[d], nts_idx=bc[d].nts_idx, first_max=[int(np.argmax(bc[d].corr_abs[8 * b:8 * b + 8])) + 1 for b in range(4)]))
    ppm_equal = all(bc[d].carrier_ppm == dem[d].fcch_carrier_ppm for d in range(D) if bc[d].flags in (0, 8))
    L.gsmcal_debug_set(3, 1)
    bcch()
    stages = gsmcal.api.last_batch_stage_ms()
    demod()
    stages_without = gsmcal.api.last_batch_stage_ms()
    L.gsmcal_debug_set(3, 4)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        bcch()
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and any(k in ev.name for k in ("demod", "fde_template")):
            key = ev.name.split("(")[0].split("<")[0].replace("void ", "")
            dt = (ev.device_time if hasattr(ev, "device_time") else ev.cuda_time) / 1e3
            kern[key] = kern.get(key, 0.0) + dt
    out = dict(
        card=smi, streams=D, n_iq=n_iq, reps=a.reps,
        workload="demod_batch_time.py's: synthetic 10 s streams, seeds 0.., normal training sequence code seed % 8, device-resident (44 GB at 1024 streams)",
        calibrate_demod_batch_ms=dict(median=statistics.median(t_dem), min=min(t_dem), max=max(t_dem), all=t_dem),
        calibrate_demod_bcch_batch_ms=dict(median=statistics.median(t_bc), min=min(t_bc), max=max(t_bc), all=t_bc),
        bcch_increment_ms_median=statistics.median(t_bc) - statistics.median(t_dem),
        stage_ms_one_group=stages, stage_ms_one_group_without_bcch=stages_without, demod_kernel_ms_one_group=kern,
        bcch_kernel_ms=kern.get("bcch_demod_batch_kernel"),
        bcch_flags_histogram={str(k): v for k, v in sorted(flags.items())},
        nts_idx_equals_tsc_plus_1=hit, nts_idx_equals_tsc_plus_1_share=hit / D,
        flag0_streams_missing_their_tsc=missed,
        bcch_carrier_ppm_equals_fcch_carrier_ppm=ppm_equal,
        timing="host clock around each call (the call returns after its stream has drained); per-kernel times: torch.profiler CUDA activity, separate run")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("card", "calibrate_demod_batch_ms", "calibrate_demod_bcch_batch_ms", "bcch_increment_ms_median", "stage_ms_one_group",
                                          "bcch_kernel_ms", "bcch_flags_histogram", "nts_idx_equals_tsc_plus_1_share", "flag0_streams_missing_their_tsc")}, indent=1))


if __name__ == "__main__":
    main()
