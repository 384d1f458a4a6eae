"""Time gsmcal_calibrate_carrier_fit_batch against gsmcal_calibrate_batch on 1024 synthetic 10 s streams (random_spec seeds 0..,
generated on the GPU and resident in HBM: 44 GB, far above L2), and write profiles/carrier_fit_1gpu.json.

Alternates the two calls (host clock ending in the call's own stream synchronise; medians of --reps), then one run with a single
stream group (debug key 3 = 1) for the stage breakdown, then one torch.profiler run for the per-kernel CUDA times of the carrier stage.
carrier_fit_row_kernel's FP64 rate: its counted work over its profiled time, against gsmcal_fp64_peak (a register-only DFMA kernel)
measured in the same call.  Counted work per row whose grid ran: 29 grid points x 928 samples x 14 FP64 operations (complex
multiply-add 8, rotation step 6); per row that also ran Newton: 5 steps x 928 samples x 23 (y times the rotation 6, S0 2, S1 4, m^2 1,
S2 4, rotation step 6).  Also: how carrier_fit_ppm and total_carrier_ppm compare with the injected ppm, and the card's name and power
limit read in the same call."""
import argparse
import ctypes as C
import json
import math
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
from gsmcal._lib import CarrierFitResult, StreamResult, lib  # noqa: E402

N_IQ_10S = 21666667
FS = gsmcal.api.SYMBOL_RATE * 8
FLOP_GRID = 29 * 928 * 14
FLOP_NEWTON = 5 * 928 * 23


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=1024)
    ap.add_argument("--n-iq", type=int, default=N_IQ_10S)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "carrier_fit_1gpu.json"))
    a = ap.parse_args()
    if gsmcal.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    D, n_iq = a.streams, a.n_iq
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    raw = torch.empty((D, 2 * n_iq), dtype=torch.uint8, device="cuda")
    specs = [synth.random_spec(d, n_iq) for d in range(D)]
    for d in range(D):
        synth.generate_stream(specs[d], "cuda", raw[d])
    torch.cuda.synchronize()
    coef = gsmcal.fir1(46, 200e3 / FS)
    tpl = gsmcal.gsm_SCH_training_sequence_gen(8)
    L = lib()
    cap = gsmcal.max_bursts(n_iq)
    res, cf = (StreamResult * D)(), (CarrierFitResult * D)()
    rf = np.empty((D, cap), dtype=np.uint8)
    vp = lambda x: x.ctypes.data_as(C.c_void_p)                       # noqa: E731
    args = [C.c_void_p(raw.data_ptr()), 1, n_iq, D, 957.4e6, vp(tpl), vp(coef), len(coef), 8, 8, C.cast(res, C.c_void_p), None, None, None, None, None]

    def plain():
        rc = L.gsmcal_calibrate_batch(*args)
        assert rc == 0, L.gsmcal_last_error()

    def timed():
        rc = L.gsmcal_calibrate_carrier_fit_batch(*args, C.cast(cf, C.c_void_p), None, None, vp(rf))
        assert rc == 0, L.gsmcal_last_error()

    for f in (plain, timed, plain, timed):
        f()
    t_plain, t_timed = [], []
    for _ in range(a.reps):
        for f, acc in ((plain, t_plain), (timed, t_timed)):
            t0 = time.perf_counter(); f(); torch.cuda.synchronize(); acc.append((time.perf_counter() - t0) * 1e3)
    rows = [rf[d, :max(cf[d].n_fcch, 0)] for d in range(D)]
    n_rows = sum(len(r) for r in rows)
    n_grid = sum(int((r != 4).sum()) for r in rows)
    n_newton = sum(int(((r == 0) | (r == 16)).sum()) for r in rows)
    n_fit = sum(int((r == 0).sum()) for r in rows)
    flags = {}
    for d in range(D):
        flags[cf[d].flags] = flags.get(cf[d].flags, 0) + 1
    fitted = [d for d in range(D) if math.isfinite(cf[d].carrier_fit_ppm)]
    err_fit = [abs(cf[d].carrier_fit_ppm - specs[d].carrier_ppm) for d in fitted]
    err_chain = [abs(res[d].total_carrier_ppm - specs[d].carrier_ppm) for d in fitted]
    drift = [abs(cf[d].drift_ppm_per_s) for d in fitted]
    rms = [cf[d].rms_hz for d in fitted]
    L.gsmcal_debug_set(3, 1)
    timed()
    stages = gsmcal.api.last_batch_stage_ms()
    plain()
    stages_without = gsmcal.api.last_batch_stage_ms()
    L.gsmcal_debug_set(3, 4)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        timed()
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and any(k in ev.name for k in ("carrier_fit", "demod_compact")):
            key = ev.name.split("(")[0].split("<")[0].replace("void ", "")
            dt = (ev.device_time if hasattr(ev, "device_time") else ev.cuda_time) / 1e3
            kern[key] = kern.get(key, 0.0) + dt
    fp64 = C.c_double(0.0)
    L.gsmcal_fp64_peak(C.byref(fp64), None)
    k_ms = kern.get("carrier_fit_row_kernel")
    flop = FLOP_GRID * n_grid + FLOP_NEWTON * n_newton
    tflops = flop / (k_ms * 1e-3) / 1e12 if k_ms else None
    pct = lambda v, q: float(np.percentile(v, q)) if v else None     # noqa: E731
    stat = lambda v: dict(max=max(v, default=None), median=statistics.median(v) if v else None, p95=pct(v, 95))     # noqa: E731
    out = dict(
        card=smi, streams=D, n_iq=n_iq, reps=a.reps,
        workload="synthetic 10 s streams, random_spec seeds 0.., device-resident (44 GB at 1024 streams)",
        calibrate_batch_ms=dict(median=statistics.median(t_plain), min=min(t_plain), max=max(t_plain), all=t_plain),
        calibrate_carrier_fit_batch_ms=dict(median=statistics.median(t_timed), min=min(t_timed), max=max(t_timed), all=t_timed),
        carrier_increment_ms_median=statistics.median(t_timed) - statistics.median(t_plain),
        stage_ms_one_group=stages, stage_ms_one_group_without_carrier=stages_without, carrier_kernel_ms_one_group=kern,
        fcch_rows=n_rows, rows_grid=n_grid, rows_newton=n_newton, rows_fitted=n_fit, flop_grid_per_row=FLOP_GRID,
        flop_newton_per_row=FLOP_NEWTON, counted_gflop=flop / 1e9,
        carrier_row_kernel_ms=k_ms, carrier_row_kernel_fp64_tflops=tflops, fp64_peak_tflops_measured=fp64.value,
        carrier_row_kernel_share_of_fp64_peak=(tflops / fp64.value) if tflops and fp64.value > 0 else None,
        carrier_flags_histogram={str(k): v for k, v in sorted(flags.items())},
        carrier_fit_ppm_vs_injected=dict(streams=len(fitted), **stat(err_fit)),
        total_carrier_ppm_vs_injected=stat(err_chain),
        drift_ppm_per_s_abs=stat(drift), fit_rms_hz=stat(rms),
        timing="host clock around each call (the call returns after its stream has drained); per-kernel times: torch.profiler CUDA activity, separate run")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("card", "calibrate_batch_ms", "calibrate_carrier_fit_batch_ms", "carrier_increment_ms_median", "stage_ms_one_group",
                                          "carrier_kernel_ms_one_group", "fcch_rows", "counted_gflop", "carrier_row_kernel_fp64_tflops",
                                          "carrier_row_kernel_share_of_fp64_peak", "fp64_peak_tflops_measured", "carrier_flags_histogram",
                                          "carrier_fit_ppm_vs_injected", "total_carrier_ppm_vs_injected", "drift_ppm_per_s_abs")}, indent=1))


if __name__ == "__main__":
    main()
