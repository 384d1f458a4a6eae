"""Time gsmcal_calibrate_demod_batch against gsmcal_calibrate_batch on the config-5 workload of bench.py (1024 synthetic 10 s streams,
seeds 0.., generated on the GPU and resident in HBM: 44 GB, far above L2) and write profiles/demod_batch_1gpu.json.

Alternates the two calls (host clock ending in the call's own stream synchronise), then one run with a single stream group (debug key
3 = 1) for the stage breakdown, then one torch.profiler run for the per-kernel CUDA times of the demod stage.  FMAs per burst come
from the formula below (algorithmic count: complex MAC = 4 FMA, complex x real = 2, butterfly / twiddle cmul = 4)."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (os.path.join(ROOT, "multi-rtl-sdr-calibration_b200"), os.path.join(ROOT, "oracle")):
    sys.path.insert(0, p)

import torch  # noqa: E402

import gsmcal  # noqa: E402
from gsmcal import synth  # noqa: E402
from gsmcal._lib import DemodResult, StreamResult, lib  # noqa: E402

N_IQ_10S = 21666667
FS = gsmcal.api.SYMBOL_RATE * 8


def fma_per_sch_burst(osr=8, n_taps=47):
    N, M = 194 * osr, 2 * osr
    log2m = M.bit_length() - 1
    def dft(n_terms):
        return M * 48 * n_terms * 4 + 2 * 48 * M * 4 + 97 * (M // 2) * log2m * 4
    return dict(loader_fir=(N + 3) * n_taps * 2, derotate=N * 4, dft_received_training=dft(24), dft_x=dft(48), ifft=dft(48),
                divisions=2 * N * 8, branch_correlations=194 * 16 * osr * 4)


def fma_per_fcch_burst(osr=8):
    N, M = 148 * osr, 4 * osr                # N = 37 * M
    log2m = M.bit_length() - 1
    return dict(derotate=N * 4, row_ffts=37 * (M // 2) * log2m * 4 + N * 4, all_bins=N * 37 * 4, phasors=N * 8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=1024)
    ap.add_argument("--n-iq", type=int, default=N_IQ_10S)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "demod_batch_1gpu.json"))
    a = ap.parse_args()
    if gsmcal.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    D, n_iq = a.streams, a.n_iq
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    raw = torch.empty((D, 2 * n_iq), dtype=torch.uint8, device="cuda")
    for d in range(D):
        synth.generate_stream(synth.random_spec(d, n_iq), "cuda", raw[d])
    torch.cuda.synchronize()
    coef = gsmcal.fir1(46, 200e3 / FS)
    tpl = gsmcal.gsm_SCH_training_sequence_gen(8)
    L = lib()
    res, dem = (StreamResult * D)(), (DemodResult * D)()
    vp = lambda x: x.ctypes.data_as(C.c_void_p)                       # noqa: E731
    args = [C.c_void_p(raw.data_ptr()), 1, n_iq, D, 957.4e6, vp(tpl), vp(coef), len(coef), 8, 8, C.cast(res, C.c_void_p), None, None, None, None, None]

    def cal():
        rc = L.gsmcal_calibrate_batch(*args)
        assert rc == 0, L.gsmcal_last_error()

    def demod():
        rc = L.gsmcal_calibrate_demod_batch(*args, C.cast(dem, C.c_void_p), None, None, None, None, None, None, None)
        assert rc == 0, L.gsmcal_last_error()

    for f in (cal, demod, cal, demod):
        f()
    t_cal, t_dem = [], []
    for _ in range(a.reps):
        for f, acc in ((cal, t_cal), (demod, t_dem)):
            t0 = time.perf_counter(); f(); torch.cuda.synchronize(); acc.append((time.perf_counter() - t0) * 1e3)
    n_sch = sum(max(dem[d].n_sch_ok, 0) for d in range(D))
    n_fcch = sum(max(dem[d].n_fcch, 0) for d in range(D))
    flags = {}
    for d in range(D):
        flags[dem[d].flags] = flags.get(dem[d].flags, 0) + 1
    L.gsmcal_debug_set(3, 1)
    demod()
    stages = gsmcal.api.last_batch_stage_ms()
    L.gsmcal_debug_set(3, 4)
    fp64 = C.c_double()
    L.gsmcal_fp64_peak(C.byref(fp64), None)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        demod()
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and any(k in ev.name for k in ("demod", "fde_template")):
            key = ev.name.split("(")[0].split("<")[0].replace("void ", "")
            dt = (ev.device_time if hasattr(ev, "device_time") else ev.cuda_time) / 1e3
            kern[key] = kern.get(key, 0.0) + dt
    sch_f, fcch_f = fma_per_sch_burst(), fma_per_fcch_burst()
    fma_total = n_sch * sum(sch_f.values()) + n_fcch * sum(fcch_f.values())
    kernel_ms = sum(v for k, v in kern.items() if "sch_demod_batch" in k or "fcch_demod_batch" in k)
    out = dict(
        card=smi, streams=D, n_iq=n_iq, reps=a.reps, workload="bench.py config 5: synthetic 10 s streams, seeds 0.., device-resident (44 GB at 1024 streams)",
        calibrate_batch_ms=dict(median=statistics.median(t_cal), min=min(t_cal), max=max(t_cal), all=t_cal),
        calibrate_demod_batch_ms=dict(median=statistics.median(t_dem), min=min(t_dem), max=max(t_dem), all=t_dem),
        demod_increment_ms_median=statistics.median(t_dem) - statistics.median(t_cal),
        stage_ms_one_group=stages, demod_kernel_ms_one_group=kern,
        sch_rows_demodulated=n_sch, fcch_rows_demodulated=n_fcch, demod_flags_histogram={str(k): v for k, v in flags.items()},
        fma_per_sch_burst=sch_f, fma_per_fcch_burst=fcch_f, fma_total=fma_total,
        fp64_peak_tflops_measured=fp64.value,
        demod_kernels_tflops=(2 * fma_total / (kernel_ms * 1e-3) / 1e12) if kernel_ms else None,
        demod_kernels_share_of_fp64_peak=(2 * fma_total / (kernel_ms * 1e-3) / 1e12 / fp64.value) if kernel_ms and fp64.value else None,
        timing="host clock around each call (the call returns after its stream has drained); per-kernel times: torch.profiler CUDA activity, separate run")
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("card", "calibrate_batch_ms", "calibrate_demod_batch_ms", "demod_increment_ms_median", "stage_ms_one_group",
                                          "demod_kernel_ms_one_group", "demod_kernels_tflops", "fp64_peak_tflops_measured")}, indent=1))


if __name__ == "__main__":
    main()
