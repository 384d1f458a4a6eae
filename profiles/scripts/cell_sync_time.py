"""Time gsmcal_calibrate_cell_batch against gsmcal_calibrate_batch and gsmcal_calibrate_sch_decode_batch on 1024 synthetic 10 s streams
(random_spec seeds 0.., each with a BSIC and a frame number set so that its SCH bursts carry real coded bits; generated on the GPU and
resident in HBM: 44 GB, far above L2), and write profiles/cell_sync_1gpu.json.

Alternates the three calls (host clock ending in the call's own stream synchronise; medians of --reps), then one run with a single stream
group (debug key 3 = 1) for the stage breakdown, then one torch.profiler run for the per-kernel CUDA times of stage [6].  For both
decoding calls: the row pass rate (CRC and fields), the hamming histogram of the rows that passed, and the streams whose winner has the
injected BSIC and frame clock.  The card's name and power limit are read in the same call."""
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
from gsmcal._lib import CarrierFitResult, DemodResult, SchDecodeResult, StreamResult, lib  # noqa: E402

N_IQ_10S = 21666667
FS = gsmcal.api.SYMBOL_RATE * 8
FILTER_DELAY = -23.0                    # the 47-tap channel filter's group delay, carried by pos_info (DESIGN.md 6b)


def decode_stats(sd, ham, rfl, specs):
    D = len(specs)
    rows = [(int(ham[d, i]), int(rfl[d, i])) for d in range(D) for i in range(max(sd[d].n_sch, 0))]
    hist, flags = {}, {}
    for h, f in rows:
        flags[f] = flags.get(f, 0) + 1
        if f == 0:
            hist[h] = hist.get(h, 0) + 1
    n_ok = flags.get(0, 0)
    right = [d for d in range(D) if sd[d].n_agree > 0 and sd[d].bsic == specs[d].bsic
             and abs(sd[d].frame_clock_start - synth.true_frame_clock_start(specs[d]) - FILTER_DELAY) <= 1.0]
    wrong = [d for d in range(D) if sd[d].n_agree > 0 and d not in set(right)]
    err = {}
    for d in range(D):
        if sd[d].n_agree > 0 and sd[d].bsic == specs[d].bsic:
            e = sd[d].frame_clock_start - synth.true_frame_clock_start(specs[d])
            err[e] = err.get(e, 0) + 1
    return dict(sch_rows=len(rows), rows_passing_crc_and_fields=n_ok, row_pass_rate=n_ok / len(rows) if rows else None,
                row_flags_histogram={str(k): v for k, v in sorted(flags.items())},
                hamming_histogram_of_passing_rows={str(k): v for k, v in sorted(hist.items())},
                streams_with_winner=sum(1 for d in range(D) if sd[d].n_agree > 0), streams_n_agree_ge_2=sum(1 for d in range(D) if sd[d].n_agree >= 2),
                streams_bsic_and_frame_clock_right=len(right), streams_with_a_wrong_winner=len(wrong),
                streams_wrong_bsic=sum(1 for d in wrong if sd[d].bsic != specs[d].bsic),
                frame_clock_error_histogram_right_bsic={str(k): v for k, v in sorted(err.items())},
                wrong_winner_seeds=wrong[:40],
                streams_every_row_decoded=sum(1 for d in range(D) if sd[d].n_sch > 0 and sd[d].n_agree == sd[d].n_sch),
                streams_with_disagree=sum(1 for d in range(D) if sd[d].flags & 8), streams_uncorrected=sum(1 for d in range(D) if sd[d].flags & 16))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=1024)
    ap.add_argument("--n-iq", type=int, default=N_IQ_10S)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "cell_sync_1gpu.json"))
    a = ap.parse_args()
    if gsmcal.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    D, n_iq = a.streams, a.n_iq
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    raw = torch.empty((D, 2 * n_iq), dtype=torch.uint8, device="cuda")
    specs = [dataclasses.replace(synth.random_spec(d, n_iq), bsic=d % 64, fn0=51 * ((d * 7919) % 50000)) for d in range(D)]
    for d in range(D):
        synth.generate_stream(specs[d], "cuda", raw[d])
    torch.cuda.synchronize()
    coef = gsmcal.fir1(46, 200e3 / FS)
    tpl = gsmcal.gsm_SCH_training_sequence_gen(8)
    L = lib()
    cap = gsmcal.max_bursts(n_iq)
    res, dem, cf = (StreamResult * D)(), (DemodResult * D)(), (CarrierFitResult * D)()
    sd_old, sd_new = (SchDecodeResult * D)(), (SchDecodeResult * D)()
    ham_old, rfl_old = np.empty((D, cap), dtype=np.uint8), np.empty((D, cap), dtype=np.uint8)
    ham_new, rfl_new = np.empty((D, cap), dtype=np.uint8), np.empty((D, cap), dtype=np.uint8)
    df = np.empty((D, cap))
    pos_info = np.empty((D, 6 * cap, 2))
    vp = lambda x: x.ctypes.data_as(C.c_void_p)                       # noqa: E731
    args = [C.c_void_p(raw.data_ptr()), 1, n_iq, D, 957.4e6, vp(tpl), vp(coef), len(coef), 8, 8, C.cast(res, C.c_void_p), None, None, None,
            vp(pos_info), None]

    def batch():
        assert L.gsmcal_calibrate_batch(*args) == 0, L.gsmcal_last_error()

    def decode():
        rc = L.gsmcal_calibrate_sch_decode_batch(*args, C.cast(dem, C.c_void_p), *[None] * 7, None, None, C.cast(sd_old, C.c_void_p), None, None,
                                                 vp(ham_old), vp(rfl_old))
        assert rc == 0, L.gsmcal_last_error()

    def cell():
        rc = L.gsmcal_calibrate_cell_batch(*args, C.cast(cf, C.c_void_p), None, None, None, C.cast(sd_new, C.c_void_p), None, None, None, vp(df),
                                           None, None, vp(ham_new), vp(rfl_new))
        assert rc == 0, L.gsmcal_last_error()

    calls = (("calibrate_batch", batch), ("calibrate_sch_decode_batch", decode), ("calibrate_cell_batch", cell))
    for _, f in calls + calls:
        f()
    times = {k: [] for k, _ in calls}
    for _ in range(a.reps):
        for k, f in calls:
            t0 = time.perf_counter(); f(); torch.cuda.synchronize(); times[k].append((time.perf_counter() - t0) * 1e3)
    L.gsmcal_debug_set(3, 1)
    cell()
    stages = gsmcal.api.last_batch_stage_ms()
    L.gsmcal_debug_set(3, 4)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        cell()
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and any(k in ev.name for k in ("sch_decode", "sch_demod", "demod_compact", "carrier_fit")):
            key = ev.name.split("(")[0].split("<")[0].replace("void ", "")
            dt = (ev.device_time if hasattr(ev, "device_time") else ev.cuda_time) / 1e3
            kern[key] = kern.get(key, 0.0) + dt
    dfs = np.concatenate([df[d, :max(sd_new[d].n_sch, 0)] for d in range(D)])
    dfs = dfs[np.isfinite(dfs)]
    out = dict(
        card=smi, streams=D, n_iq=n_iq, reps=a.reps,
        workload="synthetic 10 s streams, random_spec seeds 0.. with bsic = seed % 64 and fn0 = 51 * (seed * 7919 % 50000), device-resident "
                 "(44 GB at 1024 streams)",
        call_ms={k: dict(median=statistics.median(v), min=min(v), max=max(v), all=v) for k, v in times.items()},
        stage_ms_one_group=stages, stage6_kernel_ms=kern,
        sch_df_hz=dict(rows=int(dfs.size), min=float(dfs.min()) if dfs.size else None, median=float(np.median(dfs)) if dfs.size else None,
                       max=float(dfs.max()) if dfs.size else None),
        calibrate_sch_decode_batch=decode_stats(sd_old, ham_old, rfl_old, specs),
        calibrate_cell_batch=decode_stats(sd_new, ham_new, rfl_new, specs),
        timing="host clock around each call (the call returns after its stream has drained), the three calls alternating; per-kernel times: "
               "torch.profiler CUDA activity, separate run")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items() if k not in ("workload", "timing")}, indent=1))


if __name__ == "__main__":
    main()
