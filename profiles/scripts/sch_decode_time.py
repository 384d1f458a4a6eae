"""Time gsmcal_calibrate_sch_decode_batch against gsmcal_calibrate_demod_batch on 1024 synthetic 10 s streams (random_spec seeds 0..,
each with a BSIC and a frame number set so that its SCH bursts carry real coded bits; generated on the GPU and resident in HBM: 44 GB, far
above L2), and write profiles/sch_decode_1gpu.json.

Alternates the two calls (host clock ending in the call's own stream synchronise; medians of --reps), then one run of each with a single
stream group (debug key 3 = 1) for the stage breakdown, then one torch.profiler run for the per-kernel CUDA times of stage [6].  Also the
row CRC pass rate, the hamming histogram of the rows that passed, the streams with a winner / with DISAGREE / whose winner matches the
injected BSIC and frame clock, and the card's name and power limit read in the same call."""
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
from gsmcal._lib import DemodResult, SchDecodeResult, StreamResult, lib  # noqa: E402

N_IQ_10S = 21666667
FS = gsmcal.api.SYMBOL_RATE * 8


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=1024)
    ap.add_argument("--n-iq", type=int, default=N_IQ_10S)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sch_decode_1gpu.json"))
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
    res, dem, sd = (StreamResult * D)(), (DemodResult * D)(), (SchDecodeResult * D)()
    ham, rfl = np.empty((D, cap), dtype=np.uint8), np.empty((D, cap), dtype=np.uint8)
    pos_info = np.empty((D, 6 * cap, 2))
    vp = lambda x: x.ctypes.data_as(C.c_void_p)                       # noqa: E731
    args = [C.c_void_p(raw.data_ptr()), 1, n_iq, D, 957.4e6, vp(tpl), vp(coef), len(coef), 8, 8, C.cast(res, C.c_void_p), None, None, None,
            vp(pos_info), None, C.cast(dem, C.c_void_p)] + [None] * 7

    def demod():
        rc = L.gsmcal_calibrate_demod_batch(*args)
        assert rc == 0, L.gsmcal_last_error()

    def decode():
        rc = L.gsmcal_calibrate_sch_decode_batch(*args, None, None, C.cast(sd, C.c_void_p), None, None, vp(ham), vp(rfl))
        assert rc == 0, L.gsmcal_last_error()

    for f in (demod, decode, demod, decode):
        f()
    t_demod, t_decode = [], []
    for _ in range(a.reps):
        for f, acc in ((demod, t_demod), (decode, t_decode)):
            t0 = time.perf_counter(); f(); torch.cuda.synchronize(); acc.append((time.perf_counter() - t0) * 1e3)
    rows = [(int(ham[d, i]), int(rfl[d, i])) for d in range(D) for i in range(max(sd[d].n_sch, 0))]
    row_flags = {}
    for _, f in rows:
        row_flags[f] = row_flags.get(f, 0) + 1
    hist = {}
    for h, f in rows:
        if f == 0:
            hist[h] = hist.get(h, 0) + 1
    stream_flags = {}
    for d in range(D):
        stream_flags[sd[d].flags] = stream_flags.get(sd[d].flags, 0) + 1
    winners = [d for d in range(D) if sd[d].n_agree > 0]
    trusted = [d for d in winners if sd[d].n_agree >= 2]
    err = [sd[d].frame_clock_start - synth.true_frame_clock_start(specs[d]) for d in trusted]
    right = [d for d in trusted if sd[d].bsic == specs[d].bsic]
    L.gsmcal_debug_set(3, 1)
    decode()
    stages = gsmcal.api.last_batch_stage_ms()
    demod()
    stages_without = gsmcal.api.last_batch_stage_ms()
    L.gsmcal_debug_set(3, 4)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        decode()
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and any(k in ev.name for k in ("sch_decode", "sch_demod", "demod_compact", "fcch_demod")):
            key = ev.name.split("(")[0].split("<")[0].replace("void ", "")
            dt = (ev.device_time if hasattr(ev, "device_time") else ev.cuda_time) / 1e3
            kern[key] = kern.get(key, 0.0) + dt
    n_ok = sum(1 for _, f in rows if f == 0)
    out = dict(
        card=smi, streams=D, n_iq=n_iq, reps=a.reps,
        workload="synthetic 10 s streams, random_spec seeds 0.. with bsic = seed % 64 and fn0 = 51 * (seed * 7919 % 50000), device-resident "
                 "(44 GB at 1024 streams)",
        calibrate_demod_batch_ms=dict(median=statistics.median(t_demod), min=min(t_demod), max=max(t_demod), all=t_demod),
        calibrate_sch_decode_batch_ms=dict(median=statistics.median(t_decode), min=min(t_decode), max=max(t_decode), all=t_decode),
        decode_increment_ms_median=statistics.median(t_decode) - statistics.median(t_demod),
        stage_ms_one_group=stages, stage_ms_one_group_without_decode=stages_without, stage6_kernel_ms=kern,
        sch_decode_kernel_ms=kern.get("sch_decode_batch_kernel"),
        sch_rows=len(rows), rows_passing_crc_and_fields=n_ok, row_pass_rate=n_ok / len(rows) if rows else None,
        row_flags_histogram={str(k): v for k, v in sorted(row_flags.items())},
        hamming_histogram_of_passing_rows={str(k): v for k, v in sorted(hist.items())},
        stream_flags_histogram={str(k): v for k, v in sorted(stream_flags.items())},
        streams_with_winner=len(winners), streams_with_disagree=sum(1 for d in range(D) if sd[d].flags & 8),
        streams_n_agree_ge_2=len(trusted), of_those_bsic_right=len(right),
        frame_clock_error_samples=dict(min=min(err, default=None), max=max(err, default=None)),
        timing="host clock around each call (the call returns after its stream has drained); per-kernel times: torch.profiler CUDA activity, separate run")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items() if k not in ("workload", "timing")}, indent=1))


if __name__ == "__main__":
    main()
