"""Time gsmcal_calibrate_sysinfo_batch against gsmcal_calibrate_cell_batch on 1024 synthetic 10 s streams (random_spec seeds 0.., each
with a BSIC, a frame number and its System Information: SI3 on the even TCs, SI4 on the odd ones, with a CGI per stream; generated on
the GPU and resident in HBM: 44 GB, far above L2), and write profiles/sysinfo_1gpu.json.

Alternates the two calls (host clock ending in the call's own stream synchronise; medians of --reps), then one run with a single stream
group (debug key 3 = 1) for the stage breakdown, then one torch.profiler run for the per-kernel CUDA times of stage [6].  Reports the
share of complete BCCH blocks that pass the Fire check, the block flag histogram and the streams whose SI3 vote gives the injected CGI.
The card's name and power limit are read in the same call."""
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
from gsmcal._lib import CarrierFitResult, SchDecodeResult, StreamResult, SysinfoResult, lib  # noqa: E402

N_IQ_10S = 21666667
FS = gsmcal.api.SYMBOL_RATE * 8


def cgi(d):
    """(ci, mcc, mnc, lac, mnc_digits) of stream d's cell: 2- and 3-digit MNCs alternate"""
    return (0x100 + 37 * d) & 0xFFFF, 200 + d % 700, d % 100, (0x3000 + 11 * d) & 0xFFFF, 2 + d % 2


def spec(d, n_iq):
    ci, mcc, mnc, lac, nd = cgi(d)
    si3, si4 = synth.si3_message(ci, mcc, mnc, lac, nd), synth.si4_message(mcc, mnc, lac, nd)
    return dataclasses.replace(synth.random_spec(d, n_iq), bsic=d % 64, tsc=(d % 64) & 7, fn0=51 * ((d * 7919) % 50000),
                               sysinfo=tuple(si3 if tc % 2 == 0 else si4 for tc in range(8)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=1024)
    ap.add_argument("--n-iq", type=int, default=N_IQ_10S)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sysinfo_1gpu.json"))
    a = ap.parse_args()
    if gsmcal.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    D, n_iq = a.streams, a.n_iq
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    raw = torch.empty((D, 2 * n_iq), dtype=torch.uint8, device="cuda")
    specs = [spec(d, n_iq) for d in range(D)]
    for d in range(D):
        synth.generate_stream(specs[d], "cuda", raw[d])
    torch.cuda.synchronize()
    coef = gsmcal.fir1(46, 200e3 / FS)
    tpl = gsmcal.gsm_SCH_training_sequence_gen(8)
    nts = np.ascontiguousarray(gsmcal.api.gsm_normal_training_sequence_gen(8).T)
    L = lib()
    cap = gsmcal.max_bursts(n_iq)
    res, cf, sd, si = (StreamResult * D)(), (CarrierFitResult * D)(), (SchDecodeResult * D)(), (SysinfoResult * D)()
    pos_info = np.empty((D, 6 * cap, 2))
    bfl, btc = np.empty((D, cap), dtype=np.uint8), np.empty((D, cap), dtype=np.uint8)
    pay, lag = np.empty((D, cap, 23), dtype=np.uint8), np.empty((D, cap, 4), dtype=np.int8)
    vp = lambda x: x.ctypes.data_as(C.c_void_p)                       # noqa: E731
    args = [C.c_void_p(raw.data_ptr()), 1, n_iq, D, 957.4e6, vp(tpl), vp(coef), len(coef), 8, 8, C.cast(res, C.c_void_p), None, None, None,
            vp(pos_info), None, C.cast(cf, C.c_void_p), None, None, None, C.cast(sd, C.c_void_p)] + [None] * 8

    def cell():
        assert L.gsmcal_calibrate_cell_batch(*args) == 0, L.gsmcal_last_error()

    def sysinfo():
        rc = L.gsmcal_calibrate_sysinfo_batch(*args, vp(nts), C.cast(si, C.c_void_p), vp(lag), None, None, None, vp(btc), vp(bfl), None, vp(pay))
        assert rc == 0, L.gsmcal_last_error()

    calls = (("calibrate_cell_batch", cell), ("calibrate_sysinfo_batch", sysinfo))
    for _, f in calls + calls:
        f()
    times = {k: [] for k, _ in calls}
    for _ in range(a.reps):
        for k, f in calls:
            t0 = time.perf_counter(); f(); torch.cuda.synchronize(); times[k].append((time.perf_counter() - t0) * 1e3)
    L.gsmcal_debug_set(3, 1)
    sysinfo()
    stages = gsmcal.api.last_batch_stage_ms()
    L.gsmcal_debug_set(3, 4)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sysinfo()
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and any(k in ev.name for k in ("bcch_", "sch_decode", "sch_demod", "demod_compact", "carrier_fit")):
            key = ev.name.split("(")[0].split("<")[0].replace("void ", "")
            dt = (ev.device_time if hasattr(ev, "device_time") else ev.cuda_time) / 1e3
            kern[key] = kern.get(key, 0.0) + dt
    flags, n_full, n_full_ok, n_payload_right, lags = {}, 0, 0, 0, {}
    for d in range(D):
        for b in range(max(si[d].n_blocks, 0)):
            f = int(bfl[d, b])
            flags[f] = flags.get(f, 0) + 1
            if f & 8 or btc[d, b] == 255:
                continue
            n_full += 1
            n_full_ok += (f & 5) == 0
            n_payload_right += f == 0 and bytes(pay[d, b]) == specs[d].sysinfo[btc[d, b]]
            for k in range(4):
                lags[int(lag[d, b, k])] = lags.get(int(lag[d, b, k]), 0) + 1
    voted = [d for d in range(D) if si[d].n_blocks >= 0 and not si[d].flags & 16]                  # the step ran and an SI3 won
    right = [d for d in voted if (si[d].ci, si[d].mcc, si[d].mnc, si[d].lac, si[d].mnc_digits) == cgi(d)]
    out = dict(
        card=smi, streams=D, n_iq=n_iq, reps=a.reps,
        workload="synthetic 10 s streams, random_spec seeds 0.. with bsic = seed % 64, tsc = bsic & 7, fn0 = 51 * (seed * 7919 % 50000) and "
                 "SI3 / SI4 of a per-stream CGI on the even / odd TCs, device-resident (44 GB at 1024 streams)",
        call_ms={k: dict(median=statistics.median(v), min=min(v), max=max(v), all=v) for k, v in times.items()},
        stage_ms_one_group=stages, stage6_kernel_ms=kern,
        blocks=sum(flags.values()), block_flags_histogram={str(k): v for k, v in sorted(flags.items())},
        complete_blocks_of_streams_with_a_cell=n_full, complete_blocks_passing_fire=n_full_ok,
        fire_pass_share=n_full_ok / n_full if n_full else None, blocks_with_the_injected_payload=n_payload_right,
        lag_histogram={str(k): v for k, v in sorted(lags.items())},
        streams_not_run=sum(1 for d in range(D) if si[d].n_blocks < 0), streams_no_cell=sum(1 for d in range(D) if si[d].flags & 4),
        streams_with_a_cell=sum(1 for d in range(D) if sd[d].bsic >= 0), streams_no_si3=sum(1 for d in range(D) if si[d].flags & 16),
        streams_with_an_si3_cgi=len(voted), streams_with_the_right_cgi=len(right), streams_with_a_wrong_cgi=len(voted) - len(right),
        streams_with_si3_disagree=sum(1 for d in range(D) if si[d].flags & 32),
        timing="host clock around each call (the call returns after its stream has drained), the two calls alternating; per-kernel times: "
               "torch.profiler CUDA activity, separate run")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items() if k not in ("workload", "timing")}, indent=1))


if __name__ == "__main__":
    main()
