"""Time the SCH stage with the fp32 screen of sch_corr_kernel (debug key 24 = 0) against the fp64 correlation of every lag (= 1) on 1024
synthetic 10 s streams (seeds 0.., generated on the GPU and resident in HBM: 44 GB, far above L2), and write profiles/sch_screen_1gpu.json.

One stream group (debug key 3 = 1) so that gsmcal_last_batch_stage_ms reports the stages one after the other.  The two modes alternate
in one process; each call's whole time (host clock ending in a synchronise) and its "sch" stage time are recorded.  Also records the
screen's counters (bursts decided, candidate histogram, fallbacks), whether both modes returned identical records, and the card's name,
power limit and SM clock read in the same call."""
import argparse
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
from gsmcal._lib import lib  # noqa: E402

N_IQ_10S = 21666667
FS = gsmcal.api.SYMBOL_RATE * 8


def smi():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()


def summary(v):
    return dict(median=statistics.median(v), min=min(v), max=max(v), all=v)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=1024)
    ap.add_argument("--n-iq", type=int, default=N_IQ_10S)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sch_screen_1gpu.json"))
    a = ap.parse_args()
    if gsmcal.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    D, n_iq = a.streams, a.n_iq
    card_before = smi()
    raw = torch.empty((D, 2 * n_iq), dtype=torch.uint8, device="cuda")
    for d in range(D):
        synth.generate_stream(synth.random_spec(d, n_iq), "cuda", raw[d])
    torch.cuda.synchronize()
    coef = gsmcal.fir1(46, 200e3 / FS)
    tpl = gsmcal.gsm_SCH_training_sequence_gen(8)
    L = lib()
    L.gsmcal_debug_set(3, 1)

    def run(mode):
        assert L.gsmcal_debug_set(24, mode) == 0
        t0 = time.perf_counter()
        out = gsmcal.calibrate_batch(None, 957.4e6, tpl, coef, device_ptr=raw.data_ptr(), n_iq=n_iq, n_streams=D)
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3
        g = L.gsmcal_debug_get
        stats = dict(screened=g(120), fallback=g(121), candidates_hist={str(c): g(121 + c) for c in range(1, 9)})
        return out, ms, gsmcal.api.last_batch_stage_ms(), stats

    try:
        first = {m: run(m) for m in (0, 1)}                                # warm-up, and the records to compare
        same = True
        for s0, s1 in zip(first[0][0], first[1][0]):
            for k in s0:
                if not np.array_equal(np.asarray(s0[k]), np.asarray(s1[k])):
                    same = False
        call, sch, stats = {0: [], 1: []}, {0: [], 1: []}, {}
        for _ in range(a.reps):
            for m in (0, 1):
                _, ms, st, stats[m] = run(m)
                call[m].append(ms)
                sch[m].append(st["sch"])
        stages = {m: run(m)[2] for m in (0, 1)}
    finally:
        L.gsmcal_debug_set(24, 0)
        L.gsmcal_debug_set(3, 4)
    out = dict(
        card_before=card_before, card_after=smi(), streams=D, n_iq=n_iq, reps=a.reps,
        workload="synthetic 10 s streams, seeds 0.., device-resident (44 GB at 1024 streams), one stream group (debug key 3 = 1)",
        sch_stage_ms_screen=summary(sch[0]), sch_stage_ms_fp64=summary(sch[1]),
        sch_stage_saving_ms_median=statistics.median(sch[1]) - statistics.median(sch[0]),
        call_ms_screen=summary(call[0]), call_ms_fp64=summary(call[1]),
        stage_ms_screen=stages[0], stage_ms_fp64=stages[1],
        screen_counters=stats[0], fp64_counters=stats[1],
        records_identical=same,
        timing="sch: gsmcal_last_batch_stage_ms (CUDA events around the stage); call: host clock around the call, ending in a synchronise")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("card_before", "sch_stage_ms_screen", "sch_stage_ms_fp64", "sch_stage_saving_ms_median",
                                          "call_ms_screen", "call_ms_fp64", "screen_counters", "records_identical")}, indent=1))


if __name__ == "__main__":
    main()
