#!/usr/bin/env python
"""bench.py - calibrated IQ MSamples/s of the GSM sync/calibration hot path (BASELINE.json metric).

Workload = BASELINE config 5 itself at every N: 1024 synthetic dongle streams x 10 s (21,666,667 IQ at 2.1667 MS/s,
uint8) through the full FCCH/SCH/ppm pipeline (gsm_sync_demod.m:107-124: raw2iq -> FIR -> FCCH coarse -> FCCH fine ->
SCH -> post-SCH carrier -> ppm), sharded as contiguous blocks of 1024/N streams per GPU (strong scaling; all 1024 =
44.4 GB of uint8 fit one B200).  Streams are independent (SURVEY.md 8e): no data-path collective, only the 88-byte
per-stream result records are all-gathered over NCCL.  One step = one pass over all 1024 streams.

  value : whole-job MS/s with the uint8 captures resident in HBM when the timed region starts
  e2e   : the same through the C-ABI call with HOST (pinned) buffers, H2D + result D2H inside the region
  --impl reference : the CPU oracle (NumPy restatement of the reference .m files; MATLAB/Octave are probed for and
                     absent in this image) on all host cores; every step is a bounded sample of the SAME workload:
                     `cores` whole 10 s streams of the 1024
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import shutil
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(ROOT, "multi-rtl-sdr-calibration_b200"), os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

SYMBOL_RATE = (1625.0 / 6.0) * 1e3
FS = SYMBOL_RATE * 8
CARRIER = 957.4e6
N_IQ_10S = 21666667
TOTAL_STREAMS = 1024                 # BASELINE config 5
SUB_BATCH = 512                      # streams per submitted batch (2 batches in flight)
METRIC = "calibrated IQ MSamples/s"

# Algorithmic fp64 work per FCCH burst (FMA counts; one FMA = 2 flop) of the osr-8 kernels, DESIGN.md section 4 derives them.  Only
# the arithmetic the algorithm needs is counted - FIR taps x samples, Horner DFT accumulations, correlation MACs, the per-sample
# complex multiplies of the tone stage; slides, certificates, index math, reductions and conversions are NOT, so `achieved` is a
# lower bound of the FP64 instruction rate (ncu's pipe-active figure sits beside it in the roofline object).
FMA_PER_BURST = {
    "fine_fir": 2208 * 47 * 2,                    # 47-tap FIR over the 2208-sample search window, once per burst (fine_core8_kernel)
    "fine_pass": 2208 * 8 * 4,                    # chunk sums of one pass: 8 tracked bins, Horner, 4 FMA per sample and bin
    "fine_tier2": 2208 * 64 * 5 + 1025 * 64 * 8,  # 64-bin band kernel on the cached window: piece sums + slide
    "tone1": 1184 * (8 * 4 + 4 * 4 + 4 + 4 + 4),  # 8-bin Horner band DFT, 4 gate bins, gate phasor, integer-bin derotation, phasor ratios
    "tone2": 1184 * (8 * 4 + 4 + 4),              # post-SCH stage: no gate
    "sch": 646 * 47 * 2 + 89 * 512 * 4,           # FIR of the SCH window + 89-lag x 512-tap correlation
}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def profile_facts():
    """Numbers that come from committed ncu captures (profiles/roofline_facts.json, written by profiles/summarize.py --facts):
    dram bytes per launch of the HBM-bound kernel, fp64 pipe utilisation of the burst kernels."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_facts.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def probe_reference_runtimes():
    """BASELINE.md section 2 / SURVEY 8d: the reference's own function files could be timed under GNU Octave or MATLAB if either
    were installed on the box.  Neither is in this image; the probe is recorded in the JSON line either way."""
    found = {k: shutil.which(k) for k in ("octave", "octave-cli", "matlab", "mkoctfile")}
    return {"found": {k: v for k, v in found.items() if v}, "probed": sorted(found),
            "used": "none - CPU arm is oracle/gsmcal_oracle.py (NumPy/SciPy restatement); oracle/run_reference.m is the recipe "
                    "for a box that has Octave" if not any(found.values()) else "present but the harness only times the oracle"}


class ClockSampler:
    """SM clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe): NVML polled every 5 ms from a
    thread (the timed region is short); nvidia-smi is the fallback."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []
        self.sm, self.mx, self.reasons, self.power = [], [], set(), []
        self.stop_flag = threading.Event()
        self.nvml = None
        self.active = threading.Event()

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        names = {"hw_slowdown": n.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": n.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": n.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": n.nvmlClocksThrottleReasonSwPowerCap}
        while not self.stop_flag.is_set():
            if self.active.is_set():
                try:
                    self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
                    self.mx.append(float(n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)))
                    self.power.append(n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0)
                    mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                    for k, bit in names.items():
                        if mask & bit:
                            self.reasons.add(k)
                except Exception:
                    pass
            time.sleep(0.005)

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag.set()
            self.thread.join(timeout=1)
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                    "reasons": sorted(self.reasons), "samples": len(self.sm), "power_w_max": max(self.power) if self.power else None,
                    "source": "nvml, 5 ms period, timed region only"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 100 (warm-up + timed region)"}


def workload_config(n_gpus, streams_per_gpu=None, n_iq=N_IQ_10S, scaling="strong"):
    spg = streams_per_gpu if streams_per_gpu is not None else TOTAL_STREAMS // max(n_gpus, 1)
    total = spg * n_gpus
    name = "BASELINE config 5" if (total == TOTAL_STREAMS and n_iq == N_IQ_10S) else "BASELINE config 5 (reduced by flags)"
    return {"workload": f"{name}: {total} synthetic dongle streams x {n_iq / FS:.1f} s ({n_iq} IQ @ 2.1667 MS/s uint8), "
                        f"full FCCH/SCH/ppm pipeline (gsm_sync_demod.m:107-124), {spg} streams per GPU",
            "streams_per_gpu": spg, "streams_total": total, "iq_per_stream": n_iq,
            "carrier_hz": CARRIER, "fir": "fir1(46, 200e3/fs)", "oversampling": 8, "seeds": f"0..{total - 1}",
            "l2": f"inputs ({spg * 2 * n_iq / 1e9:.1f} GB per GPU) are far larger than the 126 MB L2; no flush needed",
            "parallelism": f"contiguous blocks of streams over {n_gpus} GPU(s); all_gather of 88-byte result records only"}


# ---------------------------------------------------------------------------------------------------
# CPU reference arm: the oracle over a process pool (one whole stream per worker per step)
# ---------------------------------------------------------------------------------------------------
_WORKER = {}


def _oracle_init(n, counter):
    """Pool initializer: every worker process generates and keeps ONE synthetic stream of the workload (untimed)."""
    import gsmcal_oracle as oracle
    from gsmcal import synth
    import torch
    torch.set_num_threads(1)
    with counter.get_lock():
        seed = counter.value                 # stream `seed` of the 1024 (the GPU arm's rank-0 streams use the same seeds)
        counter.value += 1
    _WORKER["raw"] = synth.generate_stream(synth.random_spec(seed, n)).numpy()
    _WORKER["tpl"] = oracle.gsm_SCH_training_sequence_gen(8)
    _WORKER["coef"] = oracle.fir1(46, 200e3 / FS)


def _oracle_worker(_):
    import gsmcal_oracle as oracle
    res = oracle.calibrate_stream(_WORKER["raw"], CARRIER, _WORKER["tpl"], _WORKER["coef"])
    return len(res["pos_info"])


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[v] = "1"
    import multiprocessing as mp
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    workers = max(1, min(cores, 64))
    n = args.n_iq                    # whole streams of the workload (10 s): same config as the GPU arm, `workers` of the 1024 per step
    ctx = mp.get_context("fork")
    counter = ctx.Value("i", 0)
    jobs = list(range(workers))
    with ctx.Pool(workers, initializer=_oracle_init, initargs=(n, counter)) as pool:
        for _ in range(args.warmup):
            pool.map(_oracle_worker, jobs, chunksize=1)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            rows = pool.map(_oracle_worker, jobs, chunksize=1)
        dt = time.perf_counter() - t0
    value = workers * n * args.steps / dt / 1e6
    spg = args.streams if args.streams else None
    sample = (f"each step = {workers} whole streams (seeds 0..{workers - 1}) of the workload's {TOTAL_STREAMS}, {n} IQ ({n / FS:.1f} s) each, "
              f"one oracle process per host core; pos_info rows per stream {min(rows)}..{max(rows)}; the oracle materialises "
              "r (filtered, resampled, derotated complex128 streams) as the reference does")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "MS/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak" if args.weak else "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.gpus, spg, n, "weak" if args.weak else "strong"),
            "cpu_baseline": {"value": value, "unit": "MS/s", "cores": workers, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "MS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "reference_runtime_probe": probe_reference_runtimes(),
            "note": "MATLAB/Octave absent: the reference arm is oracle/gsmcal_oracle.py (NumPy/SciPy fp64 restatement of the .m files)"}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# oracle agreement on the timed workload (side leg, outside every timed region)
# ---------------------------------------------------------------------------------------------------
def _agree_worker(job):
    """(index, raw uint8) -> (index, oracle result without the materialised stream).  Runs in a spawned process (no CUDA)."""
    idx, raw = job
    for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[v] = "1"
    import gsmcal_oracle as oracle
    tpl = oracle.gsm_SCH_training_sequence_gen(8)
    coef = oracle.fir1(46, 200e3 / FS)
    ref = oracle.calibrate_stream(raw, CARRIER, tpl, coef)
    ref.pop("r_final", None)
    return idx, ref


def outcome_of(n_coarse, n_fcch, n_pos_info, flags):
    if n_coarse < 0:
        return "no_fcch_found"
    if n_coarse < 5:
        return "fewer_than_5_coarse_hits"
    if n_fcch < 0:
        return "fine_spacing_fail" if flags & 1 else ("fine_snr_gate" if flags & 2 else "fine_sentinel")
    if n_fcch < 5:
        return "fewer_than_5_fcch"
    if n_pos_info < 0:
        return "sch_edge_abort" if flags & 4 else "sch_sentinel"
    if flags & 8:
        return "sch_spacing_fail"
    if flags & 16:
        return "post_few_bcch"
    return "calibrated"


def same_result(got, ref):
    ok = (np.array_equal(got["coarse_pos"], ref["coarse_pos"]) and np.array_equal(got["fcch_pos"], ref["fcch_pos"])
          and np.array_equal(got["pos_info"], ref["pos_info"]))
    for k in ("sampling_ppm", "carrier_ppm"):
        for a, b in zip(got[k], ref[k]):
            ok = ok and ((a == b) if math.isinf(b) else abs(a - b) < 1e-3)
    for k in ("total_sampling_ppm", "total_carrier_ppm"):
        ok = ok and ((got[k] == ref[k]) if math.isinf(ref[k]) else abs(got[k] - ref[k]) < 1e-3)
    return bool(ok)


def oracle_agreement(gsmcal, raw, res, n_iq, tpl, coef, count, workers):
    """Every stream of this rank that did NOT fully calibrate plus evenly spaced others (>= `count` in total): the batched
    CUDA pipeline's full outputs (positions, pos_info, ppm) against oracle.calibrate_stream on a process pool."""
    import multiprocessing as mp
    D = raw.shape[0]
    outcomes = [outcome_of(r.n_coarse, r.n_fcch, r.n_pos_info, r.flags) for r in res]
    hist = {}
    for o in outcomes:
        hist[o] = hist.get(o, 0) + 1
    # every outcome kind is represented: round-robin over the non-calibrating kinds (up to 3/4 of the budget, rare kinds first), the rest
    # evenly spaced fully calibrating streams
    by_kind = {}
    for d in range(D):
        if outcomes[d] != "calibrated":
            by_kind.setdefault(outcomes[d], []).append(d)
    pick, budget = [], (3 * count) // 4
    kinds = sorted(by_kind, key=lambda k_: len(by_kind[k_]))
    i_ = 0
    while len(pick) < budget and any(by_kind[k_] for k_ in kinds):
        k_ = kinds[i_ % len(kinds)]
        if by_kind[k_]:
            pick.append(by_kind[k_].pop(0))
        i_ += 1
    cal = [d for d in range(D) if outcomes[d] == "calibrated"]
    if cal:
        want = max(0, count - len(pick))
        pick += [cal[i] for i in sorted(set(np.linspace(0, len(cal) - 1, num=min(len(cal), want)).astype(int).tolist()))]
    pick = sorted(set(pick))
    got = {}
    for d in pick:
        got[d] = gsmcal.calibrate_batch(None, CARRIER, tpl, coef, device_ptr=raw[d].data_ptr(), n_iq=n_iq, n_streams=1)[0]
    jobs = [(d, raw[d].cpu().numpy()) for d in pick]
    t0 = time.perf_counter()
    with mp.get_context("spawn").Pool(max(1, min(workers, len(jobs)))) as pool:
        refs = dict(pool.map(_agree_worker, jobs, chunksize=1))
    dt = time.perf_counter() - t0
    bad = [d for d in pick if not same_result(got[d], refs[d])]
    checked_hist = {}
    for d in pick:
        checked_hist[outcomes[d]] = checked_hist.get(outcomes[d], 0) + 1
    return {"oracle_agrees": f"{len(pick) - len(bad)}/{len(pick)}", "mismatching_streams": bad, "checked_streams": pick,
            "checked_outcomes": checked_hist, "outcome_histogram_rank0": hist, "oracle_wall_s": dt,
            "compared": "coarse_pos, fcch_pos, pos_info bit-exact; sampling/carrier ppm (both stages and totals) within 1e-3"}


def dump_outputs(out_dir, res, record_type):
    """What the timed path hands its caller: the per-stream result records (gsmcal_calibrate_batch_collect), in stream order, one
    float64 array per record field (counts, flags and lengths are integers, exact in float64), so two builds can be compared field by
    field on the same seeded inputs.

    A stream that does not calibrate reports its ppm as inf (the reference's "no estimate", FCCH_fine_correction.m:8-15), so every
    floating-point field is written finite: <field>.npy holds 0 where the value is not finite and <field>_nonfinite.npy says which
    value it was (0 finite, 1 +inf, -1 -inf, 2 nan)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, ctype in record_type._fields_:
        vals = [getattr(r, name) for r in res]
        a = np.array([list(v) if isinstance(v, C.Array) else v for v in vals], dtype=np.float64)
        if (ctype._type_ if issubclass(ctype, C.Array) else ctype) is C.c_double:
            code = np.select([np.isposinf(a), np.isneginf(a), np.isnan(a)], [1.0, -1.0, 2.0], 0.0)
            np.save(os.path.join(out_dir, name + "_nonfinite.npy"), code)
            a = np.where(code == 0, a, 0.0)
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------------
def numa_pin(local_rank):
    """Pin this process (and the pinned host allocations it makes afterwards, first-touch) to the NUMA node of its GPU."""
    info = {"applied": False}
    try:
        import torch
        prop = torch.cuda.get_device_properties(local_rank)
        bus, dom, dev_id = getattr(prop, "pci_bus_id", None), getattr(prop, "pci_domain_id", 0), getattr(prop, "pci_device_id", 0)
        if bus is None:
            return info
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev_id:02x}.0"
        with open(os.path.join(path, "numa_node")) as f:
            node = int(f.read().strip())
        info["pci"], info["numa_node"] = os.path.basename(path), node
        if node < 0:
            return info
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
            info["applied"], info["cpus"] = True, len(allowed)
    except Exception as ex:      # noqa: BLE001
        info["error"] = repr(ex)
    return info


def run_ingest(args):
    """Loopback rtl_tcp replay -> pinned double-buffered ingest -> gsmcal_calibrate_batch(HOST), wall clock (host path)."""
    import gsmcal
    from gsmcal import ingest, synth
    from gsmcal.rtl_tcp_replay import ReplayDongle
    D, n_iq = args.ingest, min(args.n_iq, 2_166_667)
    gsmcal.set_device(0)
    specs = [synth.random_spec(d, n_iq) for d in range(D)]
    raw = synth.generate_batch(specs, device="cuda").cpu().numpy()
    srvs = [ReplayDongle(raw[d]) for d in range(D)]
    coef, tpl = gsmcal.fir1(46, 200e3 / FS), gsmcal.gsm_SCH_training_sequence_gen(8)
    try:
        with ingest.DongleIngest([(s.host, s.port) for s in srvs], n_iq, CARRIER, FS, n_threads=min(16, os.cpu_count() or 1)) as ing:
            locked, t0, k = 0, None, 0
            for buf in ing.captures(args.warmup + args.steps):
                if k == args.warmup:
                    t0 = time.perf_counter()
                res = gsmcal.calibrate_batch(buf, CARRIER, tpl, coef, details=False)
                locked = sum(1 for r in res if r.total_sampling_ppm == r.total_sampling_ppm and abs(r.total_sampling_ppm) < 1e9)
                k += 1
            dt = time.perf_counter() - t0
    finally:
        for s in srvs:
            s.close()
    rate = args.steps * D * n_iq / dt / 1e6
    print(json.dumps({"metric": "ingested + calibrated IQ MSamples/s (loopback rtl_tcp replay, wall clock)", "value": rate,
                      "unit": "MS/s", "dongles": D, "n_iq_per_capture": n_iq, "captures": args.steps,
                      "ms_per_capture": 1e3 * dt / args.steps, "realtime_dongles_equiv": rate * 1e6 / FS,
                      "locked_streams_last_capture": locked, "socket_gbs": 2 * rate / 1e3,
                      "note": "bounded by the Python replay servers + loopback TCP on the host cores, not by the GPU"}))


# ---------------------------------------------------------------------------------------------------
# BASELINE configs 1-4: the drop-in call sequences the reference scripts make, wall clock, next to the oracle on the same arrays
# ---------------------------------------------------------------------------------------------------
def _cfg_chain_worker(job):
    raw, = job
    import gsmcal_oracle as oracle
    tpl = oracle.gsm_SCH_training_sequence_gen(8)
    coef = oracle.fir1(46, 200e3 / FS)
    t0 = time.perf_counter()
    ref = oracle.calibrate_stream(raw, CARRIER, tpl, coef)
    return time.perf_counter() - t0, ref["total_sampling_ppm"], ref["total_carrier_ppm"], len(ref["pos_info"])


def _cfg_scan_worker(job):
    raw, order = job
    import gsmcal_oracle as oracle
    coef = oracle.fir1(order, 200e3 / FS)
    t0 = time.perf_counter()
    snr, num_hit, _, _ = oracle.fcch_scan_channel(raw, coef)
    return time.perf_counter() - t0, snr, num_hit


def _cfg_power_worker(job):
    cols, coef, decim = job
    import gsmcal_oracle as oracle
    t0 = time.perf_counter()
    p = oracle.band_power(cols, coef, decim)
    return time.perf_counter() - t0, p


def dropin_chain(gsmcal, raw_cols, tpl, coef):
    """gsm_sync_demod.m:107-124 function by function through the drop-in entry points (host arrays in and out of every call)."""
    r = gsmcal.raw2iq(raw_cols)                                  # :107
    r = gsmcal.fir_filter(coef, r)                               # :110
    out = []
    for i in range(r.shape[1]):                                  # :112
        col = np.ascontiguousarray(r[:, i])
        pos, _ = gsmcal.FCCH_coarse_position(col[::64], 8)      # :117
        fpos, r1, sp1, cp1 = gsmcal.FCCH_fine_correction(col, pos, 8, CARRIER)             # :118
        pinfo, r2, sp2 = gsmcal.SCH_corr_rate_correction(r1, fpos, tpl, 8)                # :119
        r3, cp2 = gsmcal.carrier_correct_post_SCH(r2, pinfo, 8, CARRIER)                  # :120
        out.append((gsmcal.total_ppm_calculation([sp1, sp2]), gsmcal.total_ppm_calculation([cp1, cp2]), len(pinfo)))   # :123-124
    return out


def run_configs(gsmcal, synth, workers, quick=False):
    """Timings for BASELINE configs 1-4 (config 5 is the main line).  Wall clock around the calls a MATLAB caller would make
    (pageable host arrays, H2D/D2H inside every call) and around the oracle on the same arrays (process pool, `workers` cores)."""
    import multiprocessing as mp
    import gsmcal_oracle as oracle
    out = {}
    tpl, coef = gsmcal.gsm_SCH_training_sequence_gen(8), gsmcal.fir1(46, 200e3 / FS)
    pool = mp.get_context("spawn").Pool(workers)

    def chain_case(name, D, n, note):
        specs = [synth.random_spec(5000 + d, n) for d in range(D)]
        raw = synth.generate_batch(specs, device="cuda").cpu().numpy()
        cols = raw.T                                             # 2N x D as the script holds it (column-major, like a MATLAB matrix: no copy)
        dropin_chain(gsmcal, cols[:, :1], tpl, coef)             # warm-up (allocations, module load)
        t0 = time.perf_counter(); got = dropin_chain(gsmcal, cols, tpl, coef); t_drop = time.perf_counter() - t0
        gsmcal.calibrate_batch(raw[:1], CARRIER, tpl, coef, details=False)
        t0 = time.perf_counter(); res = gsmcal.calibrate_batch(raw, CARRIER, tpl, coef, details=False); t_batch = time.perf_counter() - t0
        t0 = time.perf_counter(); refs = pool.map(_cfg_chain_worker, [(raw[d],) for d in range(D)], chunksize=1); t_pool = time.perf_counter() - t0
        agree = all(abs(g[0] - r[1]) < 1e-3 and abs(g[1] - r[2]) < 1e-3 and g[2] == r[3] for g, r in zip(got, refs)
                    if math.isfinite(r[1]) and math.isfinite(r[2]))
        agree_b = all(abs(res[d].total_sampling_ppm - refs[d][1]) < 1e-3 for d in range(D) if math.isfinite(refs[d][1]))
        iq = D * n
        out[name] = {"what": note, "streams": D, "iq_per_stream": n,
                     "dropin_chain_MSps": iq / t_drop / 1e6, "dropin_chain_s": t_drop,
                     "calibrate_batch_host_MSps": iq / t_batch / 1e6, "calibrate_batch_s": t_batch,
                     "oracle_MSps_one_core": n / (sum(r[0] for r in refs) / D) / 1e6, "oracle_pool_MSps": iq / t_pool / 1e6, "oracle_pool_cores": min(workers, D),
                     "speedup_dropin_vs_one_core": (iq / t_drop) / (n / (sum(r[0] for r in refs) / D)),
                     "results_agree_with_oracle": bool(agree and agree_b),
                     "bytes_materialised_per_iq": 178, "note": "drop-in chain = 178 B/sample through pageable host arrays, PCIe both ways in every call"}

    try:
        chain_case("1", 2, 1020000, "gsm_sync_demod.m:107-124, 2 dongles x 1,020,000 IQ (the script's own size)")
        if not quick:
            chain_case("3", 8, N_IQ_10S, "gsm_sync_demod.m:107-124, 8 dongles x 10 s on one GPU")
        # config 2: multi_rtl_sdr_gsm_FCCH_scanner.m:132-136,163-186 - 126 frequencies x 640,000 IQ, fir1(30), /64, coarse + acceptance
        n, nf = 640000, 126
        specs = []
        for c in range(nf):
            if c % 10 == 3:
                specs.append(synth.StreamSpec(seed=6000 + c, n_samples=n, sampling_ppm=float((c % 7) * 5 - 15), carrier_ppm=float((c % 5) * 4 - 8),
                                              snr_db=18.0, start_offset=float(1000 * c)))
            else:
                specs.append(synth.StreamSpec(seed=6000 + c, n_samples=n, noise_only=True))
        raw = synth.generate_batch(specs, device="cuda").cpu().numpy()
        coef30 = gsmcal.fir1(30, 200e3 / FS)
        gsmcal.fcch_scan(raw[:2], coef30)
        t0 = time.perf_counter(); snr, num_hit, _ = gsmcal.fcch_scan(raw, coef30); t_gpu = time.perf_counter() - t0
        t0 = time.perf_counter(); refs = pool.map(_cfg_scan_worker, [(raw[c], 30) for c in range(nf)], chunksize=2); t_pool = time.perf_counter() - t0
        agree = all(num_hit[c] == refs[c][2] and abs(snr[c] - refs[c][1]) < 1e-9 for c in range(nf))
        out["2"] = {"what": "multi_rtl_sdr_gsm_FCCH_scanner.m:132-136,163-186: 126 frequencies (935:0.2:960 MHz) x 640,000 IQ, fir1(30), /64, FCCH_coarse_position + acceptance",
                    "channels": nf, "iq_per_channel": n, "gsmcal_fcch_scan_MSps": nf * n / t_gpu / 1e6, "gsmcal_fcch_scan_s": t_gpu,
                    "oracle_MSps_one_core": n / (sum(r[0] for r in refs) / nf) / 1e6, "oracle_pool_MSps": nf * n / t_pool / 1e6, "oracle_pool_cores": workers,
                    "channels_with_carrier": int(sum(1 for c in range(nf) if num_hit[c] > 0)), "results_agree_with_oracle": bool(agree)}
        # config 4: scan_band_power_spectrum.m:80-85 (251 x 2 x 12,288 IQ) and multi_rtl_sdr_split_scanner.m:154-156 (501 x 204,800 IQ, fir1(63), /20)
        rng = np.random.default_rng(44)
        a = np.clip(np.round(rng.standard_normal((502, 2 * 12288)) * 20 + 127.5), 0, 255).astype(np.uint8).T     # column-major 24576 x 502
        gsmcal.band_power(a[:, :2])
        t0 = time.perf_counter(); p_gpu = gsmcal.band_power(a); t_gpu = time.perf_counter() - t0
        t0 = time.perf_counter(); p_ref = oracle.band_power(a); t_ref = time.perf_counter() - t0
        b = np.clip(np.round(rng.standard_normal((501, 2 * 204800)) * 20 + 127.5), 0, 255).astype(np.uint8).T   # column-major 409600 x 501
        coef63 = gsmcal.fir1(63, 0.05 / 2.048)
        gsmcal.band_power(b[:, :2], coef63, 20)
        t0 = time.perf_counter(); q_gpu = gsmcal.band_power(b, coef63, 20); t_gpu2 = time.perf_counter() - t0
        chunks = [(np.ascontiguousarray(b[:, i:i + 32]), coef63, 20) for i in range(0, 501, 32)]
        t0 = time.perf_counter(); q_parts = pool.map(_cfg_power_worker, chunks, chunksize=1); t_pool = time.perf_counter() - t0
        q_ref = np.concatenate([p for _, p in q_parts])
        out["4"] = {"what": "scan_band_power_spectrum.m:80-85 (251 freq x 2 dongles x 12,288 IQ, mean power) and multi_rtl_sdr_split_scanner.m:154-156 (501 freq x 204,800 IQ, fir1(63), /20, mean power)",
                    "band_power_MSps": 502 * 12288 / t_gpu / 1e6, "band_power_oracle_MSps_one_core": 502 * 12288 / t_ref / 1e6,
                    "split_scanner_MSps": 501 * 204800 / t_gpu2 / 1e6, "split_scanner_oracle_MSps_one_core": 501 * 204800 / sum(t for t, _ in q_parts) / 1e6,
                    "split_scanner_oracle_pool_MSps": 501 * 204800 / t_pool / 1e6, "oracle_pool_cores": workers,
                    "results_agree_with_oracle": bool(np.max(np.abs(p_gpu - p_ref) / p_ref) < 1e-12 and np.max(np.abs(q_gpu - q_ref) / q_ref) < 1e-12)}
    finally:
        pool.close(); pool.join()
    return out


# ---------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--streams", type=int, default=0, help="streams per GPU (default: 1024 / n_gpus = BASELINE config 5, strong scaling)")
    ap.add_argument("--weak", action="store_true", help="128 streams per GPU at every N (round-1 shard mode, weak scaling)")
    ap.add_argument("--n-iq", type=int, default=N_IQ_10S)
    ap.add_argument("--sub-batch", type=int, default=SUB_BATCH, help="streams per submitted batch")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-r-correct", action="store_true", help="skip the figure that also materialises r_correct")
    ap.add_argument("--no-oracle-check", action="store_true")
    ap.add_argument("--oracle-check", type=int, default=32, help="streams of the timed workload compared with the oracle (side leg)")
    ap.add_argument("--configs", default="auto", choices=["auto", "on", "off", "quick"], help="timings of BASELINE configs 1-4 (auto: on at N=1)")
    ap.add_argument("--groups", type=int, default=4, help="stream groups per batch inside the synchronous call")
    ap.add_argument("--pipeline", type=int, default=2, help="batches in flight through gsmcal_calibrate_batch_submit/_collect (1 = the synchronous call)")
    ap.add_argument("--submit-groups", type=int, default=1, help="stream groups inside each submitted batch (pipelined mode)")
    ap.add_argument("--persist-colsum", type=int, default=None)
    ap.add_argument("--no-hi-prio", action="store_true")
    ap.add_argument("--stages", action="store_true", help="also time the materialising per-stage kernels (raw2iq, FIR, resample, derotate)")
    ap.add_argument("--debug", action="append", default=[], metavar="KEY=VALUE", help="gsmcal_debug_set(KEY, VALUE) before the run (A/B of kernel paths, see include/gsmcal.h)")
    ap.add_argument("--ingest", type=int, default=0, metavar="D",
                    help="instead of the benchmark: D loopback rtl_tcp replay servers -> gsmcal.ingest -> calibrate (SURVEY 8(f) row 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result records of the last timed step (rank 0's streams) as DIR/<field>.npy, float64 and finite "
                         "(a non-finite value is stored as 0, with its kind in DIR/<field>_nonfinite.npy)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.weak and not args.streams:
        args.streams = 128
    if args.impl == "reference":
        return run_reference(args)
    if args.ingest:
        return run_ingest(args)

    import torch
    import torch.distributed as dist
    import gsmcal
    from gsmcal import synth
    from gsmcal._lib import StreamResult, lib

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    numa = numa_pin(local_rank)
    gsmcal.set_device(local_rank)
    if world > 1:
        # NCCL's kernels on a high-priority stream: at normal priority the 11 KB record gather would queue behind the 10^5 blocks of the
        # running fine search (kernels of different streams are dispatched in arrival order)
        try:
            opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), pg_options=opts)
        except Exception:      # noqa: BLE001
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    host_cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)

    D = args.streams if args.streams else max(1, TOTAL_STREAMS // world)
    n_iq = args.n_iq
    sub = max(1, min(args.sub_batch, D))
    n_sub = (D + sub - 1) // sub
    scaling = "weak" if args.weak else "strong"
    specs = [synth.random_spec(rank * D + d, n_iq) for d in range(D)]
    t_gen = time.perf_counter()
    raw = torch.empty((D, 2 * n_iq), dtype=torch.uint8, device=dev)
    for d, sp in enumerate(specs):
        synth.generate_stream(sp, dev, raw[d])
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t_gen
    coef = gsmcal.fir1(46, 200e3 / FS)
    tpl = gsmcal.gsm_SCH_training_sequence_gen(8)
    L = lib()
    L.gsmcal_debug_set(3, args.groups)
    L.gsmcal_debug_set(6, 0 if args.no_hi_prio else 1)
    if args.persist_colsum is not None:
        L.gsmcal_debug_set(7, args.persist_colsum)
    L.gsmcal_debug_set(8, args.submit_groups)
    for kv in args.debug:
        k_, _, v_ = kv.partition("=")
        L.gsmcal_debug_set(int(k_), int(v_))
    stream = torch.cuda.current_stream()
    rec_bytes = C.sizeof(StreamResult)
    gathered = torch.empty((world * sub * rec_bytes,), dtype=torch.uint8, device=dev) if world > 1 else None
    row_bytes = 2 * n_iq

    gathers = []                 # (work handle, source tensor) of the record gathers in flight

    def gather(records, in_flight=False):
        """the only exchange on the path: fixed-size per-stream result records over NCCL/NVLink.  in_flight (the submit/collect pipeline):
        asynchronous, because the caller's stream must not wait for it - the next batch's front is ordered behind that stream and has to
        start under the running burst kernels - and the handles are waited for by gather_wait() before the step's clock stops."""
        if world > 1:
            b = bytearray(bytes(records))
            b.extend(b"\0" * (sub * rec_bytes - len(b)))
            t = torch.frombuffer(b, dtype=torch.uint8).to(dev, non_blocking=True)
            if in_flight:
                gathers.append((dist.all_gather_into_tensor(gathered, t, async_op=True), t))
            else:
                dist.all_gather_into_tensor(gathered, t)

    def gather_wait():
        for wk, _t in gathers:
            wk.wait()
        gathers.clear()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    depth = max(1, min(4, args.pipeline))

    def sync_step(groups=None):
        """all D streams of this rank in ONE synchronous call"""
        res = gsmcal.calibrate_batch(None, CARRIER, tpl, coef, device_ptr=raw.data_ptr(), n_iq=n_iq, n_streams=D,
                                     cuda_stream=stream.cuda_stream, details=False)
        return res

    class Pipe:
        """sub-batches of `sub` streams through submit/collect, `depth` in flight (continuous-capture operation): the column sums
        and the latency-bound burst chain of batch i+1 run under the FP64 kernels of batch i.  Every batch is submitted AND
        collected (results on the host, records gathered) inside run()."""

        def __init__(self):
            self.pend = [None] * depth
            self.ctr = 0
            self.last = [None] * n_sub

        def _finish(self, slot):
            b, p = self.pend[slot]
            r = p.collect()
            self.pend[slot] = None
            gather(r, in_flight=True)
            self.last[b] = r

        def run(self, k):
            for _ in range(k):
                for b in range(n_sub):
                    if depth == 1:
                        d0 = b * sub
                        nd = min(sub, D - d0)
                        r = gsmcal.calibrate_batch(None, CARRIER, tpl, coef, device_ptr=raw.data_ptr() + d0 * row_bytes, n_iq=n_iq, n_streams=nd,
                                                   cuda_stream=stream.cuda_stream, details=False)
                        gather(r)
                        self.last[b] = r
                        continue
                    slot = self.ctr % depth
                    self.ctr += 1
                    if self.pend[slot] is not None:
                        self._finish(slot)
                    d0 = b * sub
                    nd = min(sub, D - d0)
                    self.pend[slot] = (b, gsmcal.calibrate_batch_submit(slot, raw.data_ptr() + d0 * row_bytes, n_iq, nd, CARRIER, tpl, coef,
                                                                        cuda_stream=stream.cuda_stream))
            for j in range(depth):                       # drain in submission order
                slot = (self.ctr + j) % depth
                if self.pend[slot] is not None:
                    self._finish(slot)
            gather_wait()                                # every rank holds every record before the clock stops
            return [r for part in self.last if part is not None for r in part]

    pipe = Pipe()
    sampler = ClockSampler(local_rank)
    sampler.start()
    res = pipe.run(args.warmup)
    barrier()
    gsmcal.launch_count(reset=True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.active.set()
    torch.cuda.profiler.start()          # ncu --profile-from-start off sees only the timed region
    ev0.record(stream)
    res = pipe.run(args.steps)           # returns after the last batch's results are on the host
    ev1.record(stream)
    barrier()
    torch.cuda.profiler.stop()
    sampler.active.clear()
    clocks = sampler.stop()
    launches = gsmcal.launch_count()
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, StreamResult)
    pipelined_phases = None
    if "13=1" in args.debug:                      # phase cycles of the last two batches of the timed run (the one before the last ran under the next front)
        cn = ["staging", "fir", "energies_k0", "chunk_sums", "prefix", "segment_starts", "diff_slide", "argmax", "certificate"]
        tn = ["cache_load", "interp_levels", "energy_k0", "horner_band", "totals_argmax", "derot_unit_phasors", "ratio_atan2", "gate_horner", "gate_sums"]
        pipelined_phases = {}
        for off_, which_ in ((150, "batch_before_last"), (50, "last_batch")):
            ent = {}
            for base_, label_, nm in ((0, "core8", cn), (16, "tone8_fine", tn), (32, "tone8_post", tn)):
                nb_ = max(1, int(L.gsmcal_debug_get(off_ + base_ + 15)))
                ent[label_] = {n_: round(int(L.gsmcal_debug_get(off_ + base_ + i_)) / nb_, 1) for i_, n_ in enumerate(nm)}
                ent[label_]["total"] = round(sum(ent[label_].values()), 1)
            steps_ = max(1, int(L.gsmcal_debug_get(off_ + 48 + 7)))
            ent["coarse_chain_per_step"] = {n_: round(int(L.gsmcal_debug_get(off_ + 48 + i_)) / steps_, 1) for i_, n_ in
                                            enumerate(["prefetch_wait", "fir_fast", "fir_slow", "decision_after_snr", "window_snr"])}
            ent["coarse_chain_per_step"]["steps_per_block"] = round(steps_ / max(1, int(L.gsmcal_debug_get(off_ + 48 + 6))), 1)
            pipelined_phases[which_] = ent
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_per_step = ms / args.steps
    total_iq = world * D * n_iq
    value = total_iq / (ms_per_step * 1e-3) / 1e6
    n_ok = sum(1 for r in res if outcome_of(r.n_coarse, r.n_fcch, r.n_pos_info, r.flags) == "calibrated" and math.isfinite(r.total_sampling_ppm))

    # ---- the same steps through ONE synchronous call per step (all D streams, 4 stream groups), outside the timed region ----
    sync_call = None
    if world == 1:
        try:
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            sync_step(); torch.cuda.synchronize()
            n_sync = max(2, min(args.steps, 5))
            s0.record(stream)
            for _ in range(n_sync):
                sync_step()
            s1.record(stream)
            torch.cuda.synchronize()
            ms_sync = s0.elapsed_time(s1) / n_sync
            sync_call = {"ms_per_step": ms_sync, "value": D * n_iq / (ms_sync * 1e-3) / 1e6, "unit": "MS/s",
                         "note": f"gsmcal_calibrate_batch, all {D} streams in one call, {args.groups} stream groups"}
        except Exception as ex:      # noqa: BLE001
            sync_call = {"error": repr(ex)}

    # ---- per-stage CUDA-event times: strictly sequential passes (1 stream group) over all D streams, outside the timed region ----
    stage_acc = {}
    L.gsmcal_debug_set(3, 1)
    n_prof = 2
    tiers = {"tier2": 0, "tier3": 0}
    for _ in range(n_prof):
        sync_step()
        for k, v in gsmcal.api.last_batch_stage_ms().items():
            stage_acc[k] = stage_acc.get(k, 0.0) + v
        tiers = {"tier2": int(L.gsmcal_debug_get(2)), "tier3": int(L.gsmcal_debug_get(1)),
                 "tier1_proven_after_passes": {str(p_): int(L.gsmcal_debug_get(10 + p_)) for p_ in range(1, 9)},
                 "tier1_left_open": int(L.gsmcal_debug_get(10))}
        if "13=1" in args.debug:                 # per-phase cycles of fine_core8_kernel (thread 0 of every block, clock64)
            names = ["staging", "fir", "energies_k0", "chunk_sums", "prefix", "segment_starts", "diff_slide", "argmax", "certificate"]
            blocks = max(1, int(L.gsmcal_debug_get(65)))
            tiers["core8_phase_cycles_per_block"] = {n_: int(L.gsmcal_debug_get(50 + i_)) / blocks for i_, n_ in enumerate(names)}
            tiers["core8_blocks"] = blocks
            tnames = ["cache_load", "interp_levels", "energy_k0", "horner_band", "totals_argmax", "derot_unit_phasors", "ratio_atan2", "gate_horner", "gate_sums"]
            for base_, label_ in ((66, "tone8_fine"), (82, "tone8_post")):
                tb = max(1, int(L.gsmcal_debug_get(base_ + 15)))
                tiers[label_ + "_phase_cycles_per_block"] = {n_: int(L.gsmcal_debug_get(base_ + i_)) / tb for i_, n_ in enumerate(tnames)}
    L.gsmcal_debug_set(3, args.groups)
    stage_ms = {k: v / n_prof for k, v in stage_acc.items()}

    # ---- rooflines -------------------------------------------------------------------------------------
    facts = profile_facts()
    fp64 = C.c_double(0.0)
    L.gsmcal_fp64_peak(C.byref(fp64), C.c_void_p(stream.cuda_stream))
    n_bursts = sum(max(r.n_coarse, 0) for r in res if r.n_coarse >= 5)
    n_tone1 = sum(max(r.n_fcch, 0) for r in res)
    hist = tiers.get("tier1_proven_after_passes", {})
    open_b = tiers.get("tier1_left_open", 0)
    n_pass_total = sum(int(p_) * n_ for p_, n_ in hist.items()) + open_b * int(L.gsmcal_debug_get(40) or 8)   # passes executed over all bursts
    if n_pass_total <= 0:
        n_pass_total = n_bursts
    fine_fma = n_bursts * FMA_PER_BURST["fine_fir"] + n_pass_total * FMA_PER_BURST["fine_pass"] + tiers["tier2"] * FMA_PER_BURST["fine_tier2"]
    stage_flop = {"fine_peak": 2.0 * fine_fma, "fine_tone": 2.0 * n_tone1 * FMA_PER_BURST["tone1"], "sch": 2.0 * n_tone1 * FMA_PER_BURST["sch"],
                  "post": 2.0 * n_tone1 * FMA_PER_BURST["tone2"]}
    stage_tflops = {k: stage_flop[k] / (stage_ms[k] * 1e-3) / 1e12 for k in stage_flop if stage_ms.get(k)}
    burst_stages = [k for k in ("fine_peak", "fine_tone", "sch", "post") if k in stage_ms]
    dominant = max(burst_stages, key=lambda k: stage_ms[k]) if burst_stages else None
    hbm_peak, peak_src = measured_peaks()
    colsum_gbs = (D * 2 * n_iq) / (stage_ms.get("colsum_u8", float("nan")) * 1e-3) / 1e9
    roofline = None
    if dominant:
        roofline = {"kernel": {"fine_peak": "fine_core8_kernel (+ fine_peak_band_kernel for the bursts it cannot certify)",
                               "fine_tone": "tone8_kernel", "sch": "sch_corr_kernel", "post": "tone8_kernel"}[dominant],
                    "stage": dominant, "bound": "fp64", "achieved": stage_tflops.get(dominant), "peak": fp64.value, "unit": "TFLOP/s",
                    "frac": (stage_tflops.get(dominant) / fp64.value) if fp64.value else None,
                    "peak_source": "measured here: gsmcal_fp64_peak (register-only DFMA kernel, CUDA events); MEASURED_PEAKS.json has no FP64 figure",
                    "algorithmic_flop_per_launch": stage_flop[dominant], "ms": stage_ms[dominant],
                    "counted": "FIR taps x samples, Horner DFT accumulations of every executed pass, band-kernel sums and slides, correlation MACs "
                               "(FMA_PER_BURST in bench.py, DESIGN.md section 4); tier-1 slides, certificates, index math, reductions are not counted",
                    "ncu_fp64_pipe_active_pct": facts.get("fp64_pipe_active_pct", {}).get(dominant),
                    "ncu_l1_data_pipe_pct": facts.get("l1_data_pipe_pct", {}).get(dominant),
                    "ncu_issue_active_pct": facts.get("issue_active_pct", {}).get(dominant),
                    "ncu_note": "the L1/shared-memory data pipe (complex128 operands: every 16-byte access of a warp is 4 wavefronts) is busier than the FP64 "
                                "pipe in every burst kernel; utilisation of all stages in ncu_all_stages",
                    "ncu_all_stages": {k: {"fp64_pipe_pct": facts.get("fp64_pipe_active_pct", {}).get(k), "l1_data_pipe_pct": facts.get("l1_data_pipe_pct", {}).get(k),
                                           "issue_active_pct": facts.get("issue_active_pct", {}).get(k)} for k in burst_stages},
                    "traffic": (int(facts["dram_bytes_per_launch"][dominant] * D / facts["streams_profiled"])
                                if facts.get("dram_bytes_per_launch", {}).get(dominant) and facts.get("streams_profiled") else None),
                    "traffic_source": (facts.get("source", "") + "; scaled by streams per launch") if facts else None,
                    "all_burst_stages_tflops": stage_tflops,
                    "all_burst_stages_frac": {k: v / fp64.value for k, v in stage_tflops.items()} if fp64.value else None}
    ratio = facts.get("colsum_dram_ratio")
    roofline_hbm = {"kernel": "colsum_u8_kernel", "bound": "hbm", "achieved": colsum_gbs, "peak": hbm_peak, "unit": "GB/s",
                    "frac": colsum_gbs / hbm_peak, "traffic": int(D * 2 * n_iq * ratio) if ratio else None,
                    "traffic_source": facts.get("colsum_source"), "peak_source": peak_src, "algorithmic_bytes_per_launch": D * 2 * n_iq,
                    "note": "the only whole-stream (HBM-proportional) pass of the fused pipeline, 2 B per IQ sample"}
    hbm_floor_ms = D * 2 * n_iq / (hbm_peak * 1e9) * 1e3
    whole_path = {"hbm_floor_ms_per_step": hbm_floor_ms, "frac_of_hbm_floor": hbm_floor_ms / ms_per_step if ms_per_step else None,
                  "note": "2 B per IQ sample read once is the HBM floor of the whole path on one rank; the step is bound by the burst kernels (FP64 + shared-memory pipes)"}

    # ---- the same pipeline when it also MATERIALISES r_correct (what the reference chain and the oracle produce on the way and hand
    #      to SCH_demod, gsm_sync_demod.m:120,145): gsmcal_calibrate_batch_r writes it in one fused pass, 2 B in + 16 B out per sample ----
    with_r = None
    if not args.no_r_correct:
        try:
            sub_r = max(1, min(D, 64))
            r_buf = torch.empty((sub_r, n_iq), dtype=torch.complex128, device=dev)

            def step_r():
                for c0 in range(0, D, sub_r):
                    nd = min(sub_r, D - c0)
                    rr = gsmcal.calibrate_batch(None, CARRIER, tpl, coef, device_ptr=raw.data_ptr() + c0 * row_bytes, n_iq=n_iq, n_streams=nd,
                                                cuda_stream=stream.cuda_stream, details=False, r_device_ptr=r_buf.data_ptr())
                    gather(rr)
            step_r()
            barrier()
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n_r = 2
            r0.record(stream)
            for _ in range(n_r):
                step_r()
            r1.record(stream)
            barrier()
            ms_r = r0.elapsed_time(r1) / n_r
            if world > 1:
                t = torch.tensor([ms_r], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms_r = float(t.item())
            gbs = D * n_iq * 18 / (ms_r * 1e-3) / 1e9
            with_r = {"value": total_iq / (ms_r * 1e-3) / 1e6, "unit": "MS/s", "ms_per_step": ms_r, "steps": n_r,
                      "algorithmic_bytes_per_iq": 18, "achieved_GBs_per_gpu": gbs, "frac_hbm": gbs / measured_peaks()[0],
                      "streams_per_call": sub_r, "r_correct_bytes_per_step": D * n_iq * 16,
                      "api": "gsmcal_calibrate_batch_r, r_correct written to a device buffer (complex128, reused per call)",
                      "note": "like-for-like with the CPU arm, which materialises the corrected stream; bounded by the fp64 47-tap FIR "
                              "(94 DFMA per sample), not by HBM"}
            del r_buf
            torch.cuda.empty_cache()
        except Exception as ex:      # noqa: BLE001
            with_r = {"error": repr(ex)}

    # ---- e2e: same call with host buffers -----------------------------------------------------------------
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(torch, dist, gsmcal, L, StreamResult, raw, D, n_iq, tpl, coef, stream, dev, world, rank, total_iq, rec_bytes, barrier, gather, sub, args, numa)

    # ---- optional: materialising per-stage kernels (the drop-in functions' device work) ------------------
    stages = None
    if args.stages and rank == 0:
        torch.cuda.profiler.start()
        stages = stage_rooflines(torch, gsmcal, L, raw, n_iq, coef, stream, hbm_peak)
        torch.cuda.profiler.stop()

    # ---- CPU baseline on this box's host cores (rank 0, N=1 only): the oracle on ONE stream of the workload ----
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        import gsmcal_oracle as oracle
        raw0 = raw[0].cpu().numpy()
        t0 = time.perf_counter()
        ref = oracle.calibrate_stream(raw0, CARRIER, tpl, coef)
        dt = time.perf_counter() - t0
        same = bool(res[0].n_pos_info == len(ref["pos_info"]) and abs(res[0].total_sampling_ppm - ref["total_sampling_ppm"]) < 1e-3
                    and abs(res[0].total_carrier_ppm - ref["total_carrier_ppm"]) < 1e-3)
        cpu_baseline = {"value": n_iq / dt / 1e6, "unit": "MS/s", "cores": 1, "kind": "port",
                        "sample": f"stream 0 of the workload ({n_iq} IQ, {n_iq / FS:.1f} s) through oracle/gsmcal_oracle.py, single thread, {dt:.1f} s",
                        "host_cores": host_cores, "gpu_result_matches_oracle": same}

    # ---- parity of the timed workload against the oracle (rank 0; every non-calibrating stream + evenly spaced others) ----
    agreement = None
    if rank == 0 and not args.no_oracle_check and args.oracle_check > 0:
        try:
            agreement = oracle_agreement(gsmcal, raw, res, n_iq, tpl, coef, args.oracle_check, host_cores)
        except Exception as ex:      # noqa: BLE001
            agreement = {"error": repr(ex)}

    configs = None
    want_cfg = args.configs in ("on", "quick") or (args.configs == "auto" and world == 1)
    if rank == 0 and want_cfg:
        del raw
        torch.cuda.empty_cache()
        try:
            configs = run_configs(gsmcal, synth, host_cores, quick=(args.configs == "quick"))
        except Exception as ex:      # noqa: BLE001
            configs = {"error": repr(ex)}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "MS/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f64",
                "data": "synthetic", "config": dict(workload_config(world, D, n_iq, scaling), batches_in_flight=depth, streams_per_submitted_batch=sub,
                               pipeline=("staggered batches (library default): the burst kernels of batch k+1 start when batch k is done; its column sums "
                                         "(one-warp TMA-ring kernel) and burst chain run on a high-priority stream under the burst kernels of batch k"
                                         if not any(k.startswith("16=0") for k in args.debug) else "two batches in lockstep (debug key 16=0)")),
                "clocks": clocks, "e2e": e2e, "with_r_correct": with_r, "gpu_launches": int(launches),
                "roofline": roofline, "roofline_hbm": roofline_hbm, "whole_path": whole_path, "fp64_peak_tflops_measured": fp64.value,
                "cpu_baseline": cpu_baseline, "stage_ms": stage_ms, "stage_ms_note": f"sequential pass over all {D} streams of rank 0 (one stream group)",
                "streams_fully_calibrated": f"{n_ok}/{D} on rank 0", "oracle_agreement": agreement, "synchronous_call": sync_call,
                "fine_search_allbin_fallback_bursts": tiers["tier3"], "fine_search_64bin_tier2_bursts": tiers["tier2"], "bursts_rank0": n_bursts,
                "pipelined_phase_cycles_per_block": pipelined_phases,
                "fine_search_tier1": {k: tiers.get(k) for k in ("tier1_proven_after_passes", "tier1_left_open", "core8_phase_cycles_per_block", "core8_blocks",
                                                                 "tone8_fine_phase_cycles_per_block", "tone8_post_phase_cycles_per_block") if k in tiers},
                "debug_keys": args.debug,
                "configs": configs, "reference_runtime_probe": probe_reference_runtimes(), "synthetic_generation_s": t_gen}
        if stages is not None:
            line["stage_rooflines"] = stages
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_e2e(torch, dist, gsmcal, L, StreamResult, raw, D, n_iq, tpl, coef, stream, dev, world, rank, total_iq, rec_bytes, barrier, gather, sub, args, numa):
    """The C-ABI call a user makes, fed from HOST memory: gsmcal_calibrate_batch(raw_mem = HOST); H2D of the step's captures and
    D2H of the result records inside the timed region.  Pinned memory is the headline; the same from pageable memory (what a
    MATLAB mxArray is) and a bare concurrent-memcpy bound are reported beside it."""
    row = 2 * n_iq
    need = D * row
    try:
        with open("/proc/meminfo") as f:
            avail = next(int(ln.split()[1]) * 1024 for ln in f if ln.startswith("MemAvailable"))
    except Exception:
        avail = 0
    chunk = D
    while chunk > 1 and (chunk * row * world * 1.5 > avail or chunk * row > 48e9):
        chunk = (chunk + 1) // 2
    n_chunks = (D + chunk - 1) // chunk
    host = torch.empty((chunk, row), dtype=torch.uint8, pin_memory=True)
    host.copy_(raw[:chunk])
    torch.cuda.synchronize()
    host_np = host.numpy()
    resbuf = (StreamResult * chunk)()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def step_host(arr_np):
        for c in range(n_chunks):
            nd = min(chunk, D - c * chunk)
            rc = L.gsmcal_calibrate_batch(arr_np.ctypes.data_as(C.c_void_p), 0, n_iq, nd, CARRIER, tpl.ctypes.data_as(C.c_void_p),
                                          coef.ctypes.data_as(C.c_void_p), len(coef), 8, 8, C.cast(resbuf, C.c_void_p),
                                          None, None, None, None, C.c_void_p(stream.cuda_stream))
            if rc != 0:
                raise RuntimeError(L.gsmcal_last_error().decode())
            for i in range(0, nd, sub):
                gather((StreamResult * min(sub, nd - i)).from_buffer(resbuf, i * rec_bytes))

    def timed(fn, steps):
        fn()
        barrier()
        t0 = time.perf_counter()
        ev0.record(stream)
        for _ in range(steps):
            fn()
        ev1.record(stream)
        barrier()
        wall = (time.perf_counter() - t0) * 1e3
        ems = max(ev0.elapsed_time(ev1), wall)          # host-side staging counts: the larger of device and wall time
        if world > 1:
            t = torch.tensor([ems], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ems = float(t.item())
        return ems / steps

    e_steps = max(2, min(args.steps, 3 if D >= 512 else 5))
    ms_pinned = timed(lambda: step_host(host_np), e_steps)
    e2e = {"value": total_iq / (ms_pinned * 1e-3) / 1e6, "unit": "MS/s", "h2d_bytes_per_step": need,
           "d2h_bytes_per_step": D * rec_bytes, "steps": e_steps, "ms_per_step": ms_pinned,
           "h2d_gbs_achieved": need / (ms_pinned * 1e-3) / 1e9,
           "api": "gsmcal_calibrate_batch(raw_mem=HOST) from pinned host memory" + ("" if n_chunks == 1 else f", {n_chunks} calls of {chunk} streams per step (one pinned buffer of {chunk} streams re-sent; host memory bound)"),
           "numa": numa}
    # bare bound: nothing but the concurrent pinned H2D copies of the same bytes on every rank
    try:
        dst = raw[:chunk]

        def bare():
            for c in range(n_chunks):
                nd = min(chunk, D - c * chunk)
                dst[:nd].copy_(host[:nd], non_blocking=True)
            torch.cuda.current_stream().synchronize()
        ms_bare = timed(bare, e_steps)
        e2e["h2d_gbs_bare"] = need / (ms_bare * 1e-3) / 1e9
        e2e["frac_of_bare_copy_bound"] = ms_bare / ms_pinned
        e2e["bound"] = ("host-to-device transfer: uint8 IQ is already the wire format; `h2d_gbs_bare` is what concurrent cudaMemcpyAsync from the same "
                        "pinned buffers reaches on this box at this N with no compute at all")
    except Exception as ex:      # noqa: BLE001
        e2e["h2d_bare_error"] = repr(ex)
    # pageable input: what gsm_calibrate_batch's MEX gateway hands over (an mxArray); the library stages it through its pinned ring
    try:
        pg_rows = min(chunk, 128)
        pageable = np.empty((pg_rows, row), dtype=np.uint8)
        pageable[:] = host_np[:pg_rows]

        def step_pg():
            rc = L.gsmcal_calibrate_batch(pageable.ctypes.data_as(C.c_void_p), 0, n_iq, pg_rows, CARRIER, tpl.ctypes.data_as(C.c_void_p),
                                          coef.ctypes.data_as(C.c_void_p), len(coef), 8, 8, C.cast(resbuf, C.c_void_p),
                                          None, None, None, None, C.c_void_p(stream.cuda_stream))
            if rc != 0:
                raise RuntimeError(L.gsmcal_last_error().decode())
        if world == 1:
            ms_pg = timed(step_pg, 3)
            e2e["pageable"] = {"value": pg_rows * n_iq / (ms_pg * 1e-3) / 1e6, "unit": "MS/s", "streams": pg_rows, "ms_per_call": ms_pg,
                               "h2d_gbs_achieved": pg_rows * row / (ms_pg * 1e-3) / 1e9,
                               "api": "gsmcal_calibrate_batch(raw_mem=HOST) from PAGEABLE host memory (numpy / mxArray)"}
    except Exception as ex:      # noqa: BLE001
        e2e["pageable"] = {"error": repr(ex)}
    del host
    return e2e


def stage_rooflines(torch, gsmcal, L, raw, n_iq, coef, stream, hbm_peak):
    """Times the whole-stream kernels behind the drop-in functions on device-resident buffers (CUDA events)."""
    cols = 8
    n = n_iq
    dev = raw.device
    a = torch.empty((cols, n, 2), dtype=torch.float64, device=dev)
    b = torch.empty((cols, n, 2), dtype=torch.float64, device=dev)
    cptr = coef.ctypes.data_as(C.c_void_p)
    out = {}
    spec = [("colsum_u8", 0, raw, a, 2), ("raw2iq_store", 1, raw, a, 18), ("fir47_c128", 2, a, b, 32), ("raw2iq_fir47_fused", 3, raw, b, 18),
            ("resample_interp1", 4, a, b, 32), ("derotate", 5, a, b, 32), ("raw2iq_fir47_decim64", 6, raw, b, 2.25)]
    for name, stage, src, dst, bytes_per_iq in spec:
        def run():
            rc = L.gsmcal_stage_launch(stage, C.c_void_p(src.data_ptr()), C.c_void_p(dst.data_ptr()), n, cols, cptr, len(coef), C.c_void_p(stream.cuda_stream))
            if rc != 0:
                raise RuntimeError(L.gsmcal_last_error().decode())
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 5
        e0.record(stream)
        for _ in range(reps):
            run()
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        gbs = cols * n * bytes_per_iq / (ms * 1e-3) / 1e9
        out[name] = {"ms": ms, "GS_per_s": cols * n / (ms * 1e-3) / 1e9, "algorithmic_bytes_per_iq": bytes_per_iq, "achieved_GBs": gbs, "frac_hbm": gbs / hbm_peak}
    return out


if __name__ == "__main__":
    main()
