#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 GNSS baseband engine (and of the reference CPU path).

  python bench.py --gpus N --steps K --warmup W            our arm (one rank per GPU under torchrun)
  python bench.py --impl reference --gpus N --steps K ...   the reference's own C receiver on host cores
  python bench.py ... --dump-outputs DIR                    also writes rank 0's receiver state after the last timed step
                                                            (seeded inputs: two builds can be compared array for array)

Metric (BASELINE.json): tracking channel*Msamples/s = streams x 12 channels x complex samples / time,
closed loop (correlator + channel logic) included.  Workload: BASELINE config 5 -- 64 independent
synthetic IF streams x 12 channels x 10 s -- resident on EACH GPU (the largest single-GPU tracking
configuration; weak scaling: N GPUs track 64*N streams, streams never leave their GPU).  The way the
config shards itself over eight GPUs (8 streams per GPU) and config 2 (one stream) are reported beside
it under "tracking_other_shapes".  One step = one pass of the whole workload.
Acquisition cells/s for configs 1, 3 and 4 are measured outside the timed steps and reported under
"acq" in the same JSON line.

`value`  : inputs already resident in HBM, device-timed (CUDA events on the launching stream).
`e2e`    : the same pass through the C ABI call that takes HOST buffers
           (gnssb200_track_run_host: pinned host record -> H2D -> kernels -> D2H of the dump records).
`roofline`: HBM form, algorithmic bytes = 0.5 B (packed 2+2 bit) or 2 B (int8) per complex sample per
           stream, divided by the tracking kernel's launch duration; see DESIGN.md for why this path
           is instruction-issue bound long before it is HBM bound (`roofline_issue` is that form).
`cpu_baseline`: the reference C receiver (oracle/_ref, compiled from the reference's own sources) on
           one host core, on stream 0 of this rank's workload copied back from the GPU; its dump
           records are also compared bit for bit with the GPU's.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NS = 8192  # complex samples per block, OSG/osgnss_next_step.c:150
FS = 16_000_000


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--streams-per-gpu", type=int, default=64)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--fmt", default="packed2", choices=["packed2", "int8"])
    ap.add_argument("--no-acq", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the extra tracking shapes (C2 single stream, 64 streams on one GPU)")
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="length of the stream sample the CPU baseline processes")
    ap.add_argument("--ref-sample-seconds", type=float, default=1.0, help="per-stream sample of the reference arm")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the receivers' state after the last timed step as DIR/rx_<field>.npy (float64), to compare two builds")
    return ap.parse_args()


# --------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (NVML, same fields as the
    nvidia-smi line of B200_PROFILING.md: clocks.sm, clocks.max.sm, clocks_event_reasons.*)."""

    def __init__(self, gpu_index: int):
        import threading

        self.gpu = gpu_index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = threading.Thread(target=self._run, daemon=True)
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            # honour CUDA_VISIBLE_DEVICES-free torchrun launches: LOCAL_RANK == physical index on this box
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def _run(self):
        nv = self.nv
        bits = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8)),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40)),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20)),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)),
        }
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = int(get_reasons(self.h))
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.01)

    def start(self):
        if self.ok:
            self._thread.start()

    def stop(self):
        if self.ok:
            self._stop.set()
            self._thread.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic_per_sample(fmt: str):
    """DRAM bytes per complex stream-sample of the tracking kernel from the committed ncu capture."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if not os.path.exists(p):
        return None
    with open(p) as f:
        d = json.load(f)
    return d.get(f"track_dram_bytes_per_stream_sample_{fmt}")


def profile_constant(key: str):
    """A per-unit figure taken from a committed ncu capture (profiles/roofline_traffic.json)."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if not os.path.exists(p):
        return None
    with open(p) as f:
        return json.load(f).get(key)


def dump_rx(out_dir: str, rx) -> None:
    """Every field of the receivers' state (what gnssb200_download_rx returns to the caller) as out_dir/rx_<field>.npy
    in float64, leading axis = stream.  A 64-bit integer field gets a last axis of two, (high 32 bits, low 32 bits), so
    that every value stays exact."""
    os.makedirs(out_dir, exist_ok=True)
    a = np.ctypeslib.as_array(rx)

    def walk(arr, prefix):
        for name in arr.dtype.names:
            if name == "pad_":
                continue
            v = arr[name]
            if v.dtype.names:
                walk(v, f"{prefix}{name}_")
                continue
            if v.dtype.itemsize == 8 and v.dtype.kind in "iu":
                v = np.stack([v >> 32, v & 0xFFFFFFFF], axis=-1)
            np.save(os.path.join(out_dir, f"{prefix}{name}.npy"), v.astype(np.float64))

    walk(a, "rx_")


# --------------------------------------------------------------------------------------------------
def run_reference(args):
    """Reference arm: the reference's own C receiver (oracle/_ref) on all host cores, one process per
    stream, on a bounded per-stream sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from multiprocessing import get_context

    from oracle import oracle_api

    oracle_api.build()
    n_streams = args.streams_per_gpu * args.gpus
    cores = os.cpu_count() or 1
    workers = min(cores, n_streams)
    nblk = int(args.ref_sample_seconds * FS / NS)
    # input: stream records of the same scenarios as our arm (seeds 5000+s), generated with the NumPy generator
    # (gnss_sdr_ru_b200/synth.py) inside each worker -- nothing in this process tree loads libgnssb200.so or CUDA.
    ctx = get_context("fork")
    times = []
    with ctx.Pool(workers) as pool:  # records first, in parallel, handed back to this process ...
        for i, r in enumerate(pool.map(_ref_make_record, [(i, nblk) for i in range(workers)], chunksize=1)):
            _REF_RECORDS[i] = r
    with ctx.Pool(workers) as pool:  # ... so that the workers forked now all inherit every record
        for it in range(args.warmup + args.steps):
            res = pool.map(_ref_worker, [(i, nblk) for i in range(workers)], chunksize=1)
            dt = max(r for r in res)  # processing time of the slowest worker
            if it >= args.warmup:
                times.append(dt)
    t = sum(times) / len(times)
    value = workers * 12 * NS * nblk / t / 1e6
    line = {
        "impl": "reference", "metric": "tracking channel*Msamples/s", "value": value, "unit": "channel*Msamples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": f"C5: {args.streams_per_gpu} streams x 12 ch on each GPU, GPS L1 C/A closed-loop tracking",
                   "sample": f"{workers} streams x {args.ref_sample_seconds:g} s each (one process per stream)"},
        "cpu_baseline": {"value": value, "unit": "channel*Msamples/s", "cores": workers, "kind": "reference",
                         "sample": f"{workers} streams x 12 ch x {args.ref_sample_seconds:g} s, reference C receiver (gcc -O2), one process per stream"},
        "e2e": {"value": value, "unit": "channel*Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


_REF_RECORDS = {}  # per worker process: stream index -> (record, scenario)


def _ref_record(i, nblk):
    if i not in _REF_RECORDS:
        from gnss_sdr_ru_b200.scenarios import gps_tracking_scenario
        from gnss_sdr_ru_b200.synth import make_record

        sc = gps_tracking_scenario(5000 + i)
        _REF_RECORDS[i] = (make_record(sc.sats, NS * nblk, seed=5000 + i), sc)
    return _REF_RECORDS[i]


def _ref_make_record(job):
    return _ref_record(*job)


def _ref_worker(job):
    i, nblk = job
    rec, sc = _ref_record(i, nblk)  # generated here if the pool handed this stream to another worker than before
    from oracle import oracle_api

    ref = oracle_api.RefReceiver()
    ref.cold_allocate(sc.prns)
    for ch, (prn, n) in enumerate(zip(sc.prns, sc.n_freq)):
        if prn > 0:
            ref.warm_start(ch, n)
    t0 = time.perf_counter()
    ref.run(rec, NS, nblk)
    return time.perf_counter() - t0


# --------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.lib import check, lib
    from gnss_sdr_ru_b200.receiver import TrackingEngine
    from gnss_sdr_ru_b200.scenarios import apply_tracking_scenario, gps_tracking_scenario, synth_sat_array

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the engine has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    S = args.streams_per_gpu
    nblk = int(args.seconds * FS / NS)  # 19531 for 10 s
    fmt = abi.FMT_PACKED2 if args.fmt == "packed2" else abi.FMT_INT8_IQ
    bytes_per_sample = 0.5 if fmt == abi.FMT_PACKED2 else 2.0
    stream_bytes = int(NS * nblk * bytes_per_sample)
    L = lib()
    eng = TrackingEngine(n_streams=S, device=local)
    scs = [gps_tracking_scenario(5000 + rank * S + s) for s in range(S)]
    d_if = torch.empty((S, stream_bytes), dtype=torch.uint8, device=dev)
    arr, nsat = synth_sat_array(scs)
    check(L.gnssb200_synth(eng.h, d_if.data_ptr(), d_if.stride(0), fmt, S, NS * nblk, C.addressof(arr), nsat, 1234 + rank, None), "gnssb200_synth")

    initial_rx = []  # the receivers' start state, built once: every step starts from the same registers

    def reset_state():
        if not initial_rx:
            for s in range(S):
                L.gnssb200_rx_init(C.byref(eng.rx[s]), C.byref(eng.cfg))
                apply_tracking_scenario(eng, s, scs[s])
            initial_rx.append(bytes(eng.rx))
        else:
            C.memmove(eng.rx, initial_rx[0], len(initial_rx[0]))
        eng.upload()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    stream = torch.cuda.current_stream()
    kernel_ms = []

    def step():
        reset_state()
        eng.run_device(d_if.data_ptr(), d_if.stride(0), nblk, NS, fmt, stream=stream.cuda_stream)

    # ---- device-resident timing ----
    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = eng.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        step()
        stream.synchronize()
        kernel_ms.append(eng.last_kernel_ms())
    ev1.record(stream)
    barrier()
    clocks = sampler.stop()
    launches = eng.launch_count() - launches0
    t_ms = ev0.elapsed_time(ev1)
    t = torch.tensor([t_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t_ms_max = float(t.item())
    total_chan_samples = world * S * 12 * NS * nblk
    value = total_chan_samples * args.steps / (t_ms_max * 1e-3) / 1e6
    eng.download()
    states = [int(eng.rx[s].chan[ch].state) for s in range(S) for ch in range(12)]
    if args.dump_outputs and rank == 0:
        dump_rx(args.dump_outputs, eng.rx)

    # ---- end to end through the host-buffer C ABI call ----
    h_if = torch.empty((S, stream_bytes), dtype=torch.uint8).pin_memory()
    h_if.copy_(d_if)
    cap = int(args.seconds * 1000) + 64
    h_dumps = torch.empty((S, 12, cap, 48), dtype=torch.uint8).pin_memory()
    h_cnt = torch.zeros((S, 12), dtype=torch.int32).pin_memory()

    def e2e_step():
        reset_state()
        h_cnt.zero_()
        check(L.gnssb200_track_run_host(eng.h, h_if.data_ptr(), h_if.stride(0), fmt, NS, nblk, h_dumps.data_ptr(), cap, h_cnt.data_ptr()),
              "gnssb200_track_run_host")

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = total_chan_samples * args.steps / float(te.item()) / 1e6
    h2d = S * stream_bytes + S * C.sizeof(abi.Rx)
    d2h = S * 12 * cap * 48 + S * 12 * 4
    # the ceiling of that figure on this box: every rank copying the same pinned records at the same time and nothing
    # else (what the host's memory system and the PCIe links deliver to N GPUs at once)
    barrier()
    for _ in range(2):
        d_if.copy_(h_if, non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(3):
        d_if.copy_(h_if, non_blocking=True)
    torch.cuda.synchronize()
    tc = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tc, op=dist.ReduceOp.MAX)
    barrier()
    h2d_gbs = 3 * S * stream_bytes / float(tc.item()) / 1e9  # per GPU, at the pace of the slowest rank
    e2e_ceiling = total_chan_samples / (S * stream_bytes / (h2d_gbs * 1e9)) / 1e6

    # ---- roofline of the tracking kernel ----
    peak, peak_src = load_peaks()
    k_ms = sum(kernel_ms) / len(kernel_ms)
    alg_bytes = S * NS * nblk * bytes_per_sample
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9
    tr = measured_traffic_per_sample(args.fmt)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": (tr * S * NS * nblk) if tr else None, "peak_source": peak_src,
                "kernel": "track_ws_kernel", "kernel_ms": k_ms, "algorithmic_bytes_per_launch": alg_bytes,
                "note": "instruction-issue bound, not HBM bound (DESIGN.md 4.1); the issue form of the same launch is under roofline_issue"}
    # issue-slot form: warp-instructions the kernel executes per channel-sample (ncu smsp__inst_executed.sum of the
    # committed capture, profiles/roofline_traffic.json) x channel-samples / launch time, against 4 issue slots per
    # SM per clock at the SM clock sampled during the timed region
    wi = profile_constant("track_warp_inst_per_channel_sample_" + args.fmt)
    roofline_issue = None
    if wi:
        sm_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6
        ach = wi * S * 12 * NS * nblk / (k_ms * 1e-3)
        roofline_issue = {"bound": "issue", "achieved": ach / 1e12, "peak": 148 * 4 * sm_hz / 1e12, "unit": "T warp-inst/s",
                          "frac": ach / (148 * 4 * sm_hz), "warp_inst_per_channel_sample": wi,
                          "source": "ncu smsp__inst_executed.sum of the same launch shape (profiles/)"}
        # the same two figures inside `roofline`, the object the driver keeps
        roofline["issue_frac"] = roofline_issue["frac"]
        roofline["warp_inst_per_channel_sample"] = wi

    # ---- BASELINE config 5 as written: 64 streams in TOTAL, sharded over the ranks (strong scaling) ----
    strong = None
    if 64 % world == 0:
        S5 = 64 // world
        eng5 = TrackingEngine(n_streams=S5, device=local)
        scs5, d5 = scs[:S5], d_if[:S5]  # this rank's share: the first 64/N of the streams it already holds

        for s in range(S5):
            L.gnssb200_rx_init(C.byref(eng5.rx[s]), C.byref(eng5.cfg))
            apply_tracking_scenario(eng5, s, scs5[s])
        initial5 = bytes(eng5.rx)

        def step5():
            C.memmove(eng5.rx, initial5, len(initial5))
            eng5.upload()
            eng5.run_device(d5.data_ptr(), d5.stride(0), nblk, NS, fmt, stream=stream.cuda_stream)

        for _ in range(2):
            step5()
        barrier()
        e50, e51 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n5 = max(2, min(args.steps, 5))
        e50.record(stream)
        for _ in range(n5):
            step5()
        e51.record(stream)
        barrier()
        t5 = torch.tensor([e50.elapsed_time(e51)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t5, op=dist.ReduceOp.MAX)
        v5 = 64 * 12 * NS * nblk * n5 / (float(t5.item()) * 1e-3) / 1e6
        strong = {"streams_total": 64, "streams_per_gpu": S5, "value": v5, "unit": "channel*Msamples/s", "scaling": "strong",
                  "vs_weak_per_gpu": v5 / (value / world), "note": "vs_weak_per_gpu / n_gpus = strong-scaling efficiency"}
        eng5.close()

    # ---- two more tracking shapes, reported beside the headline (not part of the timed steps) ----
    also = None
    if not args.no_also:
        also = {}
        shapes = (("C2_single_stream_12ch_10s", 1, args.seconds, fmt), ("C5_shard_8_streams_per_gpu", 8, args.seconds, fmt),
                  ("256_streams_on_one_gpu", 256, min(args.seconds, 2.0), fmt),
                  # the reference's own file format (int8 I,Q, 2 B per sample; osgnss_next_step.c:172) instead of the packed wire format
                  ("C5_64_streams_int8_input", 64, min(args.seconds, 2.0), abi.FMT_INT8_IQ))
        for name, S2, secs, fmt2 in shapes:
            bps2 = 0.5 if fmt2 == abi.FMT_PACKED2 else 2.0
            nb2 = int(secs * FS / NS)
            eng2 = TrackingEngine(n_streams=S2, device=local)
            scs2 = [gps_tracking_scenario(7000 + rank * 64 + s) for s in range(S2)]
            sb2 = int(NS * nb2 * bps2)
            d2 = torch.empty((S2, sb2), dtype=torch.uint8, device=dev)
            arr2, nsat2 = synth_sat_array(scs2)
            check(L.gnssb200_synth(eng2.h, d2.data_ptr(), d2.stride(0), fmt2, S2, NS * nb2, C.addressof(arr2), nsat2, 99 + rank, None), "gnssb200_synth")
            best = None
            for it in range(3):
                for s in range(S2):
                    L.gnssb200_rx_init(C.byref(eng2.rx[s]), C.byref(eng2.cfg))
                    apply_tracking_scenario(eng2, s, scs2[s])
                eng2.upload()
                eng2.run_device(d2.data_ptr(), d2.stride(0), nb2, NS, fmt2, stream=stream.cuda_stream)
                stream.synchronize()
                ms = eng2.last_kernel_ms()
                best = ms if best is None or ms < best else best
            also[name] = {"streams": S2, "seconds": secs, "kernel_ms": best, "input_format": "packed2" if fmt2 == abi.FMT_PACKED2 else "int8",
                          "channel_Msamples_per_s": S2 * 12 * NS * nb2 / (best * 1e-3) / 1e6,
                          "hbm_frac": S2 * NS * nb2 * bps2 / (best * 1e-3) / 1e9 / load_peaks()[0]}
            eng2.close()
            del d2
        # GLONASS channels of the integer correlator (SURVEY 8f rank 4): 64 streams x 12 GLONASS satellites on distinct
        # frequency channels, closed loop; 15.7 samples per half chip -> the 16-slot segment loop of the same kernel
        from gnss_sdr_ru_b200.lib import default_cfg
        from gnss_sdr_ru_b200.scenarios import glonass_tracking_scenario

        secs_g = min(args.seconds, 2.0)
        nbg = int(secs_g * FS / NS)
        engg = TrackingEngine(n_streams=S, device=local, cfg=default_cfg(glonass_carrier_if=1.0e6))
        scg = [glonass_tracking_scenario(8000 + rank * S + s) for s in range(S)]
        dg = torch.empty((S, NS * nbg // 2), dtype=torch.uint8, device=dev)
        arrg, nsatg = synth_sat_array(scg)
        check(L.gnssb200_synth(engg.h, dg.data_ptr(), dg.stride(0), abi.FMT_PACKED2, S, NS * nbg, C.addressof(arrg), nsatg, 555 + rank, None), "gnssb200_synth")
        bestg = None
        for it in range(3):
            for s in range(S):
                L.gnssb200_rx_init(C.byref(engg.rx[s]), C.byref(engg.cfg))
                apply_tracking_scenario(engg, s, scg[s])
            engg.upload()
            engg.run_device(dg.data_ptr(), dg.stride(0), nbg, NS, abi.FMT_PACKED2, stream=stream.cuda_stream)
            stream.synchronize()
            ms = engg.last_kernel_ms()
            bestg = ms if bestg is None or ms < bestg else bestg
        engg.download()
        stg = [int(engg.rx[s].chan[ch].state) for s in range(S) for ch in range(12)]
        also["glonass_integer_tracking_64_streams"] = {"streams": S, "channels": 12 * S, "seconds": secs_g, "kernel_ms": bestg,
                                                       "channel_Msamples_per_s": S * 12 * NS * nbg / (bestg * 1e-3) / 1e6,
                                                       "channels_past_confirm_at_end": sum(1 for x in stg if x >= 3)}
        engg.close()
        del dg
        # C1 integer path (SURVEY 8d): GP2021-semantics serial search, detection threshold out of reach,
        # 500 Hz bins; one dump of one channel = one search cell (PRN x Doppler bin x half-chip delay)
        from gnss_sdr_ru_b200.lib import default_cfg

        secs = min(args.seconds, 3.0)
        nb3 = int(secs * FS / NS)
        eng3 = TrackingEngine(n_streams=S, device=local, cfg=default_cfg(acq_thresh=2**30, freq_bin_width=500.0))
        for s in range(S):
            eng3.simple_cold_allocate(s, [1 + (12 * s + c) % 32 for c in range(12)])
            for c in range(12):
                eng3.rx[s].chan[c].search_max_f = 20
        eng3.upload()
        cnt3 = torch.zeros((S, 12), dtype=torch.int32, device=dev)
        dmp3 = torch.empty((S, 12, int(secs * 1000) + 64, 48), dtype=torch.uint8, device=dev)
        eng3.run_device(d_if.data_ptr(), d_if.stride(0), nb3, NS, fmt, d_dumps_ptr=dmp3.data_ptr(), dump_cap=dmp3.shape[2],
                        d_count_ptr=cnt3.data_ptr(), stream=stream.cuda_stream)
        stream.synchronize()
        ms3 = eng3.last_kernel_ms()
        cells3 = int(cnt3.sum().item())
        also["C1_integer_serial_search"] = {"streams": S, "channels": 12 * S, "seconds": secs, "kernel_ms": ms3, "cells": cells3,
                                            "cells_per_s": cells3 / (ms3 * 1e-3),
                                            "note": "threshold out of reach, 500 Hz bins, search_max_f=20; reference C receiver: ~18e3 cells/s per core"}
        eng3.close()
        # drop-in layer: the reference's own call, Sim_GP2021_int(IF, 8192) with a host buffer, synchronous (one H2D, one
        # 12-CTA launch, one register-file read-back per 512 us of signal) -- what the unchanged C receiver gets
        try:
            from gnss_sdr_ru_b200.receiver import DropInCorrelator

            dc = DropInCorrelator()
            for c_, p_ in enumerate([27, 9, 3, 5, 7, 11, 13, 17, 19, 23, 29, 31]):
                dc.ch_cntl(c_, p_)
                dc.ch_carrier(c_, int(eng.cfg.gps_carrier_ref))
                dc.ch_code(c_, int(eng.cfg.gps_code_ref))
            one = np.ascontiguousarray((np.arange(2 * NS) % 4 * 2 - 3).astype(np.int8))
            for _ in range(50):
                dc.Sim_GP2021_int(one, NS)
            ncall = 2000
            t0 = time.perf_counter()
            for _ in range(ncall):
                dc.Sim_GP2021_int(one, NS)
            dtc = (time.perf_counter() - t0) / ncall
            also["dropin_Sim_GP2021_int_host_call"] = {"us_per_call": dtc * 1e6, "channel_Msamples_per_s": 12 * NS / dtc / 1e6,
                                                       "real_time_factor": 512e-6 / dtc,
                                                       "note": "synchronous per-block call of the reference's own entry point (12 channels); the reference C code needs ~435 us per call on one core"}
        except Exception as ex:
            also["dropin_Sim_GP2021_int_host_call"] = {"error": repr(ex)}
        # SURVEY 8f rank 1: floating-point (Scilab) tracking, 8 GLONASS channels x 2 s, FP64
        from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine, TrackSettings
        from gnss_sdr_ru_b200.scenarios import TrackScenario
        from gnss_sdr_ru_b200.synth import Sat

        fsats = [Sat(system="glonass", prn=k, cn0_dbhz=48.0, doppler_hz=400.0 * k, code_phase_chips=37.0 * (k + 8),
                     data_seed=50 + k, data_rate_hz=100.0) for k in (-7, -5, -3, -1, 0, 2, 4, 6)]
        fms = 2000
        fn = 16000 * (fms + 8)
        frec = torch.empty(2 * fn, dtype=torch.uint8, device=dev)
        farr, fns = synth_sat_array([TrackScenario(sats=fsats, prns=[], n_freq=[])])
        check(L.gnssb200_synth(eng.h, frec.data_ptr(), 2 * fn, abi.FMT_INT8_IQ, 1, fn, C.addressof(farr), fns, 77, None), "gnssb200_synth")
        fchan = [dict(FCH=s_.prn, acquiredFreq=1e6 + 562500.0 * s_.prn + s_.doppler_hz + 30.0,
                      codePhase=int(round((511.0 - s_.code_phase_chips % 511.0) * 16000.0 / 511.0)) % 16000 + 1) for s_ in fsats]
        fout = torch.zeros((len(fchan), fms, 13), dtype=torch.float64, device=dev)
        fdone = torch.zeros(len(fchan), dtype=torch.int32, device=dev)
        ste = SoftTrackingEngine(handle=eng.h)
        for it in range(2):
            ste.tracking_device(frec.data_ptr(), fn, fchan, TrackSettings(msToProcess=fms), fout.data_ptr(), fdone.data_ptr())
        fms_t = ste.last_kernel_ms()
        ip = fout[:, -200:, 1].abs().mean(dim=1).cpu().numpy()
        qp = fout[:, -200:, 4].abs().mean(dim=1).cpu().numpy()
        also["scilab_float_tracking_glonass"] = {"channels": len(fchan), "ms": fms, "kernel_ms": fms_t,
                                                 "channel_Msamples_per_s": len(fchan) * 16000.0 * fms / (fms_t * 1e-3) / 1e6,
                                                 "channels_locked": int((ip > 3 * qp).sum()), "dtype": "f64"}

    # ---- acquisition (configs 1, 3, 4), outside the timed steps ----
    acq = None
    if not args.no_acq:
        acq = bench_acquisition(eng, dev, rank, world, clocks, no_cpu=args.no_cpu)

    # ---- CPU baseline (rank 0): reference C receiver on stream 0, plus bit-exact check of the GPU dumps ----
    cpu = None
    parity = None
    if rank == 0 and not args.no_cpu:
        cpu, parity = cpu_baseline(args, d_if, fmt, scs, h_dumps, h_cnt, nblk)

    torch.cuda.synchronize()
    eng.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    line = {
        "metric": "tracking channel*Msamples/s", "value": value, "unit": "channel*Msamples/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_ms_max / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": f"C5: {S} streams x 12 ch x {args.seconds:g} s on each GPU, GPS L1 C/A closed-loop tracking "
                               f"(search/confirm/pull-in/track), 8192-sample blocks",
                   "input_format": args.fmt, "l2": "inputs larger than L2 (%.0f MB per GPU per step)" % (S * stream_bytes / 1e6),
                   "streams_per_gpu": S, "blocks_per_stream": nblk,
                   "channels_tracking_at_end": sum(1 for x in states if x == 4), "channels": len(states),
                   "c5_strong": strong},
        "e2e": {"value": e2e_value, "unit": "channel*Msamples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "h2d_GBs_per_gpu_all_ranks_copying": h2d_gbs, "copy_bound_ceiling": e2e_ceiling, "frac_of_ceiling": e2e_value / e2e_ceiling},
        "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "roofline_issue": roofline_issue, "cpu_baseline": cpu, "parity_vs_reference": parity,
        "acq": acq, "tracking_other_shapes": also,
    }
    if acq:  # compact copy inside `roofline` (the driver keeps that object): FP32 fraction and cells/s per acquisition config
        roofline["acq"] = {k[:2]: {"fp32_frac": round(v["fp32_frac"], 4), "Gcells_s": round(v["cells_per_s"] / 1e9, 2),
                                   "e2e_Gcells_s": round(v.get("e2e_cells_per_s", 0.0) / 1e9, 2)}
                           for k, v in acq.items() if k.startswith("C")}
    print(json.dumps(line))


def bench_acquisition(eng, dev, rank, world, clocks, no_cpu=False):
    """acq cells/s for BASELINE configs 1, 3, 4 on device-resident records.  With several ranks the
    (sv, bin) grid is sharded (row r -> rank r % world) and the row tables are all-gathered (NCCL)."""
    import torch
    import torch.distributed as dist

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine, Settings
    from gnss_sdr_ru_b200.lib import check, lib
    from gnss_sdr_ru_b200.scenarios import gps_acq_scenario, glonass_acq_scenario, gps_weak_acq_scenario, TrackScenario, synth_sat_array

    L = lib()
    ae = AcquisitionEngine(handle=eng.h)
    sm_mhz = (clocks.get("sm_mhz") or 1965.0)
    fp32_peak = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12  # TFLOP/s at the clock seen under load
    out = {}
    N = 16000
    # C1 reads the packed 2+2-bit GPS1A-sampler format (BASELINE config 1), C3 the int8 I,Q file of the Scilab receiver
    cases = [
        ("C1_gps_1ms_32prn_41bins", Settings.gps(acqSearchBand=20.0, acqCohIntegration=1), gps_acq_scenario(1001), 1001,
         dict(B=2, K=1, T=1), abi.FMT_PACKED2),
        ("C3_glonass_5ms_14fch_121bins", Settings.glonass(), glonass_acq_scenario(3003), 3003, dict(B=2, K=1, T=5), abi.FMT_INT8_IQ),
        ("C4_gps_10ms_x20_32prn_401bins", Settings.gps(acqSearchBand=20.0, acqCohIntegration=10, n_noncoh=20),
         gps_weak_acq_scenario(4004), 4004, dict(B=1, K=20, T=10), abi.FMT_INT8_IQ),
    ]
    # bounded CPU samples (about 5-15 s each on one core): which code entries (and, for config 4, which Doppler
    # bins: one PRN of it keeps the restatement busy for two minutes) the restatement processes
    cpu_sample = {"C1_gps_1ms_32prn_41bins": (list(range(1, 33)), None),
                  "C3_glonass_5ms_14fch_121bins": (list(range(-7, 7)), None),
                  "C4_gps_10ms_x20_32prn_401bins": ([21], list(range(292, 332)))} if not no_cpu else {}
    for name, st, sats, seed, fl, afmt in cases:
        n = ae.samples_needed(st)
        n4 = (n + 3) // 4 * 4
        rec_bytes = 2 * n4 if afmt == abi.FMT_INT8_IQ else n4 // 2
        rec = torch.empty(rec_bytes, dtype=torch.uint8, device=dev)
        arr, nsat = synth_sat_array([TrackScenario(sats=sats, prns=[], n_freq=[])])
        check(L.gnssb200_synth(eng.h, rec.data_ptr(), rec_bytes, afmt, 1, n4, C.addressof(arr), nsat, seed, None), "synth")
        nb = ae.num_bins(st)
        n_sv = len(st.acqSatelliteList)
        rows = torch.zeros(n_sv * nb * 16, dtype=torch.uint8, device=dev)
        reps = 3
        times = []
        for it in range(reps + 1):
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            ae.search_device(rec.data_ptr(), n4, st, rows.data_ptr(), fmt=afmt, part_index=rank, part_count=world)
            if world > 1:
                # merge partitions: all-gather the row tables, keep the rows each rank owns
                gathered = torch.empty(world * rows.numel(), dtype=torch.uint8, device=dev)
                dist.all_gather_into_tensor(gathered, rows)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if it > 0:
                times.append(dt)
        t = torch.tensor([min(times)], dtype=torch.float64, device=dev)
        if world > 1:
            from gnss_sdr_ru_b200.partition import merge_row_tables

            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            merged = merge_row_tables(gathered.cpu().numpy().view(abi.ACQ_ROW_DTYPE).reshape(world, n_sv * nb))
        else:
            merged = rows.cpu().numpy().view(abi.ACQ_ROW_DTYPE)
        res, amb = ae.finalize(st, merged)
        found = sorted(int(r.sv) for r in res if r.sv != 0 or (st.system == "glonass" and r.peakMetric > st.acqThreshold))
        cells = n_sv * nb * N
        G = n_sv * nb
        n_base = G if st.system == "glonass" else nb  # SURVEY 8d: C3 counts one forward spectrum per (FCH, bin)
        flops = fl["B"] * fl["K"] * (n_base * (8 * fl["T"] * N + 5 * N * np.log2(N)) + G * (6 * N + 5 * N * np.log2(N) + 3 * N))
        tt = float(t.item())
        # end to end through the C ABI call that takes a HOST record: H2D of the record, search, row table back, peak logic
        e2e_cells = None
        if rank == 0:
            from gnss_sdr_ru_b200.synth import unpack2

            host_rec = rec.cpu().numpy()
            pinned = torch.from_numpy(host_rec).pin_memory().numpy()
            ae.acquisition(pinned, st, fmt=afmt)
            te = []
            for _ in range(3):
                t0 = time.perf_counter()
                r_host = ae.acquisition(pinned, st, fmt=afmt)
                te.append(time.perf_counter() - t0)
            e2e_cells = cells / min(te)
        cpu_acq = None
        if rank == 0 and cpu_sample.get(name):
            # CPU side (SURVEY 8d): the NumPy float64 restatement of acquisition.sci (numpy.fft = pocketfft, one
            # thread) on a bounded sample of the same record -- a subset of the PRN / frequency-channel list (and of
            # the Doppler bins for config 4) -- which doubles as a full-size parity check of those entries
            from oracle import pcps_oracle

            sub, bins = cpu_sample[name]
            host = host_rec.view(np.int8)[: 2 * n] if afmt == abi.FMT_INT8_IQ else unpack2(host_rec)[: 2 * n]
            kw = dict(acqSearchBand=st.acqSearchBand, acqCohIntegration=st.acqCohIntegration, svList=list(sub), n_noncoh=st.n_noncoh)
            ost = pcps_oracle.AcqSettings.glonass(**kw) if st.system == "glonass" else pcps_oracle.AcqSettings.gps(**kw)
            by_sv = {int(sv): i for i, sv in enumerate(st.acqSatelliteList)}
            x = pcps_oracle.to_complex(host)
            t0 = time.perf_counter()
            if bins is None:
                ora = pcps_oracle.acquisition(x, ost)
                dtc = time.perf_counter() - t0
                same = all(int(res[by_sv[int(sv)]].bin) == o["bin"] and int(res[by_sv[int(sv)]].codePhaseRaw) == o["codePhaseRaw"]
                           and abs(res[by_sv[int(sv)]].peakMetric - o["peakMetric"]) <= 1e-4 * o["peakMetric"] for sv, o in zip(sub, ora))
                ccells = len(sub) * nb * N
                what = f"{len(sub)} of {n_sv} code entries, all {nb} bins"
            else:  # rows of the grid: maximum within 1e-4 and its code phase exact, row by row
                same = True
                for sv in sub:
                    orow, _ = pcps_oracle.acquisition_rows(x, ost, sv, bins=bins)
                    for b1 in bins:
                        g = merged[by_sv[int(sv)] * nb + b1 - 1]
                        same = same and abs(float(g["peak"]) - orow[b1][0]) <= 1e-4 * orow[b1][0] and int(g["code_phase"]) == orow[b1][1]
                dtc = time.perf_counter() - t0
                ccells = len(sub) * len(bins) * N
                what = f"{len(sub)} of {n_sv} code entries, {len(bins)} of {nb} bins (around the satellite's Doppler)"
            cpu_acq = {"cells_per_s": ccells / dtc, "seconds": dtc, "cores": 1, "kind": "port",
                       "sample": what + ", NumPy float64 restatement of acquisition.sci (pocketfft)",
                       "argmax_exact_and_metric_1e-4": bool(same)}
        out[name] = {"cells": cells, "cells_per_s": cells / tt, "ms": tt * 1e3, "kernel_ms_rank0": ae.last_kernel_ms(), "cpu_baseline": cpu_acq,
                     "e2e_cells_per_s": e2e_cells, "input_format": "packed2" if afmt == abi.FMT_PACKED2 else "int8",
                     "algorithmic_gflop": flops / 1e9, "fp32_tflops_achieved": flops / tt / 1e12,
                     "fp32_peak_tflops": fp32_peak * world, "fp32_frac": flops / tt / 1e12 / (fp32_peak * world),
                     "detected": found, "n_present": len(sats)}
    # ---- GPS-SDR fixed-point weak acquisition (SURVEY 8f rank 2): 32 satellites, +-10 kHz, 310 ms at 2.048 Msps ----
    if rank == 0:
        try:
            out["GPSSDR_weak_32sv_pm10kHz"] = bench_gpssdr(eng, no_cpu)
        except Exception as ex:  # never lose the headline over an extra
            out["GPSSDR_weak_32sv_pm10kHz"] = {"error": repr(ex)}
    return out


def bench_gpssdr(eng, no_cpu):
    from gnss_sdr_ru_b200 import gpssdr_codes
    from gnss_sdr_ru_b200.gpssdr_acq import Acquisition

    rng = np.random.default_rng(7007)
    chips = gpssdr_codes.prn_gen()
    n = 310 * 2048
    t = np.arange(n) / 2048000.0
    x = 8.0 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    present = [(2, 1.0, 3310.0, 400), (9, 0.5, -7420.0, 1500), (20, 0.3, 880.0, 90), (27, 0.25, -1950.0, 1977)]
    for sv, amp, dopp, off in present:
        ci = (np.floor((np.arange(n) + off) * 1023.0 / 2048.0)).astype(np.int64) % 1023
        x += amp * chips[ci, sv] * np.exp(2j * np.pi * (38400.0 + dopp) * t)
    rec = np.empty((n, 2), dtype=np.int16)
    rec[:, 0], rec[:, 1] = np.round(x.real), np.round(x.imag)
    acq = Acquisition(handle=eng.h)
    svs = list(range(32))
    acq.doAcqWeak(rec, svs, -10000, 10000)  # warm-up
    best = None
    for _ in range(3):
        t0 = time.perf_counter()
        res = acq.doAcqWeak(rec, svs, -10000, 10000)
        dt = time.perf_counter() - t0
        best = dt if best is None or dt < best else best
    cells = 32 * 20 * 4 * 10 * 2048  # satellites x kHz bins x 250 Hz offsets x 25 Hz DFT rows x code phases
    r = {"cells": cells, "cells_per_s": cells / best, "ms": best * 1e3, "call": "host buffers in, results out (H2D of the record and the code table included)",
         "dtype": "int16/int32 fixed point", "strongest": sorted(res, key=lambda d: -d["magnitude"])[0]["sv"]}
    if not no_cpu:
        from oracle import gpssdr_oracle_api as G

        o = G.GpsSdrAcquisition()
        t0 = time.perf_counter()
        o.doPrepIF(2, rec)
        w = o.doAcqWeak(gpssdr_codes.fft_codes()[2], -10000, 10000)
        dtc = time.perf_counter() - t0
        o.close()
        g = res[2]
        r["cpu_baseline"] = {"cells_per_s": (cells / 32) / dtc, "seconds": dtc, "cores": 1, "kind": "port",
                             "sample": "1 of 32 satellites, restatement of doPrepIF + doAcqWeak in the reference's portable arithmetic (gcc -O2)",
                             "bit_exact": bool((g["code_phase"], g["doppler"], g["magnitude"]) == (w["code_phase"], w["doppler"], w["magnitude"]))}
    return r


def _cpu_stream_worker(job):
    """One stream through the reference C receiver (oracle/_ref) or, where that is absent, the C restatement."""
    path, prns, n_freq, nb, cap = job
    from oracle import oracle_api

    rec = np.load(path, mmap_mode="r")
    if oracle_api.have_ref():
        ref = oracle_api.RefReceiver()
        ref.cold_allocate(prns)
        for ch, (prn, n) in enumerate(zip(prns, n_freq)):
            if prn > 0:
                ref.warm_start(ch, n)
        t0 = time.perf_counter()
        _, dumps, cnt = ref.run(rec, NS, nb, dump_cap=cap)
        return time.perf_counter() - t0, dumps, cnt
    o = oracle_api.Oracle()
    o.cold_allocate(prns)
    for ch, (prn, n) in enumerate(zip(prns, n_freq)):
        if prn > 0:
            k = o.rx.chan[ch]
            k.n_freq = n
            k.del_freq = -2 * n if n > 0 else 1 - 2 * n
            k.carrier_freq = o.cfg.gps_carrier_ref + o.cfg.d_freq * n
            o.ch_carrier(ch, k.carrier_freq)
    t0 = time.perf_counter()
    _, dumps, cnt = o.run(rec, NS, nb, dump_cap=cap)
    return time.perf_counter() - t0, dumps, cnt


def cpu_baseline(args, d_if, fmt, scs, h_dumps, h_cnt, nblk):
    """The reference on host cores, one process per stream, on stream 0 and three more of this rank's streams picked at
    random (seeded); every dump record of those streams is compared with what the end-to-end GPU pass returned."""
    import shutil
    from multiprocessing import get_context

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.synth import unpack2
    from oracle import oracle_api

    oracle_api.build()
    nb = min(nblk, int(args.cpu_seconds * FS / NS))
    S = d_if.shape[0]
    rng = np.random.default_rng(20261018)
    picks = [0] + sorted(int(x) for x in rng.choice(np.arange(1, S), size=min(3, S - 1), replace=False)) if S > 1 else [0]
    cap = h_dumps.shape[2]
    kind = "reference" if oracle_api.have_ref() else "port"
    tmp = tempfile.mkdtemp(prefix="gnssb200_cpu_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        jobs = []
        for s in picks:
            raw = d_if[s].cpu().numpy()
            rec = unpack2(raw[: NS * nb // 2]) if fmt == abi.FMT_PACKED2 else raw[: 2 * NS * nb].view(np.int8)
            path = os.path.join(tmp, f"s{s}.npy")
            np.save(path, rec)
            jobs.append((path, list(scs[s].prns), list(scs[s].n_freq), nb, cap))
        with get_context("spawn").Pool(len(jobs)) as pool:
            res = pool.map(_cpu_stream_worker, jobs, chunksize=1)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    dt = max(r[0] for r in res)
    value = len(picks) * 12 * NS * nb / dt / 1e6
    ok, compared = True, 0
    for s, (_, dumps, cnt) in zip(picks, res):
        g = h_dumps[s].numpy().view(abi.DUMP_DTYPE).reshape(12, cap)
        gc = h_cnt[s].numpy()
        for ch in range(12):
            a = g[ch, : gc[ch]]
            a = a[a["block"] < nb]
            b = dumps[ch, : cnt[ch]]
            compared += len(b)
            if len(a) != len(b) or not np.array_equal(a, b):
                ok = False
    cpu = {"value": value, "unit": "channel*Msamples/s", "cores": len(picks), "kind": kind,
           "sample": f"streams {picks} of rank 0: {nb * NS / FS:.2f} s each, one process per stream, gcc -O2",
           "per_core": value / len(picks),
           # parity of the GPU pass against this run, in the object the driver keeps
           "parity_bit_exact": bool(ok), "records_compared": int(compared), "streams_compared": picks}
    parity = {"bit_exact": bool(ok), "dump_records_compared": int(compared), "against": kind, "streams": picks}
    return cpu, parity


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
