"""Cold start of 64 receivers on one GPU: batched FFT acquisition over the streams, hand-off into the channels, tracking.

    python tools/coldstart_probe.py [--streams 64] [--seconds 10] [--reps 10]

1. Synthesises the streams on the device (gnssb200_synth, packed 2+2 bit): 8-12 GPS satellites per stream at 44-50 dB-Hz,
   Dopplers uniform in +-5 kHz, code phases uniform over the whole period, 50-bps data bits that change every second
   bit (the generator starts its bits at sample 0, not at a code epoch; bits that may change every 20 ms would put
   changes 19 or 21 dumps apart for code phases in mid-period, which the channel logic's pull-in -> tracking test
   counts as noise).
2. Times the C1 acquisition shape (32 PRNs, 41 bins of 500 Hz, 1 ms coherent) three ways, each with CUDA events and a
   host clock around a synchronise: one batched call over all streams, one single-record call per stream on the same
   CUDA stream, and batched calls over 1/8/16/32/64 streams.  G cells/s = records * 32 * 41 * 16000 / time.
3. Allocates every stream's channels from its acquisition result (gnssb200_rx_acq_allocate) and tracks the whole
   record: share of the present satellites allocated, share of allocated channels in CHANNEL_TRACKING (state 4) at the
   end, median / maximum time to a channel's first state-4 dump record.
4. The same records started the reference's way: simple_cold_allocate with the true PRNs, serial search, no warm start.
Prints one JSON object with the GPU name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

NS = 8192
CELLS_C1 = 32 * 41 * 16000


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clk = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def scenarios(S: int, seed: int):
    from gnss_sdr_ru_b200.scenarios import TrackScenario
    from gnss_sdr_ru_b200.synth import Sat

    rng = np.random.default_rng(seed)
    scs = []
    for s in range(S):
        prns = [int(p) for p in rng.choice(np.arange(1, 33), size=int(rng.integers(8, 13)), replace=False)]
        sats = [Sat(prn=p, cn0_dbhz=float(rng.uniform(44.0, 50.0)), doppler_hz=float(rng.uniform(-5000.0, 5000.0)),
                    code_phase_chips=float(rng.uniform(0.0, 1023.0)), carrier_phase_cycles=float(rng.random()),
                    data_bits=np.array([0, 0, 1, 1], dtype=np.uint8)) for p in prns]
        scs.append(TrackScenario(sats=sats, prns=[], n_freq=[]))
    return scs


def timed(fn, reps: int) -> dict:
    """median device time (CUDA events) and host time (perf_counter around a synchronise) of fn(), after one warm-up"""
    import torch

    fn()
    torch.cuda.synchronize()
    dev, host = [], []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        host.append((time.perf_counter() - t0) * 1e3)
        dev.append(e0.elapsed_time(e1))
    return {"device_ms": float(np.median(dev)), "host_ms": float(np.median(host))}


def track(eng, d_if, stride, nblk, cap):
    """runs the engine's receivers over the record; returns (dump records [S,12,cap], counts [S,12])"""
    import torch

    from gnss_sdr_ru_b200 import abi

    S = eng.n_streams
    eng.upload()
    d_dumps = torch.zeros((S, 12, cap, 48), dtype=torch.uint8, device="cuda")
    d_cnt = torch.zeros((S, 12), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    eng.run_device(d_if.data_ptr(), stride, nblk, NS, abi.FMT_PACKED2, d_dumps_ptr=d_dumps.data_ptr(), dump_cap=cap,
                   d_count_ptr=d_cnt.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    eng.download()
    return d_dumps.cpu().numpy().view(abi.DUMP_DTYPE).reshape(S, 12, cap), d_cnt.cpu().numpy(), wall


def outcome(eng, dumps, cnt, channels) -> dict:
    """channels[s] = list of (channel, prn) to score; ms to the first state-4 record (one record per 1-ms code period)"""
    n_ch = sum(len(c) for c in channels)
    locked, t4 = 0, []
    for s, chs in enumerate(channels):
        for ch, _ in chs:
            if eng.rx[s].chan[ch].state == 4:
                locked += 1
            st = dumps[s, ch, : cnt[s, ch]]["state"]
            hit = np.nonzero(st == 4)[0]
            if len(hit):
                t4.append(float(dumps[s, ch, hit[0]]["block"] + 1) * NS / 16e3)  # ms at the end of that block
    return {"channels": n_ch, "state4_at_end": locked / max(n_ch, 1), "reached_state4": len(t4),
            "ms_to_first_state4_median": float(np.median(t4)) if t4 else None,
            "ms_to_first_state4_max": float(np.max(t4)) if t4 else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=64)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--seed", type=int, default=6400)
    args = ap.parse_args()

    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine, Settings
    from gnss_sdr_ru_b200.lib import check, lib
    from gnss_sdr_ru_b200.receiver import TrackingEngine
    from gnss_sdr_ru_b200.scenarios import synth_sat_array

    if not torch.cuda.is_available():
        raise SystemExit("coldstart_probe: no CUDA device")
    out = {"tool": "coldstart_probe", **gpu_info(), "streams": args.streams, "seconds": args.seconds}
    S = args.streams
    nblk = int(round(args.seconds * 16e6 / NS))
    stride = NS * nblk // 2  # packed: two complex samples per byte
    scs = scenarios(S, args.seed)
    present = [sorted(sat.prn for sat in sc.sats) for sc in scs]
    eng = TrackingEngine(n_streams=S)
    d_if = torch.empty((S, stride), dtype=torch.uint8, device="cuda")
    arr, nsat = synth_sat_array(scs)
    check(lib().gnssb200_synth(eng.h, d_if.data_ptr(), stride, abi.FMT_PACKED2, S, NS * nblk, C.addressof(arr), nsat, args.seed, None),
          "gnssb200_synth")
    torch.cuda.synchronize()

    # ---- acquisition, C1 shape ----
    st = Settings.gps(acqSearchBand=20.0, acqCohIntegration=1)
    acq = AcquisitionEngine(handle=eng.h)
    n_acq = acq.samples_needed(st)
    nb = acq.num_bins(st)
    row_bytes = 32 * nb * 16
    d_rows = torch.zeros(S * row_bytes, dtype=torch.uint8, device="cuda")
    cs = torch.cuda.current_stream().cuda_stream
    base = d_if.data_ptr()

    def batched(R):
        return lambda: acq.search_batch_device(base, stride, R, n_acq, st, d_rows.data_ptr(), fmt=abi.FMT_PACKED2, stream=cs)

    def singles():
        for r in range(S):
            acq.search_device(base + r * stride, n_acq, st, d_rows.data_ptr() + r * row_bytes, fmt=abi.FMT_PACKED2, stream=cs)

    t_single = timed(singles, args.reps)
    t_batch = timed(batched(S), args.reps)
    kernel_ms = acq.last_kernel_ms()  # the library's own events around the kernels of the last batched call
    for t, R in ((t_single, S), (t_batch, S)):
        t["gcells_per_s"] = R * CELLS_C1 / (t["device_ms"] * 1e-3) / 1e9
    out["acq_c1"] = {"cells_per_record": CELLS_C1, f"single_calls_x{S}": t_single, f"batched_x{S}": t_batch,
                     "batched_kernels_ms": kernel_ms, "device_time_ratio_single_over_batched": t_single["device_ms"] / t_batch["device_ms"]}
    sweep = {}
    for R in (1, 8, 16, 32, 64):
        if R > S:
            continue
        t = timed(batched(R), args.reps)
        t["gcells_per_s"] = R * CELLS_C1 / (t["device_ms"] * 1e-3) / 1e9
        sweep[str(R)] = t
    out["acq_c1"]["batched_sweep"] = sweep

    # ---- hand-off + tracking ----
    results = acq.acquisition_batch(base, stride, S, n_acq, st, fmt=abi.FMT_PACKED2)
    alloc = [eng.acq_allocate(s, results[s], st) for s in range(S)]
    n_present = sum(len(p) for p in present)
    hits = sum(len(set(a) & set(p)) for a, p in zip(alloc, present))
    false = sum(len(set(a) - set(p)) for a, p in zip(alloc, present))
    cap = int(args.seconds * 1000) + 64
    dumps, cnt, wall = track(eng, d_if, stride, nblk, cap)
    out["acq_handoff"] = {"present": n_present, "allocated_present": hits, "allocated_fraction": hits / n_present,
                          "allocated_absent": false, "track_wall_s": wall,
                          **outcome(eng, dumps, cnt, [list(enumerate(a)) for a in alloc])}
    del dumps

    # ---- the reference's cold start on the same records: true PRNs, serial search from cell 0, bin 0 ----
    ref = TrackingEngine(n_streams=S)
    for s in range(S):
        ref.simple_cold_allocate(s, present[s] + [0] * (12 - len(present[s])))
    dumps, cnt, wall = track(ref, d_if, stride, nblk, cap)
    out["reference_cold_start"] = {"present": n_present, "track_wall_s": wall,
                                   **outcome(ref, dumps, cnt, [list(enumerate(p)) for p in present])}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
