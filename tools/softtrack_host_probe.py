"""Measures resumable float (Scilab) tracking of many receivers against the one-shot call.

1. Synthesises R records on the device (gnssb200_synth, 8 GLONASS or 8 GPS satellites each, the records of
   tools/softtrack_batch_probe.py) and copies them to pinned host memory.  Channels come from the true Doppler and code
   phase, msToProcess = the record length minus 8 periods.
2. Times (median of --reps after one warm-up; device-resident calls with CUDA events, the host call with a host clock
   around the synchronous call):
   (a) one gnssb200_softtrack_batch on the device-resident records;
   (b) gnssb200_softtrack_resume over device windows of 100 ms and 1 s (overlap two code periods), all windows queued
       on one stream;
   (c) gnssb200_softtrack_batch_host from the pinned records into pinned rows (the call alone, host clock) at the
       automatic window, a quarter of it and four times it;
   (d) one pinned host -> device copy of the same bytes.
3. Checks that (b) and (c) give rows and ms_done byte-identical to (a).
Prints one JSON object with the GPU name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from softtrack_batch_probe import channel, gpu_info, records  # noqa: E402

P = 16000  # samples per code period at 16 MHz (GLONASS and GPS)


def median_ms(fn, reps: int, device: bool) -> float:
    import torch

    fn()
    torch.cuda.synchronize()
    t = []
    for _ in range(reps):
        if device:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            t.append(e0.elapsed_time(e1))
        else:
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            t.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(t))


def run(system: str, fmt_name: str, R: int, seconds: float, reps: int, seed: int) -> dict:
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.lib import check, lib
    from gnss_sdr_ru_b200.scenarios import TrackScenario, synth_sat_array
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine, TrackSettings, _flat_channels

    L = lib()
    eng = SoftTrackingEngine()
    fmt = abi.FMT_PACKED2 if fmt_name == "packed" else abi.FMT_INT8_IQ
    n = int(seconds * 1000) * P
    ms = int(seconds * 1000) - 8
    row = n // 2 if fmt == abi.FMT_PACKED2 else 2 * n
    recs = records(system, R, seed)
    arr, nsat = synth_sat_array([TrackScenario(sats=s, prns=[], n_freq=[]) for s in recs])
    d = torch.empty((R, row), dtype=torch.uint8, device="cuda")
    check(L.gnssb200_synth(eng.h, d.data_ptr(), row, fmt, R, n, C.addressof(arr), nsat, seed, None), "gnssb200_synth")
    h = torch.empty((R, row), dtype=torch.uint8, pin_memory=True)
    h.copy_(d)
    chans = [[channel(s) for s in rec] for rec in recs]
    n_ch = sum(len(c) for c in chans)
    ts = TrackSettings(msToProcess=ms) if system == "glonass" else TrackSettings.gps(msToProcess=ms)
    cs = torch.cuda.current_stream().cuda_stream
    msamp = n_ch * ms * P / 1e6
    out = {"system": system, "fmt": fmt_name, "records": R, "channels": n_ch, "seconds": seconds, "record_bytes": row,
           "total_GB": R * row / 1e9}

    def rate(t):
        return {"ms": t, "ms_per_signal_s": t / seconds, "channel_Msamples_per_s": msamp / (t / 1e3)}

    # (a) one-shot
    d_out = torch.zeros((n_ch, ms, 13), dtype=torch.float64, device="cuda")
    d_done = torch.zeros(n_ch, dtype=torch.int32, device="cuda")

    def one_shot():
        eng.tracking_batch_device(d.data_ptr(), row, R, n, chans, ts, d_out.data_ptr(), d_done.data_ptr(), fmt=fmt, stream=cs)

    out["a_one_shot"] = rate(median_ms(one_shot, reps, True))
    ref_rows, ref_done = d_out.cpu().numpy(), d_done.cpu().numpy()
    ref = [(ref_rows[i, : ref_done[i]].tobytes(), int(ref_done[i])) for i in range(n_ch)]
    del d_out

    def same(rows, done) -> bool:
        return all(int(done[i]) == ref[i][1] and rows[i, : done[i]].tobytes() == ref[i][0] for i in range(n_ch))

    # (b) device windows
    states0 = bytes(eng.init_states(chans, ts, R))
    d_state = torch.empty(len(states0), dtype=torch.uint8, device="cuda")
    s_host = torch.frombuffer(bytearray(states0), dtype=torch.uint8)
    w_out = torch.zeros((n_ch, ms, 13), dtype=torch.float64, device="cuda")
    out["b_resume_device"] = {}
    for wms in (100, 1000):
        W = wms * P
        A = W - 2 * P

        def windows():
            d_state.copy_(s_host, non_blocking=False)
            first = 0
            while True:
                length = min(W, n - first)
                off = first // 2 if fmt == abi.FMT_PACKED2 else 2 * first
                eng.resume_device(d.data_ptr() + off, row, R, fmt, first, length, n, ts, d_state.data_ptr(), n_ch, w_out.data_ptr(),
                                  stream=cs)
                if first + W >= n:
                    break
                first += A

        t = median_ms(windows, reps, True)
        st = (abi.SoftTrackState * n_ch).from_buffer_copy(d_state.cpu().numpy().tobytes())
        r = rate(t)
        r["windows"] = -(-(n - W) // A) + 1 if n > W else 1
        r["identical"] = same(w_out.cpu().numpy(), np.array([s.ms_done for s in st]))
        out["b_resume_device"][f"{wms}ms"] = r
    del w_out, d
    torch.cuda.empty_cache()

    # (c) host records, rows into pinned host memory
    ch, rec = _flat_channels(chans, R)
    cfg = ts.to_c()
    h_out = torch.empty((n_ch, ms, 13), dtype=torch.float64, pin_memory=True)
    h_done = np.zeros(n_ch, dtype=np.int32)
    out["c_host_pinned"] = {}
    cap = 2 * ((512 << 20) // R) if fmt == abi.FMT_PACKED2 else ((512 << 20) // R) // 2
    auto_w = max(min(1 << 20, cap), 4 * P)  # the library's automatic window
    for name, W in (("auto", 0), ("auto/4", auto_w // 4), ("auto*4", auto_w * 4)):
        rc = []

        def host():
            rc.append(L.gnssb200_softtrack_batch_host(eng.h, C.byref(cfg), h.data_ptr(), row, R, fmt, n, ch, rec, n_ch,
                                                      h_out.data_ptr(), h_done.ctypes.data, W))

        r = rate(median_ms(host, reps, False))
        r["window_samples"] = W or auto_w
        r["return_values"] = sorted(set(rc))
        r["identical"] = same(h_out.numpy(), h_done)
        out["c_host_pinned"][name] = r
    del h_out

    # (d) the pinned copy of the same bytes
    dd = torch.empty((R, row), dtype=torch.uint8, device="cuda")
    t = median_ms(lambda: dd.copy_(h, non_blocking=True), reps, True)
    out["d_h2d_pinned"] = {"ms": t, "GB_per_s": R * row / 1e9 / (t / 1e3)}
    bound = max(out["a_one_shot"]["ms"], t)
    out["c_auto_over_max_kernel_copy"] = out["c_host_pinned"]["auto"]["ms"] / bound
    eng.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=64)
    ap.add_argument("--packed-seconds", type=float, default=10.0)
    ap.add_argument("--int8-seconds", type=float, default=2.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=8800)
    ap.add_argument("--systems", default="glonass,gps")
    args = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("softtrack_host_probe: no CUDA device")
    res = {"tool": "softtrack_host_probe", **gpu_info(), "sm_count": torch.cuda.get_device_properties(0).multi_processor_count,
           "runs": []}
    for system in args.systems.split(","):
        res["runs"].append(run(system, "packed", args.records, args.packed_seconds, args.reps, args.seed))
        if args.int8_seconds > 0:
            res["runs"].append(run(system, "int8", args.records, args.int8_seconds, args.reps, args.seed))
        print(json.dumps(res["runs"][-1]), file=sys.stderr, flush=True)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
