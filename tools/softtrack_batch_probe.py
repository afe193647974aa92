"""Measures the float (Scilab) tracking of many receivers: gnssb200_softtrack_batch at each kernel width against one
gnssb200_softtrack call per record.

1. Synthesises R records on the device (gnssb200_synth), once packed 2+2 bit and once int8 with the same seed, so both
   hold the same samples: 8 GLONASS satellites per record (distinct frequency channels, 46-50 dB-Hz, Dopplers in
   +-4 kHz, code phases over the whole period), and the same with 8 GPS satellites.
2. Channels come from the true Doppler (+30 Hz) and code phase, as preRun would list them; msToProcess = --ms.
3. Times, with CUDA events around the calls (median of --reps after one warm-up): one batched call on the packed
   records at 512, 256 and 128 threads per channel and at the automatic width, and R single-record calls on the int8
   records on the same stream.  channel*Msamples/s = channels * ms * 16000 / 1e6 / seconds.
4. Checks that every batched output is byte-identical to the single calls' (the width does not change results).
Prints one JSON object with the GPU name and power limit read in the same run.  --records-sweep adds the batched
widths for smaller R, where the channels fit one per SM.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clk = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def timed_ms(fn, reps: int) -> float:
    """median device time of fn() in ms (CUDA events on the current stream), after one warm-up"""
    import torch

    fn()
    torch.cuda.synchronize()
    t = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        t.append(e0.elapsed_time(e1))
    return float(np.median(t))


def records(system: str, R: int, seed: int):
    from gnss_sdr_ru_b200.synth import Sat

    rng = np.random.default_rng(seed)
    recs = []
    for _ in range(R):
        if system == "glonass":
            ks = rng.choice(np.arange(-7, 7), size=8, replace=False)
            recs.append([Sat(system="glonass", prn=int(k), cn0_dbhz=float(rng.uniform(46.0, 50.0)), doppler_hz=float(rng.uniform(-4000, 4000)),
                             code_phase_chips=float(rng.uniform(0, 511)), data_seed=int(rng.integers(1, 1 << 30)), data_rate_hz=100.0)
                         for k in ks])
        else:
            ps = rng.choice(np.arange(1, 33), size=8, replace=False)
            recs.append([Sat(system="gps", prn=int(p), cn0_dbhz=float(rng.uniform(46.0, 50.0)), doppler_hz=float(rng.uniform(-4000, 4000)),
                             code_phase_chips=float(rng.uniform(0, 1023)), data_seed=int(rng.integers(1, 1 << 30)))
                         for p in ps])
    return recs


def channel(sat) -> dict:
    if sat.system == "glonass":
        f, L, bias = 1e6 + 562500.0 * sat.prn + sat.doppler_hz, 511.0, 30.0
    else:
        f, L, bias = 2.42e6 + sat.doppler_hz, 1023.0, 40.0
    cp = int(round((L - sat.code_phase_chips % L) * 16000.0 / L)) % 16000 + 1
    return dict(FCH=sat.prn, acquiredFreq=f + bias, codePhase=cp)


def run(system: str, R: int, ms: int, reps: int, seed: int, singles: bool) -> dict:
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.lib import check, lib
    from gnss_sdr_ru_b200.scenarios import TrackScenario, synth_sat_array
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine, TrackSettings

    L = lib()
    eng = SoftTrackingEngine()
    n = 16000 * (ms + 8)
    recs = records(system, R, seed)
    arr, nsat = synth_sat_array([TrackScenario(sats=s, prns=[], n_freq=[]) for s in recs])
    dp = torch.empty((R, n // 2), dtype=torch.uint8, device="cuda")
    check(L.gnssb200_synth(eng.h, dp.data_ptr(), n // 2, abi.FMT_PACKED2, R, n, C.addressof(arr), nsat, seed, None), "synth")
    chans = [[channel(s) for s in rec] for rec in recs]
    n_ch = sum(len(c) for c in chans)
    ts = TrackSettings(msToProcess=ms) if system == "glonass" else TrackSettings.gps(msToProcess=ms)
    d_out = torch.zeros((n_ch, ms, 13), dtype=torch.float64, device="cuda")
    d_done = torch.zeros(n_ch, dtype=torch.int32, device="cuda")
    cs = torch.cuda.current_stream().cuda_stream
    msamp = n_ch * ms * 16000 / 1e6
    out = {"system": system, "records": R, "channels": n_ch, "ms": ms, "batch_packed": {}}
    results = {}
    for nt in (512, 256, 128, 0):
        eng.set_width(nt)

        def batch():
            eng.tracking_batch_device(dp.data_ptr(), n // 2, R, n, chans, ts, d_out.data_ptr(), d_done.data_ptr(),
                                      fmt=abi.FMT_PACKED2, stream=cs)

        t = timed_ms(batch, reps)
        out["batch_packed"][str(nt or "auto")] = {"ms": t, "channel_Msamples_per_s": msamp / (t / 1e3)}
        results[nt] = (d_out.cpu().numpy().tobytes(), d_done.cpu().numpy().tobytes())
    eng.set_width(0)
    out["widths_identical"] = all(results[nt] == results[512] for nt in results)
    out["periods_done_min"] = int(np.frombuffer(results[512][1], dtype=np.int32).min())
    if singles:
        d8 = torch.empty((R, 2 * n), dtype=torch.uint8, device="cuda")
        check(L.gnssb200_synth(eng.h, d8.data_ptr(), 2 * n, abi.FMT_INT8_IQ, R, n, C.addressof(arr), nsat, seed, None), "synth")
        s_out = torch.zeros((n_ch, ms, 13), dtype=torch.float64, device="cuda")
        s_done = torch.zeros(n_ch, dtype=torch.int32, device="cuda")
        offs = np.cumsum([0] + [len(c) for c in chans])

        def singles_fn():
            for r in range(R):
                eng.tracking_device(d8[r].data_ptr(), n, chans[r], ts, s_out[offs[r]].data_ptr(), s_done[offs[r]:].data_ptr(), stream=cs)

        t = timed_ms(singles_fn, max(2, reps // 2))
        out["single_calls_int8"] = {"ms": t, "channel_Msamples_per_s": msamp / (t / 1e3)}
        out["single_identical_to_batch"] = (s_out.cpu().numpy().tobytes(), s_done.cpu().numpy().tobytes()) == results[512]
        best = min(out["batch_packed"][k]["ms"] for k in ("512", "256", "128"))
        out["batch_speedup_over_singles"] = t / best
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=64)
    ap.add_argument("--ms", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=8800)
    ap.add_argument("--records-sweep", default="8,18,19,32", help="smaller R timed for the batched widths only ('' = none)")
    args = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("softtrack_batch_probe: no CUDA device")
    res = {"tool": "softtrack_batch_probe", **gpu_info(), "sm_count": torch.cuda.get_device_properties(0).multi_processor_count,
           "runs": []}
    for system in ("glonass", "gps"):
        res["runs"].append(run(system, args.records, args.ms, args.reps, args.seed, singles=True))
    for R in [int(x) for x in args.records_sweep.split(",") if x]:
        res["runs"].append(run("glonass", R, args.ms, args.reps, args.seed + R, singles=False))
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
