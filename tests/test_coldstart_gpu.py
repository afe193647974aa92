"""Cold start of several receivers: batched FFT acquisition over the streams, hand-off of each stream's results into its
channels (gnssb200_rx_acq_allocate), closed-loop tracking on the same device buffer.

The satellites' code phases are uniform over the whole period (the tracking scenarios instead place them where the
serial search meets them early) and no channel is warm-started: what the channels know comes from the acquisition.
Two streams are compared bit exact with the oracle started from the same allocated state; all of them must find,
confirm and track every satellite that is present.
"""
import ctypes as C

import numpy as np
import pytest

from gnss_sdr_ru_b200 import abi

pytestmark = pytest.mark.gpu
NS = 8192
NBLK = 5860  # 3.0 s
CAP = 3100   # dump records per channel: one per ms
_CFG_OVER = {False: {}, True: dict(glonass_carrier_if=1.0e6)}  # oracle configuration of a GPS / GLONASS run
# 50-bps data bits that change every second bit.  The generator starts its bits at sample 0, not at a code epoch as a
# satellite does, so with code phases spread over the whole period a bit edge can fall in the middle of a 1-ms dump,
# whose prompt sign is then noise: two changes one bit apart register 19 or 21 dumps apart, and the channel logic's
# pull-in -> tracking test (31 prompt sign changes each more than 19 dumps after the last, osgpsisr.c:602-655) starts
# counting again.  Changes two bits apart register 39-41 dumps apart whatever the code phase.
BITS = np.array([0, 0, 1, 1], dtype=np.uint8)


def _gps_streams(rng, S):
    from gnss_sdr_ru_b200.scenarios import TrackScenario
    from gnss_sdr_ru_b200.synth import Sat

    scs = []
    for s in range(S):
        prns = [int(p) for p in rng.choice(np.arange(1, 33), size=int(rng.integers(7, 10)), replace=False)]
        sats = [Sat(prn=p, cn0_dbhz=float(rng.uniform(45.0, 50.0)), doppler_hz=float(rng.uniform(-5000.0, 5000.0)),
                    code_phase_chips=float(rng.uniform(0.0, 1023.0)), carrier_phase_cycles=float(rng.random()),
                    data_bits=BITS) for p in prns]
        if s == 0:
            sats[0].doppler_hz = 230.0        # within 500 Hz of zero Doppler: Doppler bin 0 of the serial search
            sats[1].code_phase_chips = 1022.6  # chip 0 starts within the first chip: search cell 0 / 1, wraps
        scs.append(TrackScenario(sats=sats, prns=[], n_freq=[]))
    return scs


def _glonass_stream(rng):
    from gnss_sdr_ru_b200.scenarios import TrackScenario
    from gnss_sdr_ru_b200.synth import Sat

    fch = [int(k) for k in rng.choice(np.arange(-7, 7), size=6, replace=False)]
    # BITS at 50 bps rather than the 100-Hz meander, whose sign changes 10 ms apart the pull-in -> tracking test never counts
    sats = [Sat(system="glonass", prn=k, cn0_dbhz=float(rng.uniform(45.0, 50.0)), doppler_hz=float(rng.uniform(-5000.0, 5000.0)),
                code_phase_chips=float(rng.uniform(0.0, 511.0)), carrier_phase_cycles=float(rng.random()), data_bits=BITS,
                data_rate_hz=50.0) for k in fch]
    sats[0].code_phase_chips = 510.7
    return [TrackScenario(sats=sats, prns=[], n_freq=[])]


def _cold_start(scs, settings, cfg, n_compare, oracle_lib):
    import torch

    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine
    from gnss_sdr_ru_b200.lib import check, lib
    from gnss_sdr_ru_b200.receiver import TrackingEngine
    from gnss_sdr_ru_b200.scenarios import synth_sat_array

    S = len(scs)
    eng = TrackingEngine(n_streams=S, cfg=cfg)
    stride = 2 * NS * NBLK
    d_if = torch.empty((S, stride), dtype=torch.uint8, device="cuda")
    arr, nsat = synth_sat_array(scs)
    check(lib().gnssb200_synth(eng.h, d_if.data_ptr(), stride, abi.FMT_INT8_IQ, S, NS * NBLK, C.addressof(arr), nsat, 4321, None),
          "gnssb200_synth")
    acq = AcquisitionEngine(handle=eng.h)
    results = acq.acquisition_batch(d_if.data_ptr(), stride, S, acq.samples_needed(settings), settings)
    allocated = [eng.acq_allocate(s, results[s], settings) for s in range(S)]
    start = [bytes(memoryview(eng.rx[s]).cast("B")) for s in range(S)]
    eng.upload()
    d_dumps = torch.zeros((S, 12, CAP, 48), dtype=torch.uint8, device="cuda")
    d_cnt = torch.zeros((S, 12), dtype=torch.int32, device="cuda")
    eng.run_device(d_if.data_ptr(), stride, NBLK, NS, abi.FMT_INT8_IQ, d_dumps_ptr=d_dumps.data_ptr(), dump_cap=CAP,
                   d_count_ptr=d_cnt.data_ptr())
    torch.cuda.synchronize()
    eng.download()
    dumps = d_dumps.cpu().numpy().view(abi.DUMP_DTYPE).reshape(S, 12, CAP)
    cnt = d_cnt.cpu().numpy()
    for s in range(n_compare):  # bit exact against the oracle from the same allocated state
        o = oracle_lib.Oracle(oracle_lib.Oracle.default_cfg(**_CFG_OVER[cfg.glonass_carrier_if != 0.0]))
        C.memmove(C.addressof(o.rx), start[s], len(start[s]))
        n, odumps, ocnt = o.run(d_if[s].cpu().numpy().view(np.int8), NS, NBLK, dump_cap=CAP)
        assert n == NBLK
        assert np.array_equal(cnt[s], ocnt), (s, cnt[s], ocnt)
        for ch in range(12):
            a, b = dumps[s, ch, : cnt[s, ch]], odumps[ch, : ocnt[ch]]
            if a.tobytes() != b.tobytes():
                i = next(i for i in range(len(a)) if a[i].tobytes() != b[i].tobytes())
                raise AssertionError(f"stream {s} ch {ch}: first differing dump {i}: gpu {a[i]} oracle {b[i]}")
        assert bytes(memoryview(eng.rx[s]).cast("B")) == bytes(memoryview(o.rx).cast("B")), f"stream {s}: rx differs"
    return eng, allocated, dumps, cnt


def _check_behaviour(scs, eng, allocated, dumps, cnt):
    for s, sc in enumerate(scs):
        assert sorted(allocated[s]) == sorted(sat.prn for sat in sc.sats), (s, allocated[s])
        for ch in range(len(allocated[s])):
            st = dumps[s, ch, : cnt[s, ch]]["state"]
            assert (st[:8] >= 2).any(), (s, ch, allocated[s][ch], st[:12])  # confirmed within its first 8 dumps
            assert eng.rx[s].chan[ch].state == 4, (s, ch, allocated[s][ch], int(eng.rx[s].chan[ch].state))
        for ch in range(len(allocated[s]), 12):
            assert cnt[s, ch] == 0  # channels left off never dump


def test_gps_cold_start_four_streams(oracle_lib):
    from gnss_sdr_ru_b200.acquisition import Settings
    from gnss_sdr_ru_b200.lib import default_cfg

    scs = _gps_streams(np.random.default_rng(2024), 4)
    eng, allocated, dumps, cnt = _cold_start(scs, Settings.gps(), default_cfg(), 2, oracle_lib)
    _check_behaviour(scs, eng, allocated, dumps, cnt)


def test_glonass_cold_start(oracle_lib):
    from gnss_sdr_ru_b200.acquisition import Settings
    from gnss_sdr_ru_b200.lib import default_cfg

    scs = _glonass_stream(np.random.default_rng(77))
    eng, allocated, dumps, cnt = _cold_start(scs, Settings.glonass(), default_cfg(glonass_carrier_if=1.0e6), 1, oracle_lib)
    _check_behaviour(scs, eng, allocated, dumps, cnt)
