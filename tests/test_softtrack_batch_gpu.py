"""Float (Scilab) tracking batched over records, gnssb200_softtrack_batch: every channel's output is byte-identical to
gnssb200_softtrack on its record alone, at every kernel width (128 / 256 / 512 threads per channel), on int8 and on
packed 2+2-bit records (against the single call on the unpacked record), and each channel stops at its own record's
end.  One GLONASS and one GPS channel are also compared with the float64 restatement (oracle/softtrack_oracle.py),
and the GLONASS chain acquisition -> preRun -> tracking -> findTimeMarks runs for four receivers at once."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

WIDTHS = (512, 256, 128)


def _compare(res, ora, ms):
    for f in ("I_E", "I_P", "I_L", "Q_E", "Q_P", "Q_L"):
        scale = np.abs(ora["I_P"]).mean() + np.abs(ora["Q_P"]).mean()
        assert len(res[f]) == len(ora[f]) == ms
        assert np.max(np.abs(res[f] - ora[f])) <= 1e-7 * scale, (f, np.max(np.abs(res[f] - ora[f])), scale)
    assert np.max(np.abs(res["absoluteSample"] - ora["absoluteSample"])) <= 1e-6
    assert np.max(np.abs(res["carrFreq"] - ora["carrFreq"])) <= 1e-6
    assert np.max(np.abs(res["codeFreq"] - ora["codeFreq"])) <= 1e-6
    for f in ("dllDiscr", "dllDiscrFilt", "pllDiscr", "pllDiscrFilt"):
        assert np.max(np.abs(res[f] - ora[f])) <= 1e-8, f


def _same_bytes(a, b) -> bool:
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def _glo(k, dop, cp, seed):
    from gnss_sdr_ru_b200.synth import Sat

    return Sat(system="glonass", prn=k, cn0_dbhz=48.0, doppler_hz=dop, code_phase_chips=cp, data_seed=seed, data_rate_hz=100.0)


def _gps(prn, dop, cp, seed):
    from gnss_sdr_ru_b200.synth import Sat

    return Sat(system="gps", prn=prn, cn0_dbhz=48.0, doppler_hz=dop, code_phase_chips=cp, data_seed=seed)


def _channel(sat):
    """The channel list entry preRun would make for a satellite, from its true Doppler and code phase."""
    if sat.system == "glonass":
        f, L, bias = 1e6 + 562500.0 * sat.prn + sat.doppler_hz, 511.0, 30.0
    else:
        f, L, bias = 2.42e6 + sat.doppler_hz, 1023.0, 40.0
    cp = int(round((L - sat.code_phase_chips % L) * 16000.0 / L)) % 16000 + 1
    return dict(FCH=sat.prn, acquiredFreq=f + bias, codePhase=cp)


def _synth(h, sat_lists, n, fmt, seed, extra=0):
    """Records of n + extra samples synthesised on the device, one row per record (the row is the stride)."""
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.lib import check, lib
    from gnss_sdr_ru_b200.scenarios import TrackScenario, synth_sat_array

    m = n + extra
    row = 2 * m if fmt == abi.FMT_INT8_IQ else m // 2
    d = torch.zeros((len(sat_lists), row), dtype=torch.uint8, device="cuda")
    arr, nsat = synth_sat_array([TrackScenario(sats=s, prns=[], n_freq=[]) for s in sat_lists])
    check(lib().gnssb200_synth(h, d.data_ptr(), row, fmt, len(sat_lists), m, C.addressof(arr), nsat, seed, None), "gnssb200_synth")
    return d


def _single(eng, d_ptr, n, channel, ts):
    """gnssb200_softtrack on one int8 record: rows [n_ch][ms][13] and periods done [n_ch]."""
    import torch

    d_out = torch.zeros((len(channel), ts.msToProcess, 13), dtype=torch.float64, device="cuda")
    d_done = torch.zeros(len(channel), dtype=torch.int32, device="cuda")
    eng.tracking_device(d_ptr, n, channel, ts, d_out.data_ptr(), d_done.data_ptr())
    return d_out.cpu().numpy(), d_done.cpu().numpy()


def _batch_raw(eng, ts, d_ptr, stride, n_records, fmt, n, channel, chan_record, d_out=None, d_done=None):
    """gnssb200_softtrack_batch with an explicit chan_record (channels of different records may interleave).
    Returns (rc, rows, done)."""
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.lib import lib

    n_ch = len(channel)
    ch = (abi.SoftTrackChan * max(n_ch, 1))()
    rec = (C.c_int32 * max(n_ch, 1))()
    for i, c in enumerate(channel):
        ch[i].sv, ch[i].code_phase, ch[i].acquired_freq = c["FCH"], c["codePhase"], c["acquiredFreq"]
        rec[i] = chan_record[i]
    if d_out is None:
        d_out = torch.zeros((max(n_ch, 1), ts.msToProcess, 13), dtype=torch.float64, device="cuda")
        d_done = torch.zeros(max(n_ch, 1), dtype=torch.int32, device="cuda")
    cfg = ts.to_c()
    rc = lib().gnssb200_softtrack_batch(eng.h, C.byref(cfg), d_ptr, stride, n_records, fmt, n, ch, rec, n_ch, d_out.data_ptr(),
                                        d_done.data_ptr(), None)
    torch.cuda.synchronize()
    return rc, d_out.cpu().numpy(), d_done.cpu().numpy()


def _check_against_single(rows, done, channel, chan_record, ref):
    """ref[r] = (rows, done) of the single call on record r with its channels in `channel` order."""
    pos = {}
    for i, r in enumerate(chan_record):
        k = pos.get(r, 0)
        pos[r] = k + 1
        assert done[i] == ref[r][1][k], (i, r, done[i], ref[r][1][k])
        assert _same_bytes(rows[i], ref[r][0][k]), (i, r, channel[i])


def test_batch_equals_single_call_every_width():
    """Four int8 records (two GLONASS, two GPS as a second call), channels of different records interleaved:
    each channel's rows and ms_done are byte-identical to gnssb200_softtrack on its record alone, for NT = 512, 256, 128."""
    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine, TrackSettings

    ms = 300
    n = 16000 * (ms + 3)
    recs = [[_glo(-3, 1234.0, 100.7, 3), _glo(2, -2100.0, 300.2, 4), _glo(5, 640.0, 17.5, 5)],
            [_glo(-7, -330.0, 455.1, 6), _glo(0, 2890.0, 222.2, 7)],
            [_gps(3, -1500.0, 200.0, 8), _gps(17, 2200.0, 811.3, 9), _gps(32, 410.0, 5.6, 10)],
            [_gps(1, -3100.0, 1000.9, 11), _gps(7, 1750.0, 432.1, 12)]]
    eng = SoftTrackingEngine()
    d = _synth(eng.h, recs, n, abi.FMT_INT8_IQ, seed=41)
    stride = d.stride(0)
    for system, rset, ts in (("glonass", (0, 1), TrackSettings(msToProcess=ms)), ("gps", (2, 3), TrackSettings.gps(msToProcess=ms))):
        ref = {r: _single(eng, d[r].data_ptr(), n, [_channel(s) for s in recs[r]], ts) for r in rset}
        # round robin over the records: r0c0 r1c0 r0c1 r1c1 r0c2
        order = [(r, k) for k in range(3) for r in rset if k < len(recs[r])]
        channel = [_channel(recs[r][k]) for r, k in order]
        chan_record = [r for r, _ in order]
        for nt in WIDTHS:
            eng.set_width(nt)
            rc, rows, done = _batch_raw(eng, ts, d.data_ptr(), stride, len(recs), abi.FMT_INT8_IQ, n, channel, chan_record)
            assert rc == 0, (system, nt)
            assert (done == ms).all(), (system, nt, done)
            _check_against_single(rows, done, channel, chan_record, ref)
        if system == "glonass":  # the loops are locked: prompt power in the in-phase arm
            assert all(np.abs(ref[r][0][:, -100:, 1]).mean() > 5 * np.abs(ref[r][0][:, -100:, 4]).mean() for r in rset)
    eng.set_width(0)


def test_packed_equals_int8_expansion():
    """Packed records tracked in one call are byte-identical to the single call on unpack2 of each record, at every
    width; one channel starts on an odd sample."""
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine, TrackSettings
    from gnss_sdr_ru_b200.synth import unpack2

    ms = 250
    n = 16000 * (ms + 3)
    recs = [[_glo(-1, 980.0, 50.3, 21), _glo(4, -2700.0, 400.4, 22)],
            [_glo(6, 310.0, 260.8, 23), _glo(-5, -1200.0, 133.3, 24), _glo(1, 2000.0, 77.7, 25)],
            [_gps(14, 1300.0, 600.6, 26), _gps(22, -2600.0, 88.8, 27)]]
    eng = SoftTrackingEngine()
    dp = _synth(eng.h, recs, n, abi.FMT_PACKED2, seed=43)
    unpacked = [torch.from_numpy(unpack2(dp[r].cpu().numpy()).view(np.uint8)).cuda() for r in range(len(recs))]
    chans = [[_channel(s) for s in rec] for rec in recs]
    chans[0][0]["codePhase"] += chans[0][0]["codePhase"] % 2  # start sample codePhase - 1 odd
    chans[2][1]["codePhase"] += chans[2][1]["codePhase"] % 2
    assert (chans[0][0]["codePhase"] - 1) % 2 == 1 and (chans[2][1]["codePhase"] - 1) % 2 == 1
    for rset, ts in (((0, 1), TrackSettings(msToProcess=ms)), ((2,), TrackSettings.gps(msToProcess=ms))):
        ref = {r: _single(eng, unpacked[r].data_ptr(), n, chans[r], ts) for r in rset}
        channel = [c for r in rset for c in chans[r]]
        chan_record = [r for r in rset for _ in chans[r]]
        for nt in WIDTHS:
            eng.set_width(nt)
            rc, rows, done = _batch_raw(eng, ts, dp.data_ptr(), dp.stride(0), len(recs), abi.FMT_PACKED2, n, channel, chan_record)
            assert rc == 0 and (done == ms).all(), (nt, rc, done)
            _check_against_single(rows, done, channel, chan_record, ref)
    eng.set_width(0)


def test_record_end_is_per_record():
    """Every record holds n samples that end mid-period, followed by more (non-zero) samples inside the stride: each
    channel stops where the single call on its record stops.  Stride 0 runs R copies of one record."""
    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine, TrackSettings

    ms = 50
    n = 16000 * 40 + 7776
    extra = 16000 * 3
    recs = [[_glo(3, 800.0, 300.0, 31)], [_glo(-2, -900.0, 120.0, 32)], [_glo(0, 1500.0, 480.0, 33)]]
    ts = TrackSettings(msToProcess=ms)
    eng = SoftTrackingEngine()
    d = _synth(eng.h, recs, n, abi.FMT_INT8_IQ, seed=45, extra=extra)
    assert int((d[:, 2 * n :] != 0).sum().item()) == d[:, 2 * n :].numel()  # int8 samples are never 0
    near_end = dict(_channel(recs[0][0]))
    near_end["codePhase"] += 16000 * 36  # a channel that starts 36 periods into record 0: 4 periods before its end
    chans = [[_channel(recs[0][0]), near_end], [_channel(recs[1][0])], [_channel(recs[2][0])]]
    ref = {r: _single(eng, d[r].data_ptr(), n, chans[r], ts) for r in range(3)}
    assert ref[0][1][1] < 5 and all(ref[r][1][0] < 41 for r in range(3))  # every channel runs into its record's end
    channel = [chans[1][0], chans[0][0], chans[2][0], chans[0][1]]
    chan_record = [1, 0, 2, 0]
    for nt in WIDTHS:
        eng.set_width(nt)
        rc, rows, done = _batch_raw(eng, ts, d.data_ptr(), d.stride(0), 3, abi.FMT_INT8_IQ, n, channel, chan_record)
        assert rc == 0
        _check_against_single(rows, done, channel, chan_record, ref)
        # the samples after a record's end would have allowed more periods
        rc, _, longer = _batch_raw(eng, ts, d.data_ptr(), d.stride(0), 3, abi.FMT_INT8_IQ, n + extra, channel, chan_record)
        assert rc == 0 and (longer > done).all()
    eng.set_width(0)
    # stride 0: three copies of record 0
    channel = chans[0] * 3
    chan_record = [0, 0, 1, 1, 2, 2]
    rc, rows, done = _batch_raw(eng, ts, d[0].data_ptr(), 0, 3, abi.FMT_INT8_IQ, n, channel, chan_record)
    assert rc == 0
    for r in range(3):
        for k in range(2):
            assert done[2 * r + k] == ref[0][1][k] and _same_bytes(rows[2 * r + k], ref[0][0][k])


def test_packed_narrow_width_against_oracle():
    """One GLONASS and one GPS channel at 128 threads per channel on packed records, compared directly with the float64
    restatement on the unpacked record."""
    from oracle import softtrack_oracle as so
    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine, TrackSettings
    from gnss_sdr_ru_b200.synth import unpack2

    ms = 200
    n = 16000 * (ms + 3)
    recs = [[_glo(2, 1234.0, 100.7, 51)], [_gps(9, -1700.0, 345.6, 52)]]
    eng = SoftTrackingEngine()
    eng.set_width(128)
    dp = _synth(eng.h, recs, n, abi.FMT_PACKED2, seed=47)
    for r, (ts, ots) in enumerate(((TrackSettings(msToProcess=ms), so.TrackSettings(msToProcess=ms)),
                                   (TrackSettings.gps(msToProcess=ms), so.TrackSettings.gps(msToProcess=ms)))):
        chans = [[], []]
        chans[r] = [_channel(recs[r][0])]
        res = eng.tracking_batch(dp.data_ptr(), dp.stride(0), 2, n, chans, ts, fmt=abi.FMT_PACKED2)
        assert [len(x) for x in res] == [len(c) for c in chans]
        ora = so.tracking(unpack2(dp[r].cpu().numpy()), chans[r][0], ots)
        _compare(res[r][0], ora, ms)


def test_chain_many_receivers_glonass_time_marks():
    """acquisition_batch -> preRun per record -> tracking_batch_device (automatic width) -> one findTimeMarks_device over
    all channels of four packed records.  Each record has its own frequency channels, Dopplers and code phases; every
    channel's mark equals the one the single-record chain (int8, gnssb200_softtrack) finds on its record, and the
    mark repeats one string (2000 ms) later."""
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine, Settings
    from gnss_sdr_ru_b200.navbits import NAV_F64, NavBitsEngine
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine, TrackSettings, preRun
    from gnss_sdr_ru_b200.synth import Sat

    rng = np.random.default_rng(35)
    tm = np.array([-1, 1, 1, -1, 1, -1, -1, 1, -1, -1, -1, -1, 1, -1, 1, -1, 1, 1, 1, -1, 1, 1, -1, -1, -1, 1, 1, 1, 1, 1])
    ms = 4300
    n = 16000 * (ms + 20)
    fchs = [(-4, 1, 5), (-7, -1, 3), (-2, 2, 6), (-5, 0, 4)]
    recs = []
    for r, ks in enumerate(fchs):
        sats = []
        for i, k in enumerate(ks):
            string = np.concatenate([2 * rng.integers(0, 2, size=170) - 1, tm[::-1]])  # 1.7 s of symbols + 0.3 s time mark
            bits = ((1 - np.tile(string, 3)) // 2).astype(np.uint8)
            sats.append(Sat(system="glonass", prn=k, cn0_dbhz=49.0, doppler_hz=float(rng.uniform(-3000.0, 3000.0)),
                            code_phase_chips=float(rng.uniform(0.0, 511.0)), data_bits=bits, data_rate_hz=100.0))
        recs.append(sats)
    acq_eng = AcquisitionEngine()
    h = acq_eng.h
    d8 = _synth(h, recs, n, abi.FMT_INT8_IQ, seed=919)
    dp = _synth(h, recs, n, abi.FMT_PACKED2, seed=919)
    acq_set = Settings.glonass(acqSatelliteList=sorted(k for ks in fchs for k in ks))
    ts = TrackSettings(msToProcess=ms)
    eng = SoftTrackingEngine(handle=h)
    nav = NavBitsEngine(handle=h)
    n_acq = 16000 * 11

    # the single-record chain on each int8 record
    single_ch, single_rows, single_marks = [], [], []
    for r in range(len(recs)):
        acq = acq_eng.acquisition(d8[r, : 2 * n_acq].cpu().numpy().view(np.int8), acq_set)
        channel = preRun(acq, ts)
        assert sorted(c["FCH"] for c in channel) == sorted(fchs[r]), r
        rows, done = _single(eng, d8[r].data_ptr(), n, channel, ts)
        assert (done == ms).all()
        d_rows = torch.from_numpy(rows).cuda()
        first, _ = nav.findTimeMarks_device(d_rows.data_ptr() + 8, NAV_F64, ms * 13 * 8, 13 * 8, len(channel), ms)
        single_ch.append(channel)
        single_rows.append(rows)
        single_marks.append(first)

    # the batched chain on the packed records
    acqs = acq_eng.acquisition_batch(dp.data_ptr(), dp.stride(0), len(recs), n_acq, acq_set, fmt=abi.FMT_PACKED2)
    channels = [preRun(a, ts) for a in acqs]
    assert channels == single_ch
    n_ch = sum(len(c) for c in channels)
    d_out = torch.zeros((n_ch, ms, 13), dtype=torch.float64, device="cuda")
    d_done = torch.zeros(n_ch, dtype=torch.int32, device="cuda")
    eng.set_width(0)
    eng.tracking_batch_device(dp.data_ptr(), dp.stride(0), len(recs), n, channels, ts, d_out.data_ptr(), d_done.data_ptr(),
                              fmt=abi.FMT_PACKED2)
    assert d_done.cpu().tolist() == [ms] * n_ch
    first, act = nav.findTimeMarks_device(d_out.data_ptr() + 8, NAV_F64, ms * 13 * 8, 13 * 8, n_ch, ms)
    assert act == list(range(1, n_ch + 1))
    out = d_out.cpu().numpy()
    assert _same_bytes(out, np.concatenate(single_rows))
    assert np.array_equal(first, np.concatenate(single_marks))
    pat = -np.repeat(tm[::-1], 10)
    ip = out[:, :, 1]
    for ch in range(n_ch):
        k0 = int(first[ch]) - 1
        assert 1300 <= k0 <= 1900, (ch, k0)  # the first string's mark starts 1.7 s into the record, minus the code phase
        assert abs(int(np.dot(np.sign(ip[ch, k0 + 2000 : k0 + 2300]), pat))) > 290  # and again one string later


def test_invalid_arguments_leave_outputs_untouched():
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.lib import GnssB200Error
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine, TrackSettings

    ms = 10
    n = 16000 * 12
    recs = [[_glo(1, 500.0, 10.0, 61)], [_gps(5, 700.0, 20.0, 62)]]
    eng = SoftTrackingEngine()
    d = _synth(eng.h, recs, n, abi.FMT_INT8_IQ, seed=49)
    stride = d.stride(0)
    glo, gps = TrackSettings(msToProcess=ms), TrackSettings.gps(msToProcess=ms)
    cg = [_channel(recs[0][0])]
    cp = [_channel(recs[1][0])]
    d_out = torch.full((2, ms, 13), -7.5, dtype=torch.float64, device="cuda")
    d_done = torch.full((2,), -3, dtype=torch.int32, device="cuda")

    def bad(ts, channel, chan_record, n_records=2, fmt=abi.FMT_INT8_IQ, stride_=stride, n_=n):
        rc, rows, done = _batch_raw(eng, ts, d.data_ptr(), stride_, n_records, fmt, n_, channel, chan_record, d_out, d_done)
        assert rc < 0
        assert (rows == -7.5).all() and (done == -3).all()

    bad(glo, cg, [0], n_records=0)
    bad(glo, cg, [2])
    bad(glo, cg, [-1])
    bad(glo, cg, [0], fmt=abi.FMT_INT8_I)
    bad(glo, cg, [0], fmt=7)
    bad(glo, cg, [0], stride_=2 * n - 2)                        # int8 record needs 2n bytes
    bad(glo, cg, [0], fmt=abi.FMT_PACKED2, stride_=n // 2 - 1)  # packed record needs n/2 bytes
    bad(gps, [dict(cp[0], FCH=0)], [1])
    bad(gps, [dict(cp[0], FCH=33)], [1])
    bad(TrackSettings(msToProcess=ms, codeLength=1000), cg, [0])
    bad(glo, [], [])
    # the valid forms of the same call run
    rc, _, done = _batch_raw(eng, glo, d.data_ptr(), stride, 2, abi.FMT_INT8_IQ, n, cg, [0])
    assert rc == 0 and done[0] == ms
    rc, _, done = _batch_raw(eng, glo, d.data_ptr(), n // 2, 2, abi.FMT_PACKED2, n, cg, [0])
    assert rc == 0
    for w in (64, 1024, -128):
        with pytest.raises(GnssB200Error):
            eng.set_width(w)
