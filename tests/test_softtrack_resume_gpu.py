"""Resumable float tracking: gnssb200_softtrack_resume window by window and gnssb200_softtrack_batch_host from host
records give every channel's rows and ms_done byte-identical to one gnssb200_softtrack_batch call on the whole record,
at any window length and kernel width, across a checkpoint of the states to the host and onto another handle.  A channel
never reads outside its window: it stops as BEHIND or BAD_RECORD and its rows keep their sentinel."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

P = 16000  # samples per code period at 16 MHz, GLONASS and GPS


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


def _synth(h, sat_lists, n, fmt, seed, row=None):
    """Records of n samples synthesised on the device, one row per record (the row is the stride)."""
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.lib import check, lib
    from gnss_sdr_ru_b200.scenarios import TrackScenario, synth_sat_array

    m = n + (-n) % 4  # the generator writes multiples of 4 samples
    row = row or (2 * m if fmt == abi.FMT_INT8_IQ else m // 2)
    d = torch.zeros((len(sat_lists), row), dtype=torch.uint8, device="cuda")
    arr, nsat = synth_sat_array([TrackScenario(sats=s, prns=[], n_freq=[]) for s in sat_lists])
    check(lib().gnssb200_synth(h, d.data_ptr(), row, fmt, len(sat_lists), m, C.addressof(arr), nsat, seed, None), "gnssb200_synth")
    return d


def _tables(abi, channel, chan_record):
    ch = (abi.SoftTrackChan * max(len(channel), 1))()
    rec = (C.c_int32 * max(len(channel), 1))()
    for i, c in enumerate(channel):
        ch[i].sv, ch[i].code_phase, ch[i].acquired_freq = c["FCH"], c["codePhase"], c["acquiredFreq"]
        rec[i] = chan_record[i]
    return ch, rec


def _one_shot(eng, ts, d_ptr, stride, n_records, fmt, n, channel, chan_record):
    """gnssb200_softtrack_batch: (rows, done)."""
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.lib import check, lib

    ch, rec = _tables(abi, channel, chan_record)
    d_out = torch.full((len(channel), ts.msToProcess, 13), np.nan, dtype=torch.float64, device="cuda")
    d_done = torch.zeros(len(channel), dtype=torch.int32, device="cuda")
    cfg = ts.to_c()
    check(lib().gnssb200_softtrack_batch(eng.h, C.byref(cfg), d_ptr, stride, n_records, fmt, n, ch, rec, len(channel),
                                         d_out.data_ptr(), d_done.data_ptr(), None), "gnssb200_softtrack_batch")
    return d_out.cpu().numpy(), d_done.cpu().numpy()


def _states(eng, ts, channel, chan_record, n_records):
    """Initial states on the device (uint8 tensor) from gnssb200_softtrack_init."""
    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.lib import check, lib

    ch, rec = _tables(abi, channel, chan_record)
    st = (abi.SoftTrackState * len(channel))()
    cfg = ts.to_c()
    check(lib().gnssb200_softtrack_init(C.byref(cfg), ch, rec, n_records, len(channel), st), "gnssb200_softtrack_init")
    return _upload(st)


def _upload(states):
    import torch

    return torch.frombuffer(bytearray(bytes(states)), dtype=torch.uint8).cuda()


def _download(d_state):
    from gnss_sdr_ru_b200 import abi

    raw = d_state.cpu().numpy().tobytes()
    n = len(raw) // C.sizeof(abi.SoftTrackState)
    return (abi.SoftTrackState * n).from_buffer_copy(raw)


def _win_ptr(d, fmt, first):
    from gnss_sdr_ru_b200 import abi

    return d.data_ptr() + (2 * first if fmt == abi.FMT_INT8_IQ else first // 2)


def _windows(n, W, A):
    """(first, length) of windows of W samples advancing by A until one reaches sample n."""
    first = 0
    while True:
        yield first, min(W, n - first)
        if first + W >= n:
            return
        first += A


def _run_windows(eng, ts, d, stride, n_records, fmt, n, d_state, d_out, W, A, widths=(0,), record_samples=None, start=0,
                 stop=None):
    """resume over windows [start, stop) of _windows(n, W, A); the width cycles through `widths`.  Returns the count."""
    import torch

    k = 0
    for k, (first, length) in enumerate(_windows(n, W, A)):
        if k < start:
            continue
        if stop is not None and k >= stop:
            return k
        eng.set_width(widths[k % len(widths)])
        rs = n if record_samples is None else record_samples(first, length)
        eng.resume_device(_win_ptr(d, fmt, first), stride, n_records, fmt, first, length, rs, ts, d_state.data_ptr(),
                          d_state.numel() // 112, d_out.data_ptr())
    torch.cuda.synchronize()
    eng.set_width(0)
    return k + 1


def _check(rows, states, ref, idx=None):
    ref_rows, ref_done = ref
    for i in (range(len(states)) if idx is None else idx):
        k = states[i].ms_done
        assert k == ref_done[i], (i, k, ref_done[i])
        assert _same_bytes(rows[i, :k], ref_rows[i, :k]), i


def _sets():
    """Two GLONASS and two GPS records, channels of the two records of a system interleaved."""
    from gnss_sdr_ru_b200.softtrack import TrackSettings

    recs = [[_glo(-3, 1234.0, 100.7, 3), _glo(2, -2100.0, 300.2, 4), _glo(5, 640.0, 17.5, 5)],
            [_glo(-7, -330.0, 455.1, 6), _glo(0, 2890.0, 222.2, 7)],
            [_gps(3, -1500.0, 200.0, 8), _gps(17, 2200.0, 811.3, 9), _gps(32, 410.0, 5.6, 10)],
            [_gps(1, -3100.0, 1000.9, 11), _gps(7, 1750.0, 432.1, 12)]]
    out = []
    for rset, mk in (((0, 1), TrackSettings), ((2, 3), TrackSettings.gps)):
        order = [(r, k) for k in range(3) for r in rset if k < len(recs[r])]
        out.append((mk, [_channel(recs[r][k]) for r, k in order], [r for r, _ in order]))
    return recs, out


@pytest.mark.parametrize("fmt_name", ["int8", "packed"])
def test_windows_equal_one_call(fmt_name):
    """Smallest legal window (four periods, overlap two) and an irregular one with the width changing 512 -> 128 -> 256
    between windows: rows and ms_done byte-identical to gnssb200_softtrack_batch."""
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine

    fmt = abi.FMT_INT8_IQ if fmt_name == "int8" else abi.FMT_PACKED2
    ms = 120
    n = P * (ms + 3)
    recs, sets = _sets()
    eng = SoftTrackingEngine()
    d = _synth(eng.h, recs, n, fmt, seed=41)
    stride = d.stride(0)
    for mk, channel, chan_record in sets:
        ts = mk(msToProcess=ms)
        ref = _one_shot(eng, ts, d.data_ptr(), stride, len(recs), fmt, n, channel, chan_record)
        assert (ref[1] == ms).all()
        for W, A, widths in ((4 * P, 2 * P, (0,)), (3 * P + 4322, P + 4322, (512, 128, 256))):
            d_state = _states(eng, ts, channel, chan_record, len(recs))
            d_out = torch.full((len(channel), ms, 13), np.nan, dtype=torch.float64, device="cuda")
            k = _run_windows(eng, ts, d, stride, len(recs), fmt, n, d_state, d_out, W, A, widths)
            assert k >= 10
            st = _download(d_state)
            assert all(s.status == abi.SOFTTRACK_MS_DONE for s in st)
            _check(d_out.cpu().numpy(), st, ref)


def test_checkpoint_same_and_other_handle():
    """After a few windows the states go to the host and the device copy is overwritten; uploaded again, on the same
    handle and on a second one, the run continues to the same bytes."""
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine

    fmt = abi.FMT_PACKED2
    ms = 100
    n = P * (ms + 3)
    recs, sets = _sets()
    eng = SoftTrackingEngine()
    d = _synth(eng.h, recs, n, fmt, seed=42)
    stride = d.stride(0)
    W, A = 5 * P + 2000, 3 * P + 2000
    for mk, channel, chan_record in sets:
        ts = mk(msToProcess=ms)
        ref = _one_shot(eng, ts, d.data_ptr(), stride, len(recs), fmt, n, channel, chan_record)
        d_state = _states(eng, ts, channel, chan_record, len(recs))
        d_out = torch.full((len(channel), ms, 13), np.nan, dtype=torch.float64, device="cuda")
        _run_windows(eng, ts, d, stride, len(recs), fmt, n, d_state, d_out, W, A, stop=5)
        saved = _download(d_state)
        assert all(s.status == abi.SOFTTRACK_RUNNING and 0 < s.ms_done < ms for s in saved)
        rows_saved = d_out.cpu()
        d_state.fill_(0xFF)
        for other in (False, True):
            e2 = SoftTrackingEngine() if other else eng
            d_state2 = _upload(saved)
            d_out2 = rows_saved.cuda()
            _run_windows(e2, ts, d, stride, len(recs), fmt, n, d_state2, d_out2, W, A, start=5)
            _check(d_out2.cpu().numpy(), _download(d_state2), ref)
            if other:
                e2.close()


def test_ends():
    """Record end inside a window (also with a provisional record length before the last window), ms_to_process reached
    mid-window, a channel that starts beyond the first windows, stride 0, and packed records of an odd length."""
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine, TrackSettings

    eng = SoftTrackingEngine()
    recs = [[_glo(3, 800.0, 300.0, 31)], [_glo(-2, -900.0, 120.0, 32)]]
    for fmt, n in ((abi.FMT_INT8_IQ, P * 40 + 7776), (abi.FMT_PACKED2, P * 40 + 7777)):
        d = _synth(eng.h, recs, n + 3, fmt, seed=45)
        late = dict(_channel(recs[1][0]))
        late["codePhase"] += P * 12  # starts 12 periods in: beyond the first windows
        channel = [_channel(recs[0][0]), _channel(recs[1][0]), late]
        chan_record = [0, 1, 1]
        for ms, end in ((50, abi.SOFTTRACK_RECORD_END), (23, abi.SOFTTRACK_MS_DONE)):
            ts = TrackSettings(msToProcess=ms)
            late0 = dict(channel[0], codePhase=channel[0]["codePhase"] + P * 12)
            for stride, chans in ((d.stride(0), channel), (0, [channel[0], channel[0], late0])):  # stride 0: record 0 twice
                ref = _one_shot(eng, ts, d.data_ptr(), stride, 2, fmt, n, chans, chan_record)
                if end == abi.SOFTTRACK_RECORD_END:
                    assert (ref[1] < ms).all() and ref[1][2] < 30
                else:
                    assert (ref[1][:2] == ms).all()
                for provisional in (False, True):
                    d_state = _states(eng, ts, chans, chan_record, 2)
                    d_out = torch.full((3, ms, 13), np.nan, dtype=torch.float64, device="cuda")
                    rs = (lambda f, l: n if f + l >= n else 1 << 40) if provisional else None
                    _run_windows(eng, ts, d, stride, 2, fmt, n, d_state, d_out, 4 * P + 1000, 2 * P + 1000, record_samples=rs)
                    st = _download(d_state)
                    assert [s.status for s in st[:2]] == [end, end]
                    _check(d_out.cpu().numpy(), st, ref)
                    rows = d_out.cpu().numpy()
                    assert all(np.isnan(rows[i, s.ms_done :]).all() for i, s in enumerate(st))


def test_never_outside_the_window():
    """A window that begins after a channel's next block: BEHIND, no row written; a record index out of range:
    BAD_RECORD; a GPS PRN out of range: BAD_SV.  The other channels are identical to the one-shot call."""
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine, TrackSettings

    eng = SoftTrackingEngine()
    ms = 40
    n = P * (ms + 3)
    recs = [[_glo(1, 500.0, 10.0, 61)], [_glo(4, -700.0, 200.0, 62)]]
    d = _synth(eng.h, recs, n, abi.FMT_INT8_IQ, seed=49)
    stride = d.stride(0)
    ts = TrackSettings(msToProcess=ms)
    late = dict(_channel(recs[1][0]))
    late["codePhase"] += P * 5
    channel = [_channel(recs[0][0]), late]
    ref = _one_shot(eng, ts, d.data_ptr(), stride, 2, abi.FMT_INT8_IQ, n, channel, [0, 1])
    d_state = _states(eng, ts, channel, [0, 1], 2)
    d_out = torch.full((2, ms, 13), np.nan, dtype=torch.float64, device="cuda")
    # the first window starts at 2P: channel 0 (next block at < P) is behind, channel 1 (at > 5P) runs
    first = 2 * P
    eng.resume_device(_win_ptr(d, abi.FMT_INT8_IQ, first), stride, 2, abi.FMT_INT8_IQ, first, n - first, n, ts,
                      d_state.data_ptr(), 2, d_out.data_ptr())
    torch.cuda.synchronize()
    st = _download(d_state)
    assert (st[0].status, st[0].ms_done) == (abi.SOFTTRACK_BEHIND, 0)
    assert np.isnan(d_out[0].cpu().numpy()).all()
    _check(d_out.cpu().numpy(), st, ref, idx=[1])
    assert ref[1][1] < ms and st[1].status == abi.SOFTTRACK_RECORD_END
    # record index and GPS PRN out of range
    for mk, field, value, status in ((TrackSettings, "record", 2, abi.SOFTTRACK_BAD_RECORD),
                                     (TrackSettings, "record", -1, abi.SOFTTRACK_BAD_RECORD),
                                     (TrackSettings.gps, "sv", 33, abi.SOFTTRACK_BAD_SV)):
        ts2 = mk(msToProcess=ms)
        chans = [_channel(recs[0][0]), _channel(recs[1][0])] if mk is TrackSettings else \
            [dict(FCH=5, codePhase=100, acquiredFreq=2.42e6), dict(FCH=9, codePhase=200, acquiredFreq=2.42e6 + 500.0)]
        ref2 = _one_shot(eng, ts2, d.data_ptr(), stride, 2, abi.FMT_INT8_IQ, n, chans, [0, 1])
        d_state = _states(eng, ts2, chans, [0, 1], 2)
        hs = _download(d_state)
        setattr(hs[0], field, value)
        d_state = _upload(hs)
        d_out = torch.full((2, ms, 13), np.nan, dtype=torch.float64, device="cuda")
        eng.resume_device(d.data_ptr(), stride, 2, abi.FMT_INT8_IQ, 0, n, n, ts2, d_state.data_ptr(), 2, d_out.data_ptr())
        torch.cuda.synchronize()
        st = _download(d_state)
        assert (st[0].status, st[0].ms_done) == (status, 0)
        assert np.isnan(d_out[0].cpu().numpy()).all()
        _check(d_out.cpu().numpy(), st, ref2, idx=[1])


@pytest.mark.parametrize("fmt_name", ["int8", "packed"])
def test_host_call_equals_one_call(fmt_name):
    """gnssb200_softtrack_batch_host from pinned and pageable host buffers, with a small window (many windows) and the
    automatic one, and with stride 0: return value 0, rows and ms_done byte-identical to the one-shot call."""
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine

    fmt = abi.FMT_INT8_IQ if fmt_name == "int8" else abi.FMT_PACKED2
    ms = 150
    n = P * (ms + 3) + (1 if fmt == abi.FMT_PACKED2 else 0)
    recs, sets = _sets()
    eng = SoftTrackingEngine()
    d = _synth(eng.h, recs, n, fmt, seed=51)
    stride = d.stride(0)
    pageable = d.cpu().numpy()
    pinned = torch.empty(d.shape, dtype=torch.uint8, pin_memory=True)
    pinned.copy_(d.cpu())
    for mk, channel, chan_record in sets:
        ts = mk(msToProcess=ms)
        ref = _one_shot(eng, ts, d.data_ptr(), stride, len(recs), fmt, n, channel, chan_record)
        chans = [[c for c, r in zip(channel, chan_record) if r == k] for k in range(len(recs))]
        flat_ref = {}
        i = 0
        for c, r in zip(channel, chan_record):  # one-shot rows of each channel, in record-by-record order
            flat_ref.setdefault(r, []).append(i)
            i += 1
        order = [i for r in range(len(recs)) for i in flat_ref.get(r, [])]
        for buf in (pinned, pageable):
            for window in (4 * P + 3000, 0):
                res = eng.tracking_batch_host(buf, stride, len(recs), n, chans, ts, fmt=fmt, window_samples=window)
                assert eng.host_stopped == 0
                got = [x for rr in res for x in rr]
                for g, i in zip(got, order):
                    assert len(g["I_E"]) == ref[1][i]
                    for k, f in enumerate(abi.SOFTTRACK_FIELDS):
                        assert _same_bytes(g[f], ref[0][i, : ref[1][i], k]), (i, f)
    # stride 0: one host record read for every record index
    mk, channel, chan_record = sets[0]
    ts = mk(msToProcess=ms)
    one = [[c for c, r in zip(channel, chan_record) if r == 0]]
    ref = _one_shot(eng, ts, d.data_ptr(), 0, 2, fmt, n, one[0] * 2, [0] * len(one[0]) + [1] * len(one[0]))
    res = eng.tracking_batch_host(pinned[0], 0, 2, n, one * 2, ts, fmt=fmt, window_samples=4 * P)
    got = [x for rr in res for x in rr]
    assert eng.host_stopped == 0 and len(got) == len(ref[1])
    for i, g in enumerate(got):
        assert _same_bytes(g["I_P"], ref[0][i, : ref[1][i], 1]) and _same_bytes(g["absoluteSample"], ref[0][i, : ref[1][i], 12])


def test_invalid_arguments_leave_states_and_outputs_untouched():
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.lib import lib
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine, TrackSettings

    L = lib()
    eng = SoftTrackingEngine()
    ms = 10
    n = P * 12
    recs = [[_glo(1, 500.0, 10.0, 71)], [_glo(2, 700.0, 20.0, 72)]]
    d = _synth(eng.h, recs, n, abi.FMT_INT8_IQ, seed=73)
    stride = d.stride(0)
    glo = TrackSettings(msToProcess=ms)
    channel = [_channel(recs[0][0]), _channel(recs[1][0])]
    d_state = _states(eng, glo, channel, [0, 1], 2)
    state0 = d_state.clone()
    d_out = torch.full((2, ms, 13), -7.5, dtype=torch.float64, device="cuda")

    def resume(cfg=glo.to_c(), win=d.data_ptr(), wstride=stride, n_records=2, fmt=abi.FMT_INT8_IQ, first=0, length=n,
               rs=n, state=d_state.data_ptr(), n_ch=2, out=d_out.data_ptr()):
        rc = L.gnssb200_softtrack_resume(eng.h, C.byref(cfg) if cfg is not None else None, win, wstride, n_records, fmt, first,
                                         length, rs, state, n_ch, out, None)
        torch.cuda.synchronize()
        return rc

    def untouched():
        return torch.equal(d_state, state0) and (d_out == -7.5).all().item()

    bad_resume = [dict(fmt=abi.FMT_INT8_I), dict(fmt=7), dict(fmt=abi.FMT_PACKED2, first=1, wstride=n), dict(wstride=2 * n - 2),
                  dict(fmt=abi.FMT_PACKED2, wstride=n // 2 - 1), dict(n_records=0), dict(n_ch=0), dict(n_ch=-1), dict(cfg=None),
                  dict(win=None), dict(state=None), dict(out=None), dict(cfg=TrackSettings(msToProcess=ms, codeLength=1000).to_c()),
                  dict(first=-2), dict(length=-1)]
    for kw in bad_resume:
        assert resume(**kw) < 0, kw
        assert untouched(), kw
    # the host call: the invalid arguments of the one-shot call, and a window shorter than four code periods
    h_iq = d.cpu().numpy()
    ch, rec = _tables(abi, channel, [0, 1])
    h_out = np.full((2, ms, 13), -7.5)
    h_done = np.full(2, -3, dtype=np.int32)

    def host(cfg=glo.to_c(), buf=h_iq.ctypes.data, hstride=stride, n_records=2, fmt=abi.FMT_INT8_IQ, n_=n, chans=ch, crec=rec,
             n_ch=2, out=h_out.ctypes.data, done=h_done.ctypes.data, window=0):
        return L.gnssb200_softtrack_batch_host(eng.h, C.byref(cfg), buf, hstride, n_records, fmt, n_, chans, crec, n_ch, out, done,
                                               window)

    for kw in [dict(window=4 * P - 1), dict(window=-1), dict(window=1), dict(fmt=abi.FMT_INT8_I), dict(n_records=0),
               dict(crec=(C.c_int32 * 2)(0, 2)), dict(hstride=2 * n - 2), dict(n_ch=0), dict(buf=None), dict(out=None),
               dict(done=None), dict(cfg=TrackSettings(msToProcess=ms, codeLength=1000).to_c()),
               dict(cfg=TrackSettings.gps(msToProcess=ms).to_c(), chans=_tables(abi, [dict(channel[0], FCH=33)] * 2, [0, 1])[0])]:
        assert host(**kw) < 0, kw
        assert (h_out == -7.5).all() and (h_done == -3).all(), kw
    # the valid forms run
    assert resume() == 0 and not untouched()
    assert host(window=4 * P) == 0 and (h_done == ms).all()


def test_graph_capture():
    """Windows captured in a CUDA graph and replayed give the bytes of the one-shot call; on a handle without its chip
    table yet, a capture is refused (-27) instead of being broken by the table's upload."""
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.lib import lib
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine, TrackSettings

    ms = 30
    n = P * (ms + 3)
    recs = [[_glo(2, 900.0, 40.0, 81)], [_glo(-4, -1300.0, 250.0, 82)]]
    channel = [_channel(recs[0][0]), _channel(recs[1][0])]
    ts = TrackSettings(msToProcess=ms)
    fresh = SoftTrackingEngine()
    s = torch.cuda.Stream()
    x = torch.zeros(4, device="cuda")
    d_state = torch.zeros(2 * 112, dtype=torch.uint8, device="cuda")
    d_out = torch.zeros((2, ms, 13), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    g0 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g0, stream=s):
        x.add_(1.0)
        cfg = ts.to_c()
        rc = lib().gnssb200_softtrack_resume(fresh.h, C.byref(cfg), x.data_ptr(), 0, 2, abi.FMT_INT8_IQ, 0, 0, n,
                                             d_state.data_ptr(), 2, d_out.data_ptr(), s.cuda_stream)
    assert rc == -27
    fresh.close()

    eng = SoftTrackingEngine()
    d = _synth(eng.h, recs, n, abi.FMT_INT8_IQ, seed=83)
    stride = d.stride(0)
    ref = _one_shot(eng, ts, d.data_ptr(), stride, 2, abi.FMT_INT8_IQ, n, channel, [0, 1])  # builds the chip table
    d_state = _states(eng, ts, channel, [0, 1], 2)
    d_out = torch.full((2, ms, 13), np.nan, dtype=torch.float64, device="cuda")
    eng.set_width(256)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        for first, length in _windows(n, 5 * P, 3 * P):
            eng.resume_device(_win_ptr(d, abi.FMT_INT8_IQ, first), stride, 2, abi.FMT_INT8_IQ, first, length, n, ts,
                              d_state.data_ptr(), 2, d_out.data_ptr(), stream=s.cuda_stream)
    eng.set_width(0)
    assert np.isnan(d_out.cpu().numpy()).all()  # captured, not run
    g.replay()
    torch.cuda.synchronize()
    _check(d_out.cpu().numpy(), _download(d_state), ref)
