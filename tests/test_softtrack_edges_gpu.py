"""Float (Scilab) tracking against the float64 restatement (oracle/softtrack_oracle.py) where kernels go wrong: the
extreme GLONASS frequency channels and GPS PRNs at +-4-5 kHz, the code epoch on the first and the last sample of a
period, correlator spacings 0 and 0.5 chip (the pads of the chip table read every period), a hard-clipped int8 record,
a record that ends exactly on a block, 2 s through the host path across ~30 window boundaries, and sample positions
past 2^32.  Every oracle case runs at 512 and 128 threads per channel, which must give the same bytes; packed records
are compared with the oracle on their int8 expansion.  The refusals: a correlator spacing outside 0..0.5 chip, and
int8 I,Q records at an odd byte address (their samples are 2-byte loads), for float tracking and FFT acquisition --
each returns < 0 before anything is launched or written.

Tolerances are those of tests/test_softtrack_gpu.py: correlator sums within 1e-7 of the prompt scale, NCO frequencies
within 1e-6 Hz, discriminators within 1e-8, absoluteSample within 1e-6 sample, identical row counts."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

P = 16000  # samples per code period at 16 MHz, GLONASS and GPS
WIDTHS = (512, 128)
SUMS = ("I_E", "I_P", "I_L", "Q_E", "Q_P", "Q_L")


def _tol_scale(ora):
    return np.abs(ora["I_P"]).mean() + np.abs(ora["Q_P"]).mean()


def _compare(res, ora, ms):
    scale = _tol_scale(ora)
    for f in SUMS:
        assert len(res[f]) == len(ora[f]) == ms, (f, len(res[f]), len(ora[f]), ms)
        assert np.max(np.abs(res[f] - ora[f])) <= 1e-7 * scale, (f, np.max(np.abs(res[f] - ora[f])), scale)
    assert np.max(np.abs(res["absoluteSample"] - ora["absoluteSample"])) <= 1e-6
    assert np.max(np.abs(res["carrFreq"] - ora["carrFreq"])) <= 1e-6
    assert np.max(np.abs(res["codeFreq"] - ora["codeFreq"])) <= 1e-6
    for f in ("dllDiscr", "dllDiscrFilt", "pllDiscr", "pllDiscrFilt"):
        assert np.max(np.abs(res[f] - ora[f])) <= 1e-8, f


def _same_bytes(a, b) -> bool:
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def _glo(k, dop, cp, seed, cn0=48.0):
    from gnss_sdr_ru_b200.synth import Sat

    return Sat(system="glonass", prn=k, cn0_dbhz=cn0, doppler_hz=dop, code_phase_chips=cp, data_seed=seed, data_rate_hz=100.0)


def _gps(prn, dop, cp, seed, cn0=48.0):
    from gnss_sdr_ru_b200.synth import Sat

    return Sat(system="gps", prn=prn, cn0_dbhz=cn0, doppler_hz=dop, code_phase_chips=cp, data_seed=seed)


def _channel(sat):
    """The channel list entry preRun would make for a satellite, from its true Doppler and code phase."""
    if sat.system == "glonass":
        f, L, bias = 1e6 + 562500.0 * sat.prn + sat.doppler_hz, 511.0, 30.0
    else:
        f, L, bias = 2.42e6 + sat.doppler_hz, 1023.0, 40.0
    cp = int(round((L - sat.code_phase_chips % L) * 16000.0 / L)) % 16000 + 1
    return dict(FCH=sat.prn, acquiredFreq=f + bias, codePhase=cp)


def _settings(system, **kw):
    """(library settings, oracle settings) of one system."""
    from oracle import softtrack_oracle as so
    from gnss_sdr_ru_b200.softtrack import TrackSettings

    if system == "gps":
        return TrackSettings.gps(**kw), so.TrackSettings.gps(**kw)
    return TrackSettings(**kw), so.TrackSettings(**kw)


def _fmt(name):
    from gnss_sdr_ru_b200 import abi

    return abi.FMT_INT8_IQ if name == "int8" else abi.FMT_PACKED2


def _synth(h, sat_lists, n, fmt, seed):
    """Records of n samples (rounded up to 4) synthesised on the device, one row per record (the row is the stride)."""
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.lib import check, lib
    from gnss_sdr_ru_b200.scenarios import TrackScenario, synth_sat_array

    m = n + (-n) % 4
    row = 2 * m if fmt == abi.FMT_INT8_IQ else m // 2
    d = torch.zeros((len(sat_lists), row), dtype=torch.uint8, device="cuda")
    arr, nsat = synth_sat_array([TrackScenario(sats=s, prns=[], n_freq=[]) for s in sat_lists])
    check(lib().gnssb200_synth(h, d.data_ptr(), row, fmt, len(sat_lists), m, C.addressof(arr), nsat, seed, None), "gnssb200_synth")
    return d


def _oracle_iq(d, r, fmt, n):
    """The int8 I,Q values of the first n samples of record r (the int8 expansion of a packed record)."""
    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.synth import unpack2

    row = d[r].cpu().numpy()
    x = row.view(np.int8) if fmt == abi.FMT_INT8_IQ else unpack2(row)
    return x[: 2 * n]


def _tables(channel, chan_record):
    from gnss_sdr_ru_b200 import abi

    ch = (abi.SoftTrackChan * max(len(channel), 1))()
    rec = (C.c_int32 * max(len(channel), 1))()
    for i, c in enumerate(channel):
        ch[i].sv, ch[i].code_phase, ch[i].acquired_freq = c["FCH"], c["codePhase"], c["acquiredFreq"]
        rec[i] = chan_record[i]
    return ch, rec


def _res(rows, done):
    from gnss_sdr_ru_b200 import abi

    return {f: rows[: done, k] for k, f in enumerate(abi.SOFTTRACK_FIELDS)}


def _batch(eng, ts, d_ptr, stride, n_records, fmt, n, channel, chan_record):
    """gnssb200_softtrack_batch at every width of WIDTHS, which must agree byte for byte: (rows, done)."""
    import torch

    from gnss_sdr_ru_b200.lib import check, lib

    ch, rec = _tables(channel, chan_record)
    got = []
    for nt in WIDTHS:
        eng.set_width(nt)
        d_out = torch.full((len(channel), ts.msToProcess, 13), np.nan, dtype=torch.float64, device="cuda")
        d_done = torch.full((len(channel),), -1, dtype=torch.int32, device="cuda")
        cfg = ts.to_c()
        check(lib().gnssb200_softtrack_batch(eng.h, C.byref(cfg), d_ptr, stride, n_records, fmt, n, ch, rec, len(channel),
                                             d_out.data_ptr(), d_done.data_ptr(), None), "gnssb200_softtrack_batch")
        got.append((d_out.cpu().numpy(), d_done.cpu().numpy()))
    eng.set_width(0)
    for rows, done in got[1:]:
        assert np.array_equal(done, got[0][1]) and _same_bytes(rows, got[0][0]), "the kernel widths disagree"
    return got[0]


def _states(ts, channel, chan_record, n_records):
    """gnssb200_softtrack_init on the host, uploaded: a uint8 device tensor."""
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.lib import check, lib

    ch, rec = _tables(channel, chan_record)
    st = (abi.SoftTrackState * len(channel))()
    cfg = ts.to_c()
    check(lib().gnssb200_softtrack_init(C.byref(cfg), ch, rec, n_records, len(channel), st), "gnssb200_softtrack_init")
    return torch.frombuffer(bytearray(bytes(st)), dtype=torch.uint8).cuda()


def _download(d_state):
    from gnss_sdr_ru_b200 import abi

    raw = d_state.cpu().numpy().tobytes()
    return (abi.SoftTrackState * (len(raw) // C.sizeof(abi.SoftTrackState))).from_buffer_copy(raw)


def _check_against_oracle(rows, done, channel, chan_record, d, fmt, n, ots, ms_each=None):
    """Every channel of a batched run against the oracle on its record's first n samples."""
    from oracle import softtrack_oracle as so

    for i, (c, r) in enumerate(zip(channel, chan_record)):
        ora = so.tracking(_oracle_iq(d, r, fmt, n), c, ots)
        ms = ots.msToProcess if ms_each is None else ms_each[i]
        assert done[i] == ms, (c, done[i], ms)
        _compare(_res(rows[i], done[i]), ora, ms)


@pytest.mark.parametrize("fmt_name", ["int8", "packed"])
@pytest.mark.parametrize("system", ["glonass", "gps"])
def test_a_frequency_and_prn_extremes(system, fmt_name):
    """GLONASS FCH -7 and +6, GPS PRN 1 and 32, each 4-5 kHz off the IF, 300 ms."""
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine

    fmt = _fmt(fmt_name)
    ms = 300
    n = P * (ms + 3)
    if system == "glonass":
        recs = [[_glo(-7, 4800.0, 123.4, 1)], [_glo(6, -4600.0, 401.9, 2)]]
    else:
        recs = [[_gps(1, 4400.0, 77.7, 3)], [_gps(32, -4900.0, 900.1, 4)]]
    eng = SoftTrackingEngine()
    d = _synth(eng.h, recs, n, fmt, seed=101)
    ts, ots = _settings(system, msToProcess=ms)
    channel = [_channel(recs[r][0]) for r in range(2)]
    rows, done = _batch(eng, ts, d.data_ptr(), d.stride(0), 2, fmt, n, channel, [0, 1])
    _check_against_oracle(rows, done, channel, [0, 1], d, fmt, n, ots)
    if system == "glonass":  # locked: prompt power in the in-phase arm (as in test_softtrack_batch_gpu.py, GLONASS only)
        assert all(np.abs(rows[i, -100:, 1]).mean() > 5 * np.abs(rows[i, -100:, 4]).mean() for i in range(2))


def test_b_code_phase_ends():
    """The code epoch on sample 0 (codePhase 1) and on sample 15999 (codePhase 16000), GLONASS and GPS, 100 ms.  Each
    case first shows that a start one sample off moves the oracle's I_P by more than 100x the tolerance."""
    from oracle import softtrack_oracle as so
    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine

    ms = 100
    n = P * (ms + 3)
    recs = [[_glo(3, 1700.0, 0.0, 11)], [_glo(-4, -2300.0, 511.0 / P, 12)],
            [_gps(12, -1200.0, 0.0, 13)], [_gps(25, 2600.0, 1023.0 / P, 14)]]
    eng = SoftTrackingEngine()
    d = _synth(eng.h, recs, n, abi.FMT_INT8_IQ, seed=103)
    for system, rset in (("glonass", (0, 1)), ("gps", (2, 3))):
        ts, ots = _settings(system, msToProcess=ms)
        channel = [_channel(recs[r][0]) for r in rset]
        assert [c["codePhase"] for c in channel] == [1, P]
        _, short = _settings(system, msToProcess=3)
        for c, r in zip(channel, rset):
            iq = _oracle_iq(d, r, abi.FMT_INT8_IQ, n)
            base = so.tracking(iq, c, short)
            moved = so.tracking(iq, dict(c, codePhase=c["codePhase"] + (1 if c["codePhase"] == 1 else -1)), short)
            assert np.max(np.abs(moved["I_P"] - base["I_P"])) > 100 * 1e-7 * _tol_scale(base), (system, c)
        rows, done = _batch(eng, ts, d.data_ptr(), d.stride(0), len(recs), abi.FMT_INT8_IQ, n, channel, list(rset))
        _check_against_oracle(rows, done, channel, rset, d, abi.FMT_INT8_IQ, n, ots)


@pytest.mark.parametrize("system", ["glonass", "gps"])
def test_c_spacing_edges(system):
    """Correlator spacing 0 (early = prompt = late, bit for bit) and 0.5 chip, GLONASS and GPS, 200 ms.  At 0.5 the
    pads of the chip table, caCode($) in front and caCode(1) behind, are read for 8 (GPS) to 16 (GLONASS) samples of
    every period.  First the case shows that a wrong left pad moves the oracle's early sums by more than 100x the
    tolerance: caCode(1) for the GPS PRN (whose first and last chips differ); the ST code's first and last chips are
    equal, so for GLONASS the wrong pad is -caCode($)."""
    from oracle import softtrack_oracle as so
    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.codes import ca_code, st_code
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine

    ms = 200
    n = P * (ms + 3)
    recs = [[_glo(-2, 2100.0, 250.5, 21)], [_gps(19, -3300.0, 512.3, 22)]]
    eng = SoftTrackingEngine()
    d = _synth(eng.h, recs, n, abi.FMT_INT8_IQ, seed=105)
    assert st_code()[0] == st_code()[-1] and ca_code(19)[0] != ca_code(19)[-1]
    r = 0 if system == "glonass" else 1
    c = _channel(recs[r][0])
    iq = _oracle_iq(d, r, abi.FMT_INT8_IQ, n)
    _, short = _settings(system, msToProcess=5, dllCorrelatorSpacing=0.5)
    code = st_code() if system == "glonass" else ca_code(19)
    wrong = -float(code[-1]) if system == "glonass" else float(code[0])
    base, mut = so.tracking(iq, c, short), so.tracking(iq, c, short, left_pad=wrong)
    dev = max(np.max(np.abs(mut[f] - base[f])) for f in ("I_E", "Q_E"))
    assert dev > 100 * 1e-7 * _tol_scale(base), (system, dev)
    for spc in (0.0, 0.5):
        ts, ots = _settings(system, msToProcess=ms, dllCorrelatorSpacing=spc)
        rows, done = _batch(eng, ts, d.data_ptr(), d.stride(0), 2, abi.FMT_INT8_IQ, n, [c], [r])
        _check_against_oracle(rows, done, [c], [r], d, abi.FMT_INT8_IQ, n, ots)
        if spc == 0.0:  # I_E I_L and Q_E Q_L are I_P and Q_P
            assert all(_same_bytes(rows[0, :, a], rows[0, :, b]) for a, b in ((0, 1), (2, 1), (3, 4), (5, 4)))


def test_d_full_scale():
    """A hard-clipped int8 record, every I and Q -128 or 127, holding one GLONASS and one GPS satellite."""
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine

    ms = 150
    n = P * (ms + 3)
    sats = [_glo(5, -1900.0, 333.3, 31, cn0=50.0), _gps(31, 2700.0, 12.9, 32, cn0=50.0)]
    eng = SoftTrackingEngine()
    d = _synth(eng.h, [sats], n, abi.FMT_INT8_IQ, seed=107)
    v = d.view(torch.int8)
    d = torch.where(v >= 0, torch.full_like(v, 127), torch.full_like(v, -128)).view(torch.uint8)
    assert set(np.unique(d.cpu().numpy().view(np.int8)).tolist()) == {-128, 127}
    for sat, system in zip(sats, ("glonass", "gps")):
        ts, ots = _settings(system, msToProcess=ms)
        c = _channel(sat)
        rows, done = _batch(eng, ts, d.data_ptr(), d.stride(0), 1, abi.FMT_INT8_IQ, n, [c], [0])
        _check_against_oracle(rows, done, [c], [0], d, abi.FMT_INT8_IQ, n, ots)


@pytest.mark.parametrize("fmt_name", ["int8", "packed"])
def test_e_exact_record_end(fmt_name):
    """pos_k = the first sample after period k.  A record of exactly pos_k samples gives k rows (the block that ends
    on the last sample runs), one of pos_k - 1 samples k - 1 rows, both ending RECORD_END; one of the two lengths is
    odd (for packed records, a half byte at the end)."""
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine

    fmt = _fmt(fmt_name)
    k = 30
    n = P * (k + 3)
    recs = [[_glo(1, 900.0, 47.1, 41)], [_gps(8, -2200.0, 610.6, 42)]]
    eng = SoftTrackingEngine()
    d = _synth(eng.h, recs, n, fmt, seed=109)
    for r, system in enumerate(("glonass", "gps")):
        c = _channel(recs[r][0])
        ts_k, _ = _settings(system, msToProcess=k)
        d_state = _states(ts_k, [c], [r], 2)
        d_out = torch.full((1, k, 13), np.nan, dtype=torch.float64, device="cuda")
        eng.resume_device(d.data_ptr(), d.stride(0), 2, fmt, 0, n, n, ts_k, d_state.data_ptr(), 1, d_out.data_ptr())
        torch.cuda.synchronize()
        st = _download(d_state)[0]
        assert (st.status, st.ms_done) == (abi.SOFTTRACK_MS_DONE, k)
        pos_k = st.pos
        ts, ots = _settings(system, msToProcess=k + 5)
        for m, rows_want in ((pos_k, k), (pos_k - 1, k - 1)):
            rows, done = _batch(eng, ts, d.data_ptr(), d.stride(0), 2, fmt, m, [c], [r])
            _check_against_oracle(rows, done, [c], [r], d, fmt, m, ots, ms_each=[rows_want])
            assert _same_bytes(rows[0, : k - 1], d_out[0, : k - 1].cpu().numpy())
            d_state = _states(ts, [c], [r], 2)
            d_out2 = torch.full((1, k + 5, 13), np.nan, dtype=torch.float64, device="cuda")
            eng.resume_device(d.data_ptr(), d.stride(0), 2, fmt, 0, m, m, ts, d_state.data_ptr(), 1, d_out2.data_ptr())
            torch.cuda.synchronize()
            s2 = _download(d_state)[0]
            assert (s2.status, s2.ms_done) == (abi.SOFTTRACK_RECORD_END, rows_want), (system, m)


def _per_100ms(res, ora):
    """The largest deviation of each field from the oracle in every 100 ms of a run, for a failing comparison."""
    lines = []
    scale = _tol_scale(ora)
    for a in range(0, len(ora["I_P"]), 100):
        b = a + 100
        sums = max(np.max(np.abs(res[f][a:b] - ora[f][a:b])) for f in SUMS) / scale
        freq = max(np.max(np.abs(res[f][a:b] - ora[f][a:b])) for f in ("carrFreq", "codeFreq"))
        disc = max(np.max(np.abs(res[f][a:b] - ora[f][a:b])) for f in ("dllDiscr", "dllDiscrFilt", "pllDiscr", "pllDiscrFilt"))
        absd = np.max(np.abs(res["absoluteSample"][a:b] - ora["absoluteSample"][a:b]))
        lines.append(f"{a:5d}-{b:5d} ms: sums {sums:.2e} of scale, freq {freq:.2e} Hz, discr {disc:.2e}, absoluteSample {absd:.2e}")
    return "\n".join(lines)


def test_f_long_run_through_the_host_path():
    """2 s of GLONASS FCH +6 and GPS PRN 32 on packed host records, one gnssb200_softtrack_batch_host call per system
    with the automatic window (2^20 samples: about 30 window boundaries), against the oracle over all 2000 periods."""
    from oracle import softtrack_oracle as so
    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine

    fmt = abi.FMT_PACKED2
    ms = 2000
    n = P * (ms + 3)
    recs = [[_glo(6, 3100.0, 222.2, 51)], [_gps(32, -3700.0, 404.4, 52)]]
    eng = SoftTrackingEngine()
    d = _synth(eng.h, recs, n, fmt, seed=111)
    h = d.cpu().numpy()
    assert n // ((1 << 20) - 2 * P) >= 28
    for r, system in enumerate(("glonass", "gps")):
        ts, ots = _settings(system, msToProcess=ms)
        chans = [[], []]
        chans[r] = [_channel(recs[r][0])]
        got = []
        for nt in WIDTHS:
            eng.set_width(nt)
            res = eng.tracking_batch_host(h, d.stride(0), 2, n, chans, ts, fmt=fmt, window_samples=0)
            assert eng.host_stopped == 0
            got.append(res[r][0])
        eng.set_width(0)
        assert all(_same_bytes(got[0][f], got[1][f]) for f in abi.SOFTTRACK_FIELDS)
        ora = so.tracking(_oracle_iq(d, r, fmt, n), chans[r][0], ots)
        try:
            _compare(got[0], ora, ms)
        except AssertionError:
            print(f"{system}: largest deviation from the oracle per 100 ms\n" + _per_100ms(got[0], ora))
            raise


@pytest.mark.parametrize("fmt_name", ["int8", "packed"])
def test_g_positions_past_2_32(fmt_name):
    """States from init with skip_samples = 2^32, resumed window by window from win_first = 2^32 over a small buffer
    that holds record samples 2^32 .. 2^32 + n: rows 0-11 byte-identical to the same record tracked from sample 0, and
    absoluteSample 2^32 larger within one ulp at that magnitude.  One packed channel starts on an odd sample."""
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine

    fmt = _fmt(fmt_name)
    ms = 60
    n = P * (ms + 3)
    big = 1 << 32
    recs = [[_glo(-6, 1500.0, 100.0, 61), _glo(4, -800.0, 300.0, 62)], [_gps(2, 2500.0, 50.5, 63)]]
    eng = SoftTrackingEngine()
    d = _synth(eng.h, recs, n, fmt, seed=113)
    stride = d.stride(0)
    W, A = 5 * P + 1234, 3 * P + 1234
    for system, channel, chan_record in (("glonass", [_channel(s) for s in recs[0]], [0, 0]), ("gps", [_channel(recs[1][0])], [1])):
        if fmt == abi.FMT_PACKED2:
            channel[0]["codePhase"] += channel[0]["codePhase"] % 2  # pos = skip + codePhase - 1 odd
        ts, _ = _settings(system, msToProcess=ms)
        ref_rows, ref_done = _batch(eng, ts, d.data_ptr(), stride, 2, fmt, n, channel, chan_record)
        assert (ref_done == ms).all()
        ts_hi, _ = _settings(system, msToProcess=ms, skipNumberOfSamples=big)
        d_state = _states(ts_hi, channel, chan_record, 2)
        st0 = _download(d_state)
        assert [s.pos for s in st0] == [big + c["codePhase"] - 1 for c in channel]
        if fmt == abi.FMT_PACKED2:
            assert st0[0].pos % 2 == 1
        d_out = torch.full((len(channel), ms, 13), np.nan, dtype=torch.float64, device="cuda")
        first, k = 0, 0
        while True:
            length = min(W, n - first)
            eng.set_width(WIDTHS[k % 2])
            off = 2 * first if fmt == abi.FMT_INT8_IQ else first // 2
            eng.resume_device(d.data_ptr() + off, stride, 2, fmt, big + first, length, big + n, ts_hi, d_state.data_ptr(),
                              len(channel), d_out.data_ptr())
            if first + W >= n:
                break
            first, k = first + A, k + 1
        torch.cuda.synchronize()
        eng.set_width(0)
        assert k >= 10
        st = _download(d_state)
        assert [s.ms_done for s in st] == [ms] * len(channel)
        rows = d_out.cpu().numpy()
        assert _same_bytes(rows[:, :, :12], ref_rows[:, :, :12])
        hi, lo = rows[:, :, 12], ref_rows[:, :, 12]
        assert (np.abs((hi - big) - lo) <= np.spacing(hi)).all()
        assert all(s.pos > big for s in st)


def test_h_refusals_launch_nothing():
    """Spacings 0.5 + 2^-40, 1.0, -0.1 and NaN on every float-tracking call; int8 I,Q records at an odd address or with
    an odd stride on the device calls of float tracking and FFT acquisition.  Each returns < 0, launches no kernel and
    leaves the outputs' sentinel and the states as they were.  Packed records may start at any byte: at an odd address
    with an odd stride they give the bytes of the aligned copy."""
    import torch

    from gnss_sdr_ru_b200 import abi
    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine, Settings
    from gnss_sdr_ru_b200.lib import lib
    from gnss_sdr_ru_b200.softtrack import SoftTrackingEngine

    L = lib()
    ms = 10
    n = P * 12
    recs = [[_glo(1, 500.0, 10.0, 71)], [_glo(2, 700.0, 20.0, 72)]]
    eng = SoftTrackingEngine()
    d = _synth(eng.h, recs, n, abi.FMT_INT8_IQ, seed=115)
    stride = d.stride(0)
    channel = [_channel(recs[0][0]), _channel(recs[1][0])]
    ch, rec = _tables(channel, [0, 1])
    glo, _ = _settings("glonass", msToProcess=ms)
    ok = glo.to_c()
    d_state = _states(glo, channel, [0, 1], 2)
    state0 = d_state.clone()
    d_out = torch.full((2, ms, 13), -7.5, dtype=torch.float64, device="cuda")
    d_done = torch.full((2,), -3, dtype=torch.int32, device="cuda")
    h_iq = d.cpu().numpy()
    h_out = np.full((2, ms, 13), -7.5)
    h_done = np.full(2, -3, dtype=np.int32)
    hs = (abi.SoftTrackState * 2)()
    C.memset(hs, 0x5A, C.sizeof(hs))
    hs0 = bytes(hs)
    eng.set_width(0)
    L.gnssb200_softtrack_batch(eng.h, C.byref(ok), d.data_ptr(), stride, 2, abi.FMT_INT8_IQ, n, ch, rec, 2, d_out.data_ptr(),
                               d_done.data_ptr(), None)  # builds the chip table: later refusals allocate nothing either
    torch.cuda.synchronize()
    d_out.fill_(-7.5)
    d_done.fill_(-3)

    def untouched():
        torch.cuda.synchronize()
        return (torch.equal(d_state, state0) and (d_out == -7.5).all().item() and (d_done == -3).all().item()
                and (h_out == -7.5).all() and (h_done == -3).all() and bytes(hs) == hs0)

    def single(cfg=ok, iq=d.data_ptr()):
        return L.gnssb200_softtrack(eng.h, C.byref(cfg), iq, n, ch, 1, d_out.data_ptr(), d_done.data_ptr(), None)

    def batch(cfg=ok, iq=d.data_ptr(), s=stride, fmt=abi.FMT_INT8_IQ):
        return L.gnssb200_softtrack_batch(eng.h, C.byref(cfg), iq, s, 2, fmt, n, ch, rec, 2, d_out.data_ptr(), d_done.data_ptr(), None)

    def resume(cfg=ok, win=d.data_ptr(), s=stride, fmt=abi.FMT_INT8_IQ):
        return L.gnssb200_softtrack_resume(eng.h, C.byref(cfg), win, s, 2, fmt, 0, n, n, d_state.data_ptr(), 2, d_out.data_ptr(), None)

    def host(cfg=ok):
        return L.gnssb200_softtrack_batch_host(eng.h, C.byref(cfg), h_iq.ctypes.data, stride, 2, abi.FMT_INT8_IQ, n, ch, rec, 2,
                                               h_out.ctypes.data, h_done.ctypes.data, 0)

    def init(cfg=ok):
        return L.gnssb200_softtrack_init(C.byref(cfg), ch, rec, 2, 2, hs)

    def refused(want, call, **kw):
        launches = L.gnssb200_launch_count(eng.h)
        rc = call(**kw)
        assert rc == want, (call.__name__, kw, rc)
        assert L.gnssb200_launch_count(eng.h) == launches, (call.__name__, kw)
        assert untouched(), (call.__name__, kw)

    for spc in (0.5 + 2.0 ** -40, 1.0, -0.1, float("nan")):
        for system in ("glonass", "gps"):
            cfg = _settings(system, msToProcess=ms, dllCorrelatorSpacing=spc)[0].to_c()
            for call in (single, batch, resume, host, init):
                refused(-20, call, cfg=cfg)
    refused(-23, single, iq=d.data_ptr() + 1)
    refused(-23, batch, iq=d.data_ptr() + 1)
    refused(-23, batch, s=stride + 1)
    refused(-23, resume, win=d.data_ptr() + 1)
    refused(-23, resume, s=stride + 1)

    # FFT acquisition: the single and the batched search
    aeng = AcquisitionEngine(handle=eng.h)
    ast = Settings.gps(acqSearchBand=4.0, acqCohIntegration=1, acqSatelliteList=[3, 7])
    acfg = ast.to_c(0, 0)
    na = 16000 * 2
    rows_a = torch.full((2 * 2 * aeng.num_bins(ast) * 16,), 0xAB, dtype=torch.uint8, device="cuda")
    for call in (lambda: L.gnssb200_acq_search(eng.h, C.byref(acfg), d.data_ptr() + 1, abi.FMT_INT8_IQ, na, rows_a.data_ptr(), None),
                 lambda: L.gnssb200_acq_search_batch(eng.h, C.byref(acfg), d.data_ptr() + 1, stride, 2, abi.FMT_INT8_IQ, na,
                                                     rows_a.data_ptr(), None),
                 lambda: L.gnssb200_acq_search_batch(eng.h, C.byref(acfg), d.data_ptr(), 2 * na + 1, 2, abi.FMT_INT8_IQ, na,
                                                     rows_a.data_ptr(), None)):
        launches = L.gnssb200_launch_count(eng.h)
        assert call() == -15
        torch.cuda.synchronize()
        assert L.gnssb200_launch_count(eng.h) == launches and (rows_a == 0xAB).all().item()

    # the valid forms: spacing 0.5 and 0 run; packed records at an odd address with an odd stride are read as they are
    for spc in (0.0, 0.5):
        assert batch(cfg=_settings("glonass", msToProcess=ms, dllCorrelatorSpacing=spc)[0].to_c()) == 0
    dp = _synth(eng.h, recs, n, abi.FMT_PACKED2, seed=117)
    row = dp.stride(0)
    odd = torch.zeros(1 + 2 * (row + 1), dtype=torch.uint8, device="cuda")
    for r in range(2):
        odd[1 + r * (row + 1) : 1 + r * (row + 1) + row] = dp[r]
    aligned = _batch(eng, glo, dp.data_ptr(), row, 2, abi.FMT_PACKED2, n, channel, [0, 1])
    shifted = _batch(eng, glo, odd.data_ptr() + 1, row + 1, 2, abi.FMT_PACKED2, n, channel, [0, 1])
    assert (aligned[1] == ms).all() and np.array_equal(aligned[1], shifted[1]) and _same_bytes(aligned[0], shifted[0])
    rows_b = torch.zeros_like(rows_a)
    rows_c = torch.zeros_like(rows_a)
    assert L.gnssb200_acq_search_batch(eng.h, C.byref(acfg), dp.data_ptr(), row, 2, abi.FMT_PACKED2, na, rows_b.data_ptr(), None) == 0
    assert L.gnssb200_acq_search_batch(eng.h, C.byref(acfg), odd.data_ptr() + 1, row + 1, 2, abi.FMT_PACKED2, na,
                                       rows_c.data_ptr(), None) == 0
    torch.cuda.synchronize()
    assert torch.equal(rows_b, rows_c) and (rows_b != 0).any().item()
