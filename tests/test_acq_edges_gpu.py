"""FFT acquisition at its edges against the float64 restatement of acquisition.sci (oracle/pcps_oracle.py).

The records are built here so that the answer is known: A*roll(c, p) + B*roll(c, p + delta) on the carrier of one
Doppler bin, plus Gaussian noise, rounded and clipped to int8, with c the oracle's own sampled code.  By the circular
cross-correlation identity the peak of that bin's row is at 0-based code phase p, and the echo B sits on the boundary
of the second-peak window: delta = +-chip is inside it, delta = +-(chip - 1) just outside.  Peaks are placed at both
ends of the code period, including the three positions where the reference's exclusion range leaves 1..N
(undefined="circular" in the oracle, the library's definition).  Further cases: packed input, records at batch index
> 0, the first and last Doppler bins (also at 3 ms, whose 166.67 Hz bins fall into 6 frequency classes), the
best-of-two-blocks rule with equal block maxima, full-scale and clipped input, an all-zero record, and the hand-off of
edge results into the tracking channels.

Tolerances as in tests/test_acq_gpu.py: every row's peak and second within 1e-4 relative; code phase and block exact
(in a row other than the one the result is taken from, a different code phase or block is accepted only where two
maxima tie within FP32 noise); bin, code phases, frequency channel and carrier exact; peakMetric within 1e-4.
"""
import numpy as np
import pytest

from gnss_sdr_ru_b200 import abi

pytestmark = pytest.mark.gpu
RTOL = 1e-4
TIE = 1e-5  # two maxima closer than this (relative) may come out in either order from the FP32 path
N = 16000


def _po():
    from oracle import pcps_oracle as po

    return po


def _chip(system):
    return 16 if system == "gps" else 31


def _positions(chip):
    return [0, 1, chip - 2, chip - 1, chip, chip + 1, N // 2, N - chip - 2, N - chip - 1, N - chip, N - 2, N - 1]


def _settings(system, sv_list, band, coh, n_noncoh=0):
    """(library settings, oracle settings) of the same search."""
    from gnss_sdr_ru_b200.acquisition import Settings

    po = _po()
    if system == "gps":
        return (Settings.gps(acqSearchBand=band, acqCohIntegration=coh, acqSatelliteList=list(sv_list), n_noncoh=n_noncoh),
                po.AcqSettings.gps(acqSearchBand=band, acqCohIntegration=coh, svList=list(sv_list), n_noncoh=n_noncoh))
    return (Settings.glonass(acqSearchBand=band, acqCohIntegration=coh, acqSatelliteList=list(sv_list), n_noncoh=n_noncoh),
            po.AcqSettings.glonass(acqSearchBand=band, acqCohIntegration=coh, svList=list(sv_list), n_noncoh=n_noncoh))


def _signal(os_, sv, p, k1, n_ms, A=40.0, delta=None, B=20.0):
    """A*roll(c, p) (+ B*roll(c, p + delta)) on the carrier of Doppler bin k1 (1-based), n_ms periods.  The wipe-off
    multiplies by exp(+i*2*pi*f*t) (acquisition.sci), so the carrier is exp(-i*2*pi*f*t), as synth.make_record has it."""
    po = _po()
    c = po.sampled_code(os_, sv)
    one = A * np.roll(c, p)
    if delta is not None:
        one = one + B * np.roll(c, (p + delta) % N)
    n = np.arange(n_ms * N)
    return np.tile(one, n_ms) * np.exp(-2j * np.pi * po.bin_freq(os_, sv, k1) * n / os_.samplingFreq)


def _int8(x, sigma=4.0, seed=0):
    """x + complex Gaussian noise (sigma per component), rounded and clipped to int8 interleaved I,Q."""
    rng = np.random.default_rng(seed)
    x = x + sigma * (rng.standard_normal(x.size) + 1j * rng.standard_normal(x.size))
    iq = np.empty(2 * x.size, dtype=np.int8)
    iq[0::2] = np.clip(np.rint(x.real), -128, 127)
    iq[1::2] = np.clip(np.rint(x.imag), -128, 127)
    return iq


def _four_level(iq):
    """int8 I,Q quantised to +-1 / +-3 (threshold: the rms of the record), the values the packed format holds."""
    v = iq.astype(np.float64)
    t = np.sqrt(np.mean(v * v))
    return (np.where(np.abs(v) > t, 3, 1) * np.where(v >= 0, 1, -1)).astype(np.int8)


def _gpu_batch(st, recs, fmt=abi.FMT_INT8_IQ):
    """acquisition_batch of records laid end to end in one device buffer (record r at index r)."""
    import torch

    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine
    from gnss_sdr_ru_b200.synth import pack2

    bufs = [pack2(r) if fmt == abi.FMT_PACKED2 else r.view(np.uint8) for r in recs]
    stride = bufs[0].size
    n = recs[0].size // 2
    d = torch.from_numpy(np.concatenate(bufs)).cuda()
    eng = AcquisitionEngine()
    return eng.acquisition_batch(d.data_ptr(), stride, len(recs), n, st, fmt=fmt, return_rows=True)


def _oracle(iq, os_):
    po = _po()
    return po.acquisition(po.to_complex(iq), os_, undefined="circular")


def _compare(res, ora, where=""):
    """GPU result dict (with rows) against the oracle's list, every row.  `where` names the case in a failure."""
    rows = res["rows"]
    for i, o in enumerate(ora):
        for key in ("bin", "codePhaseRaw", "codePhase", "freqChannel"):
            assert int(res[key][i]) == o[key], (where, key, i, res[key][i], o[key])
        assert res["carrFreq"][i] == o["carrFreq"], (where, i, res["carrFreq"][i], o["carrFreq"])
        assert abs(res["peakMetric"][i] - o["peakMetric"]) <= RTOL * o["peakMetric"], (where, i, res["peakMetric"][i], o["peakMetric"])
        assert abs(res["peak"][i] - o["peak"]) <= RTOL * o["peak"], (where, i, res["peak"][i], o["peak"])
        assert abs(res["second"][i] - o["second"]) <= RTOL * o["second"], (where, i, res["second"][i], o["second"])
        for k1, (pk, arg, blk) in o["rows"].items():
            g = rows[i, k1 - 1]
            assert abs(g["peak"] - pk) <= RTOL * pk, (where, i, k1, g["peak"], pk)
            strict = k1 == o["bin"]  # the row the result is taken from: no escape
            bm = o["row_block_max"][k1]
            cp_same = int(g["code_phase"]) == arg
            blk_same = int(g["block"]) == blk
            assert cp_same or (not strict and abs(g["peak"] - pk) <= 1e-6 * pk), (where, i, k1, g, arg)
            assert blk_same or (not strict and len(bm) == 2 and abs(bm[0] - bm[1]) <= TIE * max(bm)), (where, i, k1, g, blk, bm)
            if cp_same and blk_same:
                s2 = o["row_second"][k1]
                assert abs(g["second"] - s2) <= RTOL * s2, (where, i, k1, g["second"], s2)


def _window_second(row, p, d_min):
    d = np.abs(np.arange(N) - p)
    return float(row[np.minimum(d, N - d) >= d_min].max())


def _assert_sensitive(iq, os_, sv, k1, p, delta, chip, second):
    """The case proves something only if moving the window edge by one sample across the echo changes the second by
    far more than the tolerance: the echo at +-chip leaves a window of distance >= chip + 1, the echo at +-(chip - 1)
    enters one of distance >= chip - 1."""
    po = _po()
    row = po.acquisition_rows(po.to_complex(iq), os_, sv, bins=[k1])[1][k1]
    assert _window_second(row, p, chip) == second
    moved = _window_second(row, p, chip + 1 if abs(delta) == chip else chip - 1)
    assert abs(moved - second) > 100 * RTOL * second, (p, delta, moved, second)


# ---- peaks at the ends of the code period, echo on the window boundary ------------------------------------------------
EDGE_CASES = [("gps", 1), ("gps", 32), ("glonass", -7), ("glonass", 6)]
DELTAS = ["+chip", "-chip", "+chip-1", "-chip+1"]


def _delta(kind, chip):
    return {"+chip": chip, "-chip": -chip, "+chip-1": chip - 1, "-chip+1": -(chip - 1)}[kind]


def _edge_records(system, sv, kind, four_level=False):
    """One record per edge position (12), the signal of `sv` in a bin that moves with the position."""
    chip = _chip(system)
    delta = _delta(kind, chip)
    if system == "gps":
        sv_list, band, coh = [1, 32], 2.0, 1  # 5 bins of 500 Hz
    else:
        sv_list, band, coh = [-7, 6], 1.0, 5  # stock 5 ms, 11 bins of 100 Hz
    st, os_ = _settings(system, sv_list, band, coh)
    nb = _po().num_bins(os_)
    cases, recs = [], []
    for j, p in enumerate(_positions(chip)):
        k1 = 1 + j % nb
        iq = _int8(_signal(os_, sv, p, k1, 2 * coh, delta=delta), seed=1000 * j + chip + sv)
        recs.append(_four_level(iq) if four_level else iq)
        cases.append((p, k1))
    return st, os_, sv_list.index(sv), delta, chip, cases, recs


def _check_edge_batch(system, sv, kind, fmt):
    st, os_, i_sv, delta, chip, cases, recs = _edge_records(system, sv, kind, four_level=fmt == abi.FMT_PACKED2)
    outs = _gpu_batch(st, recs, fmt)
    assert len(outs) == len(recs)
    for (p, k1), iq, res in zip(cases, recs, outs):
        ora = _oracle(iq, os_)
        o = ora[i_sv]
        assert (o["bin"], o["codePhaseRaw"], o["freqChannel"]) == (k1, p + 1, sv), (p, k1, o["bin"], o["codePhaseRaw"])
        _assert_sensitive(iq, os_, sv, k1, p, delta, chip, o["second"])
        _compare(res, ora, where=f"peak at 0-based {p}, echo at {delta:+d}, bin {k1}")


@pytest.mark.parametrize("kind", DELTAS)
@pytest.mark.parametrize("system,sv", EDGE_CASES)
def test_edge_positions_int8_batched(oracle_lib, system, sv, kind):
    """All 12 edge positions as one batched search (R = 12): GPS 1 ms / 5 bins, GLONASS stock 5 ms / 11 bins."""
    _check_edge_batch(system, sv, kind, abi.FMT_INT8_IQ)


@pytest.mark.parametrize("kind", DELTAS)
@pytest.mark.parametrize("system,sv", [("gps", 1), ("glonass", -7)])
def test_edge_positions_packed(oracle_lib, system, sv, kind):
    """The same positions quantised to +-1 / +-3 and searched in the packed 2+2-bit format."""
    _check_edge_batch(system, sv, kind, abi.FMT_PACKED2)


def test_edge_positions_gps_stock_settings(oracle_lib):
    """Stock GPS settings (4 ms coherent, 14 kHz, 113 bins) at both ends of the period, single-record host call."""
    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine

    chip = 16
    st, os_ = _settings("gps", [32], 14.0, 4)
    eng = AcquisitionEngine()
    for j, (p, delta) in enumerate([(0, chip), (chip, -chip), (chip, -(chip - 1)), (N - chip - 1, chip - 1),
                                    (N - 1, -chip), (N - 1, chip - 1)]):
        k1 = [1, 57, 113][j % 3]
        iq = _int8(_signal(os_, 32, p, k1, 8, delta=delta), seed=77 + j)
        res = eng.acquisition(iq, st, return_rows=True)
        ora = _oracle(iq, os_)
        assert (ora[0]["bin"], ora[0]["codePhaseRaw"]) == (k1, p + 1)
        _assert_sensitive(iq, os_, 32, k1, p, delta, chip, ora[0]["second"])
        _compare(res, ora)


# ---- Doppler grid edges -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_noncoh", [0, 3])
def test_gps_3ms_first_and_last_bin(oracle_lib, n_noncoh):
    """3 ms over 7 kHz: 43 bins of 166.67 Hz (6 frequency classes); PRN 3 in bin 1, PRN 19 in bin 43, where the
    circular shift of the base spectrum is largest.  Stock best-of-two and 3 ms x 3 non-coherent."""
    st, os_ = _settings("gps", [3, 19, 24], 7.0, 3, n_noncoh=n_noncoh)
    assert _po().num_bins(os_) == 43
    n_ms = 3 * (3 if n_noncoh else 2)
    x = _signal(os_, 3, 1234, 1, n_ms, A=25.0) + _signal(os_, 19, 15000, 43, n_ms, A=25.0)
    iq = _int8(x, sigma=6.0, seed=3)
    res = _gpu_batch(st, [iq])[0]
    ora = _oracle(iq, os_)
    assert [(o["bin"], o["codePhaseRaw"], o["freqChannel"]) for o in ora[:2]] == [(1, 1235, 3), (43, 15001, 19)]
    assert ora[2]["freqChannel"] == 0
    _compare(res, ora)


def test_glonass_first_and_last_bin(oracle_lib):
    """Stock GLONASS (5 ms, 12 kHz, 121 bins): FCH -7 in its first bin, FCH +6 in its last."""
    st, os_ = _settings("glonass", [-7, 0, 6], 12.0, 5)
    x = _signal(os_, -7, 3000, 1, 10, A=25.0) + _signal(os_, 6, 11000, 121, 10, A=25.0)
    iq = _int8(x, sigma=6.0, seed=5)
    res = _gpu_batch(st, [iq])[0]
    ora = _oracle(iq, os_)
    assert [(o["bin"], o["codePhaseRaw"], o["freqChannel"]) for o in (ora[0], ora[2])] == [(1, 3001, -7), (121, 11001, 6)]
    _compare(res, ora)


# ---- best of two blocks ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("flip,want", [(None, 1), (0, 1), (1, 0)])
def test_block_rule(oracle_lib, flip, want):
    """Stock mode keeps block 0 only if its maximum is strictly larger (acquisition.sci:130).  Bit-identical blocks:
    both sides keep block 1 in every row.  A sign flip in the middle of a block: the other block is kept."""
    st, os_ = _settings("gps", [5], 2.0, 1)
    x = _signal(os_, 5, 5000, 3, 1)
    rng = np.random.default_rng(11)
    x = x + 4.0 * (rng.standard_normal(N) + 1j * rng.standard_normal(N))
    x = np.tile(x, 2)
    if flip is not None:
        x[flip * N + N // 2 : (flip + 1) * N] *= -1
    iq = _int8(x, sigma=0.0)
    res = _gpu_batch(st, [iq])[0]
    ora = _oracle(iq, os_)
    assert ora[0]["rows"][3][2] == want and int(res["rows"][0, 2]["block"]) == want
    if flip is None:
        assert all(r[2] == 1 for r in ora[0]["rows"].values())
        assert (res["rows"]["block"] == 1).all()
    _compare(res, ora)


# ---- full scale ------------------------------------------------------------------------------------------------------------
def test_full_scale_clipped_noncoherent(oracle_lib):
    """C4 shape (10 ms x 20 non-coherent) over 1 kHz (21 bins), a signal far beyond int8 hard-clipped to [-128, 127]."""
    st, os_ = _settings("gps", [22], 1.0, 10, n_noncoh=20)
    assert _po().num_bins(os_) == 21
    iq = _int8(_signal(os_, 22, 9876, 7, 200, A=300.0), sigma=20.0, seed=9)
    assert (iq == -128).any() and (iq == 127).any() and np.mean(np.abs(iq.astype(int)) >= 127) > 0.3
    res = _gpu_batch(st, [iq])[0]
    ora = _oracle(iq, os_)
    assert (ora[0]["bin"], ora[0]["codePhaseRaw"]) == (7, 9877)
    _compare(res, ora)


def test_full_scale_clipped_1ms(oracle_lib):
    """The same at 1 ms (5 bins of 500 Hz), -128 in both I and Q."""
    st, os_ = _settings("gps", [22, 23], 2.0, 1)
    iq = _int8(_signal(os_, 22, 15990, 2, 2, A=300.0), sigma=20.0, seed=10)
    assert (iq[0::2] == -128).any() and (iq[1::2] == -128).any() and (iq == 127).any()
    res = _gpu_batch(st, [iq])[0]
    ora = _oracle(iq, os_)
    assert (ora[0]["bin"], ora[0]["codePhaseRaw"]) == (2, 15991)
    _compare(res, ora)


# ---- all-zero record -------------------------------------------------------------------------------------------------------
def test_zero_record_is_not_detected(oracle_lib):
    """Peak and second are 0, so peakMetric is 0/0 = NaN on both sides, and NaN is not above the threshold: nothing is
    detected, and the hand-off allocates no channel (every channel off, as the restatement in test_acq_allocate has it)."""
    from test_acq_allocate import _restated, _results, _rx_bytes

    from gnss_sdr_ru_b200.receiver import TrackingEngine

    st, os_ = _settings("gps", [1, 32], 2.0, 1)
    iq = np.zeros(2 * 2 * N, dtype=np.int8)
    res = _gpu_batch(st, [iq])[0]
    with np.errstate(invalid="ignore", divide="ignore"):
        ora = _oracle(iq, os_)
    for i, o in enumerate(ora):
        assert np.isnan(res["peakMetric"][i]) and np.isnan(o["peakMetric"])
        assert int(res["freqChannel"][i]) == 0 == o["freqChannel"]
        assert int(res["codePhase"][i]) == 0 == o["codePhase"] and res["carrFreq"][i] == 0.0 == o["carrFreq"]
        assert (int(res["bin"][i]), int(res["codePhaseRaw"][i])) == (o["bin"], o["codePhaseRaw"]) == (1, 1)
        assert res["peak"][i] == 0.0 == o["peak"] and res["second"][i] == 0.0 == o["second"]
    assert (res["rows"]["peak"] == 0).all() and (res["rows"]["second"] == 0).all()
    eng = TrackingEngine(n_streams=1)
    assert eng.acq_allocate(0, res, st) == []
    entries = [(float(res["carrFreq"][i]), int(res["codePhase"][i]), float(res["peakMetric"][i])) for i in range(2)]
    want_rx, want_sv = _restated(oracle_lib, {}, st, _results(entries))
    assert want_sv == [0] * abi.N_CHANNELS
    assert _rx_bytes(eng.rx[0]) == _rx_bytes(want_rx)
    assert all(eng.rx[0].reg_write[ch << 3] == 0 for ch in range(abi.N_CHANNELS))
    eng.close()


# ---- hand-off of edge results ---------------------------------------------------------------------------------------------
def test_handoff_of_edge_results(oracle_lib):
    """GPU results with peaks at P = 1, P = N and P = 17 (GPS; the reference's exclusion range leaves 1..N there)
    started as channels: the receiver is byte-identical to the restatement in tests/test_acq_allocate.py."""
    from test_acq_allocate import _restated, _results, _rx_bytes

    from gnss_sdr_ru_b200.receiver import TrackingEngine

    st, os_ = _settings("gps", [1, 7, 32], 2.0, 1)
    x = _signal(os_, 1, 0, 2, 2, A=25.0) + _signal(os_, 7, 16, 5, 2, A=25.0) + _signal(os_, 32, N - 1, 1, 2, A=25.0)
    iq = _int8(x, sigma=6.0, seed=12)
    res = _gpu_batch(st, [iq])[0]
    ora = _oracle(iq, os_)
    assert [o["codePhase"] for o in ora] == [1, 17, N]
    _compare(res, ora)
    eng = TrackingEngine(n_streams=1)
    sv = eng.acq_allocate(0, res, st)
    assert sorted(sv) == [1, 7, 32]
    entries = [(float(res["carrFreq"][i]), int(res["codePhase"][i]), float(res["peakMetric"][i])) for i in range(3)]
    want_rx, want_sv = _restated(oracle_lib, {}, st, _results(entries))
    assert sv == want_sv[:3]
    assert _rx_bytes(eng.rx[0]) == _rx_bytes(want_rx)
    eng.close()
