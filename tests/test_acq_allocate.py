"""gnssb200_rx_acq_allocate: FFT acquisition results -> channels of the integer receiver (host code, no GPU).

Every case builds a result table by hand, runs the library's hand-off on a freshly initialised receiver and compares
the whole gnssb200_rx byte for byte with a restatement of the rule of include/gnssb200.h written out again here on
top of the oracle's own cold_allocate / ch_carrier / ch_code_slew.
"""
import ctypes as C
import math

import numpy as np
import pytest

from gnss_sdr_ru_b200 import abi

G = abi.PRN_GLONASS


def _rx_bytes(rx):
    return bytes(memoryview(rx).cast("B"))


def _round(x):  # llround: halves away from zero
    return int(math.copysign(math.floor(abs(x) + 0.5), x))


def _cfg(**over):
    from gnss_sdr_ru_b200.lib import default_cfg

    return default_cfg(**over)


def _results(entries):
    """entries: (carrFreq, codePhase, peakMetric) per sv of the list."""
    res = (abi.AcqResult * len(entries))()
    for r, (f, cp, m) in zip(res, entries):
        r.carrFreq, r.codePhase, r.peakMetric = f, cp, m
    return res


def _allocate(cfg, settings, res):
    from gnss_sdr_ru_b200.lib import lib

    L = lib()
    rx = abi.Rx()
    L.gnssb200_rx_init(C.byref(rx), C.byref(cfg))
    acq = settings.to_c()
    sv_out = (C.c_int32 * abi.N_CHANNELS)()
    n = L.gnssb200_rx_acq_allocate(C.byref(rx), C.byref(cfg), C.byref(acq), res, sv_out)
    return n, rx, list(sv_out)


def _restated(oracle_lib, cfg_over, settings, res):
    """The hand-off as include/gnssb200.h defines it, on the oracle's register helpers."""
    o = oracle_lib.Oracle(oracle_lib.Oracle.default_cfg(**cfg_over))
    c = o.cfg
    glo = settings.system == "glonass"
    svs = settings.acqSatelliteList
    det = [i for i in range(len(svs)) if res[i].peakMetric > settings.acqThreshold]
    det = sorted(det, key=lambda i: -res[i].peakMetric)[:12]  # sorted() is stable: ties keep list order
    o.cold_allocate([(G if glo else svs[i]) for i in det] + [0] * (12 - len(det)))
    resol = c.clock_mult * c.samp_rate / 2.0 ** c.carrier_nco_bits
    P = 1022 if glo else 2046
    for ch, i in enumerate(det):
        k = o.rx.chan[ch]
        fch = svs[i] if glo else 0
        if glo:
            k.carrier_cold_corr = fch * int(562500.0 / resol)
        ref = (c.glonass_carrier_ref if glo else c.gps_carrier_ref) + k.carrier_cold_corr
        k.carrier_freq = ref + _round((res[i].carrFreq - settings.IF - fch * settings.L1_IF_step) / resol)
        nf = max(-5, min(5, _round((k.carrier_freq - ref) / c.d_freq)))
        k.n_freq = nf
        k.del_freq = -2 * nf if nf > 0 else 1 - 2 * nf
        o.ch_carrier(ch, k.carrier_freq)
        cell = _round((res[i].codePhase - 1) * 2.0 * settings.codeFreqBasis / settings.samplingFreq) % P
        a = (cell + 1) % P
        o.ch_code_slew(ch, a - 2 if a >= 2 else 0)
        k.codes = 0
    return o.rx, [svs[i] for i in det] + [0] * (12 - len(det))


def _check(oracle_lib, settings, entries, cfg_over=None):
    cfg_over = cfg_over or {}
    res = _results(entries)
    n, rx, sv_out = _allocate(_cfg(**cfg_over), settings, res)
    want_rx, want_sv = _restated(oracle_lib, cfg_over, settings, res)
    assert n == min(12, sum(e[2] > settings.acqThreshold for e in entries))
    assert sv_out == want_sv
    assert _rx_bytes(rx) == _rx_bytes(want_rx)
    return n, rx, sv_out


def _gps(svs):
    from gnss_sdr_ru_b200.acquisition import Settings

    return Settings.gps(acqCohIntegration=1, acqSearchBand=20.0, acqSatelliteList=list(svs))


def test_order_by_peak_metric_with_ties(oracle_lib):
    st = _gps([3, 7, 9, 14, 19, 22])
    entries = [(2.42e6 + 1500.0, 4001, 5.0), (2.42e6 - 2500.0, 9000, 8.0), (2.42e6 + 250.0, 12000, 5.0),
               (2.42e6, 100, 2.0), (2.42e6 - 9500.0, 16000, 8.0), (2.42e6 + 6200.0, 1, 3.5)]
    n, rx, sv = _check(oracle_lib, st, entries)
    assert n == 5 and sv[:5] == [7, 19, 3, 9, 22]
    assert [rx.reg_write[ch << 3] for ch in range(6)] == [7, 19, 3, 9, 22, 0]
    assert rx.chan[3].n_freq == 0 and rx.chan[4].n_freq == 5  # 6.2 kHz: nearest bin clamped to search_max_f


def test_more_than_twelve_detections(oracle_lib):
    rng = np.random.default_rng(3)
    svs = list(range(1, 21))
    st = _gps(svs)
    entries = [(2.42e6 + float(rng.uniform(-9000, 9000)), int(rng.integers(1, 16001)), float(rng.uniform(3.5, 20.0)))
               for _ in svs]
    n, _, sv = _check(oracle_lib, st, entries)
    assert n == 12
    want = [svs[i] for i in np.argsort([-e[2] for e in entries], kind="stable")[:12]]
    assert sv == want


def test_none_detected(oracle_lib):
    st = _gps([1, 2, 3, 4])
    # 3.0 is not > 3.0; NaN (0/0 of an all-zero record) is not either
    n, rx, sv = _check(oracle_lib, st, [(0.0, 0, 1.5), (0.0, 0, 2.9), (0.0, 0, 3.0), (0.0, 0, math.nan)])
    assert n == 0 and sv == [0] * 12
    assert all(rx.reg_write[ch << 3] == 0 for ch in range(12))  # every channel off


def test_glonass_fch_zero_and_minus_seven(oracle_lib):
    from gnss_sdr_ru_b200.acquisition import Settings

    st = Settings.glonass(acqSatelliteList=[-7, -3, 0, 5])
    f = lambda k, fd: 1.0e6 + k * 562500.0 + fd  # noqa: E731
    entries = [(f(-7, -1250.0), 300, 6.0), (f(-3, 0.0), 0, 2.0), (f(0, 2100.0), 15999, 9.0), (f(5, 400.0), 8000, 4.0)]
    n, rx, sv = _check(oracle_lib, st, entries, cfg_over=dict(glonass_carrier_if=1.0e6))
    assert n == 3 and sv[:3] == [0, -7, 5]
    assert all(rx.reg_write[ch << 3] == G for ch in range(3)) and rx.chan[0].system == 1
    assert rx.chan[1].carrier_cold_corr == -7 * 7549747 and rx.chan[0].carrier_cold_corr == 0


@pytest.mark.parametrize("system", ["gps", "glonass"])
def test_code_phase_at_the_period_edges(oracle_lib, system):
    """tau within one chip of 0 and of the end of the period: the search cell wraps modulo P."""
    from gnss_sdr_ru_b200.acquisition import Settings

    cps = [1, 2, 9, 16, 31, 15970, 15985, 15992, 15999, 16000]
    if system == "gps":
        st, over, f0 = _gps(range(1, len(cps) + 1)), {}, 2.42e6
    else:
        st, over, f0 = Settings.glonass(acqSatelliteList=list(range(-5, -5 + len(cps)))), dict(glonass_carrier_if=1.0e6), None
    entries = [((f0 if f0 else 1.0e6 + sv * 562500.0) + 100.0 * i, cp, 10.0 - 0.1 * i)
               for i, (sv, cp) in enumerate(zip(st.acqSatelliteList, cps))]
    _, rx, _ = _check(oracle_lib, st, entries, cfg_over=over)
    slews = [rx.reg_write[(ch << 3) + 0x84] for ch in range(len(cps))]
    P = 2046 if system == "gps" else 1022
    assert all(0 <= s <= P - 3 for s in slews)
    assert slews[0] == 0 and slews[-1] == 0  # chip 0 at sample 0 or one sample before the period's end: no slew


@pytest.mark.parametrize("what", ["samp_freq", "IF", "code_freq", "IF_step", "prn"])
def test_mismatch_is_refused_and_leaves_rx_untouched(what):
    from gnss_sdr_ru_b200.acquisition import Settings
    from gnss_sdr_ru_b200.lib import lib

    L = lib()
    if what == "IF_step":
        st, cfg = Settings.glonass(L1_IF_step=562000.0, acqSatelliteList=[0]), _cfg(glonass_carrier_if=1.0e6)
    else:
        st, cfg = _gps([5]), _cfg()
        if what == "samp_freq":
            st.samplingFreq = 16.368e6
        elif what == "IF":
            st.IF = 4.092e6
        elif what == "code_freq":
            st.codeFreqBasis = 1.0229e6
        else:
            st.acqSatelliteList = [33]
    rx = abi.Rx()
    L.gnssb200_rx_init(C.byref(rx), C.byref(cfg))
    rx.chan[2].state = 4  # anything the call must not touch
    before = _rx_bytes(rx)
    acq = st.to_c()
    assert L.gnssb200_rx_acq_allocate(C.byref(rx), C.byref(cfg), C.byref(acq), _results([(2.42e6, 10, 9.0)]), None) < 0
    assert _rx_bytes(rx) == before
    assert b"gnssb200_rx_acq_allocate" in L.gnssb200_last_error_string()
