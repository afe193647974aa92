"""The NumPy restatement of acquisition.sci: regression against its committed fixture and checks of the
rules it restates (bin grid, sampled code, exclusion ranges).  Parity of this path is unpinned by any
reference output (oracle/pcps_oracle.py header)."""
import os

import numpy as np

from gnss_sdr_ru_b200.synth import unpack2

HERE = os.path.dirname(os.path.abspath(__file__))


def test_grid_and_code_rules(oracle_lib):
    from oracle import pcps_oracle as po

    g = po.AcqSettings.glonass()
    assert po.samples_per_code(g) == 16000 and po.num_bins(g) == 121  # SURVEY 8a S1
    assert po.bin_freq(g, -7, 1) == 1e6 - 7 * 562500 - 6000 and po.bin_freq(g, 6, 121) == 1e6 + 6 * 562500 + 6000
    s = po.AcqSettings.gps(acqSearchBand=20.0, acqCohIntegration=1)
    assert po.num_bins(s) == 41 and po.bin_freq(s, 1, 1) == 2.42e6 - 10000 and po.bin_freq(s, 1, 41) == 2.42e6 + 10000
    w = po.AcqSettings.gps(acqSearchBand=20.0, acqCohIntegration=10, n_noncoh=20)
    assert po.num_bins(w) == 401 and po.samples_needed(w) == 200 * 16000
    c = po.sampled_code(s, 1)
    assert c.shape == (16000,) and set(np.unique(c)) == {-1.0, 1.0}
    # 16000/1023 = 15.64 samples per chip: first chip covers samples 0..14 (ceil rule), last sample = chip 1023
    from gnss_sdr_ru_b200.codes import ca_code

    assert (c[:15] == ca_code(1)[0]).all() and c[15] == ca_code(1)[1] and c[-1] == ca_code(1)[1022]


def test_exclusion_ranges(oracle_lib):
    from oracle import pcps_oracle as po

    s = po.AcqSettings.gps()
    n = 16000
    r = po.exclusion_range(s, 5000)
    assert r[0] == 1 and 4984 in r and 4985 not in r and 5015 not in r and 5016 in r and r[-1] == n
    r = po.exclusion_range(s, 3)  # e1 < 2: range wraps past the end
    assert r[0] == 19 and r[-1] == n + 3 - 16
    r = po.exclusion_range(s, 15990)  # e2 > n
    assert r[0] == 15990 + 16 - n and r[-1] == 15990 - 16
    g = po.AcqSettings.glonass()
    assert po.exclusion_range(g, 5000)[-1] == n and 5031 in po.exclusion_range(g, 5000) and 5030 not in po.exclusion_range(g, 5000)


def test_second_peak_window_is_the_reference_range_except_at_three_positions(oracle_lib):
    """For every peak position P of both systems, the circular window (distance >= chip) equals the reference's
    exclusion range, except at the three positions where that range leaves 1..N (Scilab stops there; this library
    defines them by the circular rule).  A change of either rule shows up in the list below."""
    from oracle import pcps_oracle as po

    n = 16000
    undefined = []
    for s in (po.AcqSettings.gps(), po.AcqSettings.glonass()):
        chip = 16 if s.system == "gps" else 31
        for P in range(1, n + 1):
            w = po.second_peak_window(s, P)
            r = po.exclusion_range(s, P)
            if r.min() < 1 or r.max() > n:
                undefined.append((s.system, P))
                assert len(r) == len(w) and not np.array_equal(r, w)  # the same count, one index outside 1..N
            else:
                assert np.array_equal(np.sort(r), w), (s.system, P)
            assert len(w) == n - 2 * chip + 1
    assert undefined == [("gps", 17), ("glonass", 32), ("glonass", 15969)]


def test_undefined_positions_raise_or_follow_the_circular_rule(oracle_lib):
    """A peak at GPS P = 17 raises by default, as the reference does; undefined="circular" gives the second peak
    over second_peak_window, which holds sample 1 (circular distance 16 from the peak)."""
    import pytest

    from oracle import pcps_oracle as po

    s = po.AcqSettings.gps(acqSearchBand=1.0, acqCohIntegration=1, svList=[1])
    c = po.sampled_code(s, 1)
    n = np.arange(2 * 16000)
    # peak at 1-based 17, echo at 1, on the carrier of the middle bin (the wipe-off multiplies by exp(+i*2*pi*f*t))
    x = np.tile(np.roll(c, 16) * 40 + c * 20, 2) * np.exp(-2j * np.pi * s.IF * n / s.samplingFreq)
    with pytest.raises(IndexError):
        po.acquisition(x, s)
    r = po.acquisition(x, s, undefined="circular")[0]
    assert r["codePhaseRaw"] == 17
    full = po.acquisition_rows(x, s, 1)[1][r["bin"]]
    assert r["second"] == full[0] and r["second"] == max(full[po.second_peak_window(s, 17) - 1])
    assert r["row_second"][r["bin"]] == r["second"]


def test_oracle_regression_fixture(oracle_lib):
    from oracle import pcps_oracle as po

    g = np.load(os.path.join(HERE, "golden", "acq_golden.npz"))
    rec = unpack2(g["packed"])
    s = po.AcqSettings.gps(acqSearchBand=float(g["band"]), acqCohIntegration=int(g["coh"]), svList=[int(x) for x in g["sv"]])
    res = po.acquisition(po.to_complex(rec), s)
    assert [r["bin"] for r in res] == [int(x) for x in g["bin"]]
    assert [r["codePhaseRaw"] for r in res] == [int(x) for x in g["codePhaseRaw"]]
    assert np.allclose([r["peakMetric"] for r in res], g["peakMetric"], rtol=1e-9)
    assert [r["codePhase"] for r in res] == [int(x) for x in g["codePhase"]]
    assert res[0]["carrFreq"] == float(g["carrFreq"][0]) and res[1]["codePhase"] == 0  # PRN 6 absent -> below threshold
