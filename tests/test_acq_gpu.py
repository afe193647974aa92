"""GPU parity of the FFT acquisition against the NumPy float64 restatement of acquisition.sci.

Tolerances (north star): argmax (sv, Doppler bin, code phase) exact; floating-point peak metrics
within 1e-4 relative.  The GPU path is FP32 with a different (folded / shifted-spectrum)
formulation, the oracle is the reference's own formulation in float64.
"""
import numpy as np
import pytest

from gnss_sdr_ru_b200 import abi

pytestmark = pytest.mark.gpu
RTOL = 1e-4


def _check(res, ora, rows_gpu, nb, check_rows=True):
    for i, o in enumerate(ora):
        assert int(res["bin"][i]) == o["bin"], (i, res["bin"][i], o["bin"])
        assert int(res["codePhaseRaw"][i]) == o["codePhaseRaw"], (i, res["codePhaseRaw"][i], o["codePhaseRaw"])
        assert abs(res["peakMetric"][i] - o["peakMetric"]) <= RTOL * o["peakMetric"], (i, res["peakMetric"][i], o["peakMetric"])
        assert abs(res["peak"][i] - o["peak"]) <= RTOL * o["peak"]
        assert abs(res["second"][i] - o["second"]) <= RTOL * o["second"]
        assert int(res["codePhase"][i]) == o["codePhase"]
        assert int(res["freqChannel"][i]) == o["freqChannel"]
        assert res["carrFreq"][i] == o["carrFreq"]
        if check_rows:
            for b in range(nb):
                pk, arg, blk = o["rows"][b + 1]
                g = rows_gpu[i, b]
                assert abs(g["peak"] - pk) <= RTOL * pk, (i, b, g["peak"], pk)
                # argmax / block must agree unless two maxima tie within fp32 noise
                assert int(g["code_phase"]) == arg or abs(g["peak"] - pk) <= 1e-6 * pk, (i, b, g, arg)
                bm = o["row_block_max"][b + 1]
                assert int(g["block"]) == blk or (len(bm) == 2 and abs(bm[0] - bm[1]) <= 1e-5 * max(bm)), (i, b, g, blk, bm)
                # the second peak of the row, in the window around the row's own argmax
                if int(g["code_phase"]) == arg and int(g["block"]) == blk:
                    s2 = o["row_second"][b + 1]
                    assert abs(g["second"] - s2) <= RTOL * s2, (i, b, g["second"], s2)


def test_gps_acq_1ms(oracle_lib):
    """C1 shape (1 ms coherent, +-10 kHz, 500 Hz bins) on 6 PRNs, 4 of them present."""
    from oracle import pcps_oracle as po
    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine, Settings
    from gnss_sdr_ru_b200.scenarios import gps_acq_scenario
    from gnss_sdr_ru_b200.synth import make_record

    sats = gps_acq_scenario(1001, prns=(3, 9, 22, 31))
    rec = make_record(sats, 16000 * 3, seed=1001)
    svs = [3, 5, 9, 22, 31, 32]
    st = Settings.gps(acqSearchBand=20.0, acqCohIntegration=1, acqSatelliteList=svs)
    eng = AcquisitionEngine()
    res = eng.acquisition(rec, st, return_rows=True)
    os_ = po.AcqSettings.gps(acqSearchBand=20.0, acqCohIntegration=1, svList=svs)
    ora = po.acquisition(po.to_complex(rec), os_)
    assert eng.num_bins(st) == po.num_bins(os_) == 41
    _check(res, ora, res["rows"], 41)
    found = {int(s) for s in res["freqChannel"] if s}
    assert found == {3, 9, 22, 31}


def test_gps_acq_packed(oracle_lib):
    from oracle import pcps_oracle as po
    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine, Settings
    from gnss_sdr_ru_b200.scenarios import gps_acq_scenario
    from gnss_sdr_ru_b200.synth import make_record, pack2

    sats = gps_acq_scenario(77, prns=(7, 14))
    rec = make_record(sats, 16000 * 9, seed=77)
    svs = [7, 14, 19]
    st = Settings.gps(acqSearchBand=14.0, acqCohIntegration=4, acqSatelliteList=svs)  # stock GPS settings
    eng = AcquisitionEngine()
    res = eng.acquisition(pack2(rec), st, fmt=abi.FMT_PACKED2, return_rows=True)
    os_ = po.AcqSettings.gps(acqSearchBand=14.0, acqCohIntegration=4, svList=svs)
    ora = po.acquisition(po.to_complex(rec), os_)
    _check(res, ora, res["rows"], po.num_bins(os_))


def test_glonass_acq_stock(oracle_lib):
    """C3 shape: stock GLONASS settings (5 ms, 12 kHz, 121 bins) on 4 of the 14 frequency channels."""
    from oracle import pcps_oracle as po
    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine, Settings
    from gnss_sdr_ru_b200.scenarios import glonass_acq_scenario
    from gnss_sdr_ru_b200.synth import make_record

    sats = glonass_acq_scenario(3003, channels=(-7, 0, 5))
    rec = make_record(sats, 16000 * 11, seed=3003)
    fch = [-7, -3, 0, 5]
    st = Settings.glonass(acqSatelliteList=fch)
    eng = AcquisitionEngine()
    res = eng.acquisition(rec, st, return_rows=True)
    os_ = po.AcqSettings.glonass(svList=fch)
    ora = po.acquisition(po.to_complex(rec), os_)
    assert eng.num_bins(st) == 121
    _check(res, ora, res["rows"], 121)
    assert {int(s) for s, m in zip(res["freqChannel"], res["peakMetric"]) if m > 3.0} >= {-7, 5}


def test_gps_acq_noncoherent(oracle_lib):
    """C4 shape scaled down: 2 ms coherent x 5 non-coherent, 250 Hz bins over +-2 kHz."""
    from oracle import pcps_oracle as po
    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine, Settings
    from gnss_sdr_ru_b200.scenarios import gps_acq_scenario
    from gnss_sdr_ru_b200.synth import make_record

    sats = gps_acq_scenario(4004, prns=(11, 25), cn0=(36.0, 38.0), doppler_span=1800.0)
    rec = make_record(sats, 16000 * 10, seed=4004)
    svs = [11, 12, 25]
    st = Settings.gps(acqSearchBand=4.0, acqCohIntegration=2, acqSatelliteList=svs, n_noncoh=5)
    eng = AcquisitionEngine()
    res = eng.acquisition(rec, st, return_rows=True)
    os_ = po.AcqSettings.gps(acqSearchBand=4.0, acqCohIntegration=2, svList=svs, n_noncoh=5)
    ora = po.acquisition(po.to_complex(rec), os_)
    _check(res, ora, res["rows"], po.num_bins(os_))


def test_acq_partition_merge(oracle_lib):
    """Rows computed in 3 partitions and merged equal the single-partition table (multi-GPU sharding rule)."""
    import torch

    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine, Settings
    from gnss_sdr_ru_b200.scenarios import gps_acq_scenario
    from gnss_sdr_ru_b200.synth import make_record

    sats = gps_acq_scenario(5, prns=(1, 2))
    rec = make_record(sats, 16000 * 3, seed=5)
    st = Settings.gps(acqSearchBand=6.0, acqCohIntegration=1, acqSatelliteList=[1, 2, 3])
    eng = AcquisitionEngine()
    nb = eng.num_bins(st)
    d_iq = torch.from_numpy(rec.view(np.uint8)).cuda()
    full = torch.zeros(3 * nb * 16, dtype=torch.uint8, device="cuda")
    eng.search_device(d_iq.data_ptr(), rec.size // 2, st, full.data_ptr())
    torch.cuda.synchronize()
    full_np = full.cpu().numpy().view(abi.ACQ_ROW_DTYPE)
    merged = None
    for p in range(3):
        part = torch.zeros_like(full)
        eng.search_device(d_iq.data_ptr(), rec.size // 2, st, part.data_ptr(), part_index=p, part_count=3)
        torch.cuda.synchronize()
        pn = part.cpu().numpy().view(abi.ACQ_ROW_DTYPE).copy()
        if merged is None:
            merged = pn
        else:
            take = pn["peak"] >= 0
            assert not (take & (merged["peak"] >= 0)).any()
            merged[take] = pn[take]
    assert (merged["peak"] >= 0).all()
    assert np.array_equal(merged, full_np)


def test_acq_vs_committed_fixture():
    import os

    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine, Settings

    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "acq_golden.npz"))
    st = Settings.gps(acqSearchBand=float(g["band"]), acqCohIntegration=int(g["coh"]), acqSatelliteList=[int(x) for x in g["sv"]])
    res = AcquisitionEngine().acquisition(g["packed"], st, fmt=abi.FMT_PACKED2, return_rows=True)
    assert [int(x) for x in res["bin"]] == [int(x) for x in g["bin"]]
    assert [int(x) for x in res["codePhaseRaw"]] == [int(x) for x in g["codePhaseRaw"]]
    assert np.allclose(res["peakMetric"], g["peakMetric"], rtol=RTOL)
    assert np.allclose(res["rows"]["peak"], g["rows"][:, :, 0], rtol=RTOL)


def test_c1_full_grid_vs_oracle(oracle_lib):
    """BASELINE config 1 at full size: 32 PRNs x 41 bins x 16000 code phases (21.0 M cells)."""
    from oracle import pcps_oracle as po
    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine, Settings
    from gnss_sdr_ru_b200.scenarios import gps_acq_scenario
    from gnss_sdr_ru_b200.synth import make_record

    rec = make_record(gps_acq_scenario(1001), 16000 * 3, seed=1001)
    st = Settings.gps(acqSearchBand=20.0, acqCohIntegration=1)
    eng = AcquisitionEngine()
    res = eng.acquisition(rec, st, return_rows=True)
    assert eng.cells(st) == 32 * 41 * 16000
    ora = po.acquisition(po.to_complex(rec), po.AcqSettings.gps(acqSearchBand=20.0, acqCohIntegration=1))
    _check(res, ora, res["rows"], 41)


def test_c3_half_grid_vs_oracle(oracle_lib):
    """BASELINE config 3 settings (5 ms, 12 kHz, 121 bins) on 7 of the 14 frequency channels
    (the float64 oracle needs ~2 s per channel)."""
    from oracle import pcps_oracle as po
    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine, Settings
    from gnss_sdr_ru_b200.scenarios import glonass_acq_scenario
    from gnss_sdr_ru_b200.synth import make_record

    rec = make_record(glonass_acq_scenario(3003), 16000 * 11, seed=3003)
    fch = [-7, -5, -4, -1, 0, 3, 6]
    st = Settings.glonass(acqSatelliteList=fch)
    res = AcquisitionEngine().acquisition(rec, st, return_rows=True)
    ora = po.acquisition(po.to_complex(rec), po.AcqSettings.glonass(svList=fch))
    _check(res, ora, res["rows"], 121)


def test_c4_full_size_vs_oracle(oracle_lib):
    """BASELINE config 4 at its own settings and signal levels (10 ms coherent x 20 non-coherent, 401 bins of 50 Hz,
    satellites at 28-33 dB-Hz as generated) against the float64 restatement in the reference's formulation
    (160000-point FFTs, one wipe-off + FFT per bin and block): the weakest satellite of the record (PRN 32,
    28.2 dB-Hz), one at 31.2 dB-Hz and a PRN that is not in the record -- Doppler bin and code phase exact, peak and
    peakMetric within 1e-4, every one of the 401 row maxima within 1e-4.  One process per PRN (about two minutes each)."""
    import multiprocessing as mp

    from oracle import pcps_oracle as po
    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine, Settings
    from gnss_sdr_ru_b200.scenarios import gps_weak_acq_scenario
    from gnss_sdr_ru_b200.synth import make_record

    sats = gps_weak_acq_scenario(4004)
    assert min(s.cn0_dbhz for s in sats) < 29.0 and sum(s.cn0_dbhz <= 33.0 for s in sats) == 4
    rec = make_record(sats, 16000 * 200, seed=4004)
    svs = [32, 22, 5]
    assert {32, 22} <= {s.prn for s in sats} and 5 not in {s.prn for s in sats}
    jobs = [(rec, po.AcqSettings.gps(acqSearchBand=20.0, acqCohIntegration=10, n_noncoh=20, svList=[sv])) for sv in svs]
    with mp.get_context("spawn").Pool(len(svs)) as pool:
        pending = pool.map_async(po.acquisition_job, jobs)
        st = Settings.gps(acqSearchBand=20.0, acqCohIntegration=10, n_noncoh=20, acqSatelliteList=svs)
        eng = AcquisitionEngine()
        assert eng.num_bins(st) == 401
        res = eng.acquisition(rec, st, return_rows=True)
        ora = [r[0] for r in pending.get(timeout=1500)]
    _check(res, ora, res["rows"], 401)
    # what the threshold makes of them is part of the result: same decision on both sides
    assert [int(x) for x in res["freqChannel"]] == [o["freqChannel"] for o in ora]
    assert int(res["freqChannel"][1]) == 22 and int(res["freqChannel"][2]) == 0


def test_c4_full_size_finds_the_generated_satellites():
    """BASELINE config 4 at full size (32 PRN x 401 bins, 10 ms x 20 non-coherent, 205 M cells), all 32 PRNs: a
    size-independent property beside the oracle comparison above -- every satellite the generator put into the
    record at >= 31 dB-Hz is detected at its true Doppler bin and code phase, no absent PRN is reported."""
    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine, Settings
    from gnss_sdr_ru_b200.scenarios import gps_weak_acq_scenario
    from gnss_sdr_ru_b200.synth import make_record

    sats = gps_weak_acq_scenario(4004)  # signal levels as BASELINE config 4 states them: 28-33 dB-Hz and two at 45
    rec = make_record(sats, 16000 * 200, seed=4004)
    st = Settings.gps(acqSearchBand=20.0, acqCohIntegration=10, n_noncoh=20)
    res = AcquisitionEngine().acquisition(rec, st)
    for s in sats:
        if s.cn0_dbhz < 31.0:  # 200 ms without data-bit handling does not lift these over the threshold of 3 (the float64
            continue           # restatement agrees: test_c4_full_size_vs_oracle compares PRN 32 at 28.2 dB-Hz)
        i = s.prn - 1
        assert int(res["freqChannel"][i]) == s.prn, (s.prn, res["peakMetric"][i])
        assert abs(res["carrFreq"][i] - (2.42e6 + s.doppler_hz)) <= 50.0
        # code phase: the record starts at chip `code_phase_chips`; the replica aligns at sample
        # (1023 - phase) * 16000/1023 (mod 16000), 1-based in the result
        want = ((1023.0 - s.code_phase_chips) % 1023.0) * 16000.0 / 1023.0
        d = abs(((res["codePhase"][i] - 1) - want + 8000.0) % 16000.0 - 8000.0)
        assert d <= 16.0, (s.prn, res["codePhase"][i], want)
    absent = [p for p in range(1, 33) if p not in {s.prn for s in sats}]
    assert sum(int(res["freqChannel"][p - 1]) != 0 for p in absent) == 0
