"""gnssb200_acq_search_batch: R records in one call give exactly the row tables of R single-record searches.

The batched kernels compute every (record, sv, bin) row with the same arithmetic as a single-record call, so the tables
must be byte-identical, not merely close.  One record of a batch is also checked against the float64 restatement of
acquisition.sci with the rules of tests/test_acq_gpu.py (argmax exact, 1e-4 relative).
"""
import numpy as np
import pytest

from gnss_sdr_ru_b200 import abi

pytestmark = pytest.mark.gpu
R = 5
PAD = 4096  # stride = record bytes + PAD: the records do not touch


def _records(settings, fmt, n_ms, seed):
    """R records with different satellites, in one device buffer with a stride larger than a record."""
    import torch

    from gnss_sdr_ru_b200.scenarios import glonass_acq_scenario, gps_acq_scenario
    from gnss_sdr_ru_b200.synth import make_record, pack2

    n = 16000 * n_ms
    recs = []
    for r in range(R):
        if settings.system == "gps":
            prns = [int(p) for p in np.random.default_rng(seed + r).choice(settings.acqSatelliteList, 3, replace=False)]
            sats = gps_acq_scenario(seed + r, prns=prns)
        else:
            fch = [int(k) for k in np.random.default_rng(seed + r).choice(settings.acqSatelliteList, 3, replace=False)]
            sats = glonass_acq_scenario(seed + r, channels=fch)
        rec = make_record(sats, n, seed=seed + r)
        recs.append(pack2(rec) if fmt == abi.FMT_PACKED2 else rec.view(np.uint8))
    stride = recs[0].size + PAD
    buf = np.zeros(R * stride, dtype=np.uint8)
    for r, rec in enumerate(recs):
        buf[r * stride : r * stride + rec.size] = rec
    return torch.from_numpy(buf).cuda(), stride, n, recs


def _tables(eng, settings, d_buf, stride, n, fmt, part_index=0, part_count=0):
    """(batched [R][n_sv][n_bins], per-record [R][n_sv][n_bins]) as host row arrays."""
    import torch

    nb, n_sv = eng.num_bins(settings), len(settings.acqSatelliteList)
    bat = torch.zeros(R * n_sv * nb * 16, dtype=torch.uint8, device="cuda")
    eng.search_batch_device(d_buf.data_ptr(), stride, R, n, settings, bat.data_ptr(), fmt=fmt, part_index=part_index,
                            part_count=part_count)
    one = torch.zeros_like(bat)
    for r in range(R):
        eng.search_device(d_buf.data_ptr() + r * stride, n, settings, one.data_ptr() + r * n_sv * nb * 16, fmt=fmt,
                          part_index=part_index, part_count=part_count)
    torch.cuda.synchronize()
    view = lambda t: t.cpu().numpy().view(abi.ACQ_ROW_DTYPE).reshape(R, n_sv, nb)  # noqa: E731
    return view(bat), view(one)


def _settings(case):
    from gnss_sdr_ru_b200.acquisition import Settings

    if case in ("c1_int8", "c1_packed"):
        return Settings.gps(acqSearchBand=20.0, acqCohIntegration=1), 3
    if case == "glonass":
        return Settings.glonass(), 11
    return Settings.gps(acqSearchBand=4.0, acqCohIntegration=2, acqSatelliteList=[4, 11, 12, 25, 30], n_noncoh=5), 10


@pytest.mark.parametrize("case", ["c1_int8", "c1_packed", "glonass", "noncoherent"])
def test_batch_equals_single_record_calls(case):
    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine

    st, n_ms = _settings(case)
    fmt = abi.FMT_PACKED2 if case == "c1_packed" else abi.FMT_INT8_IQ
    eng = AcquisitionEngine()
    d_buf, stride, n, _ = _records(st, fmt, n_ms, seed=100 + len(case))
    bat, one = _tables(eng, st, d_buf, stride, n, fmt)
    assert (bat["peak"] >= 0).all()
    assert bat.tobytes() == one.tobytes()
    # the records differ, so do their tables: the batch did not read one record R times
    assert len({bat[r].tobytes() for r in range(R)}) == R


def test_batch_partitions_merge_to_the_full_table():
    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine, Settings

    st = Settings.gps(acqSearchBand=6.0, acqCohIntegration=1, acqSatelliteList=[1, 2, 3, 5, 8])
    eng = AcquisitionEngine()
    d_buf, stride, n, _ = _records(st, abi.FMT_INT8_IQ, 3, seed=7)
    full, _ = _tables(eng, st, d_buf, stride, n, abi.FMT_INT8_IQ)
    merged = None
    for p in range(3):
        bat, one = _tables(eng, st, d_buf, stride, n, abi.FMT_INT8_IQ, part_index=p, part_count=3)
        assert bat.tobytes() == one.tobytes()
        if merged is None:
            merged = bat.copy()
        else:
            take = bat["peak"] >= 0
            assert not (take & (merged["peak"] >= 0)).any()
            merged[take] = bat[take]
    assert merged.tobytes() == full.tobytes()


def test_one_record_batch_is_the_single_search_and_stride_zero_repeats_it():
    import torch

    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine

    st, _ = _settings("c1_int8")
    eng = AcquisitionEngine()
    d_buf, stride, n, _ = _records(st, abi.FMT_INT8_IQ, 3, seed=31)
    nb, n_sv = eng.num_bins(st), len(st.acqSatelliteList)
    single = torch.zeros(n_sv * nb * 16, dtype=torch.uint8, device="cuda")
    eng.search_device(d_buf.data_ptr(), n, st, single.data_ptr())
    one = torch.zeros_like(single)
    eng.search_batch_device(d_buf.data_ptr(), stride, 1, n, st, one.data_ptr())
    rep = torch.zeros(R * single.numel(), dtype=torch.uint8, device="cuda")
    eng.search_batch_device(d_buf.data_ptr(), 0, R, n, st, rep.data_ptr())
    torch.cuda.synchronize()
    s = single.cpu().numpy().tobytes()
    assert one.cpu().numpy().tobytes() == s
    rp = rep.cpu().numpy()
    assert all(rp[r * single.numel() : (r + 1) * single.numel()].tobytes() == s for r in range(R))


def test_batch_record_vs_float64_restatement(oracle_lib):
    """Record 3 of a batch (acquisition_batch: one copy back, finalize per record) against pcps_oracle."""
    from oracle import pcps_oracle as po
    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine, Settings

    svs = [3, 9, 14, 22, 31, 32]
    st = Settings.gps(acqSearchBand=20.0, acqCohIntegration=1, acqSatelliteList=svs)
    eng = AcquisitionEngine()
    d_buf, stride, n, recs = _records(st, abi.FMT_INT8_IQ, 3, seed=1001)
    outs = eng.acquisition_batch(d_buf.data_ptr(), stride, R, n, st, return_rows=True)
    assert len(outs) == R
    res = outs[3]
    ora = po.acquisition(po.to_complex(recs[3].view(np.int8)), po.AcqSettings.gps(acqSearchBand=20.0, acqCohIntegration=1,
                                                                                 svList=svs))
    for i, o in enumerate(ora):
        assert int(res["bin"][i]) == o["bin"] and int(res["codePhaseRaw"][i]) == o["codePhaseRaw"], i
        assert abs(res["peakMetric"][i] - o["peakMetric"]) <= 1e-4 * o["peakMetric"], i
        assert abs(res["peak"][i] - o["peak"]) <= 1e-4 * o["peak"], i
        assert int(res["codePhase"][i]) == o["codePhase"] and int(res["freqChannel"][i]) == o["freqChannel"]
        assert res["carrFreq"][i] == o["carrFreq"]
    # acquisition_batch's record 3 is acquisition() of that record
    single = eng.acquisition(recs[3].view(np.int8), st)
    for key in ("carrFreq", "codePhase", "peakMetric", "freqChannel", "bin", "codePhaseRaw"):
        assert np.array_equal(single[key], res[key]), key


def test_batch_argument_checks():
    import torch

    from gnss_sdr_ru_b200.acquisition import AcquisitionEngine
    from gnss_sdr_ru_b200.lib import GnssB200Error

    st, _ = _settings("c1_int8")
    eng = AcquisitionEngine()
    n = 16000 * 2
    d = torch.zeros(2 * n * 2, dtype=torch.uint8, device="cuda")
    rows = torch.zeros(2 * 32 * 41 * 16, dtype=torch.uint8, device="cuda")
    with pytest.raises(GnssB200Error):
        eng.search_batch_device(d.data_ptr(), 2 * n, 0, n, st, rows.data_ptr())
    with pytest.raises(GnssB200Error):  # int8: 2 bytes per sample
        eng.search_batch_device(d.data_ptr(), 2 * n - 2, 2, n, st, rows.data_ptr())
    with pytest.raises(GnssB200Error):  # packed: two complex samples per byte
        eng.search_batch_device(d.data_ptr(), n // 2 - 1, 2, n, st, rows.data_ptr(), fmt=abi.FMT_PACKED2)
    eng.search_batch_device(d.data_ptr(), n // 2, 2, n, st, rows.data_ptr(), fmt=abi.FMT_PACKED2)
    torch.cuda.synchronize()
