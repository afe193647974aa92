"""Pins the CPU restatement (oracle/gp2021_oracle.c) against the REFERENCE ITSELF.

* live: the reference C receiver compiled from its own sources (oracle/_ref, only where
  /root/reference exists) -- every register after every block, channel state after every gpsisr;
* golden: tests/golden/ref_track_golden.npz, outputs of that compiled reference on a seeded record
  (travels to the GPU box).
"""
import os

import numpy as np
import pytest

from gnss_sdr_ru_b200 import abi
from gnss_sdr_ru_b200.synth import unpack2

HERE = os.path.dirname(os.path.abspath(__file__))
NS = 8192


def _golden():
    g = np.load(os.path.join(HERE, "golden", "ref_track_golden.npz"))
    return g, unpack2(g["packed"])


def test_oracle_matches_golden_reference_outputs(oracle_lib):
    g, rec = _golden()
    o = oracle_lib.Oracle()
    o.cold_allocate([int(p) for p in g["prns"]])
    for ch, nf in g["warm"]:
        k = o.rx.chan[int(ch)]
        nf = int(nf)
        k.n_freq, k.del_freq, k.codes = nf, (-2 * nf if nf > 0 else 1 - 2 * nf), 0
        k.carrier_freq = o.cfg.gps_carrier_ref + o.cfg.d_freq * nf
        o.ch_carrier(int(ch), k.carrier_freq)
    cap = g["dumps"].shape[1]
    n, dumps, cnt = o.run(rec, int(g["nsamp"]), int(g["nblk"]), dump_cap=cap)
    assert np.array_equal(cnt, g["cnt"])
    assert np.array_equal(dumps, g["dumps"].view(abi.DUMP_DTYPE).reshape(dumps.shape))
    assert np.array_equal(np.array(o.rx.reg_read[:]), g["reg_read"])
    assert np.array_equal(np.array(o.rx.reg_write[:]), g["reg_write"])


@pytest.mark.skipif(not os.path.isdir("/root/reference"), reason="needs the reference sources to compile oracle/_ref")
def test_oracle_matches_live_reference_closed_loop(oracle_lib, track_record):
    rec, _ = track_record
    nblk = 900
    ref = oracle_lib.RefReceiver()
    o = oracle_lib.Oracle()
    prns = [27, 0, 0, 31, 0, 0, 0, 0, 9, 0, 32, 5]
    ref.cold_allocate(prns)
    o.cold_allocate(prns)
    for ch, nf in ((0, 1), (8, -1), (10, 1)):
        ref.warm_start(ch, nf)
        k = o.rx.chan[ch]
        k.n_freq, k.del_freq, k.codes = nf, (-2 * nf if nf > 0 else 1 - 2 * nf), 0
        k.carrier_freq = o.cfg.gps_carrier_ref + o.cfg.d_freq * nf
        o.ch_carrier(ch, k.carrier_freq)
    skip = {"pad_", "accum", "prev_accum", "mean_early", "mean_prompt", "mean_late"}
    names = [f for f, _ in abi.Chan._fields_ if f not in skip]
    for b in range(nblk):
        blk = rec[2 * NS * b : 2 * NS * (b + 1)]
        ref.sim(blk, NS)
        o.sim(blk, NS)
        rr, rw = ref.regs()
        assert np.array_equal(rr, np.array(o.rx.reg_read[:])), b
        assert np.array_equal(rw, np.array(o.rx.reg_write[:])), b
        ref.gpsisr()
        o.gpsisr()
        rr, rw = ref.regs()
        assert np.array_equal(rw, np.array(o.rx.reg_write[:])), b
        for ch in (0, 3, 8, 10, 11):
            rc, oc = ref.chan[ch], o.rx.chan[ch]
            for n in names:
                rv = getattr(rc, n)
                if isinstance(rv, bytes):
                    rv = int.from_bytes(rv, "little", signed=True) if rv else 0
                assert rv == getattr(oc, n), (b, ch, n)
            g_, c_ = ref.gpchan[ch], o.rx.corr[ch]
            assert (g_.int_carrier_phase, g_.int_carrier_cycle, g_.int_code_phase, g_.int_code_half_chip) == (
                c_.carrier_phase, c_.carrier_cycle, c_.code_phase, c_.half_chip), (b, ch)


@pytest.mark.skipif(not os.path.isdir("/root/reference"), reason="needs the reference sources to compile oracle/_ref")
def test_oracle_matches_live_reference_full_acq_to_track(oracle_lib, track_record):
    """native loops on both sides over the whole record: search -> confirm -> pull-in -> tracking"""
    rec, nblk = track_record
    ref = oracle_lib.RefReceiver()
    o = oracle_lib.Oracle()
    prns = [27, 0, 0, 31, 0, 0, 0, 0, 9, 0, 32, 5]
    ref.cold_allocate(prns)
    o.cold_allocate(prns)
    for ch, nf in ((0, 1), (8, -1), (10, 1)):
        ref.warm_start(ch, nf)
        k = o.rx.chan[ch]
        k.n_freq, k.del_freq, k.codes = nf, (-2 * nf if nf > 0 else 1 - 2 * nf), 0
        k.carrier_freq = o.cfg.gps_carrier_ref + o.cfg.d_freq * nf
        o.ch_carrier(ch, k.carrier_freq)
    _, rd, rc = ref.run(rec, NS, nblk, dump_cap=2000)
    _, od, oc = o.run(rec, NS, nblk, dump_cap=2000)
    assert np.array_equal(rc, oc)
    assert np.array_equal(rd, od)
    assert int(o.rx.chan[0].state) == 4 and int(o.rx.chan[8].state) == 4 and int(o.rx.chan[10].state) == 4


# what the compiled reference derives at start-up (BASELINE.md section 2): gps_carrier_ref, gps_code_ref, d_freq and the
# loop-filter gains FLL_a_PLL_i1..3, DLL_i1..2
REF_CONSTANTS = dict(gps_carrier_ref=32480690, gps_code_ref=6865236, d_freq=13421,
                     FLL_a_PLL_i1=925, FLL_a_PLL_i2=895, FLL_a_PLL_i3=75, DLL_i1=35, DLL_i2=35)


def test_oracle_config_constants_match_reference(oracle_lib):
    """the restatement's derived configuration equals the values the compiled reference derives"""
    cfg = oracle_lib.Oracle.default_cfg()
    assert (cfg.gps_carrier_ref, cfg.gps_code_ref, cfg.d_freq) == tuple(REF_CONSTANTS[n] for n in ("gps_carrier_ref", "gps_code_ref", "d_freq"))
    assert [cfg.pll_i1, cfg.pll_i2, cfg.pll_i3, cfg.dll_i1, cfg.dll_i2] == [
        REF_CONSTANTS[n] for n in ("FLL_a_PLL_i1", "FLL_a_PLL_i2", "FLL_a_PLL_i3", "DLL_i1", "DLL_i2")]
