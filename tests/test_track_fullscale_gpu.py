"""GPU tracking kernels at full-scale input and at the code-table edges, against the oracle (bit exact).

The other tracking tests feed typical signals (+-1/+-3 or uniform random int8, mean zero).  Here:

1. a worst-case int8 record generated from the oracle's own state: before every block the per-sample closed forms
   (SURVEY.md Appendix A) give each sample's prompt code bit and LO phase, and the sample is set so that code bit x ival
   is -381 .. -384 on every sample -- near the largest value a 16-bit lane of the packed I,Q sums can take per sample.  Runs
   of 11 half-chip segments of such samples reach about 33.5 k on the prompt I lane, past what unpack_lanes can split;
2. simple saturated records (constant, alternating, random full scale, packed all +-3), GLONASS channel included;
3. PRN registers 32 and 33 with slews that walk them past the end of row 33, where a GPS channel must read 0 and not
   the GLONASS ST code of row 35.

Every kernel form that can read the input is run; every dump record and the whole final receiver state must equal the
oracle's (_compare_run of test_track_gpu.py).
"""
import ctypes as C

import numpy as np
import pytest

from gnss_sdr_ru_b200 import abi
from test_track_gpu import _compare_run, _rx_bytes

pytestmark = pytest.mark.gpu

LO_I = np.array([-1, 1, 2, 2, 1, -1, -2, -2])  # correlator.c:203-204
LO_Q = np.array([2, 2, 1, -1, -2, -2, -1, 1])
WORD_2P29 = int(2**29 / 80) + 1  # code NCO word whose kinc (= 80 x word) is just above 2^29: 8 samples per half chip
WC_PRNS = [27, 0, 0, 0, 0, 0, 0, 0, 9, 0, 0, 0]
WC_OVER = dict(acq_thresh=2**30, tic_period=0.0123)  # the channels keep searching: the code words stay put


def _setup_wc(o_or_eng, s=None):
    if s is None:
        o_or_eng.cold_allocate(WC_PRNS)
        o_or_eng.ch_code(0, WORD_2P29)
    else:
        o_or_eng.simple_cold_allocate(s, WC_PRNS)
        o_or_eng.ch_code(s, 0, WORD_2P29)


def _bits_row(oracle_lib, reg, n=8192):
    L = oracle_lib.Oracle.lib()
    return np.array([[L.orc_code_bit(w, reg, h) for h in range(n)] for w in range(3)], dtype=np.int64)


def _block_walk(rx, ch, ns, tab):
    """closed forms of one block for channel ch from the state before it: LO phase, E/P/L bits and pre-dump flag per
    sample (the walk serial_block does)"""
    g, W, b8 = rx.corr[ch], rx.reg_write, ch << 3
    cinc = ((W[b8 + 3] << 16) + W[b8 + 4]) & 0xFFFFFFFF
    kinc = (((W[b8 + 5] << 16) + W[b8 + 6]) << 1) & 0xFFFFFFFF
    dump_at = W[b8 + 0x84] + (1022 if W[b8] == abi.PRN_GLONASS else 2046)
    hc0 = g.half_chip & 0xFFFF
    i = np.arange(ns, dtype=np.uint64)
    k = (((np.uint64(g.carrier_phase) + i * np.uint64(cinc)) & np.uint64(0xFFFFFFFF)) >> np.uint64(29)).astype(np.int64)
    wb = ((np.uint64(g.code_phase) + i * np.uint64(kinc)) >> np.uint64(32)).astype(np.int64)
    w1 = 1 if hc0 + 1 >= dump_at else dump_at - hc0
    inA = wb < w1
    rel = wb - w1
    hh = np.where(inA, hc0 + wb, np.where(rel == 0, hc0 + w1, rel))
    assert hc0 + wb.max() < 65536 and rel.max() < dump_at  # no uint16 wrap, at most one dump in the block
    return k, tab[:, hh], inA, wb


def _mix(k, I, Q):
    return LO_I[k] * I + LO_Q[k] * Q, LO_Q[k] * I - LO_I[k] * Q


def worst_case_record(oracle_lib, ns, nblk, real=False, ch=0):
    """int8 record (I,Q interleaved, or I only) whose every sample drives channel ch's prompt I lane to -384 / -381,
    generated block by block from the oracle's state; returns the record and the number of blocks in which some run of
    11 consecutive segments sums to more than 32767 in magnitude on that lane"""
    o = oracle_lib.Oracle(oracle_lib.Oracle.default_cfg(**WC_OVER))
    _setup_wc(o)
    tab = _bits_row(oracle_lib, o.rx.reg_write[ch << 3])
    out = np.zeros((nblk, ns * (1 if real else 2)), dtype=np.int8)
    over = 0
    for b in range(nblk):
        k, (cE, cP, cL), inA, wb = _block_walk(o.rx, ch, ns, tab)
        # sign -c * sgn(lo): -128 where that is negative, +127 where it is positive
        I = np.where(cP * np.sign(LO_I[k]) > 0, -128, 127)
        Q = np.zeros_like(I) if real else np.where(cP * np.sign(LO_Q[k]) > 0, -128, 127)
        if real:
            out[b] = I
            vi, vq = LO_I[k] * I, LO_Q[k] * I  # correlator.c:217-224
        else:
            out[b, 0::2], out[b, 1::2] = I, Q
            vi, vq = _mix(k, I, Q)
        cv = cP * vi
        assert (cv < 0).all() and (-cv).min() >= (127 if real else 381)
        seg = np.bincount(wb, weights=cv).astype(np.int64)
        if len(seg) >= 11 and np.abs(np.convolve(seg, np.ones(11, dtype=np.int64), "valid")).max() > 32767:
            over += 1
        # the walk is the correlator: its six sums equal the oracle's for this block
        sums = np.array([[(c * v)[m].sum() for c in (cL, cP, cE) for v in (vi, vq)] for m in (inA, ~inA)], dtype=np.int64)
        before = np.array(o.rx.corr[ch].acc[:], dtype=np.int64)
        o.sim(out[b], ns, 0 if real else 1)
        dumped = bool((o.rx.reg_read[0x82] >> ch) & 1)
        assert dumped == (not inA.all())
        after = np.array(o.rx.corr[ch].acc[:], dtype=np.int64)
        if dumped:
            assert np.array_equal(np.array(o.rx.reg_read[(ch << 3) + 0x84 : (ch << 3) + 0x8A]), before + sums[0]), b
            assert np.array_equal(after, sums[1]), b
        else:
            assert np.array_equal(after, before + sums[0]), b
        o.gpsisr()
    return out.reshape(-1), over


class RealOracle:
    """oracle front end for I-only records (orc_sim_gp2021 with iq = 0; orc_run reads I,Q pairs): the same dump records
    as orc_run"""

    def __init__(self, oracle_lib, cfg):
        self.o = oracle_lib.Oracle(cfg)
        self.rx, self.cfg = self.o.rx, self.o.cfg

    def run(self, rec, ns, nblk, dump_cap=0):
        dumps = np.zeros((12, dump_cap), dtype=abi.DUMP_DTYPE)
        cnt = np.zeros(12, dtype=np.int32)
        for b in range(nblk):
            if self.rx.halted:
                return b, dumps, cnt
            block = int(self.rx.blocks_done)
            self.o.sim(rec[b * ns : (b + 1) * ns], ns, 0)
            st = self.rx.reg_read[0x82]
            if self.o.gpsisr():
                return b, dumps, cnt
            W = self.rx.reg_write
            for ch in range(12):
                if not (st >> ch) & 1 or cnt[ch] >= dump_cap:
                    continue
                d, j, b8, k = dumps[ch], cnt[ch], ch << 3, self.rx.chan[ch]
                d["block"][j], d["ch"][j], d["state"][j] = block, ch, k.state
                d["acc"][j] = self.rx.reg_read[b8 + 0x84 : b8 + 0x8A]
                d["carrier_incr"][j] = ((W[b8 + 3] << 16) + W[b8 + 4]) & 0xFFFFFFFF
                d["code_incr"][j] = ((W[b8 + 5] << 16) + W[b8 + 6]) & 0xFFFFFFFF
                d["n_freq"][j], d["codes"][j], d["slew"][j] = k.n_freq, k.codes, W[b8 + 0x84]
                cnt[ch] += 1
        return nblk, dumps, cnt


_RECORDS = {}


def _wc(oracle_lib, ns, nblk, real=False):
    key = (ns, nblk, real)
    if key not in _RECORDS:
        _RECORDS[key] = worst_case_record(oracle_lib, ns, nblk, real)
    return _RECORDS[key]


def _pair(oracle_lib, S, over, setup_eng, setup_orc, oracle_cls=None):
    from gnss_sdr_ru_b200.lib import default_cfg
    from gnss_sdr_ru_b200.receiver import TrackingEngine

    eng = TrackingEngine(n_streams=S, cfg=default_cfg(**over))
    orcs = []
    for s in range(S):
        cfg = oracle_lib.Oracle.default_cfg(**over)
        o = oracle_cls(oracle_lib, cfg) if oracle_cls else oracle_lib.Oracle(cfg)
        setup_orc(o.o if oracle_cls else o)
        setup_eng(eng, s)
        assert _rx_bytes(eng.rx[s]) == _rx_bytes(o.rx)
        orcs.append(o)
    eng.upload()
    return eng, orcs


# (form, occupancy, streams, block length): the segment kernel (form 3; form 0 with 13 x 12 channels > 148 SMs, i.e.
# two channels per SM, picks it as the 64-stream benchmark does), fixed runs, the barrier kernel, the generic kernel
WC_FORMS = [(3, 0, 1, 8192), (0, 0, 13, 8192), (2, 0, 1, 8192), (2, 3, 1, 8192), (1, 0, 1, 8192), (0, 0, 1, 16000), (0, 0, 1, 777)]


def test_worst_case_record_reaches_the_lane_limit(oracle_lib):
    """the generator models the correlator (checked block by block inside) and the record overflows an 11-segment run
    of the prompt I lane in most blocks"""
    rec, over = _wc(oracle_lib, 8192, 120)
    assert over >= 100, over
    rec, over = _wc(oracle_lib, 16000, 60)
    assert over >= 50, over


@pytest.mark.parametrize("form,occ,S,ns", WC_FORMS)
def test_worst_case_int8_record(oracle_lib, form, occ, S, ns):
    nblk = {8192: 120, 16000: 60, 777: 900}[ns]
    rec, _ = _wc(oracle_lib, ns, nblk)
    eng, orcs = _pair(oracle_lib, S, WC_OVER, _setup_wc, _setup_wc)
    eng.set_track_variant(form, occ)
    dumps, cnt = _compare_run(eng, orcs, np.stack([rec] * S), nblk, fmt=abi.FMT_INT8_IQ, cap=1000, ns=ns)
    assert cnt[0, 0] >= (nblk * ns) // 16400 - 1  # one dump per code period on the target channel


@pytest.mark.parametrize("form", [0, 1])
def test_worst_case_int8_real_record(oracle_lib, form):
    nblk = 120
    rec, over = _wc(oracle_lib, 8192, nblk, real=True)
    eng, orcs = _pair(oracle_lib, 1, WC_OVER, _setup_wc, _setup_wc, oracle_cls=RealOracle)
    eng.set_track_variant(form, 0)
    _compare_run(eng, orcs, rec[None, :], nblk, fmt=abi.FMT_INT8_I, cap=200, ns=8192)


# ---- simple saturated records --------------------------------------------------------------------------------------
SIMPLE_PRNS = [27, abi.PRN_GLONASS, 0, 31, 0, 0, 0, 0, 9, 0, 32, 5]
SIMPLE_OVER = dict(tic_period=0.0123, acq_thresh=1100, glonass_carrier_if=1.0e6)


def _simple(kind, n):
    rng = np.random.default_rng(["random_full", "packed_pm3"].index(kind) if kind in ("random_full", "packed_pm3") else 0)
    iq = np.empty(2 * n, dtype=np.int8)
    if kind == "const_neg":
        iq[:] = -128
    elif kind == "const_pos":
        iq[:] = 127
    elif kind == "alternate":
        iq.reshape(-1, 2)[0::2] = -128
        iq.reshape(-1, 2)[1::2] = 127
    elif kind == "random_full":
        iq[:] = rng.choice(np.array([-128, 127], dtype=np.int8), 2 * n)
    elif kind == "packed_pm3":
        iq[:] = rng.choice(np.array([-3, 3], dtype=np.int8), 2 * n)
    return iq


def _setup_simple(carrier0):
    def orc(o):
        o.cold_allocate(SIMPLE_PRNS)
        if carrier0:
            for ch, p in enumerate(SIMPLE_PRNS):
                if p:
                    o.ch_carrier(ch, 0)

    def eng(e, s):
        e.simple_cold_allocate(s, SIMPLE_PRNS)
        if carrier0:
            for ch, p in enumerate(SIMPLE_PRNS):
                if p:
                    e.ch_carrier(s, ch, 0)

    return eng, orc


SIMPLE_CASES = ([(kind, form, occ, ns) for kind in ("const_neg", "const_pos", "alternate", "random_full")
                 for form, occ, ns in ((3, 0, 8192), (2, 0, 8192), (2, 3, 8192), (1, 0, 8192), (0, 0, 777))] +
                [("packed_pm3", form, 0, 8192) for form in (0, 2, 3, 4, 5)])


@pytest.mark.parametrize("kind,form,occ,ns", SIMPLE_CASES)
def test_saturated_records(oracle_lib, kind, form, occ, ns):
    """saturated input on every kernel form: GPS and GLONASS channels (int8 GLONASS blocks take the per-sample path of
    the segment kernel, packed ones the 16-slot loop), search, confirm, pull-in with accumulators near the int16 limits
    of the channel logic; random full scale with carrier word 0 (the LO phase stays put)"""
    from gnss_sdr_ru_b200.synth import pack2

    nblk = 300 if ns == 8192 else 1500
    iq = _simple(kind, ns * nblk)
    packed = kind == "packed_pm3"
    se, so = _setup_simple(kind == "random_full")
    eng, orcs = _pair(oracle_lib, 1, SIMPLE_OVER, se, so)
    eng.set_track_variant(form, occ)
    _compare_run(eng, orcs, iq[None, :], nblk, fmt=abi.FMT_PACKED2 if packed else abi.FMT_INT8_IQ,
                 packed=pack2(iq)[None, :] if packed else None, cap=400, ns=ns)


# ---- code-table row edges ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("form,packed", [(3, False), (2, False), (1, False), (3, True)])
def test_gps_rows_past_row_33_read_zero(oracle_lib, form, packed):
    """PRN register 33 with slews >= 2047 and register 32 with slews >= 4093 walk their channels past the end of row 33
    (half chip 4092 / 6138): there a GPS channel reads 0, not the GLONASS ST code of row 35.  Register 33 also at three
    times the code rate (several dumps per block: the serial path).  Short runs between slew writes on both sides, the
    whole receiver state compared after every run."""
    from gnss_sdr_ru_b200.lib import default_cfg
    from gnss_sdr_ru_b200.receiver import TrackingEngine
    from gnss_sdr_ru_b200.synth import pack2

    rng = np.random.default_rng(300 + form + (7 if packed else 0))
    over = dict(tic_period=0.0037, acq_thresh=1500)
    prns = [33, 32, 27, 33, 0, 0, 0, 0, 9, 0, 32, abi.PRN_GLONASS]
    eng = TrackingEngine(n_streams=1, cfg=default_cfg(**over))
    o = oracle_lib.Oracle(oracle_lib.Oracle.default_cfg(**over))
    eng.simple_cold_allocate(0, prns)
    o.cold_allocate(prns)
    fast = int(o.cfg.gps_code_ref) * 3
    eng.ch_code(0, 3, fast)
    o.ch_code(3, fast)
    L = eng.L
    lo = {0: 2047, 1: 4093, 3: 2047, 10: 4093}
    periods = dict.fromkeys(lo, 0)
    pending = dict.fromkeys(lo, False)
    NS = 8192
    for it in range(45):
        for ch, low in lo.items():
            if o.rx.reg_write[(ch << 3) + 0x84] <= 1:  # the last slew was consumed by a dump
                periods[ch] += pending[ch]
                v = int(rng.integers(low, low + 2500))
                L.gnssb200_ch_code_slew(C.byref(eng.rx[0]), ch, v)
                o.ch_code_slew(ch, v)
                pending[ch] = True
        assert _rx_bytes(eng.rx[0]) == _rx_bytes(o.rx)
        nblk = int(rng.integers(1, 6))
        iq = rng.choice(np.array([-3, -1, 1, 3], dtype=np.int8), size=2 * NS * nblk)
        eng.upload()
        eng.set_track_variant(form, 0)
        if packed:
            eng.run_host(pack2(iq)[None, :], nblk, NS, abi.FMT_PACKED2, dump_cap=0)
        else:
            eng.run_host(iq[None, :], nblk, NS, abi.FMT_INT8_IQ, dump_cap=0)
        eng.download()
        n, _, _ = o.run(iq, NS, nblk)
        assert n == nblk
        got, want = eng.rx[0], o.rx
        for name, _ in abi.Rx._fields_:
            ga, wa = getattr(got, name), getattr(want, name)
            gb = bytes(memoryview(ga).cast("B")) if hasattr(ga, "_length_") or isinstance(ga, C.Structure) else ga
            wb = bytes(memoryview(wa).cast("B")) if hasattr(wa, "_length_") or isinstance(wa, C.Structure) else wa
            assert gb == wb, f"iteration {it} ({nblk} blocks): rx.{name} differs"
    assert min(periods.values()) >= 2, periods  # every channel walked past row 33 at least twice
