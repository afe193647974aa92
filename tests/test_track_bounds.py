"""Edges of the tracking correlator that typical signals never reach (CPU only, no GPU).

1. Lane width.  Every correlator loop carries I and Q in one 32-bit int as ``ival + 65536*qval`` and splits the sum
   with ``unpack_lanes`` (track_common.cuh), which is exact only while each 16-bit lane stays within +-32767.  For every
   ``track_ws_kernel`` / ``track_loop_kernel`` instantiation that track.cu launches (read from the source, so a new one
   cannot escape), the samples summed into one packed int times the largest per-sample lane value of the format it
   reads must stay within that bound -- and a NumPy model of the packed int32 arithmetic (the segment partition of
   track_seg.cuh, the fixed sample runs) on full-scale samples chosen per LO phase and code bit must give the exact sums.
2. Code-table rows.  A GPS PRN register reads its row with the reference's flat spill-over into the rows after it, up
   to the end of row 33; from there on it reads 0 (the reference has 33 rows).  The GLONASS ST code of row 35 is read
   only by ``GNSSB200_PRN_GLONASS``.  Checked on the oracle against a table built here from the IS-GPS-200 G2 taps and
   the GLONASS ICD register.
"""
import os
import re

import numpy as np
import pytest

from gnss_sdr_ru_b200 import abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TRACK_CU = os.path.join(ROOT, "gnss_sdr_ru_b200", "csrc", "track.cu")

LANE_MAX = 32767
BLOCK_MAX = 8192  # the warp-specialised kernel's largest block
LO_I = np.array([-1, 1, 2, 2, 1, -1, -2, -2])  # correlator.c:203-204
LO_Q = np.array([2, 2, 1, -1, -2, -2, -1, 1])
FMT_NAMES = {"GNSSB200_FMT_INT8_IQ": abi.FMT_INT8_IQ, "GNSSB200_FMT_PACKED2": abi.FMT_PACKED2, "-1": -1}


def _sample_values(fmt):
    """(I, Q) pairs a format can deliver"""
    if fmt == abi.FMT_PACKED2:
        v = np.array([1, -1, 3, -3])
        return np.array([(i, q) for i in v for q in v])
    if fmt == abi.FMT_INT8_I:
        return np.array([(i, 0) for i in range(-128, 128)])
    v = np.arange(-128, 128)
    return np.stack(np.meshgrid(v, v), -1).reshape(-1, 2)


def lane_max(fmt):
    """largest |ival| or |qval| one sample of the format adds to a lane (correlator.c:214-215); fmt -1 = any format"""
    if fmt == -1:
        return max(lane_max(f) for f in (abi.FMT_INT8_IQ, abi.FMT_PACKED2, abi.FMT_INT8_I))
    iq = _sample_values(fmt)
    best = 0
    for k in range(8):
        ival = LO_I[k] * iq[:, 0] + LO_Q[k] * iq[:, 1]
        qval = LO_Q[k] * iq[:, 0] - LO_I[k] * iq[:, 1]
        best = max(best, int(np.abs(ival).max()), int(np.abs(qval).max()))
    return best


def launched_kernels():
    """(kind, fmt, run forms) of every tracking-kernel instantiation track.cu launches.  A run form is (threads, segments
    per thread, samples per segment) for the half-chip-segment loop, (None, samples, 1) for a fixed run of samples."""
    src = open(TRACK_CU).read()
    out = {}
    for kind, args in re.findall(r"\b(track_ws_kernel|track_loop_kernel)<([^<>]*)><<<", src):
        a = [x.strip() for x in args.split(",")]
        if kind == "track_ws_kernel":
            fmt, ct = FMT_NAMES[a[1]], int(a[2])
            segh = int(a[3]) if len(a) > 3 else 0
            if segh:  # track_ws.cuh: 7-8 samples per half chip; packed input also 15-16 (GLONASS) at (H*8+15)/16 segments
                forms = [(ct, segh, 8)]
                if fmt == abi.FMT_PACKED2:
                    forms.append((ct, (segh * 8 + 15) // 16, 16))
            else:
                forms = [(None, BLOCK_MAX // ct, 1)]
        else:  # track_loop_kernel<MAXT, MINB, FMT, TMA, SPT = 32>
            fmt = FMT_NAMES[a[2]]
            forms = [(None, int(a[4]) if len(a) > 4 else 32, 1)]
        out[f"{kind}<{args.replace(' ', '')}>"] = (kind, fmt, forms)
    return out


KERNELS = launched_kernels()


def test_every_form_of_track_cu_is_found():
    """the regex sees the launches: both kernels, both staged formats, the generic variant, segment and fixed runs"""
    kinds = {k for k, _, _ in KERNELS.values()}
    fmts = {f for _, f, _ in KERNELS.values()}
    assert kinds == {"track_ws_kernel", "track_loop_kernel"} and fmts == {abi.FMT_INT8_IQ, abi.FMT_PACKED2, -1}
    assert any(t is not None for _, _, forms in KERNELS.values() for t, _, _ in forms)
    assert len(KERNELS) >= 15


def test_lane_maxima():
    assert lane_max(abi.FMT_INT8_IQ) == 384 and lane_max(abi.FMT_PACKED2) == 9 and lane_max(abi.FMT_INT8_I) == 256


def test_every_launched_ws_kernel_has_its_shared_memory_opt_in():
    src = open(TRACK_CU).read()
    opted = {a.replace(" ", "") for a in re.findall(r"cudaFuncSetAttribute\(track_ws_kernel<([^<>]*)>", src)}
    for name, (kind, _, _) in KERNELS.items():
        if kind == "track_ws_kernel":
            assert name[len("track_ws_kernel<") : -1] in opted, name


@pytest.mark.parametrize("name", sorted(KERNELS))
def test_packed_lanes_cannot_overflow(name):
    """samples summed into one packed int before unpack_lanes x the format's largest lane value <= 32767"""
    _, fmt, forms = KERNELS[name]
    for _, runs, slots in forms:
        n = runs * slots
        assert n * lane_max(fmt) <= LANE_MAX, f"{name}: {n} samples x {lane_max(fmt)} per lane can reach {n * lane_max(fmt)}"


# ---- NumPy model of the packed arithmetic ------------------------------------------------------------------------
def w32(x):
    return ((int(x) + 2**31) % 2**32) - 2**31


def unpack_lanes(packed):
    """track_common.cuh unpack_lanes on an int32"""
    lo = ((packed & 0xFFFF) ^ 0x8000) - 0x8000
    return lo, w32(packed - lo) >> 16


def closed_form_index(n, kph0, kinc, hc0, w1, stale_idx):
    """per-sample code-table index and pre/post-dump class (SURVEY.md Appendix A)"""
    i = np.arange(n, dtype=np.uint64)
    wb = ((np.uint64(kph0) + i * np.uint64(kinc)) >> np.uint64(32)).astype(np.int64)
    inA = wb < w1
    rel = wb - w1
    return np.where(inA, hc0 + wb, np.where(rel == 0, stale_idx, rel)), inA


def brute(v, kph0, kinc, hc0, w1, stale_idx, tbl, n):
    """exact sums of code bit x value before (A) and after (B) the dump"""
    hh, inA = closed_form_index(n, kph0, kinc, hc0, w1, stale_idx)
    bits = tbl[hh]
    return int((bits[inA] * v[inA]).sum()), int((bits[~inA] * v[~inA]).sum())


def seg_start(m, kph0, kinc):
    x = np.float64(m) * 4294967296.0 + (-np.float64(kph0) - 0.5)
    return int(np.float64(x) * (np.float64(1.0) / np.float64(kinc))) + 1


def seg_model(v, kph0, kinc, hc0, w1, stale_idx, tbl, n, NT, H, SLOTS=8, packed=False):
    """seg_block (track_seg.cuh): thread runs of H whole segments, the dump hand-over to thread NT-1, head and tail one
    sample per lane.  packed=False: exact sums of v.  packed=True: v holds (ival, qval) rows; every run is summed as
    ival + 65536*qval in int32 (per segment, times the code bit, over the run) and split by unpack_lanes like the kernel."""
    wtot = (kph0 + n * kinc) >> 32
    NF = wtot - 1 if wtot > 0 else 0
    A, B = np.zeros(2, dtype=np.int64), np.zeros(2, dtype=np.int64)
    pv = (v[:, 0] + 65536 * v[:, 1]) if packed else v
    alias = tbl.copy()
    alias[0] = tbl[stale_idx]
    for tid in range(NT):
        if tid < NT - 1:
            first = tid * H
            m0 = 1 + first
            nv = min(NF - first, H) if NF > first else 0
            if m0 < w1 < m0 + nv:
                nv = w1 - m0
        else:
            m0, nv = 1, 0
            if w1 >= 2:
                ts = (w1 - 2) // H
                first = ts * H
                end = 1 + first + (min(NF - first, H) if NF > first else 0)
                if ts < NT - 1 and w1 < end:
                    m0, nv = w1, end - w1
        if nv == 0:
            m0 = 1
        clsB = m0 >= w1
        if clsB:
            rel = m0 - w1
            src, base = (alias, 0) if rel == 0 else (tbl, rel)
        else:
            src, base = tbl, hc0 + m0
        s = seg_start(m0, kph0, kinc)
        exact = -((-(m0 * 2**32 - kph0)) // kinc)
        assert s == exact, (s, exact)
        ks = (kph0 + s * kinc) % 2**32
        assert ks < kinc
        acc = 0
        for j in range(H):
            u = ks + (SLOTS - 1) * kinc
            full = u < 2**32
            cnt = SLOTS if full else SLOTS - 1
            ks = (u + (kinc if full else 0)) % 2**32
            if j < nv:
                assert s + cnt <= n
                acc += int(src[base + j]) * int(pv[s : s + cnt].sum())
            s += cnt
        part = np.array(unpack_lanes(w32(acc)) if packed else (acc, 0), dtype=np.int64)
        if clsB:
            B += part
        else:
            A += part
    OWNED = (NT - 1) * H
    head_end = n if wtot == 0 else min(seg_start(1, kph0, kinc), n)
    mt = 1 + min(NF, OWNED)
    tail_start = n if mt > wtot else min(seg_start(mt, kph0, kinc), n)
    for i in list(range(head_end)) + list(range(tail_start, n)):
        wb = (kph0 + i * kinc) >> 32
        one = v[i] if packed else np.array([v[i], 0])
        if wb < w1:
            A += int(tbl[hc0 + wb]) * one
        else:
            rel = wb - w1
            B += int(tbl[stale_idx if rel == 0 else rel]) * one
    return (int(A[0]), int(B[0])) if not packed else (tuple(int(x) for x in A), tuple(int(x) for x in B))


def fixed_run_model(v, kph0, kinc, hc0, w1, stale_idx, tbl, n, spt):
    """fixed-run form: spt consecutive samples per thread summed as packed int32 with the per-sample code bit; the chunk
    that contains the dump is re-evaluated sample by sample"""
    hh, inA = closed_form_index(n, kph0, kinc, hc0, w1, stale_idx)
    bits = tbl[hh].astype(np.int64)
    A, B = np.zeros(2, dtype=np.int64), np.zeros(2, dtype=np.int64)
    for i0 in range(0, n, spt):
        sl = slice(i0, min(i0 + spt, n))
        if inA[sl].all() or not inA[sl].any():
            acc = w32(int((bits[sl] * (v[sl, 0] + 65536 * v[sl, 1])).sum()))
            part = np.array(unpack_lanes(acc), dtype=np.int64)
        else:
            part = None
            for i in range(sl.start, sl.stop):
                (A if inA[i] else B)[:] += bits[i] * v[i]
        if part is not None:
            (A if inA[sl.start] else B)[:] += part
    return tuple(int(x) for x in A), tuple(int(x) for x in B)


def full_scale(fmt, bits, k):
    """samples that push the lane of code bit x ival to its limit on every sample: I of sign -c * sgn(lo_i[k]) and Q of
    sign -c * sgn(lo_q[k]) (c = the code bit), at full scale (-128 / +127 for int8, -3 / +3 packed)"""
    neg, pos = {abi.FMT_INT8_IQ: (-128, 127), abi.FMT_PACKED2: (-3, 3), abi.FMT_INT8_I: (-128, 127)}[fmt]
    c = np.where(bits >= 0, 1, -1)
    I = np.where(c * np.sign(LO_I[k]) > 0, neg, pos)
    Q = np.where(c * np.sign(LO_Q[k]) > 0, neg, pos) if fmt != abi.FMT_INT8_I else np.zeros_like(I)
    return I, Q


def mixed(fmt, bits, k):
    """(ival, qval) per sample of the full-scale input (correlator.c:214-215)"""
    I, Q = full_scale(fmt, bits, k)
    return np.stack([LO_I[k] * I + LO_Q[k] * Q, LO_Q[k] * I - LO_I[k] * Q], axis=1).astype(np.int64)


def _code_rows():
    """a prompt row: +-1 over three rows (the spill-over reads), as the kernels see it"""
    rng = np.random.default_rng(7)
    return rng.choice(np.array([-1, 1]), 3 * 2046 + 64)


def _block_params(rng, n, slots, it):
    if slots == 8:  # 7 or 8 samples per half chip; the bottom of the range gives 8 almost everywhere
        kinc = [2**29 + 48, 549218880, int(rng.integers(2**29, 2**32 // 7 + 1))][it % 3]
        period = 2046
    else:
        kinc = [2**28 + 48, 274340960, int(rng.integers(2**28, 2**32 // 15 + 1))][it % 3]
        period = 1022
    kph0 = int(rng.integers(0, 2**32))
    wtot = (kph0 + n * kinc) >> 32
    hc0 = int(rng.integers(0, period))
    w1 = (period - hc0 if hc0 < period - 1 else 1) if it % 2 else int(rng.integers(1, max(2, wtot + 3)))
    cinc = [0, 649613800, int(rng.integers(0, 2**32))][it % 3]
    return kinc, kph0, hc0, w1, hc0 + w1, int(rng.integers(0, 2**32)), cinc


SEG_FORMS = sorted({(fmt, t, h, slots) for _, fmt, forms in KERNELS.values() for t, h, slots in forms if t is not None})
RUN_FORMS = sorted({(fmt, h) for _, fmt, forms in KERNELS.values() for t, h, slots in forms if t is None})


@pytest.mark.parametrize("fmt,NT,H,slots", SEG_FORMS)
def test_segment_partition_reproduces_the_closed_forms(fmt, NT, H, slots):
    """thread ownership, float64 start samples and the dump hand-over of the segment form sum every sample exactly once
    with its own code bit, on random block parameters (ints: no lane packing)"""
    rng = np.random.default_rng(NT * 100 + H * 10 + slots)
    tbl = rng.integers(-1, 2, 4096)
    for it in range(12):
        n = int(rng.choice([8192, 8192, 4000, 6000, 512, 64]))
        kinc, kph0, hc0, w1, stale, _, _ = _block_params(rng, n, slots, it)
        v = rng.integers(-9, 10, n)
        assert brute(v, kph0, kinc, hc0, w1, stale, tbl, n) == seg_model(v, kph0, kinc, hc0, w1, stale, tbl, n, NT, H, slots)


@pytest.mark.parametrize("fmt,NT,H,slots", SEG_FORMS)
def test_segment_loop_packed_arithmetic_at_full_scale(fmt, NT, H, slots):
    """the packed int32 sums of the segment form on full-scale samples (every sample at the lane's limit, with the sign
    of its code bit) equal the exact sums: no lane carries into the other"""
    rng = np.random.default_rng(11 + NT + H + slots)
    tbl = np.concatenate([_code_rows(), np.zeros(2304 + 2048, dtype=np.int64)])
    for it in range(6):
        n = 8192
        kinc, kph0, hc0, w1, stale, cph0, cinc = _block_params(rng, n, slots, it)
        hh, _ = closed_form_index(n, kph0, kinc, hc0, w1, stale)
        k = ((cph0 + np.arange(n, dtype=np.uint64) * np.uint64(cinc)) % np.uint64(2**32) >> np.uint64(29)).astype(np.int64)
        v = mixed(fmt, tbl[hh], k)
        want_a = [brute(v[:, c], kph0, kinc, hc0, w1, stale, tbl, n) for c in (0, 1)]
        got = seg_model(v, kph0, kinc, hc0, w1, stale, tbl, n, NT, H, slots, packed=True)
        assert (got[0], got[1]) == ((want_a[0][0], want_a[1][0]), (want_a[0][1], want_a[1][1])), (
            f"fmt {fmt} {NT} threads x {H} segments: packed sums {got}, exact {want_a}")


@pytest.mark.parametrize("fmt,spt", RUN_FORMS)
def test_fixed_runs_packed_arithmetic_at_full_scale(fmt, spt):
    fmts = [abi.FMT_INT8_IQ, abi.FMT_PACKED2, abi.FMT_INT8_I] if fmt == -1 else [fmt]
    rng = np.random.default_rng(spt)
    tbl = np.concatenate([_code_rows(), np.zeros(2304 + 2048, dtype=np.int64)])
    for f in fmts:
        for it in range(3):
            n = 8192
            kinc, kph0, hc0, w1, stale, cph0, cinc = _block_params(rng, n, 8, it)
            hh, _ = closed_form_index(n, kph0, kinc, hc0, w1, stale)
            k = ((cph0 + np.arange(n, dtype=np.uint64) * np.uint64(cinc)) % np.uint64(2**32) >> np.uint64(29)).astype(np.int64)
            v = mixed(f, tbl[hh], k)
            want = [brute(v[:, c], kph0, kinc, hc0, w1, stale, tbl, n) for c in (0, 1)]
            got = fixed_run_model(v, kph0, kinc, hc0, w1, stale, tbl, n, spt)
            assert got == ((want[0][0], want[1][0]), (want[0][1], want[1][1])), (f, spt, got, want)


def test_full_scale_samples_reach_the_lane_limit():
    """the model input is what the lane bound assumes: code bit x ival is -381 .. -384 (int8 I,Q) or -9 (packed) on every
    sample; I-only samples give -127 |lo_i| or -128 |lo_i|, at most -256"""
    bits = np.repeat(np.array([1, -1]), 8)
    k = np.tile(np.arange(8), 2)
    for fmt, lo in ((abi.FMT_INT8_IQ, 381), (abi.FMT_PACKED2, 9), (abi.FMT_INT8_I, 127)):
        I, Q = full_scale(fmt, bits, k)
        assert I.min() >= -128 and I.max() <= 127 and Q.min() >= -128 and Q.max() <= 127
        cv = bits * mixed(fmt, bits, k)[:, 0]
        assert (-cv >= lo).all() and -cv.min() == lane_max(fmt), (fmt, cv)


# ---- code-table rows --------------------------------------------------------------------------------------------
HALF = 2046
G2_TAPS = [(2, 6), (3, 7), (4, 8), (5, 9), (1, 9), (2, 10), (1, 8), (2, 9), (3, 10), (2, 3), (3, 4), (5, 6), (6, 7), (7, 8),
           (8, 9), (9, 10), (1, 4), (2, 5), (3, 6), (4, 7), (5, 8), (6, 9), (1, 3), (4, 6), (5, 7), (6, 8), (7, 9), (8, 10),
           (1, 6), (2, 7), (3, 8), (4, 9)]  # IS-GPS-200 Table 3-Ia, G2 code phase selection, PRN 1..32


def ca_code(prn):
    """C/A code chips (0/1) from the G1 / G2 shift registers with the G2 phase-selector taps"""
    g1, g2 = [1] * 10, [1] * 10
    a, b = G2_TAPS[prn - 1]
    out = []
    for _ in range(1023):
        out.append(g1[9] ^ g2[a - 1] ^ g2[b - 1])
        f1 = g1[2] ^ g1[9]
        f2 = g2[1] ^ g2[2] ^ g2[5] ^ g2[7] ^ g2[8] ^ g2[9]
        g1, g2 = [f1] + g1[:9], [f2] + g2[:9]
    return np.array(out)


def st_code():
    """GLONASS ST code (ICD L1/L2 FDMA 3.3.2.2): 1 + x^5 + x^9, all ones, output of the 7th stage"""
    r = [1] * 9  # stages 1..9
    out = []
    for _ in range(511):
        out.append(r[6])
        r = [r[4] ^ r[8]] + r[:8]
    return np.array(out)


def flat_table():
    """(3, 37 * 2046) E/P/L: rows 1..32 C/A, row 35 the ST code (1022 entries), everything else 0"""
    t = np.zeros((3, 37 * HALF), dtype=np.int64)
    for prn in range(1, 33):
        c = 2 * ca_code(prn) - 1
        h = np.arange(HALF)
        for w in range(3):
            t[w, prn * HALF : (prn + 1) * HALF] = c[((h + w) % HALF) >> 1]
    s = 2 * st_code() - 1
    h = np.arange(1022)
    for w in range(3):
        t[w, 35 * HALF : 35 * HALF + 1022] = s[((h + w) % 1022) >> 1]
    return t


def test_code_generators():
    """first ten chips of PRN 1 / 2 / 32 (IS-GPS-200, octal 1440 / 1620 / 1712), ST code balance"""
    for prn, octal in ((1, 0o1440), (2, 0o1620), (32, 0o1712)):
        assert int("".join(map(str, ca_code(prn)[:10])), 2) == octal
    assert st_code().sum() == 256


def _oracle_bits(L, reg, hs):
    return np.array([[L.orc_code_bit(w, reg, int(h)) for h in hs] for w in range(3)])


def _want_bits(t, reg, hs):
    base, end = (35 * HALF, 37 * HALF) if reg == abi.PRN_GLONASS else (reg * HALF, 34 * HALF)
    f = base + np.asarray(hs)
    ok = f < end
    return np.where(ok, t[:, np.where(ok, f, 0)], 0)


def test_gps_rows_spill_over_up_to_row_33_then_zero(oracle_lib):
    L = oracle_lib.Oracle.lib()
    t = flat_table()
    for reg in list(range(1, 34)):
        end_h = 34 * HALF - reg * HALF
        hs = sorted(set(list(range(0, 40)) + list(range(HALF - 20, HALF + 20)) + list(range(end_h - 30, end_h + 30)) +
                        list(range(35 * HALF - reg * HALF - 5, 35 * HALF - reg * HALF + 1030)) + [2 * HALF, 20000, 65535]))
        hs = [h for h in hs if h >= 0]
        got = _oracle_bits(L, reg, hs)
        assert np.array_equal(got, _want_bits(t, reg, hs)), f"PRN register {reg}"
        # the same through orc_code_bits
        for h in hs[::7]:
            assert oracle_lib.Oracle.code_bits(reg, h) == tuple(int(x) for x in _want_bits(t, reg, [h])[:, 0])


def test_gps_register_never_reads_the_glonass_row(oracle_lib):
    """register 33 at half chip 4100 and register 32 at 6200 lie in row 35: the flat table holds ST-code bits there,
    a GPS channel reads 0"""
    t = flat_table()
    for reg, h in ((33, 4100), (32, 6200), (33, 4092), (32, 6138)):
        assert t[:, reg * HALF + h].any()
        assert oracle_lib.Oracle.code_bits(reg, h) == (0, 0, 0), (reg, h)
        assert [oracle_lib.Oracle.lib().orc_code_bit(w, reg, h) for w in range(3)] == [0, 0, 0]


def test_glonass_register_reads_its_st_row_then_zero(oracle_lib):
    L = oracle_lib.Oracle.lib()
    t = flat_table()
    hs = list(range(0, 2 * HALF + 40)) + [4 * HALF, 65535]
    got = _oracle_bits(L, abi.PRN_GLONASS, hs)
    assert np.array_equal(got, _want_bits(t, abi.PRN_GLONASS, hs))
    assert got[:, :1022].all() and not got[:, 1022:].any()
