"""gnssb200_softtrack_state (no GPU): the ctypes mirror matches the header field by field, and gnssb200_softtrack_init
builds the state every channel has before its first code period (tracking.sci:226-250) and validates like
gnssb200_softtrack_batch."""
import ctypes as C
import os
import subprocess
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_state_layout_matches_header():
    from gnss_sdr_ru_b200 import abi

    fields = [f for f, _ in abi.SoftTrackState._fields_]
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "gnssb200.h"\nint main(void){printf("%zu"' + \
        "".join(' " %zu"' for _ in fields) + ", sizeof(gnssb200_softtrack_state)" + \
        "".join(f", offsetof(gnssb200_softtrack_state, {f})" for f in fields) + ");return 0;}\n"
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "s.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), os.path.join(d, "s.c"), "-o", os.path.join(d, "s")])
        out = [int(x) for x in subprocess.check_output([os.path.join(d, "s")]).split()]
    assert out == [C.sizeof(abi.SoftTrackState)] + [getattr(abi.SoftTrackState, f).offset for f in fields]
    assert C.sizeof(abi.SoftTrackState) == 112


def _chans(abi, rows):
    ch = (abi.SoftTrackChan * len(rows))()
    for i, (sv, cp, f) in enumerate(rows):
        ch[i].sv, ch[i].code_phase, ch[i].acquired_freq = sv, cp, f
    return ch


def test_init_states():
    from gnss_sdr_ru_b200 import abi, lib
    from gnss_sdr_ru_b200.softtrack import TrackSettings

    L = lib.lib()
    rows = [(-7, 1, 1e6 - 7 * 562500.0 + 1234.5), (6, 16000, 1e6 + 6 * 562500.0 - 0.25), (0, 8123, 1e6 + 3000.0)]
    ts = TrackSettings(skipNumberOfSamples=48000, msToProcess=20)
    cfg = ts.to_c()
    rec = (C.c_int32 * 3)(2, 0, 2)
    st = (abi.SoftTrackState * 3)()
    assert L.gnssb200_softtrack_init(C.byref(cfg), _chans(abi, rows), rec, 3, 3, st) == 0
    for i, (sv, cp, f) in enumerate(rows):
        s = st[i]
        assert (s.codeFreq, s.remCodePhase, s.carrFreq, s.remCarrPhase) == (0.511e6, 0.0, f, 0.0)
        assert (s.oldCodeNco, s.oldCodeError, s.oldCarrNco, s.oldCarrError) == (0.0, 0.0, 0.0, 0.0)
        assert (s.I1, s.Q1, s.carrFreqBasis) == (0.001, 0.001, f)
        assert (s.pos, s.sv, s.record, s.ms_done, s.status) == (48000 + cp - 1, sv, rec[i], 0, abi.SOFTTRACK_RUNNING)
    # chan_record NULL: every channel in record 0
    assert L.gnssb200_softtrack_init(C.byref(cfg), _chans(abi, rows), None, 1, 3, st) == 0
    assert [s.record for s in st] == [0, 0, 0]


def test_init_invalid_arguments_leave_states_untouched():
    from gnss_sdr_ru_b200 import abi, lib
    from gnss_sdr_ru_b200.softtrack import TrackSettings

    L = lib.lib()
    glo, gps = TrackSettings(msToProcess=5).to_c(), TrackSettings.gps(msToProcess=5).to_c()
    st = (abi.SoftTrackState * 2)()
    C.memset(st, 0x5A, C.sizeof(st))
    before = bytes(st)
    ok = _chans(abi, [(3, 10, 1e6), (5, 20, 2e6)])
    rec = (C.c_int32 * 2)(0, 1)

    def bad(want, cfg, chans=ok, chan_record=rec, n_records=2, n_ch=2, states=st):
        assert L.gnssb200_softtrack_init(C.byref(cfg) if cfg is not None else None, chans, chan_record, n_records, n_ch, states) == want
        assert bytes(st) == before

    bad(-20, None)
    bad(-20, glo, chans=None)
    bad(-20, glo, states=None)
    bad(-20, glo, n_ch=0)
    bad(-20, glo, n_records=0)
    bad(-20, TrackSettings(msToProcess=0).to_c())
    bad(-20, TrackSettings(msToProcess=5, codeLength=1000).to_c())
    bad(-21, gps, chans=_chans(abi, [(3, 10, 1e6), (33, 20, 2e6)]))
    bad(-21, gps, chans=_chans(abi, [(0, 10, 1e6), (5, 20, 2e6)]))
    bad(-24, glo, chan_record=(C.c_int32 * 2)(0, 2))
    bad(-24, glo, chan_record=(C.c_int32 * 2)(-1, 0))
    assert L.gnssb200_softtrack_init(C.byref(gps), ok, rec, 2, 2, st) == 0
