"""Host-side mirror of the Scilab receivers' ``[trackResults, channel] = tracking(fid, channel, settings)``
and ``channel = preRun(acqResults, settings)`` (SCI/GLONASS/L1/tracking.sci, include/preRun.sci:66-81).
Setting and result field names follow the reference; the computation is csrc/softtrack.cu."""
from __future__ import annotations

import ctypes as C
import sys
from dataclasses import dataclass

import numpy as np

from . import abi
from .lib import GnssB200Error, check, lib


@dataclass
class TrackSettings:
    system: str = "glonass"
    samplingFreq: float = 16e6
    IF: float = 1e6
    L1_IF_step: float = 0.5625e6
    GLONASS_zero_channel: float = 1602e6
    codeFreqBasis: float = 0.511e6
    codeLength: int = 511
    skipNumberOfSamples: int = 0
    msToProcess: int = 1000
    numberOfChannels: int = 8
    dllDampingRatio: float = 0.7
    dllNoiseBandwidth: float = 0.5
    dllCorrelatorSpacing: float = 0.05
    pllNoiseBandwidth: float = 25.0
    fllNoiseBandwidth: float = 250.0

    @staticmethod
    def gps(**kw):
        d = dict(system="gps", IF=2.42e6, L1_IF_step=0.0, codeFreqBasis=1.023e6, codeLength=1023,
                 dllNoiseBandwidth=0.1, dllCorrelatorSpacing=0.2)  # SCI/GPS/L1/initSettings.sci:91-98
        d.update(kw)
        return TrackSettings(**d)

    def to_c(self) -> abi.SoftTrackCfg:
        c = abi.SoftTrackCfg()
        c.system = abi.SYS_GPS if self.system == "gps" else abi.SYS_GLONASS
        c.code_length = self.codeLength
        c.samp_freq = self.samplingFreq
        c.IF = self.IF
        c.IF_step = self.L1_IF_step
        c.glonass_zero_channel = self.GLONASS_zero_channel
        c.code_freq = self.codeFreqBasis
        c.dll_damping_ratio = self.dllDampingRatio
        c.dll_noise_bandwidth = self.dllNoiseBandwidth
        c.dll_correlator_spacing = self.dllCorrelatorSpacing
        c.pll_noise_bandwidth = self.pllNoiseBandwidth
        c.fll_noise_bandwidth = self.fllNoiseBandwidth
        c.skip_samples = self.skipNumberOfSamples
        c.ms_to_process = self.msToProcess
        return c


def preRun(acqResults: dict, settings: TrackSettings) -> list:
    """Channel list from acquisition results, strongest peakMetric first (preRun.sci:66-81)."""
    order = np.argsort(-np.asarray(acqResults["peakMetric"]), kind="stable")
    n = min(settings.numberOfChannels, int(np.sum(np.asarray(acqResults["carrFreq"]) != 0)))
    return [dict(SVN=int(i) + 1, FCH=int(acqResults["freqChannel"][i]), acquiredFreq=float(acqResults["carrFreq"][i]),
                 codePhase=int(acqResults["codePhase"][i]), status="T") for i in order[:n]]


def _track_results(out: np.ndarray, done: np.ndarray, channel: list) -> list:
    """trackResults dicts of the rows [n_ch][ms][13] and periods done [n_ch] of the channels in `channel`."""
    res = []
    for i, c in enumerate(channel):
        r = {f: out[i, : done[i], k].copy() for k, f in enumerate(abi.SOFTTRACK_FIELDS)}
        r["SVN"], r["FCH"], r["status"] = c.get("SVN", 0), c["FCH"], c.get("status", "T")
        res.append(r)
    return res


def _per_record(out: np.ndarray, done: np.ndarray, channels: list) -> list:
    """One trackResults list per record from the rows and periods of the flat channel list."""
    res, i = [], 0
    for chl in channels:
        res.append(_track_results(out[i : i + len(chl)], done[i : i + len(chl)], chl))
        i += len(chl)
    return res


def _flat_channels(channels: list, n_records: int):
    """The channel table and chan_record of one preRun channel list per record, flattened record by record."""
    if len(channels) != n_records:
        raise ValueError("channels must hold one channel list per record")
    flat = [(r, c) for r, chl in enumerate(channels) for c in chl]
    ch = (abi.SoftTrackChan * len(flat))()
    rec = (C.c_int32 * len(flat))()
    for i, (r, c) in enumerate(flat):
        ch[i].sv = c["FCH"]
        ch[i].code_phase = c["codePhase"]
        ch[i].acquired_freq = c["acquiredFreq"]
        rec[i] = r
    return ch, rec


class SoftTrackingEngine:
    def __init__(self, device: int = 0, handle=None):
        self.L = lib()
        self._own = handle is None
        if handle is None:
            handle = self.L.gnssb200_open(device, None)
            if not handle:
                raise GnssB200Error("gnssb200_open failed: " + (self.L.gnssb200_last_error_string() or b"?").decode())
        self.h = handle

    def close(self):
        if self._own and self.h:
            self.L.gnssb200_close(self.h)
        self.h = None

    def __del__(self):
        if sys is None or sys.is_finalizing():
            return
        try:
            self.close()
        except Exception:
            pass

    def tracking_device(self, d_iq_ptr: int, n_samples: int, channel: list, settings: TrackSettings, d_out_ptr: int,
                        d_ms_done_ptr: int, stream: int = 0):
        ch = (abi.SoftTrackChan * len(channel))()
        for i, c in enumerate(channel):
            ch[i].sv = c["FCH"]
            ch[i].code_phase = c["codePhase"]
            ch[i].acquired_freq = c["acquiredFreq"]
        cfg = settings.to_c()
        check(self.L.gnssb200_softtrack(self.h, C.byref(cfg), d_iq_ptr, n_samples, ch, len(channel), d_out_ptr, d_ms_done_ptr,
                                        stream or None), "gnssb200_softtrack")

    def tracking(self, iq_int8: np.ndarray, channel: list, settings: TrackSettings) -> list:
        """Host record in, list of trackResults dicts (one per channel) out."""
        import torch

        buf = np.ascontiguousarray(iq_int8, dtype=np.int8)
        d_iq = torch.from_numpy(buf.view(np.uint8)).cuda()
        n_ch = len(channel)
        d_out = torch.zeros((n_ch, settings.msToProcess, 13), dtype=torch.float64, device="cuda")
        d_done = torch.zeros(n_ch, dtype=torch.int32, device="cuda")
        self.tracking_device(d_iq.data_ptr(), buf.size // 2, channel, settings, d_out.data_ptr(), d_done.data_ptr())
        return _track_results(d_out.cpu().numpy(), d_done.cpu().numpy(), channel)

    def tracking_batch_device(self, d_iq_ptr: int, stride: int, n_records: int, n_samples: int, channels: list,
                              settings: TrackSettings, d_out_ptr: int, d_ms_done_ptr: int, fmt: int = abi.FMT_INT8_IQ,
                              stream: int = 0):
        """gnssb200_softtrack_batch: record r at d_iq_ptr + r*stride (stride 0: one record n_records times) in fmt
        (FMT_INT8_IQ or FMT_PACKED2).  channels holds one preRun channel list per record; they are tracked as one
        flat list, record by record, into d_out [n_ch][msToProcess][13] and d_ms_done [n_ch].  Synchronous on `stream`."""
        ch, rec = _flat_channels(channels, n_records)
        cfg = settings.to_c()
        check(self.L.gnssb200_softtrack_batch(self.h, C.byref(cfg), d_iq_ptr, stride, n_records, fmt, n_samples, ch, rec, len(ch),
                                              d_out_ptr, d_ms_done_ptr, stream or None), "gnssb200_softtrack_batch")

    def tracking_batch(self, d_iq_ptr: int, stride: int, n_records: int, n_samples: int, channels: list, settings: TrackSettings,
                       fmt: int = abi.FMT_INT8_IQ) -> list:
        """tracking() of n_records device-resident records in one call: one list of trackResults dicts per record."""
        import torch

        n_ch = sum(len(chl) for chl in channels)
        if len(channels) != n_records:
            raise ValueError("channels must hold one channel list per record")
        if n_ch == 0:
            return [[] for _ in channels]
        dev = torch.device("cuda", torch.cuda.current_device())
        d_out = torch.zeros((n_ch, settings.msToProcess, 13), dtype=torch.float64, device=dev)
        d_done = torch.zeros(n_ch, dtype=torch.int32, device=dev)
        self.tracking_batch_device(d_iq_ptr, stride, n_records, n_samples, channels, settings, d_out.data_ptr(), d_done.data_ptr(),
                                   fmt=fmt, stream=torch.cuda.current_stream().cuda_stream)
        return _per_record(d_out.cpu().numpy(), d_done.cpu().numpy(), channels)

    def init_states(self, channels: list, settings: TrackSettings, n_records: int):
        """gnssb200_softtrack_init: the state of every channel before its first code period, as a ctypes array of
        abi.SoftTrackState (host memory).  channels holds one preRun channel list per record, flattened record by record
        as in tracking_batch_device."""
        ch, rec = _flat_channels(channels, n_records)
        states = (abi.SoftTrackState * len(ch))()
        cfg = settings.to_c()
        check(self.L.gnssb200_softtrack_init(C.byref(cfg), ch, rec, n_records, len(ch), states), "gnssb200_softtrack_init")
        return states

    def resume_device(self, d_win_ptr: int, win_stride: int, n_records: int, fmt: int, win_first: int, win_samples: int,
                      record_samples: int, settings: TrackSettings, d_state_ptr: int, n_ch: int, d_out_ptr: int, stream: int = 0):
        """gnssb200_softtrack_resume: continue the n_ch device states d_state_ptr through samples [win_first, win_first +
        win_samples) of every record (record r's window at d_win_ptr + r*win_stride), rows into d_out [n_ch][msToProcess][13].
        Asynchronous on `stream`."""
        cfg = settings.to_c()
        check(self.L.gnssb200_softtrack_resume(self.h, C.byref(cfg), d_win_ptr, win_stride, n_records, fmt, win_first, win_samples,
                                               record_samples, d_state_ptr, n_ch, d_out_ptr, stream or None),
              "gnssb200_softtrack_resume")

    def tracking_batch_host(self, h_iq, stride: int, n_records: int, n_samples: int, channels: list, settings: TrackSettings,
                            fmt: int = abi.FMT_INT8_IQ, window_samples: int = 0) -> list:
        """tracking_batch on records in host memory (a numpy array or a CPU torch tensor, pinned for copies that overlap
        the tracking), staged window by window: one list of trackResults dicts per record.  The number of channels
        stopped because a block was longer than the windows' overlap (normally 0) is left in self.host_stopped."""
        if hasattr(h_iq, "data_ptr"):
            if h_iq.is_cuda or not h_iq.is_contiguous():
                raise ValueError("h_iq must be a contiguous host tensor")
            ptr = h_iq.data_ptr()
        else:
            h_iq = np.ascontiguousarray(h_iq)
            ptr = h_iq.ctypes.data
        ch, rec = _flat_channels(channels, n_records)
        n_ch = len(ch)
        if n_ch == 0:
            return [[] for _ in channels]
        out = np.zeros((n_ch, settings.msToProcess, 13), dtype=np.float64)
        done = np.zeros(n_ch, dtype=np.int32)
        cfg = settings.to_c()
        rc = self.L.gnssb200_softtrack_batch_host(self.h, C.byref(cfg), ptr, stride, n_records, fmt, n_samples, ch, rec, n_ch,
                                                  out.ctypes.data, done.ctypes.data, window_samples)
        if rc < 0:
            check(rc, "gnssb200_softtrack_batch_host")
        self.host_stopped = rc
        return _per_record(out, done, channels)

    def set_width(self, threads: int):
        """Threads per channel of the batched call: 0 automatic, 128, 256 or 512.  Results do not depend on it."""
        check(self.L.gnssb200_set_softtrack_width(self.h, threads), "gnssb200_set_softtrack_width")

    def last_kernel_ms(self) -> float:
        return float(self.L.gnssb200_last_kernel_ms(self.h))
