"""Host-side mirror of the Scilab receivers' ``acqResults = acquisition(longSignal, settings)``.

Field and setting names follow SCI/{GPS,GLONASS}/L1/initSettings.sci:41-136 and
acquisition.sci:1-198 (samplingFreq, IF, L1_IF_step, codeFreqBasis, codeLength, acqSearchBand,
acqCohIntegration, acqThreshold, acqSatelliteList / acqFCHList; results carrFreq, codePhase,
peakMetric, freqChannel).  The computation happens in libgnssb200.so (csrc/acq.cu); this module only
marshals arguments.  No CPU implementation exists here.
"""
from __future__ import annotations

import ctypes as C
import sys
from dataclasses import dataclass, field

import numpy as np

from . import abi
from .lib import GnssB200Error, check, lib


@dataclass
class Settings:
    system: str = "gps"
    samplingFreq: float = 16.0e6
    IF: float = 2.42e6
    L1_IF_step: float = 0.0
    codeFreqBasis: float = 1.023e6
    codeLength: int = 1023
    acqSearchBand: float = 14.0
    acqCohIntegration: int = 4
    acqThreshold: float = 3.0
    acqSatelliteList: list = field(default_factory=lambda: list(range(1, 33)))  # acqFCHList for GLONASS
    n_noncoh: int = 0  # extension (BASELINE config 4): sum of K consecutive blocks instead of best-of-two

    @staticmethod
    def gps(**kw):
        return Settings(**kw)

    @staticmethod
    def glonass(**kw):
        d = dict(system="glonass", IF=1.0e6, L1_IF_step=0.5625e6, codeFreqBasis=0.511e6, codeLength=511,
                 acqSearchBand=12.0, acqCohIntegration=5, acqSatelliteList=list(range(-7, 7)))
        d.update(kw)
        return Settings(**d)

    def to_c(self, part_index: int = 0, part_count: int = 0) -> abi.AcqCfg:
        c = abi.AcqCfg()
        c.system = abi.SYS_GPS if self.system == "gps" else abi.SYS_GLONASS
        c.samp_freq = self.samplingFreq
        c.IF = self.IF
        c.IF_step = self.L1_IF_step
        c.code_freq = self.codeFreqBasis
        c.code_length = self.codeLength
        c.search_band_khz = self.acqSearchBand
        c.coh_ms = self.acqCohIntegration
        c.n_noncoh = self.n_noncoh
        c.threshold = self.acqThreshold
        c.n_sv = len(self.acqSatelliteList)
        for i, sv in enumerate(self.acqSatelliteList):
            c.sv[i] = int(sv)
        c.part_index = part_index
        c.part_count = part_count
        return c


def _results(res) -> dict:
    """acqResults fields of a gnssb200_acq_result array (the form acquisition() returns)."""
    return dict(
        carrFreq=np.array([r.carrFreq for r in res]),
        codePhase=np.array([r.codePhase for r in res]),
        peakMetric=np.array([r.peakMetric for r in res]),
        freqChannel=np.array([r.sv for r in res]),
        bin=np.array([r.bin for r in res]),
        codePhaseRaw=np.array([r.codePhaseRaw for r in res]),
        peak=np.array([r.peak for r in res]),
        second=np.array([r.second for r in res]),
    )


class AcquisitionEngine:
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
        if sys is None or sys.is_finalizing():  # CUDA may already be torn down at interpreter exit
            return
        try:
            self.close()
        except Exception:
            pass

    def num_bins(self, settings: Settings) -> int:
        c = settings.to_c()
        return int(self.L.gnssb200_acq_num_bins(C.byref(c)))

    def samples_needed(self, settings: Settings) -> int:
        c = settings.to_c()
        return int(self.L.gnssb200_acq_samples_needed(C.byref(c)))

    def cells(self, settings: Settings) -> int:
        """cells = (#PRN or #FCH) x #Doppler bins x #code phases (SURVEY.md 8d)."""
        return len(settings.acqSatelliteList) * self.num_bins(settings) * 16000

    def acquisition(self, longSignal: np.ndarray, settings: Settings, fmt: int = abi.FMT_INT8_IQ, return_rows=False):
        """longSignal: int8 interleaved I,Q host array (or packed bytes with fmt=FMT_PACKED2)."""
        c = settings.to_c()
        buf = np.ascontiguousarray(longSignal)
        n_samples = buf.size // 2 if fmt == abi.FMT_INT8_IQ else buf.size * 2
        n_sv = len(settings.acqSatelliteList)
        res = (abi.AcqResult * n_sv)()
        nb = self.num_bins(settings)
        rows = np.zeros((n_sv, nb), dtype=abi.ACQ_ROW_DTYPE)
        check(self.L.gnssb200_acq_pcps_host(self.h, C.byref(c), buf.ctypes.data, fmt, n_samples, res, rows.ctypes.data),
              "gnssb200_acq_pcps_host")
        out = _results(res)
        if return_rows:
            out["rows"] = rows
        return out

    def search_device(self, d_iq_ptr: int, n_samples: int, settings: Settings, d_rows_ptr: int, fmt: int = abi.FMT_INT8_IQ,
                      part_index: int = 0, part_count: int = 0, stream: int = 0):
        c = settings.to_c(part_index, part_count)
        check(self.L.gnssb200_acq_search(self.h, C.byref(c), d_iq_ptr, fmt, n_samples, d_rows_ptr, stream or None),
              "gnssb200_acq_search")

    def search_batch_device(self, d_iq_ptr: int, stride: int, n_records: int, n_samples: int, settings: Settings, d_rows_ptr: int,
                            fmt: int = abi.FMT_INT8_IQ, part_index: int = 0, part_count: int = 0, stream: int = 0):
        """gnssb200_acq_search_batch: record r at d_iq_ptr + r*stride (stride 0: one record searched n_records times),
        row tables [n_records][n_sv][n_bins] at d_rows_ptr.  Asynchronous on `stream`."""
        c = settings.to_c(part_index, part_count)
        check(self.L.gnssb200_acq_search_batch(self.h, C.byref(c), d_iq_ptr, stride, n_records, fmt, n_samples, d_rows_ptr,
                                               stream or None), "gnssb200_acq_search_batch")

    def acquisition_batch(self, d_iq_ptr: int, stride: int, n_records: int, n_samples: int, settings: Settings,
                          fmt: int = abi.FMT_INT8_IQ, return_rows=False):
        """acquisition() of n_records device-resident records in one batched search: one copy of all row tables to the
        host, then the peak / second-peak / threshold logic per record.  Returns one dict per record."""
        import torch

        nb = self.num_bins(settings)
        n_sv = len(settings.acqSatelliteList)
        dev = torch.device("cuda", torch.cuda.current_device())
        d_rows = torch.empty(n_records * n_sv * nb * np.dtype(abi.ACQ_ROW_DTYPE).itemsize, dtype=torch.uint8, device=dev)
        self.search_batch_device(d_iq_ptr, stride, n_records, n_samples, settings, d_rows.data_ptr(), fmt=fmt,
                                 stream=torch.cuda.current_stream().cuda_stream)
        rows = d_rows.cpu().numpy().view(abi.ACQ_ROW_DTYPE).reshape(n_records, n_sv, nb)
        outs = []
        for r in range(n_records):
            res, _ = self.finalize(settings, rows[r])
            out = _results(res)
            if return_rows:
                out["rows"] = rows[r]
            outs.append(out)
        return outs

    def finalize(self, settings: Settings, rows: np.ndarray):
        c = settings.to_c()
        n_sv = len(settings.acqSatelliteList)
        res = (abi.AcqResult * n_sv)()
        r = np.ascontiguousarray(rows)
        amb = self.L.gnssb200_acq_finalize(C.byref(c), r.ctypes.data, res)
        return res, amb

    def acquisition_distributed(self, d_iq_ptr: int, n_samples: int, settings: Settings, fmt: int = abi.FMT_INT8_IQ, group=None,
                                return_rows=False):
        """acquisition() with the (sv, Doppler bin) grid sharded over the ranks of a torch.distributed group (one
        process per GPU, the record resident on every GPU): this rank searches rows r % world == rank, one all-gather
        of the 16-byte row tables (NCCL when the group is an NCCL group), then every rank runs the same peak /
        second-peak / threshold logic on the merged table.  Returns the same dict as acquisition() on every rank."""
        import torch
        import torch.distributed as dist

        from .partition import merge_row_tables

        world = dist.get_world_size(group)
        rank = dist.get_rank(group)
        nb = self.num_bins(settings)
        n_sv = len(settings.acqSatelliteList)
        dev = torch.device("cuda", torch.cuda.current_device())
        rows = torch.zeros(n_sv * nb * np.dtype(abi.ACQ_ROW_DTYPE).itemsize, dtype=torch.uint8, device=dev)
        self.search_device(d_iq_ptr, n_samples, settings, rows.data_ptr(), fmt=fmt, part_index=rank, part_count=world,
                           stream=torch.cuda.current_stream().cuda_stream)
        gathered = torch.empty(world * rows.numel(), dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(gathered, rows, group=group)
        merged = merge_row_tables(gathered.cpu().numpy().view(abi.ACQ_ROW_DTYPE).reshape(world, n_sv * nb))
        res, _ = self.finalize(settings, merged)
        out = _results(res)
        if return_rows:
            out["rows"] = merged.reshape(n_sv, nb)
        return out

    def last_kernel_ms(self) -> float:
        return float(self.L.gnssb200_last_kernel_ms(self.h))

    def launch_count(self) -> int:
        return int(self.L.gnssb200_launch_count(self.h))
