"""Host-side mirror of the reference receiver's correlator / channel interface, backed by the GPU.

Names follow the reference (OSG/gp2021/gp2021.h:7-18, OSG/correlator/correlator.h:8-9,
OSG/osgnss_next_step.c:41-84): ``ch_cntl``, ``ch_carrier``, ``ch_code``, ``ch_code_slew``,
``ch_epoch_load``, ``simple_cold_allocate``, ``correlator_init``, ``Sim_GP2021_int``.

* :class:`DropInCorrelator` -- the library's drop-in symbols exactly as the reference C host would
  call them (one receiver, one block per call, host buffers).
* :class:`TrackingEngine` -- the batched closed loop: S receivers x 12 channels resident on the GPU.
"""
from __future__ import annotations

import ctypes as C
import sys

import numpy as np

from . import abi
from .lib import GnssB200Error, check, default_cfg, lib

NSAMP_DEFAULT = 8192  # SAMP_RATE*interr_int/1e6, OSG/osgnss_next_step.c:150


class DropInCorrelator:
    """correlator_init / Sim_GP2021_int / REG_read / REG_write of libgnssb200.so (process-global)."""

    def __init__(self, tic_period: float = 0.0):
        self.L = lib()
        self.REG_read = (C.c_int * 256).in_dll(self.L, "REG_read")
        self.REG_write = (C.c_int * 256).in_dll(self.L, "REG_write")
        C.memset(self.REG_read, 0, 1024)
        C.memset(self.REG_write, 0, 1024)
        self.cfg = default_cfg(tic_period=tic_period)
        self.L.correlator_init(C.c_double(tic_period))

    # register accessors with the reference's masking (gp2021.c:11-14): data -> unsigned short
    def _put(self, addr: int, data: int):
        self.REG_write[addr] = data & 0xFFFF

    def ch_cntl(self, ch, data):
        self._put(ch << 3, data)

    def ch_code_slew(self, ch, data):
        self._put((ch << 3) + 0x84, data)

    def ch_epoch_load(self, ch, data):
        self._put((ch << 3) + 7, data)

    def _nco(self, addr, freq, bits):
        w = int(freq) << (32 - bits)
        w = int(float(w) * self.cfg.clock_mult)
        self._put(addr, w >> 16)
        self._put(addr + 1, w & 0xFFFF)

    def ch_carrier(self, ch, freq):
        self._nco((ch << 3) + 3, freq, self.cfg.carrier_nco_bits)

    def ch_code(self, ch, freq):
        self._nco((ch << 3) + 5, freq, self.cfg.code_nco_bits)

    def Sim_GP2021_int(self, IF: np.ndarray, nsamp: int):
        buf = np.ascontiguousarray(IF, dtype=np.int8)
        self.L.Sim_GP2021_int(buf.ctypes.data, nsamp)

    def regs(self):
        return np.array(self.REG_read[:], dtype=np.int32), np.array(self.REG_write[:], dtype=np.int32)


class TrackingEngine:
    """S independent receivers (IF streams) x 12 channels, closed loop on one GPU."""

    def __init__(self, n_streams: int = 1, device: int = 0, cfg: abi.Cfg | None = None):
        self.L = lib()
        self.cfg = cfg if cfg is not None else default_cfg()
        self.h = self.L.gnssb200_open(device, C.byref(self.cfg))
        if not self.h:
            raise GnssB200Error(
                "gnssb200_open failed: " + (self.L.gnssb200_last_error_string() or b"?").decode()
            )
        self.n_streams = n_streams
        check(self.L.gnssb200_set_streams(self.h, n_streams), "gnssb200_set_streams")
        self.rx = (abi.Rx * n_streams)()
        for s in range(n_streams):
            self.L.gnssb200_rx_init(C.byref(self.rx[s]), C.byref(self.cfg))

    def close(self):
        if self.h:
            self.L.gnssb200_close(self.h)
            self.h = None

    def __del__(self):
        if sys is None or sys.is_finalizing():  # CUDA may already be torn down at interpreter exit
            return
        try:
            self.close()
        except Exception:
            pass

    # ---- reference-named host helpers, acting on the host copy of receiver `s` -------------
    def simple_cold_allocate(self, s: int, prns):
        arr = (C.c_int32 * abi.N_CHANNELS)(*prns)
        self.L.gnssb200_rx_cold_allocate(C.byref(self.rx[s]), C.byref(self.cfg), arr)

    def ch_cntl(self, s, ch, data):
        self.L.gnssb200_ch_cntl(C.byref(self.rx[s]), ch, data)

    def ch_carrier(self, s, ch, freq):
        self.L.gnssb200_ch_carrier(C.byref(self.rx[s]), C.byref(self.cfg), ch, freq)

    def ch_code(self, s, ch, freq):
        self.L.gnssb200_ch_code(C.byref(self.rx[s]), C.byref(self.cfg), ch, freq)

    def ch_code_slew(self, s, ch, data):
        self.L.gnssb200_ch_code_slew(C.byref(self.rx[s]), ch, data)

    def ch_epoch_load(self, s, ch, data):
        self.L.gnssb200_ch_epoch_load(C.byref(self.rx[s]), ch, data)

    def warm_start(self, s: int, ch: int, n_freq: int):
        """Put a searching channel at the start of Doppler bin `n_freq`, as ch_acq
        (osgpsisr.c:443-449) leaves it when it enters that bin."""
        k = self.rx[s].chan[ch]
        k.n_freq = n_freq
        # del_freq sequence 1,-2,3,-4..: after reaching n the next step is -(2n) for n>0, 1-2n for n<=0
        k.del_freq = -2 * n_freq if n_freq > 0 else 1 - 2 * n_freq
        ref = self.cfg.glonass_carrier_ref if k.system else self.cfg.gps_carrier_ref
        k.carrier_freq = ref + k.carrier_cold_corr + self.cfg.d_freq * n_freq
        k.codes = 0
        self.ch_carrier(s, ch, k.carrier_freq)

    def set_glonass_channel(self, s: int, ch: int, fch: int):
        """Frequency channel of a GLONASS correlator channel (allocated with PRN register abi.PRN_GLONASS): the FDMA
        offset fch * 562.5 kHz in carrier-NCO units goes into carrier_cold_corr -- the correction the channel logic adds
        to the reference word (osgpsisr.c:446,454); the firmware's GLNS_L1_CARR_REF_STEP = 7549747 at 16 MHz x 5."""
        k = self.rx[s].chan[ch]
        res = self.cfg.clock_mult * self.cfg.samp_rate / 2.0 ** self.cfg.carrier_nco_bits
        k.carrier_cold_corr = int(fch * int(562500.0 / res))
        self.ch_carrier(s, ch, self.cfg.glonass_carrier_ref + k.carrier_cold_corr)

    def acq_allocate(self, s: int, result: dict, settings) -> list:
        """gnssb200_rx_acq_allocate on the host copy of receiver `s` (freshly initialised): channels from one record's
        acquisition result (a dict as AcquisitionEngine.acquisition returns it, for the same acquisition `settings`),
        detected satellites strongest first.  Returns the PRN / frequency channel of each allocated channel."""
        n_sv = len(settings.acqSatelliteList)
        res = (abi.AcqResult * n_sv)()
        for i in range(n_sv):
            r = res[i]
            r.carrFreq = float(result["carrFreq"][i])
            r.codePhase = int(result["codePhase"][i])
            r.sv = int(result["freqChannel"][i])
            r.peakMetric = float(result["peakMetric"][i])
            r.bin = int(result["bin"][i])
            r.codePhaseRaw = int(result["codePhaseRaw"][i])
            r.peak = float(result["peak"][i])
            r.second = float(result["second"][i])
        c = settings.to_c()
        sv_out = (C.c_int32 * abi.N_CHANNELS)()
        n = self.L.gnssb200_rx_acq_allocate(C.byref(self.rx[s]), C.byref(self.cfg), C.byref(c), res, sv_out)
        if n < 0:
            check(n, "gnssb200_rx_acq_allocate")
        return [int(v) for v in sv_out[:n]]

    def upload(self):
        check(self.L.gnssb200_upload_rx(self.h, 0, self.n_streams, C.addressof(self.rx)), "gnssb200_upload_rx")

    def download(self):
        check(self.L.gnssb200_download_rx(self.h, 0, self.n_streams, C.addressof(self.rx)), "gnssb200_download_rx")

    # ---- runs ----------------------------------------------------------------------------
    def set_stage_blocks(self, blocks: int):
        """blocks per stream and staging chunk of run_host (0 = automatic); results do not depend on it"""
        check(self.L.gnssb200_set_stage_blocks(self.h, blocks), "gnssb200_set_stage_blocks")

    def readback_fallbacks(self) -> int:
        return int(self.L.gnssb200_readback_fallbacks(self.h))

    def run_host(self, iq: np.ndarray, nblocks: int, nsamp: int = NSAMP_DEFAULT, fmt: int = abi.FMT_INT8_IQ,
                 dump_cap: int = 0):
        """iq: (S, bytes) host array.  Returns (dumps[S,12,cap], counts[S,12]) when dump_cap > 0."""
        buf = np.ascontiguousarray(iq)
        if buf.ndim == 1:
            buf = buf.reshape(1, -1)
        assert buf.shape[0] == self.n_streams
        dumps = cnt = None
        dp = cp = None
        if dump_cap:
            dumps = np.zeros((self.n_streams, abi.N_CHANNELS, dump_cap), dtype=abi.DUMP_DTYPE)
            cnt = np.zeros((self.n_streams, abi.N_CHANNELS), dtype=np.int32)
            dp, cp = dumps.ctypes.data, cnt.ctypes.data
        check(
            self.L.gnssb200_track_run_host(self.h, buf.ctypes.data, buf.strides[0], fmt, nsamp, nblocks, dp, dump_cap, cp),
            "gnssb200_track_run_host",
        )
        return dumps, cnt

    def run_device(self, d_if_ptr: int, stride: int, nblocks: int, nsamp: int = NSAMP_DEFAULT,
                   fmt: int = abi.FMT_INT8_IQ, d_dumps_ptr: int = 0, dump_cap: int = 0, d_count_ptr: int = 0,
                   stream: int = 0):
        """Asynchronous run on device-resident samples (raw device pointers, e.g. tensor.data_ptr())."""
        check(
            self.L.gnssb200_track_run(self.h, d_if_ptr, stride, fmt, nsamp, nblocks, d_dumps_ptr or None, dump_cap,
                                      d_count_ptr or None, stream or None),
            "gnssb200_track_run",
        )

    def set_track_slice(self, blocks: int):
        """blocks per work-queue slice of the tracking kernel (0 = automatic); results do not depend on it"""
        check(self.L.gnssb200_set_track_slice(self.h, blocks), "gnssb200_set_track_slice")

    def set_track_variant(self, form: int = 0, occ: int = 0):
        """kernel form (0 auto, 1 barrier kernel, 2 fixed sample runs, 3/4/5 half-chip segments x 96/192/384 threads) and
        occupancy variant (0 auto); results do not depend on it"""
        check(self.L.gnssb200_set_track_variant(self.h, form, occ), "gnssb200_set_track_variant")

    def launch_count(self) -> int:
        return int(self.L.gnssb200_launch_count(self.h))

    def last_kernel_ms(self) -> float:
        return float(self.L.gnssb200_last_kernel_ms(self.h))


def acq_serial(handle, d_if_ptr: int, fmt: int, n_samples: int, prn_list, search_max_f: int = 5, max_prn_delay: int = 2045,
               cells_cap: int = 4096):
    """gnssb200_acq_serial: exhaustive GP2021-semantics serial-search cell map of a device-resident record.
    Returns {prn: structured array of (prn, n_freq, codes, ip, qp, rss)}."""
    L = lib()
    prn = np.ascontiguousarray(prn_list, dtype=np.int32)
    cells = np.zeros((len(prn), cells_cap), dtype=abi.SERIAL_CELL_DTYPE)
    n = np.zeros(len(prn), dtype=np.int32)
    check(L.gnssb200_acq_serial(handle, d_if_ptr, fmt, n_samples, prn.ctypes.data, len(prn), search_max_f, max_prn_delay, cells.ctypes.data,
                                cells_cap, n.ctypes.data), "gnssb200_acq_serial")
    return {int(p): cells[i, : n[i]].copy() for i, p in enumerate(prn)}


def acq_serial_distributed(handle, d_if_ptr: int, fmt: int, n_samples: int, prn_list, search_max_f: int = 5, max_prn_delay: int = 2045,
                           cells_cap: int = 4096, group=None):
    """acq_serial with the PRN list sharded over the ranks of a torch.distributed group (entry i on rank i % world, the
    record resident on every GPU) and one all-gather of the cell tables; every rank returns the complete map."""
    import torch
    import torch.distributed as dist

    from .partition import merge_cell_maps, prns_of_rank

    world, rank = dist.get_world_size(group), dist.get_rank(group)
    mine = prns_of_rank(list(prn_list), rank, world)
    per_rank = (len(prn_list) + world - 1) // world
    cells = np.zeros((per_rank, cells_cap), dtype=abi.SERIAL_CELL_DTYPE)
    n = np.zeros(per_rank, dtype=np.int32)
    if mine:
        got = acq_serial(handle, d_if_ptr, fmt, n_samples, mine, search_max_f, max_prn_delay, cells_cap)
        for j, p in enumerate(mine):
            n[j] = len(got[p])
            cells[j, : n[j]] = got[p]
    dev = torch.device("cuda", torch.cuda.current_device())
    t_cells = torch.from_numpy(cells.view(np.uint8).reshape(-1)).to(dev)
    t_n = torch.from_numpy(n).to(dev)
    g_cells = torch.empty(world * t_cells.numel(), dtype=torch.uint8, device=dev)
    g_n = torch.empty(world * per_rank, dtype=torch.int32, device=dev)
    dist.all_gather_into_tensor(g_cells, t_cells, group=group)
    dist.all_gather_into_tensor(g_n, t_n, group=group)
    gc = g_cells.cpu().numpy().view(abi.SERIAL_CELL_DTYPE).reshape(world, per_rank, cells_cap)
    return merge_cell_maps(gc, g_n.cpu().numpy().reshape(world, per_rank), list(prn_list), world)


def serial_search_cell_map(dumps: np.ndarray, counts: np.ndarray):
    """Turn the dump records of a run with the detection threshold out of reach into the GP2021-semantics
    search cell map {(stream, channel): array of (n_freq, code delay in half chips, IP, QP, rss)}.
    One dump = one cell (SURVEY.md Appendix A, "serial-search schedule"); the record of a dump carries the
    bin / delay the channel moved to AFTER the dump, so cell k is described by record k-1."""
    out = {}
    S, nch, _ = dumps.shape
    for s in range(S):
        for ch in range(nch):
            d = dumps[s, ch, : counts[s, ch]]
            if len(d) < 2:
                continue
            ip = d["acc"][1:, 2].astype(np.int64)
            qp = d["acc"][1:, 3].astype(np.int64)
            a, b = np.abs(ip), np.abs(qp)
            rss = np.where(a > b, a + (b >> 1), b + (a >> 1))  # rss(), osgpsisr.c:77-91
            out[(s, ch)] = np.stack([d["n_freq"][:-1].astype(np.int64), d["codes"][:-1].astype(np.int64), ip, qp, rss], axis=1)
    return out
