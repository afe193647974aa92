"""Loader for libgnssb200.so (the C ABI of include/gnssb200.h).

The library is built in-tree by ``gnss_sdr_ru_b200/csrc/build.sh`` (nvcc, sm_100a).  There is no
CPU implementation behind this module: if the shared object is missing, or no CUDA device can be
opened, the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

from . import abi

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# GNSSB200_LIB: another build of the same library (A/B timing of kernel variants, tools/ab_variants.sh); still no CPU path
SO_PATH = os.environ.get("GNSSB200_LIB") or os.path.join(PKG_DIR, "libgnssb200.so")

_lib = None


class GnssB200Error(RuntimeError):
    pass


def build(force: bool = False) -> str:
    """Compile the CUDA extension for sm_100a (works without a GPU: nvcc cross-compiles)."""
    script = os.path.join(PKG_DIR, "csrc", "build.sh")
    if force:
        subprocess.check_call(["rm", "-rf", os.path.join(PKG_DIR, "csrc", "build")])
    subprocess.check_call(["bash", script], stdout=subprocess.DEVNULL)
    return SO_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise GnssB200Error(
            f"{SO_PATH} is missing: build it with gnss_sdr_ru_b200/csrc/build.sh (there is no CPU fallback)"
        )
    L = C.CDLL(SO_PATH)  # RTLD_LOCAL: the drop-in symbols must not interpose on other libraries in the process
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    P = C.POINTER
    L.gnssb200_last_error.restype = C.c_int
    L.gnssb200_last_error_string.restype = C.c_char_p
    L.gnssb200_cfg_default.argtypes = [P(abi.Cfg)]
    L.gnssb200_cfg_derive.argtypes = [P(abi.Cfg)]
    L.gnssb200_rx_init.argtypes = [P(abi.Rx), P(abi.Cfg)]
    L.gnssb200_rx_cold_allocate.argtypes = [P(abi.Rx), P(abi.Cfg), P(i32)]
    L.gnssb200_ch_cntl.argtypes = [P(abi.Rx), C.c_int, C.c_int]
    L.gnssb200_ch_carrier.argtypes = [P(abi.Rx), P(abi.Cfg), C.c_int, i64]
    L.gnssb200_ch_code.argtypes = [P(abi.Rx), P(abi.Cfg), C.c_int, i64]
    L.gnssb200_ch_code_slew.argtypes = [P(abi.Rx), C.c_int, C.c_int]
    L.gnssb200_ch_epoch_load.argtypes = [P(abi.Rx), C.c_int, C.c_uint]
    L.gnssb200_open.argtypes = [C.c_int, P(abi.Cfg)]
    L.gnssb200_open.restype = vp
    L.gnssb200_close.argtypes = [vp]
    L.gnssb200_set_streams.argtypes = [vp, C.c_int]
    L.gnssb200_upload_rx.argtypes = [vp, C.c_int, C.c_int, vp]
    L.gnssb200_download_rx.argtypes = [vp, C.c_int, C.c_int, vp]
    L.gnssb200_track_run.argtypes = [vp, vp, C.c_size_t, C.c_int, C.c_int, i64, vp, C.c_int, vp, vp]
    L.gnssb200_set_stage_blocks.argtypes = [vp, i64]
    L.gnssb200_readback_fallbacks.argtypes = [vp]
    L.gnssb200_readback_fallbacks.restype = i64
    L.gnssb200_track_run_host.argtypes = [vp, vp, C.c_size_t, C.c_int, C.c_int, i64, vp, C.c_int, vp]
    L.gnssb200_set_track_slice.argtypes = [vp, i64]
    L.gnssb200_set_track_variant.argtypes = [vp, C.c_int, C.c_int]
    L.gnssb200_track_check_failures.argtypes = [vp]
    L.gnssb200_acq_serial.argtypes = [vp, vp, C.c_int, i64, vp, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp]
    L.gnssb200_launch_count.argtypes = [vp]
    L.gnssb200_launch_count.restype = i64
    L.gnssb200_last_kernel_ms.argtypes = [vp]
    L.gnssb200_last_kernel_ms.restype = C.c_float
    L.gnssb200_synth.argtypes = [vp, vp, C.c_size_t, C.c_int, C.c_int, i64, vp, C.c_int, C.c_uint64, vp]
    L.gnssb200_softtrack.argtypes = [vp, P(abi.SoftTrackCfg), vp, i64, vp, C.c_int, vp, vp, vp]
    L.gnssb200_isr_math_eval.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp]
    for f in (L.gnssb200_find_preambles, L.gnssb200_find_time_marks):
        f.argtypes = [vp, vp, C.c_int, i64, i64, C.c_int, C.c_int, vp, vp, vp, vp]
    L.gnssb200_ingest_open.argtypes = [vp, C.c_int, C.c_int, C.c_int, i64, C.c_int]
    L.gnssb200_ingest_open.restype = vp
    L.gnssb200_ingest_close.argtypes = [vp]
    L.gnssb200_ingest_write.argtypes = [vp, vp, i64]
    L.gnssb200_ingest_write.restype = i64
    L.gnssb200_ingest_finish.argtypes = [vp]
    L.gnssb200_ingest_pump.argtypes = [vp, i64]
    L.gnssb200_ingest_pump.restype = i64
    L.gnssb200_ingest_status.argtypes = [vp, P(abi.IngestStat)]
    L.gnssb200_ingest_sync.argtypes = [vp, vp, vp]
    L.gnssb200_gpssdr_acquire.argtypes = [vp, vp, C.c_int, C.c_double, vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, vp]
    L.gnssb200_gpssdr_acquire_medium.argtypes = [vp, vp, vp, C.c_int, C.c_double, vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, vp]
    L.correlator_init.argtypes = [C.c_double]
    L.Sim_GP2021_int.argtypes = [vp, C.c_long]
    if hasattr(L, "gnssb200_acq_search"):
        L.gnssb200_acq_num_bins.argtypes = [P(abi.AcqCfg)]
        L.gnssb200_acq_samples_needed.argtypes = [P(abi.AcqCfg)]
        L.gnssb200_acq_samples_needed.restype = i64
        L.gnssb200_acq_search.argtypes = [vp, P(abi.AcqCfg), vp, C.c_int, i64, vp, vp]
        L.gnssb200_acq_finalize.argtypes = [P(abi.AcqCfg), vp, vp]
        L.gnssb200_acq_pcps_host.argtypes = [vp, P(abi.AcqCfg), vp, C.c_int, i64, vp, vp]
    if hasattr(L, "gnssb200_acq_search_batch"):
        L.gnssb200_acq_search_batch.argtypes = [vp, P(abi.AcqCfg), vp, C.c_size_t, C.c_int, C.c_int, i64, vp, vp]
        L.gnssb200_rx_acq_allocate.argtypes = [P(abi.Rx), P(abi.Cfg), P(abi.AcqCfg), vp, vp]
    if hasattr(L, "gnssb200_softtrack_batch"):
        L.gnssb200_softtrack_batch.argtypes = [vp, P(abi.SoftTrackCfg), vp, C.c_size_t, C.c_int, C.c_int, i64, vp, vp, C.c_int,
                                               vp, vp, vp]
        L.gnssb200_set_softtrack_width.argtypes = [vp, C.c_int]
    if hasattr(L, "gnssb200_softtrack_resume"):
        L.gnssb200_softtrack_init.argtypes = [P(abi.SoftTrackCfg), vp, vp, C.c_int, C.c_int, vp]
        L.gnssb200_softtrack_resume.argtypes = [vp, P(abi.SoftTrackCfg), vp, C.c_size_t, C.c_int, C.c_int, i64, i64, i64, vp,
                                                C.c_int, vp, vp]
        L.gnssb200_softtrack_batch_host.argtypes = [vp, P(abi.SoftTrackCfg), vp, C.c_size_t, C.c_int, C.c_int, i64, vp, vp,
                                                    C.c_int, vp, vp, i64]
    _lib = L
    return L


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().gnssb200_last_error_string()
        raise GnssB200Error(f"{what} failed (rc={rc}): {msg.decode() if msg else '?'}")


def default_cfg(**over) -> abi.Cfg:
    L = lib()
    cfg = abi.Cfg()
    L.gnssb200_cfg_default(C.byref(cfg))
    for k, v in over.items():
        setattr(cfg, k, v)
    L.gnssb200_cfg_derive(C.byref(cfg))
    return cfg
