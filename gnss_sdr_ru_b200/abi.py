"""ctypes mirror of include/gnssb200.h (struct layouts must match the header field for field)."""
from __future__ import annotations

import ctypes as C

N_CHANNELS = 12

FMT_INT8_IQ = 0
FMT_PACKED2 = 1
FMT_INT8_I = 2
PRN_GLONASS = 1 << 10  # PRN register value that selects the GLONASS ST code (gnssb200.h)

SYS_GPS = 0
SYS_GLONASS = 1

STATE_NAMES = {0: "off", 1: "acquisition", 2: "confirm", 3: "pull_in", 4: "tracking"}


class Cfg(C.Structure):
    _fields_ = [
        ("samp_rate", C.c_double),
        ("clock_mult", C.c_double),
        ("gps_carrier_if", C.c_double),
        ("gps_code_f", C.c_double),
        ("freq_bin_width", C.c_double),
        ("tic_period", C.c_double),
        ("carrier_nco_bits", C.c_int32),
        ("code_nco_bits", C.c_int32),
        ("acq_thresh", C.c_int32),
        ("interr_int_us", C.c_int32),
        ("Bnp", C.c_int64),
        ("Bnf", C.c_int64),
        ("Bnd", C.c_int64),
        ("pll_integ_ms", C.c_int64),
        ("dll_integ_ms", C.c_int64),
        ("gps_carrier_ref", C.c_int64),
        ("gps_code_ref", C.c_int64),
        ("d_freq", C.c_int64),
        ("tic_ref", C.c_int64),
        ("pll_i1", C.c_int32),
        ("pll_i2", C.c_int32),
        ("pll_i3", C.c_int32),
        ("dll_i1", C.c_int32),
        ("dll_i2", C.c_int32),
        ("pad_", C.c_int32),
        ("glonass_carrier_if", C.c_double),
        ("glonass_code_f", C.c_double),
        ("glonass_carrier_ref", C.c_int64),
        ("glonass_code_ref", C.c_int64),
    ]


class Chan(C.Structure):
    _fields_ = [
        ("state", C.c_int32),
        ("accum", C.c_int16 * 6),
        ("prev_accum", C.c_int16 * 6),
        ("mean_early", C.c_int64),
        ("mean_prompt", C.c_int64),
        ("mean_late", C.c_int64),
        ("cross", C.c_int64),
        ("dot", C.c_int64),
        ("carrError", C.c_int64),
        ("oldCarrError", C.c_int64),
        ("freqError", C.c_int64),
        ("carrNco", C.c_int64),
        ("oldCarrNco", C.c_int64),
        ("carrFreq", C.c_int64),
        ("carrFreqBasis", C.c_int64),
        ("codeError", C.c_int64),
        ("oldCodeError", C.c_int64),
        ("codeFreq", C.c_int64),
        ("codeFreqBasis", C.c_int64),
        ("codeNco", C.c_int64),
        ("oldCodeNco", C.c_int64),
        ("ch_time", C.c_int64),
        ("n_freq", C.c_int32),
        ("i_confirm", C.c_int32),
        ("n_thresh", C.c_int32),
        ("codes", C.c_int32),
        ("del_freq", C.c_int32),
        ("CN0", C.c_int32),
        ("carrier_freq", C.c_int64),
        ("carrier_cold_corr", C.c_int64),
        ("sign_pos", C.c_int32),
        ("prev_sign_pos", C.c_int32),
        ("sign_count", C.c_int32),
        ("ms_count", C.c_int32),
        ("ms_set", C.c_int32),
        ("ms_sign", C.c_uint64),
        ("bit", C.c_int32),
        ("search_max_PRN_delay", C.c_int32),
        ("search_max_f", C.c_int32),
        ("system", C.c_int32),
    ]


class Corr(C.Structure):
    _fields_ = [
        ("carrier_phase", C.c_uint32),
        ("carrier_cycle", C.c_uint32),
        ("code_phase", C.c_uint32),
        ("half_chip", C.c_uint32),
        ("acc", C.c_int32 * 6),
        ("ms_counter", C.c_int32),
        ("bit_counter", C.c_int32),
    ]


class Rx(C.Structure):
    _fields_ = [
        ("reg_read", C.c_int32 * 256),
        ("reg_write", C.c_int32 * 256),
        ("corr", Corr * N_CHANNELS),
        ("chan", Chan * N_CHANNELS),
        ("tic", C.c_int64),
        ("blocks_done", C.c_int64),
        ("halted", C.c_int32),
        ("pad_", C.c_int32),
    ]


class Dump(C.Structure):
    _fields_ = [
        ("block", C.c_int32),
        ("ch", C.c_int16),
        ("state", C.c_int16),
        ("acc", C.c_int32 * 6),
        ("carrier_incr", C.c_uint32),
        ("code_incr", C.c_uint32),
        ("n_freq", C.c_int16),
        ("codes", C.c_int16),
        ("slew", C.c_int32),
    ]


class SynthSat(C.Structure):
    _fields_ = [
        ("system", C.c_int32),
        ("prn", C.c_int32),
        ("cn0_dbhz", C.c_double),
        ("samp_rate", C.c_double),
        ("carrier_hz", C.c_double),
        ("code_hz", C.c_double),
        ("code_phase_chips", C.c_double),
        ("carrier_phase_cycles", C.c_double),
        ("data_seed", C.c_int32),
        ("pad_", C.c_int32),
        ("data_rate_hz", C.c_double),
        ("data_bits", C.c_void_p),
        ("n_data_bits", C.c_int64),
    ]


class AcqCfg(C.Structure):
    _fields_ = [
        ("system", C.c_int32),
        ("samp_freq", C.c_double),
        ("IF", C.c_double),
        ("IF_step", C.c_double),
        ("code_freq", C.c_double),
        ("code_length", C.c_int32),
        ("search_band_khz", C.c_double),
        ("coh_ms", C.c_int32),
        ("n_noncoh", C.c_int32),
        ("threshold", C.c_double),
        ("n_sv", C.c_int32),
        ("sv", C.c_int32 * 64),
        ("part_index", C.c_int32),
        ("part_count", C.c_int32),
    ]


class AcqRow(C.Structure):
    _fields_ = [
        ("peak", C.c_float),
        ("code_phase", C.c_int32),
        ("second", C.c_float),
        ("block", C.c_int32),
    ]


class AcqResult(C.Structure):
    _fields_ = [
        ("carrFreq", C.c_double),
        ("codePhase", C.c_int32),
        ("sv", C.c_int32),
        ("peakMetric", C.c_double),
        ("bin", C.c_int32),
        ("codePhaseRaw", C.c_int32),
        ("peak", C.c_float),
        ("second", C.c_float),
    ]


class SoftTrackCfg(C.Structure):
    _fields_ = [
        ("system", C.c_int32),
        ("code_length", C.c_int32),
        ("samp_freq", C.c_double),
        ("IF", C.c_double),
        ("IF_step", C.c_double),
        ("glonass_zero_channel", C.c_double),
        ("code_freq", C.c_double),
        ("dll_damping_ratio", C.c_double),
        ("dll_noise_bandwidth", C.c_double),
        ("dll_correlator_spacing", C.c_double),
        ("pll_noise_bandwidth", C.c_double),
        ("fll_noise_bandwidth", C.c_double),
        ("skip_samples", C.c_int64),
        ("ms_to_process", C.c_int32),
        ("pad_", C.c_int32),
    ]


class SoftTrackChan(C.Structure):
    _fields_ = [("sv", C.c_int32), ("code_phase", C.c_int32), ("acquired_freq", C.c_double)]


class SoftTrackState(C.Structure):
    """gnssb200_softtrack_state: one float-tracking channel between two code periods."""
    _fields_ = [("codeFreq", C.c_double), ("remCodePhase", C.c_double), ("carrFreq", C.c_double), ("remCarrPhase", C.c_double),
                ("oldCodeNco", C.c_double), ("oldCodeError", C.c_double), ("oldCarrNco", C.c_double), ("oldCarrError", C.c_double),
                ("I1", C.c_double), ("Q1", C.c_double), ("carrFreqBasis", C.c_double), ("pos", C.c_int64), ("sv", C.c_int32),
                ("record", C.c_int32), ("ms_done", C.c_int32), ("status", C.c_int32)]


# gnssb200_softtrack_state.status
SOFTTRACK_RUNNING, SOFTTRACK_RECORD_END, SOFTTRACK_MS_DONE = 0, 1, 2
SOFTTRACK_BEHIND, SOFTTRACK_BAD_RECORD, SOFTTRACK_BAD_SV = -1, -2, -3


class IngestStat(C.Structure):
    _fields_ = [("bytes_loaded", C.c_int64), ("bytes_output", C.c_int64), ("bytes_in_buffer", C.c_int64), ("ring_bytes", C.c_int64),
                ("blocks_done", C.c_int64), ("finished", C.c_int32), ("overflow", C.c_int32)]


class SerialCell(C.Structure):
    _fields_ = [("prn", C.c_int16), ("n_freq", C.c_int16), ("codes", C.c_int32), ("ip", C.c_int32), ("qp", C.c_int32), ("rss", C.c_int32)]


SERIAL_CELL_DTYPE = [("prn", "<i2"), ("n_freq", "<i2"), ("codes", "<i4"), ("ip", "<i4"), ("qp", "<i4"), ("rss", "<i4")]


class GpsSdrResult(C.Structure):
    _fields_ = [("sv", C.c_int32), ("type", C.c_int32), ("code_phase", C.c_int32), ("doppler", C.c_int32), ("magnitude", C.c_uint32),
                ("success", C.c_int32)]


SOFTTRACK_FIELDS = ("I_E", "I_P", "I_L", "Q_E", "Q_P", "Q_L", "carrFreq", "codeFreq", "dllDiscr", "dllDiscrFilt",
                    "pllDiscr", "pllDiscrFilt", "absoluteSample")

assert C.sizeof(Dump) == 48
DUMP_DTYPE = [
    ("block", "<i4"),
    ("ch", "<i2"),
    ("state", "<i2"),
    ("acc", "<i4", (6,)),
    ("carrier_incr", "<u4"),
    ("code_incr", "<u4"),
    ("n_freq", "<i2"),
    ("codes", "<i2"),
    ("slew", "<i4"),
]
ACQ_ROW_DTYPE = [("peak", "<f4"), ("code_phase", "<i4"), ("second", "<f4"), ("block", "<i4")]
