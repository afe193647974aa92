/*
 * gnssb200.h -- C ABI of libgnssb200.so, the B200 (sm_100a) GNSS baseband engine.
 *
 * Plain C: pointers, sizes and fixed-width structs only.  Two layers:
 *
 *  (1) DROP-IN layer: the exact symbols the reference C receiver binds for its correlator
 *      (OSG = trunk/GNSS_SOFTWARE_RECEIVERS/POSTPROCESSING_RECEIVERS/osgnss_next_step/src):
 *        OSG/correlator/correlator.h:4   int REG_read[256], REG_write[256];
 *        OSG/correlator/correlator.h:8   void correlator_init(double tic_period);
 *        OSG/correlator/correlator.h:9   void Sim_GP2021_int(char *IF, long nsamp);
 *      A host program written against correlator.h links against libgnssb200.so instead of
 *      correlator.c and runs unchanged (INTEGRATION.md shows the link line).
 *
 *  (2) BATCHED layer (gnssb200_*): many independent IF streams x 12 channels, closed loop
 *      (correlator + the integer channel logic of OSG/isr/osgpsisr.c) resident on the GPU, and the
 *      FFT parallel-code-phase acquisition modelled on SCI/{GPS,GLONASS}/L1/acquisition.sci.
 *
 * No CPU fallback exists: every entry point fails (non-zero return, gnssb200_last_error()) when no
 * CUDA device is usable; the two void drop-in functions print to stderr and abort().
 */
#ifndef GNSSB200_H_
#define GNSSB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GNSSB200_N_CHANNELS 12 /* OSG/include/globals.h:7 */

/* ---------------------------------------------------------------------------------------------
 * (1) drop-in layer
 * ------------------------------------------------------------------------------------------- */
extern int REG_read[256], REG_write[256]; /* replaces OSG/correlator/correlator.h:4 (library owns them) */

/* replaces OSG/correlator/correlator.c:107-132.  Also writes the host program's globals
 * Carrier_DCO_Delta, Code_DCO_Delta, gps_code_ref, gps_carrier_ref, glonass_code_ref,
 * glonass_carrier_ref, d_freq (OSG/include/globals.h:38-49) when the host defines them (weak refs),
 * reading freq_bin_width (globals.h:54) the same way. */
void correlator_init(double tic_period);

/* replaces OSG/correlator/correlator.c:148-316.  IF: host buffer of 2*nsamp int8 (I,Q interleaved),
 * or nsamp int8 when the host global use_iq_processing (globals.h:56) is 0.  Synchronous: REG_read /
 * REG_write are up to date on return; IF may be overwritten afterwards. */
void Sim_GP2021_int(char *IF, long nsamp);

/* 0 = ok; otherwise the cudaError_t (or a negative library code) of the most recent failure. */
int gnssb200_last_error(void);
const char *gnssb200_last_error_string(void);

/* ---------------------------------------------------------------------------------------------
 * (2) batched layer -- tracking
 * ------------------------------------------------------------------------------------------- */

/* Receiver constants.  Mirrors the tunable globals of OSG/include/globals.h:7-63 plus the values
 * correlator_init / init_tracking_loops_parameter derive from them. */
typedef struct gnssb200_cfg {
  double samp_rate;        /* SAMP_RATE 16e6                      globals.h:12 */
  double clock_mult;       /* SYSTEM_CLOCK_MULTIPLIER 5           globals.h:13 */
  double gps_carrier_if;   /* GPS_CARRIER_IF 2.42e6               globals.h:16 */
  double gps_code_f;       /* GPS_CODE_F 1023000                  globals.h:17 */
  double freq_bin_width;   /* 1000 Hz                             globals.h:54 */
  double tic_period;       /* value passed to correlator_init (the stock main passes int 0) */
  int32_t carrier_nco_bits;/* CARRIER_NCO_DIGIT_CAPACITY 30       globals.h:20 */
  int32_t code_nco_bits;   /* CODE_NCO_DIGIT_CAPACITY 29          globals.h:21 */
  int32_t acq_thresh;      /* 1800                                globals.h:36 */
  int32_t interr_int_us;   /* 512                                 globals.h:51 */
  int64_t Bnp, Bnf, Bnd;   /* 25, 1400, 2                         globals.h:59-61 */
  int64_t pll_integ_ms, dll_integ_ms; /* 1, 1                     globals.h:62-63 */
  /* derived (filled by gnssb200_cfg_derive; same arithmetic as the reference) */
  int64_t gps_carrier_ref, gps_code_ref, d_freq;   /* correlator.c:114-121 */
  int64_t tic_ref;                                 /* correlator.c:124 */
  int32_t pll_i1, pll_i2, pll_i3, dll_i1, dll_i2;  /* osgpsisr.c:252-342 */
  int32_t pad_;
  /* GLONASS channels of the integer correlator (see GNSSB200_PRN_GLONASS below) */
  double glonass_carrier_if; /* GLONASS_CARRIER_IF 0.0e6            globals.h:19 */
  double glonass_code_f;     /* GLONASS_CODE_F 511000               globals.h:20 */
  int64_t glonass_carrier_ref, glonass_code_ref; /* derived, correlator.c:116-118 */
} gnssb200_cfg;

/* GLONASS in the integer correlator.  The C reference carries only the hooks (glonass_code_ref /
 * glonass_carrier_ref, correlator.c:116-118; chan[].system "for future use", structs.h:88; "1021 for GLONASS",
 * osgnss_next_step.c:54); the behaviour is the one of the correlator the C code emulates, NAM/rtl/code_gen.v:
 * writing bit 10 of the PRN register selects the 511-chip ST code (g3 register, :121-139) and a code period of
 * 1022 half chips (:236-272) -- the firmware's `outpw(PRN_KEY, 1<<10)`.  Here: a channel whose PRN register holds
 * GNSSB200_PRN_GLONASS correlates against the ST-code row of the E/P/L table (built like the C/A rows,
 * correlator.c:84-89, with 1022 for 2046; entries past the row are 0) and dumps every 1022 + slew half chips;
 * a channel with chan.system = 1 takes glonass_code_ref / glonass_carrier_ref where the channel logic of
 * osgpsisr.c uses the GPS ones, its frequency-channel offset k*562.5 kHz goes into carrier_cold_corr. */
#define GNSSB200_PRN_GLONASS (1 << 10)

void gnssb200_cfg_default(gnssb200_cfg *cfg); /* reference defaults (globals.h) */
void gnssb200_cfg_derive(gnssb200_cfg *cfg);  /* correlator_init + init_tracking_loops_parameter */

/* Per-channel host-side logic state: the fields of struct tracking_channel
 * (OSG/include/structs.h:86-128) that the acquisition/confirm/pull-in/track state machine uses.
 * C 'long' is int64 here (the oracle is the LP64 build of the reference, SURVEY.md 7.3). */
typedef struct gnssb200_chan {
  int32_t state;            /* tracking_enum: 0 off 1 acq 2 confirm 3 pull-in 4 tracking */
  int16_t accum[6];         /* i_prompt q_prompt i_late q_late i_early q_early (structs.h:54-61) */
  int16_t prev_accum[6];
  int64_t mean_early, mean_prompt, mean_late; /* accum_mean */
  int64_t cross, dot;
  int64_t carrError, oldCarrError, freqError;
  int64_t carrNco, oldCarrNco, carrFreq, carrFreqBasis;
  int64_t codeError, oldCodeError, codeFreq, codeFreqBasis, codeNco, oldCodeNco;
  int64_t ch_time;
  int32_t n_freq, i_confirm, n_thresh, codes, del_freq;
  int32_t CN0;
  int64_t carrier_freq, carrier_cold_corr;
  int32_t sign_pos, prev_sign_pos, sign_count;
  int32_t ms_count, ms_set;
  uint64_t ms_sign;
  int32_t bit;
  int32_t search_max_PRN_delay, search_max_f;
  int32_t system;           /* channel_gnss_system_enum: 0 GPS, 1 GLONASS (structs.h:78-88) */
} gnssb200_chan;

/* Per-channel correlator state: struct gp2021_channel + ms/bit counters
 * (OSG/correlator/correlator.c:33,36-47). */
typedef struct gnssb200_corr {
  uint32_t carrier_phase, carrier_cycle, code_phase;
  uint32_t half_chip;       /* uint16_t in the reference */
  int32_t acc[6];           /* order of REG_read offsets: IL QL IP QP IE QE (correlator.c:15-20) */
  int32_t ms_counter, bit_counter;
} gnssb200_corr;

/* Everything one receiver (one IF stream) owns. */
typedef struct gnssb200_rx {
  int32_t reg_read[256];
  int32_t reg_write[256];
  gnssb200_corr corr[GNSSB200_N_CHANNELS];
  gnssb200_chan chan[GNSSB200_N_CHANNELS];
  int64_t tic;              /* correlator.c:30 (tic_ref lives in cfg) */
  int64_t blocks_done;      /* number of Sim_GP2021_int-equivalent blocks processed so far */
  int32_t halted;           /* 1 once a dumping channel was found in CHANNEL_OFF (osgpsisr.c:383-386: exit(0)) */
  int32_t pad_;
} gnssb200_rx;

/* One record per correlator dump (one per channel per code period). */
typedef struct gnssb200_dump {
  int32_t block;            /* index of the block (Sim_GP2021_int call) in which the dump fell */
  int16_t ch;
  int16_t state;            /* chan.state AFTER gpsisr handled this dump */
  int32_t acc[6];           /* IL QL IP QP IE QE, full int32 as stored in REG_read */
  uint32_t carrier_incr;    /* (REG_write[+3]<<16)+REG_write[+4] after gpsisr */
  uint32_t code_incr;       /* (REG_write[+5]<<16)+REG_write[+6] after gpsisr */
  int16_t n_freq;
  int16_t codes;
  int32_t slew;             /* REG_write[ch*8+0x84] after gpsisr */
} gnssb200_dump;            /* 48 bytes */

/* Host helpers that mirror the reference's register accessors on a gnssb200_rx
 * (OSG/gp2021/gp2021.c:74-130): same masking to 16 bits, same <<(32-N) * 5 scaling. */
void gnssb200_rx_init(gnssb200_rx *rx, const gnssb200_cfg *cfg); /* zero + correlator_init state */
void gnssb200_rx_cold_allocate(gnssb200_rx *rx, const gnssb200_cfg *cfg,
                               const int32_t prn[GNSSB200_N_CHANNELS]); /* osgnss_next_step.c:41-84 */
void gnssb200_ch_cntl(gnssb200_rx *rx, int ch, int data);
void gnssb200_ch_carrier(gnssb200_rx *rx, const gnssb200_cfg *cfg, int ch, int64_t freq);
void gnssb200_ch_code(gnssb200_rx *rx, const gnssb200_cfg *cfg, int ch, int64_t freq);
void gnssb200_ch_code_slew(gnssb200_rx *rx, int ch, int data);
void gnssb200_ch_epoch_load(gnssb200_rx *rx, int ch, unsigned data);

typedef struct gnssb200_handle gnssb200_handle;

#define GNSSB200_FMT_INT8_IQ   0 /* int8 I,Q interleaved: 2 bytes / complex sample */
#define GNSSB200_FMT_PACKED2   1 /* 2+2 bit: I0 Q0 I1 Q1 in one byte, LSB first, code {0:+1,1:-1,2:+3,3:-3} */
#define GNSSB200_FMT_INT8_I    2 /* int8 real samples (use_iq_processing = 0 path, correlator.c:217-224) */

/* device: CUDA device ordinal.  Returns NULL on failure (see gnssb200_last_error). */
gnssb200_handle *gnssb200_open(int device, const gnssb200_cfg *cfg);
void gnssb200_close(gnssb200_handle *h);

/* Number of receivers (streams) resident on the device; (re)allocates device state. */
int gnssb200_set_streams(gnssb200_handle *h, int n_streams);
int gnssb200_upload_rx(gnssb200_handle *h, int first, int count, const gnssb200_rx *rx);
int gnssb200_download_rx(gnssb200_handle *h, int first, int count, gnssb200_rx *rx);

/* Closed-loop tracking / serial search on device memory.
 *   d_if          device pointer; stream s starts at d_if + s*stream_stride_bytes
 *   fmt           GNSSB200_FMT_*
 *   nsamp         complex samples per block (the reference uses 8192 = 512 us, osgnss_next_step.c:150)
 *   nblocks       blocks to process per stream (each = one Sim_GP2021_int + gpsisr of the reference)
 *   d_dumps       device buffer of n_streams*12*dump_cap records, or NULL; channel (s,ch) writes at
 *                 [(s*12+ch)*dump_cap + k]
 *   d_dump_count  device int32[n_streams*12], number of records written per channel (may be NULL)
 *   cuda_stream   a cudaStream_t passed as void* (NULL = default stream).  Asynchronous.
 * Blocks continue from the state left by the previous call (rx.blocks_done advances).  Calls on one handle must
 * be ordered (same CUDA stream, or synchronised by the caller); only runs on disjoint receivers issued through
 * gnssb200_ingest_* may overlap. */
int gnssb200_track_run(gnssb200_handle *h, const void *d_if, size_t stream_stride_bytes, int fmt,
                       int nsamp, int64_t nblocks, gnssb200_dump *d_dumps, int dump_cap,
                       int32_t *d_dump_count, void *cuda_stream);

/* The same from host memory (copies in, runs, copies records out, synchronises): the record is staged through two
 * device buffers chunk by chunk, the copy of chunk c+1 under the kernels of chunk c; h_dumps / h_dump_count
 * (in: counts to continue from, may be NULL = 0; out: counts after the run) are host arrays laid out like their
 * device counterparts above.  Pinned (cudaHostAlloc / cudaHostRegister) buffers give full PCIe speed and let the dump
 * records travel back while later chunks still run; pageable buffers give the same results without the overlap. */
int gnssb200_track_run_host(gnssb200_handle *h, const void *h_if, size_t stream_stride_bytes, int fmt,
                            int nsamp, int64_t nblocks, gnssb200_dump *h_dumps, int dump_cap,
                            int32_t *h_dump_count);

/* GP2021-semantics serial search as an exhaustive cell map (SURVEY.md 8b): every PRN of prn_list gets a channel that
 * searches like ch_acq (OSG/isr/osgpsisr.c:424-459) with the detection threshold out of reach -- 2045 (or
 * max_prn_delay) half-chip code delays per Doppler bin, bins 0,+1,-1,+2,... up to +-search_max_f of width
 * cfg.freq_bin_width -- over the whole device-resident record (fmt INT8_IQ or PACKED2, n_samples complex samples, 8192
 * per block).  One dump = one cell: cells[p*cells_cap + k] describes the k-th cell of prn_list[p]
 * (the bin / delay the channel was in, the prompt sums of that dump and rss(IP,QP), osgpsisr.c:77-91);
 * n_cells[p] = cells completed (at most cells_cap are stored).  The handle's own receivers are not touched. */
typedef struct gnssb200_serial_cell {
  int16_t prn, n_freq;      /* PRN, Doppler bin index (carrier = gps_carrier_ref + n_freq * d_freq) */
  int32_t codes;            /* code delay in half chips */
  int32_t ip, qp, rss;
} gnssb200_serial_cell;
int gnssb200_acq_serial(gnssb200_handle *h, const void *d_if, int fmt, int64_t n_samples, const int32_t *prn_list, int n_prn,
                        int search_max_f, int max_prn_delay, gnssb200_serial_cell *cells, int cells_cap, int32_t *n_cells);

/* Scheduling knob of the tracking kernel: the blocks of every channel are cut into slices of `blocks`
 * blocks that are handed to CTAs through a work queue (keeps all SMs busy whatever the channel count).
 * 0 = automatic (slices of 512 KB of samples per stream -- 128 blocks of packed, 32 of int8 input -- so the slices in
 * flight stay L2 resident, from four channels per SM on; one slice per channel below).  Results do not depend on it. */
int gnssb200_set_track_slice(gnssb200_handle *h, int64_t blocks);

/* Which form of the tracking kernel runs (results do not depend on it; tests and A/B measurements use it).
 * form: 0 automatic; 1 the barrier-synchronised kernel; 2 warp-specialised, fixed runs of 32 / 64 samples per
 * thread; 3 / 4 / 5 warp-specialised, half-chip segments with 96 / 192 / 384 correlator threads (packed input).
 * occ: 0 automatic, else the resident-CTAs-per-SM variant (2..6) that would be chosen for that many channels per SM. */
int gnssb200_set_track_variant(gnssb200_handle *h, int form, int occ);

/* Libraries built with -DTRACK_CHECK verify on the device every shared-memory address the correlator warps form and the
 * work-queue / ring hand-over invariants; this returns the number of violations since the last call (and the count per
 * check in out[8] when it is not NULL), -1 when the library was built without the checks. */
int gnssb200_track_check_failures(unsigned out[8]);

/* Host-buffer pipeline of gnssb200_track_run_host: blocks per stream and staging chunk (0 = automatic, about 384
 * blocks, at least 32 MiB per chunk); results do not depend on it.  The dump records of a multi-chunk run are read
 * back window by window while later chunks are still running when h_dumps is pinned (or registered) host memory;
 * gnssb200_readback_fallbacks counts the runs whose records did not stay inside the predicted windows and were
 * read back again in one piece (correct either way, see csrc/api.cu). */
int gnssb200_set_stage_blocks(gnssb200_handle *h, int64_t blocks);
int64_t gnssb200_readback_fallbacks(const gnssb200_handle *h);

/* Number of kernels this library has launched since open (bench.py reports it as gpu_launches). */
int64_t gnssb200_launch_count(const gnssb200_handle *h);
/* Device time (ms, CUDA events on the launching stream) of the most recent track/acq kernel
 * sequence; valid after the stream was synchronised. */
float gnssb200_last_kernel_ms(gnssb200_handle *h);

/* Diagnostics: evaluates the device ISR's integer helpers element-wise on host arrays of length n:
 *   atan_out[i] = fix_atan2(y[i], x[i])            OSG/isr/osgpsisr.c:199-231 (int32 operands)
 *   sqrt_out[i] = sqrt_newton(L[i])                 osgpsisr.c:148-178
 *   div_out[i]  = num[i] / den[i] (C truncation)    the DLL discriminator division, osgpsisr.c:586,743
 *                 for abs(num) < 2^30, 0 < den < 2^20
 * so tests can compare them with the reference's own helpers on arbitrary arguments. */
int gnssb200_isr_math_eval(gnssb200_handle *h, int n, const int32_t *y, const int32_t *x, int32_t *atan_out,
                           const int64_t *L, uint32_t *sqrt_out, const int32_t *num, const int32_t *den,
                           int32_t *div_out);

/* ---------------------------------------------------------------------------------------------
 * synthetic IF records generated on the device (bench / test input, not part of the hot path).
 * Signal model of SIM/glonass_l3_generator.sce:60-186 + AWGN: per emitter
 * A*code(t)*data(t)*exp(-i(2*pi*f*t+phi0)), A = sqrt(10^(CN0/10)/fs), unit-power complex noise,
 * 2-bit quantiser -> {-3,-1,+1,+3}.
 * ------------------------------------------------------------------------------------------- */
typedef struct gnssb200_synth_sat {
  int32_t system;           /* GNSSB200_SYS_GPS (0) / GNSSB200_SYS_GLONASS (1) */
  int32_t prn;              /* GPS PRN 1..32 (ignored for GLONASS: one ST code) */
  double cn0_dbhz;          /* <= 0: emitter absent */
  double samp_rate;
  double carrier_hz;        /* IF + Doppler */
  double code_hz;           /* chipping rate including code Doppler */
  double code_phase_chips;  /* code phase of sample 0 */
  double carrier_phase_cycles;
  int32_t data_seed;        /* 0: no data modulation (unless data_bits is given) */
  int32_t pad_;
  double data_rate_hz;      /* 50 (GPS) / 100 (GLONASS meander) */
  const uint8_t *data_bits; /* optional HOST array of explicit data bits (0/1), repeated cyclically; NULL: pseudo-random bits from data_seed */
  int64_t n_data_bits;
} gnssb200_synth_sat;

/* sats: [n_streams * n_sats].  fmt INT8_IQ or PACKED2; n_samples multiple of 4.  Synchronous. */
int gnssb200_synth(gnssb200_handle *h, void *d_out, size_t stream_stride_bytes, int fmt, int n_streams,
                   int64_t n_samples, const gnssb200_synth_sat *sats, int n_sats, uint64_t seed,
                   void *cuda_stream);

/* ---------------------------------------------------------------------------------------------
 * (2) batched layer -- FFT parallel-code-phase acquisition
 *     modelled on acqResults = acquisition(longSignal, settings)
 *     SCI/GLONASS/L1/acquisition.sci:1-198, SCI/GPS/L1/acquisition.sci
 * ------------------------------------------------------------------------------------------- */
#define GNSSB200_SYS_GPS     0
#define GNSSB200_SYS_GLONASS 1

typedef struct gnssb200_acq_cfg {
  int32_t system;           /* GNSSB200_SYS_* : code table and chip length of the second-peak window */
  double samp_freq;         /* settings.samplingFreq   16e6 */
  double IF;                /* settings.IF             GPS 2.42e6 / GLONASS 1e6 */
  double IF_step;           /* settings.L1_IF_step     GLONASS 562500, GPS 0 */
  double code_freq;         /* settings.codeFreqBasis  1.023e6 / 0.511e6 */
  int32_t code_length;      /* settings.codeLength     1023 / 511 */
  double search_band_khz;   /* settings.acqSearchBand */
  int32_t coh_ms;           /* settings.acqCohIntegration */
  int32_t n_noncoh;         /* 0/1: stock "better of two blocks"; K>=2: sum of K consecutive blocks (config 4) */
  double threshold;         /* settings.acqThreshold   3.0 */
  int32_t n_sv;             /* entries in sv[] */
  int32_t sv[64];           /* PRN list (GPS) or frequency-channel list k=-7..6 (GLONASS) */
  /* partition of the (sv, bin) grid for multi-GPU runs: this process handles global rows
   * r with r % part_count == part_index, r = sv_index*n_bins + bin */
  int32_t part_index, part_count;
} gnssb200_acq_cfg;

typedef struct gnssb200_acq_row {   /* one (sv, Doppler bin) row of the search grid */
  float peak;               /* max over code phases of the kept block */
  int32_t code_phase;       /* 0-based first argmax (Scilab's is this + 1) */
  float second;             /* max over the code phases at circular distance >= 1 chip (16 GPS / 31 GLONASS samples)
                             * from this row's own argmax: the window of acquisition.sci:151-168 wherever its index
                             * ranges stay inside 1..N.  At 1-based argmax 17 (GPS), 32 and 15969 (GLONASS) they
                             * do not and Scilab stops; there the same circular rule is an extension of this library */
  int32_t block;            /* which block was kept (0/1); 0 for non-coherent mode */
} gnssb200_acq_row;

typedef struct gnssb200_acq_result { /* one per sv, layout of acqResults */
  double carrFreq;          /* 0 when below threshold */
  int32_t codePhase;        /* 1-based, 0 when below threshold */
  int32_t sv;               /* PRN / frequency channel (freqChannel); 0 when below threshold */
  double peakMetric;
  int32_t bin;              /* 1-based frequencyBinIndex of the peak (always filled) */
  int32_t codePhaseRaw;     /* 1-based code phase of the peak (always filled) */
  float peak, second;
} gnssb200_acq_result;

/* Number of Doppler bins for a configuration: round(band*2*Tcoh)+1 (acquisition.sci:66-67). */
int gnssb200_acq_num_bins(const gnssb200_acq_cfg *cfg);
/* Samples the record must hold: n_noncoh<=1 -> 2*coh_ms ms, else n_noncoh*coh_ms ms. */
int64_t gnssb200_acq_samples_needed(const gnssb200_acq_cfg *cfg);

/* Grid search on a device-resident int8 I,Q record (fmt INT8_IQ or PACKED2).  An INT8_IQ record must start on an
 * even byte address (its samples are read as 2-byte loads); a PACKED2 record may start anywhere.
 *   d_rows   device buffer [n_sv * n_bins] of rows; only this partition's rows are written
 *            (others keep peak = -1).  Multi-GPU callers all-gather this table (NCCL) and then call
 *            gnssb200_acq_finalize on the merged table.
 * Asynchronous on cuda_stream. */
int gnssb200_acq_search(gnssb200_handle *h, const gnssb200_acq_cfg *cfg, const void *d_iq, int fmt,
                        int64_t n_samples, gnssb200_acq_row *d_rows, void *cuda_stream);

/* The same search over R = n_records records with the same settings in one call (gnssb200_acq_search is the case
 * R = 1).  Record r starts at d_iq + r*record_stride_bytes (0 = every record is the same buffer), e.g. the stream
 * buffer that gnssb200_track_run then consumes; a non-zero stride must cover the bytes n_samples takes in fmt.
 * INT8_IQ: d_iq and the stride must be even (-15 otherwise, as for a short stride).
 *   d_rows   device [R][n_sv][n_bins]: record r's table is laid out exactly like gnssb200_acq_search's, with the same
 *            partition rule (part_index / part_count).
 * The handle's workspace holds the base spectra of all R records: R * n_cls * K * 128 KB, n_cls = the number of
 * distinct Doppler-bin frequencies modulo 1 kHz, K = 2 (stock) or n_noncoh -- 0.5 MB per record for 1 ms / 500 Hz
 * bins, about 51 MB per record for 10 ms x 20 non-coherent / 50 Hz bins.  A failed allocation is returned as an error.
 * Asynchronous on cuda_stream. */
int gnssb200_acq_search_batch(gnssb200_handle *h, const gnssb200_acq_cfg *cfg, const void *d_iq, size_t record_stride_bytes,
                              int n_records, int fmt, int64_t n_samples, gnssb200_acq_row *d_rows, void *cuda_stream);

/* Peak / second-peak / threshold logic of acquisition.sci:145-191 on a complete host row table. */
int gnssb200_acq_finalize(const gnssb200_acq_cfg *cfg, const gnssb200_acq_row *h_rows,
                          gnssb200_acq_result *results /* [n_sv] */);

/* Convenience: host record in, results out (search + finalize, single GPU, synchronises). */
int gnssb200_acq_pcps_host(gnssb200_handle *h, const gnssb200_acq_cfg *cfg, const void *h_iq, int fmt,
                           int64_t n_samples, gnssb200_acq_result *results, gnssb200_acq_row *h_rows_opt);

/* Hand-off of one record's FFT acquisition results to the channels of the integer receiver.  The C reference has no
 * such hand-off (its main starts channels with simple_cold_allocate and a PRN list fixed in advance, then searches
 * serially); this is an extension of this library, defined as follows.
 *
 * rx must be freshly initialised (gnssb200_rx_init) for the record the acquisition ran on, starting at its sample 0.
 * The detected entries (peakMetric > acq->threshold; FCH 0 counts) are ordered by peakMetric, strongest first, ties
 * in list order, and at most 12 are kept -- the order of SCI/x/include/preRun.sci:66-81.  gnssb200_rx_cold_allocate
 * gives entry i channel i (PRN register = the GPS PRN, or GNSSB200_PRN_GLONASS); the other channels stay off.  Then,
 * with res = clock_mult*samp_rate/2^carrier_nco_bits, d = cfg->d_freq and llround() rounding halves away from 0:
 *   carrier   GLONASS: carrier_cold_corr = fch * (int64)(562500/res), as for any GLONASS channel.
 *             carrier_freq = ref + carrier_cold_corr + llround((carrFreq - IF - fch*IF_step) / res), ref the GPS or
 *             GLONASS carrier reference word, written to the carrier NCO.  The channel confirms and pulls in from the
 *             acquired frequency, whatever bin it is in (reference quirk Q2 does not arise).
 *             n_freq = llround((carrier_freq - ref - carrier_cold_corr) / d) clamped to +-search_max_f,
 *             del_freq = -2*n_freq (n_freq > 0) or 1 - 2*n_freq, as when the serial search enters bin n_freq.
 *   code      tau = codePhase - 1 is the sample at which chip 0 starts.  Search cell k = llround(tau*2*code_f/fs) mod P
 *             (P = 2046 half chips for GPS, 1022 for GLONASS; a satellite with code phase theta chips at sample 0 has
 *             k = 2*(code_length - theta)).  The prompt replica runs one half chip ahead of early, so it meets chip 0
 *             at code delay a = (k + 1) mod P.  The channel starts the serial search two cells before that:
 *             k0 = a - 2 (0 when a < 2), written as code slew k0 -- the first period lasts P + k0 half chips, dump 1
 *             tests delay k0, dump 2 delay k0 + 1, dump 3 delay a -- with codes = 0, so a whole sweep of the bin at
 *             the acquired frequency follows if the satellite is missed.  Dump 0 always tests delay 0; a satellite
 *             within a cell of it may be confirmed there first, fail the confirmation at delay k0 and be found
 *             again a few dumps later.
 * Returns the number of channels allocated (0..12), or < 0 -- rx untouched -- when acq and cfg disagree (sampling
 * rate, IF, code rate, GLONASS IF step of 562.5 kHz) or an argument is invalid.  Channels 0..n-1 are allocated, the
 * others stay off; ch_sv_out[12] (may be NULL) receives the PRN / FCH of each channel (0 for channels left off). */
int gnssb200_rx_acq_allocate(gnssb200_rx *rx, const gnssb200_cfg *cfg, const gnssb200_acq_cfg *acq,
                             const gnssb200_acq_result *res /* [acq->n_sv] */, int32_t ch_sv_out[GNSSB200_N_CHANNELS]);

/* ---------------------------------------------------------------------------------------------
 * (2) batched layer -- floating-point tracking of the Scilab receivers (SURVEY.md 8f, rank 1)
 *     [trackResults, channel] = tracking(fid, channel, settings)
 *     SCI/GLONASS/L1/tracking.sci:226-400, SCI/GPS/L1/tracking.sci; channel list as built by
 *     SCI/x/include/preRun.sci:66-81 from acqResults.
 * ------------------------------------------------------------------------------------------- */
typedef struct gnssb200_softtrack_cfg {
  int32_t system;                 /* GNSSB200_SYS_* */
  int32_t code_length;            /* settings.codeLength */
  double samp_freq;               /* settings.samplingFreq */
  double IF;                      /* settings.IF */
  double IF_step;                 /* settings.L1_IF_step (GLONASS) */
  double glonass_zero_channel;    /* settings.GLONASS_zero_channel 1602e6 */
  double code_freq;               /* settings.codeFreqBasis */
  double dll_damping_ratio, dll_noise_bandwidth;
  double dll_correlator_spacing;  /* settings.dllCorrelatorSpacing, chips: 0 <= spacing <= 0.5 (NaN is invalid), so
                                   * the early and late chips stay inside the period padded by one chip each side */
  double pll_noise_bandwidth, fll_noise_bandwidth;
  int64_t skip_samples;           /* settings.skipNumberOfBytes in complex samples */
  int32_t ms_to_process;          /* settings.msToProcess */
  int32_t pad_;
} gnssb200_softtrack_cfg;

typedef struct gnssb200_softtrack_chan {   /* one entry of the `channel` struct array */
  int32_t sv;                     /* PRN (GPS) / FCH (GLONASS) */
  int32_t code_phase;             /* channel.codePhase, 1-based sample */
  double acquired_freq;           /* channel.acquiredFreq */
} gnssb200_softtrack_chan;

#define GNSSB200_SOFTTRACK_FIELDS 13 /* I_E I_P I_L Q_E Q_P Q_L carrFreq codeFreq dllDiscr dllDiscrFilt pllDiscr pllDiscrFilt absoluteSample */

/* d_iq: device int8 I,Q record (the whole file) at an even byte address; d_out: device double
 * [n_ch][ms_to_process][13]; d_ms_done: device int32 [n_ch] = code periods actually processed (fewer if the record
 * ends).  Returns < 0 and writes nothing for -20 (NULL pointer, n_ch <= 0, ms_to_process <= 0, code length other than
 * 511 / 1023, dll_correlator_spacing outside 0..0.5 or NaN), -21 (GPS PRN outside 1..32), -23 (odd d_iq).
 * Synchronous on cuda_stream. */
int gnssb200_softtrack(gnssb200_handle *h, const gnssb200_softtrack_cfg *cfg, const void *d_iq, int64_t n_samples,
                       const gnssb200_softtrack_chan *chans, int n_ch, double *d_out, int32_t *d_ms_done,
                       void *cuda_stream);

/* The float tracking of gnssb200_softtrack for channels spread over R = n_records records with the same settings.
 * Record r starts at d_iq + r*record_stride_bytes (0: every record is the same buffer) and holds n_samples complex
 * samples in fmt (INT8_IQ or PACKED2); a non-zero stride must cover them.  Channel i reads record chan_record[i]:
 * it starts at cfg->skip_samples + chans[i].code_phase - 1 of that record and stops at that record's end.
 * d_out [n_ch][ms_to_process][13] and d_ms_done [n_ch] are laid out exactly as gnssb200_softtrack's, and each
 * channel's values are bit-identical to gnssb200_softtrack on its record alone (after unpacking, for PACKED2),
 * whatever kernel width runs.  Returns < 0 and writes nothing to d_out / d_ms_done when an argument is invalid:
 * -20 (NULL pointer, n_ch <= 0, ms_to_process <= 0, a code length other than 511 / 1023, dll_correlator_spacing
 * outside 0..0.5 or NaN), -21 (a GPS PRN outside 1..32), -22 (another fmt), -23 (n_records < 1, a stride that does not
 * cover a record, or for INT8_IQ an odd d_iq or an odd stride), -24 (a chan_record out of range).
 * Synchronous on cuda_stream. */
int gnssb200_softtrack_batch(gnssb200_handle *h, const gnssb200_softtrack_cfg *cfg, const void *d_iq,
                             size_t record_stride_bytes, int n_records, int fmt, int64_t n_samples,
                             const gnssb200_softtrack_chan *chans, const int32_t *chan_record, int n_ch,
                             double *d_out, int32_t *d_ms_done, void *cuda_stream);

/* Threads per channel of gnssb200_softtrack_batch and gnssb200_softtrack_resume: 0 automatic, else 128, 256 or 512.
 * Results do not depend on it.  Automatic: the width whose CTAs finish all channels in the fewest waves, weighted by
 * the measured time of a wave at that width -- 512 while every channel has an SM of its own, narrower beyond that
 * (DESIGN §4.3). */
int gnssb200_set_softtrack_width(gnssb200_handle *h, int threads);

/* Resumable float tracking.  gnssb200_softtrack_state holds one channel between two code periods: everything the
 * tracking loop carries from one period to the next.  The block size is not stored; the kernel recomputes it as
 * (int)ceil((code_length - remCodePhase) / (codeFreq / samp_freq)), the expression of the loop itself, and doubles
 * round-trip exactly through memory.  So a channel tracked window by window (gnssb200_softtrack_resume), or
 * checkpointed to the host and continued on another handle, gives rows and ms_done byte-identical to
 * gnssb200_softtrack_batch on the whole record, at any kernel width. */
#define GNSSB200_SOFTTRACK_RUNNING     0  /* not finished: paused at a window end (or not started yet) */
#define GNSSB200_SOFTTRACK_RECORD_END  1  /* the next block passes the record end (pos + blksize > record_samples) */
#define GNSSB200_SOFTTRACK_MS_DONE     2  /* ms_done reached ms_to_process */
#define GNSSB200_SOFTTRACK_BEHIND     -1  /* pos < win_first: the next block starts before the window; nothing was read */
#define GNSSB200_SOFTTRACK_BAD_RECORD -2  /* record outside 0..n_records-1; nothing was read */
#define GNSSB200_SOFTTRACK_BAD_SV     -3  /* GPS PRN outside 1..32; nothing was read */

typedef struct gnssb200_softtrack_state {
  double codeFreq, remCodePhase;  /* code NCO */
  double carrFreq, remCarrPhase;  /* carrier NCO */
  double oldCodeNco, oldCodeError, oldCarrNco, oldCarrError;  /* loop-filter memory */
  double I1, Q1;                  /* the FLL's previous prompt sums; 0.001 before period 1 */
  double carrFreqBasis;           /* channel.acquiredFreq */
  int64_t pos;                    /* first sample of the next block, in the channel's record */
  int32_t sv;                     /* PRN (GPS) / FCH (GLONASS) */
  int32_t record;                 /* record index */
  int32_t ms_done;                /* rows written so far: the next row is d_out[ch][ms_done] */
  int32_t status;                 /* GNSSB200_SOFTTRACK_* */
} gnssb200_softtrack_state;

/* The state every channel has before its first code period: codeFreq = code_freq, carrFreq = carrFreqBasis =
 * acquired_freq, remainders and loop memory 0, I1 = Q1 = 0.001, pos = skip_samples + code_phase - 1,
 * record = chan_record[i] (NULL: 0), status RUNNING.  Host code, no device.  Validates as gnssb200_softtrack_batch:
 * -20 (NULL pointer, n_ch <= 0, n_records < 1, ms_to_process <= 0, code length other than 511 / 1023,
 * dll_correlator_spacing outside 0..0.5 or NaN), -21 (GPS PRN outside 1..32), -24 (chan_record out of range); states
 * are untouched then. */
int gnssb200_softtrack_init(const gnssb200_softtrack_cfg *cfg, const gnssb200_softtrack_chan *chans,
                            const int32_t *chan_record, int n_records, int n_ch, gnssb200_softtrack_state *states);

/* Track the n_ch channels of d_state [n_ch] (device) through one window of samples: samples
 * [win_first, win_first + win_samples) of every record.  Record r's window starts at d_win + r*win_stride_bytes
 * (0: every record is the same buffer).  INT8_IQ: sample k at byte 2*(k - win_first).  PACKED2: sample k is nibble
 * k & 1 of byte (k >> 1) - (win_first >> 1); win_first must be even.
 * A channel runs code periods while ms_done < ms_to_process, its next block [pos, pos + blksize) lies inside the window
 * and pos + blksize <= record_samples (the reference's end rule).  A block that runs past the window end pauses the
 * channel (status RUNNING, state unchanged), and a later window continues it; consecutive windows must overlap by at
 * least the block length.  record_samples may be any value at or past the window end while the record's true length
 * is not yet known; the end rule applies from the call that passes the true length.  A channel whose pos lies before
 * win_first stops as BEHIND, one with a record index out of range as BAD_RECORD: nothing is read or written for them
 * but the status.  Channels whose status is RECORD_END or MS_DONE are left untouched.  Rows go to
 * d_out [n_ch][ms_to_process][13], row ms_done of the channel, the layout of gnssb200_softtrack_batch.
 * Uses the width of gnssb200_set_softtrack_width (or the automatic width); it may change between windows.
 * Device pointers and scalars only, asynchronous on cuda_stream.  It can be captured in a CUDA graph once the handle
 * holds its chip table, i.e. after any float-tracking call on the handle (gnssb200_softtrack*, or one resume outside
 * the capture); under capture without it the call returns -27.  Returns < 0 and launches
 * nothing for: -22 (fmt other than INT8_IQ / PACKED2, packed input with an odd win_first), -23 (a non-zero stride
 * shorter than the window's bytes; INT8_IQ with an odd d_win or an odd stride), -20 (n_records < 1, n_ch <= 0,
 * win_first < 0, win_samples < 0, ms_to_process <= 0, a NULL pointer, a code length other than 511 / 1023,
 * dll_correlator_spacing outside 0..0.5 or NaN). */
int gnssb200_softtrack_resume(gnssb200_handle *h, const gnssb200_softtrack_cfg *cfg, const void *d_win,
                              size_t win_stride_bytes, int n_records, int fmt, int64_t win_first, int64_t win_samples,
                              int64_t record_samples, gnssb200_softtrack_state *d_state, int n_ch, double *d_out,
                              void *cuda_stream);

/* gnssb200_softtrack_batch on records in host memory: h_iq is a host buffer (record r at h_iq + r*record_stride_bytes,
 * 0: one record), h_out [n_ch][ms_to_process][13] and h_ms_done [n_ch] are host arrays; only rows [0, ms_done) of a
 * channel are written.  The records are staged window by window through two device buffers of one window of all
 * records each (cudaMemcpy2DAsync on a copy stream), the copy of window k+1 under the tracking of window k.
 * Consecutive windows overlap by two nominal code periods, 2*ceil(code_length*samp_freq/code_freq) samples, so a
 * channel paused at a window end finds its next block whole in the next window.  Device memory: the two staging
 * buffers, the rows and the states; the records are never resident whole.  Pinned host memory (cudaHostAlloc /
 * cudaHostRegister) gives the overlap; pageable memory gives the same results without it.
 * window_samples: samples per window, 0 automatic (2^20 samples, fewer if one window of all records would pass 512 MiB; DESIGN §4.3); below four
 * nominal code periods it is invalid; a window longer than the record is cut to the record.  Returns 0, or the number
 * of channels that ended BEHIND at pos >= 0 -- a block longer than the overlap, or a diverged loop whose block size
 * turned non-positive and walked pos back before a later window (the one-shot call would run such a channel on towards
 * sample 0) -- whose rows up to that point are still those of the one-shot call; or < 0 for the invalid arguments of
 * gnssb200_softtrack_batch (h_iq and the stride may be odd: windows are staged into aligned device buffers) and an
 * invalid window_samples (-26), with h_out / h_ms_done untouched.  Synchronous. */
int gnssb200_softtrack_batch_host(gnssb200_handle *h, const gnssb200_softtrack_cfg *cfg, const void *h_iq,
                                  size_t record_stride_bytes, int n_records, int fmt, int64_t n_samples,
                                  const gnssb200_softtrack_chan *chans, const int32_t *chan_record, int n_ch,
                                  double *h_out, int32_t *h_ms_done, int64_t window_samples);

/* ---------------------------------------------------------------------------------------------
 * (2) batched layer -- streaming ingest (SURVEY.md 8f, rank 4): a circular buffer between a sample
 *     producer and the GPU channel loop of ONE stream of the handle, modelled on
 *     FE/PC_SIDE_SOFTWARE/WIN/GPS1A_SAMPLER/src/CircularBuffer.h:9-193 and the collector / writer threads of
 *     win32_sampler.h:232-364 (the writer thread's place is taken by the tracking kernel).
 *     One producer thread may call _write/_finish while one consumer thread calls _pump/_sync/_status.
 * ------------------------------------------------------------------------------------------- */
typedef struct gnssb200_ingest gnssb200_ingest;
typedef struct gnssb200_ingest_stat {
  int64_t bytes_loaded;     /* TotBytesLoaded */
  int64_t bytes_output;     /* TotBytesOutput (handed to the GPU) */
  int64_t bytes_in_buffer;  /* DataLeftInBuffer() */
  int64_t ring_bytes;       /* CircularBufferSize */
  int64_t blocks_done;      /* 512-us blocks tracked so far */
  int32_t finished;         /* FinishedFillingBuffer */
  int32_t overflow;         /* CircularBufferOverFlow */
} gnssb200_ingest_stat;

/* stream: index of the receiver (0 .. n_streams-1) this ingest feeds; ring_blocks: ring capacity in blocks of
 * nsamp samples (the ring is pinned host memory); dump_cap: dump records kept per channel (0: none). */
gnssb200_ingest *gnssb200_ingest_open(gnssb200_handle *h, int stream, int fmt, int nsamp, int64_t ring_blocks, int dump_cap);
void gnssb200_ingest_close(gnssb200_ingest *g);
/* Producer: all-or-nothing copy into the ring.  Returns bytes, or 0 after raising the overflow flag. */
int64_t gnssb200_ingest_write(gnssb200_ingest *g, const void *data, int64_t bytes);
void gnssb200_ingest_finish(gnssb200_ingest *g);
/* Consumer: tracks the whole blocks available in one contiguous run (<= max_blocks if > 0).  Returns the number
 * of blocks launched (0: none available), < 0 on error.  Asynchronous with respect to the kernels. */
int64_t gnssb200_ingest_pump(gnssb200_ingest *g, int64_t max_blocks);
int gnssb200_ingest_status(gnssb200_ingest *g, gnssb200_ingest_stat *out);
/* Waits for the issued kernels; copies records [12][dump_cap] and counts [12] to the host (either may be NULL). */
int gnssb200_ingest_sync(gnssb200_ingest *g, gnssb200_dump *h_dumps, int32_t *h_count);

/* ---------------------------------------------------------------------------------------------
 * (2) batched layer -- start of the navigation message in the tracking output (SURVEY.md 8f, rank 3)
 *     GPS      [firstSubFrame, activeChnList] = findPreambles(trkRslt_status, trkRslt_I_P, n)
 *              SCI/GPS/L1/findPreambles.sci:30-169 with SCI/GPS/L1/include/navPartyChk.sci:57-99
 *     GLONASS  [firstString, activeChnList]   = findTimeMarks(trkRslt_status, trkRslt_I_P, n)
 *              SCI/GLONASS/L1/findTimeMarks.sci:25-66
 * d_ip: DEVICE buffer holding the prompt in-phase value of (channel ch, code period ms) at byte offset
 * ch*ch_stride_bytes + ms*ms_stride_bytes: a double (dtype GNSSB200_NAV_F64, e.g. field I_P of the
 * gnssb200_softtrack output: ch_stride = ms_to_process*13*8, ms_stride = 13*8, base + 8) or an int32
 * (GNSSB200_NAV_I32, e.g. acc[2] of the gnssb200_dump records: ch_stride = dump_cap*48, ms_stride = 48,
 * base + 16).  active_in[ch] != 0 <=> trackResults(ch).status ~= '-' (NULL: all active).
 * Outputs (host): first_*[ch] = the reference's 1-based millisecond index, 0 when nothing valid was found;
 * active_out[ch] = 1 for channels that keep a valid start (may be NULL).  Synchronises cuda_stream.
 * ------------------------------------------------------------------------------------------- */
#define GNSSB200_NAV_F64 0
#define GNSSB200_NAV_I32 1
int gnssb200_find_preambles(gnssb200_handle *h, const void *d_ip, int dtype, int64_t ch_stride_bytes, int64_t ms_stride_bytes,
                            int n_ch, int n_ms, const int32_t *active_in, int32_t *first_subframe, int32_t *active_out,
                            void *cuda_stream);
int gnssb200_find_time_marks(gnssb200_handle *h, const void *d_ip, int dtype, int64_t ch_stride_bytes, int64_t ms_stride_bytes,
                             int n_ch, int n_ms, const int32_t *active_in, int32_t *first_string, int32_t *active_out,
                             void *cuda_stream);

/* ---------------------------------------------------------------------------------------------
 * (2) batched layer -- GPS-SDR fixed-point FFT acquisition (SURVEY.md 8f, rank 2), bit exact with the
 *     reference's portable arithmetic (RT = trunk/GNSS_SOFTWARE_RECEIVERS/REALTIME_RECEIVERS/GPS/
 *     GPS_SDR_REAL_TIME_GPS_RECEIVER):
 *       Acq_Command_S Acquisition::doAcqStrong(int32 sv, int32 doppmin, int32 doppmax)  RT/objects/acquisition.cpp:244
 *       Acq_Command_S Acquisition::doAcqWeak  (int32 sv, int32 doppmin, int32 doppmax)  RT/objects/acquisition.cpp:433
 *     each preceded by Acquisition::doPrepIF(type, buff) (:182), for a list of satellites in one call.
 * iq         host buffer of complex int16 (i, q) at 2.048 Msps as doPrepIF receives it: 1 ms (type 0, strong)
 *            or 310 ms (type 2, weak)
 * fif        intermediate frequency the wipe-off tables are built for (IF_FREQUENCY 38400, signaldef.h:34)
 * prn_codes  the pre-FFT'd code table PRN_Codes (RT/accessories/prn_codes.h): [n_codes][2048] complex int16;
 *            gnss_sdr_ru_b200/gpssdr_codes.py regenerates it
 * sv_list    0-based rows of that table (the reference's _sv), n_sv of them
 * doppmin, doppmax  Hz, searched kHz bins lcv = doppmin/1000 .. doppmax/1000 - 1 (within +-100 kHz)
 * results[i] the fields doAcq* fills in Acq_Command_S (RT/includes/structs.h:130-162)
 * ------------------------------------------------------------------------------------------- */
typedef struct gnssb200_gpssdr_result {
  int32_t sv;
  int32_t type;        /* ACQ_TYPE_STRONG 0 / ACQ_TYPE_MEDIUM 1 / ACQ_TYPE_WEAK 2 */
  int32_t code_phase;  /* samples at 2.048 Msps */
  int32_t doppler;     /* Hz */
  uint32_t magnitude;
  int32_t success;     /* magnitude > THRESH_* (all 0 in the reference, config.h:72-74) */
} gnssb200_gpssdr_result;
int gnssb200_gpssdr_acquire(gnssb200_handle *h, const int16_t *iq, int type, double fif, const int16_t *prn_codes, int n_codes,
                            const int32_t *sv_list, int n_sv, int doppmin, int doppmax, gnssb200_gpssdr_result *results);

/* Acq_Command_S Acquisition::doAcqMedium(int32 sv, int32 doppmin, int32 doppmax)  RT/objects/acquisition.cpp:309,
 * preceded by doPrepIF(ACQ_TYPE_MEDIUM, iq) with iq = 10 ms (20480 complex int16): 10 ms coherent, ten 25 Hz
 * post-correlation DFT rows, kHz bins doppmin/1000 .. doppmax/1000 INCLUSIVE (:325), result type 1.
 * The reference reads spectrum rows lcv2*20 + lcv3 (:340) while a 10-ms preparation fills rows offset*10 + ms
 * (:186-234): lcv2 = 0 sees the 0 Hz rows, lcv2 = 1 the 500 Hz rows (and reports them as +250 Hz), lcv2 = 2, 3
 * see rows 40-49 and 60-69, which keep what an EARLIER preparation of the same Acquisition object wrote.  That
 * history is an input here: prior_iq / prior_type (0, 1 or 2; NULL = a new object whose row storage is zero)
 * is the buffer of the last doPrepIF that ran before this one, e.g. the 310 ms of the preceding weak search. */
int gnssb200_gpssdr_acquire_medium(gnssb200_handle *h, const int16_t *iq, const int16_t *prior_iq, int prior_type, double fif,
                                   const int16_t *prn_codes, int n_codes, const int32_t *sv_list, int n_sv, int doppmin,
                                   int doppmax, gnssb200_gpssdr_result *results);

#ifdef __cplusplus
}
#endif
#endif /* GNSSB200_H_ */
