// common.cuh -- shared declarations of libgnssb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/gnssb200.h"

#define NCH GNSSB200_N_CHANNELS
#define HALF_CHIPS 2046
#define TABLE_ROWS 37                       // rows 0, 33, 34 and 36 are zero (SURVEY.md 7.3 Q3); row 35 = GLONASS ST code
#define TABLE_ENTRIES (TABLE_ROWS * HALF_CHIPS)
#define GLO_ROW 35                          // E/P/L of the 511-chip ST code: 1022 entries, the rest of the row is zero
#define GLO_HALF_CHIPS 1022

// PRN register -> first entry of the channel's row in the flat E/P/L table (-1: no code, all reads give 0) and the
// number of half chips after which the channel dumps.  GPS rows are addressed by the register value itself like in
// correlator.c:193-198 (0..33; 0 and 33 are zero rows); GNSSB200_PRN_GLONASS selects the ST-code row.
__host__ __device__ __forceinline__ long long code_table_base(int prn_reg) {
  if (prn_reg == GNSSB200_PRN_GLONASS) return (long long)GLO_ROW * HALF_CHIPS;
  return (prn_reg >= 0 && prn_reg <= 33) ? (long long)prn_reg * HALF_CHIPS : -1;
}
// End of what a channel may read: a GPS row spills over into the rows after it like the reference's flat reads, but
// only up to the end of row 33 (the reference has 33 rows; reads past the zero row 33 give 0, never the ST code of row
// 35).  Only the GLONASS row reaches into rows 35 and 36.
#define GPS_TABLE_END (34 * HALF_CHIPS)
__host__ __device__ __forceinline__ long long code_row_end(int prn_reg) { return prn_reg == GNSSB200_PRN_GLONASS ? TABLE_ENTRIES : GPS_TABLE_END; }
__host__ __device__ __forceinline__ int code_period(int prn_reg) { return prn_reg == GNSSB200_PRN_GLONASS ? GLO_HALF_CHIPS : HALF_CHIPS; }
__host__ __device__ __forceinline__ bool code_has_fast_row(int prn_reg) { return (prn_reg >= 1 && prn_reg <= 32) || prn_reg == GNSSB200_PRN_GLONASS; }

// library-wide error slot (api.cu)
void gnssb200_set_error(int code, const char *what, const char *file, int line);
#define CUDA_TRY(expr)                                                        \
  do {                                                                        \
    cudaError_t e__ = (expr);                                                 \
    if (e__ != cudaSuccess) {                                                 \
      gnssb200_set_error((int)e__, cudaGetErrorString(e__), __FILE__, __LINE__); \
      return (int)e__;                                                        \
    }                                                                         \
  } while (0)

struct gnssb200_handle {
  int device;
  gnssb200_cfg cfg;
  int n_streams;
  gnssb200_rx *d_rx;          // [n_streams]
  int32_t *d_chan_flags;      // [n_streams*12] bit0: dumped in the last block, bit1: halted
  long long track_slice;      // blocks per work-queue slice of the tracking kernel; 0 = automatic (gnssb200_set_track_slice)
  int track_form, track_occ;  // kernel form / occupancy variant forced by gnssb200_set_track_variant (0 = automatic)
  int softtrack_width;        // threads per channel of gnssb200_softtrack_batch (gnssb200_set_softtrack_width; 0 = automatic)
  void *d_sched;              // work queue of track_ws_kernel: headers / TIC counters / slots / dump counters per channel
  uint32_t *d_code_table;     // [TABLE_ENTRIES+1] packed E | P<<8 | L<<16 (int8 each), last entry 0
  int8_t *d_chips;            // [33][1024] chips as +-1: row 0 GLONASS ST code, rows 1..32 GPS C/A (chip_table, synth.cu)
  cudaEvent_t ev0, ev1;
  long long launches;
  float serial_ms;            // device time of the last gnssb200_acq_serial run
  // acquisition workspace (acq.cu)
  void *acq_ws;
  // staging of gnssb200_track_run_host (api.cu), kept between calls
  uint8_t *stage[2];
  size_t stage_cap;
  gnssb200_dump *stage_dumps;
  size_t stage_dumps_cap;
  int32_t *stage_cnt;
  size_t stage_cnt_cap;
  cudaStream_t s_copy, s_comp;
  cudaEvent_t ev_copied[2], ev_used[2];
  cudaStream_t s_back;        // device -> host stream of the dump-record windows (gnssb200_track_run_host)
  int32_t *h_snap;            // pinned: dump counts after every chunk
  size_t h_snap_cap;
  long long stage_blocks;     // blocks per stream and staging chunk; 0 = automatic (gnssb200_set_stage_blocks)
  long long back_fallbacks;   // host-buffer runs that had to repeat the dump read-back in one piece
};

// track.cu
int track_launch(gnssb200_handle *h, int first_stream, int n_streams, const void *d_if, size_t stride, int fmt,
                 int nsamp, long long nblocks, int run_isr, gnssb200_dump *d_dumps, int dump_cap,
                 int32_t *d_dump_count, cudaStream_t st);
void build_code_table_host(uint32_t *table /* TABLE_ENTRIES+1 */);
size_t track_sched_bytes(int n_streams);

// synth.cu: the handle's chip table (built on first use, freed by gnssb200_close)
int chip_table(gnssb200_handle *h, const int8_t **d_chips);

// acq.cu
void acq_free_workspace(gnssb200_handle *h);
