// track.cu -- GP2021-style E/P/L correlator bank + closed channel loop on the device.
//
// What it replaces: Sim_GP2021_int (OSG/correlator/correlator.c:148-316) followed by gpsisr
// (OSG/isr/osgpsisr.c:360-408) once per 512 us block, for S independent IF streams x 12 channels.
//
// Two kernels share the arithmetic below (closed-form NCO starts, grouped code taps, dump rules, device ISR):
//
//   track_ws_kernel    the hot path (8192-sample blocks or shorter, 16-byte aligned, int8 I,Q or packed 2+2 bit):
//                      warp-specialised -- correlator warps + one control lane per CTA, decoupled by mbarriers,
//                      samples staged by the TMA engine, ISR bookkeeping after the next block's parameters are
//                      published -- and scheduled through a (channel, time-slice) work queue.  Described where
//                      it is defined.
//   track_loop_kernel  the generic variant (any block length, unaligned or ragged records, I-only input; also
//                      selectable with GNSSB200_TRACK_WS=0 for A/B runs): one CTA per (stream, channel) for the
//                      whole run, barrier-synchronised: TMA double buffering, 32 samples per thread per pass,
//                      warp-shuffle + shared-atomic reduction, lane 0 of warp 0 as the ISR lane.
//
// Per block, both: every thread takes consecutive complex samples, starts its carrier/code NCOs from the closed
// form phase(i) = phase0 + i*incr (SURVEY.md Appendix A) and walks them with the exact integer arithmetic of the
// reference: 8-phase LO (phase>>29), complex mix, +-1 E/P/L taps at half-chip spacing.  I and Q products ride in
// one 32-bit register as two 16-bit lanes.  Samples go four at a time: with 4*kinc < 2^32 at most one code-NCO
// carry falls inside a group, so the group contributes old_bits*S_old + new_bits*S_new -- 6 IMADs and one table
// read per 4 samples.  At most one dump per block on this path; the single straddling chunk is re-evaluated
// sample-per-lane by its warp from the closed forms.
//
// Register values the fast path cannot express (a second dump inside one block, slews beyond the table window,
// PRN outside 1..32, ...) take the serial path: one lane walks the block with the literal per-sample loop.  It is
// still device code; there is no CPU fallback.
#include "track_common.cuh"
#include "track_loop.cuh"
#include "track_ws.cuh"

// one thread per stream: status words, TIC counter and block counter after a run
__global__ void track_finish_kernel(gnssb200_rx *rx, const int32_t *chan_flags, int first_stream, int n_streams,
                                    int nsamp, long long nblocks, long long tic_ref) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_streams) return;
  const int s = first_stream + t;
  gnssb200_rx *r = rx + s;
  if (nblocks <= 0 || r->halted) return;
  int status = 0, halted = 0;
  for (int ch = 0; ch < NCH; ch++) {
    const int f = chan_flags[s * NCH + ch];
    if (f & 1) status |= 1 << ch;
    if (f & 2) halted = 1;
  }
  long long tic = r->tic;
  int tic_count = -1;
  for (long long b = 0; b < nblocks; b++) {
    if (tic < nsamp) {
      tic_count = (int)tic;
      tic += tic_ref - nsamp;
    } else {
      tic -= nsamp;
      tic_count = -1;
    }
  }
  r->tic = tic;
  r->reg_read[0x82] = status;                        // correlator.c:309
  r->reg_read[0x83] = (tic_count > -1) ? 0x2000 : 0; // :312-315
  r->blocks_done += nblocks;
  if (halted) r->halted = 1;
}

// ---- diagnostics: the device ISR's integer helpers on arrays (tests/test_isr_math.py) -----------------
__global__ void isr_math_kernel(int n, const int *y, const int *x, int *at, const long long *L, unsigned *sq, const int *num,
                                const int *den, int *dv) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  at[i] = dev_atan2_i32(y[i], x[i]);
  sq[i] = dev_isqrt(L[i]);
  dv[i] = dev_div_small(num[i], den[i]);
}

extern "C" int gnssb200_isr_math_eval(gnssb200_handle *h, int n, const int32_t *y, const int32_t *x, int32_t *atan_out,
                                      const int64_t *L, uint32_t *sqrt_out, const int32_t *num, const int32_t *den,
                                      int32_t *div_out) {
  if (!h || n <= 0) return 0;
  CUDA_TRY(cudaSetDevice(h->device));
  int *d_i = nullptr;
  long long *d_L = nullptr;
  CUDA_TRY(cudaMalloc(&d_i, (size_t)n * 7 * sizeof(int)));
  CUDA_TRY(cudaMalloc(&d_L, (size_t)n * sizeof(long long)));
  int *dy = d_i, *dx = d_i + n, *dat = d_i + 2 * (size_t)n, *dnum = d_i + 3 * (size_t)n, *dden = d_i + 4 * (size_t)n,
      *ddv = d_i + 5 * (size_t)n;
  unsigned *dsq = (unsigned *)(d_i + 6 * (size_t)n);
  CUDA_TRY(cudaMemcpy(dy, y, (size_t)n * 4, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(dx, x, (size_t)n * 4, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(dnum, num, (size_t)n * 4, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(dden, den, (size_t)n * 4, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(d_L, L, (size_t)n * 8, cudaMemcpyHostToDevice));
  isr_math_kernel<<<(n + 255) / 256, 256>>>(n, dy, dx, dat, d_L, dsq, dnum, dden, ddv);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpy(atan_out, dat, (size_t)n * 4, cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaMemcpy(sqrt_out, dsq, (size_t)n * 4, cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaMemcpy(div_out, ddv, (size_t)n * 4, cudaMemcpyDeviceToHost));
  cudaFree(d_i);
  cudaFree(d_L);
  h->launches += 1;
  return 0;
}

// TRACK_CHECK builds: violations counted by the kernels since the last call (-1: the library was built without the checks)
extern "C" int gnssb200_track_check_failures(unsigned out[8]) {
#ifdef TRACK_CHECK
  unsigned h[8], z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (cudaMemcpyFromSymbol(h, g_track_check_fail, sizeof h) != cudaSuccess) return -2;
  cudaMemcpyToSymbol(g_track_check_fail, z, sizeof z);
  int n = 0;
  for (int i = 0; i < 8; i++) {
    if (out) out[i] = h[i];
    n += (int)h[i];
  }
  return n;
#else
  (void)out;
  return -1;
#endif
}

// ---- host side -----------------------------------------------------------------------------------
void build_code_table_host(uint32_t *table) {
  // C/A Gold codes, G2 register start states per PRN (IS-GPS-200; same values as correlator.c:67-71),
  // replicas at half-chip spacing: early[h]=c[h>>1], prompt[h]=c[((h+1)%2046)>>1], late[h]=c[((h+2)%2046)>>1]
  static const int g2_start[33] = {0x000, 0x3f6, 0x3ec, 0x3d8, 0x3b0, 0x04b, 0x096, 0x2cb, 0x196, 0x32c, 0x3ba,
                                   0x374, 0x1d0, 0x3a0, 0x340, 0x280, 0x100, 0x113, 0x226, 0x04c, 0x098, 0x130,
                                   0x260, 0x267, 0x338, 0x270, 0x0e0, 0x1c0, 0x380, 0x22b, 0x056, 0x0ac, 0x158};
  for (int i = 0; i <= TABLE_ENTRIES; i++) table[i] = 0;
  for (int prn = 1; prn <= 32; prn++) {
    int chip[1023];
    int g1 = 0x1FF, g2 = g2_start[prn];
    chip[0] = 1;
    for (int c = 1; c < 1023; c++) {
      chip[c] = (g1 ^ g2) & 1;
      g1 = (g1 >> 1) | (((g1 << 2) ^ (g1 << 9)) & 0x200);
      g2 = (g2 >> 1) | (((g2 << 1) ^ (g2 << 2) ^ (g2 << 5) ^ (g2 << 7) ^ (g2 << 8) ^ (g2 << 9)) & 0x200);
    }
    for (int h = 0; h < HALF_CHIPS; h++) {
      const int e = 2 * chip[(h % HALF_CHIPS) >> 1] - 1;
      const int p = 2 * chip[((h + 1) % HALF_CHIPS) >> 1] - 1;
      const int l = 2 * chip[((h + 2) % HALF_CHIPS) >> 1] - 1;
      table[prn * HALF_CHIPS + h] = (uint32_t)(e & 0xff) | ((uint32_t)(p & 0xff) << 8) | ((uint32_t)(l & 0xff) << 16);
    }
  }
  {  // GLONASS ST code as NAM/rtl/code_gen.v:121-133 generates it: nine-stage register, all ones after the PRN-key
     // write, output stage g3[2], feedback g3[4]^g3[0] (= SCI/GLONASS/L1/include/generateSTcode.sci:35-42); replicas at
     // half-chip spacing like the C/A rows with the period 1022
    int chip[511];
    unsigned g3 = 0x1FF;
    for (int c = 0; c < 511; c++) {
      chip[c] = (g3 >> 2) & 1;
      g3 = (g3 >> 1) | ((((g3 >> 4) ^ g3) & 1u) << 8);
    }
    for (int h = 0; h < GLO_HALF_CHIPS; h++) {
      const int e = 2 * chip[(h % GLO_HALF_CHIPS) >> 1] - 1;
      const int p = 2 * chip[((h + 1) % GLO_HALF_CHIPS) >> 1] - 1;
      const int l = 2 * chip[((h + 2) % GLO_HALF_CHIPS) >> 1] - 1;
      table[GLO_ROW * HALF_CHIPS + h] = (uint32_t)(e & 0xff) | ((uint32_t)(p & 0xff) << 8) | ((uint32_t)(l & 0xff) << 16);
    }
  }
}

size_t track_sched_bytes(int n_streams) {  // work-queue storage for a handle with n_streams receivers
  return sizeof(SchedQueue) * (size_t)n_streams + (size_t)n_streams * NCH * (8 + 8 + 4) + 256;
}

int track_launch(gnssb200_handle *h, int first_stream, int n_streams, const void *d_if, size_t stride, int fmt,
                 int nsamp, long long nblocks, int run_isr, gnssb200_dump *d_dumps, int dump_cap,
                 int32_t *d_dump_count, cudaStream_t st) {
  if (n_streams <= 0 || nblocks <= 0) return 0;
  TrackArgs a;
  a.rx = h->d_rx;
  a.chan_flags = h->d_chan_flags;
  a.code_table = h->d_code_table;
  a.d_if = (const uint8_t *)d_if - (size_t)first_stream * stride;  // kernel indexes by absolute stream
  a.stride = stride;
  a.fmt = fmt;
  a.nsamp = nsamp;
  a.nblocks = nblocks;
  a.run_isr = run_isr;
  a.first_stream = first_stream;
  a.dumps = d_dumps;
  a.dump_cap = dump_cap;
  a.dump_count = d_dump_count;
  a.sched = nullptr;
  a.k1 = 1u;
  a.k8 = 8u;
  a.k128 = 128u;
  a.k2048 = 2048u;
  static_cast<gnssb200_cfg &>(a.cfg) = h->cfg;
  {
    const double m = h->cfg.clock_mult;
    const long long im = (long long)m;
    a.cfg.mult_i = ((double)im == m && im > -1024 && im < 1024) ? (int)im : 0;
    const gnssb200_cfg &c = h->cfg;
    auto ab = [](long long v) { return v < 0 ? -v : v; };
    const bool pll_ok = (ab(c.pll_i1) + ab(c.pll_i2)) * (1ll << 17) + ab(c.pll_i3) * (1ll << 16) < (1ll << 31);
    const bool dll_ok = (ab((long long)c.dll_i1 + 1) + ab(c.dll_i2)) * (1ll << 17) < (1ll << 31);
    const int shc = 32 - c.carrier_nco_bits, shk = 32 - c.code_nco_bits;
    a.cfg.fast32 = (a.cfg.mult_i != 0 && pll_ok && dll_ok && shc >= 0 && shc <= 8 && shk >= 0 && shk <= 8) ? 1 : 0;
  }
  const int grid = n_streams * NCH;
  const int spt = 32;
  int threads = (nsamp + spt - 1) / spt;  // track_loop_kernel: 32 samples per thread per pass
  threads = ((threads + 31) / 32) * 32;
  if (threads > 1024) threads = 1024;
  if (threads < 32) threads = 32;
  // TMA staging needs 16-byte aligned blocks that fit one tile per CTA pass
  const size_t blk_bytes = fmt == GNSSB200_FMT_INT8_IQ ? (size_t)nsamp * 2 : (fmt == GNSSB200_FMT_PACKED2 ? (size_t)nsamp / 2 : (size_t)nsamp);
  const bool aligned = (((uintptr_t)d_if | stride | blk_bytes) & 15) == 0 && (nsamp % 8) == 0;
  static int no_tma = -1;
  if (no_tma < 0) {
    const char *e = getenv("GNSSB200_TRACK_NO_TMA");
    no_tma = (e && atoi(e)) ? 1 : 0;
  }
  const int use_tma = (aligned && !no_tma && nsamp <= 256 * spt && blk_bytes <= 16384) ? 1 : 0;
  const int tile_bytes = use_tma ? (int)((blk_bytes + 127) & ~(size_t)127) : 0;
  const size_t dyn = (size_t)2 * tile_bytes + ((use_tma && fmt == GNSSB200_FMT_PACKED2) ? 128 * 32 * 4 : 0);
  static bool attr_done[64] = {};  // the opt-in is per device
  if (h->device < 0 || h->device >= 64 || !attr_done[h->device]) {
    CUDA_TRY(cudaFuncSetAttribute(track_loop_kernel<256, 2, GNSSB200_FMT_INT8_IQ, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 16384 + 256));
    CUDA_TRY(cudaFuncSetAttribute(track_loop_kernel<256, 2, GNSSB200_FMT_PACKED2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 3 * 16384 + 256));
    if (h->device >= 0 && h->device < 64) attr_done[h->device] = true;
  }
  static int force_occ = -1;  // GNSSB200_TRACK_OCC: force the resident-CTAs-per-SM variant (experiments)
  if (force_occ < 0) {
    const char *e = getenv("GNSSB200_TRACK_OCC");
    force_occ = e ? atoi(e) : 0;
  }
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
  const bool hot = use_tma && nsamp <= 8192 && (fmt == GNSSB200_FMT_INT8_IQ || fmt == GNSSB200_FMT_PACKED2);
  static int use_ws = -1;
  if (use_ws < 0) {
    const char *e = getenv("GNSSB200_TRACK_WS");
    use_ws = e ? atoi(e) : 1;
  }
  // gnssb200_set_track_variant: 0 automatic, 1 the barrier-synchronised kernel, 2 fixed sample runs, 3/4/5 half-chip
  // segments with 96 / 192 / 384 correlator threads
  static int env_form = -1;  // GNSSB200_TRACK_FORM: the same selection for handles that did not choose (experiments)
  if (env_form < 0) {
    const char *e = getenv("GNSSB200_TRACK_FORM");
    env_form = e ? atoi(e) : 0;
  }
  const int form = h->track_form ? h->track_form : env_form;
  if (form != 1 && use_ws && hot) {  // warp-specialised variant: correlator warps + control lane
    constexpr int DSM_I8 = 2 * 16384 + 256, DSM_PK = 3 * 16384 + 256;
    // the shared-memory opt-in is a per-device attribute of each kernel
    static bool aws[64] = {};
    if (h->device < 0 || h->device >= 64 || !aws[h->device]) {
      CUDA_TRY(cudaFuncSetAttribute(track_ws_kernel<2, GNSSB200_FMT_INT8_IQ, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, DSM_I8));
      CUDA_TRY(cudaFuncSetAttribute(track_ws_kernel<3, GNSSB200_FMT_INT8_IQ, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, DSM_I8));
      CUDA_TRY(cudaFuncSetAttribute(track_ws_kernel<5, GNSSB200_FMT_INT8_IQ, 128, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, DSM_I8));
      CUDA_TRY(cudaFuncSetAttribute(track_ws_kernel<2, GNSSB200_FMT_PACKED2, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, DSM_PK));
      CUDA_TRY(cudaFuncSetAttribute(track_ws_kernel<3, GNSSB200_FMT_PACKED2, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, DSM_PK));
      CUDA_TRY(cudaFuncSetAttribute(track_ws_kernel<1, GNSSB200_FMT_PACKED2, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, DSM_PK));
      CUDA_TRY(cudaFuncSetAttribute(track_ws_kernel<4, GNSSB200_FMT_PACKED2, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, DSM_PK));
      CUDA_TRY(cudaFuncSetAttribute(track_ws_kernel<6, GNSSB200_FMT_PACKED2, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, DSM_PK));
      CUDA_TRY(cudaFuncSetAttribute(track_ws_kernel<5, GNSSB200_FMT_PACKED2, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, DSM_PK));
      CUDA_TRY(cudaFuncSetAttribute(track_ws_kernel<4, GNSSB200_FMT_PACKED2, 96, 11>, cudaFuncAttributeMaxDynamicSharedMemorySize, DSM_PK));
      CUDA_TRY(cudaFuncSetAttribute(track_ws_kernel<5, GNSSB200_FMT_PACKED2, 96, 11>, cudaFuncAttributeMaxDynamicSharedMemorySize, DSM_PK));
      CUDA_TRY(cudaFuncSetAttribute(track_ws_kernel<6, GNSSB200_FMT_PACKED2, 96, 11>, cudaFuncAttributeMaxDynamicSharedMemorySize, DSM_PK));
      CUDA_TRY(cudaFuncSetAttribute(track_ws_kernel<3, GNSSB200_FMT_PACKED2, 192, 6>, cudaFuncAttributeMaxDynamicSharedMemorySize, DSM_PK));
      CUDA_TRY(cudaFuncSetAttribute(track_ws_kernel<5, GNSSB200_FMT_PACKED2, 192, 6>, cudaFuncAttributeMaxDynamicSharedMemorySize, DSM_PK));
      CUDA_TRY(cudaFuncSetAttribute(track_ws_kernel<6, GNSSB200_FMT_PACKED2, 192, 6>, cudaFuncAttributeMaxDynamicSharedMemorySize, DSM_PK));
      CUDA_TRY(cudaFuncSetAttribute(track_ws_kernel<2, GNSSB200_FMT_PACKED2, 384, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, DSM_PK));
      if (h->device >= 0 && h->device < 64) aws[h->device] = true;
    }
    // Work queue: every channel's blocks are cut into slices of slice_blocks; one CTA per (channel, slice)
    // item, items handed out through the FIFO so that a channel's slices run in order.
    static long long env_slice = -1;
    if (env_slice < 0) {
      const char *e = getenv("GNSSB200_TRACK_SLICE");
      env_slice = e ? atoll(e) : 0;
    }
    // Slicing pays where the GPU is throughput bound (four or more channels per SM): there it keeps every SM
    // full to the end.  With few channels each channel's latency is the limit, tickets land on SMs at random
    // (two running CTAs may share an SM next to an idle one), so those runs stay one item per channel.
    const int per_sm_need = (grid + sms - 1) / sms;
    // Slice length: 512 KB of samples per stream (128 blocks of packed, 32 of int8 input), so that the slices in flight
    // (one per stream, shared by its 12 channels) stay L2 resident: with 128-block slices of int8 input (2 MB x 64
    // streams) the channels of a stream no longer found each other's tiles in L2 and DRAM reads were 3.4 x the record
    // (ncu; 1.6 x at 32 blocks for 4 % of the speed, the price of 4 x as many slice hand-overs).
    long long auto_slice = (512 * 1024) / (long long)(blk_bytes ? blk_bytes : 1);
    auto_slice = auto_slice < 8 ? 8 : (auto_slice > 128 ? 128 : auto_slice);
    const long long slice_blocks = h->track_slice > 0 ? h->track_slice : (env_slice > 0 ? env_slice : (per_sm_need >= 4 ? auto_slice : nblocks));
    const unsigned nslices = (unsigned)((nblocks + slice_blocks - 1) / slice_blocks);
    const size_t n_all = (size_t)h->n_streams * NCH;
    uint8_t *base = (uint8_t *)h->d_sched;
    SchedQueue *qd = reinterpret_cast<SchedQueue *>(base) + first_stream;  // one header per possible first stream
    long long *tic = reinterpret_cast<long long *>(base + sizeof(SchedQueue) * (size_t)h->n_streams) + (size_t)first_stream * NCH;
    SchedSlot *slots = reinterpret_cast<SchedSlot *>(base + sizeof(SchedQueue) * (size_t)h->n_streams + 8 * n_all) + (size_t)first_stream * NCH;
    int32_t *dcnt = reinterpret_cast<int32_t *>(base + sizeof(SchedQueue) * (size_t)h->n_streams + 16 * n_all) + (size_t)first_stream * NCH;
    if (nslices > 1) {
      sched_init_kernel<<<(grid + 255) / 256, 256, 0, st>>>(qd, (unsigned)grid, nslices, slice_blocks, tic, dcnt, slots);
      CUDA_TRY(cudaGetLastError());
      h->launches += 1;
      a.sched = qd;
    }
    const unsigned items = (unsigned)grid * nslices;
    // CTAs per SM the channels ask for -> variant (registers / samples per thread)
    const int occ = h->track_occ ? h->track_occ : force_occ;
    const int per_sm = occ ? occ : (grid + sms - 1) / sms;
    // Half-chip segments need 7 or 8 samples per half chip: decided from the nominal code NCO word of this
    // configuration (a block whose word left that range is still handled, sample by sample, inside the kernel).
    bool seg = false;
    if ((fmt == GNSSB200_FMT_PACKED2 || fmt == GNSSB200_FMT_INT8_IQ) && form != 2) {
      const int shk = 32 - h->cfg.code_nco_bits;
      if (shk >= 0 && shk < 32) {
        const long long w = (long long)((double)((long long)h->cfg.gps_code_ref << shk) * h->cfg.clock_mult);  // gp2021.c:100-118
        const unsigned long long kinc = ((unsigned long long)(w & 0xffffffffll)) << 1;
        seg = kinc >= (1ull << 29) && 7ull * kinc <= (1ull << 32);
      }
      static int env_seg = -1;
      if (env_seg < 0) {
        const char *e = getenv("GNSSB200_TRACK_SEG");
        env_seg = e ? atoi(e) : 1;
      }
      if (!env_seg && form == 0) seg = false;
      // Up to one channel per SM the run is bound by each channel's own block-to-block latency, and there 256 threads
      // with 32 consecutive samples each finish a block sooner than 96 threads with 11 segments each (measured, 2 s of
      // signal: 1 stream 63 k vs 52 k, 8 streams 494 k vs 412 k channel*Msamples/s; from 16 streams on the segment
      // form is ahead: 721 k vs 691 k, 64 streams 1865 k vs 1436 k).
      if (form == 0 && per_sm <= 1) seg = false;
      if (form >= 3) seg = true;  // forced: out-of-range blocks take the per-sample form inside the kernel
    }
    const size_t dyn_seg = dyn + 2048;  // slack to start the mixer table on a 2048-byte boundary
    // segment form on int8 I,Q samples; 224 bytes of read-ahead behind the second tile.  Eight segments per thread: a
    // thread sums up to 8 x 8 samples of up to 384 per 16-bit lane before it unpacks them (24576 <= 32767 for any int8
    // input; eleven segments could reach 33792 and carry into the other lane).  127 x 8 = 1016 of the ~1048 segments
    // of an 8192-sample block are owned, the rest is the tail.
    if (fmt == GNSSB200_FMT_INT8_IQ && seg && (form == 0 || form == 3))
      track_ws_kernel<5, GNSSB200_FMT_INT8_IQ, 128, 8><<<items, 160, dyn + 256, st>>>(a, tile_bytes);
    else if (fmt == GNSSB200_FMT_INT8_IQ && per_sm >= 3)
      track_ws_kernel<3, GNSSB200_FMT_INT8_IQ, 256><<<items, 288, dyn, st>>>(a, tile_bytes);
    else if (fmt == GNSSB200_FMT_INT8_IQ)
      track_ws_kernel<2, GNSSB200_FMT_INT8_IQ, 256><<<items, 288, dyn, st>>>(a, tile_bytes);
    else if (seg && form == 5)
      track_ws_kernel<2, GNSSB200_FMT_PACKED2, 384, 3><<<items, 416, dyn_seg, st>>>(a, tile_bytes);
    else if (seg && form == 4 && per_sm >= 6)
      track_ws_kernel<6, GNSSB200_FMT_PACKED2, 192, 6><<<items, 224, dyn_seg, st>>>(a, tile_bytes);
    else if (seg && form == 4 && per_sm >= 4)
      track_ws_kernel<5, GNSSB200_FMT_PACKED2, 192, 6><<<items, 224, dyn_seg, st>>>(a, tile_bytes);
    else if (seg && form == 4)
      track_ws_kernel<3, GNSSB200_FMT_PACKED2, 192, 6><<<items, 224, dyn_seg, st>>>(a, tile_bytes);
    else if (seg && per_sm >= 6)
      track_ws_kernel<6, GNSSB200_FMT_PACKED2, 96, 11><<<items, 128, dyn_seg, st>>>(a, tile_bytes);
    else if (seg && per_sm == 5)
      track_ws_kernel<5, GNSSB200_FMT_PACKED2, 96, 11><<<items, 128, dyn_seg, st>>>(a, tile_bytes);
    else if (seg)
      track_ws_kernel<4, GNSSB200_FMT_PACKED2, 96, 11><<<items, 128, dyn_seg, st>>>(a, tile_bytes);
    // fixed sample runs: 64 samples per thread only when they tile the block (a thread always takes its whole run)
    else if (occ == 6 && nsamp % 64 == 0)
      track_ws_kernel<6, GNSSB200_FMT_PACKED2, 128><<<items, 160, dyn, st>>>(a, tile_bytes);
    else if (per_sm >= 5 && nsamp % 64 == 0)  // five resident CTAs of 72 registers beat six of 64 (spills) by 1-4 % under the work queue
      track_ws_kernel<5, GNSSB200_FMT_PACKED2, 128><<<items, 160, dyn, st>>>(a, tile_bytes);
    else if (per_sm == 4 && nsamp % 64 == 0)
      track_ws_kernel<4, GNSSB200_FMT_PACKED2, 128><<<items, 160, dyn, st>>>(a, tile_bytes);
    else if (per_sm >= 3)
      track_ws_kernel<3, GNSSB200_FMT_PACKED2, 256><<<items, 288, dyn, st>>>(a, tile_bytes);
    else if (occ == 1 && nsamp % 16 == 0)  // 512 threads x 16 samples (experiments: shorter blocks for lone channels)
      track_ws_kernel<1, GNSSB200_FMT_PACKED2, 512><<<items, 544, dyn, st>>>(a, tile_bytes);
    else
      track_ws_kernel<2, GNSSB200_FMT_PACKED2, 256><<<items, 288, dyn, st>>>(a, tile_bytes);
  } else
  if (hot && fmt == GNSSB200_FMT_INT8_IQ)  // GNSSB200_TRACK_WS=0: the barrier-synchronised predecessor, kept for A/B runs
    track_loop_kernel<256, 2, GNSSB200_FMT_INT8_IQ, true><<<grid, threads, dyn, st>>>(a, tile_bytes);
  else if (hot)
    track_loop_kernel<256, 2, GNSSB200_FMT_PACKED2, true><<<grid, threads, dyn, st>>>(a, tile_bytes);
  else
    track_loop_kernel<1024, 1, -1, false><<<grid, threads, 0, st>>>(a, 0);
  CUDA_TRY(cudaGetLastError());
  track_finish_kernel<<<(n_streams + 127) / 128, 128, 0, st>>>(h->d_rx, h->d_chan_flags, first_stream, n_streams, nsamp,
                                                               nblocks, h->cfg.tic_ref);
  CUDA_TRY(cudaGetLastError());
  h->launches += 2;
  return 0;
}
