// softtrack.cu -- the Scilab receivers' floating-point tracking (SURVEY.md 8f rank 1):
// [trackResults, channel] = tracking(fid, channel, settings),
// SCI/GLONASS/L1/tracking.sci:226-400 and SCI/GPS/L1/tracking.sci (SCI = trunk/GNSS_SOFTWARE_RECEIVERS/
// POSTPROCESSING_SCILAB_RECEIVERS): one code period per iteration, block size ceil((L-rem)/step),
// float carrier / code NCOs, early/prompt/late sums, FLL-assisted PLL and DLL in double precision.
//
// One CTA per channel (channels are independent and each is sequential in time).  Every sample of a
// block is independent given the block's NCO state, so threads stride over the block (coalesced int8
// loads), evaluate the carrier with a double-precision sincos of the reference's own argument
// expression, index the code with ceil() exactly like the reference, and six double sums are reduced
// by shuffles; lane 0 runs the discriminators / loop filters and publishes the next block's state.
// FP64 throughout: the loop is a feedback system in doubles in the reference, FP32 would not track it.
//
// Virtual lanes: the arithmetic is defined by FTRK_LANES = 512 lanes.  Lane v takes samples v, v+512, ... of a
// block and its sums are reduced per warp of 32 lanes into red[v/32][q], then summed in warp order by thread 0.
// A CTA of NT threads (512, 256 or 128) runs lanes t, t+NT, ... one after another on thread t, so every width
// forms the same sums in the same order: the width is a scheduling choice, the results do not depend on it.
#include <math.h>

#include <vector>

#include "common.cuh"

#define FTRK_LANES 512
#define FTRK_WARPS (FTRK_LANES / 32)

struct FtrkArgs {
  const uint8_t *win;   // record r's window at win + r*win_stride; sample k at offset k - win_first (DESIGN §4.3)
  size_t win_stride;
  int n_records;
  long long win_first, win_end, record_samples;
  const int8_t *chips;  // [33][1024]
  gnssb200_softtrack_state *state;  // [n_ch]
  double *out;          // [n_ch][ms][13]
  int32_t *ms_done;     // [n_ch] or NULL: the one-shot calls' copy of state.ms_done
  int ms;
  int glonass;
  int code_len;
  double fs, IF, IF_step, zero_channel, code_freq_basis, spc;
  double k1, k2, k3, tau1, tau2;
};

struct FtrkState {
  double codeFreq, remCodePhase, carrFreq, remCarrPhase;
  long long pos;
  const uint8_t *rec;
  int blksize;
  int run;
  int code_row;
};

__device__ __forceinline__ double warp_sum_d(double v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// complex sample k of a window (k counted from the window's first sample, which is even for packed input): int8 I,Q,
// or the packed nibble (byte[k>>1] >> 4*(k&1)) & 15 with I in bits 0-1 and Q in bits 2-3, code {0:+1, 1:-1, 2:+3,
// 3:-3} (DESIGN §3, sample_at in acq.cu)
template <int FMT>
__device__ __forceinline__ void ftrk_sample(const uint8_t *rec, long long k, double &I, double &Q) {
  if (FMT == GNSSB200_FMT_PACKED2) {
    const unsigned c = ((unsigned)__ldg(rec + (k >> 1)) >> (4 * (int)(k & 1))) & 15u;
    I = (double)(((c & 2u) ? 3 : 1) * ((c & 1u) ? -1 : 1));
    Q = (double)(((c & 8u) ? 3 : 1) * ((c & 4u) ? -1 : 1));
  } else {
    const char2 v = __ldg(reinterpret_cast<const char2 *>(rec) + k);
    I = (double)v.x;
    Q = (double)v.y;
  }
}

// What a channel does next, from its state between two periods: GNSSB200_SOFTTRACK_* and whether it runs the block
// [pos, pos + blksize) now (only RUNNING channels whose block lies inside the window do).
__device__ __forceinline__ int ftrk_next(const FtrkArgs &a, long long pos, int blksize, int ms_done, int *run) {
  *run = 0;
  if (ms_done >= a.ms) return GNSSB200_SOFTTRACK_MS_DONE;
  if (pos < a.win_first) return GNSSB200_SOFTTRACK_BEHIND;
  if (pos + blksize > a.record_samples) return GNSSB200_SOFTTRACK_RECORD_END;
  *run = pos + blksize <= a.win_end;
  return GNSSB200_SOFTTRACK_RUNNING;
}

template <int NT, int FMT>
__global__ void __launch_bounds__(NT) softtrack_kernel(const FtrkArgs a) {
  static_assert(FTRK_LANES % NT == 0 && NT % 32 == 0, "a CTA runs whole warps of virtual lanes");
  __shared__ double code[1023 + 2];
  __shared__ FtrkState st;
  __shared__ double red[FTRK_WARPS][6];
  const int ch = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
  const int L = a.code_len;
  // loop state that only lane 0 needs
  gnssb200_softtrack_state *sp = a.state + ch;
  double oldCodeNco = 0.0, oldCodeError = 0.0, oldCarrNco = 0.0, oldCarrError = 0.0;
  double I1 = 0.0, Q1 = 0.0, carrFreqBasis = 0.0;
  int sv = 0, done = 0, status = 0;
  bool live = false;  // thread 0: the state is not final (RECORD_END and MS_DONE are; such a channel is left as it is)
  if (tid == 0) {
    status = sp->status;
    live = status <= GNSSB200_SOFTTRACK_RUNNING;
    st.run = 0;
    if (live) {
      oldCodeNco = sp->oldCodeNco;
      oldCodeError = sp->oldCodeError;
      oldCarrNco = sp->oldCarrNco;
      oldCarrError = sp->oldCarrError;
      I1 = sp->I1;
      Q1 = sp->Q1;
      carrFreqBasis = sp->carrFreqBasis;
      sv = sp->sv;
      done = sp->ms_done;
      const int record = sp->record;
      st.codeFreq = sp->codeFreq;
      st.remCodePhase = sp->remCodePhase;
      st.carrFreq = sp->carrFreq;
      st.remCarrPhase = sp->remCarrPhase;
      st.pos = sp->pos;
      st.code_row = a.glonass ? 0 : sv;
      st.rec = a.win + (size_t)record * a.win_stride;
      const double step = st.codeFreq / a.fs;
      st.blksize = (int)ceil(((double)L - st.remCodePhase) / step);
      if (record < 0 || record >= a.n_records)
        status = GNSSB200_SOFTTRACK_BAD_RECORD;
      else if (!a.glonass && (sv < 1 || sv > 32))
        status = GNSSB200_SOFTTRACK_BAD_SV;
      else
        status = ftrk_next(a, st.pos, st.blksize, done, &st.run);
    }
  }
  __syncthreads();
  if (st.run) {
    // caCode = [caCode($) caCode caCode(1)]  (tracking.sci:171-175)
    for (int i = tid; i < L + 2; i += NT) {
      const int k = (i == 0) ? L - 1 : (i == L + 1 ? 0 : i - 1);
      code[i] = (double)a.chips[st.code_row * 1024 + k];
    }
    __syncthreads();
  }
  const uint8_t *rec = st.rec;
  double *out = a.out + (size_t)ch * a.ms * 13;
  while (st.run) {
    const double codeFreq = st.codeFreq, rem = st.remCodePhase, carrFreq = st.carrFreq, remCarr = st.remCarrPhase;
    const long long pos = st.pos, wpos = pos - a.win_first;
    const int blksize = st.blksize;
    const double step = codeFreq / a.fs;            // codePhaseStep
    const double w = (carrFreq * 2.0) * M_PI;       // (carrFreq * 2.0 * %pi)
    const double remE = rem - a.spc, remL = rem + a.spc;
    // Carrier replica exp(i*trigarg), trigarg = ((carrFreq*2*pi) .* time) + remCarrPhase (tracking.sci:288-291).
    // A lane's samples are FTRK_LANES apart, i.e. a fixed phase step apart: one double-precision sincos of the
    // reference's own argument for its first sample, one for the step, then a complex rotation per sample
    // (4 FP64 multiply-adds instead of a ~100-instruction sincos; 31 rotations add ~1e-15 of relative error, the
    // reference's own argument carries ~1e-12 rad of rounding at 6000 rad).
    double sd, cd;
    sincos(__dmul_rn(w, __ddiv_rn((double)FTRK_LANES, a.fs)), &sd, &cd);
#pragma unroll 1
    for (int v = tid; v < FTRK_LANES; v += NT) {   // virtual lanes of this thread, one after another
      double s[6] = {0, 0, 0, 0, 0, 0};               // I_E Q_E I_P Q_P I_L Q_L
      double sn = 0.0, cs = 1.0;
      if (v < blksize) sincos(__dadd_rn(__dmul_rn(w, __ddiv_rn((double)v, a.fs)), remCarr), &sn, &cs);
      for (int j = v; j < blksize; j += FTRK_LANES) {
        double I, Q;
        ftrk_sample<FMT>(rec, wpos + j, I, Q);
        // carrsig .* rawSignal, carrsig = exp(%i*trigarg); qBaseband = real, iBaseband = imag
        const double qb = __dsub_rn(__dmul_rn(cs, I), __dmul_rn(sn, Q));
        const double ib = __dadd_rn(__dmul_rn(cs, Q), __dmul_rn(sn, I));
        const double dj = (double)j;
        const double e = code[(int)ceil(__dadd_rn(remE, __dmul_rn(dj, step)))];   // caCode(ceil(tcode)+1), 1-based
        const double p = code[(int)ceil(__dadd_rn(rem, __dmul_rn(dj, step)))];
        const double l = code[(int)ceil(__dadd_rn(remL, __dmul_rn(dj, step)))];
        // The multiply-adds are written out as the compiler contracted them before the width became a template
        // parameter, so that every instantiation rounds the same way.
        s[0] = __fma_rn(e, ib, s[0]);
        s[1] = __fma_rn(e, qb, s[1]);
        s[2] = __fma_rn(p, ib, s[2]);
        s[3] = __fma_rn(p, qb, s[3]);
        s[4] = __fma_rn(l, ib, s[4]);
        s[5] = __fma_rn(l, qb, s[5]);
        // advance the replica by FTRK_LANES samples: cs*cd - sn*sd, sn*cd + cs*sd
        const double c2 = __fma_rn(cs, cd, -__dmul_rn(sn, sd)), s2 = __fma_rn(cs, sd, __dmul_rn(sn, cd));
        cs = c2;
        sn = s2;
      }
#pragma unroll
      for (int q = 0; q < 6; q++) {
        const double r = warp_sum_d(s[q]);
        if (lane == 0) red[v >> 5][q] = r;
      }
    }
    __syncthreads();
    if (tid == 0) {
      double t[6];
      for (int q = 0; q < 6; q++) {
        double acc = 0.0;
        for (int wv = 0; wv < FTRK_WARPS; wv++) acc += red[wv][q];
        t[q] = acc;
      }
      const double I_E = t[0], Q_E = t[1], I_P = t[2], Q_P = t[3], I_L = t[4], Q_L = t[5];
      // tracking.sci:301-303, 309-312
      const double newRem = __dadd_rn(__dadd_rn(rem, __dmul_rn((double)(blksize - 1), step)), step) - (double)L;
      const double last = __dadd_rn(__dmul_rn(w, __ddiv_rn((double)blksize, a.fs)), remCarr);
      const double newRemCarr = __dsub_rn(last, __dmul_rn(trunc(last / (2 * M_PI)), 2 * M_PI));
      // FLL-assisted PLL (:327-347)
      const double I2 = I1, Q2 = Q1;
      I1 = I_P;
      Q1 = Q_P;
      const double cross = I1 * Q2 - I2 * Q1;
      const double dot = fabs(I1 * I2 + Q1 * Q2);
      const double freqError = atan2(cross, dot) / M_PI;
      const double carrError = atan(Q_P / I_P) / (2.0 * M_PI);
      const double carrNco = oldCarrNco + a.k1 * carrError - a.k2 * oldCarrError - a.k3 * freqError;
      oldCarrNco = carrNco;
      oldCarrError = carrError;
      const double newCarrFreq = carrFreqBasis + carrNco;
      // DLL (:352-371)
      const double sE = sqrt(I_E * I_E + Q_E * Q_E), sL = sqrt(I_L * I_L + Q_L * Q_L);
      const double codeError = (sE - sL) / (sE + sL);
      const double codeNco = oldCodeNco + (a.tau2 / a.tau1) * (codeError - oldCodeError) + codeError * (0.001 / a.tau1);
      oldCodeNco = codeNco;
      oldCodeError = codeError;
      double newCodeFreq;
      if (a.glonass)
        newCodeFreq = a.code_freq_basis - codeNco +
                      (newCarrFreq - (a.IF + a.IF_step * sv)) / ((a.zero_channel + sv * a.IF_step) / a.code_freq_basis);
      else
        newCodeFreq = a.code_freq_basis - codeNco + ((newCarrFreq - a.IF) / 1540);
      const long long newPos = pos + blksize;
      double *o = out + (size_t)done * 13;
      o[0] = I_E; o[1] = I_P; o[2] = I_L; o[3] = Q_E; o[4] = Q_P; o[5] = Q_L;
      o[6] = newCarrFreq; o[7] = newCodeFreq; o[8] = codeError; o[9] = codeNco; o[10] = carrError; o[11] = carrNco;
      o[12] = (double)newPos - newRem * (a.fs / 1000) / (double)L;   // absoluteSample (:380-384)
      st.codeFreq = newCodeFreq;
      st.remCodePhase = newRem;
      st.carrFreq = newCarrFreq;
      st.remCarrPhase = newRemCarr;
      st.pos = newPos;
      const double nstep = newCodeFreq / a.fs;
      st.blksize = (int)ceil(((double)L - newRem) / nstep);
      done++;
      status = ftrk_next(a, newPos, st.blksize, done, &st.run);
    }
    __syncthreads();
  }
  if (tid == 0) {  // the state after the last period run, also at a pause
    if (live) {
      sp->codeFreq = st.codeFreq;
      sp->remCodePhase = st.remCodePhase;
      sp->carrFreq = st.carrFreq;
      sp->remCarrPhase = st.remCarrPhase;
      sp->oldCodeNco = oldCodeNco;
      sp->oldCodeError = oldCodeError;
      sp->oldCarrNco = oldCarrNco;
      sp->oldCarrError = oldCarrError;
      sp->I1 = I1;
      sp->Q1 = Q1;
      sp->pos = st.pos;
      sp->ms_done = done;
      sp->status = status;
    }
    if (a.ms_done) a.ms_done[ch] = sp->ms_done;
  }
}

template <int NT>
static void ftrk_launch_nt(int fmt, int n_ch, cudaStream_t st, const FtrkArgs &a) {
  if (fmt == GNSSB200_FMT_PACKED2)
    softtrack_kernel<NT, GNSSB200_FMT_PACKED2><<<n_ch, NT, 0, st>>>(a);
  else
    softtrack_kernel<NT, GNSSB200_FMT_INT8_IQ><<<n_ch, NT, 0, st>>>(a);
}

template <int NT>
static int ftrk_ctas_per_sm(int fmt, int *occ) {
  if (fmt == GNSSB200_FMT_PACKED2)
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, softtrack_kernel<NT, GNSSB200_FMT_PACKED2>, NT, 0));
  else
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, softtrack_kernel<NT, GNSSB200_FMT_INT8_IQ>, NT, 0));
  return 0;
}

// Threads per channel chosen by gnssb200_softtrack_batch when the handle leaves it open (gnssb200_set_softtrack_width
// 0).  A channel's run is a chain of code periods, so the call takes (waves of CTAs) x (time of one wave), a wave
// being the CTAs resident at once.  Measured on a B200 (DESIGN §4.3), a full wave of 512 / 256 / 128-thread CTAs
// takes 1 : 1.7 : 2.25 of the time of a full wave at 512 threads, and 1 / 3 / 5 CTAs of these widths fit an SM
// (cudaOccupancy*).  The width with the fewest wave-times wins (the wider on a tie); with 148 SMs that is 512 up to
// 148 channels, 256 up to 444, 128 up to 740, and beyond that whichever of 256 and 128 needs fewer wave-times.
static int ftrk_auto_width(gnssb200_handle *h, int fmt, int n_ch, int *nt_out) {
  static const int widths[3] = {512, 256, 128};
  static const double wave_cost[3] = {1.0, 1.7, 2.25};
  int n_sm = 0;
  CUDA_TRY(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, h->device));
  double best = 0.0;
  for (int k = 0; k < 3; k++) {
    int occ = 0;
    if (int rc = (k == 0 ? ftrk_ctas_per_sm<512>(fmt, &occ) : k == 1 ? ftrk_ctas_per_sm<256>(fmt, &occ) : ftrk_ctas_per_sm<128>(fmt, &occ)))
      return rc;
    const long long slots = (long long)(occ > 0 ? occ : 1) * n_sm;
    const double cost = (double)((n_ch + slots - 1) / slots) * wave_cost[k];
    if (k == 0 || cost < best) {
      best = cost;
      *nt_out = widths[k];
    }
  }
  return 0;
}

static FtrkArgs ftrk_args(const gnssb200_softtrack_cfg *cfg) {
  FtrkArgs a = {};
  a.ms = cfg->ms_to_process;
  a.glonass = cfg->system == GNSSB200_SYS_GLONASS ? 1 : 0;
  a.code_len = cfg->code_length;
  a.fs = cfg->samp_freq;
  a.IF = cfg->IF;
  a.IF_step = cfg->IF_step;
  a.zero_channel = cfg->glonass_zero_channel;
  a.code_freq_basis = cfg->code_freq;
  a.spc = cfg->dll_correlator_spacing;
  {  // calcLoopCoef.sci:38-43 (k = 1.0), calcFLLPLLLoopCoef.sci:36-38 (T = 0.001)
    const double zeta = cfg->dll_damping_ratio, LBW = cfg->dll_noise_bandwidth;
    const double Wn = LBW * 8 * zeta / (4 * zeta * zeta + 1);
    a.tau1 = 1.0 / (Wn * Wn);
    a.tau2 = 2.0 * zeta / Wn;
    const double T = 0.001, p = cfg->pll_noise_bandwidth / 0.53;
    a.k1 = T * (p * p) + 1.414 * p;
    a.k2 = 1.414 * p;
    a.k3 = T * (cfg->fll_noise_bandwidth / 0.25);
  }
  return a;
}

// One window of the tracking kernel for the n_ch states of d_state; arguments validated by the callers.  nt: threads
// per channel, 0 = the handle's width (or the automatic one).  Asynchronous on st.
static int ftrk_window(gnssb200_handle *h, const gnssb200_softtrack_cfg *cfg, const void *d_win, size_t win_stride,
                       int n_records, int fmt, int64_t win_first, int64_t win_samples, int64_t record_samples,
                       gnssb200_softtrack_state *d_state, int n_ch, double *d_out, int32_t *d_ms_done, cudaStream_t st,
                       int nt) {
  CUDA_TRY(cudaSetDevice(h->device));
  const int8_t *d_chips = nullptr;
  if (int rc = chip_table(h, &d_chips)) return rc;
  if (nt == 0) nt = h->softtrack_width;
  if (nt == 0)
    if (int rc = ftrk_auto_width(h, fmt, n_ch, &nt)) return rc;
  FtrkArgs a = ftrk_args(cfg);
  a.win = (const uint8_t *)d_win;
  a.win_stride = win_stride;
  a.n_records = n_records;
  a.win_first = win_first;
  a.win_end = win_first + win_samples;
  a.record_samples = record_samples;
  a.chips = d_chips;
  a.state = d_state;
  a.out = d_out;
  a.ms_done = d_ms_done;
  if (nt == 128)
    ftrk_launch_nt<128>(fmt, n_ch, st, a);
  else if (nt == 256)
    ftrk_launch_nt<256>(fmt, n_ch, st, a);
  else
    ftrk_launch_nt<512>(fmt, n_ch, st, a);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  return 0;
}

static int ftrk_bad(int rc, const char *what) {
  gnssb200_set_error(rc, what, __FILE__, __LINE__);
  return rc;
}

// The correlator spacing the kernel can read: 0 <= spc <= 0.5 chip (NaN fails).  The early / prompt / late chips are
// code[ceil(rem -+ spc + j*step)] of the padded period code[0..L+1] = [caCode($) caCode caCode(1)], for the samples
// j = 0..blksize-1 of a block.  blksize = ceil((L - rem) / step) puts rem + j*step in [rem, L), and the remainder
// carried into the next block, rem + blksize*step - L, lies in [0, step), both up to rounding: rem is exactly 0 in
// period 1 and can be a few 1e-13 below 0 after it.  The early index ceil(rem - spc) >= 0 needs spc < 1 + rem, the
// late index ceil(t + spc) <= L + 1 (t < L) needs spc <= 1 less the rounding of t.  With rem a little below 0 no bound
// just under 1 chip is airtight; 0.5 chip each side, the widest conventional spacing (10x the GLONASS default 0.05,
// 2.5x the GPS one 0.2), leaves half a chip for rounding.  (The reference stops on an index outside the padded code:
// Scilab raises on index 0 or L + 3.)
static bool ftrk_spacing_ok(const gnssb200_softtrack_cfg *cfg) {
  return cfg->dll_correlator_spacing >= 0.0 && cfg->dll_correlator_spacing <= 0.5;
}

// int8 I,Q samples are read as 2-byte char2 loads, which need an even address: the record base and its stride must be
// even.  Packed records are read byte by byte and may start anywhere.
static bool ftrk_aligned(int fmt, const void *base, size_t stride) {
  return fmt != GNSSB200_FMT_INT8_IQ || !(((uintptr_t)base | stride) & 1);
}

extern "C" int gnssb200_softtrack_init(const gnssb200_softtrack_cfg *cfg, const gnssb200_softtrack_chan *chans,
                                       const int32_t *chan_record, int n_records, int n_ch, gnssb200_softtrack_state *states) {
  if (!cfg || !chans || !states || n_ch <= 0 || n_records < 1 || cfg->ms_to_process <= 0 ||
      (cfg->code_length != 511 && cfg->code_length != 1023) || !ftrk_spacing_ok(cfg))
    return ftrk_bad(-20, "gnssb200_softtrack_init: bad arguments");
  if (cfg->system != GNSSB200_SYS_GLONASS)
    for (int i = 0; i < n_ch; i++)
      if (chans[i].sv < 1 || chans[i].sv > 32) return ftrk_bad(-21, "gnssb200_softtrack_init: GPS PRN must be 1..32");
  if (chan_record)
    for (int i = 0; i < n_ch; i++)
      if (chan_record[i] < 0 || chan_record[i] >= n_records) return ftrk_bad(-24, "gnssb200_softtrack_init: chan_record out of range");
  for (int i = 0; i < n_ch; i++) {  // tracking.sci:226-250: the loop state before period 1
    gnssb200_softtrack_state s = {};
    s.codeFreq = cfg->code_freq;
    s.carrFreq = chans[i].acquired_freq;
    s.I1 = 0.001;
    s.Q1 = 0.001;
    s.carrFreqBasis = chans[i].acquired_freq;
    s.pos = cfg->skip_samples + (int64_t)(chans[i].code_phase - 1);
    s.sv = chans[i].sv;
    s.record = chan_record ? chan_record[i] : 0;
    s.status = GNSSB200_SOFTTRACK_RUNNING;
    states[i] = s;
  }
  return 0;
}

// The one-shot tracking of n_ch channels spread over records d_iq + rec*stride (chan_record NULL: every channel in
// record 0): init and one window that covers the whole record.  Arguments are validated by the callers.  Synchronous
// on cuda_stream.
static int softtrack_run(gnssb200_handle *h, const gnssb200_softtrack_cfg *cfg, const void *d_iq, size_t stride,
                         int n_records, int fmt, int64_t n_samples, const gnssb200_softtrack_chan *chans,
                         const int32_t *chan_record, int n_ch, double *d_out, int32_t *d_ms_done, void *cuda_stream, int nt) {
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  std::vector<gnssb200_softtrack_state> hs(n_ch);
  if (int rc = gnssb200_softtrack_init(cfg, chans, chan_record, n_records, n_ch, hs.data())) return rc;
  gnssb200_softtrack_state *d_state = nullptr;
  CUDA_TRY(cudaMalloc(&d_state, sizeof(gnssb200_softtrack_state) * n_ch));
  int rc = 0;
  cudaError_t e = cudaMemcpyAsync(d_state, hs.data(), sizeof(gnssb200_softtrack_state) * n_ch, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaEventRecord(h->ev0, st);
  if (e == cudaSuccess)
    rc = ftrk_window(h, cfg, d_iq, stride, n_records, fmt, 0, n_samples, n_samples, d_state, n_ch, d_out, d_ms_done, st, nt);
  if (e == cudaSuccess && !rc) e = cudaEventRecord(h->ev1, st);
  if (e == cudaSuccess && !rc) e = cudaStreamSynchronize(st);  // hs / d_state lifetimes
  cudaFree(d_state);
  if (rc) return rc;
  CUDA_TRY(e);
  return 0;
}

extern "C" int gnssb200_softtrack(gnssb200_handle *h, const gnssb200_softtrack_cfg *cfg, const void *d_iq, int64_t n_samples,
                                  const gnssb200_softtrack_chan *chans, int n_ch, double *d_out, int32_t *d_ms_done,
                                  void *cuda_stream) {
  if (!h || !cfg || !d_iq || !chans || n_ch <= 0 || !d_out || !d_ms_done || cfg->ms_to_process <= 0 ||
      (cfg->code_length != 511 && cfg->code_length != 1023) ||  // the kernel's chip buffer holds one ST or C/A period
      !ftrk_spacing_ok(cfg)) {
    gnssb200_set_error(-20, "gnssb200_softtrack: bad arguments", __FILE__, __LINE__);
    return -20;
  }
  if (!ftrk_aligned(GNSSB200_FMT_INT8_IQ, d_iq, 0))
    return ftrk_bad(-23, "gnssb200_softtrack: an int8 I,Q record must start on an even byte address");
  if (cfg->system != GNSSB200_SYS_GLONASS)
    for (int i = 0; i < n_ch; i++)
      if (chans[i].sv < 1 || chans[i].sv > 32) {
        gnssb200_set_error(-21, "gnssb200_softtrack: GPS PRN must be 1..32", __FILE__, __LINE__);
        return -21;
      }
  return softtrack_run(h, cfg, d_iq, 0, 1, GNSSB200_FMT_INT8_IQ, n_samples, chans, nullptr, n_ch, d_out, d_ms_done,
                       cuda_stream, FTRK_LANES);
}

static size_t ftrk_bytes(int fmt, int64_t n) { return fmt == GNSSB200_FMT_INT8_IQ ? (size_t)n * 2 : ((size_t)n + 1) / 2; }

// The argument checks of gnssb200_softtrack_batch and gnssb200_softtrack_batch_host (d_iq / h_iq, d_out / h_out, ...)
static int ftrk_check_batch(const char *fn, gnssb200_handle *h, const gnssb200_softtrack_cfg *cfg, const void *iq,
                            size_t record_stride_bytes, int n_records, int fmt, int64_t n_samples,
                            const gnssb200_softtrack_chan *chans, const int32_t *chan_record, int n_ch, const double *out,
                            const int32_t *ms_done) {
  char msg[160];
  if (!h || !cfg || !iq || !chans || !chan_record || n_ch <= 0 || !out || !ms_done || cfg->ms_to_process <= 0 ||
      (cfg->code_length != 511 && cfg->code_length != 1023) || !ftrk_spacing_ok(cfg) || n_samples < 0) {
    snprintf(msg, sizeof msg, "%s: bad arguments", fn);
    return ftrk_bad(-20, msg);
  }
  if (cfg->system != GNSSB200_SYS_GLONASS)
    for (int i = 0; i < n_ch; i++)
      if (chans[i].sv < 1 || chans[i].sv > 32) {
        snprintf(msg, sizeof msg, "%s: GPS PRN must be 1..32", fn);
        return ftrk_bad(-21, msg);
      }
  if (fmt != GNSSB200_FMT_INT8_IQ && fmt != GNSSB200_FMT_PACKED2) {
    snprintf(msg, sizeof msg, "%s: fmt must be INT8_IQ or PACKED2", fn);
    return ftrk_bad(-22, msg);
  }
  if (n_records < 1 || (record_stride_bytes != 0 && record_stride_bytes < ftrk_bytes(fmt, n_samples))) {
    snprintf(msg, sizeof msg, "%s: n_records < 1, or a record stride shorter than n_samples in fmt", fn);
    return ftrk_bad(-23, msg);
  }
  for (int i = 0; i < n_ch; i++)
    if (chan_record[i] < 0 || chan_record[i] >= n_records) {
      snprintf(msg, sizeof msg, "%s: chan_record out of range", fn);
      return ftrk_bad(-24, msg);
    }
  return 0;
}

extern "C" int gnssb200_softtrack_batch(gnssb200_handle *h, const gnssb200_softtrack_cfg *cfg, const void *d_iq,
                                        size_t record_stride_bytes, int n_records, int fmt, int64_t n_samples,
                                        const gnssb200_softtrack_chan *chans, const int32_t *chan_record, int n_ch,
                                        double *d_out, int32_t *d_ms_done, void *cuda_stream) {
  if (int rc = ftrk_check_batch("gnssb200_softtrack_batch", h, cfg, d_iq, record_stride_bytes, n_records, fmt, n_samples,
                                chans, chan_record, n_ch, d_out, d_ms_done))
    return rc;
  if (!ftrk_aligned(fmt, d_iq, record_stride_bytes))
    return ftrk_bad(-23, "gnssb200_softtrack_batch: int8 I,Q records need an even d_iq and an even record stride");
  return softtrack_run(h, cfg, d_iq, record_stride_bytes, n_records, fmt, n_samples, chans, chan_record, n_ch, d_out,
                       d_ms_done, cuda_stream, 0);
}

extern "C" int gnssb200_softtrack_resume(gnssb200_handle *h, const gnssb200_softtrack_cfg *cfg, const void *d_win,
                                         size_t win_stride_bytes, int n_records, int fmt, int64_t win_first,
                                         int64_t win_samples, int64_t record_samples, gnssb200_softtrack_state *d_state,
                                         int n_ch, double *d_out, void *cuda_stream) {
  if (!h || !cfg || !d_win || !d_state || !d_out || n_ch <= 0 || n_records < 1 || win_first < 0 || win_samples < 0 ||
      cfg->ms_to_process <= 0 || (cfg->code_length != 511 && cfg->code_length != 1023) || !ftrk_spacing_ok(cfg))
    return ftrk_bad(-20, "gnssb200_softtrack_resume: bad arguments");
  if (fmt != GNSSB200_FMT_INT8_IQ && fmt != GNSSB200_FMT_PACKED2)
    return ftrk_bad(-22, "gnssb200_softtrack_resume: fmt must be INT8_IQ or PACKED2");
  if (fmt == GNSSB200_FMT_PACKED2 && (win_first & 1))
    return ftrk_bad(-22, "gnssb200_softtrack_resume: a packed window must start on an even sample");
  if (win_stride_bytes != 0 && win_stride_bytes < ftrk_bytes(fmt, win_samples))
    return ftrk_bad(-23, "gnssb200_softtrack_resume: a window stride shorter than win_samples in fmt");
  if (!ftrk_aligned(fmt, d_win, win_stride_bytes))
    return ftrk_bad(-23, "gnssb200_softtrack_resume: int8 I,Q windows need an even d_win and an even window stride");
  if (!h->d_chips) {  // the handle's chip table is built by a synchronous upload, which a stream capture cannot hold
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaStreamIsCapturing((cudaStream_t)cuda_stream, &cap));
    if (cap != cudaStreamCaptureStatusNone)
      return ftrk_bad(-27, "gnssb200_softtrack_resume: capture needs one float-tracking call on the handle before it");
  }
  return ftrk_window(h, cfg, d_win, win_stride_bytes, n_records, fmt, win_first, win_samples, record_samples, d_state, n_ch,
                     d_out, nullptr, (cudaStream_t)cuda_stream, 0);
}

// Automatic window of gnssb200_softtrack_batch_host: 2^20 samples (65.5 ms at 16 Msps), fewer if a staging buffer would
// pass 512 MiB.  Measured on a B200 with 64 records x 8 channels (DESIGN §4.3): 2^20 samples was the fastest of 2^18,
// 2^20 and 2^22 for int8 (128 MiB buffers) and of 2^20, 2^22 and 2^24 for packed (32 MiB), 1.03-1.12x the larger of the
// kernel time and the copy time.  Longer windows leave a longer first copy and last kernel without overlap.
#define FTRK_AUTO_WINDOW_SAMPLES (1LL << 20)
#define FTRK_MAX_STAGE_BYTES ((size_t)512 << 20)

extern "C" int gnssb200_softtrack_batch_host(gnssb200_handle *h, const gnssb200_softtrack_cfg *cfg, const void *h_iq,
                                             size_t stride, int n_records, int fmt, int64_t n_samples,
                                             const gnssb200_softtrack_chan *chans, const int32_t *chan_record, int n_ch,
                                             double *h_out, int32_t *h_ms_done, int64_t window_samples) {
  if (int rc = ftrk_check_batch("gnssb200_softtrack_batch_host", h, cfg, h_iq, stride, n_records, fmt, n_samples, chans,
                                chan_record, n_ch, h_out, h_ms_done))
    return rc;
  // nominal code period P; windows overlap by 2P (even for packed input, so every window starts on an even sample)
  const double period = ceil((double)cfg->code_length * cfg->samp_freq / cfg->code_freq);
  const long long P = period >= 1.0 && period < 1e9 ? (long long)period : 0;
  if (P == 0 || window_samples < 0 || (window_samples > 0 && window_samples < 4 * P))
    return ftrk_bad(-26, "gnssb200_softtrack_batch_host: window_samples must be 0 or at least four code periods");
  const bool packed = fmt == GNSSB200_FMT_PACKED2;
  const long long O = packed ? (2 * P + 1) & ~1LL : 2 * P;
  const int rows_copied = stride ? n_records : 1;  // stride 0: one record, read n_records times
  long long W = window_samples;
  if (W == 0) {
    const long long rec_bytes = (long long)(FTRK_MAX_STAGE_BYTES / rows_copied);
    const long long cap = packed ? 2 * rec_bytes : rec_bytes / 2;
    W = FTRK_AUTO_WINDOW_SAMPLES < cap ? FTRK_AUTO_WINDOW_SAMPLES : cap;
    if (W < 4 * P) W = 4 * P;
  }
  if (W > n_samples) W = n_samples;  // one window holds the whole record: staging memory follows the input
  long long A = W - O;  // advance from one window to the next
  if (packed) A &= ~1LL;
  const size_t wbytes = ftrk_bytes(fmt, W);
  const size_t dpitch = (wbytes + 255) & ~(size_t)255;
  CUDA_TRY(cudaSetDevice(h->device));
  int rc = 0;
  auto fail = [&](cudaError_t e, int line) {
    gnssb200_set_error((int)e, cudaGetErrorString(e), __FILE__, line);
    rc = (int)e;
  };
#define TRY_(x)                                       \
  do {                                                \
    cudaError_t e_ = (x);                             \
    if (e_ != cudaSuccess && !rc) fail(e_, __LINE__); \
  } while (0)
  // the handle's staging streams, events and buffers, shared with gnssb200_track_run_host (both synchronise)
  if (!h->s_copy) {
    TRY_(cudaStreamCreateWithFlags(&h->s_copy, cudaStreamNonBlocking));
    TRY_(cudaStreamCreateWithFlags(&h->s_comp, cudaStreamNonBlocking));
    TRY_(cudaStreamCreateWithFlags(&h->s_back, cudaStreamNonBlocking));
    for (int i = 0; i < 2; i++) {
      TRY_(cudaEventCreateWithFlags(&h->ev_copied[i], cudaEventDisableTiming));
      TRY_(cudaEventCreateWithFlags(&h->ev_used[i], cudaEventDisableTiming));
    }
  }
  const size_t stage_need = dpitch * rows_copied + 256;
  if (!rc && stage_need > h->stage_cap) {
    for (int i = 0; i < 2; i++) {
      cudaFree(h->stage[i]);
      h->stage[i] = nullptr;
      TRY_(cudaMalloc(&h->stage[i], stage_need));
    }
    h->stage_cap = rc ? 0 : stage_need;
  }
  std::vector<gnssb200_softtrack_state> hs(n_ch);
  if (!rc) rc = gnssb200_softtrack_init(cfg, chans, chan_record, n_records, n_ch, hs.data());
  gnssb200_softtrack_state *d_state = nullptr;
  double *d_out = nullptr;
  const size_t ch_rows = (size_t)cfg->ms_to_process * GNSSB200_SOFTTRACK_FIELDS;
  if (!rc) TRY_(cudaMalloc(&d_state, sizeof(gnssb200_softtrack_state) * n_ch));
  if (!rc) TRY_(cudaMalloc(&d_out, sizeof(double) * ch_rows * n_ch));
  cudaStream_t s_copy = h->s_copy, s_comp = h->s_comp;
  if (!rc)
    TRY_(cudaMemcpyAsync(d_state, hs.data(), sizeof(gnssb200_softtrack_state) * n_ch, cudaMemcpyHostToDevice, s_comp));
  if (!rc) TRY_(cudaEventRecord(h->ev0, s_comp));
  for (long long k = 0, first = 0; !rc; k++, first += A) {
    const long long len = n_samples - first < W ? n_samples - first : W;
    const int buf = (int)(k & 1);
    if (k >= 2) TRY_(cudaStreamWaitEvent(s_copy, h->ev_used[buf], 0));  // the kernel of window k-2 is done with it
    const size_t lbytes = ftrk_bytes(fmt, len);
    if (lbytes)
      TRY_(cudaMemcpy2DAsync(h->stage[buf], dpitch, (const uint8_t *)h_iq + (packed ? first / 2 : 2 * first),
                             stride ? stride : lbytes, lbytes, rows_copied, cudaMemcpyHostToDevice, s_copy));
    TRY_(cudaEventRecord(h->ev_copied[buf], s_copy));
    TRY_(cudaStreamWaitEvent(s_comp, h->ev_copied[buf], 0));
    if (!rc)
      rc = ftrk_window(h, cfg, h->stage[buf], stride ? dpitch : 0, n_records, fmt, first, len, n_samples, d_state, n_ch,
                       d_out, nullptr, s_comp, 0);
    TRY_(cudaEventRecord(h->ev_used[buf], s_comp));
    if (first + W >= n_samples) break;
  }
  if (!rc) TRY_(cudaEventRecord(h->ev1, s_comp));
  if (!rc)
    TRY_(cudaMemcpyAsync(hs.data(), d_state, sizeof(gnssb200_softtrack_state) * n_ch, cudaMemcpyDeviceToHost, s_comp));
  if (s_comp) TRY_(cudaStreamSynchronize(s_comp));
  if (s_copy) TRY_(cudaStreamSynchronize(s_copy));
  int stopped = 0;
  if (!rc) {
    for (int i = 0; i < n_ch && !rc; i++) {
      if (hs[i].ms_done > 0)
        TRY_(cudaMemcpyAsync(h_out + ch_rows * i, d_out + ch_rows * i, sizeof(double) * GNSSB200_SOFTTRACK_FIELDS * hs[i].ms_done,
                             cudaMemcpyDeviceToHost, s_comp));
      // the last window reaches the record end, so every channel ends RECORD_END or MS_DONE unless a block was
      // longer than the overlap; a pos before sample 0 stops the one-shot call as well
      if (hs[i].status == GNSSB200_SOFTTRACK_BEHIND && hs[i].pos >= 0) stopped++;
    }
    TRY_(cudaStreamSynchronize(s_comp));
    if (!rc)
      for (int i = 0; i < n_ch; i++) h_ms_done[i] = hs[i].ms_done;
  }
  cudaFree(d_state);
  cudaFree(d_out);
#undef TRY_
  return rc ? rc : stopped;
}

extern "C" int gnssb200_set_softtrack_width(gnssb200_handle *h, int threads) {
  if (!h || (threads != 0 && threads != 128 && threads != 256 && threads != 512)) {
    gnssb200_set_error(-25, "gnssb200_set_softtrack_width: threads must be 0, 128, 256 or 512", __FILE__, __LINE__);
    return -25;
  }
  h->softtrack_width = threads;
  return 0;
}
