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

struct FtrkChanDev {
  int sv;               // PRN (GPS) or frequency channel (GLONASS)
  int code_row;         // row in the chip table (0: GLONASS ST code, 1..32: C/A)
  double acquired_freq;
  long long start;      // first complex sample of the channel in its record (skip + codePhase - 1)
  long long rec_off;    // byte offset of the channel's record from FtrkArgs::iq
};

struct FtrkArgs {
  const uint8_t *iq;
  long long n_samples;  // of every record
  const int8_t *chips;  // [33][1024]
  const FtrkChanDev *chan;
  double *out;          // [n_ch][ms][13]
  int32_t *ms_done;     // [n_ch]
  int ms;
  int glonass;
  int code_len;
  double fs, IF, IF_step, zero_channel, code_freq_basis, spc;
  double k1, k2, k3, tau1, tau2;
};

struct FtrkState {
  double codeFreq, remCodePhase, carrFreq, remCarrPhase;
  long long pos;
  int blksize;
  int stop;
};

__device__ __forceinline__ double warp_sum_d(double v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// complex sample k of a record: int8 I,Q, or the packed nibble (byte[k>>1] >> 4*(k&1)) & 15 with I in bits 0-1 and
// Q in bits 2-3, code {0:+1, 1:-1, 2:+3, 3:-3} (DESIGN §3, sample_at in acq.cu)
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

template <int NT, int FMT>
__global__ void __launch_bounds__(NT) softtrack_kernel(const FtrkArgs a) {
  static_assert(FTRK_LANES % NT == 0 && NT % 32 == 0, "a CTA runs whole warps of virtual lanes");
  __shared__ double code[1023 + 2];
  __shared__ FtrkState st;
  __shared__ double red[FTRK_WARPS][6];
  const int ch = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
  const FtrkChanDev c = a.chan[ch];
  const uint8_t *rec = a.iq + c.rec_off;
  const int L = a.code_len;
  // caCode = [caCode($) caCode caCode(1)]  (tracking.sci:171-175)
  for (int i = tid; i < L + 2; i += NT) {
    const int k = (i == 0) ? L - 1 : (i == L + 1 ? 0 : i - 1);
    code[i] = (double)a.chips[c.code_row * 1024 + k];
  }
  // loop state that only lane 0 needs
  double oldCodeNco = 0.0, oldCodeError = 0.0, oldCarrNco = 0.0, oldCarrError = 0.0;
  double I1 = 0.001, Q1 = 0.001;
  const double carrFreqBasis = c.acquired_freq;
  if (tid == 0) {
    st.codeFreq = a.code_freq_basis;
    st.remCodePhase = 0.0;
    st.carrFreq = c.acquired_freq;
    st.remCarrPhase = 0.0;
    st.pos = c.start;
    st.stop = 0;
    const double step = st.codeFreq / a.fs;
    st.blksize = (int)ceil(((double)L - st.remCodePhase) / step);
    if (st.pos < 0 || st.pos + st.blksize > a.n_samples) st.stop = 1;
  }
  __syncthreads();
  double *out = a.out + (size_t)ch * a.ms * 13;
  int done = 0;
  for (int it = 0; it < a.ms; it++) {
    if (st.stop) break;
    const double codeFreq = st.codeFreq, rem = st.remCodePhase, carrFreq = st.carrFreq, remCarr = st.remCarrPhase;
    const long long pos = st.pos;
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
        ftrk_sample<FMT>(rec, pos + j, I, Q);
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
                      (newCarrFreq - (a.IF + a.IF_step * c.sv)) / ((a.zero_channel + c.sv * a.IF_step) / a.code_freq_basis);
      else
        newCodeFreq = a.code_freq_basis - codeNco + ((newCarrFreq - a.IF) / 1540);
      const long long newPos = pos + blksize;
      double *o = out + (size_t)it * 13;
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
      if (newPos + st.blksize > a.n_samples) st.stop = 1;
    }
    done = it + 1;
    __syncthreads();
  }
  if (tid == 0) a.ms_done[ch] = done;
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

// The tracking of n_ch channels spread over records d_iq + rec*stride; chan_record NULL: every channel in record 0.
// Arguments are validated by the callers.  Synchronous on cuda_stream.
static int softtrack_run(gnssb200_handle *h, const gnssb200_softtrack_cfg *cfg, const void *d_iq, size_t stride, int fmt,
                         int64_t n_samples, const gnssb200_softtrack_chan *chans, const int32_t *chan_record, int n_ch,
                         double *d_out, int32_t *d_ms_done, void *cuda_stream, int nt) {
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const int8_t *d_chips = nullptr;
  if (int rc = chip_table(h, &d_chips)) return rc;
  const bool glo = cfg->system == GNSSB200_SYS_GLONASS;
  std::vector<FtrkChanDev> hc(n_ch);
  for (int i = 0; i < n_ch; i++) {
    hc[i].sv = chans[i].sv;
    hc[i].code_row = glo ? 0 : chans[i].sv;
    hc[i].acquired_freq = chans[i].acquired_freq;
    hc[i].start = cfg->skip_samples + (int64_t)(chans[i].code_phase - 1);
    hc[i].rec_off = chan_record ? (long long)((size_t)chan_record[i] * stride) : 0;
  }
  FtrkChanDev *d_ch = nullptr;
  CUDA_TRY(cudaMalloc(&d_ch, sizeof(FtrkChanDev) * n_ch));
  cudaError_t e = cudaMemcpyAsync(d_ch, hc.data(), sizeof(FtrkChanDev) * n_ch, cudaMemcpyHostToDevice, st);
  if (e != cudaSuccess) {
    cudaFree(d_ch);
    CUDA_TRY(e);
  }
  FtrkArgs a;
  a.iq = (const uint8_t *)d_iq;
  a.n_samples = n_samples;
  a.chips = d_chips;
  a.chan = d_ch;
  a.out = d_out;
  a.ms_done = d_ms_done;
  a.ms = cfg->ms_to_process;
  a.glonass = glo ? 1 : 0;
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
  e = cudaEventRecord(h->ev0, st);
  if (e == cudaSuccess) {
    if (nt == 128)
      ftrk_launch_nt<128>(fmt, n_ch, st, a);
    else if (nt == 256)
      ftrk_launch_nt<256>(fmt, n_ch, st, a);
    else
      ftrk_launch_nt<512>(fmt, n_ch, st, a);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaEventRecord(h->ev1, st);
  if (e == cudaSuccess) {
    h->launches++;
    e = cudaStreamSynchronize(st);  // hc / d_ch lifetimes
  }
  cudaFree(d_ch);
  CUDA_TRY(e);
  return 0;
}

extern "C" int gnssb200_softtrack(gnssb200_handle *h, const gnssb200_softtrack_cfg *cfg, const void *d_iq, int64_t n_samples,
                                  const gnssb200_softtrack_chan *chans, int n_ch, double *d_out, int32_t *d_ms_done,
                                  void *cuda_stream) {
  if (!h || !cfg || !d_iq || !chans || n_ch <= 0 || !d_out || !d_ms_done || cfg->ms_to_process <= 0 ||
      (cfg->code_length != 511 && cfg->code_length != 1023)) {  // the kernel's chip buffer holds one ST or C/A period
    gnssb200_set_error(-20, "gnssb200_softtrack: bad arguments", __FILE__, __LINE__);
    return -20;
  }
  if (cfg->system != GNSSB200_SYS_GLONASS)
    for (int i = 0; i < n_ch; i++)
      if (chans[i].sv < 1 || chans[i].sv > 32) {
        gnssb200_set_error(-21, "gnssb200_softtrack: GPS PRN must be 1..32", __FILE__, __LINE__);
        return -21;
      }
  return softtrack_run(h, cfg, d_iq, 0, GNSSB200_FMT_INT8_IQ, n_samples, chans, nullptr, n_ch, d_out, d_ms_done, cuda_stream,
                       FTRK_LANES);
}

extern "C" int gnssb200_softtrack_batch(gnssb200_handle *h, const gnssb200_softtrack_cfg *cfg, const void *d_iq,
                                        size_t record_stride_bytes, int n_records, int fmt, int64_t n_samples,
                                        const gnssb200_softtrack_chan *chans, const int32_t *chan_record, int n_ch,
                                        double *d_out, int32_t *d_ms_done, void *cuda_stream) {
  if (!h || !cfg || !d_iq || !chans || !chan_record || n_ch <= 0 || !d_out || !d_ms_done || cfg->ms_to_process <= 0 ||
      (cfg->code_length != 511 && cfg->code_length != 1023) || n_samples < 0) {
    gnssb200_set_error(-20, "gnssb200_softtrack_batch: bad arguments", __FILE__, __LINE__);
    return -20;
  }
  if (cfg->system != GNSSB200_SYS_GLONASS)
    for (int i = 0; i < n_ch; i++)
      if (chans[i].sv < 1 || chans[i].sv > 32) {
        gnssb200_set_error(-21, "gnssb200_softtrack_batch: GPS PRN must be 1..32", __FILE__, __LINE__);
        return -21;
      }
  if (fmt != GNSSB200_FMT_INT8_IQ && fmt != GNSSB200_FMT_PACKED2) {
    gnssb200_set_error(-22, "gnssb200_softtrack_batch: fmt must be INT8_IQ or PACKED2", __FILE__, __LINE__);
    return -22;
  }
  const size_t rec_bytes = fmt == GNSSB200_FMT_INT8_IQ ? (size_t)n_samples * 2 : ((size_t)n_samples + 1) / 2;
  if (n_records < 1 || (record_stride_bytes != 0 && record_stride_bytes < rec_bytes)) {
    gnssb200_set_error(-23, "gnssb200_softtrack_batch: n_records < 1, or a record stride shorter than n_samples in fmt",
                       __FILE__, __LINE__);
    return -23;
  }
  for (int i = 0; i < n_ch; i++)
    if (chan_record[i] < 0 || chan_record[i] >= n_records) {
      gnssb200_set_error(-24, "gnssb200_softtrack_batch: chan_record out of range", __FILE__, __LINE__);
      return -24;
    }
  int nt = h->softtrack_width;
  if (nt == 0) {
    CUDA_TRY(cudaSetDevice(h->device));
    if (int rc = ftrk_auto_width(h, fmt, n_ch, &nt)) return rc;
  }
  return softtrack_run(h, cfg, d_iq, record_stride_bytes, fmt, n_samples, chans, chan_record, n_ch, d_out, d_ms_done,
                       cuda_stream, nt);
}

extern "C" int gnssb200_set_softtrack_width(gnssb200_handle *h, int threads) {
  if (!h || (threads != 0 && threads != 128 && threads != 256 && threads != 512)) {
    gnssb200_set_error(-25, "gnssb200_set_softtrack_width: threads must be 0, 128, 256 or 512", __FILE__, __LINE__);
    return -25;
  }
  h->softtrack_width = threads;
  return 0;
}
