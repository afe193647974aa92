// acq.cu -- FFT parallel-code-phase acquisition on the device.
//
// Replaces acqResults = acquisition(longSignal, settings) of the Scilab receivers
// (SCI/GLONASS/L1/acquisition.sci:49-191, SCI/GPS/L1/acquisition.sci; SCI = trunk/
// GNSS_SOFTWARE_RECEIVERS/POSTPROCESSING_SCILAB_RECEIVERS) for the search grid
// (PRN or frequency channel) x Doppler bin x code phase.
//
// Formulation (exact identities, SURVEY.md 7.3):
//  * the code replica is periodic with N = 16000 samples and only lags 1..N are kept
//    (acquisition.sci:72,131,134), so  ifft(fft(carrier.*signal).*conj(fft(code_rep)))[tau]  equals the
//    N-point circular correlation of the sample-wise SUM of the Tcoh wiped-off 1-ms segments with one
//    code period: one 16000-point FFT pair instead of a Tcoh*16000-point pair;
//  * bins whose frequencies differ by a multiple of fs/N = 1 kHz differ only by a circular shift of
//    that folded spectrum, so the forward transforms are done once per (frequency class, block)
//    ("base spectra") and every (sv, bin) row costs one multiply + one inverse FFT per block.
//
// Kernels (all use fft16k::ifft, 400 threads, one CTA per SM, transform resident in shared memory):
//  acq_code_kernel  C[code][k]      = conj(fft(code))           = unnormalised inverse DFT of the real code
//  acq_base_kernel  X[r][cls][b][k] = fft(sum_m s_r[n+mN] e^{i theta})  (wipe-off + fold + unpack fused in the loads)
//  acq_rows_kernel  per (record, sv, bin): y = ifft(X_r[(k-shift) mod N] * C[k]); |y|^2/N^2; block choice or
//                   non-coherent sum in registers; max / first argmax / second peak at circular distance >= 1 chip.
// A call searches R records with the same settings (gnssb200_acq_search_batch; the single-record entry point is R = 1):
// the row descriptors, class increments and code spectra do not depend on the record, only the X base and the output
// table do.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "common.cuh"
#include "fft16k.cuh"

using fft16k::Tables;

struct AcqRowDesc {
  int32_t out_index;  // sv_index * n_bins + bin
  int32_t code;       // code spectrum index
  int32_t cls;        // frequency class (base spectrum)
  int32_t shift;      // circular shift in bins, 0..N-1
};

struct AcqWorkspace {
  gnssb200_acq_cfg cfg;      // configuration the cached tables belong to
  bool codes_valid = false;
  int n_codes = 0, n_cls = 0, n_blocks = 0, n_rows = 0, n_bins = 0;
  int8_t *d_code_samples = nullptr;  // [n_codes][N]
  float2 *d_C = nullptr;             // [n_codes][N]
  float2 *d_X = nullptr;             // [R][n_cls][n_blocks][N]
  size_t X_cap = 0;
  float2 *d_tw16k = nullptr, *d_tw800 = nullptr;
  AcqRowDesc *d_rows = nullptr;
  size_t rows_cap = 0;
  unsigned long long *d_cls_inc = nullptr;  // [n_cls] carrier phase increment, cycles * 2^64
  size_t cls_cap = 0;
  gnssb200_acq_row *d_out_tmp = nullptr;  // for the host convenience call
  size_t out_cap = 0;
  uint8_t *d_iq_stage = nullptr;  // record staging of gnssb200_acq_pcps_host, kept between calls
  size_t iq_cap = 0;
};

// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void sample_at(const uint8_t *iq, int fmt, long long i, float &I, float &Q) {
  if (fmt == GNSSB200_FMT_INT8_IQ) {
    const char2 v = __ldg(reinterpret_cast<const char2 *>(iq) + i);
    I = (float)v.x;
    Q = (float)v.y;
  } else {  // packed 2-bit: 2 complex samples per byte, I0 Q0 I1 Q1, LSB first, {0:+1,1:-1,2:+3,3:-3}
    const uint32_t b = __ldg(iq + (i >> 1)) >> ((i & 1) * 4);
    const float val[4] = {1.f, -1.f, 3.f, -3.f};
    I = val[b & 3];
    Q = val[(b >> 2) & 3];
  }
}

__global__ void __launch_bounds__(fft16k::THREADS, 1)
acq_code_kernel(const int8_t *code_samples, float2 *C, Tables tb) {
  extern __shared__ float2 sm[];
  const int8_t *code = code_samples + (size_t)blockIdx.x * fft16k::N;
  float2 *out = C + (size_t)blockIdx.x * fft16k::N;
  fft16k::ifft(
      sm, tb, [&](int n) { return make_float2((float)code[n], 0.f); },
      [&](int tau0, float2(&v)[fft16k::R3]) {
#pragma unroll
        for (int kb = 0; kb < fft16k::R3; kb++) out[tau0 + 400 * kb] = v[kb];
      });
}

// grid = R * n_cls * n_blocks, record r at iq + r*rec_stride.  X = fft(x) = conj(ifft_unnorm(conj(x))),
// x[n] = sum_{m<T} s[blk*T*N + n + m*N] * exp(+i*2*pi*f*(n+m*N)/fs)      (acquisition.sci:62-63,111,115-116)
__global__ void __launch_bounds__(fft16k::THREADS, 1)
acq_base_kernel(const uint8_t *iq_base, size_t rec_stride, int fmt, int coh_ms, int n_cls, int n_blocks,
                const unsigned long long *cls_inc, float2 *X, Tables tb) {
  extern __shared__ float2 sm[];
  const int per_rec = n_cls * n_blocks;
  const int rec = blockIdx.x / per_rec, cb = blockIdx.x % per_rec;
  const int cls = cb / n_blocks, blk = cb % n_blocks;
  const uint8_t *iq = iq_base + (size_t)rec * rec_stride;
  const unsigned long long inc = cls_inc[cls];
  const long long base = (long long)blk * coh_ms * fft16k::N;
  float2 *out = X + (size_t)blockIdx.x * fft16k::N;
  fft16k::ifft(
      sm, tb,
      [&](int n) {
        float re = 0.f, im = 0.f;
        for (int m = 0; m < coh_ms; m++) {
          const long long i = (long long)n + (long long)m * fft16k::N;
          float I, Q;
          sample_at(iq, fmt, base + i, I, Q);
          const unsigned long long ph = (unsigned long long)i * inc;  // cycles, 64-bit fraction
          float sn, cs;
          sincospif((float)(int)(ph >> 32) * (1.0f / 2147483648.0f), &sn, &cs);
          // (I + iQ)(cs + i sn)
          re += I * cs - Q * sn;
          im += I * sn + Q * cs;
        }
        return make_float2(re, -im);  // conj(x)
      },
      [&](int tau0, float2(&v)[fft16k::R3]) {
#pragma unroll
        for (int kb = 0; kb < fft16k::R3; kb++) out[tau0 + 400 * kb] = make_float2(v[kb].x, -v[kb].y);
      });
}

// ---- CTA-wide (max value, smallest index) ------------------------------------------------------
__device__ __forceinline__ unsigned long long pack_key(float v, int idx) {
  return ((unsigned long long)__float_as_uint(v) << 32) | (unsigned)(0x7fffffff - idx);  // v >= 0
}
__device__ __forceinline__ unsigned long long block_max_key(unsigned long long key, unsigned long long *red) {
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
    key = other > key ? other : key;
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
  __syncthreads();
  if (lane == 0) red[warp] = key;
  __syncthreads();
  unsigned long long k = lane < nw ? red[lane] : 0ull;
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long other = __shfl_xor_sync(0xffffffffu, k, o);
    k = other > k ? other : k;
  }
  return k;  // same in every thread
}

struct AcqRowsArgs {
  const AcqRowDesc *rows;
  int n_rows;        // descriptors per record; work item i = record i / n_rows, descriptor i % n_rows
  int n_items;       // R * n_rows
  size_t x_rec;      // elements of X per record: n_cls * n_blocks * N
  size_t out_rec;    // rows of the output table per record: n_sv * n_bins
  const float2 *X;   // [R][cls][blocks][N]
  const float2 *C;   // [code][N]
  int n_blocks;      // 2 (stock) or K (non-coherent)
  int noncoh;        // 0: keep the block with the larger maximum; 1: sum all blocks
  int chip;          // round(fs/codeFreqBasis): 16 GPS, 31 GLONASS
  gnssb200_acq_row *out;  // [R][n_sv][n_bins]
  Tables tb;
};

// is 0-based code phase t searched for the second peak, given the peak at 0-based p?  Circular distance >= chip:
// the window of acquisition.sci:151-168 at every peak where its index ranges stay inside 1..N.  At the three peaks
// where they do not (1-based GPS 17, GLONASS 32 and 15969; Scilab stops with an error) this is an extension of the
// library: the same circular rule.
__device__ __forceinline__ bool second_peak_allowed(int t, int p, int chip) {
  const int d = abs(t - p);
  return min(d, fft16k::N - d) >= chip;
}

__global__ void __launch_bounds__(fft16k::THREADS, 1) acq_rows_kernel(const AcqRowsArgs a) {
  extern __shared__ float2 sm[];
  __shared__ unsigned long long red[16];
  const float scale = 1.0f / ((float)fft16k::N * (float)fft16k::N);  // Scilab ifft carries 1/N
  for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
    const int rec = item / a.n_rows;
    const AcqRowDesc d = a.rows[item - rec * a.n_rows];
    const float2 *C = a.C + (size_t)d.code * fft16k::N;
    const float2 *Xr = a.X + (size_t)rec * a.x_rec;
    float acc[fft16k::R3];
#pragma unroll
    for (int kb = 0; kb < fft16k::R3; kb++) acc[kb] = 0.f;
    float best_peak = -1.f, best_second = 0.f;
    int best_arg = 0, best_blk = 0;
    int my_tau0 = 0;
    for (int blk = 0; blk < a.n_blocks; blk++) {
      const float2 *X = Xr + ((size_t)d.cls * a.n_blocks + blk) * fft16k::N;
      float mag[fft16k::R3];
      fft16k::ifft(
          sm, a.tb,
          [&](int k) {
            int src = k - d.shift;
            src += (src < 0) ? fft16k::N : 0;
            return fft16k::cmul(__ldg(X + src), __ldg(C + k));
          },
          [&](int tau0, float2(&v)[fft16k::R3]) {
            my_tau0 = tau0;
#pragma unroll
            for (int kb = 0; kb < fft16k::R3; kb++) mag[kb] = (v[kb].x * v[kb].x + v[kb].y * v[kb].y) * scale;
          });
      if (a.noncoh) {
#pragma unroll
        for (int kb = 0; kb < fft16k::R3; kb++) acc[kb] += mag[kb];
        if (blk + 1 < a.n_blocks) continue;
#pragma unroll
        for (int kb = 0; kb < fft16k::R3; kb++) mag[kb] = acc[kb];
      }
      // max / first argmax over the 16000 code phases
      unsigned long long key = 0;
#pragma unroll
      for (int kb = 0; kb < fft16k::R3; kb++) {
        const unsigned long long k2 = pack_key(mag[kb], my_tau0 + 400 * kb);
        key = k2 > key ? k2 : key;
      }
      key = block_max_key(key, red);
      const float peak = __uint_as_float((unsigned)(key >> 32));
      const int arg = 0x7fffffff - (int)(unsigned)(key & 0xffffffffu);
      // second peak at circular distance >= 1 chip from this row's own peak
      unsigned long long key2 = 0;
#pragma unroll
      for (int kb = 0; kb < fft16k::R3; kb++) {
        const int t = my_tau0 + 400 * kb;
        if (second_peak_allowed(t, arg, a.chip)) {
          const unsigned long long k2 = pack_key(mag[kb], t);
          key2 = k2 > key2 ? k2 : key2;
        }
      }
      key2 = block_max_key(key2, red);
      const float second = __uint_as_float((unsigned)(key2 >> 32));
      // stock rule: block 1 only if max(block1) > max(block2), strictly (acquisition.sci:130)
      if (blk == 0 || a.noncoh || !(best_peak > peak)) {
        best_peak = peak;
        best_second = second;
        best_arg = arg;
        best_blk = a.noncoh ? 0 : blk;
      }
    }
    if (threadIdx.x == 0) {
      gnssb200_acq_row r;
      r.peak = best_peak;
      r.code_phase = best_arg;
      r.second = best_second;
      r.block = best_blk;
      a.out[(size_t)rec * a.out_rec + d.out_index] = r;
    }
  }
}

__global__ void acq_fill_rows_kernel(gnssb200_acq_row *rows, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    gnssb200_acq_row r;
    r.peak = -1.f;
    r.code_phase = 0;
    r.second = 0.f;
    r.block = 0;
    rows[i] = r;
  }
}

// ---------------------------------------------------------------------------------------------
// host side
static int scilab_round(double x) { return (int)(x < 0 ? -floor(-x + 0.5) : floor(x + 0.5)); }

extern "C" int gnssb200_acq_num_bins(const gnssb200_acq_cfg *c) {
  return scilab_round(c->search_band_khz * 2 * c->coh_ms) + 1;  // acquisition.sci:66-67
}
static int acq_blocks(const gnssb200_acq_cfg *c) { return c->n_noncoh <= 1 ? 2 : c->n_noncoh; }
extern "C" int64_t gnssb200_acq_samples_needed(const gnssb200_acq_cfg *c) {
  const int n = scilab_round(c->samp_freq / (c->code_freq / c->code_length));
  return (int64_t)acq_blocks(c) * c->coh_ms * n;
}
static double acq_bin_freq(const gnssb200_acq_cfg *c, int sv, int k1) {  // frqBins(k1), :105-108
  const double base = c->IF + (c->system == GNSSB200_SYS_GLONASS ? sv * c->IF_step : 0.0);
  return base - (c->search_band_khz / 2) * 1000 + (1000.0 / (2 * c->coh_ms)) * (k1 - 1);
}

// C/A chips (+-1) for PRN, from the correlator table (early[2c] = chip c); ST code for GLONASS
static void code_chips(int system, int sv, std::vector<int8_t> &chips) {
  if (system == GNSSB200_SYS_GPS) {
    std::vector<uint32_t> table(TABLE_ENTRIES + 1);
    build_code_table_host(table.data());
    chips.resize(1023);
    for (int c = 0; c < 1023; c++) chips[c] = (int8_t)(table[sv * HALF_CHIPS + 2 * c] & 0xff);
  } else {  // generateSTcode.sci:35-42
    chips.resize(511);
    int reg[9];
    for (int i = 0; i < 9; i++) reg[i] = 1;
    for (int c = 0; c < 511; c++) {
      chips[c] = (int8_t)(2 * reg[6] - 1);
      const int fb = reg[4] ^ reg[8];
      for (int i = 8; i > 0; i--) reg[i] = reg[i - 1];
      reg[0] = fb;
    }
  }
}

void acq_free_workspace(gnssb200_handle *h) {
  AcqWorkspace *w = (AcqWorkspace *)h->acq_ws;
  if (!w) return;
  cudaFree(w->d_code_samples);
  cudaFree(w->d_C);
  cudaFree(w->d_X);
  cudaFree(w->d_tw16k);
  cudaFree(w->d_tw800);
  cudaFree(w->d_rows);
  cudaFree(w->d_cls_inc);
  cudaFree(w->d_out_tmp);
  cudaFree(w->d_iq_stage);
  delete w;
  h->acq_ws = nullptr;
}

static bool same_code_setup(const gnssb200_acq_cfg &a, const gnssb200_acq_cfg &b) {
  if (a.system != b.system || a.samp_freq != b.samp_freq || a.code_freq != b.code_freq || a.code_length != b.code_length ||
      a.n_sv != b.n_sv)
    return false;
  return a.system == GNSSB200_SYS_GLONASS || memcmp(a.sv, b.sv, sizeof(int32_t) * a.n_sv) == 0;
}

// cudaMalloc into a workspace slot; the slot is empty (nullptr, capacity 0) unless the allocation succeeded
template <typename T>
static cudaError_t ws_reserve(T *&p, size_t &cap, size_t n) {
  if (n <= cap) return cudaSuccess;
  cudaFree(p);
  p = nullptr;
  cap = 0;
  const cudaError_t e = cudaMalloc(&p, n * sizeof(T));
  if (e != cudaSuccess) {
    p = nullptr;
    return e;
  }
  cap = n;
  return cudaSuccess;
}

extern "C" int gnssb200_acq_search_batch(gnssb200_handle *h, const gnssb200_acq_cfg *cfg, const void *d_iq, size_t record_stride_bytes,
                                         int n_records, int fmt, int64_t n_samples, gnssb200_acq_row *d_rows_out, void *cuda_stream) {
  if (!h || !cfg || !d_iq || !d_rows_out) {
    gnssb200_set_error(-10, "gnssb200_acq_search: null argument", __FILE__, __LINE__);
    return -10;
  }
  const int N = scilab_round(cfg->samp_freq / (cfg->code_freq / cfg->code_length));
  if (N != fft16k::N) {
    gnssb200_set_error(-11, "gnssb200_acq_search: samples per code must be 16000 (fs 16 MHz, 1 ms codes)", __FILE__, __LINE__);
    return -11;
  }
  if (fmt != GNSSB200_FMT_INT8_IQ && fmt != GNSSB200_FMT_PACKED2) {
    gnssb200_set_error(-12, "gnssb200_acq_search: format must be INT8_IQ or PACKED2", __FILE__, __LINE__);
    return -12;
  }
  if (cfg->n_sv <= 0 || cfg->n_sv > 64 || cfg->coh_ms <= 0 || n_samples < gnssb200_acq_samples_needed(cfg)) {
    gnssb200_set_error(-13, "gnssb200_acq_search: bad sv list / coherent time / record too short", __FILE__, __LINE__);
    return -13;
  }
  const size_t rec_bytes = fmt == GNSSB200_FMT_INT8_IQ ? (size_t)n_samples * 2 : ((size_t)n_samples + 1) / 2;
  if (n_records < 1 || (record_stride_bytes != 0 && record_stride_bytes < rec_bytes)) {
    gnssb200_set_error(-15, "gnssb200_acq_search_batch: n_records < 1, or a record stride shorter than n_samples in fmt",
                       __FILE__, __LINE__);
    return -15;
  }
  // sample_at reads an int8 I,Q sample as one 2-byte char2 load: the records must start on even addresses
  if (fmt == GNSSB200_FMT_INT8_IQ && (((uintptr_t)d_iq | record_stride_bytes) & 1)) {
    gnssb200_set_error(-15, "gnssb200_acq_search_batch: int8 I,Q records need an even d_iq and an even record stride",
                       __FILE__, __LINE__);
    return -15;
  }
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  if (!h->acq_ws) h->acq_ws = new AcqWorkspace();
  AcqWorkspace &w = *(AcqWorkspace *)h->acq_ws;
  const int n_bins = gnssb200_acq_num_bins(cfg);
  const int K = acq_blocks(cfg);
  const size_t smem = fft16k::SMEM_BYTES;
  // the opt-in is an attribute of the kernel on the current device: set it per call (a handle may live on any device)
  CUDA_TRY(cudaFuncSetAttribute(acq_code_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  CUDA_TRY(cudaFuncSetAttribute(acq_base_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  CUDA_TRY(cudaFuncSetAttribute(acq_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // ---- twiddle tables (once) ----
  if (!w.d_tw16k) {
    std::vector<float2> t1(fft16k::M), t2(fft16k::R3);
    for (int n = 0; n < fft16k::M; n++) {
      const double ang = 2.0 * M_PI * n / fft16k::N;
      t1[n] = make_float2((float)cos(ang), (float)sin(ang));
    }
    for (int b = 0; b < fft16k::R3; b++) {
      const double ang = 2.0 * M_PI * b / fft16k::M;
      t2[b] = make_float2((float)cos(ang), (float)sin(ang));
    }
    size_t c1 = 0, c2 = 0;
    cudaError_t e = ws_reserve(w.d_tw16k, c1, t1.size());
    if (e == cudaSuccess) e = ws_reserve(w.d_tw800, c2, t2.size());
    if (e == cudaSuccess) e = cudaMemcpyAsync(w.d_tw16k, t1.data(), t1.size() * sizeof(float2), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(w.d_tw800, t2.data(), t2.size() * sizeof(float2), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);  // pageable host vectors
    if (e != cudaSuccess) {
      cudaFree(w.d_tw16k);
      cudaFree(w.d_tw800);
      w.d_tw16k = w.d_tw800 = nullptr;
      CUDA_TRY(e);
    }
  }
  const Tables tb{w.d_tw16k, w.d_tw800};
  // ---- code spectra (cached per code setup) ----
  if (!w.codes_valid || !same_code_setup(w.cfg, *cfg)) {
    const int n_codes = cfg->system == GNSSB200_SYS_GLONASS ? 1 : cfg->n_sv;
    std::vector<int8_t> samples((size_t)n_codes * N);
    const double ts = 1.0 / cfg->samp_freq, tc = 1.0 / cfg->code_freq;
    for (int c = 0; c < n_codes; c++) {
      std::vector<int8_t> chips;
      const int sv = cfg->sv[c];
      if (cfg->system == GNSSB200_SYS_GPS && (sv < 1 || sv > 32)) {
        gnssb200_set_error(-14, "gnssb200_acq_search: GPS PRN must be 1..32", __FILE__, __LINE__);
        return -14;
      }
      code_chips(cfg->system, sv, chips);
      for (int i = 1; i <= N; i++) {  // makeCaTable.sci:62-66 / makeStTable.sci:60-63
        int idx = (int)ceil((ts * i) / tc);
        if (i == N) idx = cfg->code_length;
        samples[(size_t)c * N + i - 1] = chips[idx - 1];
      }
    }
    w.codes_valid = false;
    size_t c1 = 0, c2 = 0;  // exact sizes: the spectra are rebuilt whenever the code setup changes
    CUDA_TRY(ws_reserve(w.d_code_samples, c1, samples.size()));
    CUDA_TRY(ws_reserve(w.d_C, c2, samples.size()));
    CUDA_TRY(cudaMemcpyAsync(w.d_code_samples, samples.data(), samples.size(), cudaMemcpyHostToDevice, st));
    acq_code_kernel<<<n_codes, fft16k::THREADS, smem, st>>>(w.d_code_samples, w.d_C, tb);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(st));  // `samples` goes out of scope
    h->launches++;
    w.n_codes = n_codes;
    w.codes_valid = true;
  }
  w.cfg = *cfg;
  // ---- frequency classes and row descriptors ----
  std::vector<double> cls_f0;       // lowest frequency seen in each class
  std::vector<double> cls_frac;     // f mod 1000
  std::vector<AcqRowDesc> rows;
  const int part_count = cfg->part_count > 0 ? cfg->part_count : 1;
  const int part_index = cfg->part_count > 0 ? cfg->part_index : 0;
  const double bin_hz = cfg->samp_freq / N;  // 1000 Hz
  for (int s = 0; s < cfg->n_sv; s++) {
    for (int b = 0; b < n_bins; b++) {
      const double f = acq_bin_freq(cfg, cfg->sv[s], b + 1);
      double frac = fmod(f, bin_hz);
      if (frac < 0) frac += bin_hz;
      int cls = -1;
      for (size_t c = 0; c < cls_frac.size(); c++) {
        double dd = fabs(cls_frac[c] - frac);
        dd = std::min(dd, bin_hz - dd);
        if (dd < 1e-6) {
          cls = (int)c;
          break;
        }
      }
      if (cls < 0) {
        cls = (int)cls_frac.size();
        cls_frac.push_back(frac);
        cls_f0.push_back(f);
      }
      const long long j = llround((f - cls_f0[cls]) / bin_hz);
      const int r = s * n_bins + b;
      if (r % part_count != part_index) continue;
      AcqRowDesc d;
      d.out_index = r;
      d.code = cfg->system == GNSSB200_SYS_GLONASS ? 0 : s;
      d.cls = cls;
      d.shift = (int)(((j % N) + N) % N);
      rows.push_back(d);
    }
  }
  const int n_cls = (int)cls_f0.size();
  std::vector<unsigned long long> inc(n_cls);
  for (int c = 0; c < n_cls; c++) {
    double x = cls_f0[c] / cfg->samp_freq;  // cycles per sample
    x -= floor(x);
    inc[c] = (unsigned long long)(x * 18446744073709551616.0);
  }
  const int R = n_records;
  const size_t x_rec = (size_t)n_cls * K * N;
  // the workspace X holds the base spectra of every record of the call: R * n_cls * K * 128 KB
  CUDA_TRY(ws_reserve(w.d_cls_inc, w.cls_cap, (size_t)n_cls));
  CUDA_TRY(ws_reserve(w.d_X, w.X_cap, x_rec * R));
  CUDA_TRY(ws_reserve(w.d_rows, w.rows_cap, rows.size()));
  CUDA_TRY(cudaMemcpyAsync(w.d_cls_inc, inc.data(), sizeof(unsigned long long) * n_cls, cudaMemcpyHostToDevice, st));
  if (!rows.empty())
    CUDA_TRY(cudaMemcpyAsync(w.d_rows, rows.data(), sizeof(AcqRowDesc) * rows.size(), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaStreamSynchronize(st));  // pageable host vectors
  w.n_cls = n_cls;
  w.n_blocks = K;
  w.n_rows = (int)rows.size();
  w.n_bins = n_bins;

  CUDA_TRY(cudaEventRecord(h->ev0, st));
  const size_t out_rec = (size_t)cfg->n_sv * n_bins;
  const int total_rows = (int)(out_rec * R);
  acq_fill_rows_kernel<<<(total_rows + 255) / 256, 256, 0, st>>>(d_rows_out, total_rows);
  acq_base_kernel<<<R * n_cls * K, fft16k::THREADS, smem, st>>>((const uint8_t *)d_iq, record_stride_bytes, fmt, cfg->coh_ms, n_cls,
                                                                 K, w.d_cls_inc, w.d_X, tb);
  CUDA_TRY(cudaGetLastError());
  h->launches += 2;
  if (!rows.empty()) {
    AcqRowsArgs a;
    a.rows = w.d_rows;
    a.n_rows = (int)rows.size();
    a.n_items = a.n_rows * R;
    a.x_rec = x_rec;
    a.out_rec = out_rec;
    a.X = w.d_X;
    a.C = w.d_C;
    a.n_blocks = K;
    a.noncoh = cfg->n_noncoh >= 2 ? 1 : 0;
    a.chip = scilab_round(cfg->samp_freq / cfg->code_freq);
    a.out = d_rows_out;
    a.tb = tb;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
    const int grid = std::min(a.n_items, sms);
    acq_rows_kernel<<<grid, fft16k::THREADS, smem, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
  }
  CUDA_TRY(cudaEventRecord(h->ev1, st));
  return 0;
}

extern "C" int gnssb200_acq_search(gnssb200_handle *h, const gnssb200_acq_cfg *cfg, const void *d_iq, int fmt, int64_t n_samples,
                                   gnssb200_acq_row *d_rows_out, void *cuda_stream) {
  return gnssb200_acq_search_batch(h, cfg, d_iq, 0, 1, fmt, n_samples, d_rows_out, cuda_stream);
}

// acquisition.sci:145-191 on the complete (sv x bin) row table
extern "C" int gnssb200_acq_finalize(const gnssb200_acq_cfg *cfg, const gnssb200_acq_row *rows, gnssb200_acq_result *res) {
  const int n_bins = gnssb200_acq_num_bins(cfg);
  int ambiguous = 0;
  for (int s = 0; s < cfg->n_sv; s++) {
    const gnssb200_acq_row *r = rows + (size_t)s * n_bins;
    float peak = -1.f;
    for (int b = 0; b < n_bins; b++) peak = r[b].peak > peak ? r[b].peak : peak;
    int bin = 0;
    while (bin < n_bins && r[bin].peak != peak) bin++;  // first row attaining the maximum
    int code_phase = fft16k::N;                          // first column attaining it, over all rows
    for (int b = 0; b < n_bins; b++)
      if (r[b].peak == peak && r[b].code_phase < code_phase) code_phase = r[b].code_phase;
    if (code_phase != r[bin].code_phase) ambiguous++;    // exact float tie across rows (never seen on noise)
    gnssb200_acq_result &o = res[s];
    o.peak = peak;
    o.second = r[bin].second;
    o.peakMetric = (double)peak / (double)r[bin].second;
    o.bin = bin + 1;
    o.codePhaseRaw = code_phase + 1;
    o.carrFreq = 0.0;
    o.codePhase = 0;
    o.sv = 0;
    if (o.peakMetric > cfg->threshold) {
      o.codePhase = code_phase + 1;
      o.carrFreq = acq_bin_freq(cfg, cfg->sv[s], bin + 1);
      o.sv = cfg->sv[s];
    }
  }
  return ambiguous;
}

extern "C" int gnssb200_acq_pcps_host(gnssb200_handle *h, const gnssb200_acq_cfg *cfg, const void *h_iq, int fmt, int64_t n_samples,
                                      gnssb200_acq_result *results, gnssb200_acq_row *h_rows_opt) {
  if (!h || !cfg) return -10;
  CUDA_TRY(cudaSetDevice(h->device));
  const size_t bytes = fmt == GNSSB200_FMT_INT8_IQ ? (size_t)n_samples * 2 : (size_t)n_samples / 2;
  if (!h->acq_ws) h->acq_ws = new AcqWorkspace();
  AcqWorkspace &w = *(AcqWorkspace *)h->acq_ws;
  const int total = cfg->n_sv * gnssb200_acq_num_bins(cfg);
  if (total <= 0 || n_samples <= 0 || !h_iq) return -10;
  // staging buffers live in the handle: no allocation (and no implicit device synchronisation of a free) per call
  if (bytes + 16 > w.iq_cap) {
    cudaFree(w.d_iq_stage);
    w.d_iq_stage = nullptr;
    w.iq_cap = 0;
    CUDA_TRY(cudaMalloc(&w.d_iq_stage, bytes + 16));
    w.iq_cap = bytes + 16;
  }
  if (sizeof(gnssb200_acq_row) * (size_t)total > w.out_cap) {
    cudaFree(w.d_out_tmp);
    w.d_out_tmp = nullptr;
    w.out_cap = 0;
    CUDA_TRY(cudaMalloc(&w.d_out_tmp, sizeof(gnssb200_acq_row) * (size_t)total));
    w.out_cap = sizeof(gnssb200_acq_row) * (size_t)total;
  }
  uint8_t *d_iq = w.d_iq_stage;
  gnssb200_acq_row *d_rows = w.d_out_tmp;
  CUDA_TRY(cudaMemcpy(d_iq, h_iq, bytes, cudaMemcpyHostToDevice));
  int rc = gnssb200_acq_search(h, cfg, d_iq, fmt, n_samples, d_rows, nullptr);
  std::vector<gnssb200_acq_row> rows(total);
  if (!rc) {
    cudaError_t e = cudaMemcpy(rows.data(), d_rows, sizeof(gnssb200_acq_row) * total, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) {
      gnssb200_set_error((int)e, cudaGetErrorString(e), __FILE__, __LINE__);
      rc = (int)e;
    }
  }
  if (rc) return rc;
  if (h_rows_opt) memcpy(h_rows_opt, rows.data(), sizeof(gnssb200_acq_row) * total);
  gnssb200_acq_finalize(cfg, rows.data(), results);
  return 0;
}
