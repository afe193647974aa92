// api.cu -- C ABI of libgnssb200.so (include/gnssb200.h): handle management, host-side register
// helpers, the batched tracking entry points and the drop-in correlator symbols of the reference
// (OSG/correlator/correlator.h:4,8,9).
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <vector>

#include "common.cuh"

// ---------------------------------------------------------------------------------------------
static thread_local int g_err_code = 0;
static thread_local char g_err_text[512] = "";

void gnssb200_set_error(int code, const char *what, const char *file, int line) {
  g_err_code = code;
  snprintf(g_err_text, sizeof g_err_text, "%s (%s:%d)", what, file, line);
}
extern "C" int gnssb200_last_error(void) { return g_err_code; }
extern "C" const char *gnssb200_last_error_string(void) { return g_err_text; }

// ---------------------------------------------------------------------------------------------
// configuration: OSG/include/globals.h defaults; correlator_init (correlator.c:107-125);
// init_tracking_loops_parameter (osgnss_next_step.c:99-107 -> osgpsisr.c:252-342)
extern "C" void gnssb200_cfg_default(gnssb200_cfg *c) {
  memset(c, 0, sizeof *c);
  c->samp_rate = 16.0e6;
  c->clock_mult = 5.0;
  c->gps_carrier_if = 2.42e6;
  c->gps_code_f = 1023000.0;
  c->freq_bin_width = 1000.0;
  c->tic_period = 0.0;
  c->carrier_nco_bits = 30;
  c->code_nco_bits = 29;
  c->acq_thresh = 1800;
  c->interr_int_us = 512;
  c->Bnp = 25;
  c->Bnf = 1400;
  c->Bnd = 2;
  c->pll_integ_ms = 1;
  c->dll_integ_ms = 1;
  c->glonass_carrier_if = 0.0;
  c->glonass_code_f = 511000.0;
}

extern "C" void gnssb200_cfg_derive(gnssb200_cfg *c) {
  const double carr_res = c->clock_mult * c->samp_rate / pow(2.0, (double)c->carrier_nco_bits);
  const double code_res = c->clock_mult * c->samp_rate / pow(2.0, (double)c->code_nco_bits);
  c->gps_code_ref = (int64_t)(c->gps_code_f / code_res);
  c->gps_carrier_ref = (int64_t)(c->gps_carrier_if / carr_res);
  c->glonass_code_ref = (int64_t)(c->glonass_code_f / code_res);        // correlator.c:117
  c->glonass_carrier_ref = (int64_t)(c->glonass_carrier_if / carr_res);  // correlator.c:118
  c->d_freq = (int64_t)((double)(int)c->freq_bin_width / carr_res);
  c->tic_ref = (int64_t)(c->samp_rate * c->tic_period);
  const double a2 = 1.414;
  {
    const double wp = (double)c->Bnp / 0.53, wf = (double)c->Bnf / 0.25, T = (double)c->pll_integ_ms / 1000;
    const double scale = (double)(1 << c->carrier_nco_bits) / (c->samp_rate * c->clock_mult);
    c->pll_i1 = (int32_t)((T * (wp * wp) + a2 * wp) * scale);
    c->pll_i2 = (int32_t)((a2 * wp) * scale);
    c->pll_i3 = (int32_t)((T * wf) * scale);
  }
  {
    const double w = (double)c->Bnd / 0.53, T = (double)c->dll_integ_ms / 1000;
    const double scale = (double)(1 << c->code_nco_bits) / (c->samp_rate * c->clock_mult);
    c->dll_i1 = (int32_t)((T * (w * w) + a2 * w) * scale);
    c->dll_i2 = (int32_t)((a2 * w) * scale);
  }
}

// register accessors on a host-side gnssb200_rx (OSG/gp2021/gp2021.c:11-14,74-130)
static inline void host_put16(gnssb200_rx *rx, int addr, int data) { rx->reg_write[addr & 0xff] = (int)(uint16_t)data; }
extern "C" void gnssb200_ch_cntl(gnssb200_rx *rx, int ch, int data) { host_put16(rx, ch << 3, data); }
extern "C" void gnssb200_ch_code_slew(gnssb200_rx *rx, int ch, int data) { host_put16(rx, (ch << 3) + 0x84, data); }
extern "C" void gnssb200_ch_epoch_load(gnssb200_rx *rx, int ch, unsigned data) { host_put16(rx, (ch << 3) + 7, (int)data); }
static void host_put_nco(gnssb200_rx *rx, int addr, int64_t freq, int bits, double mult) {
  int64_t w = freq << (32 - bits);
  w = (int64_t)((double)w * mult);
  host_put16(rx, addr, (int)(w >> 16));
  host_put16(rx, addr + 1, (int)(w & 0xffff));
}
extern "C" void gnssb200_ch_carrier(gnssb200_rx *rx, const gnssb200_cfg *c, int ch, int64_t freq) {
  host_put_nco(rx, (ch << 3) + 3, freq, c->carrier_nco_bits, c->clock_mult);
}
extern "C" void gnssb200_ch_code(gnssb200_rx *rx, const gnssb200_cfg *c, int ch, int64_t freq) {
  host_put_nco(rx, (ch << 3) + 5, freq, c->code_nco_bits, c->clock_mult);
}
extern "C" void gnssb200_rx_init(gnssb200_rx *rx, const gnssb200_cfg *c) {
  memset(rx, 0, sizeof *rx);
  rx->tic = c->tic_ref;
}
extern "C" void gnssb200_rx_cold_allocate(gnssb200_rx *rx, const gnssb200_cfg *c, const int32_t prn[GNSSB200_N_CHANNELS]) {
  for (int ch = 0; ch < NCH; ch++) {
    gnssb200_chan *k = &rx->chan[ch];
    gnssb200_ch_cntl(rx, ch, 0);
    gnssb200_ch_carrier(rx, c, ch, c->gps_carrier_ref);
    gnssb200_ch_code(rx, c, ch, c->gps_code_ref);
    k->state = 1;
    k->carrier_cold_corr = 0;
    k->del_freq = 1;
    k->n_freq = 0;
    k->search_max_PRN_delay = 2045;
    k->search_max_f = 5;
    k->ms_set = 0;
  }
  for (int ch = 0; ch < NCH; ch++) {
    if (prn[ch] <= 0) continue;
    gnssb200_ch_cntl(rx, ch, prn[ch]);
    if (prn[ch] == GNSSB200_PRN_GLONASS) {  // the hooks of the reference put to use (gnssb200.h)
      gnssb200_chan *k = &rx->chan[ch];
      k->system = 1;
      k->search_max_PRN_delay = 1021;  // osgnss_next_step.c:54
      gnssb200_ch_carrier(rx, c, ch, c->glonass_carrier_ref);
      gnssb200_ch_code(rx, c, ch, c->glonass_code_ref);
    }
  }
}

// FFT acquisition results -> channels (definition in gnssb200.h; not in the reference)
extern "C" int gnssb200_rx_acq_allocate(gnssb200_rx *rx, const gnssb200_cfg *c, const gnssb200_acq_cfg *acq,
                                        const gnssb200_acq_result *res, int32_t ch_sv_out[GNSSB200_N_CHANNELS]) {
  const char *bad = nullptr;
  const bool glo = acq && acq->system == GNSSB200_SYS_GLONASS;
  if (!rx || !c || !acq || !res || acq->n_sv < 1 || acq->n_sv > 64 || (acq->system != GNSSB200_SYS_GPS && !glo))
    bad = "gnssb200_rx_acq_allocate: bad arguments";
  else if (acq->samp_freq != c->samp_rate)
    bad = "gnssb200_rx_acq_allocate: acquisition and receiver sampling rates differ";
  else if (acq->IF != (glo ? c->glonass_carrier_if : c->gps_carrier_if))
    bad = "gnssb200_rx_acq_allocate: acquisition and receiver IF differ";
  else if (acq->code_freq != (glo ? c->glonass_code_f : c->gps_code_f))
    bad = "gnssb200_rx_acq_allocate: acquisition and receiver code rates differ";
  else if (glo && acq->IF_step != 562500.0)
    bad = "gnssb200_rx_acq_allocate: GLONASS IF step must be 562.5 kHz";
  for (int i = 0; !bad && !glo && i < acq->n_sv; i++)
    if (acq->sv[i] < 1 || acq->sv[i] > 32) bad = "gnssb200_rx_acq_allocate: GPS PRN must be 1..32";
  if (bad) {
    gnssb200_set_error(-20, bad, __FILE__, __LINE__);
    return -20;
  }
  std::vector<int> order;  // detected entries, strongest first, ties in list order
  for (int i = 0; i < acq->n_sv; i++)
    if (res[i].peakMetric > acq->threshold) order.push_back(i);
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return res[a].peakMetric > res[b].peakMetric; });
  const int n = order.size() < NCH ? (int)order.size() : NCH;
  int32_t prn[NCH];
  for (int ch = 0; ch < NCH; ch++) {
    prn[ch] = ch < n ? (glo ? GNSSB200_PRN_GLONASS : acq->sv[order[ch]]) : 0;
    if (ch_sv_out) ch_sv_out[ch] = ch < n ? acq->sv[order[ch]] : 0;
  }
  gnssb200_rx_cold_allocate(rx, c, prn);
  const double res_hz = c->clock_mult * c->samp_rate / pow(2.0, (double)c->carrier_nco_bits);
  const int P = glo ? GLO_HALF_CHIPS : HALF_CHIPS;
  for (int ch = 0; ch < n; ch++) {
    const gnssb200_acq_result &r = res[order[ch]];
    const int fch = glo ? acq->sv[order[ch]] : 0;
    gnssb200_chan *k = &rx->chan[ch];
    // carrier: the acquired frequency in NCO units
    if (glo) k->carrier_cold_corr = (int64_t)fch * (int64_t)(562500.0 / res_hz);
    const int64_t ref = (glo ? c->glonass_carrier_ref : c->gps_carrier_ref) + k->carrier_cold_corr;
    k->carrier_freq = ref + llround((r.carrFreq - acq->IF - fch * acq->IF_step) / res_hz);
    long long nf = llround((double)(k->carrier_freq - ref) / (double)c->d_freq);
    nf = nf > k->search_max_f ? k->search_max_f : (nf < -k->search_max_f ? -k->search_max_f : nf);
    k->n_freq = (int32_t)nf;
    k->del_freq = nf > 0 ? (int32_t)(-2 * nf) : (int32_t)(1 - 2 * nf);
    gnssb200_ch_carrier(rx, c, ch, k->carrier_freq);
    // code: the prompt replica (one half chip ahead of early) meets chip 0 at delay a = cell + 1; start two cells before
    const long long cell = llround((double)(r.codePhase - 1) * 2.0 * acq->code_freq / acq->samp_freq) % P;
    const int a = (int)((cell + 1) % P);
    const int k0 = a >= 2 ? a - 2 : 0;
    gnssb200_ch_code_slew(rx, ch, k0);
    k->codes = 0;  // a whole sweep of the bin at the acquired frequency before the search moves on
  }
  return n;
}

// ---------------------------------------------------------------------------------------------
extern "C" gnssb200_handle *gnssb200_open(int device, const gnssb200_cfg *cfg) {
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    gnssb200_set_error(e != cudaSuccess ? (int)e : -1, "no CUDA device (libgnssb200 has no CPU path)", __FILE__, __LINE__);
    return nullptr;
  }
  if ((e = cudaSetDevice(device)) != cudaSuccess) {
    gnssb200_set_error((int)e, cudaGetErrorString(e), __FILE__, __LINE__);
    return nullptr;
  }
  gnssb200_handle *h = new gnssb200_handle();
  memset(h, 0, sizeof *h);
  h->device = device;
  if (cfg)
    h->cfg = *cfg;
  else {
    gnssb200_cfg_default(&h->cfg);
    gnssb200_cfg_derive(&h->cfg);
  }
  std::vector<uint32_t> table(TABLE_ENTRIES + 1);
  build_code_table_host(table.data());
  if ((e = cudaMalloc(&h->d_code_table, table.size() * 4)) != cudaSuccess ||
      (e = cudaMemcpy(h->d_code_table, table.data(), table.size() * 4, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaEventCreate(&h->ev0)) != cudaSuccess || (e = cudaEventCreate(&h->ev1)) != cudaSuccess) {
    gnssb200_set_error((int)e, cudaGetErrorString(e), __FILE__, __LINE__);
    cudaFree(h->d_code_table);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    delete h;
    return nullptr;
  }
  return h;
}

extern "C" void gnssb200_close(gnssb200_handle *h) {
  if (!h) return;
  cudaSetDevice(h->device);
  acq_free_workspace(h);
  cudaFree(h->d_rx);
  cudaFree(h->d_chan_flags);
  cudaFree(h->d_sched);
  cudaFree(h->d_code_table);
  cudaFree(h->d_chips);
  for (int i = 0; i < 2; i++) {
    cudaFree(h->stage[i]);
    if (h->ev_copied[i]) cudaEventDestroy(h->ev_copied[i]);
    if (h->ev_used[i]) cudaEventDestroy(h->ev_used[i]);
  }
  cudaFree(h->stage_dumps);
  cudaFree(h->stage_cnt);
  if (h->s_copy) cudaStreamDestroy(h->s_copy);
  if (h->s_back) cudaStreamDestroy(h->s_back);
  if (h->h_snap) cudaFreeHost(h->h_snap);
  if (h->s_comp) cudaStreamDestroy(h->s_comp);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  delete h;
}

extern "C" int gnssb200_set_streams(gnssb200_handle *h, int n) {
  CUDA_TRY(cudaSetDevice(h->device));
  if (n == h->n_streams) return 0;
  cudaFree(h->d_rx);
  cudaFree(h->d_chan_flags);
  cudaFree(h->d_sched);
  h->d_rx = nullptr;
  h->d_chan_flags = nullptr;
  h->d_sched = nullptr;
  h->n_streams = 0;
  if (n > 0) {
    CUDA_TRY(cudaMalloc(&h->d_rx, sizeof(gnssb200_rx) * (size_t)n));
    CUDA_TRY(cudaMalloc(&h->d_chan_flags, sizeof(int32_t) * NCH * (size_t)n));
    CUDA_TRY(cudaMemset(h->d_rx, 0, sizeof(gnssb200_rx) * (size_t)n));
    CUDA_TRY(cudaMemset(h->d_chan_flags, 0, sizeof(int32_t) * NCH * (size_t)n));
    CUDA_TRY(cudaMalloc(&h->d_sched, track_sched_bytes(n)));
    h->n_streams = n;
  }
  return 0;
}

static int check_range(gnssb200_handle *h, int first, int count) {
  if (first < 0 || count < 0 || first + count > h->n_streams) {
    gnssb200_set_error(-2, "stream range outside gnssb200_set_streams()", __FILE__, __LINE__);
    return -2;
  }
  return 0;
}
extern "C" int gnssb200_upload_rx(gnssb200_handle *h, int first, int count, const gnssb200_rx *rx) {
  if (check_range(h, first, count)) return -2;
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaMemcpy(h->d_rx + first, rx, sizeof(gnssb200_rx) * (size_t)count, cudaMemcpyHostToDevice));
  return 0;
}
extern "C" int gnssb200_download_rx(gnssb200_handle *h, int first, int count, gnssb200_rx *rx) {
  if (check_range(h, first, count)) return -2;
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaMemcpy(rx, h->d_rx + first, sizeof(gnssb200_rx) * (size_t)count, cudaMemcpyDeviceToHost));
  return 0;
}

// Serial search as a cell map: a private handle with the detection threshold out of reach, one channel per PRN, the
// shared record read with stride 0 by every receiver, then the dump records turned into cells (the record of dump
// k carries the bin / delay the channel moved to AFTER that dump, so cell k is described by record k-1).
extern "C" int gnssb200_acq_serial(gnssb200_handle *h, const void *d_if, int fmt, int64_t n_samples, const int32_t *prn_list, int n_prn,
                                   int search_max_f, int max_prn_delay, gnssb200_serial_cell *cells, int cells_cap, int32_t *n_cells) {
  if (!h || !d_if || !prn_list || n_prn <= 0 || !cells || cells_cap <= 0 || !n_cells || n_samples < 8192) {
    gnssb200_set_error(-8, "gnssb200_acq_serial: bad arguments", __FILE__, __LINE__);
    return -8;
  }
  gnssb200_cfg cfg = h->cfg;
  cfg.acq_thresh = 0x7fffffff;
  gnssb200_handle *t = gnssb200_open(h->device, &cfg);
  if (!t) return gnssb200_last_error();
  const int S = (n_prn + NCH - 1) / NCH, nsamp = 8192;
  const long long nblocks = n_samples / nsamp;
  const int dump_cap = cells_cap + 1;
  int rc = gnssb200_set_streams(t, S);
  std::vector<gnssb200_rx> rx(S);
  for (int s = 0; s < S && !rc; s++) {
    int32_t prn[NCH];
    for (int c = 0; c < NCH; c++) prn[c] = (s * NCH + c < n_prn) ? prn_list[s * NCH + c] : 0;
    gnssb200_rx_init(&rx[s], &cfg);
    gnssb200_rx_cold_allocate(&rx[s], &cfg, prn);
    for (int c = 0; c < NCH; c++) {
      rx[s].chan[c].search_max_f = search_max_f;
      rx[s].chan[c].search_max_PRN_delay = max_prn_delay > 0 ? max_prn_delay : 2045;
    }
  }
  if (!rc) rc = gnssb200_upload_rx(t, 0, S, rx.data());
  gnssb200_dump *d_dumps = nullptr;
  int32_t *d_cnt = nullptr;
  std::vector<gnssb200_dump> dumps((size_t)S * NCH * dump_cap);
  std::vector<int32_t> cnt((size_t)S * NCH);
  cudaError_t e = cudaSuccess;
  if (!rc) e = cudaMalloc(&d_dumps, dumps.size() * sizeof(gnssb200_dump));
  if (!rc && e == cudaSuccess) e = cudaMalloc(&d_cnt, cnt.size() * sizeof(int32_t));
  if (!rc && e == cudaSuccess) e = cudaMemset(d_cnt, 0, cnt.size() * sizeof(int32_t));
  if (!rc && e == cudaSuccess) rc = gnssb200_track_run(t, d_if, 0 /* every receiver reads the same record */, fmt, nsamp, nblocks, d_dumps, dump_cap, d_cnt, nullptr);
  if (!rc && e == cudaSuccess) e = cudaMemcpy(dumps.data(), d_dumps, dumps.size() * sizeof(gnssb200_dump), cudaMemcpyDeviceToHost);
  if (!rc && e == cudaSuccess) e = cudaMemcpy(cnt.data(), d_cnt, cnt.size() * sizeof(int32_t), cudaMemcpyDeviceToHost);
  if (!rc && e == cudaSuccess) {
    h->launches += t->launches;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, t->ev0, t->ev1) == cudaSuccess) h->serial_ms = ms;
  }
  cudaFree(d_dumps);
  cudaFree(d_cnt);
  gnssb200_close(t);
  if (e != cudaSuccess) {
    gnssb200_set_error((int)e, cudaGetErrorString(e), __FILE__, __LINE__);
    return (int)e;
  }
  if (rc) return rc;
  for (int p = 0; p < n_prn; p++) {
    const gnssb200_dump *d = &dumps[(size_t)p * dump_cap];
    const int n = cnt[p] < dump_cap ? cnt[p] : dump_cap;
    int k = 0;
    for (int i = 1; i < n && k < cells_cap; i++, k++) {
      gnssb200_serial_cell &c = cells[(size_t)p * cells_cap + k];
      c.prn = (int16_t)prn_list[p];
      c.n_freq = d[i - 1].n_freq;
      c.codes = d[i - 1].codes;
      c.ip = d[i].acc[2];
      c.qp = d[i].acc[3];
      const long long a = c.ip < 0 ? -(long long)c.ip : c.ip, b = c.qp < 0 ? -(long long)c.qp : c.qp;
      c.rss = (int32_t)(a > b ? a + (b >> 1) : b + (a >> 1));  // rss(), osgpsisr.c:77-91
    }
    n_cells[p] = k;
  }
  return 0;
}

extern "C" int gnssb200_set_track_slice(gnssb200_handle *h, int64_t blocks) {
  if (!h || blocks < 0) return -1;
  h->track_slice = blocks;
  return 0;
}

extern "C" int gnssb200_set_track_variant(gnssb200_handle *h, int form, int occ) {
  if (!h || form < 0 || form > 5 || occ < 0 || occ > 8) return -1;
  h->track_form = form;
  h->track_occ = occ;
  return 0;
}

extern "C" int gnssb200_set_stage_blocks(gnssb200_handle *h, int64_t blocks) {
  if (!h || blocks < 0) return -1;
  h->stage_blocks = blocks;
  return 0;
}

extern "C" int64_t gnssb200_readback_fallbacks(const gnssb200_handle *h) { return h ? h->back_fallbacks : -1; }

extern "C" int64_t gnssb200_launch_count(const gnssb200_handle *h) { return h->launches; }

extern "C" float gnssb200_last_kernel_ms(gnssb200_handle *h) {
  float ms = -1.f;
  if (cudaEventElapsedTime(&ms, h->ev0, h->ev1) != cudaSuccess) return -1.f;
  return ms;
}

static size_t fmt_bytes(int fmt, long long nsamples) {
  return fmt == GNSSB200_FMT_INT8_IQ ? (size_t)nsamples * 2 : (fmt == GNSSB200_FMT_PACKED2 ? (size_t)nsamples / 2 : (size_t)nsamples);
}

extern "C" int gnssb200_track_run(gnssb200_handle *h, const void *d_if, size_t stride, int fmt, int nsamp, int64_t nblocks,
                                  gnssb200_dump *d_dumps, int dump_cap, int32_t *d_dump_count, void *cuda_stream) {
  if (!h || h->n_streams <= 0) {
    gnssb200_set_error(-3, "gnssb200_track_run: no streams configured", __FILE__, __LINE__);
    return -3;
  }
  if (fmt < 0 || fmt > 2 || nsamp <= 0 || (fmt == GNSSB200_FMT_PACKED2 && (nsamp & 1))) {
    gnssb200_set_error(-4, "gnssb200_track_run: bad format / block size", __FILE__, __LINE__);
    return -4;
  }
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  CUDA_TRY(cudaEventRecord(h->ev0, st));
  int rc = track_launch(h, 0, h->n_streams, d_if, stride, fmt, nsamp, nblocks, 1, d_dumps, dump_cap, d_dump_count, st);
  if (rc) return rc;
  CUDA_TRY(cudaEventRecord(h->ev1, st));
  return 0;
}

// Host-buffer variant.  The record is streamed through two device staging buffers in chunks of
// blocks: the H2D copy of chunk c+1 (copy stream) overlaps the kernels of chunk c (compute stream);
// receiver state stays on the device between chunks.  Pass pinned host memory for full PCIe speed.
// Dump records go back while the run is still in progress (third stream, the other PCIe direction): after every
// chunk the window of record indices that chunk can have written -- one record per code period, so indices
// [count before, count after) sit around first_block * nsamp / samp_rate * 1000 -- is copied for all channels at
// once (2-D copy), margins of 16 records either side.  The exact counts after every chunk come back too; the
// host checks afterwards that every chunk's records lay inside that chunk's window and otherwise repeats the
// read-back in one piece (channels resumed at very different counts, a receiver whose code period is not 1 ms).
// Host buffers that are not pinned take the one-piece path from the start (an "async" copy to pageable memory
// would block the loop that feeds the pipeline).
extern "C" int gnssb200_track_run_host(gnssb200_handle *h, const void *h_if, size_t stride, int fmt, int nsamp, int64_t nblocks,
                                       gnssb200_dump *h_dumps, int dump_cap, int32_t *h_dump_count) {
  if (!h || h->n_streams <= 0) {
    gnssb200_set_error(-3, "gnssb200_track_run_host: no streams configured", __FILE__, __LINE__);
    return -3;
  }
  if (fmt < 0 || fmt > 2 || nsamp <= 0 || (fmt == GNSSB200_FMT_PACKED2 && (nsamp & 1))) {
    gnssb200_set_error(-4, "gnssb200_track_run_host: bad format / block size", __FILE__, __LINE__);
    return -4;
  }
  CUDA_TRY(cudaSetDevice(h->device));
  const int S = h->n_streams;
  const size_t blk_bytes = fmt_bytes(fmt, nsamp);
  // Two staging buffers of about 384 blocks per stream each (>= 32 MiB, <= 512 MiB): long enough that the
  // per-launch prologue of the channel kernel (code-table row, state load / store) stays negligible, short enough
  // that the first copy and the last kernel, which overlap with nothing, stay small (64 streams x 10 s, copy bound:
  // 1.172 M channel*Msamples/s end to end with 1024 blocks, 1.197 M with 512, 1.203 M with 384).
  static long long env_blocks = -1;  // GNSSB200_STAGE_BLOCKS overrides the chunk length (blocks per stream)
  if (env_blocks < 0) {
    const char *e = getenv("GNSSB200_STAGE_BLOCKS");
    env_blocks = (e && atoll(e) > 0) ? atoll(e) : 0;
  }
  size_t stage_target = blk_bytes * (size_t)S * (size_t)(env_blocks ? env_blocks : 384);
  if (stage_target < ((size_t)32 << 20)) stage_target = (size_t)32 << 20;
  if (stage_target > ((size_t)512 << 20)) stage_target = (size_t)512 << 20;
  long long chunk = (long long)(stage_target / (blk_bytes * (size_t)S));
  if (h->stage_blocks > 0) chunk = h->stage_blocks;  // exact, for tests of the chunked pipeline
  else if (chunk < 16) chunk = 16;
  if (chunk > nblocks) chunk = nblocks;
  const size_t dstride = (blk_bytes * (size_t)chunk + 255) & ~(size_t)255;
  int rc = 0;
  auto fail = [&](cudaError_t e, int line) {
    gnssb200_set_error((int)e, cudaGetErrorString(e), __FILE__, line);
    rc = (int)e;
  };
#define TRY_(x)                         \
  do {                                  \
    cudaError_t e_ = (x);               \
    if (e_ != cudaSuccess && !rc) fail(e_, __LINE__); \
  } while (0)
  if (!h->s_copy) {
    TRY_(cudaStreamCreateWithFlags(&h->s_copy, cudaStreamNonBlocking));
    TRY_(cudaStreamCreateWithFlags(&h->s_comp, cudaStreamNonBlocking));
    TRY_(cudaStreamCreateWithFlags(&h->s_back, cudaStreamNonBlocking));
    for (int i = 0; i < 2; i++) {
      TRY_(cudaEventCreateWithFlags(&h->ev_copied[i], cudaEventDisableTiming));
      TRY_(cudaEventCreateWithFlags(&h->ev_used[i], cudaEventDisableTiming));
    }
  }
  if (!rc && dstride * S + 256 > h->stage_cap) {
    for (int i = 0; i < 2; i++) {
      cudaFree(h->stage[i]);
      h->stage[i] = nullptr;
      TRY_(cudaMalloc(&h->stage[i], dstride * S + 256));
    }
    h->stage_cap = rc ? 0 : dstride * S + 256;
  }
  const bool want = h_dumps && dump_cap > 0;
  if (want && !rc) {
    const size_t need = sizeof(gnssb200_dump) * (size_t)S * NCH * dump_cap;
    if (need > h->stage_dumps_cap) {
      cudaFree(h->stage_dumps);
      h->stage_dumps = nullptr;
      TRY_(cudaMalloc(&h->stage_dumps, need));
      h->stage_dumps_cap = rc ? 0 : need;
    }
    if (sizeof(int32_t) * S * NCH > h->stage_cnt_cap) {
      cudaFree(h->stage_cnt);
      h->stage_cnt = nullptr;
      TRY_(cudaMalloc(&h->stage_cnt, sizeof(int32_t) * S * NCH));
      h->stage_cnt_cap = rc ? 0 : sizeof(int32_t) * S * NCH;
    }
  }
  uint8_t **d_stage = h->stage;
  gnssb200_dump *d_dumps = want ? h->stage_dumps : nullptr;
  int32_t *d_cnt = want ? h->stage_cnt : nullptr;
  cudaStream_t s_copy = h->s_copy, s_comp = h->s_comp;
  cudaEvent_t *ev_copied = h->ev_copied, *ev_used = h->ev_used;
  if (want && !rc) {
    if (h_dump_count)
      TRY_(cudaMemcpyAsync(d_cnt, h_dump_count, sizeof(int32_t) * S * NCH, cudaMemcpyHostToDevice, s_comp));
    else
      TRY_(cudaMemsetAsync(d_cnt, 0, sizeof(int32_t) * S * NCH, s_comp));
  }
  // windowed read-back of the dump records: only into pinned host memory
  const long long nchunks = nblocks > 0 ? (nblocks + chunk - 1) / chunk : 0;
  const int NR = S * NCH;
  bool windows = want && !rc && nchunks > 1 && h->cfg.samp_rate > 0;
  if (windows) {
    cudaPointerAttributes pa;
    if (cudaPointerGetAttributes(&pa, h_dumps) != cudaSuccess || pa.type != cudaMemoryTypeHost) {
      cudaGetLastError();
      windows = false;
    }
  }
  if (windows && sizeof(int32_t) * NR * (size_t)nchunks > h->h_snap_cap) {
    if (h->h_snap) cudaFreeHost(h->h_snap);
    h->h_snap = nullptr;
    TRY_(cudaHostAlloc((void **)&h->h_snap, sizeof(int32_t) * NR * (size_t)nchunks, cudaHostAllocDefault));
    h->h_snap_cap = rc ? 0 : sizeof(int32_t) * NR * (size_t)nchunks;
  }
  long long cnt0_min = 0, cnt0_max = 0;  // counts the run starts from (host memory, readable now)
  std::vector<int32_t> cnt0;
  // A continued run (h_dump_count given) only appends: the records a channel already holds, [0, cnt0[i]), stay the
  // caller's.  Nothing below column cnt0_min is copied back; what the copies overwrite between cnt0_min and a
  // channel's own cnt0[i] (the staging buffer need not hold those records) is saved here and put back at the end.
  std::vector<gnssb200_dump> keep;
  if (want && h_dump_count) {
    cnt0.assign(h_dump_count, h_dump_count + NR);
    cnt0_min = cnt0_max = cnt0[0] < 0 ? 0 : (cnt0[0] > dump_cap ? dump_cap : cnt0[0]);
    for (int i = 0; i < NR; i++) {
      const long long v = cnt0[i] < 0 ? 0 : (cnt0[i] > dump_cap ? dump_cap : cnt0[i]);
      cnt0_min = v < cnt0_min ? v : cnt0_min;
      cnt0_max = v > cnt0_max ? v : cnt0_max;
    }
    for (int i = 0; i < NR; i++) {
      const long long v = cnt0[i] < 0 ? 0 : (cnt0[i] > dump_cap ? dump_cap : cnt0[i]);
      keep.insert(keep.end(), h_dumps + (size_t)i * dump_cap + cnt0_min, h_dumps + (size_t)i * dump_cap + v);
    }
  }
  const long long col0 = cnt0_min;  // first column any read-back touches
  const double rec_per_block = (double)nsamp * 1000.0 / h->cfg.samp_rate;  // one dump per code period (1 ms)
  const long long MARGIN = 16;
  auto win_lo = [&](long long b0) {
    const long long v = cnt0_min + (long long)floor((double)b0 * rec_per_block) - MARGIN;
    return v < col0 ? col0 : (v > dump_cap ? (long long)dump_cap : v);
  };
  auto win_hi = [&](long long b1) {
    const long long v = cnt0_max + (long long)ceil((double)b1 * rec_per_block) + MARGIN;
    return v > dump_cap ? (long long)dump_cap : v;
  };
  cudaStream_t s_back = h->s_back;
  if (!rc) TRY_(cudaEventRecord(h->ev0, s_comp));
  int c = 0;
  for (long long b0 = 0; b0 < nblocks && !rc; b0 += chunk, c++) {
    const long long nb = (nblocks - b0 < chunk) ? nblocks - b0 : chunk;
    const int buf = c & 1;
    if (c >= 2) TRY_(cudaStreamWaitEvent(s_copy, ev_used[buf], 0));  // kernels of chunk c-2 are done with it
    TRY_(cudaMemcpy2DAsync(d_stage[buf], dstride, (const uint8_t *)h_if + (size_t)b0 * blk_bytes, stride, blk_bytes * (size_t)nb, S,
                           cudaMemcpyHostToDevice, s_copy));
    TRY_(cudaEventRecord(ev_copied[buf], s_copy));
    TRY_(cudaStreamWaitEvent(s_comp, ev_copied[buf], 0));
    if (!rc) rc = track_launch(h, 0, S, d_stage[buf], dstride, fmt, nsamp, nb, 1, d_dumps, want ? dump_cap : 0, d_cnt, s_comp);
    if (windows && !rc)  // exact counts after this chunk: 4 bytes per channel, in stream order right behind its kernels
      TRY_(cudaMemcpyAsync(h->h_snap + (size_t)c * NR, d_cnt, sizeof(int32_t) * NR, cudaMemcpyDeviceToHost, s_comp));
    TRY_(cudaEventRecord(ev_used[buf], s_comp));
    if (windows && !rc) {
      const long long lo = win_lo(b0), hi = win_hi(b0 + nb);
      TRY_(cudaStreamWaitEvent(s_back, ev_used[buf], 0));
      if (hi > lo)
        TRY_(cudaMemcpy2DAsync(h_dumps + lo, sizeof(gnssb200_dump) * (size_t)dump_cap, d_dumps + lo, sizeof(gnssb200_dump) * (size_t)dump_cap,
                               sizeof(gnssb200_dump) * (size_t)(hi - lo), NR, cudaMemcpyDeviceToHost, s_back));
    }
  }
  if (!rc) TRY_(cudaEventRecord(h->ev1, s_comp));
  if (!rc && want) {
    if (!windows && dump_cap > col0)
      TRY_(cudaMemcpy2DAsync(h_dumps + col0, sizeof(gnssb200_dump) * (size_t)dump_cap, d_dumps + col0, sizeof(gnssb200_dump) * (size_t)dump_cap,
                             sizeof(gnssb200_dump) * (size_t)(dump_cap - col0), NR, cudaMemcpyDeviceToHost, s_comp));
    if (h_dump_count) TRY_(cudaMemcpyAsync(h_dump_count, d_cnt, sizeof(int32_t) * S * NCH, cudaMemcpyDeviceToHost, s_comp));
  }
  if (s_comp) TRY_(cudaStreamSynchronize(s_comp));
  if (s_copy) TRY_(cudaStreamSynchronize(s_copy));
  if (s_back) TRY_(cudaStreamSynchronize(s_back));
  if (windows && !rc) {
    // every chunk's records [count before, count after) must lie inside the window copied after that chunk
    bool ok = true;
    long long b0 = 0;
    for (long long cc = 0; cc < nchunks && ok; cc++, b0 += chunk) {
      const long long nb = (nblocks - b0 < chunk) ? nblocks - b0 : chunk;
      const long long lo = win_lo(b0), hi = win_hi(b0 + nb);
      const int32_t *after = h->h_snap + (size_t)cc * NR;
      const int32_t *before = cc ? h->h_snap + (size_t)(cc - 1) * NR : (cnt0.empty() ? nullptr : cnt0.data());
      for (int i = 0; i < NR; i++) {
        const long long f = before ? before[i] : 0, t = after[i];
        if (t > f && (f < lo || t > hi)) {
          ok = false;
          break;
        }
      }
    }
    if (!ok) {
      h->back_fallbacks++;
      if (dump_cap > col0)
        TRY_(cudaMemcpy2D(h_dumps + col0, sizeof(gnssb200_dump) * (size_t)dump_cap, d_dumps + col0, sizeof(gnssb200_dump) * (size_t)dump_cap,
                          sizeof(gnssb200_dump) * (size_t)(dump_cap - col0), NR, cudaMemcpyDeviceToHost));
    }
  }
  if (!keep.empty()) {  // the caller's earlier records between cnt0_min and each channel's own start
    size_t k = 0;
    for (int i = 0; i < NR; i++) {
      const long long v = cnt0[i] < 0 ? 0 : (cnt0[i] > dump_cap ? dump_cap : cnt0[i]);
      for (long long j = cnt0_min; j < v; j++) h_dumps[(size_t)i * dump_cap + j] = keep[k++];
    }
  }
#undef TRY_
  return rc;
}

// ---------------------------------------------------------------------------------------------
// drop-in layer: the reference's own correlator symbols
extern "C" {
int REG_read[256], REG_write[256];

// globals the reference's host program defines under '#define MAIN' (OSG/include/globals.h:38-56).
// Weak: present when linked into the reference receiver, absent when loaded through ctypes.
extern double Carrier_DCO_Delta __attribute__((weak));
extern double Code_DCO_Delta __attribute__((weak));
extern long gps_code_ref __attribute__((weak));
extern long gps_carrier_ref __attribute__((weak));
extern long glonass_code_ref __attribute__((weak));
extern long glonass_carrier_ref __attribute__((weak));
extern long d_freq __attribute__((weak));
extern double freq_bin_width __attribute__((weak));
extern int use_iq_processing __attribute__((weak));
}

struct DropIn {
  gnssb200_handle *h = nullptr;
  uint8_t *d_if = nullptr, *h_if = nullptr;  // staging (pinned host / device)
  size_t if_cap = 0;
  int32_t *h_regs = nullptr;                 // pinned 512 ints: reg_read | reg_write
  cudaStream_t st = nullptr;
};
static DropIn g_drop;

[[noreturn]] static void dropin_die(const char *where) {
  fprintf(stderr, "libgnssb200: %s failed: %s -- no CPU fallback, aborting\n", where, gnssb200_last_error_string());
  abort();
}

extern "C" void correlator_init(double tic_period) {
  gnssb200_cfg cfg;
  gnssb200_cfg_default(&cfg);
  cfg.tic_period = tic_period;
  if (&freq_bin_width) cfg.freq_bin_width = freq_bin_width;
  gnssb200_cfg_derive(&cfg);
  // what correlator.c:110-121 leaves in the host's globals
  if (&Carrier_DCO_Delta) Carrier_DCO_Delta = cfg.clock_mult * cfg.samp_rate / pow(2.0, (double)cfg.carrier_nco_bits);
  if (&Code_DCO_Delta) Code_DCO_Delta = cfg.clock_mult * cfg.samp_rate / pow(2.0, (double)cfg.code_nco_bits);
  if (&gps_code_ref) gps_code_ref = (long)cfg.gps_code_ref;
  if (&gps_carrier_ref) gps_carrier_ref = (long)cfg.gps_carrier_ref;
  if (&glonass_code_ref) glonass_code_ref = (long)(511000.0 / (cfg.clock_mult * cfg.samp_rate / pow(2.0, (double)cfg.code_nco_bits)));
  if (&glonass_carrier_ref) glonass_carrier_ref = (long)(0.0e6 / (cfg.clock_mult * cfg.samp_rate / pow(2.0, (double)cfg.carrier_nco_bits)));
  if (&d_freq) d_freq = (long)cfg.d_freq;

  if (g_drop.h) {
    gnssb200_close(g_drop.h);
    g_drop.h = nullptr;
  }
  const char *dev = getenv("GNSSB200_DEVICE");
  g_drop.h = gnssb200_open(dev ? atoi(dev) : 0, &cfg);
  if (!g_drop.h) dropin_die("gnssb200_open");
  if (gnssb200_set_streams(g_drop.h, 1)) dropin_die("gnssb200_set_streams");
  gnssb200_rx *rx = new gnssb200_rx;
  gnssb200_rx_init(rx, &cfg);  // memset(gpchan) + tic = tic_ref (correlator.c:124-128)
  memcpy(rx->reg_read, REG_read, sizeof REG_read);
  memcpy(rx->reg_write, REG_write, sizeof REG_write);
  int rc = gnssb200_upload_rx(g_drop.h, 0, 1, rx);
  delete rx;
  if (rc) dropin_die("gnssb200_upload_rx");
  if (!g_drop.st && cudaStreamCreateWithFlags(&g_drop.st, cudaStreamNonBlocking) != cudaSuccess) dropin_die("cudaStreamCreate");
  if (!g_drop.h_regs && cudaMallocHost(&g_drop.h_regs, 2048) != cudaSuccess) dropin_die("cudaMallocHost");
}

extern "C" void Sim_GP2021_int(char *IF, long nsamp) {
  DropIn &d = g_drop;
  if (!d.h) {
    gnssb200_set_error(-5, "Sim_GP2021_int before correlator_init", __FILE__, __LINE__);
    dropin_die("Sim_GP2021_int");
  }
  if (nsamp <= 0) {
    // No samples: the reference's sample loop does not run, but the call still moves the TIC counter
    // (correlator.c:155-165), applies pending epoch loads (:175-180) and rewrites both status words (:309-315).
    gnssb200_rx *rx = new gnssb200_rx;
    if (gnssb200_download_rx(d.h, 0, 1, rx)) dropin_die("gnssb200_download_rx");
    memcpy(rx->reg_read, REG_read, sizeof REG_read);
    memcpy(rx->reg_write, REG_write, sizeof REG_write);
    long long tic_count;
    if (rx->tic < (long long)nsamp) {
      tic_count = rx->tic;
      rx->tic += d.h->cfg.tic_ref - (long long)nsamp;
    } else {
      rx->tic -= (long long)nsamp;
      tic_count = -1;
    }
    for (int ch = 0; ch < NCH; ch++) {
      const int reg = ch << 3;
      if (rx->reg_write[reg + 7] != -1) {
        rx->reg_read[reg + 7] = rx->reg_write[reg + 7];
        rx->corr[ch].ms_counter = rx->reg_write[reg + 7] & 0xff;
        rx->corr[ch].bit_counter = rx->reg_write[reg + 7] >> 8;
        rx->reg_write[reg + 7] = -1;
      }
    }
    rx->reg_read[0x82] = 0;
    rx->reg_read[0x83] = tic_count > -1 ? 0x2000 : 0;
    const int rc = gnssb200_upload_rx(d.h, 0, 1, rx);
    memcpy(REG_read, rx->reg_read, sizeof REG_read);
    memcpy(REG_write, rx->reg_write, sizeof REG_write);
    delete rx;
    if (rc) dropin_die("gnssb200_upload_rx");
    return;
  }
  const int fmt = (&use_iq_processing && !use_iq_processing) ? GNSSB200_FMT_INT8_I : GNSSB200_FMT_INT8_IQ;
  const size_t bytes = fmt_bytes(fmt, nsamp);
  cudaError_t e;
  if (bytes > d.if_cap) {
    cudaFree(d.d_if);
    cudaFreeHost(d.h_if);
    d.if_cap = (bytes + 4095) & ~(size_t)4095;
    if ((e = cudaMalloc(&d.d_if, d.if_cap)) != cudaSuccess || (e = cudaMallocHost(&d.h_if, d.if_cap)) != cudaSuccess) {
      gnssb200_set_error((int)e, cudaGetErrorString(e), __FILE__, __LINE__);
      dropin_die("staging allocation");
    }
  }
  memcpy(d.h_if, IF, bytes);
  memcpy(d.h_regs, REG_read, 1024);
  memcpy(d.h_regs + 256, REG_write, 1024);
  // reg_read | reg_write are the first 2 KiB of gnssb200_rx
  e = cudaMemcpyAsync(d.h->d_rx, d.h_regs, 2048, cudaMemcpyHostToDevice, d.st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d.d_if, d.h_if, bytes, cudaMemcpyHostToDevice, d.st);
  if (e != cudaSuccess) {
    gnssb200_set_error((int)e, cudaGetErrorString(e), __FILE__, __LINE__);
    dropin_die("H2D copy");
  }
  if (track_launch(d.h, 0, 1, d.d_if, 0, fmt, (int)nsamp, 1, /*run_isr=*/0, nullptr, 0, nullptr, d.st)) dropin_die("track_launch");
  e = cudaMemcpyAsync(d.h_regs, d.h->d_rx, 2048, cudaMemcpyDeviceToHost, d.st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(d.st);
  if (e != cudaSuccess) {
    gnssb200_set_error((int)e, cudaGetErrorString(e), __FILE__, __LINE__);
    dropin_die("kernel / D2H copy");
  }
  memcpy(REG_read, d.h_regs, 1024);
  memcpy(REG_write, d.h_regs + 256, 1024);
}
