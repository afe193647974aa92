/*
 * gp2021_oracle.c -- TEST INFRASTRUCTURE ONLY (oracle).  Not part of the product; nothing under
 * gnss_sdr_ru_b200/ links, loads or calls this file.  Only tests/, __graft_entry__.smoke() and the
 * cpu_baseline leg of bench.py use it.
 *
 * A sequential CPU restatement of the reference C receiver's hot path, written against the same
 * plain-C state structs as the GPU library (include/gnssb200.h) so that whole receiver states can
 * be compared byte for byte.  Reference = /root/reference, OSG =
 * trunk/GNSS_SOFTWARE_RECEIVERS/POSTPROCESSING_RECEIVERS/osgnss_next_step/src.
 *
 * Pinned (tests/test_oracle_vs_ref.py) against the reference itself compiled from its own sources
 * (oracle/_ref/libosgnss_ref34.so, recipe oracle/build_ref.sh): REG_read/REG_write after every
 * block, channel state after every gpsisr, on synthetic records and random register pokes; and
 * against the reference's golden LO sequences NAM/sci/{i,q}_carr.dat (tests/test_golden_lo.py).
 * Semantics are those of the LP64 build (C long = 64 bit).
 *
 * One documented deviation, shared with libosgnss_ref34.so: reads past a PRN's 2046-entry row
 * continue into the next row as in the reference (flat indexing), and past row 33 return 0
 * (the reference's arrays are [33][2046]; reading further is undefined there).  The GLONASS
 * ST-code row (35) lies behind that end: only GNSSB200_PRN_GLONASS reads it, a GPS row never
 * spills into it.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "../include/gnssb200.h"

#define NCH GNSSB200_N_CHANNELS
#define HALF_CHIPS 2046
#define TABLE_ROWS 37 /* rows 0, 33, 34, 36 zero; row 35: GLONASS ST code (1022 entries, then zeros) */
#define GLO_ROW 35
#define GLO_HALF_CHIPS 1022

static int8_t tab_early[TABLE_ROWS * HALF_CHIPS];
static int8_t tab_prompt[TABLE_ROWS * HALF_CHIPS];
static int8_t tab_late[TABLE_ROWS * HALF_CHIPS];
static int tables_ready;

/* OSG/correlator/correlator.c:63-91 -- G1/G2 shift registers with per-PRN G2 start states. */
static void build_tables(void) {
  static const int g2_start[33] = {0x000, 0x3f6, 0x3ec, 0x3d8, 0x3b0, 0x04b, 0x096, 0x2cb, 0x196, 0x32c, 0x3ba,
                                   0x374, 0x1d0, 0x3a0, 0x340, 0x280, 0x100, 0x113, 0x226, 0x04c, 0x098, 0x130,
                                   0x260, 0x267, 0x338, 0x270, 0x0e0, 0x1c0, 0x380, 0x22b, 0x056, 0x0ac, 0x158};
  if (tables_ready) return;
  memset(tab_early, 0, sizeof tab_early);
  memset(tab_prompt, 0, sizeof tab_prompt);
  memset(tab_late, 0, sizeof tab_late);
  for (int prn = 1; prn <= 32; prn++) {
    int8_t chip[1023];
    int g1 = 0x1FF, g2 = g2_start[prn];
    chip[0] = 1; /* :75 first chip forced */
    for (int k = 1; k < 1023; k++) {
      chip[k] = (int8_t)((g1 ^ g2) & 1);
      int f1 = ((g1 << 2) ^ (g1 << 9)) & 0x200;
      g1 = (g1 >> 1) | f1;
      int f2 = ((g2 << 1) ^ (g2 << 2) ^ (g2 << 5) ^ (g2 << 7) ^ (g2 << 8) ^ (g2 << 9)) & 0x200;
      g2 = (g2 >> 1) | f2;
    }
    for (int h = 0; h < HALF_CHIPS; h++) { /* :84-89 half-chip spaced E/P/L replicas */
      tab_early[prn * HALF_CHIPS + h] = (int8_t)(2 * chip[((h + 0) % HALF_CHIPS) >> 1] - 1);
      tab_prompt[prn * HALF_CHIPS + h] = (int8_t)(2 * chip[((h + 1) % HALF_CHIPS) >> 1] - 1);
      tab_late[prn * HALF_CHIPS + h] = (int8_t)(2 * chip[((h + 2) % HALF_CHIPS) >> 1] - 1);
    }
  }
  { /* GLONASS ST code: the g3 register of NAM/rtl/code_gen.v:121-133 (all ones after the PRN-key write, output
       g3[2], feedback g3[4]^g3[0], shifting towards bit 0); replicas like the C/A rows with the period 1022.
       An extension: the C reference has only the hooks for it (include/gnssb200.h, GNSSB200_PRN_GLONASS). */
    int8_t chip[511];
    unsigned g3 = 0x1FF;
    for (int k = 0; k < 511; k++) {
      chip[k] = (int8_t)((g3 >> 2) & 1);
      unsigned fb = ((g3 >> 4) ^ g3) & 1u;
      g3 = (g3 >> 1) | (fb << 8);
    }
    for (int h = 0; h < GLO_HALF_CHIPS; h++) {
      tab_early[GLO_ROW * HALF_CHIPS + h] = (int8_t)(2 * chip[((h + 0) % GLO_HALF_CHIPS) >> 1] - 1);
      tab_prompt[GLO_ROW * HALF_CHIPS + h] = (int8_t)(2 * chip[((h + 1) % GLO_HALF_CHIPS) >> 1] - 1);
      tab_late[GLO_ROW * HALF_CHIPS + h] = (int8_t)(2 * chip[((h + 2) % GLO_HALF_CHIPS) >> 1] - 1);
    }
  }
  tables_ready = 1;
}

/* PRN register -> first entry of the channel's row (-1: no code) and its dump period in half chips */
static long code_table_base(int prn_reg) {
  if (prn_reg == GNSSB200_PRN_GLONASS) return (long)GLO_ROW * HALF_CHIPS;
  return (prn_reg >= 0 && prn_reg <= 33) ? (long)prn_reg * HALF_CHIPS : -1;
}
static int code_period(int prn_reg) { return prn_reg == GNSSB200_PRN_GLONASS ? GLO_HALF_CHIPS : HALF_CHIPS; }
/* first flat index a PRN register may no longer read: a GPS row spills over up to the end of row 33 (34 rows, as in
   libosgnss_ref34.so), the GLONASS row up to the end of the table */
static long code_row_end(int prn_reg) { return prn_reg == GNSSB200_PRN_GLONASS ? (long)TABLE_ROWS * HALF_CHIPS : 34L * HALF_CHIPS; }
static long long carrier_ref_of(const gnssb200_chan *k, const gnssb200_cfg *c) { return k->system ? c->glonass_carrier_ref : c->gps_carrier_ref; }
static long long code_ref_of(const gnssb200_chan *k, const gnssb200_cfg *c) { return k->system ? c->glonass_code_ref : c->gps_code_ref; }

/* E/P/L entry (which = 0 early, 1 prompt, 2 late) of half chip h for a PRN register value: for tests of the tables */
/* flat table read with the reference's row spill-over; at or past `end` (code_row_end) -> 0 */
static inline int tab_at(const int8_t *t, long flat, long end) {
  return (flat >= 0 && flat < end) ? t[flat] : 0;
}

int orc_code_bit(int which, int prn_reg, int h) {
  build_tables();
  const long base = code_table_base(prn_reg);
  if (base < 0) return 0;
  const int8_t *t = which == 0 ? tab_early : (which == 1 ? tab_prompt : tab_late);
  return tab_at(t, base + h, code_row_end(prn_reg));
}

/* 8-phase LO of the carrier mixer, OSG/correlator/correlator.c:203-204 (= NAM/rtl/carrier_nco.v:21-25) */
static const int lo_i[8] = {-1, 1, 2, 2, 1, -1, -2, -2};
static const int lo_q[8] = {2, 2, 1, -1, -2, -2, -1, 1};
void orc_lo_table(int phase, int out[2]) {
  out[0] = lo_i[phase & 7];
  out[1] = lo_q[phase & 7];
}

/* expose for tests: E/P/L at (PRN register, h) */
void orc_code_bits(int prn, int h, int out[3]) {
  for (int w = 0; w < 3; w++) out[w] = orc_code_bit(w, prn, h);
}

/* ------------------------------------------------------------------------------------------- */
/* configuration: OSG/include/globals.h defaults, correlator.c:107-125, osgpsisr.c:252-342        */
void orc_cfg_default(gnssb200_cfg *c) {
  memset(c, 0, sizeof *c);
  c->samp_rate = 16.0e6;
  c->clock_mult = 5.0;
  c->gps_carrier_if = 2.42e6;
  c->gps_code_f = 1023000.0;
  c->freq_bin_width = 1000.0;
  c->tic_period = 0.0; /* int tic_period = 0.1 -> 0 (globals.h:52) */
  c->carrier_nco_bits = 30;
  c->code_nco_bits = 29;
  c->acq_thresh = 1800;
  c->interr_int_us = 512;
  c->Bnp = 25;
  c->Bnf = 1400;
  c->Bnd = 2;
  c->pll_integ_ms = 1;
  c->dll_integ_ms = 1;
  c->glonass_carrier_if = 0.0;   /* globals.h:19 */
  c->glonass_code_f = 511000.0;  /* globals.h:20 */
}

void orc_cfg_derive(gnssb200_cfg *c) {
  double carr_delta = c->clock_mult * c->samp_rate / pow(2.0, c->carrier_nco_bits);
  double code_delta = c->clock_mult * c->samp_rate / pow(2.0, c->code_nco_bits);
  c->gps_code_ref = (int64_t)(c->gps_code_f / code_delta);
  c->gps_carrier_ref = (int64_t)(c->gps_carrier_if / carr_delta);
  c->glonass_code_ref = (int64_t)(c->glonass_code_f / code_delta);       /* correlator.c:117 */
  c->glonass_carrier_ref = (int64_t)(c->glonass_carrier_if / carr_delta); /* correlator.c:118 */
  c->d_freq = (int64_t)((int)c->freq_bin_width / carr_delta); /* (int) binds to freq_bin_width, :121 */
  c->tic_ref = (int64_t)(c->samp_rate * c->tic_period);
  /* loop filters, Kaplan & Hegarty pp.179-183 as coded at osgpsisr.c:252-342 */
  {
    double wnp = c->Bnp / 0.53, wnf = c->Bnf / 0.25, T = (double)c->pll_integ_ms / 1000, a2 = 1.414;
    double k1 = T * (wnp * wnp) + a2 * wnp, k2 = a2 * wnp, k3 = T * wnf;
    double g = (double)(1 << c->carrier_nco_bits) / (c->samp_rate * c->clock_mult);
    c->pll_i1 = (int)(k1 * g);
    c->pll_i2 = (int)(k2 * g);
    c->pll_i3 = (int)(k3 * g);
  }
  {
    double w = c->Bnd / 0.53, T = (double)c->dll_integ_ms / 1000, a2 = 1.414;
    double k1 = T * (w * w) + a2 * w, k2 = a2 * w;
    double g = (double)(1 << c->code_nco_bits) / (c->samp_rate * c->clock_mult);
    c->dll_i1 = (int)(k1 * g);
    c->dll_i2 = (int)(k2 * g);
  }
}

/* ------------------------------------------------------------------------------------------- */
/* register accessors: OSG/gp2021/gp2021.c                                                       */
static inline void put16(gnssb200_rx *rx, int addr, int data) { /* outpwd(): unsigned short data, :11-14 */
  rx->reg_write[addr & 0xffff] = (uint16_t)data;
}
static inline int get16(const gnssb200_rx *rx, int addr) { /* from_gps(): short, :24-28 */
  return (int16_t)rx->reg_read[addr];
}
void orc_ch_cntl(gnssb200_rx *rx, int ch, int data) { put16(rx, ch << 3, data); }
void orc_ch_code_slew(gnssb200_rx *rx, int ch, int data) { put16(rx, (ch << 3) + 0x84, data); }
void orc_ch_epoch_load(gnssb200_rx *rx, int ch, unsigned data) { put16(rx, (ch << 3) + 7, (int)data); }
static void put_nco(gnssb200_rx *rx, const gnssb200_cfg *c, int addr, int64_t freq, int bits) {
  /* :80-118  freq << (32-bits), times the clock multiplier in double, back to long, split hi/lo */
  int64_t w = freq << (32 - bits);
  w = (int64_t)((double)w * c->clock_mult);
  put16(rx, addr, (int)(w >> 16));
  put16(rx, addr + 1, (int)(w & 0xffff));
}
void orc_ch_carrier(gnssb200_rx *rx, const gnssb200_cfg *c, int ch, int64_t freq) {
  put_nco(rx, c, (ch << 3) + 3, freq, c->carrier_nco_bits);
}
void orc_ch_code(gnssb200_rx *rx, const gnssb200_cfg *c, int ch, int64_t freq) {
  put_nco(rx, c, (ch << 3) + 5, freq, c->code_nco_bits);
}

/* correlator_init state + zeroed registers (REG_* are BSS in the reference) */
void orc_rx_init(gnssb200_rx *rx, const gnssb200_cfg *c) {
  build_tables();
  memset(rx, 0, sizeof *rx);
  rx->tic = c->tic_ref; /* correlator.c:125 */
}

/* reset_all_correlator_channles + simple_cold_allocate, osgnss_next_step.c:41-84, generalised to a
 * PRN list (prn[ch] <= 0 leaves the channel idle) */
void orc_rx_cold_allocate(gnssb200_rx *rx, const gnssb200_cfg *c, const int32_t prn[NCH]) {
  for (int ch = 0; ch < NCH; ch++) {
    gnssb200_chan *k = &rx->chan[ch];
    orc_ch_cntl(rx, ch, 0);
    orc_ch_carrier(rx, c, ch, c->gps_carrier_ref);
    orc_ch_code(rx, c, ch, c->gps_code_ref);
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
    orc_ch_cntl(rx, ch, prn[ch]);
    if (prn[ch] == GNSSB200_PRN_GLONASS) { /* the reference's hooks put to use: system flag, 1021 delays, GLONASS words */
      gnssb200_chan *k = &rx->chan[ch];
      k->system = 1;
      k->search_max_PRN_delay = 1021; /* osgnss_next_step.c:54 */
      orc_ch_carrier(rx, c, ch, c->glonass_carrier_ref);
      orc_ch_code(rx, c, ch, c->glonass_code_ref);
    }
  }
}

/* ------------------------------------------------------------------------------------------- */
/* Sim_GP2021_int: OSG/correlator/correlator.c:148-316                                            */
void orc_sim_gp2021(gnssb200_rx *rx, const gnssb200_cfg *c, const int8_t *IF, long nsamp, int iq) {
  int tic_count;
  int status = 0;
  build_tables();

  if (rx->tic < nsamp) { /* :155-165 */
    tic_count = (int)rx->tic;
    rx->tic += c->tic_ref - nsamp;
  } else {
    rx->tic -= nsamp;
    tic_count = -1;
  }

  for (int ch = 0; ch < NCH; ch++) {
    const int base = ch << 3;
    int *W = rx->reg_write, *R = rx->reg_read;
    gnssb200_corr *g = &rx->corr[ch];
    const int dump_at = W[base + 0x84] + code_period(W[base]); /* :172, read once per block (1022 for a GLONASS channel) */

    if (W[base + 7] != -1) { /* :177-182 epoch load */
      R[base + 7] = W[base + 7];
      g->ms_counter = W[base + 7] & 0xff;
      g->bit_counter = W[base + 7] >> 8;
      W[base + 7] = -1;
    }
    if (W[base] <= 0) continue; /* :185 idle channel */

    const uint32_t cinc = (uint32_t)((W[base + 3] << 16) + W[base + 4]); /* :187 */
    const uint32_t kinc = (uint32_t)((W[base + 5] << 16) + W[base + 6]) << 1; /* :189,:245 */
    const long row = code_table_base(W[base]) >= 0 ? code_table_base(W[base]) : (long)TABLE_ROWS * HALF_CHIPS; /* no code: reads give 0 */
    const long row_end = code_row_end(W[base]);
    uint16_t hc = (uint16_t)g->half_chip;
    int bp = tab_at(tab_prompt, row + hc, row_end), bl = tab_at(tab_late, row + hc, row_end),
        be = tab_at(tab_early, row + hc, row_end); /* :196-198 */
    const int8_t *p = IF;

    for (long i = 0; i < nsamp; i++) {
      const int k = g->carrier_phase >> 29; /* :206 */
      int vi, vq;
      if (iq) { /* :210-215 */
        int si = *p++, sq = *p++;
        vq = lo_q[k] * si - lo_i[k] * sq;
        vi = lo_i[k] * si + lo_q[k] * sq;
      } else { /* :217-224 */
        int s = *p++;
        vi = s * lo_i[k];
        vq = s * lo_q[k];
      }
      /* accumulators in REG_read order IL QL IP QP IE QE (:227-232) */
      g->acc[0] += bl * vi;
      g->acc[1] += bl * vq;
      g->acc[2] += bp * vi;
      g->acc[3] += bp * vq;
      g->acc[4] += be * vi;
      g->acc[5] += be * vq;

      { /* carrier NCO :235-240 */
        uint32_t before = g->carrier_phase;
        g->carrier_phase += cinc;
        if (g->carrier_phase < before) g->carrier_cycle++;
      }
      { /* code NCO :243-282 */
        uint32_t before = g->code_phase;
        g->code_phase += kinc;
        if (g->code_phase < before) {
          hc++;
          bp = tab_at(tab_prompt, row + hc, row_end);
          bl = tab_at(tab_late, row + hc, row_end);
          be = tab_at(tab_early, row + hc, row_end);
          if (hc >= dump_at) {
            for (int a = 0; a < 6; a++) {
              R[base + 0x84 + a] = g->acc[a];
              g->acc[a] = 0;
            }
            W[base + 0x84] = 0; /* slew consumed */
            hc = 0;
            status |= 1 << ch;
            g->ms_counter++;
            if (g->ms_counter == 20) g->bit_counter = (g->bit_counter + 1) % 50;
            g->ms_counter %= 20;
            R[base + 7] = g->ms_counter + (g->bit_counter << 8);
          }
        }
      }
      if (i == tic_count) { /* :286-303 measurement latch */
        R[base + 4] = R[base + 7];
        R[base + 3] = (int)(g->carrier_phase >> 22);
        R[base + 1] = hc;
        R[base + 5] = (int)(g->code_phase >> 22);
        R[base + 2] = (int)(g->carrier_cycle & 0xffff);
        R[base + 6] = (int)(g->carrier_cycle >> 16);
        g->carrier_cycle = 0;
      }
    }
    g->half_chip = hc;
  }
  rx->reg_read[0x82] = status;                        /* :309 */
  rx->reg_read[0x83] = (tic_count > -1) ? 0x2000 : 0; /* :312-315 */
  rx->blocks_done++;
}

/* ------------------------------------------------------------------------------------------- */
/* integer helpers: OSG/isr/osgpsisr.c:77-91, 148-178, 199-231                                    */
static int64_t iabs_trunc(int64_t v) { return (int64_t)abs((int)v); } /* the reference calls int abs() on longs */

static int64_t mag_approx(int64_t a, int64_t b) {
  int64_t c = iabs_trunc(a), d = iabs_trunc(b);
  if (c == 0 && d == 0) return 0;
  return (c > d) ? (d >> 1) + c : (c >> 1) + d;
}

static unsigned isqrt_newton(int64_t L) {
  int64_t t, div;
  unsigned r = (unsigned)L;
  if (L <= 0) return 0;
  if (L & 0xFFFF0000L)
    div = (L & 0xFF000000L) ? 0x3FFF : 0x3FF;
  else
    div = (L & 0x0FF00L) ? 0x3F : ((L > 4) ? 0x7 : L);
  for (;;) {
    t = L / div + div;
    div = t >> 1;
    div += t & 1;
    if ((int64_t)r > div)
      r = (unsigned)div;
    else {
      if (1 / r == r - 1 && 1 % r == 0) r--;
      return r;
    }
  }
}

unsigned orc_isqrt(long L) { return isqrt_newton((int64_t)L); }

static int64_t atan2_fix(int64_t y, int64_t x) { /* 1 rad = 16384 */
  const int64_t half_pi = 25736, pi = 51472;
  int64_t n, n3, res = 0;
  if (x == 0 && y == 0) return 0;
  if (x > 0 && x >= iabs_trunc(y)) {
    n = (y << 14) / x;
    n3 = ((((n * n) >> 14) * n) >> 13) / 9;
    res = n - n3;
  } else if (x <= 0 && -x >= iabs_trunc(y)) {
    n = (y << 14) / x;
    n3 = ((((n * n) >> 14) * n) >> 13) / 9;
    if (y > 0)
      res = n - n3 + pi;
    else
      res = n - n3 - pi;
  } else if (y > 0 && y > iabs_trunc(x)) {
    n = (x << 14) / y;
    n3 = ((((n * n) >> 14) * n) >> 13) / 9;
    res = half_pi - n + n3;
  } else if (y < 0 && -y > iabs_trunc(x)) {
    n = (x << 14) / y;
    n3 = ((((n * n) >> 14) * n) >> 13) / 9;
    res = -n + n3 - half_pi;
  }
  return res;
}

long orc_atan2(long y, long x) { return (long)atan2_fix((int64_t)y, (int64_t)x); }

static inline int sgn(int64_t v) { return v > 0 ? 1 : (v == 0 ? 0 : -1); }

enum { A_IP = 0, A_QP, A_IL, A_QL, A_IE, A_QE }; /* order of gnssb200_chan.accum[] */

/* ch_acq, osgpsisr.c:424-459 */
static void isr_search(gnssb200_rx *rx, const gnssb200_cfg *c, int ch) {
  gnssb200_chan *k = &rx->chan[ch];
  if (abs(k->n_freq) <= k->search_max_f) {
    int64_t pm = mag_approx(k->accum[A_IP], k->accum[A_QP]);
    if (pm > c->acq_thresh) {
      k->state = 2;
      k->i_confirm = 0;
      k->n_thresh = 0;
      k->mean_early = k->mean_prompt = k->mean_late = 0;
    } else {
      orc_ch_code_slew(rx, ch, 1);
      k->codes += 1;
    }
    if (k->codes == k->search_max_PRN_delay) {
      k->n_freq += k->del_freq;
      k->del_freq = -(k->del_freq + sgn(k->del_freq));
      k->carrier_freq = carrier_ref_of(k, c) + k->carrier_cold_corr + c->d_freq * k->n_freq;
      orc_ch_carrier(rx, c, ch, k->carrier_freq);
      k->codes = 0;
    }
  } else {
    k->n_freq = 0;
    k->del_freq = 1;
    k->carrier_freq = carrier_ref_of(k, c) + k->carrier_cold_corr + c->d_freq * k->n_freq;
    orc_ch_carrier(rx, c, ch, k->carrier_freq);
    k->codes = 0;
  }
  k->CN0 = 0;
}

/* ch_confirm, osgpsisr.c:475-518 (CONFIRM_M 3, N_OF_M_THRESH 2) */
static void isr_confirm(gnssb200_rx *rx, const gnssb200_cfg *c, int ch) {
  gnssb200_chan *k = &rx->chan[ch];
  int64_t pm = mag_approx(k->accum[A_IP], k->accum[A_QP]);
  int64_t lm = mag_approx(k->accum[A_IL], k->accum[A_QL]);
  int64_t em = mag_approx(k->accum[A_IE], k->accum[A_QE]);
  k->mean_early += em;
  k->mean_prompt += pm;
  k->mean_late += lm;
  if (pm > c->acq_thresh) k->n_thresh++;
  if (k->i_confirm == 3) {
    if (k->n_thresh >= 2) {
      k->state = 3;
      k->CN0 = 0;
      k->ch_time = 0;
      k->ms_set = 0;
      k->oldCarrNco = k->oldCodeNco = k->oldCarrError = k->oldCodeError = 0;
      k->codeFreqBasis = code_ref_of(k, c);
      k->carrFreqBasis = k->carrier_freq;
      k->sign_pos = k->prev_sign_pos = 0;
    } else
      k->state = 1;
  }
  k->i_confirm++;
}

/* the FLL-assisted PLL and DLL updates shared by pull-in and track, osgpsisr.c:539-597 / 696-754 */
static void isr_loops(gnssb200_rx *rx, const gnssb200_cfg *c, int ch) {
  gnssb200_chan *k = &rx->chan[ch];
  const int ip = k->accum[A_IP], qp = k->accum[A_QP], pip = k->prev_accum[A_IP], pqp = k->prev_accum[A_QP];
  const int ie = k->accum[A_IE], qe = k->accum[A_QE], il = k->accum[A_IL], ql = k->accum[A_QL];

  if (ip != 0 && qp != 0 && pip != 0 && pqp != 0) {
    k->cross = ip * pqp - pip * qp;                  /* int arithmetic as in the reference */
    k->dot = labs((long)(ip * pip + qp * pqp));
    k->cross >>= 8;
    k->dot >>= 8;
    k->freqError = atan2_fix(k->cross, k->dot);
    k->carrError = atan2_fix((int64_t)(qp * sgn(ip)), labs((long)ip)) / 2;
  } else {
    k->freqError = 0;
    k->carrError = k->oldCarrError;
  }
  k->carrNco = k->oldCarrNco + (c->pll_i1 * k->carrError - c->pll_i2 * k->oldCarrError - c->pll_i3 * k->freqError) / 51472;
  k->oldCarrNco = k->carrNco;
  k->oldCarrError = k->carrError;
  k->carrFreq = k->carrFreqBasis + k->carrNco;
  orc_ch_carrier(rx, c, ch, k->carrFreq);

  if (ie != 0 && qe != 0 && il != 0 && ql != 0) {
    unsigned se = isqrt_newton(ie * ie + qe * qe), sl = isqrt_newton(il * il + ql * ql);
    k->codeError = se;
    k->codeError = k->codeError - sl;
    k->codeError = 8192 * k->codeError;
    k->codeError = k->codeError / ((int)se + (int)sl);
  } else
    k->codeError = k->oldCodeError;
  k->codeNco = k->oldCodeNco + (((c->dll_i1 + 1) * k->codeError - c->dll_i2 * k->oldCodeError) / 8192);
  k->oldCodeNco = k->codeNco;
  k->oldCodeError = k->codeError;
  k->codeFreq = k->codeFreqBasis - k->codeNco;
  orc_ch_code(rx, c, ch, k->codeFreq);
}

/* ch_pull_in, osgpsisr.c:535-673 (debug test vectors are host-side bookkeeping, not state) */
static void isr_pull_in(gnssb200_rx *rx, const gnssb200_cfg *c, int ch) {
  gnssb200_chan *k = &rx->chan[ch];
  const int ip = k->accum[A_IP], pip = k->prev_accum[A_IP];
  isr_loops(rx, c, ch);

  if (sgn(ip) == -sgn(pip)) { /* :602-613 */
    k->prev_sign_pos = k->sign_pos;
    k->sign_pos = (int)k->ch_time;
    if (k->sign_pos - k->prev_sign_pos > 19)
      k->sign_count++;
    else
      k->sign_count = 0;
  }
  k->ms_count++; /* :617-634 */
  if ((sgn(ip) == -1 && (k->ms_sign & 0xfffff) == 0x00000) || (sgn(ip) == 1 && (k->ms_sign & 0xfffff) == 0xfffff)) {
    if (sgn(ip) == -sgn(pip)) {
      k->ms_count = 0;
      orc_ch_epoch_load(rx, ch, 0x1);
      k->ms_set = 1;
    }
  }
  k->ms_sign <<= 1;
  if (ip < 0) k->ms_sign |= 1;
  k->ms_count %= 20;

  k->ch_time++;
  if (k->sign_count > 30 && k->ms_set) k->state = 4; /* :651-655 */
  if (k->ch_time == 3000) {                            /* :656-671 */
    k->del_freq = 1;
    k->n_freq = 0;
    orc_ch_carrier(rx, c, ch, carrier_ref_of(k, c));
    orc_ch_code(rx, c, ch, code_ref_of(k, c));
    k->codes = 0;
    k->ch_time = 0;
    k->state = 1;
  }
}

/* ch_track, osgpsisr.c:692-768 */
static void isr_track(gnssb200_rx *rx, const gnssb200_cfg *c, int ch) {
  gnssb200_chan *k = &rx->chan[ch];
  isr_loops(rx, c, ch);
  k->ms_count = (k->ms_count + 1) % 20;
  if (k->ms_count == 19) k->bit = k->accum[A_IP] > 0 ? 1 : 0;
}

/* gpsisr, osgpsisr.c:360-408.  Returns 1 if the reference would have exit(0)ed (CHANNEL_OFF). */
int orc_gpsisr(gnssb200_rx *rx, const gnssb200_cfg *c) {
  uint16_t astat = (uint16_t)get16(rx, 0x82);
  for (int ch = 0; ch < NCH; ch++) {
    if (!(astat & (1u << ch))) continue;
    gnssb200_chan *k = &rx->chan[ch];
    memcpy(k->prev_accum, k->accum, sizeof k->accum);
    k->accum[A_IE] = (int16_t)get16(rx, (ch << 3) + 0x88);
    k->accum[A_QE] = (int16_t)get16(rx, (ch << 3) + 0x89);
    k->accum[A_IP] = (int16_t)get16(rx, (ch << 3) + 0x86);
    k->accum[A_QP] = (int16_t)get16(rx, (ch << 3) + 0x87);
    k->accum[A_IL] = (int16_t)get16(rx, (ch << 3) + 0x84);
    k->accum[A_QL] = (int16_t)get16(rx, (ch << 3) + 0x85);
  }
  for (int ch = 0; ch < NCH; ch++) {
    if (!(astat & (1u << ch))) continue;
    switch (rx->chan[ch].state) {
      case 0: rx->halted = 1; return 1;
      case 1: isr_search(rx, c, ch); break;
      case 2: isr_confirm(rx, c, ch); break;
      case 3: isr_pull_in(rx, c, ch); break;
      case 4: isr_track(rx, c, ch); break;
      default: break;
    }
  }
  return 0;
}

/* ------------------------------------------------------------------------------------------- */
/* closed loop over a record, logging one gnssb200_dump per dump (the main loop of
 * osgnss_next_step.c:168-184 without the display).  dumps: [12][dump_cap].  Returns blocks run.   */
long orc_run(gnssb200_rx *rx, const gnssb200_cfg *c, const int8_t *IF, long nsamp, long nblocks,
             gnssb200_dump *dumps, int dump_cap, int32_t *dump_count) {
  long b;
  for (b = 0; b < nblocks && !rx->halted; b++) {
    int32_t block_index = (int32_t)rx->blocks_done;
    orc_sim_gp2021(rx, c, IF + 2 * nsamp * b, nsamp, 1);
    int status = rx->reg_read[0x82];
    int halted = orc_gpsisr(rx, c);
    if (halted) break;
    if (!dumps) continue;
    for (int ch = 0; ch < NCH; ch++) {
      if (!(status & (1 << ch))) continue;
      if (dump_count[ch] >= dump_cap) continue;
      gnssb200_dump *d = &dumps[(long)ch * dump_cap + dump_count[ch]++];
      const int *W = rx->reg_write;
      d->block = block_index;
      d->ch = (int16_t)ch;
      d->state = (int16_t)rx->chan[ch].state;
      for (int a = 0; a < 6; a++) d->acc[a] = rx->reg_read[(ch << 3) + 0x84 + a];
      d->carrier_incr = (uint32_t)((W[(ch << 3) + 3] << 16) + W[(ch << 3) + 4]);
      d->code_incr = (uint32_t)((W[(ch << 3) + 5] << 16) + W[(ch << 3) + 6]);
      d->n_freq = (int16_t)rx->chan[ch].n_freq;
      d->codes = (int16_t)rx->chan[ch].codes;
      d->slew = W[(ch << 3) + 0x84];
    }
  }
  return b;
}
