// track_seg.cuh -- the half-chip-segment form of the correlator inner loop (track_ws_kernel, packed 2+2-bit input).
//
// The reference multiplies every mixed sample by the three code bits (correlator.c:227-232).  The bits only change
// when the code NCO wraps (:243-250), and a wrap starts a new half chip, so with S_m = sum of the mixer outputs of the
// samples the block sees between wrap m and wrap m+1 ("segment" m)
//     accum = sum_m bits[h(m)] * S_m                                        (exact: integer sums reordered)
// A thread owns H consecutive segments instead of a fixed run of samples: per sample only the mixer look-up is
// left (one table read, five address instructions), the three multiplies by E/P/L happen once per half chip, and the
// per-sample question "did the code NCO wrap here" disappears: with 2^29 <= kinc and 7*kinc <= 2^32 every full
// segment has 7 or 8 samples, decided by one carry of `ks + 7*kinc`.  Dump boundaries are wrap boundaries, so a
// segment never straddles a dump.  What threads cannot own as whole segments -- the head segment (it began in the
// previous block), the tail (cut by the block end) -- is evaluated one sample per lane by the closed forms.
#pragma once
#include "track_common.cuh"

struct __align__(16) BlockParams {
  uint32_t cph0, kph0, cinc, kinc;
  uint32_t hc0, w1, stale_idx, stale_bits;
  int mode, event;
  uint32_t wtot;  // code-NCO wraps over the block = index of the tail segment
  uint32_t seg;   // segment form that applies to the block's code NCO word: 1 = 7 or 8 samples per half chip, 2 = 15 or 16, 0 = neither
  double dinv;    // 1.0 / kinc, correctly rounded
  uint32_t kseg;  // (samples per full segment - 1) * kinc: the addend whose carry tells a short segment from a long one
  uint32_t pad;
};
static_assert(sizeof(BlockParams) == 64, "BlockParams: four 16-byte rows");

// Build knobs of the 8-slot segment loop (A/B builds: EXTRA_NVCC_FLAGS=-DSEG_U2=0, tools/ab_variants.sh).
// SEG_U2 = 1: two segments per loop round -- no register move of the prefetched table entry, half the loop control
// and half the re-loads of the kernel parameters k1 / k2048: 78 -> 75 instructions per segment, 1.84 -> 1.93 M
// channel*Msamples/s at 64 streams.  SEG_PIN = 1: the loop's three run-time constants (7*kinc, k1, k2048) read from
// shared memory through volatile loads, so that ptxas cannot re-create them inside the loop (it does, to save
// registers: three issue slots per segment); 73 instructions per segment, but 8 bytes of spills at the 80-register
// cap of six resident CTAs -- measured slower (1.91 M with SEG_U2, 1.82 M without), kept as a knob only.
// Also measured and not kept: three / four segments per round (1.65 / 1.57 M: 375 / 525 instructions of loop code with
// the leading segments, the warps of a scheduler spread over it); two per round with an odd run entering at the second
// half instead of a separate leading segment (1.82 M: the entry costs two branches and a reconvergence pair per
// round) or running a twelfth, idle slot (1.83 M); the eighth-sample flag through add.cc / subc (spills).
#ifndef SEG_U2
#define SEG_U2 1
#endif
#ifndef SEG_PIN  // the volatile reads (measured on their own and with the paired rounds: 1.3 % / 1.0 % slower -- off)
#define SEG_PIN 0
#endif

__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
  uint32_t t;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(t) : "r"(addr));
  return t;
}

// kinc for which every full segment holds 7 or 8 samples: a segment starts with code phase ks < kinc and ends with
// the sample whose step wraps, n = ceil((2^32 - ks) / kinc); n >= 7 for all ks < kinc iff 7*kinc <= 2^32, n <= 8 iff
// 8*kinc >= 2^32
__device__ __forceinline__ bool seg_kinc_ok(uint32_t kinc) { return kinc >= (1u << 29) && 7ull * kinc <= (1ull << 32); }
// the same with 15 or 16 samples per half chip (the 511-kHz GLONASS ST code at 16 Msps: 15.66)
__device__ __forceinline__ bool seg_kinc_ok16(uint32_t kinc) { return kinc >= (1u << 28) && 15ull * kinc <= (1ull << 32); }

// first sample of segment m >= 1: s = ceil((m*2^32 - kph0) / kinc) = floor((x - 0.5) / kinc) + 1 with x = m*2^32 -
// kph0 >= 1.  In doubles: x - 0.5 is exact (x < 2^44), (x - 0.5)/kinc is at least 0.5/kinc > 2^-31 away from every
// integer, the computed product is off by less than 2^13 * 2^-51 -- truncation gives the exact floor.
__device__ __forceinline__ uint32_t seg_start(uint32_t m, double nk05 /* -kph0 - 0.5 */, double dinv) {
  const double x = fma((double)m, 4294967296.0, nk05);
  return (uint32_t)(x * dinv) + 1u;
}

// H whole segments starting at sample s: q = bit address of the sample's 4-bit code in shared memory (8 * byte
// address of the tile + 4*s), cph / ks = carrier / code NCO phase at s (ks < kinc), hp = shared-memory byte address
// of the first segment's code-table entry (consecutive entries follow), nvalid = segments that count.
// Sums come back as two 16-bit lanes (ival + 65536*qval), |lane| <= 8*H*9 for packed samples (|ival|, |qval| <= 9
// per sample); unpack_lanes is exact while |lane| <= 32767 (tests/test_track_bounds.py checks every launched H).
struct SegBounds {  // shared-memory windows the loop may touch (TRACK_CHECK builds)
  uint32_t tile_lo, tile_hi, bits_lo, bits_hi, vlut_lo, vlut_hi;
};
template <int H>
__device__ __forceinline__ void correlate_segments(uint32_t q, uint32_t cph, uint32_t ks, const uint32_t cinc, const uint32_t kinc,
                                                   const uint32_t k7, const uint32_t hp, const int nvalid, const uint32_t vlut_lane,
                                                   const PipeK K, int &accE, int &accP, int &accL, const SegBounds bnd,
                                                   const uint32_t kseg_addr /* shared: this block's 7*kinc */,
                                                   const uint32_t kconst_addr /* shared: {k1, k2048} */) {
  int aE = 0, aP = 0, aL = 0;
  TCHECK(0, ks < kinc || nvalid == 0);                                    // a run starts on a code-NCO wrap
  TCHECK(1, hp >= bnd.bits_lo && hp + 4u * (H + 1) <= bnd.bits_hi + 4u);  // code-table entries of the run (+ one read ahead)
  // Software pipelined: the two sample words and the code-table entry of segment j+1 are fetched while segment j is
  // evaluated.  Rolled on purpose (#pragma unroll 1): unrolled H times every warp streams through > 10 KB of code per
  // block and the warps of an SM, each somewhere else in it, keep missing the instruction cache (ncu: a sixth of the
  // stalled warp-cycles were `no_instructions`, 13 % slower).
  // Pipe balance (ncu + SASS): ALU and FMA pipes both take one warp instruction per two cycles; the loop is written so
  // that neither carries much more than half of the ~75 instructions of a segment: LO phase by shift (IMAD.HI is slow),
  // table address and the "eighth sample" selections as multiply-adds by the 0/1 flag `e8`.
  uint32_t a0 = (q >> 3) & ~3u;
  TCHECK(2, a0 >= bnd.tile_lo && a0 + 8u <= bnd.tile_hi);
  uint32_t lo = lds_u32(a0), hi = lds_u32(a0 + 4);
  uint32_t t = lds_u32(hp);
  uint32_t hq = hp;                                      // running table address: the loop counter
  const uint32_t hq_valid = hp + 4u * (uint32_t)nvalid;  // segments at or past it do not count
  const uint32_t hq_end = hp + 4u * (uint32_t)H;
#if SEG_PIN
  uint32_t k7r, k1r, k2048r;
  asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(k7r) : "r"(kseg_addr));
  asm volatile("ld.volatile.shared.v2.u32 {%0, %1}, [%2];" : "=r"(k1r), "=r"(k2048r) : "r"(kconst_addr));
  TCHECK(0, k7r == k7 && k1r == K.k1 && k2048r == K.k2048);
#else
  const uint32_t k7r = k7, k1r = K.k1, k2048r = K.k2048;
#endif
  // one segment: tc = its code-table entry (fetched a segment earlier), tn receives the next one
#define SEG_BODY(tc, tn)                                                                                             \
  {                                                                                                                  \
    /* eight 4-bit sample codes from bit address q (two aligned words, funnel shift by q mod 32) */                  \
    const uint32_t wd = __funnelshift_r(lo, hi, q);                                                                  \
    /* 7 or 8 samples: the segment ends with the sample whose code step wraps; e8 = 1 when there are eight */        \
    uint32_t u, c;                                                                                                   \
    asm("add.cc.u32 %0, %2, %3;\n\taddc.u32 %1, 0, 0;" : "=r"(u), "=r"(c) : "r"(ks), "r"(k7r));                    \
    const uint32_t e8 = k1r - c;                                                                                     \
    ks = e8 * kinc + u;                                                                                              \
    q = e8 * 4u + (q + 28u);                                                                                         \
    /* next segment's words and table entry (one segment past the run in the last round: still inside the windows) */ \
    const uint32_t a = (q >> 3) & ~3u;                                                                               \
    TCHECK(2, a >= bnd.tile_lo && a + 8u <= bnd.tile_hi); /* sample window inside the tile (+ read-ahead slack) */   \
    lo = lds_u32(a);                                                                                                 \
    hi = lds_u32(a + 4);                                                                                             \
    tn = lds_u32(hq + 4u);                                                                                           \
    int v[8];                                                                                                        \
    _Pragma("unroll") for (int k = 0; k < 8; k++) {                                                                  \
      /* entry offset = (phase*16 + code) * 128 bytes + lane*4 */                                                    \
      uint32_t sh;                                                                                                   \
      if (k == 0)                                                                                                    \
        sh = wd << 7;                                                                                                \
      else if (k == 1)                                                                                               \
        sh = wd << 3;                                                                                                \
      else                                                                                                           \
        sh = wd >> (4 * k - 7);                                                                                      \
      uint32_t ca;                                                                                                   \
      asm("lop3.b32 %0, %1, 0x780, %2, 0xEA;" : "=r"(ca) : "r"(sh), "r"(vlut_lane)); /* (sh & 0x780) | vlut_lane */  \
      const uint32_t eaddr = (cph >> 29) * k2048r + ca; /* LO phase = top three bits of the carrier NCO */           \
      TCHECK(3, eaddr >= bnd.vlut_lo && eaddr + 4u <= bnd.vlut_hi); /* mixer table entry */                          \
      v[k] = (int)lds_u32(eaddr);                                                                                    \
      if (k < 7) cph += cinc;                                                                                        \
    }                                                                                                                \
    cph = e8 * cinc + cph;                                                                                           \
    const int S = (int)e8 * v[7] + (((v[0] + v[1] + v[2]) + (v[3] + v[4] + v[5])) + v[6]);                           \
    if (hq < hq_valid) {                                                                                             \
      aE += sext8(tc, 0) * S;                                                                                        \
      aP += sext8(tc, 1) * S;                                                                                        \
      aL += sext8(tc, 2) * S;                                                                                        \
    }                                                                                                                \
    hq += 4u;                                                                                                        \
  }
#if SEG_U2
  uint32_t t2;
  if (H & 1) {  // an odd run length: one segment ahead of the pairs
    SEG_BODY(t, t2)
    t = t2;
  }
  if (H > 1) {
#pragma unroll 1
    do {
      SEG_BODY(t, t2)
      SEG_BODY(t2, t)
    } while (hq != hq_end);
  }
#else
#pragma unroll 1
  do {
    uint32_t t_next;
    SEG_BODY(t, t_next)
    t = t_next;
  } while (hq != hq_end);
#endif
#undef SEG_BODY
  accE = aE;
  accP = aP;
  accL = aL;
}

// The segment loop on int8 I,Q samples (the reference's own file format, 2 bytes per sample): the
// mixer is the reference's two multiplications per output (correlator.c:214-215) with the LO pair
// (ival + 65536*qval coefficients of I and Q, fill_lo_lut) read from an 8-entry shared table -- one LDS.64, two
// PRMT sign extensions, two IMADs per sample -- and the three code multiplications once per half chip as above.
// q = bit address of the sample's I byte (8 * tile address + 16*s): a segment's 16 bytes come from five aligned words.
// One int8 sample adds up to 2*128 + 1*128 = 384 to a lane (|lo_i| + |lo_q| = 3), so the run is exact for any int8
// input only while 8*H*384 <= 32767, i.e. H <= 10 (a full-scale run of 11 segments reaches 33792 and carries into the
// other lane).
template <int H>
__device__ __forceinline__ void correlate_segments_i8(uint32_t q, uint32_t cph, uint32_t ks, const uint32_t cinc, const uint32_t kinc,
                                                      const uint32_t k7, const uint32_t hp, const int nvalid, const uint32_t lut_addr,
                                                      const PipeK K, int &accE, int &accP, int &accL, const SegBounds bnd) {
  static_assert(8 * H * 384 <= 32767, "int8 segment run: a 16-bit lane of the packed sums can overflow");
  int aE = 0, aP = 0, aL = 0;
  TCHECK(0, ks < kinc || nvalid == 0);
  TCHECK(1, hp >= bnd.bits_lo && hp + 4u * (H + 1) <= bnd.bits_hi + 4u);
  uint32_t hq = hp;
  const uint32_t hq_valid = hp + 4u * (uint32_t)nvalid;
  const uint32_t hq_end = hp + 4u * (uint32_t)H;
#pragma unroll 1
  do {
    const uint32_t a = (q >> 3) & ~3u;
    TCHECK(2, a >= bnd.tile_lo && a + 20u <= bnd.tile_hi);
    uint32_t w[5];
#pragma unroll
    for (int i = 0; i < 5; i++) w[i] = lds_u32(a + 4u * i);
    const uint32_t t = lds_u32(hq);
    uint32_t x[4];  // eight samples as (I0, Q0, I1, Q1) bytes: the window starts on a word or in its middle
#pragma unroll
    for (int i = 0; i < 4; i++) x[i] = __funnelshift_r(w[i], w[i + 1], q);
    uint32_t u, c;
    asm("add.cc.u32 %0, %2, %3;\n\taddc.u32 %1, 0, 0;" : "=r"(u), "=r"(c) : "r"(ks), "r"(k7));
    const uint32_t e8 = K.k1 - c;
    ks = e8 * kinc + u;
    q = e8 * 16u + (q + 112u);
    int v[8];
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const int I = sext8(x[k >> 1], (k & 1) * 2), Q = sext8(x[k >> 1], (k & 1) * 2 + 1);
      uint32_t lx, ly;
      asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(lx), "=r"(ly) : "r"((cph >> 29) * K.k8 + lut_addr));
      v[k] = I * (int)lx + Q * (int)ly;  // ival + 65536*qval
      if (k < 7) cph += cinc;
    }
    cph = e8 * cinc + cph;
    const int S = (int)e8 * v[7] + (((v[0] + v[1] + v[2]) + (v[3] + v[4] + v[5])) + v[6]);
    if (hq < hq_valid) {
      aE += sext8(t, 0) * S;
      aP += sext8(t, 1) * S;
      aL += sext8(t, 2) * S;
    }
    hq += 4u;
  } while (hq != hq_end);
  accE = aE;
  accP = aP;
  accL = aL;
}

// The same for code NCO rates with 15 or 16 samples per half chip (GLONASS channels): sixteen 4-bit codes per segment
// from three aligned words, the sixteenth sample conditional.  k15 = 15 * kinc.
template <int H>
__device__ __forceinline__ void correlate_segments16(uint32_t q, uint32_t cph, uint32_t ks, const uint32_t cinc, const uint32_t kinc,
                                                     const uint32_t k15, const uint32_t hp, const int nvalid, const uint32_t vlut_lane,
                                                     const PipeK K, int &accE, int &accP, int &accL, const SegBounds bnd) {
  int aE = 0, aP = 0, aL = 0;
  TCHECK(0, ks < kinc || nvalid == 0);
  TCHECK(1, hp >= bnd.bits_lo && hp + 4u * (H + 1) <= bnd.bits_hi + 4u);
  uint32_t hq = hp;
  const uint32_t hq_valid = hp + 4u * (uint32_t)nvalid;
  const uint32_t hq_end = hp + 4u * (uint32_t)H;
#pragma unroll 1
  do {
    const uint32_t a = (q >> 3) & ~3u;
    TCHECK(2, a >= bnd.tile_lo && a + 12u <= bnd.tile_hi);
    const uint32_t w0 = lds_u32(a), w1 = lds_u32(a + 4), w2 = lds_u32(a + 8);
    const uint32_t t = lds_u32(hq);
    const uint32_t wd[2] = {__funnelshift_r(w0, w1, q), __funnelshift_r(w1, w2, q)};
    uint32_t u, c;
    asm("add.cc.u32 %0, %2, %3;\n\taddc.u32 %1, 0, 0;" : "=r"(u), "=r"(c) : "r"(ks), "r"(k15));
    const uint32_t e16 = K.k1 - c;  // 1: sixteen samples
    ks = e16 * kinc + u;
    q = e16 * 4u + (q + 60u);
    int S = 0;
#pragma unroll
    for (int half = 0; half < 2; half++) {
      int v[8];
#pragma unroll
      for (int k = 0; k < 8; k++) {
        uint32_t sh;
        if (k == 0)
          sh = wd[half] << 7;
        else if (k == 1)
          sh = wd[half] << 3;
        else
          sh = wd[half] >> (4 * k - 7);
        uint32_t ca;
        asm("lop3.b32 %0, %1, 0x780, %2, 0xEA;" : "=r"(ca) : "r"(sh), "r"(vlut_lane));
        const uint32_t eaddr = (cph >> 29) * K.k2048 + ca;
        TCHECK(3, eaddr >= bnd.vlut_lo && eaddr + 4u <= bnd.vlut_hi);
        v[k] = (int)lds_u32(eaddr);
        if (half == 0 || k < 7) cph += cinc;
      }
      S += ((v[0] + v[1] + v[2]) + (v[3] + v[4] + v[5])) + v[6] + (half == 0 ? v[7] : (int)e16 * v[7]);
    }
    cph = e16 * cinc + cph;
    if (hq < hq_valid) {
      aE += sext8(t, 0) * S;
      aP += sext8(t, 1) * S;
      aL += sext8(t, 2) * S;
    }
    hq += 4u;
  } while (hq != hq_end);
  accE = aE;
  accP = aP;
  accL = aL;
}

// One sample from the closed forms (SURVEY.md Appendix A rules A2-A6) into the A (up to the dump) or B sums.
struct SampleCtx {
  uint32_t cph0, kph0, cinc, kinc, hc0, w1, stale_idx;
  const uint8_t *tile;
  const uint32_t *tbl;
  const uint2 *lut;
  int fmt;
};
__device__ __forceinline__ void eval_sample(const SampleCtx &c, int i, int (&sumA)[6], int (&sumB)[6], bool &anyB) {
  const unsigned long long ki = (unsigned long long)c.kph0 + (unsigned long long)i * c.kinc;
  const uint32_t wb = (uint32_t)(ki >> 32);
  const bool inA = wb < c.w1;
  const uint32_t rel = wb - c.w1;
  const uint32_t hh = inA ? c.hc0 + wb : (rel == 0 ? c.stale_idx : rel);
  TCHECK(5, hh < SMEM_TBL);
  const uint32_t t = c.tbl[hh];
  int I, Q;
  load_sample(c.tile, c.fmt, i, I, Q);
  const uint2 ab = c.lut[(c.cph0 + (uint32_t)i * c.cinc) >> 29];
  const int v = I * (int)ab.x + Q * (int)ab.y;
  int vi, vq;
  unpack_lanes(v, vi, vq);
  const int cE = sext8(t, 0), cP = sext8(t, 1), cL = sext8(t, 2);
  if (inA) {
    sumA[0] += cL * vi; sumA[1] += cL * vq; sumA[2] += cP * vi;
    sumA[3] += cP * vq; sumA[4] += cE * vi; sumA[5] += cE * vq;
  } else {
    sumB[0] += cL * vi; sumB[1] += cL * vq; sumB[2] += cP * vi;
    sumB[3] += cP * vq; sumB[4] += cE * vi; sumB[5] += cE * vq;
    anyB = true;
  }
}

// One block on the segment path, one correlator thread of NT.  Threads 0..NT-2 own the full segments
// 1 + tid*H ... ; a thread whose run contains the dump keeps the part before it and hands the rest to thread NT-1
// (which has no segments of its own), so every thread's sums belong to one side of the dump.  Warp 0 evaluates the
// head segment and whatever follows the owned segments (the tail) one sample per lane.
template <int NT, int H, int SLOTS = 8, bool I8 = false>
__device__ __forceinline__ void seg_block(const BlockParams &p, const SampleCtx &sc, const uint32_t tile_addr, const uint32_t tbl_addr,
                                          const uint32_t alias_addr, const uint32_t vlut_lane, const PipeK K, const int nsamp,
                                          const int ptid, int (&sumA)[6], int (&sumB)[6], bool &anyB, const SegBounds bnd_in,
                                          const uint32_t kseg_addr = 0, const uint32_t kconst_addr = 0) {
  // Which run of segments a thread owns: consecutive runs start 43 bytes apart in the tile (H = 11), i.e. lanes l and
  // l+3 of a warp would read the same bank (4-way conflicts on the two window loads of every segment); stepping
  // through the runs with stride 7 spreads a warp over the banks (2-way).
  constexpr int STEP = NT == 96 ? 7 : 1;
  const int tid = (ptid * STEP) % NT;
  const uint32_t wtot = p.wtot, w1 = p.w1;
  const uint32_t NF = wtot > 0 ? wtot - 1 : 0;  // full segments: 1 .. NF
  constexpr uint32_t OWNED = (uint32_t)(NT - 1) * H;
  const double nk05 = -(double)p.kph0 - 0.5;
  uint32_t m0, nv;
  if (tid < NT - 1) {
    const uint32_t first = (uint32_t)tid * H;
    m0 = 1 + first;
    nv = NF > first ? min(NF - first, (uint32_t)H) : 0u;
    if (m0 < w1 && w1 < m0 + nv) nv = w1 - m0;  // the run contains the dump: keep the part before it
  } else {
    // the part after the dump of the thread whose run contains it
    m0 = 1;
    nv = 0;
    if (w1 >= 2) {
      const uint32_t ts = (w1 - 2) / H, first = ts * H;
      const uint32_t end = 1 + first + (NF > first ? min(NF - first, (uint32_t)H) : 0u);
      if (ts < (uint32_t)(NT - 1) && w1 < end) {
        m0 = w1;
        nv = end - w1;
      }
    }
  }
  if (nv == 0) m0 = 1;  // idle: every address stays in bounds
  const bool clsB = m0 >= w1;
  uint32_t hp;
  if (clsB) {
    const uint32_t rel = m0 - w1;  // first half chip after the dump: stale bits, then tbl[1], tbl[2], ... (rule A6)
    hp = rel == 0 ? alias_addr : tbl_addr + 4u * rel;
  } else
    hp = tbl_addr + 4u * (p.hc0 + m0);
  const uint32_t s = seg_start(m0, nk05, p.dinv);
  SegBounds bnd = bnd_in;
  if (clsB && m0 == w1) {  // alias table of this ring slot
    bnd.bits_lo = alias_addr;
    bnd.bits_hi = alias_addr + 4u * 48u;
  }
  TCHECK(4, nv == 0 || s + (uint32_t)(SLOTS - 1) * nv <= (uint32_t)nsamp);  // owned segments lie inside the block
  int pE, pP, pL;
  if constexpr (I8)  // vlut_lane carries the shared address of the LO table here
    correlate_segments_i8<H>(8u * tile_addr + 16u * s, p.cph0 + s * p.cinc, p.kph0 + s * p.kinc, p.cinc, p.kinc, 7u * p.kinc, hp, (int)nv,
                             vlut_lane, K, pE, pP, pL, bnd);
  else if constexpr (SLOTS == 16)
    correlate_segments16<H>(8u * tile_addr + 4u * s, p.cph0 + s * p.cinc, p.kph0 + s * p.kinc, p.cinc, p.kinc, 15u * p.kinc, hp, (int)nv,
                            vlut_lane, K, pE, pP, pL, bnd);
  else
    correlate_segments<H>(8u * tile_addr + 4u * s, p.cph0 + s * p.cinc, p.kph0 + s * p.kinc, p.cinc, p.kinc, 7u * p.kinc, hp, (int)nv,
                          vlut_lane, K, pE, pP, pL, bnd, kseg_addr, kconst_addr);
  {
    int v[6];
    unpack_lanes(pL, v[0], v[1]);
    unpack_lanes(pP, v[2], v[3]);
    unpack_lanes(pE, v[4], v[5]);
    if (clsB) {
#pragma unroll
      for (int q = 0; q < 6; q++) sumB[q] += v[q];
      anyB |= nv != 0;
    } else {
#pragma unroll
      for (int q = 0; q < 6; q++) sumA[q] += v[q];
    }
  }
  if (ptid < 32) {
    // head: segment 0 = samples before the first wrap; tail: from the first segment nobody owns to the block end
    const uint32_t head_end = wtot == 0 ? (uint32_t)nsamp : min(seg_start(1, nk05, p.dinv), (uint32_t)nsamp);
    const uint32_t mt = 1 + min(NF, OWNED);
    const uint32_t tail_start = mt > wtot ? (uint32_t)nsamp : min(seg_start(mt, nk05, p.dinv), (uint32_t)nsamp);
    const uint32_t total = head_end + ((uint32_t)nsamp - tail_start);
    for (uint32_t e = (uint32_t)ptid; e < total; e += 32) {
      const uint32_t i = e < head_end ? e : tail_start + (e - head_end);
      eval_sample(sc, (int)i, sumA, sumB, anyB);
    }
  }
}

// a block whose code NCO does not fit the segment form: every sample from the closed forms, NT lanes
template <int NT>
__device__ __forceinline__ void generic_block(const SampleCtx &sc, const int nsamp, const int tid, int (&sumA)[6], int (&sumB)[6],
                                              bool &anyB) {
  for (int i = tid; i < nsamp; i += NT) eval_sample(sc, i, sumA, sumB, anyB);
}
