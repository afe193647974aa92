// track_common.cuh -- what both channel-loop kernels share: block parameters, sample loading / unpacking, TMA and
// mbarrier helpers, the per-thread correlation loops, the end-of-block rules (dump, TIC latch, next-block
// parameters), the literal serial block.  See track.cu for the overview.
#pragma once
#include "isr_device.cuh"


// -DTRACK_CHECK: every shared-memory address the correlator warps form and every queue / ring invariant is checked on
// the device; violations are counted in g_track_check_fail (read through gnssb200_track_check_failures).  This pool
// has compute-sanitizer closed, so this build is what the address / hand-over evidence in profiles/ comes from.
__device__ unsigned g_track_check_fail[8];
#ifdef TRACK_CHECK
#define TCHECK(slot, cond) do { if (!(cond)) atomicAdd(&g_track_check_fail[slot], 1u); } while (0)
#else
#define TCHECK(slot, cond) do { } while (0)
#endif

#define MODE_STOP (-1)
#define MODE_IDLE 0
#define MODE_FAST 1
#define MODE_SERIAL 2

// Shared-memory copy of the channel's code-table row plus the start of the next one (the reference's
// spill-over reads).  Table indices of a closed-form block stay below hc0 + w1 (= the dump position, 2046 +
// slew) before the dump and below the half chips one block spans (~1050) after it, each plus the few entries
// a chunk reads ahead; larger slews take the serial path.
#define SMEM_TBL 2304
// The copies of that window (track_ws_kernel, track_loop_kernel) are bounded by TABLE_ENTRIES only: for the fast rows
// (PRN 1..32, GLONASS) the window never reaches a row the register may not read (serial_block, which follows any slew,
// bounds every read by code_row_end).
static_assert(32 * HALF_CHIPS + SMEM_TBL <= GPS_TABLE_END, "the shared code-table window of PRN 32 reaches past row 33");

struct StepParams {
  uint32_t cph0, kph0, cinc, kinc;
  uint32_t hc0, w1, stale_idx, slew_dump;
  int mode;
  int tic_count;
  uint32_t stale_bits;   // table entry at stale_idx
  uint32_t cyc_pending;  // carrier wraps of quiet blocks not yet added to gnssb200_corr.carrier_cycle
  long long tic;         // value of the TIC down-counter after this block's tic_count was derived
};

struct TrackArgs {
  gnssb200_rx *rx;
  int32_t *chan_flags;
  const uint32_t *code_table;
  const uint8_t *d_if;
  size_t stride;
  int fmt, nsamp;
  long long nblocks;
  int run_isr;
  int first_stream;
  gnssb200_dump *dumps;
  int dump_cap;
  int32_t *dump_count;
  DevCfg cfg;
  // 1, 8, 128, 2048 as run-time values: multiplying by them keeps address arithmetic of the hot loop on the
  // FMA pipe (IMAD) instead of the ALU pipe (SHF/LOP3/IADD3), which is the busier one (ptxas would turn a
  // multiplication by a literal power of two back into a shift)
  uint32_t k1, k8, k128, k2048;
  struct SchedQueue *sched;  // work queue of this launch (track_ws_kernel)
};

// byte k of w, sign extended, in one PRMT: selector nibble k copies the byte, nibble k|8 replicates
// its sign bit (PTX prmt default mode).  Inline PTX because __byte_perm() documents only 3 selector bits.
__device__ __forceinline__ int sext8(uint32_t w, int k) {
  const uint32_t sel = 0x8880u | (uint32_t)(k * 0x1111);
  int r;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(w), "r"(0u), "r"(sel));
  return r;
}

// 8-phase LO of the GP2021 / Namuru carrier NCO (correlator.c:203-204, NAM/rtl/carrier_nco.v:21-25),
// stored so that  I*lut.x + Q*lut.y = ival + 65536*qval  with
//   ival = i_lo*I + q_lo*Q,  qval = q_lo*I - i_lo*Q   (correlator.c:214-215)
// The small tables below are nibbles of a literal (entry k = sign-extended nibble k): a `const int t[8]` indexed at run
// time is a stack array, i.e. local-memory stores and loads in every thread's prologue.
__device__ __forceinline__ int nib(uint32_t packed, int k) { return (int)(packed << (28 - 4 * k)) >> 28; }
__device__ __forceinline__ int lo_i(int k) { return nib(0xEEF1221Fu, k); }  // {-1, 1, 2, 2, 1, -1, -2, -2}
__device__ __forceinline__ int lo_q(int k) { return nib(0x1FEEF122u, k); }  // {2, 2, 1, -1, -2, -2, -1, 1}
__device__ __forceinline__ int sample_val(uint32_t code) { return nib(0xD3F1u, (int)(code & 3u)); }  // {1, -1, 3, -3}, win32_sampler.h:45-55
__device__ __forceinline__ void fill_lo_lut(uint2 *lut) {
  if (threadIdx.x < 8) {
    int k = threadIdx.x;
    lut[k].x = (uint32_t)(lo_i(k) + 65536 * lo_q(k));
    lut[k].y = (uint32_t)(lo_q(k) - 65536 * lo_i(k));
  }
}

__device__ __forceinline__ size_t bytes_for(int fmt, long long nsamples) {
  return fmt == GNSSB200_FMT_INT8_IQ ? (size_t)nsamples * 2 : (fmt == GNSSB200_FMT_PACKED2 ? (size_t)nsamples / 2 : (size_t)nsamples);
}

// one complex sample from a block, any format (slow, used by the serial path, tails, straddle fix-up)
__device__ __forceinline__ void load_sample(const uint8_t *blk, int fmt, int i, int &I, int &Q) {
  if (fmt == GNSSB200_FMT_INT8_IQ) {
    const int8_t *p = (const int8_t *)blk + 2 * (size_t)i;
    I = p[0];
    Q = p[1];
  } else if (fmt == GNSSB200_FMT_PACKED2) {
    uint32_t b = blk[i >> 1] >> ((i & 1) * 4);
    I = sample_val(b);  // FE/.../win32_sampler.h:45-55
    Q = sample_val(b >> 2);
  } else {
    I = ((const int8_t *)blk)[i];
    Q = 0;
  }
}

// SPT consecutive samples starting at i0 -> SPT/2 words of (I0,Q0,I1,Q1) int8
// One packed byte (I0 Q0 I1 Q1 as 2-bit codes, LSB first) -> int8 word (I0,Q0,I1,Q1).  The four codes are
// spread into selector nibbles and one PRMT picks the values {+1,-1,+3,-3} from a register table:
// no shared-memory look-up, no bank conflicts.
__device__ __forceinline__ uint32_t unpack_byte(uint32_t b) {
  uint32_t x = (b | (b << 4)) & 0x0F0Fu;
  x = (x | (x << 2)) & 0x3333u;
  return __byte_perm(0xFD03FF01u, 0u, x);  // bytes: code0 -> 0x01, code1 -> 0xFF, code2 -> 0x03, code3 -> 0xFD
}

template <bool SMEM, class T>
__device__ __forceinline__ T ld_in(const T *p) {
  if constexpr (SMEM)
    return *p;  // shared-memory tile written by the TMA engine
  else
    return __ldg(p);
}

template <int SPT, bool SMEM = false>
__device__ __forceinline__ void load_chunk(const uint8_t *blk, int fmt, int i0, int nsamp, bool aligned,
                                           const uint32_t *unpack_lut, uint32_t (&w)[SPT / 2]) {
  if (i0 + SPT <= nsamp && aligned) {
    if (fmt == GNSSB200_FMT_INT8_IQ) {
      const uint4 *p = reinterpret_cast<const uint4 *>(blk + 2 * (size_t)i0);
#pragma unroll
      for (int q = 0; q < SPT / 8; q++) {
        uint4 v = ld_in<SMEM>(p + q);
        w[4 * q + 0] = v.x;
        w[4 * q + 1] = v.y;
        w[4 * q + 2] = v.z;
        w[4 * q + 3] = v.w;
      }
    } else if (fmt == GNSSB200_FMT_PACKED2) {
      // SPT/2 bytes; each byte -> one word through the 256-entry shared LUT
      const uint32_t *p = reinterpret_cast<const uint32_t *>(blk + (size_t)(i0 >> 1));
#pragma unroll
      for (int q = 0; q < SPT / 8; q++) {
        uint32_t v = ld_in<SMEM>(p + q);
        w[4 * q + 0] = unpack_byte(v & 0xff);
        w[4 * q + 1] = unpack_byte((v >> 8) & 0xff);
        w[4 * q + 2] = unpack_byte((v >> 16) & 0xff);
        w[4 * q + 3] = unpack_byte(v >> 24);
      }
    } else {
      const uint32_t *p = reinterpret_cast<const uint32_t *>(blk + (size_t)i0);
#pragma unroll
      for (int q = 0; q < SPT / 4; q++) {
        uint32_t v = ld_in<SMEM>(p + q);
        w[2 * q + 0] = __byte_perm(v, 0, 0x4140);  // (I0,0,I1,0)
        w[2 * q + 1] = __byte_perm(v, 0, 0x4342);
      }
    }
  } else {
#pragma unroll
    for (int q = 0; q < SPT / 2; q++) {
      uint32_t word = 0;
#pragma unroll
      for (int e = 0; e < 2; e++) {
        int i = i0 + 2 * q + e;
        if (i < nsamp) {
          int I, Q;
          load_sample(blk, fmt, i, I, Q);
          word |= ((uint32_t)(I & 0xff) | ((uint32_t)(Q & 0xff) << 8)) << (16 * e);
        }
      }
      w[q] = word;
    }
  }
}

// ---- TMA / mbarrier helpers (sm_90+ PTX) ----------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  uint32_t ok;
  // a plain test first: in the steady state the phase has completed long ago, and test_wait answers
  // faster than try_wait (which may suspend the thread for a hardware time slice)
  asm volatile(
      "{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  while (!ok) {
#ifdef MBAR_HINT
    // with a suspend-time hint the waiting warp sleeps in the barrier unit instead of polling through the issue port
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity), "r"((uint32_t)MBAR_HINT)
        : "memory");
#else
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
#endif
  }
}

// The per-thread hot loop: SPT samples in groups of four.  Requires 1 <= kinc and 4*kinc < 2^32
// (checked by prepare_block), so at most one code-NCO carry falls inside a group: samples before it
// use the current E/P/L bits, samples after it the next table entry (correlator.c:227-250).
template <int SPT>
__device__ __forceinline__ void correlate_chunk(const uint32_t (&w)[SPT / 2], uint32_t cph, uint32_t kph,
                                                const uint32_t cinc, const uint32_t kinc, const uint32_t *tbl,
                                                uint32_t h, uint32_t bits, const uint2 *lut, int &accE, int &accP,
                                                int &accL) {
  int oE = sext8(bits, 0), oP = sext8(bits, 1), oL = sext8(bits, 2);
  int aE = 0, aP = 0, aL = 0;
  uint32_t hp = smem_u32(tbl + h);
  const uint32_t t1 = 0u - kinc, t2 = 0u - 2u * kinc, t3 = 0u - 3u * kinc, k4 = 4u * kinc;
#pragma unroll
  for (int g8 = 0; g8 < SPT / 8; g8++) {
    // eight LO look-ups in flight before the first product (shared-memory latency ~30 cycles)
    uint2 ab[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
      ab[j] = lut[cph >> 29];
      cph += cinc;
    }
    int v[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const uint32_t word = w[(8 * g8 + j) >> 1];
      const int I = sext8(word, (j & 1) * 2), Q = sext8(word, (j & 1) * 2 + 1);
      v[j] = I * (int)ab[j].x + Q * (int)ab[j].y;  // ival + 65536*qval
    }
#pragma unroll
    for (int g = 0; g < 2; g++) {
      // sample j >= 1 still sees the old bits iff no carry happened in samples 0..j-1: kph + j*kinc < 2^32
      const bool m1 = kph < t1, m2 = kph < t2, m3 = kph < t3;
      int so = v[4 * g], sn = 0;
      if (m1) so += v[4 * g + 1]; else sn += v[4 * g + 1];
      if (m2) so += v[4 * g + 2]; else sn += v[4 * g + 2];
      if (m3) so += v[4 * g + 3]; else sn += v[4 * g + 3];
      uint32_t carry;
      asm("add.cc.u32 %0, %0, %2;\n\taddc.u32 %1, 0, 0;" : "+r"(kph), "=r"(carry) : "r"(k4));
      hp += carry << 2;
      uint32_t t;
      asm("ld.shared.u32 %0, [%1];" : "=r"(t) : "r"(hp));
      const int nE = sext8(t, 0), nP = sext8(t, 1), nL = sext8(t, 2);
      aE += oE * so + nE * sn;
      aP += oP * so + nP * sn;
      aL += oL * so + nL * sn;
      oE = nE;
      oP = nP;
      oL = nL;
    }
  }
  accE = aE;
  accP = aP;
  accL = aL;
}

// Packed-native variant of the hot loop (GNSSB200_FMT_PACKED2, 32 samples = 16 bytes per thread): the
// 4-bit sample code (I,Q) and the 3-bit LO phase index a table of the finished mixer outputs
//   vlut[phase*16 + code][lane] = I*A[phase] + Q*B[phase]   (= ival + 65536*qval, exact small integers),
// replicated per lane so the look-up is bank-conflict free.  No unpack, no multiplies in the mixer.
struct PipeK {
  uint32_t k1, k8, k128, k2048;
};
template <int SPT>
__device__ __forceinline__ void correlate_chunk_packed(const uint32_t (&p)[SPT / 8], uint32_t cph, uint32_t kph,
                                                       const uint32_t cinc, const uint32_t kinc, const uint32_t *tbl,
                                                       uint32_t h, uint32_t bits, const uint32_t vlut_lane /* smem byte address of vlut[0][lane] */,
                                                       const PipeK K, int &accE, int &accP, int &accL) {
  int oE = sext8(bits, 0), oP = sext8(bits, 1), oL = sext8(bits, 2);
  int aE = 0, aP = 0, aL = 0;
  uint32_t hp = smem_u32(tbl + h);
  const uint32_t t1 = 0u - kinc, t2 = 0u - 2u * kinc, t3 = 0u - 3u * kinc, k4 = 4u * kinc;
#pragma unroll
  for (int g8 = 0; g8 < SPT / 8; g8++) {
    const uint32_t word = p[g8];
    // the eight 4-bit sample codes of this word as bytes: even samples in we, odd samples in wo
    const uint32_t we = word & 0x0F0F0F0Fu, wo = (word >> 4) & 0x0F0F0F0Fu;
    int v[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
      // entry offset = (phase*16 + code) * 128 bytes.  One PRMT on the ALU pipe (the code byte); the LO phase
      // (top three bits of the carrier NCO), both scalings and the NCO step are IMADs on the FMA pipe.
      const uint32_t code = __byte_perm((j & 1) ? wo : we, 0u, 0x4440u | (uint32_t)(j >> 1));
      const uint32_t idx = __umulhi(cph, K.k8);
      const uint32_t addr = idx * K.k2048 + (code * K.k128 + vlut_lane);
      uint32_t t;
      asm("ld.shared.u32 %0, [%1];" : "=r"(t) : "r"(addr));
      v[j] = (int)t;
      cph = cinc * K.k1 + cph;
    }
#pragma unroll
    for (int g = 0; g < 2; g++) {
      const bool m1 = kph < t1, m2 = kph < t2, m3 = kph < t3;
      int so = v[4 * g], sn = 0;
      if (m1) so += v[4 * g + 1]; else sn += v[4 * g + 1];
      if (m2) so += v[4 * g + 2]; else sn += v[4 * g + 2];
      if (m3) so += v[4 * g + 3]; else sn += v[4 * g + 3];
      uint32_t carry;
      asm("add.cc.u32 %0, %0, %2;\n\taddc.u32 %1, 0, 0;" : "+r"(kph), "=r"(carry) : "r"(k4));
      hp += carry << 2;
      uint32_t t;
      asm("ld.shared.u32 %0, [%1];" : "=r"(t) : "r"(hp));
      const int nE = sext8(t, 0), nP = sext8(t, 1), nL = sext8(t, 2);
      aE += oE * so + nE * sn;
      aP += oP * so + nP * sn;
      aL += oL * so + nL * sn;
      oE = nE;
      oP = nP;
      oL = nL;
    }
  }
  accE = aE;
  accP = aP;
  accL = aL;
}

__device__ __forceinline__ void unpack_lanes(int packed, int &lo, int &hi) {
  lo = (int)(short)(packed & 0xffff);
  hi = (packed - lo) >> 16;
}

// ---- lane-0 bookkeeping -----------------------------------------------------------------------
struct ChanShared {
  gnssb200_chan k;
  gnssb200_corr g;
  ChRegs r;
  long long tic;
  int dumped_last;
  int halted;
  int dump_count;
};

// epoch-counter load request of the host logic, applied at the start of a block (correlator.c:177-182)
__device__ __forceinline__ void apply_epoch_load(ChanShared &cs) {
  ChRegs &r = cs.r;
  if (r.w_epoch != -1) {
    r.r_meas[7] = r.w_epoch;
    cs.g.ms_counter = r.w_epoch & 0xff;
    cs.g.bit_counter = r.w_epoch >> 8;
    r.w_epoch = -1;
  }
}

// correlator parameters of the next block, part 1: what the correlator state alone decides (TIC
// down-counter, NCO phases, half-chip count) -- independent of the channel's write registers
__device__ __forceinline__ void prepare_block_state(ChanShared &cs, StepParams &sp, const TrackArgs &a) {
  const long long n = a.nsamp;
  if (cs.tic < n) {  // correlator.c:155-165
    sp.tic_count = (int)cs.tic;
    cs.tic += a.cfg.tic_ref - n;
  } else {
    cs.tic -= n;
    sp.tic_count = -1;
  }
  sp.tic = cs.tic;
  sp.cyc_pending = 0;
  sp.cph0 = cs.g.carrier_phase;
  sp.kph0 = cs.g.code_phase;
  sp.hc0 = cs.g.half_chip & 0xffff;
}
// part 2: NCO increments, dump position and path selection from the write registers
__device__ __forceinline__ void prepare_block_regs(ChanShared &cs, StepParams &sp, const TrackArgs &a, int tbl_prn) {
  const long long n = a.nsamp;
  ChRegs &r = cs.r;
  if (r.w_prn <= 0) {
    sp.mode = MODE_IDLE;
    return;
  }
  sp.cinc = (uint32_t)((r.w_carr_hi << 16) + r.w_carr_lo);
  sp.kinc = (uint32_t)((r.w_code_hi << 16) + r.w_code_lo) << 1;
  const long long slew_dump = (long long)r.w_slew + code_period(r.w_prn);  // :172 (1022 for a GLONASS channel)
  sp.slew_dump = (uint32_t)slew_dump;
  const long long w1 = ((long long)sp.hc0 + 1 >= slew_dump) ? 1 : slew_dump - sp.hc0;
  const unsigned long long wtot = ((unsigned long long)sp.kph0 + (unsigned long long)n * sp.kinc) >> 32;
  sp.w1 = (uint32_t)w1;
  sp.stale_idx = (uint32_t)(sp.hc0 + w1);
  bool fast = (r.w_prn == tbl_prn) && code_has_fast_row(r.w_prn) && slew_dump >= 1 && slew_dump < 65536 &&
              (long long)wtot < w1 + slew_dump && (wtot + 40) < SMEM_TBL && (sp.hc0 + w1 + 40) < SMEM_TBL &&
              n < (1ll << 30) && sp.kinc >= 1u && sp.kinc < (1u << 30);
  sp.mode = fast ? MODE_FAST : MODE_SERIAL;
}
__device__ __forceinline__ void prepare_block_params(ChanShared &cs, StepParams &sp, const TrackArgs &a, int tbl_prn) {
  prepare_block_state(cs, sp, a);
  prepare_block_regs(cs, sp, a, tbl_prn);
}

__device__ __forceinline__ void prepare_block(ChanShared &cs, StepParams &sp, const TrackArgs &a, int tbl_prn) {
  apply_epoch_load(cs);
  prepare_block_params(cs, sp, a, tbl_prn);
}

// dump side effects common to both paths (correlator.c:252-281)
__device__ __forceinline__ void apply_dump_counters(ChanShared &cs) {
  gnssb200_corr &g = cs.g;
  cs.r.w_slew = 0;
  g.ms_counter++;
  if (g.ms_counter == 20) g.bit_counter = (g.bit_counter + 1) % 50;
  g.ms_counter %= 20;
  cs.r.r_meas[7] = g.ms_counter + (g.bit_counter << 8);
}

// End-of-block rules of the closed-form path, split in two: everything that follows from the block's
// parameters alone (dump or not, counters, half-chip count, TIC latch, NCO phases) ...
__device__ __forceinline__ void finalize_state(ChanShared &cs, const StepParams &sp, int nsamp) {
  gnssb200_corr &g = cs.g;
  ChRegs &r = cs.r;
  const unsigned long long n = (unsigned long long)nsamp;
  const unsigned long long kend = (unsigned long long)sp.kph0 + n * sp.kinc;
  const unsigned long long cend = (unsigned long long)sp.cph0 + n * sp.cinc;
  const uint32_t wtot = (uint32_t)(kend >> 32);
  const bool dumped = sp.w1 <= wtot;
  const int epoch_before = r.r_meas[7];
  if (dumped) {
    apply_dump_counters(cs);
    g.half_chip = wtot - sp.w1;
  } else {
    g.half_chip = sp.hc0 + wtot;
  }
  cs.dumped_last = dumped ? 1 : 0;
  const uint32_t ctot = (uint32_t)(cend >> 32);
  if (sp.tic_count >= 0 && sp.tic_count < nsamp) {  // measurement latch, :286-303
    const unsigned long long m = (unsigned long long)sp.tic_count + 1;
    const unsigned long long kt = (unsigned long long)sp.kph0 + m * sp.kinc;
    const unsigned long long ct = (unsigned long long)sp.cph0 + m * sp.cinc;
    const uint32_t wa = (uint32_t)(kt >> 32), cw = (uint32_t)(ct >> 32);
    const bool by_tic = dumped && sp.w1 <= wa;
    r.r_meas[4] = by_tic ? r.r_meas[7] : epoch_before;
    r.r_meas[3] = (int)((uint32_t)ct >> 22);
    r.r_meas[1] = (int)(by_tic ? wa - sp.w1 : sp.hc0 + wa);
    r.r_meas[5] = (int)((uint32_t)kt >> 22);
    const uint32_t cyc = g.carrier_cycle + cw;
    r.r_meas[2] = (int)(cyc & 0xffff);
    r.r_meas[6] = (int)(cyc >> 16);
    g.carrier_cycle = ctot - cw;
  } else {
    g.carrier_cycle += ctot;
  }
  g.carrier_phase = (uint32_t)cend;
  g.code_phase = (uint32_t)kend;
}
// ... and the accumulators, which need the block's sums: A = samples up to the dump (or all of them),
// B = samples after it.  Requires cs.dumped_last from finalize_state.
__device__ __forceinline__ void finalize_acc(ChanShared &cs, const int (&A)[6], const int (&B)[6]) {
  gnssb200_corr &g = cs.g;
  if (cs.dumped_last) {
#pragma unroll
    for (int q = 0; q < 6; q++) {
      cs.r.r_acc[q] = g.acc[q] + A[q];
      g.acc[q] = B[q];
    }
  } else {
#pragma unroll
    for (int q = 0; q < 6; q++) g.acc[q] += A[q] + B[q];
  }
}
__device__ __forceinline__ void finalize_fast(ChanShared &cs, const StepParams &sp, const int (&A)[6], const int (&B)[6], int nsamp) {
  finalize_state(cs, sp, nsamp);
  finalize_acc(cs, A, B);
}

// literal per-sample walk of one block by a single lane (any register contents)
__device__ __noinline__ void serial_block(ChanShared &cs, const StepParams &sp, const uint32_t *code_table, int fmt, int nsamp,
                                          const uint8_t *blk) {
  gnssb200_corr &g = cs.g;
  ChRegs &r = cs.r;
  const long long row = code_table_base(r.w_prn), row_end = code_row_end(r.w_prn);
  const int dump_at = r.w_slew + code_period(r.w_prn);
  uint16_t hc = (uint16_t)g.half_chip;
  auto bits_at = [&](uint16_t hh) -> uint32_t {
    long long f = row + hh;
    return (row >= 0 && f < row_end) ? code_table[f] : 0u;
  };
  uint32_t t = bits_at(hc);
  int cE = sext8(t, 0), cP = sext8(t, 1), cL = sext8(t, 2);
  int dumped = 0;
  for (int i = 0; i < nsamp; i++) {
    const int k = g.carrier_phase >> 29;
    int I, Q;
    load_sample(blk, fmt, i, I, Q);
    const int vq = lo_q(k) * I - lo_i(k) * Q;
    const int vi = lo_i(k) * I + lo_q(k) * Q;
    g.acc[0] += cL * vi;
    g.acc[1] += cL * vq;
    g.acc[2] += cP * vi;
    g.acc[3] += cP * vq;
    g.acc[4] += cE * vi;
    g.acc[5] += cE * vq;
    uint32_t before = g.carrier_phase;
    g.carrier_phase += sp.cinc;
    if (g.carrier_phase < before) g.carrier_cycle++;
    before = g.code_phase;
    g.code_phase += sp.kinc;
    if (g.code_phase < before) {
      hc++;
      t = bits_at(hc);
      cE = sext8(t, 0);
      cP = sext8(t, 1);
      cL = sext8(t, 2);
      if (hc >= dump_at) {
        for (int q = 0; q < 6; q++) {
          r.r_acc[q] = g.acc[q];
          g.acc[q] = 0;
        }
        apply_dump_counters(cs);
        hc = 0;
        dumped = 1;
      }
    }
    if (i == sp.tic_count) {
      r.r_meas[4] = r.r_meas[7];
      r.r_meas[3] = (int)(g.carrier_phase >> 22);
      r.r_meas[1] = hc;
      r.r_meas[5] = (int)(g.code_phase >> 22);
      r.r_meas[2] = (int)(g.carrier_cycle & 0xffff);
      r.r_meas[6] = (int)(g.carrier_cycle >> 16);
      g.carrier_cycle = 0;
    }
  }
  g.half_chip = hc;
  cs.dumped_last = dumped;
}

__device__ __forceinline__ void after_block(ChanShared &cs, const TrackArgs &a, int s, int ch, long long block_index) {
  if (!cs.dumped_last) return;
  if (a.run_isr) {
    if (dev_gpsisr_channel(cs.k, cs.r, a.cfg)) {
      cs.halted = 1;
      return;
    }
  }
  if (a.dumps && cs.dump_count < a.dump_cap) {
    // 48-byte record written as three 16-byte stores
    gnssb200_dump *out = &a.dumps[((size_t)s * NCH + ch) * a.dump_cap + cs.dump_count];
    int4 q0, q1, q2;
    q0.x = (int)block_index;
    q0.y = (int)(uint16_t)(int16_t)ch | ((int)(uint16_t)(int16_t)cs.k.state << 16);
    q0.z = cs.r.r_acc[0];
    q0.w = cs.r.r_acc[1];
    q1.x = cs.r.r_acc[2];
    q1.y = cs.r.r_acc[3];
    q1.z = cs.r.r_acc[4];
    q1.w = cs.r.r_acc[5];
    q2.x = (cs.r.w_carr_hi << 16) + cs.r.w_carr_lo;
    q2.y = (cs.r.w_code_hi << 16) + cs.r.w_code_lo;
    q2.z = (int)(uint16_t)(int16_t)cs.k.n_freq | ((int)(uint16_t)(int16_t)cs.k.codes << 16);
    q2.w = cs.r.w_slew;
    int4 *o4 = reinterpret_cast<int4 *>(out);
    o4[0] = q0;
    o4[1] = q1;
    o4[2] = q2;
    cs.dump_count++;
  }
}

// sum over the warp of six ints (butterfly); result valid in every lane
__device__ __forceinline__ void warp_sum6(int (&v)[6]) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int q = 0; q < 6; q++) v[q] += __shfl_xor_sync(0xffffffffu, v[q], o);
  }
}

