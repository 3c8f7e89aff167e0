// Fused SWTPG kernels for sm_100a: 14-bit unpack -> frugal pedestal -> [RS | FIR] -> threshold hit finding -> TP list.
//
// One warp owns one 64-channel group for the whole batch (time is a sequential recurrence per channel; parallelism
// comes from channels and links only, SURVEY.md §5). Frame bytes reach the warp through a private ring of shared-
// memory stages filled by the TMA engine (cp.async.bulk + mbarrier complete_tx), so no thread ever waits on a
// global load inside the tick loop and no block-wide barrier exists.
//
// Algorithms are policy structs with the same shape:
//   struct Algo { load(state, lane); seed(S); tick<...>(S, ctx, t); store(state, lane); }
// `Scalar*` policies do the arithmetic one channel at a time in 32-bit registers, exactly as written in the
// reference (any configuration); `Packed*` policies are the production fast paths on packed s16x2 registers and are
// selected by the host only for configurations inside their documented validity range (swtpg_capi.cu: classify_config).
#pragma once

#include "swtpg_device.cuh"

namespace swtpg {

// ---- HBM-resident per-group state (struct of arrays: [group][var][lane], u32 = two packed channels) -------------
enum StateVar
{
  SV_MEDIAN = 0,
  SV_ACCUM,
  SV_PREV,
  SV_CHARGE,
  SV_TOVER,
  SV_PEAK_ADC,
  SV_PEAK_TIME,
  SV_Q25,
  SV_Q75,
  SV_A25,
  SV_A75,
  SV_RS,
  SV_MED_RS,
  SV_ACC_RS,
  SV_RS_FACTOR,
  SV_RING0, // .. SV_RING0 + 7
  SV_THRESHOLD = SV_RING0 + 8, // u16x2 hit threshold by lane of the ADC-threshold algorithms (swtpg_set_link_thresholds), written by
                               // swtpg_start; FIR + IQR and WIB2 AbsRS read KernelParams::threshold instead
  SV_COUNT
};
constexpr uint32_t kStateWordsPerGroup = SV_COUNT * 32;
constexpr uint32_t kFlagInitialized = 1u;

struct KernelParams
{
  const uint8_t* frames;   // link-major units
  const uint32_t* n_units; // per link, or nullptr = units_stride everywhere
  uint32_t units_stride;
  uint32_t n_links;        // links this launch works on: its configuration group's
  const uint32_t* link_ids; // [n_links] the group's links (ascending), nullptr = links 0 .. n_links-1. Work item i of the launch
                            // is link link_ids[i mod n_links]; frames, n_units, state, flags, link_done, TPs and dumps are
                            // indexed by that link
  uint32_t* state;         // [n_groups][SV_COUNT][32]
  uint32_t* group_flags;   // [n_groups]: bit 0 initialized, bits 8..10 FIR ring phase (absTimeModNTAPS)
  uint32_t* link_cursor;   // [2] {links claimed beyond each warp's first, warps finished}; zero between launches (WIBEth kernel)
  uint32_t* link_done;     // [links of the handle] slices of the link finished in THIS launch; zero between launches (wibeth_kernel, sliced)
  uint32_t parts_log2;     // wibeth_kernel: a link's units are handed out in 2^parts_log2 consecutive slices (0 = whole links)
  uint32_t slice_geom;     // ... of equal length (0) or halving: n/2, n/4, ..., and the rest (1). The host always asks for halving
                           // slices; the equal-slice arm stays because removing it changed the compiled tick loop of every
                           // wibeth_kernel and measured slower on B200 (AbsRS 2.6 %, SimpleThreshold 0.8 %)
  TpSink sink;
  int16_t* pedestal_out;   // debug dumps [link][unit][tick][channel] or nullptr
  int16_t* waveform_out;
  // configuration (swtpg_config)
  uint32_t threshold;      // u16
  int32_t acc_limit;       // i16
  uint32_t acc_limit_neg;  // -acc_limit as its own parameter: the integer tracker's IMAD then takes it straight from the constant
                           // bank (derived from acc_limit in the kernel it costs a register or a negation per group of ticks)
  int32_t rs_scale;        // i16
  int32_t tap_exponent;
  int32_t taps[8];
  uint32_t wib2_adc_offset;
  uint32_t debug_flags;    // bit 0: PackedFirIqr always takes its exact-threshold tier (configurations outside the comparator's range)
  uint32_t all_ones;       // 0xFFFFFFFF: a constant the compiler cannot fold, so that it stays in ONE register (VIADDMNMX takes a
                           // single immediate; ptxas otherwise re-materialises the -1 operand with a move in front of every use)
  uint32_t one;            // 1: multiplier of the adds that are to run on the FMA pipe as IMAD (see fma_add below)
};

// Pipe steering. Measured with ncu on every kernel of this file: the ALU pipe (LOP3, SHF, PRMT, IADD3, VIMNMX, VIADDMNMX, HSET2,
// ISETP, SEL: half issue rate) is 70-75 % busy while the FMA pipe (IMAD, VIADD.16x2, HFMA2, HADD2: half rate as well) idles at
// 25-30 %, and ptxas turns `a + b` into IADD3 (ALU) or IMAD.IADD (FMA) by its own alternation. An add written as a * ONE + b with
// ONE = 1 read from the kernel parameters cannot be strength-reduced and is an IMAD: the add runs on the idle pipe.
// Used by the FIR + IQR trackers (WIB2 layout 30.5 -> 31.8 % of the HBM peak); the SimpleThreshold step keeps plain adds (steered:
// 1 % slower, profiles/r02_integer_accumulators.txt).
__device__ __forceinline__ uint32_t
fma_add(uint32_t a, uint32_t b, uint32_t one)
{
  return a * one + b;
}
__device__ __forceinline__ uint32_t
fma_sub(uint32_t a, uint32_t b, uint32_t minus_one)
{ // a - b
  return b * minus_one + a;
}

struct TickCtx
{
  uint64_t ts;      // timestamp of the current unit
  uint32_t tick_base; // ticks of this batch before the current unit (FIR ring phase)
  uint32_t link;
  uint32_t chan0;   // frame channel of this lane's low half
  uint32_t unit;    // index of the current unit inside the batch
  const uint8_t* link_base;
  HitStage* stage;  // warp-private hit staging (packed policies)
  const KernelParams* p;
};

// =====================================================================================================================
// Scalar policies: the reference arithmetic, one channel at a time. Used for configurations outside the packed fast
// paths' validity range and as the in-kernel statement of the semantics (cf. oracle/swtpg_oracle.c).
// =====================================================================================================================

// wibeth/tpg/UtilsAVX2.hpp:24-74 for one lane; mask = lane participates
__device__ __forceinline__ void
frugal_scalar(int& median, int s, int& accum, int L, bool mask)
{
  int to_add = s > median ? 1 : (s == median ? 0 : -1);
  if (!mask)
    to_add = 0;
  accum = wrap16(accum + to_add);
  const bool is_gt = accum > L;
  const int b = wrap16(-L); // _mm256_set1_epi16(-1 * acclimit)
  const int sa = b < 0 ? wrap16(-accum) : (b == 0 ? 0 : accum); // _mm256_sign_epi16
  const bool is_lt = sa > L;
  int step = is_gt ? 1 : 0;
  if (is_lt)
    step = -1;
  if (!mask)
    step = 0;
  median = sat16(median + step);
  if ((is_gt || is_lt) && mask)
    accum = 0;
}

// Threshold of the FIR + IQR finder for the two channels of a lane: the 16-bit lanes of `sigma * multiplier * threshold`
// evaluated the way GCC evaluates `__m256i * int` — as 4 x int64 lanes (wib2/tpg/ProcessAVX2FIR.hpp:208, SURVEY H7): the
// sigmas of 4 adjacent register POSITIONS form one u64 that is multiplied mod 2^64, so carries run from one position into
// the next. Position q of a register holds channel perm[q] of its 16 (perm = {0..7,15,8..14}). Whole warp calls;
// sig_packed = this lane's two sigmas (s16x2), lane = index inside the 64-channel group.
__device__ __noinline__ uint32_t
iqr_threshold_exact(uint32_t sig_packed, uint32_t lane, int multiplier, uint32_t threshold)
{
  uint32_t sig8[8];
#pragma unroll
  for (int j = 0; j < 8; ++j)
    sig8[j] = __shfl_sync(0xFFFFFFFFu, sig_packed, int((lane & ~7u) + j));
  const uint64_t K = uint64_t(int64_t(int16_t(multiplier))) * uint64_t(threshold); // (sigma*mult)*thr mod 2^64
  int th[2];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int ch16 = int(2 * (lane & 7u)) + h;                           // channel within the 16-channel register
    const int pos = ch16 < 8 ? ch16 : (ch16 == 15 ? 8 : ch16 + 1);       // inverse of perm {0..7,15,8..14}
    const int g = pos >> 2, jj = pos & 3;
    uint64_t v = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int pp = 4 * g + i;
      const int cc = pp < 8 ? pp : (pp == 8 ? 15 : pp - 1);              // perm
      uint32_t w = 0;
#pragma unroll
      for (int q = 0; q < 8; ++q)
        w = (cc >> 1) == q ? sig8[q] : w;
      const uint64_t s16 = (cc & 1) ? (w >> 16) : (w & 0xFFFFu);
      v |= s16 << (16 * i);
    }
    v *= K;
    th[h] = int(int16_t(uint16_t(v >> (16 * jj))));
  }
  return pack2(th[0], th[1]);
}

struct ChanRegs
{ // one channel, unpacked
  int median, accum, prev, charge, tover, peak_adc, peak_time;
  int q25, q75, a25, a75;
  int rs, med_rs, acc_rs, rs_factor;
  int ring[8];
  int threshold; // SV_THRESHOLD as int16, like the reference's signed compare against (int16)threshold
};

template<int ALGO, bool WIB2>
struct ScalarAlgo
{
  static constexpr int kGroupUnroll = 1;
  static constexpr bool kNeedsUnitTs = true; // tick() emits TPs with TickCtx::ts; the packed policies stage hits, and
                                             // HitStage::flush reads the unit's timestamp itself
  // One-warp-per-CTA WIBEth launch (launch_wibeth_geo): kWarpsPerSm persistent warps per SM (0 = as many as fit); from
  // kFullLoadWarpsPerSm x SMs + kFullLoadExtraLinks links on, kFullLoadWarpsPerSm and slices even for whole rounds (0 = never).
  static constexpr int kWarpsPerSm = 0;
  static constexpr int kFullLoadWarpsPerSm = 0;
  static constexpr int kFullLoadExtraLinks = 0;
  static constexpr int kQuadCtasPerSm = 0; // WIBEth: > 0 = run wibeth_quad_kernel (CTA of 4 links + producer warp) with that many CTAs per SM
  static constexpr int kWib2MinCtas = 1;   // WIB2: minimum CTAs per SM the register allocation must allow
  ChanRegs c[2];
  uint32_t kphase; // FIR ring phase

  __device__ __forceinline__ void load(const uint32_t* st, uint32_t lane, uint32_t flags)
  {
    auto ld = [&](int v) { return st[v * 32 + lane]; };
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      auto g = [&](int v) { uint32_t w = ld(v); return h ? hi16s(w) : lo16s(w); };
      ChanRegs& r = c[h];
      r.median = g(SV_MEDIAN); r.accum = g(SV_ACCUM); r.prev = g(SV_PREV) & 0xFFFF; r.charge = g(SV_CHARGE) & 0xFFFF;
      r.tover = g(SV_TOVER) & 0xFFFF; r.peak_adc = g(SV_PEAK_ADC) & 0xFFFF; r.peak_time = g(SV_PEAK_TIME) & 0xFFFF;
      r.q25 = g(SV_Q25); r.q75 = g(SV_Q75); r.a25 = g(SV_A25); r.a75 = g(SV_A75);
      r.rs = g(SV_RS); r.med_rs = g(SV_MED_RS); r.acc_rs = g(SV_ACC_RS); r.rs_factor = g(SV_RS_FACTOR);
#pragma unroll
      for (int j = 0; j < 8; ++j)
        r.ring[j] = g(SV_RING0 + j);
      if constexpr (ALGO != SWTPG_ALGO_FIR_IQR && !(WIB2 && ALGO == SWTPG_ALGO_ABS_RS)) // these compare against an IQR sigma
        r.threshold = g(SV_THRESHOLD);
    }
    kphase = (flags >> 8) & 7u;
  }
  __device__ __forceinline__ void store(uint32_t* st, uint32_t lane, uint32_t) const
  {
    auto put = [&](int v, int lo, int hi) { st[v * 32 + lane] = pack2(lo, hi); };
    put(SV_MEDIAN, c[0].median, c[1].median); put(SV_ACCUM, c[0].accum, c[1].accum); put(SV_PREV, c[0].prev, c[1].prev);
    put(SV_CHARGE, c[0].charge, c[1].charge); put(SV_TOVER, c[0].tover, c[1].tover);
    put(SV_PEAK_ADC, c[0].peak_adc, c[1].peak_adc); put(SV_PEAK_TIME, c[0].peak_time, c[1].peak_time);
    put(SV_Q25, c[0].q25, c[1].q25); put(SV_Q75, c[0].q75, c[1].q75); put(SV_A25, c[0].a25, c[1].a25); put(SV_A75, c[0].a75, c[1].a75);
    put(SV_RS, c[0].rs, c[1].rs); put(SV_MED_RS, c[0].med_rs, c[1].med_rs); put(SV_ACC_RS, c[0].acc_rs, c[1].acc_rs);
#pragma unroll
    for (int j = 0; j < 8; ++j)
      put(SV_RING0 + j, c[0].ring[j], c[1].ring[j]);
  }
  __device__ __forceinline__ uint32_t phase_after(uint32_t ticks) const { return (kphase + ticks) & 7u; }
  __device__ __forceinline__ void configure(const KernelParams&) {}
  static __device__ __forceinline__ uint32_t sample(const uint32_t* row, const PairPos& pp) { return extract_pair(row, pp); }
  template<int ROW_WORDS = 28>
  __device__ __forceinline__ void begin_chunk(const uint32_t*, const PairPos&) {}
  template<bool WIB2_UNITS = false>
  __device__ __forceinline__ void finish_link(const TickCtx&) {}
  template<bool WIB2_UNITS>
  static __device__ __forceinline__ void flush(const HitStage&, const TpSink&, const uint8_t*, uint32_t, uint32_t, bool = true) {} // emits directly

  // setState: pedestal = first sample, quartiles +-20 (wibeth/tpg/ProcessingInfo.hpp:116-144)
  __device__ __forceinline__ void seed(uint32_t S)
  {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int ped = h ? int(S >> 16) : int(S & 0xFFFFu);
      c[h].median = ped;
      c[h].q25 = wrap16(ped - 20);
      c[h].q75 = wrap16(ped + 20);
    }
  }

  template<int G, bool DUMP, int ROW_WORDS = 28, bool WIB2_UNITS = false>
  __device__ __forceinline__ void group(const uint32_t* rows, const PairPos& pp, const TickCtx& ctx, int t0, uint32_t* ped_out,
                                        uint32_t* wav_out, bool /*more*/)
  {
#pragma unroll
    for (int g = 0; g < G; ++g) {
      uint32_t ped, wav;
      tick(extract_pair(rows + g * ROW_WORDS, pp), ctx, t0 + g, (ctx.chan0 >> 1) & 31u, ped, wav);
      if constexpr (DUMP) {
        ped_out[g] = ped;
        wav_out[g] = wav;
      }
    }
  }

  // One tick for both channels of the lane. Returns {pedestal u16x2, waveform s16x2} through refs (debug dumps).
  __device__ __forceinline__ void tick(uint32_t S, const TickCtx& ctx, int t, uint32_t lane, uint32_t& ped_out, uint32_t& wav_out)
  {
    const KernelParams& p = *ctx.p;
    int ped[2], wav[2];
    if constexpr (ALGO == SWTPG_ALGO_FIR_IQR) {
      // wib2/tpg/ProcessAVX2FIR.hpp:103-283
      const int multiplier = 1 << p.tap_exponent;
      const int adc_max = 32767 / multiplier;
      const int sigma_max = (1 << 15) / (multiplier * 5);
      int sigma[2], filt[2];
      const uint32_t kk = (kphase + ctx.tick_base + uint32_t(t)) & 7u; // absTimeModNTAPS at this tick
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        ChanRegs& r = c[h];
        const int raw = h ? int(S >> 16) : int(S & 0xFFFFu);
        const bool is_gt = raw > r.median, is_lt = raw < r.median;
        frugal_scalar(r.q25, raw, r.a25, 10, is_lt);
        frugal_scalar(r.q75, raw, r.a75, 10, is_gt);
        frugal_scalar(r.median, raw, r.accum, 10, true);
        int x = wrap16(raw - r.median);
        int sg = wrap16(r.q75 - r.q25);
        sg = sg > sigma_max ? sigma_max : sg;
        sigma[h] = sg;
        x = x > adc_max ? adc_max : x;
        int f = 0;
#pragma unroll
        for (int j = 0; j < 7; ++j) {
          int rv = 0; // ring[(j + kphase + t) & 7] without dynamic register indexing
#pragma unroll
          for (int q = 0; q < 8; ++q)
            rv = (((j + kk) & 7) == q) ? r.ring[q] : rv;
          f = wrap16(f + wrap16(p.taps[j] * rv));
        }
#pragma unroll
        for (int q = 0; q < 8; ++q)
          if (kk == q)
            r.ring[q] = x;
        filt[h] = f;
        ped[h] = r.median;
        wav[h] = f;
      }
      // Threshold = 16-bit lane of a 64-bit-lane product over 4 adjacent AVX2 register POSITIONS (SURVEY H7).
      const uint32_t th2 = iqr_threshold_exact(pack2(sigma[0], sigma[1]), lane, multiplier, p.threshold);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int th = h ? hi16s(th2) : lo16s(th2);
        ChanRegs& r = c[h];
        const bool over = filt[h] > th;
        const bool left = r.prev && !over;
        r.charge = sat16(int(int16_t(r.charge)) + ((over ? filt[h] : 0) >> p.tap_exponent)) & 0xFFFF;
        r.tover = sat16(int(int16_t(r.tover)) + (over ? 1 : 0)) & 0xFFFF;
        if (left) {
          emit_wib2(p.sink, ctx.ts, t, uint32_t(r.charge), uint32_t(r.tover), ctx.chan0 + h, ctx.link);
          r.charge = r.tover = 0;
        }
        r.prev = over ? 0xFFFF : 0;
      }
    } else if constexpr (WIB2 && ALGO == SWTPG_ALGO_ABS_RS) {
      // wib2/tpg/ProcessRSAVX2.hpp:24-330: quartile trackers as in the FIR finder, running sum with the literal factors
      // R = 8 and scale = 5 (:29-33), every frugal limit 10, threshold sigma * info.threshold on 4 x int64 lanes (:198),
      // charge accumulates adds(RS, medianRS) >> tap_exponent (:210-213).
      const int multiplier = 1 << p.tap_exponent;
      const int sigma_max = (1 << 15) / (multiplier * int(p.threshold)); // threshold >= 1 (checked by the host)
      int sigma[2], lv[2];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        ChanRegs& r = c[h];
        const int raw = h ? int(S >> 16) : int(S & 0xFFFFu);
        const bool is_gt = raw > r.median, is_lt = raw < r.median;
        frugal_scalar(r.q25, raw, r.a25, 10, is_lt);
        frugal_scalar(r.q75, raw, r.a75, 10, is_gt);
        frugal_scalar(r.median, raw, r.accum, 10, true);
        const int x = wrap16(raw - r.median);
        const int first = wrap16(r.rs * 8);
        const int second = wrap16((x < 0 ? wrap16(-x) : x) * 5);
        int rs = wrap16((((wrap16(first + second) * 3276) >> 14) + 1) >> 1); // _mm256_mulhrs_epi16(sum, 32768/10)
        frugal_scalar(r.med_rs, rs, r.acc_rs, 10, true);
        rs = wrap16(rs - r.med_rs);
        r.rs = rs;
        lv[h] = rs;
        int sg = wrap16(r.q75 - r.q25);
        sigma[h] = sg > sigma_max ? sigma_max : sg;
        ped[h] = r.median;
        wav[h] = rs;
      }
      const uint32_t th2 = iqr_threshold_exact(pack2(sigma[0], sigma[1]), lane, 1, p.threshold);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        ChanRegs& r = c[h];
        const int th = h ? hi16s(th2) : lo16s(th2);
        const bool over = lv[h] > th;
        const bool left = r.prev && !over;
        const int temp = sat16(lv[h] + r.med_rs);
        r.charge = sat16(int(int16_t(r.charge)) + ((over ? temp : 0) >> p.tap_exponent)) & 0xFFFF;
        r.tover = sat16(int(int16_t(r.tover)) + (over ? 1 : 0)) & 0xFFFF;
        if (left) {
          emit_wib2(p.sink, ctx.ts, t, uint32_t(r.charge), uint32_t(r.tover), ctx.chan0 + h, ctx.link);
          r.charge = r.tover = 0;
        }
        r.prev = over ? 0xFFFF : 0;
      }
    } else {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        ChanRegs& r = c[h];
        const int raw = h ? int(S >> 16) : int(S & 0xFFFFu);
        const int L = (WIB2 && ALGO == SWTPG_ALGO_SIMPLE_THRESHOLD) ? 10 : p.acc_limit; // wib2/tpg/ProcessAVX2.hpp:79
        frugal_scalar(r.median, raw, r.accum, L, true);
        const int x = wrap16(raw - r.median);
        int level = x; // what the threshold sees
        if constexpr (ALGO == SWTPG_ALGO_ABS_RS || ALGO == SWTPG_ALGO_STANDARD_RS) {
          // wibeth/tpg/ProcessAbsRSAVX2.hpp:137-159, ProcessStandardRSAVX2.hpp:140-144
          const int first = wrap16(r.rs * int(int16_t(r.rs_factor)));
          const int ax = x < 0 ? wrap16(-x) : x;
          const int sum = ALGO == SWTPG_ALGO_STANDARD_RS ? wrap16(first + x) : wrap16(first + wrap16(ax * p.rs_scale));
          int rs = wrap16((((sum * 3276) >> 14) + 1) >> 1); // _mm256_mulhrs_epi16(sum, 32768/10)
          frugal_scalar(r.med_rs, rs, r.acc_rs, p.acc_limit, true);
          rs = wrap16(rs - r.med_rs);
          r.rs = rs;
          level = rs;
        }
        const bool over = level > r.threshold; // the channel's own threshold (SV_THRESHOLD)
        const bool left = r.prev && !over;
        if constexpr (WIB2) { // wib2/tpg/ProcessAVX2.hpp:104-121
          r.charge = sat16(int(int16_t(r.charge)) + ((over ? x : 0) >> p.tap_exponent)) & 0xFFFF;
          r.tover = sat16(int(int16_t(r.tover)) + (over ? 1 : 0)) & 0xFFFF;
          if (left) {
            emit_wib2(p.sink, ctx.ts, t, uint32_t(r.charge), uint32_t(r.tover), ctx.chan0 + h, ctx.link);
            r.charge = r.tover = 0;
          }
        } else { // wibeth/tpg/ProcessAVX2.hpp:114-204
          if constexpr (ALGO == SWTPG_ALGO_SIMPLE_THRESHOLD)
            r.charge = wrap16(int(int16_t(r.charge)) + (over ? x : 0)) & 0xFFFF; // add_epi16 wraps (H3)
          else
            r.charge = sat16(int(int16_t(r.charge)) + (over ? x : 0)) & 0xFFFF;  // adds_epi16
          if (x > int(int16_t(r.peak_adc))) { // not gated by `over` (H6)
            r.peak_adc = x & 0xFFFF;
            r.peak_time = r.tover;
          }
          r.tover = sat16(int(int16_t(r.tover)) + (over ? 1 : 0)) & 0xFFFF;
          if (left) {
            emit_wibeth(p.sink, ctx.ts, t, uint32_t(r.charge), uint32_t(r.tover), uint32_t(r.peak_adc), uint32_t(r.peak_time),
                        ctx.chan0 + h, ctx.link);
            r.charge = r.tover = r.peak_adc = r.peak_time = 0;
          }
        }
        r.prev = over ? 0xFFFF : 0;
        ped[h] = r.median;
        wav[h] = level;
      }
    }
    ped_out = pack2(ped[0], ped[1]);
    wav_out = pack2(wav[0], wav[1]);
  }
};

// =====================================================================================================================
// Packed fast path: SimpleThreshold on either frame layout (wibeth/tpg/ProcessAVX2.hpp:23-229, wib2/tpg/ProcessAVX2.hpp:24-200),
// two channels per 32-bit register.
// Validity (checked by the host before selecting it): 1 <= L <= 1000 and 0 <= threshold <= 32767.
//   * median m stays in [0, 16383] (it only ever steps towards samples, which are 14-bit), so adds_epi16 on it never
//     saturates;
//   * with a constant L >= 1 the accumulator is in [-L, L] between ticks, so "acc > L" <=> acc == L+1 and
//     "-acc > L" <=> acc == -(L+1);
//   * pedestal-subtracted samples s' are in [-16383, 16383] and threshold / peak_adc are non-negative, which is the
//     operand range gt2_mask_nonneg requires.
// Register forms:
//   Sb  = S - 16384           the sample as extract_pair_biased delivers it (bits 14, 15 forced to one), and
//   Mq  = 16385 - median      so that  Sb + Mq = s' + 1  ("sp1": the pedestal-subtracted sample, biased by one),
//                             clamp(Sb + Mq, 0, 2) = sign(s - m) + 1 is a single VIADDMNMX.S16x2.RELU, and Mq stays in
//                             [2, 16385]: it never passes through 0x0000 / 0xFFFF, so its +-1 steps are ONE 32-bit
//                             three-input add (IADD3) — no carry or borrow can cross the halves;
//   A   = accumulator + L     a small non-negative integer per half ([0, 2L]), so that sums with the sign code are plain
//                             32-bit adds (see pedestal_step);
//   PK1 = peak_adc + 1        compared against sp1;   thr1 = threshold + 1 likewise;   Tn = -tover, PTn = -peak_time.
// The recurrence median(t) -> median(t+1) is the critical path of a link (time is sequential per channel). Everything else
// is taken off that path by a two-stage software pipeline inside group(): the raw words of the NEXT group's rows are loaded before this
// group's arithmetic starts (prefetch across the quiet-test branch), and the quiet test / hit bookkeeping of a group is
// DEFERRED by one group, so that it is scheduled in the shadow of the next group's pedestal chain.
// =====================================================================================================================
// PIPE = true: the two-stage software pipeline, the form every WIBEth SimpleThreshold launch runs (a warp runs at the speed of
// its dependent chain; since the accumulator reset is one IMAD that chain is short enough for 20 such warps per SM to beat 28
// straight-line ones); PIPE = false: straight-line groups, fewer registers and instructions — the WIB2 kernel's form and the
// base of the running-sum policies.
template<bool PIPE>
struct PackedSimpleT
{
  static constexpr int kGroupUnroll = 4;
  static constexpr bool kNeedsUnitTs = false;
  // Launch of the pipelined form (see ScalarAlgo; the running sums set their own): 4 persistent warps per sub-partition below one
  // round of links (92 registers; profiles/r02_simple_pipeline_sweep.txt), from 2960 links on B200 (20 x 148 SMs) 5 and slices
  // for whole rounds too (profiles/r02_pipelined_full_load_probe.txt, r02_warps_crossover_probe.txt): a launch below one link per
  // warp of the 20-per-SM grid is bound by what ONE warp does per tick. 2960 links: 66.5 % of the HBM peak with 20 warps per SM
  // against 64.2 % with 16; 2500 links: 56.7 / 58.2 %.
  static constexpr int kWarpsPerSm = 16;
  static constexpr int kFullLoadWarpsPerSm = 20;
  static constexpr int kFullLoadExtraLinks = 0;
  static constexpr int kQuadCtasPerSm = 0; // one warp per CTA: the CTA form measured slower for this policy (65.4 % against
                                           // 68.2 % of the HBM peak at 5920 links, profiles/r02_quad_form_probe.txt)
  static constexpr int kWib2MinCtas = 5;
  static constexpr bool kWib2Fields = false; // which process_swtpg_hits derives the TP fields (and whether the peak is tracked)
  uint32_t Mq, A, prev, C, Tn, PK1, PTn;
  uint32_t cUp, cDn, thr1; // fp16 constants of the running sums' RS tracker (PackedRsWibEth::frugal)
  uint32_t cLn, c2L, cLL, kM1; // -L, (2L, 2L), (L, L); 0xFFFFFFFF in a register
  uint32_t shift, shmask; // WIB2 flavour only
  uint32_t raw[8];        // software pipeline: words of the next group's four rows ...
  uint32_t dsp[4], dwhen; // ... and the deferred group: its four s' + 1 and (unit << 6 | first tick); dvalid below
  bool dvalid;

  static __device__ __forceinline__ uint32_t sample(const uint32_t* row, const PairPos& pp) { return extract_pair_biased(row, pp); }

  __device__ __forceinline__ void configure(const KernelParams& p)
  {
    const uint32_t L = uint32_t(p.acc_limit) & 0xFFFFu;
    const uint32_t up = L + 1u;            // acc == L + 1       (as an fp16 subnormal: value * 2^-24 == bit pattern)
    const uint32_t dn = 0x8000u | L;       // -L: addend of the "acc - L" / "-acc - L" saturating tests (sign-magnitude)
    cUp = up | (up << 16);
    cDn = dn | (dn << 16);
    cLn = p.acc_limit_neg;
    cLL = L * 0x00010001u;
    c2L = 2u * L * 0x00010001u;
    kM1 = p.all_ones;
    shift = shmask = 0;
  }
  // thr1 of a lane's two channels from their SV_THRESHOLD row (0..32767 per half): each half clamped to `max` first, where any
  // larger threshold is never exceeded, then + 1. Once per work item, so the tick loop is the same as with one threshold.
  static __device__ __forceinline__ uint32_t thr1_of(uint32_t row, uint32_t max)
  {
    return add2(minu2(row, max * 0x00010001u), 0x00010001u);
  }
  // Register form of the running sums' RS accumulator (PackedRsWibEth): (acc - 1) as the bit pattern of an fp16x2 subnormal
  // (value * 2^-24, sign-magnitude).
  static __device__ __forceinline__ uint32_t acc_to_reg(uint32_t v)
  {
    v = add2(v, 0xFFFFFFFFu);
    const uint32_t neg = (v & 0x80008000u) >> 15; // 1 per negative half
    const uint32_t m = neg * 0xFFFFu;             // 0xFFFF per negative half
    return (add2(v ^ m, neg) & 0x7FFF7FFFu) | (m & 0x80008000u);
  }
  static __device__ __forceinline__ uint32_t acc_from_reg(uint32_t v)
  {
    const uint32_t neg = (v & 0x80008000u) >> 15;
    const uint32_t m = neg * 0xFFFFu;
    return add2(add2((v & 0x7FFF7FFFu) ^ m, neg), 0x00010001u);
  }
  __device__ __forceinline__ void load(const uint32_t* st, uint32_t lane, uint32_t)
  {
    Mq = add2(~st[SV_MEDIAN * 32 + lane], 0x40024002u); // ~m = -m - 1
    A = add2(st[SV_ACCUM * 32 + lane], cLL);            // acc + L in [0, 2L]
    prev = st[SV_PREV * 32 + lane];
    C = st[SV_CHARGE * 32 + lane];
    Tn = neg2(st[SV_TOVER * 32 + lane]);
    PK1 = add2(st[SV_PEAK_ADC * 32 + lane], 0x00010001u);
    PTn = neg2(st[SV_PEAK_TIME * 32 + lane]);
    thr1 = thr1_of(st[SV_THRESHOLD * 32 + lane], 16383u); // s' <= 16383
    dvalid = false;
    dwhen = 0u;
#pragma unroll
    for (int g = 0; g < 4; ++g)
      dsp[g] = 0u; // s' = -1: below every threshold and every PK1, so an empty pipeline stage changes nothing
  }
  __device__ __forceinline__ uint32_t median() const { return add2(~Mq, 0x40024002u); } // 16385 - Mq
  __device__ __forceinline__ void store(uint32_t* st, uint32_t lane, uint32_t) const
  {
    st[SV_MEDIAN * 32 + lane] = median();
    st[SV_ACCUM * 32 + lane] = add2(A, neg2(cLL));
    st[SV_PREV * 32 + lane] = prev;
    st[SV_CHARGE * 32 + lane] = C;
    st[SV_TOVER * 32 + lane] = neg2(Tn);
    st[SV_PEAK_ADC * 32 + lane] = add2(PK1, 0xFFFFFFFFu);
    st[SV_PEAK_TIME * 32 + lane] = neg2(PTn);
  }
  __device__ __forceinline__ uint32_t phase_after(uint32_t) const { return 0; }
  __device__ __forceinline__ void seed(uint32_t Sb) { Mq = add2(~Sb, 0x00020002u); } // 16385 - S = 1 - Sb
  template<bool WIB2_UNITS>
  static __device__ __forceinline__ void flush(const HitStage& h, const TpSink& k, const uint8_t* link_base, uint32_t link, uint32_t lane,
                                               bool everything = true)
  {
    h.template flush<WIB2_UNITS, false>(k, link_base, link, lane, everything);
  }

  // frugal streaming median (wibeth/tpg/UtilsAVX2.hpp:38-73) + pedestal subtraction (ProcessAVX2.hpp:85): Sb -> s' + 1.
  // The accumulator biased by +L is a small non-negative number per half, like the sign code, so their sum is a plain 32-bit
  // add (either pipe); one clamp takes out the two step values, the difference is the step D in {-1, 0, +1} per half held as
  // ONE 32-bit integer (the low half may borrow from the high one — harmless, only linear 32-bit operations consume it and their
  // results have non-negative halves again), and the accumulator returns to L where it stepped through one IMAD. Two
  // instructions on the ALU pipe, two (one without the final add) on the FMA pipe, three that issue on either; the fp16-subnormal
  // accumulator of round 1 had 2 / 5 / 1 and measured slower (profiles/r02_integer_accumulators.txt).
  __device__ __forceinline__ uint32_t pedestal_step(uint32_t Sb)
  {
    const uint32_t sg1 = addclamp2(Sb, Mq, 0x00020002u);        // sign(s - m) + 1 in {0,1,2}
    const uint32_t U = A + sg1;                                 // acc' + L + 1 in [0, 2L + 2]
    const uint32_t c = addclamp2(U, kM1, c2L);                  // clamp(acc' + L, 0, 2L)
    const uint32_t D = U - c - 0x00010001u;                     // the step
    A = cLn * D + c;                                            // back to L where it stepped: c - L D as ONE IMAD with -L from the
                                                                // constant bank (written c - L * D ptxas negates D first: 62
                                                                // instead of 59 instructions per quiet 4-tick group, 2-5 % slower
                                                                // for the chain-bound forms, profiles/r02_step_form_probe.txt)
    Mq -= D;                                                    // (steering these adds to the FMA pipe measured 1 % slower here)
    return add2(Sb, Mq);                                        // s' + 1 with the UPDATED median
  }
  __device__ __forceinline__ uint32_t over_mask(uint32_t sp1) const { return gt2_mask_nonneg(sp1, thr1); } // (:97-98)

  // Hit bookkeeping of one tick (:102-207). A lane on which a channel ends a hit parks its packed registers in the warp's
  // staging buffer and resets (lane-divergent); accepted iff hit_charge != 0 (src/wibeth/WIBEthFrameProcessor.cpp:520),
  // which flush() decides on the masked charge.
  __device__ __forceinline__ void hit_update(uint32_t sp1, const TickCtx& ctx, uint32_t unit, uint32_t t)
  {
    const uint32_t over = over_mask(sp1);
    const uint32_t left = prev & ~over;                 //                                  (:102)
    C = add2(C, add2(sp1, 0xFFFFFFFFu) & over);         // wrapping charge                  (:114-118)
    const uint32_t gtp = gt2_mask_nonneg(sp1, PK1);     // un-gated peak tracking           (:134-136)
    PK1 = max2(PK1, sp1);
    PTn = (Tn & gtp) | (PTn & ~gtp);                    // peak_time = tover BEFORE increment
    Tn = addmax2(Tn, over, 0x80018001u);                // tover = adds(tover, 1): -tover >= -32767   (:139-140)
    prev = over;
    if (left != 0u) {                                   //                                  (:154-204)
      ctx.stage->push(HitStage::meta(ctx.chan0, unit, t), C & left, neg2(Tn), add2(PK1, 0xFFFFFFFFu), neg2(PTn));
      C &= ~left;
      Tn &= ~left;
      PK1 = (PK1 & ~left) | (left & 0x00010001u);
      PTn &= ~left;
    }
  }

  // Quiet test and hit bookkeeping of four ticks, two tiers (results identical in both):
  //  QUIET — no channel of the warp is inside a hit and none goes over threshold in the group (by far the most common case on
  //     physical noise): per channel charge = tover = peak_time = 0 stay 0 and only the un-gated peak tracker moves,
  //     peak_adc = max(peak_adc, max_g s'_g), because with tover == 0 every peak update writes peak_time = 0 again
  //     (ProcessAVX2.hpp:134-136). Outside a hit peak_adc <= threshold (it restarts from 0 when a hit ends and every sample
  //     since was not over), so "new peak > threshold" <=> "some sample of the group is over".
  //  otherwise per-tick bookkeeping for the whole warp.
  template<bool WIB2_UNITS>
  __device__ __forceinline__ void hits_of_group(const uint32_t (&sp)[4], const TickCtx& ctx, uint32_t unit, uint32_t t0, bool valid)
  {
    const uint32_t pk = __vimax3_s16x2(__vimax3_s16x2(sp[0], sp[1], sp[2]), sp[3], PK1);
    const uint32_t busy = over_mask(pk) | prev; // some tick of the group over threshold, or still inside a hit
    if (__builtin_expect(!__any_sync(0xFFFFFFFFu, busy != 0u), 1)) {
      PK1 = pk;
      return;
    }
    if (!valid) // empty pipeline stage (first group of a link) while a hit carried over from the previous batch is still open
      return;
#pragma unroll
    for (int g = 0; g < 4; ++g)
      hit_update(sp[g], ctx, unit, t0 + uint32_t(g));
    if (ctx.stage->must_flush())
      flush<WIB2_UNITS>(*ctx.stage, ctx.p->sink, ctx.link_base, ctx.link, (ctx.chan0 >> 1) & 31u, false); // whole 32-pair rounds only
  }

  // First group of a chunk: its rows' words come straight from shared memory (the copy has just landed).
  template<int ROW_WORDS = 28>
  __device__ __forceinline__ void begin_chunk(const uint32_t* rows, const PairPos& pp)
  {
    if constexpr (PIPE) {
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        raw[2 * g] = rows[g * ROW_WORDS + pp.w0];
        raw[2 * g + 1] = rows[g * ROW_WORDS + pp.w1];
      }
    }
  }

  // G consecutive ticks. `more`: another group of the same chunk follows (its rows are prefetched before the branch).
  template<int G, bool DUMP, int ROW_WORDS = 28, bool WIB2_UNITS = false>
  __device__ __forceinline__ void group(const uint32_t* rows, const PairPos& pp, const TickCtx& ctx, int t0, uint32_t* ped_out,
                                        uint32_t* wav_out, bool more)
  {
    static_assert(G == 4, "max tree and pipeline registers are written for 4 ticks");
    uint32_t sp[G], Sb[G];
    if constexpr (PIPE) {
#pragma unroll
      for (int g = 0; g < G; ++g)
        Sb[g] = extract_pair_biased_from(raw[2 * g], raw[2 * g + 1], pp.sh);
      if (more) // the loads of the next group are in flight while this group's recurrence runs
        begin_chunk<ROW_WORDS>(rows + G * ROW_WORDS, pp);
    } else {
#pragma unroll
      for (int g = 0; g < G; ++g)
        Sb[g] = extract_pair_biased(rows + g * ROW_WORDS, pp);
    }
    // The pedestal recurrence never reads hit state: one branch-free dependent chain.
#pragma unroll
    for (int g = 0; g < G; ++g) {
      sp[g] = pedestal_step(Sb[g]);
      if constexpr (DUMP) {
        ped_out[g] = median();
        wav_out[g] = add2(sp[g], 0xFFFFFFFFu);
      }
    }
    if constexpr (PIPE) {
      // ... and in its shadow the quiet test (max tree, compare, vote) of the PREVIOUS group, which is independent of it
      hits_of_group<WIB2_UNITS>(dsp, ctx, dwhen >> 6, dwhen & 63u, dvalid);
#pragma unroll
      for (int g = 0; g < G; ++g)
        dsp[g] = sp[g];
      dwhen = (ctx.unit << 6) | uint32_t(t0);
      dvalid = true;
    } else {
      hits_of_group<WIB2_UNITS>(sp, ctx, ctx.unit, uint32_t(t0), true);
    }
  }
  // End of a link (before the staged hits are flushed and the state is stored): drain the pipeline.
  template<bool WIB2_UNITS = false>
  __device__ __forceinline__ void finish_link(const TickCtx& ctx)
  {
    if constexpr (PIPE) {
      if (dvalid)
        hits_of_group<WIB2_UNITS>(dsp, ctx, dwhen >> 6, dwhen & 63u, true);
      dvalid = false;
    }
  }
};
using PackedSimpleWibEth = PackedSimpleT<false>;
using PackedSimpleWibEthPipe = PackedSimpleT<true>;

// =====================================================================================================================
// WIB2 SimpleThreshold (wib2/tpg/ProcessAVX2.hpp:24-200). Same pedestal recurrence with the limit fixed at 10 (:79); charge
// accumulates (over ? s' : 0) >> tap_exponent with signed saturation (:110-112), no peak tracking, hit block = {chan, t,
// charge, tover}. Validity: 0 <= threshold <= 32767. Straight-line groups only: the CTA form caps the registers for five CTAs
// per SM, and the pipelined form measured 7 % slower there (profiles/r02_simple_pipeline_sweep.txt).
// =====================================================================================================================
struct PackedSimpleWib2 : PackedSimpleWibEth
{
  static constexpr bool kWib2Fields = true;
  template<bool WIB2_UNITS>
  static __device__ __forceinline__ void flush(const HitStage& h, const TpSink& k, const uint8_t* link_base, uint32_t link, uint32_t lane,
                                               bool everything = true)
  {
    h.template flush<WIB2_UNITS, true>(k, link_base, link, lane, everything);
  }

  __device__ __forceinline__ void configure(const KernelParams& p)
  {
    KernelParams q = p;
    q.acc_limit = 10; // wib2/tpg/ProcessAVX2.hpp:79
    q.acc_limit_neg = 0u - 10u;
    PackedSimpleWibEth::configure(q);
    shift = uint32_t(p.tap_exponent);
    const uint32_t m = 0xFFFFu >> shift;
    shmask = m | (m << 16);
  }
  __device__ __forceinline__ void hit_update(uint32_t sp1, const TickCtx& ctx, uint32_t unit, uint32_t t)
  {
    const uint32_t over = over_mask(sp1);
    const uint32_t left = prev & ~over;
    // over => s' > threshold >= 0: both halves of the masked value are non-negative, so the arithmetic shift is a logical one
    const uint32_t add = ((add2(sp1, 0xFFFFFFFFu) & over) >> shift) & shmask;
    C = minu2(add2(C, add), 0x7FFF7FFFu);               // adds_epi16 of two non-negative halves
    Tn = addmax2(Tn, over, 0x80018001u);                // tover = adds(tover, 1)
    prev = over;
    if (left != 0u) {
      // accepted iff hit_charge != 0 (src/wib2/WIB2FrameProcessor.cpp:429): decided in flush on the masked charge
      ctx.stage->push(HitStage::meta(ctx.chan0, unit, t), C & left, neg2(Tn));
      C &= ~left;
      Tn &= ~left;
    }
  }
  template<bool WIB2_UNITS>
  __device__ __forceinline__ void hits_of_group(const uint32_t (&sp)[4], const TickCtx& ctx, uint32_t unit, uint32_t t0, bool valid)
  {
    const uint32_t mx = __vimax3_s16x2(__vimax3_s16x2(sp[0], sp[1], sp[2]), sp[3], sp[3]);
    const uint32_t busy = over_mask(mx) | prev;
    if (__builtin_expect(!__any_sync(0xFFFFFFFFu, busy != 0u), 1))
      return; // nothing but the pedestal moves outside hits
    if (!valid)
      return;
#pragma unroll
    for (int g = 0; g < 4; ++g)
      hit_update(sp[g], ctx, unit, t0 + uint32_t(g));
    if (ctx.stage->must_flush())
      flush<WIB2_UNITS>(*ctx.stage, ctx.p->sink, ctx.link_base, ctx.link, (ctx.chan0 >> 1) & 31u, false); // whole 32-pair rounds only
  }
  template<int G, bool DUMP, int ROW_WORDS, bool WIB2_UNITS>
  __device__ __forceinline__ void group(const uint32_t* rows, const PairPos& pp, const TickCtx& ctx, int t0, uint32_t* ped_out,
                                        uint32_t* wav_out, bool /*more*/)
  {
    static_assert(G == 4, "max tree is written for 4 ticks");
    uint32_t sp[G];
#pragma unroll
    for (int g = 0; g < G; ++g) {
      sp[g] = pedestal_step(extract_pair_biased(rows + g * ROW_WORDS, pp));
      if constexpr (DUMP) {
        ped_out[g] = median();
        wav_out[g] = add2(sp[g], 0xFFFFFFFFu);
      }
    }
    hits_of_group<WIB2_UNITS>(sp, ctx, ctx.unit, uint32_t(t0), true);
  }
};

// =====================================================================================================================
// Packed fast path: WIBEth running-sum finders — AbsRS (wibeth/tpg/ProcessAbsRSAVX2.hpp:21-345) and StandardRS
// (wibeth/tpg/ProcessStandardRSAVX2.hpp:23-). Per tick and channel:
//   s' = raw - median                                     (frugal pedestal as in SimpleThreshold)
//   sum = RS * R + |s'| * scale      (AbsRS, :137-150)    or   RS * R + s'   (StandardRS, :140-144)   — mullo / add, mod 2^16
//   RS  = mulhrs(sum, 32768/10)                           (UtilsAVX2.hpp:77-81: round(sum / 10))
//   RS -= median_RS  after a second frugal update on RS   (:152-159)
//   threshold on RS; charge accumulates s' with signed saturation (:204); peak tracking on s' as in SimpleThreshold.
// The two 16-bit multiplies are done per half with 32-bit IMADs (only the low 16 bits of a product are used, so the packed
// register itself is the low-half operand and no sign extension is needed); mulhrs is sign-extend + IMAD + shift per half.
// |RS| <= 3277 by construction, so the RS median lives in [-3277, 3277] and the packed sign tests cannot overflow.
// Validity: 1 <= L <= 1000, 0 <= threshold <= 32767; any per-channel memory factor and any scale factor.
// =====================================================================================================================
template<bool STANDARD>
struct PackedRsWibEth : PackedSimpleWibEth
{
  static constexpr int kGroupUnroll = 2;
  // AbsRS: 4 warps per sub-partition beat 5 by 3 % (same sweep). Above one round of a 20-per-SM grid, 20 warps per SM with
  // halving slices, whole rounds included: AbsRS 28.7 -> 30.4 % of the HBM peak at 5920 links (its own 16 per SM hold for whole
  // links: 20 unsliced 26.9 %), StandardRS 35.4 -> 36.7 % (profiles/r02_warps_crossover_probe.txt).
  static constexpr int kWarpsPerSm = STANDARD ? 20 : 16;
  static constexpr int kFullLoadExtraLinks = 1;
  uint32_t RS1, MRq, AR;     // RS + 1 (carried value, after median subtraction); 1 - median_RS; (acc_RS - 1) as fp16 subnormal
  int f_lo, f_hi, nf_lo, nf_hi, scale;
  template<int ROW_WORDS = 28>
  __device__ __forceinline__ void begin_chunk(const uint32_t*, const PairPos&) {}
  template<bool WIB2_UNITS = false>
  __device__ __forceinline__ void finish_link(const TickCtx&) {}

  __device__ __forceinline__ void configure(const KernelParams& p)
  {
    PackedSimpleWibEth::configure(p);
    scale = p.rs_scale;
  }
  __device__ __forceinline__ void load(const uint32_t* st, uint32_t lane, uint32_t flags)
  {
    PackedSimpleWibEth::load(st, lane, flags);
    // RS - median_RS is in [-6554, 6554]: a larger threshold is never exceeded (and stays inside the comparator's range)
    thr1 = thr1_of(st[SV_THRESHOLD * 32 + lane], 6555u);
    RS1 = add2(st[SV_RS * 32 + lane], 0x00010001u);
    MRq = add2(~st[SV_MED_RS * 32 + lane], 0x00020002u);
    AR = acc_to_reg(st[SV_ACC_RS * 32 + lane]);
    const uint32_t f = st[SV_RS_FACTOR * 32 + lane];
    f_lo = lo16s(f);
    f_hi = hi16s(f);
    nf_lo = -f_lo; // RS * R = (RS + 1) * R - R: the "- R" rides on an IMAD addend
    nf_hi = -f_hi;
  }
  __device__ __forceinline__ void store(uint32_t* st, uint32_t lane, uint32_t k) const
  {
    PackedSimpleWibEth::store(st, lane, k);
    st[SV_RS * 32 + lane] = add2(RS1, 0xFFFFFFFFu);
    st[SV_MED_RS * 32 + lane] = add2(~MRq, 0x00020002u);
    st[SV_ACC_RS * 32 + lane] = acc_from_reg(AR);
  }
  // frugal update of (Mq_, A_) = (1 - median, accumulator - 1) with sample S; returns S - median + 1 with the updated median.
  // Used for the median of the RUNNING SUM, which lives in [-3277, 3277]: its register passes through zero, so the two step
  // flags are added as packed halves (two VIADD.16x2) instead of the one 32-bit add the raw pedestal gets away with.
  __device__ __forceinline__ uint32_t frugal(uint32_t S, uint32_t& Mq_, uint32_t& A_) const
  {
    const uint32_t sg1 = addclamp2(S, Mq_, 0x00020002u);
    const uint32_t T = hadd2_bits(A_, sg1);
    const uint32_t upm = eq2_mask(T, cUp);
    const uint32_t dn1 = hfma2_sat_bits(T, 0xBC00BC00u, cDn);
    A_ = hfma2_bits(ne2_abs_one(T, cUp), T, 0x80018001u);
    Mq_ = add2(add2(Mq_, upm), dn1);
    return add2(S, Mq_);
  }
  // _mm256_mulhrs_epi16(v, 3276) for the 16-bit value in the LOW half of `w` (upper half ignored): ((v * 3276 >> 14) + 1) >> 1
  // = (v * 3276 + 2^14) >> 15, which fits 32-bit arithmetic (|v * 3276| < 2^27).
  static __device__ __forceinline__ int mulhrs_low(uint32_t w)
  {
    return (int(int16_t(uint16_t(w))) * 3276 + 16384) >> 15;
  }
  // One tick: sp1 = s' + 1 (pedestal-subtracted sample, biased), returns RS - median_RS + 1
  __device__ __forceinline__ uint32_t rs_step(uint32_t sp1)
  {
    const uint32_t x = add2(sp1, 0xFFFFFFFFu);
    uint32_t lo, hi;
    if constexpr (STANDARD) {
      lo = uint32_t(int(RS1) * f_lo + int(x) + nf_lo);                       // low 16 bits: RS * R + s'
      hi = uint32_t(int(RS1 >> 16) * f_hi + int(x >> 16) + nf_hi);
    } else {
      const uint32_t ax = max2(x, neg2(x));                                  // |s'| (s' > -32768)
      lo = uint32_t(int(RS1) * f_lo + (int(ax) * scale + nf_lo));            // low 16 bits: RS * R + |s'| * scale
      hi = uint32_t(int(RS1 >> 16) * f_hi + (int(ax >> 16) * scale + nf_hi));
    }
    const int r_lo = mulhrs_low(lo), r_hi = mulhrs_low(hi);
    const uint32_t rs = __byte_perm(uint32_t(r_lo), uint32_t(r_hi), 0x5410);  // pack the two low halves
    RS1 = frugal(rs, MRq, AR);                                               // second pedestal, on the running sum
    return RS1;
  }

  __device__ __forceinline__ void hit_update(uint32_t sp1, uint32_t lv1, const TickCtx& ctx, int t)
  {
    const uint32_t over = gt2_mask_nonneg(lv1, thr1);
    const uint32_t left = prev & ~over;
    const uint32_t xm = add2(sp1, 0xFFFFFFFFu) & over;
    // adds_epi16 (:204); s' may be negative here. Packed wrapping add, then repair the (rare) halves that overflowed:
    // overflow <=> both operands have the same sign and the sum's sign differs.
    const uint32_t Cw = add2(C, xm);
    const uint32_t ovf = ~(C ^ xm) & (C ^ Cw) & 0x80008000u;
    if (__builtin_expect(ovf != 0u, 0))
      C = pack2(sat16(lo16s(C) + lo16s(xm)), sat16(hi16s(C) + hi16s(xm)));
    else
      C = Cw;
    const uint32_t gtp = gt2_mask_nonneg(sp1, PK1);                          // un-gated peak tracking on s'
    PK1 = max2(PK1, sp1);
    PTn = (Tn & gtp) | (PTn & ~gtp);
    Tn = addmax2(Tn, over, 0x80018001u);
    prev = over;
    if (left != 0u) {
      ctx.stage->push(HitStage::meta(ctx.chan0, ctx.unit, uint32_t(t)), C & left, neg2(Tn), add2(PK1, 0xFFFFFFFFu), neg2(PTn));
      C &= ~left;
      Tn &= ~left;
      PK1 = (PK1 & ~left) | (left & 0x00010001u);
      PTn &= ~left;
    }
  }

  template<int G, bool DUMP, int ROW_WORDS = 28, bool WIB2_UNITS = false>
  __device__ __forceinline__ void group(const uint32_t* rows, const PairPos& pp, const TickCtx& ctx, int t0, uint32_t* ped_out,
                                        uint32_t* wav_out, bool /*more*/)
  {
    static_assert(G == 4, "max trees below are written for 4 ticks");
    uint32_t sp[G], lv[G];
#pragma unroll
    for (int g = 0; g < G; ++g) {
      sp[g] = pedestal_step(extract_pair_biased(rows + g * ROW_WORDS, pp));
      lv[g] = rs_step(sp[g]);
      if constexpr (DUMP) {
        ped_out[g] = median();
        wav_out[g] = add2(lv[g], 0xFFFFFFFFu);
      }
    }
    const uint32_t mxl = __vimax3_s16x2(__vimax3_s16x2(lv[0], lv[1], lv[2]), lv[3], lv[3]);
    const uint32_t busy = gt2_mask_nonneg(mxl, thr1) | prev;
    if (__builtin_expect(!__any_sync(0xFFFFFFFFu, busy != 0u), 1)) {
      // outside hits only the un-gated peak tracker moves (peak_time = tover = 0 is rewritten with 0)
      PK1 = __vimax3_s16x2(__vimax3_s16x2(sp[0], sp[1], sp[2]), sp[3], PK1);
      return;
    }
#pragma unroll
    for (int g = 0; g < G; ++g)
      hit_update(sp[g], lv[g], ctx, t0 + g);
    if (ctx.stage->must_flush())
      flush<WIB2_UNITS>(*ctx.stage, ctx.p->sink, ctx.link_base, ctx.link, (ctx.chan0 >> 1) & 31u, false); // whole 32-pair rounds only
  }
};

// =====================================================================================================================
// Packed fast path: FIR matched filter + IQR threshold (wib2/tpg/ProcessAVX2FIR.hpp:21-314), on either frame layout.
// Three frugal trackers per channel (quartiles on the lanes below / above the OLD median, then the median, all with
// L = 10, :108-125), sigma = min(q75 - q25, sigmaMax), s' = min(s - median, adcMax), the 7-tap filter over the ring
// (which excludes the two newest samples, :160-201), threshold sigma * multiplier * threshold, charge += filt >> exponent.
//
// Validity (checked by the host): taps == {1,6,15,20,15,6,1,0}, 1 <= tap_exponent <= 10, sigmaMax * multiplier * threshold
// < 2^16. What makes it fast:
//   * the taps firwin_int(7, 0.1, 64) produces are the binomial row (1+z)^6, so the filter is six cascaded two-tap adders:
//     6 packed adds per tick instead of 7 multiply-adds on a rotating ring, and every add wraps mod 2^16 exactly like the
//     reference's mullo/add chain (ring homomorphism). The carried state stays the reference's ring: it is converted to
//     cascade registers when a link is loaded and back when it is stored, which also removes the ring phase from the loop;
//   * the three trackers keep integer accumulators biased to small non-negative numbers, and the median and q25 live as
//     16385 - value against the biased sample Sb = S - 16384, inside [2, 16405] for every input. q75 can start above the
//     14-bit range (seeded at first sample + 20, up to 16403), so 16385 - q75 reaches -18 and a +-1 step of the low half
//     between 0xFFFF and 0x0000 would carry into the odd channel's half: its low half lives as 49153 - q75 against
//     Sb - 0x8000 instead, inside [32750, 49152] (the high half's carry out of bit 31 is lost, so it keeps 16385 - q75).
//     None of the +-1 steps can then carry between the halves (track() lists the instructions). They replaced fp16x2-subnormal
//     accumulators whose step flags came out of the fp16 pipe, with the two quartile trackers merged into one step or kept
//     separate: both forms measured slower (profiles/r02_integer_accumulators.txt);
//   * sigma is only needed where the threshold is: the quiet test works with a lower bound of the group's sigmas taken from the
//     quartiles after its last tick (sigma moves by at most one per tick, because at most one quartile moves), and the per-tick
//     values are formed from the saved quartile registers only in a group that turns out busy;
//   * while every sigma of the warp is >= 0 the 64-bit-lane product equals the per-channel product (no carries between
//     positions, SURVEY H7) and is one packed IMAD; a warp that sees a negative sigma in a 4-tick group recomputes that
//     group's thresholds with iqr_threshold_exact.
// =====================================================================================================================
struct PackedFirIqr
{
  static constexpr int kGroupUnroll = 2;
  static constexpr bool kNeedsUnitTs = false;
  static constexpr int kWarpsPerSm = 12; // 3 warps per sub-partition: 3 % faster than the 16 its 128 registers allow (same sweep)
  static constexpr int kWib2MinCtas = 5;
  static constexpr int kQuadCtasPerSm = 4; // CTA form, 16 consumer warps per SM (measured: 4 CTAs 29.8 %, 5 CTAs 27.8 %, profiles/r02_fir_forms.txt)
                                           // (64 registers instead of 109; profiles/r01_quad_vs_warp.txt)
  // Mq = 16385 - median, Q25n = 16385 - q25, Q75p = {49153 - q75 (low half), 16385 - q75 (high half)}, A = acc + 10,
  // A25 = acc25 + 10, A75 = acc75 + 11.
  uint32_t Mq, A, Q25n, A25, Q75p, A75;
  uint32_t kM1, kP1; // 0xFFFFFFFF and 1 in registers the compiler cannot see through (KernelParams::all_ones, one)
  static constexpr uint32_t kQ75Bias = 0x4002C002u; // ~q75 + {49154, 16386} = Q75p, and back
  uint32_t d1, d2, d3, d4, d5, d6, o1, o2; // cascade: d_j = previous input of stage j, o1/o2 = previous two outputs
  uint32_t prev, C, Tn;
  uint32_t xmax, sig3max, K, Kneg3, shift, shmask, thr_cfg, mult;

  static __device__ __forceinline__ uint32_t sample(const uint32_t* row, const PairPos& pp) { return extract_pair_biased(row, pp); }
  template<int ROW_WORDS = 28>
  __device__ __forceinline__ void begin_chunk(const uint32_t*, const PairPos&) {}
  template<bool WIB2_UNITS = false>
  __device__ __forceinline__ void finish_link(const TickCtx&) {}
  // fp16-subnormal constants of PackedRsIqrWib2's RS tracker (L = 10)
  static constexpr uint32_t kNegTiny = 0x80018001u; // -2^-24 per half
  static constexpr uint32_t kUp = 0x000B000Bu;      // (L+1) * 2^-24
  static constexpr uint32_t kNegL = 0x800A800Au;    // -L
  static constexpr uint32_t kNegOne = 0xBC00BC00u;

  template<bool WIB2_UNITS>
  static __device__ __forceinline__ void flush(const HitStage& h, const TpSink& k, const uint8_t* link_base, uint32_t link, uint32_t lane,
                                               bool everything = true)
  {
    h.template flush<WIB2_UNITS, true>(k, link_base, link, lane, everything); // FIR hit blocks carry {chan, t, charge, tover} only
  }
  __device__ __forceinline__ void configure(const KernelParams& p)
  {
    mult = 1u << p.tap_exponent;
    const uint32_t adc_max = 32767u / mult;                   // wib2/tpg/ProcessingInfo.hpp:93
    const uint32_t sigma_max = (1u << 15) / (mult * 5u);      // ProcessAVX2FIR.hpp:36
    xmax = adc_max * 0x00010001u;
    sig3max = (sigma_max + 3u) * 0x00010001u;
    thr_cfg = p.threshold;
    K = mult * p.threshold;
    Kneg3 = 0u - 3u * K * 0x00010001u;                        // -(3K, 3K) as ONE 32-bit integer (see threshold())
    shift = uint32_t(p.tap_exponent);
    const uint32_t m = 0xFFFFu >> shift;
    shmask = m | (m << 16);
    kM1 = p.all_ones;
    kP1 = p.one;
  }
  static __device__ __forceinline__ uint32_t to_sm(uint32_t v)
  { // two's complement s16x2 -> sign-magnitude (= bit pattern of value * 2^-24 as fp16), |v| <= 1023; PackedRsIqrWib2's RS tracker
    const uint32_t neg = (v & 0x80008000u) >> 15, m = neg * 0xFFFFu;
    return (add2(v ^ m, neg) & 0x7FFF7FFFu) | (m & 0x80008000u);
  }
  static __device__ __forceinline__ uint32_t from_sm(uint32_t v)
  {
    const uint32_t neg = (v & 0x80008000u) >> 15, m = neg * 0xFFFFu;
    return add2((v & 0x7FFF7FFFu) ^ m, neg);
  }
  __device__ __forceinline__ void cascade(uint32_t x)
  {
    const uint32_t y1 = add2(x, d1), y2 = add2(y1, d2), y3 = add2(y2, d3), y4 = add2(y3, d4), y5 = add2(y4, d5), y6 = add2(y5, d6);
    d1 = x; d2 = y1; d3 = y2; d4 = y3; d5 = y4; d6 = y5;
    o2 = o1;
    o1 = y6;
  }
  // the three trackers and the hit state, HBM form <-> register form (shared by the policies derived from this one)
  __device__ __forceinline__ void load_trackers(const uint32_t* st, uint32_t lane)
  {
    Mq = add2(~st[SV_MEDIAN * 32 + lane], 0x40024002u);       // ~m = -m - 1
    Q25n = add2(~st[SV_Q25 * 32 + lane], 0x40024002u);
    A = add2(st[SV_ACCUM * 32 + lane], 0x000A000Au);
    Q75p = add2(~st[SV_Q75 * 32 + lane], kQ75Bias);
    A25 = add2(st[SV_A25 * 32 + lane], 0x000A000Au);
    A75 = add2(st[SV_A75 * 32 + lane], 0x000B000Bu);
    prev = st[SV_PREV * 32 + lane];
    C = st[SV_CHARGE * 32 + lane];
    Tn = neg2(st[SV_TOVER * 32 + lane]);
  }
  __device__ __forceinline__ void store_trackers(uint32_t* st, uint32_t lane) const
  {
    st[SV_MEDIAN * 32 + lane] = median();
    st[SV_Q25 * 32 + lane] = add2(~Q25n, 0x40024002u);
    st[SV_ACCUM * 32 + lane] = add2(A, 0xFFF6FFF6u);
    st[SV_Q75 * 32 + lane] = add2(~Q75p, kQ75Bias);
    st[SV_A25 * 32 + lane] = add2(A25, 0xFFF6FFF6u);
    st[SV_A75 * 32 + lane] = add2(A75, 0xFFF5FFF5u);
    st[SV_PREV * 32 + lane] = prev;
    st[SV_CHARGE * 32 + lane] = C;
    st[SV_TOVER * 32 + lane] = neg2(Tn);
  }
  __device__ __forceinline__ void load(const uint32_t* st, uint32_t lane, uint32_t flags)
  {
    load_trackers(st, lane);
    // ring -> cascade: replay the ring's 8 samples, oldest first, through an empty cascade (the state only depends on them)
    const uint32_t k = (flags >> 8) & 7u; // next slot to be written = oldest sample
    kphase0 = k;
    d1 = d2 = d3 = d4 = d5 = d6 = o1 = o2 = 0u;
    for (uint32_t i = 0; i < 8; ++i)
      cascade(st[(SV_RING0 + ((k + i) & 7u)) * 32 + lane]);
  }
  __device__ __forceinline__ uint32_t median() const { return add2(~Mq, 0x40024002u); } // 16385 - Mq
  __device__ __forceinline__ void store(uint32_t* st, uint32_t lane, uint32_t k_end) const
  {
    store_trackers(st, lane);
    // cascade -> ring, by running the cascade backwards: with Y[j] = y_j one tick ago (y_0 = the sample itself),
    // y_{j-1}(two ticks ago) = Y[j] - Y[j-1]; every step back in time loses the top stage, and y_0 is the ring entry.
    uint32_t Y[7] = { d1, d2, d3, d4, d5, d6, o1 };
    int top = 6;             // Y[0..top] valid
    uint32_t known_top = o2; // y_6 two ticks ago
#pragma unroll
    for (uint32_t i = 0; i < 8; ++i) {
      st[(SV_RING0 + ((k_end + 7u - i) & 7u)) * 32 + lane] = Y[0]; // sample i+1 ticks ago
      uint32_t Z[7] = {};
#pragma unroll
      for (int jj = 1; jj <= 6; ++jj)
        if (jj <= top)
          Z[jj - 1] = add2(Y[jj], neg2(Y[jj - 1]));
      if (i == 0) { // the column two ticks ago still has its top entry (o2)
        Z[6] = known_top;
      } else {
        top -= 1;
      }
#pragma unroll
      for (int jj = 0; jj < 7; ++jj)
        Y[jj] = Z[jj];
    }
  }
  uint32_t kphase0;
  __device__ __forceinline__ uint32_t phase_after(uint32_t ticks) const { return (kphase0 + ticks) & 7u; }
  // setState: pedestal = first sample, quartiles +-20 (wib2/tpg/ProcessingInfo.hpp:101-141)
  __device__ __forceinline__ void seed(uint32_t Sb) // Sb = ped - 16384
  {
    Mq = add2(~Sb, 0x00020002u);               // 16385 - ped = 1 - Sb
    Q25n = add2(~Sb, 0x00160016u);             // 16385 - (ped - 20)
    Q75p = add2(~Sb, 0xFFEE7FEEu);             // {49153, 16385} - (ped + 20)
  }

  // The three frugal trackers of one tick (Sb = raw - 16384). Returns 16385 - median, updated: see sp1_of / clamped_sample.
  // A frugal accumulator stays in [-10, 10] between ticks, so biased by +10 it is a small NON-NEGATIVE number in each half, and so
  // are the sign codes {0,1,2}: sums of such values are plain 32-bit adds (IADD3 issues on either pipe at twice the rate of the
  // packed-16x2 and fp16x2 instructions) because nothing carries between the halves. One tracker step is
  //     U = B + sign + 1                      acc' + 11 in [0, 22]                                         IADD3
  //     c = clamp(U - 1, 0, 20)               acc' + 10 without the two step values                        VIADDMNMX.RELU
  //     D = U - 1 - c                         the step, -1 / 0 / +1 per half, as ONE 32-bit integer        IADD3
  //     B = c - 10 D  (or U - 11 D)           back to 10 (11) where it stepped                             IMAD
  //     Q = Q - D                             16385 - quantile follows                                     IADD3
  // D is a "true integer" d_hi * 65536 + d_lo whose low half may be negative (its bit pattern then borrows from the high half);
  // that is harmless because only LINEAR 32-bit operations consume it and every result they produce has non-negative halves
  // again, for which the 32-bit value and the packed value coincide — provided Q's low half stays clear of 0xFFFF / 0x0000, which
  // is why q75's low half has its own bias (Q75p) and meets the sample as Sb - 0x8000 (one more IMAD per tick). The quartile
  // enables (:119-121: sample below / above the OLD median) cost no select: the clamp's upper bound is 2 on the enabled halves and
  // 0 elsewhere, which turns the sign code into 0 there, and the missing +1 comes from n1 (q25, "+10" form) or is taken back out
  // by g1 (q75, "+11" form).
  // Per tick: 8 ALU-pipe instructions (sign tests, clamps, enables), 4-5 on the FMA pipe, 10 adds that go to whichever is free
  // — against 13 / 8 / 2 for the fp16-subnormal form with merged quartile trackers and 9 / 14 / 3 with separate ones. The
  // three-input adds stay IADD3s: as two IMADs each on the FMA pipe they gained nothing (profiles/r02_fma_steering_probe.txt, u3).
  __device__ __forceinline__ uint32_t track(uint32_t Sb)
  {
    const uint32_t sg1 = addclamp2(Sb, Mq, 0x00020002u);              // sign(raw - median) + 1, OLD median   (:108-117)
    // q25 on the halves below the OLD median (:119)
    const uint32_t n1 = min2(sg1, 0x00010001u);                       // 0 where below, 1 elsewhere
    const uint32_t s25 = addclamp2(Sb, Q25n, n1 * (kM1 + kM1) + 0x00020002u); // bound 2 - 2 n1 (IMAD): sign(raw - q25) + 1 where enabled, else 0
    const uint32_t U25 = A25 + s25 + n1;                              // acc25' + 11
    const uint32_t c25 = addclamp2(U25, kM1, 0x00140014u);
    const uint32_t D25 = U25 - c25 - 0x00010001u;
    A25 = c25 - 10u * D25;
    Q25n = fma_sub(Q25n, D25, kM1);
    // q75 on the halves above it (:121)
    const uint32_t g1 = __viaddmax_s16x2_relu(sg1, kM1, 0u);          // 1 where above, 0 elsewhere
    const uint32_t Sb75 = fma_add(Sb, 0xFFFF8000u, kP1);             // low half S - 49152 (0xC000 | S - 0x8000: no borrow)
    const uint32_t s75 = addclamp2(Sb75, Q75p, fma_add(g1, g1, kP1)); // bound 2 g1: sign(raw - q75) + 1 where enabled, else 0
    const uint32_t U75 = A75 + s75 - g1;                              // acc75' + 11
    const uint32_t c75 = addclamp2(U75, kM1, 0x00140014u);
    const uint32_t D75 = U75 - c75 - 0x00010001u;
    A75 = U75 - 11u * D75;
    Q75p = fma_sub(Q75p, D75, kM1);
    // median (:125)
    const uint32_t U = fma_add(sg1, A, kP1);
    const uint32_t cm = addclamp2(U, kM1, 0x00140014u);
    const uint32_t D = U - cm - 0x00010001u;
    A = cm - 10u * D;
    Mq = fma_sub(Mq, D, kM1);
    return Mq;
  }
  // min(q75 - q25, sigmaMax) + 3 (:131-134) from a pair of quartile registers (Q75p, Q25n)
  __device__ __forceinline__ uint32_t sig3_of(uint32_t q75p, uint32_t q25n) const
  {
    return addmin2(add2(~q75p, 0x00048004u), q25n, sig3max);          // -(16385 - q75) + 3 = ~Q75p + {32772, 4}
  }
  // One tick: returns the filter output of this tick.
  // s' + 1 = raw - median + 1 from what track() returns
  static __device__ __forceinline__ uint32_t sp1_of(uint32_t Sb, uint32_t tr)
  {
    return add2(Sb, tr);
  }
  // min(raw - median, adcMax) (:128,142) from what track() returns
  __device__ __forceinline__ uint32_t clamped_sample(uint32_t Sb, uint32_t tr) const
  {
    return addmin2(Sb, fma_add(tr, 0xFFFEFFFFu, kP1), xmax);         // tr = 16385 - median >= 2: the -1 is a plain 32-bit add
  }
  __device__ __forceinline__ uint32_t tick(uint32_t Sb)
  {
    const uint32_t x = clamped_sample(Sb, track(Sb));
    const uint32_t filt = o2;                                         // window = samples t-8 .. t-2          (:160-201)
    cascade(x);
    return filt;
  }
  // sigma * multiplier * threshold for sigma >= 0: (sig3 - 3) * K per half, as one 32-bit multiply-add — no carry crosses
  // the halves because each half of sig3 * K is >= 3K and < 2^16 + 3K... the host checks (sigmaMax + 3) * K < 2^16.
  __device__ __forceinline__ uint32_t threshold(uint32_t sig3) const { return sig3 * K + Kneg3; }

  template<bool EXACT>
  __device__ __forceinline__ void hit_update(uint32_t filt, uint32_t thr, const TickCtx& ctx, int t)
  {
    uint32_t over;
    if constexpr (EXACT) // any threshold value: plain signed compares
      over = (lo16s(filt) > lo16s(thr) ? 0xFFFFu : 0u) | (hi16s(filt) > hi16s(thr) ? 0xFFFF0000u : 0u);
    else
      over = gt2_mask_bf16(max2(filt, 0u), thr);          // 0 <= thr <= 32640                        (:208)
    const uint32_t left = prev & ~over;                   //                                           (:210)
    uint32_t add;
    if constexpr (EXACT)
      add = pack2((lo16s(filt & over)) >> shift, (hi16s(filt & over)) >> shift);
    else
      add = ((filt & over) >> shift) & shmask;            // over => filt > thr >= 0: arithmetic == logical shift (:221-223)
    if constexpr (EXACT)
      C = pack2(sat16(lo16s(C) + lo16s(add)), sat16(hi16s(C) + hi16s(add)));
    else
      C = minu2(add2(C, add), 0x7FFF7FFFu);               // adds_epi16 of two non-negative halves
    Tn = addmax2(Tn, over, 0x80018001u);                  // tover = adds(tover, 1)                    (:236-237)
    prev = over;
    if (left != 0u) {                                     //                                           (:251-281)
      // accepted iff hit_charge != 0 (src/wib2/WIB2FrameProcessor.cpp:429): decided in flush on the masked charge
      ctx.stage->push(HitStage::meta(ctx.chan0, ctx.unit, uint32_t(t)), C & left, neg2(Tn));
      C &= ~left;
      Tn &= ~left;
    }
  }

  // Quiet test and hit bookkeeping of one 4-tick group, given its filter outputs and the quartile registers after each tick.
  template<int G, bool WIB2_UNITS>
  __device__ __forceinline__ void finish_group(const uint32_t (&filt)[G], const uint32_t (&q75v)[G], const uint32_t (&q25v)[G], const TickCtx& ctx,
                                               int t0)
  {
    // Conservative quiet test: the largest filter output of the group against the threshold of a LOWER BOUND of its sigmas.
    // At most one quartile moves per tick, by one, so every sigma of the group is >= sigma(last tick) - 3.
    const uint32_t mx = __vimax3_s16x2(__vimax3_s16x2(filt[0], filt[1], filt[2]), filt[3], 0u);
    const uint32_t lo3 = add2(sig3_of(q75v[G - 1], q25v[G - 1]), 0xFFFDFFFDu); // (bound of min(sigma, sigmaMax)) + 3
    uint32_t neg = addmin2(lo3, 0xFFFDFFFDu, 0u);        // non-zero <=> the bound is negative: some sigma MAY be below zero
    if (ctx.p->debug_flags & 1u)
      neg = 0xFFFFFFFFu;
    const uint32_t busy = gt2_mask_bf16(mx, threshold(lo3)) | prev | neg;
    if (__builtin_expect(!__any_sync(0xFFFFFFFFu, busy != 0u), 1))
      return; // nothing but the trackers and the filter moves outside hits
    uint32_t sig3[G];
#pragma unroll
    for (int g = 0; g < G; ++g)
      sig3[g] = sig3_of(q75v[g], q25v[g]);
    const uint32_t smin = __vimin3_s16x2(__vimin3_s16x2(sig3[0], sig3[1], sig3[2]), sig3[3], sig3[3]);
    uint32_t really_neg = addmin2(smin, 0xFFFDFFFDu, 0u); // min(sigma, 0) of the group: non-zero <=> some sigma < 0
    if (ctx.p->debug_flags & 1u)
      really_neg = 0xFFFFFFFFu;
    if (__any_sync(0xFFFFFFFFu, really_neg != 0u)) { // rare: carries between the positions of a 64-bit lane (H7)
#pragma unroll
      for (int g = 0; g < G; ++g) {
        const uint32_t th = iqr_threshold_exact(add2(sig3[g], 0xFFFDFFFDu), (ctx.chan0 >> 1) & 31u, int(mult), thr_cfg);
        hit_update<true>(filt[g], th, ctx, t0 + g);
      }
    } else {
#pragma unroll
      for (int g = 0; g < G; ++g)
        hit_update<false>(filt[g], threshold(sig3[g]), ctx, t0 + g);
    }
    if (ctx.stage->must_flush())
      flush<WIB2_UNITS>(*ctx.stage, ctx.p->sink, ctx.link_base, ctx.link, (ctx.chan0 >> 1) & 31u, false); // whole 32-pair rounds only
  }

  template<int G, bool DUMP, int ROW_WORDS = 28, bool WIB2_UNITS = false>
  __device__ __forceinline__ void group(const uint32_t* rows, const PairPos& pp, const TickCtx& ctx, int t0, uint32_t* ped_out,
                                        uint32_t* wav_out, bool /*more*/)
  {
    static_assert(G == 4, "trees below are written for 4 ticks");
    uint32_t filt[G], q75v[G], q25v[G];
#pragma unroll
    for (int g = 0; g < G; ++g) {
      filt[g] = tick(extract_pair_biased(rows + g * ROW_WORDS, pp));
      q75v[g] = Q75p;
      q25v[g] = Q25n;
      if constexpr (DUMP) {
        ped_out[g] = median();
        wav_out[g] = filt[g];
      }
    }
    finish_group<G, WIB2_UNITS>(filt, q75v, q25v, ctx, t0);
  }
};

// =====================================================================================================================
// Packed FIR + IQR for ARBITRARY taps (any int16 taps[0..6], e.g. firwin_int at another multiplier, or a user-supplied filter):
// same trackers, threshold and hit bookkeeping as PackedFirIqr, but the filter is the reference's multiply-add chain
//   filt = sum_{j<7} taps[j] * prev_samp[(j + k) % 8]        (mullo_epi16 / add_epi16, mod 2^16; ProcessAVX2FIR.hpp:160-201)
// on a window of the last 8 clamped samples held in registers, oldest first (w[0] = s(t-8) ... w[7] = s(t-1); the ring phase
// only matters when the state is loaded and stored). Products are 32-bit IMADs whose low 16 bits are the wrapped result, so
// the packed register itself is the low-half operand; a half-swapped copy of every window entry serves the high half.
// 14 IMAD + 2 PRMT per tick instead of the binomial cascade's 6 adds.
// =====================================================================================================================
struct PackedFirIqrAnyTaps : PackedFirIqr
{
  static constexpr int kQuadCtasPerSm = 4; // CTA form, 16 consumer warps per SM: 6 % faster than one warp per CTA
  uint32_t w[8], ws[8]; // window and its half-swapped twin
  int tap[7];

  __device__ __forceinline__ void configure(const KernelParams& p)
  {
    PackedFirIqr::configure(p);
#pragma unroll
    for (int j = 0; j < 7; ++j)
      tap[j] = p.taps[j];
  }
  static __device__ __forceinline__ uint32_t swap_halves(uint32_t v) { return __byte_perm(v, v, 0x1032); }
  __device__ __forceinline__ void load(const uint32_t* st, uint32_t lane, uint32_t flags)
  {
    load_trackers(st, lane);
    const uint32_t k = (flags >> 8) & 7u; // next slot to be written = oldest sample
    kphase0 = k;
#pragma unroll
    for (uint32_t i = 0; i < 8; ++i) {
      w[i] = st[(SV_RING0 + ((k + i) & 7u)) * 32 + lane];
      ws[i] = swap_halves(w[i]);
    }
  }
  __device__ __forceinline__ void store(uint32_t* st, uint32_t lane, uint32_t k_end) const
  {
    store_trackers(st, lane);
#pragma unroll
    for (uint32_t i = 0; i < 8; ++i)
      st[(SV_RING0 + ((k_end + i) & 7u)) * 32 + lane] = w[i]; // w[0] is the oldest = the slot written next
  }
  __device__ __forceinline__ uint32_t tick(uint32_t Sb)
  {
    const uint32_t x = clamped_sample(Sb, track(Sb));
    int lo = 0, hi = 0;
#pragma unroll
    for (int j = 0; j < 7; ++j) {
      lo += tap[j] * int(w[j]);   // low 16 bits: taps[j] * (low half), any upper bits are discarded below
      hi += tap[j] * int(ws[j]);
    }
    const uint32_t filt = __byte_perm(uint32_t(lo), uint32_t(hi), 0x5410);
#pragma unroll
    for (int j = 0; j < 7; ++j) {
      w[j] = w[j + 1];
      ws[j] = ws[j + 1];
    }
    w[7] = x;
    ws[7] = swap_halves(x);
    return filt;
  }

  template<int G, bool DUMP, int ROW_WORDS = 28, bool WIB2_UNITS = false>
  __device__ __forceinline__ void group(const uint32_t* rows, const PairPos& pp, const TickCtx& ctx, int t0, uint32_t* ped_out,
                                        uint32_t* wav_out, bool /*more*/)
  {
    static_assert(G == 4, "trees below are written for 4 ticks");
    uint32_t filt[G], q75v[G], q25v[G];
#pragma unroll
    for (int g = 0; g < G; ++g) {
      filt[g] = tick(extract_pair_biased(rows + g * ROW_WORDS, pp));
      q75v[g] = Q75p;
      q25v[g] = Q25n;
      if constexpr (DUMP) {
        ped_out[g] = median();
        wav_out[g] = filt[g];
      }
    }
    finish_group<G, WIB2_UNITS>(filt, q75v, q25v, ctx, t0);
  }
};

// =====================================================================================================================
// Packed fast path: WIB2 AbsRS (wib2/tpg/ProcessRSAVX2.hpp:24-330) — the IQR threshold of the FIR finder applied to an absolute
// running sum. Per tick and channel:
//   quartile / median trackers exactly as PackedFirIqr (every limit 10, :100-126);  s' = raw - median
//   RS = mulhrs(RS * 8 + |s'| * 5, 32768/10)      literal factors (:29-33,:137-150), mullo / add mod 2^16
//   RS -= median_RS after a frugal update of median_RS with RS (:152-159)
//   sigma = min(q75 - q25, sigmaMax), sigmaMax = 2^15 / (multiplier * threshold) (:36);  over = RS > sigma * threshold (:198)
//   charge = adds(charge, (over ? adds(RS, median_RS) : 0) >> tap_exponent) (:210-213);  tover = adds(tover, over)
// |RS before subtraction| <= 3277 (mulhrs of a 16-bit value by 3276), so adds(RS, median_RS) is that value again and never
// saturates. The threshold is one packed IMAD while every sigma of the warp is >= 0 (as in PackedFirIqr); a group that sees a
// negative sigma recomputes it with the reference's 4 x int64-lane semantics. Validity (checked by the host):
// 1 <= tap_exponent <= 10, threshold >= 1, (sigmaMax + 3) * threshold < 2^16.
// =====================================================================================================================
struct PackedRsIqrWib2 : PackedFirIqr
{
  static constexpr int kGroupUnroll = 1;
  static constexpr int kWib2MinCtas = 1;
  uint32_t RS1, MRq, AR; // RS + 1 (after median subtraction); 1 - median_RS; (acc_RS - 1) as fp16 subnormal

  __device__ __forceinline__ void configure(const KernelParams& p)
  {
    PackedFirIqr::configure(p);
    const uint32_t sigma_max = (1u << 15) / (mult * p.threshold); // ProcessRSAVX2.hpp:36
    sig3max = (sigma_max + 3u) * 0x00010001u;
    K = p.threshold;                                             // sigma * info.threshold: no multiplier (:198)
    Kneg3 = 0u - 3u * K * 0x00010001u;
  }
  __device__ __forceinline__ void load(const uint32_t* st, uint32_t lane, uint32_t)
  {
    load_trackers(st, lane);
    RS1 = add2(st[SV_RS * 32 + lane], 0x00010001u);
    MRq = add2(~st[SV_MED_RS * 32 + lane], 0x00020002u);
    AR = to_sm(add2(st[SV_ACC_RS * 32 + lane], 0xFFFFFFFFu));
    kphase0 = 0;
  }
  __device__ __forceinline__ void store(uint32_t* st, uint32_t lane, uint32_t) const
  {
    store_trackers(st, lane);
    st[SV_RS * 32 + lane] = add2(RS1, 0xFFFFFFFFu);
    st[SV_MED_RS * 32 + lane] = add2(~MRq, 0x00020002u);
    st[SV_ACC_RS * 32 + lane] = add2(from_sm(AR), 0x00010001u);
  }
  __device__ __forceinline__ uint32_t phase_after(uint32_t) const { return 0; }

  // One tick: sp1 = s' + 1. Returns RS - median_RS + 1 and, in `raw_rs`, the running sum before the subtraction.
  __device__ __forceinline__ uint32_t rs_step(uint32_t sp1, uint32_t& raw_rs)
  {
    const uint32_t x = add2(sp1, 0xFFFFFFFFu);
    const uint32_t ax = max2(x, neg2(x));                                     // |s'|
    // low 16 bits per half: RS * 8 + |s'| * 5, with RS = RS1 - 1 (the packed registers serve as low-half operands)
    const uint32_t lo = uint32_t(int(RS1) * 8 + (int(ax) * 5 - 8));
    const uint32_t hi = uint32_t(int(RS1 >> 16) * 8 + (int(ax >> 16) * 5 - 8));
    const int r_lo = PackedRsWibEth<false>::mulhrs_low(lo), r_hi = PackedRsWibEth<false>::mulhrs_low(hi);
    raw_rs = __byte_perm(uint32_t(r_lo), uint32_t(r_hi), 0x5410);
    // frugal update of median_RS with the new running sum (limit 10), then subtract
    const uint32_t sg1 = addclamp2(raw_rs, MRq, 0x00020002u);
    const uint32_t T = hadd2_bits(AR, sg1);
    const uint32_t upm = eq2_mask(T, kUp);
    const uint32_t dn1 = hfma2_sat_bits(T, kNegOne, kNegL);
    AR = hfma2_bits(ne2_abs_one(T, kUp), T, kNegTiny);
    MRq = add2(add2(MRq, upm), dn1);
    RS1 = add2(raw_rs, MRq);
    return RS1;
  }

  template<bool EXACT>
  __device__ __forceinline__ void hit_update(uint32_t lv1, uint32_t raw_rs, uint32_t thr, const TickCtx& ctx, int t)
  {
    const uint32_t lv = add2(lv1, 0xFFFFFFFFu);
    uint32_t over;
    if constexpr (EXACT)
      over = (lo16s(lv) > lo16s(thr) ? 0xFFFFu : 0u) | (hi16s(lv) > hi16s(thr) ? 0xFFFF0000u : 0u);
    else
      over = gt2_mask_bf16(max2(lv, 0u), thr);            // 0 <= thr <= 32640                        (:198-200)
    const uint32_t left = prev & ~over;
    // (over ? adds(RS, median_RS) : 0) >> tap_exponent, arithmetic per half (the sum may be negative): offset-binary trick
    const uint32_t u = (add2(raw_rs & over, 0x80008000u) >> shift) & shmask;
    const uint32_t bias = (0x8000u >> shift) * 0x00010001u;
    const uint32_t add = add2(u, neg2(bias));
    const uint32_t Cw = add2(C, add);                     // adds_epi16: wrapping add + repair of the rare overflowing halves
    const uint32_t ovf = ~(C ^ add) & (C ^ Cw) & 0x80008000u;
    if (__builtin_expect(ovf != 0u, 0))
      C = pack2(sat16(lo16s(C) + lo16s(add)), sat16(hi16s(C) + hi16s(add)));
    else
      C = Cw;
    Tn = addmax2(Tn, over, 0x80018001u);                  // tover = adds(tover, 1)
    prev = over;
    if (left != 0u) {
      // accepted iff hit_charge != 0 (src/wib2/WIB2FrameProcessor.cpp:429): decided in flush on the masked charge
      ctx.stage->push(HitStage::meta(ctx.chan0, ctx.unit, uint32_t(t)), C & left, neg2(Tn));
      C &= ~left;
      Tn &= ~left;
    }
  }

  template<int G, bool DUMP, int ROW_WORDS = 28, bool WIB2_UNITS = false>
  __device__ __forceinline__ void group(const uint32_t* rows, const PairPos& pp, const TickCtx& ctx, int t0, uint32_t* ped_out,
                                        uint32_t* wav_out, bool /*more*/)
  {
    static_assert(G == 4, "trees below are written for 4 ticks");
    uint32_t lv[G], rs[G], sig3[G];
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const uint32_t Sb = extract_pair_biased(rows + g * ROW_WORDS, pp);
      lv[g] = rs_step(sp1_of(Sb, track(Sb)), rs[g]);
      sig3[g] = sig3_of(Q75p, Q25n);
      if constexpr (DUMP) {
        ped_out[g] = median();
        wav_out[g] = add2(lv[g], 0xFFFFFFFFu);
      }
    }
    // conservative quiet test: largest RS of the group (biased by one: still conservative) vs the threshold of its smallest sigma
    const uint32_t mx = __vimax3_s16x2(__vimax3_s16x2(lv[0], lv[1], lv[2]), lv[3], 0u);
    const uint32_t smin = __vimin3_s16x2(__vimin3_s16x2(sig3[0], sig3[1], sig3[2]), sig3[3], sig3[3]);
    uint32_t neg = addmin2(smin, 0xFFFDFFFDu, 0u); // min(sigma, 0) of the group: non-zero <=> some sigma < 0
    if (ctx.p->debug_flags & 1u)
      neg = 0xFFFFFFFFu;
    const uint32_t busy = gt2_mask_bf16(mx, threshold(smin)) | prev | neg;
    if (__builtin_expect(!__any_sync(0xFFFFFFFFu, busy != 0u), 1))
      return; // nothing but the trackers and the running sum moves outside hits
    if (__any_sync(0xFFFFFFFFu, neg != 0u)) { // rare: carries between the positions of a 64-bit lane (H7)
#pragma unroll
      for (int g = 0; g < G; ++g) {
        const uint32_t th = iqr_threshold_exact(add2(sig3[g], 0xFFFDFFFDu), (ctx.chan0 >> 1) & 31u, 1, thr_cfg);
        hit_update<true>(lv[g], rs[g], th, ctx, t0 + g);
      }
    } else {
#pragma unroll
      for (int g = 0; g < G; ++g)
        hit_update<false>(lv[g], rs[g], threshold(sig3[g]), ctx, t0 + g);
    }
    if (ctx.stage->must_flush())
      flush<WIB2_UNITS>(*ctx.stage, ctx.p->sink, ctx.link_base, ctx.link, (ctx.chan0 >> 1) & 31u, false); // whole 32-pair rounds only
  }
};

// =====================================================================================================================
// What the three kernels share: a link's place in the batch, the shared-memory layout, and the consumer side of a work item
// (its close, the cursor re-arm). Each kernel keeps its own producer and hand-out logic, and its own chunk step (seed, group
// loop, debug dumps): as one shared function it changed ptxas's register allocation of the one-warp-per-CTA kernel (92 -> 94
// registers for the production policy) and of the WIB2 kernel. For the same reason the one-warp-per-CTA kernel also writes out
// its hit-staging placement and cursor re-arm; every instance compiles to the same SASS as with them written out per kernel.
// =====================================================================================================================
__device__ __forceinline__ uint32_t
units_of(const KernelParams& p, uint32_t link)
{
  return p.n_units ? p.n_units[link] : p.units_stride;
}
template<uint32_t UNIT_BYTES> // a WIBEth frame or a WIB2 superchunk
__device__ __forceinline__ const uint8_t*
base_of(const KernelParams& p, uint32_t link)
{
  return p.frames + size_t(link) * p.units_stride * UNIT_BYTES;
}

// Dynamic shared memory of one CTA: [stages | mbarriers | hit staging (16 B + 4 B per record) of each consumer warp | hit
// counters | link FIFO].
template<size_t STAGE_BYTES, size_t BAR_BYTES, int HIT_WARPS, size_t FIFO_BYTES>
struct SmemLayout
{
  static constexpr size_t align16(size_t x) { return (x + 15) & ~size_t(15); }
  static constexpr size_t bars = align16(STAGE_BYTES);
  static constexpr size_t hits = align16(bars + BAR_BYTES);
  static constexpr size_t aux = hits + size_t(HIT_WARPS) * HitStage::kCap * 16;
  static constexpr size_t counts = aux + size_t(HIT_WARPS) * HitStage::kCap * 4;
  static constexpr size_t fifo = align16(counts + size_t(HIT_WARPS) * 4);
  static constexpr size_t total = fifo + FIFO_BYTES;

  static __device__ __forceinline__ void place_hits(HitStage& h, uint8_t* smem, uint32_t warp)
  {
    h.buf = reinterpret_cast<uint4*>(smem + hits) + size_t(warp) * HitStage::kCap;
    h.aux = reinterpret_cast<uint32_t*>(smem + aux) + size_t(warp) * HitStage::kCap;
    h.cnt = reinterpret_cast<uint32_t*>(smem + counts) + warp;
  }
};

// End of a work item: drain the policy's software pipeline, flush the staged hits (records carry unit indices of THIS link),
// store the state of 64-channel group `group` and its FIR ring phase after `ticks` ticks.
template<bool WIB2_UNITS, class Algo>
__device__ __forceinline__ void
close_item(Algo& algo, const TickCtx& ctx, const HitStage& hits, uint32_t* st, uint32_t group, uint32_t ticks, uint32_t lane)
{
  const KernelParams& p = *ctx.p;
  algo.template finish_link<WIB2_UNITS>(ctx);
  Algo::template flush<WIB2_UNITS>(hits, p.sink, ctx.link_base, ctx.link, lane);
  const uint32_t k_end = algo.phase_after(ticks);
  algo.store(st, lane, k_end);
  if (lane == 0)
    p.group_flags[group] = kFlagInitialized | (k_end << 8);
}

// One lane of each of the launch's `participants` calls this after its last claim: the last one out re-arms the cursor for the
// next launch (launches of one handle are stream-ordered: state is carried).
__device__ __forceinline__ void
rearm_cursor(const KernelParams& p, uint32_t participants)
{
  __threadfence();
  if (atomicAdd(p.link_cursor + 1, 1u) == participants - 1u) {
    p.link_cursor[0] = 0u;
    p.link_cursor[1] = 0u;
  }
}

// Ring of both WIBEth forms: 2 stages of 32 ticks per link (7 KB). Measured best on B200 (profiles/r01_geometry_sweep.txt): the
// kernels are issue-bound, so deeper rings do not help.
constexpr int kWibEthRowBytes = 112;
constexpr int kWibEthStages = 2, kWibEthChunkTicks = 32;
constexpr uint32_t kWibEthChunkBytes = kWibEthRowBytes * kWibEthChunkTicks;
constexpr uint32_t kWibEthChunksPerUnit = 64 / kWibEthChunkTicks;
static_assert(64 % kWibEthChunkTicks == 0, "chunk must divide the frame");

// =====================================================================================================================
// WIBEth kernel: persistent single-warp CTAs, one link (64 channels) at a time per warp, private TMA ring of chunk stages.
// Warp w of the grid starts on link w; every further link is CLAIMED from a global cursor when the warp's producer runs
// out of chunks, so links go to whichever warp is free first: a warp that shares its SM sub-partition with one more
// neighbour, or that drew longer links in a ragged batch, simply takes fewer of them. The ring is refilled by lane 0 from
// a producer cursor that runs kWibEthStages chunks ahead of the consumer ACROSS link boundaries, so a warp never drains its
// pipeline between links; the producer hands the links it chose to the consumer through a small warp-uniform FIFO. Single-warp
// CTAs let the block scheduler spread the resident warps evenly over an SM's four sub-partitions.
// =====================================================================================================================
constexpr uint32_t kWibEthFifo = 8; // links in flight; power of two; in shared memory so the tick loop carries no registers for it
using WibEthSmem = SmemLayout<size_t(kWibEthStages) * kWibEthChunkBytes, size_t(kWibEthStages) * 8, 1, kWibEthFifo * 4>;

// Whole warp: wait until *counter == want (acquire: what the publishing warp stored before its release is visible afterwards).
__device__ __noinline__ void
wait_for_slices(const uint32_t* counter, uint32_t want)
{
  uint32_t seen;
  for (;;) {
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(counter) : "memory");
    if (__all_sync(0xFFFFFFFFu, seen == want))
      break;
    __nanosleep(200);
  }
}

template<class Algo, bool DUMP>
__global__ void __launch_bounds__(32, 1)
wibeth_kernel(const KernelParams p)
{
  constexpr int NSTAGE = kWibEthStages;
  constexpr uint32_t kChunkBytes = kWibEthChunkBytes, kChunksPerUnit = kWibEthChunksPerUnit;
  extern __shared__ __align__(128) uint8_t smem[];

  // the warp's index (0) through a shuffle: without it ptxas allocates the tick loop's registers differently (92 -> 94 for the
  // production policy)
  const uint32_t warp = __shfl_sync(0xFFFFFFFFu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31u;
  const uint32_t warps_total = gridDim.x;
  const uint32_t first_link = blockIdx.x + warp; // this warp's first work item
  const uint32_t n_items = p.n_links << p.parts_log2;
  if (first_link >= n_items)
    return;

  uint8_t* stages = smem + size_t(warp) * NSTAGE * kChunkBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + WibEthSmem::bars) + warp * NSTAGE;
  HitStage hits;
  hits.buf = reinterpret_cast<uint4*>(smem + WibEthSmem::hits) + size_t(warp) * HitStage::kCap;
  hits.aux = reinterpret_cast<uint32_t*>(smem + WibEthSmem::aux) + size_t(warp) * HitStage::kCap;
  hits.cnt = reinterpret_cast<uint32_t*>(smem + WibEthSmem::counts) + warp;

  // Producer cursor: the next chunk to request is pr_src; pr_left chunks remain in link pr_link. Every lane keeps the same
  // (warp-uniform) copy, so the bookkeeping runs on the uniform datapath; only lane 0 talks to the mbarrier / copy engine
  // and to the global link cursor.
  // FIFO of links the producer has started and the consumer has not: the producer is at most NSTAGE chunks ahead and every
  // link it starts has >= kChunksPerUnit chunks, so at most ceil(NSTAGE / kChunksPerUnit) + 1 links are in flight.
  static_assert((NSTAGE + kChunksPerUnit - 1) / kChunksPerUnit + 1 <= kWibEthFifo, "link FIFO too short for this ring geometry");
  volatile uint32_t* fifo = reinterpret_cast<volatile uint32_t*>(smem + WibEthSmem::fifo) + warp * kWibEthFifo;
  uint32_t fifo_head = 0, fifo_n = 0;
  auto fifo_push = [&](uint32_t link) { // whole warp, converged; every lane holds the same `link`
    if (lane == 0)
      fifo[(fifo_head + fifo_n) & (kWibEthFifo - 1u)] = link;
    ++fifo_n;
    __syncwarp();
  };
  auto fifo_pop = [&]() -> uint32_t {
    const uint32_t link = fifo[fifo_head];
    fifo_head = (fifo_head + 1u) & (kWibEthFifo - 1u);
    --fifo_n;
    return link;
  };
  // Work items: item i = slice (i / n_links) of the group's link (i % n_links); slice k of a link with n units is its units
  // [k n >> parts_log2, (k + 1) n >> parts_log2), or, with slice_geom, halving slices (what the launch's last round leaves idle is
  // at most one LAST slice, so small last slices shorten the tail without more state round trips per link). Items are claimed
  // in increasing order, so every first slice is handed out before any second one.
  auto slice_of = [&](uint32_t item, uint32_t& link, uint32_t& u0, uint32_t& u1) -> uint32_t { // returns the slice number
    uint32_t part = 0;
    link = item;
    while (link >= p.n_links) { // at most 7 rounds; warp-uniform
      link -= p.n_links;
      ++part;
    }
    if (p.link_ids != nullptr) // one configuration group of several: its (item mod n_links)-th link
      link = p.link_ids[link];
    const uint32_t n = units_of(p, link);
    if (p.slice_geom) { // halving slices: n/2, n/4, ... and the rest (slice k starts ceil(n / 2^k) units before the end)
      u0 = n - ((n + (1u << part) - 1u) >> part);
      u1 = part + 1u == (1u << p.parts_log2) ? n : n - ((n + (2u << part) - 1u) >> (part + 1u));
    } else {
      u0 = (part * n) >> p.parts_log2;
      u1 = ((part + 1u) * n) >> p.parts_log2;
    }
    return part;
  };
  // How many of the slices before `part` hold units (with fewer units than slices some are empty and never run). Equal slices:
  // below one unit per slice every non-empty one holds exactly one, so u0 of them; halving slices: slice k < last is empty
  // unless n > 2^k. The last slice is never empty in either scheme (it re-arms the link's counter).
  auto slices_before = [&](uint32_t link, uint32_t part, uint32_t u0) -> uint32_t {
    if (!p.slice_geom)
      return min(part, u0);
    const uint32_t n = units_of(p, link);
    return min(part, n > 1u ? 32u - uint32_t(__clz(int(n - 1u))) : 0u);
  };
  // same value in every lane -> uniform register, so that the producer's per-chunk bookkeeping stays on the uniform datapath
  auto uniform = [](uint32_t v) { return __reduce_max_sync(0xFFFFFFFFu, v); };
  bool pr_done = false; // the cursor has run past the last item
  uint32_t pr_left = 0, pr_in_unit = 0, pr_slot = 0;
  const uint8_t* pr_src = nullptr;
  auto pr_start = [&](uint32_t item) { // point the producer at an item (pr_left stays 0 if it is empty)
    uint32_t link, u0, u1;
    slice_of(item, link, u0, u1);
    pr_left = uniform((u1 - u0) * kChunksPerUnit);
    if (pr_left != 0) {
      fifo_push(item);
      pr_src = base_of<SWTPG_WIBETH_FRAME_BYTES>(p, uniform(link)) + size_t(uniform(u0)) * SWTPG_WIBETH_FRAME_BYTES + 32;
      pr_in_unit = 0;
    }
  };
  auto claim = [&]() -> uint32_t { // next unclaimed item (items 0 .. warps_total-1 are the warps' first ones)
    uint32_t k = 0;
    if (lane == 0)
      k = atomicAdd(p.link_cursor, 1u);
    return warps_total + __reduce_add_sync(0xFFFFFFFFu, k); // REDUX: the result lands in a uniform register
  };
  pr_start(first_link);
  auto produce = [&]() { // request one more chunk, if any item is left for this warp (whole warp calls, converged)
    if (__builtin_expect(pr_left == 0, 0)) { // item exhausted (or empty): claim the next one that has data
      if (pr_done)
        return;
      do {
        const uint32_t item = claim();
        if (item >= n_items) {
          pr_done = true;
          return;
        }
        pr_start(item);
      } while (pr_left == 0);
    }
    if (elect_one()) {
      mbar_arrive_expect_tx(&bars[pr_slot], kChunkBytes);
      bulk_g2s(stages + pr_slot * kChunkBytes, pr_src, kChunkBytes, &bars[pr_slot]);
    }
    pr_slot = pr_slot + 1 == NSTAGE ? 0 : pr_slot + 1;
    pr_src += kChunkBytes;
    if (++pr_in_unit == kChunksPerUnit) { // skip the 32 header bytes of the next frame
      pr_in_unit = 0;
      pr_src += 32;
    }
    --pr_left;
  };

  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < NSTAGE; ++s)
      mbar_init(&bars[s], 1);
    *hits.cnt = 0u;
    fence_mbar_init();
  }
  __syncwarp();
  for (int s = 0; s < NSTAGE; ++s)
    produce();

  Algo algo;
  algo.configure(p);
  const PairPos pp = pair_pos(lane);
  TickCtx ctx;
  ctx.p = &p;
  ctx.chan0 = 2 * lane;
  ctx.ts = 0;
  ctx.stage = &hits;

  uint32_t stg = 0, phase = 0; // consumer position in the ring and its mbarrier phase
  while (fifo_n != 0) { // the producer started this link NSTAGE chunks ago (or at start-up)
    uint32_t link, u0, n_units; // n_units: end of the slice
    const uint32_t part = slice_of(fifo_pop(), link, u0, n_units);
    const uint8_t* link_base = base_of<SWTPG_WIBETH_FRAME_BYTES>(p, link);
    uint32_t* st = p.state + size_t(link) * kStateWordsPerGroup;
    // A later slice of a link continues from the state its predecessor stored: wait until the NON-EMPTY slices before it are
    // done (with fewer units than slices some are empty and never run: exactly min(part, u0) of the earlier ones are not). By
    // the time a second slice is claimed every first one was handed out a whole round ago, so this hardly ever spins; it cannot
    // dead-lock because every warp of the persistent grid is resident and items are taken in dependency order.
    if (part != 0u && u0 != 0u) {
      const uint32_t before = slices_before(link, part, u0);
      wait_for_slices(p.link_done + link, before); // out of line: the spin must not cost the tick loop registers
    }
    const uint32_t flags = *reinterpret_cast<volatile uint32_t*>(p.group_flags + link);
    algo.load(st, lane, flags);
    bool need_seed = !(flags & kFlagInitialized);
    ctx.link = link;
    ctx.link_base = link_base;

    for (uint32_t unit = u0; unit < n_units; ++unit) {
      ctx.tick_base = 0u; // 64 ticks per unit = 0 mod 8: the FIR ring phase at a unit's first tick is the slice's initial one
      ctx.unit = unit;
      if constexpr (Algo::kNeedsUnitTs) // DAQEthHeader word 1 = timestamp (docs/README.md:81)
        ctx.ts = *reinterpret_cast<const unsigned long long*>(link_base + size_t(unit) * SWTPG_WIBETH_FRAME_BYTES + 8);
#pragma unroll 1
      for (int t0 = 0; t0 < 64; t0 += kWibEthChunkTicks) {
        mbar_wait(&bars[stg], phase);
        const uint32_t* rows = reinterpret_cast<const uint32_t*>(stages + stg * kChunkBytes);
        if (need_seed) {
          algo.seed(Algo::sample(rows, pp));
          need_seed = false;
        }
        constexpr int G = 4;
        constexpr int kGroupUnroll = Algo::kGroupUnroll;
        algo.begin_chunk(rows, pp);
#pragma unroll kGroupUnroll
        for (int tt = 0; tt < kWibEthChunkTicks; tt += G) {
          uint32_t ped[G], wav[G];
          algo.template group<G, DUMP>(rows + tt * (kWibEthRowBytes / 4), pp, ctx, t0 + tt, ped, wav, tt + G < kWibEthChunkTicks);
          if constexpr (DUMP) {
#pragma unroll
            for (int g = 0; g < G; ++g) {
              const size_t o = ((size_t(link) * p.units_stride + unit) * 64 + size_t(t0 + tt + g)) * 32 + lane; // u32 = 2 channels
              if (p.pedestal_out)
                reinterpret_cast<uint32_t*>(p.pedestal_out)[o] = ped[g];
              if (p.waveform_out)
                reinterpret_cast<uint32_t*>(p.waveform_out)[o] = wav[g];
            }
          }
        }
        // Every lane's loads from this stage have completed (their values were consumed above), so after the warp barrier
        // the stage can be handed back to the copy engine: a read-then-async-write hand-off needs no proxy fence.
        __syncwarp();
        produce();
        if (++stg == NSTAGE) {
          stg = 0;
          phase ^= 1u;
        }
      }
    }

    close_item<false>(algo, ctx, hits, st, link, (n_units - u0) * 64u, lane);
    if (p.parts_log2 != 0u) { // publish the state to the warp that runs the link's next slice; the last slice re-arms the counter
      __threadfence(); // every lane's (the release alone measured the same, profiles/r02_step_form_probe.txt)
      __syncwarp();    // orders the lanes' stores before lane 0's release, which is cumulative
      if (lane == 0) {
        const uint32_t done = part + 1u == (1u << p.parts_log2) ? 0u : slices_before(link, part, u0) + 1u;
        asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p.link_done + link), "r"(done) : "memory");
      }
    }
  }
  if (lane == 0) {
    const uint32_t active = min(warps_total, n_items);
    __threadfence();
    if (atomicAdd(p.link_cursor + 1, 1u) == active - 1u) {
      p.link_cursor[0] = 0u;
      p.link_cursor[1] = 0u;
    }
  }
}

// =====================================================================================================================
// WIBEth kernel, CTA form: 4 consumer warps + 1 producer warp work on a QUAD of 4 links in lock-step (the structure of the
// WIB2 kernel below, where one link is four warps wide). A stage of the CTA-wide ring holds one chunk of each of the four links
// (four bulk copies signalled on ONE `full` barrier, released through ONE `empty` barrier with an
// arrival per consumer), so a consumer's per-chunk bookkeeping is a barrier wait and an arrive — the ring cursor, the
// source addresses and the link hand-out (first quad by block index, every further one claimed from the device-side cursor
// four links at a time, published through a small FIFO) live in the producer warp, once per quad instead of once per link.
// Ragged batches: a quad runs for the longest of its links; a consumer whose link is shorter (or absent) only keeps step.
// =====================================================================================================================
constexpr int kQuad = 4;
constexpr uint32_t kNoLink = 0xFFFFFFFFu; // quad position without a link (past the end of the group)
constexpr uint32_t kQuadFifo = 4; // quads in flight: the producer is at most NSTAGE chunks ahead, a quad has >= kChunksPerUnit chunks
// per stage one chunk of each link and the two barriers; per FIFO entry 4 link ids, the quad's length in units, padding
using WibEthQuadSmem = SmemLayout<size_t(kWibEthStages) * kQuad * kWibEthChunkBytes, size_t(kWibEthStages) * 16, kQuad, kQuadFifo * 32>;

template<class Algo, bool DUMP>
__global__ void __launch_bounds__((kQuad + 1) * 32)
wibeth_quad_kernel(const KernelParams p)
{
  constexpr int NSTAGE = kWibEthStages;
  constexpr uint32_t kChunkBytes = kWibEthChunkBytes, kChunksPerUnit = kWibEthChunksPerUnit;
  static_assert((NSTAGE + kChunksPerUnit - 1) / kChunksPerUnit + 2 <= kQuadFifo, "quad FIFO too short for this ring geometry");
  extern __shared__ __align__(128) uint8_t smem[];
  using L = WibEthQuadSmem;
  const uint32_t warp = __shfl_sync(0xFFFFFFFFu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31u;
  uint8_t* stages = smem;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + L::bars);
  uint64_t* empty = full + NSTAGE;
  volatile uint32_t* fifo = reinterpret_cast<volatile uint32_t*>(smem + L::fifo); // [kQuadFifo][8]: links[4], units of the longest
  HitStage hits;
  L::place_hits(hits, smem, warp);

  auto link_of = [&](uint32_t item) -> uint32_t { return p.link_ids != nullptr ? p.link_ids[item] : item; }; // the group's item-th link

  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < NSTAGE; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], kQuad);
    }
    fence_mbar_init();
  }
  if (lane == 0 && warp < kQuad)
    *hits.cnt = 0u;
  __syncthreads(); // the only CTA-wide barrier: mbarriers visible before anyone waits on them

  if (warp == kQuad) { // ---- producer warp (one lane) ----
    if (lane != 0)
      return;
    uint32_t slot = 0, round = 0, pushed = 0;
    auto wait_slot = [&]() { // all four consumers released the stage's previous contents
      if (round != 0)
        mbar_wait(&empty[slot], (round - 1u) & 1u);
    };
    uint32_t first_link = blockIdx.x * kQuad; // the CTA's first quad (work items); every further one is claimed from the cursor
    for (bool first = true;;) {
      uint32_t nu[kQuad], longest = 0;
      for (;;) { // next quad that has data
        if (!first)
          first_link = gridDim.x * kQuad + atomicAdd(p.link_cursor, uint32_t(kQuad));
        first = false;
        longest = 0;
        if (first_link >= p.n_links)
          break;
#pragma unroll
        for (int c = 0; c < kQuad; ++c) { // a group's last quad may be partial
          nu[c] = first_link + c < p.n_links ? units_of(p, link_of(first_link + c)) : 0u;
          longest = max(longest, nu[c]);
        }
        if (longest != 0)
          break;
      }
      volatile uint32_t* entry = fifo + (pushed & (kQuadFifo - 1u)) * 8u;
      if (first_link >= p.n_links) { // end marker: a stage that completes without data
        wait_slot();
        entry[4] = 0u;
        entry[5] = 1u;
        mbar_arrive(&full[slot]);
        break;
      }
      const uint8_t* src0 = p.frames + 32;                                        // link l of the quad: + l * link_stride
      const size_t link_stride = size_t(p.units_stride) * SWTPG_WIBETH_FRAME_BYTES;
      for (uint32_t unit = 0; unit < longest; ++unit) {
        for (uint32_t ch = 0; ch < kChunksPerUnit; ++ch) {
          wait_slot();
          if (unit == 0 && ch == 0) { // published before the arrive below releases it to the consumers
#pragma unroll
            for (int c = 0; c < kQuad; ++c)
              entry[c] = first_link + c < p.n_links ? link_of(first_link + c) : kNoLink;
            entry[4] = longest;
            entry[5] = 0u;
            ++pushed;
          }
          uint32_t bytes = 0;
#pragma unroll
          for (int c = 0; c < kQuad; ++c)
            bytes += unit < nu[c] ? kChunkBytes : 0u;
          mbar_arrive_expect_tx(&full[slot], bytes);
          const uint8_t* src = src0 + size_t(unit) * SWTPG_WIBETH_FRAME_BYTES + ch * kChunkBytes;
#pragma unroll
          for (int c = 0; c < kQuad; ++c)
            if (unit < nu[c])
              bulk_g2s(stages + (slot * kQuad + c) * kChunkBytes, src + link_of(first_link + c) * link_stride, kChunkBytes, &full[slot]);
          if (++slot == NSTAGE) {
            slot = 0;
            ++round;
          }
        }
      }
    }
    rearm_cursor(p, gridDim.x);
    return;
  }

  // ---- consumer warps: warp c works on link c of every quad ----
  Algo algo;
  algo.configure(p);
  const PairPos pp = pair_pos(lane);
  TickCtx ctx;
  ctx.p = &p;
  ctx.chan0 = 2 * lane;
  ctx.ts = 0;
  ctx.stage = &hits;

  uint32_t stg = 0, phase = 0; // consumer position in the ring and the full barrier's phase
  for (uint32_t popped = 0;; ++popped) {
    mbar_wait(&full[stg], phase); // first chunk of the next quad, or the end marker
    const volatile uint32_t* entry = fifo + (popped & (kQuadFifo - 1u)) * 8u;
    if (entry[5] != 0u)
      break;
    // the position's link through a reduction: a uniform register, as the link index was before groups (ptxas otherwise
    // needs up to 7 more registers for this kernel)
    const uint32_t link = __reduce_max_sync(0xFFFFFFFFu, entry[warp]), longest = entry[4];
    const uint32_t n_units = link != kNoLink ? units_of(p, link) : 0u;
    const uint8_t* link_base = base_of<SWTPG_WIBETH_FRAME_BYTES>(p, link != kNoLink ? link : 0u);
    uint32_t* st = p.state + size_t(link) * kStateWordsPerGroup;
    uint32_t flags = 0;
    bool need_seed = false;
    if (n_units != 0) {
      flags = p.group_flags[link];
      algo.load(st, lane, flags);
      need_seed = !(flags & kFlagInitialized);
    }
    ctx.link = link;
    ctx.link_base = link_base;

    for (uint32_t unit = 0; unit < longest; ++unit) {
      const bool mine = unit < n_units;
      ctx.tick_base = unit * 64u;
      ctx.unit = unit;
      if constexpr (Algo::kNeedsUnitTs) {
        if (mine) // DAQEthHeader word 1 = timestamp (docs/README.md:81)
          ctx.ts = *reinterpret_cast<const unsigned long long*>(link_base + size_t(unit) * SWTPG_WIBETH_FRAME_BYTES + 8);
      }
#pragma unroll 1
      for (int t0 = 0; t0 < 64; t0 += kWibEthChunkTicks) {
        if (unit != 0 || t0 != 0)
          mbar_wait(&full[stg], phase);
        if (mine) {
          const uint32_t* rows = reinterpret_cast<const uint32_t*>(stages + (stg * kQuad + warp) * kChunkBytes);
          if (need_seed) {
            algo.seed(Algo::sample(rows, pp));
            need_seed = false;
          }
          constexpr int G = 4;
          constexpr int kGroupUnroll = Algo::kGroupUnroll;
          algo.begin_chunk(rows, pp);
#pragma unroll kGroupUnroll
          for (int tt = 0; tt < kWibEthChunkTicks; tt += G) {
            uint32_t ped[G], wav[G];
            algo.template group<G, DUMP>(rows + tt * (kWibEthRowBytes / 4), pp, ctx, t0 + tt, ped, wav, tt + G < kWibEthChunkTicks);
            if constexpr (DUMP) {
#pragma unroll
              for (int g = 0; g < G; ++g) {
                const size_t o = ((size_t(link) * p.units_stride + unit) * 64 + size_t(t0 + tt + g)) * 32 + lane; // u32 = 2 channels
                if (p.pedestal_out)
                  reinterpret_cast<uint32_t*>(p.pedestal_out)[o] = ped[g];
                if (p.waveform_out)
                  reinterpret_cast<uint32_t*>(p.waveform_out)[o] = wav[g];
              }
            }
          }
        }
        // Every lane's loads from this stage have completed (their values were consumed above), so after the warp barrier
        // the stage can be handed back to the copy engine: a read-then-async-write hand-off needs no proxy fence.
        __syncwarp();
        if (lane == 0)
          mbar_arrive(&empty[stg]);
        if (++stg == NSTAGE) {
          stg = 0;
          phase ^= 1u;
        }
      }
    }

    if (n_units != 0)
      close_item<false>(algo, ctx, hits, st, link, n_units * 64u, lane);
  }
}

// =====================================================================================================================
// WIB2 kernel: one CTA of 4 consumer warps + 1 producer warp per link (256 channels), persistent over links. A superchunk
// (12 frames x 472 B) is one 5664-byte bulk copy into a CTA-wide ring; consumer warp w works on channels 64w..64w+63 (112
// bytes of every frame's ADC block). full[s]: the copy engine's complete_tx; empty[s]: one arrival per consumer warp. The
// producer warp (one lane; it sleeps on the empty barriers and issues no other instructions) walks the same link/unit
// CTA's links — the first by block index, every further one claimed from the device-side cursor, published to the consumers
// through a small FIFO — and refills a stage as soon as all four consumers have released it — so no consumer ever waits for
// another consumer, only for data (before: warp 0 refilled between its own superchunks and 13 % of all warp time was spent waiting
// on full barriers, profiles/r01_wib2_simple_ncu_full.txt).
// =====================================================================================================================
constexpr int kWib2FrameWords = SWTPG_WIB2_FRAME_BYTES / 4; // 118
constexpr int kWib2Warps = 4;
constexpr uint32_t kWib2Fifo = 8;           // links in flight: the producer is at most NSTAGE superchunks ahead (+ the end marker)
constexpr uint32_t kNoMoreLinks = 0xFFFFFFFFu;

template<int NSTAGE> // per stage one superchunk and the two barriers
using Wib2Smem = SmemLayout<size_t(NSTAGE) * SWTPG_WIB2_SUPERCHUNK_BYTES, size_t(NSTAGE) * 16, kWib2Warps, kWib2Fifo * 4>;

// Algo::kWib2MinCtas caps the registers so that that many CTAs fit an SM (5 = 25 warps): +1 % for SimpleThreshold, +2 % for
// FIR + IQR, -3.5 % for the running sum, which therefore leaves it at 1 (gpurun_out/var30: measured per policy).
template<class Algo, int NSTAGE, bool DUMP>
__global__ void __launch_bounds__((kWib2Warps + 1) * 32, Algo::kWib2MinCtas)
wib2_kernel(const KernelParams p)
{
  constexpr uint32_t kUnit = SWTPG_WIB2_SUPERCHUNK_BYTES;
  extern __shared__ __align__(128) uint8_t smem[];
  using L = Wib2Smem<NSTAGE>;
  const uint32_t warp = __shfl_sync(0xFFFFFFFFu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31u;
  uint8_t* stages = smem;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + L::bars);
  uint64_t* empty = full + NSTAGE;
  HitStage hits;
  L::place_hits(hits, smem, warp);

  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < NSTAGE; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], kWib2Warps);
    }
    fence_mbar_init();
  }
  if (lane == 0 && warp < kWib2Warps)
    *hits.cnt = 0u;
  __syncthreads(); // the only CTA-wide barrier: mbarriers visible before anyone waits on them

  volatile uint32_t* fifo = reinterpret_cast<volatile uint32_t*>(smem + L::fifo);
  if (warp == kWib2Warps) { // producer warp: one lane feeds the ring and decides which links this CTA works on
    if (lane != 0)
      return;
    static_assert(NSTAGE + 2 <= int(kWib2Fifo), "link FIFO too short for this ring depth");
    uint32_t slot = 0, round = 0, pushed = 0;
    auto wait_slot = [&]() { // all four consumers released the stage's previous contents
      if (round != 0)
        mbar_wait(&empty[slot], (round - 1u) & 1u);
    };
    uint32_t item = blockIdx.x; // the CTA's first work item; every further one is claimed from the cursor (as in wibeth_kernel)
    for (bool first = true;; first = false) {
      uint32_t n_units = 0, link = 0;
      for (;;) {
        if (!first)
          item = gridDim.x + atomicAdd(p.link_cursor, 1u);
        first = false;
        if (item >= p.n_links)
          break;
        link = p.link_ids != nullptr ? p.link_ids[item] : item; // the group's item-th link
        n_units = units_of(p, link);
        if (n_units != 0)
          break;
      }
      if (item >= p.n_links) { // end marker: a stage that completes without data
        wait_slot();
        fifo[pushed & (kWib2Fifo - 1u)] = kNoMoreLinks;
        mbar_arrive(&full[slot]);
        break;
      }
      const uint8_t* src = base_of<kUnit>(p, link);
      for (uint32_t unit = 0; unit < n_units; ++unit, src += kUnit) {
        wait_slot();
        if (unit == 0) // published before the arrive below releases it to the consumers
          fifo[pushed++ & (kWib2Fifo - 1u)] = link;
        mbar_arrive_expect_tx(&full[slot], kUnit);
        bulk_g2s(stages + slot * kUnit, src, kUnit, &full[slot]);
        if (++slot == NSTAGE) {
          slot = 0;
          ++round;
        }
      }
    }
    rearm_cursor(p, gridDim.x);
    return;
  }

  Algo algo;
  algo.configure(p);
  const PairPos pp = pair_pos(lane);
  TickCtx ctx;
  ctx.p = &p;
  ctx.chan0 = 64 * warp + 2 * lane;
  ctx.ts = 0;
  ctx.stage = &hits;
  const uint32_t row0 = p.wib2_adc_offset / 4 + warp * 28; // word offset of this warp's 112 bytes inside a frame

  uint32_t stg = 0, phase = 0;       // consumer ring position / full-barrier phase
  for (uint32_t popped = 0;; ++popped) {
    mbar_wait(&full[stg], phase);    // first superchunk of the next link, or the end marker
    const uint32_t link = fifo[popped & (kWib2Fifo - 1u)];
    if (link == kNoMoreLinks)
      break;
    const uint32_t n_units = units_of(p, link);
    const uint8_t* link_base = base_of<kUnit>(p, link);
    const uint32_t group = link * kWib2Warps + warp;
    uint32_t* st = p.state + size_t(group) * kStateWordsPerGroup;
    const uint32_t flags = p.group_flags[group];
    algo.load(st, lane, flags);
    bool need_seed = !(flags & kFlagInitialized);
    ctx.link = link;
    ctx.link_base = link_base;

    for (uint32_t unit = 0; unit < n_units; ++unit) {
      ctx.tick_base = unit * 12u;
      ctx.unit = unit;
      if (unit != 0)
        mbar_wait(&full[stg], phase);
      const uint32_t* sc = reinterpret_cast<const uint32_t*>(stages + stg * kUnit);
      if constexpr (Algo::kNeedsUnitTs)
        ctx.ts = uint64_t(sc[1]) | (uint64_t(sc[2]) << 32); // WIB2Frame::get_timestamp, first frame (:350-351)
      const uint32_t* rows = sc + row0;
      if (need_seed) {
        algo.seed(Algo::sample(rows, pp));
        need_seed = false;
      }
      constexpr int G = 4;
      algo.template begin_chunk<kWib2FrameWords>(rows, pp);
#pragma unroll
      for (int tt = 0; tt < 12; tt += G) {
        uint32_t ped[G], wav[G];
        algo.template group<G, DUMP, kWib2FrameWords, true>(rows + tt * kWib2FrameWords, pp, ctx, tt, ped, wav, tt + G < 12);
        if constexpr (DUMP) {
#pragma unroll
          for (int g = 0; g < G; ++g) {
            const size_t o = ((size_t(link) * p.units_stride + unit) * 12 + size_t(tt + g)) * 128 + warp * 32 + lane; // u32 = 2 channels
            if (p.pedestal_out)
              reinterpret_cast<uint32_t*>(p.pedestal_out)[o] = ped[g];
            if (p.waveform_out)
              reinterpret_cast<uint32_t*>(p.waveform_out)[o] = wav[g];
          }
        }
      }
      __syncwarp(); // this warp is done with the stage
      if (lane == 0)
        mbar_arrive(&empty[stg]);
      if (++stg == NSTAGE) {
        stg = 0;
        phase ^= 1u;
      }
    }

    close_item<true>(algo, ctx, hits, st, group, n_units * 12u, lane);
  }
}

} // namespace swtpg
