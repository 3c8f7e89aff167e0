// Device-side building blocks of the fused SWTPG kernels (sm_100a).
//
// Data model (DESIGN.md §3): a "group" is 64 consecutive channels = one tick row of 112 bytes = one warp.
// Lane l of the warp owns the channel PAIR (2l, 2l+1) of the group: 28 contiguous bits of the row. All per-channel
// quantities live packed two-to-a-register as s16x2 / u16x2 (low half = even channel), so the reference's 16-bit
// AVX2 lane arithmetic maps onto Blackwell's packed-16x2 integer instructions (VIADD.16x2, VIMNMX.S16x2,
// VIADDMNMX.S16x2, HSET2) — see profiles/r01_ubench_pipes.txt for their measured issue rates.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/swtpg.h"

namespace swtpg {

// ---- packed 16x2 primitives ------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t
add2(uint32_t a, uint32_t b)
{ // per-half wrapping add: VIADD.16x2 (_mm256_add_epi16)
  uint32_t r;
  asm("add.s16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ uint32_t
max2(uint32_t a, uint32_t b)
{
  uint32_t r;
  asm("max.s16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ uint32_t
min2(uint32_t a, uint32_t b)
{
  uint32_t r;
  asm("min.s16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ uint32_t
minu2(uint32_t a, uint32_t b)
{ // per-half UNSIGNED min
  uint32_t r;
  asm("min.u16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ uint32_t
addmax2(uint32_t a, uint32_t b, uint32_t c)
{ // max(a + b, c) per signed half: one VIADDMNMX.S16x2
  uint32_t r;
  asm("{.reg .b32 t; add.s16x2 t, %1, %2; max.s16x2 %0, t, %3;}" : "=r"(r) : "r"(a), "r"(b), "r"(c));
  return r;
}
__device__ __forceinline__ uint32_t
addmin2(uint32_t a, uint32_t b, uint32_t c)
{ // min(a + b, c) per signed half
  uint32_t r;
  asm("{.reg .b32 t; add.s16x2 t, %1, %2; min.s16x2 %0, t, %3;}" : "=r"(r) : "r"(a), "r"(b), "r"(c));
  return r;
}
__device__ __forceinline__ uint32_t
addclamp2(uint32_t a, uint32_t b, uint32_t hi)
{ // clamp(a + b, 0, hi) per signed half in ONE instruction (DPX: VIADDMNMX.S16x2.RELU)
  return __viaddmin_s16x2_relu(a, b, hi);
}
__device__ __forceinline__ uint32_t
neg2(uint32_t a)
{ // per-half two's complement negate
  return add2(~a, 0x00010001u);
}
// Per-half "a > b" as 0xFFFF / 0x0000, computed by the half2 comparator (HSET2) on the BIT PATTERNS. Valid as a
// signed-integer compare when b is in [0, 0x7BFF] and a is either in [0, 0x7BFF] (finite non-negative halves order
// like their bit patterns; subnormals are not flushed) or negative (sign bit set: a negative half or a NaN, both of
// which compare "not greater"). All call sites below document why their operands stay in that range.
__device__ __forceinline__ uint32_t
gt2_mask_nonneg(uint32_t a, uint32_t b)
{
  uint32_t r;
  asm("set.gt.u32.f16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
// fp16x2 add on raw bit patterns. On subnormal operands (|pattern & 0x7FFF| <= 0x3FF) this is exact sign-magnitude integer
// arithmetic executed by the FMA pipe (HADD2/HFMA2, denormals are not flushed).
__device__ __forceinline__ uint32_t
hadd2_bits(uint32_t a, uint32_t b)
{
  uint32_t r;
  asm("add.rn.f16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
// Per-half fp16 "a == b" as 0xFFFF / 0x0000 (HSET2.EQ); on subnormal patterns an integer equality test (+0 == -0).
__device__ __forceinline__ uint32_t
eq2_mask(uint32_t a, uint32_t b)
{
  uint32_t r;
  asm("set.eq.u32.f16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
// fp16x2 fused multiply-add on raw bit patterns (no flush-to-zero), and its [0, 1]-saturating form.
__device__ __forceinline__ uint32_t
hfma2_bits(uint32_t a, uint32_t b, uint32_t c)
{
  uint32_t r;
  asm("fma.rn.f16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
  return r;
}
__device__ __forceinline__ uint32_t
hfma2_sat_bits(uint32_t a, uint32_t b, uint32_t c)
{
  uint32_t r;
  asm("fma.rn.sat.f16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
  return r;
}
// Per half: 1.0 (0x3C00) where |a| != b, else 0.0 — one HSET2.BF with the |.| operand modifier.
__device__ __forceinline__ uint32_t
ne2_abs_one(uint32_t a, uint32_t b)
{
  uint32_t r;
  asm("{.reg .b32 t; abs.f16x2 t, %1; set.ne.f16x2.f16x2 %0, t, %2;}" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
// Per-half "a > b" as 0xFFFF / 0x0000 for 0 <= a <= 32767 and 0 <= b <= 32640, computed by the bf16 comparator on the bit
// patterns (HSET2.BF16_V2.GTU): non-negative bf16 values order like their patterns up to +inf = 0x7F80 = 32640; patterns
// above that are NaNs, for which the "or unordered" flavour answers true — and a > 32640 >= b is indeed true.
__device__ __forceinline__ uint32_t
gt2_mask_bf16(uint32_t a, uint32_t b)
{
  uint32_t r;
  asm("set.gtu.u32.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ uint32_t
pack2(int lo, int hi)
{
  return (uint32_t(lo) & 0xFFFFu) | (uint32_t(hi) << 16);
}
__device__ __forceinline__ int
lo16s(uint32_t v)
{
  return int(int16_t(v & 0xFFFFu));
}
__device__ __forceinline__ int
hi16s(uint32_t v)
{
  return int(int16_t(v >> 16));
}
__device__ __forceinline__ int
wrap16(int x)
{
  return int(int16_t(uint16_t(x)));
}
__device__ __forceinline__ int
sat16(int x)
{
  return x > 32767 ? 32767 : (x < -32768 ? -32768 : x);
}

// ---- async bulk copy + mbarrier (TMA engine, SASS UBLKCP / SYNCS) -------------------------------------------------
__device__ __forceinline__ uint32_t
smem_u32(const void* p)
{
  return uint32_t(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void
mbar_init(uint64_t* bar, uint32_t count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void
fence_mbar_init()
{
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void
fence_proxy_async()
{ // order this thread's earlier generic-proxy smem accesses before later async-proxy (bulk copy) writes
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void
mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes)
{
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void
mbar_arrive(uint64_t* bar)
{
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void
bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar)
{ // 16-byte aligned on both sides, bytes % 16 == 0
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// One lane of the (converged) warp, chosen by the hardware: lets ptxas issue the bulk copy from uniform registers without
// the lane-serialising loop it builds around `if (lane == 0)`.
__device__ __forceinline__ bool
elect_one()
{
  uint32_t pred;
  asm volatile("{\n.reg .pred P;\nelect.sync _|P, 0xFFFFFFFF;\nselp.u32 %0, 1, 0, P;\n}" : "=r"(pred));
  return pred != 0;
}
// Also the producer warps' wait on their `empty` barriers: try_wait parks the thread in hardware, so this loop is as fast as a
// suspend-time hint and faster than a nanosleep back-off (measured, profiles/r02_producer_wait.txt).
__device__ __forceinline__ void
mbar_wait(uint64_t* bar, uint32_t parity)
{
  asm volatile("{\n"
               ".reg .pred p;\n"
               "WAIT_%=:\n"
               "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
               "@p bra DONE_%=;\n"
               "bra WAIT_%=;\n"
               "DONE_%=:\n"
               "}" ::"r"(smem_u32(bar)),
               "r"(parity)
               : "memory");
}

// ---- 14-bit pair extraction ---------------------------------------------------------------------------------------
// Lane l's pair occupies bits [28 l, 28 l + 28) of the 896-bit little-endian row (channel c at bits [14c, 14c+14):
// fddetdataformats get_adc; reference unpack: wibeth/tpg/FrameExpand.hpp:84-186). Word index and shift are per-lane
// constants; the second word is clamped so lane 31 (shift 4, bits 868..895 all in word 27) never reads past the row.
struct PairPos
{
  uint32_t w0, w1, sh;
};
__device__ __forceinline__ PairPos
pair_pos(uint32_t lane)
{
  PairPos p;
  p.w0 = (28u * lane) >> 5;
  p.sh = (28u * lane) & 31u;
  p.w1 = p.w0 + 1u > 27u ? 27u : p.w0 + 1u;
  return p;
}
__device__ __forceinline__ uint32_t
extract_pair(const uint32_t* row, const PairPos& pp)
{
  const uint32_t x = __funnelshift_r(row[pp.w0], row[pp.w1], pp.sh); // 28 payload bits + 4 junk bits on top
  return (x & 0x3FFFu) | ((x << 2) & 0x3FFF0000u);                   // -> u16x2 {adc(2l), adc(2l+1)}
}

// The same pair with 0x4000 subtracted from each half (bits 14 and 15 forced to one: S - 16384 in two's complement), at the same
// cost — SHF + shift + 2 LOP3. The packed SimpleThreshold / running-sum policies keep "16385 - median" instead of "1 - median",
// so that the median register never passes through 0x0000 / 0xFFFF and its +-1 steps can be ONE 32-bit three-input add
// (no carry or borrow ever crosses the halves); the bias cancels in S' + Mq' = s - median + 1.
__device__ __forceinline__ uint32_t
extract_pair_biased_from(uint32_t lo_word, uint32_t hi_word, uint32_t sh)
{
  const uint32_t x = __funnelshift_r(lo_word, hi_word, sh);
  const uint32_t u = x | 0xFFFFC000u;            // low half: field 0 | 0xC000; high half: all ones
  return u & ((x << 2) | 0xC000FFFFu);           // high half: field 1 | 0xC000; low half kept
}
__device__ __forceinline__ uint32_t
extract_pair_biased(const uint32_t* row, const PairPos& pp)
{
  return extract_pair_biased_from(row[pp.w0], row[pp.w1], pp.sh);
}

// ---- TP emission -----------------------------------------------------------------------------------------------------
struct TpSink
{
  swtpg_tp* buf;
  unsigned int* count;
  uint32_t cap;
};
// Appends one record. Device order is arbitrary (atomic cursor); the host sorts by (time_start, link, channel).
__device__ __forceinline__ void
emit_tp(const TpSink& k, uint64_t time_start, uint64_t time_peak, uint32_t tot, uint32_t integral, uint32_t peak, uint32_t chan,
        uint32_t link)
{
  const unsigned idx = atomicAdd(k.count, 1u);
  if (idx < k.cap) {
    uint4* d = reinterpret_cast<uint4*>(k.buf + idx);
    d[0] = make_uint4(uint32_t(time_start), uint32_t(time_start >> 32), uint32_t(time_peak), uint32_t(time_peak >> 32));
    d[1] = make_uint4(tot, integral, (peak & 0xFFFFu) | (chan << 16), link);
  }
}
// WIBEth TP fields: src/wibeth/WIBEthFrameProcessor.cpp:520-545 (accepted iff hit_charge != 0)
__device__ __forceinline__ void
emit_wibeth(const TpSink& k, uint64_t ts, int t_end, uint32_t charge, uint32_t tover, uint32_t peak_adc, uint32_t peak_time,
            uint32_t chan, uint32_t link)
{
  if (charge == 0)
    return;
  const uint64_t t0 = ts + uint64_t(32ll * (int64_t(t_end) - int64_t(tover)));
  emit_tp(k, t0, t0 + 32ull * peak_time, 32u * tover, charge, peak_adc, chan, link);
}
// WIB2 TP fields: src/wib2/WIB2FrameProcessor.cpp:429-455
__device__ __forceinline__ void
emit_wib2(const TpSink& k, uint64_t ts, int t_end, uint32_t charge, uint32_t tover, uint32_t chan, uint32_t link)
{
  if (charge == 0)
    return;
  const uint64_t t0 = ts + uint64_t(32ll * (int64_t(t_end) - int64_t(tover)));
  const uint64_t t1 = ts + uint64_t(32ll * int64_t(t_end));
  emit_tp(k, t0, (t0 + t1) / 2, uint32_t(int64_t(tover) * 32), charge, (charge / 20u) & 0xFFFFu, chan, link);
}

// ---- per-warp hit staging -----------------------------------------------------------------------------------------
// The tick loop only parks raw PAIR records in a warp-private shared-memory buffer: a lane on which at least one of its two
// channels ends a hit takes a slot with a shared-memory atomic (lane-divergent code, one site per tick; ptxas aggregates
// the atomic over the lanes that take the branch together) and writes its packed registers as they are — 20 bytes:
//   {meta = frame channel of the low half | tick << 8 | unit << 14, charge & left, tover, peak_adc} + {peak_time}.
// A half whose masked charge is zero produced no TP (it did not end, or its hit has hit_charge == 0, which the reference's
// decode drops: src/wibeth/WIBEthFrameProcessor.cpp:520, src/wib2/WIB2FrameProcessor.cpp:429). Splitting pairs into
// records, the 64-bit TP arithmetic, the global cursor atomic (one per flush, not per hit) and the 32-byte
// record stores happen in flush(), with all 32 lanes converting one pair each (ballot-free: one warp prefix sum).
constexpr uint32_t kHitUnitBits = 18; // units per batch must stay below 2^18 (checked by swtpg_create)

struct HitStage
{
  static constexpr uint32_t kCap = 160;               // pair records; a 4-tick group parks at most one per lane and tick = 128,
  static constexpr uint32_t kFlushAbove = kCap - 128; // so checking once per group with <= kCap-128 parked never overflows
  uint4* buf;                                 // warp-private, kCap entries
  uint32_t* aux;                              // warp-private, kCap entries (peak_time pairs)
  uint32_t* cnt;                              // warp-private counter in shared memory

  static __device__ __forceinline__ uint32_t meta(uint32_t chan0, uint32_t unit, uint32_t t_end)
  {
    return chan0 | (t_end << 8) | (unit << 14);
  }
  // Any subset of lanes may call. charge_left = charge & left (per half), the other words are the packed state registers.
  __device__ __forceinline__ void push(uint32_t m, uint32_t charge_left, uint32_t tover, uint32_t peak, uint32_t ptime) const
  {
    const uint32_t slot = atomicAdd(cnt, 1u);
    buf[slot] = make_uint4(m, charge_left, tover, peak);
    aux[slot] = ptime;
  }
  __device__ __forceinline__ void push(uint32_t m, uint32_t charge_left, uint32_t tover) const // finders without peak tracking
  {
    const uint32_t slot = atomicAdd(cnt, 1u);
    buf[slot] = make_uint4(m, charge_left, tover, 0u);
  }
  // Warp-uniform (every lane reads the same word); the warp is converged at both call sites.
  __device__ __forceinline__ uint32_t count() const { return *reinterpret_cast<volatile uint32_t*>(cnt); }
  __device__ __forceinline__ bool must_flush() const
  {
    __syncwarp();
    return count() > kFlushAbove;
  }

  // Converts and writes out everything staged (see flush_hits). Whole warp calls, converged.
  template<bool WIB2_UNITS, bool WIB2_FIELDS>
  __device__ __forceinline__ void flush(const TpSink& k, const uint8_t* link_base, uint32_t link, uint32_t lane, bool everything) const;
};

// Pair records -> swtpg_tp. Out of line (cold) and all-by-value, so the caller keeps its state in registers.
//   WIB2_UNITS : where the unit's timestamp lives — WIBEthFrame DAQEthHeader word 1 (docs/README.md:81) or
//                WIB2Frame::get_timestamp of the superchunk's first frame (bytes 4..11, src/wib2/WIB2FrameProcessor.cpp:350-351)
//   WIB2_FIELDS: which process_swtpg_hits derives the fields — src/wibeth/WIBEthFrameProcessor.cpp:520-545 (peak from the
//                tracked peak) or src/wib2/WIB2FrameProcessor.cpp:429-455 (time_peak = middle of the hit, adc_peak = integral/20)
template<bool WIB2_UNITS, bool WIB2_FIELDS>
__device__ __noinline__ void
flush_hits(uint4* buf, uint32_t* aux, uint32_t* cnt, swtpg_tp* out, unsigned int* out_count, uint32_t out_cap, const uint8_t* link_base,
           uint32_t link, uint32_t lane, bool everything)
{
  __syncwarp();
  const uint32_t parked = *reinterpret_cast<volatile uint32_t*>(cnt);
  // In the middle of a link only whole rounds of 32 pairs are written out (every lane busy in every round); the tail stays
  // parked — at most 31 records, within the room a group needs — and moves to the front of the buffer. The end of a link
  // writes out everything.
  const uint32_t n = everything ? parked : parked & ~31u;
  if (n == 0)
    return;
  // Pass 1: how many TPs the parked pairs hold, then ONE reservation in the global list. The atomic's round trip overlaps
  // the loads and the prefix arithmetic of the first 32 pairs: its result is only read when the first record is stored.
  uint32_t mine = 0;
  for (uint32_t i = lane; i < n; i += 32) {
    const uint32_t c = buf[i].y;
    mine += uint32_t((c & 0xFFFFu) != 0u) + uint32_t((c >> 16) != 0u);
  }
  const uint32_t total = __reduce_add_sync(0xFFFFFFFFu, mine);
  unsigned base = 0;
  if (total != 0 && lane == 0)
    base = atomicAdd(out_count, total);
  bool have_base = false;
  uint32_t done = 0; // TPs of the pairs before this lane's (prefix over whole 32-pair rounds)
  const uint32_t below = (1u << lane) - 1u;
  for (uint32_t i0 = 0; i0 < n && total != 0; i0 += 32) { // whole warp: one pair record per lane
    const uint32_t i = i0 + lane;
    uint4 r = make_uint4(0u, 0u, 0u, 0u);
    uint32_t pt2 = 0u;
    if (i < n) {
      r = buf[i];
      if constexpr (!WIB2_FIELDS)
        pt2 = aux[i];
    }
    const bool have_lo = (r.y & 0xFFFFu) != 0u, have_hi = (r.y >> 16) != 0u;
    const uint32_t b_lo = __ballot_sync(0xFFFFFFFFu, have_lo), b_hi = __ballot_sync(0xFFFFFFFFu, have_hi);
    uint32_t idx = done + __popc(b_lo & below) + __popc(b_hi & below);
    done += __popc(b_lo) + __popc(b_hi);
    const uint32_t chan0 = r.x & 0xFFu, t_end = (r.x >> 8) & 0x3Fu, unit = r.x >> 14;
    uint64_t ts = 0;
    if (have_lo || have_hi) {
      if constexpr (WIB2_UNITS) {
        const uint32_t* hdr = reinterpret_cast<const uint32_t*>(link_base + size_t(unit) * SWTPG_WIB2_SUPERCHUNK_BYTES + 4);
        ts = uint64_t(hdr[0]) | (uint64_t(hdr[1]) << 32);
      } else {
        ts = *reinterpret_cast<const unsigned long long*>(link_base + size_t(unit) * SWTPG_WIBETH_FRAME_BYTES + 8);
      }
    }
    if (!have_base) {
      base = __shfl_sync(0xFFFFFFFFu, base, 0);
      have_base = true;
    }
    idx += base;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (!(h ? have_hi : have_lo))
        continue;
      const uint32_t charge = h ? r.y >> 16 : r.y & 0xFFFFu, tover = h ? r.z >> 16 : r.z & 0xFFFFu;
      const uint64_t t0 = ts + uint64_t(32ll * (int64_t(t_end) - int64_t(tover)));
      if (idx < out_cap) {
        uint4* d = reinterpret_cast<uint4*>(out + idx);
        uint64_t tp;
        uint32_t pk;
        if constexpr (WIB2_FIELDS) {
          tp = (t0 + (ts + uint64_t(32ll * int64_t(t_end)))) / 2;
          pk = (charge / 20u) & 0xFFFFu;
        } else {
          tp = t0 + 32ull * (h ? pt2 >> 16 : pt2 & 0xFFFFu);
          pk = h ? r.w >> 16 : r.w & 0xFFFFu;
        }
        d[0] = make_uint4(uint32_t(t0), uint32_t(t0 >> 32), uint32_t(tp), uint32_t(tp >> 32));
        d[1] = make_uint4(32u * tover, charge, pk | ((chan0 + uint32_t(h)) << 16), link);
      }
      ++idx;
    }
  }
  __syncwarp();
  const uint32_t rest = parked - n; // < 32
  uint4 r = make_uint4(0u, 0u, 0u, 0u);
  uint32_t pt2 = 0u;
  if (lane < rest) {
    r = buf[n + lane];
    if constexpr (!WIB2_FIELDS)
      pt2 = aux[n + lane];
  }
  __syncwarp();
  if (lane < rest) {
    buf[lane] = r;
    if constexpr (!WIB2_FIELDS)
      aux[lane] = pt2;
  }
  if (lane == 0)
    *reinterpret_cast<volatile uint32_t*>(cnt) = rest;
  __syncwarp();
}

template<bool WIB2_UNITS, bool WIB2_FIELDS>
__device__ __forceinline__ void
HitStage::flush(const TpSink& k, const uint8_t* link_base, uint32_t link, uint32_t lane, bool everything) const
{
  flush_hits<WIB2_UNITS, WIB2_FIELDS>(buf, aux, cnt, k.buf, k.count, k.cap, link_base, link, lane, everything);
}

} // namespace swtpg
