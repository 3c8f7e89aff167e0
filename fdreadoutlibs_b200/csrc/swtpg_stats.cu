// Per-channel statistics of the raw ADC values: one streaming read of every batch after its TPG launches, on the same stream.
//   SWTPG_FLAG_ADC_STATS      per (link, frame channel): samples, sum, sum of squares, minimum and maximum, into 32-byte
//                             accumulators in HBM (swtpg_handle::d_adc_stats), copied out by swtpg_read_adc_stats.
//   SWTPG_FLAG_NOISE_SPECTRA  per (link, frame channel): the segments counted and the circular lag sums of each segment,
//                             lag[tau] = sum_t x[t] x[(t + tau) mod N] for tau = 0..N/2 (swtpg_handle::d_noise_lags), copied out by
//                             swtpg_read_noise_lags; swtpg_noise_power turns them into the averaged periodogram on the host.
// With both flags one kernel reads the batch once.
//   SWTPG_FLAG_CHANNEL_COVARIANCE  per link: samples, the sum of every channel and the sums of products of every pair of its
//                             channels (swtpg_handle::d_channel_products), copied out by swtpg_read_channel_products;
//                             swtpg_channel_covariance turns them into covariance and correlation matrices on the host. A kernel
//                             of its own (channel_products_kernel: a CTA-wide tile of all channels on the integer tensor cores),
//                             launched after the statistics kernel.
#include "swtpg_device.cuh"
#include "swtpg_handle.h"

#include <algorithm>

using namespace swtpg;

namespace {

constexpr uint32_t kStatsWarps = 4;       // warps per CTA
constexpr uint32_t kStatsMaxUnits = 64;   // units per work item at most: keeps the per-item sums in 32 bits (64 x 64 x 16383 < 2^32)
constexpr uint32_t kStatsItemsPerSm = 48; // work items per SM a launch aims for (a few links are split finer, down to one unit)

// Noise-spectrum segments: one WIBEth frame (64 ticks), four WIB2 superchunks (48 ticks).
template<bool WIB2>
struct Segment
{
  static constexpr uint32_t kUnits = WIB2 ? SWTPG_WIB2_NOISE_SEGMENT_TICKS / SWTPG_WIB2_TICKS : 1;
  static constexpr uint32_t kTicks = WIB2 ? SWTPG_WIB2_NOISE_SEGMENT_TICKS : SWTPG_WIBETH_NOISE_SEGMENT_TICKS;
  static constexpr uint32_t kLags = kTicks / 2 + 1;
  // per warp, lane-private columns: the segment's pairs [kTicks][32] (u16x2), then the item's lag sums [kLags][2][32] (u64)
  static constexpr uint32_t kSmemBytes = kTicks * 32 * 4 + kLags * 2 * 32 * 8;
};
static_assert(SWTPG_WIB2_NOISE_SEGMENT_TICKS % SWTPG_WIB2_TICKS == 0 && SWTPG_WIBETH_NOISE_SEGMENT_TICKS == SWTPG_WIBETH_TICKS, "segments are whole units");

// Adds the circular lags of one staged segment to the lane's lag sums, one channel of its pair after the other. Products are
// below 2^28: 16 of them are summed in 32 bits, then added in 64 bits.
template<bool WIB2>
__device__ __forceinline__ void
add_segment_lags(const uint32_t* __restrict__ seg, unsigned long long* __restrict__ lags, uint32_t lane)
{
  using Sg = Segment<WIB2>;
  constexpr uint32_t N = Sg::kTicks;
  static_assert(N % 16 == 0, "the 32-bit partial sums take 16 ticks each");
#pragma unroll 1
  for (uint32_t half = 0; half < 2; ++half) {
    uint32_t x[N];
#pragma unroll
    for (uint32_t t = 0; t < N; ++t)
      x[t] = (seg[t * 32 + lane] >> (16 * half)) & 0xFFFFu;
#pragma unroll
    for (uint32_t tau = 0; tau < Sg::kLags; ++tau) {
      unsigned long long s = 0;
#pragma unroll
      for (uint32_t t0 = 0; t0 < N; t0 += 16) {
        uint32_t q = 0;
#pragma unroll
        for (uint32_t t = t0; t < t0 + 16; ++t)
          q += x[t] * x[(t + tau) % N];
        s += q;
      }
      lags[(tau * 2 + half) * 32 + lane] += s;
    }
  }
}

// Work item i of the launch: link i / (groups * parts), its 64-channel group, and units [part * chunk, part * chunk + chunk).
// One warp per item; lane l owns frame channels 64 g + 2l and 64 g + 2l + 1, extracted from each 112-byte row by extract_pair.
// kStats: sums of squares of 16 ticks fit in 32 bits (16 x 16383^2 < 2^32); they go to 64-bit registers after at most that many.
// kSpectra: each unit's pairs are staged in the warp's shared memory; a full segment adds its lags to the item's sums there (lane
// l reads and writes only its own column), which merge into HBM once per channel. The launch makes a WIB2 chunk a multiple of
// the segment's 4 units, so segments start at unit 0 of the link and only a link's last 1-3 units can be left over (not counted).
template<bool WIB2, bool kStats, bool kSpectra>
__global__ void __launch_bounds__(kStatsWarps * 32)
adc_stats_kernel(const uint8_t* __restrict__ frames, const uint32_t* __restrict__ n_units, uint32_t units_stride, uint32_t n_links,
                 uint32_t parts, uint32_t chunk, uint32_t adc_offset, swtpg_adc_stats* __restrict__ acc, swtpg_noise_lags* __restrict__ lag_acc)
{
  constexpr uint32_t kGroups = WIB2 ? SWTPG_WIB2_CHANNELS / 64 : 1;
  constexpr uint32_t kTicks = WIB2 ? SWTPG_WIB2_TICKS : SWTPG_WIBETH_TICKS;
  constexpr uint32_t kUnitBytes = WIB2 ? SWTPG_WIB2_SUPERCHUNK_BYTES : SWTPG_WIBETH_FRAME_BYTES;
  constexpr uint32_t kTickBytes = WIB2 ? SWTPG_WIB2_FRAME_BYTES : 112; // distance between consecutive rows of one group
  constexpr uint32_t kSqTicks = WIB2 ? kTicks : 16;                    // ticks summed in 32 bits before the 64-bit add
  using Sg = Segment<WIB2>;
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t item = blockIdx.x * kStatsWarps + (threadIdx.x >> 5);
  if (item >= n_links * kGroups * parts)
    return;
  const uint32_t link = item / (kGroups * parts);
  const uint32_t g = (item / parts) % kGroups;
  const uint32_t part = item % parts;
  const uint32_t units = n_units ? n_units[link] : units_stride;
  const uint32_t u0 = part * chunk;
  const uint32_t u1 = min(units, u0 + chunk);
  if (u0 >= u1)
    return;
  const PairPos pp = pair_pos(lane);
  const uint32_t row0 = WIB2 ? adc_offset + g * 112u : 32u; // byte offset of the group's first row inside a unit
  const uint8_t* base = frames + (size_t(link) * units_stride + u0) * kUnitBytes + row0;
  uint32_t sum_lo = 0, sum_hi = 0, mn = 0xFFFFFFFFu, mx = 0;
  uint64_t sq_lo = 0, sq_hi = 0;
  uint32_t* seg = nullptr;
  unsigned long long* lags = nullptr;
  if constexpr (kSpectra) {
    extern __shared__ __align__(16) uint8_t stats_smem[];
    seg = reinterpret_cast<uint32_t*>(stats_smem + (threadIdx.x >> 5) * Sg::kSmemBytes);
    lags = reinterpret_cast<unsigned long long*>(seg + Sg::kTicks * 32);
    for (uint32_t i = 0; i < Sg::kLags * 2; ++i)
      lags[i * 32 + lane] = 0;
  }
  for (uint32_t u = u0; u < u1; ++u, base += kUnitBytes) {
    uint32_t* useg = nullptr;
    if constexpr (kSpectra)
      useg = seg + ((u - u0) % Sg::kUnits) * kTicks * 32;
#pragma unroll
    for (uint32_t t0 = 0; t0 < kTicks; t0 += kSqTicks) {
      uint32_t q_lo = 0, q_hi = 0;
#pragma unroll
      for (uint32_t t = t0; t < t0 + kSqTicks; ++t) {
        const uint32_t* row = reinterpret_cast<const uint32_t*>(base + t * kTickBytes);
        const uint32_t pair = extract_pair(row, pp); // u16x2 {adc(2l), adc(2l+1)}
        if constexpr (kSpectra)
          useg[t * 32 + lane] = pair;
        if constexpr (kStats) {
          const uint32_t lo = pair & 0xFFFFu, hi = pair >> 16;
          sum_lo += lo;
          sum_hi += hi;
          q_lo += lo * lo;
          q_hi += hi * hi;
          mn = __vminu2(mn, pair);
          mx = __vmaxu2(mx, pair);
        }
      }
      if constexpr (kStats) {
        sq_lo += q_lo;
        sq_hi += q_hi;
      }
    }
    if constexpr (kSpectra)
      if ((u - u0) % Sg::kUnits == Sg::kUnits - 1)
        add_segment_lags<WIB2>(seg, lags, lane);
  }
  if constexpr (kStats) {
    // One merge per channel per item. Minimum and maximum both merge by atomicMax: the minimum is kept as 16383 - min, so zeroed
    // accumulators are an empty window (swtpg_read_adc_stats turns the encoding back).
    const unsigned long long samples = (unsigned long long)(u1 - u0) * kTicks;
    swtpg_adc_stats* a = acc + (size_t(link) * kGroups + g) * 64 + 2 * lane;
    auto merge = [&](swtpg_adc_stats* c, uint32_t sum, uint64_t sq, uint32_t lo, uint32_t hi) {
      atomicAdd(reinterpret_cast<unsigned long long*>(&c->samples), samples);
      atomicAdd(reinterpret_cast<unsigned long long*>(&c->sum), (unsigned long long)sum);
      atomicAdd(reinterpret_cast<unsigned long long*>(&c->sum_sq), (unsigned long long)sq);
      unsigned* ext = reinterpret_cast<unsigned*>(c) + 6; // the last 8 bytes: {16383 - min, max} as two words
      atomicMax(ext, 0x3FFFu - lo);
      atomicMax(ext + 1, hi);
    };
    merge(a, sum_lo, sq_lo, mn & 0xFFFFu, mx & 0xFFFFu);
    merge(a + 1, sum_hi, sq_hi, mn >> 16, mx >> 16);
  }
  if constexpr (kSpectra) {
    const unsigned long long segments = (u1 - u0) / Sg::kUnits;
    if (segments == 0)
      return;
    swtpg_noise_lags* l = lag_acc + (size_t(link) * kGroups + g) * 64 + 2 * lane;
    for (uint32_t half = 0; half < 2; ++half) {
      atomicAdd(reinterpret_cast<unsigned long long*>(&l[half].segments), segments);
      for (uint32_t tau = 0; tau < Sg::kLags; ++tau)
        atomicAdd(reinterpret_cast<unsigned long long*>(&l[half].lag[tau]), lags[(tau * 2 + half) * 32 + lane]);
    }
  }
}

template<bool WIB2, bool kStats, bool kSpectra>
cudaError_t
launch_form(unsigned grid, cudaStream_t s, const uint8_t* f, const uint32_t* d_nunits, uint32_t units_stride, uint32_t n_links, uint32_t parts,
            uint32_t chunk, uint32_t adc_offset, swtpg_handle* h)
{
  constexpr uint32_t smem = kSpectra ? kStatsWarps * Segment<WIB2>::kSmemBytes : 0;
  if constexpr (smem > 48 * 1024) {
    static int set_on[64]; // per device: the opt-in above 48 KB of dynamic shared memory is done
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess)
      return e;
    if (!set_on[dev]) {
      if ((e = cudaFuncSetAttribute(adc_stats_kernel<WIB2, kStats, kSpectra>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem))) != cudaSuccess)
        return e;
      set_on[dev] = 1;
    }
  }
  adc_stats_kernel<WIB2, kStats, kSpectra><<<grid, kStatsWarps * 32, smem, s>>>(f, d_nunits, units_stride, n_links, parts, chunk, adc_offset,
                                                                               h->d_adc_stats, h->d_noise_lags);
  return cudaGetLastError();
}

template<bool WIB2>
cudaError_t
launch_format(unsigned grid, cudaStream_t s, const uint8_t* f, const uint32_t* d_nunits, uint32_t units_stride, uint32_t n_links, uint32_t parts,
              uint32_t chunk, uint32_t adc_offset, swtpg_handle* h)
{
  if (!h->d_noise_lags)
    return launch_form<WIB2, true, false>(grid, s, f, d_nunits, units_stride, n_links, parts, chunk, adc_offset, h);
  if (!h->d_adc_stats)
    return launch_form<WIB2, false, true>(grid, s, f, d_nunits, units_stride, n_links, parts, chunk, adc_offset, h);
  return launch_form<WIB2, true, true>(grid, s, f, d_nunits, units_stride, n_links, parts, chunk, adc_offset, h);
}

// ---- channel products (SWTPG_FLAG_CHANNEL_COVARIANCE) ----------------------------------------------------------------------
constexpr uint32_t kProdWarps = 8;       // warps per CTA: 4 x 2 warp tiles of 16 x 32 products cover a 64 x 64 channel block
constexpr uint32_t kProdMaxUnits = 64;   // units per work item at most: keeps the byte-plane sums in 32 bits (static_assert below)
// Units per work item at least. An item ends with one 64-bit atomicAdd per product of its block (2080 for a WIBEth link, 4096
// for an off-diagonal WIB2 block) against 64 x 64 x ticks products of MMA work: split finer, the merges would set the time.
constexpr uint32_t kProdMinUnits = 16;
constexpr uint32_t kProdItemsPerSm = 8;  // work items (CTAs) per SM a launch aims for, as far as kProdMinUnits allows

template<bool WIB2>
struct ProductSlab
{
  static constexpr uint32_t kUnits = WIB2 ? 8 : 1; // units staged at once: 96 (WIB2) or 64 ticks, three or two K-steps of 32
  static constexpr uint32_t kTicks = kUnits * (WIB2 ? SWTPG_WIB2_TICKS : SWTPG_WIBETH_TICKS);
  static constexpr uint32_t kSteps = kTicks / 32;
  // One channel's row of a byte plane, 4 ticks per word, padded so that the stride is 4 x an odd number of words: the MMA
  // fragment loads (8 rows x 4 words) and the staging stores (4 channel pairs x 8 words) of a warp hit 32 different banks.
  static constexpr uint32_t kRowWords = kTicks / 4 + 4;
  static constexpr uint32_t kGroups = WIB2 ? 2 : 1; // 64-channel groups staged: I, and J of an off-diagonal block
};
static_assert(ProductSlab<false>::kTicks % 32 == 0 && ProductSlab<true>::kTicks % 32 == 0, "a slab is whole K-steps");
static_assert(ProductSlab<false>::kRowWords % 8 == 4 && ProductSlab<true>::kRowWords % 8 == 4, "conflict-free row stride");
// An item's HL + LH byte-plane sums, the largest, stay below 2^31: 2 x ticks x 255^2.
static_assert(2ull * kProdMaxUnits * SWTPG_WIBETH_TICKS * 255 * 255 < (1ull << 31), "int32 accumulators would overflow");
static_assert(kProdMaxUnits % ProductSlab<true>::kUnits == 0 && kProdMinUnits % ProductSlab<true>::kUnits == 0, "whole slabs");

// d += a b over one m16n8k32 tile: u8 x u8 products summed in s32 (IMMA.16832.U8.U8).
__device__ __forceinline__ void
imma_u8(int32_t (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2])
{
  asm("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+r"(d[0]), "+r"(d[1]), "+r"(d[2]), "+r"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

// Work item i of the launch: link i / (kPairs * parts), units [part * chunk, part * chunk + chunk) with part = i / kPairs % parts,
// and the pair (I, J), I <= J, of 64-channel groups with index i % kPairs: a WIBEth link is the one block (0, 0), a WIB2 link
// has 4 diagonal and 6 off-diagonal blocks. One CTA per item.
// Exact split: x < 2^14 is 256 h + l with bytes h = x >> 8 and l = x & 0xFF, so sum x_i x_j = 2^16 HH + 2^8 (HL + LH) + LL,
// each a sum of u8 x u8 products. The CTA stages a slab of ticks of groups I and J as byte planes [channel][tick] in shared memory
// (4 ticks per word, which is the layout of both MMA fragments: A row-major and B column-major are channel-major with ticks
// contiguous), then warp w sums rows 16 (w % 4) .. + 15 against columns 32 (w / 4) .. + 31 of the block over K-steps of 32 ticks.
// A diagonal block sums HH and LL only on tiles that touch the upper triangle, and HL in full (its LH is HL transposed); an
// off-diagonal block sums all four, HL and LH into one accumulator. At the end of the item the terms are combined in 64 bits and
// merged into HBM with 64-bit atomics, once per product of the block; samples come from block (0, 0) and the sums of a group's
// channels from its diagonal block.
template<bool WIB2>
__global__ void __launch_bounds__(kProdWarps * 32)
channel_products_kernel(const uint8_t* __restrict__ frames, const uint32_t* __restrict__ n_units, uint32_t units_stride, uint32_t parts,
                        uint32_t chunk, uint32_t adc_offset, unsigned long long* __restrict__ acc)
{
  using Sl = ProductSlab<WIB2>;
  constexpr uint32_t C = WIB2 ? SWTPG_WIB2_CHANNELS : SWTPG_WIBETH_CHANNELS;
  constexpr uint32_t kGroups = C / 64;
  constexpr uint32_t kPairs = kGroups * (kGroups + 1) / 2;
  constexpr uint32_t kWords = SWTPG_CHANNEL_PRODUCTS_WORDS(C);
  constexpr uint32_t kTicks = WIB2 ? SWTPG_WIB2_TICKS : SWTPG_WIBETH_TICKS;
  constexpr uint32_t kUnitBytes = WIB2 ? SWTPG_WIB2_SUPERCHUNK_BYTES : SWTPG_WIBETH_FRAME_BYTES;
  constexpr uint32_t kTickBytes = WIB2 ? SWTPG_WIB2_FRAME_BYTES : 112; // distance between consecutive rows of one group
  static_assert(kTicks % 4 == 0, "a staged word of 4 ticks never spans two units");
  __shared__ uint32_t planes[Sl::kGroups][2][64][Sl::kRowWords]; // [I / J][high / low byte][channel of the group][tick / 4]
  __shared__ int32_t mid[64][65];                                // the item's HL (+ LH) sums, transposed for a diagonal block

  const uint32_t pair = blockIdx.x % kPairs;
  const uint32_t part = (blockIdx.x / kPairs) % parts;
  const uint32_t link = blockIdx.x / (kPairs * parts);
  uint32_t I = 0, r = pair;
  while (r >= kGroups - I) {
    r -= kGroups - I;
    ++I;
  }
  const uint32_t J = I + r;
  const bool diag = I == J;
  const uint32_t units = n_units ? n_units[link] : units_stride;
  const uint32_t u0 = part * chunk;
  const uint32_t u1 = min(units, u0 + chunk);
  if (u0 >= u1)
    return;
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  // staging: the thread's lane pair sp (channels 2 sp and 2 sp + 1 of a group) and words sq + 8 k of each plane row of a slab
  const uint32_t sp = warp * 4 + (lane >> 3), sq = lane & 7u;
  const PairPos pp = pair_pos(sp);
  // MMA fragments (PTX m16n8k32 .u8): g = row of A / column of B, tig = word of 4 ticks within each half K-step
  const uint32_t mi = warp & 3u, nh = warp >> 2, g = lane >> 2, tig = lane & 3u;
  const uint32_t sb = WIB2 && !diag ? 1 : 0; // staged plane set of group J
  int32_t hh[4][4] = {}, hl[4][4] = {}, ll[4][4] = {};
  uint32_t sum_a = 0, sum_b = 0;
  const uint8_t* link_frames = frames + size_t(link) * units_stride * kUnitBytes;

  for (uint32_t us = u0; us < u1; us += Sl::kUnits) {
    for (uint32_t s = 0; s < (diag ? 1u : 2u); ++s) {
      const uint32_t row0 = WIB2 ? adc_offset + (s ? J : I) * 112u : 32u; // byte offset of the group's first row inside a unit
#pragma unroll
      for (uint32_t k = 0; k < Sl::kSteps; ++k) {
        const uint32_t q = sq + 8 * k, t = 4 * q; // word q: ticks t .. t + 3 of the slab, all in unit us + t / kTicks
        const uint32_t u = us + t / kTicks;
        uint32_t p[4] = { 0, 0, 0, 0 }; // past the item's units: zeros, which add nothing
        if (u < u1) {
          const uint8_t* row = link_frames + size_t(u) * kUnitBytes + row0 + (t % kTicks) * kTickBytes;
#pragma unroll
          for (uint32_t j = 0; j < 4; ++j)
            p[j] = extract_pair(reinterpret_cast<const uint32_t*>(row + j * kTickBytes), pp); // u16x2 {adc(2 sp), adc(2 sp + 1)}
        }
        if (diag) {
          sum_a += (p[0] & 0xFFFFu) + (p[1] & 0xFFFFu) + (p[2] & 0xFFFFu) + (p[3] & 0xFFFFu);
          sum_b += (p[0] >> 16) + (p[1] >> 16) + (p[2] >> 16) + (p[3] >> 16);
        }
        const uint32_t a01 = __byte_perm(p[0], p[1], 0x5140), a23 = __byte_perm(p[2], p[3], 0x5140); // {l0, l1, h0, h1} of 2 sp
        const uint32_t b01 = __byte_perm(p[0], p[1], 0x7362), b23 = __byte_perm(p[2], p[3], 0x7362); // of 2 sp + 1
        planes[s][0][2 * sp][q] = __byte_perm(a01, a23, 0x7632);
        planes[s][1][2 * sp][q] = __byte_perm(a01, a23, 0x5410);
        planes[s][0][2 * sp + 1][q] = __byte_perm(b01, b23, 0x7632);
        planes[s][1][2 * sp + 1][q] = __byte_perm(b01, b23, 0x5410);
      }
    }
    __syncthreads();
#pragma unroll
    for (uint32_t k = 0; k < Sl::kSteps; ++k) {
      const uint32_t w = 8 * k + tig, ra = 16 * mi + g;
      const uint32_t ah[4] = { planes[0][0][ra][w], planes[0][0][ra + 8][w], planes[0][0][ra][w + 4], planes[0][0][ra + 8][w + 4] };
      const uint32_t al[4] = { planes[0][1][ra][w], planes[0][1][ra + 8][w], planes[0][1][ra][w + 4], planes[0][1][ra + 8][w + 4] };
#pragma unroll
      for (uint32_t n = 0; n < 4; ++n) {
        const uint32_t nt = 4 * nh + n, rb = 8 * nt + g;
        const uint32_t bh[2] = { planes[sb][0][rb][w], planes[sb][0][rb][w + 4] };
        const uint32_t bl[2] = { planes[sb][1][rb][w], planes[sb][1][rb][w + 4] };
        imma_u8(hl[n], ah, bl);
        if (!diag)
          imma_u8(hl[n], al, bh);
        if (!diag || 8 * nt + 7 >= 16 * mi) { // the tile touches the upper triangle
          imma_u8(hh[n], ah, bh);
          imma_u8(ll[n], al, bl);
        }
      }
    }
    __syncthreads();
  }

  // C fragment element e of tile n: row 16 mi + g (+ 8 for e >= 2), column 8 nt + 2 tig (+ 1 for odd e)
#pragma unroll
  for (uint32_t n = 0; n < 4; ++n)
#pragma unroll
    for (uint32_t e = 0; e < 4; ++e)
      mid[16 * mi + g + 8 * (e >> 1)][8 * (4 * nh + n) + 2 * tig + (e & 1)] = hl[n][e];
  __syncthreads();
  unsigned long long* a = acc + size_t(link) * kWords;
#pragma unroll
  for (uint32_t n = 0; n < 4; ++n)
#pragma unroll
    for (uint32_t e = 0; e < 4; ++e) {
      const uint32_t rr = 16 * mi + g + 8 * (e >> 1), cc = 8 * (4 * nh + n) + 2 * tig + (e & 1);
      if (diag && rr > cc)
        continue;
      // all sums are of non-negative products, below 2^31 (HL + LH below 2^32 for a diagonal block)
      const uint64_t m = diag ? uint64_t(uint32_t(mid[rr][cc])) + uint32_t(mid[cc][rr]) : uint64_t(uint32_t(mid[rr][cc]));
      const uint64_t v = (uint64_t(uint32_t(hh[n][e])) << 16) + (m << 8) + uint32_t(ll[n][e]);
      const uint32_t i = 64 * I + rr, j = 64 * J + cc;
      atomicAdd(a + 1 + C + i * (2 * C + 1 - i) / 2 + (j - i), (unsigned long long)v);
    }
  if (diag) {
    for (uint32_t o = 1; o < 8; o <<= 1) { // the 8 lanes of lane pair sp
      sum_a += __shfl_xor_sync(0xFFFFFFFFu, sum_a, o);
      sum_b += __shfl_xor_sync(0xFFFFFFFFu, sum_b, o);
    }
    if (sq == 0) {
      atomicAdd(a + 1 + 64 * I + 2 * sp, (unsigned long long)sum_a);
      atomicAdd(a + 1 + 64 * I + 2 * sp + 1, (unsigned long long)sum_b);
    }
    if (I == 0 && threadIdx.x == 0)
      atomicAdd(a, (unsigned long long)(u1 - u0) * kTicks);
  }
}

template<bool WIB2>
cudaError_t
launch_products(int sms, cudaStream_t s, const uint8_t* f, const uint32_t* d_nunits, uint32_t units_stride, uint32_t adc_offset, swtpg_handle* h)
{
  constexpr uint32_t kGroups = (WIB2 ? SWTPG_WIB2_CHANNELS : SWTPG_WIBETH_CHANNELS) / 64;
  const uint32_t n = h->cfg.n_links * (kGroups * (kGroups + 1) / 2);
  const uint32_t want = (uint32_t(sms) * kProdItemsPerSm + n - 1) / n;
  uint32_t parts = std::max(want, (units_stride + kProdMaxUnits - 1) / kProdMaxUnits);
  parts = std::max(1u, std::min(parts, units_stride));
  uint32_t chunk = std::max((units_stride + parts - 1) / parts, kProdMinUnits);
  chunk = std::min(kProdMaxUnits, (chunk + ProductSlab<WIB2>::kUnits - 1) / ProductSlab<WIB2>::kUnits * ProductSlab<WIB2>::kUnits);
  parts = (units_stride + chunk - 1) / chunk;
  const uint64_t grid = uint64_t(n) * parts;
  if (grid == 0)
    return cudaSuccess;
  channel_products_kernel<WIB2><<<unsigned(grid), kProdWarps * 32, 0, s>>>(f, d_nunits, units_stride, parts, chunk, adc_offset,
                                                                          reinterpret_cast<unsigned long long*>(h->d_channel_products));
  return cudaGetLastError();
}

} // namespace

cudaError_t
swtpg_internal::launch_channel_stats(swtpg_handle* h, const void* d_frames, const uint32_t* d_nunits, uint32_t units_stride, cudaStream_t s)
{
  static int sm_count[64]; // per device, 0 = not queried yet
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess)
    return e;
  if (dev < 0 || dev >= 64)
    return cudaErrorInvalidDevice;
  if (sm_count[dev] == 0) {
    int sms = 0;
    if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess)
      return e;
    sm_count[dev] = std::max(1, sms);
  }
  const bool wib2 = h->cfg.format == SWTPG_FORMAT_WIB2;
  const uint32_t n = h->cfg.n_links * h->groups_per_link;
  // Split each link's units so that a few links (one APA = 40 links) still fill the GPU, into chunks of at most kStatsMaxUnits.
  const uint32_t want = (uint32_t(sm_count[dev]) * kStatsItemsPerSm + n - 1) / n;
  uint32_t parts = std::max(want, (units_stride + kStatsMaxUnits - 1) / kStatsMaxUnits);
  parts = std::max(1u, std::min(parts, units_stride));
  uint32_t chunk = (units_stride + parts - 1) / parts;
  if (wib2 && h->d_noise_lags) // whole segments from unit 0 of the link; still at most kStatsMaxUnits, a multiple of 4
    chunk = (chunk + Segment<true>::kUnits - 1) / Segment<true>::kUnits * Segment<true>::kUnits;
  parts = (units_stride + chunk - 1) / chunk;
  const uint64_t items = uint64_t(n) * parts;
  const unsigned grid = unsigned((items + kStatsWarps - 1) / kStatsWarps);
  const uint8_t* f = static_cast<const uint8_t*>(d_frames);
  std::lock_guard<std::mutex> lk(h->stats_mu); // no read can fall between this launch and the record of ev_stats
  if (h->stats_stream && h->stats_stream != s && (e = cudaStreamWaitEvent(s, h->ev_stats, 0)) != cudaSuccess)
    return e;
  if (h->d_adc_stats || h->d_noise_lags) {
    e = wib2 ? launch_format<true>(grid, s, f, d_nunits, units_stride, h->cfg.n_links, parts, chunk, h->cfg.wib2_adc_offset, h)
             : launch_format<false>(grid, s, f, d_nunits, units_stride, h->cfg.n_links, parts, chunk, 0, h);
    if (e != cudaSuccess)
      return e;
  }
  if (h->d_channel_products) {
    e = wib2 ? launch_products<true>(sm_count[dev], s, f, d_nunits, units_stride, h->cfg.wib2_adc_offset, h)
             : launch_products<false>(sm_count[dev], s, f, d_nunits, units_stride, 0, h);
    if (e != cudaSuccess)
      return e;
  }
  h->stats_stream = s;
  return cudaEventRecord(h->ev_stats, s);
}
