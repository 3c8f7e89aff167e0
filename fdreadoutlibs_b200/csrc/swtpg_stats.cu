// Per-channel statistics of the raw ADC values: one streaming read of every batch after its TPG launches, on the same stream.
//   SWTPG_FLAG_ADC_STATS      per (link, frame channel): samples, sum, sum of squares, minimum and maximum, into 32-byte
//                             accumulators in HBM (swtpg_handle::d_adc_stats), copied out by swtpg_read_adc_stats.
//   SWTPG_FLAG_NOISE_SPECTRA  per (link, frame channel): the segments counted and the circular lag sums of each segment,
//                             lag[tau] = sum_t x[t] x[(t + tau) mod N] for tau = 0..N/2 (swtpg_handle::d_noise_lags), copied out by
//                             swtpg_read_noise_lags; swtpg_noise_power turns them into the averaged periodogram on the host.
// With both flags one kernel reads the batch once.
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
  e = wib2 ? launch_format<true>(grid, s, f, d_nunits, units_stride, h->cfg.n_links, parts, chunk, h->cfg.wib2_adc_offset, h)
           : launch_format<false>(grid, s, f, d_nunits, units_stride, h->cfg.n_links, parts, chunk, 0, h);
  if (e != cudaSuccess)
    return e;
  h->stats_stream = s;
  return cudaEventRecord(h->ev_stats, s);
}
