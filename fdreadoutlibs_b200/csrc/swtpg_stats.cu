// Per-channel ADC statistics (SWTPG_FLAG_ADC_STATS): one streaming read of every batch after its TPG launches, on the same stream.
// It accumulates, per (link, frame channel), the samples, sum, sum of squares, minimum and maximum of the raw 14-bit ADC values
// into 32-byte accumulators in HBM (swtpg_handle::d_adc_stats), which swtpg_read_adc_stats copies out by windows.
#include "swtpg_device.cuh"
#include "swtpg_handle.h"

#include <algorithm>

using namespace swtpg;

namespace {

constexpr uint32_t kStatsWarps = 4;       // warps per CTA
constexpr uint32_t kStatsMaxUnits = 64;   // units per work item at most: keeps the per-item sums in 32 bits (64 x 64 x 16383 < 2^32)
constexpr uint32_t kStatsItemsPerSm = 48; // work items per SM a launch aims for (a few links are split finer, down to one unit)

// Work item i of the launch: link i / (groups * parts), its 64-channel group, and units [part * chunk, part * chunk + chunk).
// One warp per item; lane l owns frame channels 64 g + 2l and 64 g + 2l + 1, extracted from each 112-byte row by extract_pair.
// Sums of squares of 16 ticks fit in 32 bits (16 x 16383^2 < 2^32); they go to 64-bit registers after at most that many.
template<bool WIB2>
__global__ void __launch_bounds__(kStatsWarps * 32)
adc_stats_kernel(const uint8_t* __restrict__ frames, const uint32_t* __restrict__ n_units, uint32_t units_stride, uint32_t n_links,
                 uint32_t parts, uint32_t chunk, uint32_t adc_offset, swtpg_adc_stats* __restrict__ acc)
{
  constexpr uint32_t kGroups = WIB2 ? SWTPG_WIB2_CHANNELS / 64 : 1;
  constexpr uint32_t kTicks = WIB2 ? SWTPG_WIB2_TICKS : SWTPG_WIBETH_TICKS;
  constexpr uint32_t kUnitBytes = WIB2 ? SWTPG_WIB2_SUPERCHUNK_BYTES : SWTPG_WIBETH_FRAME_BYTES;
  constexpr uint32_t kTickBytes = WIB2 ? SWTPG_WIB2_FRAME_BYTES : 112; // distance between consecutive rows of one group
  constexpr uint32_t kSqTicks = WIB2 ? kTicks : 16;                    // ticks summed in 32 bits before the 64-bit add
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
  for (uint32_t u = u0; u < u1; ++u, base += kUnitBytes) {
#pragma unroll
    for (uint32_t t0 = 0; t0 < kTicks; t0 += kSqTicks) {
      uint32_t q_lo = 0, q_hi = 0;
#pragma unroll
      for (uint32_t t = t0; t < t0 + kSqTicks; ++t) {
        const uint32_t* row = reinterpret_cast<const uint32_t*>(base + t * kTickBytes);
        const uint32_t pair = extract_pair(row, pp); // u16x2 {adc(2l), adc(2l+1)}
        const uint32_t lo = pair & 0xFFFFu, hi = pair >> 16;
        sum_lo += lo;
        sum_hi += hi;
        q_lo += lo * lo;
        q_hi += hi * hi;
        mn = __vminu2(mn, pair);
        mx = __vmaxu2(mx, pair);
      }
      sq_lo += q_lo;
      sq_hi += q_hi;
    }
  }
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

} // namespace

cudaError_t
swtpg_internal::launch_adc_stats(swtpg_handle* h, const void* d_frames, const uint32_t* d_nunits, uint32_t units_stride, cudaStream_t s)
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
  const uint32_t chunk = (units_stride + parts - 1) / parts;
  parts = (units_stride + chunk - 1) / chunk;
  const uint64_t items = uint64_t(n) * parts;
  const unsigned grid = unsigned((items + kStatsWarps - 1) / kStatsWarps);
  const uint8_t* f = static_cast<const uint8_t*>(d_frames);
  std::lock_guard<std::mutex> lk(h->stats_mu); // no read can fall between this launch and the record of ev_stats
  if (h->stats_stream && h->stats_stream != s && (e = cudaStreamWaitEvent(s, h->ev_stats, 0)) != cudaSuccess)
    return e;
  if (wib2)
    adc_stats_kernel<true><<<grid, kStatsWarps * 32, 0, s>>>(f, d_nunits, units_stride, h->cfg.n_links, parts, chunk, h->cfg.wib2_adc_offset,
                                                             h->d_adc_stats);
  else
    adc_stats_kernel<false><<<grid, kStatsWarps * 32, 0, s>>>(f, d_nunits, units_stride, h->cfg.n_links, parts, chunk, 0, h->d_adc_stats);
  if ((e = cudaGetLastError()) != cudaSuccess)
    return e;
  h->stats_stream = s;
  return cudaEventRecord(h->ev_stats, s);
}
