// Host runtime behind include/swtpg.h: device buffers, kernel selection and the batch entry points. The streaming path
// (swtpg_submit ... swtpg_poll) lives in swtpg_stream.cu. Plain CUDA runtime; no torch, no CPU compute fallback.
#include "swtpg_handle.h"
#include "swtpg_kernels.cuh"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

using namespace swtpg;
using swtpg_internal::ConfGroup;
using swtpg_internal::fail;
using swtpg_internal::Policy;
using swtpg_internal::TpgConf;

// Layouts the ctypes binding (fdreadoutlibs_b200/_lib.py, frames.py) relies on.
static_assert(sizeof(swtpg_tp) == 32, "swtpg_tp must stay 32 bytes (two 16-byte device stores)");
static_assert(sizeof(swtpg_config) == 72, "swtpg_config layout changed: bump SWTPG_ABI_VERSION and the bindings");
static_assert(sizeof(swtpg_channel_state) == 48, "swtpg_channel_state layout changed");
static_assert(sizeof(swtpg_counters) == 80, "swtpg_counters layout changed");
static_assert(sizeof(swtpg_link_config) == 36, "swtpg_link_config layout changed");
static_assert(sizeof(swtpg_adc_stats) == 32, "swtpg_adc_stats layout changed");
static_assert(sizeof(swtpg_noise_lags) == 272, "swtpg_noise_lags layout changed");
static_assert(SWTPG_CHANNEL_PRODUCTS_WORDS(SWTPG_WIBETH_CHANNELS) == 2145 && SWTPG_CHANNEL_PRODUCTS_WORDS(SWTPG_WIB2_CHANNELS) == 33153,
              "swtpg_read_channel_products layout changed");

namespace {
thread_local std::string g_create_error;
thread_local std::string g_error_copy;
}
void
swtpg_internal::set_create_error(const char* msg)
{
  g_create_error = msg;
}

namespace {

// ---- kernel launch table ------------------------------------------------------------------------------------------
// CTAs of persistent kernel K the whole GPU holds at once (SMs x resident CTAs per SM, the latter capped at `cap` if cap > 0),
// and the SM count. Queried once per kernel and device.
template<auto K>
cudaError_t
residency(int threads, size_t smem, int cap, unsigned* resident, unsigned* sms)
{
  static int res[64], sm[64]; // 0 = not queried yet
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess)
    return e;
  if (dev < 0 || dev >= 64)
    return cudaErrorInvalidDevice;
  if (res[dev] == 0) {
    e = cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess)
      return e;
    int per_sm = 0, n = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, K, threads, smem);
    if (e != cudaSuccess)
      return e;
    e = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess)
      return e;
    if (cap > 0) // the policy's measured optimum, if the device holds that many
      per_sm = std::min(per_sm, cap);
    sm[dev] = std::max(1, n);
    res[dev] = std::max(1, per_sm * n);
  }
  *resident = unsigned(res[dev]);
  *sms = unsigned(sm[dev]);
  return cudaSuccess;
}

// One-warp-per-CTA form of the WIBEth kernel, persistent: at most as many CTAs as the device holds at once; warps claim links
// dynamically (wibeth_kernel), so the grid only has to load every SM sub-partition alike: a multiple of 4 single-warp CTAs per
// SM, capped at the policy's warps per SM (20 on B200: 5 warps per sub-partition; a 21st warp would make one sub-partition of
// every SM 20 % slower than its neighbours — profiles/README.md). From the policy's full-load link count on it runs its
// full-load warps per SM and slices the links even when their number is a whole multiple of the persistent warps.
template<class Algo, bool DUMP>
cudaError_t
launch_wibeth_geo(const KernelParams& kp, cudaStream_t s)
{
  constexpr auto k = wibeth_kernel<Algo, DUMP>;
  constexpr size_t smem = WibEthSmem::total;
  unsigned resident = 0, sms = 0;
  const cudaError_t e = residency<k>(32, smem, 0, &resident, &sms);
  if (e != cudaSuccess)
    return e;
  const bool full_load = Algo::kFullLoadWarpsPerSm > 0 && kp.n_links >= Algo::kFullLoadWarpsPerSm * sms + Algo::kFullLoadExtraLinks;
  const unsigned warps_per_sm = full_load ? Algo::kFullLoadWarpsPerSm : Algo::kWarpsPerSm;
  const unsigned per_sm = resident / sms;
  unsigned even = per_sm >= 4 ? per_sm / 4 * 4 : per_sm;
  if (warps_per_sm > 0) // the measured optimum, if the device holds that many
    even = std::min(even, warps_per_sm);
  const unsigned grid = std::min<unsigned>(std::min<unsigned>(kp.n_links, even * sms), resident);
  // More links than persistent warps = several rounds of links per warp, and whatever the last round leaves idle is lost (round 2,
  // straight-line SimpleThreshold policy: 6000 links on 4144 warps 64.9 % of the HBM peak, 8288 = two full rounds 73.0 %). Handing
  // the links out in 4 HALVING slices (n/2, n/4, n/8, n/8 units) makes the rounds short, at the price of the extra state round
  // trips (about 3 % per launch): what the launch's last round leaves idle is at most one LAST slice, so small last slices shorten
  // the tail without more round trips per link than four equal ones (pipelined SimpleThreshold policy at 20 warps per SM, 5920
  // links: whole links 68.9 %, equal slices 70.8 %, halving 73.1 %; 6000 links 71.0 -> 73.3 %; AbsRS + 2.5 %;
  // profiles/r02_halving_slices_probe.txt).
  //   * Below full load a link count that is a whole number of rounds keeps whole links (straight-line form, 8288 links: 73.0 %
  //     against 70.8 % sliced); at full load the policies gain from slices even then.
  // A launch that cannot fill the GPU keeps whole links: time is sequential per link, slices could only wait for each other.
  KernelParams kq = kp;
  unsigned parts = 1;
  if (kp.n_links > grid && (full_load || kp.n_links % grid != 0))
    parts = std::max(1u, std::min(4u, kp.units_stride / 16u));
  // Test hook: SWTPG_PARTS=n hands every launch out in n slices (at most 8), so that the GPU suite can run its cases with every
  // link sliced (tests/test_gpu_parity.py::test_links_handed_out_in_slices).
  static const int parts_override = [] { const char* e = getenv("SWTPG_PARTS"); return e ? atoi(e) : 0; }();
  if (parts_override > 0)
    parts = std::min(unsigned(parts_override), 8u);
  kq.parts_log2 = 0;
  while ((2u << kq.parts_log2) <= parts) // the largest power of two not above it
    ++kq.parts_log2;
  kq.slice_geom = 1u; // halving slices
  k<<<grid, 32, smem, s>>>(kq);
  return cudaGetLastError();
}

// CTA form of the WIBEth kernel (wibeth_quad_kernel): 4 consumer warps + 1 producer warp per quad of links.
template<class Algo, bool DUMP>
cudaError_t
launch_wibeth_quad(const KernelParams& kp, cudaStream_t s)
{
  constexpr auto k = wibeth_quad_kernel<Algo, DUMP>;
  constexpr size_t smem = WibEthQuadSmem::total;
  unsigned resident = 0, sms = 0;
  const cudaError_t e = residency<k>((kQuad + 1) * 32, smem, Algo::kQuadCtasPerSm, &resident, &sms);
  if (e != cudaSuccess)
    return e;
  const unsigned quads = (kp.n_links + kQuad - 1) / kQuad;
  const unsigned grid = std::min<unsigned>(quads, resident); // persistent CTAs claim quads dynamically
  k<<<grid, (kQuad + 1) * 32, smem, s>>>(kp);
  return cudaGetLastError();
}

// Which form of the WIBEth kernel a policy runs is a measured choice (profiles/r01_quad_vs_warp.txt): the CTA form is 14 % faster
// for FIR + IQR (ptxas needs 64 registers instead of 109 for it, so 20 consumer warps fit an SM), the one-warp-per-CTA form
// 2-5 % faster for SimpleThreshold and the running sums (the quad's lock-step costs more than the producer bookkeeping it
// saves).
// WIBEth SimpleThreshold, the production algorithm, runs the software-pipelined form of its policy (prefetch of the next group's
// rows + deferred quiet test, PackedSimpleT<true>, 92 registers) on every launch since its dependent chain lost an instruction
// (the accumulator reset as one IMAD): with 20 warps per SM and halving slices it beats the straight-line form with 28 at every
// link count — 5920 links 73.1 % against 67.8 % of the HBM peak, 6000 links 73.3 / 67.8 %, 8288 links 74.3 / 73.2 %, 4440 links
// 72.1 / 67.6 % — except on a dense-hit batch (20.2 / 21.0 %) (profiles/r02_simple_pipeline_sweep.txt,
// profiles/r02_halving_slices_probe.txt).
template<class Algo, bool DUMP>
cudaError_t
launch_wibeth(const KernelParams& kp, cudaStream_t s)
{
  if constexpr (Algo::kQuadCtasPerSm > 0)
    return launch_wibeth_quad<Algo, DUMP>(kp, s);
  else
    return launch_wibeth_geo<Algo, DUMP>(kp, s);
}

// WIB2: one CTA (4 consumer warps + 1 producer warp) per link at a time, ring of 4 superchunks; persistent over links.
template<class Algo, bool DUMP>
cudaError_t
launch_wib2(const KernelParams& kp, cudaStream_t s)
{
  constexpr int kStages = 4;
  constexpr auto k = wib2_kernel<Algo, kStages, DUMP>;
  constexpr size_t smem = Wib2Smem<kStages>::total;
  unsigned resident = 0, sms = 0;
  const cudaError_t e = residency<k>((kWib2Warps + 1) * 32, smem, 0, &resident, &sms);
  if (e != cudaSuccess)
    return e;
  const unsigned grid = std::min<unsigned>(kp.n_links, resident); // persistent CTAs claim links dynamically
  k<<<grid, (kWib2Warps + 1) * 32, smem, s>>>(kp); // 4 consumer warps + the producer warp
  return cudaGetLastError();
}

template<bool DUMP>
cudaError_t
launch(Policy policy, const KernelParams& kp, cudaStream_t s)
{
  switch (policy) {
    case Policy::WibEthSimple: return launch_wibeth<PackedSimpleWibEthPipe, DUMP>(kp, s);
    case Policy::WibEthAbsRs: return launch_wibeth<PackedRsWibEth<false>, DUMP>(kp, s);
    case Policy::WibEthStandardRs: return launch_wibeth<PackedRsWibEth<true>, DUMP>(kp, s);
    case Policy::WibEthFir: return launch_wibeth<PackedFirIqr, DUMP>(kp, s);
    case Policy::WibEthFirAnyTaps: return launch_wibeth<PackedFirIqrAnyTaps, DUMP>(kp, s);
    case Policy::WibEthScalarSimple: return launch_wibeth<ScalarAlgo<SWTPG_ALGO_SIMPLE_THRESHOLD, false>, DUMP>(kp, s);
    case Policy::WibEthScalarAbsRs: return launch_wibeth<ScalarAlgo<SWTPG_ALGO_ABS_RS, false>, DUMP>(kp, s);
    case Policy::WibEthScalarStandardRs: return launch_wibeth<ScalarAlgo<SWTPG_ALGO_STANDARD_RS, false>, DUMP>(kp, s);
    case Policy::WibEthScalarFir: return launch_wibeth<ScalarAlgo<SWTPG_ALGO_FIR_IQR, false>, DUMP>(kp, s);
    case Policy::Wib2Simple: return launch_wib2<PackedSimpleWib2, DUMP>(kp, s);
    case Policy::Wib2AbsRs: return launch_wib2<PackedRsIqrWib2, DUMP>(kp, s);
    case Policy::Wib2Fir: return launch_wib2<PackedFirIqr, DUMP>(kp, s);
    case Policy::Wib2FirAnyTaps: return launch_wib2<PackedFirIqrAnyTaps, DUMP>(kp, s);
    case Policy::Wib2ScalarSimple: return launch_wib2<ScalarAlgo<SWTPG_ALGO_SIMPLE_THRESHOLD, true>, DUMP>(kp, s);
    case Policy::Wib2ScalarAbsRs: return launch_wib2<ScalarAlgo<SWTPG_ALGO_ABS_RS, true>, DUMP>(kp, s);
    case Policy::Wib2ScalarFir: return launch_wib2<ScalarAlgo<SWTPG_ALGO_FIR_IQR, true>, DUMP>(kp, s);
  }
  return cudaErrorNotSupported;
}

// Kernel parameters of one configuration group's launch.
KernelParams
make_params(const swtpg_handle* h, const ConfGroup& g, const void* d_frames, const uint32_t* d_nunits, uint32_t stride, swtpg_tp* d_tps,
            unsigned* d_count, int16_t* ped, int16_t* wav)
{
  const TpgConf& c = h->confs[g.conf];
  KernelParams kp{};
  kp.frames = static_cast<const uint8_t*>(d_frames);
  kp.n_units = d_nunits;
  kp.units_stride = stride;
  kp.n_links = g.n_links;
  kp.link_ids = g.d_links;
  kp.state = h->d_state;
  kp.group_flags = h->d_flags;
  kp.link_cursor = g.d_cursor;
  kp.link_done = h->d_link_cursor + 2 * SWTPG_MAX_LINK_CONFIGS;
  kp.parts_log2 = 0;
  kp.sink.buf = d_tps;
  kp.sink.count = d_count;
  kp.sink.cap = h->tp_capacity;
  kp.pedestal_out = ped;
  kp.waveform_out = wav;
  kp.threshold = c.threshold;
  kp.acc_limit = c.frugal_acc_limit;
  kp.acc_limit_neg = 0u - (uint32_t(c.frugal_acc_limit) & 0xFFFFu);
  kp.rs_scale = int16_t(c.rs_scale_factor);
  kp.tap_exponent = c.tap_exponent;
  for (int i = 0; i < 8; ++i)
    kp.taps[i] = c.fir_taps[i];
  kp.wib2_adc_offset = h->cfg.wib2_adc_offset;
  kp.debug_flags = c.fir_force_exact ? 1u : 0u;
  kp.all_ones = 0xFFFFFFFFu;
  kp.one = 1u;
  return kp;
}

// One batch = one launch per configuration group. The groups run one after another on the same stream, never concurrently:
// a warp's first work item is fixed by its warp index rather than claimed, so a later slice of a link can wait for a warp of
// its own grid that is not resident yet. Every persistent grid is sized to the whole GPU, so two sliced grids running at once
// could fill the SMs with warps that all spin on warps of their own grid which can never become resident: a deadlock.
template<bool DUMP>
cudaError_t
launch_groups(const swtpg_handle* h, const void* d_frames, const uint32_t* d_nunits, uint32_t stride, swtpg_tp* d_tps, unsigned* d_count,
              int16_t* ped, int16_t* wav, cudaStream_t s)
{
  for (const ConfGroup& g : h->conf_groups) {
    const cudaError_t e = launch<DUMP>(h->confs[g.conf].policy, make_params(h, g, d_frames, d_nunits, stride, d_tps, d_count, ped, wav), s);
    if (e != cudaSuccess)
      return e;
  }
  return cudaSuccess;
}

// The configuration groups of the links' current configurations (swtpg_start): one per entry of h->confs in use, its links in
// ascending order. A handle whose links all run one configuration launches as before any link had its own: link_ids = nullptr.
swtpg_status
form_conf_groups(swtpg_handle* h)
{
  std::vector<uint32_t> links;
  std::vector<ConfGroup> groups;
  for (uint32_t c = 0; c < h->confs.size(); ++c) {
    const size_t first = links.size();
    for (uint32_t l = 0; l < h->cfg.n_links; ++l)
      if (h->link_conf[l] == c)
        links.push_back(l);
    if (links.size() == first)
      continue;
    ConfGroup g;
    g.conf = c;
    g.n_links = uint32_t(links.size() - first);
    g.d_links = h->d_group_links + first;
    g.d_cursor = h->d_link_cursor + 2 * groups.size();
    groups.push_back(g);
  }
  if (groups.size() == 1)
    groups[0].d_links = nullptr;
  else
    SW_CUDA(h, cudaMemcpyAsync(h->d_group_links, links.data(), links.size() * 4, cudaMemcpyHostToDevice, h->stream));
  SW_CUDA(h, cudaStreamSynchronize(h->stream));
  h->conf_groups = std::move(groups);
  h->conf_groups_stale = false;
  return SWTPG_OK;
}

// The SV_RS_FACTOR row (u16x2 by lane) of 64-channel state group g: the link's per-channel table h->h_rs_factor where it has one,
// else its configuration's factor.
void
rs_factor_row(const swtpg_handle* h, uint32_t g, uint32_t* row)
{
  const uint32_t link = g / h->groups_per_link, sub = g % h->groups_per_link;
  for (uint32_t lane = 0; lane < 32; ++lane) {
    uint32_t lo = h->link_rs_factor[link], hi = lo;
    if (h->h_rs_factor && h->rs_table_link[link]) {
      const uint16_t* f = h->h_rs_factor + size_t(link) * h->channels + sub * 64 + 2 * lane;
      lo = f[0];
      hi = f[1];
    }
    row[lane] = lo | (hi << 16);
  }
}

swtpg_status
reset_state(swtpg_handle* h)
{
  // Fresh zeroed ChanState (wibeth/tpg/ProcessingInfo.hpp:23-40) + per-channel RS memory factor (setState :131) + per-channel
  // hit threshold: the link's table, else its configuration's threshold, so that every link has a valid row
  std::vector<uint32_t> st(size_t(h->n_groups) * kStateWordsPerGroup, 0u);
  for (uint32_t g = 0; g < h->n_groups; ++g) {
    rs_factor_row(h, g, &st[size_t(g) * kStateWordsPerGroup + SV_RS_FACTOR * 32]);
    const uint32_t link = g / h->groups_per_link, sub = g % h->groups_per_link;
    const std::vector<uint16_t>& table = h->link_thresholds[link];
    for (uint32_t lane = 0; lane < 32; ++lane) {
      uint32_t lo = h->confs[h->link_conf[link]].threshold, hi = lo;
      if (!table.empty()) {
        lo = table[sub * 64 + 2 * lane];
        hi = table[sub * 64 + 2 * lane + 1];
      }
      st[size_t(g) * kStateWordsPerGroup + SV_THRESHOLD * 32 + lane] = lo | (hi << 16);
    }
  }
  SW_CUDA(h, cudaMemcpyAsync(h->d_state, st.data(), st.size() * 4, cudaMemcpyHostToDevice, h->stream));
  SW_CUDA(h, cudaMemsetAsync(h->d_flags, 0, size_t(h->n_groups) * 4, h->stream));
  SW_CUDA(h, cudaMemsetAsync(h->d_link_cursor, 0, (2 * SWTPG_MAX_LINK_CONFIGS + size_t(h->cfg.n_links)) * sizeof(uint32_t), h->stream));
  SW_CUDA(h, cudaStreamSynchronize(h->stream));
  return SWTPG_OK;
}

// swtpg_start: every window starts empty, after the statistics work of the previous run (reset_state then waits for the stream).
swtpg_status
reset_channel_stats(swtpg_handle* h)
{
  std::lock_guard<std::mutex> lk(h->stats_mu);
  if (h->stats_stream && h->stats_stream != h->stream)
    SW_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_stats, 0));
  const size_t n = size_t(h->cfg.n_links) * h->channels;
  if (h->d_adc_stats)
    SW_CUDA(h, cudaMemsetAsync(h->d_adc_stats, 0, n * sizeof(swtpg_adc_stats), h->stream));
  if (h->d_noise_lags)
    SW_CUDA(h, cudaMemsetAsync(h->d_noise_lags, 0, n * sizeof(swtpg_noise_lags), h->stream));
  if (h->d_channel_products)
    SW_CUDA(h, cudaMemsetAsync(h->d_channel_products, 0, size_t(h->cfg.n_links) * h->products_words * sizeof(uint64_t), h->stream));
  SW_CUDA(h, cudaEventRecord(h->ev_stats, h->stream));
  h->stats_stream = h->stream;
  return SWTPG_OK;
}

// Rewrites the SV_RS_FACTOR rows of links [link0, link0 + n) (rs_factor_row): ONE strided
// asynchronous copy on the compute stream, i.e. ordered before every kernel launched after this call and after every kernel
// launched before it. The source is pageable, so the runtime has staged it when the call returns.
swtpg_status
upload_rs_factor_rows(swtpg_handle* h, uint32_t link0, uint32_t n)
{
  const uint32_t g0 = link0 * h->groups_per_link, ng = n * h->groups_per_link;
  std::vector<uint32_t> rows(size_t(ng) * 32);
  for (uint32_t g = 0; g < ng; ++g)
    rs_factor_row(h, g0 + g, &rows[size_t(g) * 32]);
  SW_CUDA(h, cudaMemcpy2DAsync(h->d_state + size_t(g0) * kStateWordsPerGroup + SV_RS_FACTOR * 32, size_t(kStateWordsPerGroup) * 4, rows.data(), 128,
                               128, ng, cudaMemcpyHostToDevice, h->stream));
  return SWTPG_OK;
}

swtpg_status
check_batch_args(swtpg_handle* h, const void* frames, const uint32_t* n_units, uint32_t stride)
{
  if (!h)
    return SWTPG_ERR_INVALID_ARG;
  if (!h->started)
    return fail(h, SWTPG_ERR_STATE, "swtpg_start has not been called");
  if (!frames && stride)
    return fail(h, SWTPG_ERR_INVALID_ARG, "frames is NULL");
  if (stride > h->cfg.max_units)
    return fail(h, SWTPG_ERR_INVALID_ARG, "units_stride exceeds cfg.max_units");
  if (n_units)
    for (uint32_t l = 0; l < h->cfg.n_links; ++l)
      if (n_units[l] > stride)
        return fail(h, SWTPG_ERR_INVALID_ARG, "n_units[link] exceeds units_stride");
  return SWTPG_OK;
}

// Enqueue one batch on `s`: n_units upload, counter reset, kernel (timed with events on the same stream).
swtpg_status
enqueue_batch(swtpg_handle* h, const void* d_frames, const uint32_t* n_units, uint32_t stride, cudaStream_t s, bool dump)
{
  const uint32_t* d_nu = nullptr;
  uint64_t units = 0;
  if (n_units) {
    // pinned source, double-buffered: the copy that last read this buffer (two calls ago) must have finished
    const uint32_t turn = h->nunits_turn++ & 1u;
    SW_CUDA(h, cudaEventSynchronize(h->ev_nunits[turn]));
    memcpy(h->h_nunits[turn], n_units, size_t(h->cfg.n_links) * 4);
    SW_CUDA(h, cudaMemcpyAsync(h->d_nunits, h->h_nunits[turn], size_t(h->cfg.n_links) * 4, cudaMemcpyHostToDevice, s));
    SW_CUDA(h, cudaEventRecord(h->ev_nunits[turn], s));
    d_nu = h->d_nunits;
    for (uint32_t l = 0; l < h->cfg.n_links; ++l)
      units += n_units[l];
  } else {
    units = uint64_t(stride) * h->cfg.n_links;
  }
  SW_CUDA(h, cudaMemsetAsync(h->d_count, 0, sizeof(unsigned), s));
  if (stride) {
    int16_t* ped = dump ? h->d_ped : nullptr;
    int16_t* wav = dump ? h->d_wav : nullptr;
    SW_CUDA(h, cudaEventRecord(h->ev0, s));
    SW_CUDA(h, dump ? launch_groups<true>(h, d_frames, d_nu, stride, h->d_tps, h->d_count, ped, wav, s)
                    : launch_groups<false>(h, d_frames, d_nu, stride, h->d_tps, h->d_count, ped, wav, s));
    SW_CUDA(h, cudaEventRecord(h->ev1, s));
    h->timed = true;
    if (h->channel_stats())
      SW_CUDA(h, swtpg_internal::launch_channel_stats(h, d_frames, d_nu, stride, s));
  }
  h->last_stream = s;
  h->counters.units_processed += units;
  h->counters.samples_processed += units * h->channels * h->ticks;
  h->counters.batches++;
  return SWTPG_OK;
}

swtpg_status
fetch(swtpg_handle* h, cudaStream_t s, swtpg_tp* out, size_t cap, size_t* n_out)
{
  SW_CUDA(h, cudaMemcpyAsync(h->h_count, h->d_count, sizeof(unsigned), cudaMemcpyDeviceToHost, s));
  SW_CUDA(h, cudaStreamSynchronize(s));
  const size_t found = *h->h_count;
  const size_t stored = std::min<size_t>(found, h->tp_capacity);
  const size_t n = std::min(stored, cap);
  const swtpg_tp* src = h->d_tps;
  bool finish_on_host = false;
  std::unique_lock<std::mutex> sorter_lock; // the ordered list lives in the sorter's buffer until our copy has completed
  if (h->sorter && n && out) {
    const swtpg_status st = swtpg_internal::sort_tps_device(h, h->sorter, h->d_tps, stored, s, &src, &finish_on_host, &sorter_lock);
    if (st != SWTPG_OK)
      return st;
  }
  if (n && out)
    SW_CUDA(h, cudaMemcpyAsync(out, src, n * sizeof(swtpg_tp), cudaMemcpyDeviceToHost, s));
  SW_CUDA(h, cudaStreamSynchronize(s));
  if (sorter_lock.owns_lock())
    sorter_lock.unlock();
  if (finish_on_host && n == stored)
    swtpg_sort_tps(out, n); // equal keys / keys wider than 64 bits: the host's tie-break makes both orderings identical
  if (n_out)
    *n_out = found;
  h->counters.tps_emitted += found;
  h->counters.d2h_bytes += n * sizeof(swtpg_tp) + sizeof(unsigned);
  if (found > stored)
    h->counters.tps_dropped_overflow += found - stored;
  if (found > n)
    return fail(h, SWTPG_ERR_OVERFLOW, "more TPs than capacity");
  return SWTPG_OK;
}

// Checks one TPG configuration of a handle of `format`, normalises it and picks the policy that runs it (the packed fast paths'
// validity ranges). swtpg_create and swtpg_set_link_config both go through here. On failure *why says what is wrong.
swtpg_status
classify_config(int32_t format, const swtpg_link_config& in, TpgConf* out, const char** why)
{
  const bool wib2 = format == SWTPG_FORMAT_WIB2;
  if (in.algorithm < SWTPG_ALGO_SIMPLE_THRESHOLD || in.algorithm > SWTPG_ALGO_FIR_IQR)
    return *why = "unknown tpg_algorithm (reference: TPGAlgorithmInexistent)", SWTPG_ERR_UNSUPPORTED;
  if (wib2 && in.algorithm == SWTPG_ALGO_STANDARD_RS)
    return *why = "StandardRS does not exist for the WIB2 format (reference: SimpleThreshold and AbsRS only)", SWTPG_ERR_UNSUPPORTED;
  if (wib2 && in.algorithm == SWTPG_ALGO_ABS_RS && in.threshold == 0)
    return *why = "WIB2 AbsRS needs threshold >= 1 (sigmaMax = 2^15 / (multiplier * threshold))", SWTPG_ERR_INVALID_ARG;
  if (in.tap_exponent > 14)
    return *why = "tap_exponent out of range", SWTPG_ERR_INVALID_ARG;
  TpgConf c;
  c.algorithm = in.algorithm;
  c.threshold = in.threshold;
  c.frugal_acc_limit = in.frugal_acc_limit;
  c.rs_scale_factor = in.rs_scale_factor;
  c.tap_exponent = in.tap_exponent == 0 ? 6 : in.tap_exponent;
  bool any_tap = false;
  for (int i = 0; i < 8; ++i) {
    c.fir_taps[i] = in.fir_taps[i];
    any_tap |= in.fir_taps[i] != 0;
  }
  if (!any_tap) { // src/wib2/WIB2FrameProcessor.cpp:93-94
    swtpg_firwin_int(7, 0.1, 1 << c.tap_exponent, c.fir_taps);
    c.fir_taps[7] = 0;
  }
  // The policy: a packed fast path where the configuration is inside its validity range (see the policy), else the reference
  // arithmetic (ScalarAlgo).
  auto by_format = [wib2](Policy wibeth, Policy wib2_policy) { return wib2 ? wib2_policy : wibeth; };
  const bool acc_ok = c.frugal_acc_limit >= 1 && c.frugal_acc_limit <= 1000;
  const bool thr_ok = c.threshold <= 32767;
  // The packed IQR-threshold trackers (FIR + IQR, WIB2 AbsRS) need 1 <= tap_exponent <= 10. They build sigma * K with one
  // multiply-add (no carry between the halves while (sigmaMax + 3) * K < 2^16) and compare through the bf16 comparator, which
  // orders like signed int16 only up to 32640. Beyond that the reference's _mm256_cmpgt_epi16 sees the product as a NEGATIVE
  // int16 once a channel's IQR is large enough, so such configurations run the same packed trackers with the exact-threshold
  // tier (plain signed compares on the 64-bit-lane product) forced on for every group.
  const bool iqr_ok = c.tap_exponent >= 1 && c.tap_exponent <= 10;
  const uint32_t mult = 1u << c.tap_exponent;
  auto exact_tier = [](uint64_t sigma_max, uint64_t K) { return !((sigma_max + 3) * K < 65536 && sigma_max * K <= 32640); };
  switch (c.algorithm) {
    case SWTPG_ALGO_SIMPLE_THRESHOLD:
      c.policy = thr_ok && (wib2 || acc_ok) ? by_format(Policy::WibEthSimple, Policy::Wib2Simple)
                                            : by_format(Policy::WibEthScalarSimple, Policy::Wib2ScalarSimple);
      break;
    case SWTPG_ALGO_ABS_RS:
      if (wib2) { // K = threshold (>= 1, checked above), sigmaMax = 2^15 / (multiplier * threshold)
        c.policy = iqr_ok ? Policy::Wib2AbsRs : Policy::Wib2ScalarAbsRs;
        c.fir_force_exact = iqr_ok && exact_tier((1u << 15) / (uint64_t(mult) * c.threshold), c.threshold);
      } else {
        c.policy = thr_ok && acc_ok ? Policy::WibEthAbsRs : Policy::WibEthScalarAbsRs;
      }
      break;
    case SWTPG_ALGO_STANDARD_RS: c.policy = thr_ok && acc_ok ? Policy::WibEthStandardRs : Policy::WibEthScalarStandardRs; break;
    case SWTPG_ALGO_FIR_IQR: { // K = multiplier * threshold, sigmaMax = 2^15 / (multiplier * 5): threshold <= 5 at exponent 6
      static const int16_t kBinomial[8] = { 1, 6, 15, 20, 15, 6, 1, 0 };
      const bool binomial = memcmp(c.fir_taps, kBinomial, sizeof kBinomial) == 0; // the cascade, else the multiply-add chain
      c.policy = !iqr_ok  ? by_format(Policy::WibEthScalarFir, Policy::Wib2ScalarFir)
                 : binomial ? by_format(Policy::WibEthFir, Policy::Wib2Fir)
                            : by_format(Policy::WibEthFirAnyTaps, Policy::Wib2FirAnyTaps);
      c.fir_force_exact = iqr_ok && exact_tier((1u << 15) / (mult * 5u), uint64_t(mult) * c.threshold);
      break;
    }
  }
  *out = c;
  return SWTPG_OK;
}

// Whether a link running `algorithm` may have a per-channel threshold table: the algorithms whose threshold is in ADC counts. FIR +
// IQR and WIB2 AbsRS multiply it by an IQR sigma on 4 x int64 lanes that carry between neighbouring channels (iqr_threshold_exact),
// where a per-channel multiplier has no reference meaning.
bool
threshold_table_allowed(int32_t format, int32_t algorithm)
{
  return algorithm != SWTPG_ALGO_FIR_IQR && !(format == SWTPG_FORMAT_WIB2 && algorithm == SWTPG_ALGO_ABS_RS);
}

// Whether links of configurations a and b can run in one launch: they agree in every field their algorithm reads (the kernel
// parameters the policies of launch() consume). The policy follows from those fields. rs_memory_factor is per-link state
// (SV_RS_FACTOR rows), not a kernel parameter, so it never splits a group.
bool
same_group(int32_t format, const TpgConf& a, const TpgConf& b)
{
  if (a.algorithm != b.algorithm || a.threshold != b.threshold)
    return false;
  const bool wib2 = format == SWTPG_FORMAT_WIB2;
  const bool acc = !wib2 && a.algorithm != SWTPG_ALGO_FIR_IQR; // WIB2 and the FIR finder hard-wire 10 (wib2/tpg/ProcessAVX2.hpp:79)
  const bool scale = !wib2 && a.algorithm == SWTPG_ALGO_ABS_RS; // StandardRS adds s' unscaled (ProcessStandardRSAVX2.hpp:140-144)
  const bool exponent = wib2 || a.algorithm == SWTPG_ALGO_FIR_IQR; // the charge shift of WIB2, the multiplier of FIR + IQR
  const bool taps = a.algorithm == SWTPG_ALGO_FIR_IQR;
  if (acc && a.frugal_acc_limit != b.frugal_acc_limit)
    return false;
  if (scale && a.rs_scale_factor != b.rs_scale_factor)
    return false;
  if (exponent && a.tap_exponent != b.tap_exponent)
    return false;
  if (taps && memcmp(a.fir_taps, b.fir_taps, sizeof a.fir_taps) != 0)
    return false;
  return true;
}

// swtpg_read_adc_stats / swtpg_read_noise_lags / swtpg_read_channel_products: copies the window of links [link0, link0 + n_links)
// of a device accumulator d[n_links][per_link] to the pinned mirror hbuf and, on reset, zeroes it, in stream order. The caller
// holds read_mu and has checked the arguments; returns when hbuf holds the window.
template<typename T>
swtpg_status
read_window(swtpg_handle* h, T* d, T* hbuf, uint32_t link0, uint32_t n_links, size_t per_link, int reset)
{
  const size_t first = size_t(link0) * per_link, n = size_t(n_links) * per_link;
  {
    // Copy and reset are enqueued back to back on the stream of the last batch: a batch enqueued meanwhile falls after both.
    std::lock_guard<std::mutex> lk(h->stats_mu);
    const cudaStream_t s = h->stats_stream ? h->stats_stream : h->stream;
    SW_CUDA(h, cudaMemcpyAsync(hbuf + first, d + first, n * sizeof(T), cudaMemcpyDeviceToHost, s));
    if (reset) {
      SW_CUDA(h, cudaMemsetAsync(d + first, 0, n * sizeof(T), s));
      SW_CUDA(h, cudaEventRecord(h->ev_stats, s));
      h->stats_stream = s;
    }
    SW_CUDA(h, cudaEventRecord(h->ev_stats_read, s));
  }
  SW_CUDA(h, cudaEventSynchronize(h->ev_stats_read));
  return SWTPG_OK;
}

swtpg_status
check_read_args(swtpg_handle* h, uint32_t link0, uint32_t n_links, const void* out, const void* acc, const char* no_flag)
{
  if (!h)
    return fail(nullptr, SWTPG_ERR_INVALID_ARG, "handle is NULL");
  if (!out)
    return fail(h, SWTPG_ERR_INVALID_ARG, "out is NULL");
  if (!acc)
    return fail(h, SWTPG_ERR_STATE, no_flag);
  if (uint64_t(link0) + n_links > h->cfg.n_links)
    return fail(h, SWTPG_ERR_INVALID_ARG, "link0 + n_links exceeds cfg.n_links");
  return SWTPG_OK;
}

} // namespace

cudaError_t
swtpg_internal::launch_batch_kernel(swtpg_handle* h, const void* d_frames, const uint32_t* d_nunits, uint32_t units_stride, swtpg_tp* d_tps,
                                    unsigned* d_count, cudaStream_t s)
{
  return launch_groups<false>(h, d_frames, d_nunits, units_stride, d_tps, d_count, nullptr, nullptr, s);
}

extern "C" void swtpg_internal_ingest_counts(swtpg_handle* h, uint64_t* zero_copy, uint64_t* staged); // swtpg_stream.cu

extern "C" {

uint32_t
swtpg_abi_version(void)
{
  return SWTPG_ABI_VERSION;
}

const char*
swtpg_status_string(swtpg_status s)
{
  switch (s) {
    case SWTPG_OK: return "ok";
    case SWTPG_ERR_INVALID_ARG: return "invalid argument";
    case SWTPG_ERR_CUDA: return "CUDA error / no usable device";
    case SWTPG_ERR_BUSY: return "busy (back-pressure)";
    case SWTPG_ERR_OVERFLOW: return "TP buffer overflow";
    case SWTPG_ERR_STATE: return "invalid call sequence";
    case SWTPG_ERR_UNSUPPORTED: return "unsupported algorithm/format";
  }
  return "unknown";
}

const char*
swtpg_last_error(const swtpg_handle* h)
{
  if (!h)
    return g_create_error.c_str();
  swtpg_handle* hh = const_cast<swtpg_handle*>(h);
  std::lock_guard<std::mutex> lk(hh->err_mu);
  g_error_copy = hh->last_error; // per-thread copy: another thread may fail (and rewrite the text) at any time
  return g_error_copy.c_str();
}

int
swtpg_device_available(void)
{
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
    cudaGetLastError();
    return 0;
  }
  for (int d = 0; d < n; ++d) {
    int major = 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, d) == cudaSuccess && major == 10)
      return 1;
  }
  return 0;
}

swtpg_status
swtpg_create(const swtpg_config* cfg, swtpg_handle** out)
{
  if (!cfg || !out)
    return fail(nullptr, SWTPG_ERR_INVALID_ARG, "cfg/out is NULL");
  *out = nullptr;
  if (cfg->struct_size != sizeof(swtpg_config))
    return fail(nullptr, SWTPG_ERR_INVALID_ARG, "swtpg_config.struct_size mismatch");
  if (cfg->n_links == 0 || cfg->max_units == 0)
    return fail(nullptr, SWTPG_ERR_INVALID_ARG, "n_links and max_units must be > 0");
  if (cfg->max_units >= (1u << kHitUnitBits))
    return fail(nullptr, SWTPG_ERR_INVALID_ARG, "max_units must stay below 2^18 units per batch (hit records carry the unit index in 18 bits)");
  if (cfg->format != SWTPG_FORMAT_WIBETH && cfg->format != SWTPG_FORMAT_WIB2)
    return fail(nullptr, SWTPG_ERR_UNSUPPORTED, "unknown frame format");
  swtpg_link_config own{};
  own.struct_size = sizeof own;
  own.algorithm = cfg->algorithm;
  own.threshold = cfg->threshold;
  own.frugal_acc_limit = cfg->frugal_acc_limit;
  own.rs_memory_factor = cfg->rs_memory_factor;
  own.rs_scale_factor = cfg->rs_scale_factor;
  memcpy(own.fir_taps, cfg->fir_taps, sizeof own.fir_taps);
  own.tap_exponent = cfg->tap_exponent;
  TpgConf conf;
  const char* why = nullptr;
  const swtpg_status cs = classify_config(cfg->format, own, &conf, &why);
  if (cs != SWTPG_OK)
    return fail(nullptr, cs, why);
  if (cfg->wib2_adc_offset % 4 != 0 || cfg->wib2_adc_offset > SWTPG_WIB2_FRAME_BYTES - 448)
    return fail(nullptr, SWTPG_ERR_INVALID_ARG, "wib2_adc_offset must be a multiple of 4 and leave room for the 448-byte ADC block");
  if (cfg->flags & ~(SWTPG_FLAG_SORTED_TPS | SWTPG_FLAG_ADC_STATS | SWTPG_FLAG_NOISE_SPECTRA | SWTPG_FLAG_CHANNEL_COVARIANCE))
    return fail(nullptr, SWTPG_ERR_INVALID_ARG, "unknown bits in swtpg_config.flags");

  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
    cudaGetLastError();
    return fail(nullptr, SWTPG_ERR_CUDA, "no CUDA device visible (this library has no CPU fallback)");
  }
  if (cfg->device < 0 || cfg->device >= ndev)
    return fail(nullptr, SWTPG_ERR_INVALID_ARG, "device ordinal out of range");
  SW_CUDA((swtpg_handle*)nullptr, cudaSetDevice(cfg->device));
  int major = 0;
  SW_CUDA((swtpg_handle*)nullptr, cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, cfg->device));
  if (major != 10)
    return fail(nullptr, SWTPG_ERR_CUDA, "device is not compute capability 10.x (kernels are sm_100a only)");

  std::unique_ptr<swtpg_handle> h(new (std::nothrow) swtpg_handle);
  if (!h)
    return fail(nullptr, SWTPG_ERR_INVALID_ARG, "out of host memory");
  h->cfg = *cfg;
  const bool wib2 = cfg->format == SWTPG_FORMAT_WIB2;
  h->unit_bytes = wib2 ? SWTPG_WIB2_SUPERCHUNK_BYTES : SWTPG_WIBETH_FRAME_BYTES;
  h->channels = wib2 ? SWTPG_WIB2_CHANNELS : SWTPG_WIBETH_CHANNELS;
  h->ticks = wib2 ? SWTPG_WIB2_TICKS : SWTPG_WIBETH_TICKS;
  h->groups_per_link = h->channels / 64;
  h->n_groups = cfg->n_links * h->groups_per_link;
  if (h->cfg.n_slots == 0)
    h->cfg.n_slots = 4; // measured: 2 slots 38.0, 3 slots 45.4, 4 slots 47.1, 6 slots 47.2 GB/s (profiles/r02_streaming_slots_probe.txt)
  if (h->cfg.n_slots < 2)
    return fail(nullptr, SWTPG_ERR_INVALID_ARG, "n_slots must be >= 2");
  h->cfg.tap_exponent = conf.tap_exponent;
  memcpy(h->cfg.fir_taps, conf.fir_taps, sizeof conf.fir_taps);
  if (h->cfg.wib2_adc_offset == 0)
    h->cfg.wib2_adc_offset = 20;
  h->confs.assign(1, conf);
  h->conf_links.assign(1, cfg->n_links);
  h->link_conf.assign(cfg->n_links, 0);
  h->link_rs_factor.assign(cfg->n_links, cfg->rs_memory_factor);
  h->link_thresholds.assign(cfg->n_links, {});
  h->rs_table_link.assign(cfg->n_links, 0);
  // TP buffer: explicit, else samples/128 per batch clamped to [64 Ki, 16 Mi] records (physical TP rates are orders of
  // magnitude below one per 128 samples; the high-occupancy stress configuration sets tp_capacity itself).
  const uint64_t samples = uint64_t(cfg->n_links) * cfg->max_units * h->channels * h->ticks;
  uint64_t cap = cfg->tp_capacity ? cfg->tp_capacity : std::min<uint64_t>(std::max<uint64_t>(samples / 128, 1u << 16), 1u << 24);
  cap = std::min<uint64_t>(cap, std::max<uint64_t>(samples / 2, 1));
  h->tp_capacity = uint32_t(cap);
  swtpg_handle* hp = h.get();
  SW_CUDA(hp, cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  SW_CUDA(hp, cudaEventCreate(&h->ev0));
  SW_CUDA(hp, cudaEventCreate(&h->ev1));
  SW_CUDA(hp, cudaMalloc(&h->d_state, size_t(h->n_groups) * kStateWordsPerGroup * 4));
  SW_CUDA(hp, cudaMalloc(&h->d_flags, size_t(h->n_groups) * 4));
  SW_CUDA(hp, cudaMalloc(&h->d_link_cursor, (2 * SWTPG_MAX_LINK_CONFIGS + size_t(h->cfg.n_links)) * sizeof(uint32_t)));
  SW_CUDA(hp, cudaMemset(h->d_link_cursor, 0, (2 * SWTPG_MAX_LINK_CONFIGS + size_t(h->cfg.n_links)) * sizeof(uint32_t)));
  SW_CUDA(hp, cudaMalloc(&h->d_group_links, size_t(h->cfg.n_links) * sizeof(uint32_t)));
  SW_CUDA(hp, cudaMalloc(&h->d_tps, size_t(h->tp_capacity) * sizeof(swtpg_tp)));
  SW_CUDA(hp, cudaMalloc(&h->d_count, sizeof(unsigned)));
  SW_CUDA(hp, cudaMallocHost(&h->h_count, sizeof(unsigned)));
  SW_CUDA(hp, cudaMalloc(&h->d_nunits, size_t(cfg->n_links) * 4));
  for (int i = 0; i < 2; ++i) {
    SW_CUDA(hp, cudaMallocHost(&h->h_nunits[i], size_t(cfg->n_links) * 4));
    SW_CUDA(hp, cudaEventCreateWithFlags(&h->ev_nunits[i], cudaEventDisableTiming));
  }
  if (cfg->flags & SWTPG_FLAG_SORTED_TPS)
    h->sorter = swtpg_internal::sorter_create();
  if (cfg->flags & SWTPG_FLAG_ADC_STATS) {
    const size_t bytes = size_t(cfg->n_links) * h->channels * sizeof(swtpg_adc_stats);
    SW_CUDA(hp, cudaMalloc(&h->d_adc_stats, bytes));
    SW_CUDA(hp, cudaMemset(h->d_adc_stats, 0, bytes));
    SW_CUDA(hp, cudaMallocHost(&h->h_adc_stats, bytes));
  }
  if (cfg->flags & SWTPG_FLAG_NOISE_SPECTRA) {
    const size_t bytes = size_t(cfg->n_links) * h->channels * sizeof(swtpg_noise_lags);
    SW_CUDA(hp, cudaMalloc(&h->d_noise_lags, bytes));
    SW_CUDA(hp, cudaMemset(h->d_noise_lags, 0, bytes));
    SW_CUDA(hp, cudaMallocHost(&h->h_noise_lags, bytes));
  }
  h->products_words = SWTPG_CHANNEL_PRODUCTS_WORDS(h->channels);
  if (cfg->flags & SWTPG_FLAG_CHANNEL_COVARIANCE) {
    const size_t bytes = size_t(cfg->n_links) * h->products_words * sizeof(uint64_t);
    SW_CUDA(hp, cudaMalloc(&h->d_channel_products, bytes));
    SW_CUDA(hp, cudaMemset(h->d_channel_products, 0, bytes));
    SW_CUDA(hp, cudaMallocHost(&h->h_channel_products, bytes));
  }
  if (h->channel_stats()) {
    SW_CUDA(hp, cudaEventCreateWithFlags(&h->ev_stats, cudaEventDisableTiming));
    SW_CUDA(hp, cudaEventCreateWithFlags(&h->ev_stats_read, cudaEventDisableTiming));
  }
  *out = h.release();
  return SWTPG_OK;
}

void
swtpg_destroy(swtpg_handle* h)
{
  if (!h)
    return;
  cudaSetDevice(h->cfg.device);
  swtpg_internal::engine_destroy(h); // joins the streaming threads, unregisters latency buffers
  cudaDeviceSynchronize();
  for (auto& b : h->bounce) {
    for (int i = 0; i < 2; ++i) {
      if (b.buf[i]) cudaFreeHost(b.buf[i]);
      if (b.free_ev[i]) cudaEventDestroy(b.free_ev[i]);
    }
    if (b.done) cudaEventDestroy(b.done);
    if (b.stream) cudaStreamDestroy(b.stream);
  }
  if (h->d_state) cudaFree(h->d_state);
  if (h->d_flags) cudaFree(h->d_flags);
  if (h->d_link_cursor) cudaFree(h->d_link_cursor);
  if (h->d_group_links) cudaFree(h->d_group_links);
  if (h->d_tps) cudaFree(h->d_tps);
  if (h->d_count) cudaFree(h->d_count);
  if (h->h_count) cudaFreeHost(h->h_count);
  if (h->d_nunits) cudaFree(h->d_nunits);
  for (int i = 0; i < 2; ++i) {
    if (h->h_nunits[i]) cudaFreeHost(h->h_nunits[i]);
    if (h->ev_nunits[i]) cudaEventDestroy(h->ev_nunits[i]);
  }
  if (h->d_frames) cudaFree(h->d_frames);
  if (h->d_ped) cudaFree(h->d_ped);
  if (h->d_wav) cudaFree(h->d_wav);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->stream) cudaStreamDestroy(h->stream);
  if (h->sorter) swtpg_internal::sorter_destroy(h->sorter);
  if (h->d_adc_stats) cudaFree(h->d_adc_stats);
  if (h->h_adc_stats) cudaFreeHost(h->h_adc_stats);
  if (h->d_noise_lags) cudaFree(h->d_noise_lags);
  if (h->h_noise_lags) cudaFreeHost(h->h_noise_lags);
  if (h->d_channel_products) cudaFree(h->d_channel_products);
  if (h->h_channel_products) cudaFreeHost(h->h_channel_products);
  if (h->ev_stats) cudaEventDestroy(h->ev_stats);
  if (h->ev_stats_read) cudaEventDestroy(h->ev_stats_read);
  delete[] h->h_rs_factor;
  delete h;
}

swtpg_status
swtpg_start(swtpg_handle* h)
{
  if (!h)
    return SWTPG_ERR_INVALID_ARG;
  SW_CUDA(h, cudaSetDevice(h->cfg.device));
  swtpg_status s = SWTPG_OK;
  if (h->conf_groups_stale && (s = form_conf_groups(h)) != SWTPG_OK)
    return s;
  if (h->channel_stats() && (s = reset_channel_stats(h)) != SWTPG_OK)
    return s;
  s = reset_state(h);
  if (s != SWTPG_OK)
    return s;
  s = swtpg_internal::engine_reset(h); // streaming path: idle, rings empty, undelivered TPs of the previous run dropped
  if (s != SWTPG_OK)
    return s;
  h->counters.reset();
  h->timed = false;
  h->started = true;
  return SWTPG_OK;
}

swtpg_status
swtpg_stop(swtpg_handle* h)
{
  if (!h)
    return SWTPG_ERR_INVALID_ARG;
  swtpg_status s = swtpg_sync(h);
  h->started = false;
  return s;
}

swtpg_status
swtpg_set_rs_memory_factor(swtpg_handle* h, const uint16_t* by_link_channel)
{
  if (!h)
    return SWTPG_ERR_INVALID_ARG;
  delete[] h->h_rs_factor;
  h->h_rs_factor = nullptr;
  if (by_link_channel) {
    const size_t n = size_t(h->cfg.n_links) * h->channels;
    h->h_rs_factor = new uint16_t[n];
    memcpy(h->h_rs_factor, by_link_channel, n * sizeof(uint16_t));
  }
  std::fill(h->rs_table_link.begin(), h->rs_table_link.end(), by_link_channel ? 1 : 0);
  if (h->started) { // only the factor rows change; carried state is preserved
    SW_CUDA(h, cudaSetDevice(h->cfg.device));
    return upload_rs_factor_rows(h, 0, h->cfg.n_links);
  }
  return SWTPG_OK;
}

swtpg_status
swtpg_set_link_rs_memory_factor(swtpg_handle* h, uint32_t link, const uint16_t* by_channel)
{
  if (!h || !by_channel || link >= h->cfg.n_links)
    return SWTPG_ERR_INVALID_ARG;
  {
    std::lock_guard<std::mutex> lk(h->engine_mu); // several links' threads may arrive here with their first frames
    if (!h->h_rs_factor) // the other links keep their configuration's factor (rs_table_link)
      h->h_rs_factor = new uint16_t[size_t(h->cfg.n_links) * h->channels];
    memcpy(h->h_rs_factor + size_t(link) * h->channels, by_channel, size_t(h->channels) * sizeof(uint16_t));
    h->rs_table_link[link] = 1;
  }
  if (!h->started)
    return SWTPG_OK; // swtpg_start uploads the table
  SW_CUDA(h, cudaSetDevice(h->cfg.device));
  return upload_rs_factor_rows(h, link, 1);
}

swtpg_status
swtpg_set_link_config(swtpg_handle* h, uint32_t link, const swtpg_link_config* c)
{
  if (!h)
    return fail(nullptr, SWTPG_ERR_INVALID_ARG, "handle is NULL");
  if (h->started)
    return fail(h, SWTPG_ERR_STATE, "a link's configuration can only change while the handle is stopped");
  if (link >= h->cfg.n_links)
    return fail(h, SWTPG_ERR_INVALID_ARG, "link out of range");
  TpgConf conf = h->confs[0];
  uint16_t rs_factor = h->cfg.rs_memory_factor;
  if (c) {
    if (c->struct_size != sizeof(swtpg_link_config))
      return fail(h, SWTPG_ERR_INVALID_ARG, "swtpg_link_config.struct_size mismatch");
    const char* why = nullptr;
    const swtpg_status s = classify_config(h->cfg.format, *c, &conf, &why);
    if (s != SWTPG_OK)
      return fail(h, s, why);
    rs_factor = c->rs_memory_factor;
  }
  std::lock_guard<std::mutex> lk(h->engine_mu); // links' conf() calls may arrive from several threads
  if (!h->link_thresholds[link].empty() && !threshold_table_allowed(h->cfg.format, conf.algorithm))
    return fail(h, SWTPG_ERR_UNSUPPORTED, "the link has a per-channel threshold table, which its new algorithm cannot use (clear it first)");
  const uint32_t old = h->link_conf[link];
  --h->conf_links[old];
  auto in_use = [&](uint32_t i) { return i == 0 || h->conf_links[i] != 0; }; // the handle's own always counts
  uint32_t at = uint32_t(h->confs.size());
  for (uint32_t i = 0; i < h->confs.size() && at == h->confs.size(); ++i)
    if (in_use(i) && same_group(h->cfg.format, h->confs[i], conf))
      at = i;
  for (uint32_t i = 1; i < h->confs.size() && at == h->confs.size(); ++i)
    if (!in_use(i))
      at = i; // a free entry
  if (at == h->confs.size()) {
    if (at == SWTPG_MAX_LINK_CONFIGS) {
      ++h->conf_links[old];
      return fail(h, SWTPG_ERR_INVALID_ARG, "more than SWTPG_MAX_LINK_CONFIGS distinct link configurations");
    }
    h->confs.push_back(conf);
    h->conf_links.push_back(0);
  } else if (!in_use(at)) {
    h->confs[at] = conf;
  }
  ++h->conf_links[at];
  h->link_conf[link] = uint8_t(at);
  h->link_rs_factor[link] = rs_factor;
  h->conf_groups_stale = true;
  return SWTPG_OK;
}

swtpg_status
swtpg_set_link_thresholds(swtpg_handle* h, uint32_t link, const uint16_t* by_channel)
{
  if (!h)
    return fail(nullptr, SWTPG_ERR_INVALID_ARG, "handle is NULL");
  if (h->started)
    return fail(h, SWTPG_ERR_STATE, "a link's thresholds can only change while the handle is stopped");
  if (link >= h->cfg.n_links)
    return fail(h, SWTPG_ERR_INVALID_ARG, "link out of range");
  std::lock_guard<std::mutex> lk(h->engine_mu); // links' conf() calls may arrive from several threads
  if (!by_channel) {
    h->link_thresholds[link].clear();
    return SWTPG_OK;
  }
  for (uint32_t c = 0; c < h->channels; ++c)
    if (by_channel[c] > 32767u)
      return fail(h, SWTPG_ERR_INVALID_ARG, "a per-channel threshold is above 32767");
  if (!threshold_table_allowed(h->cfg.format, h->confs[h->link_conf[link]].algorithm))
    return fail(h, SWTPG_ERR_UNSUPPORTED, "per-channel thresholds exist for SimpleThreshold and the WIBEth running sums only");
  h->link_thresholds[link].assign(by_channel, by_channel + h->channels);
  return SWTPG_OK;
}

swtpg_status
swtpg_process_device(swtpg_handle* h, const void* d_frames, const uint32_t* n_units, uint32_t units_stride, void* stream)
{
  swtpg_status s = check_batch_args(h, d_frames, n_units, units_stride);
  if (s != SWTPG_OK)
    return s;
  if (reinterpret_cast<uintptr_t>(d_frames) & 15u)
    return fail(h, SWTPG_ERR_INVALID_ARG, "d_frames must be 16-byte aligned (bulk-copy source)");
  SW_CUDA(h, cudaSetDevice(h->cfg.device));
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : h->stream;
  return enqueue_batch(h, d_frames, n_units, units_stride, st, false);
}

swtpg_status
swtpg_fetch_tps(swtpg_handle* h, swtpg_tp* out, size_t cap, size_t* n_out)
{
  if (!h)
    return SWTPG_ERR_INVALID_ARG;
  if (!h->last_stream)
    return fail(h, SWTPG_ERR_STATE, "no batch has been processed");
  SW_CUDA(h, cudaSetDevice(h->cfg.device));
  return fetch(h, h->last_stream, out, cap, n_out);
}

double
swtpg_last_kernel_ms(swtpg_handle* h)
{
  if (!h || !h->timed)
    return -1.0;
  if (cudaEventSynchronize(h->ev1) != cudaSuccess)
    return -1.0;
  float ms = 0;
  if (cudaEventElapsedTime(&ms, h->ev0, h->ev1) != cudaSuccess)
    return -1.0;
  return double(ms);
}

// Copy of one payload into pinned memory (csrc/swtpg_hostutil.cpp: non-temporal stores where the CPU has AVX2).
extern "C" void swtpg_stage_copy(void* dst, const void* src, size_t bytes);

// Host-to-device copy of a PAGEABLE source. cudaMemcpyAsync would stage it through the driver's own bounce buffer on one
// thread (11 GB/s on the bench box against 55 GB/s from pinned memory); here a few worker threads copy 4 MB chunks into their
// own pinned double buffers with non-temporal stores and queue the DMA of each chunk on their own stream, so the host copies
// of later chunks overlap the transfers of earlier ones. The handle's stream then waits for every worker's last transfer.
constexpr size_t kBounceChunk = size_t(4) << 20;
constexpr size_t kBounceMinBytes = size_t(16) << 20;

static bool
is_pageable(const void* p)
{
  cudaPointerAttributes a{};
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return true;
  }
  return a.type == cudaMemoryTypeUnregistered;
}

static swtpg_status
staged_h2d(swtpg_handle* h, uint8_t* d_dst, const uint8_t* src, size_t bytes)
{
  if (h->bounce.empty()) {
    const unsigned hw = std::max(2u, std::thread::hardware_concurrency());
    const unsigned workers = std::min(8u, hw / 2);
    std::vector<swtpg_handle::Bounce> b(workers);
    for (auto& w : b) {
      for (int i = 0; i < 2; ++i) {
        SW_CUDA(h, cudaMallocHost(&w.buf[i], kBounceChunk));
        SW_CUDA(h, cudaEventCreateWithFlags(&w.free_ev[i], cudaEventDisableTiming));
      }
      SW_CUDA(h, cudaEventCreateWithFlags(&w.done, cudaEventDisableTiming));
      SW_CUDA(h, cudaStreamCreateWithFlags(&w.stream, cudaStreamNonBlocking));
    }
    h->bounce = std::move(b);
  }
  const size_t n_chunks = (bytes + kBounceChunk - 1) / kBounceChunk;
  const size_t workers = h->bounce.size();
  std::vector<cudaError_t> err(workers, cudaSuccess);
  std::vector<std::thread> threads;
  const int device = h->cfg.device;
  for (size_t t = 0; t < workers; ++t)
    threads.emplace_back([&, t]() {
      swtpg_handle::Bounce& w = h->bounce[t];
      cudaError_t e = cudaSetDevice(device);
      unsigned used = 0;
      for (size_t c = t; c < n_chunks && e == cudaSuccess; c += workers, ++used) {
        const int slot = int(used & 1u);
        if (used >= 2)
          e = cudaEventSynchronize(w.free_ev[slot]); // the transfer that last read this buffer has finished
        if (e != cudaSuccess)
          break;
        const size_t off = c * kBounceChunk, len = std::min(kBounceChunk, bytes - off);
        swtpg_stage_copy(w.buf[slot], src + off, len);
        e = cudaMemcpyAsync(d_dst + off, w.buf[slot], len, cudaMemcpyHostToDevice, w.stream);
        if (e == cudaSuccess)
          e = cudaEventRecord(w.free_ev[slot], w.stream);
      }
      if (e == cudaSuccess)
        e = cudaEventRecord(w.done, w.stream);
      err[t] = e;
    });
  for (auto& th : threads)
    th.join();
  for (size_t t = 0; t < workers; ++t) {
    SW_CUDA(h, err[t]);
    SW_CUDA(h, cudaStreamWaitEvent(h->stream, h->bounce[t].done, 0));
  }
  return SWTPG_OK;
}

static swtpg_status
process_host_impl(swtpg_handle* h, const void* frames, const uint32_t* n_units, uint32_t stride, swtpg_tp* out, size_t cap, size_t* n_out,
                  int16_t* ped_out, int16_t* wav_out, bool dump)
{
  swtpg_status s = check_batch_args(h, frames, n_units, stride);
  if (s != SWTPG_OK)
    return s;
  SW_CUDA(h, cudaSetDevice(h->cfg.device));
  const size_t bytes = size_t(h->cfg.n_links) * stride * h->unit_bytes;
  if (bytes > h->d_frames_bytes) {
    if (h->d_frames)
      cudaFree(h->d_frames);
    h->d_frames = nullptr;
    h->d_frames_bytes = 0;
    SW_CUDA(h, cudaMalloc(&h->d_frames, bytes));
    h->d_frames_bytes = bytes;
  }
  const size_t dump_elems = size_t(h->cfg.n_links) * stride * h->ticks * h->channels;
  if (dump && dump_elems > h->d_dump_elems) {
    if (h->d_ped) cudaFree(h->d_ped);
    if (h->d_wav) cudaFree(h->d_wav);
    h->d_ped = h->d_wav = nullptr;
    h->d_dump_elems = 0;
    SW_CUDA(h, cudaMalloc(&h->d_ped, dump_elems * 2));
    SW_CUDA(h, cudaMalloc(&h->d_wav, dump_elems * 2));
    h->d_dump_elems = dump_elems;
  }
  if (dump && dump_elems) {
    SW_CUDA(h, cudaMemsetAsync(h->d_ped, 0, dump_elems * 2, h->stream));
    SW_CUDA(h, cudaMemsetAsync(h->d_wav, 0, dump_elems * 2, h->stream));
  }
  if (bytes >= kBounceMinBytes && is_pageable(frames)) {
    s = staged_h2d(h, h->d_frames, static_cast<const uint8_t*>(frames), bytes);
    if (s != SWTPG_OK)
      return s;
  } else if (bytes) {
    SW_CUDA(h, cudaMemcpyAsync(h->d_frames, frames, bytes, cudaMemcpyHostToDevice, h->stream));
  }
  h->counters.h2d_bytes += bytes;
  s = enqueue_batch(h, h->d_frames, n_units, stride, h->stream, dump);
  if (s != SWTPG_OK)
    return s;
  s = fetch(h, h->stream, out, cap, n_out);
  if (dump && dump_elems) {
    if (ped_out)
      SW_CUDA(h, cudaMemcpy(ped_out, h->d_ped, dump_elems * 2, cudaMemcpyDeviceToHost));
    if (wav_out)
      SW_CUDA(h, cudaMemcpy(wav_out, h->d_wav, dump_elems * 2, cudaMemcpyDeviceToHost));
  }
  return s;
}

swtpg_status
swtpg_process_host(swtpg_handle* h, const void* frames, const uint32_t* n_units, uint32_t units_stride, swtpg_tp* out, size_t cap,
                   size_t* n_out)
{
  return process_host_impl(h, frames, n_units, units_stride, out, cap, n_out, nullptr, nullptr, false);
}

swtpg_status
swtpg_process_host_debug(swtpg_handle* h, const void* frames, const uint32_t* n_units, uint32_t units_stride, swtpg_tp* out, size_t cap,
                         size_t* n_out, int16_t* pedestal_out, int16_t* waveform_out)
{
  return process_host_impl(h, frames, n_units, units_stride, out, cap, n_out, pedestal_out, waveform_out, true);
}

swtpg_status
swtpg_sync(swtpg_handle* h)
{
  if (!h)
    return SWTPG_ERR_INVALID_ARG;
  SW_CUDA(h, cudaSetDevice(h->cfg.device));
  swtpg_status s = swtpg_internal::engine_quiesce(h); // streaming path: every dispatched batch has delivered its TPs to the ready queue
  if (s != SWTPG_OK)
    return s;
  SW_CUDA(h, cudaStreamSynchronize(h->stream));
  if (h->last_stream && h->last_stream != h->stream)
    SW_CUDA(h, cudaStreamSynchronize(h->last_stream));
  return SWTPG_OK;
}

swtpg_status
swtpg_dump_state(swtpg_handle* h, uint32_t link, swtpg_channel_state* out)
{
  if (!h || !out || link >= h->cfg.n_links)
    return SWTPG_ERR_INVALID_ARG;
  SW_CUDA(h, cudaSetDevice(h->cfg.device));
  swtpg_status s = swtpg_sync(h);
  if (s != SWTPG_OK)
    return s;
  std::vector<uint32_t> st(size_t(h->groups_per_link) * kStateWordsPerGroup);
  std::vector<uint32_t> fl(h->groups_per_link);
  SW_CUDA(h, cudaMemcpy(st.data(), h->d_state + size_t(link) * h->groups_per_link * kStateWordsPerGroup, st.size() * 4, cudaMemcpyDeviceToHost));
  SW_CUDA(h, cudaMemcpy(fl.data(), h->d_flags + size_t(link) * h->groups_per_link, fl.size() * 4, cudaMemcpyDeviceToHost));
  for (uint32_t c = 0; c < h->channels; ++c) {
    const uint32_t g = c / 64, lane = (c % 64) / 2, hi = c & 1;
    auto get = [&](int v) -> uint16_t {
      const uint32_t w = st[size_t(g) * kStateWordsPerGroup + size_t(v) * 32 + lane];
      return uint16_t(hi ? (w >> 16) : (w & 0xFFFFu));
    };
    swtpg_channel_state& o = out[c];
    memset(&o, 0, sizeof o);
    o.pedestal = int16_t(get(SV_MEDIAN));
    o.accum = int16_t(get(SV_ACCUM));
    o.quantile25 = int16_t(get(SV_Q25));
    o.quantile75 = int16_t(get(SV_Q75));
    o.accum25 = int16_t(get(SV_A25));
    o.accum75 = int16_t(get(SV_A75));
    o.rs = int16_t(get(SV_RS));
    o.pedestal_rs = int16_t(get(SV_MED_RS));
    o.accum_rs = int16_t(get(SV_ACC_RS));
    o.rs_memory_factor = get(SV_RS_FACTOR);
    o.prev_was_over = get(SV_PREV);
    o.hit_charge = get(SV_CHARGE);
    o.hit_tover = get(SV_TOVER);
    o.hit_peak_adc = get(SV_PEAK_ADC);
    o.hit_peak_time = get(SV_PEAK_TIME);
    o.initialized = uint16_t(fl[g] & kFlagInitialized);
    for (int j = 0; j < 8; ++j)
      o.prev_samp[j] = int16_t(get(SV_RING0 + j));
  }
  return SWTPG_OK;
}

swtpg_status
swtpg_read_adc_stats(swtpg_handle* h, uint32_t link0, uint32_t n_links, swtpg_adc_stats* out, int reset)
{
  swtpg_status st = check_read_args(h, link0, n_links, out, h ? h->d_adc_stats : nullptr, "the handle was created without SWTPG_FLAG_ADC_STATS");
  if (st != SWTPG_OK || n_links == 0)
    return st;
  SW_CUDA(h, cudaSetDevice(h->cfg.device));
  std::lock_guard<std::mutex> rd(h->read_mu);
  if ((st = read_window(h, h->d_adc_stats, h->h_adc_stats, link0, n_links, h->channels, reset)) != SWTPG_OK)
    return st;
  const size_t first = size_t(link0) * h->channels, n = size_t(n_links) * h->channels;
  for (size_t i = 0; i < n; ++i) {
    const swtpg_adc_stats& a = h->h_adc_stats[first + i];
    uint32_t ext[2];
    memcpy(ext, &a.min, sizeof ext); // {16383 - min, max} (swtpg_handle::d_adc_stats)
    swtpg_adc_stats& o = out[i];
    o.samples = a.samples;
    o.sum = a.sum;
    o.sum_sq = a.sum_sq;
    o.min = a.samples ? uint16_t(0x3FFFu - ext[0]) : 0;
    o.max = a.samples ? uint16_t(ext[1]) : 0;
    o.reserved = 0;
  }
  return SWTPG_OK;
}

swtpg_status
swtpg_read_noise_lags(swtpg_handle* h, uint32_t link0, uint32_t n_links, swtpg_noise_lags* out, int reset)
{
  swtpg_status st = check_read_args(h, link0, n_links, out, h ? h->d_noise_lags : nullptr, "the handle was created without SWTPG_FLAG_NOISE_SPECTRA");
  if (st != SWTPG_OK || n_links == 0)
    return st;
  SW_CUDA(h, cudaSetDevice(h->cfg.device));
  std::lock_guard<std::mutex> rd(h->read_mu);
  if ((st = read_window(h, h->d_noise_lags, h->h_noise_lags, link0, n_links, h->channels, reset)) != SWTPG_OK)
    return st;
  memcpy(out, h->h_noise_lags + size_t(link0) * h->channels, size_t(n_links) * h->channels * sizeof(swtpg_noise_lags));
  return SWTPG_OK;
}

swtpg_status
swtpg_read_channel_products(swtpg_handle* h, uint32_t link0, uint32_t n_links, uint64_t* out, int reset)
{
  swtpg_status st = check_read_args(h, link0, n_links, out, h ? h->d_channel_products : nullptr,
                                    "the handle was created without SWTPG_FLAG_CHANNEL_COVARIANCE");
  if (st != SWTPG_OK || n_links == 0)
    return st;
  SW_CUDA(h, cudaSetDevice(h->cfg.device));
  std::lock_guard<std::mutex> rd(h->read_mu);
  if ((st = read_window(h, h->d_channel_products, h->h_channel_products, link0, n_links, h->products_words, reset)) != SWTPG_OK)
    return st;
  memcpy(out, h->h_channel_products + size_t(link0) * h->products_words, size_t(n_links) * h->products_words * sizeof(uint64_t));
  return SWTPG_OK;
}

swtpg_status
swtpg_get_counters(swtpg_handle* h, swtpg_counters* out)
{
  if (!h || !out)
    return SWTPG_ERR_INVALID_ARG;
  out->units_processed = h->counters.units_processed.load();
  out->samples_processed = h->counters.samples_processed.load();
  out->tps_emitted = h->counters.tps_emitted.load();
  out->tps_dropped_overflow = h->counters.tps_dropped_overflow.load();
  out->batches = h->counters.batches.load();
  out->submit_busy = h->counters.submit_busy.load();
  out->h2d_bytes = h->counters.h2d_bytes.load();
  out->d2h_bytes = h->counters.d2h_bytes.load();
  swtpg_internal_ingest_counts(h, &out->units_zero_copy, &out->units_staged);
  return SWTPG_OK;
}

swtpg_status
swtpg_sort_stats(swtpg_handle* h, double* last_ms, double* total_ms, uint64_t* lists, uint64_t* finished_on_host)
{
  if (!h)
    return SWTPG_ERR_INVALID_ARG;
  swtpg_internal::sorter_stats(h->sorter, last_ms, total_ms, lists, finished_on_host);
  return SWTPG_OK;
}

void*
swtpg_alloc_pinned(size_t bytes, int write_combined)
{
  void* p = nullptr;
  const unsigned flags = cudaHostAllocPortable | (write_combined ? cudaHostAllocWriteCombined : 0u);
  if (bytes == 0 || cudaHostAlloc(&p, bytes, flags) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}

void
swtpg_free_pinned(void* p)
{
  if (p && cudaFreeHost(p) != cudaSuccess)
    cudaGetLastError();
}

} // extern "C"
