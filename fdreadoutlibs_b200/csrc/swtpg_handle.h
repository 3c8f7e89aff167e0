// Internal layout of swtpg_handle, shared by the translation units behind include/swtpg.h:
//   swtpg_capi.cu    create / destroy / start / stop, the batch entry points and the kernel launch table
//   swtpg_stream.cu  the streaming path (swtpg_submit ... swtpg_poll): per-link rings, dispatcher and completion threads,
//                    the gather kernel that pulls frames out of pinned host memory
//   swtpg_stats.cu   the per-channel statistics kernel (SWTPG_FLAG_ADC_STATS, SWTPG_FLAG_NOISE_SPECTRA) and the channel
//                    products kernel (SWTPG_FLAG_CHANNEL_COVARIANCE)
// Not installed; nothing outside csrc/ includes it.
#pragma once

#include "../../include/swtpg.h"

#include <cuda_runtime.h>

#include <atomic>
#include <cstdio>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

namespace swtpg_internal {
struct StreamEngine;
struct TpSorter;

// One TPG configuration (swtpg_create's or a link's, swtpg_set_link_config), normalised — default taps and tap exponent
// filled in — and classified: which policy of the launch table runs it. classify_config (swtpg_capi.cu) is the only place
// that makes one.
// The kernel policy a configuration runs (launch, swtpg_capi.cu): a packed fast path (swtpg_kernels.cuh) where the configuration
// is inside its validity range, else ScalarAlgo, the reference arithmetic.
enum class Policy : uint8_t
{
  WibEthSimple,     // PackedSimpleWibEthPipe
  WibEthAbsRs,      // PackedRsWibEth<false>
  WibEthStandardRs, // PackedRsWibEth<true>
  WibEthFir,        // PackedFirIqr: binomial taps
  WibEthFirAnyTaps, // PackedFirIqrAnyTaps
  WibEthScalarSimple,
  WibEthScalarAbsRs,
  WibEthScalarStandardRs,
  WibEthScalarFir,
  Wib2Simple,     // PackedSimpleWib2
  Wib2AbsRs,      // PackedRsIqrWib2
  Wib2Fir,        // PackedFirIqr
  Wib2FirAnyTaps, // PackedFirIqrAnyTaps
  Wib2ScalarSimple,
  Wib2ScalarAbsRs,
  Wib2ScalarFir,
};

struct TpgConf
{
  int32_t algorithm = 0;
  uint16_t threshold = 0;
  int16_t frugal_acc_limit = 0;
  uint16_t rs_scale_factor = 0;
  int16_t fir_taps[SWTPG_MAX_TAPS] = {};
  uint8_t tap_exponent = 0;
  Policy policy = Policy::WibEthScalarSimple;
  bool fir_force_exact = false; // packed FIR / WIB2-AbsRS trackers with the exact-threshold tier on every group (classify_config)
};

// Links of one handle whose configurations run as one launch of the batch kernel (formed at swtpg_start).
struct ConfGroup
{
  uint32_t conf = 0;                  // index into swtpg_handle::confs
  uint32_t n_links = 0;
  const uint32_t* d_links = nullptr;  // the group's links in ascending order; nullptr = every link of the handle
  uint32_t* d_cursor = nullptr;       // its own {claimed, finished} pair of the kernels' dynamic link hand-out
};
}

struct swtpg_handle
{
  swtpg_config cfg{};
  uint32_t unit_bytes = 0, channels = 0, ticks = 0, groups_per_link = 0, n_groups = 0;
  uint32_t tp_capacity = 0;
  std::atomic<bool> started{ false };

  // TPG configurations: confs[0] is the handle's own (swtpg_create), the others come from swtpg_set_link_config; link l runs
  // confs[link_conf[l]]. No two entries in use run the same (same_group), and there are at most SWTPG_MAX_LINK_CONFIGS.
  std::vector<swtpg_internal::TpgConf> confs;
  std::vector<uint32_t> conf_links;    // links using each entry of confs; an entry other than 0 with none is free
  std::vector<uint8_t> link_conf;      // [n_links]
  std::vector<uint16_t> link_rs_factor; // [n_links] rs_memory_factor of each link's configuration
  // [n_links] per-channel hit thresholds of swtpg_set_link_thresholds, by frame channel; empty = the configuration's threshold.
  // Only links whose algorithm compares ADC counts have one (threshold_table_allowed); swtpg_start writes the SV_THRESHOLD rows.
  std::vector<std::vector<uint16_t>> link_thresholds;
  // Configuration groups: one per entry of confs in use, formed by swtpg_start when a link's configuration has changed, and
  // frozen while the handle is started (the streaming engine's threads read them without a lock, so swtpg_set_link_config
  // refuses to run then).
  std::vector<swtpg_internal::ConfGroup> conf_groups;
  bool conf_groups_stale = true;
  uint32_t* d_group_links = nullptr;   // [n_links]: the groups' link lists, back to back

  cudaStream_t stream = nullptr; // batch path + all kernels (state is carried batch to batch: kernels are ordered)
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  bool timed = false;
  cudaStream_t last_stream = nullptr;

  uint32_t* d_state = nullptr;
  uint32_t* d_flags = nullptr;
  uint32_t* d_link_cursor = nullptr; // SWTPG_MAX_LINK_CONFIGS x {claimed, finished}: dynamic link hand-out of the kernels, one
                                     // pair per configuration group, self-resetting; followed by [n_links] slices done per link
                                     // (wibeth_kernel's sliced hand-out, self-resetting too)
  swtpg_tp* d_tps = nullptr;
  unsigned* d_count = nullptr;
  unsigned* h_count = nullptr;
  uint32_t* d_nunits = nullptr;
  // ragged lengths of the batch entry points: two pinned buffers used alternately, each guarded by the event of the copy that
  // last read it (back-to-back swtpg_process_device calls must not overwrite lengths an earlier async copy still reads)
  uint32_t* h_nunits[2] = { nullptr, nullptr };
  cudaEvent_t ev_nunits[2] = { nullptr, nullptr };
  uint32_t nunits_turn = 0;
  uint8_t* d_frames = nullptr;
  size_t d_frames_bytes = 0;
  int16_t* d_ped = nullptr;
  int16_t* d_wav = nullptr;
  size_t d_dump_elems = 0;
  uint16_t* h_rs_factor = nullptr; // [n_links][channels] or null
  std::vector<uint8_t> rs_table_link; // [n_links] 1 = the link's rows of h_rs_factor were set (else its configuration's factor)
  swtpg_internal::TpSorter* sorter = nullptr; // SWTPG_FLAG_SORTED_TPS: device-side ordering of TP lists (swtpg_sort.cu)

  // SWTPG_FLAG_ADC_STATS (null without it). d_adc_stats[n_links][channels] holds the current window of every channel in the
  // layout of swtpg_adc_stats, except its last 8 bytes: {16383 - min, max} as two 32-bit words, so that zeroed memory is an empty
  // window and both merge by atomicMax.
  swtpg_adc_stats* d_adc_stats = nullptr;
  swtpg_adc_stats* h_adc_stats = nullptr; // pinned, same size
  // SWTPG_FLAG_NOISE_SPECTRA (null without it): d_noise_lags[n_links][channels], the current window in the layout of swtpg_noise_lags.
  swtpg_noise_lags* d_noise_lags = nullptr;
  swtpg_noise_lags* h_noise_lags = nullptr; // pinned, same size
  // SWTPG_FLAG_CHANNEL_COVARIANCE (null without it): d_channel_products[n_links][SWTPG_CHANNEL_PRODUCTS_WORDS(channels)], the
  // current window in the layout of swtpg_read_channel_products.
  uint64_t* d_channel_products = nullptr;
  uint64_t* h_channel_products = nullptr; // pinned, same size
  uint32_t products_words = 0;            // SWTPG_CHANNEL_PRODUCTS_WORDS(channels)
  // Any of the three flags (all null without them). Every statistics kernel and every read runs in one order: each waits for
  // ev_stats, which is recorded after the last of them on stats_stream, when it runs on another stream. stats_mu guards those two
  // and keeps a read's copy and reset together; read_mu serialises reads (the pinned mirrors, ev_stats_read).
  cudaEvent_t ev_stats = nullptr, ev_stats_read = nullptr;
  cudaStream_t stats_stream = nullptr;
  std::mutex stats_mu, read_mu;
  bool channel_stats() const { return d_adc_stats || d_noise_lags || d_channel_products; } // every batch gets a launch_channel_stats

  // streaming path (swtpg_stream.cu), created on the first swtpg_submit / swtpg_register_buffer
  std::mutex engine_mu;
  std::atomic<swtpg_internal::StreamEngine*> engine{ nullptr };

  // bounce pipeline of swtpg_process_host for pageable sources: per worker two pinned buffers, a stream and events
  struct Bounce
  {
    uint8_t* buf[2] = { nullptr, nullptr };
    cudaEvent_t free_ev[2] = { nullptr, nullptr };
    cudaEvent_t done = nullptr;
    cudaStream_t stream = nullptr;
  };
  std::vector<Bounce> bounce;

  // counters behind swtpg_get_counters: written by the caller's threads and by the engine's threads
  struct Counters
  {
    std::atomic<uint64_t> units_processed{ 0 }, samples_processed{ 0 }, tps_emitted{ 0 }, tps_dropped_overflow{ 0 }, batches{ 0 },
      submit_busy{ 0 }, h2d_bytes{ 0 }, d2h_bytes{ 0 };
    void reset()
    {
      units_processed = samples_processed = tps_emitted = tps_dropped_overflow = batches = submit_busy = h2d_bytes = d2h_bytes = 0;
    }
  } counters;

  // last failure text: any thread may set it, swtpg_last_error hands out a per-thread copy
  std::mutex err_mu;
  std::string last_error;
  void set_error(const char* msg)
  {
    std::lock_guard<std::mutex> lk(err_mu);
    last_error = msg;
  }
};

namespace swtpg_internal {

void set_create_error(const char* msg);

inline swtpg_status
fail(swtpg_handle* h, swtpg_status s, const char* msg)
{
  if (h)
    h->set_error(msg);
  else
    set_create_error(msg);
  return s;
}

#define SW_CUDA(h, call)                                                                                                          \
  do {                                                                                                                            \
    cudaError_t e_ = (call);                                                                                                      \
    if (e_ != cudaSuccess) {                                                                                                      \
      char buf_[512];                                                                                                             \
      snprintf(buf_, sizeof buf_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__);                    \
      swtpg_internal::fail((h), SWTPG_ERR_CUDA, buf_);                                                                            \
      return SWTPG_ERR_CUDA;                                                                                                      \
    }                                                                                                                             \
  } while (0)

// swtpg_capi.cu: launches the handle's fused kernel over one batch laid out link-major in device memory
// ([n_links][units_stride][unit_bytes], d_nunits = per-link valid units or nullptr) on stream `s`. TPs go to d_tps / d_count.
cudaError_t launch_batch_kernel(swtpg_handle* h, const void* d_frames, const uint32_t* d_nunits, uint32_t units_stride, swtpg_tp* d_tps,
                                unsigned* d_count, cudaStream_t s);

// swtpg_stats.cu: adds one batch, laid out as for launch_batch_kernel, to the per-channel ADC statistics (SWTPG_FLAG_ADC_STATS)
// and noise lags (SWTPG_FLAG_NOISE_SPECTRA) the handle keeps, in one read of the batch on stream `s`, then to its channel products
// (SWTPG_FLAG_CHANNEL_COVARIANCE) in a second kernel, after the statistics work of earlier batches and reads whatever stream that
// ran on.
cudaError_t launch_channel_stats(swtpg_handle* h, const void* d_frames, const uint32_t* d_nunits, uint32_t units_stride, cudaStream_t s);

// swtpg_sort.cu: device-side ordering of a batch's TP list (SWTPG_FLAG_SORTED_TPS)
TpSorter* sorter_create();
void sorter_destroy(TpSorter* s);
void sorter_stats(const TpSorter* s, double* last_ms, double* total_ms, uint64_t* calls, uint64_t* host_fallbacks);
swtpg_status sort_tps_device(swtpg_handle* h, TpSorter* st, const swtpg_tp* d_tps, size_t n, cudaStream_t s, const swtpg_tp** out,
                             bool* finish_on_host, std::unique_lock<std::mutex>* lock);

// swtpg_stream.cu
void engine_destroy(swtpg_handle* h);          // stops the threads, frees everything (swtpg_destroy)
swtpg_status engine_reset(swtpg_handle* h);    // swtpg_start: idle engine, empty rings
swtpg_status engine_quiesce(swtpg_handle* h);  // swtpg_sync: every dispatched batch has completed

} // namespace swtpg_internal
