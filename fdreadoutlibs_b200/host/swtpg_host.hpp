// Host-side C++ face of the B200 SWTPG: the frame-processor plug-ins of DUNE-DAQ/fdreadoutlibs with their own method
// names and behaviour, with the body of find_hits replaced by calls into the C ABI (include/swtpg.h).
//
// Citations `path:line` are into the reference repository. Everything that the reference gets from packages that are
// not part of it (readoutlibs, iomanager, opmonlib, ers, detchannelmaps, trgdataformats, fddetdataformats) is restated
// here as the smallest stand-in that lets the plug-in logic be compiled, driven and tested on its own:
//   readoutlibs::TaskRawDataProcessorModel<T>   -> TaskRawDataProcessorModel<T> (pre tasks inline, post tasks inline)
//   iomanager sender "tp_out"                   -> TpSink (std::function try_send)
//   readoutinfo::RawDataProcessorInfo           -> RawDataProcessorInfo (POD)
//   detchannelmaps::TPCChannelMap               -> ChannelMap (std::function)
//   trgdataformats::TriggerPrimitive            -> TriggerPrimitive (field-for-field; byte layout unpinned)
//   ers issues (FDReadoutIssues.hpp:27-46)      -> exceptions for conf-time issues, counters for data-path issues
#pragma once

#include "../../include/swtpg.h"

#include <array>
#include <atomic>
#include <chrono>
#include <cstdint>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <set>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

namespace swtpg {
namespace host {

// ---- records and payloads on the boundary ---------------------------------------------------------------------------
// trgdataformats::TriggerPrimitive as the reference fills it (src/wibeth/WIBEthFrameProcessor.cpp:540-549).
struct TriggerPrimitive
{
  enum class Type : uint32_t { kUnknown = 0, kTPC = 1, kPDS = 2 };
  enum class Algorithm : uint32_t { kUnknown = 0, kTPCDefault = 1, kSimpleThreshold = 2, kAbsRunningSum = 3, kRunningSum = 4 };
  uint16_t version = 1;
  uint64_t time_start = 0, time_peak = 0, time_over_threshold = 0;
  uint32_t channel = 0, adc_integral = 0;
  uint16_t adc_peak = 0, detid = 0;
  Type type = Type::kUnknown;
  Algorithm algorithm = Algorithm::kUnknown;
  uint16_t flag = 0;
};
// SURVEY.md 8(b): trgdataformats is not part of the snapshot; its TriggerPrimitive is a 56-byte record — the 16-bit version
// first (padded to 8), three 64-bit times, channel and adc_integral (32 bit), adc_peak and detid (16 bit), the two 32-bit enums
// and the 16-bit flag word (restated from memory of trgdataformats/TriggerPrimitive.hpp). Same members, same order, so the
// restatement must come out at the same size; the byte layout itself stays unpinned (parity is asserted on field tuples).
static_assert(sizeof(TriggerPrimitive) == 56, "TriggerPrimitive restatement drifted from the 56-byte record of trgdataformats");
// include/fdreadoutlibs/TriggerPrimitiveTypeAdapter.hpp:19-71: ordering by (time_start, channel)
struct TriggerPrimitiveTypeAdapter
{
  TriggerPrimitive tp;
  bool operator<(const TriggerPrimitiveTypeAdapter& o) const
  {
    return tp.time_start != o.tp.time_start ? tp.time_start < o.tp.time_start : tp.channel < o.tp.channel;
  }
  uint64_t get_first_timestamp() const { return tp.time_start; }
};

// DAQEthHeader of fddetdataformats (bit positions restated from memory; unpinned — same statement as oracle/shim).
struct DAQEthHeader
{
  uint64_t version : 6, det_id : 6, crate_id : 10, slot_id : 4, stream_id : 8, reserved : 6, seq_id : 12, block_length : 12;
  uint64_t timestamp;
};
// include/fdreadoutlibs/DUNEWIBEthTypeAdapter.hpp:22-96
struct DUNEWIBEthTypeAdapter
{
  char data[SWTPG_WIBETH_FRAME_BYTES];
  DAQEthHeader* header() { return reinterpret_cast<DAQEthHeader*>(data); }
  const DAQEthHeader* header() const { return reinterpret_cast<const DAQEthHeader*>(data); }
  uint64_t get_first_timestamp() const { return header()->timestamp; }
  void set_first_timestamp(uint64_t ts) { header()->timestamp = ts; }
  size_t get_num_frames() const { return 1; }
  size_t get_payload_size() const { return sizeof data; }
  static constexpr uint64_t expected_tick_difference = 2048, samples_per_frame = 64, samples_tick_difference = 32;
};
static_assert(sizeof(DUNEWIBEthTypeAdapter) == 7200, "DUNEWIBEthTypeAdapter.hpp:98");
// WIB2Frame header of fddetdataformats (restated; word 0 bit fields + 64-bit timestamp in words 1-2).
struct WIB2Header
{
  uint32_t version : 6, detector_id : 6, crate : 10, slot : 4, link : 6;
  uint32_t timestamp_1, timestamp_2;
};
// include/fdreadoutlibs/DUNEWIBSuperChunkTypeAdapter.hpp:22-98
struct DUNEWIBSuperChunkTypeAdapter
{
  char data[SWTPG_WIB2_SUPERCHUNK_BYTES];
  WIB2Header* header(size_t frame = 0) { return reinterpret_cast<WIB2Header*>(data + frame * SWTPG_WIB2_FRAME_BYTES); }
  const WIB2Header* header(size_t frame = 0) const { return reinterpret_cast<const WIB2Header*>(data + frame * SWTPG_WIB2_FRAME_BYTES); }
  uint64_t get_first_timestamp() const { return uint64_t(header()->timestamp_1) | (uint64_t(header()->timestamp_2) << 32); }
  void set_timestamp(size_t frame, uint64_t ts)
  {
    header(frame)->timestamp_1 = uint32_t(ts);
    header(frame)->timestamp_2 = uint32_t(ts >> 32);
  }
  size_t get_num_frames() const { return 12; }
  static constexpr uint64_t expected_tick_difference = 32, samples_tick_difference = 32;
};
static_assert(sizeof(DUNEWIBSuperChunkTypeAdapter) == 5664, "DUNEWIBSuperChunkTypeAdapter.hpp:100");

// ---- configuration / monitoring PODs ----------------------------------------------------------------------------------
// The fields of readoutlibs' RawDataProcessorConf that the TPC processors read (src/wibeth/WIBEthFrameProcessor.cpp:175-230).
struct RawDataProcessorConf
{
  uint32_t source_id = 0;
  std::string tpg_algorithm = "SimpleThreshold";
  bool enable_simple_threshold_on_collection = false;
  float tpg_rs_memory_factor = 0.8f; // x10 inside conf()
  float tpg_rs_scale_factor = 2.0f;  // 10/x inside conf()
  int16_t tpg_frugal_streaming_accumulator_limit = 10;
  uint64_t tp_timeout = 100000;
  std::vector<uint32_t> tpg_channel_mask;
  uint16_t tpg_threshold = 100;
  uint16_t crate_id = 0, slot_id = 0, link_id = 0;
  bool enable_tpg = true;
  std::string channel_map_name = "linear";
  bool emulator_mode = false;
  bool correct_channel_lookup = false; // false: index the position-ordered LUT with the frame channel, as production does (H2)
  // Not a reference field: hit threshold per plane, indexed by get_plane_from_offline_channel (0 = collection); -1 = tpg_threshold.
  // conf() resolves it into a per-frame-channel table through the channel map and the configured crate / slot / link ids
  // (swtpg_set_link_thresholds). SimpleThreshold and the WIBEth running sums only.
  std::array<int32_t, 3> tpg_plane_threshold{ -1, -1, -1 };
  // Back-pressure from the GPU pipeline: false = drop the frame and count it (what a full queue does to the reference's
  // try_send); true = wait for a staging slot (file replay / emulators, where losing data is worse than stalling).
  bool block_on_backpressure = false;
};
// readoutinfo::RawDataProcessorInfo + TPChannelInfo as get_info fills them (src/wibeth/WIBEthFrameProcessor.cpp:237-292)
struct RawDataProcessorInfo
{
  uint64_t num_seq_id_errors = 0;
  int32_t min_seq_id_jump = 0, max_seq_id_jump = 0;
  uint64_t num_ts_errors = 0;
  double rate_tp_hits = 0; // kHz
  uint64_t num_tps_sent = 0, num_tps_suppressed_too_long = 0, num_tps_send_failed = 0, num_frames_dropped_busy = 0;
  uint32_t top_channels[10] = {};
  uint32_t top_channel_tps[10] = {};
  uint32_t n_top = 0;
};
// FDReadoutIssues.hpp:27-31 / :41-46
struct TPGAlgorithmInexistent : std::runtime_error
{
  explicit TPGAlgorithmInexistent(const std::string& a) : std::runtime_error("The selected algorithm does not exist: " + a + " . Check your configuration file and seelect either SWTPG or AbsRS.") {}
};
struct LinkMisconfiguration
{
  uint32_t crate, slot, stream, exp_crate, exp_slot, exp_stream;
};
// readoutlibs::FrameErrorRegistry: named error intervals
struct FrameErrorRegistry
{
  struct ErrorInterval { uint64_t start, end; };
  void add_error(const std::string& name, ErrorInterval iv)
  {
    std::lock_guard<std::mutex> lk(mu);
    errors[name] = iv;
    ++counts[name];
  }
  std::mutex mu;
  std::map<std::string, ErrorInterval> errors;
  std::map<std::string, uint64_t> counts;
};
// detchannelmaps::TPCChannelMap::get_offline_channel_from_crate_slot_stream_chan
using ChannelMap = std::function<uint32_t(uint32_t crate, uint32_t slot, uint32_t stream, uint32_t chan)>;
ChannelMap make_map(const std::string& name); // "linear" | "reversed" stand-ins (see .cpp); unknown names throw
// detchannelmaps::TPCChannelMap::get_plane_from_offline_channel. Stand-in: an APA-like 2560-channel period, planes
// 1, 2 (induction) and 0 (collection, the last 992 channels) — only "plane == 0" matters to the reference (:445).
inline uint32_t
get_plane_from_offline_channel(uint32_t offline_channel)
{
  const uint32_t c = offline_channel % 2560u;
  return c < 800u ? 1u : (c < 1568u ? 2u : 0u);
}
// iomanager sender: non-blocking try_send
using TpSink = std::function<bool(TriggerPrimitiveTypeAdapter&&)>;

// ---- readoutlibs::TaskRawDataProcessorModel stand-in -------------------------------------------------------------------
template<class ReadoutType>
class TaskRawDataProcessorModel
{
public:
  explicit TaskRawDataProcessorModel(std::unique_ptr<FrameErrorRegistry>& reg) : m_error_registry(reg) {}
  virtual ~TaskRawDataProcessorModel() = default;
  virtual void conf(const RawDataProcessorConf& c) { m_emulator_mode = c.emulator_mode; }
  virtual void start() {}
  virtual void stop() {}
  // consumer thread: pre tasks synchronously, then (after the latency-buffer insert) the post tasks. The real model runs
  // each post task on its own thread behind an SPSC queue; the stand-in calls them inline.
  void preprocess_item(ReadoutType* item)
  {
    for (auto& t : m_pre)
      t(item);
  }
  void postprocess_item(const ReadoutType* item)
  {
    for (auto& t : m_post)
      t(item);
  }
  uint64_t get_last_daq_time() const { return m_last_processed_daq_ts.load(); }

protected:
  void add_preprocess_task(std::function<void(ReadoutType*)> t) { m_pre.push_back(std::move(t)); }
  void add_postprocess_task(std::function<void(const ReadoutType*)> t) { m_post.push_back(std::move(t)); }
  void reset_tasks()
  {
    m_pre.clear();
    m_post.clear();
  }
  std::unique_ptr<FrameErrorRegistry>& m_error_registry;
  bool m_emulator_mode = false;
  std::atomic<uint64_t> m_last_processed_daq_ts{ 0 };

private:
  std::vector<std::function<void(ReadoutType*)>> m_pre;
  std::vector<std::function<void(const ReadoutType*)>> m_post;
};

// Not a reference type: ADC statistics of one channel of a link over one window of swtpg_read_adc_stats, reported under the
// offline channel that channel's TPs carry. rms = sqrt(sum_sq / samples - mean^2); all zero when samples == 0.
struct ChannelAdcStats
{
  uint32_t offline_channel = 0;
  uint64_t samples = 0;
  double mean = 0, rms = 0;
  uint16_t min = 0, max = 0;
};

// Not a reference type: the noise power spectrum of one channel of a link over one window of swtpg_read_noise_lags (swtpg_noise_power
// of its lags), reported under the offline channel that channel's TPs carry. power[k] is bin k at k x 1.953125 MHz / N, in ADC
// counts^2 (the mean over segments of |rfft|^2 / N): N / 2 + 1 = 33 bins for WIBEth, 25 for WIB2 (the rest zero); all zero when
// segments == 0.
struct ChannelNoiseSpectrum
{
  uint32_t offline_channel = 0;
  uint64_t segments = 0;
  double power[SWTPG_WIBETH_NOISE_SEGMENT_TICKS / 2 + 1] = {};
};

// Not a reference type: the channel covariance of a link over one window of swtpg_read_channel_products (swtpg_channel_covariance
// of its products). Row and column c are frame channel c, reported under the offline channel offline_channel[c] that its TPs
// carry. covariance and correlation are C x C row-major, full and symmetric: ADC counts^2, and NaN where a channel has no variance.
struct ChannelCovariance
{
  uint64_t samples = 0;
  std::vector<uint32_t> offline_channel;
  std::vector<double> covariance, correlation;
};

// ---- the GPU pipeline shared by the links of one device -------------------------------------------------------------------
class FrameProcessorBase;
// One swtpg_handle per GPU; every frame processor attached to it owns one link index. Any link's post-processing thread
// may drain completed batches: records are routed to the processor of their link (swtpg_tp.link).
class TpgEngine
{
public:
  // flags: SWTPG_FLAG_* of include/swtpg.h (SWTPG_FLAG_SORTED_TPS: every link's block of a delivered batch is in time order)
  TpgEngine(int device, swtpg_format format, uint32_t n_links, uint32_t superchunk_units, uint32_t n_slots = 4, uint32_t tp_capacity = 0,
            uint32_t flags = SWTPG_FLAG_NONE);
  ~TpgEngine();
  TpgEngine(const TpgEngine&) = delete;
  uint32_t attach(FrameProcessorBase* p);      // conf(): returns the link index
  // conf() of the processor attached as `link`: the first one creates the handle with its parameters, every later one sets its
  // own link's (swtpg_set_link_config), so links of one device may run different algorithms and thresholds. Before start().
  void configure(uint32_t link, const swtpg_config& algo);
  void start();                                // idempotent per run: the first processor to start creates the handle state
  void stop();                                 // flush + drain; the last processor to stop ends the run
  // per-position RS memory factor of one link, by FRAME channel (src/wibeth/WIBEthFrameProcessor.cpp:437-456 + setState)
  void set_link_memory_factor(uint32_t link, const uint16_t* by_channel, uint32_t n_channels);
  // per-channel hit thresholds of one link, by FRAME channel (swtpg_set_link_thresholds); nullptr = the link's tpg_threshold.
  // Before start(), like configure().
  void set_link_thresholds(uint32_t link, const uint16_t* by_channel, uint32_t n_channels);
  // swtpg_read_adc_stats of one link: out[n_channels] by frame channel (an engine created with SWTPG_FLAG_ADC_STATS). After conf().
  void read_adc_stats(uint32_t link, swtpg_adc_stats* out, uint32_t n_channels, bool reset);
  // swtpg_read_noise_lags of one link: out[n_channels] by frame channel (an engine created with SWTPG_FLAG_NOISE_SPECTRA). After conf().
  void read_noise_lags(uint32_t link, swtpg_noise_lags* out, uint32_t n_channels, bool reset);
  // swtpg_read_channel_products of one link: out[words], words = SWTPG_CHANNEL_PRODUCTS_WORDS of its channels (an engine created
  // with SWTPG_FLAG_CHANNEL_COVARIANCE). After conf().
  void read_channel_products(uint32_t link, uint64_t* out, size_t words, bool reset);
  swtpg_format format() const { return swtpg_format(m_cfg.format); }
  // false = back-pressure (the link's ring is full). wait_us > 0: sleep up to that long for room first (swtpg_submit_wait)
  bool submit(uint32_t link, const void* unit, size_t bytes, uint64_t wait_us = 0);
  // Zero-copy ingest: the latency buffer(s) the constframeptrs point into (swtpg_register_buffer). After conf().
  void register_latency_buffer(void* base, size_t bytes);
  void unregister_latency_buffer(void* base);
  // TPs of completed batches -> process_swtpg_hits of their links' processors. While the engine runs this is the job of its
  // own delivery thread (swtpg_poll_wait: asleep until a batch completes), so no link thread ever polls or contends for it;
  // drain(true) is what stop() uses: flush, then deliver until the library reports nothing pending, in flight or ready.
  void drain(bool wait = false);
  swtpg_handle* handle() { return m_h; }
  uint32_t n_links() const { return m_cfg.n_links; }

private:
  swtpg_config m_cfg{};
  swtpg_handle* m_h = nullptr;
  bool m_configured = false;
  std::vector<FrameProcessorBase*> m_procs;
  std::mutex m_mu, m_drain_mu;
  uint32_t m_started = 0;
  std::vector<swtpg_tp> m_buf, m_sorted;
  std::vector<uint32_t> m_link_count;
  std::thread m_delivery;
  std::atomic<bool> m_delivery_quit{ false };
  size_t deliver_once(uint64_t wait_us);
};

class FrameProcessorBase
{
public:
  virtual ~FrameProcessorBase() = default;
  virtual void process_swtpg_hits(const swtpg_tp* tps, size_t n) = 0; // records of THIS link, any order
};

// ---- the link plumbing both TPC formats share ----------------------------------------------------------------------------
// What WIBEthFrameProcessor and WIB2FrameProcessor of the reference each write out in full: the link's attachment in conf(),
// the TPG part of start / stop / get_info, the per-channel tables built on the first frame, the submit of find_hits and the
// TriggerPrimitive tail of process_swtpg_hits. kChannels: frame channels of one payload. kCountEveryTp: num_tps_sent and the
// hit rate count every record that passed the mask, whatever tp_timeout or tp_out made of it (WIB2,
// src/wib2/WIB2FrameProcessor.cpp:469-470), rather than only the records tp_out accepted (WIBEth).
template<class ReadoutType, class FrameHandler, uint32_t kChannels, bool kCountEveryTp>
class TpcFrameProcessor : public TaskRawDataProcessorModel<ReadoutType>, public FrameProcessorBase
{
  static_assert((kChannels & (kChannels - 1)) == 0, "a record's frame channel is its channel field modulo kChannels");

public:
  using inherited = TaskRawDataProcessorModel<ReadoutType>;
  using frameptr = ReadoutType*;
  using constframeptr = const ReadoutType*;

  void init(TpSink tp_out) { m_tp_sink = std::move(tp_out); } // reference: get_iom_sender("tp_out")
  void start() override;
  void stop() override;
  void get_info(RawDataProcessorInfo& info);
  // Not in the reference: the ADC statistics of this link's channels since the last reset (engine flag SWTPG_FLAG_ADC_STATS), by
  // the offline channel its TPs carry, masked channels included. Empty until the first frame has built the channel map.
  void get_adc_stats(std::vector<ChannelAdcStats>& out, bool reset);
  // Not in the reference: the noise power spectra of this link's channels since the last reset (engine flag
  // SWTPG_FLAG_NOISE_SPECTRA), by the offline channel its TPs carry, masked channels included. Empty until the first frame has
  // built the channel map.
  void get_noise_spectra(std::vector<ChannelNoiseSpectrum>& out, bool reset);
  // Not in the reference: the covariance and correlation of this link's channels since the last reset (engine flag
  // SWTPG_FLAG_CHANNEL_COVARIANCE), rows in frame-channel order under the offline channel its TPs carry, masked channels
  // included. Empty (no rows) until the first frame has built the channel map.
  void get_channel_covariance(ChannelCovariance& out, bool reset);
  void process_swtpg_hits(const swtpg_tp* tps, size_t n) override; // fed with device TP records
  FrameHandler* handler() { return m_frame_handler.get(); }

protected:
  TpcFrameProcessor(std::unique_ptr<FrameErrorRegistry>& error_registry, std::shared_ptr<TpgEngine> engine);
  // The rest of conf() once the caller has parsed its algorithm into `a` and registered its pre-process tasks: the link's
  // tp_timeout, channel mask, ids and back-pressure policy, and with enable_tpg its engine link, configuration, threshold
  // table and the post-process task find_hits.
  void conf_link(const RawDataProcessorConf& config, const swtpg_config& a, std::function<void(constframeptr)> find_hits);
  // First frame: the offline channel offline_of(c) that records of frame channel c are reported with, its mask flag, a zeroed
  // rate counter; then get_info, get_adc_stats, get_noise_spectra and get_channel_covariance may read them.
  template<class OfflineOf>
  void set_channel_tables(OfflineOf offline_of)
  {
    for (uint32_t c = 0; c < kChannels; ++c) {
      m_offline_of_channel[c] = offline_of(c);
      m_masked[c] = m_channel_mask_set.count(m_offline_of_channel[c]) ? 1 : 0;
      m_tp_channel_rate[c].store(0, std::memory_order_relaxed);
    }
    m_maps_ready.store(true, std::memory_order_release);
  }
  // The frame is only borrowed for the duration of find_hits: swtpg_submit copies it into the pinned staging slot — unless it
  // lies in a latency buffer registered with the engine, which the copy engine then reads directly (zero-copy ingest).
  // Non-blocking by default, like the reference's try_send: a full ring drops the frame and counts it. With
  // block_on_backpressure the thread SLEEPS until the completion thread has freed ring space (swtpg_submit_wait). TPs come
  // back through the engine's delivery thread (process_swtpg_hits), never through this thread.
  void submit(constframeptr fp, uint32_t link)
  {
    if (!m_block) {
      if (!m_engine->submit(link, fp->data, sizeof fp->data))
        ++m_frames_dropped;
    } else {
      while (!m_engine->submit(link, fp->data, sizeof fp->data, 100000)) {
      }
    }
  }

  std::shared_ptr<TpgEngine> m_engine;
  std::unique_ptr<FrameHandler> m_frame_handler;
  TpSink m_tp_sink;
  ChannelMap m_channel_map;
  bool m_tpg_enabled = false, m_block = false;
  TriggerPrimitive::Algorithm m_tp_algo = TriggerPrimitive::Algorithm::kUnknown; // never assigned for WIB2 (wib2/WIB2FrameProcessor.hpp:137)
  uint64_t m_tp_max_width = 0;
  std::set<uint32_t> m_channel_mask_set;
  uint32_t m_crate_no = 0, m_slot_no = 0, m_link_no = 0, m_det_id = 0;
  // m_tp_channel_rate_map of the reference, kept as one counter per FRAME channel (the key of every record) and turned into
  // (offline channel -> count) pairs in get_info; the channel mask likewise is looked up once per channel
  std::array<std::atomic<uint32_t>, kChannels> m_tp_channel_rate{};
  std::array<uint32_t, kChannels> m_offline_of_channel{};
  std::array<uint8_t, kChannels> m_masked{};
  std::atomic<bool> m_maps_ready{ false };
  uint64_t m_previous_ts = 0, m_current_ts = 0;
  std::atomic<uint64_t> m_ts_error_ctr{ 0 }, m_new_tps{ 0 }, m_tpg_hits_count{ 0 }, m_tps_suppressed_too_long{ 0 }, m_tps_send_failed{ 0 },
    m_frames_dropped{ 0 };
  std::chrono::time_point<std::chrono::high_resolution_clock> m_t0;
};

// ---- WIBEth ---------------------------------------------------------------------------------------------------------------
// include/fdreadoutlibs/wibeth/WIBEthFrameProcessor.hpp:45-71. The handler keeps its role (per-link TPG resources) but the
// resources are now a link slot of the engine instead of a hit buffer + ProcessingInfo.
class WIBEthFrameHandler
{
public:
  bool first_hit = true;
  std::array<uint32_t, 64> register_channel_map{}; // position p -> offline channel (RegisterToChannelNumber.cpp:35-122)
  uint32_t link = 0;
  void reset() { first_hit = true; }
};

// include/fdreadoutlibs/wibeth/WIBEthFrameProcessor.hpp:73-205
class WIBEthFrameProcessor : public TpcFrameProcessor<DUNEWIBEthTypeAdapter, WIBEthFrameHandler, SWTPG_WIBETH_CHANNELS, false>
{
public:
  WIBEthFrameProcessor(std::unique_ptr<FrameErrorRegistry>& error_registry, std::shared_ptr<TpgEngine> engine)
    : TpcFrameProcessor(error_registry, std::move(engine))
  {
  }

  void conf(const RawDataProcessorConf& cfg) override;                 // (:172-235)
  void start() override;                                                // (:111-144)
  void get_info(RawDataProcessorInfo& info);                            // (:237-292)
  void sequence_check(frameptr fp);                                     // (:298-353)
  void timestamp_check(frameptr fp);                                    // (:359-405)
  void find_hits(constframeptr fp, WIBEthFrameHandler* frame_handler); // (:410-476)

  const std::vector<LinkMisconfiguration>& misconfigurations() const { return m_misconf; }

private:
  bool m_enable_simple_threshold_on_collection = false, m_correct_lookup = false;
  uint16_t m_tpg_rs_memory_factor = 0;
  std::vector<LinkMisconfiguration> m_misconf;
  uint16_t m_previous_seq_id = 0, m_current_seq_id = 0;
  std::atomic<uint64_t> m_seq_id_error_ctr{ 0 };
  std::atomic<int16_t> m_seq_id_min_jump{ 0 }, m_seq_id_max_jump{ 0 };
};

// ---- WIB2 -----------------------------------------------------------------------------------------------------------------
// include/fdreadoutlibs/wib2/WIB2FrameProcessor.hpp:45-175. The reference runs two handlers (register_selector 0/1, 128
// channels each) on two post-processing threads; the device processes the whole 256-channel superchunk, so one task remains.
class WIB2FrameHandler
{
public:
  bool first_hit = true;
  uint32_t link = 0;
  void reset() { first_hit = true; }
};

class WIB2FrameProcessor : public TpcFrameProcessor<DUNEWIBSuperChunkTypeAdapter, WIB2FrameHandler, SWTPG_WIB2_CHANNELS, true>
{
public:
  WIB2FrameProcessor(std::unique_ptr<FrameErrorRegistry>& error_registry, std::shared_ptr<TpgEngine> engine)
    : TpcFrameProcessor(error_registry, std::move(engine))
  {
  }

  void conf(const RawDataProcessorConf& cfg) override;                // src/wib2/WIB2FrameProcessor.cpp:196-229
  void timestamp_check(frameptr fp);                                   // (:293-340)
  void find_hits(constframeptr fp, WIB2FrameHandler* frame_handler); // (:345-396)
};

extern template class TpcFrameProcessor<DUNEWIBEthTypeAdapter, WIBEthFrameHandler, SWTPG_WIBETH_CHANNELS, false>;
extern template class TpcFrameProcessor<DUNEWIBSuperChunkTypeAdapter, WIB2FrameHandler, SWTPG_WIB2_CHANNELS, true>;

// ---- downstream of the path: TPs -> time-ordered TPSets -------------------------------------------------------------------
// trigger::TPSet as send_tp_sets fills it (src/TPCTPRequestHandler.cpp:145-165)
struct TPSet
{
  enum class Type : uint32_t { kUnknown = 0, kPayload = 1, kHeartbeat = 2 };
  uint64_t seqno = 0;
  uint32_t run_number = 0;
  uint32_t origin = 0; // source id
  Type type = Type::kUnknown;
  uint64_t start_time = 0, end_time = 0;
  std::vector<TriggerPrimitive> objects;
};
// The fields of readoutlibs' ReadoutModelConf that TPCTPRequestHandler::conf reads (src/TPCTPRequestHandler.cpp:20-28)
struct ReadoutModelConf
{
  uint32_t source_id = 0;
  uint32_t tpset_transmission_rate_hz = 100;
  uint64_t tpset_min_latency_ticks = 100000;
  int tardy_tp_quiet_time_at_start_sec = 10;
};
struct TPRequestHandlerInfo // the readoutinfo fields get_info fills (:57-82)
{
  uint64_t num_tps_sent = 0, num_tpsets_sent = 0, num_tps_in_tpsets_send_failed = 0, num_tpsets_send_failed = 0, num_tps_suppressed_tardy = 0,
           num_heartbeats = 0;
};
using TPSetSink = std::function<bool(TPSet&&)>;

// include/fdreadoutlibs/TPCTPRequestHandler.hpp:57-108 + src/TPCTPRequestHandler.cpp: the consumer of the (merged) TP stream.
// The skip-list latency buffer of readoutlibs is restated as an ordered multiset keyed like TriggerPrimitiveTypeAdapter
// (time_start, channel); the periodic sender thread is one explicit call per cycle (send_tp_sets_once), so the windowing
// logic can be driven deterministically. This is what bounds the GPU batching latency: a TP whose time_start is below the
// published cut-off when it arrives is "tardy" and dropped (readoutlibs ReadoutModel consults get_cutoff_timestamp()).
class TPCTPRequestHandler
{
public:
  void init(TPSetSink tpset_out) { m_tpset_sink = std::move(tpset_out); }
  void conf(const ReadoutModelConf& c);
  void start(uint32_t run_number);
  void stop();
  void get_info(TPRequestHandlerInfo& info);
  uint64_t get_cutoff_timestamp() const { return m_cutoff_timestamp.load(); }
  bool supports_cutoff_timestamp() const { return true; }
  void report_tardy_packet(const TriggerPrimitiveTypeAdapter& packet, int64_t tardy_ticks);
  // what ReadoutModel's consumer does with an arriving TP: tardy check against the cut-off, else latency-buffer insert
  bool receive(TriggerPrimitiveTypeAdapter&& tp);
  // one iteration of the sender thread's loop body (:108-191); returns true if a TPSet (payload or heartbeat) was produced
  bool send_tp_sets_once();
  size_t occupancy() const { return m_latency_buffer.size(); }
  // latency-buffer clean-up stand-in: forget TPs older than `ts` (the skip-list request handler pops them periodically)
  void pop_older_than(uint64_t ts);

private:
  std::multiset<TriggerPrimitiveTypeAdapter> m_latency_buffer;
  TPSetSink m_tpset_sink;
  uint32_t m_source_id = 0, m_run_number = 0;
  int m_tp_set_sender_sleep_us = 10000, m_tardy_tp_quiet_time_at_start_sec = 10;
  uint64_t m_ts_set_sender_offset_ticks = 0, m_next_tpset_seqno = 0;
  uint64_t m_start_win_ts = 0;
  bool m_first_cycle = true;
  std::atomic<uint64_t> m_new_tps{ 0 }, m_new_tpsets{ 0 }, m_new_tps_in_tpsets_send_failed{ 0 }, m_new_tpsets_send_failed{ 0 },
    m_new_tps_suppressed_tardy{ 0 }, m_new_heartbeats{ 0 }, m_late_warnings{ 0 };
  std::atomic<uint64_t> m_cutoff_timestamp{ 0 };
  std::chrono::time_point<std::chrono::high_resolution_clock> m_run_start_timepoint;
};

} // namespace host
} // namespace swtpg
