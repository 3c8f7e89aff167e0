// Implementation of the host-side frame processors (see swtpg_host.hpp). Plain C++17; the only dependency is the C ABI of
// libswtpg_b200.so. There is no CPU hit finder here: without a device, TpgEngine::start throws.
#include "swtpg_host.hpp"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <ctime>
#include <thread>
#include <variant>

namespace swtpg {
namespace host {

namespace {
// Lane l of AVX2 register r holds frame channel 16r + kPerm[l] (unittest/WIBEthFrameExpansion_test.cxx:111,124)
constexpr int kPerm[16] = { 0, 1, 2, 3, 4, 5, 6, 7, 15, 8, 9, 10, 11, 12, 13, 14 };
inline uint32_t
position_to_frame_channel(uint32_t pos)
{
  return (pos & ~15u) | uint32_t(kPerm[pos & 15u]);
}
void
check(swtpg_handle* h, swtpg_status s, const char* what)
{
  if (s != SWTPG_OK)
    throw std::runtime_error(std::string(what) + ": " + swtpg_status_string(s) + " — " + (swtpg_last_error(h) ? swtpg_last_error(h) : ""));
}
} // namespace

ChannelMap
make_map(const std::string& name)
{
  // detchannelmaps is not part of the reference repository. "linear" numbers the channels of consecutive streams
  // consecutively inside a (crate, slot); "reversed" additionally flips each group of 64 (exercises a non-monotonic map).
  if (name == "linear")
    return [](uint32_t crate, uint32_t slot, uint32_t stream, uint32_t chan) { return ((crate * 8 + slot) * 64 + stream) * 64 + chan; };
  if (name == "reversed")
    return [](uint32_t crate, uint32_t slot, uint32_t stream, uint32_t chan) { return ((crate * 8 + slot) * 64 + stream) * 64 + (63 - (chan & 63)) + (chan & ~63u); };
  throw std::runtime_error("unknown channel map: " + name);
}

// ---- TpgEngine ------------------------------------------------------------------------------------------------------
TpgEngine::TpgEngine(int device, swtpg_format format, uint32_t n_links, uint32_t superchunk_units, uint32_t n_slots, uint32_t tp_capacity,
                     uint32_t flags)
{
  m_cfg.struct_size = sizeof m_cfg;
  m_cfg.device = device;
  m_cfg.format = format;
  m_cfg.n_links = n_links;
  m_cfg.max_units = superchunk_units;
  m_cfg.n_slots = n_slots;
  m_cfg.tp_capacity = tp_capacity;
  m_cfg.flags = flags;
  m_procs.assign(n_links, nullptr);
  m_buf.resize(1 << 16);
}

TpgEngine::~TpgEngine()
{
  if (m_h)
    swtpg_destroy(m_h);
}

uint32_t
TpgEngine::attach(FrameProcessorBase* p)
{
  std::lock_guard<std::mutex> lk(m_mu);
  for (uint32_t i = 0; i < m_procs.size(); ++i)
    if (m_procs[i] == p)
      return i;
  for (uint32_t i = 0; i < m_procs.size(); ++i)
    if (!m_procs[i]) {
      m_procs[i] = p;
      return i;
    }
  throw std::runtime_error("TpgEngine: more frame processors than links");
}

void
TpgEngine::configure(uint32_t link, const swtpg_config& a)
{
  std::lock_guard<std::mutex> lk(m_mu);
  if (m_configured) { // every link parses its own RawDataProcessorConf (src/wibeth/WIBEthFrameProcessor.cpp:175-230)
    swtpg_link_config c{};
    c.struct_size = sizeof c;
    c.algorithm = a.algorithm;
    c.threshold = a.threshold;
    c.frugal_acc_limit = a.frugal_acc_limit;
    c.rs_memory_factor = a.rs_memory_factor;
    c.rs_scale_factor = a.rs_scale_factor;
    memcpy(c.fir_taps, a.fir_taps, sizeof c.fir_taps);
    c.tap_exponent = a.tap_exponent;
    check(m_h, swtpg_set_link_config(m_h, link, &c), "swtpg_set_link_config");
    return;
  }
  m_cfg.algorithm = a.algorithm;
  m_cfg.threshold = a.threshold;
  m_cfg.frugal_acc_limit = a.frugal_acc_limit;
  m_cfg.rs_memory_factor = a.rs_memory_factor;
  m_cfg.rs_scale_factor = a.rs_scale_factor;
  swtpg_handle* h = nullptr;
  const swtpg_status s = swtpg_create(&m_cfg, &h);
  if (s != SWTPG_OK)
    throw std::runtime_error(std::string("swtpg_create: ") + swtpg_status_string(s) + " — " + swtpg_last_error(nullptr));
  m_h = h;
  m_configured = true;
}

void
TpgEngine::start()
{
  std::lock_guard<std::mutex> lk(m_mu);
  if (!m_h)
    throw std::runtime_error("TpgEngine::start before conf");
  if (m_started++ == 0) {
    check(m_h, swtpg_start(m_h), "swtpg_start");
    m_delivery_quit = false;
    m_delivery = std::thread([this] { // hands TPs to the links' processors as batches complete; asleep in between
      while (!m_delivery_quit.load(std::memory_order_acquire)) {
        try {
          std::lock_guard<std::mutex> dl(m_drain_mu);
          deliver_once(2000);
        } catch (const std::exception&) {
          return; // the next call into the engine (submit / stop) reports the failure
        }
      }
    });
  }
}

void
TpgEngine::stop()
{
  {
    std::lock_guard<std::mutex> lk(m_mu);
    if (m_started == 0 || --m_started != 0)
      return;
  }
  m_delivery_quit.store(true, std::memory_order_release);
  if (m_delivery.joinable())
    m_delivery.join();
  drain(true); // flush the ragged tail, deliver everything that is left
  check(m_h, swtpg_stop(m_h), "swtpg_stop");
}

void
TpgEngine::set_link_memory_factor(uint32_t link, const uint16_t* by_channel, uint32_t)
{
  // one small asynchronous copy for this link's rows, ordered on the compute stream; no engine-wide lock, no other link waits
  check(m_h, swtpg_set_link_rs_memory_factor(m_h, link, by_channel), "swtpg_set_link_rs_memory_factor");
}

void
TpgEngine::read_adc_stats(uint32_t link, swtpg_adc_stats* out, uint32_t n_channels, bool reset)
{
  const uint32_t channels = m_cfg.format == SWTPG_FORMAT_WIB2 ? SWTPG_WIB2_CHANNELS : SWTPG_WIBETH_CHANNELS;
  if (n_channels != channels)
    throw std::invalid_argument("TpgEngine::read_adc_stats: one entry per frame channel of the link");
  check(m_h, swtpg_read_adc_stats(m_h, link, 1, out, reset ? 1 : 0), "swtpg_read_adc_stats");
}

void
TpgEngine::read_noise_lags(uint32_t link, swtpg_noise_lags* out, uint32_t n_channels, bool reset)
{
  const uint32_t channels = m_cfg.format == SWTPG_FORMAT_WIB2 ? SWTPG_WIB2_CHANNELS : SWTPG_WIBETH_CHANNELS;
  if (n_channels != channels)
    throw std::invalid_argument("TpgEngine::read_noise_lags: one entry per frame channel of the link");
  check(m_h, swtpg_read_noise_lags(m_h, link, 1, out, reset ? 1 : 0), "swtpg_read_noise_lags");
}

void
TpgEngine::read_channel_products(uint32_t link, uint64_t* out, size_t words, bool reset)
{
  const uint32_t channels = m_cfg.format == SWTPG_FORMAT_WIB2 ? SWTPG_WIB2_CHANNELS : SWTPG_WIBETH_CHANNELS;
  if (words != SWTPG_CHANNEL_PRODUCTS_WORDS(channels))
    throw std::invalid_argument("TpgEngine::read_channel_products: SWTPG_CHANNEL_PRODUCTS_WORDS words of the link");
  check(m_h, swtpg_read_channel_products(m_h, link, 1, out, reset ? 1 : 0), "swtpg_read_channel_products");
}

void
TpgEngine::set_link_thresholds(uint32_t link, const uint16_t* by_channel, uint32_t n_channels)
{
  const uint32_t channels = m_cfg.format == SWTPG_FORMAT_WIB2 ? SWTPG_WIB2_CHANNELS : SWTPG_WIBETH_CHANNELS;
  if (by_channel && n_channels != channels)
    throw std::invalid_argument("TpgEngine::set_link_thresholds: one threshold per frame channel of the link");
  check(m_h, swtpg_set_link_thresholds(m_h, link, by_channel), "swtpg_set_link_thresholds");
}

static bool
has_plane_thresholds(const RawDataProcessorConf& config)
{
  const auto& plane = config.tpg_plane_threshold;
  return plane[0] >= 0 || plane[1] >= 0 || plane[2] >= 0;
}

// The per-frame-channel table of RawDataProcessorConf::tpg_plane_threshold: channel c of the link (crate, slot, link) takes the
// threshold of its plane, or tpg_threshold where that is -1. Empty when no plane has its own.
static std::vector<uint16_t>
plane_threshold_table(const RawDataProcessorConf& config, const ChannelMap& map, uint32_t channels)
{
  std::vector<uint16_t> table;
  const auto& plane = config.tpg_plane_threshold;
  if (!has_plane_thresholds(config))
    return table;
  for (int32_t t : plane)
    if (t > 32767)
      throw std::invalid_argument("tpg_plane_threshold: above 32767");
  for (uint32_t c = 0; c < channels; ++c) {
    const int32_t t = plane[get_plane_from_offline_channel(map(config.crate_id, config.slot_id, config.link_id, c))];
    table.push_back(t >= 0 ? uint16_t(t) : config.tpg_threshold);
  }
  return table;
}

bool
TpgEngine::submit(uint32_t link, const void* unit, size_t bytes, uint64_t wait_us)
{
  const swtpg_status s = wait_us ? swtpg_submit_wait(m_h, link, unit, bytes, wait_us) : swtpg_submit(m_h, link, unit, bytes);
  if (s == SWTPG_ERR_BUSY)
    return false;
  check(m_h, s, "swtpg_submit");
  return true;
}

void
TpgEngine::register_latency_buffer(void* base, size_t bytes)
{
  std::lock_guard<std::mutex> lk(m_mu);
  if (!m_h)
    throw std::runtime_error("TpgEngine::register_latency_buffer before conf");
  check(m_h, swtpg_register_buffer(m_h, base, bytes), "swtpg_register_buffer");
}

void
TpgEngine::unregister_latency_buffer(void* base)
{
  std::lock_guard<std::mutex> lk(m_mu);
  if (m_h)
    check(m_h, swtpg_unregister_buffer(m_h, base), "swtpg_unregister_buffer");
}

// One poll (sleeping up to wait_us for a completed batch) and the hand-over of its records: a counting sort by link, then one
// process_swtpg_hits call per link that has any. Caller holds m_drain_mu.
size_t
TpgEngine::deliver_once(uint64_t wait_us)
{
  size_t n = 0;
  const swtpg_status s = wait_us ? swtpg_poll_wait(m_h, m_buf.data(), m_buf.size(), &n, wait_us) : swtpg_poll(m_h, m_buf.data(), m_buf.size(), &n);
  if (s != SWTPG_OK && s != SWTPG_ERR_OVERFLOW)
    check(m_h, s, "swtpg_poll");
  if (n == 0)
    return 0;
  const size_t n_links = m_procs.size();
  m_link_count.assign(n_links + 1, 0u);
  for (size_t i = 0; i < n; ++i)
    if (m_buf[i].link < n_links)
      ++m_link_count[m_buf[i].link + 1];
  for (size_t l = 0; l < n_links; ++l)
    m_link_count[l + 1] += m_link_count[l];
  m_sorted.resize(m_buf.size());
  {
    std::vector<uint32_t>& at = m_link_count; // running write positions: at[l] ends up as the END of link l's block
    for (size_t i = 0; i < n; ++i)
      if (m_buf[i].link < n_links)
        m_sorted[at[m_buf[i].link]++] = m_buf[i];
  }
  size_t begin = 0;
  for (size_t l = 0; l < n_links; ++l) {
    const size_t end = m_link_count[l];
    if (end > begin && m_procs[l])
      m_procs[l]->process_swtpg_hits(m_sorted.data() + begin, end - begin);
    begin = end;
  }
  return n;
}

void
TpgEngine::drain(bool wait)
{
  std::unique_lock<std::mutex> lk(m_drain_mu, std::defer_lock);
  if (wait)
    lk.lock();
  else if (!lk.try_lock())
    return; // the delivery thread (or another caller) is at it
  if (!wait) {
    for (int pass = 0; pass < 4 && deliver_once(0); ++pass) {
    }
    return;
  }
  // stop(): everything submitted must come out. The loop ends on the library's own bookkeeping — nothing pending, nothing in
  // flight, nothing ready — never on "a poll brought no records" (a batch without TPs is still a batch in flight).
  for (;;) {
    const swtpg_status fs = swtpg_flush(m_h); // BUSY: every batch waits to be polled — deliver, then flush again
    if (fs != SWTPG_OK && fs != SWTPG_ERR_BUSY)
      check(m_h, fs, "swtpg_flush");
    if (fs == SWTPG_OK)
      check(m_h, swtpg_sync(m_h), "swtpg_sync");
    while (deliver_once(0)) {
    }
    uint64_t pending = 0;
    uint32_t in_flight = 0, ready = 0;
    check(m_h, swtpg_stream_status(m_h, &pending, &in_flight, &ready), "swtpg_stream_status");
    if (fs == SWTPG_OK && pending == 0 && in_flight == 0 && ready == 0)
      return;
  }
}

// ---- TpcFrameProcessor ------------------------------------------------------------------------------------------------
namespace {
ChannelAdcStats
channel_adc_stats(uint32_t offline_channel, const swtpg_adc_stats& a)
{
  ChannelAdcStats o;
  o.offline_channel = offline_channel;
  o.samples = a.samples;
  if (a.samples) {
    // variance = (n sum_sq - sum^2) / n^2, the numerator exact in 128 bits
    const unsigned __int128 n = a.samples, num = n * a.sum_sq - (unsigned __int128)a.sum * a.sum;
    o.mean = double(a.sum) / double(a.samples);
    o.rms = std::sqrt(double(num) / (double(a.samples) * double(a.samples)));
    o.min = a.min;
    o.max = a.max;
  }
  return o;
}
} // namespace

template<class R, class H, uint32_t kChannels, bool kCountEveryTp>
TpcFrameProcessor<R, H, kChannels, kCountEveryTp>::TpcFrameProcessor(std::unique_ptr<FrameErrorRegistry>& error_registry,
                                                                     std::shared_ptr<TpgEngine> engine)
  : inherited(error_registry)
  , m_engine(std::move(engine))
  , m_frame_handler(std::make_unique<H>())
{
}

template<class R, class H, uint32_t kChannels, bool kCountEveryTp>
void
TpcFrameProcessor<R, H, kChannels, kCountEveryTp>::conf_link(const RawDataProcessorConf& config, const swtpg_config& a,
                                                             std::function<void(constframeptr)> find_hits)
{
  m_tp_max_width = config.tp_timeout;
  m_channel_mask_set.insert(config.tpg_channel_mask.begin(), config.tpg_channel_mask.end());
  m_crate_no = config.crate_id;
  m_slot_no = config.slot_id;
  m_link_no = config.link_id;
  m_block = config.block_on_backpressure;
  if (config.enable_tpg) {
    m_tpg_enabled = true;
    m_channel_map = make_map(config.channel_map_name);
    m_frame_handler->link = m_engine->attach(this);
    m_engine->configure(m_frame_handler->link, a);
    // the table must be in place before start(), so it comes from the configured ids rather than the first frame's header (a
    // WIBEth link whose frames carry other ids is reported as a LinkMisconfiguration)
    const std::vector<uint16_t> table = plane_threshold_table(config, m_channel_map, kChannels);
    m_engine->set_link_thresholds(m_frame_handler->link, table.empty() ? nullptr : table.data(), uint32_t(table.size()));
    inherited::add_postprocess_task(std::move(find_hits));
  }
  inherited::conf(config);
}

template<class R, class H, uint32_t kChannels, bool kCountEveryTp>
void
TpcFrameProcessor<R, H, kChannels, kCountEveryTp>::start()
{
  if (m_tpg_enabled) {
    m_tps_suppressed_too_long = 0;
    m_tps_send_failed = 0;
    m_frames_dropped = 0;
    m_frame_handler->reset(); // = initialize(): fresh per-link resources; the device state is zeroed by swtpg_start
    m_engine->start();
  }
  m_previous_ts = m_current_ts = 0;
  m_ts_error_ctr = 0;
  m_t0 = std::chrono::high_resolution_clock::now();
  m_new_tps = 0;
  m_tpg_hits_count = 0;
  inherited::start();
}

template<class R, class H, uint32_t kChannels, bool kCountEveryTp>
void
TpcFrameProcessor<R, H, kChannels, kCountEveryTp>::stop()
{
  inherited::stop();
  if (m_tpg_enabled) {
    m_engine->stop(); // flushes the partially filled superchunk and delivers the remaining TPs through process_swtpg_hits
    m_frame_handler->reset();
  }
}

template<class R, class H, uint32_t kChannels, bool kCountEveryTp>
void
TpcFrameProcessor<R, H, kChannels, kCountEveryTp>::get_info(RawDataProcessorInfo& info)
{
  info = RawDataProcessorInfo{};
  info.num_ts_errors = m_ts_error_ctr.load();
  const auto now = std::chrono::high_resolution_clock::now();
  if (m_tpg_enabled) {
    const uint64_t new_hits = m_tpg_hits_count.exchange(0);
    const double seconds = std::chrono::duration_cast<std::chrono::microseconds>(now - m_t0).count() / 1000000.;
    info.rate_tp_hits = seconds > 0 ? new_hits / seconds / 1000. : 0;
    info.num_tps_sent = m_new_tps.exchange(0);
    info.num_tps_suppressed_too_long = m_tps_suppressed_too_long.exchange(0);
    info.num_tps_send_failed = m_tps_send_failed.exchange(0);
    info.num_frames_dropped_busy = m_frames_dropped.exchange(0);
    // the ten channels with the most TPs since the last call, then reset (src/wibeth/WIBEthFrameProcessor.cpp:263-284): the
    // reference keeps a std::map keyed by offline channel and sorts its pairs by count; ties keep the map's (ascending channel) order
    if (m_maps_ready.load(std::memory_order_acquire)) {
      std::map<uint32_t, int> rate;
      for (uint32_t c = 0; c < kChannels; ++c)
        rate[m_offline_of_channel[c]] += int(m_tp_channel_rate[c].exchange(0, std::memory_order_relaxed));
      std::vector<std::pair<uint32_t, int>> v(rate.begin(), rate.end());
      std::stable_sort(v.begin(), v.end(), [](const auto& x, const auto& y) { return x.second > y.second; });
      info.n_top = uint32_t(std::min<size_t>(10, v.size()));
      for (uint32_t i = 0; i < info.n_top; ++i) {
        info.top_channels[i] = v[i].first;
        info.top_channel_tps[i] = uint32_t(v[i].second);
      }
    }
  }
  m_t0 = now;
}

template<class R, class H, uint32_t kChannels, bool kCountEveryTp>
void
TpcFrameProcessor<R, H, kChannels, kCountEveryTp>::get_adc_stats(std::vector<ChannelAdcStats>& out, bool reset)
{
  out.clear();
  if (!m_maps_ready.load(std::memory_order_acquire))
    return;
  swtpg_adc_stats s[kChannels];
  m_engine->read_adc_stats(m_frame_handler->link, s, kChannels, reset);
  for (uint32_t c = 0; c < kChannels; ++c)
    out.push_back(channel_adc_stats(m_offline_of_channel[c], s[c]));
}

template<class R, class H, uint32_t kChannels, bool kCountEveryTp>
void
TpcFrameProcessor<R, H, kChannels, kCountEveryTp>::get_noise_spectra(std::vector<ChannelNoiseSpectrum>& out, bool reset)
{
  out.clear();
  if (!m_maps_ready.load(std::memory_order_acquire))
    return;
  std::vector<swtpg_noise_lags> lags(kChannels);
  std::vector<double> power(kChannels * (SWTPG_WIBETH_NOISE_SEGMENT_TICKS / 2 + 1));
  m_engine->read_noise_lags(m_frame_handler->link, lags.data(), kChannels, reset);
  const swtpg_format fmt = m_engine->format();
  const size_t bins = (fmt == SWTPG_FORMAT_WIB2 ? SWTPG_WIB2_NOISE_SEGMENT_TICKS : SWTPG_WIBETH_NOISE_SEGMENT_TICKS) / 2 + 1;
  check(nullptr, swtpg_noise_power(lags.data(), kChannels, fmt, power.data()), "swtpg_noise_power");
  out.resize(kChannels);
  for (uint32_t c = 0; c < kChannels; ++c) {
    out[c].offline_channel = m_offline_of_channel[c];
    out[c].segments = lags[c].segments;
    std::copy(power.begin() + c * bins, power.begin() + (c + 1) * bins, out[c].power);
  }
}

template<class R, class H, uint32_t kChannels, bool kCountEveryTp>
void
TpcFrameProcessor<R, H, kChannels, kCountEveryTp>::get_channel_covariance(ChannelCovariance& out, bool reset)
{
  out = ChannelCovariance{};
  if (!m_maps_ready.load(std::memory_order_acquire))
    return;
  std::vector<uint64_t> products(SWTPG_CHANNEL_PRODUCTS_WORDS(kChannels));
  m_engine->read_channel_products(m_frame_handler->link, products.data(), products.size(), reset);
  out.samples = products[0];
  out.offline_channel.assign(m_offline_of_channel.begin(), m_offline_of_channel.end());
  out.covariance.resize(size_t(kChannels) * kChannels);
  out.correlation.resize(size_t(kChannels) * kChannels);
  check(nullptr, swtpg_channel_covariance(products.data(), 1, m_engine->format(), out.covariance.data(), out.correlation.data()),
        "swtpg_channel_covariance");
}

template<class R, class H, uint32_t kChannels, bool kCountEveryTp>
void
TpcFrameProcessor<R, H, kChannels, kCountEveryTp>::process_swtpg_hits(const swtpg_tp* tps, size_t n)
{
  uint64_t nhits = 0;
  for (size_t i = 0; i < n; ++i) {
    const swtpg_tp& r = tps[i];
    const uint32_t c = r.channel & (kChannels - 1);
    if (m_masked[c]) // offline channel in tpg_channel_mask (src/wibeth/WIBEthFrameProcessor.cpp:528)
      continue;
    TriggerPrimitiveTypeAdapter tp;
    tp.tp.time_start = r.time_start;
    tp.tp.time_peak = r.time_peak;
    tp.tp.time_over_threshold = r.time_over_threshold;
    tp.tp.channel = m_offline_of_channel[c];
    tp.tp.adc_integral = r.adc_integral;
    tp.tp.adc_peak = r.adc_peak;
    tp.tp.detid = uint16_t(m_det_id);
    tp.tp.type = TriggerPrimitive::Type::kTPC;
    tp.tp.algorithm = m_tp_algo;
    tp.tp.version = 1;
    bool sent = false;
    if (tp.tp.time_over_threshold > m_tp_max_width)
      m_tps_suppressed_too_long++; // reference: ers::warning(TPTooLong)
    else if (!m_tp_sink || !m_tp_sink(std::move(tp)))
      m_tps_send_failed++; // reference: ers::warning(FailedToSendTP)
    else
      sent = true;
    if (kCountEveryTp || sent) {
      m_new_tps++;
      ++nhits;
    }
    m_tp_channel_rate[c].fetch_add(1, std::memory_order_relaxed);
  }
  m_tpg_hits_count += nhits;
}

template class TpcFrameProcessor<DUNEWIBEthTypeAdapter, WIBEthFrameHandler, SWTPG_WIBETH_CHANNELS, false>;
template class TpcFrameProcessor<DUNEWIBSuperChunkTypeAdapter, WIB2FrameHandler, SWTPG_WIB2_CHANNELS, true>;

// ---- WIBEthFrameProcessor ---------------------------------------------------------------------------------------------
void
WIBEthFrameProcessor::conf(const RawDataProcessorConf& config)
{
  swtpg_config a{};
  if (config.tpg_algorithm == "SimpleThreshold") {
    m_tp_algo = TriggerPrimitive::Algorithm::kSimpleThreshold;
    a.algorithm = SWTPG_ALGO_SIMPLE_THRESHOLD;
  } else if (config.tpg_algorithm == "AbsRS") {
    m_tp_algo = TriggerPrimitive::Algorithm::kAbsRunningSum;
    a.algorithm = SWTPG_ALGO_ABS_RS;
    m_enable_simple_threshold_on_collection = config.enable_simple_threshold_on_collection;
  } else if (config.tpg_algorithm == "StandardRS") {
    m_tp_algo = TriggerPrimitive::Algorithm::kRunningSum;
    a.algorithm = SWTPG_ALGO_STANDARD_RS;
    m_enable_simple_threshold_on_collection = config.enable_simple_threshold_on_collection;
  } else {
    throw TPGAlgorithmInexistent(config.tpg_algorithm);
  }
  // Running-sum factors travel as integers x10 (src/wibeth/WIBEthFrameProcessor.cpp:199-206)
  m_tpg_rs_memory_factor = uint16_t(10 * config.tpg_rs_memory_factor);
  a.rs_memory_factor = m_tpg_rs_memory_factor;
  a.rs_scale_factor = config.tpg_rs_scale_factor != 0 ? uint16_t(10 / config.tpg_rs_scale_factor) : 0;
  a.frugal_acc_limit = config.tpg_frugal_streaming_accumulator_limit;
  a.threshold = config.tpg_threshold;
  m_correct_lookup = config.correct_channel_lookup;
  inherited::reset_tasks();
  inherited::add_preprocess_task([this](frameptr fp) { sequence_check(fp); });
  inherited::add_preprocess_task([this](frameptr fp) { timestamp_check(fp); });
  conf_link(config, a, [this](constframeptr fp) { find_hits(fp, m_frame_handler.get()); });
}

void
WIBEthFrameProcessor::start()
{
  TpcFrameProcessor::start();
  m_seq_id_error_ctr = 0;
}

void
WIBEthFrameProcessor::get_info(RawDataProcessorInfo& info)
{
  TpcFrameProcessor::get_info(info);
  info.num_seq_id_errors = m_seq_id_error_ctr.load();
  info.min_seq_id_jump = m_seq_id_min_jump.exchange(0);
  info.max_seq_id_jump = m_seq_id_max_jump.exchange(0);
}

void
WIBEthFrameProcessor::sequence_check(frameptr fp)
{
  if (inherited::m_emulator_mode) { // emulated data: stamp the geo id and a perfectly incrementing sequence id
    DAQEthHeader* h = fp->header();
    h->crate_id = m_crate_no;
    h->slot_id = m_slot_no;
    h->stream_id = m_link_no;
    h->seq_id = m_previous_seq_id & 0xfff; // one frame per payload: (previous + i) with i = 0, as in the reference (:311)
  }
  m_current_seq_id = uint16_t(fp->header()->seq_id);
  const uint16_t expected_seq_id = uint16_t((m_previous_seq_id + fp->get_num_frames()) & 0xfff);
  int16_t delta_seq_id = int16_t(m_current_seq_id - expected_seq_id);
  if (delta_seq_id > 0x800)
    delta_seq_id -= 0x1000;
  else if (delta_seq_id < -0x7ff)
    delta_seq_id += 0x1000;
  if (delta_seq_id != 0) {
    ++m_seq_id_error_ctr;
    m_seq_id_max_jump = std::max(delta_seq_id, m_seq_id_max_jump.load());
    m_seq_id_min_jump = std::min(delta_seq_id, m_seq_id_min_jump.load());
    m_error_registry->add_error("SEQUENCE_ID_JUMP", FrameErrorRegistry::ErrorInterval{ expected_seq_id, m_current_seq_id });
  }
  m_previous_seq_id = m_current_seq_id;
}

void
WIBEthFrameProcessor::timestamp_check(frameptr fp)
{
  const uint64_t frame_tick_difference = DUNEWIBEthTypeAdapter::expected_tick_difference * fp->get_num_frames();
  if (inherited::m_emulator_mode) {
    DAQEthHeader* h = fp->header();
    h->crate_id = m_crate_no;
    h->slot_id = m_slot_no;
    h->stream_id = m_link_no;
    h->timestamp = m_previous_ts + frame_tick_difference;
  }
  m_current_ts = fp->get_first_timestamp();
  if (m_current_ts - m_previous_ts != frame_tick_difference) {
    ++m_ts_error_ctr;
    m_error_registry->add_error("MISSING_FRAMES", FrameErrorRegistry::ErrorInterval{ m_previous_ts + frame_tick_difference, m_current_ts });
  }
  m_previous_ts = m_current_ts;
  m_last_processed_daq_ts = m_current_ts;
}

void
WIBEthFrameProcessor::find_hits(constframeptr fp, WIBEthFrameHandler* frame_handler)
{
  if (!fp)
    return;
  const DAQEthHeader* hdr = fp->header();
  if (frame_handler->first_hit) {
    // Register-position -> offline channel map, built from the first frame's geo id (RegisterToChannelNumber.cpp:35-122):
    // position p of the expanded registers holds frame channel 16(p/16) + perm[p%16].
    for (uint32_t p = 0; p < 64; ++p)
      frame_handler->register_channel_map[p] = m_channel_map(hdr->crate_id, hdr->slot_id, hdr->stream_id, position_to_frame_channel(p));
    m_det_id = uint32_t(hdr->det_id);
    if (hdr->crate_id != m_crate_no || hdr->slot_id != m_slot_no || hdr->stream_id != m_link_no)
      m_misconf.push_back({ uint32_t(hdr->crate_id), uint32_t(hdr->slot_id), uint32_t(hdr->stream_id), m_crate_no, m_slot_no, m_link_no });
    // H2 (SURVEY.md): production indexes the POSITION-ordered map with the FRAME channel the AVX2 code emits (:527)
    set_channel_tables([&](uint32_t c) {
      return m_correct_lookup ? m_channel_map(hdr->crate_id, hdr->slot_id, hdr->stream_id, c) : frame_handler->register_channel_map[c];
    });
    if (m_enable_simple_threshold_on_collection) { // collection channels run with R = 0, i.e. a plain threshold (:441-450)
      uint16_t factor[64];
      for (uint32_t c = 0; c < 64; ++c) {
        const uint32_t offline = m_channel_map(hdr->crate_id, hdr->slot_id, hdr->stream_id, c);
        factor[c] = get_plane_from_offline_channel(offline) == 0 ? uint16_t(0) : m_tpg_rs_memory_factor;
      }
      m_engine->set_link_memory_factor(frame_handler->link, factor, 64);
    }
    frame_handler->first_hit = false;
  }
  submit(fp, frame_handler->link);
}

// ---- WIB2FrameProcessor ---------------------------------------------------------------------------------------------
void
WIB2FrameProcessor::conf(const RawDataProcessorConf& config)
{
  swtpg_config a{};
  if (config.tpg_algorithm == "SimpleThreshold")
    a.algorithm = SWTPG_ALGO_SIMPLE_THRESHOLD;
  else if (config.tpg_algorithm == "AbsRS") // src/wib2/WIB2FrameProcessor.cpp:388-392
    a.algorithm = SWTPG_ALGO_ABS_RS;
  else if (config.tpg_algorithm == "FIR") // the FIR + IQR finder the reference ships in wib2/tpg/ProcessAVX2FIR.hpp
    a.algorithm = SWTPG_ALGO_FIR_IQR;
  else
    throw TPGAlgorithmInexistent(config.tpg_algorithm);
  // FIR + IQR and AbsRS multiply the threshold by an IQR sigma
  if (config.enable_tpg && has_plane_thresholds(config) && a.algorithm != SWTPG_ALGO_SIMPLE_THRESHOLD)
    throw std::invalid_argument("tpg_plane_threshold: WIB2 supports per-plane thresholds with SimpleThreshold only");
  a.threshold = config.tpg_threshold;
  a.frugal_acc_limit = 10;
  inherited::reset_tasks();
  inherited::add_preprocess_task([this](frameptr fp) { timestamp_check(fp); });
  conf_link(config, a, [this](constframeptr fp) { find_hits(fp, m_frame_handler.get()); });
}

void
WIB2FrameProcessor::timestamp_check(frameptr fp)
{
  const uint64_t tick = DUNEWIBSuperChunkTypeAdapter::expected_tick_difference;
  const uint64_t superchunk_tick_difference = tick * fp->get_num_frames();
  if (inherited::m_emulator_mode) {
    uint64_t ts_next = m_previous_ts + superchunk_tick_difference;
    for (size_t i = 0; i < fp->get_num_frames(); ++i) {
      WIB2Header* h = fp->header(i);
      h->crate = m_crate_no;
      h->slot = m_slot_no;
      h->link = m_link_no;
      fp->set_timestamp(i, ts_next);
      ts_next += tick;
    }
  }
  m_current_ts = fp->get_first_timestamp();
  if (m_current_ts - m_previous_ts != superchunk_tick_difference) {
    ++m_ts_error_ctr;
    m_error_registry->add_error("MISSING_FRAMES", FrameErrorRegistry::ErrorInterval{ m_previous_ts + superchunk_tick_difference, m_current_ts });
  }
  m_previous_ts = m_current_ts;
  m_last_processed_daq_ts = m_current_ts;
}

void
WIB2FrameProcessor::find_hits(constframeptr fp, WIB2FrameHandler* frame_handler)
{
  if (!fp)
    return;
  if (frame_handler->first_hit) {
    const WIB2Header* h = fp->header();
    m_det_id = h->detector_id;
    // WIB2's AVX2 code emits the register POSITION and the map is position-ordered (src/wib2/WIB2FrameProcessor.cpp:367-368),
    // so the reported channel is the true offline channel of the frame channel: a frame-channel-ordered map is equivalent.
    set_channel_tables([&](uint32_t c) { return m_channel_map(h->crate, h->slot, h->link, c); });
    frame_handler->first_hit = false;
  }
  submit(fp, frame_handler->link);
}

// ---- TPCTPRequestHandler ----------------------------------------------------------------------------------------------
void
TPCTPRequestHandler::conf(const ReadoutModelConf& c)
{
  m_source_id = c.source_id;
  m_tp_set_sender_sleep_us = int(1000000 / std::max<uint32_t>(1, c.tpset_transmission_rate_hz));
  m_ts_set_sender_offset_ticks = c.tpset_min_latency_ticks;
  m_tardy_tp_quiet_time_at_start_sec = c.tardy_tp_quiet_time_at_start_sec;
}

void
TPCTPRequestHandler::start(uint32_t run_number)
{
  m_new_tps = 0;
  m_new_tpsets = 0;
  m_new_tps_in_tpsets_send_failed = 0;
  m_new_tpsets_send_failed = 0;
  m_new_tps_suppressed_tardy = 0;
  m_new_heartbeats = 0;
  m_latency_buffer.clear();
  m_run_number = run_number;
  m_cutoff_timestamp.store(0);
  m_first_cycle = true;
  m_start_win_ts = 0;
  m_next_tpset_seqno = 0;
  m_run_start_timepoint = std::chrono::high_resolution_clock::now();
}

void
TPCTPRequestHandler::stop()
{
  m_cutoff_timestamp.store(0);
}

void
TPCTPRequestHandler::get_info(TPRequestHandlerInfo& info)
{
  info.num_tps_sent = m_new_tps.exchange(0);
  info.num_tpsets_sent = m_new_tpsets.exchange(0);
  info.num_tps_in_tpsets_send_failed = m_new_tps_in_tpsets_send_failed.exchange(0);
  info.num_tpsets_send_failed = m_new_tpsets_send_failed.exchange(0);
  info.num_tps_suppressed_tardy = m_new_tps_suppressed_tardy.exchange(0);
  info.num_heartbeats = m_new_heartbeats.exchange(0);
}

void
TPCTPRequestHandler::report_tardy_packet(const TriggerPrimitiveTypeAdapter&, int64_t)
{
  ++m_new_tps_suppressed_tardy;
  const auto now = std::chrono::high_resolution_clock::now();
  if (std::chrono::duration_cast<std::chrono::seconds>(now - m_run_start_timepoint).count() > m_tardy_tp_quiet_time_at_start_sec)
    ++m_late_warnings; // reference: ers::warning(DataPacketArrivedTooLate), muted during the quiet time after start (:88-96)
}

bool
TPCTPRequestHandler::receive(TriggerPrimitiveTypeAdapter&& tp)
{
  const uint64_t cutoff = get_cutoff_timestamp();
  if (tp.get_first_timestamp() < cutoff) {
    report_tardy_packet(tp, int64_t(cutoff - tp.get_first_timestamp()));
    return false;
  }
  m_latency_buffer.insert(std::move(tp));
  return true;
}

void
TPCTPRequestHandler::pop_older_than(uint64_t ts)
{
  while (!m_latency_buffer.empty() && m_latency_buffer.begin()->get_first_timestamp() < ts)
    m_latency_buffer.erase(m_latency_buffer.begin());
}

bool
TPCTPRequestHandler::send_tp_sets_once()
{
  if (m_latency_buffer.empty())
    return false;
  const uint64_t newest_ts = m_latency_buffer.rbegin()->get_first_timestamp();
  const uint64_t oldest_ts = m_latency_buffer.begin()->get_first_timestamp();
  if (m_first_cycle) {
    m_start_win_ts = oldest_ts;
    m_first_cycle = false;
  }
  if (!(newest_ts - m_start_win_ts > m_ts_set_sender_offset_ticks))
    return false;
  const uint64_t end_win_ts = newest_ts - m_ts_set_sender_offset_ticks;
  // get_fragment_pieces(start, end): every element with start <= time_start < end, in (time_start, channel) order
  TPSet tpset;
  TriggerPrimitiveTypeAdapter lo;
  lo.tp.time_start = m_start_win_ts;
  lo.tp.channel = 0;
  for (auto it = m_latency_buffer.lower_bound(lo); it != m_latency_buffer.end() && it->get_first_timestamp() < end_win_ts; ++it)
    tpset.objects.push_back(it->tp);
  const size_t num_tps = tpset.objects.size();
  tpset.run_number = m_run_number;
  tpset.type = num_tps > 0 ? TPSet::Type::kPayload : TPSet::Type::kHeartbeat;
  tpset.origin = m_source_id;
  tpset.start_time = num_tps ? tpset.objects.front().time_start : m_start_win_ts;
  tpset.end_time = num_tps ? tpset.objects.back().time_start : end_win_ts;
  tpset.seqno = m_next_tpset_seqno++;
  m_cutoff_timestamp.store(tpset.end_time);
  if (!m_tpset_sink || !m_tpset_sink(std::move(tpset))) {
    m_new_tps_in_tpsets_send_failed += num_tps; // reference: ers::warning(FailedToSendTPSet)
    ++m_new_tpsets_send_failed;
  } else {
    m_new_tps += num_tps;
    ++m_new_tpsets;
  }
  if (num_tps == 0)
    m_new_heartbeats++;
  m_start_win_ts = end_win_ts; // remember what we sent for the next loop
  return true;
}

} // namespace host
} // namespace swtpg

// =====================================================================================================================
// C test harness (tests/test_host_shim.py drives the classes above through ctypes): one engine + n frame processors with
// in-memory "tp_out" queues. Not part of the drop-in surface.
// =====================================================================================================================
using namespace swtpg::host;

struct swtpg_host_conf
{
  int32_t device, format; // swtpg_format
  uint32_t n_links, superchunk_units;
  char tpg_algorithm[32];
  float tpg_rs_memory_factor, tpg_rs_scale_factor;
  uint16_t tpg_threshold;
  int16_t tpg_frugal_streaming_accumulator_limit;
  uint64_t tp_timeout;
  uint32_t channel_mask[16];
  uint32_t n_mask;
  uint16_t crate_id, slot_id, first_link_id;
  uint8_t enable_tpg, emulator_mode, correct_channel_lookup, reversed_map, enable_simple_threshold_on_collection, block_on_backpressure;
  uint8_t count_only_sink; // 1: tp_out only counts what it accepts (throughput runs: no queue growth)
  uint8_t n_slots;         // staging depth of the engine in superchunks (0 = 4)
  uint32_t sink_capacity; // per link; try_send fails beyond it (0 = unbounded)
};

// The TPG fields of one link's RawDataProcessorConf, overriding those of swtpg_host_conf (swtpg_host_create with links).
struct swtpg_host_link_conf
{
  char tpg_algorithm[32];
  float tpg_rs_memory_factor, tpg_rs_scale_factor;
  uint16_t tpg_threshold;
  int16_t tpg_frugal_streaming_accumulator_limit;
  int32_t tpg_plane_threshold[3]; // -1 = tpg_threshold
};

struct swtpg_host_tp
{
  uint64_t time_start, time_peak, time_over_threshold;
  uint32_t channel, adc_integral;
  uint16_t adc_peak, detid;
  uint32_t type, algorithm;
  uint16_t version, flag;
};

using WIBEthProcessors = std::vector<std::unique_ptr<WIBEthFrameProcessor>>;
using WIB2Processors = std::vector<std::unique_ptr<WIB2FrameProcessor>>;

struct swtpg_host
{
  std::shared_ptr<TpgEngine> engine;
  std::vector<std::unique_ptr<FrameErrorRegistry>> regs;
  std::variant<WIBEthProcessors, WIB2Processors> procs; // one processor per link, all of the engine's format
  std::vector<std::vector<TriggerPrimitiveTypeAdapter>> queues;
  std::vector<std::unique_ptr<std::mutex>> qmu;
  uint32_t sink_capacity = 0;
  bool count_only = false;
  std::atomic<uint64_t> accepted{ 0 };
  std::string error;
};

static thread_local std::string g_host_error;

// f(processors) with the handle's processor vector: the format is resolved once per C call, not once per payload.
template<class F>
static decltype(auto)
with_processors(swtpg_host* h, F&& f)
{
  return std::visit(std::forward<F>(f), h->procs);
}

// Payload `index` of an array of P's frames through the consumer path of processor p: the pre-process tasks (may rewrite the
// header in emulator mode — the buffer is the caller's, as the latency buffer element is in the reference), then the
// post-process task.
template<class P>
static void
push_payload(P& p, void* payloads, size_t index)
{
  auto* fp = static_cast<typename P::frameptr>(payloads) + index;
  p.preprocess_item(fp);
  p.postprocess_item(fp);
}

extern "C" {

const char*
swtpg_host_last_error(void)
{
  return g_host_error.c_str();
}

// links: NULL, or links[n_links], each frame processor's conf() with its own TPG fields (one engine, links with different
// configurations). flags: SWTPG_FLAG_* for the engine's handle (SWTPG_FLAG_ADC_STATS: the processors' get_adc_stats;
// SWTPG_FLAG_NOISE_SPECTRA: their get_noise_spectra; SWTPG_FLAG_CHANNEL_COVARIANCE: their get_channel_covariance).
swtpg_host*
swtpg_host_create(const swtpg_host_conf* c, const swtpg_host_link_conf* links, uint32_t flags)
{
  try {
    auto h = std::make_unique<swtpg_host>();
    h->engine = std::make_shared<TpgEngine>(c->device, swtpg_format(c->format), c->n_links, c->superchunk_units, c->n_slots ? c->n_slots : 4u,
                                            0u, flags);
    h->sink_capacity = c->sink_capacity;
    h->count_only = c->count_only_sink != 0;
    h->queues.resize(c->n_links);
    h->regs.resize(c->n_links); // the processors keep REFERENCES to these unique_ptrs (as the reference's model does): no reallocation later
    if (c->format != SWTPG_FORMAT_WIBETH)
      h->procs.emplace<WIB2Processors>();
    for (uint32_t l = 0; l < c->n_links; ++l) {
      h->qmu.push_back(std::make_unique<std::mutex>());
      h->regs[l] = std::make_unique<FrameErrorRegistry>();
      RawDataProcessorConf rc;
      rc.tpg_algorithm = c->tpg_algorithm;
      rc.tpg_threshold = c->tpg_threshold;
      rc.tpg_rs_memory_factor = c->tpg_rs_memory_factor;
      rc.tpg_rs_scale_factor = c->tpg_rs_scale_factor;
      rc.tpg_frugal_streaming_accumulator_limit = c->tpg_frugal_streaming_accumulator_limit;
      rc.tp_timeout = c->tp_timeout;
      rc.tpg_channel_mask.assign(c->channel_mask, c->channel_mask + std::min<uint32_t>(c->n_mask, 16));
      rc.crate_id = c->crate_id;
      rc.slot_id = c->slot_id;
      rc.link_id = uint16_t(c->first_link_id + l);
      rc.enable_tpg = c->enable_tpg != 0;
      rc.emulator_mode = c->emulator_mode != 0;
      rc.correct_channel_lookup = c->correct_channel_lookup != 0;
      rc.channel_map_name = c->reversed_map ? "reversed" : "linear";
      rc.enable_simple_threshold_on_collection = c->enable_simple_threshold_on_collection != 0;
      rc.block_on_backpressure = c->block_on_backpressure != 0;
      if (links) {
        rc.tpg_algorithm = links[l].tpg_algorithm;
        rc.tpg_threshold = links[l].tpg_threshold;
        rc.tpg_rs_memory_factor = links[l].tpg_rs_memory_factor;
        rc.tpg_rs_scale_factor = links[l].tpg_rs_scale_factor;
        rc.tpg_frugal_streaming_accumulator_limit = links[l].tpg_frugal_streaming_accumulator_limit;
        std::copy(links[l].tpg_plane_threshold, links[l].tpg_plane_threshold + 3, rc.tpg_plane_threshold.begin());
      }
      swtpg_host* hp = h.get();
      auto sink = [hp, l](TriggerPrimitiveTypeAdapter&& tp) {
        if (hp->count_only) {
          hp->accepted.fetch_add(1, std::memory_order_relaxed);
          return true;
        }
        std::lock_guard<std::mutex> lk(*hp->qmu[l]);
        if (hp->sink_capacity && hp->queues[l].size() >= hp->sink_capacity)
          return false;
        hp->queues[l].push_back(std::move(tp));
        return true;
      };
      with_processors(hp, [&](auto& procs) {
        using P = typename std::decay_t<decltype(procs)>::value_type::element_type;
        procs.push_back(std::make_unique<P>(h->regs[l], h->engine));
        procs.back()->init(sink);
        procs.back()->conf(rc);
      });
    }
    return h.release();
  } catch (const TPGAlgorithmInexistent& e) {
    g_host_error = std::string("TPGAlgorithmInexistent: ") + e.what();
  } catch (const std::exception& e) {
    g_host_error = e.what();
  }
  return nullptr;
}

void
swtpg_host_destroy(swtpg_host* h)
{
  delete h;
}

int
swtpg_host_start(swtpg_host* h)
{
  try {
    with_processors(h, [](auto& procs) {
      for (auto& p : procs)
        p->start();
    });
    return 0;
  } catch (const std::exception& e) {
    g_host_error = e.what();
    return -1;
  }
}

int
swtpg_host_stop(swtpg_host* h)
{
  try {
    with_processors(h, [](auto& procs) {
      for (auto& p : procs)
        p->stop();
    });
    return 0;
  } catch (const std::exception& e) {
    g_host_error = e.what();
    return -1;
  }
}

// One payload of one link through the consumer path
int
swtpg_host_push(swtpg_host* h, uint32_t link, void* payload)
{
  try {
    with_processors(h, [&](auto& procs) { push_payload(*procs[link], payload, 0); });
    return 0;
  } catch (const std::exception& e) {
    g_host_error = e.what();
    return -1;
  }
}

// The reference's threading model: one consumer/post-processing thread per link, all running concurrently. Each thread pushes
// its link's n_units payloads (payloads: [n_links][n_units][unit_bytes], modified in place by the pre-process tasks).
int
swtpg_host_push_parallel(swtpg_host* h, void* payloads, uint32_t n_units)
{
  const size_t n_links = h->queues.size();
  std::vector<std::string> errors(n_links);
  with_processors(h, [&](auto& procs) {
    std::vector<std::thread> threads;
    for (size_t l = 0; l < n_links; ++l)
      threads.emplace_back([=, &errors, &procs]() {
        try {
          for (uint32_t u = 0; u < n_units; ++u)
            push_payload(*procs[l], payloads, l * n_units + u);
        } catch (const std::exception& e) {
          errors[l] = e.what();
        }
      });
    for (auto& t : threads)
      t.join();
  });
  for (auto& e : errors)
    if (!e.empty()) {
      g_host_error = e;
      return -1;
    }
  return 0;
}

// A readout host the way it is built: a FEW consumer threads, each serving many links. Thread t owns links t, t + T, ...; it
// walks them round-robin, `burst` consecutive payloads per link and turn, each through the pre-process tasks (sequence /
// timestamp checks) and the post-process task (find_hits). pace > 0 runs against the clock: payload g of every link is due
// g * period / pace after the start (period = one payload's worth of detector time: 2048 ticks of 16 ns for a WIBEth frame,
// 12 x 32 ticks for a WIB2 superchunk), a burst is pushed when its last payload is due, and the thread SLEEPS until then —
// so the CPU time it reports is the work, not the waiting. `passes` walks over the same payload array again (emulator mode
// keeps the timestamps running). Fills wall seconds and the feeder threads' summed CPU seconds.
struct swtpg_host_feed_stats
{
  double wall_s, feeder_cpu_s;
  uint64_t payloads, late_bursts;
};

int
swtpg_host_push_feeders(swtpg_host* h, void* payloads, uint32_t n_units, uint32_t n_threads, uint32_t burst, double pace, uint32_t passes,
                        swtpg_host_feed_stats* out)
{
  const size_t n_links = h->queues.size();
  const double period_s = (std::holds_alternative<WIBEthProcessors>(h->procs) ? 2048.0 : 12.0 * 32.0) / 62.5e6;
  n_threads = std::max<uint32_t>(1, std::min<uint32_t>(n_threads, uint32_t(n_links)));
  burst = std::max<uint32_t>(1, std::min(burst, n_units));
  std::vector<std::string> errors(n_threads);
  std::vector<double> cpu(n_threads, 0.0);
  std::vector<uint64_t> late(n_threads, 0);
  const auto t_start = std::chrono::steady_clock::now() + std::chrono::milliseconds(2);
  with_processors(h, [&](auto& procs) {
    std::vector<std::thread> threads;
    for (uint32_t t = 0; t < n_threads; ++t)
      threads.emplace_back([=, &errors, &cpu, &late, &procs]() {
        try {
          for (uint32_t pass = 0; pass < passes; ++pass)
            for (uint32_t u0 = 0; u0 < n_units; u0 += burst) {
              const uint32_t u1 = std::min(n_units, u0 + burst);
              if (pace > 0) {
                const double due_s = (double(pass) * n_units + u1) * period_s / pace;
                const auto due = t_start + std::chrono::duration_cast<std::chrono::steady_clock::duration>(std::chrono::duration<double>(due_s));
                if (std::chrono::steady_clock::now() < due)
                  std::this_thread::sleep_until(due);
                else
                  ++late[t];
              }
              for (size_t l = t; l < n_links; l += n_threads)
                for (uint32_t u = u0; u < u1; ++u)
                  push_payload(*procs[l], payloads, l * n_units + u);
            }
          timespec ts{};
          clock_gettime(CLOCK_THREAD_CPUTIME_ID, &ts);
          cpu[t] = double(ts.tv_sec) + 1e-9 * double(ts.tv_nsec);
        } catch (const std::exception& e) {
          errors[t] = e.what();
        }
      });
    for (auto& th : threads)
      th.join();
  });
  const double wall = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
  for (auto& e : errors)
    if (!e.empty()) {
      g_host_error = e;
      return -1;
    }
  if (out) {
    out->wall_s = wall;
    out->feeder_cpu_s = 0;
    out->late_bursts = 0;
    for (uint32_t t = 0; t < n_threads; ++t) {
      out->feeder_cpu_s += cpu[t];
      out->late_bursts += late[t];
    }
    out->payloads = uint64_t(passes) * n_units * n_links;
  }
  return 0;
}

// the engine's swtpg_counters (units by address / by copy, batches, bytes)
int
swtpg_host_counters(swtpg_host* h, swtpg_counters* out)
{
  return h->engine->handle() && swtpg_get_counters(h->engine->handle(), out) == SWTPG_OK ? 0 : -1;
}

// device time of the streaming path's gather and TPG kernels (swtpg_stream_timing)
int
swtpg_host_stream_timing(swtpg_host* h, double* gather_ms, double* kernel_ms, uint64_t* batches)
{
  return h->engine->handle() && swtpg_stream_timing(h->engine->handle(), gather_ms, kernel_ms, batches) == SWTPG_OK ? 0 : -1;
}

// TPs accepted by the count-only sinks so far
uint64_t
swtpg_host_tp_count(swtpg_host* h)
{
  return h->accepted.load();
}

size_t
swtpg_host_take_tps(swtpg_host* h, uint32_t link, swtpg_host_tp* out, size_t cap)
{
  std::lock_guard<std::mutex> lk(*h->qmu[link]);
  auto& q = h->queues[link];
  const size_t n = std::min(cap, q.size());
  for (size_t i = 0; i < n; ++i) {
    const TriggerPrimitive& t = q[i].tp;
    out[i] = { t.time_start, t.time_peak, t.time_over_threshold, t.channel, t.adc_integral, t.adc_peak, t.detid, uint32_t(t.type),
               uint32_t(t.algorithm), t.version, t.flag };
  }
  q.erase(q.begin(), q.begin() + long(n));
  return n;
}

void
swtpg_host_get_info(swtpg_host* h, uint32_t link, RawDataProcessorInfo* info)
{
  with_processors(h, [&](auto& procs) { procs[link]->get_info(*info); });
}

uint64_t
swtpg_host_error_count(swtpg_host* h, uint32_t link, const char* name)
{
  std::lock_guard<std::mutex> lk(h->regs[link]->mu);
  auto it = h->regs[link]->counts.find(name);
  return it == h->regs[link]->counts.end() ? 0 : it->second;
}

uint32_t
swtpg_host_misconfigurations(swtpg_host* h, uint32_t link)
{
  const auto* eth = std::get_if<WIBEthProcessors>(&h->procs);
  return eth ? uint32_t((*eth)[link]->misconfigurations().size()) : 0u;
}

uint64_t
swtpg_host_last_daq_time(swtpg_host* h, uint32_t link)
{
  return with_processors(h, [&](auto& procs) { return procs[link]->get_last_daq_time(); });
}

// Zero-copy ingest: register / unregister the array the pushed payloads live in (the "latency buffer")
int
swtpg_host_register_buffer(swtpg_host* h, void* base, size_t bytes, int on)
{
  try {
    if (on)
      h->engine->register_latency_buffer(base, bytes);
    else
      h->engine->unregister_latency_buffer(base);
  } catch (const std::exception& e) {
    g_host_error = e.what();
    return -1;
  }
  return 0;
}

// ChannelAdcStats of a link's processor: out[cap] (64 WIBEth / 256 WIB2 entries, none before the first frame); the entry count, -1 on error
static_assert(sizeof(ChannelAdcStats) == 40, "hostshim.HOST_ADC_STATS_DTYPE mirrors ChannelAdcStats");
int
swtpg_host_adc_stats(swtpg_host* h, uint32_t link, int reset, ChannelAdcStats* out, uint32_t cap)
{
  try {
    std::vector<ChannelAdcStats> v;
    with_processors(h, [&](auto& procs) { procs.at(link)->get_adc_stats(v, reset != 0); });
    const size_t n = std::min<size_t>(v.size(), cap);
    std::copy(v.begin(), v.begin() + n, out);
    return int(n);
  } catch (const std::exception& e) {
    g_host_error = e.what();
    return -1;
  }
}

// ChannelNoiseSpectrum of a link's processor: out[cap] (64 WIBEth / 256 WIB2 entries, none before the first frame); the entry count, -1 on error
static_assert(sizeof(ChannelNoiseSpectrum) == 280, "hostshim.HOST_NOISE_SPECTRUM_DTYPE mirrors ChannelNoiseSpectrum");
int
swtpg_host_noise_spectra(swtpg_host* h, uint32_t link, int reset, ChannelNoiseSpectrum* out, uint32_t cap)
{
  try {
    std::vector<ChannelNoiseSpectrum> v;
    with_processors(h, [&](auto& procs) { procs.at(link)->get_noise_spectra(v, reset != 0); });
    const size_t n = std::min<size_t>(v.size(), cap);
    std::copy(v.begin(), v.begin() + n, out);
    return int(n);
  } catch (const std::exception& e) {
    g_host_error = e.what();
    return -1;
  }
}

// ChannelCovariance of a link's processor into samples, offline[cap] and covariance / correlation [cap][cap] (either may be NULL):
// the channel count (64 WIBEth / 256 WIB2, 0 before the first frame), -1 on error or when cap is too small
int
swtpg_host_channel_covariance(swtpg_host* h, uint32_t link, int reset, uint64_t* samples, uint32_t* offline, double* covariance,
                              double* correlation, uint32_t cap)
{
  try {
    ChannelCovariance v;
    with_processors(h, [&](auto& procs) { procs.at(link)->get_channel_covariance(v, reset != 0); });
    const size_t n = v.offline_channel.size();
    if (n > cap)
      throw std::invalid_argument("swtpg_host_channel_covariance: cap is below the link's channel count");
    if (samples)
      *samples = v.samples;
    if (offline)
      std::copy(v.offline_channel.begin(), v.offline_channel.end(), offline);
    if (covariance)
      std::copy(v.covariance.begin(), v.covariance.end(), covariance);
    if (correlation)
      std::copy(v.correlation.begin(), v.correlation.end(), correlation);
    return int(n);
  } catch (const std::exception& e) {
    g_host_error = e.what();
    return -1;
  }
}

// position -> offline channel map of a link (after its first frame)
void
swtpg_host_register_channel_map(swtpg_host* h, uint32_t link, uint32_t* out64)
{
  if (const auto* eth = std::get_if<WIBEthProcessors>(&h->procs))
    for (int p = 0; p < 64; ++p)
      out64[p] = (*eth)[link]->handler()->register_channel_map[size_t(p)];
}

// ---- TPCTPRequestHandler harness ---------------------------------------------------------------------------------------------
struct swtpg_host_tpsets
{
  TPCTPRequestHandler handler;
  std::vector<TPSet> sent;
  uint32_t sink_capacity = 0;
};
struct swtpg_host_tpset_hdr
{
  uint64_t seqno, start_time, end_time;
  uint32_t run_number, origin, type, n_objects;
};

swtpg_host_tpsets*
swtpg_host_tpsets_create(uint32_t source_id, uint32_t rate_hz, uint64_t min_latency_ticks, uint32_t run_number, uint32_t sink_capacity)
{
  auto* h = new swtpg_host_tpsets;
  h->sink_capacity = sink_capacity;
  h->handler.init([h](TPSet&& s) {
    if (h->sink_capacity && h->sent.size() >= h->sink_capacity)
      return false;
    h->sent.push_back(std::move(s));
    return true;
  });
  ReadoutModelConf c;
  c.source_id = source_id;
  c.tpset_transmission_rate_hz = rate_hz;
  c.tpset_min_latency_ticks = min_latency_ticks;
  h->handler.conf(c);
  h->handler.start(run_number);
  return h;
}

void
swtpg_host_tpsets_destroy(swtpg_host_tpsets* h)
{
  delete h;
}

// feeds n harness TP records (e.g. taken from a frame processor's tp_out); returns how many were accepted (not tardy)
size_t
swtpg_host_tpsets_receive(swtpg_host_tpsets* h, const swtpg_host_tp* tps, size_t n)
{
  size_t ok = 0;
  for (size_t i = 0; i < n; ++i) {
    TriggerPrimitiveTypeAdapter a;
    a.tp.time_start = tps[i].time_start;
    a.tp.time_peak = tps[i].time_peak;
    a.tp.time_over_threshold = tps[i].time_over_threshold;
    a.tp.channel = tps[i].channel;
    a.tp.adc_integral = tps[i].adc_integral;
    a.tp.adc_peak = tps[i].adc_peak;
    a.tp.detid = tps[i].detid;
    a.tp.type = TriggerPrimitive::Type(tps[i].type);
    a.tp.algorithm = TriggerPrimitive::Algorithm(tps[i].algorithm);
    ok += h->handler.receive(std::move(a)) ? 1 : 0;
  }
  return ok;
}

int
swtpg_host_tpsets_cycle(swtpg_host_tpsets* h)
{
  return h->handler.send_tp_sets_once() ? 1 : 0;
}

uint64_t
swtpg_host_tpsets_cutoff(swtpg_host_tpsets* h)
{
  return h->handler.get_cutoff_timestamp();
}

size_t
swtpg_host_tpsets_count(swtpg_host_tpsets* h)
{
  return h->sent.size();
}

// header of sent TPSet i and (if objs != NULL) its first `cap` objects
int
swtpg_host_tpsets_get(swtpg_host_tpsets* h, size_t i, swtpg_host_tpset_hdr* hdr, swtpg_host_tp* objs, size_t cap)
{
  if (i >= h->sent.size())
    return -1;
  const TPSet& s = h->sent[i];
  *hdr = { s.seqno, s.start_time, s.end_time, s.run_number, s.origin, uint32_t(s.type), uint32_t(s.objects.size()) };
  for (size_t k = 0; objs && k < std::min(cap, s.objects.size()); ++k) {
    const TriggerPrimitive& t = s.objects[k];
    objs[k] = { t.time_start, t.time_peak, t.time_over_threshold, t.channel, t.adc_integral, t.adc_peak, t.detid, uint32_t(t.type),
                uint32_t(t.algorithm), t.version, t.flag };
  }
  return 0;
}

void
swtpg_host_tpsets_info(swtpg_host_tpsets* h, TPRequestHandlerInfo* info)
{
  h->handler.get_info(*info);
}

} // extern "C"
