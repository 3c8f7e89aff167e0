// Streaming path behind include/swtpg.h (swtpg_submit / swtpg_submit_wait / swtpg_register_buffer / swtpg_flush / swtpg_poll /
// swtpg_poll_wait): what a readout application's per-link post-processing threads drive, one payload at a time.
//
//   producers (one thread per link at a time, lock-free)      dispatcher thread                 completion thread
//   ----------------------------------------------------      -----------------                 -----------------
//   swtpg_submit: append the unit's DEVICE-VISIBLE address     when a link has a full            waits (sleeping) for a batch's
//   to the link's ring — the payload itself if it lies in      superchunk / time-out / flush:    gather -> frees the ring space,
//   a registered latency buffer (zero-copy), else its copy     take what every link has,         wakes blocked producers;
//   in the link's pinned staging ring — and bump `head`.       build the pointer table,          waits for the TP count -> copies
//                                                              enqueue gather + TPG kernel       the TPs out -> ready queue
//
// There is no all-links barrier: batches are ragged (0 .. max_units units per link), so a slow or dead link never holds the
// others back, and flush is just "dispatch now" — safe against concurrent submits because the dispatcher only ever takes
// whole units below a `head` it has read with acquire semantics.
//
// The host-to-device transfer is ONE kernel per batch (gather_units_tma): SM-issued copies read every unit where it lies in
// pinned, mapped host memory through a per-unit pointer table and lay the batch out link-major in HBM for the fused TPG
// kernel. No per-link cudaMemcpyAsync calls (round 1 issued one per link and run), no staging pass for registered buffers.
#include "swtpg_handle.h"

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <thread>

extern "C" void swtpg_stage_copy(void* dst, const void* src, size_t bytes); // swtpg_hostutil.cpp

namespace swtpg_internal {

// ---- gather kernels ---------------------------------------------------------------------------------------------------
struct GatherItem
{
  const uint8_t* src; // device-visible address of the unit in pinned host memory (16-byte aligned)
  uint64_t dst_off;   // byte offset inside the batch's link-major device buffer
};

__device__ __forceinline__ uint32_t
g_smem_u32(const void* p)
{
  return uint32_t(__cvta_generic_to_shared(p));
}

// TMA form: one thread per CTA runs a ring of STAGES bulk copies host -> shared memory (mbarrier complete_tx) and forwards
// every landed unit with a bulk copy shared memory -> HBM. STAGES - 1 units (7200 B each) are in flight per CTA, which is what
// covers the host link's latency; nothing but the one thread's bookkeeping is ever issued on the SM.
template<int STAGES>
__global__ void __launch_bounds__(32)
gather_units_tma(const GatherItem* __restrict__ items, uint32_t n, uint8_t* __restrict__ dst, uint32_t bytes)
{
  extern __shared__ __align__(128) uint8_t g_smem[];
  uint64_t* bar = reinterpret_cast<uint64_t*>(g_smem + size_t(STAGES) * bytes);
  if (threadIdx.x != 0)
    return;
#pragma unroll
  for (int s = 0; s < STAGES; ++s)
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(g_smem_u32(&bar[s])));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  const uint32_t first = blockIdx.x, step = gridDim.x;
  const uint32_t mine = first < n ? (n - first + step - 1) / step : 0;
  auto load = [&](uint32_t k) { // k-th unit of this CTA
    const uint32_t s = k % STAGES;
    const uint8_t* src = items[first + k * step].src;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(g_smem_u32(&bar[s])), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(g_smem_u32(g_smem + size_t(s) * bytes)),
                 "l"(src), "r"(bytes), "r"(g_smem_u32(&bar[s]))
                 : "memory");
  };
  for (uint32_t k = 0; k < mine && k < STAGES - 1; ++k)
    load(k);
  for (uint32_t k = 0; k < mine; ++k) {
    const uint32_t s = k % STAGES, parity = (k / STAGES) & 1u;
    asm volatile("{\n.reg .pred p;\nGW_%=:\nmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n@p bra GD_%=;\nbra GW_%=;\nGD_%=:\n}" ::"r"(
                   g_smem_u32(&bar[s])),
                 "r"(parity), "r"(100000u)
                 : "memory");
    const uint64_t off = items[first + k * step].dst_off;
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst + off), "r"(g_smem_u32(g_smem + size_t(s) * bytes)), "r"(bytes)
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); // the store of unit k-1 has read its stage: refill that one
    if (k + STAGES - 1 < mine)
      load(k + STAGES - 1);
  }
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ---- engine -----------------------------------------------------------------------------------------------------------
using Clock = std::chrono::steady_clock;

struct alignas(64) LinkQ
{
  // written by the link's producer thread
  std::atomic<uint64_t> head{ 0 }; // units delivered
  uint32_t slot = 0;               // head % ring_units
  uint64_t range_epoch = 0;        // cached registered range of this link's payloads (a link's payloads come from one latency buffer)
  uintptr_t range_lo = 0, range_hi = 0;
  intptr_t range_delta = 0;        // device-visible address = host address + delta
  uintptr_t gap_lo = 0, gap_hi = 0; // cached MISS: the unregistered gap between ranges the link's last staged payload lay in
  uint64_t n_zero_copy = 0, n_staged = 0; // units of this link submitted by address / by copy (summed by swtpg_get_counters)
  // written by the engine's threads
  alignas(64) std::atomic<uint64_t> tail{ 0 }; // units whose gather has completed: their ring slots are free again
  std::atomic<uint64_t> dispatched{ 0 };       // units handed to a batch
  uint32_t dslot = 0;                          // dispatched % ring_units
};

struct Batch
{
  uint8_t* d_frames = nullptr; // [n_links][max_units][unit_bytes]
  swtpg_tp* d_tps = nullptr;
  swtpg_tp* h_tps = nullptr;   // pinned
  unsigned* d_count = nullptr;
  unsigned* h_count = nullptr; // pinned
  uint32_t* h_nunits = nullptr; // pinned [n_links]
  uint32_t* d_nunits = nullptr;
  GatherItem* h_items = nullptr; // pinned [n_links * max_units]
  GatherItem* d_items = nullptr;
  uint32_t n_items = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev_gather = nullptr, ev_kernel = nullptr, ev_count = nullptr, ev_tps = nullptr;
  cudaEvent_t ev_up = nullptr;                  // pointer table and lengths are on the device (the gather stream waits for it)
  cudaEvent_t ev_g0 = nullptr, ev_k0 = nullptr; // timing: start of the gather / of the TPG kernel (device clocks, swtpg_stream_timing)
  cudaEvent_t ev_stats = nullptr;               // the statistics kernel has read d_frames (swtpg_handle::channel_stats only)
  uint32_t n_ready = 0, n_taken = 0;
  bool overflow = false;
  bool released = false; // the release thread has handed the batch's ring slots back (guarded by StreamEngine::mu)
};

struct StreamEngine
{
  swtpg_handle* h = nullptr;
  uint32_t n_links = 0, M = 0, R = 0, unit_bytes = 0;
  std::unique_ptr<LinkQ[]> links;
  std::unique_ptr<const uint8_t*[]> ring_ptr; // [n_links][R]: device-visible address of every pending unit
  std::atomic<uint8_t*> stage{ nullptr };     // pinned, mapped [n_links][R][unit_bytes]; allocated by the first staged submit
  uint8_t* stage_dev = nullptr;
  std::mutex stage_mu;

  struct Range
  {
    uintptr_t lo, hi;
    intptr_t delta;
    bool ours; // this handle pinned it (cudaHostRegister) and unpins it again
  };
  std::vector<Range> ranges;
  std::mutex ranges_mu;
  std::atomic<uint64_t> ranges_epoch{ 0 };

  std::vector<std::unique_ptr<Batch>> batches;
  std::mutex mu; // queues, requests, condition variables below
  std::condition_variable cv_dispatch, cv_complete, cv_release, cv_ready, cv_space, cv_flush;
  std::deque<Batch*> free_q, inflight_q, release_q, ready_q;
  uint32_t building = 0; // batches taken from free_q that have not reached inflight_q yet
  std::atomic<bool> kicked{ false };
  std::atomic<uint32_t> space_waiters{ 0 };
  uint64_t flush_req = 0, flush_done = 0;
  bool reset_req = false, stalled_on_poll = false, quit = false;
  std::atomic<int> thread_status{ SWTPG_OK };
  std::atomic<uint64_t> gather_us{ 0 }, kernel_us{ 0 }, timed_batches{ 0 };
  std::thread dispatcher, releaser, completer;
  std::mutex poll_mu; // one poller at a time
  std::chrono::microseconds timeout{ 5000 };

  cudaStream_t gather_stream = nullptr; // the gathers of all batches run one after the other on this stream

  void kick()
  {
    if (!kicked.exchange(true, std::memory_order_acq_rel)) {
      std::lock_guard<std::mutex> lk(mu);
      cv_dispatch.notify_one();
    }
  }
  void thread_fail(const char* what, cudaError_t e)
  {
    char buf[256];
    snprintf(buf, sizeof buf, "streaming engine: %s failed: %s", what, cudaGetErrorString(e));
    h->set_error(buf);
    thread_status.store(SWTPG_ERR_CUDA);
    std::lock_guard<std::mutex> lk(mu);
    cv_ready.notify_all();
    cv_flush.notify_all();
    cv_space.notify_all();
  }
  cudaError_t launch_gather(Batch& b);
  cudaError_t enqueue(Batch& b);
  void dispatcher_main();
  void releaser_main();
  void completer_main();
};

namespace {

constexpr int kGatherStages = 8;
constexpr unsigned kGatherCtas = 64;

void
free_batch(Batch& b)
{
  if (b.d_frames) cudaFree(b.d_frames);
  if (b.d_tps) cudaFree(b.d_tps);
  if (b.h_tps) cudaFreeHost(b.h_tps);
  if (b.d_count) cudaFree(b.d_count);
  if (b.h_count) cudaFreeHost(b.h_count);
  if (b.h_nunits) cudaFreeHost(b.h_nunits);
  if (b.d_nunits) cudaFree(b.d_nunits);
  if (b.h_items) cudaFreeHost(b.h_items);
  if (b.d_items) cudaFree(b.d_items);
  if (b.ev_gather) cudaEventDestroy(b.ev_gather);
  if (b.ev_kernel) cudaEventDestroy(b.ev_kernel);
  if (b.ev_g0) cudaEventDestroy(b.ev_g0);
  if (b.ev_up) cudaEventDestroy(b.ev_up);
  if (b.ev_k0) cudaEventDestroy(b.ev_k0);
  if (b.ev_count) cudaEventDestroy(b.ev_count);
  if (b.ev_tps) cudaEventDestroy(b.ev_tps);
  if (b.ev_stats) cudaEventDestroy(b.ev_stats);
  if (b.stream) cudaStreamDestroy(b.stream);
}

} // namespace

cudaError_t
StreamEngine::launch_gather(Batch& b)
{
  if (b.n_items == 0)
    return cudaSuccess;
  const unsigned grid = std::min<unsigned>(kGatherCtas, b.n_items);
  const size_t smem = size_t(kGatherStages) * unit_bytes + kGatherStages * 8;
  gather_units_tma<kGatherStages><<<grid, 32, smem, gather_stream>>>(b.d_items, b.n_items, b.d_frames, unit_bytes);
  return cudaGetLastError();
}

// Everything a batch needs on the device, in order: pointer table + ragged lengths up on the batch's own stream, gather on the
// engine's gather stream (behind the previous batch's gather, overlapping its TPG kernel), TPG kernel on the handle's compute stream (state is carried: kernels of
// consecutive batches must run in order), TP count back on the batch's stream.
cudaError_t
StreamEngine::enqueue(Batch& b)
{
  cudaError_t e;
#define TRY(x)                                                                                                                    \
  if ((e = (x)) != cudaSuccess)                                                                                                   \
  return e
  TRY(cudaMemcpyAsync(b.d_items, b.h_items, size_t(b.n_items) * sizeof(GatherItem), cudaMemcpyHostToDevice, b.stream));
  TRY(cudaMemcpyAsync(b.d_nunits, b.h_nunits, size_t(n_links) * 4, cudaMemcpyHostToDevice, b.stream));
  TRY(cudaEventRecord(b.ev_up, b.stream));
  TRY(cudaStreamWaitEvent(gather_stream, b.ev_up, 0));
  TRY(cudaEventRecord(b.ev_g0, gather_stream));
  TRY(launch_gather(b));
  TRY(cudaEventRecord(b.ev_gather, gather_stream));
  TRY(cudaStreamWaitEvent(b.stream, b.ev_gather, 0));
  TRY(cudaMemsetAsync(b.d_count, 0, sizeof(unsigned), b.stream));
  TRY(cudaStreamWaitEvent(h->stream, b.ev_gather, 0));
  TRY(cudaEventRecord(b.ev_k0, h->stream));
  TRY(launch_batch_kernel(h, b.d_frames, b.d_nunits, M, b.d_tps, b.d_count, h->stream));
  TRY(cudaEventRecord(b.ev_kernel, h->stream));
  if (h->channel_stats()) { // after ev_kernel (stream timing is the TPG kernel's alone), and before ev_count: the batch is not reused earlier
    TRY(launch_channel_stats(h, b.d_frames, b.d_nunits, M, h->stream));
    TRY(cudaEventRecord(b.ev_stats, h->stream));
  }
  TRY(cudaStreamWaitEvent(b.stream, h->channel_stats() ? b.ev_stats : b.ev_kernel, 0));
  TRY(cudaMemcpyAsync(b.h_count, b.d_count, sizeof(unsigned), cudaMemcpyDeviceToHost, b.stream));
  TRY(cudaEventRecord(b.ev_count, b.stream));
#undef TRY
  return cudaSuccess;
}

void
StreamEngine::dispatcher_main()
{
  cudaSetDevice(h->cfg.device);
  std::unique_lock<std::mutex> lk(mu);
  bool have_pending_since = false;
  Clock::time_point pending_since{};
  for (;;) {
    cv_dispatch.wait_for(lk, timeout, [&] { return quit || reset_req || kicked.load(std::memory_order_acquire) || flush_req > flush_done; });
    if (quit)
      return;
    kicked.store(false, std::memory_order_release);
    if (reset_req) { // swtpg_start: nothing is in flight (the caller quiesced first) and nobody submits
      cv_ready.wait(lk, [&] { return quit || (inflight_q.empty() && building == 0); });
      if (quit)
        return;
      while (!ready_q.empty()) { // undelivered TPs of the previous run are dropped with it
        free_q.push_back(ready_q.front());
        ready_q.pop_front();
      }
      for (uint32_t l = 0; l < n_links; ++l) {
        LinkQ& q = links[l];
        q.head.store(0);
        q.tail.store(0);
        q.dispatched.store(0);
        q.slot = q.dslot = 0;
        q.n_zero_copy = q.n_staged = 0;
      }
      have_pending_since = false;
      gather_us = kernel_us = timed_batches = 0;
      reset_req = false;
      cv_flush.notify_all();
      continue;
    }
    const uint64_t ticket = flush_req;
    const bool flushing = ticket > flush_done;
    lk.unlock();
    for (;;) { // one batch per turn while there is a reason to dispatch
      uint64_t total = 0;
      bool any_full = false;
      for (uint32_t l = 0; l < n_links; ++l) {
        const uint64_t avail = links[l].head.load(std::memory_order_acquire) - links[l].dispatched.load(std::memory_order_relaxed);
        any_full |= avail >= M;
        total += std::min<uint64_t>(avail, M);
      }
      if (total == 0) {
        have_pending_since = false;
        break;
      }
      const Clock::time_point now = Clock::now();
      if (!have_pending_since) {
        have_pending_since = true;
        pending_since = now;
      }
      if (!(any_full || flushing || now - pending_since >= timeout))
        break;
      lk.lock();
      while (free_q.empty() && !quit) {
        stalled_on_poll = inflight_q.empty() && building == 0; // every batch holds TPs nobody has polled: only swtpg_poll helps
        if (stalled_on_poll)
          cv_flush.notify_all();
        cv_dispatch.wait(lk);
      }
      stalled_on_poll = false;
      if (quit)
        return;
      Batch* b = free_q.front();
      free_q.pop_front();
      ++building;
      lk.unlock();
      // take what every link has NOW (more may have arrived while waiting for a batch)
      uint32_t n = 0;
      for (uint32_t l = 0; l < n_links; ++l) {
        LinkQ& q = links[l];
        const uint64_t done = q.dispatched.load(std::memory_order_relaxed);
        const uint32_t take = uint32_t(std::min<uint64_t>(q.head.load(std::memory_order_acquire) - done, M));
        b->h_nunits[l] = take;
        const uint8_t* const* ring = ring_ptr.get() + size_t(l) * R;
        uint32_t s = q.dslot;
        const uint64_t row = uint64_t(l) * M * unit_bytes;
        for (uint32_t u = 0; u < take; ++u) {
          b->h_items[n++] = GatherItem{ ring[s], row + uint64_t(u) * unit_bytes };
          s = s + 1 == R ? 0 : s + 1;
        }
        q.dslot = s;
        if (take)
          q.dispatched.store(done + take, std::memory_order_release);
      }
      b->n_items = n;
      b->n_ready = b->n_taken = 0;
      b->overflow = false;
      const cudaError_t e = enqueue(*b);
      if (e != cudaSuccess)
        thread_fail("batch dispatch", e);
      h->counters.units_processed += n;
      h->counters.samples_processed += uint64_t(n) * h->channels * h->ticks;
      h->counters.h2d_bytes += uint64_t(n) * unit_bytes;
      h->counters.batches++;
      have_pending_since = false;
      lk.lock();
      --building;
      b->released = false;
      inflight_q.push_back(b);
      release_q.push_back(b);
      cv_complete.notify_one();
      cv_release.notify_one();
      lk.unlock();
      if (e != cudaSuccess)
        break;
    }
    lk.lock();
    if (flushing) {
      flush_done = std::max(flush_done, ticket);
      cv_flush.notify_all();
    }
  }
}

// Ring space comes back the moment a batch's gather has finished — the frames are in HBM, so the units' ring slots (and the
// borrow of zero-copy units) end there — independently of how long the TPG kernel and the TP read-back of earlier batches
// take: its own thread, asleep in cudaEventSynchronize in between.
void
StreamEngine::releaser_main()
{
  cudaSetDevice(h->cfg.device);
  std::unique_lock<std::mutex> lk(mu);
  for (;;) {
    cv_release.wait(lk, [&] { return quit || !release_q.empty(); });
    if (release_q.empty())
      return; // quit
    Batch* b = release_q.front();
    release_q.pop_front();
    lk.unlock();
    const cudaError_t e = cudaEventSynchronize(b->ev_gather);
    for (uint32_t l = 0; l < n_links; ++l)
      if (b->h_nunits[l])
        links[l].tail.fetch_add(b->h_nunits[l], std::memory_order_release);
    if (e != cudaSuccess)
      thread_fail("gather", e);
    lk.lock();
    b->released = true;
    cv_complete.notify_all();
    if (space_waiters.load(std::memory_order_acquire) != 0)
      cv_space.notify_all();
  }
}

void
StreamEngine::completer_main()
{
  cudaSetDevice(h->cfg.device);
  std::unique_lock<std::mutex> lk(mu);
  for (;;) {
    cv_complete.wait(lk, [&] { return quit || !inflight_q.empty(); });
    if (inflight_q.empty())
      return; // quit
    Batch* b = inflight_q.front(); // stays at the front until it is complete (swtpg_sync waits for the queue to empty)
    lk.unlock();
    cudaError_t e = cudaEventSynchronize(b->ev_count);
    if (e == cudaSuccess) {
      const unsigned found = *b->h_count;
      const unsigned stored = std::min<unsigned>(found, h->tp_capacity);
      const swtpg_tp* src = b->d_tps;
      bool finish_on_host = false;
      std::unique_lock<std::mutex> sorter_lock;
      if (h->sorter && stored > 1 &&
          sort_tps_device(h, h->sorter, b->d_tps, stored, b->stream, &src, &finish_on_host, &sorter_lock) != SWTPG_OK)
        e = cudaErrorUnknown; // the text is in the handle's last error already
      if (stored && e == cudaSuccess)
        e = cudaMemcpyAsync(b->h_tps, src, size_t(stored) * sizeof(swtpg_tp), cudaMemcpyDeviceToHost, b->stream);
      if (e == cudaSuccess)
        e = cudaEventRecord(b->ev_tps, b->stream);
      if (e == cudaSuccess)
        e = cudaEventSynchronize(b->ev_tps);
      if (sorter_lock.owns_lock())
        sorter_lock.unlock();
      if (finish_on_host && e == cudaSuccess)
        swtpg_sort_tps(b->h_tps, stored);
      b->n_ready = stored;
      b->overflow = found > stored;
      float g_ms = 0.f, k_ms = 0.f; // device time the gather and the TPG kernel of this batch took (both have completed)
      if (cudaEventElapsedTime(&g_ms, b->ev_g0, b->ev_gather) == cudaSuccess && cudaEventElapsedTime(&k_ms, b->ev_k0, b->ev_kernel) == cudaSuccess) {
        gather_us.fetch_add(uint64_t(g_ms * 1000.f), std::memory_order_relaxed);
        kernel_us.fetch_add(uint64_t(k_ms * 1000.f), std::memory_order_relaxed);
        timed_batches.fetch_add(1, std::memory_order_relaxed);
      } else {
        cudaGetLastError();
      }
      h->counters.tps_emitted += found;
      h->counters.d2h_bytes += uint64_t(stored) * sizeof(swtpg_tp) + sizeof(unsigned);
      if (found > stored)
        h->counters.tps_dropped_overflow += found - stored;
    }
    if (e != cudaSuccess)
      thread_fail("batch completion", e);
    lk.lock();
    cv_complete.wait(lk, [&] { return b->released || quit; }); // its ring slots are back (the release thread reads h_nunits)
    inflight_q.pop_front();
    ready_q.push_back(b);
    cv_ready.notify_all();
    cv_dispatch.notify_all(); // a dispatcher waiting for a free batch re-evaluates "only swtpg_poll can help now"
    if (quit && inflight_q.empty())
      return;
  }
}

namespace {

swtpg_status
engine_create(swtpg_handle* h, StreamEngine** out)
{
  std::lock_guard<std::mutex> lk(h->engine_mu);
  if (StreamEngine* e = h->engine.load(std::memory_order_acquire)) {
    *out = e;
    return SWTPG_OK;
  }
  SW_CUDA(h, cudaSetDevice(h->cfg.device));
  std::unique_ptr<StreamEngine> e(new StreamEngine);
  e->h = h;
  e->n_links = h->cfg.n_links;
  e->M = h->cfg.max_units;
  e->R = h->cfg.n_slots * h->cfg.max_units;
  e->unit_bytes = h->unit_bytes;
  e->timeout = std::chrono::microseconds(h->cfg.dispatch_timeout_us ? h->cfg.dispatch_timeout_us : 5000u);
  e->links.reset(new LinkQ[e->n_links]);
  e->ring_ptr.reset(new const uint8_t*[size_t(e->n_links) * e->R]());
  // One gather stream for all batches: their gathers run one after the other. Side by side (each on its batch's stream) they
  // share the host link worse than they use it one at a time: 45.4-46.8 against 48.2-48.8 GB/s at 240 links with 3-6 slots
  // (profiles/r02_gather_serial_probe.txt).
  SW_CUDA(h, cudaStreamCreateWithFlags(&e->gather_stream, cudaStreamNonBlocking));
  const size_t smem = size_t(kGatherStages) * e->unit_bytes + kGatherStages * 8;
  SW_CUDA(h, cudaFuncSetAttribute(gather_units_tma<kGatherStages>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  const size_t fbytes = size_t(e->n_links) * e->M * e->unit_bytes;
  const size_t n_items = size_t(e->n_links) * e->M;
  auto cleanup = [&]() {
    for (auto& b : e->batches)
      free_batch(*b);
    cudaStreamDestroy(e->gather_stream);
  };
  for (uint32_t i = 0; i < h->cfg.n_slots; ++i) {
    e->batches.emplace_back(new Batch);
    Batch& b = *e->batches.back();
    cudaError_t ce = cudaSuccess;
    auto ok = [&](cudaError_t x) { return ce == cudaSuccess ? (ce = x) == cudaSuccess : false; };
    ok(cudaMalloc(&b.d_frames, fbytes));
    ok(cudaMalloc(&b.d_tps, size_t(h->tp_capacity) * sizeof(swtpg_tp)));
    ok(cudaMallocHost(&b.h_tps, size_t(h->tp_capacity) * sizeof(swtpg_tp)));
    ok(cudaMalloc(&b.d_count, sizeof(unsigned)));
    ok(cudaMallocHost(&b.h_count, sizeof(unsigned)));
    ok(cudaMallocHost(&b.h_nunits, size_t(e->n_links) * 4));
    ok(cudaMalloc(&b.d_nunits, size_t(e->n_links) * 4));
    ok(cudaMallocHost(&b.h_items, n_items * sizeof(GatherItem)));
    ok(cudaMalloc(&b.d_items, n_items * sizeof(GatherItem)));
    ok(cudaStreamCreateWithFlags(&b.stream, cudaStreamNonBlocking));
    // blocking-sync events: the completion thread sleeps in cudaEventSynchronize instead of spinning on a core
    ok(cudaEventCreateWithFlags(&b.ev_gather, cudaEventBlockingSync));
    ok(cudaEventCreateWithFlags(&b.ev_kernel, cudaEventDefault));
    ok(cudaEventCreate(&b.ev_g0));
    ok(cudaEventCreateWithFlags(&b.ev_up, cudaEventDisableTiming));
    ok(cudaEventCreate(&b.ev_k0));
    ok(cudaEventCreateWithFlags(&b.ev_count, cudaEventDisableTiming | cudaEventBlockingSync));
    ok(cudaEventCreateWithFlags(&b.ev_tps, cudaEventDisableTiming | cudaEventBlockingSync));
    if (h->channel_stats())
      ok(cudaEventCreateWithFlags(&b.ev_stats, cudaEventDisableTiming));
    if (ce != cudaSuccess) {
      cleanup();
      SW_CUDA(h, ce);
    }
    e->free_q.push_back(&b);
  }
  StreamEngine* ep = e.release();
  ep->dispatcher = std::thread([ep] { ep->dispatcher_main(); });
  ep->releaser = std::thread([ep] { ep->releaser_main(); });
  ep->completer = std::thread([ep] { ep->completer_main(); });
  h->engine.store(ep, std::memory_order_release);
  *out = ep;
  return SWTPG_OK;
}

// Pinned, mapped staging ring for units that do not lie in a registered buffer; allocated by the first such submit.
swtpg_status
ensure_stage(swtpg_handle* h, StreamEngine* e)
{
  std::lock_guard<std::mutex> lk(e->stage_mu);
  if (e->stage.load(std::memory_order_acquire))
    return SWTPG_OK;
  SW_CUDA(h, cudaSetDevice(h->cfg.device));
  uint8_t* p = nullptr;
  SW_CUDA(h, cudaHostAlloc(&p, size_t(e->n_links) * e->R * e->unit_bytes, cudaHostAllocMapped | cudaHostAllocPortable));
  uint8_t* d = nullptr;
  SW_CUDA(h, cudaHostGetDevicePointer(&d, p, 0));
  e->stage_dev = d;
  e->stage.store(p, std::memory_order_release);
  return SWTPG_OK;
}

// Device-visible address of [unit, unit + bytes) if it lies inside a registered range and is 16-byte aligned (the bulk copy's
// requirement), else nullptr. Lock-free on the hot path: the link keeps the last range it hit.
inline const uint8_t*
registered_address(StreamEngine* e, LinkQ& q, const void* unit, size_t bytes)
{
  const uint64_t epoch = e->ranges_epoch.load(std::memory_order_acquire);
  if (epoch == 0)
    return nullptr; // nothing was ever registered
  const uintptr_t a = reinterpret_cast<uintptr_t>(unit);
  if (a & 15u)
    return nullptr;
  if (q.range_epoch == epoch) {
    if (a >= q.range_lo && a + bytes <= q.range_hi)
      return reinterpret_cast<const uint8_t*>(a + uintptr_t(q.range_delta));
    if (a >= q.gap_lo && a + bytes <= q.gap_hi)
      return nullptr; // cached miss: inside the same unregistered gap as the link's last staged payload
  }
  // first payload of the link, or the set of ranges changed, or the payload lies somewhere else than the last one
  std::lock_guard<std::mutex> lk(e->ranges_mu);
  q.range_epoch = e->ranges_epoch.load(std::memory_order_relaxed);
  uintptr_t below = 0, above = ~uintptr_t(0);
  for (const auto& r : e->ranges) {
    if (a >= r.lo && a + bytes <= r.hi) {
      q.range_lo = r.lo;
      q.range_hi = r.hi;
      q.range_delta = r.delta;
      return reinterpret_cast<const uint8_t*>(a + uintptr_t(r.delta));
    }
    if (r.hi <= a)
      below = std::max(below, r.hi);
    else if (r.lo >= a + bytes)
      above = std::min(above, r.lo);
    else { // straddles a range boundary: staged, and not cached
      below = a;
      above = a;
    }
  }
  q.gap_lo = below;
  q.gap_hi = above;
  return nullptr;
}

swtpg_status
submit_impl(swtpg_handle* h, uint32_t link, const void* unit, size_t bytes, uint64_t timeout_us)
{
  if (!h || !unit)
    return SWTPG_ERR_INVALID_ARG;
  if (!h->started.load(std::memory_order_acquire))
    return fail(h, SWTPG_ERR_STATE, "swtpg_start has not been called");
  if (link >= h->cfg.n_links || bytes != h->unit_bytes)
    return fail(h, SWTPG_ERR_INVALID_ARG, "bad link index or unit size");
  StreamEngine* e = h->engine.load(std::memory_order_acquire);
  if (!e) {
    const swtpg_status s = engine_create(h, &e);
    if (s != SWTPG_OK)
      return s;
  }
  if (e->thread_status.load(std::memory_order_relaxed) != SWTPG_OK)
    return swtpg_status(e->thread_status.load());
  LinkQ& q = e->links[link];
  const uint64_t head = q.head.load(std::memory_order_relaxed); // one producer thread per link
  if (head - q.tail.load(std::memory_order_acquire) >= e->R) {
    bool room = false;
    if (timeout_us) { // sleep until the completion thread has freed ring space (or the time is up)
      e->kick();      // whatever is pending has to go out for that to happen
      std::unique_lock<std::mutex> lk(e->mu);
      e->space_waiters.fetch_add(1, std::memory_order_acq_rel);
      room = e->cv_space.wait_for(lk, std::chrono::microseconds(timeout_us), [&] {
        return head - q.tail.load(std::memory_order_acquire) < e->R || e->quit || e->thread_status.load() != SWTPG_OK;
      });
      e->space_waiters.fetch_sub(1, std::memory_order_acq_rel);
      room = room && head - q.tail.load(std::memory_order_acquire) < e->R;
    }
    if (!room) {
      h->counters.submit_busy.fetch_add(1, std::memory_order_relaxed);
      return SWTPG_ERR_BUSY; // ring full: the caller drops or retries, like a failed try_send
    }
  }
  const size_t idx = size_t(link) * e->R + q.slot;
  const uint8_t* dev = registered_address(e, q, unit, bytes);
  if (!dev) { // not in a registered latency buffer: the payload is only borrowed for this call, so it is copied
    uint8_t* st = e->stage.load(std::memory_order_acquire);
    if (!st) {
      const swtpg_status s = ensure_stage(h, e);
      if (s != SWTPG_OK)
        return s;
      st = e->stage.load(std::memory_order_acquire);
    }
    swtpg_stage_copy(st + idx * e->unit_bytes, unit, bytes);
    dev = e->stage_dev + idx * e->unit_bytes;
    ++q.n_staged;
  } else {
    ++q.n_zero_copy;
  }
  e->ring_ptr[idx] = dev;
  q.slot = q.slot + 1 == e->R ? 0 : q.slot + 1;
  q.head.store(head + 1, std::memory_order_release);
  if (head + 1 - q.dispatched.load(std::memory_order_relaxed) >= e->M && !e->kicked.load(std::memory_order_relaxed))
    e->kick(); // this link has a full superchunk: wake the dispatcher (once; it takes every link's pending units)
  return SWTPG_OK;
}

swtpg_status
poll_impl(swtpg_handle* h, swtpg_tp* out, size_t cap, size_t* n_out, uint64_t timeout_us)
{
  if (n_out)
    *n_out = 0;
  if (!h || (!out && cap))
    return SWTPG_ERR_INVALID_ARG;
  StreamEngine* e = h->engine.load(std::memory_order_acquire);
  if (!e)
    return SWTPG_OK;
  std::lock_guard<std::mutex> pl(e->poll_mu);
  std::unique_lock<std::mutex> lk(e->mu);
  if (timeout_us && e->ready_q.empty())
    e->cv_ready.wait_for(lk, std::chrono::microseconds(timeout_us), [&] { return !e->ready_q.empty() || e->quit || e->thread_status.load() != SWTPG_OK; });
  size_t n = 0;
  swtpg_status ret = SWTPG_OK;
  while (!e->ready_q.empty()) {
    Batch* b = e->ready_q.front(); // only this (serialised) function pops the queue, so `b` stays valid without the lock
    lk.unlock();
    const uint32_t take = uint32_t(std::min<size_t>(cap - n, b->n_ready - b->n_taken));
    if (take)
      memcpy(out + n, b->h_tps + b->n_taken, size_t(take) * sizeof(swtpg_tp));
    n += take;
    b->n_taken += take;
    if (b->overflow) {
      b->overflow = false;
      ret = fail(h, SWTPG_ERR_OVERFLOW, "device TP buffer overflow: raise swtpg_config.tp_capacity");
    }
    lk.lock();
    if (b->n_taken < b->n_ready)
      break; // caller's buffer is full; the rest comes with the next poll
    e->ready_q.pop_front();
    e->free_q.push_back(b);
    e->cv_dispatch.notify_one(); // the dispatcher may be waiting for a free batch
  }
  lk.unlock();
  if (n_out)
    *n_out = n;
  if (ret == SWTPG_OK && e->thread_status.load() != SWTPG_OK)
    ret = swtpg_status(e->thread_status.load());
  return ret;
}

} // namespace

void
engine_destroy(swtpg_handle* h)
{
  StreamEngine* e = h->engine.exchange(nullptr);
  if (!e)
    return;
  {
    std::lock_guard<std::mutex> lk(e->mu);
    e->quit = true;
    e->cv_dispatch.notify_all();
    e->cv_complete.notify_all();
    e->cv_release.notify_all();
    e->cv_ready.notify_all();
    e->cv_space.notify_all();
    e->cv_flush.notify_all();
  }
  if (e->dispatcher.joinable())
    e->dispatcher.join();
  if (e->releaser.joinable())
    e->releaser.join();
  if (e->completer.joinable())
    e->completer.join();
  cudaDeviceSynchronize();
  for (auto& b : e->batches)
    free_batch(*b);
  if (uint8_t* st = e->stage.load())
    cudaFreeHost(st);
  for (const auto& r : e->ranges)
    if (r.ours && cudaHostUnregister(reinterpret_cast<void*>(r.lo)) != cudaSuccess)
      cudaGetLastError();
  cudaStreamDestroy(e->gather_stream);
  delete e;
}

swtpg_status
engine_quiesce(swtpg_handle* h)
{
  StreamEngine* e = h->engine.load(std::memory_order_acquire);
  if (!e)
    return SWTPG_OK;
  std::unique_lock<std::mutex> lk(e->mu);
  e->cv_ready.wait(lk, [&] { return (e->inflight_q.empty() && e->building == 0) || e->quit || e->thread_status.load() != SWTPG_OK; });
  return swtpg_status(e->thread_status.load());
}

swtpg_status
engine_reset(swtpg_handle* h)
{
  StreamEngine* e = h->engine.load(std::memory_order_acquire);
  if (!e)
    return SWTPG_OK;
  std::unique_lock<std::mutex> lk(e->mu);
  e->reset_req = true;
  e->cv_dispatch.notify_all();
  e->cv_flush.wait(lk, [&] { return !e->reset_req || e->quit; });
  return SWTPG_OK;
}

} // namespace swtpg_internal

using namespace swtpg_internal;

extern "C" {

swtpg_status
swtpg_submit(swtpg_handle* h, uint32_t link, const void* unit, size_t bytes)
{
  return submit_impl(h, link, unit, bytes, 0);
}

swtpg_status
swtpg_submit_wait(swtpg_handle* h, uint32_t link, const void* unit, size_t bytes, uint64_t timeout_us)
{
  return submit_impl(h, link, unit, bytes, timeout_us);
}

swtpg_status
swtpg_register_buffer(swtpg_handle* h, void* base, size_t bytes)
{
  if (!h || !base || bytes == 0)
    return SWTPG_ERR_INVALID_ARG;
  StreamEngine* e = h->engine.load(std::memory_order_acquire);
  if (!e) {
    const swtpg_status s = engine_create(h, &e);
    if (s != SWTPG_OK)
      return s;
  }
  SW_CUDA(h, cudaSetDevice(h->cfg.device));
  bool ours = true;
  cudaError_t ce = cudaHostRegister(base, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped);
  if (ce != cudaSuccess) {
    // already page-locked — by another handle (two GPUs sharing one latency buffer: "already registered") or by
    // cudaHostAlloc / swtpg_alloc_pinned ("invalid value")? Then it only has to be looked up, not pinned again.
    cudaGetLastError();
    cudaPointerAttributes attr{};
    if (cudaPointerGetAttributes(&attr, base) != cudaSuccess || attr.type != cudaMemoryTypeHost) {
      cudaGetLastError();
      SW_CUDA(h, ce);
    }
    ours = false;
  }
  void* dev = nullptr;
  ce = cudaHostGetDevicePointer(&dev, base, 0);
  if (ce != cudaSuccess) {
    if (ours)
      cudaHostUnregister(base);
    SW_CUDA(h, ce);
  }
  std::lock_guard<std::mutex> lk(e->ranges_mu);
  const uintptr_t lo = reinterpret_cast<uintptr_t>(base);
  e->ranges.push_back({ lo, lo + bytes, intptr_t(reinterpret_cast<uintptr_t>(dev)) - intptr_t(lo), ours });
  e->ranges_epoch.fetch_add(1, std::memory_order_release);
  return SWTPG_OK;
}

swtpg_status
swtpg_unregister_buffer(swtpg_handle* h, void* base)
{
  if (!h || !base)
    return SWTPG_ERR_INVALID_ARG;
  StreamEngine* e = h->engine.load(std::memory_order_acquire);
  if (!e)
    return fail(h, SWTPG_ERR_INVALID_ARG, "buffer was not registered with this handle");
  const uintptr_t lo = reinterpret_cast<uintptr_t>(base);
  {
    std::lock_guard<std::mutex> lk(e->ranges_mu);
    if (std::find_if(e->ranges.begin(), e->ranges.end(), [lo](const StreamEngine::Range& r) { return r.lo == lo; }) == e->ranges.end())
      return fail(h, SWTPG_ERR_INVALID_ARG, "buffer was not registered with this handle");
  }
  // no gather may still have to read from it: dispatch what is pending, then wait for the device
  if (h->started.load()) {
    const swtpg_status fs = swtpg_flush(h);
    if (fs != SWTPG_OK)
      return fs;
  }
  swtpg_status st = swtpg_sync(h);
  if (st != SWTPG_OK)
    return st;
  bool ours = false;
  {
    std::lock_guard<std::mutex> lk(e->ranges_mu);
    auto it = std::find_if(e->ranges.begin(), e->ranges.end(), [lo](const StreamEngine::Range& r) { return r.lo == lo; });
    if (it == e->ranges.end())
      return fail(h, SWTPG_ERR_INVALID_ARG, "buffer was not registered with this handle");
    ours = it->ours;
    e->ranges.erase(it);
    e->ranges_epoch.fetch_add(1, std::memory_order_release);
  }
  if (ours && cudaHostUnregister(base) != cudaSuccess)
    cudaGetLastError(); // already gone
  return SWTPG_OK;
}

swtpg_status
swtpg_flush(swtpg_handle* h)
{
  if (!h)
    return SWTPG_ERR_INVALID_ARG;
  if (!h->started.load())
    return fail(h, SWTPG_ERR_STATE, "swtpg_start has not been called");
  StreamEngine* e = h->engine.load(std::memory_order_acquire);
  if (!e)
    return SWTPG_OK;
  std::unique_lock<std::mutex> lk(e->mu);
  const uint64_t ticket = ++e->flush_req;
  e->cv_dispatch.notify_all();
  e->cv_flush.wait(lk, [&] { return e->flush_done >= ticket || e->stalled_on_poll || e->quit || e->thread_status.load() != SWTPG_OK; });
  if (e->thread_status.load() != SWTPG_OK)
    return swtpg_status(e->thread_status.load());
  if (e->flush_done < ticket)
    return fail(h, SWTPG_ERR_BUSY, "every batch holds TPs that have not been polled: swtpg_poll, then flush again");
  return SWTPG_OK;
}

swtpg_status
swtpg_poll(swtpg_handle* h, swtpg_tp* out, size_t cap, size_t* n_out)
{
  return poll_impl(h, out, cap, n_out, 0);
}

swtpg_status
swtpg_poll_wait(swtpg_handle* h, swtpg_tp* out, size_t cap, size_t* n_out, uint64_t timeout_us)
{
  return poll_impl(h, out, cap, n_out, timeout_us);
}

swtpg_status
swtpg_stream_timing(swtpg_handle* h, double* gather_ms, double* kernel_ms, uint64_t* batches)
{
  if (!h)
    return SWTPG_ERR_INVALID_ARG;
  double g = 0, k = 0;
  uint64_t n = 0;
  if (StreamEngine* e = h->engine.load(std::memory_order_acquire)) {
    g = double(e->gather_us.load()) * 1e-3;
    k = double(e->kernel_us.load()) * 1e-3;
    n = e->timed_batches.load();
  }
  if (gather_ms)
    *gather_ms = g;
  if (kernel_ms)
    *kernel_ms = k;
  if (batches)
    *batches = n;
  return SWTPG_OK;
}

// units submitted by address (zero-copy) and by staging copy since swtpg_start; used by swtpg_get_counters
void
swtpg_internal_ingest_counts(swtpg_handle* h, uint64_t* zero_copy, uint64_t* staged)
{
  *zero_copy = *staged = 0;
  if (StreamEngine* e = h->engine.load(std::memory_order_acquire))
    for (uint32_t l = 0; l < e->n_links; ++l) {
      *zero_copy += e->links[l].n_zero_copy;
      *staged += e->links[l].n_staged;
    }
}

swtpg_status
swtpg_stream_status(swtpg_handle* h, uint64_t* units_pending, uint32_t* batches_in_flight, uint32_t* batches_ready)
{
  if (!h)
    return SWTPG_ERR_INVALID_ARG;
  uint64_t pending = 0;
  uint32_t inflight = 0, ready = 0;
  if (StreamEngine* e = h->engine.load(std::memory_order_acquire)) {
    for (uint32_t l = 0; l < e->n_links; ++l)
      pending += e->links[l].head.load(std::memory_order_acquire) - e->links[l].dispatched.load(std::memory_order_acquire);
    std::lock_guard<std::mutex> lk(e->mu);
    inflight = uint32_t(e->inflight_q.size()) + e->building;
    ready = uint32_t(e->ready_q.size());
  }
  if (units_pending)
    *units_pending = pending;
  if (batches_in_flight)
    *batches_in_flight = inflight;
  if (batches_ready)
    *batches_ready = ready;
  return SWTPG_OK;
}

} // extern "C"
