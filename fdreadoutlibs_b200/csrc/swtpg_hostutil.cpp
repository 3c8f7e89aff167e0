// Host-only pieces of libswtpg_b200.so (plain g++; no CUDA): the staging copy of swtpg_submit, the FIR tap design, the
// host-side ordering / merge of TP lists, the noise power spectra of swtpg_noise_power and the covariance matrices of
// swtpg_channel_covariance.
#include "../../include/swtpg.h"

#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <cstring>
#include <limits>
#include <vector>

// ---- staging copy ------------------------------------------------------------------------------------------------------
// Copy of one payload (frame / superchunk) into the pinned staging slot of the streaming path (swtpg_submit).
// The destination is written once by the CPU and read once by the GPU's copy engine, so it should neither be pulled into the
// cache first (read-for-ownership) nor stay there: non-temporal stores. Plain C++ (g++), because nvcc's host front end does
// not accept the AVX intrinsics headers.
#if defined(__x86_64__)
#include <immintrin.h>

__attribute__((target("avx2"))) static void
stage_copy_avx2(char* d, const char* s, size_t bytes)
{
  size_t i = 0;
  for (; i + 128 <= bytes; i += 128) {
    const __m256i a = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(s + i));
    const __m256i b = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(s + i + 32));
    const __m256i c = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(s + i + 64));
    const __m256i e = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(s + i + 96));
    _mm256_stream_si256(reinterpret_cast<__m256i*>(d + i), a);
    _mm256_stream_si256(reinterpret_cast<__m256i*>(d + i + 32), b);
    _mm256_stream_si256(reinterpret_cast<__m256i*>(d + i + 64), c);
    _mm256_stream_si256(reinterpret_cast<__m256i*>(d + i + 96), e);
  }
  for (; i + 32 <= bytes; i += 32)
    _mm256_stream_si256(reinterpret_cast<__m256i*>(d + i), _mm256_loadu_si256(reinterpret_cast<const __m256i*>(s + i)));
  if (i < bytes)
    memcpy(d + i, s + i, bytes - i);
  _mm_sfence(); // the slot may be handed to the copy engine by another thread right after
}
#endif

extern "C" __attribute__((visibility("hidden"))) void
swtpg_stage_copy(void* dst, const void* src, size_t bytes)
{
#if defined(__x86_64__)
  static const bool avx2 = __builtin_cpu_supports("avx2");
  if (avx2 && (reinterpret_cast<uintptr_t>(dst) & 31u) == 0) {
    stage_copy_avx2(static_cast<char*>(dst), static_cast<const char*>(src), bytes);
    return;
  }
#endif
  memcpy(dst, src, bytes);
}

// ---- TP ordering ----------------------------------------------------------------------------------------------------------
static inline bool
tp_less(const swtpg_tp& a, const swtpg_tp& b)
{
  if (a.time_start != b.time_start) return a.time_start < b.time_start;
  if (a.link != b.link) return a.link < b.link;
  if (a.channel != b.channel) return a.channel < b.channel;
  if (a.time_over_threshold != b.time_over_threshold) return a.time_over_threshold < b.time_over_threshold;
  if (a.adc_integral != b.adc_integral) return a.adc_integral < b.adc_integral;
  // the remaining fields, so that the order is total: records that tie on everything above (only possible when a link delivers
  // the same timestamps twice) come out the same way whatever order the device emitted them in
  if (a.time_peak != b.time_peak) return a.time_peak < b.time_peak;
  return a.adc_peak < b.adc_peak;
}

// Host-side ordering of a batch's TP list. A 64-frame batch of 148 APAs carries ~0.5 M records: std::sort needs ~110 ms for
// them, more than the batch's whole host-to-device copy. The keys are narrow, though — time_start spans the batch (a few
// 10^5 ticks), link < n_links, channel < 256 — so (time_start - min, link, channel) packs into one 64-bit integer, and an LSD
// radix sort of (key, index) pairs with 11-bit digits followed by one gather orders the list in ~10 ms. Ties on the key
// (which cannot come out of one handle) are ordered like tp_less afterwards; lists whose keys do not fit fall back to std::sort.
static unsigned
bit_length(uint64_t v)
{
  unsigned b = 0;
  while (v) {
    ++b;
    v >>= 1;
  }
  return b;
}

static void
sort_tps_impl(swtpg_tp* a, size_t n)
{
  if (n < 2)
    return;
  if (n < 4096 || n > 0xFFFFFFFFull) {
    std::stable_sort(a, a + n, tp_less);
    return;
  }
  uint64_t tmin = a[0].time_start, tmax = a[0].time_start;
  uint32_t lmax = 0;
  uint16_t cmax = 0;
  for (size_t i = 0; i < n; ++i) {
    tmin = std::min(tmin, a[i].time_start);
    tmax = std::max(tmax, a[i].time_start);
    lmax = std::max(lmax, a[i].link);
    cmax = std::max(cmax, a[i].channel);
  }
  const unsigned cb = bit_length(cmax), lb = bit_length(lmax), tb = bit_length(tmax - tmin), bits = cb + lb + tb;
  if (bits > 64) {
    std::stable_sort(a, a + n, tp_less);
    return;
  }
  struct KV
  {
    uint64_t key;
    uint32_t idx, pad;
  };
  constexpr unsigned kDigit = 11, kBuckets = 1u << kDigit, kMaxPasses = (64 + kDigit - 1) / kDigit;
  const unsigned passes = (bits + kDigit - 1) / kDigit;
  // scratch is kept per calling thread between calls (grow-only): a batch-sized sort per superchunk would otherwise spend most
  // of its time faulting in 64 n bytes of fresh pages
  thread_local std::vector<unsigned char> scratch;
  const size_t need = 2 * n * sizeof(KV) + n * sizeof(swtpg_tp) + 64;
  if (scratch.size() < need)
    scratch.resize(need + need / 4);
  unsigned char* base = scratch.data() + ((64 - (reinterpret_cast<uintptr_t>(scratch.data()) & 63)) & 63);
  KV* kv = reinterpret_cast<KV*>(base);
  KV* kv2 = kv + n;
  swtpg_tp* out = reinterpret_cast<swtpg_tp*>(kv2 + n);
  std::vector<uint32_t> hist(size_t(kMaxPasses) * kBuckets, 0u); // all digit histograms in the pass that builds the keys
  for (size_t i = 0; i < n; ++i) {
    const uint64_t t = a[i].time_start - tmin;
    const uint64_t key = (tb ? t << (lb + cb) : 0) | (uint64_t(a[i].link) << cb) | a[i].channel;
    kv[i].key = key;
    kv[i].idx = uint32_t(i);
    for (unsigned p = 0; p < passes; ++p)
      ++hist[p * kBuckets + ((key >> (p * kDigit)) & (kBuckets - 1))];
  }
  KV *src = kv, *dst = kv2;
  for (unsigned p = 0; p < passes; ++p) {
    uint32_t* h = hist.data() + size_t(p) * kBuckets;
    uint32_t sum = 0;
    bool trivial = false;
    for (unsigned d = 0; d < kBuckets; ++d) {
      trivial |= h[d] == n; // every key has the same digit: nothing to do
      const uint32_t c = h[d];
      h[d] = sum;
      sum += c;
    }
    if (trivial)
      continue;
    const unsigned shift = p * kDigit;
    for (size_t i = 0; i < n; ++i)
      dst[h[(src[i].key >> shift) & (kBuckets - 1)]++] = src[i];
    std::swap(src, dst);
  }
  for (size_t i = 0; i < n; ++i)
    out[i] = a[src[i].idx];
  for (size_t i = 0; i < n;) { // runs of equal (time_start, link, channel): order the rest of tp_less, keeping input order on full ties
    size_t j = i + 1;
    while (j < n && src[j].key == src[i].key)
      ++j;
    if (j - i > 1)
      std::stable_sort(out + i, out + j, tp_less);
    i = j;
  }
  memcpy(a, out, n * sizeof(swtpg_tp));
}

extern "C" void
swtpg_sort_tps(swtpg_tp* tps, size_t n)
{
  if (tps && n > 1)
    sort_tps_impl(tps, n);
}

extern "C" void
swtpg_merge_sorted(const swtpg_tp* const* lists, const size_t* n, size_t k, swtpg_tp* out)
{
  // The lists are sorted like swtpg_sort_tps; ties are resolved by list index (stable across GPUs). A tree of two-way merges
  // of neighbouring runs: every level streams the records once (sequential reads and writes, one mostly-predictable comparison
  // on time_start per record), ceil(log2 k) levels, ping-pong between `out` and one scratch buffer arranged so that the last
  // level lands in `out`. std::merge takes equal elements from its first range first, and runs stay in list order, so the
  // result is what a stable sort of the concatenation gives (which is what this function did before, 10x slower).
  struct Run
  {
    const swtpg_tp* p;
    size_t n;
  };
  std::vector<Run> runs;
  size_t total = 0;
  for (size_t i = 0; i < k; ++i)
    if (n[i]) {
      runs.push_back({ lists[i], n[i] });
      total += n[i];
    }
  if (runs.empty())
    return;
  if (runs.size() == 1) {
    memcpy(out, runs[0].p, total * sizeof(swtpg_tp));
    return;
  }
  unsigned levels = 0;
  for (size_t r = runs.size(); r > 1; r = (r + 1) / 2)
    ++levels;
  thread_local std::vector<swtpg_tp> scratch; // grow-only, like the sort's
  if (levels > 1 && scratch.size() < total)
    scratch.resize(total + total / 4);
  for (unsigned level = 1; level <= levels; ++level) {
    swtpg_tp* w = ((levels - level) & 1u) ? scratch.data() : out;
    std::vector<Run> next;
    size_t pos = 0;
    for (size_t i = 0; i < runs.size(); i += 2) {
      if (i + 1 < runs.size()) {
        std::merge(runs[i].p, runs[i].p + runs[i].n, runs[i + 1].p, runs[i + 1].p + runs[i + 1].n, w + pos, tp_less);
        next.push_back({ w + pos, runs[i].n + runs[i + 1].n });
      } else { // odd run out: carried to this level's buffer so that the next level's inputs never alias its output
        memcpy(w + pos, runs[i].p, runs[i].n * sizeof(swtpg_tp));
        next.push_back({ w + pos, runs[i].n });
      }
      pos += next.back().n;
    }
    runs.swap(next);
  }
}

extern "C" int
swtpg_firwin_int(int n, double cutoff, int multiplier, int16_t* taps)
{ // src/wib2/tpg/DesignFIR.cpp:20-68 (host, double precision; runs once per start in the reference)
  if (n < 2 || n > 64 || !taps)
    return -1;
  const double pi = 3.14159265358979323846;
  std::vector<double> v(size_t(n), 0.0);
  double sum = 0;
  const int alpha = n / 2;
  for (int m = 0; m < n; ++m) {
    const double w = 0.54 - 0.46 * std::cos(2.0 * pi * m / (n - 1));
    const double x = cutoff * (m - alpha);
    v[size_t(m)] = w * (x == 0 ? 1.0 : std::sin(pi * x) / (pi * x));
    sum += v[size_t(m)];
  }
  for (int m = 0; m < n; ++m)
    taps[m] = int16_t(std::round(multiplier * (v[size_t(m)] / sum)));
  return n;
}

// ---- noise power spectra -------------------------------------------------------------------------------------------------
// swtpg_noise_power (include/swtpg.h): the cosine transform of the circular lag sums of swtpg_read_noise_lags.
extern "C" swtpg_status
swtpg_noise_power(const swtpg_noise_lags* in, size_t n, int format, double* power)
{
  if ((!in || !power) && n)
    return SWTPG_ERR_INVALID_ARG;
  if (format != SWTPG_FORMAT_WIBETH && format != SWTPG_FORMAT_WIB2)
    return SWTPG_ERR_UNSUPPORTED;
  const int N = int(format == SWTPG_FORMAT_WIB2 ? SWTPG_WIB2_NOISE_SEGMENT_TICKS : SWTPG_WIBETH_NOISE_SEGMENT_TICKS);
  const int bins = N / 2 + 1;
  const double kPi = 3.14159265358979323846;
  std::vector<double> c(size_t(bins) * bins); // c[k][tau]: weight of lag[tau] in bin k (1, 2 cos(2 pi k tau / N), cos(pi k))
  for (int k = 0; k < bins; ++k)
    for (int tau = 0; tau < bins; ++tau)
      c[size_t(k) * bins + tau] = (tau == 0 || tau == N / 2 ? 1.0 : 2.0) * std::cos(2 * kPi * ((k * tau) % N) / N);
  for (size_t i = 0; i < n; ++i) {
    const swtpg_noise_lags& a = in[i];
    double* p = power + i * size_t(bins);
    if (a.segments == 0) {
      std::fill(p, p + bins, 0.0);
      continue;
    }
    const double scale = 1.0 / (double(N) * double(a.segments));
    double p0 = 0;
    for (int tau = 0; tau < bins; ++tau)
      p0 += c[size_t(tau)] * double(a.lag[tau]);
    p[0] = p0 * scale;
    // k >= 1: the weights sum to 0, so lag[tau] - lag[0] (exact in int64: 0 <= lag[tau] <= lag[0] < 2^63) gives the same sum
    // without the pedestal's N x 900^2 per segment drowning the noise in rounding.
    double d[SWTPG_WIBETH_NOISE_SEGMENT_TICKS / 2 + 1];
    for (int tau = 0; tau < bins; ++tau)
      d[tau] = double(int64_t(a.lag[tau]) - int64_t(a.lag[0]));
    for (int k = 1; k < bins; ++k) {
      double s = 0;
      for (int tau = 1; tau < bins; ++tau)
        s += c[size_t(k) * bins + tau] * d[tau];
      p[k] = s * scale;
    }
  }
  return SWTPG_OK;
}

// ---- channel covariance ------------------------------------------------------------------------------------------------------
// swtpg_channel_covariance (include/swtpg.h): covariance and correlation matrices of the channel products of
// swtpg_read_channel_products.
extern "C" swtpg_status
swtpg_channel_covariance(const uint64_t* in, size_t n_links, int format, double* covariance, double* correlation)
{
  if (!in)
    return SWTPG_ERR_INVALID_ARG;
  if (format != SWTPG_FORMAT_WIBETH && format != SWTPG_FORMAT_WIB2)
    return SWTPG_ERR_UNSUPPORTED;
  const size_t C = format == SWTPG_FORMAT_WIB2 ? SWTPG_WIB2_CHANNELS : SWTPG_WIBETH_CHANNELS;
  const size_t words = SWTPG_CHANNEL_PRODUCTS_WORDS(C);
  const double nan = std::numeric_limits<double>::quiet_NaN();
  std::vector<__int128> num(C * C);
  for (size_t l = 0; l < n_links; ++l) {
    const uint64_t* w = in + l * words;
    const __int128 n = w[0];
    const uint64_t* sum = w + 1;
    // num_ij = n P_ij - S_i S_j exactly: n < 2^36, P_ij < 2^64 and S_i < 2^50 keep both terms below 2^100
    for (size_t i = 0, k = 1 + C; i < C; ++i)
      for (size_t j = i; j < C; ++j, ++k)
        num[i * C + j] = num[j * C + i] = n * __int128(w[k]) - __int128(sum[i]) * __int128(sum[j]);
    const double n2 = double(w[0]) * double(w[0]);
    for (size_t i = 0; i < C; ++i)
      for (size_t j = 0; j < C; ++j) {
        const size_t o = (l * C + i) * C + j;
        const __int128 vi = num[i * C + i], vj = num[j * C + j];
        if (covariance)
          covariance[o] = w[0] ? double(num[i * C + j]) / n2 : 0.0; // a variance of 0 makes num_ij 0 (Cauchy-Schwarz)
        if (correlation)
          correlation[o] = vi > 0 && vj > 0 ? std::clamp(double(num[i * C + j]) / std::sqrt(double(vi) * double(vj)), -1.0, 1.0) : nan;
      }
  }
  return SWTPG_OK;
}
