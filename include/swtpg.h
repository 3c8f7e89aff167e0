/*
 * swtpg.h — C ABI of the B200-native software trigger-primitive generator (libswtpg_b200.so).
 *
 * This is the drop-in boundary for ONE path of DUNE-DAQ/fdreadoutlibs: what happens inside
 * WIBEthFrameProcessor::find_hits / WIB2FrameProcessor::find_hits, i.e.
 *   14-bit unpack -> frugal-streaming pedestal -> [running sum | FIR] -> threshold hit finding -> TriggerPrimitive fields.
 * Every entry point names the reference interface it replaces (paths relative to the reference repository root).
 * Plain C: POD structs, pointers and sizes, integer status codes; no exceptions cross this boundary and no
 * torch / CUDA types appear in any signature (streams and device pointers travel as void*).
 *
 * There is no CPU fallback: every compute entry point fails with SWTPG_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef SWTPG_H_
#define SWTPG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SWTPG_ABI_VERSION 2u

/* Frame geometry restated from the reference (sizes pinned by static_asserts there). */
#define SWTPG_WIBETH_FRAME_BYTES 7200u /* include/fdreadoutlibs/DUNEWIBEthTypeAdapter.hpp:20-22,98 */
#define SWTPG_WIBETH_CHANNELS 64u
#define SWTPG_WIBETH_TICKS 64u        /* wibeth/tpg/TPGConstants_wibeth.hpp:22 (FRAMES_PER_MSG) */
#define SWTPG_WIBETH_TS_PER_FRAME 2048u /* DUNEWIBEthTypeAdapter.hpp:93 */
#define SWTPG_WIB2_FRAME_BYTES 472u
#define SWTPG_WIB2_SUPERCHUNK_BYTES 5664u /* include/fdreadoutlibs/DUNEWIBSuperChunkTypeAdapter.hpp:18-22,100 */
#define SWTPG_WIB2_CHANNELS 256u
#define SWTPG_WIB2_TICKS 12u          /* wib2/tpg/TPGConstants_wib2.hpp:30 (FRAMES_PER_MSG) */
#define SWTPG_TS_PER_TICK 32u         /* DUNEWIBEthTypeAdapter.hpp:95, DUNEWIBSuperChunkTypeAdapter.hpp:97 */
#define SWTPG_MAX_TAPS 8u

typedef enum swtpg_status
{
  SWTPG_OK = 0,
  SWTPG_ERR_INVALID_ARG = 1,
  SWTPG_ERR_CUDA = 2,       /* no usable device / CUDA runtime error; see swtpg_last_error() */
  SWTPG_ERR_BUSY = 3,       /* back-pressure: staging ring full (reference: FailedToSendTP-style drop, never blocks) */
  SWTPG_ERR_OVERFLOW = 4,   /* more TPs than the caller's / the device buffer's capacity; count is still reported */
  SWTPG_ERR_STATE = 5,      /* call sequence violated (e.g. submit before start) */
  SWTPG_ERR_UNSUPPORTED = 6 /* reference: TPGAlgorithmInexistent (include/fdreadoutlibs/FDReadoutIssues.hpp:27-31) */
} swtpg_status;

typedef enum swtpg_format
{
  SWTPG_FORMAT_WIBETH = 0, /* unit = one 7200-B WIBEthFrame: 64 channels x 64 ticks */
  SWTPG_FORMAT_WIB2 = 1    /* unit = one 5664-B superchunk of 12 WIB2 frames: 256 channels x 12 ticks */
} swtpg_format;

/* tpg_algorithm strings of the reference (src/wibeth/WIBEthFrameProcessor.cpp:180-197) plus the FIR+IQR finder that
 * the reference ships for WIB2/ProtoWIB (include/fdreadoutlibs/wib2/tpg/ProcessAVX2FIR.hpp). */
typedef enum swtpg_algorithm
{
  SWTPG_ALGO_SIMPLE_THRESHOLD = 0, /* "SimpleThreshold": wibeth/tpg/ProcessAVX2.hpp, wib2/tpg/ProcessAVX2.hpp */
  SWTPG_ALGO_ABS_RS = 1,           /* "AbsRS":      wibeth/tpg/ProcessAbsRSAVX2.hpp, wib2/tpg/ProcessRSAVX2.hpp */
  SWTPG_ALGO_STANDARD_RS = 2,      /* "StandardRS": wibeth/tpg/ProcessStandardRSAVX2.hpp */
  SWTPG_ALGO_FIR_IQR = 3           /* FIR matched filter + IQR threshold: wib2/tpg/ProcessAVX2FIR.hpp */
} swtpg_algorithm;

/* One trigger primitive as emitted by the device: the fields process_swtpg_hits derives per hit
 * (src/wibeth/WIBEthFrameProcessor.cpp:523-545, src/wib2/WIB2FrameProcessor.cpp:431-455) BEFORE the
 * register->offline-channel LUT, channel mask and tp_timeout filters, which stay on the host shim.
 * `channel` is the frame channel (WIBEth 0..63, WIB2 0..255); see DESIGN.md "H2". 32 bytes. */
typedef struct swtpg_tp
{
  uint64_t time_start;          /* 62.5 MHz ticks: ts(frame of hit end) + 32*(t_end - tover) */
  uint64_t time_peak;
  uint32_t time_over_threshold; /* 32 * samples over threshold */
  uint32_t adc_integral;
  uint16_t adc_peak;
  uint16_t channel;
  uint32_t link;                /* index of the link inside this handle (0..n_links-1) */
} swtpg_tp;

/* Mirrors the fields of readoutlibs' RawDataProcessorConf that the hot path consumes
 * (src/wibeth/WIBEthFrameProcessor.cpp:175-230) and the handler constants
 * (include/fdreadoutlibs/wibeth/WIBEthFrameProcessor.hpp:69, wib2/WIB2FrameProcessor.hpp:68-69). */
typedef struct swtpg_config
{
  uint32_t struct_size;      /* = sizeof(swtpg_config); lets the ABI grow */
  int32_t device;            /* CUDA device ordinal */
  int32_t format;            /* swtpg_format */
  int32_t algorithm;         /* swtpg_algorithm */
  uint32_t n_links;          /* independent links owned by this handle (one reference FrameProcessor each) */
  uint32_t max_units;        /* superchunk length: units (frames / WIB2 superchunks) per link per batch, < 2^18 */
  uint32_t tp_capacity;      /* device TP buffer, records per batch; 0 = sized for the worst case */
  uint32_t n_slots;          /* staging-ring depth of the streaming path (>= 2); 0 = 4 */
  uint16_t threshold;        /* tpg_threshold (ADC; sigma units for FIR_IQR) */
  int16_t frugal_acc_limit;  /* tpg_frugal_streaming_accumulator_limit (WIB2 and FIR paths hard-wire 10) */
  uint16_t rs_memory_factor; /* already x10, as conf() scales it (WIBEthFrameProcessor.cpp:202) */
  uint16_t rs_scale_factor;  /* already 10/x (WIBEthFrameProcessor.cpp:206) */
  int16_t fir_taps[SWTPG_MAX_TAPS]; /* FIR_IQR only; all-zero = firwin_int(7,0.1,64)+{0} = {1,6,15,20,15,6,1,0} */
  uint8_t tap_exponent;      /* m_tpg_tap_exponent = 6 */
  uint8_t reserved0[3];
  uint32_t wib2_adc_offset;  /* byte offset of adc_words inside a WIB2 frame; 0 = 20 */
  uint32_t flags;            /* SWTPG_FLAG_* */
  uint32_t dispatch_timeout_us; /* streaming path: units that have waited this long are dispatched even if no link has a full
                                   superchunk yet (a stalled or dead link never holds the others back); 0 = 5000 */
} swtpg_config;

#define SWTPG_FLAG_NONE 0u
/* The TP list of every batch (swtpg_process_host, swtpg_fetch_tps, swtpg_poll*) comes back ordered by (time_start, link,
 * channel) — the order TriggerPrimitiveTypeAdapter::operator< imposes downstream
 * (include/fdreadoutlibs/TriggerPrimitiveTypeAdapter.hpp:26-29) — ordered ON THE DEVICE before it crosses the host link (an LSD
 * radix sort of packed keys in HBM), identical to what swtpg_sort_tps makes of the unordered list. Lists of one handle can
 * then be merged across GPUs with swtpg_merge_sorted without a host sort. */
#define SWTPG_FLAG_SORTED_TPS 1u
/* Per-channel ADC statistics of every link (swtpg_read_adc_stats): one extra read of every batch on the device, after its TPG kernel
 * and on the same stream. Without the flag nothing is allocated or launched for them. */
#define SWTPG_FLAG_ADC_STATS 2u
/* Per-channel noise spectra of every link (swtpg_read_noise_lags, swtpg_noise_power): the circular lag sums of fixed segments of
 * every channel, accumulated on the device by the same extra read of every batch as SWTPG_FLAG_ADC_STATS (with both flags the batch
 * is read once). Without the flag nothing is allocated or launched for them. */
#define SWTPG_FLAG_NOISE_SPECTRA 8u /* bit 4u stays unassigned: swtpg_create keeps refusing it */
/* Noise-spectrum segment lengths in ticks: one WIBEth frame, four WIB2 superchunks. */
#define SWTPG_WIBETH_NOISE_SEGMENT_TICKS 64u
#define SWTPG_WIB2_NOISE_SEGMENT_TICKS 48u
/* Channel-to-channel covariance of every link (swtpg_read_channel_products, swtpg_channel_covariance): the sums of products of
 * every pair of channels of a link, accumulated on the device by a kernel of its own after the statistics read of every batch
 * and on the same stream. Without the flag nothing is allocated or launched for them. */
#define SWTPG_FLAG_CHANNEL_COVARIANCE 32u /* bits 4u and 16u stay unassigned: swtpg_create keeps refusing them */
/* uint64_t words per link of swtpg_read_channel_products for a link of `channels` frame channels: 2145 (WIBEth), 33153 (WIB2). */
#define SWTPG_CHANNEL_PRODUCTS_WORDS(channels) (1u + (channels) + (channels) * ((channels) + 1u) / 2u)

/* Per-channel carried state, by frame channel: ChanState of wibeth/tpg/ProcessingInfo.hpp:20-66 and
 * wib2/tpg/ProcessingInfo.hpp:20-68. Used for parity dumps only. */
typedef struct swtpg_channel_state
{
  int16_t pedestal, accum;
  int16_t quantile25, quantile75, accum25, accum75;
  int16_t rs, pedestal_rs, accum_rs;
  uint16_t rs_memory_factor;
  uint16_t prev_was_over, hit_charge, hit_tover, hit_peak_adc, hit_peak_time;
  uint16_t initialized; /* 0 until the first unit seeded the pedestal (setState) */
  int16_t prev_samp[SWTPG_MAX_TAPS];
} swtpg_channel_state;

/* Counters behind the opmon fields of get_info (src/wibeth/WIBEthFrameProcessor.cpp:237-292). */
typedef struct swtpg_counters
{
  uint64_t units_processed;  /* frames / superchunks */
  uint64_t samples_processed;
  uint64_t tps_emitted;
  uint64_t tps_dropped_overflow;
  uint64_t batches;
  uint64_t submit_busy;      /* swtpg_submit calls refused with SWTPG_ERR_BUSY */
  uint64_t h2d_bytes, d2h_bytes;
  uint64_t units_zero_copy;  /* streaming path: units read where they lay in a registered latency buffer ... */
  uint64_t units_staged;     /* ... and units copied into the pinned staging ring by swtpg_submit */
} swtpg_counters;

typedef struct swtpg_handle swtpg_handle;

uint32_t swtpg_abi_version(void);
const char* swtpg_status_string(swtpg_status s);
/* Thread-local text of the last failure on this handle (NULL handle: last create failure). */
const char* swtpg_last_error(const swtpg_handle* h);
/* 1 if a CUDA device of compute capability 10.x is visible, else 0. Never throws, never initialises a context. */
int swtpg_device_available(void);

/* Replaces WIBEthFrameHandler::initialize / WIB2FrameHandler::initialize (buffers, taps, ProcessingInfo):
 * src/wibeth/WIBEthFrameProcessor.cpp:74-91, src/wib2/WIB2FrameProcessor.cpp:90-120. */
swtpg_status swtpg_create(const swtpg_config* cfg, swtpg_handle** out);
void swtpg_destroy(swtpg_handle* h);

/* Replaces the TPG part of FrameProcessor::start / ::stop: fresh zeroed ChanState, first_hit re-armed
 * (src/wibeth/WIBEthFrameProcessor.cpp:111-154, 67-72). */
swtpg_status swtpg_start(swtpg_handle* h);
swtpg_status swtpg_stop(swtpg_handle* h);

/* Per-position RS memory factor of AbsRS / StandardRS, by frame channel: [n_links][channels]
 * (src/wibeth/WIBEthFrameProcessor.cpp:437-456). NULL = cfg.rs_memory_factor everywhere. Call before the first unit. */
swtpg_status swtpg_set_rs_memory_factor(swtpg_handle* h, const uint16_t* by_link_channel);
/* The same for ONE link: by_channel[channels]. This is what a frame processor calls from find_hits on its first frame
 * (WIBEthFrameProcessor.cpp:437-456 runs per link): one small asynchronous copy ordered on the compute stream, thread-safe
 * against the other links' calls and against batches in flight. */
swtpg_status swtpg_set_link_rs_memory_factor(swtpg_handle* h, uint32_t link, const uint16_t* by_channel);

/* Per-link TPG configuration. Every frame processor of the reference parses its own RawDataProcessorConf
 * (src/wibeth/WIBEthFrameProcessor.cpp:175-230), so two links of one application may run different algorithms or thresholds.
 * Links whose configurations agree in every field their algorithm reads form one configuration group; each group is one
 * launch of the batch kernel, and the groups of a batch run one after another on the same stream. */
#define SWTPG_MAX_LINK_CONFIGS 16u /* distinct configurations per handle, the handle's own included */
typedef struct swtpg_link_config
{
  uint32_t struct_size;      /* = sizeof(swtpg_link_config) */
  int32_t algorithm;         /* swtpg_algorithm */
  uint16_t threshold;
  int16_t frugal_acc_limit;
  uint16_t rs_memory_factor, rs_scale_factor; /* already x10 / 10/x, as in swtpg_config */
  int16_t fir_taps[SWTPG_MAX_TAPS];           /* all zero = firwin_int(7, 0.1, 1 << tap_exponent) + {0} */
  uint8_t tap_exponent;      /* 0 = 6 */
  uint8_t reserved0[3];
} swtpg_link_config;
/* The TPG parameters of ONE link (the rest of its conf(): src/wibeth/WIBEthFrameProcessor.cpp:175-230). NULL = back to the
 * handle's swtpg_config. Only while the handle is not started (before swtpg_start or after swtpg_stop): SWTPG_ERR_STATE
 * otherwise. Takes effect at the next swtpg_start, which gives every link fresh state. SWTPG_ERR_INVALID_ARG for a bad
 * struct_size, link >= n_links, a field out of range or a configuration that would make more than SWTPG_MAX_LINK_CONFIGS
 * distinct ones (configurations that differ only in fields their algorithm does not read, or only in rs_memory_factor,
 * count as one); SWTPG_ERR_UNSUPPORTED for an unknown algorithm or StandardRS on WIB2, as swtpg_create. A per-channel table
 * of swtpg_set_*rs_memory_factor takes precedence over the link's rs_memory_factor, as over the handle's. */
swtpg_status swtpg_set_link_config(swtpg_handle* h, uint32_t link, const swtpg_link_config* c);

/* Per-channel thresholds of ONE link, by frame channel: by_channel[SWTPG_*_CHANNELS], each 0..32767 (ADC counts above the
 * pedestal, or above the RS median). NULL = back to the threshold of the link's configuration. An extension of the reference,
 * which applies one tpg_threshold to every channel of a frame processor: induction and collection planes, or a hot channel,
 * can have their own without a configuration per threshold (and without masking the channel).
 *   - Only while the handle is not started (SWTPG_ERR_STATE otherwise); takes effect at the next swtpg_start, like
 *     swtpg_set_link_config. The table stays until NULL or swtpg_destroy: it survives swtpg_stop / swtpg_start and later
 *     swtpg_set_link_config calls, and takes precedence over the threshold of the link's configuration.
 *   - SWTPG_ERR_INVALID_ARG for a NULL handle, link >= n_links or an entry above 32767.
 *   - SWTPG_ERR_UNSUPPORTED for a table on a link whose algorithm is FIR_IQR or WIB2 AbsRS: there the threshold multiplies an
 *     IQR sigma. swtpg_set_link_config refuses the same way to move a link that has a table to one of those algorithms
 *     (a NULL that returns it to such a handle configuration included). A refused call changes nothing; NULL is always accepted.
 *   - Tables do not split configuration groups: a link's thresholds are per-channel state, like its RS memory factors. */
swtpg_status swtpg_set_link_thresholds(swtpg_handle* h, uint32_t link, const uint16_t* by_channel);

/*
 * Batch entry points. `frames` is link-major: unit u of link l starts at ((l * units_stride) + u) * unit_bytes.
 * n_units[l] <= units_stride <= cfg.max_units valid units for link l (ragged batches allowed; NULL = all links
 * have units_stride units). State is carried from the previous batch per link, exactly as ProcessingInfo carries
 * it from frame to frame. TPs come back unordered; sort with swtpg_sort_tps for (time_start, link, channel) order.
 *
 * Together these replace the body of find_hits: expand_wibeth_adcs + setState on the first frame +
 * m_assigned_tpg_algorithm_function + process_swtpg_hits' field arithmetic
 * (src/wibeth/WIBEthFrameProcessor.cpp:410-476,478-549; src/wib2/WIB2FrameProcessor.cpp:345-396,398-458).
 */
/* Host buffers (pageable or pinned): H2D copy, kernel, D2H of the TP list, all inside the call. Pinned or registered sources
 * are read by the copy engine directly; pageable sources of 16 MB and more go through a pipeline of pinned bounce buffers
 * filled by a few worker threads (3.6x the rate of a plain cudaMemcpy from pageable memory on the bench box). */
swtpg_status swtpg_process_host(swtpg_handle* h, const void* frames, const uint32_t* n_units, uint32_t units_stride,
                                swtpg_tp* out, size_t cap, size_t* n_out);
/* Frames already resident in HBM. `stream` is a cudaStream_t; NULL = the handle's own (non-blocking) stream — to run on
 * the legacy default stream pass cudaStreamLegacy, i.e. (void*)1. Asynchronous: the caller orders the producer of
 * d_frames before this call on that stream. TPs stay on the device until swtpg_fetch_tps. */
swtpg_status swtpg_process_device(swtpg_handle* h, const void* d_frames, const uint32_t* n_units, uint32_t units_stride,
                                  void* stream);
/* Waits for the last swtpg_process_device, copies its TPs out. *n_out = TPs found (may exceed cap: OVERFLOW). */
swtpg_status swtpg_fetch_tps(swtpg_handle* h, swtpg_tp* out, size_t cap, size_t* n_out);
/* Device time of the last batch kernel in milliseconds (CUDA events on the launching stream); < 0 if none. */
double swtpg_last_kernel_ms(swtpg_handle* h);

/* Parity dump of the intermediate waveforms the reference can print (docs/README.md:31-36 "save-adc"):
 * same as swtpg_process_host, plus per sample the pedestal AFTER its frugal update and the waveform the
 * threshold is applied to (pedestal-subtracted ADC, running sum, or FIR output), both int16,
 * laid out [link][unit][tick][channel] over units_stride units per link. Either may be NULL. */
swtpg_status swtpg_process_host_debug(swtpg_handle* h, const void* frames, const uint32_t* n_units, uint32_t units_stride,
                                      swtpg_tp* out, size_t cap, size_t* n_out, int16_t* pedestal_out, int16_t* waveform_out);

/*
 * Streaming entry points: what a FrameProcessor's post-processing thread calls once per payload.
 *
 * Every link owns a ring of n_slots * max_units pending units. swtpg_submit appends one unit of `link` to that link's ring —
 * the payload's address if it lies in a latency buffer registered with swtpg_register_buffer (zero-copy), else a copy of it
 * in the link's pinned staging ring (the reference's constframeptr is only borrowed for the duration of find_hits) — and
 * returns; it takes no lock and never blocks: SWTPG_ERR_BUSY when that link's ring is full (the reference's failed try_send).
 * One producer thread per link at a time, any number of links concurrently.
 *
 * A dispatcher thread inside the library turns pending units into batches: as soon as ANY link has a full superchunk
 * (cfg.max_units units), or pending units have waited cfg.dispatch_timeout_us, or on swtpg_flush, every link contributes what
 * it has delivered so far (0 .. max_units units: batches are ragged, per-link state is carried from batch to batch exactly as
 * ProcessingInfo carries it from frame to frame). So links advance independently; a silent link does not hold back the TPs
 * of the others. A batch is: ONE gather kernel that pulls the units out of pinned host memory through a per-unit pointer
 * table (no per-link copy calls) -> the fused TPG kernel -> the TP list back to pinned host memory. A completion thread frees
 * the ring space of a batch as soon as its gather has finished (which also ends the borrow of zero-copy units) and queues
 * the batch's TPs; swtpg_poll hands them out, oldest batch first. It replaces the per-hit m_tp_sink->try_send loop's source
 * (src/wibeth/WIBEthFrameProcessor.cpp:555). At most n_slots batches exist at a time: un-polled TPs back-pressure the ring.
 */
swtpg_status swtpg_submit(swtpg_handle* h, uint32_t link, const void* unit, size_t bytes);
/* Like swtpg_submit, but waits (sleeping, not spinning) up to timeout_us for room in the link's ring; SWTPG_ERR_BUSY on
 * time-out. For file replay and emulators, where stalling the source is right and dropping frames is not. */
swtpg_status swtpg_submit_wait(swtpg_handle* h, uint32_t link, const void* unit, size_t bytes, uint64_t timeout_us);
/*
 * Zero-copy ingest. The constframeptr a post-processing task receives points INTO the link's latency buffer
 * (readoutlibs IterableQueueModel / FixedRateQueueModel: one contiguous array of payloads; SURVEY.md 8b "Ownership").
 * Registering that array here (cudaHostRegister, mapped) makes swtpg_submit record the payload's address instead of copying
 * it: the batch's gather kernel reads the unit where it lies, over the host link. Units outside every registered range (or
 * not 16-byte aligned) are still copied, so both kinds may be mixed. Contract: a submitted unit must stay unmodified until
 * its batch's gather has completed — at most n_slots superchunks after the submit, milliseconds against a latency buffer's
 * seconds of retention; swtpg_flush + swtpg_sync (or stop) end every such borrow. Any number of ranges (one per link is
 * typical). swtpg_unregister_buffer flushes and waits for the handle to drain first.
 */
swtpg_status swtpg_register_buffer(swtpg_handle* h, void* base, size_t bytes);
swtpg_status swtpg_unregister_buffer(swtpg_handle* h, void* base);
/* Dispatches everything submitted so far (ragged batch), returns when it has been handed to the device. Safe against
 * concurrent swtpg_submit calls (units submitted meanwhile may or may not be included). SWTPG_ERR_BUSY if all n_slots
 * batches hold TPs nobody has polled yet: poll, then flush again. */
swtpg_status swtpg_flush(swtpg_handle* h);
/* TPs of completed batches, oldest first, without blocking. *n_out = records written (<= cap); call again for more. */
swtpg_status swtpg_poll(swtpg_handle* h, swtpg_tp* out, size_t cap, size_t* n_out);
/* The same, but sleeps up to timeout_us until at least one completed batch is available. */
swtpg_status swtpg_poll_wait(swtpg_handle* h, swtpg_tp* out, size_t cap, size_t* n_out, uint64_t timeout_us);
/* Blocks until every dispatched batch has completed (used by stop and by tests). */
swtpg_status swtpg_sync(swtpg_handle* h);
/* Streaming path bookkeeping: units submitted but not yet dispatched, batches dispatched but not yet completed, completed
 * batches waiting for swtpg_poll. Any pointer may be NULL. */
swtpg_status swtpg_stream_status(swtpg_handle* h, uint64_t* units_pending, uint32_t* batches_in_flight, uint32_t* batches_ready);
/* Device time (CUDA events) the completed batches of the streaming path spent in the gather kernel — the host-link transfer —
 * and in the fused TPG kernel since swtpg_start, and how many batches that covers. Monitoring / bench aid. */
swtpg_status swtpg_stream_timing(swtpg_handle* h, double* gather_ms, double* kernel_ms, uint64_t* batches);

/* Carried state of one link, by frame channel (ChanState parity). out has SWTPG_*_CHANNELS entries. */
swtpg_status swtpg_dump_state(swtpg_handle* h, uint32_t link, swtpg_channel_state* out);

/* Statistics of the raw ADC values of one channel (frame channel, as swtpg_tp.channel) over one window. 32 bytes.
 * pedestal = sum / samples, RMS noise = sqrt(sum_sq / samples - pedestal^2). An extension of the reference, whose opmon reports
 * only the TP rate per channel: the noise that a per-channel threshold (swtpg_set_link_thresholds) is usually a multiple of,
 * and saturated (max 16383) or dead (min == max) channels. */
typedef struct swtpg_adc_stats
{
  uint64_t samples;      /* samples of this channel in the window */
  uint64_t sum;          /* sum of the raw 14-bit ADC values */
  uint64_t sum_sq;       /* sum of their squares: exact while samples < 2^36 (9.7 h of one channel's data) */
  uint16_t min, max;     /* raw ADC extremes; both 0 when samples == 0 */
  uint32_t reserved;
} swtpg_adc_stats;
/* out[n_links][SWTPG_*_CHANNELS] for links link0 .. link0 + n_links - 1 (handles created with SWTPG_FLAG_ADC_STATS). Every sample of
 * every valid unit (u < n_units[l]) of every batch, from every batch entry point and the streaming path, is counted once.
 *   - A window holds exactly the batches enqueued before the read that ends it: the read is ordered like a batch, on the stream of
 *     the last batch, and waits only for that work. reset != 0 starts the next window of these links at that point, so every batch
 *     falls into exactly one window, also while the streaming path dispatches batches or other threads read other links.
 *   - swtpg_start zeroes every window; after swtpg_stop they stay readable; before the first batch they read as zeros.
 *   - SWTPG_ERR_STATE on a handle created without the flag; SWTPG_ERR_INVALID_ARG for a NULL handle or out, or for
 *     link0 + n_links > cfg.n_links. */
swtpg_status swtpg_read_adc_stats(swtpg_handle* h, uint32_t link0, uint32_t n_links, swtpg_adc_stats* out, int reset);

/* Noise lags of one channel (frame channel, as swtpg_tp.channel) over one window. 272 bytes. An extension of the reference: what
 * the noise is (white, a coherent line, low-frequency pickup), from which a threshold or the FIR taps of a channel are chosen.
 * A segment is N consecutive ticks of one batch: N = SWTPG_WIBETH_NOISE_SEGMENT_TICKS (one frame) or
 * SWTPG_WIB2_NOISE_SEGMENT_TICKS (four superchunks; a WIB2 link's valid units of a batch are cut into groups of four from its
 * first unit, and a remainder of 1-3 superchunks is not counted). A segment never spans two batches. With x the raw 14-bit ADC
 * values of a segment,
 *   lag[tau] = sum over segments of sum_{t<N} x[t] x[(t + tau) mod N],  tau = 0 .. N/2,
 * the circular lags, whose cosine transform is the segment's |rfft(x)|^2 (swtpg_noise_power). WIB2 fills lag[0..24] and leaves
 * the rest 0. The sums are exact while lag[0] < 2^63, i.e. segments < 5.3e8 (4.9 h of one channel's data at 1.953125 MHz). */
typedef struct swtpg_noise_lags
{
  uint64_t segments; /* segments of this channel in the window */
  uint64_t lag[33];  /* circular lag sums, tau = 0 .. N/2 */
} swtpg_noise_lags;
/* out[n_links][SWTPG_*_CHANNELS] for links link0 .. link0 + n_links - 1 (handles created with SWTPG_FLAG_NOISE_SPECTRA). Windows,
 * their order against batches and the streaming path, resets, swtpg_start, swtpg_stop and the errors are those of
 * swtpg_read_adc_stats; a read of one kind ends no window of the other kind. */
swtpg_status swtpg_read_noise_lags(swtpg_handle* h, uint32_t link0, uint32_t n_links, swtpg_noise_lags* out, int reset);
/* The averaged periodogram with a rectangular window of n entries of swtpg_read_noise_lags of a handle of `format`: power[n][N/2+1],
 * bin k at k * 1.953125 MHz / N, the mean over segments of |rfft(x)_k|^2 / N:
 *   P_k = (lag[0] + 2 sum_{tau=1}^{N/2-1} lag[tau] cos(2 pi k tau / N) + lag[N/2] cos(pi k)) / (N segments).
 * For k >= 1 lag[0] is subtracted from every lag in exact integers first (the cosine weights sum to 0), so the pedestal does not
 * swamp the noise. Bin 0 keeps the pedestal: by Parseval the N bins of the full periodogram sum to lag[0] / segments. An entry with
 * no segments gives zeros. A pure host function; SWTPG_ERR_INVALID_ARG for NULL pointers, SWTPG_ERR_UNSUPPORTED for an unknown
 * format. */
swtpg_status swtpg_noise_power(const swtpg_noise_lags* in, size_t n, int format, double* power);

/* Channel products of one link over one window: SWTPG_CHANNEL_PRODUCTS_WORDS(C) uint64_t words, C = SWTPG_*_CHANNELS, by frame
 * channel (as swtpg_tp.channel). An extension of the reference: whether a channel's noise is shared with other channels (pickup
 * common to the channels of one front-end ASIC or FEMB), which no per-channel statistic shows and which a threshold at k x RMS
 * fires on whole groups of channels for. With x_c[t] the raw 14-bit ADC values of channel c over the window's ticks t,
 *   [0]                   samples, the ticks counted (every channel of a link sees every tick)
 *   [1 + c]               sum[c] = sum_t x_c[t],                      c = 0 .. C-1
 *   [1 + C + k(i, j)]     products[i][j] = sum_t x_i[t] x_j[t],       i <= j, upper triangle row-major:
 *                         k(i, j) = i C - i (i - 1) / 2 + (j - i)
 * The sums are exact while samples < 2^36 (9.7 h of one link's data). They are of raw values, so hits and cosmic tracks, which
 * correlate neighbouring channels too, are in them: read the matrix over quiet windows. */
/* out[n_links][SWTPG_CHANNEL_PRODUCTS_WORDS(C)] for links link0 .. link0 + n_links - 1 (handles created with
 * SWTPG_FLAG_CHANNEL_COVARIANCE). Windows, their order against batches and the streaming path, resets, swtpg_start, swtpg_stop and
 * the errors are those of swtpg_read_adc_stats; a read of one kind ends no window of another kind. */
swtpg_status swtpg_read_channel_products(swtpg_handle* h, uint32_t link0, uint32_t n_links, uint64_t* out, int reset);
/* Covariance and Pearson correlation of n_links entries of swtpg_read_channel_products of a handle of `format`: covariance and
 * correlation [n_links][C][C], full and symmetric, either may be NULL. With n = samples, S = sum, P = products,
 *   num_ij = n P_ij - S_i S_j   (formed exactly in 128-bit integers: the pedestal's n x 900^2 per product would otherwise
 *                                swamp the noise's covariance in rounding)
 *   covariance_ij  = num_ij / n^2                 (population covariance, numpy.cov(bias=True))
 *   correlation_ij = num_ij / sqrt(num_ii num_jj) (clipped to [-1, 1] against rounding, as numpy.corrcoef)
 * Where a variance is 0 (a dead or constant channel, a link without samples) the covariance is 0 and the correlation NaN. A pure
 * host function; SWTPG_ERR_INVALID_ARG for a NULL in, SWTPG_ERR_UNSUPPORTED for an unknown format. */
swtpg_status swtpg_channel_covariance(const uint64_t* in, size_t n_links, int format, double* covariance, double* correlation);
swtpg_status swtpg_get_counters(swtpg_handle* h, swtpg_counters* out);
/* SWTPG_FLAG_SORTED_TPS bookkeeping: device time (CUDA events, includes the 16-byte read-back of the key range) of the last
 * ordered list and of all lists since swtpg_create, how many lists were ordered on the device, and how many of them the host
 * had to finish (equal keys, or keys wider than 64 bits: links whose timestamps are unrelated). Any pointer may be NULL. */
swtpg_status swtpg_sort_stats(swtpg_handle* h, double* last_ms, double* total_ms, uint64_t* lists, uint64_t* finished_on_host);

/* Page-locked host memory for frame buffers handed to swtpg_process_host (or used as a latency buffer without a later
 * swtpg_register_buffer). write_combined != 0 asks for write-combined pages: the CPU only ever WRITES frames there (reads are
 * very slow) and the device's reads do not snoop the CPU caches, which matters when several GPUs of one host ingest at once.
 * Returns NULL on failure. */
void* swtpg_alloc_pinned(size_t bytes, int write_combined);
void swtpg_free_pinned(void* p);

/* Host-side ordering of a TP list by (time_start, link, channel): the order TriggerPrimitiveTypeAdapter::operator<
 * imposes downstream (include/fdreadoutlibs/TriggerPrimitiveTypeAdapter.hpp:26-29). In place. */
void swtpg_sort_tps(swtpg_tp* tps, size_t n);
/* k-way merge of already sorted per-GPU TP lists into `out` (capacity sum of n[i]): the host-side time-ordered
 * merge that follows link sharding across GPUs. */
void swtpg_merge_sorted(const swtpg_tp* const* lists, const size_t* n, size_t k, swtpg_tp* out);

/* firwin_int of src/wib2/tpg/DesignFIR.cpp:57-68 (host, double precision): taps[n]. Returns n. */
int swtpg_firwin_int(int n, double cutoff, int multiplier, int16_t* taps);

#ifdef __cplusplus
}
#endif
#endif /* SWTPG_H_ */
