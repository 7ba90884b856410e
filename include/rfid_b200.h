/* rfid_b200.h -- C-ABI of the B200-native Gen2 receive/decode chain.
 *
 * This is the drop-in boundary: a plain-C shared library (librfid_b200.so) whose
 * entry points are what the reference's three GNU Radio blocks would bind if
 * their work() loops were replaced by GPU calls.  Nothing like it exists in the
 * reference (it has no FFI); each entry point cites the reference interface it
 * replaces (paths relative to /root/reference/gr-rfid).
 *
 *   reference                                   | replaced by
 *   --------------------------------------------+--------------------------------------
 *   filter.fir_filter_ccc(5,[1]*25)             | rfid_b200_mf_work      (block mode)
 *     apps/reader.py:65,75 (GNU Radio, external)|   + fused into rfid_b200_decode_capture
 *   gate_impl::general_work  lib/gate_impl.cc:85| rfid_b200_gate_work    (block mode)
 *   tag_decoder_impl::general_work              | rfid_b200_decoder_work (block mode)
 *     lib/tag_decoder_impl.cc:196               |
 *   whole RX chain on a recorded capture        | rfid_b200_decode_capture (capture mode)
 *   READER_STATS bookkeeping                    | rfid_b200_reduce_stats
 *     lib/tag_decoder_impl.cc:269-288,329-387   |
 *
 * Conventions: every function returns 0 on success or a negative RFID_B200_E*
 * code (rfid_b200_strerror() names it); no exception crosses the boundary; no
 * torch/C++ types appear in a signature.  Complex samples are interleaved
 * float32 I,Q (GNU Radio gr_complex / the on-disk format of
 * misc/data/file_source_test, apps/reader.py:102).  There is NO CPU fallback:
 * rfid_b200_create() fails with RFID_B200_ENODEV when no sm_100 device is
 * usable.
 */
#ifndef RFID_B200_H
#define RFID_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RFID_B200_API __attribute__((visibility("default")))

#define RFID_B200_ABI_VERSION 1

/* error codes */
enum {
  RFID_B200_OK = 0,
  RFID_B200_EINVAL = -1,   /* bad argument */
  RFID_B200_ENODEV = -2,   /* no usable sm_100 CUDA device */
  RFID_B200_ENOMEM = -3,   /* host or device allocation failed */
  RFID_B200_ECUDA = -4,    /* CUDA runtime error (see rfid_b200_last_cuda_error) */
  RFID_B200_ECAPACITY = -5 /* caller-provided output buffer too small */
};

/* window kinds (reference: DECODER_DECODE_RN16 / DECODER_DECODE_EPC, include/rfid/global_vars.h:34) */
enum { RFID_B200_RN16 = 0, RFID_B200_EPC = 1 };

/* Configuration.  Defaults reproduce apps/reader.py:52-65 + include/rfid/global_vars.h:72-143. */
typedef struct rfid_b200_params {
  int32_t adc_rate;    /* raw complex sample rate, Hz            (reader.py:53  -> 2000000) */
  int32_t decim;       /* matched-filter decimation              (reader.py:54  -> 5)       */
  int32_t ntaps;       /* boxcar length = half an FM0 symbol     (reader.py:65  -> 25)      */
  int32_t fixed_q;     /* slots per round = 2^fixed_q            (global_vars.h:72 -> 0)    */
  int32_t max_queries; /* stop after this many Query/QueryRep    (global_vars.h:76 -> 1000) */
  int32_t max_tags;    /* stop after more than this many unique tags (global_vars.h:100 -> 100) */
  int32_t device;      /* CUDA device ordinal */
  int32_t reserved;
} rfid_b200_params;

/* One capture segment: a contiguous range of RAW samples that is decoded as an
 * independent stream with freshly constructed gate state (SURVEY.md section 8e). */
typedef struct rfid_b200_segment {
  uint64_t offset; /* first raw complex sample */
  uint32_t length; /* number of raw complex samples */
  uint32_t reserved;
} rfid_b200_segment;

/* One decoded window (64 bytes).  Everything the reference's tag_decoder
 * derives from one ungated window, including the quantities it keeps private
 * (score = local `max` in tag_sync, tag_decoder_impl.cc:81,94-98). */
typedef struct rfid_b200_window_result {
  int32_t segment;    /* index into the segment table */
  int32_t window;     /* ordinal inside the segment: even = RN16, odd = EPC (SURVEY.md 3.5) */
  int32_t open_index; /* decimated index (segment relative) of the first ungated sample, gate_impl.cc:164-175 */
  int32_t length;     /* n_samples_to_ungate, gate_impl.cc:115,121 */
  int32_t kind;       /* RFID_B200_RN16 / RFID_B200_EPC */
  int32_t sync_index; /* argmax offset of the preamble correlation, tag_decoder_impl.cc:85-100 */
  float score;        /* |c(sync_index)|^2, tag_decoder_impl.cc:94 */
  float h_re, h_im;   /* channel estimate h_est, tag_decoder_impl.cc:103 */
  float T;            /* EPC half-symbol period T_global, tag_decoder_impl.cc:166-169; 0 for RN16 */
  int32_t crc_ok;     /* EPC: 1 pass / 0 fail (check_crc, tag_decoder_impl.cc:401-445); RN16: -1 */
  int32_t tag_id;     /* EPC: bits[104..111] as an integer, tag_decoder_impl.cc:348-352; RN16: the 16-bit RN16 */
  uint8_t bits[16];   /* decoded bits, MSB first; RN16 uses bits[0..1], EPC all 16 bytes */
} rfid_b200_window_result;

/* READER_STATS as a plain struct (include/rfid/global_vars.h:36-53). */
#define RFID_B200_MAX_TAGS 256
typedef struct rfid_b200_stats {
  int32_t n_queries_sent;
  int32_t cur_inventory_round;
  int32_t cur_slot_number;
  int32_t max_slot_number;
  int32_t n_epc_correct;
  int32_t n_windows;      /* windows that entered the statistics */
  int32_t terminated;     /* 1 once the reference's stop rule fired, gate_impl.cc:101-109 */
  int32_t n_unique_tags;
  int32_t tag_id[RFID_B200_MAX_TAGS];    /* ascending (std::map order) */
  int32_t tag_reads[RFID_B200_MAX_TAGS];
} rfid_b200_stats;

typedef struct rfid_b200_ctx rfid_b200_ctx;

RFID_B200_API int rfid_b200_abi_version(void);
RFID_B200_API const char* rfid_b200_strerror(int code);
RFID_B200_API const char* rfid_b200_last_cuda_error(const rfid_b200_ctx* ctx);
RFID_B200_API void rfid_b200_default_params(rfid_b200_params* p);

/* Context: one per block instance (block mode) or per decode stream (capture mode).
 * A capture-mode call on another stream than the context's previous one waits for
 * everything queued on that previous stream, which must therefore still exist.
 * Replaces the constructors gate_impl.cc:41-70 / tag_decoder_impl.cc:50-62 and the
 * process-global reader_state (global_vars.cc:34-54). */
RFID_B200_API int rfid_b200_create(const rfid_b200_params* p, rfid_b200_ctx** out);
RFID_B200_API void rfid_b200_destroy(rfid_b200_ctx* ctx);

/* Derived sample counts (gate_impl.cc:48-53,115,121; tag_decoder_impl.cc:60). */
RFID_B200_API int rfid_b200_window_length(const rfid_b200_ctx* ctx, int kind);
RFID_B200_API int rfid_b200_fs_dec(const rfid_b200_ctx* ctx);

/* ---------------- capture mode (throughput path) ----------------
 * Decode nseg independent segments of a raw capture that is ALREADY RESIDENT in
 * device memory: matched filter + decimation, gate, tag_decoder, all on the GPU,
 * asynchronously on `stream` (a cudaStream_t passed as void*; NULL = default).
 * d_iq: device pointer, interleaved float32 I,Q.  d_segs: device pointer to nseg
 * segment descriptors.  d_results: device buffer of nseg*max_windows_per_segment
 * records; record k of segment s lands at d_results[s*max_windows_per_segment+k].
 * d_counts: device int32[nseg], number of windows found per segment.
 * Windows beyond max_windows_per_segment are counted but not stored. */
RFID_B200_API int rfid_b200_decode_capture(rfid_b200_ctx* ctx, const float* d_iq, size_t n_raw,
                                           const rfid_b200_segment* d_segs, int nseg,
                                           int max_windows_per_segment,
                                           rfid_b200_window_result* d_results, int32_t* d_counts,
                                           void* stream);

/* Same, but every pointer is a HOST pointer: copies in, decodes, copies the
 * records out, synchronises.  This is the end-to-end call a reference user makes
 * on a recorded file (apps/reader.py:102-112 in DEBUG mode). */
RFID_B200_API int rfid_b200_decode_capture_host(rfid_b200_ctx* ctx, const float* h_iq, size_t n_raw,
                                                const rfid_b200_segment* h_segs, int nseg,
                                                int max_windows_per_segment,
                                                rfid_b200_window_result* h_results, int32_t* h_counts);

/* Kernel launches issued by the last decode_capture call on this context. */
RFID_B200_API int rfid_b200_last_launch_count(const rfid_b200_ctx* ctx);
/* Device time (ms) of the decode kernel accumulated since the last reset, and its
 * launches, while timing is enabled.  Each launch stamps its first CTA start and
 * last CTA end on the GPU's global timer and counts end - max(start, end of the
 * previous launch): the device time it adds to a back-to-back sequence, without
 * launch latency.  Synchronises with the stream of the last timed launch. */
RFID_B200_API int rfid_b200_kernel_time(rfid_b200_ctx* ctx, int reset, float* ms_total, int* launches);
RFID_B200_API int rfid_b200_enable_kernel_timing(rfid_b200_ctx* ctx, int on);

/* Optional debug taps for capture mode (device pointers, may be NULL):
 * d_windows receives the ungated, DC-removed samples of every stored window
 * (gate output, gate_impl.cc:173,187) at a stride of rfid_b200_window_length(EPC)
 * complex samples per record slot. */
RFID_B200_API int rfid_b200_set_window_tap(rfid_b200_ctx* ctx, float* d_windows);

/* Host-side reduction of window records into READER_STATS, replaying the
 * bookkeeping of tag_decoder_impl.cc:269-288,295,329-387 and the stop rule of
 * gate_impl.cc:101-109 in stream order.  `continuous` != 0: all records belong to
 * one continuous reader session (counters carry across segments);
 * 0: every segment is its own session and the per-session stats are summed. */
RFID_B200_API int rfid_b200_reduce_stats(const rfid_b200_ctx* ctx, const rfid_b200_window_result* h_results,
                                         const int32_t* h_counts, int nseg, int max_windows_per_segment,
                                         int continuous, rfid_b200_stats* out);

/* ---------------- capture ingest (SURVEY.md section 8f, rank 2) ----------------
 * The reference decodes a recorded file (apps/reader.py:101-112, format: raw interleaved
 * float32 I,Q, misc/code/plot_signal.m:5-9) through ONE sequential gate.  Capture mode wants
 * independent segments, so a recording is first cut where nothing happens: reader commands are
 * bursts of low pulses (PW = 12 us, reader_impl.cc:55-71) separated by CW; every burst with more
 * than NUM_PULSES_COMMAND pulses arms exactly one gate window (gate_impl.cc:150-180) and the
 * window kinds alternate RN16/EPC, so a segment = `commands_per_segment` consecutive commands
 * plus the CW after each, starting `lead_us` of CW before the first.  Segment offsets are
 * multiples of `decim` (the matched filter keeps the capture's decimation phase); segment 0
 * starts at sample 0.  Decoding the segments reproduces the continuous reference run bit for
 * bit in every decision (open index, sync index, T, bits, CRC); correlation scores agree to the
 * drift of the reference's float running means (SURVEY.md 8e). */
typedef struct rfid_b200_segmenter {
  float level_frac;             /* low when |x| < level_frac * (mean |x| of the first 2^21 samples); 0.5 */
  float gap_us;                 /* CW longer than this separates two commands; 400 (> TRcal = 200 us) */
  float lead_us;                /* CW kept in front of a segment's first command; 300 (< gap_us) */
  int32_t min_pulses;           /* bursts with fewer low pulses are not commands; 6 (gate_impl.cc:164) */
  int32_t commands_per_segment; /* 2: one RN16 window + one EPC window */
  int32_t reserved[3];
} rfid_b200_segmenter;

RFID_B200_API void rfid_b200_default_segmenter(rfid_b200_segmenter* sp);

/* Segment table of a capture that is already in device memory.  sp may be NULL (defaults).
 * h_segs: HOST array of `capacity` entries; *nseg receives the number of segments (also when
 * RFID_B200_ECAPACITY is returned).  Runs on `stream` and synchronises it. */
RFID_B200_API int rfid_b200_segment_capture(rfid_b200_ctx* ctx, const float* d_iq, size_t n_raw,
                                            const rfid_b200_segmenter* sp, rfid_b200_segment* h_segs,
                                            int capacity, int* nseg, void* stream);

/* File-to-records ingest, HOST pointers: uploads the capture in 16 MiB slices (pageable memory
 * through two pinned staging buffers, registered/pinned memory directly) with the threshold
 * pass of the segmenter running behind each slice, builds the segment table, decodes it and
 * copies table, records and counts back.  h_results holds seg_capacity*max_windows_per_segment
 * records, h_counts seg_capacity ints. */
RFID_B200_API int rfid_b200_ingest_capture_host(rfid_b200_ctx* ctx, const float* h_iq, size_t n_raw,
                                                const rfid_b200_segmenter* sp, int max_windows_per_segment,
                                                rfid_b200_segment* h_segs, int seg_capacity, int* nseg,
                                                rfid_b200_window_result* h_results, int32_t* h_counts);

/* ---------------- reader TX synthesiser + closed-loop slot simulator (SURVEY.md section 8f, rank 1) ----------------
 * The reader block's PIE command waveforms (reader_impl.cc:51-125 tables, :237-372 what every
 * Gen2-logic state emits, :383-443 CRC-5) generated on the GPU, sample for sample identical to
 * what reader_impl::general_work writes to its output port (float 0.0/1.0 at the DAC rate). */
enum {
  RFID_B200_TX_START = 0,        /* START: carrier before the first Query          (reader_impl.cc:237-243) */
  RFID_B200_TX_QUERY = 1,        /* SEND_QUERY: preamble + Query + carrier         (:265-285) */
  RFID_B200_TX_QUERY_REP = 2,    /* SEND_QUERY_REP                                 (:330-344) */
  RFID_B200_TX_ACK = 3,          /* SEND_ACK: frame-sync + 01 + RN16 (arg)         (:290-320) */
  RFID_B200_TX_CW = 4,           /* SEND_CW: carrier during the EPC reply          (:322-328) */
  RFID_B200_TX_NAK = 5,          /* SEND_NAK_Q / SEND_NAK_QR                       (:245-263) */
  RFID_B200_TX_POWER_DOWN = 6,   /* POWER_DOWN                                     (:228-235) */
  RFID_B200_TX_QUERY_ADJUST = 7  /* SEND_QUERY_ADJUST                              (:346-366) */
};
typedef struct rfid_b200_tx_command {
  int32_t kind; /* RFID_B200_TX_* */
  int32_t arg;  /* ACK: the 16-bit RN16 to echo */
} rfid_b200_tx_command;

/* Waveform of a script of emissions, written to d_out (device, `capacity` floats).  *n_samples
 * receives the total length (also on RFID_B200_ECAPACITY); d_out may be NULL to query it. */
RFID_B200_API int rfid_b200_tx_synth(rfid_b200_ctx* ctx, const rfid_b200_tx_command* h_script, int n_commands,
                                     int dac_rate, float* d_out, size_t capacity, size_t* n_samples, void* stream);

/* Inventory-slot simulator: one segment = one slot = carrier, Query (slot 0 of a round) or QueryRep,
 * RN16 replies of the tags that picked this slot, ACK, EPC reply, carrier.  Signal model (SURVEY.md 8d,
 * calibrated on misc/data/file_source_test): rx = (L + sum_k g_k b_k[n]) * env[n] + w[n], env = the
 * reader waveform above held to the ADC rate and shaped by the measured TX/RX edge response, b_k = FM0
 * half-symbol levels (TAG_PREAMBLE, data, dummy 1) at BLF 40 kHz starting T1 after the command.
 * closed_loop != 0: the first part of every slot is generated and decoded by this context's receive
 * chain, the ACK echoes the RN16 that was decoded, and only a tag whose RN16 matches sends its EPC
 * (collided or empty slots therefore end in silence, as with a real reader); closed_loop == 0: the ACK
 * echoes the strongest tag's RN16.  All randomness is counter-based: segment i of the global numbering is
 * the same whichever rank generates it. */
typedef struct rfid_b200_sim_params {
  uint64_t seed;
  int32_t n_tags;      /* tags in the field (0..16); each draws a slot per inventory round */
  int32_t closed_loop;
  int32_t dac_rate;    /* reader TX rate (apps/reader.py:56 -> 1000000); adc_rate must be a multiple */
  float segment_us;    /* slot length (8480 = the recording's round period) */
  float lead_us;       /* carrier before the first command (400) */
  float noise_sigma;   /* per component (0.0030) */
  float tag_gain;      /* |g| (0.0227) */
  float tag_phase;     /* arg g, rad */
  float clock_pct;     /* tag clock tolerance, percent (0.8) */
  float leak_re, leak_im; /* carrier leakage (0.2846, -0.0349) */
  float floor_level;   /* envelope inside a low pulse (0.004) */
  int32_t reserved[2];
} rfid_b200_sim_params;

typedef struct rfid_b200_sim_truth {
  int32_t is_query;       /* 1: the slot starts with a Query, 0: QueryRep */
  int32_t n_replies;      /* tags that answered with an RN16 */
  int32_t strongest_rn16; /* RN16 of the strongest of them, -1: empty slot */
  int32_t acked_rn16;     /* RN16 in the ACK (closed loop: what the receive chain decoded), -1: no ACK sent */
  int32_t replier;        /* tag that sent its EPC, -1: none */
  int32_t reserved[3];
  uint8_t epc[16];        /* PC + EPC + CRC-16 it sent (zeros if none) */
} rfid_b200_sim_truth;

RFID_B200_API void rfid_b200_default_sim(rfid_b200_sim_params* p);
/* raw samples per segment for these settings (negative: error) */
RFID_B200_API int rfid_b200_sim_segment_length(const rfid_b200_ctx* ctx, const rfid_b200_sim_params* p);
/* Generate segments [first_segment, first_segment + nseg) into d_iq (device, nseg * segment_length
 * complex64), with their segment table (device, offsets relative to d_iq) and ground truth (device, may
 * be NULL).  Asynchronous on `stream` except for buffer growth. */
RFID_B200_API int rfid_b200_sim_capture(rfid_b200_ctx* ctx, const rfid_b200_sim_params* p, int64_t first_segment,
                                        int nseg, float* d_iq, rfid_b200_segment* d_segs,
                                        rfid_b200_sim_truth* d_truth, void* stream);

/* ---------------- block mode (GNU Radio drop-in) ----------------
 * Called from the thin host blocks' general_work(); HOST pointers, owned by the
 * scheduler, touched only during the call.  State lives in the context (device
 * memory) between calls. */

/* gate_impl::general_work (gate_impl.cc:85-200).  seek: 0 = none, 1 = the Gen2
 * logic asked for an RN16 window, 2 = for an EPC window since the previous call
 * (reader_state->gate_status SEEK flags, gate_impl.cc:112-123).  Returns through
 * *consumed / *written the values the reference passes to consume_each() and
 * returns; *closed = 1 when a window completed inside this call.  magn2_out
 * (may be NULL) receives |out|^2 per written sample (reader_state->magn_squared_samples). */
RFID_B200_API int rfid_b200_gate_work(rfid_b200_ctx* ctx, int seek, const float* in, int n_in, float* out,
                                      int out_capacity, int* consumed, int* written, int* closed,
                                      float* magn2_out);

/* tag_decoder_impl::general_work on one complete window (tag_decoder_impl.cc:223-393):
 * win = n complex samples (n >= window length of `kind`), result in *res.
 * bits_out (may be NULL): 16 (RN16) or 128 (EPC) floats in {0.,1.} exactly as the
 * reference writes them to stream port 0 (tag_decoder_impl.cc:261-266). */
RFID_B200_API int rfid_b200_decoder_work(rfid_b200_ctx* ctx, int kind, const float* win, int n,
                                         rfid_b200_window_result* res, float* bits_out);

/* fir_filter_ccc(decim,[1]*ntaps) replacement (apps/reader.py:75): canonical
 * boxcar + decimation with ntaps-1 samples of history kept in the context.
 * Writes floor((n_in + carry)/decim) outputs. */
RFID_B200_API int rfid_b200_mf_work(rfid_b200_ctx* ctx, const float* in, int n_in, float* out, int out_capacity,
                                    int* written);

#ifdef __cplusplus
}
#endif
#endif /* RFID_B200_H */
