// rfid_b200.cu -- C-ABI of the B200-native Gen2 receive chain (see include/rfid_b200.h).
// Host side: context, configuration derivation, launches, host<->device marshalling,
// READER_STATS reduction.  There is no CPU implementation of the signal path in this
// library: every entry point that produces samples or decisions launches a kernel.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <new>
#include <string>
#include <vector>

#include "rx_block.cuh"
#include "rx_common.cuh"
#include "rx_fused.cuh"
#include "rx_fused_split.cuh"
#include "rx_ingest.cuh"
#include "rx_pack.cuh"
#include "tx_synth.cuh"

using namespace rfid_b200;

struct rfid_b200_ctx {
  rfid_b200_params params;
  RxConfig cfg;
  int device;
  cudaStream_t stream;  // own stream for block mode / host-mode capture calls
  cudaStream_t copy_stream;  // host-mode capture calls: uploads of the next slice run beside the decode of this one
  cudaEvent_t ev_slice[4];
  std::string last_error;
  // capture mode
  FusedArgs layout;     // shared-memory carve-up (pointers filled per call)
  float* window_tap;
  int last_launches;
  bool timing;
  unsigned long long* d_stamps;      // kernel timing: kStampSlots launch slots {earliest CTA start, latest CTA end} (ns)
  int stamp_next;                    // slots taken since the last drain
  cudaStream_t stamp_stream;         // stream of the last timed launch
  unsigned long long last_end_ns;    // end stamp of the last drained launch
  double kernel_ms;
  int kernel_launches;
  int sm_count;
  int pack_g_override;  // RFID_B200_PACK_G (developer aid): segments per CTA of the pack kernel, 0 = automatic
  bool pack_disabled;   // RFID_B200_KERNEL=split: keep the one-CTA-per-segment kernels for every configuration
  // host-mode staging buffers
  void* d_iq; size_t d_iq_bytes;
  void* d_segs; size_t d_segs_bytes;
  void* d_res; size_t d_res_bytes;
  void* d_cnt; size_t d_cnt_bytes;
  void* d_win; size_t d_win_bytes;  // per-segment window scratch of the one-CTA-per-segment kernels
  void* d_yhist;                     // rx_pack_kernel: y history, [%nsmid][kPMaxSeg][kYW] float2
  cudaEvent_t ev_hist;               // hist_stream's work, recorded when a launch moves to another stream
  cudaStream_t hist_stream;          // stream of the last rx_pack_kernel launch
  bool hist_used;
  // block mode
  GateState* d_gate;
  GateCallOut* d_gate_out;
  void* d_in; size_t d_in_bytes;
  void* d_out; size_t d_out_bytes;
  void* d_m2; size_t d_m2_bytes;
  void* d_blk; size_t d_blk_bytes;   // block mode: [GateCallOut | out samples | |out|^2] in one block -> ONE D2H per work call
  void* h_blk; size_t h_blk_bytes;   // its pinned host mirror
  rfid_b200_window_result* d_one;
  // mf block mode
  void* d_mf; size_t d_mf_bytes; long long mf_abs0; long long mf_have; long long mf_next_n;
  // capture ingest (segmenter work buffers, pinned upload staging)
  void* d_mask; size_t d_mask_bytes;
  void* d_chunk; size_t d_chunk_bytes;  // chunk_last | prev_low | falls_before | chunk_falls
  void* d_bursts; size_t d_bursts_bytes;
  void* d_ing;  // level partials + totals
  void* h_stage[2]; cudaEvent_t ev_stage[2];
  std::vector<IngestBurst> h_bursts;
  // TX synthesiser / slot simulator
  void* d_script; size_t d_script_bytes;
  void* d_sim_res; size_t d_sim_res_bytes;
  void* d_sim_cnt; size_t d_sim_cnt_bytes;
};

namespace {

const char* kErrNames[] = {"ok", "invalid argument", "no usable sm_100 CUDA device", "out of memory", "CUDA runtime error",
                           "output buffer too small"};

int fail_cuda(rfid_b200_ctx* c, cudaError_t e, const char* what)
{
  if (c) c->last_error = std::string(what) + ": " + cudaGetErrorString(e);
  return RFID_B200_ECUDA;
}
#define CK(call)                                                   \
  do {                                                             \
    cudaError_t _e = (call);                                       \
    if (_e != cudaSuccess) return fail_cuda(ctx, _e, #call);       \
  } while (0)

int next_pow2(int v)
{
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

// Derived counts with the reference's own expression order and types
// (gate_impl.cc:48-53,115,121; tag_decoder_impl.cc:60,85,151-152; global_vars.h:110-111).
int derive_config(const rfid_b200_params& p, RxConfig& c)
{
  if (p.adc_rate <= 0 || p.decim <= 0 || p.ntaps <= 0 || p.fixed_q < 0 || p.fixed_q > 15) return RFID_B200_EINVAL;
  memset(&c, 0, sizeof(c));
  c.adc_rate = p.adc_rate; c.decim = p.decim; c.ntaps = p.ntaps;
  const int sample_rate = p.adc_rate / p.decim;  // apps/reader.py:76
  c.fs_dec = sample_rate;
  const float TAG_BIT_D = (float)(1.0 / kReaderFreq * std::pow(10, 6));
  c.n_T1 = (int)(kT1_D * (sample_rate / std::pow(10, 6)));
  c.n_PW = (int)(kPW_D * (sample_rate / std::pow(10, 6)));
  c.n_tag_bit_i = (int)(TAG_BIT_D * (sample_rate / std::pow(10, 6)));
  c.win_length = (int)(kWinSizeD * (sample_rate / std::pow(10, 6)));
  c.dc_length = (int)(kDcSizeD * (sample_rate / std::pow(10, 6)));
  c.n_tag_bit_f = (float)(TAG_BIT_D * sample_rate / std::pow(10, 6));
  c.len_epc = (kEPCBits + kTagPreambleBits) * c.n_tag_bit_i + 2 * c.n_tag_bit_i;
  c.len_rn16 = (kRN16Bits + kTagPreambleBits) * c.n_tag_bit_i + 2 * c.n_tag_bit_i;
  c.fixed_q = p.fixed_q; c.max_queries = p.max_queries; c.max_tags = p.max_tags;
  c.mf_q = p.ntaps / p.decim; c.mf_rem = p.ntaps % p.decim;
  int sr = 0;
  for (int i = 0; i < 1.5 * c.n_tag_bit_f; i++) sr++;  // tag_decoder_impl.cc:85
  c.sync_range = sr;
  const float n = c.n_tag_bit_f;
  c.t_min = (float)(n / 2.0 - n / 2.0 / 100);  // :151
  c.t_max = (float)(n / 2.0 + n / 2.0 / 100);  // :152
  // divisors for which RN(x/d) == fma(fma(-RN(x*c), d, x), c, RN(x*c)) holds for every binary32 x (exhaustive
  // check: tools/micro/verify_constdiv.c, run by tests/test_host_logic.py)
  static const int kVerifiedDivisors[] = {6, 24, 48, 50, 60, 96, 100, 125, 144, 192, 200, 300, 400};
  c.win_recip = 1.0f / (float)c.win_length;
  c.dc_recip = 1.0f / (float)c.dc_length;
  c.win_div_fast = c.dc_div_fast = 0;
  for (int d : kVerifiedDivisors) {
    if (d == c.win_length) c.win_div_fast = 1;
    if (d == c.dc_length) c.dc_div_fast = 1;
  }
  if (c.win_length < 1 || c.dc_length < 1 || c.n_tag_bit_i < 1 || c.win_length > kMaxWinLen || c.dc_length > kMaxDcLen)
    return RFID_B200_EINVAL;
  return RFID_B200_OK;
}

int align_up(int v, int a) { return (v + a - 1) / a * a; }

bool fast_path_ok(const RxConfig& c) { return c.win_length <= kTT && c.dc_length <= kTT; }

// smallest decoder stage for a window that is complete when the decode starts: the head (sync range + 6 symbols) and one
// chunk of the symbol-period search (one float per sample); the bit decisions and the rest of an RN16 window are read from
// global memory directly
int decode_stage_small(const RxConfig& c)
{
  const int head = c.sync_range + (int)(6.0f * c.n_tag_bit_f) + 2;
  const int span = (int)((float)kChunkSteps * c.t_max + 256.0f * (c.t_max - c.t_min)) + 8;
  int need = head > (span + 1) / 2 ? head : (span + 1) / 2;
  return align_up(need, 8);
}

// shared-memory carve-up of rx_fused_split_kernel: five tile stages forming one time-indexed ring
void make_layout_split(const RxConfig& c, FusedArgs& L)
{
  int off = 0;
  L.raw_stage_samples = c.decim * kTT + 2;
  L.off_raw = off; off = align_up(off + kRawStages * L.raw_stage_samples * 8, 16);
  L.bhist_size = next_pow2(kTT + c.mf_q + 2);
  L.off_bhist = off; off = align_up(off + L.bhist_size * 8 * (c.mf_rem ? 2 : 1), 16);
  L.off_tile_y = off; off += kRing * 8;
  L.off_tile_a = off; off += kRing * 4;
  L.off_tile_d = off; off += kRing * 4 + 64;          // + read-ahead pad of the running-sum loop
  L.off_etile = off; off += kS * 2 * kTT * 4 + 64;
  L.off_snap = off; off = align_up(off + c.dc_length * 8, 16);
  L.dstage_samples = decode_stage_samples(c.n_tag_bit_f);
  if (L.dstage_samples < c.len_rn16) L.dstage_samples = align_up(c.len_rn16, 8);  // an RN16 window is staged whole
  L.off_dstage = off; off = align_up(off + L.dstage_samples * 8, 16);
  L.ahist_size = L.ycl_size = 0;
  L.off_ahist = L.off_ycl = L.off_e = 0;
  L.rn16_pad = align_up(c.len_rn16, 16);
  L.win_stride = L.rn16_pad + align_up(c.len_epc, 16);
  L.smem_bytes = off;
}

void make_layout(const RxConfig& c, FusedArgs& L)
{
  if (fast_path_ok(c)) { make_layout_split(c, L); return; }
  const bool spec = false;
  int off = 0;
  L.raw_stage_samples = c.decim * kTT + 2;
  L.off_raw = off; off = align_up(off + kRawStages * L.raw_stage_samples * 8, 16);
  L.bhist_size = next_pow2(kTT + c.mf_q + 2);
  L.off_bhist = off; off = align_up(off + L.bhist_size * 8 * (c.mf_rem ? 2 : 1), 16);
  L.off_tile_y = off; off += kTileStages * kTT * 8;
  L.off_tile_a = off; off += kTileStages * kTT * 4;
  L.off_tile_d = off; off += kTileStages * kTT * 4 + 64;  // + read-ahead pad of the running-sum loop
  L.ahist_size = L.ycl_size = 0;
  L.off_ahist = L.off_ycl = L.off_e = L.off_etile = L.off_snap = 0;
  if (spec) {
    L.off_etile = off; off += kTileStages * 2 * kTT * 4 + 64;
    L.off_snap = off; off = align_up(off + c.dc_length * 8, 16);
  } else {
    L.ahist_size = next_pow2(kTT + c.win_length);
    L.off_ahist = off; off = align_up(off + L.ahist_size * 4, 16);
    L.ycl_size = next_pow2(kTT + c.dc_length);
    L.off_ycl = off; off = align_up(off + L.ycl_size * 8, 16);
    L.off_e = off; off += 2 * (kTT + 16) * 4;
  }
  // (long rings leave little shared memory: the decoder stages the window's head only and gathers the rest from L2)
  L.dstage_samples = align_up(c.sync_range + (int)(6.0f * c.n_tag_bit_f) + 2, 8);
  L.off_dstage = off; off = align_up(off + L.dstage_samples * 8, 16);
  L.rn16_pad = align_up(c.len_rn16, 16);
  L.win_stride = L.rn16_pad + align_up(c.len_epc, 16);
  L.smem_bytes = off;
}

// number of SM identifiers (%smid < %nsmid; may exceed the SM count)
__global__ void query_nsmid_kernel(unsigned* out)
{
  unsigned n;
  asm("mov.u32 %0, %%nsmid;" : "=r"(n));
  *out = n;
}

// rx_pack_kernel serves the reference configuration (block-sum matched filter with 5 blocks of 5, rings inside a tile);
// its y history must hold a whole EPC window plus the tiles warps A / B / C may be apart, and at most kPTrig windows can
// open within one tile
bool pack_ok(const RxConfig& c)
{
  return c.decim == 5 && c.mf_rem == 0 && c.mf_q == 5 && fast_path_ok(c) && c.len_rn16 >= kT2 / 2 &&
         c.len_epc + c.dc_length + 8 * kT2 <= kYW && ((c.win_length | c.dc_length) & 3) == 0 && c.dc_length <= 124 && c.win_length <= kT2 && c.n_T1 + 1 >= 32;
}

// shared-memory carve-up of rx_pack_kernel for G segments per CTA
void make_layout_pack(const RxConfig& c, int G, PackArgs& L)
{
  L.G = G;
  L.raw_stage_samples = c.decim * kTT + 2;
  int o = 0;
  L.o_raw = o; o = align_up(o + 2 * L.raw_stage_samples * 8, 16);
  L.o_tail_y = o; o = align_up(o + 2 * c.dc_length * 8, 16);
  L.o_ring_a = o; o += kRingA * 4;
  // decode stage: an RN16 window is staged whole; an EPC window needs its head and one chunk of the period search
  L.dstage_samples = decode_stage_small(c);
  if (L.dstage_samples < c.len_rn16) L.dstage_samples = align_up(c.len_rn16, 8);
  L.o_dstage = o; o = align_up(o + L.dstage_samples * 8, 16);
  L.seg_bytes = o;
  int off = 0;
  L.off_dA = off; off += kPAS * G * kPChainBuf * 4;
  L.off_dD = off; off += kPDS * 2 * G * kPChainBuf * 4;
  L.off_seg = align_up(off, 16);
  L.smem_bytes = L.off_seg + G * L.seg_bytes;
  if (L.smem_bytes < kPackMinSmem) L.smem_bytes = kPackMinSmem;   // one CTA per SM: the y history is indexed by the SM
}

int pack_segments_per_cta(const rfid_b200_ctx* ctx, int nseg);

typedef void (*fused_fn)(const FusedArgs);
fused_fn pick_kernel(const RxConfig& c)
{
  if (c.decim != 5) return nullptr;
  if (fast_path_ok(c)) {
    if (c.mf_rem == 0 && c.mf_q == 5) return rx_fused_split_kernel<5, 5>;  // the reference configuration: 25 taps
    return rx_fused_split_kernel<5, 0>;
  }
  return rx_fused_kernel<5, 0>;  // long rings (raw rates above 5 MS/s) and any tap count
}

int grow(rfid_b200_ctx* ctx, void** p, size_t* have, size_t need)
{
  if (*have >= need) return RFID_B200_OK;
  if (*p) cudaFree(*p);
  *p = nullptr; *have = 0;
  size_t want = need + need / 4 + 256;
  cudaError_t e = cudaMalloc(p, want);
  if (e != cudaSuccess) { ctx->last_error = "cudaMalloc failed"; cudaGetLastError(); return RFID_B200_ENOMEM; }
  *have = want;
  return RFID_B200_OK;
}

// Segments per CTA of rx_pack_kernel: as few CTAs as fill the device once (one CTA per SM, every SM busy for the
// whole launch); larger batches run kPMaxSeg per CTA in several waves.
int pack_segments_per_cta(const rfid_b200_ctx* ctx, int nseg)
{
  if (ctx->pack_g_override > 0) return ctx->pack_g_override;
  const int sms = ctx->sm_count > 0 ? ctx->sm_count : 148;
  int g = (nseg + sms - 1) / sms;
  if (g < 1) g = 1;
  if (g > kPMaxSeg) g = kPMaxSeg;
  return g;
}

constexpr int kStampSlots = 256;  // timed launches between two drains (a full table is drained before the next launch)

// every slot back to {~0, 0}: stamp_cta_start keeps the minimum, stamp_warp_end the maximum
cudaError_t reset_stamps(rfid_b200_ctx* ctx)
{
  const size_t slot = 2 * sizeof(unsigned long long);
  cudaError_t e = cudaMemsetAsync(ctx->d_stamps, 0xFF, kStampSlots * slot, ctx->stream);
  if (e == cudaSuccess) e = cudaMemset2DAsync(ctx->d_stamps + 1, slot, 0, sizeof(unsigned long long), kStampSlots, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  return e;
}

// Adds the launches stamped since the last drain to kernel_ms / kernel_launches and frees their slots.  A launch counts
// the device time it adds to the sequence, end - max(start, previous end): its duration when launches do not overlap,
// less the part that ran beside the previous launch when they do.
int drain_timing(rfid_b200_ctx* ctx)
{
  if (ctx->stamp_next == 0) return RFID_B200_OK;
  std::vector<unsigned long long> h(2 * (size_t)ctx->stamp_next);
  CK(cudaMemcpyAsync(h.data(), ctx->d_stamps, h.size() * sizeof(h[0]), cudaMemcpyDeviceToHost, ctx->stamp_stream));
  CK(cudaStreamSynchronize(ctx->stamp_stream));
  for (int i = 0; i < ctx->stamp_next; i++) {
    const unsigned long long start = h[2 * i], end = h[2 * i + 1];
    if (end == 0) continue;  // the launch failed
    const unsigned long long from = std::max(start, ctx->last_end_ns);
    if (end > from) ctx->kernel_ms += (double)(end - from) * 1e-6;
    ctx->last_end_ns = std::max(ctx->last_end_ns, end);
    ctx->kernel_launches++;
  }
  ctx->stamp_next = 0;
  CK(reset_stamps(ctx));
  return RFID_B200_OK;
}

}  // namespace

extern "C" {

int rfid_b200_abi_version(void) { return RFID_B200_ABI_VERSION; }

const char* rfid_b200_strerror(int code)
{
  int k = -code;
  if (k < 0 || k > 5) return "unknown error";
  return kErrNames[k];
}

const char* rfid_b200_last_cuda_error(const rfid_b200_ctx* ctx) { return ctx ? ctx->last_error.c_str() : ""; }

void rfid_b200_default_params(rfid_b200_params* p)
{
  if (!p) return;
  p->adc_rate = 2000000;  // apps/reader.py:53
  p->decim = 5;           // apps/reader.py:54
  p->ntaps = 25;          // apps/reader.py:65
  p->fixed_q = 0;         // global_vars.h:72
  p->max_queries = 1000;  // global_vars.h:76
  p->max_tags = 100;      // global_vars.h:100
  p->device = 0;
  p->reserved = 0;
}

int rfid_b200_create(const rfid_b200_params* p, rfid_b200_ctx** out)
{
  if (!p || !out) return RFID_B200_EINVAL;
  *out = nullptr;
  RxConfig cfg;
  int rc = derive_config(*p, cfg);
  if (rc) return rc;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || p->device < 0 || p->device >= ndev) { cudaGetLastError(); return RFID_B200_ENODEV; }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, p->device) != cudaSuccess || prop.major != 10) { cudaGetLastError(); return RFID_B200_ENODEV; }
  rfid_b200_ctx* ctx = new (std::nothrow) rfid_b200_ctx();
  if (!ctx) return RFID_B200_ENOMEM;
  ctx->params = *p; ctx->cfg = cfg; ctx->device = p->device;
  ctx->window_tap = nullptr; ctx->last_launches = 0; ctx->timing = false; ctx->kernel_ms = 0.0; ctx->kernel_launches = 0;
  ctx->d_stamps = nullptr; ctx->stamp_next = 0; ctx->stamp_stream = nullptr; ctx->last_end_ns = 0;
  ctx->d_iq = ctx->d_segs = ctx->d_res = ctx->d_cnt = ctx->d_in = ctx->d_out = ctx->d_m2 = ctx->d_mf = nullptr;
  ctx->d_win = nullptr; ctx->d_win_bytes = 0;
  ctx->d_yhist = nullptr;
  ctx->ev_hist = nullptr; ctx->hist_stream = nullptr; ctx->hist_used = false;
  ctx->d_blk = nullptr; ctx->d_blk_bytes = 0; ctx->h_blk = nullptr; ctx->h_blk_bytes = 0;
  ctx->d_iq_bytes = ctx->d_segs_bytes = ctx->d_res_bytes = ctx->d_cnt_bytes = ctx->d_in_bytes = ctx->d_out_bytes = ctx->d_m2_bytes = ctx->d_mf_bytes = 0;
  ctx->d_gate = nullptr; ctx->d_gate_out = nullptr; ctx->d_one = nullptr;
  ctx->mf_abs0 = 0; ctx->mf_have = 0; ctx->mf_next_n = 0;
  ctx->d_mask = ctx->d_chunk = ctx->d_bursts = ctx->d_ing = nullptr;
  ctx->d_mask_bytes = ctx->d_chunk_bytes = ctx->d_bursts_bytes = 0;
  ctx->d_script = ctx->d_sim_res = ctx->d_sim_cnt = nullptr;
  ctx->d_script_bytes = ctx->d_sim_res_bytes = ctx->d_sim_cnt_bytes = 0;
  ctx->h_stage[0] = ctx->h_stage[1] = nullptr; ctx->ev_stage[0] = ctx->ev_stage[1] = nullptr;
  memset(&ctx->layout, 0, sizeof(ctx->layout));
  make_layout(cfg, ctx->layout);
  cudaError_t e = cudaSetDevice(p->device);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
  ctx->copy_stream = nullptr;
  for (int k = 0; k < 4; k++) ctx->ev_slice[k] = nullptr;
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
  for (int k = 0; k < 4 && e == cudaSuccess; k++) e = cudaEventCreateWithFlags(&ctx->ev_slice[k], cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaMalloc((void**)&ctx->d_gate, sizeof(GateState));
  if (e == cudaSuccess) e = cudaMalloc((void**)&ctx->d_gate_out, sizeof(GateCallOut));
  if (e == cudaSuccess) e = cudaMalloc((void**)&ctx->d_one, sizeof(rfid_b200_window_result));
  if (e == cudaSuccess) e = cudaMemsetAsync(ctx->d_gate, 0, sizeof(GateState), ctx->stream);
  if (e == cudaSuccess) {
    // gate_impl ctor (gate_impl.cc:45) + initialize_reader_state (global_vars.cc:47): NEG_EDGE, first SEEK = RN16
    GateState init;
    memset(&init, 0, sizeof(init));
    init.to_ungate = cfg.len_rn16;
    e = cudaMemcpyAsync(ctx->d_gate, &init, offsetof(GateState, win_samples), cudaMemcpyHostToDevice, ctx->stream);
  }
  if (e == cudaSuccess) e = cudaMalloc((void**)&ctx->d_stamps, kStampSlots * 2 * sizeof(unsigned long long));
  if (e == cudaSuccess) e = reset_stamps(ctx);
  ctx->sm_count = prop.multiProcessorCount;
  {
    const char* ev = getenv("RFID_B200_PACK_G");
    ctx->pack_g_override = ev ? atoi(ev) : 0;
    if (ctx->pack_g_override < 0 || ctx->pack_g_override > kPMaxSeg) ctx->pack_g_override = 0;
    const char* kv = getenv("RFID_B200_KERNEL");
    ctx->pack_disabled = kv && strcmp(kv, "split") == 0;
  }
  if (e == cudaSuccess && pack_ok(cfg)) {
    // the y history of rx_pack_kernel: one region per SM identifier
    unsigned nsmid = 0, *d_n = nullptr;
    e = cudaMalloc(&d_n, sizeof(unsigned));
    if (e == cudaSuccess) {
      query_nsmid_kernel<<<1, 1, 0, ctx->stream>>>(d_n);
      e = cudaMemcpyAsync(&nsmid, d_n, sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
      cudaFree(d_n);
    }
    if (e == cudaSuccess && nsmid < (unsigned)prop.multiProcessorCount) nsmid = prop.multiProcessorCount;
    if (e == cudaSuccess) e = cudaMalloc(&ctx->d_yhist, (size_t)nsmid * kPMaxSeg * kYW * sizeof(float2));
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_hist, cudaEventDisableTiming);
  }
  if (e == cudaSuccess && pack_ok(cfg)) {
    PackArgs pl;
    make_layout_pack(cfg, kPMaxSeg, pl);
    e = cudaFuncSetAttribute((const void*)rx_pack_kernel<5, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, pl.smem_bytes);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute((const void*)rx_pack_kernel<5, 5>, cudaFuncAttributePreferredSharedMemoryCarveout,
                               cudaSharedmemCarveoutMaxShared);
  }
  fused_fn fn = pick_kernel(cfg);
  if (e == cudaSuccess && fn)
    e = cudaFuncSetAttribute((const void*)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx->layout.smem_bytes);
  if (e == cudaSuccess && fn)
    e = cudaFuncSetAttribute((const void*)fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute((const void*)decode_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             cfg.len_epc * 12 + 64);
  if (e != cudaSuccess) {
    cudaGetLastError();
    rfid_b200_destroy(ctx);
    return RFID_B200_ECUDA;
  }
  *out = ctx;
  return RFID_B200_OK;
}

void rfid_b200_destroy(rfid_b200_ctx* ctx)
{
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->h_blk) cudaFreeHost(ctx->h_blk);
  void* ptrs[] = {ctx->d_stamps, ctx->d_blk, ctx->d_win, ctx->d_yhist, ctx->d_iq, ctx->d_segs, ctx->d_res, ctx->d_cnt, ctx->d_in, ctx->d_out, ctx->d_m2, ctx->d_mf,
                  ctx->d_gate, ctx->d_gate_out, ctx->d_one, ctx->d_mask, ctx->d_chunk, ctx->d_bursts, ctx->d_ing,
                  ctx->d_script, ctx->d_sim_res, ctx->d_sim_cnt};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  for (int b = 0; b < 2; b++) {
    if (ctx->h_stage[b]) cudaFreeHost(ctx->h_stage[b]);
    if (ctx->ev_stage[b]) cudaEventDestroy(ctx->ev_stage[b]);
  }
  for (int k = 0; k < 4; k++) if (ctx->ev_slice[k]) cudaEventDestroy(ctx->ev_slice[k]);
  if (ctx->ev_hist) cudaEventDestroy(ctx->ev_hist);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

int rfid_b200_window_length(const rfid_b200_ctx* ctx, int kind)
{
  if (!ctx) return RFID_B200_EINVAL;
  return kind == RFID_B200_RN16 ? ctx->cfg.len_rn16 : ctx->cfg.len_epc;
}

int rfid_b200_fs_dec(const rfid_b200_ctx* ctx) { return ctx ? ctx->cfg.fs_dec : RFID_B200_EINVAL; }

int rfid_b200_set_window_tap(rfid_b200_ctx* ctx, float* d_windows)
{
  if (!ctx) return RFID_B200_EINVAL;
  ctx->window_tap = d_windows;
  return RFID_B200_OK;
}

int rfid_b200_enable_kernel_timing(rfid_b200_ctx* ctx, int on)
{
  if (!ctx) return RFID_B200_EINVAL;
  ctx->timing = on != 0;
  return RFID_B200_OK;
}

int rfid_b200_kernel_time(rfid_b200_ctx* ctx, int reset, float* ms_total, int* launches)
{
  if (!ctx) return RFID_B200_EINVAL;
  CK(cudaSetDevice(ctx->device));
  const int rc = drain_timing(ctx);
  if (rc) return rc;
  if (ms_total) *ms_total = (float)ctx->kernel_ms;
  if (launches) *launches = ctx->kernel_launches;
  if (reset) { ctx->kernel_ms = 0.0; ctx->kernel_launches = 0; }
  return RFID_B200_OK;
}

int rfid_b200_last_launch_count(const rfid_b200_ctx* ctx) { return ctx ? ctx->last_launches : RFID_B200_EINVAL; }

static int decode_capture_impl(rfid_b200_ctx* ctx, const float* d_iq, size_t n_raw, const rfid_b200_segment* d_segs, int nseg,
                               int max_windows_per_segment, rfid_b200_window_result* d_results, int32_t* d_counts,
                               void* stream, int seg_base);

int rfid_b200_decode_capture(rfid_b200_ctx* ctx, const float* d_iq, size_t n_raw, const rfid_b200_segment* d_segs, int nseg,
                             int max_windows_per_segment, rfid_b200_window_result* d_results, int32_t* d_counts,
                             void* stream)
{
  return decode_capture_impl(ctx, d_iq, n_raw, d_segs, nseg, max_windows_per_segment, d_results, d_counts, stream, 0);
}

static int decode_capture_impl(rfid_b200_ctx* ctx, const float* d_iq, size_t n_raw, const rfid_b200_segment* d_segs, int nseg,
                               int max_windows_per_segment, rfid_b200_window_result* d_results, int32_t* d_counts,
                               void* stream, int seg_base)
{
  if (!ctx || !d_iq || !d_segs || !d_results || !d_counts || nseg < 0 || max_windows_per_segment < 1) return RFID_B200_EINVAL;
  if ((reinterpret_cast<uintptr_t>(d_iq) & 15u) != 0) return RFID_B200_EINVAL;  // TMA bulk source alignment
  ctx->last_launches = 0;
  if (nseg == 0) return RFID_B200_OK;
  fused_fn fn = pick_kernel(ctx->cfg);
  if (!fn) { ctx->last_error = "capture mode supports decim = 5 only in this build"; return RFID_B200_EINVAL; }
  CK(cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)stream;  // NULL = the (legacy) default stream, as documented
  FusedArgs A = ctx->layout;
  const bool use_pack = pack_ok(ctx->cfg) && !ctx->pack_disabled;
  if (!use_pack) {
    // window scratch: one RN16 + one EPC window per segment (grown on demand; cudaMalloc synchronises, so a
    // caller that wants a fully asynchronous call sizes the context once with its largest batch)
    int rc = grow(ctx, &ctx->d_win, &ctx->d_win_bytes, (size_t)nseg * A.win_stride * sizeof(float2));
    if (rc) return rc;
  }
  A.win_scratch = reinterpret_cast<float2*>(ctx->d_win);
  A.iq = reinterpret_cast<const float2*>(d_iq);
  A.n_raw = n_raw;
  A.segs = d_segs;
  A.nseg = nseg;
  A.seg_base = seg_base;
  A.max_windows = max_windows_per_segment;
  A.results = d_results;
  A.counts = d_counts;
  A.window_tap = reinterpret_cast<float2*>(ctx->window_tap);
  A.cfg = ctx->cfg;
  A.stamps = nullptr;
  if (ctx->timing) {
    if (ctx->stamp_next == kStampSlots) {
      int rc = drain_timing(ctx);
      if (rc) return rc;
    }
    A.stamps = ctx->d_stamps + 2 * ctx->stamp_next++;
    ctx->stamp_stream = s;
  }
  if (use_pack) {
    PackArgs P;
    memset(&P, 0, sizeof(P));
    make_layout_pack(ctx->cfg, pack_segments_per_cta(ctx, nseg), P);
    P.iq = A.iq; P.n_raw = A.n_raw; P.segs = A.segs; P.nseg = nseg; P.seg_base = seg_base; P.max_windows = A.max_windows;
    P.results = A.results; P.counts = A.counts; P.window_tap = A.window_tap; P.y_hist = reinterpret_cast<float2*>(ctx->d_yhist);
    P.stamps = A.stamps;
    P.cfg = ctx->cfg;
    // the y history belongs to one launch at a time: a launch on another stream than the previous one waits for everything
    // queued on that stream so far (on one stream, each launch completes after the one before it, see rx_pack.cuh)
    if (ctx->hist_used && ctx->hist_stream != s) {
      CK(cudaEventRecord(ctx->ev_hist, ctx->hist_stream));
      CK(cudaStreamWaitEvent(s, ctx->ev_hist, 0));
    }
    // programmatic dependent launch: scheduled while the previous kernel of the stream still runs (rx_pack.cuh)
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t lc;
    memset(&lc, 0, sizeof(lc));
    lc.gridDim = dim3((nseg + P.G - 1) / P.G);
    lc.blockDim = dim3(32 * (4 * P.G + 2));
    lc.dynamicSmemBytes = P.smem_bytes;
    lc.stream = s;
    lc.attrs = attr;
    lc.numAttrs = 1;
    CK(cudaLaunchKernelEx(&lc, rx_pack_kernel<5, 5>, P));
    ctx->hist_stream = s; ctx->hist_used = true;
  } else {
    fn<<<nseg, fast_path_ok(ctx->cfg) ? kSplitThreads : kFusedThreads, A.smem_bytes, s>>>(A);
  }
  CK(cudaGetLastError());
  ctx->last_launches = 1;
  return RFID_B200_OK;
}

int rfid_b200_decode_capture_host(rfid_b200_ctx* ctx, const float* h_iq, size_t n_raw, const rfid_b200_segment* h_segs,
                                  int nseg, int max_windows_per_segment, rfid_b200_window_result* h_results,
                                  int32_t* h_counts)
{
  if (!ctx || !h_iq || !h_segs || !h_results || !h_counts || nseg < 0 || max_windows_per_segment < 1) return RFID_B200_EINVAL;
  if (nseg == 0) return RFID_B200_OK;
  CK(cudaSetDevice(ctx->device));
  int rc;
  const size_t res_bytes = (size_t)nseg * max_windows_per_segment * sizeof(rfid_b200_window_result);
  if ((rc = grow(ctx, &ctx->d_iq, &ctx->d_iq_bytes, n_raw * 8 + 16))) return rc;
  if ((rc = grow(ctx, &ctx->d_segs, &ctx->d_segs_bytes, (size_t)nseg * sizeof(rfid_b200_segment)))) return rc;
  if ((rc = grow(ctx, &ctx->d_res, &ctx->d_res_bytes, res_bytes))) return rc;
  if ((rc = grow(ctx, &ctx->d_cnt, &ctx->d_cnt_bytes, (size_t)nseg * 4))) return rc;
  cudaStream_t s = ctx->stream;
  CK(cudaMemcpyAsync(ctx->d_segs, h_segs, (size_t)nseg * sizeof(rfid_b200_segment), cudaMemcpyHostToDevice, s));
  CK(cudaMemsetAsync(ctx->d_res, 0, res_bytes, s));
  // Pinned source: the call is a pipeline over slices of the segment table -- upload of slice k+1 (copy stream) beside the
  // decode of slice k and the download of slice k-1's records (compute stream).  The call as a whole is bound by the
  // host -> device link (8 B per sample); the pipeline takes the decode and the record download off its tail.
  // Pageable source: one plain copy (the driver stages it synchronously anyway).
  cudaPointerAttributes attr;
  const bool pinned = cudaPointerGetAttributes(&attr, h_iq) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  cudaGetLastError();
  const int n_slices = (pinned && nseg >= 64) ? 4 : 1;
  if (n_slices == 1) CK(cudaMemcpyAsync(ctx->d_iq, h_iq, n_raw * 8, cudaMemcpyHostToDevice, s));
  int launches = 0;
  for (int k = 0; k < n_slices; k++) {
    const int b = (int)((long long)nseg * k / n_slices), e = (int)((long long)nseg * (k + 1) / n_slices);
    if (e <= b) continue;
    if (n_slices > 1) {
      unsigned long long lo = ~0ull, hi = 0;
      for (int i = b; i < e; i++) {
        const unsigned long long o = h_segs[i].offset, t = o + h_segs[i].length;
        if (o < lo) lo = o;
        if (t > hi) hi = t;
      }
      if (hi > n_raw) hi = n_raw;
      if (lo > hi) lo = hi;
      lo = lo >= 4 ? lo - 4 : 0;  // (the tile loader rounds a segment's first sample down to an even index)
      if (hi > lo) CK(cudaMemcpyAsync((char*)ctx->d_iq + lo * 8, (const char*)h_iq + lo * 8, (hi - lo) * 8, cudaMemcpyHostToDevice, ctx->copy_stream));
      CK(cudaEventRecord(ctx->ev_slice[k], ctx->copy_stream));
      CK(cudaStreamWaitEvent(s, ctx->ev_slice[k], 0));
    }
    rc = decode_capture_impl(ctx, (const float*)ctx->d_iq, n_raw, (const rfid_b200_segment*)ctx->d_segs + b, e - b,
                             max_windows_per_segment, (rfid_b200_window_result*)ctx->d_res + (size_t)b * max_windows_per_segment,
                             (int32_t*)ctx->d_cnt + b, s, b);
    if (rc) return rc;
    launches += ctx->last_launches;
    const size_t rb = (size_t)(e - b) * max_windows_per_segment * sizeof(rfid_b200_window_result);
    CK(cudaMemcpyAsync((char*)h_results + (size_t)b * max_windows_per_segment * sizeof(rfid_b200_window_result),
                       (char*)ctx->d_res + (size_t)b * max_windows_per_segment * sizeof(rfid_b200_window_result), rb,
                       cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(h_counts + b, (int32_t*)ctx->d_cnt + b, (size_t)(e - b) * 4, cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  ctx->last_launches = launches;
  return RFID_B200_OK;
}

// READER_STATS bookkeeping: tag_decoder_impl.cc:269-288 (RN16 too short), :295 (slot++ per EPC window),
// :329-365 (CRC ok), :366-387 (CRC fail), reader_impl.cc:259,336 (n_queries_sent), gate_impl.cc:101-109 (stop rule).
int rfid_b200_reduce_stats(const rfid_b200_ctx* ctx, const rfid_b200_window_result* recs, const int32_t* counts, int nseg,
                           int max_per_seg, int continuous, rfid_b200_stats* out)
{
  if (!ctx || !recs || !counts || !out || nseg < 0 || max_per_seg < 1) return RFID_B200_EINVAL;
  memset(out, 0, sizeof(*out));
  const int max_slot = 1 << ctx->cfg.fixed_q;
  out->max_slot_number = max_slot;
  std::map<int, int> tag_reads;   // what print_results() reports
  std::map<int, int> seg_reads;   // non-continuous mode: the tag_reads of the segment's own (fresh) reader_state
  int round = 1, slot = 1, nq = 1, total_q = 0;
  bool stopped = false;
  for (int s = 0; s < nseg; s++) {
    // an independent segment = a reference run with freshly constructed blocks: counters AND the unique-tag stop rule
    // (gate_impl.cc:101-104) start over; the global map only accumulates for reporting
    if (!continuous) { round = 1; slot = 1; nq = 1; stopped = false; seg_reads.clear(); }
    std::map<int, int>& rule_reads = continuous ? tag_reads : seg_reads;
    const int n = counts[s] < max_per_seg ? counts[s] : max_per_seg;
    const rfid_b200_window_result* r = recs + (size_t)s * max_per_seg;
    for (int k = 0; k < n && !stopped; k++) {
      bool next_query = false;
      if (r[k].kind == RFID_B200_RN16) {
        if (r[k].crc_ok == -2) {
          slot++;
          if (slot > max_slot) { slot = 1; round++; }
          next_query = true;
        }
      } else {
        slot++;
        if (slot > max_slot) { slot = 1; round++; }
        if (r[k].crc_ok == 1) {
          out->n_epc_correct++;
          tag_reads[r[k].tag_id]++;
          if (!continuous) seg_reads[r[k].tag_id]++;
        }
        next_query = true;
      }
      out->n_windows++;
      if (next_query) {
        nq++;
        if (nq > ctx->cfg.max_queries || (int)rule_reads.size() > ctx->cfg.max_tags) stopped = true;
      }
    }
    if (!continuous) total_q += nq;
  }
  out->n_queries_sent = continuous ? nq : total_q;
  out->cur_inventory_round = round;
  out->cur_slot_number = slot;
  out->terminated = stopped ? 1 : 0;
  out->n_unique_tags = (int)tag_reads.size();
  int k = 0;
  for (auto& kv : tag_reads) {
    if (k >= RFID_B200_MAX_TAGS) break;
    out->tag_id[k] = kv.first;
    out->tag_reads[k] = kv.second;
    k++;
  }
  return RFID_B200_OK;
}

// ------------------------------------------------------------------ capture ingest (SURVEY 8f-2)
}  // extern "C"

namespace {

constexpr size_t kUploadSamples = (size_t)1 << 21;  // 16 MiB per upload slice; multiple of kIngestChunk
constexpr size_t kLevelHead = (size_t)1 << 21;      // CW level is estimated on the head of the capture

struct SegmenterCfg {
  float level_frac;
  unsigned int gap, lead;
  int min_pulses, commands;
};

int resolve_segmenter(const rfid_b200_ctx* ctx, const rfid_b200_segmenter* sp, SegmenterCfg& o)
{
  rfid_b200_segmenter d;
  rfid_b200_default_segmenter(&d);
  if (sp) d = *sp;
  if (!(d.level_frac > 0.f && d.level_frac < 1.f) || !(d.gap_us > 0.f) || !(d.lead_us >= 0.f) || d.min_pulses < 1 ||
      d.commands_per_segment < 1)
    return RFID_B200_EINVAL;
  o.level_frac = d.level_frac;
  o.gap = (unsigned int)((double)d.gap_us * 1e-6 * ctx->cfg.adc_rate);
  o.lead = (unsigned int)((double)d.lead_us * 1e-6 * ctx->cfg.adc_rate);
  if (o.gap < 1) o.gap = 1;
  if (o.lead >= o.gap) return RFID_B200_EINVAL;  // a lead-in must not reach into the previous command
  o.min_pulses = d.min_pulses;
  o.commands = d.commands_per_segment;
  return RFID_B200_OK;
}

int ingest_alloc(rfid_b200_ctx* ctx, size_t n_raw, const SegmenterCfg& sc, long long& n_chunks, unsigned int& burst_cap)
{
  n_chunks = (long long)((n_raw + kIngestChunk - 1) / kIngestChunk);
  burst_cap = (unsigned int)(n_raw / sc.gap + 4);
  int rc;
  if ((rc = grow(ctx, &ctx->d_mask, &ctx->d_mask_bytes, (size_t)n_chunks * 32 * 4))) return rc;
  if ((rc = grow(ctx, &ctx->d_chunk, &ctx->d_chunk_bytes, (size_t)n_chunks * 28 + 64))) return rc;
  if ((rc = grow(ctx, &ctx->d_bursts, &ctx->d_bursts_bytes, (size_t)burst_cap * sizeof(IngestBurst)))) return rc;
  if (!ctx->d_ing) {
    if (cudaMalloc(&ctx->d_ing, kLevelBlocks * sizeof(double) + sizeof(IngestTotals)) != cudaSuccess) {
      cudaGetLastError();
      return RFID_B200_ENOMEM;
    }
  }
  return RFID_B200_OK;
}

struct IngestPtrs {
  double* partial; IngestTotals* tot;
  unsigned int* mask; long long* chunk_last; long long* prev_low; unsigned long long* falls_before; unsigned int* chunk_falls;
};

IngestPtrs ingest_ptrs(rfid_b200_ctx* ctx, long long n_chunks)
{
  IngestPtrs P;
  P.partial = reinterpret_cast<double*>(ctx->d_ing);
  P.tot = reinterpret_cast<IngestTotals*>(P.partial + kLevelBlocks);
  P.mask = reinterpret_cast<unsigned int*>(ctx->d_mask);
  P.chunk_last = reinterpret_cast<long long*>(ctx->d_chunk);
  P.prev_low = P.chunk_last + n_chunks;
  P.falls_before = reinterpret_cast<unsigned long long*>(P.prev_low + n_chunks);
  P.chunk_falls = reinterpret_cast<unsigned int*>(P.falls_before + n_chunks);
  return P;
}

int launch_level(rfid_b200_ctx* ctx, const float2* d_iq, size_t n_raw, const SegmenterCfg& sc, const IngestPtrs& P, cudaStream_t s)
{
  const unsigned long long n0 = n_raw < kLevelHead ? n_raw : kLevelHead;
  ingest_level_partial<<<kLevelBlocks, kLevelThreads, 0, s>>>(d_iq, n0, P.partial);
  ingest_level_final<<<1, 32, 0, s>>>(P.partial, n0, sc.level_frac, P.tot);
  CK(cudaGetLastError());
  ctx->last_launches += 2;
  return RFID_B200_OK;
}

int launch_mask(rfid_b200_ctx* ctx, const float2* d_iq, size_t n_raw, long long first_chunk, long long n, const IngestPtrs& P,
                cudaStream_t s)
{
  if (n <= 0) return RFID_B200_OK;
  long long blocks = (n + 7) / 8;
  if (blocks > 148 * 8) blocks = 148 * 8;
  ingest_mask<<<(unsigned)blocks, 256, 0, s>>>(d_iq, n_raw, first_chunk, n, P.tot, P.mask, P.chunk_last, P.chunk_falls);
  CK(cudaGetLastError());
  ctx->last_launches += 1;
  return RFID_B200_OK;
}

// scan + burst extraction + copy back; synchronises `s`
int finish_bursts(rfid_b200_ctx* ctx, long long n_chunks, unsigned int burst_cap, const SegmenterCfg& sc, const IngestPtrs& P,
                  cudaStream_t s, IngestTotals& tot)
{
  ingest_scan<<<1, 1024, 0, s>>>(n_chunks, P.chunk_last, P.chunk_falls, P.prev_low, P.falls_before, P.tot);
  long long blocks = (n_chunks + 7) / 8;
  if (blocks > 148 * 8) blocks = 148 * 8;
  ingest_bursts<<<(unsigned)blocks, 256, 0, s>>>(n_chunks, P.mask, P.prev_low, P.falls_before, sc.gap,
                                                 reinterpret_cast<IngestBurst*>(ctx->d_bursts), burst_cap, P.tot);
  CK(cudaGetLastError());
  ctx->last_launches += 2;
  CK(cudaMemcpyAsync(&tot, P.tot, sizeof(tot), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (tot.n_bursts > burst_cap) { ctx->last_error = "segmenter: burst list overflow"; return RFID_B200_ECAPACITY; }
  ctx->h_bursts.resize(tot.n_bursts);
  if (tot.n_bursts) {
    CK(cudaMemcpyAsync(ctx->h_bursts.data(), ctx->d_bursts, (size_t)tot.n_bursts * sizeof(IngestBurst), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
  }
  std::sort(ctx->h_bursts.begin(), ctx->h_bursts.end(), [](const IngestBurst& a, const IngestBurst& b) { return a.pos < b.pos; });
  return RFID_B200_OK;
}

// Pair commands into segments.  Segment j covers commands [j*C, (j+1)*C): it starts `lead` samples before its
// first command (rounded down to a multiple of decim so the matched filter keeps the capture's decimation
// phase; the first segment starts at sample 0 like the reference's continuous run) and runs up to the first
// pulse of the next segment's first command, i.e. consecutive segments overlap by the lead-in.
int build_segments(const rfid_b200_ctx* ctx, const std::vector<IngestBurst>& b, unsigned long long n_falls, size_t n_raw,
                   const SegmenterCfg& sc, rfid_b200_segment* out, int capacity, int* nseg)
{
  std::vector<unsigned long long> cmd;
  for (size_t k = 0; k < b.size(); k++) {
    const unsigned long long next_rank = k + 1 < b.size() ? b[k + 1].rank : n_falls;
    if (next_rank - b[k].rank >= (unsigned long long)sc.min_pulses) cmd.push_back(b[k].pos);
  }
  const size_t C = (size_t)sc.commands;
  const size_t ns = cmd.empty() ? (n_raw ? 1 : 0) : (cmd.size() + C - 1) / C;
  *nseg = (int)ns;
  if ((int)ns > capacity) return RFID_B200_ECAPACITY;
  const unsigned long long D = (unsigned long long)ctx->cfg.decim;
  for (size_t j = 0; j < ns; j++) {
    unsigned long long start = 0;
    if (j > 0) {
      const unsigned long long c0 = cmd[j * C];
      start = c0 > sc.lead ? c0 - sc.lead : 0;
      start -= start % D;
    }
    const unsigned long long end = (j + 1) * C < cmd.size() ? cmd[(j + 1) * C] : (unsigned long long)n_raw;
    if (end - start > 0xffffffffull) return RFID_B200_EINVAL;
    out[j].offset = start;
    out[j].length = (uint32_t)(end - start);
    out[j].reserved = 0;
  }
  return RFID_B200_OK;
}

}  // namespace

extern "C" {

void rfid_b200_default_segmenter(rfid_b200_segmenter* sp)
{
  if (!sp) return;
  memset(sp, 0, sizeof(*sp));
  sp->level_frac = 0.5f;
  sp->gap_us = 400.f;
  sp->lead_us = 300.f;
  sp->min_pulses = kNumPulsesCommand + 1;  // gate_impl.cc:164: num_pulses > NUM_PULSES_COMMAND
  sp->commands_per_segment = 2;            // RN16 window + EPC window
}

int rfid_b200_segment_capture(rfid_b200_ctx* ctx, const float* d_iq, size_t n_raw, const rfid_b200_segmenter* sp,
                              rfid_b200_segment* h_segs, int capacity, int* nseg, void* stream)
{
  if (!ctx || !d_iq || !h_segs || !nseg || capacity < 0) return RFID_B200_EINVAL;
  *nseg = 0;
  SegmenterCfg sc;
  int rc = resolve_segmenter(ctx, sp, sc);
  if (rc) return rc;
  if (n_raw == 0) return RFID_B200_OK;
  CK(cudaSetDevice(ctx->device));
  long long n_chunks;
  unsigned int burst_cap;
  if ((rc = ingest_alloc(ctx, n_raw, sc, n_chunks, burst_cap))) return rc;
  const IngestPtrs P = ingest_ptrs(ctx, n_chunks);
  cudaStream_t s = (cudaStream_t)stream;
  const float2* iq = reinterpret_cast<const float2*>(d_iq);
  ctx->last_launches = 0;
  if ((rc = launch_level(ctx, iq, n_raw, sc, P, s))) return rc;
  if ((rc = launch_mask(ctx, iq, n_raw, 0, n_chunks, P, s))) return rc;
  IngestTotals tot;
  if ((rc = finish_bursts(ctx, n_chunks, burst_cap, sc, P, s, tot))) return rc;
  return build_segments(ctx, ctx->h_bursts, tot.n_falls, n_raw, sc, h_segs, capacity, nseg);
}

int rfid_b200_ingest_capture_host(rfid_b200_ctx* ctx, const float* h_iq, size_t n_raw, const rfid_b200_segmenter* sp,
                                  int max_windows_per_segment, rfid_b200_segment* h_segs, int seg_capacity, int* nseg,
                                  rfid_b200_window_result* h_results, int32_t* h_counts)
{
  if (!ctx || !h_iq || !h_segs || !nseg || !h_results || !h_counts || seg_capacity < 0 || max_windows_per_segment < 1)
    return RFID_B200_EINVAL;
  *nseg = 0;
  SegmenterCfg sc;
  int rc = resolve_segmenter(ctx, sp, sc);
  if (rc) return rc;
  if (n_raw == 0) return RFID_B200_OK;
  if (!pick_kernel(ctx->cfg)) { ctx->last_error = "capture mode supports decim = 5 only in this build"; return RFID_B200_EINVAL; }
  CK(cudaSetDevice(ctx->device));
  long long n_chunks;
  unsigned int burst_cap;
  if ((rc = ingest_alloc(ctx, n_raw, sc, n_chunks, burst_cap))) return rc;
  if ((rc = grow(ctx, &ctx->d_iq, &ctx->d_iq_bytes, n_raw * 8 + 16))) return rc;
  const IngestPtrs P = ingest_ptrs(ctx, n_chunks);
  cudaStream_t s = ctx->stream;
  const float2* d_iq = reinterpret_cast<const float2*>(ctx->d_iq);

  // pageable sources go through two pinned staging slices so the host memcpy of slice k+1 overlaps the DMA of
  // slice k; pinned (registered) sources are DMA'd directly.  The threshold pass runs behind each slice.
  cudaPointerAttributes attr;
  bool pinned = cudaPointerGetAttributes(&attr, h_iq) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  cudaGetLastError();
  if (!pinned) {
    for (int b = 0; b < 2; b++) {
      if (!ctx->h_stage[b]) {
        if (cudaHostAlloc(&ctx->h_stage[b], kUploadSamples * 8, cudaHostAllocDefault) != cudaSuccess) {
          cudaGetLastError();
          return RFID_B200_ENOMEM;
        }
        CK(cudaEventCreateWithFlags(&ctx->ev_stage[b], cudaEventDisableTiming));
      }
    }
  }
  ctx->last_launches = 0;
  int launches = 0;
  size_t slice = 0;
  for (size_t off = 0; off < n_raw; off += kUploadSamples, slice++) {
    const size_t n = n_raw - off < kUploadSamples ? n_raw - off : kUploadSamples;
    const float* src = h_iq + 2 * off;
    if (!pinned) {
      const int b = (int)(slice & 1);
      if (slice >= 2) CK(cudaEventSynchronize(ctx->ev_stage[b]));
      memcpy(ctx->h_stage[b], src, n * 8);
      CK(cudaMemcpyAsync((char*)ctx->d_iq + off * 8, ctx->h_stage[b], n * 8, cudaMemcpyHostToDevice, s));
      CK(cudaEventRecord(ctx->ev_stage[b], s));
    } else {
      CK(cudaMemcpyAsync((char*)ctx->d_iq + off * 8, src, n * 8, cudaMemcpyHostToDevice, s));
    }
    if (off == 0 && (rc = launch_level(ctx, d_iq, n_raw, sc, P, s))) return rc;
    const long long first = (long long)(off / kIngestChunk);
    const long long cnt = (long long)((n + kIngestChunk - 1) / kIngestChunk);
    // the mask kernel treats samples beyond `off + n` as not yet present: pass the uploaded extent as n_raw
    if ((rc = launch_mask(ctx, d_iq, off + n, first, cnt, P, s))) return rc;
  }
  IngestTotals tot;
  if ((rc = finish_bursts(ctx, n_chunks, burst_cap, sc, P, s, tot))) return rc;
  launches = ctx->last_launches;
  if ((rc = build_segments(ctx, ctx->h_bursts, tot.n_falls, n_raw, sc, h_segs, seg_capacity, nseg))) return rc;
  const int ns = *nseg;
  if (ns == 0) return RFID_B200_OK;
  const size_t res_bytes = (size_t)ns * max_windows_per_segment * sizeof(rfid_b200_window_result);
  if ((rc = grow(ctx, &ctx->d_segs, &ctx->d_segs_bytes, (size_t)ns * sizeof(rfid_b200_segment)))) return rc;
  if ((rc = grow(ctx, &ctx->d_res, &ctx->d_res_bytes, res_bytes))) return rc;
  if ((rc = grow(ctx, &ctx->d_cnt, &ctx->d_cnt_bytes, (size_t)ns * 4))) return rc;
  CK(cudaMemcpyAsync(ctx->d_segs, h_segs, (size_t)ns * sizeof(rfid_b200_segment), cudaMemcpyHostToDevice, s));
  CK(cudaMemsetAsync(ctx->d_res, 0, res_bytes, s));
  rc = rfid_b200_decode_capture(ctx, (const float*)ctx->d_iq, n_raw, (const rfid_b200_segment*)ctx->d_segs, ns,
                                max_windows_per_segment, (rfid_b200_window_result*)ctx->d_res, (int32_t*)ctx->d_cnt, s);
  if (rc) return rc;
  ctx->last_launches += launches;
  CK(cudaMemcpyAsync(h_results, ctx->d_res, res_bytes, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(h_counts, ctx->d_cnt, (size_t)ns * 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return RFID_B200_OK;
}

// ------------------------------------------------------------------ TX synthesiser + slot simulator (SURVEY 8f-1)
}  // extern "C"

namespace {

// waveform table sizes with the reference's arithmetic: float sample period, float quotients, truncation
// (reader_impl.cc:51-71)
int derive_tx_timing(int dac_rate, TxTiming& T)
{
  if (dac_rate <= 0) return RFID_B200_EINVAL;
  const float sample_d = 1.0 / dac_rate * std::pow(10, 6);
  const float n_data0 = 2 * kPW_D / sample_d, n_data1 = 4 * kPW_D / sample_d, n_pw = kPW_D / sample_d;
  const float n_cw = kCW_D / sample_d, n_delim = kDELIM_D / sample_d, n_trcal = kTRCAL_D / sample_d;
  const float TAG_BIT_D = (float)(1.0 / kReaderFreq * std::pow(10, 6));
  const int RN16_D = (int)((kRN16Bits + kTagPreambleBits) * TAG_BIT_D);
  const int EPC_D = (int)((kEPCBits + kTagPreambleBits) * TAG_BIT_D);
  T.n_data0 = (int)n_data0; T.n_data1 = (int)n_data1; T.n_pw = (int)n_pw; T.n_delim = (int)n_delim;
  T.n_rtcal = (int)(n_data0 + n_data1); T.n_trcal = (int)n_trcal; T.n_cw = (int)n_cw;
  T.n_cwquery = (int)((kT1_D + kT2_D + RN16_D) / sample_d);
  T.n_cwack = (int)((3 * kT1_D + kT2_D + EPC_D) / sample_d);
  T.n_pdown = (int)(kP_DOWN_D / sample_d);
  if (T.n_pw < 1 || T.n_data0 < 2) return RFID_B200_EINVAL;
  return RFID_B200_OK;
}

// step response of the TX/RX chain measured on the recording (falling edge, raw 2 MS/s samples)
const float kEdgeFir2Msps[] = {-0.07f, 0.32f, 0.52f, 0.155f, 0.005f, 0.03f, 0.01f, 0.01f, 0.01f, 0.005f, 0.005f};

int build_sim_args(const rfid_b200_ctx* ctx, const rfid_b200_sim_params& p, SimArgs& A)
{
  memset(&A, 0, sizeof(A));
  if (p.n_tags < 0 || p.n_tags > kSimMaxTags || !(p.segment_us > 0.f) || !(p.lead_us >= 0.f) || p.dac_rate <= 0) return RFID_B200_EINVAL;
  if (ctx->cfg.adc_rate % p.dac_rate != 0) return RFID_B200_EINVAL;
  int rc = derive_tx_timing(p.dac_rate, A.T);
  if (rc) return rc;
  A.p = p;
  A.fixed_q = ctx->cfg.fixed_q;
  A.hold = ctx->cfg.adc_rate / p.dac_rate;
  A.sps = ctx->cfg.adc_rate / 1e6;
  A.dac_us = 1e6 / p.dac_rate;
  A.seg_len = (int)std::lround((double)p.segment_us * A.sps);
  A.lead_dac = (int)std::lround((double)p.lead_us / A.dac_us);
  // edge response stretched to the same duration at other ADC rates (linear interpolation, unit DC gain)
  const int n2 = (int)(sizeof(kEdgeFir2Msps) / sizeof(float));
  if (ctx->cfg.adc_rate == 2000000) {
    A.n_fir = n2;
    for (int i = 0; i < n2; i++) A.fir[i] = kEdgeFir2Msps[i];
  } else {
    int L = (int)std::lround(n2 * A.sps / 2.0);
    if (L < 3) L = 3;
    if (L > kSimMaxFir) L = kSimMaxFir;
    double sum = 0.0;
    for (int i = 0; i < L; i++) {
      const double x = (double)i * (n2 - 1) / (L - 1);
      const int i0 = (int)x;
      const int i1 = i0 + 1 < n2 ? i0 + 1 : i0;
      const double v = kEdgeFir2Msps[i0] + (kEdgeFir2Msps[i1] - kEdgeFir2Msps[i0]) * (x - i0);
      A.fir[i] = (float)v;
      sum += v;
    }
    for (int i = 0; i < L; i++) A.fir[i] = (float)(A.fir[i] / sum);
    A.n_fir = L;
  }
  A.mask_words = (A.seg_len + 31) / 32 + 1;
  if (A.seg_len < 64 || sizeof(SimShared) + 16 + (size_t)A.mask_words * 4 > 200 * 1024) return RFID_B200_EINVAL;
  return RFID_B200_OK;
}

}  // namespace

extern "C" {

int rfid_b200_tx_synth(rfid_b200_ctx* ctx, const rfid_b200_tx_command* h_script, int n_commands, int dac_rate, float* d_out,
                       size_t capacity, size_t* n_samples, void* stream)
{
  if (!ctx || !h_script || n_commands < 0 || !n_samples) return RFID_B200_EINVAL;
  TxTiming T;
  int rc = derive_tx_timing(dac_rate, T);
  if (rc) return rc;
  std::vector<unsigned long long> off((size_t)n_commands + 1, 0ull);
  for (int c = 0; c < n_commands; c++) {
    if (h_script[c].kind < RFID_B200_TX_START || h_script[c].kind > RFID_B200_TX_QUERY_ADJUST) return RFID_B200_EINVAL;
    off[c + 1] = off[c] + (unsigned long long)tx_length(T, h_script[c].kind, h_script[c].arg, ctx->cfg.fixed_q);
  }
  *n_samples = (size_t)off[n_commands];
  ctx->last_launches = 0;
  if (!d_out) return RFID_B200_OK;
  if (capacity < *n_samples) return RFID_B200_ECAPACITY;
  if (n_commands == 0) return RFID_B200_OK;
  CK(cudaSetDevice(ctx->device));
  const size_t sb = (size_t)n_commands * sizeof(rfid_b200_tx_command), ob = (size_t)n_commands * 8;
  if ((rc = grow(ctx, &ctx->d_script, &ctx->d_script_bytes, sb + ob + 16))) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  unsigned long long* d_off = reinterpret_cast<unsigned long long*>(ctx->d_script);
  rfid_b200_tx_command* d_scr = reinterpret_cast<rfid_b200_tx_command*>(d_off + n_commands);
  // pageable sources: cudaMemcpyAsync stages them before returning, so the vectors may go out of scope
  CK(cudaMemcpyAsync(d_off, off.data(), ob, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d_scr, h_script, sb, cudaMemcpyHostToDevice, s));
  tx_synth_kernel<<<n_commands, 256, 0, s>>>(T, ctx->cfg.fixed_q, d_scr, d_off, n_commands, d_out);
  CK(cudaGetLastError());
  ctx->last_launches = 1;
  return RFID_B200_OK;
}

void rfid_b200_default_sim(rfid_b200_sim_params* p)
{
  if (!p) return;
  memset(p, 0, sizeof(*p));
  p->seed = 1234;
  p->n_tags = 1;
  p->closed_loop = 1;
  p->dac_rate = 1000000;  // apps/reader.py:56
  p->segment_us = 8480.f;
  p->lead_us = 400.f;
  p->noise_sigma = 0.0030f;
  p->tag_gain = 0.0227f;
  p->tag_phase = std::atan2(0.192f, -0.981f);
  p->clock_pct = 0.8f;
  p->leak_re = 0.2846f;
  p->leak_im = -0.0349f;
  p->floor_level = 0.004f;
}

int rfid_b200_sim_segment_length(const rfid_b200_ctx* ctx, const rfid_b200_sim_params* p)
{
  if (!ctx || !p) return RFID_B200_EINVAL;
  SimArgs A;
  int rc = build_sim_args(ctx, *p, A);
  return rc ? rc : A.seg_len;
}

int rfid_b200_sim_capture(rfid_b200_ctx* ctx, const rfid_b200_sim_params* p, int64_t first_segment, int nseg, float* d_iq,
                          rfid_b200_segment* d_segs, rfid_b200_sim_truth* d_truth, void* stream)
{
  if (!ctx || !p || !d_iq || !d_segs || nseg < 0 || first_segment < 0) return RFID_B200_EINVAL;
  SimArgs A;
  int rc = build_sim_args(ctx, *p, A);
  if (rc) return rc;
  ctx->last_launches = 0;
  if (nseg == 0) return RFID_B200_OK;
  CK(cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)stream;
  const size_t smem = ((sizeof(SimShared) + 15) & ~(size_t)15) + (size_t)A.mask_words * 4;
  CK(cudaFuncSetAttribute((const void*)sim_slot_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  A.first_segment = first_segment; A.nseg = nseg;
  A.iq = reinterpret_cast<float2*>(d_iq); A.segs = d_segs; A.truth = d_truth;
  int launches = 0;
  if (!p->closed_loop) {
    A.phase = 2;
    sim_slot_kernel<<<nseg, kSimThreads, smem, s>>>(A);
    CK(cudaGetLastError());
    launches = 1;
  } else {
    // Query + RN16 replies -> decode the RN16 window with this context's receive chain -> ACK(decoded) + EPC
    if (!pick_kernel(ctx->cfg)) { ctx->last_error = "capture mode supports decim = 5 only in this build"; return RFID_B200_EINVAL; }
    if ((rc = grow(ctx, &ctx->d_sim_res, &ctx->d_sim_res_bytes, (size_t)nseg * sizeof(rfid_b200_window_result)))) return rc;
    if ((rc = grow(ctx, &ctx->d_sim_cnt, &ctx->d_sim_cnt_bytes, (size_t)nseg * 4))) return rc;
    A.phase = 0;
    sim_slot_kernel<<<nseg, kSimThreads, smem, s>>>(A);
    CK(cudaGetLastError());
    CK(cudaMemsetAsync(ctx->d_sim_res, 0, (size_t)nseg * sizeof(rfid_b200_window_result), s));
    rc = rfid_b200_decode_capture(ctx, d_iq, (size_t)nseg * A.seg_len, d_segs, nseg, 1, (rfid_b200_window_result*)ctx->d_sim_res,
                                  (int32_t*)ctx->d_sim_cnt, s);
    if (rc) return rc;
    A.phase = 1;
    A.rn16_records = (const rfid_b200_window_result*)ctx->d_sim_res;
    A.rn16_counts = (const int32_t*)ctx->d_sim_cnt;
    sim_slot_kernel<<<nseg, kSimThreads, smem, s>>>(A);
    CK(cudaGetLastError());
    launches = 3;
  }
  ctx->last_launches = launches;
  return RFID_B200_OK;
}

// ------------------------------------------------------------------ block mode
int rfid_b200_gate_work(rfid_b200_ctx* ctx, int seek, const float* in, int n_in, float* out, int out_capacity,
                        int* consumed, int* written, int* closed, float* magn2_out)
{
  if (!ctx || !in || !out || !consumed || !written || n_in < 0 || seek < 0 || seek > 2) return RFID_B200_EINVAL;
  if (out_capacity < n_in) return RFID_B200_ECAPACITY;  // the reference may write up to ninput items (gate_impl.cc:95,174,187)
  *consumed = 0; *written = 0;
  if (closed) *closed = 0;
  if (n_in == 0 && seek == 0) return RFID_B200_OK;
  CK(cudaSetDevice(ctx->device));
  int rc;
  const size_t ns = (size_t)(n_in > 0 ? n_in : 1);
  // one device block [GateCallOut (64 B) | out: ns complex | |out|^2: ns floats] and its pinned host mirror: the kernel's
  // whole result comes back with ONE copy and ONE synchronisation per work call (it was two of each)
  const size_t off_out = 64, off_m2 = off_out + ns * 8, blk = off_m2 + ns * 4;
  if ((rc = grow(ctx, &ctx->d_in, &ctx->d_in_bytes, ns * 8))) return rc;
  if ((rc = grow(ctx, &ctx->d_blk, &ctx->d_blk_bytes, blk))) return rc;
  if (ctx->h_blk_bytes < blk) {
    if (ctx->h_blk) cudaFreeHost(ctx->h_blk);
    ctx->h_blk = nullptr; ctx->h_blk_bytes = 0;
    const size_t want = blk + blk / 4 + 256;
    if (cudaHostAlloc(&ctx->h_blk, want, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return RFID_B200_ENOMEM; }
    ctx->h_blk_bytes = want;
  }
  cudaStream_t s = ctx->stream;
  char* db = (char*)ctx->d_blk;
  if (n_in) CK(cudaMemcpyAsync(ctx->d_in, in, (size_t)n_in * 8, cudaMemcpyHostToDevice, s));
  gate_block_kernel<<<1, 32, 0, s>>>(ctx->cfg, ctx->d_gate, seek, (const float2*)ctx->d_in, n_in, (float2*)(db + off_out),
                                     (float*)(db + off_m2), (GateCallOut*)db);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(ctx->h_blk, db, blk, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  GateCallOut r;
  memcpy(&r, ctx->h_blk, sizeof(r));
  if (r.written > 0) {
    memcpy(out, (char*)ctx->h_blk + off_out, (size_t)r.written * 8);
    if (magn2_out) memcpy(magn2_out, (char*)ctx->h_blk + off_m2, (size_t)r.written * 4);
  }
  *consumed = r.consumed; *written = r.written;
  if (closed) *closed = r.closed;
  ctx->last_launches = 1;
  return RFID_B200_OK;
}

int rfid_b200_decoder_work(rfid_b200_ctx* ctx, int kind, const float* win, int n, rfid_b200_window_result* res,
                           float* bits_out)
{
  if (!ctx || !win || !res || (kind != RFID_B200_RN16 && kind != RFID_B200_EPC)) return RFID_B200_EINVAL;
  const int need = kind == RFID_B200_RN16 ? ctx->cfg.len_rn16 : ctx->cfg.len_epc;
  if (n < need) return RFID_B200_EINVAL;  // the reference only fires on a complete window (tag_decoder_impl.cc:223,291)
  CK(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = grow(ctx, &ctx->d_in, &ctx->d_in_bytes, (size_t)need * 8))) return rc;
  cudaStream_t s = ctx->stream;
  CK(cudaMemcpyAsync(ctx->d_in, win, (size_t)need * 8, cudaMemcpyHostToDevice, s));
  decode_block_kernel<<<1, 32, (size_t)need * 12 + 64, s>>>(ctx->cfg, kind, (const float2*)ctx->d_in, need, ctx->d_one);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(res, ctx->d_one, sizeof(*res), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (bits_out) {
    const int nb = kind == RFID_B200_RN16 ? 16 : 128;
    for (int i = 0; i < nb; i++) bits_out[i] = (res->bits[i >> 3] >> (7 - (i & 7))) & 1 ? 1.0f : 0.0f;
  }
  ctx->last_launches = 1;
  return RFID_B200_OK;
}

int rfid_b200_mf_work(rfid_b200_ctx* ctx, const float* in, int n_in, float* out, int out_capacity, int* written)
{
  if (!ctx || !in || !out || !written || n_in < 0) return RFID_B200_EINVAL;
  *written = 0;
  CK(cudaSetDevice(ctx->device));
  const int D = ctx->cfg.decim, K = ctx->cfg.ntaps;
  const long long abs_end = ctx->mf_abs0 + ctx->mf_have + n_in;       // one past the newest sample
  const long long last_n = abs_end / D - 1;  // floor(total/decim) outputs exist so far (fixed-rate decimator)
  const long long n_out = last_n - ctx->mf_next_n + 1 > 0 ? last_n - ctx->mf_next_n + 1 : 0;
  if (n_out > out_capacity) return RFID_B200_ECAPACITY;
  int rc;
  const size_t total = (size_t)(ctx->mf_have + n_in);
  // staging buffer = carried history + new chunk
  if ((rc = grow(ctx, &ctx->d_out, &ctx->d_out_bytes, (total + 1) * 8))) return rc;
  cudaStream_t s = ctx->stream;
  if (ctx->mf_have) CK(cudaMemcpyAsync(ctx->d_out, ctx->d_mf, (size_t)ctx->mf_have * 8, cudaMemcpyDeviceToDevice, s));
  if (n_in) CK(cudaMemcpyAsync((char*)ctx->d_out + (size_t)ctx->mf_have * 8, in, (size_t)n_in * 8, cudaMemcpyHostToDevice, s));
  if (n_out > 0) {
    if ((rc = grow(ctx, &ctx->d_m2, &ctx->d_m2_bytes, (size_t)n_out * 8))) return rc;
    const int threads = 128;
    mf_block_kernel<<<(unsigned)((n_out + threads - 1) / threads), threads, 0, s>>>(
        ctx->cfg, (const float2*)ctx->d_out, ctx->mf_abs0, ctx->mf_next_n, (int)n_out, (float2*)ctx->d_m2);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, ctx->d_m2, (size_t)n_out * 8, cudaMemcpyDeviceToHost, s));
  }
  // keep what the next output still needs: samples from D*next_n - (K-1) on
  const long long next_n = ctx->mf_next_n + n_out;
  long long keep_from = (long long)D * next_n - (K - 1);
  if (keep_from < ctx->mf_abs0) keep_from = ctx->mf_abs0;
  if (keep_from > abs_end) keep_from = abs_end;
  const long long keep = abs_end - keep_from;
  if ((rc = grow(ctx, &ctx->d_mf, &ctx->d_mf_bytes, (size_t)(keep + 1) * 8))) return rc;
  if (keep) CK(cudaMemcpyAsync(ctx->d_mf, (char*)ctx->d_out + (size_t)(keep_from - ctx->mf_abs0) * 8, (size_t)keep * 8,
                               cudaMemcpyDeviceToDevice, s));
  CK(cudaStreamSynchronize(s));
  ctx->mf_abs0 = keep_from; ctx->mf_have = keep; ctx->mf_next_n = next_n;
  *written = (int)n_out;
  ctx->last_launches = n_out > 0 ? 1 : 0;
  return RFID_B200_OK;
}

}  // extern "C"
