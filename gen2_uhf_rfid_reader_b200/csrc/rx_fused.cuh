// rx_fused.cuh -- the fused capture-mode kernel: matched filter + decimation,
// gate (reader-command detection, windowing) and tag_decoder for one capture
// segment per CTA, streaming the segment through shared memory in tiles so the
// only HBM traffic is one read of every raw sample (8 B/sample) plus 64-byte
// result records.
//
// Replaces (reference gr-rfid/): filter.fir_filter_ccc(5,[1]*25) (apps/reader.py:65,75),
// gate_impl::general_work (lib/gate_impl.cc:85-200) and
// tag_decoder_impl::general_work (lib/tag_decoder_impl.cc:196-397).
//
// CTA = 4 warps with fixed roles (rotated over the hardware warps by blockIdx so that the
// latency-critical warps of co-resident CTAs spread over the four SM sub-partitions):
//   sequencer   everything that is order-dependent in the reference.  Per 128-sample tile it runs ONE
//               pass of three simultaneous float running sums -- lane 0: avg_ampl over tile k
//               (gate_impl.cc:131), lanes 1,2: dc_est.re/.im over the closed samples of tile k-1
//               (gate_impl.cc:141) -- then finishes tile k-1 (window emission with the now-known DC
//               estimate, window hand-off to the decoder) and runs thresholds + the edge/pulse state
//               machine of tile k as bit-mask hopping (a few steps per reader command).
//   workers x2  wait for the TMA bulk copy of the next raw tile, block-sum matched filter, |y|
//               (exact cabsf), amplitude-ring difference / win_length  -> tile stage.
//   decoder     decodes each closed window from shared memory (preamble correlation, channel
//               estimate, FM0 decisions, period search, CRC-16) and writes the result record.
// Hand-offs use named barriers (bar.arrive / bar.sync): a waiting warp is parked by the hardware
// and costs no issue slots; only the TMA completion uses an mbarrier (transaction count).
#pragma once

#include "rx_common.cuh"
#include "rx_decode.cuh"

namespace rfid_b200 {

#ifdef RFID_B200_PHASE_PROFILE
// developer aid: per-phase clock64() sums of the sequencer / worker warp of CTA 0..N, written to the window tap
#define PH_DECL long long ph_t0 = clock64(), ph_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#define PH_MARK(i) { long long ph_t1 = clock64(); ph_acc[i] += ph_t1 - ph_t0; ph_t0 = ph_t1; }
#define PH_DUMP(base) if (lane == 0 && A.window_tap) { long long* o = reinterpret_cast<long long*>(A.window_tap) + (size_t)blockIdx.x * 24 + (base); for (int i = 0; i < 8; i++) o[i] = ph_acc[i]; }
#else
#define PH_DECL
#define PH_MARK(i)
#define PH_DUMP(base)
#endif

constexpr int kTT = 128;          // decimated samples per tile
constexpr int kRawStages = 2;
constexpr int kTileStages = 3;    // >= 3: tile k-1 is still being finished while tile k+1 is produced
constexpr int kWorkerWarps = 2;
constexpr int kWorkerThreads = kWorkerWarps * 32;
constexpr int kFusedThreads = 32 * (2 + kWorkerWarps);
constexpr int kMaxTileEvents = 6;

// named barrier ids (immediates, so that ptxas reserves 8 and not all 16 hardware barriers per CTA)
enum : int {
  BAR_WORKERS = 1,      // the two worker warps (64)
  BAR_TILE_FULL = 2,    // +stage: workers arrive (64), sequencer syncs (32)
  BAR_TILE_EMPTY = 5    // +stage: sequencer arrives (32), workers sync (64)
};

template <int BASE>
__device__ __forceinline__ void bar_sync_stage(int s, int n)
{
  if (s == 0) asm volatile("bar.sync %0, %1;" ::"n"((int)BASE), "r"(n) : "memory");
  else if (s == 1) asm volatile("bar.sync %0, %1;" ::"n"((int)(BASE + 1)), "r"(n) : "memory");
  else asm volatile("bar.sync %0, %1;" ::"n"((int)(BASE + 2)), "r"(n) : "memory");
}
template <int BASE>
__device__ __forceinline__ void bar_arrive_stage(int s, int n)
{
  if (s == 0) asm volatile("bar.arrive %0, %1;" ::"n"((int)BASE), "r"(n) : "memory");
  else if (s == 1) asm volatile("bar.arrive %0, %1;" ::"n"((int)(BASE + 1)), "r"(n) : "memory");
  else asm volatile("bar.arrive %0, %1;" ::"n"((int)(BASE + 2)), "r"(n) : "memory");
}
__device__ __forceinline__ void bar_sync_workers()
{
  asm volatile("bar.sync 1, 64;" ::: "memory");
}

struct FusedArgs {
  const float2* iq;              // raw capture (device), 16-byte aligned
  unsigned long long n_raw;      // total samples in the capture buffer
  const rfid_b200_segment* segs;
  int nseg;
  int seg_base;                  // added to the segment index stored in the records (a call that decodes a slice of a table)
  int max_windows;               // record slots per segment
  rfid_b200_window_result* results;
  int32_t* counts;
  float2* window_tap;            // optional: ungated samples of every stored window (stride len_epc)
  float2* win_scratch;           // [nseg][win_stride]: the window being decoded (RN16 at 0, EPC at rn16_pad); L2-resident
  unsigned long long* stamps;    // launch timing slot (stamp_cta_start / stamp_warp_end), nullptr = off
  int win_stride, rn16_pad;
  int off_dstage, dstage_samples; // decoder staging buffer
  RxConfig cfg;
  // shared-memory carve-up (bytes from the dynamic smem base), computed on the host
  int off_raw, raw_stage_samples;
  int off_bhist, bhist_size;     // float2[bhist_size] (+ partial-block ring right after it when mf_rem > 0)
  int off_ahist, ahist_size;     // float[ahist_size]
  int off_tile_y, off_tile_a, off_tile_d;
  int off_ycl, ycl_size;         // float2[ycl_size]                       (generic path)
  int off_e;                     // float[2][kTT + 16]                      (generic path)
  int off_etile;                 // float[kTileStages][2][kTT] (+pad)       (fast path: workers' DC-ring differences)
  int off_snap;                  // float2[dc_length]: dc ring snapshot taken when the gate opens (fast path)
  int smem_bytes;
};

struct TileEvent {
  int type;  // 1 = gate opens at tile position pos (trigger sample), 2 = window ends before position pos
  int pos;
  int a, b, c, d;  // open: a = index of the trigger in the tile's closed-sample list, b = open index, c = store
                   // close: a = kind, b = ordinal, c = length, d = open index
};

struct FusedShared {
  uint64_t raw_full[kRawStages];
  uint64_t win_ready[2], win_free[2];  // alternate per hand-off: the sequencer may run two hand-offs ahead
  int meta_kind[2], meta_open[2], meta_ordinal[2], meta_len[2];  // double-buffered by hand-off parity
  int n_ev;
  TileEvent ev[kMaxTileEvents];
};

__device__ __forceinline__ int next_set128(unsigned long long lo, unsigned long long hi, int pos)
{
  if (pos < 64) {
    unsigned long long m = lo & (~0ull << pos);
    if (m) return __ffsll((long long)m) - 1;
    pos = 64;
  }
  if (pos < 128) {
    unsigned long long m = hi & (~0ull << (pos - 64));
    if (m) return 64 + __ffsll((long long)m) - 1;
  }
  return 128;
}

__device__ __forceinline__ void chain8(float4& u, float4& v, float& acc)
{
  acc = f_add(acc, u.x); u.x = acc;
  acc = f_add(acc, u.y); u.y = acc;
  acc = f_add(acc, u.z); u.z = acc;
  acc = f_add(acc, u.w); u.w = acc;
  acc = f_add(acc, v.x); v.x = acc;
  acc = f_add(acc, v.y); v.y = acc;
  acc = f_add(acc, v.z); v.z = acc;
  acc = f_add(acc, v.w); v.w = acc;
}

// Sequential in-place running sum: acc = acc + buf[i]; buf[i] = acc (one rounding per step, the order of
// the reference's recurrences).  The next 8 inputs are always in flight while 8 dependent adds retire, so
// the loop runs at the FADD dependency latency.  May READ up to 16 floats past buf[n-1] (callers pad).
__device__ __forceinline__ void chain_inplace(float* buf, int n, float& acc)
{
  int i = 0;
  if (n >= 16) {
    float4 a0 = *reinterpret_cast<const float4*>(buf), a1 = *reinterpret_cast<const float4*>(buf + 4);
    for (; i + 16 <= n; i += 16) {
      float4 b0 = *reinterpret_cast<const float4*>(buf + i + 8), b1 = *reinterpret_cast<const float4*>(buf + i + 12);
      chain8(a0, a1, acc);
      *reinterpret_cast<float4*>(buf + i) = a0;
      *reinterpret_cast<float4*>(buf + i + 4) = a1;
      a0 = *reinterpret_cast<const float4*>(buf + i + 16);
      a1 = *reinterpret_cast<const float4*>(buf + i + 20);
      chain8(b0, b1, acc);
      *reinterpret_cast<float4*>(buf + i + 8) = b0;
      *reinterpret_cast<float4*>(buf + i + 12) = b1;
    }
  }
  for (; i < n; i++) {
    acc = f_add(acc, buf[i]);
    buf[i] = acc;
  }
}

// raw tile geometry: segment-relative index of the first sample held in the stage buffer
template <int DECIM>
__device__ __forceinline__ long long tile_load_start(unsigned long long seg_off, int k)
{
  long long lo = (long long)DECIM * k * kTT - (DECIM - 1);
  if (lo < 0) lo = 0;
  long long abs_lo = (long long)seg_off + lo;
  abs_lo &= ~1ll;  // 16-byte aligned source
  return abs_lo - (long long)seg_off;
}

template <int DECIM>
__device__ __forceinline__ void issue_tile_load(const FusedArgs& A, const rfid_b200_segment& sg, int k, float2* stage,
                                                uint64_t* bar)
{
  const long long start = tile_load_start<DECIM>(sg.offset, k);  // may be -1
  long long hi = (long long)DECIM * ((long long)k * kTT + kTT - 1);
  if (hi > (long long)sg.length - 1) hi = (long long)sg.length - 1;
  long long count = hi - start + 1;  // samples start..hi
  long long count_al = (count + 1) & ~1ll;
  const long long abs_start = (long long)sg.offset + start;
  float2 tail = make_float2(0.f, 0.f);
  bool patch = false;
  if ((unsigned long long)(abs_start + count_al) > A.n_raw) {
    // the rounded-up copy would run one sample past the capture buffer: copy an even count and
    // fetch the last sample with a plain load
    count_al -= 2;
    tail = A.iq[abs_start + count - 1];
    patch = true;
  }
  const uint32_t bytes = (uint32_t)(count_al * 8);
  if (patch) stage[count - 1] = tail;
  mbar_arrive_expect_tx(bar, bytes);
  if (bytes) tma_load_1d(stage, A.iq + abs_start, bytes, bar);
}

// MFQ > 0: ntaps == MFQ * DECIM (compile-time unrolled block sums); MFQ == 0: generic ntaps.
// This kernel keeps explicit amplitude / closed-sample rings of any length (raw rates above 5 MS/s, where the
// reference's 250 us / 120 us windows are longer than a tile); rx_fused_split_kernel is the fast path below that.
template <int DECIM, int MFQ>
__global__ void __launch_bounds__(kFusedThreads, 8) rx_fused_kernel(const FusedArgs A)
{
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ FusedShared B;
  __shared__ unsigned warps_done;
  stamp_cta_start(A.stamps);

  const int seg = blockIdx.x;
  const int lane = threadIdx.x & 31;
  const int warp = ((threadIdx.x >> 5) + blockIdx.x) & 3;  // role: 0 sequencer, 1..2 workers, 3 decoder
  const RxConfig& C = A.cfg;
  const rfid_b200_segment sg = A.segs[seg];
  const int n_out = (int)(sg.length / DECIM);
  const int ntiles = (n_out + kTT - 1) / kTT;

  float2* raw = reinterpret_cast<float2*>(smem + A.off_raw);
  float2* bhist = reinterpret_cast<float2*>(smem + A.off_bhist);
  float2* phist = bhist + A.bhist_size;
  float* ahist = reinterpret_cast<float*>(smem + A.off_ahist);
  float2* tile_y = reinterpret_cast<float2*>(smem + A.off_tile_y);
  float* tile_a = reinterpret_cast<float*>(smem + A.off_tile_a);
  float* tile_d = reinterpret_cast<float*>(smem + A.off_tile_d);
  float2* ycl = reinterpret_cast<float2*>(smem + A.off_ycl);
  float* e_re = reinterpret_cast<float*>(smem + A.off_e);
  float* e_im = e_re + kTT + 16;
  // ungated window samples go to a per-segment global scratch (written once, read once by the decoder warp
  // of the same CTA a few microseconds later: L2 traffic, not shared memory -- that is what lets 8 CTAs fit an SM)
  float2* const win_base = A.win_scratch + (size_t)seg * A.win_stride;
  float2* const dstage = reinterpret_cast<float2*>(smem + A.off_dstage);  // decoder's staging buffer

  // ---- init: zero the history rings (win_samples / dc_samples start at 0, gate_impl.cc:55-56;
  //      x[<0] = +0 for the matched filter), set up the TMA barriers
  for (int i = threadIdx.x; i < A.bhist_size * (C.mf_rem ? 2 : 1); i += kFusedThreads) bhist[i] = make_float2(0.f, 0.f);
  for (int i = threadIdx.x; i < A.ahist_size; i += kFusedThreads) ahist[i] = 0.f;
  for (int i = threadIdx.x; i < A.ycl_size; i += kFusedThreads) ycl[i] = make_float2(0.f, 0.f);
  if (threadIdx.x == 0) {
    for (int s = 0; s < kRawStages; s++) mbar_init(&B.raw_full[s], 1);
    for (int s = 0; s < 2; s++) { mbar_init(&B.win_ready[s], 1); mbar_init(&B.win_free[s], 1); }
    B.n_ev = 0;
    warps_done = 0;
    mbar_fence_init();
  }
  __syncthreads();

  if (warp >= 1 && warp <= kWorkerWarps) {
    // =========================================================== workers
    const int wt = (warp - 1) * 32 + lane;
    if (wt == 0) {
      for (int k = 0; k < kRawStages && k < ntiles; k++)
        issue_tile_load<DECIM>(A, sg, k, raw + (size_t)k * A.raw_stage_samples, &B.raw_full[k]);
    }
    const int bmask = A.bhist_size - 1, amask = A.ahist_size - 1;
    const float winlen_f = (float)C.win_length;
    PH_DECL
    for (int k = 0; k < ntiles; k++) {
      const int rs = k % kRawStages, ts = k % kTileStages;
      const float2* stage = raw + (size_t)rs * A.raw_stage_samples;
      // stage index of raw sample x[D*n - (D-1) + j] for tile-local output t:  D*t - (D-1) + j - delta
      const int delta = (int)(tile_load_start<DECIM>(sg.offset, k) - (long long)DECIM * k * kTT);
      const int nvalid = min(kTT, n_out - k * kTT);
      PH_MARK(0)
      mbar_wait(&B.raw_full[rs], (k / kRawStages) & 1);
      PH_MARK(1)
      // ---- block sums B(n) = x[D*n-D+1 .. D*n], ascending (and the partial block when ntaps % D != 0)
#pragma unroll
      for (int r = 0; r < kTT / kWorkerThreads; r++) {
        const int t = wt + r * kWorkerThreads;
        if (t < nvalid) {
          const int n = k * kTT + t;
          const int base = DECIM * t - (DECIM - 1) - delta;
          float2 x[DECIM];
#pragma unroll
          for (int j = 0; j < DECIM; j++) {
            // only the very first block of a segment reaches before sample 0 (reads as +0)
            const bool before = (k == 0) && (DECIM * t - (DECIM - 1) + j < 0);
            x[j] = before ? make_float2(0.f, 0.f) : stage[base + j];
          }
          float2 b = x[0];
#pragma unroll
          for (int j = 1; j < DECIM; j++) b = c_add(b, x[j]);
          bhist[n & bmask] = b;
          if (MFQ == 0 && C.mf_rem) {  // P(n): newest mf_rem samples of the block, ascending (static indexing only)
            float2 p = make_float2(0.f, 0.f);
            bool started = false;
#pragma unroll
            for (int j = 0; j < DECIM; j++) {
              if (j >= DECIM - C.mf_rem) {
                p = started ? c_add(p, x[j]) : x[j];
                started = true;
              }
            }
            phist[n & bmask] = p;
          }
        }
      }
      PH_MARK(2)
      bar_sync_workers();  // raw stage rs fully consumed, block sums visible
      if (wt == 0 && k + kRawStages < ntiles)
        issue_tile_load<DECIM>(A, sg, k + kRawStages, raw + (size_t)rs * A.raw_stage_samples, &B.raw_full[rs]);
      PH_MARK(3)
      if (k >= kTileStages) bar_sync_stage<BAR_TILE_EMPTY>(ts, 96);  // the sequencer is done with tile k - 3
      PH_MARK(4)
      // ---- y[n] = ((P(n-q) + B(n-q+1)) + ...) + B(n);  a = |y|
      float a_reg[kTT / kWorkerThreads];
      float2 y_reg[kTT / kWorkerThreads];
#pragma unroll
      for (int r = 0; r < kTT / kWorkerThreads; r++) {
        const int t = wt + r * kWorkerThreads;
        a_reg[r] = 0.f;
        y_reg[r] = make_float2(0.f, 0.f);
        if (t < nvalid) {
          const int n = k * kTT + t;
          float2 y;
          if (MFQ > 0) {
            y = bhist[(n - MFQ + 1) & bmask];
#pragma unroll
            for (int m = MFQ - 2; m >= 0; m--) y = c_add(y, bhist[(n - m) & bmask]);
          } else {
            int m = n - C.mf_q + 1;
            if (C.mf_rem) {
              y = phist[(n - C.mf_q) & bmask];
            } else {
              y = bhist[m & bmask];
              m++;
            }
            for (; m <= n; m++) y = c_add(y, bhist[m & bmask]);
          }
          const float a = cabsf_ref(y.x, y.y);  // gate_impl.cc:130
          tile_y[ts * kTT + t] = y;
          tile_a[ts * kTT + t] = a;
          ahist[n & amask] = a;
          a_reg[r] = a;
          y_reg[r] = y;
        }
      }
      PH_MARK(5)
      bar_sync_workers();  // this tile's amplitudes / filtered samples visible
      PH_MARK(6)
      // ---- (a - win_samples[win_index]) / win_length   (gate_impl.cc:131)
#pragma unroll
      for (int r = 0; r < kTT / kWorkerThreads; r++) {
        const int t = wt + r * kWorkerThreads;
        if (t < nvalid) {
          const int n = k * kTT + t;
          tile_d[ts * kTT + t] = f_div(f_sub(a_reg[r], ahist[(n - C.win_length) & amask]), winlen_f);
        }
      }
      __threadfence_block();
      bar_arrive_stage<BAR_TILE_FULL>(ts, 96);
      PH_MARK(7)
    }
    if (wt == 0) { PH_DUMP(8) }
  } else if (warp == 0) {
    // =========================================================== sequencer
    float acc = 0.f;  // lane 0: avg_ampl, lane 1: dc_est.re, lane 2: dc_est.im
    // --- gate state machine (runs one tile ahead of the window emission)
    bool sig_pos = false;          // signal_state, starts NEG_EDGE (gate_impl.cc:45)
    int n_samples = 0, num_pulses = 0;
    bool gate_open = false;
    int to_ungate = C.len_rn16;    // first SEEK is for an RN16 (global_vars.cc:47, reader_impl.cc:262)
    int wcount = 0;
    int n_closed = 0;              // closed-sample ordinal (index into the DC ring stream)
    int open_idx = 0;
    bool cur_store = false;
    int nq = 1;                    // n_queries_sent after START -> SEND_QUERY (reader_impl.cc:259)
    bool terminated = false;
    int n_e = 0;                   // closed samples of the tile whose DC chain is still to run
    // --- emission state (tile k-1)
    bool f_open = false, f_store = false;
    int f_wpos = 0, n_signalled = 0, n_freed = 0;
    float2* win = win_base;
    int closed_since = C.dc_length;  // closed samples since the last window (>= dc_length: ring lookback is time-contiguous)
    float2 dc_open = make_float2(0.f, 0.f);
    const int ymask = A.ycl_size - 1;
    const float dclen_f = (float)C.dc_length;
    const int half_pw = C.n_PW / 2;
    PH_DECL

    for (int k = 0; k <= ntiles; k++) {
      const int ts = k % kTileStages;
      const int nvalid = k < ntiles ? min(kTT, n_out - k * kTT) : 0;
      float* davg = tile_d + ts * kTT;
      PH_MARK(0)
      if (k < ntiles) bar_sync_stage<BAR_TILE_FULL>(ts, 96);
      PH_MARK(1)
      // ---- 1. the three recurrences, one pass: avg_ampl over tile k, dc_est over tile k-1's closed samples
      float* pe_re = e_re;  // tile k-1's list
      float* pe_im = e_im;
      if (lane < 3) chain_inplace(lane == 0 ? davg : (lane == 1 ? pe_re : pe_im), lane == 0 ? nvalid : n_e, acc);
      __syncwarp();
      PH_MARK(2)
      // ---- 2. finish tile k-1: window emission (gate_impl.cc:173,187) and hand-off to the decoder
      if (k >= 1) {
        const int pts = (k - 1) % kTileStages;
        const float2* py = tile_y + pts * kTT;
        const int pvalid = min(kTT, n_out - (k - 1) * kTT);
        const int nev = B.n_ev;
        int pos = 0;
        for (int e = 0; e <= nev; e++) {
          const bool last = e == nev;
          const int etype = last ? 0 : B.ev[e].type;
          const int epos = last ? pvalid : B.ev[e].pos;
          if (f_open) {
            const int take = epos - pos;  // an open event cannot occur while the gate is open
            if (f_store)
              for (int j = lane; j < take; j += 32) win[f_wpos + j] = c_sub(py[pos + j], dc_open);
            f_wpos += take;
            pos = epos;
          }
          if (etype == 2) {
            // window complete: hand it to the decoder
            f_open = false;
            if (f_store) {
              __syncwarp();
              if (lane == 0) {
                const int ms = n_signalled & 1;  // the slot of hand-off n-2 is free: at most one window is outstanding
                B.meta_kind[ms] = B.ev[e].a; B.meta_ordinal[ms] = B.ev[e].b; B.meta_len[ms] = B.ev[e].c; B.meta_open[ms] = B.ev[e].d;
              }
              __threadfence();  // window samples were written to global memory
              __syncwarp();
              if (lane == 0) mbar_arrive(&B.win_ready[n_signalled & 1]);
              n_signalled++;
            }
            pos = epos;
          } else if (etype == 1) {
            // READER COMMAND DETECTED (gate_impl.cc:164-180): dc_est right after the trigger sample
            const int j = B.ev[e].a;
            dc_open = make_float2(pe_re[j], pe_im[j]);
            f_store = B.ev[e].c != 0;
            f_open = true;
            win = win_base + (B.ev[e].d ? A.rn16_pad : 0);  // RN16 and EPC windows have their own scratch areas
            if (f_store) {
              // the area is reused two windows later: at most one window may still be with the decoder
              while (n_signalled - n_freed >= 2) { mbar_wait(&B.win_free[n_freed & 1], (n_freed >> 1) & 1); n_freed++; }
              if (lane == 0) win[0] = c_sub(py[epos], dc_open);
            }
            f_wpos = 1;
            pos = epos + 1;
          }
        }
        __syncwarp();
      }
      PH_MARK(3)
      // ---- 3. thresholds + state machine of tile k; collect its closed samples for the DC chain
      n_e = 0;
      int nev = 0;
      if (k < ntiles && !terminated) {
        const float* ta = tile_a + ts * kTT;
        const float2* ty = tile_y + ts * kTT;
        unsigned lt[4], gt[4];
#pragma unroll
        for (int r = 0; r < 4; r++) {
          const int i = r * 32 + lane;
          const bool v = i < nvalid;
          const float thr = v ? f_mul(davg[i], kThreshFraction) : 0.f;  // gate_impl.cc:136
          const float a = v ? ta[i] : 0.f;
          lt[r] = __ballot_sync(0xffffffffu, v && a < thr);
          gt[r] = __ballot_sync(0xffffffffu, v && a > thr);
        }
        const unsigned long long LT_lo = lt[0] | ((unsigned long long)lt[1] << 32), LT_hi = lt[2] | ((unsigned long long)lt[3] << 32);
        const unsigned long long GT_lo = gt[0] | ((unsigned long long)gt[1] << 32), GT_hi = gt[2] | ((unsigned long long)gt[3] << 32);
        PH_MARK(4)

        int pos = 0;
        while (pos < nvalid) {
          if (!gate_open) {
            // ---- closed: hop from edge to edge (gate_impl.cc:145-162) until the tile ends or the gate opens
            const int run_start = pos;
            bool opened = false;
            while (pos < nvalid) {
              if (sig_pos) {
                const int p_fall = next_set128(LT_lo, LT_hi, pos);
                int p_open = 1 << 30;
                if (num_pulses > kNumPulsesCommand) p_open = pos + max(0, C.n_T1 - n_samples);
                if (p_fall >= nvalid && p_open >= nvalid) { n_samples += nvalid - pos; pos = nvalid; break; }
                if (p_fall <= p_open) { n_samples = 0; sig_pos = false; pos = p_fall + 1; }
                else { pos = p_open + 1; opened = true; break; }
              } else {
                const int p_rise = next_set128(GT_lo, GT_hi, pos);
                if (p_rise >= nvalid) { n_samples += nvalid - pos; pos = nvalid; break; }
                const int n_at = n_samples + (p_rise - pos + 1);
                num_pulses = (n_at > half_pw) ? num_pulses + 1 : 0;
                n_samples = 0; sig_pos = true; pos = p_rise + 1;
              }
            }
            // ---- DC tracker inputs for the closed run [run_start, pos) (gate_impl.cc:141-143); the run
            //      includes the trigger sample, as in the reference (the update precedes the open test)
            const int len = pos - run_start;
            for (int j = lane; j < len; j += 32) ycl[(n_closed + j) & ymask] = ty[run_start + j];
            __syncwarp();
            for (int j = lane; j < len; j += 32) {
              const float2 yv = ty[run_start + j];
              const float2 old = ycl[(n_closed + j - C.dc_length) & ymask];
              e_re[n_e + j] = f_div(f_sub(yv.x, old.x), dclen_f);
              e_im[n_e + j] = f_div(f_sub(yv.y, old.y), dclen_f);
            }
            n_closed += len;
            n_e += len;
            if (opened) {
              gate_open = true;
              open_idx = k * kTT + pos - 1;
              cur_store = wcount < A.max_windows;
              if (lane == 0 && nev < kMaxTileEvents) {
                TileEvent& ev = B.ev[nev];
                ev.type = 1; ev.pos = pos - 1; ev.a = n_e - 1; ev.b = open_idx; ev.c = cur_store ? 1 : 0; ev.d = wcount & 1;
              }
              nev++;
              num_pulses = 0;
              n_samples = 1;
            }
          } else {
            // ---- open: the samples pass through (gate_impl.cc:182-195); emitted one tile later
            const int take = min(to_ungate - n_samples, nvalid - pos);
            n_samples += take; pos += take;
            if (n_samples >= to_ungate) {
              gate_open = false;
              const int kind = wcount & 1;  // windows alternate RN16, EPC (SURVEY.md 3.5)
              if (lane == 0 && nev < kMaxTileEvents) {
                TileEvent& ev = B.ev[nev];
                ev.type = 2; ev.pos = pos; ev.a = kind; ev.b = wcount; ev.c = to_ungate; ev.d = open_idx;
              }
              nev++;
              wcount++;
              closed_since = 0;
              // the Gen2 logic answers (ACK after RN16 -> GATE_SEEK_EPC, Query/QueryRep after EPC ->
              // GATE_SEEK_RN16) and the next gate call applies it (gate_impl.cc:112-123)
              to_ungate = kind ? C.len_rn16 : C.len_epc;
              n_samples = 0;
              if (kind) {
                nq++;
                if (nq > C.max_queries) { terminated = true; break; }  // gate_impl.cc:101-109
              }
            }
          }
        }
      }
      if (lane == 0) B.n_ev = min(nev, kMaxTileEvents);
      __syncwarp();
      // the stage of tile k-1 (its samples fed the ring lookbacks / snapshot above) may be refilled now
      if (k >= 1 && k - 1 + kTileStages < ntiles) {
        __threadfence_block();
        bar_arrive_stage<BAR_TILE_EMPTY>((k - 1) % kTileStages, 96);
      }
      PH_MARK(5)
    }
    PH_DUMP(0)
    // ---- shut the decoder down, publish the window count
    // the exit message needs the meta slot of hand-off n-2 only
    while (n_signalled - n_freed >= 2) { mbar_wait(&B.win_free[n_freed & 1], (n_freed >> 1) & 1); n_freed++; }
    if (lane == 0) {
      B.meta_kind[n_signalled & 1] = -1;
      A.counts[seg] = wcount;
    }
    __threadfence_block();
    __syncwarp();
    if (lane == 0) mbar_arrive(&B.win_ready[n_signalled & 1]);
  } else {
    // =========================================================== decoder
    for (int j = 0;; j++) {
      while (!mbar_try_wait(&B.win_ready[j & 1], (j >> 1) & 1)) __nanosleep(400);  // idle most of the time: poll slowly
      const int kind = B.meta_kind[j & 1];
      if (kind < 0) break;
      const int ordinal = B.meta_ordinal[j & 1], open_idx = B.meta_open[j & 1], len = B.meta_len[j & 1];
      WindowDecode wd;
      const float2* win = win_base + (kind ? A.rn16_pad : 0);
      decode_window_staged(C, kind, win, len, dstage, A.dstage_samples, wd);
      rfid_b200_window_result* dst = A.results + (size_t)seg * A.max_windows + ordinal;
      if (lane == 0) store_result(dst, wd, seg + A.seg_base, ordinal, open_idx, len, kind);
#ifndef RFID_B200_PHASE_PROFILE
      if (A.window_tap) {
        float2* tap = A.window_tap + ((size_t)(seg + A.seg_base) * A.max_windows + ordinal) * C.len_epc;
        for (int p = lane; p < len; p += 32) tap[p] = __ldcg(win + p);
      }
#endif
      __syncwarp();
      if (lane == 0) mbar_arrive(&B.win_free[j & 1]);
    }
  }
  stamp_warp_end(A.stamps, &warps_done);
}

}  // namespace rfid_b200
