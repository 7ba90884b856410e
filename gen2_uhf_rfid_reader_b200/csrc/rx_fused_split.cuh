// rx_fused_split.cuh -- fast-path variant of the fused capture kernel (reference configuration and every
// rate whose amplitude / DC rings fit one tile, i.e. raw rates up to 5 MS/s).
//
// Same arithmetic as rx_fused.cuh, different schedule.  The order-dependent work of a segment is split over
// TWO warps that run concurrently, one tile apart:
//   chain    ONLY the three float running sums (lane 0: avg_ampl over tile i, gate_impl.cc:131; lanes 1,2:
//            dc_est.re/.im over the closed samples of tile i-2, gate_impl.cc:141).  This is the irreducible
//            serial part of exact replay: ~5.6 cycles per sample, nothing else on its critical path.
//   control  thresholds (ballot into 128-bit masks), the edge/pulse state machine by bit-mask hopping, the few
//            DC-ring differences that the workers could not pre-compute (tiles with gate activity), window
//            emission to the L2-resident scratch two tiles later (when dc_est at the trigger is known), window
//            hand-off to the decoder.
// plus the two workers (TMA wait, block-sum matched filter, exact |y|, ring differences) and the decoder warp.
// CTA = 5 warps; tile stages form a time-indexed ring of 5 x 128 samples.  All hand-offs are mbarriers
// (phase = use count of the stage); waits that are not on the chain<->control critical path back off.
#pragma once

#include "rx_fused.cuh"

namespace rfid_b200 {

constexpr int kS = 5;                         // tile stages
#ifndef RFID_B200_SPLIT_WORKER_WARPS
#define RFID_B200_SPLIT_WORKER_WARPS 1
#endif
constexpr int kSWWarps = RFID_B200_SPLIT_WORKER_WARPS;   // worker warps of the split kernel
constexpr int kSWThreads = kSWWarps * 32;
constexpr int kSplitWarps = 3 + kSWWarps;     // chain, control, workers, decoder
constexpr int kSplitThreads = 32 * kSplitWarps;
__device__ __forceinline__ void split_sync_workers()
{
  if (kSWWarps == 1) __syncwarp();
  else bar_sync_workers();
}
constexpr int kRing = kS * kTT;               // time-indexed ring length (samples)

struct SplitShared {
  uint64_t raw_full[kRawStages];
  uint64_t tile_full[kS];    // workers (2 arrivals)  -> chain
  uint64_t chain_done[kS];   // chain   (1)           -> control   (avg of tile i, dc of tile i-2)
  uint64_t elist_ready[kS];  // control (1)           -> chain     (closed-sample list of tile i final)
  uint64_t tile_free[kS];    // control (1)           -> workers
  uint64_t win_ready[2], win_free[2];
  int meta_kind[2], meta_open[2], meta_ordinal[2], meta_len[2];
  int progress[2];           // window samples published so far (streaming decode)
  int aborted[2];            // the capture ended inside this window: finish the decode, store nothing
  int n_e[kS];               // closed samples in the DC list of each stage
  int n_ev[kS];
  TileEvent ev[kS][kMaxTileEvents];
};

// Named (hardware) barriers for the hand-offs that are waited on all the time -- a warp parked at bar.sync costs no
// issue slots: chain -> control ("chain_done"), control -> chain ("elist_ready"), control -> decoder ("win_ready").
// Two ids each, alternating: at most two arrivals can be outstanding on any of them (see the comments at the
// arrive sites).  Ids are immediates so ptxas reserves 8 barriers per CTA, not 16.
enum : int { SBAR_WIN_READY = 2, SBAR_CHAIN_DONE = 4, SBAR_ELIST = 6 };
template <int BASE>
__device__ __forceinline__ void bar2_sync(int parity)
{
  if (parity == 0) asm volatile("bar.sync %0, 64;" ::"n"((int)BASE) : "memory");
  else asm volatile("bar.sync %0, 64;" ::"n"((int)(BASE + 1)) : "memory");
}
template <int BASE>
__device__ __forceinline__ void bar2_arrive(int parity)
{
  __threadfence_block();
  if (parity == 0) asm volatile("bar.arrive %0, 64;" ::"n"((int)BASE) : "memory");
  else asm volatile("bar.arrive %0, 64;" ::"n"((int)(BASE + 1)) : "memory");
}

// a wait that is off the critical path: poll rarely
#ifndef RFID_B200_LAZY_NS
#define RFID_B200_LAZY_NS 2000
#endif
__device__ __forceinline__ void mbar_wait_lazy(uint64_t* bar, uint32_t parity)
{
  if (mbar_try_wait(bar, parity)) return;
  while (!mbar_try_wait(bar, parity)) __nanosleep(RFID_B200_LAZY_NS);
}
// a wait on the critical path: poll back to back
__device__ __forceinline__ void mbar_wait_hot(uint64_t* bar, uint32_t parity)
{
  mbar_wait_relaxed(bar, parity, 2000);  // try_wait with a suspend hint: the hardware parks the warp until the phase flips
}

// ---- the edge/pulse state machine of one closed run, warp-parallel -------------------------------------
// The reference walks the samples one by one (gate_impl.cc:145-180):
//     n_samples++;  POS && a<thr -> NEG, n_samples=0;   NEG && a>thr -> POS, pulse bookkeeping, n_samples=0;
//     open when n_samples > T1 && POS && num_pulses > 5.
// Here: (1) the POS/NEG state before every position follows from the fall-wish / rise-wish masks by a carry
// chain -- state' = rise | (keep & state) is the carry recurrence of a binary addition, so one 128-bit add gives
// all 128 states; (2) the resulting edges (<= 32 per batch) are handled one per lane: pulse widths by a shuffle,
// the run-length of consecutive valid pulses by ballot + popc, the first position at which the gate opens by
// ballot + ffs.  Exactly the reference's decisions, O(1) warp steps per tile instead of one step per edge.
struct GateFsm {
  bool sig_pos;
  int n_samples, num_pulses;
};

__device__ __forceinline__ int kth_set_bit128(unsigned w0, unsigned w1, unsigned w2, unsigned w3, int k)
{
  const int c0 = __popc(w0), c1 = c0 + __popc(w1), c2 = c1 + __popc(w2);
  int word = 0, r = k;
  unsigned sel = w0;
  if (k >= c2) { word = 3; r = k - c2; sel = w3; }
  else if (k >= c1) { word = 2; r = k - c1; sel = w2; }
  else if (k >= c0) { word = 1; r = k - c0; sel = w1; }
  return 32 * word + (int)__fns(sel, 0, r + 1);
}

// Processes the closed samples [from, nvalid) of a tile.  Returns the position at which the gate opens
// (the trigger sample, state updated for the open gate) or -1 (state advanced to the end of the tile).
struct Mask128 { unsigned w[4]; };

__device__ __forceinline__ int fsm_closed_run(const Mask128& lt, const Mask128& gt, int from, int nvalid, int n_T1,
                                              int half_pw, GateFsm& st)
{
  const int lane = threadIdx.x & 31;
  // ---- states by carry propagation: A = rise|keep, B = rise, carry-in = current state
  unsigned F[4], R[4], X[4];
  unsigned carry = st.sig_pos ? 1u : 0u;
#pragma unroll
  for (int w = 0; w < 4; w++) {
    // positions before `from` keep the state (they belong to an earlier run / an open window)
    const int lo = from - 32 * w;
    const unsigned live = lo <= 0 ? 0xffffffffu : (lo >= 32 ? 0u : (0xffffffffu << lo));
    F[w] = lt.w[w] & live;
    R[w] = gt.w[w] & live;
    const unsigned Pk = ~(F[w] | R[w]);
    const unsigned Aw = R[w] | Pk, Bw = R[w];
    const unsigned long long sum = (unsigned long long)Aw + Bw + carry;
    X[w] = Pk ^ (unsigned)sum;  // carry INTO each bit = state before that position (A ^ B == keep)
    carry = (unsigned)(sum >> 32);
  }
  unsigned E[4], RS[4];
#pragma unroll
  for (int w = 0; w < 4; w++) {
    RS[w] = ~X[w] & R[w];          // NEG -> POS
    E[w] = (X[w] & F[w]) | RS[w];  // POS -> NEG, or rise
  }
  int pos = from;
  int remaining = __popc(E[0]) + __popc(E[1]) + __popc(E[2]) + __popc(E[3]);
  int done = 0;
  while (true) {
    const int nb = min(32, remaining);
    // candidate before the first edge of this batch (the state may already be armed)
    int first_edge = nvalid;
    int p_k = 1 << 20;
    bool is_rise = false;
    if (lane < nb) {
      p_k = kth_set_bit128(E[0], E[1], E[2], E[3], done + lane);
      const int wsel = p_k >> 5;
      const unsigned rsw = wsel == 0 ? RS[0] : (wsel == 1 ? RS[1] : (wsel == 2 ? RS[2] : RS[3]));
      is_rise = (rsw >> (p_k & 31)) & 1u;
    }
    if (nb > 0) first_edge = __shfl_sync(0xffffffffu, p_k, 0);
    if (st.sig_pos && st.num_pulses > kNumPulsesCommand) {
      const int p_open = pos + max(0, n_T1 - st.n_samples);
      if (p_open < first_edge && p_open < nvalid) {  // a falling edge at the same position wins
        st.sig_pos = true; st.num_pulses = 0; st.n_samples = 1;
        return p_open;
      }
    }
    if (nb == 0) { st.n_samples += nvalid - pos; return -1; }
    // ---- one edge per lane
    const int p_virtual = pos - 1 - st.n_samples;  // where the previous edge would sit
    int p_prev = __shfl_up_sync(0xffffffffu, p_k, 1);
    if (lane == 0) p_prev = p_virtual;
    const bool valid_rise = (lane < nb) && is_rise && (p_k - p_prev > half_pw);   // n_samples > n_samples_PW/2
    const bool bad_rise = (lane < nb) && is_rise && !(p_k - p_prev > half_pw);
    const unsigned VR = __ballot_sync(0xffffffffu, valid_rise), IR = __ballot_sync(0xffffffffu, bad_rise);
    // num_pulses after edge k: valid rises since the last invalid one (inclusive range), plus the carried
    // count if no reset happened yet
    const unsigned upto = lane == 31 ? 0xffffffffu : ((2u << lane) - 1u);
    const unsigned resets = IR & upto;
    int np;
    if (resets) {
      const int last = 31 - __clz(resets);
      np = __popc(VR & upto & ~((2u << last) - 1u));
    } else {
      np = st.num_pulses + __popc(VR & upto);
    }
    // next edge after lane k (next lane, or the first edge of the next batch, or none)
    int p_next = __shfl_down_sync(0xffffffffu, p_k, 1);
    if (lane == nb - 1) p_next = (remaining > nb) ? kth_set_bit128(E[0], E[1], E[2], E[3], done + nb) : nvalid;
    const int p_open_k = p_k + 1 + n_T1;
    const bool opens = (lane < nb) && is_rise && np > kNumPulsesCommand && p_open_k < p_next && p_open_k < nvalid;
    const unsigned OM = __ballot_sync(0xffffffffu, opens);
    if (OM) {
      const int k = __ffs(OM) - 1;
      const int p_open = __shfl_sync(0xffffffffu, p_open_k, k);
      st.sig_pos = true; st.num_pulses = 0; st.n_samples = 1;
      return p_open;
    }
    // ---- no opening in this batch: state after its last edge
    const int kl = nb - 1;
    const int p_last = __shfl_sync(0xffffffffu, p_k, kl);
    st.sig_pos = __shfl_sync(0xffffffffu, (int)is_rise, kl) != 0;
    st.num_pulses = __shfl_sync(0xffffffffu, np, kl);
    st.n_samples = 0;
    pos = p_last + 1;
    done += nb;
    remaining -= nb;
  }
}

template <int DECIM, int MFQ>
__global__ void __launch_bounds__(kSplitThreads, 7) rx_fused_split_kernel(const FusedArgs A)
{
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ SplitShared B;
  __shared__ unsigned warps_done;
  stamp_cta_start(A.stamps);

  const int seg = blockIdx.x;
  const int lane = threadIdx.x & 31;
#ifdef RFID_B200_PHASE_PROFILE
  const long long ph_begin = clock64();
#define PH_END(slot) if (lane == 0 && A.window_tap) reinterpret_cast<long long*>(A.window_tap)[(size_t)blockIdx.x * 24 + (slot)] = clock64() - ph_begin;
#else
#define PH_END(slot)
#endif
  // roles: 0 chain, 1 control, 2.. workers, last decoder
  // Fixed role per warp of the CTA (nibble w of the table = role of warp w).  The hardware already places the four
  // warps of successive CTAs on the SM's warp slots with a rotating offset (tools/warpmap.py: CTA k's warp w gets slot
  // 4k + (w + c_k) % 4), so with a fixed table every sub-partition ends up with one or two warps of each role.  Rotating
  // the roles in software on top of that can cancel the hardware's rotation and stack all running-sum warps of an SM on
  // one sub-partition.  Measured on the 1000-segment benchmark (tools/variants.sh): rotating by the CTA's ordinal on
  // its SM 81.5 us, rotating by blockIdx 70.3 us, fixed tables 66-71 us depending on the order, worker / chain /
  // control / decoder 66.1 us.
#ifndef RFID_B200_ROLE_PERM
#define RFID_B200_ROLE_PERM 0x2013
#endif
  static_assert(kSplitWarps == 4 || kSplitWarps == 5, "role table");
  const int role = kSplitWarps == 4 ? (RFID_B200_ROLE_PERM >> (4 * (3 - (threadIdx.x >> 5)))) & 0xF
                                    : ((threadIdx.x >> 5) + blockIdx.x) % kSplitWarps;
#ifdef RFID_B200_PHASE_PROFILE
  if (lane == 0 && A.window_tap) {  // where did the hardware put this warp?  (slot 24*nseg + 4*cta + role) = smid << 16 | warpid
    unsigned smid, wid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    asm volatile("mov.u32 %0, %%warpid;" : "=r"(wid));
    reinterpret_cast<long long*>(A.window_tap)[(size_t)gridDim.x * 24 + (size_t)blockIdx.x * 4 + role] = (long long)((smid << 16) | wid);
  }
#endif
  const RxConfig& C = A.cfg;
  const rfid_b200_segment sg = A.segs[seg];
  const int n_out = (int)(sg.length / DECIM);
  const int ntiles = (n_out + kTT - 1) / kTT;

  float2* raw = reinterpret_cast<float2*>(smem + A.off_raw);
  float2* bhist = reinterpret_cast<float2*>(smem + A.off_bhist);
  float2* phist = bhist + A.bhist_size;
  float2* ring_y = reinterpret_cast<float2*>(smem + A.off_tile_y);   // [kRing]
  float* ring_a = reinterpret_cast<float*>(smem + A.off_tile_a);     // [kRing]
  float* ring_d = reinterpret_cast<float*>(smem + A.off_tile_d);     // [kRing] (+pad): delta-amp, then avg_ampl in place
  float* etile = reinterpret_cast<float*>(smem + A.off_etile);       // [kS][2][kTT] (+pad): DC-ring differences, then dc_est
  float2* snap = reinterpret_cast<float2*>(smem + A.off_snap);
  float2* dstage = reinterpret_cast<float2*>(smem + A.off_dstage);  // decoder's staging buffer
  float2* const win_base = A.win_scratch + (size_t)seg * A.win_stride;

  if (MFQ == 0 || kSWWarps != 1)  // (the consecutive-mapping workers keep their block sums in registers)
    for (int i = threadIdx.x; i < A.bhist_size * (C.mf_rem ? 2 : 1); i += kSplitThreads) bhist[i] = make_float2(0.f, 0.f);
  for (int i = threadIdx.x; i < kRing; i += kSplitThreads) { ring_y[i] = make_float2(0.f, 0.f); ring_a[i] = 0.f; }
  if (threadIdx.x == 0) {
    for (int s = 0; s < kRawStages; s++) mbar_init(&B.raw_full[s], 1);
    for (int s = 0; s < kS; s++) {
      mbar_init(&B.tile_full[s], kSWWarps);
      mbar_init(&B.chain_done[s], 1);
      mbar_init(&B.elist_ready[s], 1);
      mbar_init(&B.tile_free[s], 2);  // control (done with the stage's lookbacks) + chain (window emission done)
      B.n_e[s] = 0;
      B.n_ev[s] = 0;
    }
    for (int s = 0; s < 2; s++) { mbar_init(&B.win_ready[s], 1); mbar_init(&B.win_free[s], 1); }
    warps_done = 0;
    mbar_fence_init();
  }
  __syncthreads();

  if (role >= 2 && role < 2 + kSWWarps) {
    // =========================================================== workers
    const int wt = (role - 2) * 32 + lane;
    // raw tile geometry.  Tile k >= 1 starts at raw sample D*kTT*k - (D-1) of the segment, moved down to an even
    // absolute index (16-byte TMA source); tile 0 starts at the segment's first (even-aligned) sample.  Interior
    // tiles are all alike: `fast_tiles` of them can be issued with a constant byte count and a pointer bump.
    const int odd = (int)(sg.offset & 1ull);
    const uint32_t fast_bytes = (uint32_t)((DECIM * kTT + 2 * odd) * 8);
    int fast_tiles = 0;  // tiles 1 .. fast_tiles-1 take the fast path
    {
      // tile k is "interior" when its last sample D*(k*kTT + kTT-1) exists and the rounded-up copy stays inside the capture
      const long long by_len = ((long long)sg.length - 1 - (long long)DECIM * (kTT - 1)) / ((long long)DECIM * kTT);
      const long long room = (long long)A.n_raw - (long long)sg.offset + (DECIM - 1) + odd - (DECIM * kTT + 2 * odd);
      const long long by_buf = room >= 0 ? room / ((long long)DECIM * kTT) : -1;
      long long f = (by_len < by_buf ? by_len : by_buf) + 1;
      if (sg.length < (unsigned)(DECIM * kTT)) f = 0;
      fast_tiles = f < 0 ? 0 : (f > ntiles ? ntiles : (int)f);
    }
    const float2* const fast_src = A.iq + sg.offset - (DECIM - 1) - odd;  // + D*kTT*k for tile k >= 1
    auto load_tile = [&](int k, int rs_) {
      float2* dst = raw + (size_t)rs_ * A.raw_stage_samples;
      if (k >= 1 && k < fast_tiles) {
        mbar_arrive_expect_tx(&B.raw_full[rs_], fast_bytes);
        tma_load_1d(dst, fast_src + (size_t)k * (DECIM * kTT), fast_bytes, &B.raw_full[rs_]);
      } else {
        issue_tile_load<DECIM>(A, sg, k, dst, &B.raw_full[rs_]);
      }
    };
    if (wt == 0) {
      for (int k = 0; k < kRawStages && k < ntiles; k++) load_tile(k, k);
    }
    const int bmask = A.bhist_size - 1;
    const float winlen_f = (float)C.win_length, dclen_f = (float)C.dc_length;
    float2 b_keep[MFQ > 1 ? MFQ - 1 : 1];
#pragma unroll
    for (int m = 0; m < (MFQ > 1 ? MFQ - 1 : 1); m++) b_keep[m] = make_float2(0.f, 0.f);
    PH_DECL
    int rs = 0, ts = 0;                  // k % kRawStages, k % kS
    uint32_t raw_par = 0, free_par = 1;  // (k / kRawStages) & 1, ((k / kS) & 1) ^ 1
    for (int k = 0; k < ntiles; k++) {
      const float2* stage = raw + (size_t)rs * A.raw_stage_samples;
      const int delta = -odd - (k > 0 ? DECIM - 1 : 0);  // tile_load_start(k) - D*kTT*k
      const int nvalid = min(kTT, n_out - k * kTT);
      PH_MARK(0)
      mbar_wait(&B.raw_full[rs], raw_par);
      PH_MARK(1)
      if constexpr (MFQ > 0 && kSWWarps == 1) {
        // ---- consecutive mapping: this lane owns outputs t0 .. t0+3 of the tile; block sums travel between lanes by
        // shuffle and between tiles in registers, wide shared-memory accesses throughout
        constexpr int Q = kTT / 32;
        static_assert(MFQ - 1 <= Q, "block-sum halo comes from the neighbouring lane only");
        const int t0 = Q * lane;
        const int base = DECIM * t0 - (DECIM - 1) - delta;  // stage index of x[D*t0 - (D-1)]; parity = odd
        // block sums B(n) = x[D*n-D+1 .. D*n], ascending; two outputs' worth of raw samples in registers at a time
        float2 w[MFQ - 1 + Q];
        static_assert(Q % 2 == 0 && (2 * DECIM) % 2 == 0, "");
#pragma unroll
        for (int h = 0; h < Q; h += 2) {
          float2 x[2 * DECIM];
          if (odd == 0 && k > 0) {
            const float4* p4 = reinterpret_cast<const float4*>(stage + base + DECIM * h);
#pragma unroll
            for (int j = 0; j < DECIM; j++) {
              const float4 v = p4[j];
              x[2 * j] = make_float2(v.x, v.y);
              x[2 * j + 1] = make_float2(v.z, v.w);
            }
          } else {
#pragma unroll
            for (int j = 0; j < 2 * DECIM; j++) {
              const bool before = (k == 0) && (DECIM * (t0 + h) - (DECIM - 1) + j < 0);  // before sample 0 of the segment: +0
              x[j] = before ? make_float2(0.f, 0.f) : stage[base + DECIM * h + j];
            }
          }
#pragma unroll
          for (int q = 0; q < 2; q++) {
            float2 b = x[DECIM * q];
#pragma unroll
            for (int j = 1; j < DECIM; j++) b = c_add2(b, x[DECIM * q + j]);
            w[MFQ - 1 + h + q] = b;
          }
        }
        __syncwarp();  // raw stage consumed
        if (lane == 0 && k + kRawStages < ntiles) load_tile(k + kRawStages, rs);
        PH_MARK(2)
#pragma unroll
        for (int m = 0; m < MFQ - 1; m++) {  // B(n-MFQ+1 ..) of the first outputs: the previous lane's / tile's last block sums
          const float2 mine = w[Q + m];
          const float ux = __shfl_up_sync(0xffffffffu, mine.x, 1), uy = __shfl_up_sync(0xffffffffu, mine.y, 1);
          w[m] = lane ? make_float2(ux, uy) : b_keep[m];
          b_keep[m] = make_float2(__shfl_sync(0xffffffffu, mine.x, 31), __shfl_sync(0xffffffffu, mine.y, 31));
        }
        PH_MARK(3)
        mbar_wait_lazy(&B.tile_free[ts], free_par);  // control is done with tile k - 5
        PH_MARK(4)
        float2 y[Q];
        float a[Q];
#pragma unroll
        for (int q = 0; q < Q; q++) {
          y[q] = w[q];
#pragma unroll
          for (int m = 1; m < MFQ; m++) y[q] = c_add2(y[q], w[q + m]);
          a[q] = cabsf_ref(y[q].x, y[q].y);  // gate_impl.cc:130
        }
        {
          float4* py = reinterpret_cast<float4*>(ring_y + ts * kTT + t0);
#pragma unroll
          for (int q = 0; q < Q; q += 2) py[q / 2] = make_float4(y[q].x, y[q].y, y[q + 1].x, y[q + 1].y);
          float4* pa = reinterpret_cast<float4*>(ring_a + ts * kTT + t0);
#pragma unroll
          for (int q = 0; q < Q; q += 4) pa[q / 4] = make_float4(a[q], a[q + 1], a[q + 2], a[q + 3]);
        }
        PH_MARK(5)
        __syncwarp();  // this tile's |y| and y visible to the lookbacks below
        PH_MARK(6)
        // ring differences (gate_impl.cc:131,141), all divisions in flight together; the multiply-correct quotients
        // are used when every input of the warp is inside the verified range
        float xd[Q], xr[Q], xi[Q];
        int ia = ts * kTT + t0 - C.win_length, iy = ts * kTT + t0 - C.dc_length;
        if (ia < 0) ia += kRing;
        if (iy < 0) iy += kRing;
        if (((C.win_length | C.dc_length) & 3) == 0) {  // lookback groups are aligned and never straddle the ring's end
#pragma unroll
          for (int q = 0; q < Q; q += 4) {
            const float4 oa = *reinterpret_cast<const float4*>(ring_a + ia + q);
            xd[q] = f_sub(a[q], oa.x); xd[q + 1] = f_sub(a[q + 1], oa.y);
            xd[q + 2] = f_sub(a[q + 2], oa.z); xd[q + 3] = f_sub(a[q + 3], oa.w);
          }
#pragma unroll
          for (int q = 0; q < Q; q += 2) {
            const float4 oy = *reinterpret_cast<const float4*>(ring_y + iy + q);
            xr[q] = f_sub(y[q].x, oy.x); xi[q] = f_sub(y[q].y, oy.y);
            xr[q + 1] = f_sub(y[q + 1].x, oy.z); xi[q + 1] = f_sub(y[q + 1].y, oy.w);
          }
        } else {
#pragma unroll
          for (int q = 0; q < Q; q++) {
            int ja = ia + q, jy = iy + q;
            if (ja >= kRing) ja -= kRing;
            if (jy >= kRing) jy -= kRing;
            const float2 old = ring_y[jy];
            xd[q] = f_sub(a[q], ring_a[ja]);
            xr[q] = f_sub(y[q].x, old.x);
            xi[q] = f_sub(y[q].y, old.y);
          }
        }
        // range test of all twelve dividends at once (3-input min / max)
        float mx = fabsf(xd[0]), mn = mx;
#pragma unroll
        for (int q = 0; q < Q; q++) {
          mx = fmaxf(fmaxf(mx, fabsf(xd[q])), fmaxf(fabsf(xr[q]), fabsf(xi[q])));
          mn = fminf(fminf(mn, fabsf(xd[q])), fminf(fabsf(xr[q]), fabsf(xi[q])));
        }
        const bool all_ok = C.win_div_fast && C.dc_div_fast && mn >= kDivFastMin && mx <= kDivFastMax;
        float qd[Q], qr[Q], qi[Q];
        if (__all_sync(0xffffffffu, all_ok)) {
#pragma unroll
          for (int q = 0; q < Q; q++) {
            qd[q] = f_div_fast(xd[q], winlen_f, C.win_recip);
            qr[q] = f_div_fast(xr[q], dclen_f, C.dc_recip);
            qi[q] = f_div_fast(xi[q], dclen_f, C.dc_recip);
          }
        } else {  // an exact zero, a denormal, or an unverified divisor somewhere in the warp: IEEE division
#pragma unroll
          for (int q = 0; q < Q; q++) {
            qd[q] = f_div_const(xd[q], winlen_f, C.win_recip, C.win_div_fast);
            qr[q] = f_div_const(xr[q], dclen_f, C.dc_recip, C.dc_div_fast);
            qi[q] = f_div_const(xi[q], dclen_f, C.dc_recip, C.dc_div_fast);
          }
        }
#pragma unroll
        for (int q = 0; q < Q; q += 4) {
          *reinterpret_cast<float4*>(ring_d + ts * kTT + t0 + q) = make_float4(qd[q], qd[q + 1], qd[q + 2], qd[q + 3]);
          *reinterpret_cast<float4*>(etile + (ts * 2 + 0) * kTT + t0 + q) = make_float4(qr[q], qr[q + 1], qr[q + 2], qr[q + 3]);
          *reinterpret_cast<float4*>(etile + (ts * 2 + 1) * kTT + t0 + q) = make_float4(qi[q], qi[q + 1], qi[q + 2], qi[q + 3]);
        }
      } else {
        // ---- block sums B(n) = x[D*n-D+1 .. D*n], ascending
  #pragma unroll
        for (int r = 0; r < kTT / kSWThreads; r++) {
          const int t = wt + r * kSWThreads;
          if (t < nvalid) {
            const int n = k * kTT + t;
            const int base = DECIM * t - (DECIM - 1) - delta;
            float2 x[DECIM];
            if (k == 0 && t == 0) {  // the segment's very first block reaches before sample 0: those read as +0
  #pragma unroll
              for (int j = 0; j < DECIM; j++) x[j] = j < DECIM - 1 ? make_float2(0.f, 0.f) : stage[base + j];
            } else {
  #pragma unroll
              for (int j = 0; j < DECIM; j++) x[j] = stage[base + j];
            }
            float2 b = x[0];
  #pragma unroll
            for (int j = 1; j < DECIM; j++) b = c_add2(b, x[j]);
            if (MFQ > 0) {
              bhist[MFQ - 1 + t] = b;               // bhist[0 .. MFQ-2] = the last MFQ-1 block sums of the previous tile
              if (t >= kTT - (MFQ - 1)) b_keep[0] = b;  // ... which these threads hand over after the tile
            } else {
              bhist[n & bmask] = b;
            }
            if (MFQ == 0 && C.mf_rem) {
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
        split_sync_workers();  // raw stage consumed, block sums visible
        if (wt == 0 && k + kRawStages < ntiles) load_tile(k + kRawStages, rs);
        PH_MARK(3)
        mbar_wait_lazy(&B.tile_free[ts], free_par);  // control is done with tile k - 5
        PH_MARK(4)
        float a_reg[kTT / kSWThreads];
        float2 y_reg[kTT / kSWThreads];
  #pragma unroll
        for (int r = 0; r < kTT / kSWThreads; r++) {
          const int t = wt + r * kSWThreads;
          a_reg[r] = 0.f;
          y_reg[r] = make_float2(0.f, 0.f);
          if (t < nvalid) {
            const int n = k * kTT + t;
            float2 y;
            if (MFQ > 0) {
              const float2* bp = bhist + t;  // B(n-MFQ+1) .. B(n) are bp[0 .. MFQ-1]
              y = bp[0];
  #pragma unroll
              for (int m = 1; m < MFQ; m++) y = c_add2(y, bp[m]);
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
            ring_y[ts * kTT + t] = y;
            ring_a[ts * kTT + t] = a;
            a_reg[r] = a;
            y_reg[r] = y;
          }
        }
        PH_MARK(5)
        split_sync_workers();  // this tile's |y| and y visible to both workers; every block sum has been consumed
        PH_MARK(6)
        if (MFQ > 0) {
          const int t_hi = wt + kSWThreads * (kTT / kSWThreads - 1);  // this thread's last output of the tile
          if (t_hi >= kTT - (MFQ - 1) && t_hi < nvalid) bhist[t_hi - (kTT - (MFQ - 1))] = b_keep[0];
        }
        {
          // ring differences of this thread's samples, all divisions in flight together (gate_impl.cc:131,141); the
          // multiply-correct quotients are used when every input of the warp is inside the verified range
          float xd[kTT / kSWThreads], xr[kTT / kSWThreads], xi[kTT / kSWThreads];
          bool all_ok = C.win_div_fast && C.dc_div_fast;
  #pragma unroll
          for (int r = 0; r < kTT / kSWThreads; r++) {
            const int t = wt + r * kSWThreads;
            xd[r] = xr[r] = xi[r] = 1.0f;
            if (t < nvalid) {
              int ia = ts * kTT + t - C.win_length;
              if (ia < 0) ia += kRing;
              int iy = ts * kTT + t - C.dc_length;
              if (iy < 0) iy += kRing;
              const float2 old = ring_y[iy];
              xd[r] = f_sub(a_reg[r], ring_a[ia]);
              xr[r] = f_sub(y_reg[r].x, old.x);
              xi[r] = f_sub(y_reg[r].y, old.y);
            }
            all_ok = all_ok && f_div_fast_ok(xd[r]) && f_div_fast_ok(xr[r]) && f_div_fast_ok(xi[r]);
          }
          if (__all_sync(0xffffffffu, all_ok)) {
  #pragma unroll
            for (int r = 0; r < kTT / kSWThreads; r++) {
              const int t = wt + r * kSWThreads;
              if (t < nvalid) {
                ring_d[ts * kTT + t] = f_div_fast(xd[r], winlen_f, C.win_recip);
                etile[(ts * 2 + 0) * kTT + t] = f_div_fast(xr[r], dclen_f, C.dc_recip);
                etile[(ts * 2 + 1) * kTT + t] = f_div_fast(xi[r], dclen_f, C.dc_recip);
              }
            }
          } else {  // an exact zero, a denormal, or an unverified divisor somewhere in the warp: IEEE division
  #pragma unroll
            for (int r = 0; r < kTT / kSWThreads; r++) {
              const int t = wt + r * kSWThreads;
              if (t < nvalid) {
                ring_d[ts * kTT + t] = f_div_const(xd[r], winlen_f, C.win_recip, C.win_div_fast);
                etile[(ts * 2 + 0) * kTT + t] = f_div_const(xr[r], dclen_f, C.dc_recip, C.dc_div_fast);
                etile[(ts * 2 + 1) * kTT + t] = f_div_const(xi[r], dclen_f, C.dc_recip, C.dc_div_fast);
              }
            }
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&B.tile_full[ts]);
      PH_MARK(7)
      if (++rs == kRawStages) { rs = 0; raw_par ^= 1u; }
      if (++ts == kS) { ts = 0; free_par ^= 1u; }
    }
    if (wt == 0) { PH_DUMP(8) }
    if (wt == 0) { PH_END(21) }
  } else if (role == 0) {
    // =========================================================== chain: the exact running sums, nothing else
    float acc = 0.f;  // lane 0: avg_ampl, lane 1: dc_est.re, lane 2: dc_est.im
    // window emission state (two tiles behind the state machine)
    bool f_open = false, f_store = false;
    int f_wpos = 0, n_signalled = 0, n_freed = 0, f_slot = 0, wsig_ordinal = 0;
    float2 dc_open = make_float2(0.f, 0.f);
    float2* win = win_base;
    PH_DECL
    for (int i = 0; i < ntiles + 2; i++) {
      const int s = i % kS;
      int n = 0;
      PH_MARK(0)
      float* buf = ring_d + s * kTT;
      if (i < ntiles) {
        mbar_wait(&B.tile_full[s], (i / kS) & 1);
        if (lane == 0) n = min(kTT, n_out - i * kTT);
      }
      PH_MARK(1)
      if (i >= 2) {
        const int j = i - 2, sj = j % kS;
        bar2_sync<SBAR_ELIST>(j & 1);  // control has fixed the closed-sample list of tile i-2
        if (lane == 1 || lane == 2) {
          n = B.n_e[sj];
          buf = etile + (sj * 2 + (lane - 1)) * kTT;
        }
      }
      PH_MARK(2)
      if (lane < 3) chain_inplace(buf, n, acc);
      __syncwarp();
      PH_MARK(3)
      // control syncs on chain_done(i) before it publishes elist_ready(i), which this warp needs for
      // iteration i+2: never more than two arrivals outstanding => ids alternate with i
      bar2_arrive<SBAR_CHAIN_DONE>(i & 1);
      // ---- finish tile i-2: window emission (gate_impl.cc:173,187) with the dc_est this pass just produced, and the
      //      hand-off to the decoder
      if (i >= 2) {
        const int t = i - 2, ps = t % kS;
        const float2* py = ring_y + ps * kTT;
        const float* pe_re = etile + (ps * 2 + 0) * kTT;
        const float* pe_im = pe_re + kTT;
        const int pvalid = min(kTT, n_out - t * kTT);
        const int pnev = B.n_ev[ps];
        int pos = 0;
        for (int e = 0; e <= pnev; e++) {
          const bool last = e == pnev;
          const int etype = last ? 0 : B.ev[ps][e].type;
          const int epos = last ? pvalid : B.ev[ps][e].pos;
          if (f_open) {
            const int take = epos - pos;
            if (f_store && take > 0) {
              for (int j = lane; j < take; j += 32) win[f_wpos + j] = c_sub(py[pos + j], dc_open);
              __threadfence_block();  // samples first, then the counter the decoder (same CTA) polls
              __syncwarp();
              if (lane == 0) *(volatile int*)&B.progress[f_slot] = f_wpos + take;
            }
            f_wpos += take;
            pos = epos;
          }
          if (etype == 2) {
            f_open = false;  // the decoder already has the window: it saw progress reach its length
            pos = epos;
          } else if (etype == 1) {
            const int j = B.ev[ps][e].a;
            dc_open = make_float2(pe_re[j], pe_im[j]);  // dc_est right after the trigger sample
            f_store = B.ev[ps][e].c != 0;
            f_open = true;
            win = win_base + (B.ev[ps][e].d ? A.rn16_pad : 0);
            if (f_store) {
              // the scratch area and the meta slot are reused two hand-offs later
              while (n_signalled - n_freed >= 2) { mbar_wait(&B.win_free[n_freed & 1], (n_freed >> 1) & 1); n_freed++; }
              f_slot = n_signalled & 1;
              if (lane == 0) {
                win[0] = c_sub(py[epos], dc_open);
                const int knd = B.ev[ps][e].d;
                B.meta_kind[f_slot] = knd; B.meta_ordinal[f_slot] = wsig_ordinal; B.meta_open[f_slot] = B.ev[ps][e].b;
                B.meta_len[f_slot] = knd ? C.len_epc : C.len_rn16;
                *(volatile int*)&B.progress[f_slot] = 0;
                B.aborted[f_slot] = 0;
              }
              __threadfence_block();
              __syncwarp();
              if (lane == 0) *(volatile int*)&B.progress[f_slot] = 1;
              // hand the window to the decoder NOW: it decodes while the gate is still open (streaming)
              bar2_arrive<SBAR_WIN_READY>(f_slot);
              n_signalled++;
            }
            wsig_ordinal++;
            f_wpos = 1;
            pos = epos + 1;
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&B.tile_free[ps]);  // second party of tile_free (control arrived after tile i-1's state machine)
      }
    }
    if (f_open && f_store && lane == 0) {
      // the segment ended inside a window the decoder is already working on: let it run to the end
      *(volatile int*)&B.aborted[f_slot] = 1;
      __threadfence_block();
      *(volatile int*)&B.progress[f_slot] = 1 << 30;
    }
    __syncwarp();
    while (n_signalled - n_freed >= 2) { mbar_wait(&B.win_free[n_freed & 1], (n_freed >> 1) & 1); n_freed++; }
    if (lane == 0) {
      B.meta_kind[n_signalled & 1] = -1;
    }
    __syncwarp();
    bar2_arrive<SBAR_WIN_READY>(n_signalled & 1);
    PH_DUMP(16)
    PH_END(20)
  } else if (role == 1) {
    // =========================================================== control
    bool sig_pos = false;          // signal_state, starts NEG_EDGE (gate_impl.cc:45)
    int n_samples = 0, num_pulses = 0;
    bool gate_open = false;
    int to_ungate = C.len_rn16;    // first SEEK is for an RN16 (global_vars.cc:47, reader_impl.cc:262)
    int wcount = 0, open_idx = 0;
    bool cur_store = false;
    int nq = 1;                    // n_queries_sent after START -> SEND_QUERY (reader_impl.cc:259)
    bool terminated = false;
    int closed_since = C.dc_length;
    const float dclen_f = (float)C.dc_length;
    const int half_pw = C.n_PW / 2;
    PH_DECL

    for (int i = 0; i < ntiles; i++) {
      const int s = i % kS;
      PH_MARK(0)
      bar2_sync<SBAR_CHAIN_DONE>(i & 1);  // avg_ampl of tile i and dc_est of tile i-2 are final
      PH_MARK(1)
      // ---- thresholds + state machine of tile i; make its closed-sample list final
      int nev = 0, n_e = 0;
      if (i < ntiles) {
        const int nvalid = min(kTT, n_out - i * kTT);
        const float* davg = ring_d + s * kTT;
        const float* ta = ring_a + s * kTT;
        const float2* ty = ring_y + s * kTT;
        float* er = etile + (s * 2 + 0) * kTT;
        float* ei = er + kTT;
        if (!terminated) {
          // thresholds of tile i (gate_impl.cc:136,148,154): a < 0.75 avg / a > 0.75 avg per sample, as 128-bit masks.
          // A tile that lies entirely inside an open window needs none (the gate ignores edges while it is open).
          unsigned lt[4] = {0u, 0u, 0u, 0u}, gt[4] = {0u, 0u, 0u, 0u};
          if (!(gate_open && to_ungate - n_samples > nvalid)) {
#pragma unroll
            for (int r = 0; r < 4; r++) {
              const int p = r * 32 + lane;
              const float thr = f_mul(davg[p], kThreshFraction);
              const float a = ta[p];
              lt[r] = __ballot_sync(0xffffffffu, a < thr);
              gt[r] = __ballot_sync(0xffffffffu, a > thr);
            }
            if (nvalid < kTT) {  // the segment's last, partial tile: samples past its end compare nothing
#pragma unroll
              for (int r = 0; r < 4; r++) {
                const int left = nvalid - r * 32;
                const unsigned vm = left >= 32 ? 0xffffffffu : (left > 0 ? (1u << left) - 1u : 0u);
                lt[r] &= vm;
                gt[r] &= vm;
              }
            }
          }
          PH_MARK(2)
          int pos = 0;
          while (pos < nvalid) {
            if (!gate_open) {
              // ---- closed: edges, pulse counting and the open test of this run in one warp-parallel step
              const int run_start = pos;
              int p_open = -1;
              if (sig_pos && (lt[0] | lt[1] | lt[2] | lt[3]) == 0u) {
                // carrier only (the common case): no falling edge can occur, only the open test remains
                if (num_pulses > kNumPulsesCommand) {
                  const int cand = run_start + max(0, C.n_T1 - n_samples);
                  if (cand < nvalid) { p_open = cand; num_pulses = 0; n_samples = 1; }
                }
                if (p_open < 0) n_samples += nvalid - run_start;
              } else {
                GateFsm fs = {sig_pos, n_samples, num_pulses};
                const Mask128 ltm = {{lt[0], lt[1], lt[2], lt[3]}}, gtm = {{gt[0], gt[1], gt[2], gt[3]}};
                p_open = fsm_closed_run(ltm, gtm, run_start, nvalid, C.n_T1, half_pw, fs);
                sig_pos = fs.sig_pos; n_samples = fs.n_samples; num_pulses = fs.num_pulses;
              }
              const bool opened = p_open >= 0;
              pos = opened ? p_open + 1 : nvalid;
              // ---- DC tracker inputs of the closed run [run_start, pos) (gate_impl.cc:141-143; includes the trigger)
              const int len = pos - run_start;
              if (run_start == 0 && pos == nvalid && !opened && closed_since >= C.dc_length) {
                // no gate activity and the ring lookback is time-contiguous: the workers' differences are exact
              } else {
#pragma unroll 1
                for (int j = lane; j < len; j += 32) {
                  const int p = run_start + j, m = closed_since + j;
                  const float2 yv = ty[p];
                  float2 old;
                  if (m < C.dc_length) {
                    old = snap[m];  // ring contents from before the window
                  } else {
                    int iy = s * kTT + p - C.dc_length;
                    if (iy < 0) iy += kRing;
                    old = ring_y[iy];
                  }
                  er[n_e + j] = f_div_const(f_sub(yv.x, old.x), dclen_f, C.dc_recip, C.dc_div_fast);
                  ei[n_e + j] = f_div_const(f_sub(yv.y, old.y), dclen_f, C.dc_recip, C.dc_div_fast);
                }
              }
              closed_since = min(closed_since + len, 1 << 24);
              n_e += len;
              if (opened) {
                // READER COMMAND DETECTED (gate_impl.cc:164-180): keep the dc ring as it stands now
#pragma unroll 1
                for (int j = lane; j < C.dc_length; j += 32) {
                  int iy = s * kTT + (pos - 1) - C.dc_length + 1 + j;
                  if (iy < 0) iy += kRing;
                  snap[j] = ring_y[iy];
                }
                gate_open = true;
                open_idx = i * kTT + pos - 1;
                cur_store = wcount < A.max_windows;
                if (lane == 0 && nev < kMaxTileEvents) {
                  TileEvent& ev = B.ev[s][nev];
                  ev.type = 1; ev.pos = pos - 1; ev.a = n_e - 1; ev.b = open_idx; ev.c = cur_store ? 1 : 0; ev.d = wcount & 1;
                }
                nev++;
              }
            } else {
              // ---- open: samples pass through (gate_impl.cc:182-195); emitted two tiles later
              const int take = min(to_ungate - n_samples, nvalid - pos);
              n_samples += take; pos += take;
              if (n_samples >= to_ungate) {
                gate_open = false;
                const int kind = wcount & 1;  // windows alternate RN16, EPC (SURVEY.md 3.5)
                if (lane == 0 && nev < kMaxTileEvents) {
                  TileEvent& ev = B.ev[s][nev];
                  ev.type = 2; ev.pos = pos; ev.a = kind; ev.b = wcount; ev.c = to_ungate; ev.d = open_idx;
                }
                nev++;
                wcount++;
                closed_since = 0;
                // ACK after RN16 -> GATE_SEEK_EPC, Query/QueryRep after EPC -> GATE_SEEK_RN16 (gate_impl.cc:112-123)
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
        if (lane == 0) { B.n_e[s] = n_e; B.n_ev[s] = min(nev, kMaxTileEvents); }
        __syncwarp();
        bar2_arrive<SBAR_ELIST>(i & 1);  // chain may run dc_est over this tile (its iteration i+2)
      }
      PH_MARK(3)
      // the ring lookbacks of tile i reach back into stage i-1 only: control is done with it (the chain
      // warp, which emits tile i-1's window samples, is the other party of tile_free)
      if (i >= 1 && lane == 0) mbar_arrive(&B.tile_free[(i - 1) % kS]);
      PH_MARK(4)
    }
    PH_DUMP(0)
    if (lane == 0) A.counts[seg] = wcount;
    PH_END(22)
  } else {
    // =========================================================== decoder
    for (int j = 0;; j++) {
      bar2_sync<SBAR_WIN_READY>(j & 1);  // parked by the hardware until the control warp hands a window over
      const int kind = B.meta_kind[j & 1];
      if (kind < 0) break;
      const int ordinal = B.meta_ordinal[j & 1], open_idx = B.meta_open[j & 1], len = B.meta_len[j & 1];
      const float2* win = win_base + (kind ? A.rn16_pad : 0);
      WindowDecode wd;
      decode_window_staged(C, kind, win, len, dstage, A.dstage_samples, wd, (const volatile int*)&B.progress[j & 1]);
      rfid_b200_window_result* dst = A.results + (size_t)seg * A.max_windows + ordinal;
      const bool aborted = *(volatile int*)&B.aborted[j & 1] != 0;
      if (lane == 0 && !aborted) store_result(dst, wd, seg + A.seg_base, ordinal, open_idx, len, kind);
#ifndef RFID_B200_PHASE_PROFILE
      if (A.window_tap) {
        float2* tap = A.window_tap + ((size_t)(seg + A.seg_base) * A.max_windows + ordinal) * C.len_epc;
        for (int p = lane; p < len; p += 32) tap[p] = __ldcg(win + p);
      }
#endif
      __syncwarp();
      if (lane == 0) mbar_arrive(&B.win_free[j & 1]);
    }
    PH_END(23)
  }
  stamp_warp_end(A.stamps, &warps_done);
}

}  // namespace rfid_b200
