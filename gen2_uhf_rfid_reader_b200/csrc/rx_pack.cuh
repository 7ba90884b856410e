// rx_pack.cuh -- the roofline kernel of the reference configuration (decimation 5, 25 taps, rings inside one tile):
// same arithmetic as rx_fused_split.cuh, re-scheduled around three measurements (tools/pack_profile.py, ncu):
//   * the exact replay of the gate's float running sums (avg_ampl, gate_impl.cc:131; dc_est, gate_impl.cc:141) is a
//     dependent FADD chain -- it costs the same whether 3 or 24 lanes of the warp carry a chain;
//   * everything else of a segment is one warp's worth of *latency*, not of issue slots: a warp that walks a tile through
//     matched filter, |y|, ring differences (or thresholds + the edge / pulse state machine) needs 2-3 thousand cycles per
//     pass almost independently of how many samples the pass covers;
//   * the stages of a segment have very different costs from tile to tile (the state machine costs 1 k cycles on a
//     carrier-only tile and 6 k on a tile full of reader pulses), so a lockstep hand-off per tile runs at the sum of the
//     worst stages.
// So a CTA owns G <= kPMaxSeg capture segments, one warp per role and segment, ONE chain warp for all of them, and the
// stages are coupled only through small rings with full / free barriers (mbarriers, one phase per slot use):
//   warp A0/A1[g] P1: waits for the raw half-tile (TMA bulk copies issued by the loader warp), block-sum matched filter,
//               exact |y|, amplitude / DC ring differences of 4 outputs per lane.  Writes |y| and the amplitude quotients
//               into 4-slot rings, the DC quotients into a 5-slot ring, and y itself into the segment's circular history in
//               global memory (L2 resident, kYW samples).  May run up to four tiles ahead of warp B.
//   chain warp  lane 8*c + g replays running sum c (0 avg_ampl, 1 dc_est.re, 2 dc_est.im) of segment g: avg_ampl of tile i
//               as soon as every segment's P1(i) is in, dc_est of tile j once every segment's P3(j) has fixed its list --
//               whichever is ready, both in one pass when both are; then hands dc_est at every window's trigger sample
//               to warp C.
//   warp B[g]   P3: thresholds by ballot (one mask word per lane), the edge / pulse state machine on the 256-bit masks, the
//               DC-tracker inputs of the 48 samples after a window (y read back from the history), -0.0f for the samples
//               inside windows.  Frees the |y| / quotient slot as soon as its masks are made.  Queues opening windows.
//   warp C[g]   decodes every queued window straight from the history as soon as its last sample and its dc_est exist
//               (rx_decode.cuh); dc_est is subtracted as the decoder reads the samples -- the same exact float
//               subtraction, gate_impl.cc:173,187.
//   loader      lane g streams segment g's raw samples through its two half-tile stages as warp A frees them.
// The history is indexed by the SM (one CTA per SM: the shared-memory request guarantees it, also between two launches
// that overlap under programmatic dependent launch), so its size does not depend on the number of segments of the launch;
// warp A never overwrites a sample a queued window still needs.
// Back-to-back launches overlap (programmatic dependent launch, see DESIGN §4.1): every CTA lets the next launch be
// scheduled right after the start-up barrier, so the next launch's CTAs take SMs as this launch's CTAs exit.  Before the
// first store of an output (counts: warp B, records / window tap: warp C) a warp waits for the previous launch to complete,
// since that launch may write the same buffers; the loader warp waits at its end, so no CTA exits before the previous launch
// has completed and work queued after a launch still sees every earlier launch.  The inputs (capture, segment table) need no
// wait: the previous rx_pack_kernel never writes them, and any other kernel before this one has completed when it starts.
// Shared memory per segment: 2 raw half-tile stages (10 KB), the last dc_length outputs of either half-tile (P1's DC
// lookback is a lane shuffle plus this tail), a 4-tile ring of |y| (4 KB), the decoder's stage (2 KB); per CTA the
// running-sum buffers (4 + 5x2 per segment, 1072 B each, skewed so the chain warp's 128-bit accesses are bank-conflict
// free).  HBM traffic: every raw sample is read once (evict-first), 64 B are written per window; the history (8 B per
// decimated sample, rewritten in place) lives in L2.
#pragma once

#include "rx_fused_split.cuh"

namespace rfid_b200 {

constexpr int kT2 = 2 * kTT;                 // decimated samples per tile (two half-tiles of kTT)
constexpr int kPAS = 4;                      // slots of the |y| ring and of the amplitude quotient / avg_ampl lists
constexpr int kRingA = kPAS * kT2;
constexpr int kPDS = 5;                      // DC-list slots: P1 up to four tiles ahead, P3 fix-ups, chain
constexpr int kPMaxSeg = 7;                  // segments per CTA (chain lanes 8*c + g, g < 8)
constexpr int kPChainBuf = kT2 + 12;         // floats per running-sum buffer: read-ahead pad; 1072 B = 48 mod 128
constexpr int kPackMaxThreads = 32 * (4 * kPMaxSeg + 2);   // A0, A1, B, C per segment + loader + chain
constexpr int kYW = 4096;                    // samples of y history per segment (power of two)
constexpr int kPQ = 8;                       // queue of windows that will be decoded (opened, not yet decoded)
constexpr int kPTrig = 2;                    // windows that may open within one tile (host: len_rn16 >= kT2 / 2)
constexpr int kPackMinSmem = 116 * 1024;     // request at least this much: two CTAs never share an SM (and its history),
                                             // not even CTAs of two overlapping launches

struct PackArgs {
  const float2* iq;
  unsigned long long n_raw;
  const rfid_b200_segment* segs;
  int nseg;
  int seg_base;                              // added to the segment index stored in the records
  int max_windows;
  rfid_b200_window_result* results;
  int32_t* counts;
  float2* window_tap;
  float2* y_hist;                            // [%nsmid][kPMaxSeg][kYW]
  unsigned long long* stamps;                // launch timing slot (stamp_cta_start / stamp_warp_end), nullptr = off
  RxConfig cfg;
  int G;                                     // segments per CTA of this launch
  int raw_stage_samples;
  int seg_bytes;                             // per-segment shared-memory region
  int o_raw, o_tail_y, o_ring_a, o_dstage;   // offsets inside a segment region
  int dstage_samples;
  int off_dA, off_dD, off_seg;               // offsets from the dynamic shared-memory base
  int smem_bytes;
};

struct PackSegCtl {
  rfid_b200_segment seg;     // the segment's table entry (length 0: none), read from global memory once per CTA
  uint64_t raw_full[2];      // loader (TMA transaction count) -> warp A
  uint64_t raw_empty[2];     // warps A (stage 0: A0 and A1's halo read, stage 1: A1) -> loader
  uint64_t half_rdy;         // warp A0 -> warp A1: y and |y| of the first half-tile are in the rings
  uint64_t tail_rdy;         // warp A1 -> warp A0 (next tile): second half-tile in the rings, block-sum halo in `keep`
  uint64_t freeA[kPAS];      // warp B -> warps A: masks of the tile in this slot are made, the slot may be rewritten
  float2 keep[2][4];         // the tile's last MFQ-1 block sums, by tile parity
  // windows that will be decoded, by sequence number k (slot k & (kPQ-1)): written by warp B, dc_val by the chain warp
  int q_open[kPQ], q_kind[kPQ], q_ord[kPQ];
  float2 dc_val[kPQ];
  volatile int n_opened, n_dc, n_decoded, seg_done;
  volatile int y_tiles;      // tiles whose y is complete in the history (written by warp A1, or A0 for a lone first half)
  // warp B's state that only changes at gate events (kept out of its registers)
  int b_wcount, b_nq, b_snap_base, b_queued;
  int n_e[kPDS];             // closed samples of the tile in DC-list slot (written by P3)
  int trig_n[kPDS];          // queued windows that opened in that tile: index of the trigger in the list, sequence number
  int trig_j[kPDS][kPTrig], trig_k[kPDS][kPTrig];
};
struct PackCtaCtl {
  uint64_t fullA[kPAS];      // 2G warps A -> chain: P1 of the tile is in
  uint64_t avgdone[kPAS];    // chain -> warps B: avg_ampl of the tile is final
  uint64_t p3done[kPDS];     // G warps B -> chain: the tile's DC list is final
  uint64_t dcdone[kPDS];     // chain -> warps A: the DC-list slot may be rewritten
};

#ifdef RFID_B200_PHASE_PROFILE
// developer aid (tools/pack_profile.py): absolute clock64() stamps (since CTA start) of warps A, B, C, chain of CTA 0
#define PP_DECL long long* pp_log = nullptr;
#define PP_AT(i) { if (pp_log && lane == 0) pp_log[pp_step * 8 + (i)] = clock64() - pp_cta_t0; }
#else
#define PP_DECL
#define PP_AT(i)
#endif

// hand-off waits on the critical path: the hardware parks the warp for a few dozen cycles per try
__device__ __forceinline__ void pwait(uint64_t* bar, uint32_t parity) { mbar_wait_relaxed(bar, parity, 2000); }

// ---- the edge / pulse state machine of one closed run on 256-bit masks, the eight mask words spread over lanes 0..7 ----
// Same decisions as fsm_closed_run (rx_fused_split.cuh) and therefore as the reference's sample loop
// (gate_impl.cc:145-180):
//   states     state' = rise | keep & state is the carry recurrence of a binary addition; inside a word one 64-bit add,
//              across the words the same recurrence once more (generate = the word's sum overflows with carry-in 0,
//              propagate = only with carry-in 1), i.e. one more addition on the two ballots
//   pulses     a rise at p is a valid pulse when the fall before it is more than half_pw back: no fall bit at p-1 .. p-half_pw
//   num_pulses valid rises since the last invalid one (plus the carried count while no invalid rise has occurred)
//   opening    the carried state reaches T1 before the first edge, or a rise r with num_pulses > 5 is followed by
//              n_T1 + 1 edge-free samples inside the tile (gate opens at r + 1 + n_T1; a fall there wins)
// Positions and counts are combined with redux.sync / vote (one instruction each); the reductions of the common path
// (a tile full of reader pulses, no opening) do not depend on each other, so they are in flight together.
struct GateFsm2 {
  bool sig_pos;
  int n_samples, num_pulses;
};
__device__ __forceinline__ unsigned m_below(int n) { return n <= 0 ? 0u : (n >= 32 ? 0xffffffffu : ((1u << n) - 1u)); }

// ltw / gtw: word (lane & 7) of the below- / above-threshold masks, held by the lane itself
__device__ __forceinline__ int fsm_closed_run_lanes(unsigned ltw, unsigned gtw, int from, int nvalid, int n_T1,
                                                    int half_pw, GateFsm2& st)
{
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int w = lane & 7;
  const bool own = lane < 8;
  const int base = 32 * w;
  const unsigned live = own ? ~m_below(from - base) : 0u;   // (lanes 8..31 carry empty words)
  const unsigned F = ltw & live, R = gtw & live;
  const unsigned Pk = ~(F | R);
  const unsigned long long sum0 = (unsigned long long)(R | Pk) + R, sum1 = sum0 + 1ull;
  const unsigned C0 = __ballot_sync(FULL, own && (sum0 >> 32) != 0ull) & 0xffu;
  const unsigned C1 = __ballot_sync(FULL, own && (sum1 >> 32) != 0ull) & 0xffu;
  const unsigned cv = (C1 + C0 + (st.sig_pos ? 1u : 0u)) ^ C1 ^ C0;   // bit k: carry into word k (C0 is a subset of C1)
  const unsigned X = Pk ^ (unsigned)(((cv >> w) & 1u) ? sum1 : sum0);   // state before each position
  const unsigned RS = ~X & R, FE = X & F, E = RS | FE;
  const int e_first = __reduce_min_sync(FULL, E ? base + __ffs(E) - 1 : 1024);
  const int e_last = __reduce_max_sync(FULL, E ? base + 31 - __clz(E) : -1);
  const int r_last = __reduce_max_sync(FULL, RS ? base + 31 - __clz(RS) : -1);
  const unsigned fe_prev = __shfl_up_sync(FULL, FE, 1);
  const int first_edge = e_first < nvalid ? e_first : nvalid;
  if (st.sig_pos && st.num_pulses > kNumPulsesCommand) {
    const int p_open = from + max(0, n_T1 - st.n_samples);
    if (p_open < first_edge && p_open < nvalid) {
      st.sig_pos = true; st.num_pulses = 0; st.n_samples = 1;
      return p_open;
    }
  }
  if (e_first >= nvalid) { st.n_samples += nvalid - from; return -1; }
  const unsigned fe_lo = w == 0 ? 0u : fe_prev;
  unsigned knock = 0u;
  for (int k = 1; k <= half_pw; k++) knock |= (FE << k) | (fe_lo >> (32 - k));
  unsigned VR = RS & ~knock;
  // the first edge, if it is a rise: its pulse began before the run
  if ((e_first >> 5) == w && ((RS >> (e_first & 31)) & 1u) && !(st.n_samples + (e_first - from + 1) > half_pw))
    VR &= ~(1u << (e_first & 31));
  const unsigned IR = RS & ~VR;
  const int np_in = st.num_pulses;
  const int lim = nvalid - 1 - n_T1;  // rises at or above lim cannot open the gate within this tile
  // (host: n_T1 + 1 >= 32.)  A rise that opens the gate is followed by n_T1 + 1 edge-free positions; when that is 64 or
  // more, the stretch covers a whole mask word, so a tile without an edge-free word below nvalid has no candidate.
  if (lim > 0 && (n_T1 + 1 < 64 || __any_sync(FULL, own && base < nvalid && E == 0u))) {
    auto first_of = [&](unsigned m) { return __reduce_min_sync(FULL, m ? base + __ffs(m) - 1 : 1024); };
    auto last_of = [&](unsigned m) { return __reduce_max_sync(FULL, m ? base + 31 - __clz(m) : -1); };
    auto np_at = [&](int r) {  // num_pulses right after the rise at r
      const unsigned upto = m_below(r + 1 - base);
      const int last = last_of(IR & upto);
      const unsigned rng = upto & ~m_below(last + 1 - base);
      const int cnt = __reduce_add_sync(FULL, __popc(VR & rng));
      return last >= 0 ? cnt : np_in + cnt;
    };
    // inside its own word an opening rise is the highest edge; the first edge of the words above it (suffix minimum over
    // the lanes) decides.  At most nvalid / (n_T1 + 1) rises qualify, so the loop below runs once or twice.
    const int hi = E ? 31 - __clz(E) : -1;
    const int fe = E ? base + __ffs(E) - 1 : 1024;
    int nx = __shfl_down_sync(FULL, fe, 1);
    if (w == 7) nx = 1024;
    {
      int t1 = __shfl_down_sync(FULL, nx, 1); if (w >= 6) t1 = 1024; nx = min(nx, t1);
      int t2 = __shfl_down_sync(FULL, nx, 2); if (w >= 5) t2 = 1024; nx = min(nx, t2);
      int t4 = __shfl_down_sync(FULL, nx, 4); if (w >= 3) t4 = 1024; nx = min(nx, t4);
    }
    const int rr = base + hi;
    const bool q = own && hi >= 0 && ((RS >> hi) & 1u) && rr < lim && nx > rr + 1 + n_T1;
    unsigned cand = q ? (1u << hi) : 0u;
    while (true) {
      const int r = first_of(cand);
      if (r >= 1024) break;
      if (own && (r >> 5) == w) cand &= ~(1u << (r & 31));
      const unsigned quiet_rng = m_below(r + 2 + n_T1 - base) & ~m_below(r + 1 - base);
      if (!__any_sync(FULL, (E & quiet_rng) != 0u) && np_at(r) > kNumPulsesCommand) {
        st.sig_pos = true; st.num_pulses = 0; st.n_samples = 1;
        return r + 1 + n_T1;
      }
    }
  }
  st.sig_pos = e_last == r_last;            // the last edge is a rise
  st.n_samples = nvalid - 1 - e_last;
  if (r_last >= 0) {
    // valid rises after the last invalid one: the words above the last word that holds an invalid rise, and that word's
    // bits above it
    const unsigned Lm = __ballot_sync(FULL, IR != 0u) & 0xffu;
    unsigned mine = VR;
    if (Lm) {
      const int L = 31 - __clz(Lm);
      if (w < L) mine = 0u;
      else if (w == L && IR) mine = VR & ~((2u << (31 - __clz(IR))) - 1u);
    }
    const int cnt = __reduce_add_sync(FULL, own ? __popc(mine) : 0);
    st.num_pulses = Lm ? cnt : np_in + cnt;
  }
  return -1;
}

template <int DECIM, int MFQ>
__global__ void __launch_bounds__(kPackMaxThreads, 1) rx_pack_kernel(const PackArgs A)
{
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ PackSegCtl ctl_all[kPMaxSeg];
  __shared__ PackCtaCtl cta;
  __shared__ unsigned warps_done;
  stamp_cta_start(A.stamps);
#ifdef RFID_B200_PHASE_PROFILE
  __shared__ long long pp_cta_t0;
  if (threadIdx.x == 0) pp_cta_t0 = clock64();
  int pp_step = 0;
  // per-CTA start / end on the global timer (ns): rows 512.. of the log
  unsigned long long* pp_cta = A.window_tap ? reinterpret_cast<unsigned long long*>(A.window_tap) + 512 * 8 + 2 * blockIdx.x : nullptr;
  if (pp_cta && threadIdx.x == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); pp_cta[0] = t; }
#endif

  static_assert(MFQ >= 2, "pack kernel: block-sum matched filter");
  constexpr int Q = kTT / 32;                // outputs per lane and half-tile
  static_assert(MFQ - 1 <= Q, "block-sum halo comes from the neighbouring lane only");
  static_assert(Q == 4, "four consecutive outputs per lane and half-tile");

  const int G = A.G;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int seg0 = blockIdx.x * G;
  const int g_act = min(G, A.nseg - seg0);   // segments this CTA really has
  const RxConfig& C = A.cfg;
  unsigned smid;
  asm("mov.u32 %0, %%smid;" : "=r"(smid));
  float2* const y_cta = A.y_hist + (size_t)smid * kPMaxSeg * kYW;

  float* const dA = reinterpret_cast<float*>(smem + A.off_dA);   // [kPAS][G][kPChainBuf]
  float* const dD = reinterpret_cast<float*>(smem + A.off_dD);   // [kPDS][2][G][kPChainBuf]

  // ---- init.  The loader warp initialises the raw-stage barriers itself and sends the first two half-tiles of every
  // segment on their way before it joins the start-up barrier; meanwhile the other warps initialise the hand-off barriers,
  // zero the rings (win_samples / dc_samples start at 0, gate_impl.cc:55-56) and read the segment lengths.
  int max_tiles = 0;
  if (warp == 3 * G) {
    if (lane < G) {
      PackSegCtl& c = ctl_all[lane];
      for (int s = 0; s < 2; s++) { mbar_init(&c.raw_full[s], 1); mbar_init(&c.raw_empty[s], s == 0 ? 2 : 1); }
      mbar_fence_init();
    }
    __syncwarp();
  } else {
    rfid_b200_segment sg0;       // (threads 0..G-1: the load is in flight while the barriers are initialised and the rings zeroed)
    sg0.offset = 0; sg0.length = 0; sg0.reserved = 0;
    if ((int)threadIdx.x < g_act) sg0 = A.segs[seg0 + threadIdx.x];
    if (threadIdx.x < G) {
      PackSegCtl& c = ctl_all[threadIdx.x];
      mbar_init(&c.half_rdy, 1); mbar_init(&c.tail_rdy, 1);
      for (int s = 0; s < kPAS; s++) mbar_init(&c.freeA[s], 1);
      for (int m = 0; m < 4; m++) { c.keep[0][m] = make_float2(0.f, 0.f); c.keep[1][m] = make_float2(0.f, 0.f); }
      for (int s = 0; s < kPDS; s++) { c.n_e[s] = 0; c.trig_n[s] = 0; }
      c.n_opened = 0; c.n_dc = 0; c.n_decoded = 0; c.seg_done = 0; c.y_tiles = 0;
      c.b_wcount = 0; c.b_nq = 1; c.b_snap_base = 0; c.b_queued = 0;
      mbar_fence_init();
    }
    if (threadIdx.x == 32) {
      for (int s = 0; s < kPAS; s++) { mbar_init(&cta.fullA[s], 2 * G); mbar_init(&cta.avgdone[s], 1); }
      for (int s = 0; s < kPDS; s++) { mbar_init(&cta.p3done[s], G); mbar_init(&cta.dcdone[s], 1); }
      warps_done = 0;
      mbar_fence_init();
    }
    for (int g = 0; g < G; g++) {
      unsigned char* sb = smem + A.off_seg + (size_t)g * A.seg_bytes;
      float4* ry = reinterpret_cast<float4*>(sb + A.o_tail_y);
      float4* ra = reinterpret_cast<float4*>(sb + A.o_ring_a);
      const int tid = threadIdx.x - (warp > 3 * G ? 32 : 0), nth = blockDim.x - 32;
      for (int i = tid; i < C.dc_length; i += nth) ry[i] = make_float4(0.f, 0.f, 0.f, 0.f);   // two tails of dc_length samples
      for (int i = tid; i < kRingA / 4; i += nth) ra[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (threadIdx.x < G) ctl_all[threadIdx.x].seg = sg0;
    asm volatile("bar.sync 14, %0;" ::"r"((int)blockDim.x) : "memory");   // start-up barrier (the loader joins it below)
    // the CTA holds its SM: the next launch may be scheduled (it gets SMs as this launch's CTAs exit)
    pdl_launch_dependents();
    // the CTA's barriers count every warp A / B for every tile of the longest segment
    for (int g = 0; g < g_act; g++) {
      const int n_out_g = (int)(ctl_all[g].seg.length / DECIM);
      max_tiles = max(max_tiles, (n_out_g + kT2 - 1) / kT2);
    }
  }

  if (warp < 3 * G) {
    // ======================================================================================= warps A0 / A1 (P1) and B (P3)
    const bool is_a = warp < 2 * G;
    const int ahalf = warp < G ? 0 : 1;       // which half-tile a P1 warp owns
    const int g = warp < G ? warp : (warp < 2 * G ? warp - G : warp - 2 * G);
    const bool have = g < g_act;
    const int seg = seg0 + g;
    rfid_b200_segment sg;
    sg.offset = 0; sg.length = 0; sg.reserved = 0;
    if (have) sg = ctl_all[g].seg;
    const int n_out = (int)(sg.length / DECIM);
    const int ntiles = (n_out + kT2 - 1) / kT2;
    PackSegCtl& B = ctl_all[g];
    unsigned char* sb = smem + A.off_seg + (size_t)g * A.seg_bytes;
    float2* raw = reinterpret_cast<float2*>(sb + A.o_raw);
    float2* tail_y = reinterpret_cast<float2*>(sb + A.o_tail_y);   // [2][dc_length]: the last outputs of either half-tile
    float* ring_a = reinterpret_cast<float*>(sb + A.o_ring_a);
    float2* const y_seg = y_cta + (size_t)g * kYW;
    auto bufA = [&](int tile) { return dA + (size_t)((tile % kPAS) * G + g) * kPChainBuf; };
    auto bufD = [&](int tile, int comp) { return dD + (size_t)(((tile % kPDS) * 2 + comp) * G + g) * kPChainBuf; };
    const float dclen_f = (float)C.dc_length;
    PP_DECL

    if (is_a) {
      // ------------------------------------------------------------------------------------- warps A0 / A1: P1 of one half-tile
      const int odd = (int)(sg.offset & 1ull);
      const float winlen_f = (float)C.win_length;
      const int h2 = ahalf;
#ifdef RFID_B200_PHASE_PROFILE
      if (seg == 0 && A.window_tap) pp_log = reinterpret_cast<long long*>(A.window_tap) + (h2 ? 256 * 8 : 0);
#endif
      for (int i = 0; i < max_tiles; i++) {
#ifdef RFID_B200_PHASE_PROFILE
        pp_step = i;
#endif
        PP_AT(0)
        const int k = 2 * i + h2;                      // half-tile index = tile index of the 128-sample kernels
        if (have && i < ntiles) {
          // the slots this tile is written into are free: warp B made the masks of tile i-3, the chain warp is through
          // with the DC list of tile i-4, and no queued window still needs the history samples about to be replaced
          if (i >= kPAS) pwait(&B.freeA[i % kPAS], (uint32_t)((i / kPAS - 1) & 1));
          if (i >= kPDS) pwait(&cta.dcdone[i % kPDS], (uint32_t)((i / kPDS - 1) & 1));
          if ((i + 1) * kT2 > kYW) {
            const int lowest = (i + 1) * kT2 - kYW;     // oldest history sample that survives this tile
            while (true) {
              const int nd = B.n_decoded, no = B.n_opened;
              const int need = nd < no ? B.q_open[nd & (kPQ - 1)] : 0x7fffffff;
              if (B.n_decoded == nd && need >= lowest) break;
              __nanosleep(200);
            }
          }
        } else if (i >= kPAS) {
          // nothing to compute (segment over, or no segment): keep step with the CTA so that this warp's arrival can never
          // fall into an earlier phase of the barrier
          pwait(&cta.avgdone[i % kPAS], (uint32_t)((i / kPAS - 1) & 1));
        }
        if (k * kTT < n_out) {
          const int nvalid = min(kTT, n_out - k * kTT);  // outputs of this half-tile
          const int t0 = Q * lane;
          const float2* stage = raw + (size_t)h2 * A.raw_stage_samples;
          const int delta = -odd - (k > 0 ? DECIM - 1 : 0);
          const int base = DECIM * t0 - (DECIM - 1) - delta;
          // ---- block sums B(n) = x[D*n-D+1 .. D*n], ascending
          float2 w[MFQ - 1 + Q];
          mbar_wait(&B.raw_full[h2], (uint32_t)(i & 1));
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
            } else {   // (first half-tile of a segment, odd offsets: one pass in 28 at most)
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
          // ---- the MFQ-1 block sums before this half-tile (lane 0's halo)
          float2 halo[MFQ - 1];
          if (h2 == 0) {
            // ... are the last ones of the previous tile: warp A1 left them in the keep slot (and the tile's second half in
            // the time rings, which the lookbacks below reach into)
            if (i >= 1) pwait(&B.tail_rdy, (uint32_t)((i - 1) & 1));
#pragma unroll
            for (int m = 0; m < MFQ - 1; m++) halo[m] = B.keep[(i + 1) & 1][m];
          } else {
            // ... are the last ones of the first half-tile: lanes 0..MFQ-2 recompute them from the tail of stage 0
            mbar_wait(&B.raw_full[0], (uint32_t)(i & 1));
            const float2* stage0 = raw;
            const int delta0 = -odd - (k - 1 > 0 ? DECIM - 1 : 0);
            const int tl = kTT - (MFQ - 1) + min(lane, MFQ - 2);          // output kTT-4 .. kTT-1 of half-tile 0
            const int b0 = DECIM * tl - (DECIM - 1) - delta0;
            float2 hb = stage0[b0];
#pragma unroll
            for (int j = 1; j < DECIM; j++) hb = c_add2(hb, stage0[b0 + j]);
#pragma unroll
            for (int m = 0; m < MFQ - 1; m++) halo[m] = make_float2(__shfl_sync(0xffffffffu, hb.x, m), __shfl_sync(0xffffffffu, hb.y, m));
          }
          __syncwarp();  // raw stages consumed: the loader may refill them
          if (lane == 0) { mbar_arrive(&B.raw_empty[h2]); if (h2 == 1) mbar_arrive(&B.raw_empty[0]); }
          PP_AT(1)
#pragma unroll
          for (int m = 0; m < MFQ - 1; m++) {
            const float2 mine = w[Q + m];
            const float ux = __shfl_up_sync(0xffffffffu, mine.x, 1), uy = __shfl_up_sync(0xffffffffu, mine.y, 1);
            w[m] = lane ? make_float2(ux, uy) : halo[m];
            if (h2 == 1) {  // hand the tile's last block sums to warp A0 (read after tail_rdy)
              const float ex = __shfl_sync(0xffffffffu, mine.x, 31), ey = __shfl_sync(0xffffffffu, mine.y, 31);
              if (lane == 0) B.keep[i & 1][m] = make_float2(ex, ey);
            }
          }
          // ---- y = sum of MFQ block sums (canonical order), a = |y| (gate_impl.cc:130)
          float2 y[Q];
          float a[Q];
          bool risky = false;
#pragma unroll
          for (int q = 0; q < Q; q++) {
            y[q] = w[q];
#pragma unroll
            for (int m = 1; m < MFQ; m++) y[q] = c_add2(y[q], w[q + m]);
            // outputs past the end of the segment (last, partial tile) are computed from stale shared memory: give them
            // a harmless value so that they cannot push the whole warp onto the rare exact-evaluation paths below
            if (nvalid < kTT && t0 + q >= nvalid) y[q] = make_float2(1.0f, 0.0f);
            bool rq;
            a[q] = cabsf_quick(y[q].x, y[q].y, rq);
            risky = risky || rq;
          }
          if (__any_sync(0xffffffffu, risky)) {  // rare (about one tile in 60): the exact evaluation for the whole warp
#pragma unroll
            for (int q = 0; q < Q; q++) a[q] = cabsf_ref_call(y[q].x, y[q].y);
          }
          const int ba = (i % kPAS) * kT2 + h2 * kTT;   // this half-tile's place in the |y| ring
          {
            const float4 y01 = make_float4(y[0].x, y[0].y, y[1].x, y[1].y), y23 = make_float4(y[2].x, y[2].y, y[3].x, y[3].y);
            *reinterpret_cast<float4*>(ring_a + ba + t0) = make_float4(a[0], a[1], a[2], a[3]);
            float4* hy = reinterpret_cast<float4*>(y_seg + ((i * kT2 + h2 * kTT + t0) & (kYW - 1)));   // the history
            hy[0] = y01;
            hy[1] = y23;
          }
          PP_AT(2)
          __syncwarp();  // this half-tile's |y| visible to the lookback below
          if (h2 == 1) pwait(&B.half_rdy, (uint32_t)(i & 1));   // the lookbacks reach into the first half
          // ---- ring differences (gate_impl.cc:131,141).  |y| from the time ring; y from dc_length samples back: the lane
          // dc_length / 4 below (same output slot), or -- for the first lanes -- the tail the previous half-tile left.
          // (host: window / DC lengths are multiples of 4, so the groups are aligned and never straddle the ring's end)
          float xd[Q], xr[Q], xi[Q];
          {
            int ia = ba + t0 - C.win_length;
            if (ia < 0) ia += kRingA;
            const float4 oa = *reinterpret_cast<const float4*>(ring_a + ia);
            xd[0] = f_sub(a[0], oa.x); xd[1] = f_sub(a[1], oa.y); xd[2] = f_sub(a[2], oa.z); xd[3] = f_sub(a[3], oa.w);
            const int dl = C.dc_length >> 2;                                   // lanes
            const float2* tprev = tail_y + (h2 ? 0 : C.dc_length);             // A0 reads A1's tail (previous tile), A1 reads A0's
            float4 t01 = make_float4(0.f, 0.f, 0.f, 0.f), t23 = t01;
            if (lane < dl) {
              t01 = *reinterpret_cast<const float4*>(tprev + 4 * lane);
              t23 = *reinterpret_cast<const float4*>(tprev + 4 * lane + 2);
            }
            float2 oy[Q];
#pragma unroll
            for (int q = 0; q < Q; q++) {
              oy[q].x = __shfl_up_sync(0xffffffffu, y[q].x, dl);
              oy[q].y = __shfl_up_sync(0xffffffffu, y[q].y, dl);
            }
            if (lane < dl) { oy[0] = make_float2(t01.x, t01.y); oy[1] = make_float2(t01.z, t01.w); oy[2] = make_float2(t23.x, t23.y); oy[3] = make_float2(t23.z, t23.w); }
#pragma unroll
            for (int q = 0; q < Q; q++) { xr[q] = f_sub(y[q].x, oy[q].x); xi[q] = f_sub(y[q].y, oy[q].y); }
            // this half-tile's own tail (the previous reader of that buffer is through: tail_rdy / half_rdy above)
            if (lane >= 32 - dl) {
              float4* tw = reinterpret_cast<float4*>(tail_y + (h2 ? C.dc_length : 0) + 4 * (lane - (32 - dl)));
              tw[0] = make_float4(y[0].x, y[0].y, y[1].x, y[1].y);
              tw[1] = make_float4(y[2].x, y[2].y, y[3].x, y[3].y);
            }
          }
          if (nvalid < kTT) {
#pragma unroll
            for (int q = 0; q < Q; q++)
              if (t0 + q >= nvalid) { xd[q] = 1.0f; xr[q] = 1.0f; xi[q] = 1.0f; }
          }
          // all twelve divisions in flight together; the multiply-correct quotients need every dividend in the verified range
          float mx = fabsf(xd[0]), mn = mx;
#pragma unroll
          for (int q = 0; q < Q; q++) {
            mx = fmaxf(fmaxf(mx, fabsf(xd[q])), fmaxf(fabsf(xr[q]), fabsf(xi[q])));
            mn = fminf(fminf(mn, fabsf(xd[q])), fminf(fabsf(xr[q]), fabsf(xi[q])));
          }
          const bool all_ok = C.win_div_fast && C.dc_div_fast && mn >= kDivFastMin && mx <= kDivFastMax;
          const bool warp_ok = __all_sync(0xffffffffu, all_ok);
          __syncwarp();
          // (every lane's lookback values have arrived, this half's tail is written: warp A1 may go on to the second half)
          if (h2 == 0 && lane == 0 && (k + 1) * kTT < n_out) mbar_arrive(&B.half_rdy);
          float qd[Q], qr[Q], qi[Q];
          if (warp_ok) {
#pragma unroll
            for (int q = 0; q < Q; q++) {
              qd[q] = f_div_fast(xd[q], winlen_f, C.win_recip);
              qr[q] = f_div_fast(xr[q], dclen_f, C.dc_recip);
              qi[q] = f_div_fast(xi[q], dclen_f, C.dc_recip);
            }
          } else {  // an exact zero, a denormal, or an unverified divisor somewhere in the warp: IEEE division
#pragma unroll
            for (int q = 0; q < Q; q++) {
              qd[q] = f_div_const_call(xd[q], winlen_f, C.win_recip, C.win_div_fast);
              qr[q] = f_div_const_call(xr[q], dclen_f, C.dc_recip, C.dc_div_fast);
              qi[q] = f_div_const_call(xi[q], dclen_f, C.dc_recip, C.dc_div_fast);
            }
          }
          if (nvalid < kTT) {
            // the segment's last, partial half-tile: the chain warp runs whole groups of 16 steps, so the slots past the
            // end hold -0.0f (x + -0.0f == x for every x, including both zeros: the running sum is carried unchanged)
#pragma unroll
            for (int q = 0; q < Q; q++)
              if (t0 + q >= nvalid) { qd[q] = -0.0f; qr[q] = -0.0f; qi[q] = -0.0f; }
          }
          *reinterpret_cast<float4*>(bufA(i) + h2 * kTT + t0) = make_float4(qd[0], qd[1], qd[2], qd[3]);
          *reinterpret_cast<float4*>(bufD(i, 0) + h2 * kTT + t0) = make_float4(qr[0], qr[1], qr[2], qr[3]);
          *reinterpret_cast<float4*>(bufD(i, 1) + h2 * kTT + t0) = make_float4(qi[0], qi[1], qi[2], qi[3]);
          __syncwarp();
          // second half-tile (and the halo) handed to warp A0's next tile
          if (h2 == 1 && lane == 0 && (k + 1) * kTT < n_out) mbar_arrive(&B.tail_rdy);
          // the tile's y is in the history (warp A1 got here after warp A0's half_rdy; a lone first half is the segment's last)
          if (lane == 0 && (h2 == 1 || (k + 1) * kTT >= n_out)) { __threadfence_block(); B.y_tiles = i + 1; }
        }
        PP_AT(3)
        __syncwarp();
        if (lane == 0) mbar_arrive(&cta.fullA[i % kPAS]);   // this half of tile i is ready for the chain warp
      }
      // the next launch's CTA on this SM rewrites the same history: this CTA's history stores are performed before it exits
      __threadfence();
    } else {
      // ------------------------------------------------------------------------------------- warp B: P3
      // the gate (gate_impl.cc:45, global_vars.cc:47, reader_impl.cc:259,262)
      bool sig_pos = false;
      int n_samples = 0, num_pulses = 0;
      bool gate_open = false;
      int to_ungate = C.len_rn16;
      bool terminated = false;
      bool was_quiet = true;      // the last tile with a closed run had no sample below its threshold
      int closed_since = C.dc_length;
      // (window count, queries, queue counters, ...: PackSegCtl::b_*, touched at gate events only.  b_snap_base = history
      // index of the DC ring's oldest entry when the last window opened)
      // y from the history; before the segment's first sample the rings hold +0 (gate_impl.cc:55-56)
      auto y_at = [&](int idx) { return idx >= 0 ? __ldcg(y_seg + (idx & (kYW - 1))) : make_float2(0.f, 0.f); };
#ifdef RFID_B200_PHASE_PROFILE
      if (seg == 0 && A.window_tap) pp_log = reinterpret_cast<long long*>(A.window_tap) + 64 * 8;
#endif
      for (int t = 0; t < max_tiles; t++) {
#ifdef RFID_B200_PHASE_PROFILE
        pp_step = t;
#endif
        PP_AT(0)
        pwait(&cta.avgdone[t % kPAS], (uint32_t)((t / kPAS) & 1));  // avg_ampl of tile t is final
        PP_AT(1)
        // ================================================================= P3(t): thresholds, state machine, DC list
        if (have && t < ntiles) {
          // room in the window queue for every window this tile can open (the oldest queued window has closed and its
          // dc_est is out or on its way: warp C does not depend on this warp to get through it)
          while (B.b_queued - B.n_decoded > kPQ - 1 - kPTrig) __nanosleep(200);
          const int s = t % kPDS;
          int n_e = 0, ntrig = 0;
          const int nvalid = min(kT2, n_out - t * kT2);
          const int tb = t * kT2;                     // history index of the tile's first sample
          const float* davg = bufA(t);
          const float* ta = ring_a + (t % kPAS) * kT2;
          float* er = bufD(t, 0);
          float* ei = bufD(t, 1);
          bool freed = false;
          auto release_a = [&]() {   // this tile's |y| and avg_ampl have been read for the last time
            if (!freed) { __syncwarp(); if (lane == 0) mbar_arrive(&B.freeA[t % kPAS]); freed = true; }
          };
          if (!terminated && gate_open && to_ungate - n_samples > nvalid) {
            // the whole tile lies inside an open window (gate_impl.cc:182-195): nothing to detect, no DC update
            release_a();
            n_samples += nvalid;   // (n_e = 0: the chain warp skips the tile)
          } else if (!terminated) {
            // thresholds (gate_impl.cc:136,148,154).  First a one-vote test in the lanes' natural 4-sample groups: while the
            // signal is high and no sample of the tile falls below its threshold, no edge can occur (carrier only).
            unsigned ltw = 0u, gtw = 0u;   // word (lane & 7) of the below- / above-threshold masks
            // (only tried when the previous tile was edge-free too: inside a reader command the test would fail every time)
            bool quiet = false;
            if (sig_pos && !gate_open && nvalid == kT2 && was_quiet) {
              bool below = false;
#pragma unroll
              for (int h2 = 0; h2 < 2; h2++) {
                const float4 av = *reinterpret_cast<const float4*>(davg + h2 * kTT + 4 * lane);
                const float4 aa = *reinterpret_cast<const float4*>(ta + h2 * kTT + 4 * lane);
                below = below || aa.x < f_mul(av.x, kThreshFraction) || aa.y < f_mul(av.y, kThreshFraction) ||
                        aa.z < f_mul(av.z, kThreshFraction) || aa.w < f_mul(av.w, kThreshFraction);
              }
              quiet = !__any_sync(0xffffffffu, below);
            }
            bool have_masks = false;
            auto make_masks = [&]() {
#pragma unroll
              for (int r = 0; r < 8; r++) {
                const int p = r * 32 + lane;
                const float thr = f_mul(davg[p], kThreshFraction);
                const float av = ta[p];
                const unsigned bl = __ballot_sync(0xffffffffu, av < thr), bg = __ballot_sync(0xffffffffu, av > thr);
                if ((lane & 7) == r) { ltw = bl; gtw = bg; }
              }
              if (nvalid < kT2) {
                const unsigned vm = m_below(nvalid - (lane & 7) * 32);
                ltw &= vm;
                gtw &= vm;
              }
              have_masks = true;
              release_a();
            };
            int pos = 0;
            while (pos < nvalid) {
              if (!gate_open) {
                const int run_start = pos;
                int p_open = -1;
                // (the one-vote result only covers a run that starts the tile with the signal high)
                PP_AT(4)
                if (!have_masks && !(quiet && run_start == 0)) make_masks();
                PP_AT(5)
                const bool no_lt = !__any_sync(0xffffffffu, ltw != 0u);
                was_quiet = no_lt;
                if (sig_pos && no_lt) {
                  // carrier only (the common case): no falling edge can occur, only the open test remains
                  if (num_pulses > kNumPulsesCommand) {
                    const int cand = run_start + max(0, C.n_T1 - n_samples);
                    if (cand < nvalid) { p_open = cand; num_pulses = 0; n_samples = 1; }
                  }
                  if (p_open < 0) n_samples += nvalid - run_start;
                } else {
                  GateFsm2 fs = {sig_pos, n_samples, num_pulses};
                  p_open = fsm_closed_run_lanes(ltw, gtw, run_start, nvalid, C.n_T1, C.n_PW / 2, fs);
                  sig_pos = fs.sig_pos; n_samples = fs.n_samples; num_pulses = fs.num_pulses;
                }
                PP_AT(6)
                const bool opened = p_open >= 0;
                pos = opened ? p_open + 1 : nvalid;
                // ---- DC tracker inputs of the closed run [run_start, pos) (gate_impl.cc:141-143; includes the trigger).
                // The list keeps the tile's natural positions: P1's time-contiguous differences are exact except for the
                // first dc_length samples after a window, whose ring entries date from before the window -- those are
                // recomputed here (y from the history); samples inside windows get -0.0f below (x + -0.0f == x).
                const int len = pos - run_start;
                if (closed_since < C.dc_length) {
                  const int nfix = min(len, C.dc_length - closed_since);
                  const int snap0 = B.b_snap_base;
#pragma unroll 1
                  for (int j0 = 0; j0 < nfix; j0 += 64) {
                    float2 yv[2], ov[2];
#pragma unroll
                    for (int u = 0; u < 2; u++) {
                      const int j = j0 + 32 * u + lane;
                      const bool valid = j < nfix;
                      yv[u] = y_at(tb + run_start + (valid ? j : 0));
                      ov[u] = y_at(snap0 + closed_since + (valid ? j : 0));
                    }
#pragma unroll
                    for (int u = 0; u < 2; u++) {
                      const int j = j0 + 32 * u + lane;
                      const bool valid = j < nfix;
                      const float xr = valid ? f_sub(yv[u].x, ov[u].x) : 1.0f, xi = valid ? f_sub(yv[u].y, ov[u].y) : 1.0f;
                      float qr, qi;
                      if (__all_sync(0xffffffffu, C.dc_div_fast && f_div_fast_ok(xr) && f_div_fast_ok(xi))) {
                        qr = f_div_fast(xr, dclen_f, C.dc_recip);
                        qi = f_div_fast(xi, dclen_f, C.dc_recip);
                      } else {
                        qr = f_div_const_call(xr, dclen_f, C.dc_recip, C.dc_div_fast);
                        qi = f_div_const_call(xi, dclen_f, C.dc_recip, C.dc_div_fast);
                      }
                      if (valid) { er[run_start + j] = qr; ei[run_start + j] = qi; }
                    }
                  }
                }
                PP_AT(7)
                closed_since = min(closed_since + len, 1 << 24);
                n_e = pos;
                if (opened) {
                  // READER COMMAND DETECTED (gate_impl.cc:164-180): the DC ring stands as it is now
                  gate_open = true;
                  const int open_idx = tb + pos - 1, wcount = B.b_wcount, n_queued = B.b_queued;
                  // a window is decoded when it closes inside the segment (its length is known now); windows beyond
                  // max_windows are not decoded
                  const bool cur_store = wcount < A.max_windows && ntrig < kPTrig && open_idx + to_ungate <= n_out;
                  __syncwarp();
                  if (lane == 0) {
                    B.b_snap_base = open_idx - C.dc_length + 1;
                    if (cur_store) {
                      // queue the window for warp C; dc_est right after the trigger sample follows from the chain warp
                      const int qs = n_queued & (kPQ - 1);
                      B.q_open[qs] = open_idx; B.q_kind[qs] = wcount & 1; B.q_ord[qs] = wcount;
                      B.trig_j[s][ntrig] = pos - 1; B.trig_k[s][ntrig] = n_queued;
                      B.b_queued = n_queued + 1;
                      __threadfence_block();
                      B.n_opened = n_queued + 1;
                    }
                  }
                  __syncwarp();
                  if (cur_store) ntrig++;
                }
              } else {
                // ---- open: samples pass through (gate_impl.cc:182-195); warp C reads them from the history.  They do not
                // enter the DC tracker: their list entries carry the running sums unchanged
                const int take = min(to_ungate - n_samples, nvalid - pos);
                for (int j = lane; j < take; j += 32) { er[pos + j] = -0.0f; ei[pos + j] = -0.0f; }
                n_samples += take; pos += take;
                n_e = pos;
                if (n_samples >= to_ungate) {
                  gate_open = false;
                  const int wcount = B.b_wcount, nq = B.b_nq;
                  const int kind = wcount & 1;  // windows alternate RN16, EPC (SURVEY.md 3.5)
                  __syncwarp();
                  if (lane == 0) {
                    B.b_wcount = wcount + 1;
                    if (kind) B.b_nq = nq + 1;
                  }
                  __syncwarp();
                  closed_since = 0;
                  // ACK after RN16 -> GATE_SEEK_EPC, Query/QueryRep after EPC -> GATE_SEEK_RN16 (gate_impl.cc:112-123)
                  to_ungate = kind ? C.len_rn16 : C.len_epc;
                  n_samples = 0;
                  if (kind && nq + 1 > C.max_queries) { terminated = true; break; }  // gate_impl.cc:101-109
                }
              }
            }
          }
          release_a();
          if (terminated) {
            // the list ends where the reader stopped: pad its last group of 16 with -0.0f (see P1)
            const int n16 = (n_e + 15) & ~15;
            if (lane < 16 && n_e + lane < n16) { er[n_e + lane] = -0.0f; ei[n_e + lane] = -0.0f; }
          }
          if (lane == 0) { B.n_e[s] = n_e; B.trig_n[s] = ntrig; }
        }
        PP_AT(2)
        __syncwarp();
        if (lane == 0) mbar_arrive(&cta.p3done[t % kPDS]);   // the tile's DC list is final
      }
      // ---- end of the segment (the previous launch may have written the same counts)
      pdl_wait();
      if (have && lane == 0) A.counts[seg] = B.b_wcount;
      if (lane == 0) { __threadfence_block(); B.seg_done = 1; }
    }
  } else if (warp == 3 * G + 1) {
    // ======================================================================================= chain warp
    // lane 8*c + g: running sum c (0 avg_ampl, 1 dc_est.re, 2 dc_est.im) of segment g
    const int comp = lane >> 3, g = lane & 7;
    const bool active = comp < 3 && g < g_act;
    int n_out = 0;
    if (active) n_out = (int)(ctl_all[g].seg.length / DECIM);
    float acc = 0.f;
    PP_DECL
#ifdef RFID_B200_PHASE_PROFILE
    if (blockIdx.x == 0 && A.window_tap) pp_log = reinterpret_cast<long long*>(A.window_tap) + 128 * 8;
#endif
    // avg_ampl of tile ia as soon as every segment's P1(ia) is in, dc_est of tile id as soon as every segment's P3(id) has
    // fixed its list -- whichever is ready, both in ONE convergent loop when both are
    int ia = 0, id = 0;
    while (ia < max_tiles || id < max_tiles) {
      PP_AT(0)
      bool ra = false, rd = false;
      while (true) {
        ra = ia < max_tiles && mbar_test_wait(&cta.fullA[ia % kPAS], (uint32_t)((ia / kPAS) & 1));
        rd = id < ia && mbar_test_wait(&cta.p3done[id % kPDS], (uint32_t)((id / kPDS) & 1));
        if (ra || rd) break;
        __nanosleep(20);
      }
#ifdef RFID_B200_PHASE_PROFILE
      pp_step = ra ? ia : 32 + id;
#endif
      PP_AT(1)
      {
        // branch-free selection of this lane's buffer and length
        const int n_avg = ra ? min(kT2, max(0, n_out - ia * kT2)) : 0;
        const int n_dc = (rd && active && comp > 0) ? ctl_all[g].n_e[id % kPDS] : 0;
        const int n = active ? (comp == 0 ? n_avg : n_dc) : 0;
        const int ofsA = ((ia % kPAS) * G + g) * kPChainBuf;
        const int ofsD = (((id % kPDS) * 2 + (comp - 1)) * G + g) * kPChainBuf;
        float* buf = comp == 0 ? dA + (ia < max_tiles ? ofsA : 0) : dD + (active && comp > 0 && id < max_tiles ? ofsD : 0);
        const int n16 = (n + 15) & ~15;
        __syncwarp();
        chain_inplace(buf, n16, acc);
        __syncwarp();
        if (ra) {
          if (lane == 0) mbar_arrive(&cta.avgdone[ia % kPAS]);
          ia++;
        }
        // ---- dc_est right after the trigger sample of every queued window that opened in tile id: hand it to warp C
        if (rd) {
          if (active && comp > 0) {
            PackSegCtl& S = ctl_all[g];
            const int s = id % kPDS;
            const int tn = S.trig_n[s];
            for (int e = 0; e < tn; e++) {
              const float v = buf[S.trig_j[s][e]];
              float* dst = reinterpret_cast<float*>(&S.dc_val[S.trig_k[s][e] & (kPQ - 1)]);
              dst[comp - 1] = v;
            }
          }
          __syncwarp();
          if (active && comp == 1) {
            PackSegCtl& S = ctl_all[g];
            const int tn = S.trig_n[id % kPDS];
            if (tn > 0) { __threadfence_block(); S.n_dc = S.n_dc + tn; }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&cta.dcdone[id % kPDS]);
          id++;
        }
      }
      PP_AT(2)
    }
  } else if (warp == 3 * G) {
    // ======================================================================================= loader warp
    // lane g streams the raw half-tiles of segment g through its two stages (TMA bulk copies) as warp A frees them; the
    // first two go out before the start-up barrier
    const int g = lane;
    rfid_b200_segment sg;
    sg.offset = 0; sg.length = 0; sg.reserved = 0;
    if (g < g_act) sg = A.segs[seg0 + g];
    const int n_out = (int)(sg.length / DECIM);
    const int nhalf = g < g_act ? (n_out + kTT - 1) / kTT : 0;
    PackSegCtl& B = ctl_all[g < G ? g : 0];
    float2* raw = reinterpret_cast<float2*>(smem + A.off_seg + (size_t)(g < G ? g : 0) * A.seg_bytes + A.o_raw);
    // raw half-tile geometry (as rx_fused_split.cuh)
    const int odd = (int)(sg.offset & 1ull);
    const uint32_t fast_bytes = (uint32_t)((DECIM * kTT + 2 * odd) * 8);
    int fast_tiles = 0;
    {
      const long long by_len = ((long long)sg.length - 1 - (long long)DECIM * (kTT - 1)) / ((long long)DECIM * kTT);
      const long long room = (long long)A.n_raw - (long long)sg.offset + (DECIM - 1) + odd - (DECIM * kTT + 2 * odd);
      const long long by_buf = room >= 0 ? room / ((long long)DECIM * kTT) : -1;
      long long f = (by_len < by_buf ? by_len : by_buf) + 1;
      if (sg.length < (unsigned)(DECIM * kTT)) f = 0;
      fast_tiles = f < 0 ? 0 : (f > nhalf ? nhalf : (int)f);
    }
    const float2* const fast_src = A.iq + sg.offset - (DECIM - 1) - odd;
    FusedArgs FA;  // issue_tile_load only reads iq / n_raw
    FA.iq = A.iq; FA.n_raw = A.n_raw;
    const unsigned long long pol = l2_policy_evict_first();   // every raw sample is read exactly once
    auto issue = [&](int k) {
      const int rs_ = k & 1;
      float2* dst = raw + (size_t)rs_ * A.raw_stage_samples;
      if (k >= 1 && k < fast_tiles) {
        mbar_arrive_expect_tx(&B.raw_full[rs_], fast_bytes);
        tma_load_1d_hint(dst, fast_src + (size_t)k * (DECIM * kTT), fast_bytes, &B.raw_full[rs_], pol);
      } else {
        issue_tile_load<DECIM>(FA, sg, k, dst, &B.raw_full[rs_]);
      }
    };
    for (int k = 0; k < 2 && k < nhalf; k++) issue(k);   // both stages are free at the start
    __syncwarp();
    asm volatile("bar.sync 14, %0;" ::"r"((int)blockDim.x) : "memory");   // start-up barrier
    pdl_launch_dependents();
    for (int k = 2; k < nhalf; k++) {
      mbar_wait_idle(&B.raw_empty[k & 1], (uint32_t)(((k >> 1) - 1) & 1), 100);
      issue(k);
    }
    // the CTA does not complete before the previous launch has (warps B / C may have stored nothing)
    pdl_wait();
  } else {
    // ======================================================================================= warp C: decode
    const int g = warp - 3 * G - 2;
    if (g < g_act) {
      const int seg = seg0 + g;
      PackSegCtl& B = ctl_all[g];
      unsigned char* sb = smem + A.off_seg + (size_t)g * A.seg_bytes;
      float2* dstage = reinterpret_cast<float2*>(sb + A.o_dstage);
      const float2* const y_seg = y_cta + (size_t)g * kYW;
      PP_DECL
#ifdef RFID_B200_PHASE_PROFILE
      if (seg == 0 && A.window_tap) pp_log = reinterpret_cast<long long*>(A.window_tap) + 192 * 8;
#endif
      for (int k = 0;;) {
        // the next queued window: decodable as soon as its last sample is in the history (warp A runs ahead of the gate)
        // and dc_est right after its trigger sample has come from the chain warp (two tiles after the gate opened it)
        const int done = B.seg_done;   // (read before the counter: once set, the counter is final)
        const int no = B.n_opened;
        if (no <= k) {
          if (done) break;
          __nanosleep(400);            // nothing to do until warp B opens a window
          continue;
        }
        __threadfence_block();
#ifdef RFID_B200_PHASE_PROFILE
        pp_step = k;
#endif
        PP_AT(0)
        {
          const int qs0 = k & (kPQ - 1);
          const int wend = B.q_open[qs0] + (B.q_kind[qs0] ? C.len_epc : C.len_rn16);
          while (B.y_tiles * kT2 < wend || B.n_dc <= k) __nanosleep(200);
        }
        __threadfence_block();
        const int qs = k & (kPQ - 1);
        const int kind = B.q_kind[qs], ord = B.q_ord[qs], wopen = B.q_open[qs];
        const float2 dc = B.dc_val[qs];
        const int len = kind ? C.len_epc : C.len_rn16;
        const WinSrc wv{y_seg, wopen, kYW - 1};
        PP_AT(1)
        WindowDecode wd;
#ifdef RFID_B200_PHASE_PROFILE
        decode_window_staged(C, kind, wv, len, dstage, A.dstage_samples, wd, nullptr, nullptr, dc, pp_log ? pp_log + (kind ? 60 : 61) * 8 : nullptr);
#else
        decode_window_staged(C, kind, wv, len, dstage, A.dstage_samples, wd, nullptr, nullptr, dc);
#endif
        rfid_b200_window_result* dst = A.results + (size_t)seg * A.max_windows + ord;
        if (k == 0) pdl_wait();   // the previous launch may have written the same records / window tap
        if (lane == 0) store_result(dst, wd, seg + A.seg_base, ord, wopen, len, kind);
#ifndef RFID_B200_PHASE_PROFILE
        if (A.window_tap) {
          float2* tap = A.window_tap + ((size_t)(seg + A.seg_base) * A.max_windows + ord) * C.len_epc;
          for (int p2 = lane; p2 < len; p2 += 32) tap[p2] = c_sub(__ldcg(wv.at(p2)), dc);
        }
#endif
        __syncwarp();
        k++;
        if (lane == 0) { __threadfence_block(); B.n_decoded = k; }   // warp A may reuse the window's history samples
        PP_AT(2)
      }
#ifdef RFID_B200_PHASE_PROFILE
      if (pp_cta && lane == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); atomicMax(pp_cta + 1, t); }
#endif
    }
  }
  stamp_warp_end(A.stamps, &warps_done);
}

}  // namespace rfid_b200
