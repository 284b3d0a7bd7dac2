// Fast lattice (v4): block-exponent fp32 alpha/beta recursion, eight lattice states per lane,
// packed f32x2 arithmetic, forward and backward sweeps running concurrently in one CTA and meeting
// in the middle, posterior reduction and gradient-row write-back on dedicated reducer warps.
//
// Arithmetic.  The recursion of SURVEY Appendix A is evaluated in the LINEAR domain:
//     alpha_t(s) = y_t(l'_s) * (alpha_{t-1}(s) + alpha_{t-1}(s-1) + [skip] alpha_{t-1}(s-2))
// Each lane owns eight consecutive lattice positions as fp32 mantissas plus ONE int32 power-of-two
// exponent that is renormalised after every frame, so the representable range is unbounded while
// the inner loop is FADD2/FMUL2/FFMA2 + integer exponent arithmetic: no exp/log at all (the softmax
// probabilities y come from K1).  Relative rounding error is ~6e-8 per operation independent of
// |log alpha| -- this is what keeps T=1500 utterances inside the 1e-4 gradient tolerance where an
// fp32 log-space recursion does not (DESIGN.md, "numerics").  The one weakness -- a state more than
// ~2^-110 below its lane's largest state loses bits -- is harmless unless that state could carry
// posterior mass; phase 2 bounds that mass for every lane and frame, and if the bound is not
// negligible (FLAG_PRECISION_LOST) the utterance is redone by the fp64 safe lattice in the same CTA.
//
// Packing.  The eight values of a lane live in four 64-bit registers, pair j = elements (j, j+4)
// (forward side: low word = element j; backward side: low word = element j+4).  With that pairing
// the neighbour terms of the recursion are again whole pairs -- element j-1 of pair j is pair j-1 --
// so one FADD2/FFMA2/FMUL2 (sm_100 packed fp32) advances two lattice states, and the mirrored pairing
// of the two sides makes the stored values of one side load as ready-made pairs on the other.
//
// Schedule.  One CTA per utterance, 2*(NWMAX+K) warps.  Per side: NW lattice warps (forward: alpha,
// t = 0,1,..; backward: beta on the reversed label sequence, t = T-1,T-2,..) and K helper warps.
// Phase 1: each side covers half of the frames and stores its pre-emission values to the scratch.
// Phase 2 (after one CTA barrier): each side continues through the other half, multiplies its fresh
// values with the stored ones of the opposite side -- posterior(t,s) = alpha_t(s) * beta'_t(s) / P --
// and scatters the label posteriors into a symbol-sorted shared-memory row.  The reducer warps of the
// side (one frame of the chunk each) sum that row per symbol one chunk behind the lattice warps
// (named-barrier hand-off, double buffered) and turn the softmax row K1 left in the gradient buffer
// into  grad[t,b,:] = y - occupancy  with one store per warp (small vocabularies: every touched
// symbol of the frame lies in the same 128-byte row), or one RED per (frame, symbol) (gathered mode).
// Sequential depth is T frames instead of 2T, only half of alpha and beta ever goes through HBM, and
// nothing but the recursion itself is on the critical path.
//
// Lattice layout.  Lane l of warp w holds positions base_w + 8l .. +7, base_w = w*(256-2*KX):
// consecutive warp windows overlap by a halo of 2*KX positions (KX = 16 frames, four lanes).  Dependencies
// only point downwards (s-1, s-2), so a warp can run KX frames without talking to its neighbour while
// the garbage creeping up from its window bottom stays inside the halo; every KX frames the lattice
// warps of a side exchange halo lanes through shared memory.  K = 4 frames ("chunk") is the granularity
// of the shared-memory buffers: phase 1 runs KX/K chunks between two named barriers, phase 2 meets its
// helper warps at one named barrier per chunk (posterior hand-off) and exchanges halos at every fourth.
// Neighbour states inside a warp travel by __shfl_up.  The emission rows (cp.async, two exchanges ahead)
// and the opposite side's stored records of chunk c+1 (TMA bulk copies) are fetched by the helper warps
// while chunk c computes.
#pragma once

#include "lattice_common.cuh"
#include "lattice_safe.cuh"

namespace b200ctc {

// Developer timeline trace (tools/trace_lattice.py): compiled in only with -DB200CTC_TRACE.
#ifdef B200CTC_TRACE
constexpr int kTraceCap = 4096;
__device__ long long g_trace[64 * kTraceCap];
__device__ int g_trace_cnt[64];
__device__ int g_trace_cta = 0;               // which CTA (launch index) records its timeline
__device__ long long g_cta_time[2 * 2048];   // %globaltimer at entry / exit of every CTA of the last lattice launch
__device__ __forceinline__ void trace_event(int& cnt, int tag) {
  if (blockIdx.x == g_trace_cta && (threadIdx.x & 31) == 0 && cnt < kTraceCap) {
    g_trace[(threadIdx.x >> 5) * kTraceCap + cnt] = ((long long)clock64() << 8) | tag;
    ++cnt;
    g_trace_cnt[threadIdx.x >> 5] = cnt;
  }
}
#define B200CTC_TRACE_DECL(cnt) int cnt = 0
#define B200CTC_TRACE_EVENT(cnt, tag) trace_event(cnt, tag)
#else
#define B200CTC_TRACE_DECL(cnt) int cnt = 0
#define B200CTC_TRACE_EVENT(cnt, tag) do { (void)cnt; } while (0)
#endif

constexpr int kAbortExtremeRow = 2;  // abort word: K1 flagged the utterance (nothing was written yet); 1 = redo after a lost range
constexpr int kEZero = -(1 << 28);  // exponent of an all-zero lane
constexpr int kChunk = 4;           // frames per chunk (K)
constexpr int kLaneStates = 8;      // lattice states per lane (NS)
constexpr int kRowsRing = 4;        // emission-row ring, in halo-exchange intervals (KX/K chunks each): the reducers' one, the current one, the next (landed), the one after (in flight)
constexpr int kReducers = kChunk;   // reducer warps per side: warp j takes frame j of every phase-2 chunk
// Helper warps per side.  One CTA for both sides: kReducers warps that fetch (emission rows, records) AND reduce.
// Cluster variant (one side per CTA, an SM to itself): the two jobs on different warps -- kReducers fetchers and
// kReducers reducers -- because with one or two lattice windows the helper's fetch-then-reduce chain (~1500 cycles
// per chunk) is what arrives last at the chunk barrier.
template <bool CL>
__host__ __device__ constexpr int helper_warps() { return CL ? 2 * kReducers : kReducers; }
enum HelperRole { kFetchAndReduce = 0, kFetchOnly = 1, kReduceOnly = 2 };
// Cluster variant, warps of a CTA.  Warp i issues on SM sub-partition i % 4, and the lattice warps are the latency-
// critical ones: with one or two lattice windows the helper warps take the OTHER sub-partitions (a reducer next to
// the single lattice warp of C1 cost 5 % of the step), which leaves a few warp slots idle.
template <int NWMAX>
__host__ __device__ constexpr int cluster_block_warps() { return NWMAX == 2 ? 16 : 12; }
// w: lattice window (< NWMAX), NWMAX + h for helper h (0..3 fetch, 4..7 reduce), or -1 (idle)
template <int NWMAX>
__device__ __forceinline__ int cluster_warp_role(int warp) {
  if (NWMAX >= 4) return warp;                                     // 0..3 lattice, 4..11 helpers: two per sub-partition
  const int sp = warp & 3, slot = warp >> 2;
  if (warp < NWMAX) return warp;
  if (NWMAX == 2) return sp >= 2 ? NWMAX + slot * 2 + (sp - 2) : -1;           // sub-partitions 2, 3: four helpers each
  const int h = slot * 3 + sp - 1;                                 // NWMAX == 1: sub-partitions 1, 2, 3
  return (sp != 0 && h < 2 * kReducers) ? NWMAX + h : -1;
}
// Depth D of the record ring (phase 2), in chunks: the helper warps fetch the opposite side's records D - 1
// chunks ahead.  A bulk copy out of the HBM scratch takes ~2000 cycles under load -- longer than a chunk computes --
// so with a ring of two (fetch during chunk c what chunk c + 1 reads) its latency sits on the critical path of
// some chunks (B200: C3 -2 %, C5 -6 % with four, see experiments/README.md).  Chosen per launch
// (CallParams::oth_depth, lattice.cu): the deepest of 4, 3, 2 whose shared memory still holds the longest label
// sequence of the call -- in gathered mode the capacity is 195 / 210 / 226 labels.
constexpr int kOthDepthMax = 4;

// ---------------------------------------------------------------------------------------------
// PTX helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void named_bar_sync(int id, int count) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(int id, int count) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory");
}
// ---- thread-block cluster (the two-CTA variant: alpha sweep on one SM, beta sweep on another) ----
__device__ __forceinline__ unsigned cluster_ctarank() {
  unsigned r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// All threads of both CTAs.  Release/acquire at cluster scope: global and shared writes before the barrier are
// visible to the other CTA after it; the fence also orders them against the other CTA's TMA (async proxy) reads.
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("fence.proxy.async;" ::: "memory");
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
  asm volatile("fence.proxy.async;" ::: "memory");
}
__device__ __forceinline__ int ld_peer_s32(const int* local_ptr, unsigned peer_rank) {   // the same word in the peer CTA's shared memory
  unsigned a = (unsigned)__cvta_generic_to_shared(local_ptr), pa;
  int v;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(pa) : "r"(a), "r"(peer_rank));
  asm volatile("ld.shared::cluster.s32 %0, [%1];" : "=r"(v) : "r"(pa) : "memory");
  return v;
}
__device__ __forceinline__ void cp_async_4(void* smem, const void* gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_8(void* smem, const void* gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_16(void* smem, const void* gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---- TMA 1-D bulk copy (global -> shared, completion on an mbarrier) ----
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// Bounded wait (a bulk copy that never completes must not hang the GPU): false after ~2^22 polls.
__device__ __forceinline__ bool mbar_wait(unsigned long long* bar, unsigned parity) {
  for (int it = 0; it < (1 << 22); ++it) {
    unsigned done;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n" : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    if (done) return true;
  }
  return false;
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// 2^d for d <= 0 (0 when d < -126)
__device__ __forceinline__ float pow2_neg(int d) { return __int_as_float(max(d + 127, 0) << 23); }
// 2^d clamped to [2^-127 -> 0, 2^127]
__device__ __forceinline__ float pow2_clamped(int d) { return __int_as_float(min(max(d + 127, 0), 254) << 23); }

// ---- packed fp32 pairs (FADD2 / FMUL2 / FFMA2 on sm_100) ----
typedef unsigned long long f2;
__device__ __forceinline__ f2 f2_pack(float lo, float hi) {
  f2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ float f2_lo(f2 v) {
  return __uint_as_float((unsigned)(v & 0xffffffffull));
}
__device__ __forceinline__ float f2_hi(f2 v) {
  return __uint_as_float((unsigned)(v >> 32));
}
__device__ __forceinline__ f2 f2_add(f2 a, f2 b) {
  f2 r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f2 f2_mul(f2 a, f2 b) {
  f2 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f2 f2_fma(f2 a, f2 b, f2 c) {
  f2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
// pair (element j, element j+4) in the packing of SIDE
template <int SIDE>
__device__ __forceinline__ f2 mk(float xj, float xj4) { return SIDE ? f2_pack(xj4, xj) : f2_pack(xj, xj4); }
template <int SIDE>
__device__ __forceinline__ float el_j(f2 p) { return SIDE ? f2_hi(p) : f2_lo(p); }
template <int SIDE>
__device__ __forceinline__ float el_j4(f2 p) { return SIDE ? f2_lo(p) : f2_hi(p); }
__device__ __forceinline__ float f2_max(f2 a, f2 b) {  // max over the four floats of two pairs
  return fmaxf(fmaxf(f2_lo(a), f2_hi(a)), fmaxf(f2_lo(b), f2_hi(b)));
}

// ---------------------------------------------------------------------------------------------
// geometry shared by host (shared-memory sizing) and device.  NS = kLaneStates lattice states per lane.
// ---------------------------------------------------------------------------------------------
// Frames between two halo exchanges of neighbouring lattice windows (KX).  Consecutive windows overlap by
// 2*KX positions: dependencies only point downwards (s-1, s-2), so the garbage creeping up from a window's
// bottom stays inside the overlap for KX frames.  K (frames per chunk) sets the granularity of the
// shared-memory buffers and of the hand-off with the helper warps; phase 1 needs neither between two
// exchanges and runs KX/K chunks back to back without a barrier -- every barrier costs the recursion's
// dependent chain a pipeline drain and refill (~500 cycles against 140 per frame in steady state).
constexpr int kExchangeFrames = 4 * kChunk;

__host__ __device__ inline int fast_warps_needed(int L) {
  const int P = kLaneStates * ((2 * L + 1 + kLaneStates - 1) / kLaneStates);
  const int win = 32 * kLaneStates, own = win - 2 * kExchangeFrames;
  return P <= win ? 1 : 1 + (P - win + own - 1) / own;
}
// One frame of stored records ("frame block"), the same layout in the HBM scratch and in shared memory:
// NS/4 planes of JG float4 (the packed mantissa pairs of every position group) followed by JG int32
// exponents, padded to 16 bytes -- one TMA bulk copy moves a whole frame.
__host__ __device__ inline int frame_block_bytes(int L) {
  const int JG = (2 * L + 1 + kLaneStates - 1) / kLaneStates;
  return (kLaneStates / 4) * JG * 16 + ((JG + 3) & ~3) * 4;
}
// Symbol-sorted posterior row: the label posteriors of a frame grouped by symbol (label i sits at its rank
// in (symbol, position) order), every symbol's group padded to a multiple of four slots so that the
// reducers read it with LDS.128.  The padding slots are never written and stay zero.
__host__ __device__ inline int post_label_slots(int L, int V) {
  const int n_sym = L < V - 1 ? L : V - 1;
  return (L + 3 * n_sym + 3) & ~3;
}

struct FastSideSmem {
  float* rows;      // [kRowsRing * KX/K][K][RWS]   staged emission rows (+ a zero slot at index RW)
  unsigned char* oth;   // [D][K] frame blocks   the opposite side's stored records, a ring of chunks (+ one all-zero block)
  float* post;      // [2][K][PS]              symbol-sorted label posteriors + blank partials + dump slot
  float4* halo_m;   // [2][NWMAX][HL][NS/4]    halo lanes
  int* halo_e;      // [2][NWMAX][HL]
  float* red_m;     // [NWMAX]
  int* red_e;       // [NWMAX]
  unsigned long long* mbar;   // [kReducers][kOthDepthMax]   one mbarrier per helper warp and ring slot (TMA bulk copies of the records)
};

template <int NWMAX>
__host__ __device__ inline int post_stride(int L, int V) {  // floats per frame in the post buffer
  return post_label_slots(L, V) + NWMAX * 32 + 4;
}

template <int NWMAX>
__host__ __device__ inline size_t fast_side_bytes(int L, int RW, int V, int D) {
  constexpr int HL = 2 * kExchangeFrames / kLaneStates;
  constexpr int RCH = kRowsRing * kExchangeFrames / kChunk;   // chunk slots of the emission-row ring
  size_t b = 0;
  b += (size_t)(D * kChunk + 1) * frame_block_bytes(L);      // oth (+ the zero block)
  b += (size_t)2 * NWMAX * HL * (kLaneStates / 4) * 16;      // halo_m
  b += (size_t)RCH * kChunk * (size_t)(RW + 4) * 4;          // rows
  b += 2 * (size_t)kChunk * post_stride<NWMAX>(L, V) * 4;    // post
  b += (size_t)2 * NWMAX * HL * 4;                           // halo_e
  b += NWMAX * 8;                                            // red
  b += (size_t)kReducers * kOthDepthMax * 8 + 8;             // mbar
  return (b + 15) / 16 * 16;
}
constexpr int kReducerGroups = 64;    // reducer groups of the straight-line reducer path: two per lane
constexpr int kUntouchedMaxV = 256;   // the small-vocabulary (non-gathered) lattice never sees a larger vocabulary
// Dynamic shared memory of the fast lattice for label sequences up to L with nwmax lattice windows and a record
// ring D chunks deep: the utterance-wide tables (control words, lab, sorted, seg_start, seg_sym, slot_of_label,
// seg_slot, untouched; laid out by lattice_fast_utterance) and `sides` side blocks -- 2 when one CTA runs both
// sweeps, 1 in the cluster variant.
inline size_t fast_smem_bytes(const CallParams& p, int nwmax, int sides, int L, int D) {
  const int RW = p.gathered ? em_width_of(L) : (p.V + 3) / 4 * 4;
  size_t common = (size_t)(16 + 6 * L + 16 + 4 * kReducerGroups + (p.V <= kUntouchedMaxV ? p.V : 0)) * 4;
  common = (common + 15) / 16 * 16;
  const size_t side = nwmax == 1 ? fast_side_bytes<1>(L, RW, p.V, D)
                    : nwmax == 2 ? fast_side_bytes<2>(L, RW, p.V, D) : fast_side_bytes<4>(L, RW, p.V, D);
  return common + sides * side + 16;
}
template <int NWMAX>
__device__ __forceinline__ FastSideSmem carve_fast_side(unsigned char* base, int L, int RW, int V, int D) {
  constexpr int HL = 2 * kExchangeFrames / kLaneStates;
  constexpr int RCH = kRowsRing * kExchangeFrames / kChunk;
  FastSideSmem s;
  unsigned char* p = base;
  s.oth = p;                               p += (size_t)(D * kChunk + 1) * frame_block_bytes(L);
  s.halo_m = reinterpret_cast<float4*>(p); p += (size_t)2 * NWMAX * HL * (kLaneStates / 4) * 16;
  s.rows = reinterpret_cast<float*>(p);    p += (size_t)RCH * kChunk * (size_t)(RW + 4) * 4;
  s.post = reinterpret_cast<float*>(p);    p += 2 * (size_t)kChunk * post_stride<NWMAX>(L, V) * 4;
  s.halo_e = reinterpret_cast<int*>(p);    p += (size_t)2 * NWMAX * HL * 4;
  s.red_m = reinterpret_cast<float*>(p);   p += NWMAX * 4;
  s.red_e = reinterpret_cast<int*>(p);     p += NWMAX * 4;
  p = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(p) + 7) / 8 * 8);
  s.mbar = reinterpret_cast<unsigned long long*>(p);
  return s;
}

// Utterance-wide tables (shared by both sides).
struct FastCommon {
  int* abort_flag;     // set by any thread: the fast result cannot be trusted / used
  int* lab;            // [L]
  SymbolIndex ix;      // sorted / seg_start / seg_sym / n_seg
  int* slot_of_label;  // [L]    slot of label i in the symbol-sorted posterior row
  int* seg_slot;       // [n_seg+1] first slot of every symbol's group in the posterior row (a multiple of 4)
  int* max_n4;         // [0] iterations of a reducer's group sum (16-byte chunks), [1] number of reducer groups, [2] most pieces of one symbol
  // Reducer groups (small vocabularies, <= 64 of them).  Normally one per distinct symbol; when a few symbols
  // carry most of the labels (text: the space, 'e') their slot ranges are cut into pieces of at most max_n4[0]
  // chunks that different lanes sum, so that the reducers' trip count follows the AVERAGE group, not the largest.
  int* vg_base4;       // [64] first 16-byte chunk
  int* vg_n4;          // [64] chunks
  int* vg_sym;         // [64] symbol
  int* vg_cnt;         // [64] pieces of the symbol if this is its first piece (the lane that writes the entry), else 0
  int* untouched;      // [V] vocabulary entries that are neither the blank nor a label of the utterance (rescaled rows only)
  int* n_untouched;
};

// named barrier ids (0 is __syncthreads)
__device__ __forceinline__ int bar_chunk(int side) { return 1 + side * 2; }   // lattice + helper warps of a side, once per chunk
__device__ __forceinline__ int bar_total(int side) { return 2 + side * 2; }
constexpr int kBarMidpoint = 5;
// The one rendezvous of the two sides.  Phase 1's records were written with ordinary stores (generic proxy); the
// helper warps read them back with TMA bulk copies (async proxy) right after this barrier.  A CTA barrier orders
// generic accesses only: without the proxy fence a copy of the newest records -- the frames next to the midpoint
// -- could overtake the stores and deliver what the scratch held before (found with a poisoned workspace,
// tools/stress_repro.py --poison: one utterance in a few thousand got NaN or slightly rescaled rows; invisible
// whenever the scratch still holds the same call's records).
__device__ __forceinline__ void midpoint_sync(int count) {
  asm volatile("fence.proxy.async;" ::: "memory");
  named_bar_sync(kBarMidpoint, count);
}

// ---------------------------------------------------------------------------------------------
// per-lane state of a lattice warp.  NP = NS/2 packed pairs; pair j holds elements (j, j+NP).
// Label positions are the odd elements (forward) / even elements (backward); label slot m is element
// 2m+1 / 2m; label pair u (pair index 2u+1 / 2u) holds label slots (u, u + NP/2).
// ---------------------------------------------------------------------------------------------
struct LaneConst {
  int idxB[kLaneStates / 2];   // byte offset in the emission row of the label positions (zero slot if the position is a dummy)
  int idxB_blank;              // byte offset of the blank
  f2 Kf[kLaneStates / 4];      // skip-transition factors (1.0 allowed / 0.0 not) of the label pairs
  int posB[kLaneStates / 2];   // byte offset of the label positions in the symbol-sorted posterior row (dump slot if dummy)
  int blankB;                  // byte offset of this thread's blank partial sum in the posterior row
  int recB, expB;              // byte offsets of this lane's group in a frame block: first mantissa plane, exponent
  bool owned;                  // this lane's group belongs to the warp (not to the halo) and exists
  int group;                   // global position group (pos0 / NS)
};

struct LaneState {
  f2 A[kLaneStates / 2];
  int e;
};

__device__ __forceinline__ float lds_f32(const void* base, int byte_off) {
  return *reinterpret_cast<const float*>(reinterpret_cast<const char*>(base) + byte_off);
}
__device__ __forceinline__ void sts_f32(void* base, int byte_off, float v) {
  *reinterpret_cast<float*>(reinterpret_cast<char*>(base) + byte_off) = v;
}
__device__ __forceinline__ float f2_max_all(const f2 (&v)[4]) {   // max over the 8 floats, two levels deep
  const float t1 = fmax3(f2_lo(v[0]), f2_hi(v[0]), f2_lo(v[1]));
  const float t2 = fmax3(f2_hi(v[1]), f2_lo(v[2]), f2_hi(v[2]));
  const float t3 = fmaxf(f2_lo(v[3]), f2_hi(v[3]));
  return fmax3(t1, t2, t3);
}

// One frame of the recursion for one lane.  ACC: pre-emission sums at exponent E; st: the new
// emission-weighted state, renormalised.
template <int SIDE>
__device__ __forceinline__ void lattice_frame(LaneState& st, const LaneConst& lc, const void* __restrict__ row,
                                              bool lane0, f2 (&ACC)[kLaneStates / 2], int& E) {
  constexpr int NP = kLaneStates / 2;
  const float a_top = el_j4<SIDE>(st.A[NP - 1]), a_top2 = el_j4<SIDE>(st.A[NP - 2]);
  const float n1 = __shfl_up_sync(0xffffffffu, a_top, 1);
  const float n2 = __shfl_up_sync(0xffffffffu, a_top2, 1);
  int ne = __shfl_up_sync(0xffffffffu, st.e, 1);
  // emissions: one broadcast load for the blank positions, one gather per label position
  const float yb = lds_f32(row, lc.idxB_blank);
  float y[NP];
#pragma unroll
  for (int m = 0; m < NP; ++m) y[m] = lds_f32(row, lc.idxB[m]);
  if (lane0) ne = kEZero;                      // nothing below the window: scales n1, n2 to zero
  E = max(st.e, ne);
  const float so = pow2_neg(st.e - E), sn = pow2_neg(ne - E);
  const f2 so2 = f2_pack(so, so);
  f2 As[NP];
#pragma unroll
  for (int j = 0; j < NP; ++j) As[j] = f2_mul(st.A[j], so2);
  const float b1 = n1 * sn, b2 = n2 * sn;
  const f2 Q1 = mk<SIDE>(b1, el_j<SIDE>(As[NP - 1]));   // elements (-1, NP-1)
  const f2 Q2 = mk<SIDE>(b2, el_j<SIDE>(As[NP - 2]));   // elements (-2, NP-2)
  ACC[0] = f2_add(As[0], Q1);
#pragma unroll
  for (int j = 1; j < NP; ++j) ACC[j] = f2_add(As[j], As[j - 1]);
  const f2 YB = f2_pack(yb, yb);
  f2 W[NP];
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    const bool is_label = SIDE ? (j % 2 == 0) : (j % 2 == 1);
    if (is_label) {
      const int u = j / 2;                                  // label pair u: label slots (u, u + NP/2)
      const f2 below2 = j >= 2 ? As[j - 2] : (j == 1 ? Q1 : Q2);
      ACC[j] = f2_fma(lc.Kf[u], below2, ACC[j]);
      W[j] = f2_mul(ACC[j], mk<SIDE>(y[u], y[u + NP / 2]));
    } else {
      W[j] = f2_mul(ACC[j], YB);
    }
  }
  const float mx = f2_max_all(W);
  // renormalise: largest mantissa -> [1,2).  mx == 0 (or NaN from garbage): the lane is empty.
  const int eb = __float_as_int(mx) >> 23;                       // biased exponent
  const bool nz = mx > 0.f;
  const float sc = nz ? __int_as_float((254 - eb) << 23) : 0.f;  // 2^(127-eb)
  const f2 sc2 = f2_pack(sc, sc);
#pragma unroll
  for (int j = 0; j < NP; ++j) st.A[j] = f2_mul(W[j], sc2);
  st.e = nz ? E + eb - 127 : kEZero;
}

template <int SIDE>
struct FastCtx {
  const CallParams* p;
  int b, T, L, S, JG, FB, P, NW, RW, RWS, PS, RC, D;    // FB: bytes of a frame block; D: depth of the record ring
  int w, lane, tid_side;
  FastSideSmem sm;
  unsigned char* scr;   // [T] frame blocks: stored pre-emission pairs in the READER's group order and packing
  int per_row;                                // emission rows: cp.async copies per row
  const char* st_src; int st_stride;          // this lane's element of frame t at st_src + t*st_stride (bytes)
  unsigned st_dst; int st_vecB;               // shared address of this lane's element in row 0 of the ring; bytes per copy
  __device__ __forceinline__ int frame_of(int n) const { return SIDE ? T - 1 - n : n; }
};

// Frames [t0, t1] in which the lattice-state window [ws_lo, ws_hi] intersects the reachable band
// lo_t = max(0, S - 2(T-t)) <= s < hi_t = min(S, 2(t+1)); empty (t0 > t1) when it never does.
__device__ __forceinline__ void band_frames(int ws_lo, int ws_hi, int S, int T, int& t0, int& t1) {
  ws_hi = min(ws_hi, S - 1);
  t0 = ws_lo >> 1;
  t1 = T - ((S - ws_hi + 1) >> 1);
  if (ws_lo > ws_hi) { t0 = 1; t1 = 0; }
}

// Everything a lattice warp carries through the sweep.
struct SweepState {
  LaneState st;
  LaneConst lc;
  int act_lo, act_hi;       // steps in which the warp window intersects the reachable band (chunks outside are skipped)
  int rd_hi, wr_len;        // the other side stored this lane's record of step n iff (unsigned)(rd_hi - n) < wr_len
  float inv_mP; int eP;     // total probability P = mP * 2^eP (phase 2)
  int maxbound;             // running maximum of the range-check bound (phase 2), as a power-of-two exponent
  unsigned char* wblk;      // phase 1: this lane's slot in the frame block of the current step (running pointer)
  int wstep, weoff;         // its stride per step (0 for lanes that own no group: they hit the dump block) and exponent offset
};
constexpr int kLostBound = 127 + 110 - 24 - 2;   // maxbound above this: FLAG_PRECISION_LOST

// Helper warp: prefetch the opposite side's frame block of step n into slot `slot` (= buffer * K + frame)
// of the record ring with ONE TMA bulk copy.  Records the other side never wrote (its warp skipped the
// chunk: out of the band) arrive as garbage; the lattice lanes know which of their records exist
// (SweepState::rd_hi / wr_len) and read the all-zero block instead.
template <int SIDE>
__device__ __forceinline__ void prefetch_other(const FastCtx<SIDE>& c, int slot, int n, unsigned long long* mbar) {
  if (c.lane == 0) {
    mbar_expect_tx(mbar, (unsigned)c.FB);
    bulk_g2s(c.sm.oth + (size_t)slot * c.FB, c.scr + (size_t)c.frame_of(n) * c.FB, (unsigned)c.FB, mbar);
  }
}

// Helper warp: stage the emission row of the frame of step n into row `slot` (= ring slot * K + frame).
template <int SIDE>
__device__ __forceinline__ void stage_row_at(const FastCtx<SIDE>& c, unsigned dst, const char* src) {
#pragma unroll 1
  for (int e = c.lane; e < c.per_row; e += 32) {
    const unsigned d = dst + (unsigned)(e - c.lane) * (unsigned)c.st_vecB;
    const char* g = src + (e - c.lane) * c.st_vecB;
    if (c.st_vecB == 16) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(g) : "memory");
    else if (c.st_vecB == 8) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(g) : "memory");
    else asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(g) : "memory");
  }
}
template <int SIDE>
__device__ __forceinline__ void stage_row(const FastCtx<SIDE>& c, int slot, int n) {
  stage_row_at<SIDE>(c, c.st_dst + (unsigned)(slot * c.RWS * 4), c.st_src + (long long)c.frame_of(n) * c.st_stride);
}

// Posterior of one frame for one lane: the fresh renormalised state times the stored record of the
// opposite side, normalised by P:  post = a * o * 2^(e + oe - eP) / mP.  Scatters the label
// posteriors and the blank partial sum.  Every lane of the warp runs it and stores: lanes that own no
// group scatter into the dump slot, and a cost-only call points `post` at a dump row.
// No band masks: for every state outside the reachable band at least one factor is exactly zero
// (unreachable from this side's start: a == 0; unreachable from the other side's start: the stored
// value is 0, or the record was never written and reads as zero -- prefetch_other).
// The fresh state is normalised to [1,2) per lane, so the one scale factor cannot push a product
// that matters out of the fp32 range.
template <int SIDE>
__device__ __forceinline__ void posterior_frame(SweepState& ss, const unsigned char* __restrict__ blk, int plane_bytes,
                                                void* __restrict__ post) {
  constexpr int NP = kLaneStates / 2, NH = kLaneStates / 4;
  const LaneConst& lc = ss.lc;
  const LaneState& st = ss.st;
  f2 O[NP];
#pragma unroll
  for (int h = 0; h < NH; ++h) {
    const float4 q = *reinterpret_cast<const float4*>(blk + lc.recB + h * plane_bytes);
    O[2 * h] = f2_pack(q.x, q.y);
    O[2 * h + 1] = f2_pack(q.z, q.w);
  }
  const int oe = *reinterpret_cast<const int*>(blk + lc.expB);
  const int dexp = st.e + oe - ss.eP;
  const float s = pow2_clamped(dexp) * ss.inv_mP;   // inv_mP in (0.5, 1]
  const f2 s2 = f2_pack(s, s);
  f2 PO[NP];
#pragma unroll
  for (int j = 0; j < NP; ++j) PO[j] = f2_mul(f2_mul(st.A[j], O[j]), s2);
  // Range check.  A state that sits more than 2^-110 below its lane's largest value may have lost
  // bits (on either side).  Its posterior is bounded by
  //   2^-110 * max(own lane) * max(other lane) * 2^dexp / mP,   max(own lane) in [1,2);
  // if that bound is not negligible (> 2^-24) the block-exponent result cannot be trusted.  The own
  // maximum runs over ALL states of the lane: dead states (too late to finish) share the exponent.
  // Evaluated on the exponent fields (a zero maximum has field 0 and can only lower the bound), so
  // it cannot overflow or underflow; the running maximum is tested at the chunk boundary.
  // The stored values are sums of at most three renormalised mantissas (< 6, exponent field <= 129): while
  // dexp stays below kLostBound - 129 the bound holds whatever they are, and only the (rare) lanes beyond
  // that look at their maximum.
  if (dexp > kLostBound - 130) {
    const float omax = f2_max_all(O);
    ss.maxbound = max(ss.maxbound, (__float_as_int(omax) >> 23) + dexp);
  }
  {
    f2 bacc;
    bool first = true;
#pragma unroll
    for (int j = 0; j < NP; ++j) {
      const bool is_label = SIDE ? (j % 2 == 0) : (j % 2 == 1);
      if (is_label) {
        const int u = j / 2;
        sts_f32(post, lc.posB[u], el_j<SIDE>(PO[j]));
        sts_f32(post, lc.posB[u + NP / 2], el_j4<SIDE>(PO[j]));
      } else {
        bacc = first ? PO[j] : f2_add(bacc, PO[j]);
        first = false;
      }
    }
    sts_f32(post, lc.blankB, f2_lo(bacc) + f2_hi(bacc));
  }
}

// One chunk (kc <= K frames starting at step n0; emission rows in ring slot `rslot`).  A warp whose
// window misses the reachable band in all frames of the chunk skips it (warp-uniform).
template <bool PH2, int SIDE>
__device__ __forceinline__ void run_chunk(const FastCtx<SIDE>& c, SweepState& ss, int rslot, int pbuf, int obuf,
                                          int n0, int kc, bool write_post) {
  constexpr int NP = kLaneStates / 2, NH = kLaneStates / 4;
  const LaneConst& lc = ss.lc;
  const bool lane0 = c.lane == 0;
  const char* row = reinterpret_cast<const char*>(c.sm.rows + (size_t)rslot * kChunk * c.RWS);
  const int row_bytes = c.RWS * 4;
  const bool active = n0 <= ss.act_hi && n0 + kc - 1 >= ss.act_lo;
  if (!PH2) {
    if (!active) {
      ss.wblk += (long long)ss.wstep * kc;
      return;
    }
    // scratch slot of this lane's group for the opposite side's reader (mirrored group order)
    const int plane = c.JG * 16;
    const int eoff = ss.weoff;                                    // exponent slot relative to the first mantissa plane slot
    unsigned char* blk = ss.wblk;
#pragma unroll 2
    for (int j = 0; j < kc; ++j) {
      f2 ACC[NP]; int E;
      lattice_frame<SIDE>(ss.st, lc, row, lane0, ACC, E);
      // the reader's pair j is this lane's pair NP-1-j (mirrored group, mirrored packing); lanes that
      // own no group (halo, beyond the lattice) store into the dump block: no branch in the loop
#pragma unroll
      for (int h = 0; h < NH; ++h)
        asm volatile("st.global.v2.b64 [%0], {%1, %2};" ::"l"(blk + h * plane),
                     "l"(ACC[NP - 1 - 2 * h]), "l"(ACC[NP - 2 - 2 * h]) : "memory");
      *reinterpret_cast<int*>(blk + eoff) = E;
      row += row_bytes;
      blk += ss.wstep;
    }
    ss.wblk = blk;
  } else {
    // cost-only calls (no gradient buffer) walk phase 2 for the range check: their posteriors land in one dump row
    char* post = reinterpret_cast<char*>(c.sm.post + (size_t)pbuf * kChunk * c.PS);
    const int post_bytes = write_post ? c.PS * 4 : 0;
    const bool store = write_post;
    if (active) {
      const unsigned char* blk = c.sm.oth + (size_t)obuf * kChunk * c.FB;
      const unsigned char* zero_blk = c.sm.oth + (size_t)c.D * kChunk * c.FB;
      const int plane = c.JG * 16;
#pragma unroll 2
      for (int j = 0; j < kc; ++j) {
        f2 ACC[NP]; int E;
        lattice_frame<SIDE>(ss.st, lc, row, lane0, ACC, E);
        const bool wr = (unsigned)(ss.rd_hi - (n0 + j)) < (unsigned)ss.wr_len;   // did the other side store this record?
        posterior_frame<SIDE>(ss, wr ? blk : zero_blk, plane, post);
        row += row_bytes;
        post += post_bytes;
        blk += c.FB;
      }
    } else if (store) {
#pragma unroll 1
      for (int j = 0; j < kc; ++j) {
#pragma unroll
        for (int m = 0; m < NP; ++m) sts_f32(post, lc.posB[m], 0.f);
        sts_f32(post, lc.blankB, 0.f);
        post += post_bytes;
      }
    }
  }
}

// Chunk boundary of the lattice warps: publish the halo lanes, ONE barrier with the side's lattice and
// helper warps (after it the helpers' prefetch for the next chunk has landed and the posterior buffer
// of the previous chunk is consumed), import the halo.
template <int NWMAX, int SIDE, int HW>   // HW: helper warps of the side
__device__ __forceinline__ void chunk_boundary(const FastCtx<SIDE>& c, SweepState& ss, int cc, int* abort_flag, int& tc,
                                               bool exchange = true) {
  constexpr int NH = kLaneStates / 4, HL = 2 * kExchangeFrames / kLaneStates;
  static_assert(HL * kLaneStates == 2 * kExchangeFrames && HL >= 1, "the halo must be whole lanes");
  const int hb = cc & 1, NW = c.NW, w = c.w, lane = c.lane;
  LaneState& st = ss.st;
  if (exchange && w + 1 < NW && lane >= 32 - HL) {
    const int slot = (hb * NWMAX + w) * HL + (lane - (32 - HL));
#pragma unroll
    for (int h = 0; h < NH; ++h)
      c.sm.halo_m[slot * NH + h] = make_float4(f2_lo(st.A[2 * h]), f2_hi(st.A[2 * h]), f2_lo(st.A[2 * h + 1]), f2_hi(st.A[2 * h + 1]));
    c.sm.halo_e[slot] = st.e;
  }
  if (ss.lc.owned && ss.maxbound > kLostBound) *abort_flag = 1;
  B200CTC_TRACE_EVENT(tc, 30);
  named_bar_sync(bar_chunk(SIDE), (NW + HW) * 32);
  B200CTC_TRACE_EVENT(tc, 31);
  if (exchange && w > 0 && lane < HL) {
    const int slot = (hb * NWMAX + (w - 1)) * HL + lane;
#pragma unroll
    for (int h = 0; h < NH; ++h) {
      const float4 hv = c.sm.halo_m[slot * NH + h];
      st.A[2 * h] = f2_pack(hv.x, hv.y);
      st.A[2 * h + 1] = f2_pack(hv.z, hv.w);
    }
    st.e = c.sm.halo_e[slot];
  }
}

// Total probability from the per-warp partial sums (every thread of the side, reducers included,
// evaluates the same expression on the same shared values).  Returns false when the fast path must
// give up; otherwise mP in [1,2) and eP with P = mP * 2^eP, and log2(P) for the cost.
__device__ __forceinline__ bool total_probability(const FastSideSmem& sm, int NW, float& inv_mP, int& eP, double& log2P) {
  int Emax = kEZero;
  for (int i = 0; i < NW; ++i) Emax = max(Emax, sm.red_e[i]);
  float tot = 0.f;
  for (int i = 0; i < NW; ++i) tot += sm.red_m[i] * pow2_neg(sm.red_e[i] - Emax);
  if (!(tot > 0.f) || !(tot < INFINITY) || Emax <= kEZero / 2) return false;
  const int eb = (__float_as_int(tot) >> 23) - 127;
  const float mP = tot * pow2_clamped(-eb);
  inv_mP = 1.0f / mP;
  eP = Emax + eb;
  log2P = (double)Emax + log2((double)tot);
  return true;
}

template <int NWMAX, int SIDE>
__device__ __forceinline__ void fill_ctx(FastCtx<SIDE>& c, const CallParams& p, int b, const UttMeta& m,
                                         unsigned char* side_smem, int w, int lane) {
  c.p = &p; c.b = b;
  c.T = m.T; c.L = m.L; c.S = 2 * m.L + 1; c.JG = (c.S + kLaneStates - 1) / kLaneStates; c.FB = frame_block_bytes(m.L); c.P = kLaneStates * c.JG;
  c.NW = fast_warps_needed(m.L);
  c.RW = p.gathered ? m.W : (p.V + 3) / 4 * 4;
  c.RWS = c.RW + 4;
  c.PS = post_stride<NWMAX>(m.L, p.V);
  c.RC = c.PS - NWMAX * 32 - 4;                 // label slots come first, then the blank partials, then the dump slot
  c.w = w; c.lane = lane; c.tid_side = w * 32 + lane;
  c.D = p.oth_depth;
  c.sm = carve_fast_side<NWMAX>(side_smem, m.L, c.RW, p.V, c.D);
  c.scr = p.scratch + m.scratch_off * kGroupBytes;
  const float* row_src; long long row_stride; int row_vec;
  if (p.gathered) {
    row_src = p.em + m.em_off; row_stride = m.W; row_vec = 4; c.per_row = m.W / 4;
  } else {
    row_src = p.yrows + (long long)b * p.V; row_stride = (long long)p.B * p.V;
    const uintptr_t a = reinterpret_cast<uintptr_t>(p.yrows);
    row_vec = (p.V % 4 == 0 && a % 16 == 0) ? 4 : ((p.V % 2 == 0 && a % 8 == 0) ? 2 : 1);
    c.per_row = p.V / row_vec;
  }
  c.st_vecB = row_vec * 4;
  c.st_src = reinterpret_cast<const char*>(row_src) + lane * c.st_vecB;
  c.st_stride = (int)(row_stride * 4);          // api.cu rejects mini-batches whose frame stride exceeds 2^31 bytes
  c.st_dst = (unsigned)__cvta_generic_to_shared(c.sm.rows) + (unsigned)(lane * c.st_vecB);
}

struct SidePlan {
  int M_side, nc1, nc2, n_chunks;
};
__device__ __forceinline__ SidePlan side_plan(int T, int side) {
  SidePlan s;
  s.M_side = side ? (T / 2) : (T - T / 2);      // frames this side covers in phase 1
  s.nc1 = (s.M_side + kChunk - 1) / kChunk;
  s.nc2 = (T - s.M_side + kChunk - 1) / kChunk;
  s.n_chunks = s.nc1 + s.nc2;
  return s;
}

// ---------------------------------------------------------------------------------------------
// lattice warps of one side
// ---------------------------------------------------------------------------------------------
// CL: the two sides are the two CTAs of a thread-block cluster; the one rendezvous of the sides (midpoint) then is
// a cluster barrier instead of a named barrier.
template <int NWMAX, int SIDE, bool CL>
__device__ void fast_side_sweep(const CallParams& p, int b, const UttMeta& m, const FastCommon& cm,
                                unsigned char* side_smem, int w, int lane) {
  constexpr int NP = kLaneStates / 2, NH = kLaneStates / 4;
  constexpr int H = 2 * kExchangeFrames;                     // halo positions
  constexpr int RCH = kRowsRing * kExchangeFrames / kChunk;   // chunk slots of the emission-row ring
  constexpr int HL = H / kLaneStates;                         // halo lanes
  constexpr int WIN = 32 * kLaneStates;                       // positions per warp window
  constexpr int OWN = WIN - H;
  constexpr int OWNG = OWN / kLaneStates;                     // owned groups per warp

  FastCtx<SIDE> c;
  fill_ctx<NWMAX, SIDE>(c, p, b, m, side_smem, w, lane);
  const int T = c.T, S = c.S, JG = c.JG, P = c.P, NW = c.NW;
  const int* lab = cm.lab;

  // ---- per-lane constants ----
  SweepState ss;
  LaneConst& lc = ss.lc;
  const int base_w = w * OWN;
  const int pos0 = base_w + kLaneStates * lane;
  lc.group = pos0 / kLaneStates;
  lc.owned = ((w == 0) || (lane >= HL)) && (lc.group < JG);
  lc.idxB_blank = 4 * (p.gathered ? 0 : p.blank);
  lc.blankB = 4 * (lc.owned ? c.RC + c.tid_side : c.PS - 4);
  lc.recB = min(lc.group, JG - 1) * 16;
  lc.expB = NH * JG * 16 + min(lc.group, JG - 1) * 4;
  {
    float kk[NP];
#pragma unroll
    for (int mslot = 0; mslot < NP; ++mslot) {
      const int q = pos0 + (SIDE ? 2 * mslot : 2 * mslot + 1);   // label positions of the lane
      const int s = SIDE ? (P - 1 - q) : q;
      const bool ok = (q < P) && (s >= 0) && (s < S);             // s is odd by construction
      lc.idxB[mslot] = 4 * c.RW;            // zero slot
      lc.posB[mslot] = 4 * (c.PS - 4);      // dump slot
      kk[mslot] = 0.f;
      if (ok) {
        const int li = s >> 1;
        lc.idxB[mslot] = 4 * (p.gathered ? li + 1 : lab[li]);
        if (lc.owned) lc.posB[mslot] = 4 * cm.slot_of_label[li];   // halo lanes scatter into the dump slot
        const bool sk = SIDE ? (s + 2 < S && lab[li] != lab[li + 1]) : (s >= 3 && lab[li] != lab[li - 1]);
        kk[mslot] = sk ? 1.f : 0.f;
      }
    }
#pragma unroll
    for (int u = 0; u < NP / 2; ++u) lc.Kf[u] = mk<SIDE>(kk[u], kk[u + NP / 2]);
  }
  {
    // steps in which this warp's window intersects the reachable band (the same for every lane:
    // broadcast from lane 0 so that the compiler can see the chunk-skip branch is warp-uniform)
    const int win_lo_pos = base_w, win_hi_pos = min(base_w + WIN - 1, P - 1);
    const int ws_lo = SIDE ? (P - 1 - win_hi_pos) : win_lo_pos;
    const int ws_hi = SIDE ? (P - 1 - win_lo_pos) : win_hi_pos;
    int t0, t1;
    band_frames(ws_lo, ws_hi, S, T, t0, t1);
    int a_lo = SIDE ? T - 1 - t1 : t0, a_hi = SIDE ? T - 1 - t0 : t1;
    if (t0 > t1) { a_lo = 1 << 30; a_hi = -1; }
    ss.act_lo = __shfl_sync(0xffffffffu, a_lo, 0);
    ss.act_hi = __shfl_sync(0xffffffffu, a_hi, 0);
    // which phase-1 records of this lane's group the OTHER side wrote: its warp that owns the mirrored
    // group was active in the chunk (K steps aligned at its step 0) that holds the frame
    const int G = JG - 1 - lc.group;                          // the writer's group index
    const int wo = G < 32 ? 0 : (G - HL) / OWNG;              // its owner warp (the first HL lanes of warps > 0 are halo)
    const int o_lo_pos = wo * OWN, o_hi_pos = min(wo * OWN + WIN - 1, P - 1);
    const int os_lo = SIDE ? o_lo_pos : (P - 1 - o_hi_pos);   // the writer is the opposite side
    const int os_hi = SIDE ? o_hi_pos : (P - 1 - o_lo_pos);
    band_frames(os_lo, os_hi, S, T, t0, t1);
    const int M_other = SIDE ? (T - T / 2) : (T / 2);         // frames the other side covers in phase 1
    int na = SIDE ? t0 : T - 1 - t1;                          // in the writer's steps
    int nb = min(SIDE ? t1 : T - 1 - t0, M_other - 1);
    ss.rd_hi = 0; ss.wr_len = 0;
    if (t0 <= t1 && na <= nb && lc.group < JG) {
      na = na / kChunk * kChunk;
      nb = nb / kChunk * kChunk + kChunk - 1;
      ss.rd_hi = T - 1 - na;                                  // writer step n' = T-1-n for a reader at step n
      ss.wr_len = nb - na + 1;
    }
  }
  // ---- initial state: delta on the first lattice state of this side's sweep ----
  {
    float v[kLaneStates];
#pragma unroll
    for (int i = 0; i < kLaneStates; ++i) v[i] = 0.f;
    ss.st.e = kEZero;
    const int q_start = SIDE ? (P - S) : 0;   // backward: NS*JG - S dummy positions come first
    if (w == 0 && q_start >= pos0 && q_start < pos0 + kLaneStates) {
#pragma unroll
      for (int i = 0; i < kLaneStates; ++i) if (q_start - pos0 == i) v[i] = 1.f;
      ss.st.e = 0;
    }
#pragma unroll
    for (int j = 0; j < NP; ++j) ss.st.A[j] = mk<SIDE>(v[j], v[j + NP]);
  }
  ss.maxbound = -(1 << 30); ss.inv_mP = 0.f; ss.eP = 0;
  {
    const int gm = JG - 1 - min(lc.group, JG - 1);             // the reader's (mirrored) group index
    ss.weoff = NH * JG * 16 - 12 * gm;
    ss.wstep = lc.owned ? (SIDE ? -c.FB : c.FB) : 0;
    ss.wblk = c.scr + (size_t)(lc.owned ? c.frame_of(0) : T) * c.FB + (size_t)gm * 16;   // block T: the dump block
  }
  B200CTC_TRACE_DECL(tc);
  B200CTC_TRACE_EVENT(tc, 10);

  const SidePlan pl = side_plan(T, SIDE);
  const int M_side = pl.M_side, nc2 = pl.nc2;
  int* abort_flag = cm.abort_flag;

  // the all-zero frame block (stands in for records the other side never wrote)
  for (int i = c.tid_side; i < c.FB / 4; i += NW * 32) reinterpret_cast<int*>(c.sm.oth + (size_t)c.D * kChunk * c.FB)[i] = (i >= NH * JG * 4) ? kEZero : 0;
  // zero slots of the row buffers (the helper warps stage the rows themselves)
  for (int i = c.tid_side; i < RCH * kChunk; i += NW * 32) {
    float* z = c.sm.rows + (size_t)i * c.RWS + c.RW;
    z[0] = 0.f; z[1] = 0.f; z[2] = 0.f; z[3] = 0.f;
  }
  // Step ranges: phase 1 = [0, M_side), phase 2 = [M_side, T); chunks of K steps from the start of each.
  // `rs` is the row-ring slot of the current chunk.  Everything a chunk needs (emission rows, the other
  // side's records) was fetched by the helper warps during the previous chunk.
  int rs = 0;
  B200CTC_TRACE_EVENT(tc, 1);
  constexpr int HW = helper_warps<CL>();                        // barriers: lattice warps + the side's helper warps
  named_bar_sync(bar_chunk(SIDE), (NW + HW) * 32);              // rows of chunk 0 staged, wr_tab visible

  // ================================ phase 1 ================================
  // KX/K chunks between two halo exchanges (one barrier with the helpers per exchange)
  // ... as ONE frame loop: the rows of the KX/K chunks are consecutive in the ring (an exchange interval
  // starts at a multiple of KX/K chunk slots), and the band test applies to the whole interval (a warp that
  // runs frames outside its band only writes records the reader never looks at, record_window).
  int cc = 0, xc = 0;
  for (int n0 = 0; n0 < M_side; ++xc) {
    const int kc = min(kExchangeFrames, M_side - n0), nch = (kc + kChunk - 1) / kChunk;
    B200CTC_TRACE_EVENT(tc, 2);
    run_chunk<false, SIDE>(c, ss, rs, 0, 0, n0, kc, false);
    B200CTC_TRACE_EVENT(tc, 3);
    rs = (rs + nch) & (RCH - 1);
    n0 += kc;
    cc += nch;
    chunk_boundary<NWMAX, SIDE, HW>(c, ss, xc, abort_flag, tc);
  }

  // ================================ midpoint ================================
  // Lattice and helper warps of both sides meet here exactly once: everything phase 1 stored is
  // visible afterwards.
  B200CTC_TRACE_EVENT(tc, 4);
  if (CL) cluster_sync_all(); else midpoint_sync(2 * (NW + HW) * 32);
  if (nc2 == 0) return;
  named_bar_sync(bar_chunk(SIDE), (NW + HW) * 32);              // the helpers fetched the records of the first phase-2 chunk

  // ---- total probability P = sum_s alpha_t(s) beta'_t(s) at the first phase-2 frame (state copy) ----
  {
    const int n0 = M_side;
    LaneState tmp = ss.st;
    float part = 0.f; int pe = kEZero;
    if (n0 <= ss.act_hi && n0 + min(kChunk, T - M_side) - 1 >= ss.act_lo) {   // same rule as run_chunk: the warp runs this chunk
      f2 ACC[NP]; int E;
      lattice_frame<SIDE>(tmp, lc, c.sm.rows + (size_t)rs * kChunk * c.RWS, lane == 0, ACC, E);
      if (lc.owned) {
        // no band masks: outside the band one of the two factors is exactly zero (posterior_frame)
        const bool wr = (unsigned)(ss.rd_hi - n0) < (unsigned)ss.wr_len;
        const unsigned char* blk = c.sm.oth + (wr ? (size_t)0 : (size_t)c.D * kChunk * c.FB);
        float sum = 0.f;
#pragma unroll
        for (int h = 0; h < NH; ++h) {
          const float4 q = *reinterpret_cast<const float4*>(blk + lc.recB + h * JG * 16);
          const f2 p0 = f2_mul(tmp.A[2 * h], f2_pack(q.x, q.y)), p1 = f2_mul(tmp.A[2 * h + 1], f2_pack(q.z, q.w));
          sum += (f2_lo(p0) + f2_hi(p0)) + (f2_lo(p1) + f2_hi(p1));
        }
        if (sum > 0.f) { part = sum; pe = tmp.e + *reinterpret_cast<const int*>(blk + lc.expB); }
      }
    }
    int emax = pe;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) emax = max(emax, __shfl_xor_sync(0xffffffffu, emax, o));
    float scaled = part * pow2_neg(pe - emax);
    scaled = warp_sum(scaled);
    if (lane == 0) { c.sm.red_m[w] = scaled; c.sm.red_e[w] = emax; }
    named_bar_sync(bar_total(SIDE), (NW + HW) * 32);          // lattice warps + the side's helpers
    double log2P;
    if (!total_probability(c.sm, NW, ss.inv_mP, ss.eP, log2P)) {
      // zero / underflowed / garbage total probability: the safe lattice decides
      if (c.tid_side == 0) *abort_flag = 1;
      return;                                            // every thread of the side computed the same value
    }
    if (SIDE == 1 && c.tid_side == 0) p.costs[b] = (float)(-log2P * 0.69314718055994530942);
  }
  // cost-only calls still walk phase 2 (for the range check) but neither store posteriors nor update rows
  const bool write_post = p.grads != nullptr;

  // ================================ phase 2 ================================
  int k2 = 0, ob = 0;                                  // ob: ring slot of the chunk's records, k2 mod D
  for (int n0 = M_side; n0 < T; n0 += kChunk, ++k2, ++cc) {
    const int kc = min(kChunk, T - n0), par = k2 & 1;
    B200CTC_TRACE_EVENT(tc, 13);
    run_chunk<true, SIDE>(c, ss, rs, par, ob, n0, kc, write_post);
    ob = ob + 1 == c.D ? 0 : ob + 1;
    B200CTC_TRACE_EVENT(tc, 14);
    // the barrier with the helpers is per chunk; the halo is good for KX frames after an exchange
    const bool exchange = (k2 + 1) % (kExchangeFrames / kChunk) == 0;
    chunk_boundary<NWMAX, SIDE, HW>(c, ss, xc, abort_flag, tc, exchange);
    rs = (rs + 1) & (RCH - 1);
    xc += exchange ? 1 : 0;
  }
  B200CTC_TRACE_EVENT(tc, 15);
}

// ---------------------------------------------------------------------------------------------
// helper warps of one side: prefetch for the lattice warps; per-symbol occupancy of every phase-2 frame, gradient rows
// ---------------------------------------------------------------------------------------------
// Sum of one symbol's group of the posterior row: n4 16-byte chunks starting at row4.  Every lane of the
// warp runs max_n4 (warp-uniform) iterations; chunks past the lane's own group read as zero.  Fixed order.
__device__ __forceinline__ float4 lds128(unsigned a) {   // 16 bytes at a shared-window address
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
// [a, end): the lane's group as shared-window addresses; `zero`: sixteen zero bytes (what chunks past the group read)
__device__ __forceinline__ float post_group_sum(unsigned a, unsigned end, unsigned zero, int max_n4) {
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 2
  for (int r = 0; r < max_n4; ++r, a += 16) {
    const float4 v = lds128(a < end ? a : zero);
    a0 += v.x; a1 += v.y; a2 += v.z; a3 += v.w;
  }
  return (a0 + a1) + (a2 + a3);
}

// Sum over the warp of values in [0, 1] whose total is an occupancy (<= 1): one REDUX on Q30 fixed point
// instead of five dependent shuffle+add steps (error <= 32 * 2^-31, deterministic).
__device__ __forceinline__ float warp_sum_q30(float v) {
  const int q = __float2int_rn(v * 1073741824.f);
  return (float)__reduce_add_sync(0xffffffffu, q) * (1.f / 1073741824.f);
}

// Per-symbol occupancy of one phase-2 frame (posterior row `post`, softmax row `yrow`) and the update
// of its gradient row.
struct ReducerLane {
  int sym[2], base4[2], n4[2], cnt[2];   // reducer groups lane and lane + 32 (FastCommon::vg_*)
  int nvg, mp;                           // number of groups; most pieces of one symbol
};
// SPLIT: some symbol's slots are cut into pieces (ReducerLane::mp > 1).  A separate instantiation: the combination's
// shuffles between the group sums and the stores cost the common, unsplit case 5 % of the step (B200, C1 / C2) by
// merely being there.
template <int NWMAX, bool SPLIT>
__device__ __forceinline__ void reduce_frame(const CallParams& p, const FastCommon& cm, const float* __restrict__ post,
                                             const float* __restrict__ yrow, float* __restrict__ grow, unsigned zero,
                                             int RC, int NW, int n_seg, int max_n4, const ReducerLane& rl, int lane) {
  const unsigned post_a = smem_u32(post);
  const bool gathered = p.gathered != 0;
  // blank: partial sums of the lattice threads
  float accb = 0.f;
#pragma unroll
  for (int i = 0; i < NWMAX; ++i)
    if (i < NW) accb += post[RC + i * 32 + lane];
  const float sy = p.s_y, so = p.s_occ, cl = p.c_ls;   // (1, 1, 0) unless the call carries b200ctc_options
  if (n_seg <= 64 && !gathered) {
    // small vocabularies, straight line: lane u owns reducer groups u and u + 32 (in registers)
    // (the unsplit instantiation tests lane < n_seg where the split one tests its per-lane piece counts: kept apart
    // on purpose -- the common case's code is the one that was tuned, and it moves by 1-2 % when it is touched)
    const bool own0 = SPLIT ? rl.cnt[0] > 0 : lane < n_seg, own1 = SPLIT ? rl.cnt[1] > 0 : lane + 32 < n_seg;
    float tot0 = post_group_sum(post_a + 16u * rl.base4[0], post_a + 16u * (rl.base4[0] + rl.n4[0]), zero, max_n4);
    const float y0 = own0 ? yrow[rl.sym[0]] : 0.f;
    const float yb = yrow[p.blank];
    float tot1 = 0.f, y1 = 0.f;
    if ((SPLIT ? rl.nvg : n_seg) > 32) {
      tot1 = post_group_sum(post_a + 16u * rl.base4[1], post_a + 16u * (rl.base4[1] + rl.n4[1]), zero, max_n4);
      y1 = own1 ? yrow[rl.sym[1]] : 0.f;
    }
    if (SPLIT) {
      // a symbol cut into pieces: its first piece (group v) collects the pieces v + 1 .. v + cnt - 1 in that order
      const float p0 = tot0, p1 = tot1;
      for (int j = 1; j < rl.mp; ++j) {
        const int src = (lane + j) & 31;
        const float a = __shfl_sync(0xffffffffu, p0, src), b = __shfl_sync(0xffffffffu, p1, src);
        const bool wrap = lane + j >= 32;                       // group lane + j lives in the second slot of lane `src`
        if (j < rl.cnt[0]) tot0 += wrap ? b : a;
        if (j < rl.cnt[1] && !wrap) tot1 += b;                  // group lane + 32 + j (< 64: the pieces of one symbol are consecutive)
      }
    }
    accb = warp_sum_q30(accb);
    if (own0) grow[rl.sym[0]] = fmaf(-so, tot0, fmaf(sy, y0, -cl));   // the touched symbols of a frame share one or two 128-byte rows
    if (own1) grow[rl.sym[1]] = fmaf(-so, tot1, fmaf(sy, y1, -cl));
    if (lane == 0) grow[p.blank] = fmaf(-so, accb, fmaf(sy, yb, -cl));
  } else {
    for (int u0 = 0; u0 < n_seg; u0 += 32) {
      const int u = u0 + lane;
      const int s0 = u < n_seg ? cm.seg_slot[u] : 0, s1 = u < n_seg ? cm.seg_slot[u + 1] : 0;
      const float tot = post_group_sum(post_a + 4u * s0, post_a + 4u * s1, zero, max_n4);
      if (u < n_seg) {
        const int sy_ = cm.ix.seg_sym[u];
        if (!gathered) grow[sy_] = fmaf(-so, tot, fmaf(sy, yrow[sy_], -cl));
        else grow[1 + u] = tot;                         // gathered: `grow` is the frame's emission row, now its occupancy row
      }
    }
    accb = warp_sum_q30(accb);
    if (lane == 0) {
      if (!gathered) grow[p.blank] = fmaf(-so, accb, fmaf(sy, yrow[p.blank], -cl));
      else grow[0] = accb;
    }
  }
  if (p.rescale && !gathered) {          // entries the utterance never touches: s_y * y - c_ls
    const int n_un = *cm.n_untouched;
    for (int j = lane; j < n_un; j += 32) {
      const int k = cm.untouched[j];
      grow[k] = fmaf(sy, yrow[k], -cl);
    }
  }
}

// Helper warp hj of the side owns frame hj of every chunk: during chunk c it fetches what that frame
// of chunk c+1 needs (emission row; in phase 2 the other side's records of all position groups) and,
// in phase 2, reduces the posteriors the lattice warps produced for its frame of chunk c-1 into the
// gradient row.  It meets the lattice warps at the one barrier per chunk.
template <int NWMAX, int SIDE, bool CL, bool SPLIT, int ROLE>
__device__ void fast_side_helper(const CallParams& p, int b, const UttMeta& m, const FastCommon& cm,
                                 unsigned char* side_smem, int hj, int lane) {
  static_assert(kReducers == kChunk, "one helper warp per frame of a chunk");
  constexpr bool FETCH = ROLE != kReduceOnly, REDUCE = ROLE != kFetchOnly;
  FastCtx<SIDE> c;
  fill_ctx<NWMAX, SIDE>(c, p, b, m, side_smem, NWMAX + hj, lane);
  const int T = c.T, NW = c.NW, V = p.V;
  const SidePlan pl = side_plan(T, SIDE);
  const int M_side = pl.M_side;
  const int nbar = (NW + helper_warps<CL>()) * 32;
  B200CTC_TRACE_DECL(tc);

  unsigned long long* mbar = c.sm.mbar + hj * kOthDepthMax;   // one per ring slot: slot s completes phase (q / D) & 1 for chunk q
  const int D = c.D;
  if (FETCH && lane == 0) {
    for (int s = 0; s < kOthDepthMax; ++s) mbar_init(mbar + s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();

  // Emission rows are staged two barrier intervals ahead (ring slot = chunk & (RCH - 1)), so that the
  // global-memory latency of a row never sits between the lattice warps and a barrier.
  constexpr int M = kExchangeFrames / kChunk, RCH = kRowsRing * M;
  const int nc1 = pl.nc1, n_chunks = pl.n_chunks;
  auto chunk_start = [&](int cc) { return cc < nc1 ? cc * kChunk : M_side + (cc - nc1) * kChunk; };
  int staged = 0;                                    // chunks [0, staged) have been requested
  auto stage_upto = [&](int end) {                   // one cp.async group: this warp's row of chunks [staged, end)
    if (FETCH) {
      for (; staged < min(end, n_chunks); ++staged) {
        const int n = chunk_start(staged) + hj;
        if (n < T) stage_row<SIDE>(c, (staged & (RCH - 1)) * kChunk + hj, n);   // a row past a short chunk is harmless
      }
      cp_async_commit();
    }
  };
  stage_upto(M);
  stage_upto(2 * M);
  if (FETCH) cp_async_wait<1>();
  named_bar_sync(bar_chunk(SIDE), nbar);

  // ================================ phase 1 ================================
  // one barrier per halo exchange of the lattice warps (M chunks); rows are staged two exchanges ahead
  int cc = 0;
  for (int xc = 0; cc < nc1; ++xc, cc = min(cc + M, nc1)) {
    stage_upto((xc + 3) * M);
    if (FETCH) cp_async_wait<1>();            // rows up to chunk (xc+2)*M - 1 have landed
    named_bar_sync(bar_chunk(SIDE), nbar);
  }

  // ================================ midpoint ================================
  if (CL) cluster_sync_all(); else midpoint_sync(2 * nbar);
  if (pl.nc2 == 0) return;
  // The records frame hj of phase-2 chunk q needs travel into ring slot q mod D, D - 1 chunks ahead of the lattice
  // warps (the slot is free: they finished chunk q - D before the barrier that precedes the copy).  The first D - 1
  // chunks go into slots 0 .. D - 2 here; the loop below keeps its slot and phase counters incrementally.
  const int nc2 = pl.nc2;
  for (int q = 0; FETCH && q < D - 1; ++q) {
    const int n = M_side + q * kChunk + hj;
    if (q < nc2 && n < T) prefetch_other<SIDE>(c, q * kChunk + hj, n, mbar + q);
  }
  auto landed = [&](int n, int slot, unsigned phase) {       // the copy for step n (if there was one) has arrived
    if (FETCH && n < T)
      if (!mbar_wait(mbar + slot, phase) && lane == 0) *cm.abort_flag = 1;   // never observed; the safe lattice would redo the utterance
  };
  landed(M_side + hj, 0, 0u);
  named_bar_sync(bar_chunk(SIDE), nbar);
  named_bar_sync(bar_total(SIDE), nbar);
  {
    float inv_mP; int eP; double log2P;
    if (!total_probability(c.sm, NW, inv_mP, eP, log2P)) return;
  }
  const bool reduce = REDUCE && p.grads != nullptr;

  const int n_seg = *cm.ix.n_seg, max_n4 = cm.max_n4[0];
  ReducerLane rl;                                     // this lane's reducer groups (lane, lane + 32)
  rl.nvg = SPLIT ? cm.max_n4[1] : n_seg; rl.mp = SPLIT ? cm.max_n4[2] : 1;
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int u = lane + 32 * i;
    if (SPLIT) {                                      // pieces of symbol groups (the prologue's tables)
      const bool ok = u < rl.nvg;
      rl.sym[i] = ok ? cm.vg_sym[u] : 0;
      rl.base4[i] = ok ? cm.vg_base4[u] : 0;
      rl.n4[i] = ok ? cm.vg_n4[u] : 0;
      rl.cnt[i] = ok ? cm.vg_cnt[u] : 0;
    } else {                                          // one group per symbol
      rl.sym[i] = u < n_seg ? cm.ix.seg_sym[u] : 0;
      rl.base4[i] = u < n_seg ? cm.seg_slot[u] >> 2 : 0;
      rl.n4[i] = u < n_seg ? (cm.seg_slot[u + 1] - cm.seg_slot[u]) >> 2 : 0;
      rl.cnt[i] = 0;
    }
  }

  // ================================ phase 2 ================================
  // Running addresses, advanced once per chunk: the loop holds no multiplication by a frame index.  (The helper
  // warps execute ~7 cycles per instruction next to the lattice warps; every instruction here delays the barrier.)
  // By now every chunk phase 1's look-ahead requested is a phase-2 chunk or the last chunk of phase 1.
  const int sgn = SIDE ? -1 : 1;
  // (a) emission rows: chunk `staged` is the next one to request (at most one per iteration)
  const int st_adv = sgn * kChunk * c.st_stride;
  const char* st_src = c.st_src + (long long)c.frame_of(chunk_start(staged) + hj) * c.st_stride;
  int st_n = chunk_start(staged) + hj;
  // (b) the opposite side's records: chunk k2 + D - 1 goes into ring slot (k2 - 1) mod D; chunk k2 + 1 is awaited
  const int rec_adv = sgn * kChunk * c.FB;
  int rec_n = M_side + (D - 1) * kChunk + hj;
  int f_slot = D - 1;                                          // slot of chunk k2 + D - 1
  int l_slot = 1 % D, l_n = M_side + kChunk + hj;              // slot, step and mbarrier phase of chunk k2 + 1
  unsigned l_phase = D == 1 ? 1u : 0u;
  const unsigned char* rec_src = c.scr + (long long)c.frame_of(rec_n) * c.FB;
  // (c) the row reduce_frame updates: the gradient row of the frame, or (gathered mode) the frame's emission row in
  // the workspace, which nobody reads any more once its posteriors exist and which becomes its occupancy row
  const long long out_stride = p.gathered ? (long long)m.W : (long long)p.B * V;
  float* out = (p.gathered ? p.em + m.em_off : p.grads + (long long)b * V) + (long long)c.frame_of(M_side + hj) * out_stride;
  const long long out_adv = sgn * kChunk * out_stride;
  const unsigned zero16 = smem_u32(c.sm.rows + c.RW);          // the zero slot of emission row 0
  const float* post_hj = c.sm.post + (size_t)hj * c.PS;
  const int post_half = kChunk * c.PS;                          // floats per posterior buffer
  const float* rows_hj = c.sm.rows + (size_t)hj * c.RWS;
  const int row_chunk = kChunk * c.RWS;                         // floats per chunk slot of the row ring
  const unsigned st_dst_hj = c.st_dst + (unsigned)(hj * c.RWS * 4);

  int k2 = 0;
  for (; k2 < nc2; ++k2, ++cc) {
    B200CTC_TRACE_EVENT(tc, 7);
    if (FETCH && staged < cc + 3 && staged < n_chunks) {   // chunk cc+2 (nothing to do while phase 1's look-ahead lasts)
      if (st_n < T) stage_row_at<SIDE>(c, st_dst_hj + (unsigned)((staged & (RCH - 1)) * row_chunk * 4), st_src);   // a row past a short chunk is harmless
      ++staged; st_n += kChunk; st_src += st_adv;
    }
    if (FETCH) cp_async_commit();
    if (FETCH && rec_n < T && lane == 0) {
      unsigned long long* mb = mbar + f_slot;
      mbar_expect_tx(mb, (unsigned)c.FB);
      bulk_g2s(c.sm.oth + (size_t)(f_slot * kChunk + hj) * c.FB, rec_src, (unsigned)c.FB, mb);
    }
    rec_n += kChunk; rec_src += rec_adv;
    f_slot = f_slot + 1 == D ? 0 : f_slot + 1;
    B200CTC_TRACE_EVENT(tc, 8);
    if (reduce && k2 >= 1) {                          // frame hj of the previous chunk (it was a full chunk)
      const float* post_row = post_hj + ((k2 - 1) & 1) * post_half;
      const float* y_row = rows_hj + ((cc - 1) & (RCH - 1)) * row_chunk;
      reduce_frame<NWMAX, SPLIT>(p, cm, post_row, y_row, out, zero16, c.RC, NW, n_seg, max_n4, rl, lane);
      out += out_adv;
    }
    B200CTC_TRACE_EVENT(tc, 9);
    if (FETCH) cp_async_wait<1>();
    landed(l_n, l_slot, l_phase);
    l_n += kChunk;
    if (++l_slot == D) { l_slot = 0; l_phase ^= 1u; }
    named_bar_sync(bar_chunk(SIDE), nbar);
  }
  // the last chunk
  if (reduce && M_side + (k2 - 1) * kChunk + hj < T) {
    const float* post_row = post_hj + ((k2 - 1) & 1) * post_half;
    const float* y_row = rows_hj + ((cc - 1) & (RCH - 1)) * row_chunk;
    reduce_frame<NWMAX, SPLIT>(p, cm, post_row, y_row, out, zero16, c.RC, NW, n_seg, max_n4, rl, lane);
  }
  cp_async_wait<0>();
}

// The whole fast path for one utterance; every thread of the CTA calls it.  On return the shared
// word (*smem_abort)[0] is non-zero when the utterance must be redone by the safe lattice (the
// caller reads it after a __syncthreads()).
// CL (cluster variant): the CTA holds ONE side -- the one its rank in the two-CTA cluster names -- with NWMAX
// lattice warps and kReducers helper warps; both CTAs run the (cheap) prologue.
template <int NWMAX, bool CL = false>
__device__ void lattice_fast_utterance(const CallParams& p, int b, unsigned char* smem, int** smem_abort) {
  const UttMeta m = p.meta[b];
  const int L = m.L;
  // The warp index and the number of lattice windows are warp-uniform by construction; a broadcast from lane 0
  // makes that visible to the compiler, so that the role dispatch below is no potentially divergent branch and
  // the shuffles of the frame loops need no convergence check (BRA.DIV) in front of them: measured on B200, C3
  // (four windows) 0.1967 -> 0.1930 ms per step, C2 (two windows) 0.2674 -> 0.2652, but C1 (one window, where
  // ptxas then allocates 91 registers instead of 105) 0.138 -> 0.156 -- hence only for NWMAX > 1.
  const int NW = NWMAX > 1 ? __shfl_sync(0xffffffffu, fast_warps_needed(L), 0) : fast_warps_needed(L);
  const int warp = NWMAX > 1 ? __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0) : (int)(threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const int side = CL ? (int)cluster_ctarank() : warp / (NWMAX + kReducers);
  int w = CL ? cluster_warp_role<NWMAX>(warp) : warp - side * (NWMAX + kReducers);
  // Scheduler balance: warp i issues on SM sub-partition i % 4.  Early in phase 1 (and late in phase 2)
  // only the lowest lattice windows of each side are inside the reachable band; giving the backward
  // side its windows in reverse warp order puts the two busy windows on different sub-partitions.
  if (!CL && side == 1 && w < NWMAX) w = NWMAX - 1 - w;

  // ---- shared memory: common part, then one block per side ----
  FastCommon cm;
  int* ip = reinterpret_cast<int*>(smem);
  cm.abort_flag = ip;            ip += 8;
  cm.ix.n_seg = ip;              ip += 4;
  cm.max_n4 = ip;                ip += 4;
  cm.lab = ip;                   ip += L;
  cm.ix.sorted = ip;             ip += L;
  cm.ix.seg_start = ip;          ip += L + 1;
  cm.ix.seg_sym = ip;            ip += L + 1;
  cm.slot_of_label = ip;         ip += L;
  cm.seg_slot = ip;              ip += L + 2;
  cm.vg_base4 = ip;              ip += kReducerGroups;
  cm.vg_n4 = ip;                 ip += kReducerGroups;
  cm.vg_sym = ip;                ip += kReducerGroups;
  cm.vg_cnt = ip;                ip += kReducerGroups;
  cm.n_untouched = cm.abort_flag + 4;
  cm.untouched = ip;             ip += (p.V <= kUntouchedMaxV ? p.V : 0);
  size_t common = (size_t)(reinterpret_cast<unsigned char*>(ip) - smem);
  common = (common + 15) / 16 * 16;
  const int RW = p.gathered ? m.W : (p.V + 3) / 4 * 4;
  const size_t side_bytes = fast_side_bytes<NWMAX>(L, RW, p.V, p.oth_depth);
  *smem_abort = cm.abort_flag;

  // ---- prologue (all threads of the CTA) ----
#ifdef B200CTC_TRACE
  if (blockIdx.x == g_trace_cta && threadIdx.x == 0) g_trace[63 * kTraceCap] = ((long long)clock64() << 8) | 20;
#endif
  for (int i = threadIdx.x; i < L; i += blockDim.x) cm.lab[i] = p.labels[m.lab_off + i];
  if (threadIdx.x < 8) cm.abort_flag[threadIdx.x] = 0;
  // posterior buffers start all-zero: padding slots and the blank partials of idle threads are never written
  {
    const int PS = post_stride<NWMAX>(L, p.V);
    for (int sd = 0; sd < (CL ? 1 : 2); ++sd) {
      FastSideSmem s = carve_fast_side<NWMAX>(smem + common + sd * side_bytes, L, RW, p.V, p.oth_depth);
      for (int i = threadIdx.x; i < 2 * kChunk * PS; i += blockDim.x) s.post[i] = 0.f;
    }
  }
  __syncthreads();
  build_symbol_index(cm.lab, L, p.V, cm.ix);
  // slots of the symbol-sorted posterior layout: the group of segment u starts at seg_slot[u] (padded to 4)
  {
    const int n_seg = *cm.ix.n_seg;
    if (warp == 0) {
      int base = 0, mx = 0;
      for (int u0 = 0; u0 < n_seg; u0 += 32) {
        const int u = u0 + lane;
        const int cnt = (u < n_seg) ? cm.ix.seg_start[u + 1] - cm.ix.seg_start[u] : 0;
        const int pad = (cnt + 3) & ~3;
        mx = max(mx, cnt);
        int incl = pad;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int v = __shfl_up_sync(0xffffffffu, incl, o);
          if (lane >= o) incl += v;
        }
        if (u < n_seg) cm.seg_slot[u] = base + incl - pad;
        base += __shfl_sync(0xffffffffu, incl, 31);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      if (lane == 0) cm.seg_slot[n_seg] = base;
      __syncwarp();
      // ---- reducer groups ----
      const int mx4 = (mx + 3) >> 2, tot4 = base >> 2;
      int R = mx4, nvg = n_seg, mp = 1;
      int g4[2], first4[2];
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int u = lane + 32 * i;
        const bool ok = u < n_seg && n_seg <= kReducerGroups;
        first4[i] = ok ? cm.seg_slot[u] >> 2 : 0;
        g4[i] = ok ? (cm.seg_slot[u + 1] - cm.seg_slot[u]) >> 2 : 0;
      }
      if (n_seg <= kReducerGroups && !p.gathered) {
        // The smallest piece size whose pieces still fit the lanes (one per lane while the symbols do), taken only
        // when the model says it pays: 8 instructions per chunk and group slot; the combination costs more than
        // its instruction count (two shuffles per step on the helpers' critical path), so a split has to save a
        // quarter of the reducer's loop.  Pieces(r) falls with r: bisection; exact small-integer division by
        // multiplication (g4 * r < 2^16).  Skipped outright when even the ideal split could not pay (uniform labels).
        const int limit = n_seg <= 32 ? 32 : 64, slots0 = n_seg <= 32 ? 1 : 2;
        const int cost0 = slots0 * mx4 * 8;
        auto split_cost = [](int slots, int r, int pm) { return slots * r * 8 + (pm - 1) * 12 + 16; };
        int lo = max(1, (tot4 + limit - 1) / limit), hi = mx4 - 1;
        if (lo <= hi && mx4 <= 128 && 4 * split_cost(1, lo, 2) <= 3 * cost0) {
          auto pieces = [&](int r, int& pm) {
            const unsigned m = 65536u / (unsigned)r + 1u;
            const int p0 = (int)(((unsigned)(g4[0] + r - 1) * m) >> 16), p1 = (int)(((unsigned)(g4[1] + r - 1) * m) >> 16);
            pm = __reduce_max_sync(0xffffffffu, max(p0, p1));
            return __reduce_add_sync(0xffffffffu, p0 + p1);
          };
          while (lo < hi) {                       // pieces(hi) <= n_seg <= limit always holds at hi = mx4
            const int mid = (lo + hi) >> 1;
            int pm;
            if (pieces(mid, pm) <= limit) hi = mid; else lo = mid + 1;
          }
          int pm;
          const int nv = pieces(lo, pm);
          if (nv <= limit && 4 * split_cost(nv <= 32 ? 1 : 2, lo, pm) <= 3 * cost0) { R = lo; nvg = nv; mp = pm; }
        }
        if (mp > 1) {                             // (one group per symbol: the helpers read the symbol tables themselves)
          // the pieces of symbol u follow one another; exclusive prefix over the symbols in (lane, lane + 32) order
          const unsigned m = 65536u / (unsigned)R + 1u;
          int pc[2], pre[2], run = 0;
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            pc[i] = (int)(((unsigned)(g4[i] + R - 1) * m) >> 16);
            int incl = pc[i];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
              const int v = __shfl_up_sync(0xffffffffu, incl, o);
              if (lane >= o) incl += v;
            }
            pre[i] = run + incl - pc[i];
            run += __shfl_sync(0xffffffffu, incl, 31);
          }
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            const int u = lane + 32 * i;
            for (int j = 0; j < pc[i]; ++j) {
              const int v = pre[i] + j;
              cm.vg_base4[v] = first4[i] + j * R;
              cm.vg_n4[v] = min(R, g4[i] - j * R);
              cm.vg_sym[v] = cm.ix.seg_sym[u];
              cm.vg_cnt[v] = j == 0 ? pc[i] : 0;
            }
          }
        }
      }
      if (lane == 0) { cm.max_n4[0] = R; cm.max_n4[1] = nvg; cm.max_n4[2] = mp; }
    }
    __syncthreads();
    for (int k = threadIdx.x; k < L; k += blockDim.x) {
      int lo = 0, hi = n_seg - 1;              // the segment that holds sorted position k
      while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (cm.ix.seg_start[mid] <= k) lo = mid; else hi = mid - 1;
      }
      cm.slot_of_label[cm.ix.sorted[k]] = cm.seg_slot[lo] + (k - cm.ix.seg_start[lo]);
    }
    __syncthreads();
    if (p.gathered && p.grads != nullptr && (!CL || side == 0)) {   // apply_occupancy_kernel needs the distinct symbols in global memory
      for (int u = threadIdx.x; u < n_seg; u += blockDim.x) p.sym_tab[m.sym_off + u] = cm.ix.seg_sym[u];
      if (threadIdx.x == 0) p.nseg[b] = n_seg;
    }
    // rescaled rows (b200ctc_options): the reducers rewrite EVERY entry of a live row, so they also need the
    // vocabulary entries the utterance never touches (neither the blank nor one of its labels)
    if (p.rescale && !p.gathered && p.grads != nullptr) {
      for (int k = threadIdx.x; k < p.V; k += blockDim.x) cm.untouched[k] = 1;
      __syncthreads();
      for (int u = threadIdx.x; u < n_seg; u += blockDim.x) cm.untouched[cm.ix.seg_sym[u]] = 0;
      if (threadIdx.x == 0) cm.untouched[p.blank] = 0;
      __syncthreads();
      if (warp == 0) {                       // in-place compaction (reads of a tile precede its writes; the write index never overtakes)
        int n = 0;
        for (int k0 = 0; k0 < p.V; k0 += 32) {
          const int k = k0 + lane;
          const bool keep = k < p.V && cm.untouched[k] != 0;
          const unsigned bal = __ballot_sync(0xffffffffu, keep);
          __syncwarp();
          if (keep) cm.untouched[n + __popc(bal & ((1u << lane) - 1u))] = k;
          n += __popc(bal);
          __syncwarp();
        }
        if (lane == 0) *cm.n_untouched = n;
      }
      __syncthreads();
    }
  }
#ifdef B200CTC_TRACE
  if (blockIdx.x == g_trace_cta && threadIdx.x == 0) {
    g_trace[63 * kTraceCap + 1] = ((long long)clock64() << 8) | 21;
    g_trace_cnt[63] = 2;
  }
#endif
  // Everything above needed only the host-prepared tables.  From here on K1's output is read (softmax rows,
  // gathered emissions, the extreme-row flag): wait for K1 (programmatic dependent launch, lattice.cu).
  pdl_wait_primary();
  if (p.flags[b] & FLAG_EXTREME_ROW) {      // some probability below 2^-100: the safe lattice takes the utterance
    if (threadIdx.x == 0) *cm.abort_flag = kAbortExtremeRow;
    return;
  }
  unsigned char* side_smem = smem + common + (CL ? 0 : side) * side_bytes;
  if (w >= 0 && w < NW) {
    if (side == 0) fast_side_sweep<NWMAX, 0, CL>(p, b, m, cm, side_smem, w, lane);
    else           fast_side_sweep<NWMAX, 1, CL>(p, b, m, cm, side_smem, w, lane);
  } else if (CL && w >= NWMAX) {
    // cluster variant: helper warps NWMAX .. NWMAX + 3 fetch, NWMAX + 4 .. NWMAX + 7 reduce (frame hj of every chunk each)
    const bool split = __builtin_expect(cm.max_n4[2] > 1, 0);
    const int hw = w - NWMAX;
    if (hw < kReducers) {
      if (side == 0) fast_side_helper<NWMAX, 0, CL, false, kFetchOnly>(p, b, m, cm, side_smem, hw, lane);
      else           fast_side_helper<NWMAX, 1, CL, false, kFetchOnly>(p, b, m, cm, side_smem, hw, lane);
    } else if (!split) {
      if (side == 0) fast_side_helper<NWMAX, 0, CL, false, kReduceOnly>(p, b, m, cm, side_smem, hw - kReducers, lane);
      else           fast_side_helper<NWMAX, 1, CL, false, kReduceOnly>(p, b, m, cm, side_smem, hw - kReducers, lane);
    } else {
      if (side == 0) fast_side_helper<NWMAX, 0, CL, true, kReduceOnly>(p, b, m, cm, side_smem, hw - kReducers, lane);
      else           fast_side_helper<NWMAX, 1, CL, true, kReduceOnly>(p, b, m, cm, side_smem, hw - kReducers, lane);
    }
  } else if (w >= NWMAX) {
    // (a second instantiation of the helper rather than a branch in its loop: the combination of split symbol
    // groups costs the unsplit case 5 % of the step by merely being in the loop body; out of line -- __noinline__ --
    // it costs every case 10-15 %: a 448-byte stack frame and the call ABI's register constraints)
    const bool split = __builtin_expect(cm.max_n4[2] > 1, 0);
    if (!split) {
      if (side == 0) fast_side_helper<NWMAX, 0, CL, false, kFetchAndReduce>(p, b, m, cm, side_smem, w - NWMAX, lane);
      else           fast_side_helper<NWMAX, 1, CL, false, kFetchAndReduce>(p, b, m, cm, side_smem, w - NWMAX, lane);
    } else {
      if (side == 0) fast_side_helper<NWMAX, 0, CL, true, kFetchAndReduce>(p, b, m, cm, side_smem, w - NWMAX, lane);
      else           fast_side_helper<NWMAX, 1, CL, true, kFetchAndReduce>(p, b, m, cm, side_smem, w - NWMAX, lane);
    }
  } else if (CL) {
    cluster_sync_all();          // an idle warp: the midpoint rendezvous counts every thread of the cluster
  }
  // idle warps wait at the caller's __syncthreads()
}

}  // namespace b200ctc
