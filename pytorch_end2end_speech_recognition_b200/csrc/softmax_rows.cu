// K1: row-wise softmax over the vocabulary.
//
// One pass over acts[T,B,V]: for every frame row (t,b) with t < act_lens[b] it computes the row
// log-sum-exp, writes the softmax probabilities y into the gradient buffer (the lattice kernel
// later subtracts the posterior occupancy from exactly those entries, so that
// grad = softmax - occupancy, SURVEY Appendix A), stores lse[t,b], and -- in gathered mode, for
// large vocabularies -- also writes the label-indexed emission row
//   em[t][0] = y[blank], em[t][i] = y[label_i]
// so that the lattice kernel never touches the V-wide rows again.  Rows t >= act_lens[b] and rows
// of utterances with no valid alignment are zero-filled (the reference wrapper pre-zeros grads,
// models/pytorch_v3/ctc/ctc.py:36; here that fill is fused into this pass).
//
// Logits of element type T (float, __nv_bfloat16, __half) are widened to fp32 when they are loaded; every
// kernel computes in fp32 from there on and writes fp32 rows (for a bfloat16 / float16 call into the staging
// region that launch_narrow_grads later rounds into the caller's buffer).
//
// Bound: HBM.  Algorithmic bytes per row: sizeof(T) * V read + 4V written.
#include <cstdlib>
#include <type_traits>

#include "common.cuh"

namespace b200ctc {

namespace {

constexpr float kExtremeLogProb = -69.0f;  // y < 2^-100 (natural log -69.3): outside the fast lattice's range

// ---- small vocabulary: LPR lanes per row (8, 16 or 32), the row lives in registers ---------------
// Lane q of a row's lane group holds elements q, q+LPR, q+2*LPR, ...: every load/store instruction of
// the warp touches 32/LPR rows with LPR consecutive floats each, and the reductions are log2(LPR)
// shuffle steps.  V <= LPR*NV.
template <int LPR>
__device__ __forceinline__ float group_max(float v) {
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
template <int LPR>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// The element type changes only the load: element-to-lane assignment and reduction order are those of fp32 logits,
// so a reduced-precision row gives exactly the fp32 results of its widened values.
template <typename T, int LPR, int NV>
__global__ void __launch_bounds__(256) softmax_rows_warp_kernel(CallParams p) {
  pdl_launch_dependents();   // the lattice kernel may begin its prologue now
  constexpr int RPW = 32 / LPR;                       // rows per warp
  const int lane = threadIdx.x & 31;
  const int q = lane & (LPR - 1), sub = lane / LPR;
  // grid: x over the mini-batch (RPW rows per warp, 8 warps per CTA), (y, z) = frame: no index division
  const int t = blockIdx.y + blockIdx.z * 65535;
  if (t >= p.T) return;
  int b = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * RPW + sub;
  const bool row_ok = b < p.B;
  if (!row_ok) b = p.B - 1;                           // keep the lane in the shuffles; it stores nothing
  const long long row = (long long)t * p.B + b;
  const int m_T = p.meta[b].T, m_feasible = p.meta[b].feasible;
  float* grow = (p.yrows && row_ok) ? p.yrows + row * p.V : nullptr;
  const bool live = t < m_T && m_feasible;
  const T* arow = static_cast<const T*>(p.acts) + (long long)t * p.as_t + (long long)b * p.as_b;
  float x[NV];
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int v = q + LPR * i;
    x[i] = (live && v < p.V) ? widen(__ldg(arow + v)) * p.logit_scale : -INFINITY;
    mx = fmaxf(mx, x[i]);
  }
  mx = group_max<LPR>(mx);
  if (!live) mx = 0.f;                                // avoid inf - inf in dead rows
  float s = 0.f;
  float e[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    e[i] = __expf(x[i] - mx);                         // exp(-inf) = 0 for the padding lanes
    s += e[i];
  }
  s = group_sum<LPR>(s);
  const float inv = live ? 1.0f / s : 0.f;
  const float lse = mx + logf(s);
  // any probability of the row below 2^-100?  (outside the fast lattice's range)
  bool extreme = false;
#pragma unroll
  for (int i = 0; i < NV; ++i) extreme |= (q + LPR * i < p.V) && (x[i] - lse < kExtremeLogProb);
  const unsigned ext = __ballot_sync(0xffffffffu, extreme && live && row_ok);
  if (p.xe_rows) {                                    // label smoothing: -sum_k log y_k of the row = V * lse - sum_k z_k
    float sx = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) sx += (q + LPR * i < p.V && live) ? x[i] : 0.f;
    sx = group_sum<LPR>(sx);
    if (live && row_ok && q == 0) p.xe_rows[row] = (float)p.V * lse - sx;
  }
  if (live && row_ok && q == 0) {
    p.lse[row] = lse;
    if ((ext >> (sub * LPR)) & ((LPR == 32) ? 0xffffffffu : ((1u << LPR) - 1u))) atomicOr(p.flags + b, FLAG_EXTREME_ROW);
  }
  if (grow) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int v = q + LPR * i;
      // zero for rows t >= act_lens[b] and infeasible utterances.  Small vocabularies: the plain softmax (the
      // lattice reads it as its emissions and rewrites the row); gathered mode: the row in its final form
      // minus the occupancy, which the lattice subtracts with one RED per (frame, symbol)
      if (v < p.V) grow[v] = (p.gathered && live) ? fmaf(p.s_y, e[i] * inv, -p.c_ls) : e[i] * inv;
    }
  }
  if (p.gathered) {
    // label-indexed emissions, taken from the register-resident row by shuffle (all lanes take part)
    const UttMeta m = p.meta[b];
    float* erow = p.em + m.em_off + (long long)t * m.W;
    const int* lab = p.labels + m.lab_off;
    const bool wr = live && row_ok;
    int w_max = wr ? m.W : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) w_max = max(w_max, __shfl_xor_sync(0xffffffffu, w_max, o));
    for (int base = 0; base < w_max; base += LPR) {
      const int i = base + q;
      const int sym = (!wr || i >= m.W) ? -1 : ((i == 0) ? p.blank : ((i <= m.L) ? lab[i - 1] : -1));
      float val = 0.f;
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        // every lane asks the lane of its own row that holds element sym for its k-th value
        const float cand = __shfl_sync(0xffffffffu, e[k], (lane & ~(LPR - 1)) | (sym & (LPR - 1)));
        if (sym >= 0 && sym / LPR == k) val = cand * inv;
      }
      if (wr && i < m.W) erow[i] = val;
    }
  }
}

// ---- large vocabulary: one CTA per row, the row is staged in shared memory ----------------------
constexpr int kRowThreads = 256;

// A 128-bit group of eight bfloat16 / float16 logits, widened.
template <typename T>
__device__ __forceinline__ void widen8(const uint4& u, float (&f)[8]) {
  using T2 = std::conditional_t<std::is_same_v<T, __half>, __half2, __nv_bfloat162>;
  const T2* h = reinterpret_cast<const T2*>(&u);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float2 w = widen2(h[k]);
    f[2 * k] = w.x;
    f[2 * k + 1] = w.y;
  }
}

__device__ __forceinline__ float block_reduce_max(float v, float* red) {
  v = warp_max(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = red[0];
#pragma unroll
  for (int i = 1; i < kRowThreads / 32; ++i) r = fmaxf(r, red[i]);
  __syncthreads();
  return r;
}
__device__ __forceinline__ float block_reduce_min(float v, float* red) {
  v = warp_min(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = red[0];
#pragma unroll
  for (int i = 1; i < kRowThreads / 32; ++i) r = fminf(r, red[i]);
  __syncthreads();
  return r;
}
__device__ __forceinline__ float block_reduce_sum(float v, float* red) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = 0.f;
#pragma unroll
  for (int i = 0; i < kRowThreads / 32; ++i) r += red[i];
  __syncthreads();
  return r;
}

template <typename T>
__global__ void __launch_bounds__(kRowThreads) softmax_rows_cta_kernel(CallParams p) {
  pdl_launch_dependents();   // the lattice kernel may begin its prologue now
  extern __shared__ __align__(16) float srow[];  // V widened logits (+ 16 / sizeof(T) - 1 slack for the aligned window)
  __shared__ float red[kRowThreads / 32];
  const long long row = blockIdx.x;
  const int t = (int)(row / p.B);
  const int b = (int)(row - (long long)t * p.B);
  const UttMeta m = p.meta[b];
  const int V = p.V;
  const int tid = threadIdx.x;
  float* grow = p.yrows ? p.yrows + row * V : nullptr;

  if (t >= m.T || !m.feasible) {
    if (grow) {
      // zero fill with 128-bit stores on the aligned body
      int head = (int)(((16 - ((uintptr_t)grow & 15)) & 15) >> 2);
      if (head > V) head = V;
      for (int v = tid; v < head; v += kRowThreads) grow[v] = 0.f;
      int nvec = (V - head) >> 2;
      float4* g4 = reinterpret_cast<float4*>(grow + head);
      for (int v = tid; v < nvec; v += kRowThreads) g4[v] = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int v = head + (nvec << 2) + tid; v < V; v += kRowThreads) grow[v] = 0.f;
    }
    return;
  }

  const T* arow = static_cast<const T*>(p.acts) + (long long)t * p.as_t + (long long)b * p.as_b;
  // ---- load: scalar head up to 16-byte alignment, 128-bit body, scalar tail.  The row is placed
  // in shared memory at the same phase, in elements, as in global memory so both sides stay aligned.
  constexpr int kVec = 16 / sizeof(T);                    // elements per 128-bit load
  const int phase = (int)(((uintptr_t)arow & 15) / sizeof(T));  // elements past an aligned address
  float* s = srow + phase;                                // s[v] <-> arow[v]
  int head = (kVec - phase) & (kVec - 1);
  if (head > V) head = V;
  float mx = -INFINITY, mn = INFINITY;
  const float ls = p.logit_scale;
  for (int v = tid; v < head; v += kRowThreads) {
    float x = widen(__ldg(arow + v)) * ls;
    s[v] = x;
    mx = fmaxf(mx, x);
    mn = fminf(mn, x);
  }
  if constexpr (sizeof(T) == 4) {
    const int nvec = (V - head) >> 2;
    const float4* a4 = reinterpret_cast<const float4*>(arow + head);
    float4* s4 = reinterpret_cast<float4*>(s + head);
    for (int v = tid; v < nvec; v += kRowThreads) {
      float4 x = __ldg(a4 + v);
      x.x *= ls; x.y *= ls; x.z *= ls; x.w *= ls;
      s4[v] = x;
      mx = fmaxf(fmaxf(mx, fmaxf(x.x, x.y)), fmaxf(x.z, x.w));
      mn = fminf(fminf(mn, fminf(x.x, x.y)), fminf(x.z, x.w));
    }
    for (int v = head + (nvec << 2) + tid; v < V; v += kRowThreads) {
      float x = __ldg(arow + v) * ls;
      s[v] = x;
      mx = fmaxf(mx, x);
      mn = fminf(mn, x);
    }
  } else {
    const int nvec = (V - head) / kVec;
    const uint4* a8 = reinterpret_cast<const uint4*>(arow + head);
    float4* s4 = reinterpret_cast<float4*>(s + head);
    for (int v = tid; v < nvec; v += kRowThreads) {
      float f[8];
      widen8<T>(__ldg(a8 + v), f);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        f[k] *= ls;
        mx = fmaxf(mx, f[k]);
        mn = fminf(mn, f[k]);
      }
      s4[2 * v] = make_float4(f[0], f[1], f[2], f[3]);
      s4[2 * v + 1] = make_float4(f[4], f[5], f[6], f[7]);
    }
    for (int v = head + nvec * kVec + tid; v < V; v += kRowThreads) {
      float x = widen(__ldg(arow + v)) * ls;
      s[v] = x;
      mx = fmaxf(mx, x);
      mn = fminf(mn, x);
    }
  }
  mx = block_reduce_max(mx, red);  // barriers inside also publish the staged row
  mn = block_reduce_min(mn, red);
  float sum = 0.f, sx = 0.f;
  for (int v = tid; v < V; v += kRowThreads) {
    const float x = s[v];
    float e = __expf(x - mx);
    s[v] = e;
    sum += e;
    sx += x;
  }
  sum = block_reduce_sum(sum, red);
  if (p.xe_rows) sx = block_reduce_sum(sx, red);
  const float inv = 1.0f / sum;
  const float lse = mx + logf(sum);
  if (tid == 0) {
    p.lse[row] = lse;
    if (p.xe_rows) p.xe_rows[row] = (float)V * lse - sx;
    if (mn - lse < kExtremeLogProb) atomicOr(p.flags + b, FLAG_EXTREME_ROW);
  }
  if (grow) {
    // this kernel only runs in gathered mode (V > 256): the row is written in its final form minus the occupancy
    const float sy = p.gathered ? p.s_y * inv : inv, c = p.gathered ? p.c_ls : 0.f;
    int ghead = (int)(((16 - ((uintptr_t)grow & 15)) & 15) >> 2);
    if (ghead > V) ghead = V;
    for (int v = tid; v < ghead; v += kRowThreads) grow[v] = fmaf(s[v], sy, -c);
    int gvec = (V - ghead) >> 2;
    float4* g4 = reinterpret_cast<float4*>(grow + ghead);
    for (int v = tid; v < gvec; v += kRowThreads) {
      int o = ghead + (v << 2);
      g4[v] = make_float4(fmaf(s[o], sy, -c), fmaf(s[o + 1], sy, -c), fmaf(s[o + 2], sy, -c), fmaf(s[o + 3], sy, -c));
    }
    for (int v = ghead + (gvec << 2) + tid; v < V; v += kRowThreads) grow[v] = fmaf(s[v], sy, -c);
  }
  if (p.gathered) {
    float* erow = p.em + m.em_off + (long long)t * m.W;
    const int* lab = p.labels + m.lab_off;
    for (int i = tid; i < m.W; i += kRowThreads) {
      float val = 0.f;
      if (i == 0) val = s[p.blank] * inv;
      else if (i <= m.L) val = s[__ldg(lab + i - 1)] * inv;
      erow[i] = val;
    }
  }
}


// ---- large vocabulary, streaming: persistent warps, rows arrive through per-warp rings of TMA bulk copies ----
// The CTA-per-row kernel above spends ~3600 warp instructions per row of V = 3386 (block reductions replicated in
// eight warps, barriers, short loops) and is bound by the issue slots, not by HBM: 4.0 TB/s on B200.  Here ONE WARP
// owns a row (no block-wide reduction, no CTA barrier) and keeps the next row of its own in flight with
// cp.async.bulk (global -> shared, completion on an mbarrier) while it works on the current one; warp w of the
// grid walks rows w, w + W, w + 2W, ...  A row of V floats is not 16-byte aligned in general: the copy moves the
// enclosing aligned window and the row sits `phase` floats into its stage.  Rows whose window would leave the
// logits tensor (first / last row of an unaligned tensor) are loaded with plain loads; padding frames need no
// load at all (zero fill).  The stages hold the logits in their own element type: a bfloat16 / float16 stage is
// half the size of an fp32 one.
constexpr int kStreamMaxWarps = 8;     // warps per CTA (fewer when two rows per warp do not fit the shared memory)
constexpr size_t kStreamRingBytes = 220 * 1024;   // shared memory of a CTA's stages
constexpr float kLog2e = 1.4426950408889634f;

__device__ __forceinline__ unsigned sm_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ bool stream_mbar_wait(unsigned bar, unsigned parity) {
  for (int it = 0; it < (1 << 22); ++it) {     // bounded: a copy that never completes must not hang the GPU
    unsigned done;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n" : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if (done) return true;
  }
  return false;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <typename T>
struct StreamRow {
  int t, b;
  bool live, bulk;
  const T* arow;
  int phase;              // elements between the aligned window start and the row
  unsigned bytes;         // size of the aligned window
  int L, W, lab_off;      // of the row's utterance (gathered emissions)
  long long em_off;
};
template <typename T>
__device__ __forceinline__ StreamRow<T> stream_row(const CallParams& p, unsigned row, uintptr_t acts_lo, uintptr_t acts_hi) {
  StreamRow<T> r;
  r.t = (int)(row / (unsigned)p.B);
  r.b = (int)(row - (unsigned)r.t * (unsigned)p.B);
  const UttMeta m = p.meta[r.b];
  r.live = r.t < m.T && m.feasible;
  r.L = m.L; r.W = m.W; r.lab_off = m.lab_off; r.em_off = m.em_off;
  r.arow = static_cast<const T*>(p.acts) + (long long)r.t * p.as_t + (long long)r.b * p.as_b;
  const uintptr_t a = reinterpret_cast<uintptr_t>(r.arow);
  const uintptr_t lo = a & ~(uintptr_t)15, hi = (a + (uintptr_t)p.V * sizeof(T) + 15) & ~(uintptr_t)15;
  r.phase = (int)((a - lo) / sizeof(T));
  r.bytes = (unsigned)(hi - lo);
  r.bulk = r.live && lo >= acts_lo && hi <= acts_hi;
  return r;
}

template <typename T, bool XE>   // XE: the label-smoothing row term needs sum_k z
__global__ void __launch_bounds__(kStreamMaxWarps * 32) softmax_rows_stream_kernel(CallParams p, unsigned n_rows, int stage_elems,
                                                                                  int n_warps, uintptr_t acts_lo, uintptr_t acts_hi) {
  extern __shared__ __align__(128) float stages[];   // [n_warps][2][stage_elems] elements of type T
  __shared__ unsigned long long full_bar[kStreamMaxWarps][2];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int V = p.V;
  const float ls = p.logit_scale;
  if (wid < n_warps) {
    const unsigned bar0 = sm_u32(&full_bar[wid][0]);
    if (lane == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0) : "memory");
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0 + 8) : "memory");
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    T* ring = reinterpret_cast<T*>(stages) + (size_t)wid * 2 * stage_elems;
    const unsigned first = blockIdx.x * (unsigned)n_warps + wid, stride = gridDim.x * (unsigned)n_warps;
    auto issue = [&](unsigned row, int st) {      // lane 0: request a row of this warp into stage st
      if (row >= n_rows) return;
      const StreamRow<T> r = stream_row<T>(p, row, acts_lo, acts_hi);
      if (!r.bulk) return;
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the stage was read and written through the generic proxy
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar0 + 8 * st), "r"(r.bytes) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"(sm_u32(ring + (size_t)st * stage_elems)), "l"(reinterpret_cast<const char*>(r.arow) - (int)sizeof(T) * r.phase),
                     "r"(r.bytes), "r"(bar0 + 8 * st) : "memory");
    };
    if (lane == 0) issue(first, 0);
    unsigned parity = 0;                          // bit st: the phase of the stage's mbarrier its next bulk row completes
    int st = 0;
    for (unsigned row = first; row < n_rows; row += stride, st ^= 1) {
      if (lane == 0 && row + stride > row) issue(row + stride, st ^ 1);   // the other stage: this warp finished with it (closing __syncwarp)
      const StreamRow<T> r = stream_row<T>(p, row, acts_lo, acts_hi);
      float* grow = p.yrows ? p.yrows + (long long)row * V : nullptr;
      if (!r.live) {
        if (grow) {       // zero fill with 128-bit stores on the aligned body
          int head = (int)(((16 - ((uintptr_t)grow & 15)) & 15) >> 2);
          if (head > V) head = V;
          if (lane < head) grow[lane] = 0.f;
          const int nvec = (V - head) >> 2;
          float4* g4 = reinterpret_cast<float4*>(grow + head);
#pragma unroll 4
          for (int v = lane; v < nvec; v += 32) __stcs(g4 + v, make_float4(0.f, 0.f, 0.f, 0.f));
          const int tail = head + (nvec << 2) + lane;
          if (tail < V) grow[tail] = 0.f;
        }
        continue;
      }
      T* s = ring + (size_t)st * stage_elems + r.phase;         // s[v] <-> arow[v]
      // The labels whose emissions this lane gathers at the end of the row, requested now: the ring leaves the L1
      // almost no capacity, so every one of these loads is an L2 round trip that would otherwise end the row.
      constexpr int kLabPre = 8;
      int lab_pre[kLabPre];
      if (p.gathered) {
        const int* lab = p.labels + r.lab_off;
#pragma unroll
        for (int j = 0; j < kLabPre; ++j) {
          const int i = lane + 32 * j;
          lab_pre[j] = (i >= 1 && i <= r.L) ? __ldg(lab + i - 1) : p.blank;
        }
      }
      if (r.bulk) {
        if (!stream_mbar_wait(bar0 + 8 * st, (parity >> st) & 1u)) __trap();   // never observed; fail loudly rather than read a row that did not land
        parity ^= 1u << st;
      } else {            // a row at the edge of an unaligned tensor: plain loads
        for (int v = lane; v < V; v += 32) s[v] = __ldg(r.arow + v);
        __syncwarp();
      }
      if constexpr (sizeof(T) == 4) {
        // ---- pass 1: maximum / minimum (/ sum, label smoothing) of the raw logits ----
        int head = (4 - r.phase) & 3;
        if (head > V) head = V;
        const int nvec = (V - head) >> 2, tail0 = head + (nvec << 2);
        float4* s4 = reinterpret_cast<float4*>(s + head);
        float mx = -INFINITY, mn = INFINITY, sx = 0.f;
        if (lane < head) { const float x = s[lane]; mx = x; mn = x; sx = x; }
        {
          float mx1 = -INFINITY, mn1 = INFINITY, sx1 = 0.f;
  #pragma unroll 4
          for (int v = lane; v < nvec; v += 32) {
            const float4 x = s4[v];
            mx = fmaxf(mx, fmaxf(x.x, x.y)); mx1 = fmaxf(mx1, fmaxf(x.z, x.w));
            mn = fminf(mn, fminf(x.x, x.y)); mn1 = fminf(mn1, fminf(x.z, x.w));
            if (XE) { sx += x.x + x.y; sx1 += x.z + x.w; }
          }
          mx = fmaxf(mx, mx1); mn = fminf(mn, mn1); sx += sx1;
        }
        if (tail0 + lane < V) { const float x = s[tail0 + lane]; mx = fmaxf(mx, x); mn = fminf(mn, x); sx += x; }
        mx = warp_max(mx); mn = warp_min(mn);
        if (XE) sx = warp_sum(sx);
        // z = ls * x: the scale is positive in every use (1 / temperature), a negative one swaps the extremes
        const float zmax = ls >= 0.f ? ls * mx : ls * mn, zmin = ls >= 0.f ? ls * mn : ls * mx;
        // ---- pass 2: e = exp(z - zmax) in place, row sum ----
        const float a2 = ls * kLog2e, b2 = -zmax * kLog2e;
        float sum = 0.f, sum1 = 0.f;
        if (lane < head) { const float e = ex2_approx(fmaf(s[lane], a2, b2)); s[lane] = e; sum = e; }
  #pragma unroll 4
        for (int v = lane; v < nvec; v += 32) {
          float4 x = s4[v];
          x.x = ex2_approx(fmaf(x.x, a2, b2)); x.y = ex2_approx(fmaf(x.y, a2, b2));
          x.z = ex2_approx(fmaf(x.z, a2, b2)); x.w = ex2_approx(fmaf(x.w, a2, b2));
          s4[v] = x;
          sum += x.x + x.y; sum1 += x.z + x.w;
        }
        if (tail0 + lane < V) { const float e = ex2_approx(fmaf(s[tail0 + lane], a2, b2)); s[tail0 + lane] = e; sum += e; }
        sum = warp_sum(sum + sum1);
        const float inv = 1.0f / sum;
        const float lse = zmax + logf(sum);
        if (lane == 0) {
          p.lse[row] = lse;
          if (XE) p.xe_rows[row] = (float)V * lse - ls * sx;
          if (zmin - lse < kExtremeLogProb) atomicOr(p.flags + r.b, FLAG_EXTREME_ROW);
        }
        // ---- pass 3: the row in its final form minus the occupancy (gathered mode), label-gathered emissions ----
        if (grow) {
          const float sy = p.gathered ? p.s_y * inv : inv, c = p.gathered ? p.c_ls : 0.f;
          int ghead = (int)(((16 - ((uintptr_t)grow & 15)) & 15) >> 2);
          if (ghead > V) ghead = V;
          const int gvec = (V - ghead) >> 2;
          float4* g4 = reinterpret_cast<float4*>(grow + ghead);
          if (ghead == head) {          // source and destination rows share the 16-byte phase (contiguous logits): 128-bit both ways,
            if (lane < ghead) grow[lane] = fmaf(s[lane], sy, -c);   // and every lane re-reads exactly what it wrote in pass 2
  #pragma unroll 4
            for (int v = lane; v < gvec; v += 32) {
              const float4 e = s4[v];
              __stcs(g4 + v, make_float4(fmaf(e.x, sy, -c), fmaf(e.y, sy, -c), fmaf(e.z, sy, -c), fmaf(e.w, sy, -c)));
            }
          } else {
            __syncwarp();
            if (lane < ghead) grow[lane] = fmaf(s[lane], sy, -c);
            for (int v = lane; v < gvec; v += 32) {
              const int o = ghead + (v << 2);
              __stcs(g4 + v, make_float4(fmaf(s[o], sy, -c), fmaf(s[o + 1], sy, -c), fmaf(s[o + 2], sy, -c), fmaf(s[o + 3], sy, -c)));
            }
          }
          const int gt = ghead + (gvec << 2) + lane;
          if (gt < V) grow[gt] = fmaf(s[gt], sy, -c);
        }
        __syncwarp();       // pass 2's values are visible to every lane
        if (p.gathered) {
          float* erow = p.em + r.em_off + (long long)r.t * r.W;
          const int* lab = p.labels + r.lab_off;
  #pragma unroll
          for (int j = 0; j < kLabPre; ++j) {        // i = 0: the blank; padding entries (L < i < W): zero
            const int i = lane + 32 * j;
            if (i < r.W) erow[i] = i <= r.L ? s[lab_pre[j]] * inv : 0.f;
          }
          for (int i = lane + 32 * kLabPre; i < r.W; i += 32)
            erow[i] = i <= r.L ? s[__ldg(lab + i - 1)] * inv : 0.f;
        }
      } else {
        // bfloat16 / float16: the stage keeps the raw logits (an fp32 row would not fit a half-size stage), so pass 2
        // only sums e = exp(z - zmax) and pass 3 evaluates it again from the stage: the same function of the same value
        constexpr int kVec = 8;                  // elements per 128-bit shared-memory load
        int head = (kVec - r.phase) & (kVec - 1);
        if (head > V) head = V;
        const int nvec = (V - head) / kVec, tail0 = head + nvec * kVec;
        const uint4* s8 = reinterpret_cast<const uint4*>(s + head);
        // ---- pass 1: maximum / minimum (/ sum, label smoothing) of the widened logits ----
        float mx = -INFINITY, mn = INFINITY, sx = 0.f;
        if (lane < head) { const float x = widen(s[lane]); mx = x; mn = x; sx = x; }
#pragma unroll 2
        for (int v = lane; v < nvec; v += 32) {
          float f[8];
          widen8<T>(s8[v], f);
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            mx = fmaxf(mx, f[k]);
            mn = fminf(mn, f[k]);
            if (XE) sx += f[k];
          }
        }
        if (tail0 + lane < V) { const float x = widen(s[tail0 + lane]); mx = fmaxf(mx, x); mn = fminf(mn, x); sx += x; }
        mx = warp_max(mx); mn = warp_min(mn);
        if (XE) sx = warp_sum(sx);
        const float zmax = ls >= 0.f ? ls * mx : ls * mn, zmin = ls >= 0.f ? ls * mn : ls * mx;
        // ---- pass 2: row sum of e = exp(z - zmax) ----
        const float a2 = ls * kLog2e, b2 = -zmax * kLog2e;
        auto e_of = [&](int v) { return ex2_approx(fmaf(widen(s[v]), a2, b2)); };
        float sum = 0.f, sum1 = 0.f;
        if (lane < head) sum = e_of(lane);
#pragma unroll 2
        for (int v = lane; v < nvec; v += 32) {
          float f[8];
          widen8<T>(s8[v], f);
#pragma unroll
          for (int k = 0; k < 8; k += 2) {
            sum += ex2_approx(fmaf(f[k], a2, b2));
            sum1 += ex2_approx(fmaf(f[k + 1], a2, b2));
          }
        }
        if (tail0 + lane < V) sum += e_of(tail0 + lane);
        sum = warp_sum(sum + sum1);
        const float inv = 1.0f / sum;
        const float lse = zmax + logf(sum);
        if (lane == 0) {
          p.lse[row] = lse;
          if (XE) p.xe_rows[row] = (float)V * lse - ls * sx;
          if (zmin - lse < kExtremeLogProb) atomicOr(p.flags + r.b, FLAG_EXTREME_ROW);
        }
        // ---- pass 3: the fp32 row in its final form minus the occupancy (gathered mode), label-gathered emissions ----
        if (grow) {
          const float sy = p.gathered ? p.s_y * inv : inv, c = p.gathered ? p.c_ls : 0.f;
          int ghead = (int)(((16 - ((uintptr_t)grow & 15)) & 15) >> 2);
          if (ghead > V) ghead = V;
          const int gvec = (V - ghead) >> 2;
          float4* g4 = reinterpret_cast<float4*>(grow + ghead);
          if (lane < ghead) grow[lane] = fmaf(e_of(lane), sy, -c);
#pragma unroll 4
          for (int v = lane; v < gvec; v += 32) {
            const int o = ghead + (v << 2);
            __stcs(g4 + v, make_float4(fmaf(e_of(o), sy, -c), fmaf(e_of(o + 1), sy, -c), fmaf(e_of(o + 2), sy, -c),
                                       fmaf(e_of(o + 3), sy, -c)));
          }
          const int gt = ghead + (gvec << 2) + lane;
          if (gt < V) grow[gt] = fmaf(e_of(gt), sy, -c);
        }
        if (p.gathered) {
          float* erow = p.em + r.em_off + (long long)r.t * r.W;
          const int* lab = p.labels + r.lab_off;
#pragma unroll
          for (int j = 0; j < kLabPre; ++j) {
            const int i = lane + 32 * j;
            if (i < r.W) erow[i] = i <= r.L ? e_of(lab_pre[j]) * inv : 0.f;
          }
          for (int i = lane + 32 * kLabPre; i < r.W; i += 32)
            erow[i] = i <= r.L ? e_of(__ldg(lab + i - 1)) * inv : 0.f;
        }
      }
      __syncwarp();       // closing: every lane is done with the stage
    }
  }
  // The lattice kernel may begin its prologue now.  Not earlier: its CTAs (one per utterance, most of an SM's shared
  // memory each) would sit on their SMs waiting for this grid to finish while this grid still needs them.
  pdl_launch_dependents();
}

template <typename T>
cudaError_t launch_softmax_rows_of(const CallParams& p, cudaStream_t stream) {
  const long long n_rows = (long long)p.T * p.B;
  if (p.V <= 256) {
    const int warps = 8;
    auto grid_for = [&](int rows_per_warp) {     // frames on (y, z): T up to 65535^2
      const int per_cta = warps * rows_per_warp;
      const int ty = p.T < 65535 ? p.T : 65535;
      return dim3((unsigned)((p.B + per_cta - 1) / per_cta), (unsigned)ty, (unsigned)((p.T + 65534) / 65535));
    };
    // eight elements per lane: the per-row work (reductions, 1/s, log, flags) is shared by fewer lanes -- the kernel is
    // bound by its instruction count, not by HBM (profiles/r02_softmax_ncu_summary.txt: 75 % of the issue slots)
    static const bool nv4 = std::getenv("B200CTC_K1_NV4") != nullptr;   // the previous geometry, for A/B measurements
    if (nv4 && p.V <= 32) softmax_rows_warp_kernel<T, 8, 4><<<grid_for(4), warps * 32, 0, stream>>>(p);
    else if (nv4 && p.V <= 64) softmax_rows_warp_kernel<T, 16, 4><<<grid_for(2), warps * 32, 0, stream>>>(p);
    else if (nv4 && p.V <= 128) softmax_rows_warp_kernel<T, 32, 4><<<grid_for(1), warps * 32, 0, stream>>>(p);
    else if (p.V <= 32) softmax_rows_warp_kernel<T, 4, 8><<<grid_for(8), warps * 32, 0, stream>>>(p);
    else if (p.V <= 64) softmax_rows_warp_kernel<T, 8, 8><<<grid_for(4), warps * 32, 0, stream>>>(p);
    else if (p.V <= 128) softmax_rows_warp_kernel<T, 16, 8><<<grid_for(2), warps * 32, 0, stream>>>(p);
    else softmax_rows_warp_kernel<T, 32, 8><<<grid_for(1), warps * 32, 0, stream>>>(p);
  } else {
    // streaming kernel when at least two warps with two fp32 rows each fit the shared memory (V <= 14074), else one CTA
    // per row.  The limit is the fp32 one for every element type; the ring itself is sized for the element type.
    constexpr int kVec = 16 / sizeof(T);          // elements per 16 bytes
    const int stage_f32 = (p.V + 6 + 3) & ~3;
    const bool fits = kStreamRingBytes / ((size_t)2 * stage_f32 * sizeof(float)) >= 2;
    // a window is the row plus up to kVec - 1 elements on each side, rounded to 16 bytes
    const int stage_elems = (p.V + 3 * (kVec - 1)) & ~(kVec - 1);
    const size_t per_warp = (size_t)2 * stage_elems * sizeof(T);
    int n_warps = (int)(kStreamRingBytes / per_warp);
    if (n_warps > kStreamMaxWarps) n_warps = kStreamMaxWarps;
    if (!fits || n_rows >= (1ll << 31) || std::getenv("B200CTC_SOFTMAX_CTA_PER_ROW")) {
      const size_t smem = (size_t)(p.V + kVec) * sizeof(float);
      if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(softmax_rows_cta_kernel<T>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
      }
      softmax_rows_cta_kernel<T><<<(unsigned)n_rows, kRowThreads, smem, stream>>>(p);
    } else {
      const size_t ring = per_warp * n_warps;
      auto kern = p.xe_rows ? softmax_rows_stream_kernel<T, true> : softmax_rows_stream_kernel<T, false>;
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ring);
      if (e != cudaSuccess) return e;
      static int n_sm = 0;
      if (n_sm == 0) {
        int dev = 0;
        if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
        if ((e = cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
      }
      long long grid = n_sm;                       // one CTA per SM (the ring takes most of its shared memory)
      if (grid * n_warps > n_rows) grid = (n_rows + n_warps - 1) / n_warps;
      const uintptr_t lo = reinterpret_cast<uintptr_t>(p.acts);
      const uintptr_t hi = lo + (uintptr_t)(((long long)(p.T - 1) * p.as_t + (long long)(p.B - 1) * p.as_b + p.V) * sizeof(T));
      kern<<<(unsigned)grid, kStreamMaxWarps * 32, ring, stream>>>(p, (unsigned)n_rows, stage_elems, n_warps, lo, hi);
    }
  }
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_softmax_rows(const CallParams& p, cudaStream_t stream) {
  if ((long long)p.T * p.B == 0) return cudaSuccess;
  switch (p.acts_dtype) {
    case B200CTC_BFLOAT16: return launch_softmax_rows_of<__nv_bfloat16>(p, stream);
    case B200CTC_FLOAT16: return launch_softmax_rows_of<__half>(p, stream);
    default: return launch_softmax_rows_of<float>(p, stream);
  }
}

}  // namespace b200ctc
