// K4: batched best-path (greedy) CTC decoder.
//
// Replaces the python loops of models/pytorch_v3/ctc/decoders/greedy_decoder.py:32-45:
//   :32-37  per-frame np.argmax over the vocabulary for t < x_lens[b]   -> frame_argmax kernels
//   :40     collapse repeated labels (itertools.groupby)                 \  collapse kernel
//   :43-44  drop the blank label                                         /
// np.argmax semantics are kept bit-exactly: the first index wins ties, -0.0 == +0.0, and a NaN is
// "larger" than everything (the first NaN wins).
//
// Element types: the arg-max kernels are templates on the logits' type (float, __nv_bfloat16, __half).  Widening a
// 16-bit value to fp32 is exact and monotone, so every type gives the arg-max the fp32 kernel gives on the widened
// logits, ties and NaN included.
//
// Bound: HBM (one read of the logits, 4 bytes written per frame).
#include <cstdlib>
#include <type_traits>

#include "common.cuh"

namespace b200ctc {

namespace {

// Order-preserving key: (value key << 32) | (~index).  max() over keys = np.argmax.
__device__ __forceinline__ unsigned long long argmax_key(float x, int idx) {
  unsigned int k;
  if (x != x) {
    k = 0xffffffffu;
  } else {
    x += 0.0f;  // -0.0 -> +0.0
    unsigned int bits = __float_as_uint(x);
    k = (bits & 0x80000000u) ? ~bits : (bits | 0x80000000u);
  }
  return ((unsigned long long)k << 32) | (unsigned long long)(0xffffffffu - (unsigned int)idx);
}
__device__ __forceinline__ unsigned long long umax64(unsigned long long a, unsigned long long b) {
  return a > b ? a : b;
}
__device__ __forceinline__ unsigned long long warp_max_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = umax64(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ int key_index(unsigned long long k) {
  return (int)(0xffffffffu - (unsigned int)(k & 0xffffffffull));
}

// small vocabulary: one warp per frame
template <typename E>
__global__ void __launch_bounds__(256) frame_argmax_warp_kernel(
    const E* __restrict__ logits, long long stride_b, long long stride_t,
    const int* __restrict__ lens, int T, int V, int B, int* __restrict__ out_tokens) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= (long long)B * T) return;
  const int b = (int)(row / T), t = (int)(row - (long long)b * T);
  if (t >= min(lens[b], T)) return;
  const E* x = logits + b * stride_b + t * stride_t;
  unsigned long long best = 0ull;
  for (int v = lane; v < V; v += 32) best = umax64(best, argmax_key(widen(__ldg(x + v)), v));
  best = warp_max_u64(best);
  if (lane == 0) out_tokens[row] = key_index(best);
}

// very small vocabulary (V <= 4 * LPR, LPR = 8 or 16 lanes per frame): a warp decodes 32 / LPR frames at once, so
// that one load instruction of the warp covers several short rows instead of one 120-byte row
template <typename E, int LPR>
__global__ void __launch_bounds__(256) frame_argmax_group_kernel(
    const E* __restrict__ logits, long long stride_b, long long stride_t,
    const int* __restrict__ lens, int T, int V, int B, int* __restrict__ out_tokens) {
  constexpr int RPW = 32 / LPR;
  const int lane = threadIdx.x & 31, q = lane & (LPR - 1), sub = lane / LPR;
  long long row = ((long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * RPW + sub;
  const bool in_range = row < (long long)B * T;
  if (!in_range) row = (long long)B * T - 1;                // keep the lane in the shuffles; it stores nothing
  const int b = (int)(row / T), t = (int)(row - (long long)b * T);
  const bool live = in_range && t < min(lens[b], T);
  const E* x = logits + b * stride_b + t * stride_t;
  unsigned long long best = 0ull;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int v = q + LPR * i;
    if (live && v < V) best = umax64(best, argmax_key(widen(__ldg(x + v)), v));
  }
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) best = umax64(best, __shfl_xor_sync(0xffffffffu, best, o));
  if (live && q == 0) out_tokens[row] = key_index(best);
}

// large vocabulary: one CTA per frame, 128-bit loads on the aligned body (fp32 only: the A/B alternative of the
// streaming kernel below)
__global__ void __launch_bounds__(256) frame_argmax_cta_kernel(
    const float* __restrict__ logits, long long stride_b, long long stride_t,
    const int* __restrict__ lens, int T, int V, int B, int* __restrict__ out_tokens) {
  __shared__ unsigned long long red[8];
  const long long row = blockIdx.x;
  const int b = (int)(row / T), t = (int)(row - (long long)b * T);
  if (t >= min(lens[b], T)) return;
  const float* x = logits + b * stride_b + t * stride_t;
  const int tid = threadIdx.x;
  int head = (int)(((16 - ((uintptr_t)x & 15)) & 15) >> 2);
  if (head > V) head = V;
  unsigned long long best = 0ull;
  for (int v = tid; v < head; v += 256) best = umax64(best, argmax_key(__ldg(x + v), v));
  const int nvec = (V - head) >> 2;
  const float4* x4 = reinterpret_cast<const float4*>(x + head);
  for (int i = tid; i < nvec; i += 256) {
    const float4 q = __ldg(x4 + i);
    const int v = head + (i << 2);
    best = umax64(best, argmax_key(q.x, v));
    best = umax64(best, argmax_key(q.y, v + 1));
    best = umax64(best, argmax_key(q.z, v + 2));
    best = umax64(best, argmax_key(q.w, v + 3));
  }
  for (int v = head + (nvec << 2) + tid; v < V; v += 256) best = umax64(best, argmax_key(__ldg(x + v), v));
  best = warp_max_u64(best);
  if ((tid & 31) == 0) red[tid >> 5] = best;
  __syncthreads();
  if (tid == 0) {
    unsigned long long r = red[0];
#pragma unroll
    for (int i = 1; i < 8; ++i) r = umax64(r, red[i]);
    out_tokens[row] = key_index(r);
  }
}

// large vocabulary, streaming: persistent warps, one WARP per frame row (no block reduction, no barrier), eight
// 128-bit loads in flight per lane.  The one-CTA-per-frame kernel above reads C4's logits (V = 3386) at 3.8 TB/s:
// 64 000 short-lived CTAs with three loads per thread each.
__device__ __forceinline__ float4 ldg_stream4(const float4* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ uint4 ldg_stream_u4(const uint4* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
#ifndef B200CTC_ARGMAX_IN_FLIGHT
#define B200CTC_ARGMAX_IN_FLIGHT 8
#endif
constexpr int kInFlight = B200CTC_ARGMAX_IN_FLIGHT;

// the warp's arg-max key of one fp32 row (any lane holds it on return)
__device__ __forceinline__ unsigned long long row_argmax_key(const float* x, int V, int lane) {
  int head = (int)(((16 - ((uintptr_t)x & 15)) & 15) >> 2);
  if (head > V) head = V;
  unsigned long long best = 0ull;
  if (lane < head) best = argmax_key(__ldg(x + lane), lane);
  const int nvec = (V - head) >> 2;
  const float4* x4 = reinterpret_cast<const float4*>(x + head);
  int i = lane;
  for (; i + 32 * (kInFlight - 1) < nvec; i += 32 * kInFlight) {   // kInFlight independent loads per lane before any use
    float4 q[kInFlight];
#pragma unroll
    for (int k = 0; k < kInFlight; ++k) q[k] = ldg_stream4(x4 + i + 32 * k);
#pragma unroll
    for (int k = 0; k < kInFlight; ++k) {
      const int v = head + ((i + 32 * k) << 2);
      best = umax64(best, argmax_key(q[k].x, v));
      best = umax64(best, argmax_key(q[k].y, v + 1));
      best = umax64(best, argmax_key(q[k].z, v + 2));
      best = umax64(best, argmax_key(q[k].w, v + 3));
    }
  }
  for (; i < nvec; i += 32) {
    const float4 q = ldg_stream4(x4 + i);
    const int v = head + (i << 2);
    best = umax64(best, argmax_key(q.x, v));
    best = umax64(best, argmax_key(q.y, v + 1));
    best = umax64(best, argmax_key(q.z, v + 2));
    best = umax64(best, argmax_key(q.w, v + 3));
  }
  const int tail = head + (nvec << 2) + lane;
  if (tail < V) best = umax64(best, argmax_key(__ldg(x + tail), tail));
  return warp_max_u64(best);
}

// 16-bit logits: bit pattern of +inf, and the value of a bit pattern
template <typename E> constexpr unsigned kInf16 = 0;
template <> constexpr unsigned kInf16<__nv_bfloat16> = 0x7f80u;
template <> constexpr unsigned kInf16<__half> = 0x7c00u;
template <typename E> __device__ __forceinline__ E from_bits(unsigned short h);
template <> __device__ __forceinline__ __nv_bfloat16 from_bits(unsigned short h) { return __ushort_as_bfloat16(h); }
template <> __device__ __forceinline__ __half from_bits(unsigned short h) { return __ushort_as_half(h); }

// Value key of a 16-bit logit h in the upper half of w (the lower half of w is ignored), formed on the raw bits:
// the upper 16 bits of the result are inf + |h| for h >= 0 and inf - |h| for h < 0 (mod 2^16; inf = kInf16), so
// -0 and +0 get the same key, the order is that of the values, and every NaN, of either sign and any payload, lands
// above the key of +inf, 2 * inf.  `rot_low` is inf << 16 plus what goes into the lower 16 bits.  Four
// instructions: shift, LOP3, IADD3, and the max that consumes the key.
__device__ __forceinline__ unsigned key16(unsigned w, unsigned rot_low) {
  const unsigned m = (unsigned)((int)w >> 31);
  return ((w & 0x7fff0000u) ^ m) - m + rot_low;
}

// The warp's arg-max of one 16-bit row, as a 32-bit key (value key << 16) | (0xffff - v); V <= 65536.
// The body keeps one running maximum per position j of the eight elements of a 16-byte vector, keyed by the vector
// index, so the hot loop never forms an element index; the per-lane combination below restores it.  A row whose
// maximum is a NaN is read again with the 64-bit key, where the first NaN wins whatever its payload.
template <typename E>
__device__ __forceinline__ unsigned row_argmax_key16(const E* x, int V, int lane) {
  constexpr unsigned kRot = kInf16<E> << 16;
  const unsigned short* h = reinterpret_cast<const unsigned short*>(x);
  int head = (int)(((16 - ((uintptr_t)x & 15)) & 15) >> 1);
  if (head > V) head = V;
  const int nvec = (V - head) >> 3;
  const uint4* x4 = reinterpret_cast<const uint4*>(x + head);
  unsigned acc[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};   // 0: empty (a real key has 0xffff - i > 0 in its lower half)
  auto take = [&](const uint4& q, int i) {
    const unsigned rl = kRot + 0xffffu - (unsigned)i;
    acc[0] = max(acc[0], key16(q.x << 16, rl)); acc[1] = max(acc[1], key16(q.x, rl));
    acc[2] = max(acc[2], key16(q.y << 16, rl)); acc[3] = max(acc[3], key16(q.y, rl));
    acc[4] = max(acc[4], key16(q.z << 16, rl)); acc[5] = max(acc[5], key16(q.z, rl));
    acc[6] = max(acc[6], key16(q.w << 16, rl)); acc[7] = max(acc[7], key16(q.w, rl));
  };
  int i = lane;
  for (; i + 32 * (kInFlight - 1) < nvec; i += 32 * kInFlight) {   // kInFlight independent loads per lane before any use
    uint4 q[kInFlight];
#pragma unroll
    for (int k = 0; k < kInFlight; ++k) q[k] = ldg_stream_u4(x4 + i + 32 * k);
#pragma unroll
    for (int k = 0; k < kInFlight; ++k) take(q[k], i + 32 * k);
  }
  for (; i < nvec; i += 32) take(ldg_stream_u4(x4 + i), i);
  unsigned best = 0u;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (acc[j] == 0u) continue;
    const int v = head + 8 * (int)(0xffffu - (acc[j] & 0xffffu)) + j;
    best = max(best, (acc[j] & 0xffff0000u) | (0xffffu - (unsigned)v));
  }
  if (lane < head) best = max(best, key16((unsigned)h[lane] << 16, kRot + 0xffffu - (unsigned)lane));   // 0..7 elements
  const int tail = head + (nvec << 3) + lane;                                                                 // 0..7 elements
  if (tail < V) best = max(best, key16((unsigned)h[tail] << 16, kRot + 0xffffu - (unsigned)tail));
  return __reduce_max_sync(0xffffffffu, best);
}

// The warp's arg-max key of one 16-bit row on widened values, for any V.
template <typename E>
__device__ __forceinline__ unsigned long long row_argmax_key(const E* x, int V, int lane) {
  const unsigned short* h = reinterpret_cast<const unsigned short*>(x);
  int head = (int)(((16 - ((uintptr_t)x & 15)) & 15) >> 1);
  if (head > V) head = V;
  unsigned long long best = 0ull;
  if (lane < head) best = argmax_key(widen(from_bits<E>(h[lane])), lane);
  const int nvec = (V - head) >> 3;
  const uint4* x4 = reinterpret_cast<const uint4*>(x + head);
  auto take = [&](const uint4& q, int i) {
    const int v = head + (i << 3);
    const unsigned w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      best = umax64(best, argmax_key(widen(from_bits<E>((unsigned short)(w[j] & 0xffffu))), v + 2 * j));
      best = umax64(best, argmax_key(widen(from_bits<E>((unsigned short)(w[j] >> 16))), v + 2 * j + 1));
    }
  };
  int i = lane;
  for (; i + 32 * (kInFlight - 1) < nvec; i += 32 * kInFlight) {
    uint4 q[kInFlight];
#pragma unroll
    for (int k = 0; k < kInFlight; ++k) q[k] = ldg_stream_u4(x4 + i + 32 * k);
#pragma unroll
    for (int k = 0; k < kInFlight; ++k) take(q[k], i + 32 * k);
  }
  for (; i < nvec; i += 32) take(ldg_stream_u4(x4 + i), i);
  const int tail = head + (nvec << 3) + lane;
  if (tail < V) best = umax64(best, argmax_key(widen(from_bits<E>(h[tail])), tail));
  return warp_max_u64(best);
}

// the whole row again with the 64-bit key on widened values, scalar loads (rows with a NaN only)
template <typename E>
__device__ __noinline__ int row_argmax_scalar(const E* x, int V, int lane) {
  unsigned long long best = 0ull;
  for (int v = lane; v < V; v += 32) best = umax64(best, argmax_key(widen(x[v]), v));
  return key_index(warp_max_u64(best));
}

// kNarrowKey (16-bit E, V <= 65536): the 32-bit key on raw bits; else the 64-bit key on widened values
template <typename E, bool kNarrowKey>
__global__ void __launch_bounds__(256) frame_argmax_stream_kernel(
    const E* __restrict__ logits, long long stride_b, long long stride_t,
    const int* __restrict__ lens, int T, int V, int B, int* __restrict__ out_tokens) {
  const int lane = threadIdx.x & 31;
  const long long n_rows = (long long)B * T;
  const long long n_warps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < n_rows; row += n_warps) {
    const int b = (int)(row / T), t = (int)(row - (long long)b * T);
    if (t >= min(lens[b], T)) continue;
    const E* x = logits + b * stride_b + t * stride_t;
    int token;
    if constexpr (kNarrowKey) {
      const unsigned best = row_argmax_key16(x, V, lane);
      token = (best >> 16) > 2 * kInf16<E> ? row_argmax_scalar(x, V, lane) : (int)(0xffffu - (best & 0xffffu));
    } else {
      token = key_index(row_argmax_key(x, V, lane));
    }
    if (lane == 0) out_tokens[row] = token;
  }
}

// One CTA per utterance: keep frame t iff its symbol differs from frame t-1 and is not blank;
// compact in place with a block-wide prefix sum (writes never overtake reads: compaction only
// moves tokens to lower indices and each chunk is read in full before it is written).
constexpr int kCollapseThreads = 1024;
__global__ void __launch_bounds__(kCollapseThreads) collapse_kernel(
    const int* __restrict__ lens, int T, int blank, int* __restrict__ out_tokens,
    int* __restrict__ out_lens) {
  __shared__ int warp_tot[32];
  __shared__ int base_s;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int* row = out_tokens + (long long)b * T;
  const int n = min(max(lens[b], 0), T);   // a length outside [0, T] is clamped (the reference would raise IndexError)
  if (tid == 0) base_s = 0;
  __syncthreads();
  for (int t0 = 0; t0 < n; t0 += kCollapseThreads) {
    const int t = t0 + tid;
    const int base = base_s;  // written by the previous chunk before its closing barrier
    int sym = 0, keep = 0;
    if (t < n) {
      sym = row[t];
      const int prev = (t > 0) ? row[t - 1] : -1;  // frame t-1 is still un-compacted here (see barrier below)
      keep = (sym != blank) && (t == 0 || sym != prev);
    }
    // inclusive scan of keep
    int incl = keep;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int up = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += up;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();  // all reads of this chunk (and of row[t0-1]) are done
    if (warp == 0) {
      int w = warp_tot[lane];
      int wi = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int up = __shfl_up_sync(0xffffffffu, wi, o);
        if (lane >= o) wi += up;
      }
      warp_tot[lane] = wi - w;  // exclusive
    }
    __syncthreads();
    const int pos = base + warp_tot[warp] + incl - keep;
    // In-place safety: a token moves from frame t to pos <= t.  Frame t0-1 (the next chunk's
    // "prev") is only ever overwritten by itself (pos == t means every earlier frame was kept).
    if (keep) row[pos] = sym;
    if (tid == kCollapseThreads - 1) base_s = pos + keep;
    __syncthreads();
  }
  __syncthreads();
  const int total = (n > 0) ? base_s : 0;
  if (tid == 0) out_lens[b] = total;
  for (int t = total + tid; t < T; t += kCollapseThreads) row[t] = -1;
}

// persistent grid: as many CTAs as are resident at once (eight per SM for fp32)
template <typename E, bool kNarrowKey>
cudaError_t launch_stream(const E* logits, long long stride_b, long long stride_t, const int* lens, int T, int V, int B,
                          int* out_tokens, cudaStream_t stream) {
  static int n_sm = 0, per_sm = 0;
  if (n_sm == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) n_sm = 148;
  }
  if (per_sm == 0 && cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, frame_argmax_stream_kernel<E, kNarrowKey>, 256, 0) != cudaSuccess) {
    cudaGetLastError();
    per_sm = 8;
  }
  const long long rows = (long long)B * T;
  long long grid = (long long)n_sm * per_sm;
  if (grid * 8 > rows) grid = (rows + 7) / 8;
  frame_argmax_stream_kernel<E, kNarrowKey><<<(unsigned)grid, 256, 0, stream>>>(logits, stride_b, stride_t, lens, T, V, B, out_tokens);
  return cudaGetLastError();
}

template <typename E>
cudaError_t launch_argmax(const E* logits, long long stride_b, long long stride_t, const int* lens, int T, int V, int B,
                          int* out_tokens, cudaStream_t stream) {
  const long long rows = (long long)B * T;
  if (V <= 32) {
    frame_argmax_group_kernel<E, 8><<<(unsigned)((rows + 31) / 32), 256, 0, stream>>>(logits, stride_b, stride_t, lens, T, V, B, out_tokens);
  } else if (V <= 64) {
    frame_argmax_group_kernel<E, 16><<<(unsigned)((rows + 15) / 16), 256, 0, stream>>>(logits, stride_b, stride_t, lens, T, V, B, out_tokens);
  } else if (V <= 512) {
    const unsigned grid = (unsigned)((rows + 7) / 8);
    frame_argmax_warp_kernel<E><<<grid, 256, 0, stream>>>(logits, stride_b, stride_t, lens, T, V, B, out_tokens);
  } else if (std::is_same<E, float>::value && std::getenv("B200CTC_GREEDY_CTA_PER_ROW")) {   // the previous kernel, for A/B
    // measurements of fp32 rows; 16-bit rows always stream
    frame_argmax_cta_kernel<<<(unsigned)rows, 256, 0, stream>>>(reinterpret_cast<const float*>(logits), stride_b, stride_t, lens, T, V, B, out_tokens);
  } else if constexpr (std::is_same<E, float>::value) {
    return launch_stream<E, false>(logits, stride_b, stride_t, lens, T, V, B, out_tokens, stream);
  } else if (V > 65536) {
    return launch_stream<E, false>(logits, stride_b, stride_t, lens, T, V, B, out_tokens, stream);
  } else {
    return launch_stream<E, true>(logits, stride_b, stride_t, lens, T, V, B, out_tokens, stream);
  }
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_greedy(const void* logits, int dtype, long long stride_b, long long stride_t, const int* lens,
                          int T, int V, int B, int blank, int* out_tokens, int* out_lens, cudaStream_t stream) {
  if (B == 0) return cudaSuccess;
  if ((long long)B * T > 0) {
    cudaError_t e;
    if (dtype == B200CTC_BFLOAT16)
      e = launch_argmax(static_cast<const __nv_bfloat16*>(logits), stride_b, stride_t, lens, T, V, B, out_tokens, stream);
    else if (dtype == B200CTC_FLOAT16)
      e = launch_argmax(static_cast<const __half*>(logits), stride_b, stride_t, lens, T, V, B, out_tokens, stream);
    else
      e = launch_argmax(static_cast<const float*>(logits), stride_b, stride_t, lens, T, V, B, out_tokens, stream);
    if (e != cudaSuccess) return e;
  }
  collapse_kernel<<<B, kCollapseThreads, 0, stream>>>(lens, T, blank, out_tokens, out_lens);
  return cudaGetLastError();
}

}  // namespace b200ctc
