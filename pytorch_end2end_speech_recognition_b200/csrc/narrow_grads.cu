// The last pass of a bfloat16 / float16 call: the fp32 gradient rows staged in the workspace by K1, the lattice and
// the occupancy pass are rounded once, to nearest even, into the caller's buffer of the logits' element type.  The
// gradient is formed in fp32 before this rounding: subtracting the occupancy from a softmax already rounded to
// bfloat16 would lose the whole gradient of a confident frame, where both are close to one.
//
// Bound: HBM.  Bytes per element: 4 read + 2 written, one pass, 128-bit loads and stores.
//
// Also here: the backward of such a loss, grads * grad_output in fp32 with one rounding to the gradient's type (a
// grad_output first rounded to float16 would turn a GradScaler's 2^16 into inf).  2 bytes read + 2 written per element.
#include <type_traits>

#include "common.cuh"

namespace b200ctc {

namespace {

constexpr int kNarrowThreads = 256;

__device__ __forceinline__ unsigned pack2(float lo, float hi, __nv_bfloat16*) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const unsigned*>(&h);
}
__device__ __forceinline__ unsigned pack2(float lo, float hi, __half*) {
  const __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<const unsigned*>(&h);
}
__device__ __forceinline__ void narrow_store(float x, __nv_bfloat16* d) { *d = __float2bfloat16_rn(x); }
__device__ __forceinline__ void narrow_store(float x, __half* d) { *d = __float2half_rn(x); }

// VEC: dst is 16-byte aligned; eight elements per step (two 128-bit loads, one 128-bit store), scalar tail.
template <typename T, bool VEC>
__global__ void __launch_bounds__(kNarrowThreads) narrow_grads_kernel(const float* __restrict__ src, T* __restrict__ dst,
                                                                      long long n) {
  const long long tid = (long long)blockIdx.x * kNarrowThreads + threadIdx.x;
  const long long stride = (long long)gridDim.x * kNarrowThreads;
  long long done = 0;
  if (VEC) {
    const long long n8 = n >> 3;
    const float4* s4 = reinterpret_cast<const float4*>(src);
    uint4* d8 = reinterpret_cast<uint4*>(dst);
    for (long long i = tid; i < n8; i += stride) {
      const float4 a = __ldcs(s4 + 2 * i), b = __ldcs(s4 + 2 * i + 1);
      __stcs(d8 + i, make_uint4(pack2(a.x, a.y, dst), pack2(a.z, a.w, dst), pack2(b.x, b.y, dst), pack2(b.z, b.w, dst)));
    }
    done = n8 << 3;
  }
  for (long long i = done + tid; i < n; i += stride) narrow_store(src[i], dst + i);
}

template <typename T>
cudaError_t launch_narrow_of(const float* src, T* dst, long long n, cudaStream_t stream) {
  const bool vec = (reinterpret_cast<uintptr_t>(dst) & 15) == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0;
  const long long per_thread = vec ? 8 : 1;
  long long blocks = (n / per_thread + kNarrowThreads - 1) / kNarrowThreads;
  if (blocks > 8192) blocks = 8192;            // larger inputs: grid-stride loop
  if (blocks < 1) blocks = 1;
  if (vec) narrow_grads_kernel<T, true><<<(unsigned)blocks, kNarrowThreads, 0, stream>>>(src, dst, n);
  else narrow_grads_kernel<T, false><<<(unsigned)blocks, kNarrowThreads, 0, stream>>>(src, dst, n);
  return cudaGetLastError();
}

// out[i] = grads[i] * scale[s] in fp32, rounded once; s = 0, or the utterance b = (i / V) % B when PER_UTT.  VEC: both
// buffers 16-byte aligned, eight elements per step.
template <typename T, bool VEC, bool PER_UTT>
__global__ void __launch_bounds__(kNarrowThreads) scale_grads_kernel(const T* grads, T* out,
                                                                     long long n, int V, int B,
                                                                     const float* __restrict__ scale) {
  using T2 = std::conditional_t<std::is_same_v<T, __half>, __half2, __nv_bfloat162>;
  const long long tid = (long long)blockIdx.x * kNarrowThreads + threadIdx.x;
  const long long stride = (long long)gridDim.x * kNarrowThreads;
  auto scale_of = [&](long long i) { return PER_UTT ? __ldg(scale + (i / V) % B) : __ldg(scale); };
  const float s0 = PER_UTT ? 0.f : __ldg(scale);
  long long done = 0;
  if (VEC) {
    const long long n8 = n >> 3;
    const uint4* g8 = reinterpret_cast<const uint4*>(grads);
    uint4* o8 = reinterpret_cast<uint4*>(out);
    for (long long i = tid; i < n8; i += stride) {
      const uint4 u = __ldcs(g8 + i);
      const T2* h = reinterpret_cast<const T2*>(&u);
      float f[8];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float2 w = widen2(h[k]);
        f[2 * k] = w.x;
        f[2 * k + 1] = w.y;
      }
      if (PER_UTT) {
        const long long r0 = (8 * i) / V, r1 = (8 * i + 7) / V;
        if (r0 == r1) {
          const float s = __ldg(scale + r0 % B);
#pragma unroll
          for (int k = 0; k < 8; ++k) f[k] *= s;
        } else {
#pragma unroll
          for (int k = 0; k < 8; ++k) f[k] *= scale_of(8 * i + k);
        }
      } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) f[k] *= s0;
      }
      __stcs(o8 + i, make_uint4(pack2(f[0], f[1], out), pack2(f[2], f[3], out), pack2(f[4], f[5], out),
                                pack2(f[6], f[7], out)));
    }
    done = n8 << 3;
  }
  for (long long i = done + tid; i < n; i += stride)
    narrow_store(widen(grads[i]) * (PER_UTT ? scale_of(i) : s0), out + i);
}

template <typename T>
cudaError_t launch_scale_of(const T* grads, T* out, long long n, int V, int B, const float* scale, bool per_utt,
                            cudaStream_t stream) {
  const bool vec = ((reinterpret_cast<uintptr_t>(grads) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
  long long blocks = (n / (vec ? 8 : 1) + kNarrowThreads - 1) / kNarrowThreads;
  if (blocks > 8192) blocks = 8192;            // larger inputs: grid-stride loop
  if (blocks < 1) blocks = 1;
  const dim3 grid((unsigned)blocks);
  if (vec && per_utt) scale_grads_kernel<T, true, true><<<grid, kNarrowThreads, 0, stream>>>(grads, out, n, V, B, scale);
  else if (vec) scale_grads_kernel<T, true, false><<<grid, kNarrowThreads, 0, stream>>>(grads, out, n, V, B, scale);
  else if (per_utt) scale_grads_kernel<T, false, true><<<grid, kNarrowThreads, 0, stream>>>(grads, out, n, V, B, scale);
  else scale_grads_kernel<T, false, false><<<grid, kNarrowThreads, 0, stream>>>(grads, out, n, V, B, scale);
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_scale_grads(const void* grads, void* out, int dtype, int T, int B, int V, const float* scale,
                               int n_scale, cudaStream_t stream) {
  const long long n = (long long)T * B * V;
  if (n == 0) return cudaSuccess;
  const bool per_utt = n_scale != 1;
  if (dtype == B200CTC_BFLOAT16)
    return launch_scale_of(static_cast<const __nv_bfloat16*>(grads), static_cast<__nv_bfloat16*>(out), n, V, B, scale,
                           per_utt, stream);
  if (dtype == B200CTC_FLOAT16)
    return launch_scale_of(static_cast<const __half*>(grads), static_cast<__half*>(out), n, V, B, scale, per_utt, stream);
  return cudaErrorInvalidValue;
}

cudaError_t launch_narrow_grads(const float* src, void* dst, long long n, int dtype, cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  if (dtype == B200CTC_BFLOAT16) return launch_narrow_of(src, static_cast<__nv_bfloat16*>(dst), n, stream);
  if (dtype == B200CTC_FLOAT16) return launch_narrow_of(src, static_cast<__half*>(dst), n, stream);
  return cudaErrorInvalidValue;
}

}  // namespace b200ctc
