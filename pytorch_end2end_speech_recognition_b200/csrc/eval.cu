// Evaluation kernels (SURVEY 8(f) rank 4): the steps after the decoder.
//
//  * edit_distance_kernel -- batched Levenshtein distance with the substitution / insertion / deletion counts
//    of the reference's utils/evaluation/edit_distance.py:53-126 (compute_wer: a numpy uint16 matrix filled by
//    two python loops, then a backtrace), one CTA per (reference, hypothesis) pair.  The matrix is filled along
//    anti-diagonals (cells of one diagonal are independent); only the backtrace decision of every cell is kept
//    (one byte), in the order the reference tests them (:99-117): match on the diagonal, insertion, substitution,
//    else deletion.
//  * softmax_temperature_kernel -- the fused softmax(logits / temperature) of CTC.posteriors
//    (models/pytorch_v3/ctc/ctc.py:455-502), one warp per row, online max / sum.
//
// Bound: HBM for the softmax (4V read, or 2V for 16-bit logits, + 4V written per row: probs are fp32 for every type); the edit distance is a latency-bound dynamic
// programme of (R + H) dependent steps per pair and is parallel over the mini-batch.
#include "common.cuh"

namespace b200ctc {

namespace {

constexpr int kEdThreads = 256;
enum : unsigned char { kDirNone = 0, kDirMatch = 1, kDirIns = 2, kDirSub = 3, kDirDel = 4 };

__global__ void __launch_bounds__(kEdThreads) edit_distance_kernel(
    const int* __restrict__ refs, int ref_stride, const int* __restrict__ ref_lens,
    const int* __restrict__ hyps, int hyp_stride, const int* __restrict__ hyp_lens,
    int max_ref, int max_hyp, int* __restrict__ out4, unsigned char* __restrict__ dirs_all) {
  extern __shared__ int s_diag[];                     // three anti-diagonals, indexed by the row i: [3][max_ref + 1]
  const int b = blockIdx.x, tid = threadIdx.x;
  const int R = min(max(ref_lens[b], 0), max_ref), H = min(max(hyp_lens[b], 0), max_hyp);
  const int* ref = refs + (long long)b * ref_stride;
  const int* hyp = hyps + (long long)b * hyp_stride;
  unsigned char* dirs = dirs_all + (long long)b * (max_ref + 1) * (max_hyp + 1);   // [R+1][H+1], row stride H + 1
  const int W = max_ref + 1;
  int* d2 = s_diag;          // diagonal k - 2
  int* d1 = s_diag + W;      // diagonal k - 1
  int* d0 = s_diag + 2 * W;  // diagonal k
  for (int k = 0; k <= R + H; ++k) {
    const int i_lo = max(0, k - H), i_hi = min(R, k);
    for (int i = i_lo + tid; i <= i_hi; i += kEdThreads) {
      const int j = k - i;
      int d;
      unsigned char dir;
      if (i == 0) { d = j; dir = j == 0 ? kDirNone : kDirIns; }            // d[0][j] = j  (:69-70)
      else if (j == 0) { d = i; dir = kDirDel; }                            // d[i][0] = i  (:71-72)
      else {
        const bool eq = ref[i - 1] == hyp[j - 1];
        const int diag = d2[i - 1], left = d1[i], up = d1[i - 1];
        d = eq ? diag : min(min(diag, left), up) + 1;                       // :77-83
        // backtrace decision in the reference's order (:99-117)
        if (eq && d == diag) dir = kDirMatch;
        else if (d == left + 1) dir = kDirIns;
        else if (d == diag + 1) dir = kDirSub;
        else dir = kDirDel;
      }
      d0[i] = d;
      dirs[(long long)i * (H + 1) + j] = dir;
    }
    __syncthreads();
    int* t = d2; d2 = d1; d1 = d0; d0 = t;
  }
  if (tid == 0) {
    __threadfence_block();
    const int dist = d1[R];                            // after the last rotation d1 is diagonal R + H
    int x = R, y = H, sub = 0, ins = 0, del = 0;
    while (x > 0 || y > 0) {
      const unsigned char dir = dirs[(long long)x * (H + 1) + y];
      if (dir == kDirMatch) { --x; --y; }
      else if (dir == kDirIns) { ++ins; --y; }
      else if (dir == kDirSub) { ++sub; --x; --y; }
      else { ++del; --x; }
    }
    out4[4 * b + 0] = dist;
    out4[4 * b + 1] = sub;
    out4[4 * b + 2] = ins;
    out4[4 * b + 3] = del;
  }
}

// one warp per row; V-strided online softmax (two reads of the row: the second one hits L1/L2).  E: the logits' type;
// every type keeps the fp32 element-to-lane assignment and summation order, so a 16-bit row gives bit for bit what
// the fp32 kernel gives on its widened values.
template <typename E>
__global__ void __launch_bounds__(256) softmax_temperature_kernel(
    const E* __restrict__ logits, long long stride_b, long long stride_t, int T, int V, long long rows,
    float inv_temperature, float* __restrict__ probs) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const long long b = row / T, t = row - b * T;
  const E* x = logits + b * stride_b + t * stride_t;
  float m = -INFINITY, s = 0.f;
  for (int v = lane; v < V; v += 32) {
    const float z = widen(__ldg(x + v)) * inv_temperature;
    const float nm = fmaxf(m, z);
    s = s * __expf(m - nm) + __expf(z - nm);
    m = nm;
  }
  const float gm = warp_max(m);
  s = warp_sum(s * __expf(m - gm));                    // lanes that saw nothing: m = -inf, s = 0 -> 0 * exp(-inf) = 0
  const float inv = 1.0f / s;
  float* y = probs + row * V;
  for (int v = lane; v < V; v += 32) y[v] = __expf(widen(__ldg(x + v)) * inv_temperature - gm) * inv;
}

}  // namespace

size_t edit_distance_workspace_bytes(int B, int max_ref, int max_hyp) {
  return (size_t)B * (size_t)(max_ref + 1) * (size_t)(max_hyp + 1);
}

cudaError_t launch_edit_distance(const int* refs, int ref_stride, const int* ref_lens, const int* hyps, int hyp_stride,
                                 const int* hyp_lens, int B, int max_ref, int max_hyp, int* out4, void* workspace,
                                 cudaStream_t stream) {
  if (B == 0) return cudaSuccess;
  const size_t smem = (size_t)3 * (max_ref + 1) * sizeof(int);
  if (smem > 200 * 1024) return cudaErrorInvalidConfiguration;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(edit_distance_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  edit_distance_kernel<<<B, kEdThreads, smem, stream>>>(refs, ref_stride, ref_lens, hyps, hyp_stride, hyp_lens, max_ref,
                                                        max_hyp, out4, reinterpret_cast<unsigned char*>(workspace));
  return cudaGetLastError();
}

cudaError_t launch_softmax_temperature(const void* logits, int dtype, long long stride_b, long long stride_t, int T, int V,
                                       int B, float inv_temperature, float* probs, cudaStream_t stream) {
  const long long rows = (long long)B * T;
  if (rows == 0) return cudaSuccess;
  const long long grid = (rows + 7) / 8;
  if (grid > 0x7fffffffLL) return cudaErrorInvalidConfiguration;
  if (dtype == B200CTC_BFLOAT16)
    softmax_temperature_kernel<<<(unsigned)grid, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(logits), stride_b,
                                                                   stride_t, T, V, rows, inv_temperature, probs);
  else if (dtype == B200CTC_FLOAT16)
    softmax_temperature_kernel<<<(unsigned)grid, 256, 0, stream>>>(static_cast<const __half*>(logits), stride_b, stride_t,
                                                                   T, V, rows, inv_temperature, probs);
  else
    softmax_temperature_kernel<<<(unsigned)grid, 256, 0, stream>>>(static_cast<const float*>(logits), stride_b, stride_t,
                                                                   T, V, rows, inv_temperature, probs);
  return cudaGetLastError();
}

}  // namespace b200ctc
