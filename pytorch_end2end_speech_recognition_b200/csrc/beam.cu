// CTC prefix beam search on the GPU (SURVEY 8(f) rank 3), one CTA per utterance.
//
// Restates models/pytorch_v3/ctc/decoders/beam_search_decoder.py:33-124 (no language model: alpha = beta = 0,
// the only mode the reference implements): the beam holds prefixes with the log-probabilities of ending in blank
// (p_b) and in a non-blank (p_nb); every frame each prefix is kept ("stay": :75-81 for the blank, :105-109 for a
// repeated last symbol) and extended by every non-blank symbol (:86-101); candidates that denote the same prefix
// are merged (the reference's dict keyed by the prefix tuple); the beam_width best by logaddexp(p_b, p_nb) survive
// (:113-116, python's stable sort: ties keep the order in which the dict first saw the prefix).
//
// Arithmetic: float64 on the float32 log-probabilities, numpy's logaddexp formula -- what the reference computes
// under the numpy it was written for (a python float plus a float32 scalar is a float64 there).  Prefixes are
// nodes of a trie in global memory (parent, symbol); an extension coincides with a kept prefix exactly when that
// prefix's node is the child (parent = the extended prefix, symbol = the appended one), so merging needs no
// hashing.  Selection: beam_width rounds of a block-wide arg-max over the candidate scores with the reference's
// tie order (score descending, then first touch in its (symbol, beam entry) loop nest).
#include "common.cuh"

namespace b200ctc {

namespace {

constexpr int kBeamThreads = 256;
constexpr int kMaxBeam = 64;
constexpr double kLogE2 = 0.693147180559945309417232121458176568;

__device__ __forceinline__ double logaddexp64(double x, double y) {   // numpy: npy_logaddexp
  if (x == y) return x + kLogE2;
  const double tmp = x - y;
  if (tmp > 0) return x + log1p(exp(-tmp));
  if (tmp <= 0) return y + log1p(exp(tmp));
  return tmp;   // NaN
}

struct Best {
  double score;
  long long seq;   // tie order (smaller first); < 0: nothing
  int idx;         // >= 0: extension candidate i * V + c; < 0: stay candidate -(j + 1)
};
__device__ __forceinline__ bool better(const Best& a, const Best& b) {   // a before b in the reference's sort
  if (b.seq < 0) return a.seq >= 0;
  if (a.seq < 0) return false;
  if (a.score != b.score) return a.score > b.score;
  return a.seq < b.seq;
}

// E: the log-probabilities' type (float, __nv_bfloat16, __half).  A 16-bit value widens exactly to the float64 the
// arithmetic uses, so the result is the fp32 kernel's on the widened values.
template <typename E>
__global__ void __launch_bounds__(kBeamThreads) beam_search_kernel(
    const E* __restrict__ log_probs, long long stride_b, long long stride_t, const int* __restrict__ lens,
    int T, int V, int blank, int beam_width, double* __restrict__ cand_all, int2* __restrict__ nodes_all,
    int* __restrict__ out_tokens, int* __restrict__ out_lens, float* __restrict__ out_scores) {
  __shared__ double s_pb[2][kMaxBeam], s_pnb[2][kMaxBeam];      // current / next beam
  __shared__ int s_node[2][kMaxBeam], s_last[2][kMaxBeam];      // trie node of the prefix, its last symbol (-1: empty)
  __shared__ double s_stay_pb[kMaxBeam], s_stay_pnb[kMaxBeam], s_stay_tot[kMaxBeam];
  __shared__ long long s_stay_seq[kMaxBeam];
  __shared__ int s_parent_idx[kMaxBeam], s_stay_taken[kMaxBeam];
  __shared__ Best s_red[kBeamThreads / 32];
  __shared__ Best s_win;
  __shared__ int s_n_nodes;

  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n_frames = min(max(lens[b], 0), T);
  const E* lp_b = log_probs + (long long)b * stride_b;
  double* cand = cand_all + (long long)b * kMaxBeam * V;
  int2* nodes = nodes_all + (long long)b * ((long long)T * beam_width + 1);
  int cur = 0, W = 1;
  if (tid == 0) {
    s_pb[0][0] = 0.0; s_pnb[0][0] = -INFINITY; s_node[0][0] = 0; s_last[0][0] = -1;
    nodes[0] = make_int2(-1, -1);
    s_n_nodes = 1;
  }
  __syncthreads();

  for (int t = 0; t < n_frames; ++t) {
    const E* lp = lp_b + (long long)t * stride_t;
    const int nxt = cur ^ 1;
    // ---- extension candidates (prefix i, symbol c != blank): beam_search_decoder.py:86-101 ----
    for (int k = tid; k < W * V; k += kBeamThreads) {
      const int i = k / V, c = k - i * V;
      double v = INFINITY;                              // +inf: not a candidate
      if (c != blank) {
        const double p_t = (double)widen(lp[c]);
        v = (c != s_last[cur][i]) ? logaddexp64(s_pb[cur][i] + p_t, s_pnb[cur][i] + p_t) : s_pb[cur][i] + p_t;
      }
      cand[k] = v;
    }
    // which kept prefix is the child of another one in the beam?  (its extension then denotes the same prefix)
    if (tid < W) {
      const int par = nodes[s_node[cur][tid]].x;
      int pi = -1;
      for (int i = 0; i < W; ++i) pi = (s_node[cur][i] == par) ? i : pi;
      s_parent_idx[tid] = pi;
      s_stay_taken[tid] = 0;
    }
    __syncthreads();
    // ---- stay candidates: :75-81 (blank) and :105-109 (repeated last symbol), merged with the extension of the parent ----
    if (tid < W) {
      const int j = tid, e = s_last[cur][j];
      const double p_blank = (double)widen(lp[blank]);
      const double n_pb = logaddexp64(s_pb[cur][j] + p_blank, s_pnb[cur][j] + p_blank);
      double n_pnb = -INFINITY;
      long long seq = ((long long)blank * W + j) * 2;
      if (e >= 0) {
        const int pi = s_parent_idx[j];
        // the reference accumulates in beam order; logaddexp of two values is symmetric, so the order is immaterial
        if (pi >= 0) {
          n_pnb = logaddexp64(n_pnb, cand[pi * V + e]);
          cand[pi * V + e] = INFINITY;                  // that extension IS this prefix
          seq = min(seq, ((long long)e * W + pi) * 2);
        }
        n_pnb = logaddexp64(n_pnb, s_pnb[cur][j] + (double)widen(lp[e]));
        seq = min(seq, ((long long)e * W + j) * 2 + 1);
      }
      s_stay_pb[j] = n_pb; s_stay_pnb[j] = n_pnb;
      s_stay_tot[j] = logaddexp64(n_pb, n_pnb);
      s_stay_seq[j] = seq;
    }
    __syncthreads();
    // ---- the beam_width best candidates, in the reference's order (:113-116) ----
    const int n_cand_max = W * V;
    int n_new = 0;
    for (int r = 0; r < beam_width; ++r) {
      Best best; best.score = 0; best.seq = -1; best.idx = 0;
      for (int k = tid; k < n_cand_max; k += kBeamThreads) {
        const double v = cand[k];
        if (v == INFINITY) continue;
        const int i = k / V, c = k - i * V;
        Best x; x.score = v; x.seq = ((long long)c * W + i) * 2; x.idx = k;
        if (better(x, best)) best = x;
      }
      if (tid < W && !s_stay_taken[tid]) {
        Best x; x.score = s_stay_tot[tid]; x.seq = s_stay_seq[tid]; x.idx = -(tid + 1);
        if (better(x, best)) best = x;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        Best y;
        y.score = __shfl_xor_sync(0xffffffffu, best.score, o);
        y.seq = __shfl_xor_sync(0xffffffffu, best.seq, o);
        y.idx = __shfl_xor_sync(0xffffffffu, best.idx, o);
        if (better(y, best)) best = y;
      }
      if (lane == 0) s_red[warp] = best;
      __syncthreads();
      if (tid == 0) {
        Best w = s_red[0];
        for (int i = 1; i < kBeamThreads / 32; ++i) if (better(s_red[i], w)) w = s_red[i];
        s_win = w;
        if (w.seq >= 0) {
          if (w.idx < 0) {                               // a kept prefix
            const int j = -w.idx - 1;
            s_stay_taken[j] = 1;
            s_pb[nxt][r] = s_stay_pb[j]; s_pnb[nxt][r] = s_stay_pnb[j];
            s_node[nxt][r] = s_node[cur][j]; s_last[nxt][r] = s_last[cur][j];
          } else {                                       // a new prefix: one more trie node
            const int i = w.idx / V, c = w.idx - i * V;
            const int id = s_n_nodes++;
            nodes[id] = make_int2(s_node[cur][i], c);
            s_pb[nxt][r] = -INFINITY; s_pnb[nxt][r] = w.score;
            s_node[nxt][r] = id; s_last[nxt][r] = c;
            cand[w.idx] = INFINITY;
          }
        }
      }
      __syncthreads();
      if (s_win.seq < 0) break;                          // fewer candidates than beam_width
      ++n_new;
    }
    W = n_new;
    cur = nxt;
    __syncthreads();
  }
  // ---- best hypothesis: the first entry of the last beam (:118-119), read back along the trie ----
  if (tid == 0) {
    int len = 0;
    for (int n = s_node[cur][0]; n > 0; n = nodes[n].x) ++len;
    int* row = out_tokens + (long long)b * T;
    int pos = len;
    for (int n = s_node[cur][0]; n > 0; n = nodes[n].x) row[--pos] = nodes[n].y;
    for (int k = len; k < T; ++k) row[k] = -1;
    out_lens[b] = len;
    if (out_scores) out_scores[b] = (float)logaddexp64(s_pb[cur][0], s_pnb[cur][0]);
  }
}

}  // namespace

size_t beam_search_workspace_bytes(int B, int T, int V, int beam_width) {
  const size_t cand = (size_t)B * kMaxBeam * (size_t)V * sizeof(double);
  const size_t nodes = (size_t)B * ((size_t)T * beam_width + 1) * sizeof(int2);
  return (cand + 255) / 256 * 256 + nodes;
}

cudaError_t launch_beam_search(const void* log_probs, int dtype, long long stride_b, long long stride_t, const int* lens,
                               int T, int V, int B, int blank, int beam_width, int* out_tokens, int* out_lens,
                               float* out_scores, void* workspace, cudaStream_t stream) {
  if (B == 0) return cudaSuccess;
  if (beam_width < 1 || beam_width > kMaxBeam) return cudaErrorInvalidValue;
  unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
  const size_t cand = ((size_t)B * kMaxBeam * (size_t)V * sizeof(double) + 255) / 256 * 256;
  double* cand_all = reinterpret_cast<double*>(ws);
  int2* nodes_all = reinterpret_cast<int2*>(ws + cand);
  if (dtype == B200CTC_BFLOAT16)
    beam_search_kernel<<<B, kBeamThreads, 0, stream>>>(static_cast<const __nv_bfloat16*>(log_probs), stride_b, stride_t,
                                                       lens, T, V, blank, beam_width, cand_all, nodes_all, out_tokens,
                                                       out_lens, out_scores);
  else if (dtype == B200CTC_FLOAT16)
    beam_search_kernel<<<B, kBeamThreads, 0, stream>>>(static_cast<const __half*>(log_probs), stride_b, stride_t, lens, T,
                                                       V, blank, beam_width, cand_all, nodes_all, out_tokens, out_lens,
                                                       out_scores);
  else
    beam_search_kernel<<<B, kBeamThreads, 0, stream>>>(static_cast<const float*>(log_probs), stride_b, stride_t, lens, T,
                                                       V, blank, beam_width, cand_all, nodes_all, out_tokens, out_lens,
                                                       out_scores);
  return cudaGetLastError();
}

}  // namespace b200ctc
