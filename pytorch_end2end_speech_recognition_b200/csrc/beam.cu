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
//
// Shallow fusion with an n-gram language model (kLM): every prefix also carries its LM state and its score
//   S(empty) = 0,  S(prefix + c) = S(prefix) + (alpha * lnP(c | prefix) + beta)
// and candidates are ranked by logaddexp(p_b, p_nb) + S (the CTC part evolves as without the LM).  After the last
// frame the hypothesis is the entry with the largest (logaddexp(p_b, p_nb) + S) + alpha * lnP(</s> | prefix).  Each
// multiplication and addition is rounded on its own (__dmul_rn / __dadd_rn: nvcc would contract a*b+c into a DFMA,
// numpy does not).  The LM instantiation makes the trie canonical -- a node (parent, symbol) is looked up in a
// per-utterance hash table before one is created -- so node identity is sequence identity and the merge by parent
// is exact even when a prefix leaves the beam and comes back; the LM-free instantiations keep their code.
#include "common.cuh"
#include "ngram_lm.cuh"

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

// What the LM instantiation adds to the workspace and the arguments.
struct BeamLmArgs {
  LmView lm;
  double alpha, beta;
  double* keys_all;   // [B][beam_width * V] ranking key of each extension candidate, beside its CTC value in cand
  double* rows_all;   // [B][beam_width][n_words] log10 P(w | state) of the prefixes in the beam
  int* hash_all;      // [B][hash_cap] canonical trie: node ids by hash of (parent, symbol), -1 empty
  long long hash_cap;
};

// Per beam entry (current / next beam) and per new prefix of a frame.
struct BeamLmShared {
  double S[2][kMaxBeam];            // LM score of the prefix
  int state[2][kMaxBeam];           // LM state
  int row[2][kMaxBeam];             // its row in rows_all
  int par[kMaxBeam];                // next beam: the entry of the current beam it extends, -1 for a kept prefix
  int new_row[kMaxBeam];            // row to build for a new prefix, -1 for a kept one
  int chain[kMaxBeam][kMaxLmOrder];
  int chain_len[kMaxBeam];
  int row_used[kMaxBeam];
};

// The LM instantiation's shared state; only the kernels that call this allocate it.
template <bool kLM>
__device__ __forceinline__ BeamLmShared* lm_shared() { return nullptr; }
template <>
__device__ __forceinline__ BeamLmShared* lm_shared<true>() {
  __shared__ BeamLmShared s_lm;
  return &s_lm;
}

__device__ __forceinline__ unsigned trie_hash(int parent, int c) {
  const unsigned long long x = (((unsigned long long)(unsigned)parent << 32) | (unsigned)c) * 0x9E3779B97F4A7C15ull;
  return (unsigned)(x >> 32);
}

// S(prefix i + c) from S(prefix i) and the row of prefix i
__device__ __forceinline__ double lm_extended_score(const BeamLmArgs& a, double S, const double* row, int c) {
  const double lnp = __dmul_rn(row[a.lm.word_of[c]], kLn10);
  return __dadd_rn(S, __dadd_rn(__dmul_rn(a.alpha, lnp), a.beta));
}

// E: the log-probabilities' type (float, __nv_bfloat16, __half).  A 16-bit value widens exactly to the float64 the
// arithmetic uses, so the result is the fp32 kernel's on the widened values.
// kLM: shallow fusion with the n-gram model of `lma` (unused otherwise).
template <typename E, bool kLM>
__global__ void __launch_bounds__(kBeamThreads) beam_search_kernel(
    const E* __restrict__ log_probs, long long stride_b, long long stride_t, const int* __restrict__ lens,
    int T, int V, int blank, int beam_width, double* __restrict__ cand_all, int2* __restrict__ nodes_all,
    int* __restrict__ out_tokens, int* __restrict__ out_lens, float* __restrict__ out_scores, BeamLmArgs lma) {
  __shared__ double s_pb[2][kMaxBeam], s_pnb[2][kMaxBeam];      // current / next beam
  __shared__ int s_node[2][kMaxBeam], s_last[2][kMaxBeam];      // trie node of the prefix, its last symbol (-1: empty)
  __shared__ double s_stay_pb[kMaxBeam], s_stay_pnb[kMaxBeam], s_stay_tot[kMaxBeam];
  __shared__ long long s_stay_seq[kMaxBeam];
  __shared__ int s_parent_idx[kMaxBeam], s_stay_taken[kMaxBeam];
  __shared__ Best s_red[kBeamThreads / 32];
  __shared__ Best s_win;
  __shared__ int s_n_nodes;
  BeamLmShared* const L = lm_shared<kLM>();

  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n_frames = min(max(lens[b], 0), T);
  const E* lp_b = log_probs + (long long)b * stride_b;
  // per-utterance strides of beam_layout (BeamLayout): derived here rather than passed, which keeps the kernels at
  // their register counts without spills (a stride read from the parameters costs the LM-free kernel 10 registers)
  double* cand = cand_all + (long long)b * (kLM ? beam_width : kMaxBeam) * V;
  int2* nodes = nodes_all + (long long)b * ((long long)T * beam_width + 1);
  // ranking keys: the CTC value itself without the LM
  double* keys = kLM ? lma.keys_all + (long long)b * beam_width * V : cand;
  double* rows = kLM ? lma.rows_all + (long long)b * beam_width * lma.lm.n_words : nullptr;
  int* hash = kLM ? lma.hash_all + (long long)b * lma.hash_cap : nullptr;
  unsigned hash_mask = 0;
  int cur = 0, W = 1;
  if (tid == 0) {
    s_pb[0][0] = 0.0; s_pnb[0][0] = -INFINITY; s_node[0][0] = 0; s_last[0][0] = -1;
    nodes[0] = make_int2(-1, -1);
    s_n_nodes = 1;
  }
  if constexpr (kLM) {
    // a table of at least twice the nodes this utterance can create
    long long cap = 1;
    while (cap < 2 * ((long long)n_frames * beam_width + 1)) cap <<= 1;
    hash_mask = (unsigned)(cap - 1);
    for (long long k = tid; k < cap; k += kBeamThreads) hash[k] = -1;
    if (tid == 0) {
      L->S[0][0] = 0.0; L->state[0][0] = lma.lm.bos_state; L->row[0][0] = 0;
      L->new_row[0] = 0;
      L->chain_len[0] = lm_chain(lma.lm, lma.lm.bos_state, L->chain[0]);
    }
    __syncthreads();
    lm_build_rows(lma.lm, rows, L->new_row, L->chain, L->chain_len, 1);
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
      if constexpr (kLM) {
        // logaddexp(-inf, v) is v: the key of a new prefix is its p_nb plus its S
        keys[k] = c != blank
                      ? __dadd_rn(v, lm_extended_score(lma, L->S[cur][i], rows + (long long)L->row[cur][i] * lma.lm.n_words, c))
                      : INFINITY;
      }
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
          if constexpr (kLM) keys[pi * V + e] = INFINITY;
          seq = min(seq, ((long long)e * W + pi) * 2);
        }
        n_pnb = logaddexp64(n_pnb, s_pnb[cur][j] + (double)widen(lp[e]));
        seq = min(seq, ((long long)e * W + j) * 2 + 1);
      }
      s_stay_pb[j] = n_pb; s_stay_pnb[j] = n_pnb;
      s_stay_tot[j] = logaddexp64(n_pb, n_pnb);
      if constexpr (kLM) s_stay_tot[j] = __dadd_rn(s_stay_tot[j], L->S[cur][j]);
      s_stay_seq[j] = seq;
    }
    __syncthreads();
    // ---- the beam_width best candidates, in the reference's order (:113-116) ----
    const int n_cand_max = W * V;
    int n_new = 0;
    for (int r = 0; r < beam_width; ++r) {
      Best best; best.score = 0; best.seq = -1; best.idx = 0;
      for (int k = tid; k < n_cand_max; k += kBeamThreads) {
        const double v = keys[k];
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
            if constexpr (kLM) {
              L->S[nxt][r] = L->S[cur][j]; L->state[nxt][r] = L->state[cur][j]; L->row[nxt][r] = L->row[cur][j];
              L->par[r] = -1;
            }
          } else if constexpr (kLM) {                    // a new prefix: its node and LM state follow the rounds
            const int i = w.idx / V, c = w.idx - i * V;
            s_pb[nxt][r] = -INFINITY; s_pnb[nxt][r] = cand[w.idx];
            s_last[nxt][r] = c;
            L->S[nxt][r] = lm_extended_score(lma, L->S[cur][i], rows + (long long)L->row[cur][i] * lma.lm.n_words, c);
            L->par[r] = i;
            keys[w.idx] = INFINITY;
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
    if constexpr (kLM) {
      // new prefixes: the node of (parent, symbol) if the trie has it (the prefix was in the beam before), and the
      // LM state; the new prefixes of a frame are distinct sequences, so they are looked up and inserted in parallel
      const int r = tid;
      const bool is_new = r < n_new && L->par[r] >= 0;
      int parent = 0, c = 0, found = -1;
      unsigned h = 0;
      if (is_new) {
        c = s_last[nxt][r];
        parent = s_node[cur][L->par[r]];
        for (h = trie_hash(parent, c) & hash_mask;; h = (h + 1) & hash_mask) {
          const int id = __ldcg(hash + h);
          if (id < 0) break;
          const int2 nd = nodes[id];
          if (nd.x == parent && nd.y == c) { found = id; break; }
        }
        const int st = lm_next_state(lma.lm, L->state[cur][L->par[r]], lma.lm.word_of[c]);
        L->state[nxt][r] = st;
        L->chain_len[r] = lm_chain(lma.lm, st, L->chain[r]);
      }
      if (tid == 0) {   // rows: a kept prefix keeps its own, a new one takes one no kept prefix holds
        for (int q = 0; q < beam_width; ++q) L->row_used[q] = 0;
        for (int q = 0; q < n_new; ++q) if (L->par[q] < 0) L->row_used[L->row[nxt][q]] = 1;
        int f = 0;
        for (int q = 0; q < n_new; ++q) {
          if (L->par[q] < 0) { L->new_row[q] = -1; continue; }
          while (L->row_used[f]) ++f;
          L->row[nxt][q] = L->new_row[q] = f++;
        }
      }
      __syncthreads();
      if (is_new) {
        if (found < 0) {
          found = s_n_nodes + r;                          // at most beam_width new nodes a frame: T * W + 1 in all
          nodes[found] = make_int2(parent, c);
          while (atomicCAS(hash + h, -1, found) != -1) h = (h + 1) & hash_mask;
        }
        s_node[nxt][r] = found;
      }
      lm_build_rows(lma.lm, rows, L->new_row, L->chain, L->chain_len, n_new);
      __syncthreads();
      if (tid == 0) s_n_nodes += n_new;
    }
    W = n_new;
    cur = nxt;
    __syncthreads();
  }
  // ---- best hypothesis: the first entry of the last beam (:118-119), read back along the trie ----
  if (tid == 0) {
    int best = 0;
    double lm_score = 0.0;
    if constexpr (kLM) {   // with the end of sentence: the largest total, ties to the earlier entry
      for (int j = 0; j < W; ++j) {
        const double eos = rows[(long long)L->row[cur][j] * lma.lm.n_words + lma.lm.eos];
        const double f = __dadd_rn(__dadd_rn(logaddexp64(s_pb[cur][j], s_pnb[cur][j]), L->S[cur][j]),
                                   __dmul_rn(lma.alpha, __dmul_rn(eos, kLn10)));
        if (j == 0 || f > lm_score) { lm_score = f; best = j; }
      }
    }
    int len = 0;
    for (int n = s_node[cur][best]; n > 0; n = nodes[n].x) ++len;
    int* row = out_tokens + (long long)b * T;
    int pos = len;
    for (int n = s_node[cur][best]; n > 0; n = nodes[n].x) row[--pos] = nodes[n].y;
    for (int k = len; k < T; ++k) row[k] = -1;
    out_lens[b] = len;
    if (out_scores) out_scores[b] = kLM ? (float)lm_score : (float)logaddexp64(s_pb[cur][0], s_pnb[cur][0]);
  }
}

// The workspace, for the LM-free search (n_words = 0) and the LM search (n_words: the LM's row width,
// LmView::n_words).  Regions: the candidate values, the LM's ranking keys, the trie nodes, the LM's hash table and
// rows; each starts on a 256-byte boundary and an LM region is empty without the LM.
struct BeamLayout {
  long long cand_stride;   // doubles of candidates (and of keys) per utterance
  long long node_stride;   // trie nodes per utterance: the root and at most beam_width new ones a frame
  long long row_stride;    // doubles of LM rows per utterance: beam_width rows of n_words
  long long hash_cap;      // slots of the hash table per utterance: at least twice the nodes
  size_t off_keys, off_nodes, off_hash, off_rows, total;
};

BeamLayout beam_layout(int B, int T, int V, int beam_width, int n_words) {
  auto al = [](size_t x) { return (x + 255) / 256 * 256; };
  const bool lm = n_words > 0;
  BeamLayout l;
  l.cand_stride = (long long)(lm ? beam_width : kMaxBeam) * V;
  l.node_stride = (long long)T * beam_width + 1;
  l.row_stride = (long long)beam_width * n_words;
  l.hash_cap = 0;
  if (lm) {
    l.hash_cap = 1;
    while (l.hash_cap < 2 * l.node_stride) l.hash_cap <<= 1;
  }
  const size_t cand = (size_t)B * l.cand_stride * sizeof(double), nodes = (size_t)B * l.node_stride * sizeof(int2);
  l.off_keys = al(cand);
  l.off_nodes = l.off_keys + (lm ? al(cand) : 0);
  l.off_hash = l.off_nodes + al(nodes);
  l.off_rows = l.off_hash + al((size_t)B * l.hash_cap * sizeof(int));
  l.total = lm ? l.off_rows + (size_t)B * l.row_stride * sizeof(double) : l.off_nodes + nodes;
  return l;
}

// lma: the LM, alpha and beta (kLM); its workspace pointers are filled in here
template <bool kLM>
cudaError_t launch(const void* log_probs, int dtype, long long stride_b, long long stride_t, const int* lens, int T, int V,
                   int B, int blank, int beam_width, int* out_tokens, int* out_lens, float* out_scores, void* workspace,
                   BeamLmArgs lma, cudaStream_t stream) {
  if (B == 0) return cudaSuccess;
  if (beam_width < 1 || beam_width > kMaxBeam) return cudaErrorInvalidValue;
  const BeamLayout l = beam_layout(B, T, V, beam_width, kLM ? lma.lm.n_words : 0);
  unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
  double* cand = reinterpret_cast<double*>(ws);
  int2* nodes = reinterpret_cast<int2*>(ws + l.off_nodes);
  if (kLM) {
    lma.keys_all = reinterpret_cast<double*>(ws + l.off_keys);
    lma.rows_all = reinterpret_cast<double*>(ws + l.off_rows);
    lma.hash_all = reinterpret_cast<int*>(ws + l.off_hash);
    lma.hash_cap = l.hash_cap;
  }
  if (dtype == B200CTC_BFLOAT16)
    beam_search_kernel<__nv_bfloat16, kLM><<<B, kBeamThreads, 0, stream>>>(
        static_cast<const __nv_bfloat16*>(log_probs), stride_b, stride_t, lens, T, V, blank, beam_width, cand,
        nodes, out_tokens, out_lens, out_scores, lma);
  else if (dtype == B200CTC_FLOAT16)
    beam_search_kernel<__half, kLM><<<B, kBeamThreads, 0, stream>>>(
        static_cast<const __half*>(log_probs), stride_b, stride_t, lens, T, V, blank, beam_width, cand,
        nodes, out_tokens, out_lens, out_scores, lma);
  else
    beam_search_kernel<float, kLM><<<B, kBeamThreads, 0, stream>>>(
        static_cast<const float*>(log_probs), stride_b, stride_t, lens, T, V, blank, beam_width, cand,
        nodes, out_tokens, out_lens, out_scores, lma);
  return cudaGetLastError();
}

}  // namespace

size_t beam_search_workspace_bytes(int B, int T, int V, int beam_width) {
  return beam_layout(B, T, V, beam_width, 0).total;
}

cudaError_t launch_beam_search(const void* log_probs, int dtype, long long stride_b, long long stride_t, const int* lens,
                               int T, int V, int B, int blank, int beam_width, int* out_tokens, int* out_lens,
                               float* out_scores, void* workspace, cudaStream_t stream) {
  return launch<false>(log_probs, dtype, stride_b, stride_t, lens, T, V, B, blank, beam_width, out_tokens, out_lens,
                       out_scores, workspace, BeamLmArgs{}, stream);
}

size_t beam_search_lm_workspace_bytes(int B, int T, int V, int beam_width, int n_words) {
  return beam_layout(B, T, V, beam_width, n_words).total;
}

cudaError_t launch_beam_search_lm(const void* log_probs, int dtype, long long stride_b, long long stride_t,
                                  const int* lens, int T, int V, int B, int blank, int beam_width, const LmView& lm,
                                  double alpha, double beta, int* out_tokens, int* out_lens, float* out_scores,
                                  void* workspace, cudaStream_t stream) {
  BeamLmArgs a{};
  a.lm = lm;
  a.alpha = alpha;
  a.beta = beta;
  return launch<true>(log_probs, dtype, stride_b, stride_t, lens, T, V, B, blank, beam_width, out_tokens, out_lens,
                      out_scores, workspace, a, stream);
}

}  // namespace b200ctc
