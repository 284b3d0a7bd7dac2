// Token-level back-off n-gram language model on the device: the layout ngram_lm.cu builds from an ARPA file and the
// lookups the fused prefix beam search (beam.cu) makes.  No other file knows the layout.
//
// Words: the decoder ids 0..V-1 whose symbol is a unigram of the model stand for themselves; <s> is V, </s> is V+1 and
// <unk> is V+2 (unless a symbol is literally "<unk>"), so a row over words has V+3 entries.  Nodes are the n-grams
// (node 0: the empty history, whose children are the unigrams), numbered by order, then parent, then word, so the
// children of a node are contiguous and sorted by word.
#pragma once

#include "common.cuh"

namespace b200ctc {

constexpr int kMaxLmOrder = 8;
constexpr double kLn10 = 2.302585092994045684017991454684364208;   // the double nearest ln 10 (oracle/lm_ref.py: LN10)

// The number of words of a model over V decoder symbols: the width of an LM row (LmView::n_words).
constexpr int lm_n_words(int V) { return V + 3; }

struct LmNode {
  double p;          // log10 p of the n-gram
  double bo;         // log10 back-off weight of the n-gram as a history (0 when the file gives none)
  int word;          // its last word
  int first_child;   // children: [first_child, first_child + n_child)
  int n_child;
  int backoff;       // the longest proper suffix that is an n-gram (0: the empty history)
  int depth;         // number of words
  int pad_;
};

struct LmView {
  const LmNode* nodes;
  const double* uni_p;   // [n_words] log10 p of each unigram (0 for a word that is none: never read)
  const int* uni_node;   // [n_words] node of each unigram, -1 for a word that is none
  const int* word_of;    // [V] the word of each decoder id (-1 at blank)
  int n_words;           // lm_n_words(V)
  int order;             // N
  int bos_state;         // the state of the empty prefix: <s> (order >= 2) or the empty history
  int eos;               // the word </s>
};

// The child of `node` with word w, or -1: a binary search over its children.
__device__ __forceinline__ int lm_child(const LmView& lm, int node, int w) {
  if (node == 0) return lm.uni_node[w];
  const LmNode& n = lm.nodes[node];
  int lo = n.first_child, hi = n.first_child + n.n_child;
  const int end = hi;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (lm.nodes[mid].word < w) lo = mid + 1;
    else hi = mid;
  }
  return (lo < end && lm.nodes[lo].word == w) ? lo : -1;
}

// A state is the node of the longest suffix of the history (at most N-1 words) that is an n-gram.  Appending word w:
// a suffix u+w can only be an n-gram when u is one (every n-gram's history is an n-gram), and the suffixes of the
// history that are n-grams are exactly the back-off chain of the state.
__device__ __forceinline__ int lm_next_state(const LmView& lm, int s, int w) {
  for (;;) {
    if (lm.nodes[s].depth < lm.order - 1) {
      const int ch = lm_child(lm, s, w);
      if (ch >= 0) return ch;
    }
    if (s == 0) return 0;
    s = lm.nodes[s].backoff;
  }
}

// The back-off chain of state s without the empty history, shallowest first; returns its length (< kMaxLmOrder).
__device__ __forceinline__ int lm_chain(const LmView& lm, int s, int* out) {
  int n = 0;
  for (int x = s; x != 0; x = lm.nodes[x].backoff) ++n;
  int k = n;
  for (int x = s; x != 0; x = lm.nodes[x].backoff) out[--k] = x;
  return n;
}

// log10 P(w | state) for every word, for up to n states at once, by the whole block:
//   row(empty) = the unigram row;   row(s)[w] = p(s w) if s w is an n-gram, else bo(s) + row(backoff(s))[w].
// The histories longer than a state are not n-grams: their back-off weight is 0 and their term an exact +0.0, so this
// is the right-associative sum of the definition, bit for bit, and every access to a row is coalesced.
//   row_idx[r]   the row (in units of n_words doubles) that entry r's row goes to, or -1: entry r is skipped
//   chain[r]     lm_chain of entry r's state, chain_len[r] its length
// The caller synchronises the block before (the arguments are in shared memory) and after (the rows are read).
__device__ __forceinline__ void lm_build_rows(const LmView& lm, double* rows, const int* row_idx,
                                              const int (*chain)[kMaxLmOrder], const int* chain_len, int n) {
  const int NW = lm.n_words;
  int max_len = 0;
  for (int r = 0; r < n; ++r) max_len = (row_idx[r] >= 0 && chain_len[r] > max_len) ? chain_len[r] : max_len;
  for (int k = threadIdx.x; k < n * NW; k += blockDim.x) {
    const int r = k / NW, w = k - r * NW;
    if (row_idx[r] >= 0) rows[(long long)row_idx[r] * NW + w] = lm.uni_p[w];
  }
  for (int l = 0; l < max_len; ++l) {
    __syncthreads();
    for (int k = threadIdx.x; k < n * NW; k += blockDim.x) {
      const int r = k / NW, w = k - r * NW;
      if (row_idx[r] >= 0 && l < chain_len[r]) {
        double* x = rows + (long long)row_idx[r] * NW + w;
        *x = __dadd_rn(lm.nodes[chain[r][l]].bo, *x);
      }
    }
    __syncthreads();
    for (int r = 0; r < n; ++r) {
      if (row_idx[r] < 0 || l >= chain_len[r]) continue;
      const LmNode& s = lm.nodes[chain[r][l]];
      for (int k = threadIdx.x; k < s.n_child; k += blockDim.x) {
        const LmNode& ch = lm.nodes[s.first_child + k];
        rows[(long long)row_idx[r] * NW + ch.word] = ch.p;
      }
    }
  }
}

}  // namespace b200ctc

struct b200ctc_ngram_lm;

namespace b200ctc {
// ngram_lm.cu: B200CTC_STATUS_SUCCESS when `lm` was loaded for V symbols with this blank on the current device.
int ngram_lm_check(const b200ctc_ngram_lm* lm, int V, int blank);
LmView ngram_lm_view(const b200ctc_ngram_lm* lm);
}  // namespace b200ctc
