// Evaluation kernels (SURVEY 8(f) rank 4): the steps after the decoder.
//
//  * edit_distance_kernel -- batched Levenshtein distance with the substitution / insertion / deletion counts
//    of the reference's utils/evaluation/edit_distance.py:53-126 (compute_wer: a numpy uint16 matrix filled by
//    two python loops, then a backtrace), one CTA per (reference, hypothesis) pair.  The matrix is filled along
//    anti-diagonals (cells of one diagonal are independent); only the backtrace decision of every cell is kept
//    (one byte), in the order the reference tests them (:99-117): match on the diagonal, insertion, substitution,
//    else deletion.
//  * word_errors_kernel -- the same DP (edit_distance_dp) over words and over the space-free characters of
//    character-level hypotheses: the WER / CER of character models (examples/librispeech/s5/exp/metrics/
//    character.py:17-158), two CTAs per pair, words identified through a per-pair hash table.
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

// Edit distance of ref[0, R) and hyp[0, H) with the counts of the backtrace, by the whole CTA; the result is valid in
// thread 0 only.  s_diag: three anti-diagonals of W >= R + 1 ints in shared memory; dirs: (R + 1) * (H + 1) bytes of
// global memory, row stride H + 1.  ref / hyp are read with whatever loads the caller's pointers allow: a caller
// that wrote them itself passes plain pointers and must __syncthreads() first.
__device__ __forceinline__ int4 edit_distance_dp(const int* ref, int R, const int* hyp, int H, unsigned char* dirs,
                                                 int* s_diag, int W) {
  const int tid = threadIdx.x;
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
  int4 r = make_int4(0, 0, 0, 0);
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
    r = make_int4(dist, sub, ins, del);
  }
  return r;
}

__global__ void __launch_bounds__(kEdThreads) edit_distance_kernel(
    const int* __restrict__ refs, int ref_stride, const int* __restrict__ ref_lens,
    const int* __restrict__ hyps, int hyp_stride, const int* __restrict__ hyp_lens,
    int max_ref, int max_hyp, int* __restrict__ out4, unsigned char* __restrict__ dirs_all) {
  extern __shared__ int s_diag[];                     // three anti-diagonals, indexed by the row i: [3][max_ref + 1]
  const int b = blockIdx.x;
  const int R = min(max(ref_lens[b], 0), max_ref), H = min(max(hyp_lens[b], 0), max_hyp);
  const int* ref = refs + (long long)b * ref_stride;
  const int* hyp = hyps + (long long)b * hyp_stride;
  unsigned char* dirs = dirs_all + (long long)b * (max_ref + 1) * (max_hyp + 1);   // [R+1][H+1], row stride H + 1
  const int4 r = edit_distance_dp(ref, R, hyp, H, dirs, s_diag, max_ref + 1);
  if (threadIdx.x == 0) {
    out4[4 * b + 0] = r.x;
    out4[4 * b + 1] = r.y;
    out4[4 * b + 2] = r.z;
    out4[4 * b + 3] = r.w;
  }
}

// Per-pair workspace of word_errors_kernel.  A sequence of n tokens has at most (n + 1) / 2 words.  Word CTA: the
// reference's words then the hypothesis's (start, end, hash, id), the word-identity table (a power of two, at least
// twice the words) and the backtrace of the word matrix.  Character CTA: both sequences without spaces and the
// backtrace of their matrix.
struct WordErrorsLayout {
  int max_words;           // (max_ref + 1) / 2 + (max_hyp + 1) / 2
  int table_cap;
  size_t off_start, off_end, off_hash, off_id, off_table, off_wdirs, off_cref, off_chyp, off_cdirs, pair_bytes;
};

__host__ __device__ inline size_t we_align(size_t x) { return (x + 15) / 16 * 16; }

__host__ __device__ inline WordErrorsLayout word_errors_layout(int max_ref, int max_hyp) {
  WordErrorsLayout l;
  const int wr = (max_ref + 1) / 2, wh = (max_hyp + 1) / 2;
  l.max_words = wr + wh;
  int cap = 1;
  while (cap < 2 * l.max_words) cap <<= 1;
  l.table_cap = cap;
  size_t off = 0;
  l.off_start = off; off += we_align((size_t)l.max_words * sizeof(int));
  l.off_end = off;   off += we_align((size_t)l.max_words * sizeof(int));
  l.off_hash = off;  off += we_align((size_t)l.max_words * sizeof(unsigned long long));
  l.off_id = off;    off += we_align((size_t)l.max_words * sizeof(int));
  l.off_table = off; off += we_align((size_t)cap * sizeof(int));
  l.off_wdirs = off; off += we_align((size_t)(wr + 1) * (size_t)(wh + 1));
  l.off_cref = off;  off += we_align((size_t)max_ref * sizeof(int));
  l.off_chyp = off;  off += we_align((size_t)max_hyp * sizeof(int));
  l.off_cdirs = off; off += we_align((size_t)(max_ref + 1) * (size_t)(max_hyp + 1));
  l.pair_bytes = off;
  return l;
}

// Exclusive prefix sum of `flag` over the CTA's threads, offset by `carry`, which every thread then advances by the
// sum of all flags.  Called by every thread; s_warp holds kEdThreads / 32 ints.
__device__ __forceinline__ int cta_exclusive_scan(int flag, int* s_warp, int& carry) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int x = flag;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) s_warp[warp] = x;
  __syncthreads();
  int before = carry, total = 0;
#pragma unroll
  for (int w = 0; w < kEdThreads / 32; ++w) {
    const int v = s_warp[w];
    before += w < warp ? v : 0;
    total += v;
  }
  __syncthreads();                                     // s_warp is rewritten by the next call
  carry += total;
  return before + x - flag;
}

// Words of seq[0, n) (maximal runs of tokens other than `space`) as half-open [start, end) at start[base ..] and
// end[base ..]; returns their number (in every thread).
__device__ int split_words(const int* __restrict__ seq, int n, int space, int* start, int* end, int base, int* s_warp) {
  int count = 0;
  for (int p0 = 0; p0 < n; p0 += kEdThreads) {
    const int p = p0 + threadIdx.x;
    const bool in = p < n && seq[p] != space;
    const int is_first = in && (p == 0 || seq[p - 1] == space);
    const bool is_last = in && (p == n - 1 || seq[p + 1] == space);
    const int w = cta_exclusive_scan(is_first, s_warp, count) + is_first - 1;   // index of the word holding p
    if (is_first) start[base + w] = p;
    if (is_last) end[base + w] = p + 1;
  }
  return count;
}

// seq[0, n) without `space` at out[0 ..]; returns the length (in every thread).
__device__ int drop_spaces(const int* __restrict__ seq, int n, int space, int* out, int* s_warp) {
  int count = 0;
  for (int p0 = 0; p0 < n; p0 += kEdThreads) {
    const int p = p0 + threadIdx.x;
    const int keep = p < n && seq[p] != space;
    const int q = cta_exclusive_scan(keep, s_warp, count);
    if (keep) out[q] = seq[p];
  }
  return count;
}

__device__ __forceinline__ unsigned long long mix64(unsigned long long h) {   // splitmix64 finaliser
  h ^= h >> 30; h *= 0xbf58476d1ce4e5b9ULL;
  h ^= h >> 27; h *= 0x94d049bb133111ebULL;
  return h ^ (h >> 31);
}

// Grid (B, 2).  CTA (b, 0): split both sequences into words, give every word an id (equal ids <=> equal words) and
// run the edit distance over the ids.  CTA (b, 1): the edit distance of both sequences without spaces.  Everything
// a CTA reads from the workspace it wrote itself in this launch (plain loads after a __syncthreads()); the
// workspace's contents on entry do not matter.
__global__ void __launch_bounds__(kEdThreads) word_errors_kernel(
    const int* __restrict__ refs, int ref_stride, const int* __restrict__ ref_lens,
    const int* __restrict__ hyps, int hyp_stride, const int* __restrict__ hyp_lens,
    int max_ref, int max_hyp, int space, int* __restrict__ word4, int* __restrict__ char4,
    int* __restrict__ ref_counts, unsigned char* workspace) {
  extern __shared__ int s_diag[];                     // three anti-diagonals: [3][max_ref + 1]
  __shared__ int s_warp[kEdThreads / 32];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int R = min(max(ref_lens[b], 0), max_ref), H = min(max(hyp_lens[b], 0), max_hyp);
  const int* ref = refs + (long long)b * ref_stride;
  const int* hyp = hyps + (long long)b * hyp_stride;
  const WordErrorsLayout l = word_errors_layout(max_ref, max_hyp);
  unsigned char* ws = workspace + (long long)b * l.pair_bytes;

  if (blockIdx.y == 1) {
    int* cref = reinterpret_cast<int*>(ws + l.off_cref);
    int* chyp = reinterpret_cast<int*>(ws + l.off_chyp);
    const int Rc = drop_spaces(ref, R, space, cref, s_warp);
    const int Hc = drop_spaces(hyp, H, space, chyp, s_warp);
    __syncthreads();
    const int4 r = edit_distance_dp(cref, Rc, chyp, Hc, ws + l.off_cdirs, s_diag, max_ref + 1);
    if (tid == 0) {
      char4[4 * b + 0] = r.x; char4[4 * b + 1] = r.y; char4[4 * b + 2] = r.z; char4[4 * b + 3] = r.w;
      ref_counts[2 * b + 1] = Rc;
    }
    return;
  }

  int* start = reinterpret_cast<int*>(ws + l.off_start);
  int* end = reinterpret_cast<int*>(ws + l.off_end);
  unsigned long long* hash = reinterpret_cast<unsigned long long*>(ws + l.off_hash);
  int* id = reinterpret_cast<int*>(ws + l.off_id);
  int* table = reinterpret_cast<int*>(ws + l.off_table);
  for (int k = tid; k < l.table_cap; k += kEdThreads) table[k] = -1;
  const int Rw = split_words(ref, R, space, start, end, 0, s_warp);
  const int Hw = split_words(hyp, H, space, start, end, Rw, s_warp);
  const int nw = Rw + Hw;
  __syncthreads();
  // a word's tokens: words [0, Rw) are in ref, the others in hyp
  for (int w = tid; w < nw; w += kEdThreads) {
    const int* seq = w < Rw ? ref : hyp;
    const int s = start[w], e = end[w];
    unsigned long long h = 0x9e3779b97f4a7c15ULL ^ (unsigned long long)(e - s);
    for (int p = s; p < e; ++p) h = (h ^ (unsigned)seq[p]) * 0x100000001b3ULL;
    hash[w] = mix64(h);
  }
  __syncthreads();
  // Word identity: the first of a set of equal words to claim a slot on their common probe sequence is their id.
  // A probe compares tokens whenever the hashes agree, so a hash collision costs a comparison, never a wrong id.
  const unsigned mask = (unsigned)(l.table_cap - 1);
  for (int w = tid; w < nw; w += kEdThreads) {
    const int* seq = w < Rw ? ref : hyp;
    const int s = start[w], len = end[w] - s;
    const unsigned long long h = hash[w];
    for (unsigned slot = (unsigned)h & mask;; slot = (slot + 1) & mask) {
      const int other = atomicCAS(table + slot, -1, w);
      if (other < 0) { id[w] = w; break; }
      if (hash[other] != h) continue;
      const int* oseq = other < Rw ? ref : hyp;
      const int os = start[other];
      bool same = end[other] - os == len;
      for (int p = 0; same && p < len; ++p) same = oseq[os + p] == seq[s + p];
      if (same) { id[w] = other; break; }
    }
  }
  __syncthreads();
  const int4 r = edit_distance_dp(id, Rw, id + Rw, Hw, ws + l.off_wdirs, s_diag, max_ref + 1);
  if (tid == 0) {
    word4[4 * b + 0] = r.x; word4[4 * b + 1] = r.y; word4[4 * b + 2] = r.z; word4[4 * b + 3] = r.w;
    ref_counts[2 * b + 0] = Rw;
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

size_t word_errors_workspace_bytes(int B, int max_ref, int max_hyp) {
  return (size_t)B * word_errors_layout(max_ref, max_hyp).pair_bytes;
}

cudaError_t launch_word_errors(const int* refs, int ref_stride, const int* ref_lens, const int* hyps, int hyp_stride,
                               const int* hyp_lens, int B, int max_ref, int max_hyp, int space, int* word4, int* char4,
                               int* ref_counts, void* workspace, cudaStream_t stream) {
  if (B == 0) return cudaSuccess;
  const size_t smem = (size_t)3 * (max_ref + 1) * sizeof(int);
  if (smem > 200 * 1024) return cudaErrorInvalidConfiguration;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(word_errors_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  word_errors_kernel<<<dim3(B, 2), kEdThreads, smem, stream>>>(refs, ref_stride, ref_lens, hyps, hyp_stride, hyp_lens,
                                                               max_ref, max_hyp, space, word4, char4, ref_counts,
                                                               reinterpret_cast<unsigned char*>(workspace));
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
