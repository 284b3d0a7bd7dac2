// Safe lattice: fp64 log-space alpha/beta recursion, one CTA per utterance.
//
// This is the robust path of K2.  It is used (a) for utterances whose softmax rows contain
// probabilities below 2^-100 (FLAG_EXTREME_ROW), (b) when the block-exponent fast path reports a
// loss of range (FLAG_PRECISION_LOST), and (c) for label sequences longer than the fast path's
// lattice window.  It follows SURVEY Appendix A literally: alpha over all frames (stored to the
// scratch as doubles), log-likelihood from the last frame, then beta fused with the occupancy
// update of the gradient rows.  Emissions are log-probabilities acts[t,b,k] - lse[t,b] with the
// row log-sum-exp from K1, evaluated in double.  Logits of every element type are read through load_act
// (common.cuh), which widens them to fp32 as K1 does.
#pragma once

#include "lattice_common.cuh"

namespace b200ctc {

__device__ __forceinline__ double log_sum_exp3(double a, double b, double c) {
  const double m = fmax(a, fmax(b, c));
  if (m == -INFINITY) return -INFINITY;
  return m + log(exp(a - m) + exp(b - m) + exp(c - m));
}

struct SafeSmem {
  double* a0;     // [S] lattice frontier, double buffered
  double* a1;     // [S]
  float* post;    // [S] posteriors of the current frame
  int* lab;       // [L]
  SymbolIndex ix;
  double* bcast;  // [2]
};

__host__ __device__ inline size_t safe_smem_bytes(int L) {
  const size_t S = 2 * (size_t)L + 1;
  size_t bytes = 2 * S * sizeof(double) + 2 * sizeof(double);
  bytes += S * sizeof(float);
  bytes += (size_t)(4 * L + 8) * sizeof(int);
  return bytes + 64;
}

__device__ __forceinline__ SafeSmem carve_safe_smem(unsigned char* base, int L) {
  const int S = 2 * L + 1;
  SafeSmem s;
  double* d = reinterpret_cast<double*>(base);
  s.bcast = d;
  s.a0 = d + 2;
  s.a1 = s.a0 + S;
  s.post = reinterpret_cast<float*>(s.a1 + S);
  int* ip = reinterpret_cast<int*>(s.post + S);
  s.lab = ip;
  s.ix.sorted = s.lab + L;
  s.ix.seg_start = s.ix.sorted + L;
  s.ix.seg_sym = s.ix.seg_start + L + 1;
  s.ix.n_seg = s.ix.seg_sym + L + 1;
  return s;
}

// Whole-CTA routine.  `rows_dirty`: the gradient rows of this utterance no longer hold the plain
// softmax (the fast path already subtracted part of the occupancy) and must be rebuilt first.
__device__ void lattice_safe_utterance(const CallParams& p, int b, unsigned char* smem_base,
                                       bool rows_dirty) {
  const UttMeta m = p.meta[b];
  const int T = m.T, L = m.L, S = 2 * L + 1;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int V = p.V, blank = p.blank;
  SafeSmem sm = carve_safe_smem(smem_base, L);

  for (int i = tid; i < L; i += nt) sm.lab[i] = p.labels[m.lab_off + i];
  __syncthreads();
  build_symbol_index(sm.lab, L, V, sm.ix);

  const long long acts_b = (long long)b * p.as_b;   // element offset of the utterance's logits
  double* alpha = reinterpret_cast<double*>(p.scratch + m.scratch_off * kGroupBytes);
  const long long frame_stride = 4LL * m.J;  // doubles per frame in the scratch

  // Gradient rows in their final form minus the occupancy (s_y * y - c_ls; the plain softmax without
  // b200ctc_options): rebuilt when the fast path left them half-updated, and for rescaled small-vocabulary
  // calls, whose rows K1 leaves as the plain softmax for the fast lattice to read.
  const float ls = p.logit_scale;
  if ((rows_dirty || (p.rescale && !p.gathered)) && p.grads) {
    for (int t = 0; t < T; ++t) {
      const long long arow = acts_b + (long long)t * p.as_t;
      float* grow = p.grads + ((long long)t * p.B + b) * V;
      const float lse = p.lse[(long long)t * p.B + b];
      for (int v = tid; v < V; v += nt) grow[v] = fmaf(p.s_y, expf(load_act(p, arow + v) * ls - lse), -p.c_ls);
    }
    __threadfence();
    __syncthreads();
  }

  // ---- forward sweep -----------------------------------------------------------------------
  double* prev = sm.a0;
  double* cur = sm.a1;
  for (int s = tid; s < S; s += nt) prev[s] = (s == 0) ? 0.0 : -INFINITY;  // virtual frame -1
  __syncthreads();
  for (int t = 0; t < T; ++t) {
    const long long arow = acts_b + (long long)t * p.as_t;
    const double lse = (double)p.lse[(long long)t * p.B + b];
    for (int s = tid; s < S; s += nt) {
      const int sym = (s & 1) ? sm.lab[s >> 1] : blank;
      const bool skip = (s & 1) && s >= 3 && sm.lab[s >> 1] != sm.lab[(s >> 1) - 1];
      const double x0 = prev[s];
      const double x1 = (s >= 1) ? prev[s - 1] : -INFINITY;
      const double x2 = skip ? prev[s - 2] : -INFINITY;
      const double v = log_sum_exp3(x0, x1, x2) + ((double)(load_act(p, arow + sym) * ls) - lse);
      cur[s] = v;
      alpha[t * frame_stride + s] = v;
    }
    __syncthreads();
    double* tmp = prev; prev = cur; cur = tmp;
  }
  if (tid == 0) {
    double ll = prev[S - 1];
    if (S > 1) ll = log_sum_exp3(ll, prev[S - 2], -INFINITY);
    sm.bcast[0] = ll;
    p.costs[b] = (float)(-ll);  // -(-inf) = +inf when no alignment has non-zero probability
  }
  __syncthreads();
  const double ll = sm.bcast[0];
  if (!p.grads) return;
  if (!(ll > -INFINITY)) {
    // zero-probability target: same policy as an infeasible utterance (cost +inf, zero gradient)
    for (int t = 0; t < T; ++t) {
      float* grow = p.grads + ((long long)t * p.B + b) * V;
      for (int v = tid; v < V; v += nt) grow[v] = 0.f;
    }
    return;
  }

  // ---- backward sweep fused with the occupancy update ------------------------------------------
  __syncthreads();
  for (int s = tid; s < S; s += nt) prev[s] = (s == S - 1) ? 0.0 : -INFINITY;  // virtual frame T
  __syncthreads();
  const int n_seg = *sm.ix.n_seg;
  const int warp = tid >> 5, lane = tid & 31, n_warps = nt >> 5;
  for (int t = T - 1; t >= 0; --t) {
    const long long arow = acts_b + (long long)t * p.as_t;
    const double lse = (double)p.lse[(long long)t * p.B + b];
    for (int s = tid; s < S; s += nt) {
      const int sym = (s & 1) ? sm.lab[s >> 1] : blank;
      const bool skip = (s & 1) && (s + 2 < S) && sm.lab[s >> 1] != sm.lab[(s >> 1) + 1];
      const double x0 = prev[s];
      const double x1 = (s + 1 < S) ? prev[s + 1] : -INFINITY;
      const double x2 = skip ? prev[s + 2] : -INFINITY;
      const double lp = (double)(load_act(p, arow + sym) * ls) - lse;
      const double v = log_sum_exp3(x0, x1, x2) + lp;
      cur[s] = v;
      const double q = alpha[t * frame_stride + s] + v - lp - ll;
      const double pr = exp(q);
      sm.post[s] = (pr == pr && q > -INFINITY) ? (float)pr : 0.f;  // NaN (inf-inf) and -inf -> 0
    }
    __syncthreads();
    float* grow = p.grads + ((long long)t * p.B + b) * V;
    // blank: even states, one warp
    if (warp == 0) {
      float acc = 0.f;
      for (int s = 2 * lane; s < S; s += 64) acc += sm.post[s];
      acc = warp_sum(acc);
      if (lane == 0) atomicAdd(grow + blank, -p.s_occ * acc);
    }
    // label symbols: one thread per symbol segment (warps 1.. when there are several warps)
    const int first = (n_warps > 1) ? 32 : 0;
    for (int u = tid - first; u >= 0 && u < n_seg; u += nt - first) {
      float acc = 0.f;
      for (int k = sm.ix.seg_start[u]; k < sm.ix.seg_start[u + 1]; ++k)
        acc += sm.post[2 * sm.ix.sorted[k] + 1];
      atomicAdd(grow + sm.ix.seg_sym[u], -p.s_occ * acc);
    }
    __syncthreads();
    double* tmp = prev; prev = cur; cur = tmp;
  }
}

}  // namespace b200ctc
