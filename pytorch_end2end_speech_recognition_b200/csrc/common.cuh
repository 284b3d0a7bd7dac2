// Shared definitions for the B200 CTC engine (internal; the public boundary is include/b200ctc.h).
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "b200ctc.h"

namespace b200ctc {

// ---------------------------------------------------------------------------------------------
// Per-utterance plan, produced on the host (api.cu: plan_batch) and uploaded with the labels in
// one pinned->device copy.  "Lattice" vocabulary: S = 2L+1 blank-extended states, grouped four to
// a float4 ("group"); J = ceil(S/4) groups per frame.
// ---------------------------------------------------------------------------------------------
struct UttMeta {
  int T;            // frames of this utterance (act_lens[b])
  int L;            // labels of this utterance (label_lens[b])
  int lab_off;      // offset of its labels in the flat label vector
  int feasible;     // 1 iff L + repeats <= T (and T > 0 or L == 0)
  int J;            // ceil((2L+1)/4)
  int W;            // emission-row width in gathered mode: round_up(L+1, 4)
  long long scratch_off;  // offset of its alpha/beta scratch, in 32-byte units (one unit per group per frame)
  long long em_off;       // offset of its gathered emission rows, in floats (gathered mode only)
  int sym_off;            // offset of its distinct-symbol list in CallParams::sym_tab (gathered mode only)
  int pad_;
};

// Device views of one call, shared by all kernels.
struct CallParams {
  const void* acts;       // [T,B,V] logits of type acts_dtype, element (t,b,v) at acts[t*as_t + b*as_b + v]
  long long as_t, as_b;
  float* grads;           // [T,B,V] contiguous fp32 or nullptr (cost only): the caller's buffer, or the staging region of a
                          // bfloat16 / float16 call, which launch_narrow_grads rounds into the caller's buffer
  float* yrows;           // [T,B,V] where K1 leaves the softmax rows: == grads, or a workspace buffer in a cost-only call
  int T, B, V, blank;
  const UttMeta* meta;    // [B]
  const int* order;       // [B] utterances sorted by decreasing lattice work (longest first)
  const int* labels;      // flat labels (device copy)
  int* flags;             // [B] per-utterance flags written by the kernels
  int* done_counter;      // [1] utterances finished by the lattice kernel (zeroed with the plan upload)
  float* lse;             // [T*B] row log-sum-exp, natural log, time-major (t*B+b)
  float* em;              // gathered emissions (gathered mode) or nullptr
  unsigned char* scratch; // alpha/beta scratch
  float* costs;           // [B]
  float* loss_sum;        // [1] or nullptr
  int gathered;           // 1: lattice reads emissions from `em`, 0: from the softmax rows in `yrows`
  int acts_dtype;         // b200ctc_dtype_t of acts (fills what was padding: the offsets of the other fields stay)
  // Gathered mode leaves the per-symbol occupancy of frame t in the emission row em[t] it no longer needs
  // ([0] blank, [1 + u] distinct symbol u) instead of one RED per (frame, symbol) into gradient rows that have
  // long left the L2; apply_occupancy_kernel subtracts them afterwards, all frames in parallel.
  int* sym_tab;           // distinct symbols of every utterance (at meta[b].sym_off), written by the lattice prologue
  int* nseg;              // [B] their number
  int fast_l_cap;         // longest label sequence the block-exponent lattice takes (window count and shared-memory budget)
  int oth_depth;          // depth of the lattice's record ring, in chunks (2..4; prepare_lattice)
  // Fused call-site arithmetic (b200ctc_options; reference: models/pytorch_v3/ctc/ctc.py:306-307,323,329-337):
  //   z = logit_scale * acts;  grads = s_y * softmax(z) - s_occ * occupancy - c_ls   (rows t < T_b)
  //   loss_sum = loss_scale * sum_b [ ctc_w * cost_b + ls_w * sum_{t<T_b} (V * lse - sum_k z) ]
  float logit_scale, s_y, s_occ, c_ls, loss_scale, ctc_w, ls_w;
  int rescale;            // 1: s_y, s_occ, c_ls are not (1, 1, 0): every entry of a live gradient row is rewritten
  float* xe_rows;         // [T*B] V*lse - sum_k z of every live row (label smoothing only) or nullptr
  float* xe_costs;        // [B] their per-utterance sums (workspace, or the caller's ls_costs)
  // device-resident call (b200ctc_loss_and_grad_dev): the tables above are produced by plan_kernel from these
  const int* dev_label_lens;   // [B] or nullptr
  const int* dev_act_lens;     // [B]
  int label_stride;            // labels of utterance b start at labels + b * label_stride
  int max_label_len;           // bound on label_lens (sizes the per-utterance workspace regions)
};

// Programmatic dependent launch (sm_90+): K1 lets the lattice kernel start while it is still running; the
// lattice kernel does everything that needs no K1 output (labels, symbol index) and then waits for K1's
// completion and memory flush.  Both instructions are no-ops in a launch without the PDL attribute.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait_primary() { asm volatile("griddepcontrol.wait;" ::: "memory"); }


enum UttFlags : int {
  FLAG_EXTREME_ROW = 1,    // some softmax probability of the utterance is below 2^-100: use the safe lattice
  FLAG_PRECISION_LOST = 2, // the block-exponent lattice saw a live state lose range: redo with the safe lattice
  FLAG_INVALID_INPUT = 4,  // device-resident call: a label or a length of the utterance is out of range (cost NaN, zero gradient)
  FLAG_OCC_ROWS = 8        // gathered mode: the fast lattice left the utterance's occupancy in its emission rows
};

constexpr int kGroupBytes = 32;  // scratch bytes per (frame, group): the safe lattice stores 4 doubles

// scratch units (32 bytes) per frame: the safe lattice stores 4 doubles per group of four states,
// the fast lattice a little more than that for very short label sequences
__host__ __device__ inline int groups_of(int L) {
  const int j4 = (2 * L + 1 + 3) / 4, j8 = (2 * L + 1 + 7) / 8;
  // fast lattice: 32 bytes of mantissas per group of eight states + an int32 exponent row padded to 4 groups
  const int fast8 = (36 * j8 + 12 + 31) / 32;
  return j4 > fast8 ? j4 : fast8;
}
__host__ __device__ inline int em_width_of(int L) { return (L + 1 + 3) / 4 * 4; }

// Launch geometry of the lattice kernel for one call (lattice.cu: prepare_lattice).
struct LatticeCfg {
  int nwmax, l_cap, depth;   // lattice windows per sweep (1, 2, 4); longest label sequence of the fast lattice; record ring depth
  size_t smem;               // dynamic shared memory per CTA
  bool cluster;              // two CTAs per utterance (lattice_cluster_kernel)
};

// host launchers (each in its own .cu)
cudaError_t launch_softmax_rows(const CallParams& p, cudaStream_t stream);
cudaError_t prepare_lattice(CallParams& p, int max_L, LatticeCfg* cfg);   // also fills fast_l_cap and oth_depth; error when not even the safe lattice fits
cudaError_t launch_lattice(const CallParams& p, const LatticeCfg& cfg, cudaStream_t stream);
cudaError_t launch_apply_occupancy(const CallParams& p, cudaStream_t stream);
// dst[i] = src[i] rounded to nearest even in `dtype` (B200CTC_BFLOAT16 / B200CTC_FLOAT16), i < n
cudaError_t launch_narrow_grads(const float* src, void* dst, long long n, int dtype, cudaStream_t stream);
// out = grads * scale[0] (n_scale == 1) or grads[t,b,:] * scale[b] (n_scale == B), in fp32, rounded once to `dtype`
cudaError_t launch_scale_grads(const void* grads, void* out, int dtype, int T, int B, int V, const float* scale,
                               int n_scale, cudaStream_t stream);
cudaError_t launch_plan(const CallParams& p, UttMeta* meta, int* order, int* flags, cudaStream_t stream);
size_t edit_distance_workspace_bytes(int B, int max_ref, int max_hyp);
cudaError_t launch_edit_distance(const int* refs, int ref_stride, const int* ref_lens, const int* hyps, int hyp_stride,
                                 const int* hyp_lens, int B, int max_ref, int max_hyp, int* out4, void* workspace,
                                 cudaStream_t stream);
// the decoders and the posterior softmax read logits / log-probabilities of element type `dtype` (b200ctc_dtype_t)
cudaError_t launch_softmax_temperature(const void* logits, int dtype, long long stride_b, long long stride_t, int T, int V,
                                       int B, float inv_temperature, float* probs, cudaStream_t stream);
size_t beam_search_workspace_bytes(int B, int T, int V, int beam_width);
cudaError_t launch_beam_search(const void* log_probs, int dtype, long long stride_b, long long stride_t, const int* lens,
                               int T, int V, int B, int blank, int beam_width, int* out_tokens, int* out_lens,
                               float* out_scores, void* workspace, cudaStream_t stream);
cudaError_t launch_greedy(const void* logits, int dtype, long long stride_b, long long stride_t, const int* lens,
                          int T, int V, int B, int blank, int* out_tokens, int* out_lens, cudaStream_t stream);

// ---------------------------------------------------------------------------------------------
// small device helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// Logit element types: every kernel widens a logit to fp32 when it loads it and computes in fp32 from there on.
__device__ __forceinline__ float widen(float x) { return x; }
__device__ __forceinline__ float widen(__nv_bfloat16 x) { return __bfloat162float(x); }
__device__ __forceinline__ float widen(__half x) { return __half2float(x); }
__device__ __forceinline__ float2 widen2(__nv_bfloat162 x) { return __bfloat1622float2(x); }
__device__ __forceinline__ float2 widen2(__half2 x) { return __half22float2(x); }

// Logit (t,b,v) of any element type, for code that is not specialised on it (the safe lattice); `i` is the element
// offset t*as_t + b*as_b + v.
__device__ __forceinline__ float load_act(const CallParams& p, long long i) {
  if (p.acts_dtype == B200CTC_BFLOAT16) return widen(static_cast<const __nv_bfloat16*>(p.acts)[i]);
  if (p.acts_dtype == B200CTC_FLOAT16) return widen(static_cast<const __half*>(p.acts)[i]);
  return static_cast<const float*>(p.acts)[i];
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace b200ctc
