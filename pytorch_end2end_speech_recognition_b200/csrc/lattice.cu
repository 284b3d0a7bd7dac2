// K2: alpha/beta lattice recursion + posterior occupancy update of the gradient rows.
// K3 (fused into K2's last CTA): fixed-order sum of the per-utterance costs.
#include <cstdlib>

#include "common.cuh"
#include "lattice_fast.cuh"
#include "lattice_safe.cuh"

namespace b200ctc {

namespace {

// What every utterance ends with (the CTA that owns it; at least kTailThreads threads): the label-smoothing term of
// the utterance and, in the CTA that finishes last, the fixed-order sum of the costs (K3).  It reuses the dynamic
// shared memory for kTailThreads partial sums in double.
constexpr int kTailThreads = 128;   // the same summation order whatever the block size of the kernel variant
constexpr size_t kTailSmemBytes = kTailThreads * sizeof(double);
__device__ void utterance_tail(const CallParams& p, int b, const UttMeta& m, unsigned char* smem) {
  constexpr int NT = kTailThreads;
  // A CTA that never needed K1's output (infeasible or empty utterance) still must not let this kernel complete
  // before K1 does: whatever follows in the stream is ordered behind THIS kernel.  A no-op for everybody else.
  pdl_wait_primary();
  // Label smoothing (b200ctc_options): -sum_{t<T_b} sum_k log y[t,k] of this utterance from K1's per-row terms,
  // strided partial sums in double, then a tree: fixed order.
  double* part = reinterpret_cast<double*>(smem);
  if (p.xe_rows != nullptr) {
    __syncthreads();               // the utterance's own use of the shared memory is over
    if (threadIdx.x < NT) {
      double acc = 0.0;
      const int n_rows = m.feasible ? m.T : 0;     // K1 writes the term for live rows only
      for (int t = threadIdx.x; t < n_rows; t += NT) acc += (double)__ldcg(p.xe_rows + (long long)t * p.B + b);
      part[threadIdx.x] = acc;
    }
    __syncthreads();
    for (int o = NT / 2; o > 0; o >>= 1) {
      if ((int)threadIdx.x < o) part[threadIdx.x] += part[threadIdx.x + o];
      __syncthreads();
    }
    if (threadIdx.x == 0) p.xe_costs[b] = (float)part[0];
  }
  // K3, fused: the CTA that finishes last sums the per-utterance costs in a fixed order (NT strided
  // partial sums in double, then a tree), so the returned loss is bit-reproducible run to run.
  if (p.loss_sum == nullptr) return;
  __shared__ int s_last;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();                 // this CTA's cost is visible before the ticket is taken
    s_last = atomicAdd(p.done_counter, 1) == p.B - 1;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  if (threadIdx.x < NT) {
    double acc = 0.0;
    for (int i = threadIdx.x; i < p.B; i += NT) {
      double c = (double)__ldcg(p.costs + i) * (double)p.ctc_w;
      if (p.xe_rows != nullptr) c += (double)__ldcg(p.xe_costs + i) * (double)p.ls_w;
      acc += c;
    }
    part[threadIdx.x] = acc;
  }
  __syncthreads();
  for (int o = NT / 2; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) part[threadIdx.x] += part[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) *p.loss_sum = (float)(part[0] * (double)p.loss_scale);
}

// One CTA per utterance, longest lattice first (p.order): per side NWMAX lattice warps and kReducers
// reducer warps (lattice_fast.cuh).  The block-exponent fast path runs unless
// the utterance was flagged by K1 or is too long for the lattice window; when the fast path gives
// up (range lost, zero probability) the same CTA redoes the utterance with the fp64 safe path.
template <int NWMAX>
__global__ void __launch_bounds__(2 * (NWMAX + kReducers) * 32, 1) lattice_kernel(CallParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  pdl_launch_dependents();   // the plan kernel of the next device-resident call may run underneath this kernel (plan.cu)
  const int b = p.order[blockIdx.x];
  const UttMeta m = p.meta[b];
#ifdef B200CTC_TRACE
  if (threadIdx.x == 0 && blockIdx.x < 2048) {
    unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    g_cta_time[blockIdx.x * 2] = (long long)t;
  }
#endif
  if (!m.feasible) {  // K1 already zero-filled its gradient rows
    if (threadIdx.x == 0) p.costs[b] = (p.flags[b] & FLAG_INVALID_INPUT) ? NAN : INFINITY;
  } else if (m.T == 0) {  // empty utterance with an empty target: probability one
    if (threadIdx.x == 0) p.costs[b] = 0.f;
  } else {
    bool use_safe = m.L > p.fast_l_cap;   // too long for the lattice windows or for the shared-memory budget
    bool dirty = false;
    if (!use_safe) {
      // prologue (no K1 output needed), then wait for K1, then the sweeps -- unless K1 flagged an extreme row
      int* abort_word = nullptr;
      lattice_fast_utterance<NWMAX>(p, b, smem, &abort_word);
      __syncthreads();
      const int why = *abort_word;
      use_safe = why != 0;
      if (!use_safe && p.gathered && p.grads != nullptr && threadIdx.x == 0)
        atomicOr(p.flags + b, FLAG_OCC_ROWS);        // the occupancy of every frame sits in the emission rows
      if (use_safe && why != kAbortExtremeRow) {
        dirty = p.grads != nullptr;  // part of the gradient rows may already have been rewritten
        if (threadIdx.x == 0) atomicOr(p.flags + b, FLAG_PRECISION_LOST);
        __threadfence();             // order this thread's row updates before the rows are rebuilt
        __syncthreads();
      }
    } else {
      pdl_wait_primary();
    }
    if (use_safe) lattice_safe_utterance(p, b, smem, dirty);
  }

#ifdef B200CTC_TRACE
  __syncthreads();
  if (threadIdx.x == 0 && blockIdx.x < 2048) {
    unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    g_cta_time[blockIdx.x * 2 + 1] = (long long)t;
  }
#endif
  utterance_tail(p, b, m, smem);
}

// The thread-block-cluster variant: TWO CTAs per utterance, the forward sweep on one SM and the backward sweep on
// another (NWMAX lattice warps + kReducers fetching and kReducers reducing helper warps each), for mini-batches that leave at least half of the
// SMs idle.  The sides meet once, at the midpoint (a cluster barrier: everything phase 1 stored is visible to the
// other SM afterwards), and compare their abort words through distributed shared memory at the end; the CTA of
// rank 0 owns the utterance-level duties (safe lattice, flags, the tail).
template <int NWMAX>
__global__ void __launch_bounds__(cluster_block_warps<NWMAX>() * 32, 1) lattice_cluster_kernel(CallParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  pdl_launch_dependents();
  const unsigned rank = cluster_ctarank();
  const int b = p.order[blockIdx.x >> 1];
  const UttMeta m = p.meta[b];
  const bool owner = rank == 0;
  if (!m.feasible) {
    if (owner && threadIdx.x == 0) p.costs[b] = (p.flags[b] & FLAG_INVALID_INPUT) ? NAN : INFINITY;
  } else if (m.T == 0) {
    if (owner && threadIdx.x == 0) p.costs[b] = 0.f;
  } else {
    bool use_safe = m.L > p.fast_l_cap;
    bool dirty = false;
    if (!use_safe) {
      int* abort_word = nullptr;
      lattice_fast_utterance<NWMAX, true>(p, b, smem, &abort_word);
      __syncthreads();
      cluster_sync_all();                                   // both sweeps are over, both abort words final
      const int why = *abort_word | ld_peer_s32(abort_word, rank ^ 1u);
      cluster_sync_all();                                   // neither CTA reuses its shared memory before the peer has read it
      use_safe = why != 0;
      if (owner) {
        if (!use_safe && p.gathered && p.grads != nullptr && threadIdx.x == 0) atomicOr(p.flags + b, FLAG_OCC_ROWS);
        if (use_safe && why != kAbortExtremeRow) {
          dirty = p.grads != nullptr;
          if (threadIdx.x == 0) atomicOr(p.flags + b, FLAG_PRECISION_LOST);
          __threadfence();
          __syncthreads();
        }
      }
    } else {
      pdl_wait_primary();
    }
    if (use_safe && owner) lattice_safe_utterance(p, b, smem, dirty);
  }
  if (!owner) {
    pdl_wait_primary();
    return;
  }
  utterance_tail(p, b, m, smem);
}

constexpr size_t kSmemBudget = 227 * 1024 - 6 * 1024;   // dynamic shared memory: 227 KB per CTA minus the kernel's static arrays (4.4 KB)

// Two CTAs per utterance pay when every CTA gets an SM of its own: 2 * B <= number of SMs (B200CTC_CLUSTER=0 / 1
// overrides the choice, for A/B measurements).
bool want_cluster(int B) {
  static int n_sm = 0;
  if (n_sm == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) n_sm = 1;
  }
  if (const char* e = std::getenv("B200CTC_CLUSTER")) return e[0] == '1';
  return 2 * B <= n_sm;
}
int round_nw(int nw) { return nw <= 1 ? 1 : (nw <= 2 ? 2 : 4); }

template <int NWMAX>
cudaError_t launch_lattice_t(const CallParams& p, const LatticeCfg& c, cudaStream_t stream) {
  void (*kernel)(CallParams) = c.cluster ? lattice_cluster_kernel<NWMAX> : lattice_kernel<NWMAX>;
  if (c.smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c.smem);
    if (e != cudaSuccess) return e;
  }
  // programmatic dependent launch: this kernel may start while K1 (the previous kernel in the stream) runs
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(c.cluster ? 2 * p.B : p.B));
  cfg.blockDim = dim3(c.cluster ? cluster_block_warps<NWMAX>() * 32 : 2 * (NWMAX + kReducers) * 32);
  cfg.dynamicSmemBytes = c.smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  attr[1].id = cudaLaunchAttributeClusterDimension;   // the cluster variant only: the two CTAs of an utterance
  attr[1].val.clusterDim.x = 2;
  attr[1].val.clusterDim.y = 1;
  attr[1].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = c.cluster ? 2 : 1;
  return cudaLaunchKernelEx(&cfg, kernel, p);
}

// Gathered mode, after the lattice: grads[t,b,symbol] -= s_occ * occupancy for the blank and every distinct symbol
// of the utterance, one warp per frame row.  Each (frame, symbol) entry is touched once: plain read-modify-write.
__global__ void __launch_bounds__(256) apply_occupancy_kernel(CallParams p) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= (long long)p.T * p.B) return;
  const int t = (int)(row / p.B), b = (int)(row - (long long)t * p.B);
  const UttMeta m = p.meta[b];
  if (t >= m.T || !(p.flags[b] & FLAG_OCC_ROWS)) return;
  const float* occ = p.em + m.em_off + (long long)t * m.W;
  float* g = p.grads + row * p.V;
  const int* syms = p.sym_tab + m.sym_off;
  const int n = p.nseg[b];
  // One reduction per (frame, symbol) entry, performed at the L2: the warp does not wait for the gradient entry to
  // come back before it can go on (a load-modify-store here ran at 8 % of the issue slots, bound by that round trip).
  // Each entry receives exactly one addend: deterministic.
  for (int u = lane; u < n; u += 32) {
    const int k = __ldg(syms + u);
    atomicAdd(g + k, -p.s_occ * __ldcg(occ + 1 + u));
  }
  if (lane == 0) atomicAdd(g + p.blank, -p.s_occ * __ldcg(occ));
}

}  // namespace

cudaError_t launch_apply_occupancy(const CallParams& p, cudaStream_t stream) {
  const long long rows = (long long)p.T * p.B;
  if (rows == 0) return cudaSuccess;
  apply_occupancy_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, stream>>>(p);
  return cudaGetLastError();
}

// Launch geometry for a call whose longest feasible label sequence is max_L: the number of lattice windows
// per sweep (template parameter NWMAX: 1, 2 or 4), the longest label sequence the block-exponent lattice
// takes (l_cap: it must fit NWMAX windows AND the shared-memory budget -- in gathered mode the emission-row
// ring grows with the label sequence, 256 * (L + 5) bytes per side), and the dynamic shared memory.
// Longer utterances are evaluated by the fp64 safe lattice in the same launch.
cudaError_t prepare_lattice(CallParams& p, int max_L, LatticeCfg* out) {
  const size_t safe = safe_smem_bytes(max_L) > kTailSmemBytes ? safe_smem_bytes(max_L) : kTailSmemBytes;
  if (safe > kSmemBudget) return cudaErrorInvalidConfiguration;   // not even the safe lattice holds this label sequence
  // The deepest record ring whose shared memory still holds the longest label sequence; when none does, the
  // shallowest (largest capacity) and the longer utterances take the safe lattice.
  int nwmax = 1, l_cap = 0, depth = 2;
  for (int D = kOthDepthMax; D >= 2; --D) {
    nwmax = round_nw(fast_warps_needed(max_L));
    l_cap = max_L;
    // shared memory is monotonic in L (and in the row width, which follows L in gathered mode)
    while (l_cap > 0 && (fast_warps_needed(l_cap) > nwmax || fast_smem_bytes(p, nwmax, 2, l_cap, D) > kSmemBudget)) --l_cap;
    depth = D;
    if (l_cap >= max_L) break;
  }
  nwmax = round_nw(fast_warps_needed(l_cap));
  const size_t fast = fast_smem_bytes(p, nwmax, 2, l_cap, depth);
  out->nwmax = nwmax;
  out->depth = depth;
  out->l_cap = fast <= kSmemBudget ? l_cap : -1;   // -1: every utterance takes the safe lattice
  out->smem = (out->l_cap >= 0 && fast > safe) ? fast : safe;
  out->cluster = out->l_cap >= 0 && want_cluster(p.B);
  if (out->cluster) {
    // one side per CTA; at least 116 KB so that the two CTAs of a cluster cannot share an SM
    const size_t one = fast_smem_bytes(p, nwmax, 1, out->l_cap, depth);
    size_t sm = one > safe ? one : safe;
    out->smem = sm > (size_t)116 * 1024 ? sm : (size_t)116 * 1024;
  }
  p.fast_l_cap = out->l_cap;
  p.oth_depth = depth;
  return cudaSuccess;
}

cudaError_t launch_lattice(const CallParams& p, const LatticeCfg& c, cudaStream_t stream) {
  if (p.B == 0) return cudaSuccess;
  // eight lattice states per lane; one, two or four 256-state windows per sweep
  if (c.nwmax == 1) return launch_lattice_t<1>(p, c, stream);
  if (c.nwmax == 2) return launch_lattice_t<2>(p, c, stream);
  return launch_lattice_t<4>(p, c, stream);   // longer label sequences (L > 463) take the safe lattice
}

#ifdef B200CTC_TRACE
// developer hook: copies the timeline of CTA 0 of the last lattice launch and clears it
extern "C" __attribute__((visibility("default"))) int b200ctc_debug_set_trace_cta(int cta) {
  return cudaMemcpyToSymbol(g_trace_cta, &cta, sizeof(int)) == cudaSuccess ? 0 : 2;
}
extern "C" __attribute__((visibility("default"))) int b200ctc_debug_read_cta_times(long long* host, int n) {
  if (cudaDeviceSynchronize() != cudaSuccess) return 2;
  return cudaMemcpyFromSymbol(host, g_cta_time, sizeof(long long) * 2 * n) == cudaSuccess ? 0 : 2;
}
extern "C" __attribute__((visibility("default"))) int b200ctc_debug_read_trace(long long* host, int* counts) {
  if (cudaDeviceSynchronize() != cudaSuccess) return 2;
  if (cudaMemcpyFromSymbol(host, g_trace, sizeof(long long) * 64 * kTraceCap) != cudaSuccess) return 2;
  if (cudaMemcpyFromSymbol(counts, g_trace_cnt, sizeof(int) * 64) != cudaSuccess) return 2;
  static int zeros[64];
  if (cudaMemcpyToSymbol(g_trace_cnt, zeros, sizeof(zeros)) != cudaSuccess) return 2;
  return 0;
}
#endif

}  // namespace b200ctc
