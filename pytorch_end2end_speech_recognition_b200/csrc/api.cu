// C-ABI entry points (include/b200ctc.h): argument validation, batch planning (on the host for the
// warp-ctc style call with host-resident labels, by plan_kernel for the device-resident call),
// workspace carving and kernel dispatch.  No exceptions leave this file.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <new>
#include <numeric>
#include <vector>

#include "common.cuh"
#include "ngram_lm.cuh"

namespace b200ctc {

namespace {

constexpr size_t kAlign = 256;
constexpr int kStagingSlots = 4;
constexpr int kGatherMinV = 129;  // V above this: the lattice reads gathered emission rows

inline size_t align_up(size_t x) { return (x + kAlign - 1) / kAlign * kAlign; }
// The caller's workspace may have any alignment: every `_workspace` query adds kAlign bytes to what the layout needs,
// and the call lays the layout out from the first kAlign boundary of the buffer.  nullptr when fewer than `need`
// bytes follow that boundary.
unsigned char* aligned_workspace(void* workspace, size_t workspace_bytes, size_t need) {
  const size_t lost = (kAlign - reinterpret_cast<uintptr_t>(workspace) % kAlign) % kAlign;
  if (workspace_bytes < lost || workspace_bytes - lost < need) return nullptr;
  return static_cast<unsigned char*>(workspace) + lost;
}
inline bool valid_dtype(int d) { return d == B200CTC_FLOAT32 || d == B200CTC_BFLOAT16 || d == B200CTC_FLOAT16; }

// The call's host-prepared tables (utterance metadata, launch order, flags, labels: ~160 KB for C3) are
// written into a pinned staging slot and copied to a device slot of the handle on the handle's own COPY
// STREAM, at call time -- not stream-ordered behind the caller's earlier kernels.  The kernels wait for the
// copy's event.  A copy enqueued on the compute stream is issued to the copy engines only when that stream
// reaches it, i.e. after the application has already queued its prefetch of the next mini-batch of logits
// (bench.py's e2e leg, any data loader), and then waits behind 12 MB of it: +0.2 ms per call measured on
// B200 (tools/e2e_timeline.py).  Issued at call time it travels while the previous call's kernels run.
struct WorkspaceLayout {
  size_t blob_bytes;   // meta + order + flags + labels
  size_t off_meta, off_order, off_flags, off_labels;
  size_t off_lse, off_xe_rows, off_xe_costs, off_symtab, off_nseg, off_em, off_scratch;
  size_t off_staging;  // fp32 [T,B,V] gradient rows of a bfloat16 / float16 call (empty otherwise)
  size_t total;
};

struct BatchTotals {
  long long sum_labels = 0;
  long long em_floats = 0;       // sum_b T_b * W_b
  long long scratch_units = 0;   // sum_b (T_b + 1) * J_b
};

int totals_from_lens(const int* label_lens, const int* act_lens, int T, int B, BatchTotals* out) {
  BatchTotals t;
  for (int b = 0; b < B; ++b) {
    const int L = label_lens[b], Tb = act_lens[b];
    if (L < 0 || Tb < 0 || Tb > T) return B200CTC_STATUS_INVALID_VALUE;
    t.sum_labels += L;
    t.em_floats += (long long)Tb * em_width_of(L);
    t.scratch_units += (long long)(Tb + 1) * groups_of(L);   // + one dump frame block
  }
  *out = t;
  return B200CTC_STATUS_SUCCESS;
}

// Worst case of the same totals when only the shape is known (device-resident lengths).
BatchTotals totals_from_bound(int T, int B, int max_label_len) {
  BatchTotals t;
  t.sum_labels = 0;                                            // the caller's label tensor is read in place
  t.em_floats = (long long)B * T * em_width_of(max_label_len);
  t.scratch_units = (long long)B * (T + 1) * groups_of(max_label_len);
  return t;
}

// `tables_in_workspace`: the device-resident call keeps meta/order/flags in the workspace (plan_kernel writes
// them); the host call keeps them, with the labels, in the handle's staging slots.
// Small vocabularies never run the lattice in gathered mode: the `em` region then holds the softmax rows of a
// cost-only call (no gradient buffer to leave them in).  `staged`: a bfloat16 / float16 call with a gradient, whose
// kernels write fp32 rows into the staging region at the end; fp32 calls do not have it.
WorkspaceLayout make_layout(const BatchTotals& t, int T, int B, int V, long long symtab_ints, bool staged = false) {
  WorkspaceLayout w;
  size_t off = 0;
  w.off_meta = off;   off += align_up((size_t)B * sizeof(UttMeta));
  w.off_order = off;  off += align_up((size_t)B * sizeof(int));
  w.off_flags = off;  off += align_up((size_t)(B + 1) * sizeof(int));   // + the finished-utterance counter
  w.off_labels = off; off += align_up((size_t)t.sum_labels * sizeof(int));
  w.blob_bytes = off;
  w.off_lse = off;    off += align_up((size_t)T * B * sizeof(float));
  w.off_xe_rows = off; off += align_up((size_t)T * B * sizeof(float));   // label smoothing: per-row cross-entropy terms
  w.off_xe_costs = off; off += align_up((size_t)B * sizeof(float));
  w.off_symtab = off; off += align_up((size_t)(V >= kGatherMinV ? symtab_ints : 0) * sizeof(int));
  w.off_nseg = off;   off += align_up((size_t)B * sizeof(int));
  const size_t em_floats = V >= kGatherMinV ? (size_t)t.em_floats : (size_t)T * B * V;
  w.off_em = off;     off += align_up(em_floats * sizeof(float));
  w.off_scratch = off; off += align_up((size_t)t.scratch_units * kGroupBytes);
  w.off_staging = off; off += staged ? align_up((size_t)T * B * V * sizeof(float)) : 0;
  w.total = off;
  return w;
}

}  // namespace

}  // namespace b200ctc

using namespace b200ctc;

struct b200ctc_handle {
  int device;
  std::mutex mu;                    // calls on one handle are serialised
  struct Slot {
    void* host = nullptr;           // pinned staging buffer the host fills
    void* dev = nullptr;            // its device copy, read by the kernels
    size_t capacity = 0;
    cudaEvent_t copied = nullptr;   // the tables have reached `dev` (copy stream)
    cudaEvent_t done = nullptr;     // the call's kernels have finished: host and dev are reusable
    bool in_flight = false;
    // what the tables in this slot were planned for (plan cache: a call with the same lengths and labels on
    // the same stream reuses them: no planning, no host-to-device copy)
    bool planned = false;
    int T = 0, V = 0, B = 0, blank = 0, max_L = 0;
    long long sum_labels = 0;
    cudaStream_t stream = nullptr;
  } slots[kStagingSlots];
  cudaStream_t copy_stream = nullptr;
  int next_slot = 0;
  int last_slot = -1;
  bool profiling = false;
  cudaEvent_t prof[4] = {nullptr, nullptr, nullptr, nullptr};  // before softmax / lattice / cost sum, after
  bool prof_valid = false;
  const int* last_flags = nullptr;  // device pointer to the last call's flags
  int last_B = 0;
  long long plan_hits = 0, plan_misses = 0;
};

namespace {

int check_device(const b200ctc_handle* h) {
  int cur = -1;
  if (cudaGetDevice(&cur) != cudaSuccess) {
    cudaGetLastError();
    return B200CTC_STATUS_EXECUTION_FAILED;
  }
  return cur == h->device ? B200CTC_STATUS_SUCCESS : B200CTC_STATUS_INVALID_VALUE;
}

int status_of(cudaError_t e) {
  if (e == cudaSuccess) return B200CTC_STATUS_SUCCESS;
  std::fprintf(stderr, "b200ctc: CUDA error: %s\n", cudaGetErrorString(e));
  cudaGetLastError();
  return (e == cudaErrorInvalidValue || e == cudaErrorInvalidConfiguration) ? B200CTC_STATUS_UNSUPPORTED
                                                                            : B200CTC_STATUS_EXECUTION_FAILED;
}

// K1 -> K2 (whose last CTA also writes loss_sum) on `stream`, bracketed by the profiling events.  `narrow_to`: the
// caller's gradient buffer of a bfloat16 / float16 call, into which the fp32 rows at p.grads are rounded last.
int run_kernels(b200ctc_handle* h, CallParams& p, int max_L, cudaStream_t stream, void* narrow_to = nullptr) {
  h->last_flags = p.flags;
  h->last_B = p.B;
  LatticeCfg lattice;
  cudaError_t e = prepare_lattice(p, max_L, &lattice);
  if (e != cudaSuccess) return status_of(e);
  const bool prof = h->profiling;
  if (prof) cudaEventRecord(h->prof[0], stream);
  e = launch_softmax_rows(p, stream);
  if (prof) cudaEventRecord(h->prof[1], stream);
  if (e == cudaSuccess) e = launch_lattice(p, lattice, stream);
  if (prof) cudaEventRecord(h->prof[2], stream);
  if (e == cudaSuccess && p.gathered && p.grads) e = launch_apply_occupancy(p, stream);
  if (e == cudaSuccess && narrow_to) e = launch_narrow_grads(p.grads, narrow_to, (long long)p.T * p.B * p.V, p.acts_dtype, stream);
  if (prof) {
    cudaEventRecord(h->prof[3], stream);
    h->prof_valid = true;
  }
  return status_of(e);
}

void fill_common(CallParams& p, const void* acts, int64_t as_t, int64_t as_b, float* grads, int T, int V, int B,
                 int blank, float* costs, float* loss_sum, unsigned char* ws, const WorkspaceLayout& lay,
                 const b200ctc_options* o = nullptr, float* ls_costs = nullptr) {
  // fused call-site arithmetic (include/b200ctc.h, b200ctc_options); the defaults leave every result bit-identical
  const float logit_scale = o ? o->logit_scale : 1.f, lsp = o ? o->label_smoothing : 0.f;
  const float grad_scale = o ? o->grad_scale : 1.f;
  p.logit_scale = logit_scale;
  p.s_y = grad_scale;
  p.s_occ = grad_scale * (1.f - lsp);
  p.c_ls = grad_scale * lsp / (float)V;
  p.loss_scale = o ? o->loss_scale : 1.f;
  p.ctc_w = 1.f - lsp;
  p.ls_w = lsp / (float)V;
  p.rescale = (p.s_y != 1.f || p.s_occ != 1.f || p.c_ls != 0.f) ? 1 : 0;
  p.xe_rows = lsp != 0.f ? reinterpret_cast<float*>(ws + lay.off_xe_rows) : nullptr;
  p.xe_costs = ls_costs ? ls_costs : reinterpret_cast<float*>(ws + lay.off_xe_costs);
  p.sym_tab = reinterpret_cast<int*>(ws + lay.off_symtab);
  p.nseg = reinterpret_cast<int*>(ws + lay.off_nseg);
  p.acts = acts;
  p.as_t = as_t;
  p.as_b = as_b;
  p.grads = grads;
  p.T = T; p.B = B; p.V = V; p.blank = blank;
  p.lse = reinterpret_cast<float*>(ws + lay.off_lse);
  p.em = reinterpret_cast<float*>(ws + lay.off_em);
  p.scratch = ws + lay.off_scratch;
  p.costs = costs;
  p.loss_sum = loss_sum;
  p.gathered = V >= kGatherMinV ? 1 : 0;
  p.yrows = p.gathered ? grads : (grads ? grads : p.em);   // cost only, small vocabulary: the rows go to the workspace
  p.fast_l_cap = 0;
  p.oth_depth = 2;
  p.dev_label_lens = nullptr;
  p.dev_act_lens = nullptr;
  p.label_stride = 0;
  p.max_label_len = 0;
  p.acts_dtype = B200CTC_FLOAT32;
}

}  // namespace

extern "C" {

int b200ctc_version(void) { return B200CTC_VERSION; }

const char* b200ctc_status_string(int status) {
  switch (status) {
    case B200CTC_STATUS_SUCCESS: return "success";
    case B200CTC_STATUS_INVALID_VALUE: return "invalid value";
    case B200CTC_STATUS_EXECUTION_FAILED: return "CUDA execution failed";
    case B200CTC_STATUS_UNSUPPORTED: return "unsupported problem size";
    case B200CTC_STATUS_WORKSPACE_TOO_SMALL: return "workspace too small";
    default: return "unknown status";
  }
}

int b200ctc_create(b200ctc_handle** handle, int device) {
  if (!handle) return B200CTC_STATUS_INVALID_VALUE;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) {
    cudaGetLastError();
    return B200CTC_STATUS_EXECUTION_FAILED;  // no CPU fallback: a CUDA device is required
  }
  b200ctc_handle* h = new (std::nothrow) b200ctc_handle();
  if (!h) return B200CTC_STATUS_EXECUTION_FAILED;
  h->device = device;
  *handle = h;
  return B200CTC_STATUS_SUCCESS;
}

int b200ctc_destroy(b200ctc_handle* h) {
  if (!h) return B200CTC_STATUS_SUCCESS;
  for (auto& s : h->slots) {
    if (s.done) {
      if (s.in_flight) cudaEventSynchronize(s.done);
      cudaEventDestroy(s.done);
    }
    if (s.copied) cudaEventDestroy(s.copied);
    if (s.host) cudaFreeHost(s.host);
    if (s.dev) cudaFree(s.dev);
  }
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  for (auto& e : h->prof)
    if (e) cudaEventDestroy(e);
  delete h;
  return B200CTC_STATUS_SUCCESS;
}

int b200ctc_get_workspace_size(const int* label_lens, const int* act_lens, int T, int V, int B,
                               size_t* bytes) {
  if (!bytes || T < 0 || V < 1 || B < 0 || (B > 0 && (!label_lens || !act_lens)))
    return B200CTC_STATUS_INVALID_VALUE;
  BatchTotals t;
  int st = totals_from_lens(label_lens, act_lens, T, B, &t);
  if (st != B200CTC_STATUS_SUCCESS) return st;
  *bytes = make_layout(t, T, B, V, t.sum_labels).total + kAlign;
  return B200CTC_STATUS_SUCCESS;
}

int b200ctc_get_workspace_bound(int T, int V, int B, int max_label_len, size_t* bytes) {
  return b200ctc_get_workspace_bound_typed(T, V, B, max_label_len, B200CTC_FLOAT32, 1, bytes);
}

int b200ctc_get_workspace_bound_typed(int T, int V, int B, int max_label_len, int dtype, int need_grad, size_t* bytes) {
  if (!bytes || T < 0 || V < 1 || B < 0 || max_label_len < 0 || !valid_dtype(dtype)) return B200CTC_STATUS_INVALID_VALUE;
  const bool staged = dtype != B200CTC_FLOAT32 && need_grad;
  *bytes = make_layout(totals_from_bound(T, B, max_label_len), T, B, V, (long long)B * max_label_len, staged).total + kAlign;
  return B200CTC_STATUS_SUCCESS;
}

int b200ctc_loss_and_grad(b200ctc_handle* h, const float* acts, int64_t acts_stride_t,
                          int64_t acts_stride_b, float* grads, const int* flat_labels,
                          const int* label_lens, const int* act_lens, int T, int V, int B, int blank,
                          float* costs, float* loss_sum, void* workspace, size_t workspace_bytes,
                          void* stream_v) {
  if (!h || T < 0 || V < 1 || B < 0 || blank < 0 || blank >= V) return B200CTC_STATUS_INVALID_VALUE;
  std::lock_guard<std::mutex> lock(h->mu);
  int st = check_device(h);
  if (st != B200CTC_STATUS_SUCCESS) return st;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_v);
  if (B == 0) {
    if (loss_sum && cudaMemsetAsync(loss_sum, 0, sizeof(float), stream) != cudaSuccess)
      return B200CTC_STATUS_EXECUTION_FAILED;
    return B200CTC_STATUS_SUCCESS;
  }
  if (!label_lens || !act_lens || !costs || !workspace || (!acts && T > 0))
    return B200CTC_STATUS_INVALID_VALUE;

  // ---- plan on the host ----------------------------------------------------------------------
  BatchTotals tot;
  st = totals_from_lens(label_lens, act_lens, T, B, &tot);
  if (st != B200CTC_STATUS_SUCCESS) return st;
  if (tot.sum_labels > 0 && !flat_labels) return B200CTC_STATUS_INVALID_VALUE;
  if (tot.sum_labels > 0x7fffffffLL) return B200CTC_STATUS_UNSUPPORTED;
  if ((long long)B * V * 4 > 0x7fffffffLL) return B200CTC_STATUS_UNSUPPORTED;   // frame stride of the gradient rows in bytes (int32 in the lattice)
  const WorkspaceLayout lay = make_layout(tot, T, B, V, tot.sum_labels);
  unsigned char* ws = aligned_workspace(workspace, workspace_bytes, lay.total);
  if (!ws) return B200CTC_STATUS_WORKSPACE_TOO_SMALL;

  // ---- plan cache: the same lengths and labels as the previous call on this stream? ------------
  int max_L = 0;
  bool hit = false;
  if (h->last_slot >= 0) {
    b200ctc_handle::Slot& s = h->slots[h->last_slot];
    if (s.planned && s.T == T && s.V == V && s.B == B && s.blank == blank && s.stream == stream &&
        s.sum_labels == tot.sum_labels && s.capacity >= lay.blob_bytes) {
      const unsigned char* blob = reinterpret_cast<const unsigned char*>(s.host);
      const UttMeta* meta = reinterpret_cast<const UttMeta*>(blob + lay.off_meta);
      hit = true;
      for (int b = 0; b < B && hit; ++b) hit = meta[b].T == act_lens[b] && meta[b].L == label_lens[b];
      if (hit && tot.sum_labels > 0)
        hit = std::memcmp(blob + lay.off_labels, flat_labels, (size_t)tot.sum_labels * sizeof(int)) == 0;
      if (hit) max_L = s.max_L;
    }
  }

  b200ctc_handle::Slot* slotp;
  if (hit) {
    ++h->plan_hits;
    slotp = &h->slots[h->last_slot];
    // the tables are already on the device; only the per-call words (flags, finished counter) are reset,
    // stream-ordered behind the previous call that used them
    unsigned char* tab = reinterpret_cast<unsigned char*>(slotp->dev);
    if (cudaMemsetAsync(tab + lay.off_flags, 0, (size_t)(B + 1) * sizeof(int), stream) != cudaSuccess) {
      cudaGetLastError();
      return B200CTC_STATUS_EXECUTION_FAILED;
    }
  } else {
    ++h->plan_misses;
    // staging slot (pinned): reuse only after the call that last read it has completed
    h->last_slot = h->next_slot;
    slotp = &h->slots[h->next_slot];
    b200ctc_handle::Slot& slot = *slotp;
    h->next_slot = (h->next_slot + 1) % kStagingSlots;
    slot.planned = false;
    if (slot.in_flight) {
      if (cudaEventSynchronize(slot.done) != cudaSuccess) return B200CTC_STATUS_EXECUTION_FAILED;
      slot.in_flight = false;
    }
    if (slot.capacity < lay.blob_bytes) {                 // grows on demand (rare: synchronous allocation)
      if (slot.host) cudaFreeHost(slot.host);
      if (slot.dev) cudaFree(slot.dev);
      slot.host = slot.dev = nullptr;
      slot.capacity = 0;
      const size_t cap = std::max(lay.blob_bytes * 2, (size_t)1 << 16);
      if (cudaHostAlloc(&slot.host, cap, cudaHostAllocDefault) != cudaSuccess || cudaMalloc(&slot.dev, cap) != cudaSuccess) {
        cudaGetLastError();
        return B200CTC_STATUS_EXECUTION_FAILED;
      }
      slot.capacity = cap;
    }
    if ((!slot.done && cudaEventCreateWithFlags(&slot.done, cudaEventDisableTiming) != cudaSuccess) ||
        (!slot.copied && cudaEventCreateWithFlags(&slot.copied, cudaEventDisableTiming) != cudaSuccess) ||
        (!h->copy_stream && cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking) != cudaSuccess))
      return B200CTC_STATUS_EXECUTION_FAILED;

    unsigned char* blob = reinterpret_cast<unsigned char*>(slot.host);
    UttMeta* meta = reinterpret_cast<UttMeta*>(blob + lay.off_meta);
    int* order = reinterpret_cast<int*>(blob + lay.off_order);
    int* flags = reinterpret_cast<int*>(blob + lay.off_flags);
    int* labels = reinterpret_cast<int*>(blob + lay.off_labels);

    long long lab_off = 0, em_off = 0, scratch_off = 0;
    for (int b = 0; b < B; ++b) {
      const int L = label_lens[b], Tb = act_lens[b];
      const int* lab = flat_labels + lab_off;
      int repeats = 0;
      for (int i = 0; i < L; ++i) {
        const int s = lab[i];
        if (s < 0 || s >= V || s == blank) return B200CTC_STATUS_INVALID_VALUE;
        if (i > 0 && s == lab[i - 1]) ++repeats;
      }
      UttMeta& m = meta[b];
      m.T = Tb;
      m.L = L;
      m.lab_off = (int)lab_off;
      m.feasible = (L + repeats <= Tb) ? 1 : 0;
      m.J = groups_of(L);
      m.W = em_width_of(L);
      m.scratch_off = scratch_off;
      m.em_off = em_off;
      m.sym_off = (int)lab_off;
      m.pad_ = 0;
      lab_off += L;
      em_off += (long long)Tb * m.W;
      scratch_off += (long long)(Tb + 1) * m.J;
      if (m.feasible) max_L = std::max(max_L, L);
      order[b] = b;
      flags[b] = 0;
    }
    flags[B] = 0;   // finished-utterance counter (the last CTA of the lattice kernel sums the costs)
    if (tot.sum_labels > 0) std::memcpy(labels, flat_labels, (size_t)tot.sum_labels * sizeof(int));
    // longest lattice first: CTAs are dispatched in index order, so the tail of the launch is short
    std::stable_sort(order, order + B, [&](int x, int y) {
      const long long wx = (long long)meta[x].T * (2 * meta[x].L + 1) * meta[x].feasible;
      const long long wy = (long long)meta[y].T * (2 * meta[y].L + 1) * meta[y].feasible;
      return wx > wy;
    });

    // tables: host slot -> device slot on the handle's copy stream, now; the caller's stream waits for the event
    if (cudaMemcpyAsync(slot.dev, blob, lay.blob_bytes, cudaMemcpyHostToDevice, h->copy_stream) != cudaSuccess ||
        cudaEventRecord(slot.copied, h->copy_stream) != cudaSuccess ||
        cudaStreamWaitEvent(stream, slot.copied, 0) != cudaSuccess) {
      cudaGetLastError();
      return B200CTC_STATUS_EXECUTION_FAILED;
    }
    slot.planned = true;
    slot.T = T; slot.V = V; slot.B = B; slot.blank = blank; slot.max_L = max_L;
    slot.sum_labels = tot.sum_labels;
    slot.stream = stream;
  }

  b200ctc_handle::Slot& slot = *slotp;
  unsigned char* tab = reinterpret_cast<unsigned char*>(slot.dev);
  CallParams p;
  fill_common(p, acts, acts_stride_t, acts_stride_b, grads, T, V, B, blank, costs, loss_sum, ws, lay);
  p.meta = reinterpret_cast<const UttMeta*>(tab + lay.off_meta);
  p.order = reinterpret_cast<const int*>(tab + lay.off_order);
  p.flags = reinterpret_cast<int*>(tab + lay.off_flags);
  p.done_counter = p.flags + B;
  p.labels = reinterpret_cast<const int*>(tab + lay.off_labels);

  st = run_kernels(h, p, max_L, stream);
  // the slot (host and device side) is reusable once the kernels of this call have finished
  if (cudaEventRecord(slot.done, stream) == cudaSuccess) slot.in_flight = true;
  else if (st == B200CTC_STATUS_SUCCESS) st = B200CTC_STATUS_EXECUTION_FAILED;
  return st;
}

int b200ctc_loss_and_grad_dev(b200ctc_handle* h, const float* acts, int64_t acts_stride_t,
                              int64_t acts_stride_b, float* grads, const int* labels, int label_stride,
                              const int* label_lens, const int* act_lens, int T, int V, int B,
                              int max_label_len, int blank, const b200ctc_options* opts, float* costs,
                              float* loss_sum, float* ls_costs, void* workspace, size_t workspace_bytes,
                              void* stream_v) {
  return b200ctc_loss_and_grad_dev_typed(h, acts, acts_stride_t, acts_stride_b, B200CTC_FLOAT32, grads, labels,
                                         label_stride, label_lens, act_lens, T, V, B, max_label_len, blank, opts, costs,
                                         loss_sum, ls_costs, workspace, workspace_bytes, stream_v);
}

int b200ctc_loss_and_grad_dev_typed(b200ctc_handle* h, const void* acts, int64_t acts_stride_t, int64_t acts_stride_b,
                                    int acts_dtype, void* grads, const int* labels, int label_stride,
                                    const int* label_lens, const int* act_lens, int T, int V, int B, int max_label_len,
                                    int blank, const b200ctc_options* opts, float* costs, float* loss_sum,
                                    float* ls_costs, void* workspace, size_t workspace_bytes, void* stream_v) {
  if (!h || T < 0 || V < 1 || B < 0 || blank < 0 || blank >= V || max_label_len < 0 || label_stride < max_label_len ||
      !valid_dtype(acts_dtype))
    return B200CTC_STATUS_INVALID_VALUE;
  if (opts && (!(opts->logit_scale > 0.f) || !(opts->label_smoothing >= 0.f) || !(opts->label_smoothing < 1.f) ||
               opts->grad_scale != opts->grad_scale || opts->loss_scale != opts->loss_scale))
    return B200CTC_STATUS_INVALID_VALUE;
  std::lock_guard<std::mutex> lock(h->mu);
  int st = check_device(h);
  if (st != B200CTC_STATUS_SUCCESS) return st;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_v);
  if (B == 0) {
    if (loss_sum && cudaMemsetAsync(loss_sum, 0, sizeof(float), stream) != cudaSuccess)
      return B200CTC_STATUS_EXECUTION_FAILED;
    return B200CTC_STATUS_SUCCESS;
  }
  if (!label_lens || !act_lens || !costs || !workspace || (!acts && T > 0) || (!labels && max_label_len > 0))
    return B200CTC_STATUS_INVALID_VALUE;
  if ((long long)B * V * 4 > 0x7fffffffLL || (long long)B * label_stride > 0x7fffffffLL || B > 65536)
    return B200CTC_STATUS_UNSUPPORTED;
  const bool staged = acts_dtype != B200CTC_FLOAT32 && grads;
  const WorkspaceLayout lay =
      make_layout(totals_from_bound(T, B, max_label_len), T, B, V, (long long)B * max_label_len, staged);
  unsigned char* ws = aligned_workspace(workspace, workspace_bytes, lay.total);
  if (!ws) return B200CTC_STATUS_WORKSPACE_TOO_SMALL;

  CallParams p;
  // a bfloat16 / float16 gradient is formed in fp32 in the staging region and rounded into `grads` by the last kernel
  float* rows = staged ? reinterpret_cast<float*>(ws + lay.off_staging) : static_cast<float*>(grads);
  fill_common(p, acts, acts_stride_t, acts_stride_b, rows, T, V, B, blank, costs, loss_sum, ws, lay, opts, ls_costs);
  p.acts_dtype = acts_dtype;
  UttMeta* meta = reinterpret_cast<UttMeta*>(ws + lay.off_meta);
  int* order = reinterpret_cast<int*>(ws + lay.off_order);
  int* flags = reinterpret_cast<int*>(ws + lay.off_flags);
  p.meta = meta;
  p.order = order;
  p.flags = flags;
  p.done_counter = flags + B;
  p.labels = labels;
  p.dev_label_lens = label_lens;
  p.dev_act_lens = act_lens;
  p.label_stride = label_stride;
  p.max_label_len = max_label_len;

  // everything below is kernel launches on `stream`: the call can be captured into a CUDA graph
  cudaError_t e = launch_plan(p, meta, order, flags, stream);
  if (e != cudaSuccess) return status_of(e);
  return run_kernels(h, p, max_label_len, stream, staged ? grads : nullptr);
}

int b200ctc_scale_grads(const void* grads, void* out, int dtype, int T, int B, int V, const float* scale, int n_scale,
                        void* stream_v) {
  if (T < 0 || B < 0 || V < 1 || (dtype != B200CTC_BFLOAT16 && dtype != B200CTC_FLOAT16) ||
      (n_scale != 1 && n_scale != B))
    return B200CTC_STATUS_INVALID_VALUE;
  if ((long long)T * B == 0) return B200CTC_STATUS_SUCCESS;
  if (!grads || !out || !scale) return B200CTC_STATUS_INVALID_VALUE;
  return status_of(launch_scale_grads(grads, out, dtype, T, B, V, scale, n_scale, reinterpret_cast<cudaStream_t>(stream_v)));
}

int b200ctc_set_profiling(b200ctc_handle* h, int enable) {
  if (!h) return B200CTC_STATUS_INVALID_VALUE;
  std::lock_guard<std::mutex> lock(h->mu);
  if (enable) {
    for (auto& e : h->prof)
      if (!e && cudaEventCreate(&e) != cudaSuccess) return B200CTC_STATUS_EXECUTION_FAILED;
  }
  h->profiling = enable != 0;
  h->prof_valid = false;
  return B200CTC_STATUS_SUCCESS;
}

int b200ctc_get_last_kernel_ms(b200ctc_handle* h, float* ms3) {
  if (!h || !ms3 || !h->prof_valid) return B200CTC_STATUS_INVALID_VALUE;
  std::lock_guard<std::mutex> lock(h->mu);
  if (cudaEventSynchronize(h->prof[3]) != cudaSuccess) return B200CTC_STATUS_EXECUTION_FAILED;
  for (int i = 0; i < 3; ++i)
    if (cudaEventElapsedTime(ms3 + i, h->prof[i], h->prof[i + 1]) != cudaSuccess)
      return B200CTC_STATUS_EXECUTION_FAILED;
  return B200CTC_STATUS_SUCCESS;
}

int b200ctc_get_last_fallbacks(b200ctc_handle* h, int* counts3, void* stream_v) {
  if (!h || !counts3 || !h->last_flags) return B200CTC_STATUS_INVALID_VALUE;
  std::lock_guard<std::mutex> lock(h->mu);
  std::vector<int> host((size_t)h->last_B);
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_v);
  if (cudaMemcpyAsync(host.data(), h->last_flags, host.size() * sizeof(int), cudaMemcpyDeviceToHost, stream) != cudaSuccess ||
      cudaStreamSynchronize(stream) != cudaSuccess) {
    cudaGetLastError();
    return B200CTC_STATUS_EXECUTION_FAILED;
  }
  counts3[0] = counts3[1] = counts3[2] = 0;
  for (int f : host) {
    if (f & FLAG_EXTREME_ROW) ++counts3[0];
    if (f & FLAG_PRECISION_LOST) ++counts3[1];
    if (f & FLAG_INVALID_INPUT) ++counts3[2];
  }
  return B200CTC_STATUS_SUCCESS;
}

int b200ctc_get_plan_cache_stats(b200ctc_handle* h, long long* hits, long long* misses) {
  if (!h || !hits || !misses) return B200CTC_STATUS_INVALID_VALUE;
  std::lock_guard<std::mutex> lock(h->mu);
  *hits = h->plan_hits;
  *misses = h->plan_misses;
  return B200CTC_STATUS_SUCCESS;
}

int b200ctc_beam_search_workspace(int B, int T, int V, int beam_width, size_t* bytes) {
  if (!bytes || B < 0 || T < 0 || V < 1 || beam_width < 1 || beam_width > 64) return B200CTC_STATUS_INVALID_VALUE;
  *bytes = beam_search_workspace_bytes(B, T, V, beam_width) + kAlign;
  return B200CTC_STATUS_SUCCESS;
}

int b200ctc_beam_search(const float* log_probs, int64_t stride_b, int64_t stride_t, const int* lens, int T, int V,
                        int B, int blank, int beam_width, int* out_tokens, int* out_lens, float* out_scores,
                        void* workspace, size_t workspace_bytes, void* stream_v) {
  return b200ctc_beam_search_typed(log_probs, B200CTC_FLOAT32, stride_b, stride_t, lens, T, V, B, blank, beam_width,
                                   out_tokens, out_lens, out_scores, workspace, workspace_bytes, stream_v);
}

int b200ctc_beam_search_typed(const void* log_probs, int dtype, int64_t stride_b, int64_t stride_t, const int* lens, int T,
                              int V, int B, int blank, int beam_width, int* out_tokens, int* out_lens, float* out_scores,
                              void* workspace, size_t workspace_bytes, void* stream_v) {
  if (T < 0 || V < 1 || B < 0 || blank < 0 || blank >= V || beam_width < 1 || beam_width > 64 || !valid_dtype(dtype))
    return B200CTC_STATUS_INVALID_VALUE;
  if (B == 0) return B200CTC_STATUS_SUCCESS;
  if (!lens || !out_lens || !workspace || (T > 0 && (!log_probs || !out_tokens))) return B200CTC_STATUS_INVALID_VALUE;
  unsigned char* ws = aligned_workspace(workspace, workspace_bytes, beam_search_workspace_bytes(B, T, V, beam_width));
  if (!ws) return B200CTC_STATUS_WORKSPACE_TOO_SMALL;
  return status_of(launch_beam_search(log_probs, dtype, stride_b, stride_t, lens, T, V, B, blank, beam_width, out_tokens,
                                      out_lens, out_scores, ws, reinterpret_cast<cudaStream_t>(stream_v)));
}

int b200ctc_beam_search_lm_workspace(int B, int T, int V, int beam_width, size_t* bytes) {
  if (!bytes || B < 0 || T < 0 || V < 1 || beam_width < 1 || beam_width > 64) return B200CTC_STATUS_INVALID_VALUE;
  *bytes = beam_search_lm_workspace_bytes(B, T, V, beam_width, lm_n_words(V)) + kAlign;
  return B200CTC_STATUS_SUCCESS;
}

int b200ctc_beam_search_lm(const void* log_probs, int dtype, int64_t stride_b, int64_t stride_t, const int* lens, int T,
                           int V, int B, int blank, int beam_width, const b200ctc_ngram_lm* lm, double alpha, double beta,
                           int* out_tokens, int* out_lens, float* out_scores, void* workspace, size_t workspace_bytes,
                           void* stream_v) {
  if (T < 0 || V < 1 || B < 0 || blank < 0 || blank >= V || beam_width < 1 || beam_width > 64 || !valid_dtype(dtype) ||
      !std::isfinite(alpha) || !std::isfinite(beta))
    return B200CTC_STATUS_INVALID_VALUE;
  const int st = ngram_lm_check(lm, V, blank);
  if (st != B200CTC_STATUS_SUCCESS) return st;
  if (B == 0) return B200CTC_STATUS_SUCCESS;
  if (!lens || !out_lens || !workspace || (T > 0 && (!log_probs || !out_tokens))) return B200CTC_STATUS_INVALID_VALUE;
  if ((long long)T * beam_width >= 0x3fffffffLL) return B200CTC_STATUS_UNSUPPORTED;   // trie node ids and hash slots
  const LmView view = ngram_lm_view(lm);
  unsigned char* ws =
      aligned_workspace(workspace, workspace_bytes, beam_search_lm_workspace_bytes(B, T, V, beam_width, view.n_words));
  if (!ws) return B200CTC_STATUS_WORKSPACE_TOO_SMALL;
  return status_of(launch_beam_search_lm(log_probs, dtype, stride_b, stride_t, lens, T, V, B, blank, beam_width, view,
                                         alpha, beta, out_tokens, out_lens, out_scores, ws,
                                         reinterpret_cast<cudaStream_t>(stream_v)));
}

int b200ctc_edit_distance_workspace(int B, int max_ref, int max_hyp, size_t* bytes) {
  if (!bytes || B < 0 || max_ref < 0 || max_hyp < 0) return B200CTC_STATUS_INVALID_VALUE;
  *bytes = edit_distance_workspace_bytes(B, max_ref, max_hyp) + kAlign;
  return B200CTC_STATUS_SUCCESS;
}

int b200ctc_edit_distance(const int* refs, int ref_stride, const int* ref_lens, const int* hyps, int hyp_stride,
                          const int* hyp_lens, int B, int max_ref, int max_hyp, int* out4, void* workspace,
                          size_t workspace_bytes, void* stream_v) {
  if (B < 0 || max_ref < 0 || max_hyp < 0 || ref_stride < max_ref || hyp_stride < max_hyp) return B200CTC_STATUS_INVALID_VALUE;
  if (B == 0) return B200CTC_STATUS_SUCCESS;
  if (!ref_lens || !hyp_lens || !out4 || !workspace || (max_ref > 0 && !refs) || (max_hyp > 0 && !hyps))
    return B200CTC_STATUS_INVALID_VALUE;
  unsigned char* ws = aligned_workspace(workspace, workspace_bytes, edit_distance_workspace_bytes(B, max_ref, max_hyp));
  if (!ws) return B200CTC_STATUS_WORKSPACE_TOO_SMALL;
  return status_of(launch_edit_distance(refs, ref_stride, ref_lens, hyps, hyp_stride, hyp_lens, B, max_ref, max_hyp, out4,
                                        ws, reinterpret_cast<cudaStream_t>(stream_v)));
}

// sizes up to 2^29 keep the word count and table size of word_errors_layout in int
int b200ctc_word_errors_workspace(int B, int max_ref, int max_hyp, size_t* bytes) {
  if (!bytes || B < 0 || max_ref < 0 || max_hyp < 0) return B200CTC_STATUS_INVALID_VALUE;
  if (max_ref > (1 << 29) || max_hyp > (1 << 29)) return B200CTC_STATUS_UNSUPPORTED;
  const size_t pair = word_errors_workspace_bytes(1, max_ref, max_hyp);
  if (B > 0 && pair > (SIZE_MAX - kAlign) / (size_t)B) return B200CTC_STATUS_UNSUPPORTED;
  *bytes = (size_t)B * pair + kAlign;
  return B200CTC_STATUS_SUCCESS;
}

int b200ctc_word_errors(const int* refs, int ref_stride, const int* ref_lens, const int* hyps, int hyp_stride,
                        const int* hyp_lens, int B, int max_ref, int max_hyp, int space, int* word4, int* char4,
                        int* ref_counts, void* workspace, size_t workspace_bytes, void* stream_v) {
  if (B < 0 || max_ref < 0 || max_hyp < 0 || ref_stride < max_ref || hyp_stride < max_hyp) return B200CTC_STATUS_INVALID_VALUE;
  if (B == 0) return B200CTC_STATUS_SUCCESS;
  if (!ref_lens || !hyp_lens || !word4 || !char4 || !ref_counts || !workspace || (max_ref > 0 && !refs) ||
      (max_hyp > 0 && !hyps))
    return B200CTC_STATUS_INVALID_VALUE;
  size_t need = 0;
  const int st = b200ctc_word_errors_workspace(B, max_ref, max_hyp, &need);
  if (st != B200CTC_STATUS_SUCCESS) return st;
  unsigned char* ws = aligned_workspace(workspace, workspace_bytes, need - kAlign);   // the layout without the query's slack
  if (!ws) return B200CTC_STATUS_WORKSPACE_TOO_SMALL;
  return status_of(launch_word_errors(refs, ref_stride, ref_lens, hyps, hyp_stride, hyp_lens, B, max_ref, max_hyp, space,
                                      word4, char4, ref_counts, ws, reinterpret_cast<cudaStream_t>(stream_v)));
}

int b200ctc_softmax_temperature(const float* logits, int64_t stride_b, int64_t stride_t, int T, int V, int B,
                                float temperature, float* probs, void* stream_v) {
  return b200ctc_softmax_temperature_typed(logits, B200CTC_FLOAT32, stride_b, stride_t, T, V, B, temperature, probs,
                                           stream_v);
}

int b200ctc_softmax_temperature_typed(const void* logits, int dtype, int64_t stride_b, int64_t stride_t, int T, int V,
                                      int B, float temperature, float* probs, void* stream_v) {
  if (T < 0 || V < 1 || B < 0 || !(temperature > 0.f) || !valid_dtype(dtype)) return B200CTC_STATUS_INVALID_VALUE;
  if ((long long)B * T == 0) return B200CTC_STATUS_SUCCESS;
  if (!logits || !probs) return B200CTC_STATUS_INVALID_VALUE;
  return status_of(launch_softmax_temperature(logits, dtype, stride_b, stride_t, T, V, B, 1.0f / temperature, probs,
                                              reinterpret_cast<cudaStream_t>(stream_v)));
}

int b200ctc_greedy_decode(const float* logits, int64_t stride_b, int64_t stride_t, const int* lens,
                          int T, int V, int B, int blank, int* out_tokens, int* out_lens,
                          void* stream_v) {
  return b200ctc_greedy_decode_typed(logits, B200CTC_FLOAT32, stride_b, stride_t, lens, T, V, B, blank, out_tokens,
                                     out_lens, stream_v);
}

int b200ctc_greedy_decode_typed(const void* logits, int dtype, int64_t stride_b, int64_t stride_t, const int* lens, int T,
                                int V, int B, int blank, int* out_tokens, int* out_lens, void* stream_v) {
  if (T < 0 || V < 1 || B < 0 || !valid_dtype(dtype)) return B200CTC_STATUS_INVALID_VALUE;
  if (B == 0) return B200CTC_STATUS_SUCCESS;
  if (!lens || !out_lens || (T > 0 && (!logits || !out_tokens))) return B200CTC_STATUS_INVALID_VALUE;
  return status_of(launch_greedy(logits, dtype, stride_b, stride_t, lens, T, V, B, blank, out_tokens, out_lens,
                                 reinterpret_cast<cudaStream_t>(stream_v)));
}

}  // extern "C"
