// Thin PyTorch C++ extension over the C ABI (include/b200ctc.h): what replaces warp-ctc's pytorch_binding
// (tools/install_warpctc_pytorch.sh:12-18 builds `pytorch_binding/setup.py install`; reference call site
// models/pytorch_v3/ctc/ctc.py:35,39-45).  PyTorch supplies device memory, the current stream and the tensor
// checks; every computation happens behind the C ABI in libb200ctc.so.  It is the one binding of the loss
// (ctc.py); the ctypes binding (_lib.py) serves the decoders, evaluation and diagnostics on the same handles.
#include <torch/extension.h>
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>

#include <map>
#include <mutex>
#include <tuple>

#include "b200ctc.h"

namespace {

std::mutex g_mu;
std::map<int, b200ctc_handle*> g_handles;                          // one handle per device
std::map<std::pair<int, void*>, at::Tensor> g_workspaces;          // (device, stream) -> growing workspace

void check(int st, const char* what) {
  TORCH_CHECK(st == B200CTC_STATUS_SUCCESS, what, " failed: ", b200ctc_status_string(st), " (status ", st, ")");
}

b200ctc_handle* handle_of(int device) {
  std::lock_guard<std::mutex> lock(g_mu);
  auto it = g_handles.find(device);
  if (it != g_handles.end()) return it->second;
  b200ctc_handle* h = nullptr;
  check(b200ctc_create(&h, device), "b200ctc_create");
  g_handles[device] = h;
  return h;
}

at::Tensor workspace_of(int device, void* stream, size_t bytes) {
  std::lock_guard<std::mutex> lock(g_mu);
  auto key = std::make_pair(device, stream);
  auto it = g_workspaces.find(key);
  if (it == g_workspaces.end() || (size_t)it->second.numel() < bytes) {
    const int64_t n = std::max<int64_t>((int64_t)(bytes + bytes / 4), 1 << 20);
    g_workspaces[key] = at::empty({n}, at::TensorOptions().dtype(at::kByte).device(at::kCUDA, device));
    it = g_workspaces.find(key);
  }
  return it->second;
}

// `reduced`: the device-label call also takes bfloat16 and float16 logits; the host-label (warp-ctc) call is fp32 only
void check_acts(const at::Tensor& acts, bool reduced) {
  TORCH_CHECK(acts.is_cuda(), "acts must be a CUDA tensor: this engine has no CPU path");
  const auto t = acts.scalar_type();
  TORCH_CHECK(t == at::kFloat || (reduced && (t == at::kBFloat16 || t == at::kHalf)),
              reduced ? "acts must be float32, bfloat16 or float16" : "acts must be float32");
  TORCH_CHECK(acts.dim() == 3, "acts must be [T, B, V]");
}

int dtype_of(const at::Tensor& acts) {
  switch (acts.scalar_type()) {
    case at::kBFloat16: return B200CTC_BFLOAT16;
    case at::kHalf: return B200CTC_FLOAT16;
    default: return B200CTC_FLOAT32;
  }
}

// The gradient has the logits' element type; costs and the loss sum are fp32 whatever it is.

std::tuple<at::Tensor, at::Tensor, at::Tensor> outputs(const at::Tensor& acts, const c10::optional<at::Tensor>& grads,
                                                       bool need_grad, const c10::optional<at::Tensor>& costs,
                                                       const c10::optional<at::Tensor>& loss_sum) {
  const auto T = acts.size(0), B = acts.size(1), V = acts.size(2);
  at::Tensor g;
  if (need_grad) {
    if (grads.has_value()) {
      g = *grads;
      TORCH_CHECK(g.is_cuda() && g.scalar_type() == acts.scalar_type() && g.is_contiguous() && g.sizes() == acts.sizes(),
                  "grads must be a contiguous CUDA tensor shaped like acts, of its dtype");
    } else {
      g = at::empty({T, B, V}, acts.options().memory_format(at::MemoryFormat::Contiguous));
    }
  }
  at::Tensor c = costs.has_value() ? *costs : at::empty({B}, acts.options().dtype(at::kFloat));
  at::Tensor l = loss_sum.has_value() ? *loss_sum : at::empty({1}, acts.options().dtype(at::kFloat));
  return {c, l, g};
}

}  // namespace

// Device-resident labels / lengths (b200ctc_loss_and_grad_dev_typed): kernel launches only, CUDA-graph capturable.
// fp32, bfloat16 or float16 logits; the gradient is returned in their dtype.
std::tuple<at::Tensor, at::Tensor, c10::optional<at::Tensor>> loss_and_grad_dev(
    at::Tensor acts, at::Tensor labels, at::Tensor act_lens, at::Tensor label_lens, int64_t blank,
    c10::optional<at::Tensor> grads, bool need_grad, c10::optional<at::Tensor> costs, c10::optional<at::Tensor> loss_sum,
    int64_t max_label_len, double logit_scale, double label_smoothing, double loss_scale, double grad_scale,
    c10::optional<at::Tensor> ls_costs) {
  check_acts(acts, true);
  if (acts.stride(2) != 1 && acts.size(2) > 1) acts = acts.contiguous();
  const int T = (int)acts.size(0), B = (int)acts.size(1), V = (int)acts.size(2);
  TORCH_CHECK(labels.is_cuda() && labels.dim() == 2 && labels.size(0) == B, "labels must be a padded CUDA [B, Lmax] tensor");
  if (labels.scalar_type() != at::kInt || labels.stride(1) != 1) labels = labels.to(at::kInt).contiguous();
  if (act_lens.scalar_type() != at::kInt || !act_lens.is_contiguous()) act_lens = act_lens.to(at::kInt).contiguous();
  if (label_lens.scalar_type() != at::kInt || !label_lens.is_contiguous()) label_lens = label_lens.to(at::kInt).contiguous();
  TORCH_CHECK(act_lens.is_cuda() && label_lens.is_cuda() && act_lens.numel() == B && label_lens.numel() == B,
              "act_lens and label_lens must be CUDA tensors with one entry per utterance");
  const int Lmax = max_label_len >= 0 ? (int)max_label_len : (int)labels.size(1);
  TORCH_CHECK(Lmax <= labels.size(1), "max_label_len exceeds the padded label width");
  c10::cuda::CUDAGuard guard(acts.device());
  const int device = acts.get_device();
  auto [c, l, g] = outputs(acts, grads, need_grad, costs, loss_sum);
  cudaStream_t stream = at::cuda::getCurrentCUDAStream(device).stream();
  size_t bytes = 0;
  const int dtype = dtype_of(acts);
  check(b200ctc_get_workspace_bound_typed(T, V, B, Lmax, dtype, need_grad ? 1 : 0, &bytes),
        "b200ctc_get_workspace_bound_typed");
  at::Tensor ws = workspace_of(device, (void*)stream, bytes);
  b200ctc_options o{(float)logit_scale, (float)label_smoothing, (float)loss_scale, (float)grad_scale};
  const bool plain = logit_scale == 1.0 && label_smoothing == 0.0 && loss_scale == 1.0 && grad_scale == 1.0;
  check(b200ctc_loss_and_grad_dev_typed(handle_of(device), acts.data_ptr(), acts.stride(0), acts.stride(1), dtype,
                                  need_grad ? g.data_ptr() : nullptr, labels.data_ptr<int>(),
                                  (B > 0 && labels.size(1) > 0) ? (int)labels.stride(0) : Lmax,
                                  label_lens.data_ptr<int>(), act_lens.data_ptr<int>(), T, V, B, Lmax, (int)blank,
                                  plain ? nullptr : &o, c.data_ptr<float>(), l.data_ptr<float>(),
                                  ls_costs.has_value() ? ls_costs->data_ptr<float>() : nullptr, ws.data_ptr(),
                                  (size_t)ws.numel(), (void*)stream),
        "b200ctc_loss_and_grad_dev_typed");
  return {c, l, need_grad ? c10::optional<at::Tensor>(g) : c10::nullopt};
}

// Host-resident flat labels / lengths: the warp-ctc contract (b200ctc_loss_and_grad).
std::tuple<at::Tensor, at::Tensor, c10::optional<at::Tensor>> loss_and_grad_host(
    at::Tensor acts, at::Tensor labels, at::Tensor act_lens, at::Tensor label_lens, int64_t blank,
    c10::optional<at::Tensor> grads, bool need_grad, c10::optional<at::Tensor> costs, c10::optional<at::Tensor> loss_sum) {
  check_acts(acts, false);
  if (acts.stride(2) != 1 && acts.size(2) > 1) acts = acts.contiguous();
  const int T = (int)acts.size(0), B = (int)acts.size(1), V = (int)acts.size(2);
  auto host_i32 = [](at::Tensor x, const char* name) {
    TORCH_CHECK(x.dim() == 1, name, " must be 1-dimensional");
    return x.to(at::kCPU, at::kInt).contiguous();
  };
  labels = host_i32(labels, "labels");
  act_lens = host_i32(act_lens, "act_lens");
  label_lens = host_i32(label_lens, "label_lens");
  TORCH_CHECK(act_lens.numel() == B && label_lens.numel() == B, "act_lens and label_lens must have one entry per utterance");
  TORCH_CHECK(label_lens.sum().item<int64_t>() == labels.numel(), "sum(label_lens) does not match len(labels)");
  c10::cuda::CUDAGuard guard(acts.device());
  const int device = acts.get_device();
  auto [c, l, g] = outputs(acts, grads, need_grad, costs, loss_sum);
  cudaStream_t stream = at::cuda::getCurrentCUDAStream(device).stream();
  size_t bytes = 0;
  check(b200ctc_get_workspace_size(label_lens.data_ptr<int>(), act_lens.data_ptr<int>(), T, V, B, &bytes),
        "b200ctc_get_workspace_size");
  at::Tensor ws = workspace_of(device, (void*)stream, bytes);
  check(b200ctc_loss_and_grad(handle_of(device), acts.data_ptr<float>(), acts.stride(0), acts.stride(1),
                              need_grad ? g.data_ptr<float>() : nullptr, labels.data_ptr<int>(),
                              label_lens.data_ptr<int>(), act_lens.data_ptr<int>(), T, V, B, (int)blank,
                              c.data_ptr<float>(), l.data_ptr<float>(), ws.data_ptr(), (size_t)ws.numel(), (void*)stream),
        "b200ctc_loss_and_grad");
  return {c, l, need_grad ? c10::optional<at::Tensor>(g) : c10::nullopt};
}

// Backward of a loss on bfloat16 / float16 logits (b200ctc_scale_grads): grads * scale in fp32, rounded once; `scale`
// holds one value or one per utterance.
at::Tensor scale_grads(at::Tensor grads, at::Tensor scale) {
  const auto t = grads.scalar_type();
  TORCH_CHECK(grads.is_cuda() && (t == at::kBFloat16 || t == at::kHalf) && grads.is_contiguous() && grads.dim() == 3,
              "grads must be a contiguous CUDA bfloat16 or float16 [T, B, V] tensor");
  const int T = (int)grads.size(0), B = (int)grads.size(1), V = (int)grads.size(2);
  scale = scale.to(at::kFloat).contiguous();
  TORCH_CHECK(scale.is_cuda() && scale.get_device() == grads.get_device() && (scale.numel() == 1 || scale.numel() == B),
              "scale must be a CUDA tensor on the gradient's device with one value or one per utterance");
  c10::cuda::CUDAGuard guard(grads.device());
  at::Tensor out = at::empty_like(grads);
  cudaStream_t stream = at::cuda::getCurrentCUDAStream(grads.get_device()).stream();
  check(b200ctc_scale_grads(grads.data_ptr(), out.data_ptr(), dtype_of(grads), T, B, V, scale.data_ptr<float>(),
                            (int)scale.numel(), (void*)stream),
        "b200ctc_scale_grads");
  return out;
}

int64_t handle_address(int64_t device) { return (int64_t)(intptr_t)handle_of((int)device); }

void release_workspaces() {
  std::lock_guard<std::mutex> lock(g_mu);
  g_workspaces.clear();
}

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.doc() = "PyTorch binding of the B200 CTC engine's C ABI (include/b200ctc.h)";
  m.def("loss_and_grad_dev", &loss_and_grad_dev, "CTC cost and gradient, device-resident labels and lengths",
        py::arg("acts"), py::arg("labels"), py::arg("act_lens"), py::arg("label_lens"), py::arg("blank") = 0,
        py::arg("grads") = py::none(), py::arg("need_grad") = true, py::arg("costs") = py::none(),
        py::arg("loss_sum") = py::none(), py::arg("max_label_len") = -1, py::arg("logit_scale") = 1.0,
        py::arg("label_smoothing") = 0.0, py::arg("loss_scale") = 1.0, py::arg("grad_scale") = 1.0,
        py::arg("ls_costs") = py::none());
  m.def("loss_and_grad_host", &loss_and_grad_host, "CTC cost and gradient, host-resident flat labels (warp-ctc contract)",
        py::arg("acts"), py::arg("labels"), py::arg("act_lens"), py::arg("label_lens"), py::arg("blank") = 0,
        py::arg("grads") = py::none(), py::arg("need_grad") = true, py::arg("costs") = py::none(),
        py::arg("loss_sum") = py::none());
  m.def("scale_grads", &scale_grads, "grads * scale in fp32, rounded once to the bfloat16 / float16 gradient's dtype",
        py::arg("grads"), py::arg("scale"));
  m.def("handle_address", &handle_address, "address of the device's b200ctc_handle (shared with the ctypes diagnostics)");
  m.def("release_workspaces", &release_workspaces);
}
