// common.h -- helpers shared by the torch/pybind layer (ext.cpp: padding lists; fast_ops.cpp: C++ autograd
// functions behind hpc_rll.rl_utils and hpc_rll.torch_utils.network; legacy.cpp: the reference's 19 `hpc_rl_utils`
// tensor-list entry points; network.cpp: the reference's `hpc_torch_utils_network` ScatterConnection entry points).
// Nothing here computes: every function ends in a call into the C ABI (include/hpc_rll_b200.h).
#pragma once
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>
#include <torch/extension.h>

#include <vector>

#include "hpc_rll_b200.h"

namespace hpcrl {

using torch::Tensor;

inline void ck(int rc, const char* what) { TORCH_CHECK(rc == 0, what, " failed: ", hpc_rll_last_error()); }

// the reference asserts is_cuda only (hpc_rll/rl_utils/gae.py:58-59); we also check dtype and make the layout dense
inline Tensor f32(const Tensor& t, const char* name) {
    TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor (hpc version only supports cuda)");
    TORCH_CHECK_TYPE(t.scalar_type() == torch::kFloat32, name, " must be float32, got ", t.scalar_type());
    return t.contiguous();
}
inline Tensor i64(const Tensor& t, const char* name) {
    TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor (hpc version only supports cuda)");
    TORCH_CHECK_TYPE(t.scalar_type() == torch::kInt64, name, " must be int64, got ", t.scalar_type());
    return t.contiguous();
}
inline const float* fp(const Tensor& t) { return t.defined() ? t.data_ptr<float>() : nullptr; }
inline float* fpm(Tensor& t) { return t.defined() ? t.data_ptr<float>() : nullptr; }
inline const int64_t* ip(const Tensor& t) { return t.defined() ? t.data_ptr<int64_t>() : nullptr; }
inline void* cur_stream() { return c10::cuda::getCurrentCUDAStream().stream(); }

// per-call scratch from torch's caching allocator (stream-ordered reuse); call under the tensor's device guard
inline Tensor workspace(int op, int64_t T, int64_t B, int64_t N, const Tensor& like) {
    const int64_t n = static_cast<int64_t>(hpc_rll_workspace_bytes(op, T, B, N));
    return torch::empty({n < 8 ? 8 : n}, like.options().dtype(torch::kUInt8));
}

// upstream gradient of a scalar loss as a 1-element fp32 device tensor (never read on the host)
inline Tensor gscalar(const Tensor& g, const Tensor& like) {
    if (!g.defined()) return torch::zeros({1}, like.options().dtype(torch::kFloat32));
    return g.reshape({1}).to(like.device(), torch::kFloat32).contiguous();
}

void register_fast_ops(pybind11::module& m);
void register_legacy(pybind11::module& m);
void register_fast_network_ops(pybind11::module& net);
void register_network_legacy(pybind11::module& net);

}  // namespace hpcrl
