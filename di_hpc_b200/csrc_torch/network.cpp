// network.cpp -- the reference's native boundary for ScatterConnection: the two entry points of its pybind module
// `hpc_torch_utils_network` (/root/reference/src/torch_utils/network/entry.cpp:9-12, implemented in
// src/torch_utils/network/scatter_connection.cu:8-76) with the SAME names and `(inputs, outputs[, scatter_type])`
// tensor-list signatures, on top of the C ABI.  With this module importable as `hpc_torch_utils_network` the UNMODIFIED
// reference wrapper (hpc_rll/torch_utils/network/scatter_connection.py) runs on the B200 kernels.
//   ScatterConnectionForward ([x (B,M,N), location (B,M,2)], [output (B,N,H,W)], "cover" | "add")
//   ScatterConnectionBackward([grad_out (B,N,H,W), location], [grad_in (B,M,N)])
// H and W come from the output (forward) or grad_out (backward), B, M and N from x (forward) or grad_in (backward), as in
// the reference launcher.  The forward overwrites every element of `output` (the wrapper hands in its module buffer and
// the reference memsets it first).  LstmForward / LstmBackward are not provided.
#include "common.h"

namespace hpcrl {
namespace {

using TL = std::vector<Tensor>;

float* out_f32(Tensor& t, const char* name, int64_t numel) {
    TORCH_CHECK(t.is_cuda() && t.scalar_type() == torch::kFloat32 && t.is_contiguous(), name,
                " must be a contiguous float32 CUDA tensor");
    TORCH_CHECK(t.numel() == numel, name, " holds ", t.numel(), " elements, expected ", numel);
    return t.data_ptr<float>();
}

void check_location(const Tensor& loc, int64_t B, int64_t M) {
    TORCH_CHECK(loc.dim() == 3 && loc.size(0) == B && loc.size(1) == M && loc.size(2) == 2,
                "location must be (B, M, 2)=(", B, ", ", M, ", 2), got ", loc.sizes());
}

void ScatterConnectionForward(const TL& in, TL& out, const std::string& scatter_type) {
    TORCH_CHECK(in.size() >= 2 && out.size() >= 1, "ScatterConnectionForward: expected [input, location], [output]");
    TORCH_CHECK(scatter_type == "cover" || scatter_type == "add", "scatter_type must be 'cover' or 'add', got ",
                scatter_type);
    const Tensor x = f32(in[0], "input"), loc = i64(in[1], "location");
    TORCH_CHECK(x.dim() == 3, "input must be (B, M, N), got ", x.sizes());
    const int64_t B = x.size(0), M = x.size(1), N = x.size(2);
    check_location(loc, B, M);
    TORCH_CHECK(out[0].dim() == 4 && out[0].size(0) == B && out[0].size(1) == N, "output must be (B, N, H, W)");
    const int64_t H = out[0].size(2), W = out[0].size(3);
    c10::cuda::CUDAGuard guard(x.device());
    ck(hpc_rll_scatter_connection_forward(fp(x), ip(loc), out_f32(out[0], "output", B * N * H * W), B, M, N, H, W,
                                          scatter_type == "add" ? 1 : 0, cur_stream()),
       "hpc_rll_scatter_connection_forward");
}

void ScatterConnectionBackward(const TL& in, TL& out) {
    TORCH_CHECK(in.size() >= 2 && out.size() >= 1, "ScatterConnectionBackward: expected [grad_out, location], [grad_in]");
    const Tensor g = f32(in[0], "grad_out"), loc = i64(in[1], "location");
    TORCH_CHECK(g.dim() == 4, "grad_out must be (B, N, H, W), got ", g.sizes());
    TORCH_CHECK(out[0].dim() == 3, "grad_in must be (B, M, N)");
    const int64_t B = out[0].size(0), M = out[0].size(1), N = out[0].size(2), H = g.size(2), W = g.size(3);
    TORCH_CHECK(g.size(0) == B && g.size(1) == N, "grad_out must be (B, N, H, W) with B, N of grad_in");
    check_location(loc, B, M);
    c10::cuda::CUDAGuard guard(g.device());
    ck(hpc_rll_scatter_connection_backward(fp(g), ip(loc), out_f32(out[0], "grad_in", B * M * N), B, M, N, H, W,
                                           cur_stream()),
       "hpc_rll_scatter_connection_backward");
}

}  // namespace

void register_network_legacy(pybind11::module& net) {
    net.def("ScatterConnectionForward", &ScatterConnectionForward, "scatter_connection forward (CUDA)");
    net.def("ScatterConnectionBackward", &ScatterConnectionBackward, "scatter_connection backward (CUDA)");
}

}  // namespace hpcrl
