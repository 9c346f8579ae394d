// ext.cpp -- thin torch/pybind layer over the C ABI for the list-of-tensor (padding) entry points.
//
// The padding ops are dominated by per-tensor host work (collect pointers and shapes of ~64 small
// tensors, allocate outputs); doing that in Python costs more than the kernel.  This module does the
// list handling in C++ and then calls hpc_rll_pad_batch / hpc_rll_unpad_batch (include/hpc_rll_b200.h).
// It exports the 11 padding bindings of the reference's `hpc_rl_utils` module with the same names and
// signatures (/root/reference/src/rl_utils/entry.cpp:9-20, include/hpc/rll/cuda/rl_utils/entry.h:10-60), so
// the reference's own Python wrapper (hpc_rll/rl_utils/padding.py) runs on top of it unchanged.
// No kernels live here; without libhpc_rll_b200.so this module cannot load.
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>
#include <torch/extension.h>

#include <algorithm>
#include <random>
#include <vector>

#include "common.h"

namespace {

void check(int rc, const char* what) { TORCH_CHECK(rc == 0, what, " failed: ", hpc_rll_last_error()); }

void validate(const std::vector<torch::Tensor>& x, int ndim) {
    TORCH_CHECK(!x.empty(), "empty input list");
    const auto dev = x[0].device();
    TORCH_CHECK(dev.is_cuda(), "hpc version only supports cuda");
    for (const auto& t : x) {
        TORCH_CHECK(t.device() == dev, "all tensors must live on one CUDA device");
        TORCH_CHECK(t.scalar_type() == torch::kFloat32, "padding supports float32 tensors");
        TORCH_CHECK(t.dim() == ndim, "expected ", ndim, "-D tensors");
    }
}

// shapes of a list as n x ndim int64
std::vector<int64_t> shapes_of(const std::vector<torch::Tensor>& x, int ndim) {
    std::vector<int64_t> s(x.size() * ndim);
    for (size_t i = 0; i < x.size(); ++i)
        for (int d = 0; d < ndim; ++d) s[i * ndim + d] = x[i].size(d);
    return s;
}

// pads inputs[bounds[g] .. bounds[g+1]) to the per-group max; one launch for everything
std::pair<std::vector<torch::Tensor>, std::vector<torch::Tensor>> pad_groups(const std::vector<torch::Tensor>& in,
                                                                             int ndim,
                                                                             const std::vector<int64_t>& bounds,
                                                                             int value) {
    const int64_t n = static_cast<int64_t>(in.size());
    c10::cuda::CUDAGuard guard(in[0].device());
    std::vector<torch::Tensor> keep;  // contiguous versions stay alive until the launch is queued
    std::vector<const float*> src(n);
    std::vector<float*> dst(n);
    std::vector<int32_t*> msk(n);
    std::vector<int32_t> shp(n * 3, 1), pad(n * 3, 1);
    std::vector<torch::Tensor> new_x, mask;
    for (size_t g = 0; g + 1 < bounds.size(); ++g) {
        const int64_t lo = bounds[g], hi = bounds[g + 1];
        std::vector<int64_t> full(ndim + 1, 0);
        full[0] = hi - lo;
        for (int64_t i = lo; i < hi; ++i)
            for (int d = 0; d < ndim; ++d) full[d + 1] = std::max<int64_t>(full[d + 1], in[i].size(d));
        auto x = torch::empty(full, in[0].options());
        auto m = torch::empty(full, in[0].options().dtype(torch::kInt32));
        int64_t vol = 1;
        for (int d = 0; d < ndim; ++d) vol *= full[d + 1];
        for (int64_t i = lo; i < hi; ++i) {
            const torch::Tensor& t = in[i];
            if (t.is_contiguous()) {
                src[i] = t.numel() ? t.data_ptr<float>() : nullptr;
            } else {
                keep.push_back(t.contiguous());
                src[i] = keep.back().data_ptr<float>();
            }
            dst[i] = x.data_ptr<float>() + vol * (i - lo);
            msk[i] = m.data_ptr<int32_t>() + vol * (i - lo);
            for (int d = 0; d < ndim; ++d) {
                shp[i * 3 + (3 - ndim) + d] = static_cast<int32_t>(t.size(d));
                pad[i * 3 + (3 - ndim) + d] = static_cast<int32_t>(full[d + 1]);
            }
        }
        new_x.push_back(std::move(x));
        mask.push_back(std::move(m));
    }
    check(hpc_rll_pad_batch(src.data(), dst.data(), msk.data(), shp.data(), pad.data(), n, value,
                            c10::cuda::getCurrentCUDAStream().stream()),
          "hpc_rll_pad_batch");
    return {std::move(new_x), std::move(mask)};
}

std::vector<torch::Tensor> pad_forward(const std::vector<torch::Tensor>& inputs, int ndim, int value) {
    validate(inputs, ndim);
    auto r = pad_groups(inputs, ndim, {0, static_cast<int64_t>(inputs.size())}, value);
    return {r.first[0], r.second[0]};
}

std::vector<std::vector<torch::Tensor>> group_pad_forward(const std::vector<torch::Tensor>& inputs, int ndim,
                                                          const std::vector<int>& group_idx, int value) {
    validate(inputs, ndim);
    std::vector<int64_t> bounds(group_idx.begin(), group_idx.end());
    if (bounds.empty() || bounds.back() != static_cast<int64_t>(inputs.size()))
        bounds.push_back(static_cast<int64_t>(inputs.size()));
    auto r = pad_groups(inputs, ndim, bounds, value);
    return {std::move(r.first), std::move(r.second)};
}

std::vector<torch::Tensor> unpad_forward(const torch::Tensor& x_in, const std::vector<int>& shape, int ndim) {
    TORCH_CHECK(x_in.is_cuda(), "hpc version only supports cuda");
    TORCH_CHECK(x_in.scalar_type() == torch::kFloat32, "padding supports float32 tensors");
    TORCH_CHECK(x_in.dim() == ndim + 1, "expected a ", ndim + 1, "-D padded batch");
    const torch::Tensor x = x_in.contiguous();
    const int64_t n = x.size(0);
    TORCH_CHECK(static_cast<int64_t>(shape.size()) == n * ndim, "shapes must hold ", ndim, " ints per tensor");
    c10::cuda::CUDAGuard guard(x.device());
    int64_t total = 0, vol = 1;
    for (int d = 0; d < ndim; ++d) vol *= x.size(d + 1);
    std::vector<int64_t> sizes(n);
    for (int64_t i = 0; i < n; ++i) {
        int64_t s = 1;
        for (int d = 0; d < ndim; ++d) s *= shape[i * ndim + d];
        sizes[i] = s;
        total += s;
    }
    auto flat = torch::empty({total}, x.options());  // one allocation; the outputs are views of it
    std::vector<const float*> src(n);
    std::vector<float*> dst(n);
    std::vector<int32_t> shp(n * 3, 1), pad(n * 3, 1);
    std::vector<torch::Tensor> out;
    out.reserve(n);
    int64_t off = 0;
    for (int64_t i = 0; i < n; ++i) {
        src[i] = x.data_ptr<float>() + vol * i;
        dst[i] = flat.data_ptr<float>() + off;
        std::vector<int64_t> view(ndim);
        for (int d = 0; d < ndim; ++d) {
            view[d] = shape[i * ndim + d];
            shp[i * 3 + (3 - ndim) + d] = shape[i * ndim + d];
            pad[i * 3 + (3 - ndim) + d] = static_cast<int32_t>(x.size(d + 1));
        }
        out.push_back(flat.narrow(0, off, sizes[i]).view(view));
        off += sizes[i];
    }
    check(hpc_rll_unpad_batch(src.data(), dst.data(), shp.data(), pad.data(), n,
                              c10::cuda::getCurrentCUDAStream().stream()),
          "hpc_rll_unpad_batch");
    return out;
}

// ---- group splitters, reference return convention: group shapes ..., then the index vector -----------------
std::vector<std::vector<int>> pack_split(const std::vector<torch::Tensor>& x, const std::vector<int64_t>& bounds) {
    const int ndim = static_cast<int>(x[0].dim());
    std::vector<std::vector<int>> res;
    for (size_t g = 0; g + 1 < bounds.size(); ++g) {
        std::vector<int> mx(ndim, 0);
        for (int64_t i = bounds[g]; i < bounds[g + 1]; ++i)
            for (int d = 0; d < ndim; ++d) mx[d] = std::max<int>(mx[d], static_cast<int>(x[i].size(d)));
        res.push_back(mx);
    }
    res.emplace_back(bounds.begin(), bounds.end());
    return res;
}

std::vector<std::vector<int>> oracle_split_group(const std::vector<torch::Tensor>& x, int group) {
    TORCH_CHECK(!x.empty(), "empty input list");
    const int ndim = static_cast<int>(x[0].dim());
    const int64_t n = static_cast<int64_t>(x.size());
    const int g = static_cast<int>(std::min<int64_t>(group, n));
    auto shp = shapes_of(x, ndim);
    std::vector<int64_t> pos(g + 1);
    check(hpc_rll_oracle_split_group(shp.data(), n, ndim, g, pos.data()), "hpc_rll_oracle_split_group");
    return pack_split(x, pos);
}

std::vector<std::vector<int>> sample_split_group(const std::vector<torch::Tensor>& x, int group) {
    TORCH_CHECK(!x.empty(), "empty input list");
    static std::mt19937_64 rng(0x5EED);
    const int ndim = static_cast<int>(x[0].dim());
    const int64_t n = static_cast<int64_t>(x.size());
    auto shp = shapes_of(x, ndim);
    std::vector<int64_t> starts(group + 2);
    int cnt = 0;
    check(hpc_rll_sample_split_group(shp.data(), n, ndim, group, rng(), starts.data(), &cnt),
          "hpc_rll_sample_split_group");
    starts.resize(cnt + 1);
    return pack_split(x, starts);
}

// ---- whole-call entry points used by di_hpc_b200/rl_utils/padding.py (everything host-side in C++) --------
// returns (new_x, mask, flat shapes)
py::tuple pad_nd(const std::vector<torch::Tensor>& inputs, int ndim, int value) {
    validate(inputs, ndim);
    auto r = pad_groups(inputs, ndim, {0, static_cast<int64_t>(inputs.size())}, value);
    auto shp = shapes_of(inputs, ndim);
    return py::make_tuple(r.first[0], r.second[0], shp);
}

// sort by element count (stable), split (mode 0 = sample, 1 = oracle), pad every group in one launch;
// returns [tuple(new_x), tuple(mask), tuple(per-group flat shapes)] like hpc_rll/rl_utils/padding.py:39-41
py::list group_pad_nd(const std::vector<torch::Tensor>& inputs, int ndim, int group, int mode, int value) {
    validate(inputs, ndim);
    std::vector<torch::Tensor> x(inputs);
    std::stable_sort(x.begin(), x.end(), [](const torch::Tensor& a, const torch::Tensor& b) { return a.numel() < b.numel(); });
    auto split = mode == 1 ? oracle_split_group(x, group) : sample_split_group(x, group);
    std::vector<int64_t> bounds(split.back().begin(), split.back().end());
    auto r = pad_groups(x, ndim, bounds, value);
    py::tuple tx(r.first.size()), tm(r.first.size()), ts(r.first.size());
    for (size_t g = 0; g + 1 < bounds.size(); ++g) {
        std::vector<int64_t> flat;
        for (int64_t i = bounds[g]; i < bounds[g + 1]; ++i)
            for (int d = 0; d < ndim; ++d) flat.push_back(x[i].size(d));
        tx[g] = r.first[g];
        tm[g] = r.second[g];
        ts[g] = flat;
    }
    py::list out;
    out.append(tx);
    out.append(tm);
    out.append(ts);
    return out;
}

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
    hpcrl::register_fast_ops(m);  // C++ autograd functions behind hpc_rll.rl_utils (fast_ops.cpp)
    hpcrl::register_legacy(m);    // the reference's 19 hot-path `hpc_rl_utils` names (legacy.cpp)
    // hpc_rll.torch_utils.network: its autograd op and the reference's `hpc_torch_utils_network` names
    pybind11::module net = m.def_submodule("_network", "ScatterConnection (hpc_rll.torch_utils.network)");
    hpcrl::register_fast_network_ops(net);  // fast_ops.cpp
    hpcrl::register_network_legacy(net);    // network.cpp
    m.def("pad_nd", &pad_nd, "pad a list of n-D tensors: (new_x, mask, flat shapes)");
    m.def("group_pad_nd", &group_pad_nd, "sort + split + pad in one call");
    m.def("unpad_nd", [](const torch::Tensor& x, const std::vector<int>& s, int ndim) { return unpad_forward(x, s, ndim); },
          "unpad a padded batch into views of one allocation");
    m.def("sample_split_group", &sample_split_group, "sample_split_group");
    m.def("oracle_split_group", &oracle_split_group, "oracle_split_group");
    m.def("Pad1DForward", [](const std::vector<torch::Tensor>& x, const int& v) { return pad_forward(x, 1, v); },
          "Pad1D forward (CUDA)");
    m.def("Pad2DForward", [](const std::vector<torch::Tensor>& x, const int& v) { return pad_forward(x, 2, v); },
          "Pad2D forward (CUDA)");
    m.def("Pad3DForward", [](const std::vector<torch::Tensor>& x, const int& v) { return pad_forward(x, 3, v); },
          "Pad3D forward (CUDA)");
    // reference signature: (inputs, group_cnt, max_shape, group_id, group_idx, value); only group_idx is needed
    m.def("GroupPad1DForward",
          [](const std::vector<torch::Tensor>& x, const std::vector<int>&, const std::vector<int>&,
             const std::vector<int>&, const std::vector<int>& gi, const int& v) { return group_pad_forward(x, 1, gi, v); },
          "GroupPad1D forward (CUDA)");
    m.def("GroupPad2DForward",
          [](const std::vector<torch::Tensor>& x, const std::vector<int>&, const std::vector<int>&,
             const std::vector<int>&, const std::vector<int>& gi, const int& v) { return group_pad_forward(x, 2, gi, v); },
          "GroupPad2D forward (CUDA)");
    m.def("GroupPad3DForward",
          [](const std::vector<torch::Tensor>& x, const std::vector<int>&, const std::vector<int>&,
             const std::vector<int>&, const std::vector<int>& gi, const int& v) { return group_pad_forward(x, 3, gi, v); },
          "GroupPad3D forward (CUDA)");
    m.def("Unpad1DForward", [](const torch::Tensor& x, const std::vector<int>& s) { return unpad_forward(x, s, 1); },
          "Unpad1D forward (CUDA)");
    m.def("Unpad2DForward", [](const torch::Tensor& x, const std::vector<int>& s) { return unpad_forward(x, s, 2); },
          "Unpad2D forward (CUDA)");
    m.def("Unpad3DForward", [](const torch::Tensor& x, const std::vector<int>& s) { return unpad_forward(x, s, 3); },
          "Unpad3D forward (CUDA)");
}
