"""ScatterConnection on the GPU, compared BIT FOR BIT (signed zeros included) with the origin-generated fixtures and the
numpy oracle (oracle/scatter_oracle.py): the module through both bindings, the reference test shape and an
AlphaStar-sized map (the two backward regimes), collision-heavy maps, odd shapes and alignments, out-of-range entities
with NaN canaries around the outputs, every kernel variant forced by hpc_rll_debug_set_config, run-to-run
determinism, the reference's native names with NaN-prefilled outputs, a replay of the calls the unmodified reference
wrapper makes, and CUDA-graph replay."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import scatter_oracle as so
from tests._golden import GOLDEN_DIR, names
from tests._gpu import need_cuda

pytestmark = pytest.mark.gpu


def bits(t):
    return t.detach().contiguous().view(torch.int32).cpu()


def same_bits(got, want):
    """got: CUDA tensor, want: numpy fp32 array (or tensor): identical bit patterns."""
    w = torch.from_numpy(np.ascontiguousarray(want)) if isinstance(want, np.ndarray) else want.detach().cpu()
    g = got.detach().cpu().contiguous()
    assert g.shape == w.shape, (g.shape, w.shape)
    eq = g.view(torch.int32) == w.contiguous().view(torch.int32)
    assert bool(eq.all()), "%d of %d elements differ" % (int((~eq).sum()), eq.numel())


def inputs(B, M, N, H, W, seed, loc_hw=None, negzero=True):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, M, N, generator=g)
    if negzero:
        x[torch.rand(B, M, N, generator=g) < 0.05] = -0.0
    h, w = loc_hw or (H, W)
    loc = torch.stack([torch.randint(0, h, (B, M), generator=g), torch.randint(0, w, (B, M), generator=g)], dim=2)
    gout = torch.randn(B, N, H, W, generator=g)
    return x, loc, gout


def module_run(x, loc, gout, H, W, mode, binding="ext", monkeypatch=None):
    from hpc_rll.torch_utils.network.scatter_connection import ScatterConnection
    if monkeypatch is not None:
        monkeypatch.setenv("HPC_RLL_BINDING", binding)
    B, M, N = x.shape
    xd = x.cuda().requires_grad_(True)
    out = ScatterConnection(B, M, N, H, W, mode)(xd, loc.cuda())
    out.backward(gout.cuda())
    torch.cuda.synchronize()
    return out.detach(), xd.grad


def check_oracle(x, loc, gout, H, W, mode, out, gx):
    same_bits(out, so.forward(x.numpy(), loc.numpy(), H, W, mode))
    same_bits(gx, so.backward(gout.numpy(), loc.numpy(), H, W))


@pytest.mark.parametrize("binding", ["ext", "ctypes"])
@pytest.mark.parametrize("name", names("scatter"))
def test_fixture_through_the_module(name, binding, monkeypatch):
    need_cuda()
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    H, W, mode = int(z["H"]), int(z["W"]), str(z["scatter_type"])
    out, gx = module_run(torch.from_numpy(z["x"]), torch.from_numpy(z["location"]), torch.from_numpy(z["grad_out"]), H,
                         W, mode, binding, monkeypatch)
    same_bits(out, z["out"])
    same_bits(gx, z["grad_x"])


# (B, M, N, H, W, loc_hw): the reference test shape (dense map, slab backward), an AlphaStar-like map (sparse, direct
# gather, cells split over tiles), collision-heavy maps, odd planes / channel counts, single batch / entity
SHAPES = {
    "ref_256": (256, 256, 256, 16, 16, None),
    "alphastar": (64, 512, 32, 152, 160, None),
    "collide_4096_in_16": (8, 4096, 40, 4, 4, None),
    "collide_300_in_1": (3, 300, 33, 1, 1, None),
    "collide_corner_of_big_map": (4, 700, 32, 152, 160, (3, 5)),
    "odd_plane_5x7_n13": (6, 90, 13, 5, 7, None),
    "odd_plane_9x9_n1": (5, 200, 1, 9, 9, None),
    "b1": (1, 77, 64, 12, 20, None),
    "m1": (9, 1, 70, 16, 16, None),
    "n_not_mult4_big_map": (2, 64, 37, 33, 47, None),
}


@pytest.mark.parametrize("mode", ["add", "cover"])
@pytest.mark.parametrize("shape", sorted(SHAPES))
def test_shapes_match_oracle(shape, mode):
    need_cuda()
    B, M, N, H, W, hw = SHAPES[shape]
    x, loc, gout = inputs(B, M, N, H, W, seed=sum(map(ord, shape)) + len(mode), loc_hw=hw)
    out, gx = module_run(x, loc, gout, H, W, mode)
    check_oracle(x, loc, gout, H, W, mode, out, gx)


def test_misaligned_x_and_strided_inputs():
    need_cuda()
    from hpc_rll.torch_utils.network.scatter_connection import ScatterConnection
    B, M, N, H, W = 4, 50, 24, 8, 8
    x, loc, gout = inputs(B, M, N, H, W, seed=7)
    store = torch.empty(x.numel() + 1, device="cuda")
    xd = store[1:].view(B, M, N)  # 4 bytes past a 16-byte boundary
    xd.copy_(x.cuda())
    xd.requires_grad_(True)
    locd = torch.cat([loc.cuda(), loc.cuda()], dim=2)[:, :, :2]  # non-contiguous location
    for mode in ("add", "cover"):
        out = ScatterConnection(B, M, N, H, W, mode)(xd, locd)
        out.backward(gout.cuda().transpose(2, 3).contiguous().transpose(2, 3))  # contiguous values, strided view
        torch.cuda.synchronize()
        check_oracle(x, loc, gout, H, W, mode, out, xd.grad)
        xd.grad = None


def abi_run(x, loc, gout, H, W, mode, offset):
    """C ABI with NaN canaries around out and grad_x; out / grad_x start `offset` floats into their buffers."""
    from di_hpc_b200 import _abi
    L = _abi.lib()
    B, M, N = x.shape
    xd, ld, gd = x.cuda(), loc.cuda(), gout.cuda()
    n_out, n_gx = B * N * H * W, B * M * N
    so_ = torch.full((n_out + offset + 8, ), float("nan"), device="cuda")
    sg = torch.full((n_gx + offset + 8, ), float("nan"), device="cuda")
    out, gx = so_[offset:offset + n_out], sg[offset:offset + n_gx]
    s = _abi.stream_of(xd)
    _abi.check(L.hpc_rll_scatter_connection_forward(xd.data_ptr(), ld.data_ptr(), out.data_ptr(), B, M, N, H, W,
                                                    1 if mode == "add" else 0, s), "forward")
    _abi.check(L.hpc_rll_scatter_connection_backward(gd.data_ptr(), ld.data_ptr(), gx.data_ptr(), B, M, N, H, W, s),
               "backward")
    torch.cuda.synchronize()
    for store, n in ((so_, n_out), (sg, n_gx)):
        assert torch.isnan(store[:offset]).all() and torch.isnan(store[offset + n:]).all()  # nothing written outside
    return out.view(B, N, H, W), gx.view(B, M, N)


@pytest.mark.parametrize("offset", [0, 1])
@pytest.mark.parametrize("mode", ["add", "cover"])
def test_out_of_range_entities_write_nothing_and_get_zero_gradient(mode, offset):
    need_cuda()
    for (B, M, N, H, W) in ((5, 300, 36, 16, 16), (3, 400, 32, 152, 160), (2, 100, 5, 7, 9)):
        x, loc, gout = inputs(B, M, N, H, W, seed=B * M + offset)
        bad = torch.tensor([[-1, 0], [H, 0], [0, W], [0, -1], [1 << 40, 1], [-(1 << 40), 2], [2, 1 << 33],
                            [H - 1, W]])
        k = torch.randint(0, len(bad), (B, M), generator=torch.Generator().manual_seed(3))
        sel = torch.rand(B, M, generator=torch.Generator().manual_seed(4)) < 0.3
        loc[sel] = bad[k[sel]]
        out, gx = abi_run(x, loc, gout, H, W, mode, offset)
        check_oracle(x, loc, gout, H, W, mode, out, gx)
        assert bool((gx[sel.cuda()] == 0).all())


def test_every_kernel_variant_gives_the_same_bits():
    need_cuda()
    from di_hpc_b200 import _abi
    for (B, M, N, H, W) in ((32, 256, 64, 16, 16), (4, 512, 32, 152, 160), (6, 90, 13, 5, 7)):
        x, loc, gout = inputs(B, M, N, H, W, seed=11)
        for mode in ("add", "cover"):
            want_out = so.forward(x.numpy(), loc.numpy(), H, W, mode)
            want_gx = so.backward(gout.numpy(), loc.numpy(), H, W)
            try:
                for cfg in (-1, 0, 1, 2, 3):  # bit 0: forward per-thread stores, bit 1: backward direct gather
                    _abi.set_config(_abi.OP_SCATTER_CONNECTION, cfg)
                    out, gx = module_run(x, loc, gout, H, W, mode)
                    same_bits(out, want_out)
                    same_bits(gx, want_gx)
            finally:
                _abi.set_config(_abi.OP_SCATTER_CONNECTION, -1)


def test_two_calls_are_bitwise_equal():
    need_cuda()
    x, loc, gout = inputs(256, 256, 256, 16, 16, seed=5, loc_hw=(2, 2))  # 64 entities per cell
    for mode in ("add", "cover"):
        a = module_run(x, loc, gout, 16, 16, mode)
        b = module_run(x, loc, gout, 16, 16, mode)
        assert torch.equal(bits(a[0]), bits(b[0])) and torch.equal(bits(a[1]), bits(b[1]))


def test_cpp_and_ctypes_bindings_are_identical(monkeypatch):
    need_cuda()
    from di_hpc_b200 import _ext
    assert _ext.load() is not None, _ext.why_missing()
    x, loc, gout = inputs(16, 300, 48, 24, 20, seed=9, loc_hw=(6, 20))
    for mode in ("add", "cover"):
        a = module_run(x, loc, gout, 24, 20, mode, "ext", monkeypatch)
        b = module_run(x, loc, gout, 24, 20, mode, "ctypes", monkeypatch)
        assert torch.equal(bits(a[0]), bits(b[0])) and torch.equal(bits(a[1]), bits(b[1]))


@pytest.mark.parametrize("mode", ["add", "cover"])
def test_legacy_names_overwrite_nan_prefilled_outputs(mode):
    need_cuda()
    import hpc_torch_utils_network as h
    for (B, M, N, H, W) in ((8, 64, 40, 16, 16), (3, 50, 17, 7, 9)):
        x, loc, gout = inputs(B, M, N, H, W, seed=M)
        out = torch.full((B, N, H, W), float("nan"), device="cuda")
        gin = torch.full((B, M, N), float("nan"), device="cuda")
        h.ScatterConnectionForward([x.cuda(), loc.cuda()], [out], mode)
        h.ScatterConnectionBackward([gout.cuda(), loc.cuda()], [gin])
        torch.cuda.synchronize()
        check_oracle(x, loc, gout, H, W, mode, out, gin)
    with pytest.raises(RuntimeError):
        h.ScatterConnectionForward([x.cuda(), loc.cuda()], [out], "max")


def test_replay_of_the_reference_wrapper_calls():
    """tests/golden/ref_scatter_wrapper_calls.json: every call DI-hpc's hpc_rll/torch_utils/network/scatter_connection.py
    makes into `hpc_torch_utils_network`, replayed on this repository's module."""
    need_cuda()
    import hpc_torch_utils_network as h
    with open(os.path.join(GOLDEN_DIR, "ref_scatter_wrapper_calls.json")) as f:
        tr = json.load(f)
    assert tr["scenarios"]
    for name, sc in sorted(tr["scenarios"].items()):
        B, M, N = sc["inputs"]["x"]["shape"]
        H, W = sc["inputs"]["grad_out"]["shape"][2:]
        x, loc, gout = inputs(B, M, N, H, W, seed=len(name))
        ins = {"x": x.cuda(), "location": loc.cuda(), "grad_out": gout.cuda()}
        bufs = {int(k): torch.full(b["shape"], b["fill"], dtype=getattr(torch, b["dtype"]), device="cuda")
                for k, b in sc["buffers"].items()}
        get = lambda r: ins[r["input"]] if "input" in r else bufs[r["buffer"]]
        outs = []
        for c in sc["calls"]:
            o = [get(r) for r in c["outputs"]]
            getattr(h, c["fn"])([get(r) for r in c["inputs"]], o, *c["scalars"])
            outs.append(o)
        torch.cuda.synchronize()
        res = {k: outs[c][i] for k, (c, i) in sc["results"].items()}
        mode = sc["calls"][0]["scalars"][0]
        check_oracle(x, loc, gout, H, W, mode, res["out"], res["grad_x"])


def test_cuda_graph_replay():
    need_cuda()
    from hpc_rll.torch_utils.network.scatter_connection import ScatterConnection
    B, M, N, H, W = 16, 128, 64, 16, 16
    for mode in ("add", "cover"):
        mod = ScatterConnection(B, M, N, H, W, mode)
        x0, l0, _ = inputs(B, M, N, H, W, seed=1)
        graphed = torch.cuda.make_graphed_callables(mod, (x0.cuda().requires_grad_(True), l0.cuda()))
        for seed in (2, 3):
            x, loc, gout = inputs(B, M, N, H, W, seed=seed, loc_hw=(4, 16))
            xd = x.cuda().requires_grad_(True)
            out = graphed(xd, loc.cuda())
            out.backward(gout.cuda())
            torch.cuda.synchronize()
            check_oracle(x, loc, gout, H, W, mode, out, xd.grad)
