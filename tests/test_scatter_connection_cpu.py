"""ScatterConnection without a GPU: the numpy oracle against the origin-generated fixtures (bit for bit), the reference's
API surface (module, autograd function, the native `hpc_torch_utils_network` names and the arity of every call the
reference wrapper makes), argument errors of the C ABI, and the SASS of the built kernels (bulk stores, no atomics)."""
import inspect
import os

import numpy as np
import pytest

from oracle import scatter_oracle as so
from tests._golden import GOLDEN_DIR, names

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load(name):
    return np.load(os.path.join(GOLDEN_DIR, name + ".npz"))


def trace():
    import json
    with open(os.path.join(GOLDEN_DIR, "ref_scatter_wrapper_calls.json")) as f:
        return json.load(f)


@pytest.mark.parametrize("name", names("scatter"))
def test_oracle_matches_origin_bit_for_bit(name):
    z = load(name)
    H, W, mode = int(z["H"]), int(z["W"]), str(z["scatter_type"])
    out = so.forward(z["x"], z["location"], H, W, mode)
    assert out.dtype == np.float32 and out.tobytes() == z["out"].tobytes()  # bytes: -0.0 vs +0.0 counts
    gx = so.backward(z["grad_out"], z["location"], H, W)
    assert gx.dtype == np.float32 and gx.tobytes() == z["grad_x"].tobytes()


def test_fixtures_cover_signed_zeros_and_collisions():
    negzero = lambda a: int((np.signbit(a) & (a == 0)).sum())
    modes, collide = set(), 0
    for name in names("scatter"):
        z = load(name)
        modes.add(str(z["scatter_type"]))
        assert negzero(z["x"]) > 0
        if str(z["scatter_type"]) == "add":
            assert negzero(z["out"]) == 0  # the sum starts at +0.0
        cells = z["location"][..., 0] * int(z["W"]) + z["location"][..., 1]
        collide = max(collide, max(len(c) - len(np.unique(c)) for c in cells))
    assert modes == {"add", "cover"} and collide >= 900
    assert any(negzero(load(n)["out"]) > 0 for n in names("scatter") if "cover" in n)  # cover copies -0.0


def test_oracle_drops_out_of_range_entities():
    x = np.arange(1, 13, dtype=np.float32).reshape(1, 4, 3)
    loc = np.array([[[0, 0], [2, 0], [0, -1], [1, 1]]], dtype=np.int64)  # y == H, x < 0 are outside a 2x2 map
    out = so.forward(x, loc, 2, 2, "add")
    assert out[0, :, 0, 0].tolist() == [1, 2, 3] and out[0, :, 1, 1].tolist() == [10, 11, 12]
    assert out.sum() == 1 + 2 + 3 + 10 + 11 + 12
    g = so.backward(np.ones((1, 3, 2, 2), dtype=np.float32), loc, 2, 2)
    assert g[0, :, 0].tolist() == [1, 0, 0, 1]


def test_reference_api_surface():
    import hpc_rll.torch_utils.network as net
    import hpc_rll.torch_utils.network.scatter_connection as sc

    def params(fn):
        return [p for p in inspect.signature(fn).parameters if p != "self"]

    assert net.ScatterConnection is sc.ScatterConnection
    assert params(sc.ScatterConnection.__init__) == ["B", "M", "N", "H", "W", "scatter_type"]
    assert params(sc.ScatterConnection.forward) == ["x", "location"]
    assert hasattr(sc, "ScatterConnectionFunction")
    import torch
    m = sc.ScatterConnection(2, 3, 4, 5, 6, "add").cuda()  # parameter-free: .cuda() needs no device
    assert isinstance(m, torch.nn.Module) and m.H == 5 and m.W == 6
    with pytest.raises(AssertionError):
        sc.ScatterConnection(2, 3, 4, 5, 6, "max")
    with pytest.raises(ImportError):
        import hpc_rll.torch_utils.network.rnn  # noqa: F401  (LSTM stays out)


def test_native_module_names_and_arity_match_the_recorded_wrapper():
    import hpc_torch_utils_network as h
    t = trace()
    assert sorted(t["entry_cpp_bindings"]) == ["LstmBackward", "LstmForward", "ScatterConnectionBackward",
                                               "ScatterConnectionForward"]
    assert sorted(h.__all__) == ["ScatterConnectionBackward", "ScatterConnectionForward"]
    assert not hasattr(h, "LstmForward")
    used = t["wrapper_uses"]["scatter_connection"]
    assert used and all(callable(getattr(h, u)) for u in used)
    calls = [c for s in t["scenarios"].values() for c in s["calls"]]
    assert {c["fn"] for c in calls} == set(used)
    for c in calls:
        sig = getattr(h, c["fn"]).__doc__.splitlines()[0]
        assert "Sequence[torch.Tensor]" in sig and sig.count("arg") == 2 + len(c["scalars"]), (c["fn"], sig)


def test_hpc_rl_utils_names_unchanged():
    import hpc_rl_utils
    names_now = sorted(k for k in dir(hpc_rl_utils) if not k.startswith("_"))
    assert not any("catter" in k for k in names_now)
    assert len(names_now) == 43, names_now  # the reference's 30 binding names + 13 fast ops of hpc_rll.rl_utils


def test_argument_errors_are_reported_without_a_gpu():
    from di_hpc_b200 import _abi
    L = _abi.lib()
    fwd, bwd = L.hpc_rll_scatter_connection_forward, L.hpc_rll_scatter_connection_backward
    assert fwd(None, None, None, 2, 3, 4, 5, 6, 2, None) == 1  # bad mode
    assert b"mode" in L.hpc_rll_last_error()
    assert fwd(None, None, None, 2, -3, 4, 5, 6, 1, None) == 1
    assert b"negative" in L.hpc_rll_last_error()
    assert fwd(None, None, None, 2, 3, 4, 5, 6, 0, None) == 1
    assert b"null" in L.hpc_rll_last_error()
    assert fwd(None, None, None, 2, 3, 4, 1 << 20, 1 << 20, 1, None) == 1  # H*W beyond the int cell index
    assert bwd(None, None, None, 2, 3, 4, 5, -6, None) == 1
    assert bwd(None, None, None, 2, 3, 4, 5, 6, None) == 1
    # zero-size problems are no-ops (nothing to write), with any pointers
    assert fwd(None, None, None, 0, 3, 4, 5, 6, 1, None) == 0
    assert fwd(None, None, None, 2, 3, 4, 0, 6, 0, None) == 0
    assert bwd(None, None, None, 2, 0, 4, 5, 6, None) == 0
    assert L.hpc_rll_workspace_bytes(_abi.OP_SCATTER_CONNECTION, 0, 2, 4) == 0
    assert L.hpc_rll_debug_set_config(_abi.OP_SCATTER_CONNECTION, -1) == 0
    assert L.hpc_rll_launch_count() == 0


@pytest.fixture(scope="module")
def sass():
    import sys
    sys.path.insert(0, ROOT)
    from di_hpc_b200 import build
    from tools import sass_opcodes
    if sass_opcodes.cuobjdump() is None:
        pytest.skip("cuobjdump not found (neither on PATH nor in the CUDA toolkit)")
    kernels, atomics, _ = sass_opcodes.parse(build.build())
    return kernels, atomics


def test_forward_writer_stores_in_bulk(sass):
    kernels, atomics = sass
    # scatter_conn_fwd_kernel<ADD, BULK>: Lb1EE = BULK true
    bulk = {k: c for k, c in kernels.items() if "scatter_conn_fwd_kernel" in k and k.endswith("Lb1EEEvPKfPKlPfiiiiiii")}
    assert len(bulk) == 2, sorted(kernels)
    for name, c in bulk.items():
        assert c["UBLKCP"] > 0 or c["UTMASTG"] > 0, (name, dict(c))
        assert c["STG"] == 0, (name, c["STG"])  # the tile leaves through the copy engine only
    slab = [c for k, c in kernels.items() if "scatter_conn_bwd_slab_kernel" in k]
    assert slab and all(c["UBLKCP"] > 0 and c["SYNCS"] > 0 for c in slab)
    scatter = [k for k in kernels if "scatter_conn" in k]
    assert len(scatter) == 6 and not any(k in atomics for k in scatter)
