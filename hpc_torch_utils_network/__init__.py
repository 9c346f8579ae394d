"""`hpc_torch_utils_network` -- the reference's NATIVE module name for its network ops (/root/reference/setup.py:35-40,
src/torch_utils/network/entry.cpp:8-13), exporting `ScatterConnectionForward(inputs, outputs, scatter_type)` and
`ScatterConnectionBackward(inputs, outputs)` with the reference's tensor-list signatures, implemented on
libhpc_rll_b200.so (di_hpc_b200/csrc_torch/network.cpp).  With the repo root on sys.path the UNMODIFIED reference
wrapper `hpc_rll/torch_utils/network/scatter_connection.py` runs on the B200 kernels.  `LstmForward` / `LstmBackward`
are not provided (LSTM is out of scope, DESIGN.md section 8)."""
from di_hpc_b200 import _ext as _loader

_m = _loader.require()._network
ScatterConnectionForward = _m.ScatterConnectionForward
ScatterConnectionBackward = _m.ScatterConnectionBackward
__all__ = ["ScatterConnectionForward", "ScatterConnectionBackward"]
