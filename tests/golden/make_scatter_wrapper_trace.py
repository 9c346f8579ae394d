#!/usr/bin/env python
"""Record how the UNMODIFIED reference ScatterConnection wrapper (DI-hpc
``hpc_rll/torch_utils/network/scatter_connection.py``) drives its native module ``hpc_torch_utils_network``.

Same machinery as make_wrapper_trace.py (its ``Trace`` / ``Recorder`` stand-in): the wrapper runs once per scenario on
the CPU and every call it makes is stored -- binding name, input / output tensor lists (a user input by name, or a
buffer by id), scalars -- with the shape, dtype and initial fill of every buffer and which binding output the user
receives, plus the binding names ``src/torch_utils/network/entry.cpp`` exports and the names the wrapper uses.
Output: tests/golden/ref_scatter_wrapper_calls.json, replayed by tests/test_scatter_connection_gpu.py.  Re-run with a
DI-hpc checkout (nothing of it is copied into this repository):

    python tests/golden/make_scatter_wrapper_trace.py <DI-hpc checkout>
"""
import json
import os
import re
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from make_wrapper_trace import Recorder, Trace, idx, t32  # noqa: E402

OUT = os.path.join(HERE, "ref_scatter_wrapper_calls.json")
WRAPPER = os.path.join("hpc_rll", "torch_utils", "network", "scatter_connection.py")


def scenarios(native, ref_root):
    """The reference test shape (tests/test_scatter.py:9-13) in both modes and an odd-sized map.
    Each yields (name, inputs, run) with run() -> results."""
    sys.modules["hpc_torch_utils_network"] = native
    path = os.path.join(ref_root, WRAPPER)
    m = types.ModuleType("ref_wrapper_scatter_connection")
    m.__file__ = path
    with open(path) as f:  # optimize=1 compiles out the wrapper's `assert x.is_cuda`
        exec(compile(f.read(), path, "exec", optimize=1), m.__dict__)
    g = np.random.default_rng(0)
    for name, (B, M, N, H, W), mode in (("scatter_cover", (256, 256, 256, 16, 16), "cover"),
                                        ("scatter_add", (256, 256, 256, 16, 16), "add"),
                                        ("scatter_add_odd", (3, 50, 17, 7, 9), "add")):
        loc = torch.stack([idx(g, H, B, M), idx(g, W, B, M)], dim=2)

        def run(i, B=B, M=M, N=N, H=H, W=W, mode=mode):
            out = m.ScatterConnection(B, M, N, H, W, mode)(i["x"], i["location"])
            out.backward(i["grad_out"])
            return {"out": out, "grad_x": i["x"].grad}
        yield name, dict(x=t32(g, B, M, N).requires_grad_(True), location=loc, grad_out=t32(g, B, N, H, W)), run


def main(ref_root):
    native = Recorder()
    with open(os.path.join(ref_root, "src", "torch_utils", "network", "entry.cpp")) as f:
        entry = sorted(re.findall(r'm\.def\("(\w+)"', f.read()))
    with open(os.path.join(ref_root, WRAPPER)) as f:
        uses = sorted(set(re.findall(r"hpc_torch_utils_network\.(\w+)", f.read())))
    out = {"source": "DI-hpc @ a8a7734: src/torch_utils/network/entry.cpp and "
                     "hpc_rll/torch_utils/network/scatter_connection.py",
           "entry_cpp_bindings": entry, "wrapper_uses": {"scatter_connection": uses}, "scenarios": {}}
    for name, inputs, run in scenarios(native, ref_root):
        native.trace = tr = Trace(inputs)
        res = run(inputs)
        out["scenarios"][name] = {
            "module": "scatter_connection",
            "inputs": {k: {"shape": list(v.shape), "dtype": str(v.dtype).replace("torch.", "")} for k, v in inputs.items()},
            "calls": tr.calls, "buffers": tr.buffers, "results": {k: tr.locate(v) for k, v in res.items()}}
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote %s (%d scenarios)" % (OUT, len(out["scenarios"])))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: make_scatter_wrapper_trace.py <DI-hpc checkout>")
    main(sys.argv[1])
