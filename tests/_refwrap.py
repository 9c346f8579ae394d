"""The UNMODIFIED reference wrappers (hpc_rll/rl_utils/*.py of DI-hpc) as recorded calls into their native module.

Those wrappers own no arithmetic: each module registers scratch buffers and each autograd Function hands
(input list, output list, scalars) to one `hpc_rl_utils` binding and returns some of the buffers.
tests/golden/ref_wrapper_calls.json (written by tests/golden/make_wrapper_trace.py from the reference) records,
per scenario, every such call, the shape / dtype / initial fill of every buffer, and which binding output the
user receives.  `replay` issues exactly those calls against this repository's `hpc_rl_utils` shim, which is what
a DI-hpc user gets by swapping the extension under the unmodified wrappers."""
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TRACE_PATH = os.path.join(ROOT, "tests", "golden", "ref_wrapper_calls.json")

with open(TRACE_PATH) as _f:
    TRACE = json.load(_f)


def scenario(name):
    return TRACE["scenarios"][name]


def replay(name, inputs, native, device="cuda"):
    """Issue the recorded calls of scenario `name` on `native` (the `hpc_rl_utils` module) with `inputs`
    (dict of tensors named as recorded) -> dict result name -> the binding output the wrapper returns."""
    import torch
    sc = scenario(name)
    for k, spec in sc["inputs"].items():
        t = inputs[k]
        assert list(t.shape) == spec["shape"] and str(t.dtype) == "torch." + spec["dtype"], (name, k, t.shape, t.dtype)
    bufs = {int(k): torch.full(b["shape"], b["fill"], dtype=getattr(torch, b["dtype"]), device=device)
            for k, b in sc["buffers"].items()}

    def get(ref):
        return inputs[ref["input"]] if "input" in ref else bufs[ref["buffer"]]

    outs = []
    for c in sc["calls"]:
        o = [get(r) for r in c["outputs"]]
        getattr(native, c["fn"])([get(r) for r in c["inputs"]], o, *c["scalars"])
        outs.append(o)
    return {k: outs[c][i] for k, (c, i) in sc["results"].items()}
