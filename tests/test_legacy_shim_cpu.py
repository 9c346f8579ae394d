"""The native boundary of the reference: a module importable as `hpc_rl_utils` exporting the 30 binding names of
DI-hpc's src/rl_utils/entry.cpp:9-38 with tensor-list signatures.  CPU part: names, arities, and that every call the
UNMODIFIED reference wrappers make (recorded in tests/golden/ref_wrapper_calls.json) reaches a shim binding that takes
those arguments (no kernel runs without a GPU)."""
import os

import pytest

from tests import _refwrap

HOT = {"GaeForward": 4, "TdLambdaForward": 4, "TdLambdaBackward": 2, "DistNStepTdForward": 5, "DistNStepTdBackward": 2,
       "QNStepTdForward": 3, "QNStepTdBackward": 2, "QNStepTdRescaleForward": 3, "QNStepTdRescaleBackward": 2,
       "UpgoForward": 2, "UpgoBackward": 2, "VTraceForward": 7, "VTraceBackward": 2, "PPOForward": 5, "PPOBackward": 2,
       "IQNNStepTDErrorForward": 4, "IQNNStepTDErrorBackward": 2, "QRDQNNStepTDErrorForward": 3,
       "QRDQNNStepTDErrorBackward": 2}
PAD = ["sample_split_group", "oracle_split_group", "Pad1DForward", "GroupPad1DForward", "Unpad1DForward", "Pad2DForward",
       "GroupPad2DForward", "Unpad2DForward", "Pad3DForward", "GroupPad3DForward", "Unpad3DForward"]


def test_all_reference_binding_names_exist_with_reference_arity():
    import hpc_rl_utils
    for name in list(HOT) + PAD:
        assert callable(getattr(hpc_rl_utils, name)), name
    for name, nargs in HOT.items():
        sig = getattr(hpc_rl_utils, name).__doc__.splitlines()[0]
        assert sig.count("arg") == nargs, (name, sig)
        assert "Sequence[torch.Tensor]" in sig  # (inputs, outputs, floats...) like entry.h:62-165


def test_entry_cpp_lists_exactly_these_names():
    assert sorted(_refwrap.TRACE["entry_cpp_bindings"]) == sorted(list(HOT) + PAD)


@pytest.mark.parametrize("mod", ["gae", "td", "upgo", "vtrace", "ppo"])
def test_unmodified_reference_wrappers_bind_to_the_shim(mod):
    import hpc_rl_utils
    # `import hpc_rl_utils` inside the wrappers resolves to this repository's shim
    assert os.path.dirname(os.path.abspath(hpc_rl_utils.__file__)) == os.path.join(_refwrap.ROOT, "hpc_rl_utils")
    used = _refwrap.TRACE["wrapper_uses"][mod]
    assert used and all(hasattr(hpc_rl_utils, u) for u in used), used
    # every recorded call of this wrapper: (inputs, outputs, scalars...) matches the binding's arity
    calls = [c for s in _refwrap.TRACE["scenarios"].values() if s["module"] == mod for c in s["calls"]]
    assert calls and {c["fn"] for c in calls} <= set(used)
    for c in calls:
        sig = getattr(hpc_rl_utils, c["fn"]).__doc__.splitlines()[0]
        assert sig.count("arg") == 2 + len(c["scalars"]), (c["fn"], sig, c["scalars"])
