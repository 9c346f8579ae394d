#!/usr/bin/env python
"""Record how the UNMODIFIED reference wrappers (DI-hpc ``hpc_rll/rl_utils/*.py``) drive their native module.

DI-hpc's Python wrappers own no arithmetic: every ``nn.Module`` registers scratch buffers and every
``autograd.Function`` passes (input list, output list, scalars) to one ``hpc_rl_utils`` binding and returns
some of those buffers.  This script runs each wrapper once on the CPU with a recording stand-in for
``hpc_rl_utils`` and stores, per scenario of ``tests/test_legacy_shim_gpu.py``:

  calls    binding name, input / output tensor lists (a user input by name, or a buffer by id), scalars
  buffers  shape, dtype and initial fill of every tensor that is not a user input (module buffers, the
           default weights, the upstream gradients autograd hands to ``backward``)
  results  which output of which call the user receives (returned tensors, ``.grad`` of the inputs,
           ``.item()`` values)

plus the binding names ``src/rl_utils/entry.cpp`` exports and the names each wrapper file uses.  The
tests replay these calls on this repository's ``hpc_rl_utils`` shim, so they need no reference tree.
The wrappers' ``assert x.is_cuda`` lines are compiled out (``optimize=1``) so they run on the CPU.
Re-run with a DI-hpc checkout (nothing of it is copied into this repository):

    python tests/golden/make_wrapper_trace.py <DI-hpc checkout>
"""
import json
import os
import re
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "ref_wrapper_calls.json")
MODULES = ("gae", "td", "upgo", "vtrace", "ppo")


class Trace:
    """Identifies every tensor handed to a binding and marks each output with a distinct value, so that what the
    wrapper returns can be traced back to (call, output position)."""

    def __init__(self, inputs):
        self.inputs = inputs
        self.calls, self.buffers, self.keep = [], {}, []
        self.ids = {}

    def ref(self, t):
        for name, x in self.inputs.items():
            if x.data_ptr() == t.data_ptr() and x.shape == t.shape and x.dtype == t.dtype:
                return {"input": name}
        key = (t.data_ptr(), tuple(t.shape), t.dtype)
        if key not in self.ids:
            flat = t.detach().reshape(-1)
            if flat.numel() == 0 or not bool((flat == flat[0]).all()):
                raise RuntimeError("tensor %s passed to a binding is neither a user input nor constant" % (t.shape, ))
            self.ids[key] = len(self.buffers)
            self.buffers[len(self.buffers)] = {"shape": list(t.shape), "dtype": str(t.dtype).replace("torch.", ""),
                                               "fill": flat[0].item()}
            self.keep.append(t)  # no address reuse while recording
        return {"buffer": self.ids[key]}

    @staticmethod
    def marker(call, k):
        return -float(1 + 100 * call + k)

    def record(self, fn, args):
        ins, outs = args[0], args[1]
        self.calls.append({"fn": fn, "inputs": [self.ref(t) for t in ins], "outputs": [self.ref(t) for t in outs],
                           "scalars": list(args[2:])})
        for k, t in enumerate(outs):
            t.fill_(self.marker(len(self.calls) - 1, k))

    def locate(self, value):
        v = value if isinstance(value, float) else value.detach().reshape(-1)
        first = v if isinstance(v, float) else v[0].item()
        if not isinstance(v, float):
            assert bool((v == first).all()), "result is not one binding output"
        for c in range(len(self.calls)):
            for k in range(len(self.calls[c]["outputs"])):
                if first == self.marker(c, k):
                    return [c, k]
        raise RuntimeError("result %r is not a binding output" % first)


class Recorder(types.ModuleType):
    def __init__(self):
        super().__init__("hpc_rl_utils")
        self.trace = None

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)

        def call(*args):
            self.trace.record(name, args)
        return call


def load_wrappers(native, wrappers):
    sys.modules["hpc_rl_utils"] = native
    mods = {}
    for name in MODULES:
        path = os.path.join(wrappers, name + ".py")
        m = types.ModuleType("ref_wrapper_" + name)
        m.__file__ = path
        with open(path) as f:
            exec(compile(f.read(), path, "exec", optimize=1), m.__dict__)
        mods[name] = m
    return mods


def t32(g, *shape):
    return torch.from_numpy(g.standard_normal(shape, dtype=np.float32))


def idx(g, n, *shape):
    return torch.from_numpy(g.integers(0, n, shape).astype(np.int64))


def scenarios(W):
    """Shapes and calls of tests/test_legacy_shim_gpu.py::test_reference_wrappers_* (values are irrelevant: the
    wrappers never branch on data).  Each yields (name, wrapper module, inputs, run) with run() -> results."""
    g = np.random.default_rng(0)
    T, B = 1024, 64
    value, reward, weight = t32(g, T + 1, B), t32(g, T, B), t32(g, T, B)
    yield "gae", "gae", dict(value=value, reward=reward), lambda i: {"adv": W["gae"].GAE(T, B)(i["value"], i["reward"])}

    def td_lambda(i):
        loss = W["td"].TDLambda(T, B)(i["value"], i["reward"], i["weight"])
        loss.backward()
        return {"loss": loss, "grad_value": i["value"].grad}
    yield "td_lambda", "td", dict(value=value.clone().requires_grad_(True), reward=reward, weight=weight), td_lambda

    T, B, N = 64, 48, 16
    tgt, beh, act = t32(g, T, B, N), t32(g, T, B, N), idx(g, N, T, B)
    value, reward, rhos = t32(g, T + 1, B), t32(g, T, B), t32(g, T, B).abs()

    def vtrace(i):
        l = W["vtrace"].VTrace(T, B, N)(i["target_output"], i["behaviour_output"], i["action"], i["value"], i["reward"])
        (1.0 * l.policy_loss + 0.5 * l.value_loss - 0.25 * l.entropy_loss).sum().backward()
        return {"policy_loss": l.policy_loss, "value_loss": l.value_loss, "entropy_loss": l.entropy_loss,
                "grad_target_output": i["target_output"].grad, "grad_value": i["value"].grad}
    yield "vtrace", "vtrace", dict(target_output=tgt.clone().requires_grad_(True), behaviour_output=beh, action=act,
                                   value=value.clone().requires_grad_(True), reward=reward), vtrace

    def upgo(i):
        loss = W["upgo"].UPGO(T, B, N)(i["target_output"], i["rhos"], i["action"], i["reward"], i["value"])
        loss.sum().backward()
        return {"loss": loss, "grad_target_output": i["target_output"].grad}
    yield "upgo", "upgo", dict(target_output=tgt.clone().requires_grad_(True), rhos=rhos, action=act, reward=reward,
                               value=value), upgo

    Bp = 128

    def ppo(i):
        loss, info = W["ppo"].PPO(Bp, N)(i["logits_new"], i["logits_old"], i["action"], i["value_new"], i["value_old"],
                                         i["adv"], i["return"], None, 0.2, True, None)
        (loss.policy_loss + 0.5 * loss.value_loss - 0.01 * loss.entropy_loss).sum().backward()
        return {"policy_loss": loss.policy_loss, "value_loss": loss.value_loss, "entropy_loss": loss.entropy_loss,
                "approx_kl": info.approx_kl, "grad_logits_new": i["logits_new"].grad,
                "grad_value_new": i["value_new"].grad}
    yield "ppo", "ppo", dict(logits_new=t32(g, Bp, N).requires_grad_(True), logits_old=t32(g, Bp, N), action=idx(g, N, Bp),
                             value_new=t32(g, Bp).requires_grad_(True), value_old=t32(g, Bp), adv=t32(g, Bp),
                             **{"return": t32(g, Bp)}), ppo

    T, B, N = 10, 89, 7
    common = dict(action=idx(g, N, B), next_n_action=idx(g, N, B), reward=t32(g, T, B),
                  done=torch.from_numpy((g.random(B) < 0.3).astype(np.float32)), weight=t32(g, B).abs())

    def nstep(cls, *args):
        def run(i):
            loss, tde = cls(*args[0])(i["q"], i["next_n_q"], i["action"], i["next_n_action"], i["reward"], i["done"],
                                      *[i[a] if isinstance(a, str) else a for a in args[1]])
            loss.sum().backward()
            return {"loss": loss, "td_error_per_sample": tde, "grad_q": i["q"].grad}
        return run

    td = W["td"]
    for name, cls in (("q_nstep_td", td.QNStepTD), ("q_nstep_td_rescale", td.QNStepTDRescale)):
        yield name, "td", dict(q=t32(g, B, N).requires_grad_(True), next_n_q=t32(g, B, N), **common), \
            nstep(cls, (T, B, N), ("weight", 0.95))
    A = 51
    dist = torch.softmax(t32(g, B, N, A), -1)
    yield "dist_nstep_td", "td", dict(q=dist.requires_grad_(True), next_n_q=torch.softmax(t32(g, B, N, A), -1), **common), \
        nstep(td.DistNStepTD, (T, B, N, A), ("weight", 0.95, -10.0, 10.0))
    tau, tau_p = 39, 34
    yield "qrdqn_nstep_td", "td", dict(q=t32(g, B, N, tau).requires_grad_(True), next_n_q=t32(g, B, N, tau), **common), \
        nstep(td.QRDQNNStepTDError, (tau, T, B, N), (0.95, "weight"))
    yield "iqn_nstep_td", "td", dict(q=t32(g, tau, B, N).requires_grad_(True), next_n_q=t32(g, tau_p, B, N),
                                     replay_quantiles=t32(g, tau, B).abs(), **common), \
        nstep(td.IQNNStepTDError, (tau, tau_p, T, B, N), ("replay_quantiles", 0.95, 0.9, "weight"))


def main(ref_root):
    wrappers = os.path.join(ref_root, "hpc_rll", "rl_utils")
    native = Recorder()
    W = load_wrappers(native, wrappers)
    with open(os.path.join(ref_root, "src", "rl_utils", "entry.cpp")) as f:
        entry = sorted(re.findall(r'm\.def\("(\w+)"', f.read()))
    uses = {}
    for name in MODULES:
        with open(os.path.join(wrappers, name + ".py")) as f:
            uses[name] = sorted(set(re.findall(r"hpc_rl_utils\.(\w+)", f.read())))
    out = {"source": "DI-hpc @ a8a7734: src/rl_utils/entry.cpp and hpc_rll/rl_utils/{%s}.py" % ",".join(MODULES),
           "entry_cpp_bindings": entry, "wrapper_uses": uses, "scenarios": {}}
    for name, module, inputs, run in scenarios(W):
        native.trace = tr = Trace(inputs)
        res = run(inputs)
        out["scenarios"][name] = {
            "module": module,
            "inputs": {k: {"shape": list(v.shape), "dtype": str(v.dtype).replace("torch.", "")} for k, v in inputs.items()},
            "calls": tr.calls, "buffers": tr.buffers, "results": {k: tr.locate(v) for k, v in res.items()}}
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote %s (%d scenarios, %d calls)" % (OUT, len(out["scenarios"]),
                                                sum(len(s["calls"]) for s in out["scenarios"].values())))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: make_wrapper_trace.py <DI-hpc checkout>")
    main(sys.argv[1])
