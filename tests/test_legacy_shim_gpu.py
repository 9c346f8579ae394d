"""-m gpu: the reference's native boundary on the B200 kernels.

(a) `test_names_*`: each of the 19 hot-path `hpc_rl_utils` names called directly with tensor lists in the reference
    launchers' positional order (src/rl_utils/*.cu `index++`; buffers shaped as the reference modules register them),
    results compared with the oracle.
(b) `test_reference_wrappers_*`: the calls the UNMODIFIED reference wrappers (hpc_rll/rl_utils/*.py) make into their
    native module in forward + autograd backward (recorded in tests/golden/ref_wrapper_calls.json), issued on the shim
    and compared with the oracle -- what a DI-hpc user gets by swapping the extension.
"""
import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests import _refwrap
from tests._gpu import dev, host, need_cuda, rel_err, rng

pytestmark = pytest.mark.gpu
TOL = 1e-5


def close(got, want, what):
    e = rel_err(got, want)
    assert e <= TOL, "%s: rel err %.3e" % (what, e)


def z(*s):
    return torch.zeros(*s, device="cuda")


def one():
    return torch.ones(1, device="cuda")


def scan_inputs(g, T, B):
    return (g.standard_normal((T + 1, B), dtype=np.float32), g.standard_normal((T, B), dtype=np.float32),
            g.random((T, B), dtype=np.float32))


def nstep_inputs(g, T, B, N):
    return dict(action=g.integers(0, N, (B, )).astype(np.int64), next_n_action=g.integers(0, N, (B, )).astype(np.int64),
                reward=g.standard_normal((T, B), dtype=np.float32), done=(g.random(B) < 0.3).astype(np.float32),
                weight=g.random(B).astype(np.float32))


# ------------------------------------------------------------------------------------------------ (a) direct calls
def test_names_gae_and_td_lambda():
    need_cuda()
    import hpc_rl_utils as H
    T, B = 33, 260
    value, reward, weight = scan_inputs(rng(1), T, B)
    adv = z(T, B)
    H.GaeForward([dev(value), dev(reward)], [adv], 0.99, 0.97)
    close(host(adv), orc.gae_forward(value, reward, np.float32(0.99), np.float32(0.97)), "adv")
    loss, gbuf, gval = z(1), z(T, B), z(T + 1, B)
    H.TdLambdaForward([dev(value), dev(reward), dev(weight)], [loss, gbuf], 0.9, 0.8)
    H.TdLambdaBackward([one() * 1.7, gbuf], [gval])
    o = orc.td_lambda(value, reward, weight, np.float32(0.9), np.float32(0.8), 1.7)
    close(float(loss.item()), o["loss"], "loss")
    close(host(gval) * T * B, o["grad_value"] * T * B, "grad_value")
    # the reference module's default weight is ones(B) (rl_utils/td.py:160): broadcast, not read out of bounds
    H.TdLambdaForward([dev(value), dev(reward), torch.ones(B, device="cuda")], [loss, gbuf], 0.9, 0.8)
    close(float(loss.item()), orc.td_lambda(value, reward, None, np.float32(0.9), np.float32(0.8))["loss"], "loss (B,)")


@pytest.mark.parametrize("rescale", [False, True])
def test_names_q_nstep(rescale):
    need_cuda()
    import hpc_rl_utils as H
    T, B, N = 5, 300, 6
    g = rng(2 + rescale)
    inp = nstep_inputs(g, T, B, N)
    q, nq = g.standard_normal((B, N), dtype=np.float32), g.standard_normal((B, N), dtype=np.float32)
    td, loss, gbuf, gq = z(B), z(1), z(B), z(B, N)
    fwd, bwd = (H.QNStepTdRescaleForward, H.QNStepTdRescaleBackward) if rescale else (H.QNStepTdForward, H.QNStepTdBackward)
    fwd([dev(q), dev(nq), dev(inp["action"]), dev(inp["next_n_action"]), dev(inp["reward"]), dev(inp["done"]),
         dev(inp["weight"])], [td, loss, gbuf], 0.95)
    bwd([one() * 1.3, gbuf, dev(inp["action"])], [gq])
    o = orc.q_nstep_td(q, nq, inp["action"], inp["next_n_action"], inp["reward"], inp["done"], inp["weight"],
                       np.float32(0.95), rescale, 1.3)
    close(float(loss.item()), o["loss"], "loss")
    close(host(td), o["td_error_per_sample"], "td")
    close(host(gq) * B, o["grad_q"] * B, "grad_q")
    assert np.array_equal(host(gq) != 0, o["grad_q"] != 0)


def test_names_dist_nstep():
    need_cuda()
    import hpc_rl_utils as H
    T, B, N, A = 3, 200, 4, 51
    g = rng(4)
    inp = nstep_inputs(g, T, B, N)
    sm = lambda x: (np.exp(x) / np.exp(x).sum(-1, keepdims=True)).astype(np.float32)  # noqa: E731
    dist, ndist = sm(g.standard_normal((B, N, A))), sm(g.standard_normal((B, N, A)))
    td, loss, buf, gd = z(B), z(1), z(B + B * A), z(B, N, A)
    H.DistNStepTdForward([dev(dist), dev(ndist), dev(inp["action"]), dev(inp["next_n_action"]), dev(inp["reward"]),
                          dev(inp["done"]), dev(inp["weight"])], [td, loss, buf], 0.95, -10.0, 10.0)
    H.DistNStepTdBackward([one() * 0.9, buf, dev(inp["action"])], [gd])
    o = orc.dist_nstep_td(dist, ndist, inp["action"], inp["next_n_action"], inp["reward"], inp["done"], inp["weight"],
                          np.float32(0.95), -10.0, 10.0, 0.9)
    close(float(loss.item()), o["loss"], "loss")
    close(host(td), o["td_error_per_sample"], "td")
    close(host(gd) * B, o["grad_dist"] * B, "grad_dist")


def test_names_qrdqn_and_iqn():
    need_cuda()
    import hpc_rl_utils as H
    tau, tau_p, T, B, N = 39, 34, 10, 89, 7
    g = rng(5)
    inp = nstep_inputs(g, T, B, N)
    vg = g.random(B).astype(np.float32)
    q, nq = g.standard_normal((B, N, tau), dtype=np.float32), g.standard_normal((B, N, tau), dtype=np.float32)
    loss, td, gbuf, gq = z(1), z(B), z(B, tau), z(B, N, tau)  # grad_buf (B,tau): the reference's own (too small) shape
    H.QRDQNNStepTDErrorForward([dev(q), dev(nq), dev(inp["action"]), dev(inp["next_n_action"]), dev(inp["reward"]),
                                dev(inp["done"]), dev(inp["weight"]), dev(vg)],
                               [loss, td, z(B, tau, tau), z(B, tau, tau), gbuf], 0.95)
    H.QRDQNNStepTDErrorBackward([one() * 1.1, gbuf, dev(inp["weight"]), dev(inp["action"])], [gq])
    o = orc.qrdqn_nstep_td(q, nq, inp["action"], inp["next_n_action"], inp["reward"], inp["done"], inp["weight"], vg,
                           np.float32(0.95), 1.1)
    close(float(loss.item()), o["loss"], "qrdqn loss")
    close(host(td), o["td_error_per_sample"], "qrdqn td")
    close(host(gq) * B, o["grad_q"] * B, "qrdqn grad_q")
    qi, nqi = g.standard_normal((tau, B, N), dtype=np.float32), g.standard_normal((tau_p, B, N), dtype=np.float32)
    rq = g.random((tau, B)).astype(np.float32)
    gbuf, gqi = z(B, tau_p, tau), z(tau, B, N)
    H.IQNNStepTDErrorForward([dev(qi), dev(nqi), dev(inp["action"]), dev(inp["next_n_action"]), dev(inp["reward"]),
                              dev(inp["done"]), dev(rq), dev(inp["weight"]), dev(vg)],
                             [loss, td, z(B, tau_p, tau), z(B, tau_p, tau), gbuf], 0.95, 0.9)
    H.IQNNStepTDErrorBackward([one() * 0.8, gbuf, dev(inp["weight"]), dev(inp["action"])], [gqi])
    o = orc.iqn_nstep_td(qi, nqi, inp["action"], inp["next_n_action"], inp["reward"], inp["done"], rq, inp["weight"], vg,
                         np.float32(0.95), np.float32(0.9), 0.8)
    close(float(loss.item()), o["loss"], "iqn loss")
    close(host(td), o["td_error_per_sample"], "iqn td")
    close(host(gqi) * B, o["grad_q"] * B, "iqn grad_q")


def test_names_upgo_vtrace_ppo():
    need_cuda()
    import hpc_rl_utils as H
    T, B, N = 12, 70, 18
    g = rng(6)
    value, reward, weight = scan_inputs(g, T, B)
    tgt = (g.standard_normal((T, B, N)) * 1.5).astype(np.float32)
    beh = (g.standard_normal((T, B, N)) * 1.5).astype(np.float32)
    act = g.integers(0, N, (T, B)).astype(np.int64)
    rhos = (g.random((T, B)) * 2).astype(np.float32)
    # ---- upgo
    advb, metric, loss, gbuf, gt = z(T, B), z(T, B), z(1), z(T, B, N), z(T, B, N)
    H.UpgoForward([dev(tgt), dev(rhos), dev(act), dev(reward), dev(value)], [advb, metric, loss, gbuf])
    H.UpgoBackward([one() * -0.7, gbuf, advb], [gt])
    o = orc.upgo(tgt, rhos, act, reward, value, -0.7)
    close(float(loss.item()), o["loss"], "upgo loss")
    close(host(gt) * T * B, o["grad_target_output"] * T * B, "upgo grad")
    # ---- vtrace: 12 forward outputs in vtrace.cu:26-37 order, 11 backward inputs in vtrace.cu:93-103 order
    outs = [z(T, B), z(T, B), z(T, B, N), z(T, B, N), z(T, B, N), z(T, B), z(T, B), z(T, B), z(T, B), z(1), z(1), z(1)]
    H.VTraceForward([dev(tgt), dev(beh), dev(act), dev(value), dev(reward), dev(weight)], outs, 0.9, 0.8, 1.5, 0.9, 2.0)
    gv, gtt = z(T + 1, B), z(T, B, N)
    coef = [1.0, 0.5, -0.25]
    H.VTraceBackward([one() * coef[0], one() * coef[1], one() * coef[2], dev(value), dev(act), dev(weight), outs[7],
                      outs[8], outs[2], outs[3], outs[4]], [gv, gtt])
    o = orc.vtrace(tgt, beh, act, value, reward, weight, np.float32(0.9), np.float32(0.8), np.float32(1.5),
                   np.float32(0.9), np.float32(2.0), coef)
    for k, nm in enumerate(("policy_loss", "value_loss", "entropy_loss")):
        close(float(outs[9 + k].item()), o[nm], "vtrace " + nm)
    close(host(gtt) * T * B, o["grad_target_output"] * T * B, "vtrace grad_target_output")
    close(host(gv) * T * B, o["grad_value"] * T * B, "vtrace grad_value")
    # ---- ppo: 14 outputs in ppo.cu:26-39 order, 9 backward inputs in ppo.cu:80-88 order
    Bp = 257
    lo = g.standard_normal((Bp, N)).astype(np.float32)
    ln = (lo + 0.3 * g.standard_normal((Bp, N))).astype(np.float32)
    a = g.integers(0, N, (Bp, )).astype(np.int64)
    vn, vo, adv, ret, w = (g.standard_normal(Bp).astype(np.float32) for _ in range(5))
    w = np.abs(w)
    outs = [z(Bp), z(Bp), z(Bp, N), z(Bp, N), z(Bp, N), z(Bp), z(Bp), z(Bp), z(Bp), z(1), z(1), z(1), z(1), z(1)]
    for dual_ref, dual in ((3.0, 3.0), (0.0, None)):  # the reference wrapper encodes None as 0.0 (rl_utils/ppo.py:136)
        H.PPOForward([dev(ln), dev(lo), dev(a), dev(vn), dev(vo), dev(adv), dev(ret), dev(w)], outs, True, 0.2, dual_ref)
        gval, glog = z(Bp), z(Bp, N)
        c3 = [1.0, 0.5, -0.01]
        H.PPOBackward([one() * c3[0], one() * c3[1], one() * c3[2], outs[6], outs[7], outs[8], outs[2], outs[3], outs[4]],
                      [gval, glog])
        o = orc.ppo(ln, lo, a, vn, vo, adv, ret, w, np.float32(0.2), True, dual, c3)
        for k, nm in enumerate(("policy_loss", "value_loss", "entropy_loss", "approx_kl")):
            close(float(outs[9 + k].item()), o[nm], "ppo " + nm)
        assert abs(float(outs[13].item()) - o["clipfrac"]) <= 2.0 / Bp
        close(host(glog) * Bp, o["grad_logits_new"] * Bp, "ppo grad_logits_new")
        close(host(gval) * Bp, o["grad_value_new"] * Bp, "ppo grad_value_new")


# ------------------------------------------------------------------------------------------------ (b) reference wrappers
def _replay(name, **inputs):
    """the calls the unmodified reference wrapper makes in scenario `name`, issued on the shim (tests/_refwrap.py)"""
    need_cuda()
    import hpc_rl_utils
    return _refwrap.replay(name, inputs, hpc_rl_utils)


def test_reference_wrappers_gae_tdlambda():
    g = rng(11)
    T, B = 1024, 64  # tests/test_gae.py:10-11, tests/test_tdlambda.py:10-11
    value, reward, weight = scan_inputs(g, T, B)
    adv = _replay("gae", value=dev(value), reward=dev(reward))["adv"]
    close(host(adv), orc.gae_forward(value, reward, np.float32(0.99), np.float32(0.97)), "adv")
    r = _replay("td_lambda", value=dev(value), reward=dev(reward), weight=dev(weight))
    o = orc.td_lambda(value, reward, weight, np.float32(0.9), np.float32(0.8))
    close(float(r["loss"].item()), o["loss"], "loss")
    close(host(r["grad_value"]) * T * B, o["grad_value"] * T * B, "grad_value")


def test_reference_wrappers_vtrace_upgo_ppo():
    g = rng(12)
    T, B, N = 64, 48, 16
    value, reward, weight = scan_inputs(g, T, B)
    tgt = (g.standard_normal((T, B, N)) * 1.5).astype(np.float32)
    beh = (g.standard_normal((T, B, N)) * 1.5).astype(np.float32)
    act = g.integers(0, N, (T, B)).astype(np.int64)
    # weight None -> module ones; upstream gradients 1, 0.5, -0.25 of the three losses
    r = _replay("vtrace", target_output=dev(tgt), behaviour_output=dev(beh), action=dev(act), value=dev(value),
                reward=dev(reward))
    coef = [1.0, 0.5, -0.25]
    o = orc.vtrace(tgt, beh, act, value, reward, None, coef=coef)
    for nm in ("policy_loss", "value_loss", "entropy_loss"):
        close(float(r[nm].item()), o[nm], nm)
    close(host(r["grad_target_output"]) * T * B, o["grad_target_output"] * T * B, "vtrace grad_target_output")
    close(host(r["grad_value"]) * T * B, o["grad_value"] * T * B, "vtrace grad_value")
    rhos = (g.random((T, B)) * 2).astype(np.float32)
    r = _replay("upgo", target_output=dev(tgt), rhos=dev(rhos), action=dev(act), reward=dev(reward), value=dev(value))
    o = orc.upgo(tgt, rhos, act, reward, value)
    close(float(r["loss"].item()), o["loss"], "upgo loss")
    close(host(r["grad_target_output"]) * T * B, o["grad_target_output"] * T * B, "upgo grad")
    Bp = 128  # tests/test_ppo.py:11-12
    lo = g.standard_normal((Bp, N)).astype(np.float32)
    ln = (lo + 0.3 * g.standard_normal((Bp, N))).astype(np.float32)
    a = g.integers(0, N, (Bp, )).astype(np.int64)
    vn, vo, adv, ret = (g.standard_normal(Bp).astype(np.float32) for _ in range(4))
    # weight None, clip 0.2, value clip on, dual clip None; loss = policy + 0.5 value - 0.01 entropy
    r = _replay("ppo", logits_new=dev(ln), logits_old=dev(lo), action=dev(a), value_new=dev(vn), value_old=dev(vo),
                adv=dev(adv), **{"return": dev(ret)})
    o = orc.ppo(ln, lo, a, vn, vo, adv, ret, None, 0.2, True, None, [1.0, 0.5, -0.01])
    for nm in ("policy_loss", "value_loss", "entropy_loss"):
        close(float(r[nm].item()), o[nm], "ppo " + nm)
    close(float(r["approx_kl"].item()), o["approx_kl"], "approx_kl")
    close(host(r["grad_logits_new"]) * Bp, o["grad_logits_new"] * Bp, "ppo grad_logits_new")
    close(host(r["grad_value_new"]) * Bp, o["grad_value_new"] * Bp, "ppo grad_value_new")


def test_reference_wrappers_nstep_family():
    g = rng(13)
    T, B, N = 10, 89, 7
    inp = nstep_inputs(g, T, B, N)
    dv = {k: dev(v) for k, v in inp.items()}
    for rescale, name in ((False, "q_nstep_td"), (True, "q_nstep_td_rescale")):  # gamma 0.95
        q, nq = g.standard_normal((B, N), dtype=np.float32), g.standard_normal((B, N), dtype=np.float32)
        r = _replay(name, q=dev(q), next_n_q=dev(nq), **dv)
        o = orc.q_nstep_td(q, nq, inp["action"], inp["next_n_action"], inp["reward"], inp["done"], inp["weight"],
                           np.float32(0.95), rescale)
        close(float(r["loss"].item()), o["loss"], "q loss")
        close(host(r["td_error_per_sample"]), o["td_error_per_sample"], "q td")
        close(host(r["grad_q"]) * B, o["grad_q"] * B, "grad_q")
    A = 51
    sm = lambda x: (np.exp(x) / np.exp(x).sum(-1, keepdims=True)).astype(np.float32)  # noqa: E731
    dist, ndist = sm(g.standard_normal((B, N, A))), sm(g.standard_normal((B, N, A)))
    r = _replay("dist_nstep_td", q=dev(dist), next_n_q=dev(ndist), **dv)  # gamma 0.95, support [-10, 10]
    o = orc.dist_nstep_td(dist, ndist, inp["action"], inp["next_n_action"], inp["reward"], inp["done"], inp["weight"],
                          np.float32(0.95), -10.0, 10.0)
    close(float(r["loss"].item()), o["loss"], "dist loss")
    close(host(r["grad_q"]) * B, o["grad_dist"] * B, "grad_dist")
    tau, tau_p = 39, 34  # tests/test_qrdqn_nstep_td_error.py:10-14
    q, nq = g.standard_normal((B, N, tau), dtype=np.float32), g.standard_normal((B, N, tau), dtype=np.float32)
    r = _replay("qrdqn_nstep_td", q=dev(q), next_n_q=dev(nq), **dv)  # gamma 0.95, value_gamma None
    o = orc.qrdqn_nstep_td(q, nq, inp["action"], inp["next_n_action"], inp["reward"], inp["done"], inp["weight"], None,
                           np.float32(0.95))
    close(float(r["loss"].item()), o["loss"], "qrdqn loss")
    close(host(r["td_error_per_sample"]), o["td_error_per_sample"], "qrdqn td")
    close(host(r["grad_q"]) * B, o["grad_q"] * B, "qrdqn grad_q")
    qi, nqi = g.standard_normal((tau, B, N), dtype=np.float32), g.standard_normal((tau_p, B, N), dtype=np.float32)
    rq = g.random((tau, B)).astype(np.float32)
    r = _replay("iqn_nstep_td", q=dev(qi), next_n_q=dev(nqi), replay_quantiles=dev(rq), **dv)  # gamma 0.95, kappa 0.9
    o = orc.iqn_nstep_td(qi, nqi, inp["action"], inp["next_n_action"], inp["reward"], inp["done"], rq, inp["weight"], None,
                         np.float32(0.95), np.float32(0.9))
    close(float(r["loss"].item()), o["loss"], "iqn loss")
    close(host(r["td_error_per_sample"]), o["td_error_per_sample"], "iqn td")
    close(host(r["grad_q"]) * B, o["grad_q"] * B, "iqn grad_q")
