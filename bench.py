#!/usr/bin/env python
"""bench.py -- headline benchmark of the trajectory-return hot path on B200.

Metric (BASELINE.json): GAE forward+backward trajectory-steps/s at 1/2/4/8 B200, plus % of the HBM roofline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one GAE forward + one GAE adjoint over one batch of synthetic trajectories (T=1024, B=65536 per GPU,
fp32 -- BASELINE.json configs[1]) through the API north_star names: `hpc_rll.rl_utils.gae.GAE(T, B)(value, reward)`
followed by `torch.autograd.grad(adv, [value, reward], grad_adv)`.  With N GPUs every rank holds its own B=65536
shard (global batch N*65536, no data-path collective => weak scaling).

  value         whole-job steps/s, inputs resident in HBM: CUDA events around exactly K queued steps, barrier +
                synchronize on both sides, max over ranks
  module        the same step timed per call (synchronise after each) and through the raw C ABI (no autograd)
  roofline      dominant kernel's algorithmic bytes / its mean CUDA-event duration vs the measured HBM peak
  e2e           same metric through `di_hpc_b200.host.gae_fwd_bwd_host`: page-locked HOST tensors in, host tensors
                out, H2D/D2H copies inside the timed region (T-chunked carry pipeline; buffers on the GPU's NUMA node)
  ops           (N=1) the other BASELINE configs through their modules: V-trace + UPGO at C2 (T=512, B=32768, N=16),
                QR-DQN + IQN at C3 (B=1M, tau=64, N=8, nstep=5): ms, units/s, algorithmic GB/s, fraction of the bound
  c4            BASELINE configs[4] verbatim: GAE T=1024, global B=524288 sharded over the N ranks (B_local=524288/N),
                plus the NCCL scatter of the (T,B_local) slices from rank 0 as its own figure
  loss_allreduce (N>1) TD(lambda) fwd+bwd on the local shard with the scalar loss all-reduced (the only collective
                the path has): ms with and without it
  cpu_baseline  the oracle port (oracle/oracle.c, OpenMP) on this box's host cores, same workload

`--impl reference` times the CPU implementation (the oracle port: the reference's own CPU path is the Python/PyTorch
`hpc_rll.origin`, which does not exist on the GPU box) on the same config.

`--dump-outputs DIR` writes what the last timed step returned to its caller (adv, grad_value, grad_reward) as
DIR/<name>.npy, float32, restricted to a fixed seeded sample of columns (at most 16 MB per output).  The inputs are
seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

T_DEFAULT, B_DEFAULT = 1024, 65536
C4_GLOBAL_B = 524288
GAMMA, LAMBDA = 0.99, 0.97
OUT = sys.stdout
METRIC = "gae_fwd_bwd_trajectory_steps_per_sec"
UNIT = "steps/s"
# hpc_rll.origin.gae (the reference's actual CPU path) on this exact workload, measured in the BUILD container
# (8-core Xeon, torch 2.11 CPU; BASELINE.md section 4): it cannot run on the GPU box (no /root/reference there)
ORIGIN_CONTEXT = {"what": "hpc_rll.origin.gae T=1024 B=65536 fp32 on the build container's 8 host cores "
                          "(BASELINE.md sec. 4; not on this box)",
                  "forward_s": 0.72, "forward_backward_s": 148.7, "steps_per_s_fwd_bwd": 1024 * 65536 / 148.7,
                  "note": "origin's autograd backward is O(T^2 B) (origin/gae.py:36 in-place adds)"}


def workload_name(T, B):
    return "gae_fwd_bwd T=%d B=%d fp32 per GPU (BASELINE.json configs[1])" % (T, B)


def config_of(T, B, world):
    """identical in both arms (the driver's same_config check compares them)"""
    return {"workload": workload_name(T, B), "global_B": B * world, "gamma": GAMMA, "lambda": LAMBDA,
            "l2": "inputs (%.0f MB per kernel) larger than L2 (126 MB); no flush needed" % ((12 * T * B + 4 * B) / 1e6)}


def algorithmic_bytes(T, B):
    """SURVEY.md 8(d): 12 B/step forward (v, r in; adv out) + 12 B/step backward (G in; g_r, g_v out)
    + one extra (B,) row each for value[T] / grad_value[T]."""
    fwd = 12 * T * B + 4 * B
    bwd = 12 * T * B + 4 * B
    return fwd, bwd


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            with open(p) as f:
                return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled while the GPU is under load."""
    FIELDS = ("clocks.sm,clocks.max.sm,utilization.gpu,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                clk, mx, util = float(parts[0]), float(parts[1]), float(parts[2])
            except ValueError:
                continue
            smax = mx
            if util >= 20.0:
                sm.append(clk)
                for n, v in zip(names, parts[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples_under_load": len(sm)}


def cpu_baseline(T, B, reps):
    """Oracle port (C + OpenMP) on the same workload: fwd + adjoint.  The thread count is probed (all host
    threads, then fewer) and the fastest is reported with the threads it actually used."""
    import numpy as np
    from oracle import oracle as orc
    orc.build()
    ncpu = os.cpu_count() or 1
    try:
        ncpu = min(ncpu, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    rng = np.random.default_rng(1234)
    src = [rng.standard_normal((T + 1, B), dtype=np.float32), rng.standard_normal((T, B), dtype=np.float32),
           rng.standard_normal((T, B), dtype=np.float32)]

    def run(nthreads, n):
        orc.set_threads(nthreads)
        # parallel first-touch with this thread count so each thread streams pages local to its NUMA node
        value, reward, gadv = (orc.place(a) for a in src)
        orc.gae_forward(value, reward, GAMMA, LAMBDA)
        orc.gae_backward(gadv, GAMMA, LAMBDA)
        ts = []
        for _ in range(n):
            t0 = time.perf_counter()
            orc.gae_forward(value, reward, GAMMA, LAMBDA)
            orc.gae_backward(gadv, GAMMA, LAMBDA)
            ts.append(time.perf_counter() - t0)
        ts.sort()
        return ts[len(ts) // 2]

    cands = sorted({c for c in (ncpu, ncpu // 2, ncpu // 4, 32, 16, 8) if 1 <= c <= ncpu}, reverse=True)
    probe = {c: run(c, 2) for c in cands}
    best = min(probe, key=probe.get)
    med = run(best, reps)
    return {"value": T * B / med, "unit": UNIT, "cores": best, "kind": "port",
            "sample": "full workload T=%d B=%d fp32 fwd+adjoint, median of %d runs (%.1f ms each), "
                      "oracle/oracle.c OpenMP, best of thread counts %s (host has %d)"
                      % (T, B, reps, med * 1e3, {k: round(v * 1e3, 1) for k, v in probe.items()}, ncpu),
            "reference_origin_context": ORIGIN_CONTEXT}, med


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    T, B = args.T, args.B
    base, med = cpu_baseline(T, B, max(3, args.steps))
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": med * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_of(T, B, max(1, args.gpus)),
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), file=OUT, flush=True)


# --------------------------------------------------------------------------------------------------- helpers (ours)
def event_ms(torch, fn, iters):
    """mean ms of fn() over `iters` queued calls (CUDA events on the current stream, synchronised both sides)"""
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def kernel_ms(torch, fn, min_iters, min_ms=300.0):
    iters = min_iters
    while True:
        t = event_ms(torch, fn, iters) * iters
        if t >= min_ms or iters >= 1 << 16:
            return t / iters
        iters *= 4


def ops_block(torch, peak):
    """BASELINE configs[2] and [3] through the drop-in modules (forward + autograd backward), queued calls between
    CUDA events.  Algorithmic bytes: SURVEY.md 8(d).  QR-DQN / IQN are bounded by the FP32 pipes, not HBM: their
    `frac` is against the HBM bound all the same (bytes that must move / time / peak), `bound` names the real limiter."""
    from hpc_rll.rl_utils.td import IQNNStepTDError, QRDQNNStepTDError
    from hpc_rll.rl_utils.upgo import UPGO
    from hpc_rll.rl_utils.vtrace import VTrace
    dev = "cuda"
    one = torch.ones(1, device=dev)
    out = {}

    def measure(name, step, units, unit_name, alg_bytes, bound, config, iters=10):
        for _ in range(3):
            step()
        ms = min(event_ms(torch, step, iters) for _ in range(2))
        gbs = alg_bytes / (ms * 1e-3) / 1e9
        out[name] = {"config": config, "ms": ms, "value": units / (ms * 1e-3), "unit": unit_name,
                     "algorithmic_gbs": gbs, "frac_of_hbm_peak": gbs / peak, "bound": bound,
                     "api": "hpc_rll.rl_utils module forward + torch.autograd.grad"}

    # ---- C2: V-trace + UPGO, T=512, B=32768, N=16
    T, B, N = 512, 32768, 16
    g = torch.Generator(device=dev).manual_seed(7)
    tgt = torch.randn(T, B, N, device=dev, generator=g).requires_grad_(True)
    beh = torch.randn(T, B, N, device=dev, generator=g)
    act = torch.randint(0, N, (T, B), device=dev, generator=g)
    val = torch.randn(T + 1, B, device=dev, generator=g).requires_grad_(True)
    rew = torch.randn(T, B, device=dev, generator=g)
    rho = torch.rand(T, B, device=dev, generator=g) * 2
    vt, up = VTrace(T, B, N), UPGO(T, B, N)

    def vtrace_step():
        l = vt(tgt, beh, act, val, rew)
        torch.autograd.grad(l.policy_loss + 0.5 * l.value_loss - 0.01 * l.entropy_loss, [tgt, val], grad_outputs=one)

    def upgo_step():
        torch.autograd.grad(up(tgt, rho, act, rew, val.detach()), [tgt], grad_outputs=one)

    cfg2 = "T=%d B=%d N=%d fp32 (BASELINE.json configs[2])" % (T, B, N)
    measure("vtrace", vtrace_step, T * B, "steps/s", (16 * N + 52) * T * B, "hbm", cfg2)
    measure("upgo", upgo_step, T * B, "steps/s", (12 * N + 36) * T * B, "hbm", cfg2)
    del tgt, beh, act, val, rew, rho
    torch.cuda.empty_cache()

    # ---- C3: QR-DQN + IQN, B=1M, tau=tau'=64, N=8, nstep=5
    B, N, tau, nstep = 1 << 20, 8, 64, 5
    a = torch.randint(0, N, (B, ), device=dev, generator=g)
    na = torch.randint(0, N, (B, ), device=dev, generator=g)
    r = torch.randn(nstep, B, device=dev, generator=g)
    done = (torch.rand(B, device=dev, generator=g) < 0.1).float()
    w = torch.rand(B, device=dev, generator=g)
    q = torch.randn(B, N, tau, device=dev, generator=g).requires_grad_(True)
    nq = torch.randn(B, N, tau, device=dev, generator=g)
    qr = QRDQNNStepTDError(tau, nstep, B, N)

    def qrdqn_step():
        loss, _ = qr(q, nq, a, na, r, done, 0.99, w)
        torch.autograd.grad(loss, [q], grad_outputs=one)

    cfg3 = "B=%d tau=%d N=%d nstep=%d fp32 (BASELINE.json configs[3])" % (B, tau, N, nstep)
    measure("qrdqn_nstep_td_error", qrdqn_step, B, "samples/s", (8 * tau + 4 * N * tau + 4 * nstep + 32) * B,
            "instruction issue (sorted O(tau log tau) evaluation; 718 warp instructions per sample)", cfg3)
    del q, nq
    torch.cuda.empty_cache()
    qi = torch.randn(tau, B, N, device=dev, generator=g).requires_grad_(True)
    nqi = torch.randn(tau, B, N, device=dev, generator=g)
    rq = torch.rand(tau, B, device=dev, generator=g)
    iq = IQNNStepTDError(tau, tau, nstep, B, N)

    def iqn_step():
        loss, _ = iq(qi, nqi, a, na, r, done, rq, 0.99, 1.0, w)
        torch.autograd.grad(loss, [qi], grad_outputs=one)

    measure("iqn_nstep_td_error", iqn_step, B, "samples/s", (12 * N * tau + 4 * tau + 50) * B,
            "hbm + instruction issue (strided gathers touch every sector of q)", cfg3)
    del qi, nqi, rq
    torch.cuda.empty_cache()
    return out


def dump_outputs(out_dir, outputs, B, suffix=""):
    """Write the last timed step's outputs as out_dir/<name><suffix>.npy (float32).  Every output is (rows, B); a full
    one is 268 MB at the default size, so a fixed sample of whole columns (complete trajectories) is kept: the same
    seeded choice of columns in every output and every run, at most 2^22 elements (16 MB) per output."""
    import numpy as np
    import torch
    rows = max(t.shape[0] for t in outputs.values())
    ncols = min(B, max(1, (1 << 22) // rows))
    cols = np.sort(np.random.default_rng(0).choice(B, size=ncols, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        idx = torch.from_numpy(cols).to(t.device)
        a = t.detach().index_select(1, idx).float().cpu().numpy()
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)


def run_ours(args):
    import torch
    from di_hpc_b200 import _abi
    from di_hpc_b200 import host as hostapi
    from hpc_rll.rl_utils.gae import GAE

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback exists)"
    torch.cuda.set_device(local)
    # host placement for the e2e path: this rank's threads and page-locked buffers on the GPU's NUMA node
    numa_node = hostapi.bind_to_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29531")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    T, B = args.T, args.B  # per-GPU shard (weak scaling)
    K, W = args.steps, max(3, args.warmup)
    L = _abi.lib()
    dev = torch.device("cuda", local)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    value = torch.randn(T + 1, B, device=dev, generator=gen).requires_grad_(True)
    reward = torch.randn(T, B, device=dev, generator=gen).requires_grad_(True)
    gadv = torch.randn(T, B, device=dev, generator=gen)
    gae = GAE(T, B)

    def step():  # the API north_star names: module forward + autograd backward -> what its caller receives
        adv = gae(value, reward, GAMMA, LAMBDA)
        grad_value, grad_reward = torch.autograd.grad(adv, [value, reward], grad_outputs=gadv)
        return {"adv": adv, "grad_value": grad_value, "grad_reward": grad_reward}

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x, dtype=torch.float32):
        t = torch.tensor([x], device=dev, dtype=dtype)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    # each step's outputs are held until the next step returns, in warm-up as in the timed loop, so that the
    # allocator already holds both sets of output buffers when the timing starts
    for _ in range(W):
        last = step()
    # ---- timed region: exactly K steps ------------------------------------------------------
    barrier()
    n0 = _abi.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        last = step()
    e1.record()
    barrier()
    launches = _abi.launch_count() - n0
    ms_per_step = max_over_ranks(e0.elapsed_time(e1)) / K
    value_metric = T * B * world / (ms_per_step * 1e-3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last, B, "" if world == 1 else "_rank%d" % rank)
    del last

    # ---- the same step per call (synchronise after each) and through the raw C ABI (no autograd, no allocation) ----
    per_call = []
    for _ in range(min(K, 20)):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step()
        b.record()
        torch.cuda.synchronize()
        per_call.append(a.elapsed_time(b))
    per_call.sort()
    adv_b, gv_b, gr_b = torch.empty(T, B, device=dev), torch.empty(T + 1, B, device=dev), torch.empty(T, B, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    pv, pr, pg, pa, pgv, pgr = (t.data_ptr() for t in (value, reward, gadv, adv_b, gv_b, gr_b))

    def fwd():
        _abi.check(L.hpc_rll_gae_forward(pv, pr, pa, T, B, GAMMA, LAMBDA, st), "gae_forward")

    def bwd():
        _abi.check(L.hpc_rll_gae_backward(pg, pgv, pgr, T, B, GAMMA, LAMBDA, st), "gae_backward")

    def raw_step():
        fwd()
        bwd()

    raw_ms = event_ms(torch, raw_step, max(K, 20))
    fwd_b, bwd_b = algorithmic_bytes(T, B)
    peak, peak_src = hbm_peak()
    module = {"api": "hpc_rll.rl_utils.gae.GAE.forward + torch.autograd.grad (C++ autograd binding: %s)"
                     % ("yes" if __import__("di_hpc_b200._ext", fromlist=["x"]).fast() is not None else "no, ctypes"),
              "queued_ms_per_step": ms_per_step,
              "queued_frac_of_hbm_peak": (fwd_b + bwd_b) / (ms_per_step * 1e-3) / 1e9 / peak,
              "per_call_ms_median": per_call[len(per_call) // 2],
              "per_call_frac_of_hbm_peak": (fwd_b + bwd_b) / (per_call[len(per_call) // 2] * 1e-3) / 1e9 / peak,
              "raw_c_abi_ms_per_step": raw_ms}

    # ---- roofline: each kernel alone, mean CUDA-event duration on the launching stream --------
    fwd_ms = kernel_ms(torch, fwd, max(K, 20))
    bwd_ms = kernel_ms(torch, bwd, max(K, 20))
    # kernel the library picks at this width (gae.cu pick_cfg): bulk-store output from 256 columns per SM up
    stg = "_st" if B >= 256 * torch.cuda.get_device_properties(dev).multi_processor_count and \
        "HPC_RLL_CFG_GAE" not in os.environ else ""
    dom = ("gae_bwd_tma" if bwd_ms >= fwd_ms else "gae_fwd_tma") + stg
    dom_ms, dom_b = (bwd_ms, bwd_b) if bwd_ms >= fwd_ms else (fwd_ms, fwd_b)
    achieved = dom_b / (dom_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "kernel": dom, "peak_source": peak_src,
                "fwd": {"ms": fwd_ms, "gbs": fwd_b / (fwd_ms * 1e-3) / 1e9},
                "bwd": {"ms": bwd_ms, "gbs": bwd_b / (bwd_ms * 1e-3) / 1e9},
                "step": {"ms": ms_per_step, "gbs": (fwd_b + bwd_b) / (ms_per_step * 1e-3) / 1e9,
                         "frac": (fwd_b + bwd_b) / (ms_per_step * 1e-3) / 1e9 / peak}}
    tr = os.path.join(ROOT, "profiles", "gae_dram_traffic.json")
    if os.path.exists(tr):
        try:
            with open(tr) as f:
                roofline["traffic"] = json.load(f).get(dom)
        except Exception:
            pass
    clocks = sampler.stop() if sampler else None
    del adv_b, gv_b, gr_b

    # ---- e2e: host tensors through the public host API, copies inside the timed region ----------------------
    hv, hr, hg = hostapi.pinned_empty((T + 1, B), local), hostapi.pinned_empty((T, B), local), \
        hostapi.pinned_empty((T, B), local)
    hout = (hostapi.pinned_empty((T, B), local), hostapi.pinned_empty((T + 1, B), local),
            hostapi.pinned_empty((T, B), local))
    cg = torch.Generator().manual_seed(99 + rank)
    for t in (hv, hr, hg):
        t.normal_(generator=cg)

    def e2e_step():  # returns only after the results are in the host tensors
        hostapi.gae_fwd_bwd_host(hv, hr, hg, GAMMA, LAMBDA, out=hout)

    # the link ceiling WITH ALL RANKS ACTIVE: every rank copies 268 MB each way at once, 4 times (GPUs that share a
    # PCIe switch uplink or a socket's memory controllers slow each other down; this is the figure e2e can be judged by)
    dbuf_in, dbuf_out = torch.empty(T, B, device=dev), torch.empty(T, B, device=dev)
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()

    def duplex_once():
        with torch.cuda.stream(s_in):
            dbuf_in.copy_(hr, non_blocking=True)
        with torch.cuda.stream(s_out):
            hout[0].copy_(dbuf_out, non_blocking=True)

    duplex_once()
    barrier()
    t0 = time.perf_counter()
    for _ in range(4):
        duplex_once()
    barrier()
    duplex_gbs = 4 * T * B * 4 / max_over_ranks(time.perf_counter() - t0, torch.float64) / 1e9
    del dbuf_in, dbuf_out

    Ke = max(3, min(K, 10))
    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(Ke):
        e2e_step()
    barrier()
    e2e_ms = max_over_ranks(time.perf_counter() - t0, torch.float64) * 1e3 / Ke
    h2d = 4 * ((T + 1) * B + T * B + T * B)
    d2h = 4 * (T * B + (T + 1) * B + T * B)
    e2e = {"value": T * B * world / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms, "steps": Ke,
           "gbs_each_way": h2d / (e2e_ms * 1e-3) / 1e9, "numa_node": numa_node,
           "pcie_duplex_gbs_each_way_all_ranks_active": duplex_gbs,
           "frac_of_that_duplex_rate": h2d / (e2e_ms * 1e-3) / 1e9 / duplex_gbs,
           "api": "di_hpc_b200.host.gae_fwd_bwd_host -> hpc_rll_gae_fwd_bwd_host (page-locked host tensors on the GPU's "
                  "NUMA node; T-chunked H2D / kernel / D2H carry pipeline)"}
    del hv, hr, hg, hout

    # ---- C4 verbatim: global B=524288 over the N ranks, shards resident; scatter from rank 0 timed separately ------
    c4 = None
    if not args.no_extras and C4_GLOBAL_B % world == 0:
        Bl = C4_GLOBAL_B // world
        del value, reward, gadv
        torch.cuda.empty_cache()
        v4 = torch.randn(T + 1, Bl, device=dev, generator=gen).requires_grad_(True)
        r4 = torch.randn(T, Bl, device=dev, generator=gen).requires_grad_(True)
        g4 = torch.randn(T, Bl, device=dev, generator=gen)
        gae4 = GAE(T, Bl)

        def step4():
            return torch.autograd.grad(gae4(v4, r4, GAMMA, LAMBDA), [v4, r4], grad_outputs=g4)

        for _ in range(3):
            step4()
        barrier()
        k4 = max(5, min(K, 20))
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(k4):
            step4()
        b.record()
        barrier()
        ms4 = max_over_ranks(a.elapsed_time(b)) / k4
        f4, b4 = algorithmic_bytes(T, Bl)
        c4 = {"workload": "gae_fwd_bwd T=%d global B=%d sharded over %d GPU(s), B_local=%d (BASELINE.json configs[4])"
                          % (T, C4_GLOBAL_B, world, Bl),
              "ms_per_step": ms4, "value": T * C4_GLOBAL_B / (ms4 * 1e-3), "unit": UNIT, "scaling": "strong",
              "frac_of_hbm_peak_per_gpu": (f4 + b4) / (ms4 * 1e-3) / 1e9 / peak, "steps": k4}
        del v4, r4, g4
        torch.cuda.empty_cache()
        if dist is not None:
            # the (T,B_local) column slices of a global (T,B) tensor held by rank 0: contiguous per-rank blocks are
            # prepared on rank 0 (outside the timing, as a collector would) and scattered over NVLink
            shard = torch.empty(T, Bl, device=dev)
            parts = [torch.randn(T, Bl, device=dev) for _ in range(world)] if rank == 0 else None
            for _ in range(2):
                dist.scatter(shard, parts, src=0)
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            ks = 5
            for _ in range(ks):
                dist.scatter(shard, parts, src=0)
            b.record()
            barrier()
            sc_ms = max_over_ranks(a.elapsed_time(b)) / ks
            sent = 4 * T * Bl * (world - 1)
            c4["scatter"] = {"what": "NCCL scatter of ONE (T,B_local) fp32 tensor per rank from rank 0 (value and "
                                     "reward need two of these; excluded from steps/s as BASELINE.md C4 says)",
                             "ms": sc_ms, "bytes_leaving_rank0": sent, "gbs_rank0_egress": sent / (sc_ms * 1e-3) / 1e9,
                             "vs_compute": sc_ms * 2 / ms4}
            del shard, parts
            torch.cuda.empty_cache()

    # ---- the path's only collective: a loss op on the local shard, scalar all-reduced ----------------------
    loss_ar = None
    if dist is not None and not args.no_extras:
        from di_hpc_b200.sharding import P2PScalarAllReduce, all_reduce_losses, set_global_batch
        from hpc_rll.rl_utils.td import TDLambda
        vl = torch.randn(T + 1, B, device=dev, generator=gen).requires_grad_(True)
        rl = torch.randn(T, B, device=dev, generator=gen)
        tdl = set_global_batch(TDLambda(T, B), B * world)
        one = torch.ones(1, device=dev)

        def td_local():
            torch.autograd.grad(tdl(vl, rl), [vl], grad_outputs=one)

        def td_global():
            (loss, ) = all_reduce_losses([tdl(vl, rl)])
            torch.autograd.grad(loss, [vl], grad_outputs=one)

        p2p = P2PScalarAllReduce()

        def td_global_p2p():
            (loss, ) = all_reduce_losses([tdl(vl, rl)], comm=p2p)
            torch.autograd.grad(loss, [vl], grad_outputs=one)

        # same numbers from both collectives (rank-ordered fp32 sum vs NCCL's)
        la = all_reduce_losses([tdl(vl, rl)])[0].item()
        lb = all_reduce_losses([tdl(vl, rl)], comm=p2p)[0].item()
        res = {"loss_nccl": la, "loss_p2p": lb}
        for name, fn in (("local_only_ms", td_local), ("with_allreduce_ms", td_global),
                         ("with_p2p_allreduce_ms", td_global_p2p)):
            for _ in range(3):
                fn()
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(20):
                fn()
            b.record()
            barrier()
            res[name] = max_over_ranks(a.elapsed_time(b)) / 20
        res["what"] = ("TD(lambda) fwd+bwd T=%d B_local=%d, loss normalised by the global count; with_allreduce adds one "
                       "NCCL all_reduce(SUM) of the scalar loss per step, with_p2p_allreduce the NVLink peer-memory kernel "
                       "(csrc/p2p.cu) instead (di_hpc_b200.sharding.all_reduce_losses)" % (T, B))
        res["allreduce_cost_ms"] = res["with_allreduce_ms"] - res["local_only_ms"]
        res["p2p_allreduce_cost_ms"] = res["with_p2p_allreduce_ms"] - res["local_only_ms"]
        p2p.close()
        loss_ar = res
        del vl, rl
        torch.cuda.empty_cache()

    ops = None
    if world == 1 and not args.no_extras:
        try:
            del value, reward, gadv
        except NameError:
            pass
        torch.cuda.empty_cache()
        ops = ops_block(torch, peak)

    if rank == 0:
        hostapi.unbind()  # the CPU baseline gets every host core and both sockets' memory, like the reference arm
        base, _ = cpu_baseline(T, B, 5) if world == 1 else (None, None)
        line = {"metric": METRIC, "value": value_metric, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": config_of(T, B, world),
                "roofline": roofline, "module": module, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks}
        if c4 is not None:
            line["c4"] = c4
        if loss_ar is not None:
            line["loss_allreduce"] = loss_ar
        if ops is not None:
            line["ops"] = ops
        if base is not None:
            line["cpu_baseline"] = base
        print(json.dumps(line), file=OUT, flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def _claim_stdout():
    """The driver parses ONE JSON line from stdout.  Libraries (NCCL's version banner, torchrun notices)
    also write there, so stdout is pointed at stderr for the whole run and the JSON line goes to the
    saved descriptor."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(real, "w")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--T", type=int, default=T_DEFAULT)
    ap.add_argument("--B", type=int, default=B_DEFAULT, help="columns per GPU")
    ap.add_argument("--no-extras", action="store_true", help="skip the ops / c4 / loss_allreduce blocks")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs (adv, grad_value, grad_reward; a fixed sample of columns) "
                         "as DIR/<name>.npy; the inputs are seeded, so runs with the same arguments are comparable")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    global OUT
    OUT = _claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
    OUT.flush()


if __name__ == "__main__":
    main()
