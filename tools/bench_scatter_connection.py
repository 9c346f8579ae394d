"""ScatterConnection throughput on the GPU: the hpc_rll module (forward, and forward + backward) against a plain-torch
formulation of the same op with torch's autograd (what a DI-engine model runs without hpc), and ``torch.zeros`` of the
output as the write rate actually reached in the same run.  CUDA events over queued calls (best of a few windows).
Algorithmic bytes come from the shapes:
  forward  : x + location + output
  backward : location + grad_x + the 32-byte grad_out sectors the entities' cells touch (counted from the locations)
The card's name and power limit are read in the same run.

    python tools/bench_scatter_connection.py --out DIR [--iters 50] [--quick]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hpc_rll.torch_utils.network.scatter_connection import ScatterConnection  # noqa: E402

# name -> (B, M, N, H, W): the reference test shape (tests/test_scatter.py of DI-hpc; dense map, slab backward), the
# same at B=1024 (working set beyond the 126 MB L2), an AlphaStar-like map (sparse, direct-gather backward, 200 MB out)
WORKLOADS = {
    "ref_b256": (256, 256, 256, 16, 16),
    "ref_b1024": (1024, 256, 256, 16, 16),
    "alphastar_b64": (64, 512, 32, 152, 160),
}


def card():
    idx = torch.cuda.current_device()
    info = {"name": torch.cuda.get_device_name(idx)}
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(idx), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30)
        pl, clk = [v.strip() for v in r.stdout.strip().split(",")]
        info.update(power_limit_w=float(pl), max_sm_clock_mhz=float(clk))
    except Exception as e:  # noqa: BLE001
        info["power_limit_w"] = "unavailable: %s" % e
    return info


def torch_scatter(x, loc, H, W, mode):
    """plain torch with autograd: per-batch scatter along the flattened map, channel-major like the output"""
    B, M, N = x.shape
    idx = (loc[..., 0] * W + loc[..., 1]).unsqueeze(1).expand(B, N, M)
    src = x.transpose(1, 2)
    out = x.new_zeros(B, N, H * W)
    out = out.scatter_add(2, idx, src) if mode == "add" else out.scatter(2, idx, src)
    return out.view(B, N, H, W)


def timed(fn, iters, windows=5):
    """best-of-windows ms per call, `iters` calls queued back to back between two events"""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    best = None
    for _ in range(windows):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        best = ms if best is None else min(best, ms)
    return best


def touched_sector_bytes(loc, N, H, W):
    """32-byte sectors of grad_out the backward gather must read: distinct (b, cell // 8) pairs, times N planes
    (H*W*4 is a multiple of 32 for the workloads here, so every plane starts on a sector)."""
    B = loc.shape[0]
    cell = loc[..., 0] * W + loc[..., 1]
    key = torch.arange(B, device=loc.device).unsqueeze(1) * (H * W) + cell // 8
    return int(torch.unique(key).numel()) * N * 32


def bench(name, B, M, N, H, W, mode, iters):
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(B, M, N, device="cuda", generator=g)
    loc = torch.stack([torch.randint(0, H, (B, M), device="cuda", generator=g),
                       torch.randint(0, W, (B, M), device="cuda", generator=g)], dim=2)
    gout = torch.randn(B, N, H, W, device="cuda", generator=g)
    xg = x.clone().requires_grad_(True)
    mod = ScatterConnection(B, M, N, H, W, mode)
    out_b, x_b, loc_b = B * N * H * W * 4, B * M * N * 4, B * M * 2 * 8
    fwd_bytes = x_b + loc_b + out_b
    bwd_bytes = loc_b + x_b + touched_sector_bytes(loc, N, H, W)
    with torch.no_grad():
        t_fwd = timed(lambda: mod(x, loc), iters)
        t_torch_fwd = timed(lambda: torch_scatter(x, loc, H, W, mode), iters)
        t_zeros = timed(lambda: torch.zeros(B, N, H, W, device="cuda"), iters)
    t_fb = timed(lambda: torch.autograd.grad(mod(xg, loc), xg, gout), iters)
    t_torch_fb = timed(lambda: torch.autograd.grad(torch_scatter(xg, loc, H, W, mode), xg, gout), iters)
    gbs = lambda b, ms: b / ms / 1e6
    zeros_rate = gbs(out_b, t_zeros)
    r = {"workload": name, "mode": mode, "B": B, "M": M, "N": N, "H": H, "W": W,
         "fwd_bytes": fwd_bytes, "bwd_bytes": bwd_bytes,
         "hpc_fwd_ms": t_fwd, "hpc_fwd_bwd_ms": t_fb, "hpc_bwd_ms_derived": t_fb - t_fwd,
         "torch_fwd_ms": t_torch_fwd, "torch_fwd_bwd_ms": t_torch_fb, "zeros_ms": t_zeros,
         "hpc_fwd_GBps": gbs(fwd_bytes, t_fwd), "hpc_fwd_bwd_GBps": gbs(fwd_bytes + bwd_bytes, t_fb),
         "zeros_write_GBps": zeros_rate,
         "hpc_fwd_vs_zeros_rate": gbs(fwd_bytes, t_fwd) / zeros_rate,
         "fwd_bwd_speedup_vs_torch": t_torch_fb / t_fb, "fwd_speedup_vs_torch": t_torch_fwd / t_fwd}
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for bench_scatter_connection.json")
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--quick", action="store_true", help="reference shape only, few iterations")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_scatter_connection needs a CUDA device")
    os.makedirs(a.out, exist_ok=True)
    res = {"card": card(), "iters": a.iters, "results": []}
    print(json.dumps(res["card"]), flush=True)
    for name, (B, M, N, H, W) in WORKLOADS.items():
        if a.quick and name != "ref_b256":
            continue
        for mode in ("add", "cover"):
            r = bench(name, B, M, N, H, W, mode, 5 if a.quick else a.iters)
            res["results"].append(r)
            print(json.dumps(r), flush=True)
            torch.cuda.empty_cache()
    with open(os.path.join(a.out, "bench_scatter_connection.json"), "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
