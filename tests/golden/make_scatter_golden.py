#!/usr/bin/env python
"""Generate the committed ScatterConnection fixtures (tests/golden/scatter_*.npz) by RUNNING THE REFERENCE.

Runs ``hpc_rll/origin/scatter_connection.py`` of a DI-hpc checkout on the CPU (loaded read-only through
``_ref_origin.REF_ROOT``; nothing is copied) on seeded inputs and stores ``x``, ``location``, the map ``out``, a random
upstream gradient ``grad_out`` and the autograd gradient ``grad_x``, plus ``H``, ``W`` and ``scatter_type``.  Origin on
the CPU is sequential in entity order, so these pin the semantics the kernels match bit for bit
(oracle/scatter_oracle.py, DESIGN.md section 4.12).  Adds or rewrites only the scatter_*.npz files:

    python tests/golden/make_scatter_golden.py
"""
import importlib.util
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import _ref_origin  # noqa: E402


def _origin():
    path = os.path.join(_ref_origin.REF_ROOT, "hpc_rll", "origin", "scatter_connection.py")
    spec = importlib.util.spec_from_file_location("ref_origin_scatter_connection", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def case_scatter(S, name, B, M, N, H, W, scatter_type, seed, loc_hw=None):
    """x with ~5% -0.0 entries (add turns a lone -0.0 into +0.0, cover keeps it), locations drawn from the first
    loc_hw = (h, w) rows / columns (collisions), the gradient of x for a random upstream gradient of the map."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, M, N, generator=g)
    x[torch.rand(B, M, N, generator=g) < 0.05] = -0.0
    h, w = loc_hw or (H, W)
    location = torch.stack([torch.randint(0, h, (B, M), generator=g), torch.randint(0, w, (B, M), generator=g)], dim=2)
    grad_out = torch.randn(B, N, H, W, generator=g)
    xr = x.clone().requires_grad_(True)
    out = S.ScatterConnection(scatter_type)(xr, (H, W), location)
    grad_x, = torch.autograd.grad(out, xr, grad_outputs=grad_out)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), x=x.numpy(), location=location.numpy(),
                        out=out.detach().numpy(), grad_out=grad_out.numpy(), grad_x=grad_x.numpy(), H=np.asarray(H),
                        W=np.asarray(W), scatter_type=np.asarray(scatter_type))


def main():
    S = _origin()
    s = 2468
    case_scatter(S, "scatter_add_b4_m64_n8_h3w3", 4, 64, 8, 3, 3, "add", s + 1)       # heavy collisions
    case_scatter(S, "scatter_cover_b4_m64_n8_h3w3", 4, 64, 8, 3, 3, "cover", s + 2)
    case_scatter(S, "scatter_add_b2_m1000_n4_h2w2", 2, 1000, 4, 2, 2, "add", s + 3)   # 1000 entities in 4 cells
    case_scatter(S, "scatter_cover_b2_m1000_n4_h2w2", 2, 1000, 4, 2, 2, "cover", s + 4)
    case_scatter(S, "scatter_add_b3_m40_n17_h7w9", 3, 40, 17, 7, 9, "add", s + 5)     # odd plane, N % 4 != 0
    case_scatter(S, "scatter_cover_b3_m40_n17_h7w9", 3, 40, 17, 7, 9, "cover", s + 6)
    case_scatter(S, "scatter_add_b2_m24_n5_h16w16", 2, 24, 5, 16, 16, "add", s + 7)   # sparse: lone entities
    case_scatter(S, "scatter_cover_b2_m24_n5_h16w16", 2, 24, 5, 16, 16, "cover", s + 8)
    case_scatter(S, "scatter_add_b2_m48_n6_h16w16_corner", 2, 48, 6, 16, 16, "add", s + 9, loc_hw=(2, 3))
    print("wrote 9 scatter fixtures to %s" % HERE)


if __name__ == "__main__":
    main()
