"""numpy restatement of the reference's ScatterConnection.  TEST INFRASTRUCTURE ONLY (see oracle.c header).

hpc_rll/origin/scatter_connection.py:25-64 on the CPU is sequential in entity order m (torch's CPU scatter_ /
scatter_add_ walk the index in order): per batch b and cell y*W + x,
  add   : out = ((0.f + x[m0]) + x[m1]) + ...  in ascending m, fp32 (a lone -0.0 becomes +0.0)
  cover : out = x[m_last]                      (copied exactly, -0.0 stays -0.0)
  cells no entity lands on are +0.0.
The gradient of x is the gather grad_x[b, m, :] = grad_out[b, :, y, x] in both modes.  An entity outside the map writes
nothing and gets a zero gradient (this project's rule; origin has no defined behaviour there).  Pinned to origin outputs
by tests/golden/scatter_*.npz.
"""
import numpy as np


def _cells(location, H, W):
    """(B, M, 2) int64 -> (B, M) cell index, -1 outside the map."""
    y, x = location[..., 0], location[..., 1]
    inside = (y >= 0) & (y < H) & (x >= 0) & (x < W)
    return np.where(inside, y * W + x, -1)


def forward(x, location, H, W, scatter_type):
    assert scatter_type in ("cover", "add")
    x = np.asarray(x, dtype=np.float32)
    B, M, N = x.shape
    cells = _cells(np.asarray(location, dtype=np.int64), H, W)
    out = np.zeros((B, H * W, N), dtype=np.float32)
    for b in range(B):
        for m in range(M):
            c = cells[b, m]
            if c < 0:
                continue
            if scatter_type == "add":
                out[b, c] = out[b, c] + x[b, m]  # fp32 + fp32, one entity at a time
            else:
                out[b, c] = x[b, m]
    return np.ascontiguousarray(out.transpose(0, 2, 1).reshape(B, N, H, W))


def backward(grad_out, location, H, W):
    g = np.asarray(grad_out, dtype=np.float32)
    B, N = g.shape[:2]
    cells = _cells(np.asarray(location, dtype=np.int64), H, W)
    flat = g.reshape(B, N, H * W)
    gx = np.take_along_axis(flat, np.maximum(cells, 0)[:, None, :], axis=2).transpose(0, 2, 1)  # (B, M, N)
    return np.ascontiguousarray(np.where((cells >= 0)[:, :, None], gx, np.float32(0)))
