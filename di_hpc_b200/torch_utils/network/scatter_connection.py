"""ScatterConnection -- drop-in for /root/reference/hpc_rll/torch_utils/network/scatter_connection.py (class
ScatterConnection, ScatterConnectionFunction).

Same constructor ``ScatterConnection(B, M, N, H, W, scatter_type)`` and ``forward(x, location)`` as the reference
(scatter_connection.py:31-88): ``x`` (B, M, N) fp32 entity embeddings, ``location`` (B, M, 2) int64 ``(y, x)`` pairs,
result (B, N, H, W).  Results are those of hpc_rll/origin/scatter_connection.py on the CPU, bit for bit: entities apply
in ascending ``m`` -- ``'add'`` sums in that order starting from +0.0, ``'cover'`` keeps the last one -- and the
gradient of ``x`` is the gather ``grad_out[b, :, y, x]`` in both modes.  Differences, all deliberate (DESIGN.md
"Deviations"):
  * the result is a fresh tensor, not the module-owned ``output`` buffer returned by alias; B, M and N come from ``x``
    (the constructor's are kept only for API compatibility), H and W from the constructor;
  * ``'cover'`` with colliding entities is deterministic (the reference's CUDA path races) and ``'add'`` uses no
    floating-point atomics, so results are identical run to run;
  * an entity outside the H x W map writes nothing and gets a zero gradient (the reference writes out of bounds);
  * kernels run on PyTorch's current stream, with argument checks.
"""
import torch

from ... import _abi, _ext

_MODES = {'cover': 0, 'add': 1}


def _check(x, location):
    x = _abi.require_f32_cuda("x", x)
    location = _abi.require_i64_cuda("location", location)
    if x.dim() != 3:
        raise ValueError("x must be (B, M, N), got %s" % (tuple(x.shape), ))
    B, M, N = x.shape
    if location.shape != (B, M, 2):
        raise ValueError("location must be (B, M, 2)=(%d, %d, 2), got %s" % (B, M, tuple(location.shape)))
    if location.device != x.device:
        raise ValueError("x and location must live on one CUDA device")
    return x, location


class ScatterConnectionFunction(torch.autograd.Function):

    @staticmethod
    def forward(ctx, x, location, H, W, scatter_type):
        x, location = _check(x, location)
        B, M, N = x.shape
        out = torch.empty((B, N, H, W), dtype=torch.float32, device=x.device)
        with _abi.on_device(x.device):
            _abi.check(
                _abi.lib().hpc_rll_scatter_connection_forward(_abi.ptr(x), _abi.ptr(location), _abi.ptr(out), B, M, N,
                                                              H, W, _MODES[scatter_type], _abi.stream_of(x)),
                "hpc_rll_scatter_connection_forward")
        ctx.save_for_backward(location)
        ctx.N = N
        return out

    @staticmethod
    def backward(ctx, grad_out):
        location, = ctx.saved_tensors
        grad_out = _abi.require_f32_cuda("grad_out", grad_out)
        B, M, _ = location.shape
        H, W = grad_out.shape[2], grad_out.shape[3]
        grad_x = torch.empty((B, M, ctx.N), dtype=torch.float32, device=grad_out.device)
        with _abi.on_device(grad_out.device):
            _abi.check(
                _abi.lib().hpc_rll_scatter_connection_backward(_abi.ptr(grad_out), _abi.ptr(location),
                                                               _abi.ptr(grad_x), B, M, ctx.N, H, W,
                                                               _abi.stream_of(grad_out)),
                "hpc_rll_scatter_connection_backward")
        return grad_x, None, None, None, None


class ScatterConnection(torch.nn.Module):
    r"""
    Overview:
        Scatter feature to its corresponding location.
        In AlphaStar, each entity is embedded into a tensor; these tensors are scattered into a feature map of the
        map size.

    Interface:
        __init__, forward
    """

    def __init__(self, B, M, N, H, W, scatter_type) -> None:
        r"""
        Arguments:
            - B (:obj:`int`): batch size
            - M (:obj:`int`): the number of entities
            - N (:obj:`int`): the dimension of entity attributes
            - H (:obj:`int`): height of the spatial feature
            - W (:obj:`int`): width of the spatial feature
            - scatter_type (:obj:`str`): 'add' or 'cover': when two entities share a location, the later one is
              added to or covers the earlier one
        """
        super().__init__()
        self.B, self.M, self.N, self.H, self.W = B, M, N, H, W
        self.scatter_type = scatter_type
        assert self.scatter_type in ['cover', 'add']

    def forward(self, x: torch.Tensor, location: torch.Tensor) -> torch.Tensor:
        """
        Arguments:
            - x (:obj:`torch.FloatTensor`): :math:`(B, M, N)`, the entity embeddings
            - location (:obj:`torch.LongTensor`): :math:`(B, M, 2)`, each location is (y, x)
        Returns:
            - output (:obj:`torch.FloatTensor`): :math:`(B, N, H, W)`, the scattered feature map
        """
        assert (x.is_cuda)
        assert (location.is_cuda)
        fast = _ext.fast()
        if fast is not None:  # C++ autograd function (csrc_torch/fast_ops.cpp); ScatterConnectionFunction is its twin
            return fast._network.scatter_connection(x, location, int(self.H), int(self.W), _MODES[self.scatter_type])
        return ScatterConnectionFunction.apply(x, location, int(self.H), int(self.W), self.scatter_type)
