"""Grid-graph GNN stack of the roofline sweep (BASELINE.json configs[4], SURVEY.md section 8d.5).

Operator = the reference's `FrozenLakeNet.GNNLayer` (frozenlake/FrozenLakeNet.py:8-33),
`relu(bmm(adj, W x + b))`, applied to gh x gw 4-neighbour grid graphs with the symmetric
normalisation of `create_adjacency` (:68-72) and self loops.  The dense Linear runs on the
library's SGEMM, the aggregation on `azg_grid_aggregate_relu_*` (the adjacency is never
materialised); `torch.autograd.Function`s route tensors, parameters live in `nn.Linear`s.
"""
import torch
import torch.nn as nn

from . import _lib
from ._lib import ptr, stream
from .training import _Linear


class _GridAggRelu(torch.autograd.Function):
    @staticmethod
    def forward(ctx, sup, gh, gw):
        sup = sup.contiguous()
        B, n, H = sup.shape
        out = torch.empty_like(sup)
        _lib.check(_lib.lib().azg_grid_aggregate_relu_forward(ptr(sup), B, gh, gw, H, ptr(out), stream()))
        ctx.save_for_backward(out)
        ctx.g = (gh, gw)
        return out

    @staticmethod
    def backward(ctx, dout):
        (out,) = ctx.saved_tensors
        dout = dout.contiguous()
        B, n, H = out.shape
        dsup = torch.empty_like(out)
        _lib.check(_lib.lib().azg_grid_aggregate_relu_backward(ptr(dout), ptr(out), B, ctx.g[0], ctx.g[1], H, ptr(dsup), stream()))
        return dsup, None, None


def _pack(weight, transpose):
    H = weight.shape[0]
    lib = _lib.lib()
    blob = torch.empty(int(lib.azg_grid_packed_bytes(H)), dtype=torch.uint8, device=weight.device)
    _lib.check(lib.azg_grid_pack_weights(ptr(weight.detach().contiguous()), H, int(transpose), ptr(blob), stream()))
    return blob


class _GridLayerTC(torch.autograd.Function):
    """One GNNLayer as the fused tensor-core kernel (csrc/azg_grid_tc.cu): out = relu(adj (x W^T + b)).
    Backward: dx from the same kernel on (dout * [out > 0]) with the transposed weight image; the weight and bias
    gradients contract over all B*n rows (S = adj (dout * [out > 0]), dW = S^T x): on tcgen05 with MN-major operands."""

    @staticmethod
    def forward(ctx, x, weight, bias, gh, gw, prec):
        x = x.contiguous()
        B, n, H = x.shape
        lib = _lib.lib()
        out = torch.empty_like(x)
        _lib.check(lib.azg_grid_layer_tc_forward(ptr(x), ptr(_pack(weight, False)), ptr(bias.contiguous()), B, gh, gw, H, prec,
                                                 ptr(out), stream()))
        ctx.save_for_backward(x, weight, out)
        ctx.g = (gh, gw, prec)
        return out

    @staticmethod
    def backward(ctx, dout):
        x, weight, out = ctx.saved_tensors
        gh, gw, prec = ctx.g
        dout = dout.contiguous()
        B, n, H = out.shape
        lib = _lib.lib()
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            _lib.check(lib.azg_grid_layer_tc_backward_input(ptr(dout), ptr(out), ptr(_pack(weight, True)), B, gh, gw, H, prec,
                                                            ptr(dx), stream()))
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            s = torch.empty_like(out)
            _lib.check(lib.azg_grid_aggregate_relu_backward(ptr(dout), ptr(out), B, gh, gw, H, ptr(s), stream()))
            dw, db = torch.empty_like(weight), torch.empty(H, dtype=torch.float32, device=x.device)
            if H in (64, 128, 256):  # contraction over all B*n rows on the tensor cores (MN-major operands, split-K over CTAs)
                scratch = torch.empty(int(lib.azg_grid_dw_scratch_floats(H)), dtype=torch.float32, device=x.device)
                _lib.check(lib.azg_grid_layer_tc_backward_weights(ptr(s), ptr(x), B * n, H, prec, ptr(dw), ptr(db), ptr(scratch),
                                                                  stream()))
            else:
                _lib.check(lib.azg_linear_backward(ptr(s), ptr(x), ptr(weight), None, B * n, H, H, 0, None, ptr(dw), ptr(db), None,
                                                   stream()))
        return dx, dw, db, None, None, None


class GridGNNStack(nn.Module):
    """`layers` x GNNLayer(hidden, hidden) over [B, gh*gw, hidden] node features.

    precision: "bf16x3" (default; fp32-level accuracy on the tensor cores), "bf16", or "fp32" (CUDA-core SGEMM +
    separate aggregation kernel -- also the path for graphs of more than 256 nodes or other hidden sizes).  Graphs of up to
    128 nodes share 128-row tiles (128 // n graphs each), 129..256 nodes take one 256-row tile per graph.  The fused layer
    takes gh, gw >= 1 with gh*gw <= 256 (azg_grid_tc_supported); tests/test_grid_tc_layer_gpu.py checks all of its kernels
    against float64.
    The fp32 path takes any grid of up to 2^30 nodes and any hidden size divisible by 4; tests/test_grid_fp32_path_gpu.py
    checks it against float64 from 1 to 33,124 nodes and hidden 4 to 1,024."""

    def __init__(self, gh, gw, hidden, layers=2, precision="bf16x3"):
        super().__init__()
        _lib.require_device()
        self.gh, self.gw, self.hidden = gh, gw, hidden
        self.precision = _lib.PRECISIONS[precision]
        self.gnn_layers = nn.ModuleList([nn.Linear(hidden, hidden) for _ in range(layers)])
        self.fused = self.precision != _lib.PREC_FP32 and bool(_lib.lib().azg_grid_tc_supported(gh, gw, hidden))

    def forward(self, x):
        B, n, H = x.shape
        assert n == self.gh * self.gw and H == self.hidden
        for lin in self.gnn_layers:
            if self.fused:
                x = _GridLayerTC.apply(x, lin.weight, lin.bias, self.gh, self.gw, self.precision)
                continue
            sup = _Linear.apply(x.reshape(B * n, H), lin.weight, lin.bias, False)
            x = _GridAggRelu.apply(sup.reshape(B, n, H), self.gh, self.gw)
        return x
