"""Grid-graph sweep operator (BASELINE configs[4]): CUDA forward/backward of the GNNLayer stack on
grid graphs vs the oracle (torch bmm with the dense normalised adjacency)."""
import numpy as np
import pytest
import torch

from oracle import nets as onets
import torch.nn.functional as F

from azgnn_b200.gridgnn import GridGNNStack, _GridAggRelu, _GridLayerTC
from azgnn_b200.training import _Linear

pytestmark = pytest.mark.gpu
torch.backends.cuda.matmul.allow_tf32 = False


@pytest.mark.parametrize("gh,gw", [(3, 3), (4, 4), (6, 7), (7, 7), (8, 8), (16, 16)])
@pytest.mark.parametrize("hidden", [64, 128, 256])
def test_grid_gnn_forward_backward(gh, gw, hidden):
    """fp32 path: SGEMM + aggregation kernels vs the dense-adjacency oracle.  Gradients: against autograd through the oracle
    operator under the kernel's own ReLU pattern, every element (see test_fused_tensor_core_layer)."""
    torch.manual_seed(gh * 100 + hidden)
    B = 37
    n = gh * gw
    net = GridGNNStack(gh, gw, hidden, layers=2, precision="fp32").cuda()
    assert not net.fused
    x = torch.randn(B, n, hidden, device="cuda", requires_grad=True)
    with torch.no_grad():  # the per-layer outputs, through the same kernels as net(x)
        outs, h = [], x
        for lin in net.gnn_layers:
            h = _GridAggRelu.apply(_Linear.apply(h.reshape(B * n, hidden), lin.weight, lin.bias, False).reshape(B, n, hidden), gh, gw)
            outs.append(h)
    y = net(x)
    assert torch.equal(y, outs[-1])
    g = torch.randn_like(y)
    y.backward(g)
    got = [x.grad.clone()] + [p.grad.clone() for p in net.parameters()]
    x2 = x.detach().clone().requires_grad_(True)
    ws = [l.weight.detach().clone().requires_grad_(True) for l in net.gnn_layers]
    bs = [l.bias.detach().clone().requires_grad_(True) for l in net.gnn_layers]
    with torch.no_grad():
        y_ref = onets.grid_gnn_forward(ws, bs, x2, gh, gw)
    assert (y - y_ref).abs().max().item() <= 1e-5 * max(1.0, y_ref.abs().max().item())
    adj = onets.grid_adjacency(gh, gw).cuda().unsqueeze(0).expand(B, -1, -1)
    h2 = x2
    for w, b, o in zip(ws, bs, outs):
        h2 = torch.bmm(adj, F.linear(h2, w, b)) * (o > 0)
    h2.backward(g)
    ref = [x2.grad] + [t.grad for pair in zip(ws, bs) for t in pair]
    for a, b in zip(got, ref):
        assert (a - b).abs().max().item() <= 1e-4 * b.abs().max().item() + 1e-6, (a - b).abs().max().item()


@pytest.mark.parametrize("gh,gw", [(3, 3), (4, 4), (6, 7), (7, 7), (8, 8), (11, 11), (9, 15), (12, 13), (15, 16), (16, 16), (1, 200)])
@pytest.mark.parametrize("hidden", [64, 128, 256])
def test_fused_tensor_core_layer(gh, gw, hidden):
    """bf16x3 = the fused tcgen05 layer kernel.  Outputs: the fp32 contract (1e-5) against the oracle.  Gradients:
    against autograd through the oracle operator evaluated WITH THE KERNEL'S OWN ReLU pattern -- a hidden unit whose
    pre-activation is within rounding of 0 may land on either side of the ReLU in two correct implementations, and
    with a random upstream gradient one such flip moves a whole row of the weight gradient, so comparing gradients
    across different activation patterns says nothing about the backward kernels."""
    torch.manual_seed(gh * 100 + hidden)
    B = 1531 if gh * gw <= 128 else 449  # the persistent CTAs walk several tiles each (above 128 nodes: one graph per 256-row tile)
    net = GridGNNStack(gh, gw, hidden, layers=2, precision="bf16x3").cuda()
    assert net.fused
    x = torch.randn(B, gh * gw, hidden, device="cuda", requires_grad=True)
    outs, h = [], x
    for lin in net.gnn_layers:
        h = _GridLayerTC.apply(h, lin.weight, lin.bias, gh, gw, net.precision)
        outs.append(h)
    g = torch.randn_like(h)
    h.backward(g)
    got = [x.grad.clone()] + [p.grad.clone() for p in net.parameters()]
    x2 = x.detach().clone().requires_grad_(True)
    ws = [l.weight.detach().clone().requires_grad_(True) for l in net.gnn_layers]
    bs = [l.bias.detach().clone().requires_grad_(True) for l in net.gnn_layers]
    with torch.no_grad():
        y_ref = onets.grid_gnn_forward(ws, bs, x2, gh, gw)
    assert (h - y_ref).abs().max().item() <= 1e-5 * max(1.0, y_ref.abs().max().item())
    adj = onets.grid_adjacency(gh, gw).cuda().unsqueeze(0).expand(B, -1, -1)
    h2 = x2
    for w, b, o in zip(ws, bs, outs):
        h2 = torch.bmm(adj, F.linear(h2, w, b)) * (o.detach() > 0)
    h2.backward(g)
    ref = [x2.grad] + [t.grad for pair in zip(ws, bs) for t in pair]
    for a, b in zip(got, ref):
        assert (a - b).abs().max().item() <= 1e-4 * b.abs().max().item() + 1e-6, (a - b).abs().max().item()


@pytest.mark.parametrize("gh,gw", [(7, 7), (16, 16), (13, 10)])
@pytest.mark.parametrize("B", [1, 2, 3, 148 * 2 + 1])
def test_fused_layer_ragged_batches(B, gh, gw):
    """tiles with empty graph slots / a partial last tile, bf16 single-product mode at its stated tolerance (2e-2)"""
    torch.manual_seed(B)
    for precision, tol in (("bf16x3", 1e-5), ("bf16", 2e-2)):
        net = GridGNNStack(gh, gw, 128, layers=2, precision=precision).cuda()
        assert net.fused
        x = torch.randn(B, gh * gw, 128, device="cuda")
        with torch.no_grad():
            y = net(x)
            y2 = onets.grid_gnn_forward([l.weight for l in net.gnn_layers], [l.bias for l in net.gnn_layers], x, gh, gw)
        assert (y - y2).abs().max().item() <= tol * max(1.0, y2.abs().max().item())


@pytest.mark.parametrize("env", [{"AZG_GRID_TILE": "256"}, {"AZG_GRID_TILE": "128", "AZG_GRID_PAIR": "0"}])
def test_forced_tile_shapes_on_small_graphs(env):
    """The library picks the tile shape per configuration (128-row tiles, 256-row tiles where they waste fewer rows or the graph
    needs them, CTA pairs for H = 256 in bf16x3).  The switches force the other choice for graphs of up to 128 nodes:
    AZG_GRID_TILE=256 -> several graphs per 256-row tile, some straddling the half boundary; AZG_GRID_TILE=128 + AZG_GRID_PAIR=0
    -> 128-row tiles everywhere and single CTAs with streamed weights.  Read once per process -> subprocess."""
    import os
    import subprocess
    import sys
    sel = "test_fused_tensor_core_layer and (3-3 or 7-7 or 8-8 or 11-11) or test_fused_layer_ragged_batches and 7-7"
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k", sel],
                       env=dict(os.environ, **env), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout and "no tests ran" not in r.stdout


@pytest.mark.parametrize("H", [64, 128, 256])
@pytest.mark.parametrize("rows", [1, 63, 64, 65, 4097, 333333])
def test_weight_gradient_kernel_ragged_row_counts(H, rows):
    """dW = S^T X, db = colsum(S) on tcgen05 with MN-major operands: partial k-blocks, fewer k-blocks than CTAs.  bf16x3
    against the exact product, bf16 against the product of the bf16-rounded operands (what its one MMA per step
    multiplies), both at 2e-5 of the largest sum |S| |X|."""
    from azgnn_b200 import _lib
    from azgnn_b200._lib import ptr, stream
    g = torch.Generator(device="cuda").manual_seed(rows + H)
    S = torch.randn(rows, H, device="cuda", generator=g)
    X = torch.randn(rows, H, device="cuda", generator=g)
    lib = _lib.lib()
    dw, db = torch.empty(H, H, device="cuda"), torch.empty(H, device="cuda")
    scratch = torch.empty(int(lib.azg_grid_dw_scratch_floats(H)), device="cuda")
    scale = (S.double().abs().t() @ X.double().abs()).max().item() + 1.0
    for prec, want in ((_lib.PREC_BF16X3, S.double().t() @ X.double()),
                       (_lib.PREC_BF16, S.bfloat16().double().t() @ X.bfloat16().double())):
        _lib.check(lib.azg_grid_layer_tc_backward_weights(ptr(S), ptr(X), rows, H, prec, ptr(dw), ptr(db), ptr(scratch), stream()))
        assert (dw.double() - want).abs().max().item() <= 2e-5 * scale, (prec, (dw.double() - want).abs().max().item(), scale)
        assert (db.double() - S.double().sum(0)).abs().max().item() <= 1e-5 * (S.abs().sum(0).max().item() + 1.0)
