"""The fp32 path of the grid-graph stack (gridgnn.py, precision="fp32", and every graph or hidden size the fused tensor-core
layer does not take) against float64, at every shape it accepts.

The aggregation kernel (azg_train.cu, grid_aggregate_kernel) is driven through the C ABI and compared, element by element,
with a float64 reference that gathers the <= 5 neighbours of each node by index: the dense adjacency would take 8.8 GB
at 33k nodes.  The reference itself is held to oracle.nets.grid_adjacency without a GPU.  The stack (azg_linear_f32 +
aggregation, forward and backward) is compared with float64 autograd under the kernel's own ReLU pattern.

u = 2^-24 is the unit roundoff of fp32."""
import pytest
import torch
import torch.nn.functional as Fn

from oracle import nets as onets

from azgnn_b200 import _lib
from azgnn_b200._lib import ptr, stream
from azgnn_b200.gridgnn import GridGNNStack, _GridAggRelu
from azgnn_b200.training import _Linear

from helpers import aggregate64, grid_neighbours

U = 2.0 ** -24
GRID = 148 * 16  # CTAs of launch_grid_aggregate (azg_train.cu): graphs b and b + GRID are walked by the same CTA


@pytest.mark.parametrize("gh,gw", [(1, 1), (1, 2), (3, 3), (4, 7), (16, 16)])
def test_neighbour_reference_matches_dense_oracle(gh, gw):
    """The gathered reference against the dense oracle.nets.grid_adjacency (float32, cast to float64): same sparsity
    pattern, coefficients within the oracle's own float32 rounding (8 u relative), the same products with a random matrix."""
    n = gh * gw
    idx, coef = grid_neighbours(gh, gw)
    assert torch.equal(idx[:, 0], torch.arange(n))  # the self loop comes first
    ok = idx >= 0
    dense = torch.zeros(n, n, dtype=torch.float64)
    dense.index_put_((torch.arange(n)[:, None].expand(n, 5)[ok], idx[ok]), coef[ok], accumulate=True)
    want = onets.grid_adjacency(gh, gw).double()
    assert torch.equal(dense != 0, want != 0)
    assert ((dense - want).abs() <= 8 * U * dense).all(), (dense - want).abs().max().item()
    assert torch.equal(dense, dense.t())
    v = torch.randn(2, n, 3, dtype=torch.float64, generator=torch.Generator().manual_seed(n))
    got, terms = aggregate64(v, idx, coef)
    assert ((got - want @ v).abs() <= 10 * U * terms).all()
    assert torch.allclose(terms, dense @ v.abs(), rtol=1e-15, atol=0)


# ------------------------------------------------------------------------------------ aggregation through the C ABI
def _abi(v, act, gh, gw):
    """forward (act None: relu(adj v)) or backward (adj (v * (act > 0))) through the C ABI.  The output is a view into a
    buffer with a NaN guard of G floats on each side, which must come back untouched."""
    B, n, H = v.shape
    G = max(H, 256)
    buf = torch.full((B * n * H + 2 * G,), float("nan"), device="cuda")
    out = buf[G:G + B * n * H].view(B, n, H)
    lib = _lib.lib()
    if act is None:
        _lib.check(lib.azg_grid_aggregate_relu_forward(ptr(v), B, gh, gw, H, ptr(out), stream()))
    else:
        _lib.check(lib.azg_grid_aggregate_relu_backward(ptr(v), ptr(act), B, gh, gw, H, ptr(out), stream()))
    assert bool(torch.isnan(buf[:G]).all()) and bool(torch.isnan(buf[G + B * n * H:]).all()), "wrote outside [B, n, H]"
    return out


def _ratio(got, v, act, idx, coef, c=12 * U, step_floats=1 << 22):
    """max over elements of |got - ref| / (c sum_k |a_ik| |v_k|) against the float64 reference, graphs in chunks.
    c = 12 u: five fmaf roundings plus the coefficient's sqrtf, division and product.  A zero bound demands an exact 0.
    A NaN or infinite output (such as an element the kernel never wrote into the NaN-filled buffer of _abi) counts as inf."""
    B, n, H = v.shape
    step = max(1, step_floats // (n * H))
    worst = 0.0
    for b0 in range(0, B, step):
        vb = v[b0:b0 + step].double()
        if act is not None:
            vb = vb * (act[b0:b0 + step] > 0)
        ref, terms = aggregate64(vb, idx, coef)
        if act is None:
            ref = ref.clamp(min=0)
        err = (got[b0:b0 + step].double() - ref).abs()
        r = torch.where(err == 0, 0.0, err / (c * terms))  # an error on a zero bound is inf
        r = torch.where(torch.isfinite(got[b0:b0 + step]), r, float("inf"))
        worst = max(worst, r.max().item())
    return worst


def test_ratio_rejects_unwritten_outputs():
    """_ratio on the CPU: the float64 result rounded to fp32 passes; the same output with its third 256-node chunk, or one
    channel group, left NaN (what _abi's buffer holds where the kernel never writes), or with one wrong value, fails."""
    gh, gw, H = 23, 23, 32
    idx, coef = grid_neighbours(gh, gw)
    g = torch.Generator().manual_seed(1)
    sup = torch.randn(2, gh * gw, H, generator=g)
    dout = torch.randn(2, gh * gw, H, generator=g)
    act = torch.randn(2, gh * gw, H, generator=g)
    for v, a in ((sup, None), (dout, act)):
        ref, _ = aggregate64(v.double() * (a > 0) if a is not None else v.double(), idx, coef)
        good = (ref.clamp(min=0) if a is None else ref).float()
        assert _ratio(good, v, a, idx, coef) <= 1.0
        chunk, group, wrong = good.clone(), good.clone(), good.clone()
        chunk[1, 512:] = float("nan")
        group[0, :, 28:32] = float("nan")
        wrong[1, 300, 5] += 1.0
        assert _ratio(wrong, v, a, idx, coef) > 1e3
        for bad in (chunk, group, torch.full_like(good, float("nan")), torch.full_like(good, float("inf"))):
            assert _ratio(bad, v, a, idx, coef) == float("inf")


def _act(shape, gen):
    """an activation with exact zeros, negative values and -0.0 (none of them passes the mask act > 0)"""
    a = torch.randn(shape, device="cuda", generator=gen)
    r = torch.rand(shape, device="cuda", generator=gen)
    a = torch.where(r < 0.1, torch.zeros((), device="cuda"), a)
    a = torch.where((r >= 0.1) & (r < 0.2), torch.full((), -0.0, device="cuda"), a)
    a.view(-1)[:3] = torch.tensor([0.0, -0.0, -1.0])  # each kind at least once, however small the case
    return a


SHAPES = [(1, 1), (1, 2), (2, 1), (3, 3), (16, 16), (1, 257), (257, 1), (16, 17), (17, 17), (23, 23), (64, 64), (1, 5000)]
HIDDENS = [4, 12, 32, 64, 100, 256, 260, 1024]
SHAPE_CASES = [(gh, gw, H, 3) for gh, gw in SHAPES for H in HIDDENS] + [(182, 182, 4, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("gh,gw,H,B", SHAPE_CASES)
def test_aggregate_every_shape(gh, gw, H, B):
    """azg_grid_aggregate_relu_forward / _backward against float64, |err| <= 12 u sum_k |a_ik| |v_k| per element.
    Graphs of 1 to 33,124 nodes: the neighbour table holds 256 nodes, so 1x257, 257x1, 16x17 and 17x17 take two table
    chunks, 23x23 three, 64x64 16, 1x5000 20 and 182x182 130 (node indices above the 32,767 of an int16).  H / 4 = 1, 3,
    8, 16, 25, 64, 65, 256 channel groups: block shapes 16x16 (idle lanes below 16 groups), 25x10, 64x4, and one to four
    passes of the channel loop.  The backward's mask reads act > 0 at the neighbour; act holds 0, -0.0 and negatives."""
    gen = torch.Generator(device="cuda").manual_seed(gh * 10007 + gw * 31 + H)
    idx, coef = grid_neighbours(gh, gw, "cuda")
    n = gh * gw
    sup = torch.randn(B, n, H, device="cuda", generator=gen)
    dout = torch.randn(B, n, H, device="cuda", generator=gen)
    act = _act((B, n, H), gen)
    e_f = _ratio(_abi(sup, None, gh, gw), sup, None, idx, coef)
    e_b = _ratio(_abi(dout, act, gh, gw), dout, act, idx, coef)
    print(f"aggregate {gh}x{gw} H={H} B={B}: |err| / bound forward {e_f:.3f}, backward {e_b:.3f}")
    assert e_f <= 1.0 and e_b <= 1.0, (e_f, e_b)


BATCH_CASES = [(gh, gw, H, B) for gh, gw in ((7, 7), (17, 17)) for H in (32, 260) for B in (1, 3, GRID, GRID + 1, 5000)
               if B * gh * gw * H <= 1 << 26]


@pytest.mark.gpu
@pytest.mark.parametrize("gh,gw,H,B", BATCH_CASES)
def test_aggregate_batches_past_the_grid(gh, gw, H, B):
    """The kernel runs min(B, 2,368) CTAs and each walks graphs b, b + 2,368, ... (launch_grid_aggregate).  B = 1, 3,
    2,368, 2,369 (one CTA takes a second graph) and 5,000 (three graphs on some CTAs) at 7x7 (one table chunk) and 17x17
    (two chunks), H = 32 and 260 (two passes of the 64-group channel loop), B n H <= 2^26.  Graph b + 2,368 repeats the
    inputs of graph b.  Against float64 (bound of test_aggregate_every_shape); bit-exact, because no arithmetic crosses
    graphs: graph b + 2,368 equals graph b, and the first, last and 2,369th graphs evaluated alone equal their rows."""
    gen = torch.Generator(device="cuda").manual_seed(B * 7 + H + gh)
    idx, coef = grid_neighbours(gh, gw, "cuda")
    n, m = gh * gw, min(B, GRID)
    rep = torch.arange(B, device="cuda") % GRID
    sup = torch.randn(m, n, H, device="cuda", generator=gen)[rep]
    dout = torch.randn(m, n, H, device="cuda", generator=gen)[rep]
    act = _act((m, n, H), gen)[rep]
    out, dsup = _abi(sup, None, gh, gw), _abi(dout, act, gh, gw)
    e_f = _ratio(out, sup, None, idx, coef)
    e_b = _ratio(dsup, dout, act, idx, coef)
    print(f"aggregate {gh}x{gw} H={H} B={B}: |err| / bound forward {e_f:.3f}, backward {e_b:.3f}")
    assert e_f <= 1.0 and e_b <= 1.0, (e_f, e_b)
    if B > GRID:
        assert torch.equal(out[GRID:], out[:B - GRID]) and torch.equal(dsup[GRID:], dsup[:B - GRID])
    for b in sorted({0, B - 1, min(GRID, B - 1)}):
        s = slice(b, b + 1)
        assert torch.equal(_abi(sup[s].contiguous(), None, gh, gw), out[s]), b
        assert torch.equal(_abi(dout[s].contiguous(), act[s].contiguous(), gh, gw), dsup[s]), b


@pytest.mark.gpu
def test_aggregate_refusals():
    """H % 4 != 0, gh = 0, gw = 0 and graphs above 2^30 nodes raise through _lib.check in both directions, before any
    launch; B = 0 returns OK without a launch."""
    lib = _lib.lib()
    t = torch.zeros(64, device="cuda")

    def call(backward, B, gh, gw, H):
        if backward:
            return lib.azg_grid_aggregate_relu_backward(ptr(t), ptr(t), B, gh, gw, H, ptr(t), stream())
        return lib.azg_grid_aggregate_relu_forward(ptr(t), B, gh, gw, H, ptr(t), stream())

    for backward in (False, True):
        name = "azg_grid_aggregate_relu_" + ("backward" if backward else "forward")
        for args in ((1, 2, 2, 6), (1, 0, 3, 4), (1, 3, 0, 4), (1, 32769, 32769, 4), (1, 1 << 20, 1 << 11, 4)):
            torch.cuda.synchronize()
            l0 = lib.azg_launch_count()
            with pytest.raises(RuntimeError, match=name):
                _lib.check(call(backward, *args))
            assert lib.azg_launch_count() == l0, (name, args)
        l0 = lib.azg_launch_count()
        assert call(backward, 0, 2, 2, 4) == _lib.OK
        assert lib.azg_launch_count() == l0


# ------------------------------------------------------------------------------------ the stack
def _tiles(M, N):
    """128 x 128 output tiles of azg_linear_f32: below 222 it runs the training-step kernels, at 222 and above the SGEMM
    (azg_nets.cu, azg_linear_f32)"""
    return -(-M // 128) * -(-N // 128)


def _stack_batches(n, H):
    """B = 3, and the two batches whose B n rows put the Linear on each side of the 222-tile switch"""
    lo = max(B for B in range(1, 222 * 128 + 1) if _tiles(B * n, H) < 222)
    return 3, lo, lo + 1


def _stack64(x, ws, bs, masks, g, idx, coef):
    """float64 stack under the given ReLU masks: its output and the gradients of (output . g) w.r.t. x, weights, biases"""
    x = x.detach().double().requires_grad_(True)
    ws = [w.detach().double().requires_grad_(True) for w in ws]
    bs = [b.detach().double().requires_grad_(True) for b in bs]
    h = x
    for w, b, m in zip(ws, bs, masks):
        h = aggregate64(Fn.linear(h, w, b), idx, coef)[0] * m
    h.backward(g.double())
    out = {"y": h.detach(), "dx": x.grad}
    for i, (w, b) in enumerate(zip(ws, bs)):
        out[f"dW{i}"], out[f"db{i}"] = w.grad, b.grad
    return out


# c: the outputs and gradients end in contractions over H (<= 260), five neighbours and, for the weight gradients, all
# B n rows (<= 28,288), chained through two layers.  Their terms have random signs (g ~ N(0, 1)), so the rounding error
# stays far below sum|terms|; 2^-18 = 64 u, the bound of test_train_pieces_gpu.py.
C_STACK = 2.0 ** -18


@pytest.mark.gpu
@pytest.mark.parametrize("gh,gw", [(16, 16), (17, 17), (1, 300)])
@pytest.mark.parametrize("hidden", [32, 96, 128, 260])
def test_stack_forward_backward(gh, gw, hidden):
    """GridGNNStack(precision="fp32"), two layers: output, x.grad and every dW, db against float64 autograd evaluated under
    the kernel's own ReLU pattern (a pre-activation within rounding of 0 may fall on either side of the ReLU in two
    correct implementations; with the same mask on both sides every element is compared).  Bound per element: C_STACK
    times the same float64 computation on |x|, |W|, |b|, |g| (the sum of the absolute values of every term of the chained
    contractions; adj and the masks are non-negative).  16x16 takes one neighbour-table chunk, 17x17 and 1x300 two; hidden
    32 / 96 / 260 are outside the fused layer's sizes, and 128 is fp32 by choice.  B = 3 and the batches just below and at
    the 222-tile switch of azg_linear_f32 (e.g. 17x17, H = 128: 97 graphs = 220 tiles, 98 = 222)."""
    n = gh * gw
    idx, coef = grid_neighbours(gh, gw, "cuda")
    worst = {}
    for B in _stack_batches(n, hidden):
        torch.manual_seed(B * 13 + hidden + n)
        net = GridGNNStack(gh, gw, hidden, layers=2, precision="fp32").cuda()
        assert not net.fused
        x = torch.randn(B, n, hidden, device="cuda", requires_grad=True)
        with torch.no_grad():  # the per-layer outputs, through the same kernels as net(x)
            outs, h = [], x
            for lin in net.gnn_layers:
                h = _GridAggRelu.apply(_Linear.apply(h.reshape(B * n, hidden), lin.weight, lin.bias, False).reshape(B, n, hidden),
                                       gh, gw)
                outs.append(h)
        y = net(x)
        assert torch.equal(y, outs[-1])
        g = torch.randn_like(y)
        y.backward(g)
        got = {"y": y.detach(), "dx": x.grad}
        for i, lin in enumerate(net.gnn_layers):
            got[f"dW{i}"], got[f"db{i}"] = lin.weight.grad, lin.bias.grad
        ws, bs = [l.weight for l in net.gnn_layers], [l.bias for l in net.gnn_layers]
        masks = [(o > 0).double() for o in outs]
        ref = _stack64(x, ws, bs, masks, g, idx, coef)
        terms = _stack64(x.abs(), [w.abs() for w in ws], [b.abs() for b in bs], masks, g.abs(), idx, coef)
        for k in got:
            err = (got[k].double() - ref[k]).abs()
            r = torch.where(err == 0, 0.0, err / (C_STACK * terms[k]))
            r = torch.where(torch.isfinite(got[k]), r, float("inf")).max().item()
            worst[k] = max(worst.get(k, 0.0), r)
            assert r <= 1.0, (B, k, r)
    print(f"stack {gh}x{gw} H={hidden} B={_stack_batches(n, hidden)} tiles {[_tiles(B * n, hidden) for B in _stack_batches(n, hidden)]}: "
          f"max |err| / bound {worst}")


@pytest.mark.gpu
@pytest.mark.parametrize("gh,gw,H,fused", [(16, 16, 128, True), (16, 17, 128, False), (1, 257, 128, False), (8, 8, 96, False),
                                           (8, 8, 512, False)])
def test_stack_routing(gh, gw, H, fused):
    """A stack is fused exactly when azg_grid_tc_supported says so (at most 256 nodes, H in {64, 128, 256}).  A "bf16x3" or
    "bf16" stack that is not fused runs the fp32 kernels: outputs and gradients bit-identical to the "fp32" stack with the
    same weights."""
    assert bool(_lib.lib().azg_grid_tc_supported(gh, gw, H)) == fused
    torch.manual_seed(H + gh * gw)
    nets = {p: GridGNNStack(gh, gw, H, layers=2, precision=p).cuda() for p in ("fp32", "bf16x3", "bf16")}
    assert not nets["fp32"].fused
    for p in ("bf16x3", "bf16"):
        assert nets[p].fused == fused, p
        nets[p].load_state_dict(nets["fp32"].state_dict())
    if fused:
        return
    x0 = torch.randn(5, gh * gw, H, device="cuda")
    g = torch.randn_like(x0)
    res = {}
    for p, net in nets.items():
        x = x0.clone().requires_grad_(True)
        y = net(x)
        y.backward(g)
        res[p] = [y.detach(), x.grad] + [q.grad for q in net.parameters()]
    for p in ("bf16x3", "bf16"):
        for a, b in zip(res[p], res["fp32"]):
            assert torch.equal(a, b), p
