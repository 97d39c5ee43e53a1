"""Training pieces (K3) through the C ABI against float64, at the sizes training reaches and across the thresholds that
switch their code paths.  test_train_gpu.py checks them only inside whole training steps at batch <= 64.

fp32 kernels are held to scale-aware bounds, |err| <= c * sum|terms| (the sum of the absolute values of the terms the
kernel adds, computed in float64), as test_gemm_gpu.py::test_gemm_f32_matches_torch does; each test states its c.
u = 2^-24 is the unit roundoff of fp32."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as Fn

from oracle import nets as onets

from azgnn_b200 import _lib
from azgnn_b200._lib import ptr, stream

pytestmark = pytest.mark.gpu
U = 2.0 ** -24


def _launches():
    torch.cuda.synchronize()
    return _lib.lib().azg_launch_count()


# ------------------------------------------------------------------------------------ conv3x3 + ReLU
LAYERS = [(1, 32, 1), (32, 64, 1), (64, 128, 0)]  # conv1 / conv2 of both games (pad 1), TicTacToe conv3 (pad 0)


def _conv_case(B, Cin, Cout, n, pad, seed):
    """forward and backward through the ABI, float64 references and the sum|terms| of each output"""
    lib = _lib.lib()
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.relu(torch.randn(B, Cin, n, n, device="cuda", generator=g))  # post-ReLU activations, as in the nets
    if Cin == 1:
        x = torch.randint(-1, 2, (B, 1, n, n), device="cuda", generator=g).float()  # board planes
    w = torch.randn(Cout, Cin, 3, 3, device="cuda", generator=g) / (3 * Cin ** 0.5)
    b = torch.randn(Cout, device="cuda", generator=g) * 0.1
    Ho = n + 2 * pad - 2
    out = torch.empty(B, Cout, Ho, Ho, device="cuda")
    _lib.check(lib.azg_conv3x3_relu_forward(ptr(x), ptr(w), ptr(b), ptr(out), B, Cin, Cout, n, n, pad, stream()))
    dout = torch.randn(B, Cout, Ho, Ho, device="cuda", generator=g)
    din, dw, db = torch.empty_like(x), torch.empty_like(w), torch.empty_like(b)
    l0 = _launches()
    _lib.check(lib.azg_conv3x3_relu_backward(ptr(x), ptr(w), ptr(out), ptr(dout), ptr(din), ptr(dw), ptr(db), B, Cin, Cout, n, n, pad,
                                             stream()))
    launches = _launches() - l0
    xd, wd, bd = x.double(), w.double(), b.double()
    pre = Fn.conv2d(xd, wd, bd, padding=pad)
    # The backward reference takes its ReLU gate from the kernel's own forward output.  A pre-activation within rounding of
    # 0 may land on the other side of the ReLU than in float64 (test_train_gpu.py tolerates two such rows per gradient);
    # gating both sides alike removes that case, so every element is compared.
    gd = dout.double() * (out > 0)
    ga = gd.abs()
    got = {"out": out, "din": din, "dw": dw, "db": db}
    ref = {"out": torch.relu(pre), "din": torch.nn.grad.conv2d_input(x.shape, wd, gd, padding=pad),
           "dw": torch.nn.grad.conv2d_weight(xd, w.shape, gd, padding=pad), "db": gd.sum(dim=(0, 2, 3))}
    terms = {"out": Fn.conv2d(xd.abs(), wd.abs(), bd.abs(), padding=pad), "din": torch.nn.grad.conv2d_input(x.shape, wd.abs(), ga, padding=pad),
             "dw": torch.nn.grad.conv2d_weight(xd.abs(), w.shape, ga, padding=pad), "db": ga.sum(dim=(0, 2, 3))}
    ratio = {k: ((got[k].double() - ref[k]).abs() / (terms[k] + 1e-30)).max().item() for k in got}
    return ratio, launches


# c: a rounding per added term on partial sums of random-sign terms (dout ~ N(0,1)) stays far below sum|terms|; 2^-18 is
# 64 u, the same order as the 2e-6 of test_gemm_f32_matches_torch, and holds up to the 420,000-term serial sums of the
# direct weight-gradient kernel
C_CONV = 2.0 ** -18


@pytest.mark.parametrize("n", [3, 4, 5, 6, 7, 8])
@pytest.mark.parametrize("Cin,Cout,pad", LAYERS)
def test_conv3x3_relu_forward_backward(n, Cin, Cout, pad):
    """azg_conv3x3_relu_forward / _backward against float64 conv2d and its gradients (out, din, dw, db).  The backward picks
    its branch from R = B*Ho*Wo (azg_train.cu, azg_conv3x3_relu_backward: `if (R >= 256 && n_g + 2 * n_c <= 2^28)`):
    direct kernels below R = 256 (two launches with din), pack + split-K GEMM at and above it (at least five).  B =
    floor(255 / P) (R just below 256; one board when P > 255 cannot happen here), B = ceil(256 / P) (R just at or above
    256) and B = 64, P = Ho*Wo.  The third branch (direct kernels above the 2^28-element pack) is
    test_conv3x3_backward_above_the_pack_bound."""
    P = (n + 2 * pad - 2) ** 2
    for B in sorted({max(1, 255 // P), -(-256 // P), 64}):
        R = B * P
        ratio, launches = _conv_case(B, Cin, Cout, n, pad, seed=B * 131 + n * 7 + Cin)
        print(f"conv {Cin}->{Cout} pad {pad} n={n} B={B} R={R}: {launches} launches, max |err| / sum|terms| {ratio}")
        assert (launches == 2) if R < 256 else (launches >= 5), (R, launches)
        assert max(ratio.values()) <= C_CONV, ratio


@pytest.mark.parametrize("B", [8559, 8560])
def test_conv3x3_backward_above_the_pack_bound(B):
    """The pack + GEMM backward needs n_g + 2 n_c = R * (Cout + 2 * 9 * Cin) floats of scratch and runs while that is <=
    2^28 (azg_train.cu, azg_conv3x3_relu_backward).  Connect4 conv2 at n = 7 (Cin 32, Cout 64, R = 49 B): R * 640 <= 2^28
    up to B = 8,559 (pack + GEMM, at least five launches); B = 8,560 runs the direct kernels again (two launches)."""
    ratio, launches = _conv_case(B, 32, 64, 7, 1, seed=B)
    print(f"conv 32->64 n=7 B={B} R={49 * B} pack floats {49 * B * 640} (2^28 = {2 ** 28}): {launches} launches, "
          f"max |err| / sum|terms| {ratio}")
    assert (launches == 2) if 49 * B * 640 > 2 ** 28 else (launches >= 5), launches
    assert max(ratio.values()) <= C_CONV, ratio


# ------------------------------------------------------------------------------------ policy / value loss
@pytest.mark.parametrize("B", [1, 255, 256, 257, 5000])
@pytest.mark.parametrize("A", [5, 8, 10, 17, 65])
def test_policy_value_loss(B, A):
    """azg_policy_value_loss runs as ONE CTA whose 256 threads stride over the rows (policy_value_loss_kernel): B = 1,
    255 / 256 / 257 (one row per thread, then a second pass for one thread) and 5,000 (20 rows per thread); A = 5 .. 65
    (the action counts of FrozenLake, Connect4 4 / 7 and TicTacToe 4 / 8).  Logits up to +-60, target rows with zeros and
    with sums from 0.5 to 2, norm = 4 B (the data-parallel case: every rank divides by the global batch).  Against float64
    log_softmax / tanh and their autograd gradients.  Bounds, with lse the row's log-sum-exp after subtracting the max m:
    logp: (A + 4) u (|l - m| + |lse| + 1); dlogits: that error plus (A + 4) u (the serial sum(t)) relative on
    softmax * sum(t), plus 4 u |t|, over norm, plus what fp32 cannot resolve below its normal range (a softmax of e^-100
    is subnormal: 2^-126 (sum(t) + 1) / norm, and 2^-149 on the result); v: 4 u; dvraw: 16 u (2 |t_v - v| + 1) / norm; loss: the logp errors
    weighted by t plus (A + B / 256 + 12) u sum|terms| for the per-row, thread-serial and tree sums, over norm."""
    lib = _lib.lib()
    g = torch.Generator().manual_seed(B * 100 + A)
    logits = (torch.rand(B, A, generator=g) * 2 - 1) * 60
    vraw = torch.randn(B, generator=g) * 2
    tpi = torch.rand(B, A, generator=g) * (torch.rand(B, A, generator=g) > 0.3)
    tpi = tpi / tpi.sum(1, keepdim=True).clamp(min=1e-6) * (0.5 + 1.5 * torch.rand(B, 1, generator=g))
    tv = torch.rand(B, generator=g) * 2 - 1
    norm = 4.0 * B
    dev = [t.cuda().contiguous() for t in (logits, vraw, tpi, tv)]
    loss, logp, v = torch.empty(1, device="cuda"), torch.empty(B, A, device="cuda"), torch.empty(B, device="cuda")
    dlogits, dvraw = torch.empty(B, A, device="cuda"), torch.empty(B, device="cuda")
    _lib.check(lib.azg_policy_value_loss(*[ptr(t) for t in dev], B, A, norm, ptr(loss), ptr(logp), ptr(v), ptr(dlogits), ptr(dvraw),
                                         stream()))
    L = logits.double().requires_grad_(True)
    R = vraw.double().requires_grad_(True)
    t, tvd = tpi.double(), tv.double()
    lp = torch.log_softmax(L, dim=1)
    vv = torch.tanh(R)
    per_row = -(t * lp).sum(1) + (tvd - vv) ** 2
    ref_loss = per_row.sum() / norm
    ref_loss.backward()
    m = L.detach().max(1, keepdim=True).values
    lse = torch.logsumexp(L.detach() - m, dim=1, keepdim=True)
    lp_scale = (L.detach() - m).abs() + lse.abs() + 1
    lp_tol = (A + 4) * U * lp_scale
    sm_sum = lp.detach().exp() * t.sum(1, keepdim=True)
    d_tol = (sm_sum * (lp_tol + (A + 4) * U) + 4 * U * t + 2.0 ** -126 * (t.sum(1, keepdim=True) + 1)) / norm + 2.0 ** -149
    dv_tol = 16 * U * (2 * (tvd - vv.detach()).abs() + 1) / norm
    terms = (t * lp.detach()).abs().sum() + ((tvd - vv.detach()) ** 2).sum()
    loss_tol = ((t * lp_tol).sum() + (A + B / 256 + 12) * U * terms) / norm
    e = {"loss": abs(loss.item() - ref_loss.item()) / loss_tol.item(),
         "logp": ((logp.double().cpu() - lp.detach()).abs() / lp_tol).max().item(),
         "v": (v.double().cpu() - vv.detach()).abs().max().item() / (4 * U),
         "dlogits": ((dlogits.double().cpu() - L.grad).abs() / d_tol).max().item(),
         "dvraw": ((dvraw.double().cpu() - R.grad).abs() / dv_tol).max().item()}
    print(f"loss B={B} A={A}: |err| / bound {e}, loss {loss.item():.6f}")
    assert max(e.values()) <= 1.0, e


# ------------------------------------------------------------------------------------ GNNLayer
_KEYS = ("attention.0.weight", "attention.0.bias", "attention.2.weight", "attention.2.bias", "update_net.0.weight", "update_net.0.bias",
         "update_net.2.weight", "update_net.2.bias", "gate.0.weight", "gate.0.bias")  # the order of azg_gnn_layer_params


def _offset(t, shift):
    """a copy of t whose data pointer sits `shift` floats past a 16-byte boundary"""
    buf = torch.empty(t.numel() + 4, device="cuda")
    view = buf[shift:shift + t.numel()].view(t.shape)
    view.copy_(t)
    return view


def _gnn_case(P, F, shift):
    lib = _lib.lib()
    g = torch.Generator().manual_seed(P * 13 + F)
    shapes = [(128, 2 * F), (128,), (1, 128), (1,), (F, 2 * F), (F,), (F, F), (F,), (F, 2 * F), (F,)]
    params = [(torch.rand(s, generator=g) * 2 - 1) / (s[-1] ** 0.5) for s in shapes]
    f0, path = torch.randn(F, generator=g) * 0.5, torch.randn(P, F, generator=g) * 0.5
    d_out0 = torch.randn(F, generator=g)
    dp = [_offset(p.cuda(), shift) for p in params]
    grads = [_offset(torch.zeros(p.shape), shift) for p in params]
    f0d, pathd, doutd = f0.cuda(), path.cuda(), d_out0.cuda()
    out0 = torch.empty(F, device="cuda")
    d_f0 = torch.empty(F, device="cuda")
    saved = torch.empty(lib.azg_gnn_layer_saved_floats(P, F), device="cuda")
    scratch = torch.empty(lib.azg_gnn_layer_scratch_floats(P, F), device="cuda")
    cp = _lib.GNNLayerParams(*[ptr(p) for p in dp])
    cg = _lib.GNNLayerGrads(*[ptr(q) for q in grads])
    _lib.check(lib.azg_gnn_layer_forward(C.byref(cp), ptr(f0d), ptr(pathd), P, F, ptr(out0), ptr(saved), stream()))
    _lib.check(lib.azg_gnn_layer_backward(C.byref(cp), ptr(f0d), ptr(pathd), P, F, ptr(saved), ptr(doutd), ptr(d_f0), C.byref(cg),
                                          ptr(scratch), stream()))
    # float64 autograd of oracle.nets.gnn_layer on the GPU
    p64 = {k: p.cuda().double().requires_grad_(True) for k, p in zip(_KEYS, params)}
    f064 = f0.cuda().double().requires_grad_(True)
    out = onets.gnn_layer(p64, "", torch.cat([f064[None], path.cuda().double()]))
    (out[0] * d_out0.cuda().double()).sum().backward()
    got = {"out0": out0, "d_f0": d_f0, **{k: q for k, q in zip(_KEYS, grads)}}
    ref = {"out0": out[0].detach(), "d_f0": f064.grad, **{k: p64[k].grad for k in _KEYS}}
    scale = {k: ref[k].abs().max() for k in ref}
    # alpha = s / sum(s): the attention gradients are differences d_alpha_i / t - (d_alpha . s) / t^2 that cancel (exactly,
    # at P = 1).  Their scale is that of the terms before the cancellation: the gradients of the layer without the
    # normalisation (alpha = s), divided by t = sum(s).
    q64 = {k: p.cuda().double().requires_grad_(True) for k, p in zip(_KEYS, params)}
    path64, f0n = path.cuda().double(), f0.cuda().double()
    comb = torch.cat([f0n[None].expand(P, -1), path64], dim=1)
    s = torch.sigmoid(Fn.linear(torch.relu(Fn.linear(comb, q64[_KEYS[0]], q64[_KEYS[1]])), q64[_KEYS[2]], q64[_KEYS[3]]))
    cat2 = torch.cat([f0n, (path64 * s).sum(0)])
    upd = Fn.linear(torch.relu(Fn.linear(cat2, q64[_KEYS[4]], q64[_KEYS[5]])), q64[_KEYS[6]], q64[_KEYS[7]])
    ((f0n + torch.sigmoid(Fn.linear(cat2, q64[_KEYS[8]], q64[_KEYS[9]])) * upd) * d_out0.cuda().double()).sum().backward()
    t = s.detach().sum()
    for k in _KEYS[:4]:
        scale[k] = torch.maximum(scale[k], q64[k].grad.abs().max() / t)
    return {k: ((got[k].double() - ref[k]).abs().max() / scale[k].clamp(min=1e-30)).item() for k in got}


# c: every gradient here ends in contractions of length <= 2F = 8,192 or P = 1,023 whose terms have random signs, so the
# rounding error of each is about u sqrt(K) of its largest entry (5e-6 at K = 8,192); three such stages chain (attention,
# its softmax-like normalisation, the weight gradient).  Bound: 2^-14 (6e-5) of the tensor's largest entry (for the
# attention gradients, of their terms before the normalisation's cancellation; see _gnn_case).
C_GNN = 2.0 ** -14


@pytest.mark.parametrize("P", [1, 2, 63, 64, 255, 1023])
@pytest.mark.parametrize("F", [512, 1152, 3136, 4096])
def test_gnn_layer_forward_backward(P, F):
    """azg_gnn_layer_forward / _backward (GNNLayer at B = P + 1) against float64 autograd of oracle.nets.gnn_layer: out0,
    every parameter gradient and d_f0.  P = 1 and 2 (the smallest graphs), 63 / 64 (a 64-row tile of the fp32 GEMMs),
    255 and 1,023 (longer paths than any earlier test); F = 512 (TicTacToe 4x4), 1,152 (TicTacToe 5x5), 3,136 (Connect4
    7x7), 4,096 (Connect4 8x8).  |err| <= 2^-14 max|ref| per tensor (see C_GNN)."""
    e = _gnn_case(P, F, 0)
    print(f"gnn layer P={P} F={F}: max |err| / max|ref| {e}")
    assert max(e.values()) <= C_GNN, e


@pytest.mark.parametrize("P,F", [(2, 512), (64, 1152), (255, 4096)])
def test_gnn_layer_backward_unfused_fallback(P, F):
    """The backward streams each weight matrix once (rank1_bwd: weight gradient and input gradient in one pass) when
    rank1_ok holds for the gate, update_net.0 and update_net.2 matrices and their gradients (azg_train.cu,
    azg_gnn_layer_backward: `const bool fused = rank1_ok(...)`), which needs 16-byte aligned pointers.  Weight and gradient
    buffers offset by one float make rank1_ok (and gemv_rows_ok in the forward) false, so the separate GEMMs run: same
    float64 references and bound as test_gnn_layer_forward_backward."""
    e = _gnn_case(P, F, 1)
    print(f"gnn layer (unaligned weights: GEMM fallback) P={P} F={F}: max |err| / max|ref| {e}")
    assert max(e.values()) <= C_GNN, e


# ------------------------------------------------------------------------------------ FrozenLake graph aggregation
@pytest.mark.parametrize("E", [64, 128, 200])
def test_graph_mean_relu(E):
    """azg_graph_mean_relu_forward / _backward (FrozenLake's all-ones normalised adjacency, 3..5 nodes per graph) with
    node counts 3, 4 and 5 mixed in one batch of 1,000 graphs, E = 64, 128 and 200 (not a multiple of 64), against float64
    relu(adj @ sup) per graph and its gradient.  Forward bound (k + 2) u sum|terms|; the backward reference takes its ReLU
    gate from the kernel's forward output (a knife-edge pre-activation cannot flip an element), bound (k + 2) u sum|terms|."""
    lib = _lib.lib()
    B = 1000
    g = torch.Generator().manual_seed(E)
    counts = torch.randint(3, 6, (B,), generator=g, dtype=torch.int32)
    valid = (torch.arange(5)[None, :] < counts[:, None].long()).double()[..., None]  # [B, 5, 1]
    sup = (torch.randn(B, 5, E, generator=g).double() * valid).float()
    dout = (torch.randn(B, 5, E, generator=g).double() * valid).float()
    sd, cd, dd = sup.cuda(), counts.cuda(), dout.cuda()
    out, dsup = torch.empty_like(sd), torch.empty_like(sd)
    _lib.check(lib.azg_graph_mean_relu_forward(ptr(sd), ptr(cd), B, E, ptr(out), stream()))
    _lib.check(lib.azg_graph_mean_relu_backward(ptr(dd), ptr(out), ptr(cd), B, E, ptr(dsup), stream()))
    k = counts.double()[:, None, None]
    s64, d64 = sup.double(), dout.double()
    pre = s64.sum(1, keepdim=True) / k  # adj = 1/k everywhere: every valid node gets the same row
    ref_out = torch.relu(pre) * valid
    gate = (out.cpu()[:, :1] > 0).double()
    ref_dsup = gate * d64.sum(1, keepdim=True) / k * valid
    tol_f = (k + 2) * U * (s64.abs().sum(1, keepdim=True) / k) + 1e-30
    tol_b = (k + 2) * U * (d64.abs().sum(1, keepdim=True) / k) + 1e-30
    e_f = ((out.cpu().double() - ref_out).abs() / tol_f).max().item()
    e_b = ((dsup.cpu().double() - ref_dsup).abs() / tol_b).max().item()
    print(f"graph mean relu E={E}: |err| / bound forward {e_f:.3f}, backward {e_b:.3f}")
    assert e_f <= 1.0 and e_b <= 1.0
