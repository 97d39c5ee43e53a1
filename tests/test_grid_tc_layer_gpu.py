"""The fused tensor-core grid layer (csrc/azg_grid_tc.cu) against float64, element by element, in every kernel it
instantiates.  GridGNNStack runs it for "bf16x3" and "bf16" whenever gh*gw <= 256 and H is 64, 128 or 256.

    forward          out = relu(adj (x W^T + b))
    backward_input   dx  = adj ((dout * [act > 0]) W)

grid_layer_tc_kernel<H, X3, BWD, MT, PAIR>: X3 = bf16x3 (three products) or bf16 (one), BWD = backward_input, MT = 1
(128-row tiles) or 2 (256-row tiles), PAIR = a CTA pair that shares one weight operand.  The shared-memory plan
(GridSmem) decides WRES (weight images resident for the life of the CTA; otherwise every stage streams its k-block of
them from L2), EC (columns per epilogue chunk; 16 means 64-byte staging rows with XOR-swizzled 16-byte units) and NTILE
(staging tiles: 2 = two epilogue groups of four warps alternating chunks, 1 = one group of eight warps).  Each line is
two instantiations, forward and backward:

    H    X3      MT  PAIR  WRES  EC  NTILE   chosen for
    64   bf16x3  1   -     yes   32  2       <= 128 nodes, unless 256-row tiles waste fewer rows (1x1, 3x3, 11x11)
    64   bf16x3  2   -     yes   32  2       7x7, 9x9, 1x85 and everything above 128 nodes
    64   bf16    1   -     yes   32  2       <= 128 nodes, unless 256-row tiles waste far fewer rows (3x3, 7x7)
    64   bf16    2   -     yes   32  2       9x9, 1x85 and everything above 128 nodes
    128  the same four lines as H = 64
    256  bf16x3  1   pair  yes   16  2       <= 128 nodes
    256  bf16x3  1   -     no    16  2       <= 128 nodes with AZG_GRID_PAIR=0
    256  bf16x3  2   -     no    16  1       above 128 nodes; <= 128 with AZG_GRID_TILE=256
    256  bf16    1   -     yes   32  2       <= 128 nodes
    256  bf16    2   -     yes   16  2       above 128 nodes; <= 128 with AZG_GRID_TILE=256

`instantiation` mirrors the library's choice (wide_tiles, dispatch_h) and a CPU test checks that CASES reach all 26.

Reference: the operands split as split_pair (azg_tc.cuh) does, hi = bf16(x), lo = bf16(x - hi), and the products the
kernel issues (bf16x3: Xh Wh^T + Xh Wl^T + Xl Wh^T; bf16: Xh Wh^T) summed in float64, then aggregated through the
neighbour table of helpers.grid_neighbours.  Bound per element: 2^-18 adj T (T = the sum of the absolute product terms:
the fp32 accumulation in tensor memory, as in test_forward_thresholds_gpu.py::test_bf16x3_matches_its_exact_emulation)
+ 12 u (adj |D| + |rowsum b|) (the epilogue's fp32 staging, five-term gather, coefficients and fmaf, as in
test_grid_fp32_path_gpu.py).  u = 2^-24."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import nets as onets

from azgnn_b200 import _lib
from azgnn_b200._lib import ptr, stream

from helpers import aggregate64, grid_neighbours

U = 2.0 ** -24
C_MMA = 2.0 ** -18
C_EPI = 12 * U
SMS = 148  # B200: persistent CTAs of one launch (pairs: 74)
NAN = float("nan")


# ------------------------------------------------------------------------------------ which kernel runs
def wide_tiles(n, H, x3, env):
    """azg_grid_tc.cu wide_tiles: 256-row tiles above 128 nodes, or when they waste fewer rows (float32 arithmetic)"""
    if n > 128:
        return True
    if env.get("AZG_GRID_TILE") in ("256", "128"):
        return env["AZG_GRID_TILE"] == "256"
    if H > 128:
        return False
    f = np.float32
    u1 = f((128 // n) * n) / f(128.0)
    u2 = f((256 // n) * n) / f(256.0)
    return bool(u2 - u1 > f(0.1 if x3 else 0.25))


def instantiation(gh, gw, H, x3, bwd, env):
    """(H, X3, BWD, MT, PAIR) of the kernel the library launches (dispatch, dispatch_h)"""
    mt = 2 if wide_tiles(gh * gw, H, x3, env) else 1
    pair = H == 256 and x3 and mt == 1 and env.get("AZG_GRID_PAIR") != "0"
    return (H, x3, bwd, mt, pair)


ALL_INSTANTIATIONS = {(H, x3, bwd, mt, pair) for H in (64, 128, 256) for x3 in (True, False) for bwd in (False, True)
                      for mt in (1, 2) for pair in (False, True) if not pair or (H == 256 and x3 and mt == 1)}

SHAPES_128 = [(1, 1), (1, 2), (2, 1), (3, 3), (7, 7), (9, 9), (11, 11), (1, 85), (1, 128), (128, 1), (1, 129), (13, 10),
              (2, 100), (16, 16), (1, 256), (256, 1)]
SHAPES_64 = [(1, 1), (3, 3), (7, 7), (9, 9), (16, 16)]
SHAPES_256 = [(1, 1), (3, 3), (9, 9), (11, 11), (1, 129), (16, 16), (256, 1)]
ENVS = {"nopair": {"AZG_GRID_PAIR": "0"}, "tile256": {"AZG_GRID_TILE": "256"}}
CASES = ([(gh, gw, 128, "") for gh, gw in SHAPES_128] + [(gh, gw, 64, "") for gh, gw in SHAPES_64]
         + [(gh, gw, 256, "") for gh, gw in SHAPES_256]
         + [(3, 3, 256, "nopair"), (11, 11, 256, "nopair"), (9, 9, 256, "tile256"), (1, 85, 256, "tile256")])


def _case_id(c):
    return f"{c[0]}x{c[1]}-H{c[2]}" + (f"-{c[3]}" if c[3] else "")


def test_cases_cover_every_instantiation():
    """ALL_INSTANTIATIONS is what dispatch_h can launch: 26 kernels.  Every one is run by some case, in both precisions'
    own instantiations, forward and backward."""
    assert len(ALL_INSTANTIATIONS) == 26
    got = {instantiation(gh, gw, H, x3, bwd, ENVS.get(e, {})) for gh, gw, H, e in CASES for x3 in (True, False)
           for bwd in (False, True)}
    assert got == ALL_INSTANTIATIONS, sorted(ALL_INSTANTIATIONS - got)
    # 7x7 takes 256-row tiles in bf16x3 only, 9x9 in both (graph 1 across the halves); 129 nodes is the first graph that needs them
    assert instantiation(7, 7, 128, True, False, {})[3] == 2 and instantiation(7, 7, 128, False, False, {})[3] == 1
    assert instantiation(9, 9, 128, True, False, {})[3] == 2 and instantiation(9, 9, 128, False, False, {})[3] == 2
    assert instantiation(1, 128, 128, True, False, {})[3] == 1 and instantiation(1, 129, 128, False, False, {})[3] == 2


# ------------------------------------------------------------------------------------ float64 reference
def split(t):
    """fp32 -> (hi, lo) in float64 as split_pair: hi = bf16(t), lo = bf16(t - hi)"""
    hi = t.bfloat16()
    return hi.double(), (t - hi.float()).bfloat16().double()


def products(a, w, x3):
    """the (A part, B part) pairs of the kernel's tensor-core products of a [rows, K] and the B operand w [N, K]"""
    ah, al = split(a)
    wh, wl = split(w)
    return [(ah, wh), (ah, wl), (al, wh)] if x3 else [(ah, wh)]


def corrections(x3):
    """indices into products() of what a kernel could drop on one k-block: the two correction products of bf16x3, the
    only product of bf16"""
    return (1, 2) if x3 else (0,)


def emulate(x, w, b, act, idx, coef, x3, drop=None):
    """The layer as the kernel computes it, in float64, for x [B, n, H] fp32 (dout when act is given), w the [H, H] weight
    (nn.Linear: [out, in]) and b its bias (forward only).  Returns (output, bound).  drop = (product, k-block) leaves that
    one product out on that one 64-wide k-block."""
    B, n, H = x.shape
    a = x.reshape(B * n, H)
    if act is not None:  # the gate as the kernel's m > 0 ? x : 0 -- a NaN in a closed entry is dropped, not propagated
        a = torch.where(act.reshape(B * n, H) > 0, a, torch.zeros((), device=a.device))
        w = w.t()  # dx = G W = G (W^T)^T
    d = t = 0.0
    for i, (p, q) in enumerate(products(a, w, x3)):
        t = t + p.abs() @ q.abs().t()
        if drop is not None and drop[0] == i:
            p = p.clone()
            p[:, 64 * drop[1]:64 * drop[1] + 64] = 0.0
        d = d + p @ q.t()
    out, absd = aggregate64(d.view(B, n, H), idx, coef)
    bound = C_MMA * aggregate64(t.view(B, n, H), idx, coef)[0] + C_EPI * absd
    if act is None:
        rb = coef.sum(1)[:, None] * b.double()  # adj (1 b^T) = rowsum(adj) b^T
        out = (out + rb).clamp(min=0)
        bound = bound + C_EPI * rb.abs()
    return out, bound


def ratio(got, ref, bound):
    """max over elements of |got - ref| / bound.  A zero bound demands an exact match; a NaN or infinite output (such
    as an element the kernel never wrote into run()'s NaN-filled buffer) counts as an infinite error."""
    err = (got.double() - ref).abs()
    r = torch.where(err == 0, 0.0, err / bound)
    return torch.where(torch.isfinite(got), r, float("inf")).max().item()


def drop_margin(x, w, b, act, idx, coef, x3, ref, bound):
    """min over k-blocks and droppable products of max over elements of |change| / bound, where change is what leaving
    that product out on that k-block does to the output: >= 10 means such a kernel fails by ten times the bound"""
    worst = float("inf")
    for i in corrections(x3):
        for k in range(x.shape[-1] // 64):
            change = (emulate(x, w, b, act, idx, coef, x3, drop=(i, k))[0] - ref).abs()
            worst = min(worst, torch.where(change == 0, 0.0, change / bound).max().item())
    return worst


def _act(shape, gen, device):
    """a ReLU output for the gate: positive, 0, -0.0, negative and NaN entries (only the positive ones open it)"""
    a = torch.randn(shape, device=device, generator=gen)
    r = torch.rand(shape, device=device, generator=gen)
    a = torch.where(r < 0.1, torch.zeros((), device=device), a)
    a = torch.where((r >= 0.1) & (r < 0.2), torch.full((), -0.0, device=device), a)
    a = torch.where((r >= 0.2) & (r < 0.25), torch.full((), NAN, device=device), a)
    a.view(-1)[:4] = torch.tensor([0.0, -0.0, -1.0, NAN])  # each kind at least once, however small the case
    return a


def _dout(shape, act, gen, device):
    """an upstream gradient with NaN in a third of the entries the gate closes"""
    g = torch.randn(shape, device=device, generator=gen)
    r = torch.rand(shape, device=device, generator=gen)
    return torch.where(~(act > 0) & (r < 0.33), torch.full((), NAN, device=device), g)


def _weights(H, gen, device):
    w = (torch.rand(H, H, device=device, generator=gen) * 2 - 1) / H ** 0.5  # nn.Linear's init range
    b = torch.randn(H, device=device, generator=gen) * 0.5
    return w, b


# ------------------------------------------------------------------------------------ CPU checks of the reference
@pytest.mark.parametrize("gh,gw", [(1, 1), (3, 3), (2, 5), (9, 9)])
def test_emulation_matches_dense_oracle(gh, gw):
    """On bf16-representable inputs (every lo part is 0) both precisions' emulations are the exact layer: forward
    against relu(grid_adjacency (x W^T + b)) and backward against grid_adjacency ((dout * [act > 0]) W), both with the
    dense oracle.nets.grid_adjacency in float64.  The oracle's coefficients are float32 (8 u), so 10 u of the terms."""
    n, H, B = gh * gw, 128, 3
    g = torch.Generator().manual_seed(n)
    bf = lambda t: t.bfloat16().float()  # noqa: E731
    x = bf(torch.randn(B, n, H, generator=g))
    w, b = _weights(H, g, "cpu")
    w, b = bf(w), bf(b)
    act = _act((B, n, H), g, "cpu")
    dout = bf(_dout((B, n, H), act, g, "cpu"))
    idx, coef = grid_neighbours(gh, gw)
    adj = onets.grid_adjacency(gh, gw).double()
    pre = x.double() @ w.double().t() + b.double()
    gate = torch.where(act > 0, dout, torch.zeros(())).double()
    want = {False: (adj @ pre).clamp(min=0), True: adj @ (gate @ w.double())}
    terms = {False: adj @ pre.abs(), True: adj @ (gate.abs() @ w.double().abs())}
    for x3 in (True, False):
        for bwd in (False, True):
            got, _ = emulate(dout if bwd else x, w, b, act if bwd else None, idx, coef, x3)
            assert ((got - want[bwd]).abs() <= 10 * U * terms[bwd]).all(), (x3, bwd)


def test_comparison_rejects_wrong_outputs():
    """The comparison on the CPU, 9x9 graphs (three per 256-row tile, graph 1 across the halves), H = 128: the float64
    emulation rounded to fp32 passes.  It fails with one k-block's Xl Wh^T left out (bf16x3), the second half of a tile or
    one 32-column chunk left NaN (what run()'s buffer holds where the kernel never writes), or one element off by 1e-3."""
    gh, gw, H, B = 9, 9, 128, 6
    g = torch.Generator().manual_seed(3)
    idx, coef = grid_neighbours(gh, gw)
    x = torch.randn(B, gh * gw, H, generator=g)
    w, b = _weights(H, g, "cpu")
    act = _act(x.shape, g, "cpu")
    dout = _dout(x.shape, act, g, "cpu")
    for x3 in (True, False):
        for v, a in ((x, None), (dout, act)):
            ref, bound = emulate(v, w, b, a, idx, coef, x3)
            good = ref.float()
            assert ratio(good, ref, bound) <= 1.0
            if x3:
                dropped = emulate(v, w, b, a, idx, coef, x3, drop=(2, H // 64 - 1))[0].float()
                assert ratio(dropped, ref, bound) > 10.0
            assert drop_margin(v, w, b, a, idx, coef, x3, ref, bound) >= 10.0
            half, chunk, wrong = good.clone(), good.clone(), good.clone()
            half.view(-1, H)[128:3 * 81] = NAN
            chunk[:, :, 32:64] = NAN
            wrong[4, 40, 7] += 1e-3
            assert ratio(wrong, ref, bound) > 1.0
            for bad in (half, chunk):
                assert ratio(bad, ref, bound) == float("inf")


def test_shape_check_refuses_invalid_grids():
    """azg_grid_tc_supported through ctypes, no GPU needed: negative sides, a product that wraps a 32-bit int to 1
    (641 x 6,700,417 = 2^32 + 1), 0 and 257 nodes are refused; 1 and 256 nodes in either orientation, and 16x16, are
    taken at H = 64, 128 and 256 and at no other H."""
    from importlib import import_module
    lib = ctypes.CDLL(import_module("azgnn_b200.build").build())
    lib.azg_grid_tc_supported.restype = ctypes.c_int
    lib.azg_grid_tc_supported.argtypes = [ctypes.c_int] * 3
    ok = lib.azg_grid_tc_supported
    for gh, gw in ((-1, -1), (-2, -64), (-16, -16), (641, 6700417), (6700417, 641), (0, 0), (0, 5), (5, 0), (1, 257),
                   (257, 1), (-1, 1), (1, -256)):
        for H in (64, 128, 256):
            assert ok(gh, gw, H) == 0, (gh, gw, H)
    for gh, gw in ((1, 1), (1, 256), (256, 1), (16, 16), (2, 128)):
        for H in (64, 128, 256):
            assert ok(gh, gw, H) == 1, (gh, gw, H)
        for H in (0, 32, 96, 192, 512, -64):
            assert ok(gh, gw, H) == 0, (gh, gw, H)


# ------------------------------------------------------------------------------------ the kernels through the C ABI
GUARD = 256


def pack(w, transpose):
    lib = _lib.lib()
    H = w.shape[0]
    img = torch.empty(int(lib.azg_grid_packed_bytes(H)), dtype=torch.uint8, device="cuda")
    _lib.check(lib.azg_grid_pack_weights(ptr(w), H, int(transpose), ptr(img), stream()))
    return img


def run(x, img, b, act, gh, gw, prec):
    """forward (act None) or backward_input through the C ABI.  The output is a view into a buffer with a NaN guard of
    GUARD floats on each side, which must come back untouched."""
    B, n, H = x.shape
    N = B * n * H
    buf = torch.full((N + 2 * GUARD,), NAN, device="cuda")
    out = buf[GUARD:GUARD + N].view(B, n, H)
    lib = _lib.lib()
    if act is None:
        _lib.check(lib.azg_grid_layer_tc_forward(ptr(x), ptr(img), ptr(b), B, gh, gw, H, prec, ptr(out), stream()))
    else:
        _lib.check(lib.azg_grid_layer_tc_backward_input(ptr(x), ptr(act), ptr(img), B, gh, gw, H, prec, ptr(out), stream()))
    assert bool(torch.isnan(buf[:GUARD]).all()) and bool(torch.isnan(buf[GUARD + N:]).all()), "wrote outside [B, n, H]"
    return out


def _batch(n, mt, pair):
    """graphs per tile G, and a batch whose last tile is partly filled (when G > 1) and whose 151 tiles exceed the 148 CTAs
    and the 74 pairs, so each walks a second tile; 151 is odd, so the last pair's peer runs the all-zero tile"""
    G = 128 * mt // n
    return G, 150 * G + (G + 1) // 2


def _targets(n, G, mt, B):
    """graphs whose outputs are checked bit for bit: slot 0 and slot G - 1 of tile 0, the graph on the half boundary
    (rows 127 and 128) and the first one wholly in the second half of a 256-row tile, tile 1 (a pair's peer CTA), a tile
    past the first round of CTAs, and the last graph"""
    t = {0, G - 1, 127 // n, G + G // 2, SMS * G + 1, B - 1}
    if mt == 2 and -(-128 // n) < G:
        t.add(-(-128 // n))
    return sorted(s for s in t if s < B)


def _subprocess(request, env):
    """run this test case again in a child process with env set (the library reads the switches once per process)"""
    r = subprocess.run([sys.executable, "-m", "pytest", f"{os.path.abspath(__file__)}::{request.node.name}", "-q", "-s"],
                       env=dict(os.environ, **env), capture_output=True, text=True, timeout=900)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout and "skipped" not in r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("gh,gw,H,env", CASES, ids=[_case_id(c) for c in CASES])
def test_layer_matches_emulation(request, gh, gw, H, env):
    """Both precisions, forward and backward_input, one batch of _batch's size: every element within the bound of the
    module docstring against the float64 emulation, and the bound is at most a tenth of what leaving one droppable
    product out on any one k-block changes somewhere (drop_margin).  Nothing is written outside the output.  Bit for bit:
    graphs other than the _targets filled with NaN and inf (in x; in dout with the gate open) leave the targets' outputs
    unchanged and finite, each target run alone (B = 1) equals its row, and a second launch equals the first.  The
    backward's act holds 0, -0.0, negatives and NaN; its dout holds NaN where the gate is closed."""
    env = ENVS.get(env, {})
    if any(os.environ.get(k) != v for k, v in env.items()):
        return _subprocess(request, env)
    n = gh * gw
    gen = torch.Generator(device="cuda").manual_seed(n * 1009 + H)
    idx, coef = grid_neighbours(gh, gw, "cuda")
    w, b = _weights(H, gen, "cuda")
    imgs = {False: pack(w, False), True: pack(w, True)}
    report = []
    for x3, prec in ((True, _lib.PREC_BF16X3), (False, _lib.PREC_BF16)):
        _, _, _, mt, pair = instantiation(gh, gw, H, x3, False, env)
        G, B = _batch(n, mt, pair)
        targets = _targets(n, G, mt, B)
        others = torch.ones(B, dtype=torch.bool, device="cuda")
        others[targets] = False
        x = torch.randn(B, n, H, device="cuda", generator=gen)
        act = _act((B, n, H), gen, "cuda")
        dout = _dout((B, n, H), act, gen, "cuda")
        for bwd in (False, True):
            v, a = (dout, act) if bwd else (x, None)
            out = run(v, imgs[bwd], b, a, gh, gw, prec)
            ref, bound = emulate(v, w, b, a, idx, coef, x3)
            e = ratio(out, ref, bound)
            m = drop_margin(v[:SMS], w, b, a[:SMS] if bwd else None, idx, coef, x3, ref[:SMS], bound[:SMS])
            report.append(f"{'bf16x3' if x3 else 'bf16'} {'bwd' if bwd else 'fwd'} MT={mt}{' pair' if pair else ''}: "
                          f"|err| / bound {e:.3f}, drop margin {m:.1f}")
            assert e <= 1.0, report[-1]
            assert m >= 10.0, report[-1]
            assert torch.equal(run(v, imgs[bwd], b, a, gh, gw, prec), out), "two launches differ"
            vp = v.clone()
            poison = torch.where(torch.arange(B, device="cuda")[:, None, None] % 2 == 0, NAN, float("inf"))
            vp = torch.where(others[:, None, None], poison.expand_as(vp), vp)
            ap = torch.where(others[:, None, None], torch.ones((), device="cuda"), a) if bwd else None
            outp = run(vp, imgs[bwd], b, ap, gh, gw, prec)
            assert torch.equal(outp[targets], out[targets]), "another graph's NaN / inf reached a target"
            assert bool(torch.isfinite(out[targets]).all())
            for t in targets:
                s = slice(t, t + 1)
                alone = run(v[s].contiguous(), imgs[bwd], b, a[s].contiguous() if bwd else None, gh, gw, prec)
                assert torch.equal(alone, out[s]), ("graph run alone differs", t)
    print(f"grid tc {_case_id((gh, gw, H, ''))} {env or ''} B={B}: " + "; ".join(report))


@pytest.mark.gpu
def test_refusals():
    """Both entry points refuse, before any launch: precision fp32 or f16f8, H = 32, 96 or 512, negative sides, a
    product that wraps to 1, 0 and 257 nodes; the forward also refuses a NULL bias.  B = 0 returns OK without a launch."""
    lib = _lib.lib()
    t = torch.zeros(1 << 16, device="cuda")

    def call(bwd, B, gh, gw, H, prec, bias=t):
        if bwd:
            return lib.azg_grid_layer_tc_backward_input(ptr(t), ptr(t), ptr(t), B, gh, gw, H, prec, ptr(t), stream())
        return lib.azg_grid_layer_tc_forward(ptr(t), ptr(t), ptr(bias), B, gh, gw, H, prec, ptr(t), stream())

    X3 = _lib.PREC_BF16X3
    bad = [(1, 4, 4, 128, _lib.PREC_FP32), (1, 4, 4, 128, _lib.PREC_F16F8)]
    bad += [(1, 4, 4, H, X3) for H in (32, 96, 512)]
    bad += [(1, gh, gw, 128, X3) for gh, gw in ((-1, -1), (-2, -64), (-16, -16), (641, 6700417), (0, 4), (1, 257))]
    for bwd in (False, True):
        name = "azg_grid_layer_tc_" + ("backward_input" if bwd else "forward")
        cases = [(args, {}) for args in bad] + ([] if bwd else [((1, 4, 4, 128, X3), {"bias": None})])
        for args, kw in cases:
            torch.cuda.synchronize()
            l0 = lib.azg_launch_count()
            with pytest.raises(RuntimeError, match=name):
                _lib.check(call(bwd, *args, **kw))
            assert lib.azg_launch_count() == l0, (name, args, kw)
        l0 = lib.azg_launch_count()
        assert call(bwd, 0, 4, 4, 128, X3) == _lib.OK
        assert lib.azg_launch_count() == l0


@pytest.mark.gpu
@pytest.mark.parametrize("bwd", [False, True], ids=["forward", "backward"])
def test_past_2_32_elements(bwd):
    """bf16, H = 256, 16x16 graphs (MT = 2, EC = 16), B = 65,537: 2^32 + 65,536 elements per tensor (17.2 GB).  The first
    and last graphs and those on either side of element 2^31 (graphs 32,767 and 32,768) and 2^32 (65,535 and 65,536)
    against the float64 emulation, and equal to themselves run alone."""
    gh, gw, H, B = 16, 16, 256, 65537
    n, N = gh * gw, 65537 * 256 * 256
    need = (3 if bwd else 2) * (N + 2 * GUARD) * 4 + (4 << 30)
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"needs {need / 1e9:.0f} GB of free device memory, {free / 1e9:.0f} GB are free")
    targets = [0, 32767, 32768, 65535, 65536]
    gen = torch.Generator(device="cuda").manual_seed(65537 + bwd)
    idx, coef = grid_neighbours(gh, gw, "cuda")
    w, b = _weights(H, gen, "cuda")
    img = pack(w, bwd)
    v = torch.empty(B, n, H, device="cuda").normal_(generator=gen)
    a = None
    try:
        if bwd:
            a = torch.empty(B, n, H, device="cuda").normal_(generator=gen)
            for t in targets:
                a[t] = _act((n, H), gen, "cuda")
                v[t] = _dout((n, H), a[t], gen, "cuda")
        out = run(v, img, b, a, gh, gw, _lib.PREC_BF16)
        worst = 0.0
        for t in targets:
            s = slice(t, t + 1)
            vs, as_ = v[s].contiguous(), a[s].contiguous() if bwd else None
            ref, bound = emulate(vs, w, b, as_, idx, coef, False)
            worst = max(worst, ratio(out[s], ref, bound))
            assert torch.equal(run(vs, img, b, as_, gh, gw, _lib.PREC_BF16), out[s]), t
        print(f"grid tc bf16 {'bwd' if bwd else 'fwd'} 16x16 H=256 B={B}: |err| / bound {worst:.3f} at graphs {targets}")
        assert worst <= 1.0, worst
    finally:
        del v, a
        out = None
        torch.cuda.empty_cache()
