"""Forward kernels against float64 on both sides of the batch-size and shape thresholds that pick their code paths.

The small batches of test_nets_gpu.py reach one side of most thresholds; the benchmarks and self-play run on the other.
Each test names the threshold (code line and formula) and the sizes chosen on each side of it.  References are the
oracle.nets functions evaluated in float64 (they are dtype-agnostic), or the operation written in torch float64."""
import numpy as np
import pytest
import torch

from oracle import nets as onets
from oracle import rules as orules

from azgnn_b200 import _lib
from azgnn_b200.nets import B200Connect4GNNWrapper, B200FrozenLakeNet, B200TicTacToeGNNWrapper
from helpers import dotdict

pytestmark = pytest.mark.gpu

TC_PRECS = ("f16f8", "f16f8ks", "bf16x3", "bf16x3ks", "bf16")
BOTH = _lib.EVAL_STD | _lib.EVAL_GNN


def _wrapper(kind, n, **kw):
    game = (orules.Connect4Rules if kind == "c4" else orules.TicTacToeRules)(n)
    torch.manual_seed(0)
    args = dict(lr=1e-3, dropout=0.3, epochs=1, batch_size=64, gnn_layers=2, use_gnn=True, b200_precision="fp32")
    return (B200Connect4GNNWrapper if kind == "c4" else B200TicTacToeGNNWrapper)(game, dotdict(dict(args, **kw)))


def _sd64(m):
    return {k: v.detach().double().cpu() for k, v in m.state_dict().items()}


def _oracle(kind, w, boards):
    """float64 pi, v, pi_gnn, v_gnn of the reference modules for int boards [B, n, n]"""
    p, q, n = _sd64(w.nnet), _sd64(w.gnn), w.n
    bt = torch.from_numpy(np.asarray(boards).astype(np.float64))
    with torch.no_grad():
        if kind == "c4":
            pi, v = onets.c4_predict(p, bt, n)
            gpi, gv = onets.c4_predict_with_gnn(p, q, bt, n)
        else:
            pi, v = onets.ttt_predict(p, bt, n)
            gpi, gv = onets.ttt_predict_with_gnn(p, q, bt, n)
    return {"pi": pi.numpy(), "v": v.numpy(), "pi_gnn": gpi.numpy(), "v_gnn": gv.numpy()}


def _max_err(out, ref, keys=None, rows=None):
    errs = {}
    for k in keys or ref:
        got = out[k] if rows is None else out[k][rows]
        got = got.double().cpu().numpy() if torch.is_tensor(got) else np.asarray(got, dtype=np.float64)
        errs[k] = float(np.abs(got.reshape(ref[k].shape) - ref[k]).max())
    return errs


# ------------------------------------------------------------------------------------ TicTacToe im2col chunks
def _ttt_chunk(n, layer):
    """boards per im2col chunk of ttt_conv_tc (csrc/azg_gemm_tc.cu, `chunk = TTT_IMG_BYTES / (P * Kp * 2) / 256 * 256`):
    TTT_IMG_BYTES = 2^27, conv2 (pad 1): P = n^2, Kp = 320 (K = 288); conv3 (pad 0): P = (n-2)^2, Kp = 576"""
    P, Kp = (n * n, 320) if layer == 2 else ((n - 2) ** 2, 576)
    return max((2 ** 27 // (P * Kp * 2)) // 256 * 256, 256)


def _chunk_rows(B, chunk, rng, per_chunk=24):
    rows = set()
    for b0 in range(0, B, chunk):
        last = min(B, b0 + chunk) - 1
        rows.update((b0, last))
        rows.update(rng.integers(b0, last + 1, size=per_chunk).tolist())
    return rows


@pytest.mark.parametrize("n,B", [(8, 7000), (4, 30000), (3, 65536), (6, 1111), (7, 1111)])
def test_tictactoe_beyond_the_im2col_chunk(n, B):
    """ttt_conv_tc splits conv2 and conv3 into chunks of `chunk = floor(2^27 / (P*Kp*2) / 256) * 256` boards
    (azg_gemm_tc.cu, ttt_conv_tc): n = 3: 23,296 / 116,480; n = 4: 13,056 / 28,928; n = 8: 3,072 / 3,072 (conv2 / conv3).
    n = 8, B = 7,000 runs three chunks in each conv (ragged last chunk 856); n = 4, B = 30,000 three conv2 chunks and two
    conv3 chunks; n = 3, B = 65,536 is the bench_games leaf batch (three conv2 chunks, one conv3 chunk).  The second and
    later chunks bring in b0 > 0, the output offset out_nhwc + b0*P*N and the ragged last chunk.  The launch count of
    the call grows by two (im2col + GEMM) per extra chunk.  n = 6 (F = 2,048, BN = 256) and n = 7 (F = 3,200: the
    single-CTA BN = 64 GEMM with KB = 50) at the ragged B = 1,111 cover the other TicTacToe widths.
    Per chunk the first row, the last row and a random sample are compared with the float64 oracle (bf16x3: 1e-5,
    bf16: 5e-3), std and GNN predictions; those rows evaluated alone are bit-identical to the same rows of the big batch."""
    w = _wrapper("ttt", n)
    rng = np.random.default_rng(B + n)
    boards = rng.integers(-1, 2, size=(B, n, n)).astype(np.int8)
    states = w.states_from_boards(boards)
    c2, c3 = _ttt_chunk(n, 2), _ttt_chunk(n, 3)
    rows = np.array(sorted(_chunk_rows(B, c2, rng) | _chunk_rows(B, c3, rng)))
    ref = _oracle("ttt", w, boards[rows].astype(np.int64))
    trows = torch.from_numpy(rows).cuda()
    lib = _lib.lib()
    extra = (-(-B // c2) - 1) + (-(-B // c3) - 1)
    for prec, tol in ((_lib.PREC_BF16X3, 1e-5), (_lib.PREC_BF16, 5e-3)):
        w.forward_states(states[:1].contiguous(), BOTH, precision=prec)  # packs the weights
        torch.cuda.synchronize()
        l0 = lib.azg_launch_count()
        w.forward_states(states[:1].contiguous(), BOTH, precision=prec)
        l1 = lib.azg_launch_count()
        full = w.forward_states(states, BOTH, precision=prec)
        l2 = lib.azg_launch_count()
        assert (l2 - l1) - (l1 - l0) == 2 * extra, (l1 - l0, l2 - l1, extra)
        errs = _max_err(full, ref, rows=trows)
        print(f"ttt n={n} B={B} {_lib.PRECISION_NAMES[prec]}: chunks {-(-B // c2)}/{-(-B // c3)}, {len(rows)} rows, max |err| vs fp64 {errs}")
        assert max(errs.values()) <= tol, errs
        alone = w.forward_states(states[trows].contiguous(), BOTH, precision=prec)
        for k in full:
            assert torch.equal(alone[k], full[k][trows]), k
    if (n, B) == (4, 30000):  # the fp32 CUDA-core path at the same size
        o = w.forward_states(states, BOTH, precision=_lib.PREC_FP32)
        errs = _max_err(o, ref, rows=trows)
        print(f"ttt n={n} B={B} fp32: max |err| vs fp64 {errs}")
        assert max(errs.values()) <= 1e-5, errs


# ------------------------------------------------------------------------------------ Connect4 trunk tiles
def _boards_per_tile(n):
    """c4_trunk2_tc_kernel: G = (127 - (n^2 + n - 2)) / (n+1)^2 + 1 boards per 128-row tile (azg_gemm_tc.cu)"""
    return (127 - (n * n + n - 2)) // ((n + 1) ** 2) + 1


def _trunk_batches(n):
    G = _boards_per_tile(n)
    return sorted({1, 2, G + 1} | {37 * G + r for r in range(1, G)})


@pytest.mark.parametrize("n", [4, 5, 6])
def test_connect4_ragged_trunk_tiles(n):
    """c4_trunk2_tc_kernel packs G = (127 - (n^2 + n - 2)) / (n+1)^2 + 1 boards into a 128-row tile (azg_gemm_tc.cu,
    `const int G = ...`): G = 5, 3, 2 at n = 4, 5, 6.  Batches B = 37*G + r for every r = 1 .. G-1 leave a partially
    filled last tile, plus B = 1, 2 and G+1 (n = 4: 1, 2, 6, 186..189; n = 5: 1, 2, 4, 112, 113; n = 6: 1, 2, 3, 75).
    Every tensor-core precision, with and without EVAL_FOLD, against the float64 oracle at the contracts of
    test_nets_gpu.py (f16f8 / f16f8ks / bf16x3 / bf16x3ks: 1e-5, folded v_gnn 2e-5; bf16: 5e-3); a std-only call equals
    the std half of the combined call."""
    w = _wrapper("c4", n)
    worst = {}
    for B in _trunk_batches(n):
        boards = np.random.default_rng(100 * n + B).integers(-1, 2, size=(B, n, n)).astype(np.int64)
        ref = _oracle("c4", w, boards)
        states = w.states_from_boards(boards)
        for name in TC_PRECS:
            prec = _lib.PRECISIONS[name]
            only_std = w.forward_states(states, _lib.EVAL_STD, precision=prec)
            for fold in (0, _lib.EVAL_FOLD):
                o = w.forward_states(states, BOTH | fold, precision=prec)
                errs = _max_err(o, ref)
                key = (name, bool(fold))
                worst[key] = max(worst.get(key, 0.0), max(errs.values()))
                if name == "bf16":
                    assert max(errs.values()) <= 5e-3, (B, key, errs)
                else:
                    assert max(errs["pi"], errs["v"], errs["pi_gnn"]) <= 1e-5, (B, key, errs)
                    assert errs["v_gnn"] <= (2e-5 if fold else 1e-5), (B, key, errs)
                assert torch.equal(only_std["pi"], o["pi"]) and torch.equal(only_std["v"], o["v"]), (B, key)
    print(f"c4 n={n} G={_boards_per_tile(n)} B={_trunk_batches(n)}: max |err| vs fp64 per (precision, fold) {worst}")


# ------------------------------------------------------------------------------------ device row counts
@pytest.mark.parametrize("n", [4, 7])
@pytest.mark.parametrize("prec", ["f16f8", "f16f8ks", "bf16x3ks"])
@pytest.mark.parametrize("fold", [False, True])
def test_device_row_counts(n, prec, fold):
    """azg_c4_forward_dyn reads the live row count on the device: the trunk clamps B (`if (t.dyn_rows && *t.dyn_rows <
    t.B) t.B = *t.dyn_rows`), the GEMMs clamp M (`rows = *g.dyn_rows`) and the head finalisers skip `row >= *dyn_rows`
    (azg_gemm_tc.cu).  Counts 0, 1, G (boards per trunk tile: 5 at n = 4, 2 at n = 7), 127/128/129 (an m-tile), 255/256/257
    (a CTA pair's two m-tiles) and B = 700.  Live rows equal a plain call on those rows bit for bit; rows past the count
    keep their sentinel; count = 0 returns AZG_OK and writes nothing.  At count = B the outputs hold the float64 oracle's
    contract (1e-5, folded v_gnn 2e-5)."""
    B = 700
    w = _wrapper("c4", n)
    boards = np.random.default_rng(21 + n).integers(-1, 2, size=(B, n, n)).astype(np.int64)
    states = w.states_from_boards(boards)
    p = _lib.PRECISIONS[prec]
    mask = BOTH | (_lib.EVAL_FOLD if fold else 0)
    for live in sorted({0, 1, _boards_per_tile(n), 127, 128, 129, 255, 256, 257, B}):
        count = torch.tensor([live], dtype=torch.int32, device="cuda")
        out = {k: torch.full_like(v, 7.0) for k, v in w._outputs(B, mask).items()}
        w.forward_states(states, mask, precision=p, count=count, out=out)
        torch.cuda.synchronize()
        if live:
            plain = w.forward_states(states[:live].contiguous(), mask, precision=p)
            for k in plain:
                assert torch.equal(out[k][:live], plain[k]), (live, k)
        for k in out:
            assert bool((out[k][live:] == 7.0).all()), (live, k)  # untouched past the count
    ref = _oracle("c4", w, boards)
    errs = _max_err(out, ref)
    print(f"dyn rows n={n} {prec} fold={fold}: count = B max |err| vs fp64 {errs}")
    assert max(errs["pi"], errs["v"], errs["pi_gnn"]) <= 1e-5 and errs["v_gnn"] <= (2e-5 if fold else 1e-5), errs


# ------------------------------------------------------------------------------------ azg_tc_linear
def _tc_linear(A, W, b, prec, relu):
    """C = act(A W^T + b) through the C ABI; C is a view of a buffer one row longer, whose last row must stay NaN"""
    M, F = A.shape
    Mp = (M + 255) // 256 * 256
    nbytes = 2 * (Mp + F) * F * 2 + 4096
    scratch = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
    Cbuf = torch.full((M + 1, F), float("nan"), device="cuda")
    _lib.check(_lib.lib().azg_tc_linear(_lib.ptr(A), _lib.ptr(W), _lib.ptr(b), _lib.ptr(Cbuf), M, F, prec, relu, _lib.ptr(scratch),
                                        scratch.numel(), _lib.stream()))
    assert bool(torch.isnan(Cbuf[M]).all()), "azg_tc_linear wrote past row M"
    return Cbuf[:M]


def _bn(F, prec):
    """tile width: pick_bn (224 | 256 | 160) for the bf16 splits, pick_bn_f8 (224 | 160 | 128) for f16f8 (azg_gemm_tc.cu)"""
    order = (224, 160, 128) if prec.startswith("f16f8") else (224, 256, 160)
    return next(bn for bn in order if F % bn == 0)


def _linear_operands(M, F, seed, scale=0.5):
    g = torch.Generator().manual_seed(seed)
    A = torch.randn(M, F, generator=g) * scale
    W = (torch.rand(F, F, generator=g) * 2 - 1) / F ** 0.5
    b = torch.randn(F, generator=g) * 0.1
    return A, W, b


@pytest.mark.parametrize("F", [1024, 1600, 2304, 3136, 4096])
@pytest.mark.parametrize("M", [1, 127, 128, 129, 255, 256, 257, 4097])
def test_tc_linear_tile_width_table(F, M):
    """Every tile width of the tensor-core GEMM: F = 1,024 / 1,600 / 2,304 / 3,136 / 4,096 are the Connect4 widths 64 n^2 at
    n = 4..8, with BN = 256 / 160 / 256 / 224 / 256 for the bf16 splits (pick_bn) and 128 / 160 / 128 / 224 / 128 for f16f8
    (pick_bn_f8), KB = F / 64 = 16 .. 64.  M = 1, 127/128/129 (one m-tile of BM = 128), 255/256/257 (the m-tile pair of
    the 2-CTA kernel, Mp = ceil(M / 256) * 256) and 4,097.  All five tensor-core precisions against float64 with the
    tolerances of test_nets_gpu.py::test_tc_linear: bf16x3, f16f8 and their K-split forms 1e-4 against A W^T + b; bf16
    5e-5 against the product of bf16-rounded operands.  Nothing is written past row M."""
    A, W, b = _linear_operands(M, F, M * 7 + F)
    Ad, Wd, bd = A.cuda().double(), W.cuda().double(), b.cuda().double()
    relu = M % 2
    ref = Ad @ Wd.t() + bd
    refb = A.cuda().bfloat16().double() @ W.cuda().bfloat16().double().t() + bd
    if relu:
        ref, refb = ref.clamp(min=0), refb.clamp(min=0)
    errs = {}
    for name in TC_PRECS:
        got = _tc_linear(A.cuda(), W.cuda(), b.cuda(), _lib.PRECISIONS[name], relu).double()
        errs[name] = (got - (refb if name == "bf16" else ref)).abs().max().item()
    print(f"tc_linear M={M} F={F} relu={relu} BN bf16/f16f8 = {_bn(F, 'bf16x3')}/{_bn(F, 'f16f8')}: max |err| {errs}")
    assert errs["bf16"] <= 5e-5, errs
    assert max(v for k, v in errs.items() if k != "bf16") <= 1e-4, errs


@pytest.mark.parametrize("F", [1024, 3136])
def test_bf16x3_matches_its_exact_emulation(F):
    """AZG_PREC_BF16X3 pinned term by term: Xh Wh^T + Xh Wl^T + Xl Wh^T + b with Xh = bf16(X), Xl = bf16(X - Xh) (same for
    W), operands rounded in torch and accumulated in float64.  The kernel (tcgen05 kind::f16, fp32 accumulation in TMEM)
    must agree to fp32-accumulation noise, bounded by c * sum|terms| with c = 2^-18 (the accumulator rounds, by
    truncation, once per K = 16 MMA step: 3 K / 16 steps whose partial sums stay near sum|terms| / sqrt(K)).  The bound is also below a tenth of the smallest contribution of any
    one of the two correction products on any one k-block, so a kernel that drops Xl Wh^T (or Xh Wl^T) from a single
    64-wide k-block fails.  F = 1,024 (BN = 256, KB = 16) and 3,136 (BN = 224, KB = 49), M = 300 (a ragged m-tile pair)."""
    M = 300
    A, W, b = _linear_operands(M, F, 29 + F)
    got = _tc_linear(A.cuda(), W.cuda(), b.cuda(), _lib.PREC_BF16X3, 0).double()
    Ad, Wd, bd = A.cuda().double(), W.cuda().double(), b.cuda().double()
    Ah, Wh = A.bfloat16().cuda().double(), W.bfloat16().cuda().double()
    Al, Wl = (A - A.bfloat16().float()).bfloat16().cuda().double(), (W - W.bfloat16().float()).bfloat16().cuda().double()
    model = Ah @ Wh.t() + Ah @ Wl.t() + Al @ Wh.t() + bd
    terms = Ah.abs() @ Wh.abs().t() + Ah.abs() @ Wl.abs().t() + Al.abs() @ Wh.abs().t() + bd.abs()
    e_model = (got - model).abs().max().item()
    e_rel = ((got - model).abs() / terms).max().item()
    e_exact = (got - (Ad @ Wd.t() + bd)).abs().max().item()
    # the smallest, over k-blocks, of the largest change that dropping one product on that k-block would make
    kb = [slice(k, k + 64) for k in range(0, F, 64)]
    drop = min(min((Al[:, s] @ Wh[:, s].t()).abs().max().item(), (Ah[:, s] @ Wl[:, s].t()).abs().max().item()) for s in kb)
    print(f"bf16x3 F={F}: |got - emulation| {e_model:.2e} (max {e_rel:.2e} of sum|terms|), |got - fp64| {e_exact:.2e}, "
          f"smallest one-k-block correction {drop:.2e}")
    assert e_rel <= 2.0 ** -18
    assert e_model < 0.1 * drop
    assert e_exact <= 1e-4


def _e4m3(t):
    return t.clamp(-448, 448).to(torch.float8_e4m3fn).double()  # clamp = the kernel's satfinite conversion


def _f16f8_model(A, W, b):
    """fp16(x) fp16(w) + [e4m3(2^3 x) | e4m3(2^14 x_lo)] . [e4m3(2^(s+11) w_lo) | e4m3(2^s w)] * 2^-(s+14) + b, float64"""
    Ad, Wd = A.double(), W.double()
    Ah, Wh = A.half().double(), W.half().double()
    m = float(W.abs().max())
    s = int(np.floor(np.log2(448.0 / m)))
    while m * 2.0 ** s > 448.0:
        s -= 1
    while m * 2.0 ** (s + 1) <= 448.0:
        s += 1
    corr = (_e4m3(Ad * 8.0) @ _e4m3((Wd - Wh) * 2.0 ** (s + 11)).t() + _e4m3((Ad - Ah) * 2.0 ** 14) @ _e4m3(Wd * 2.0 ** s).t()) * 2.0 ** -(s + 14)
    return Ah @ Wh.t() + corr + b.double()


@pytest.mark.parametrize("mag", [0.01, 1.0, 50.0, 60.0, 500.0, 30000.0, "mixed"])
def test_f16f8_emulation_across_activation_range(mag):
    """AZG_PREC_F16F8 scales activations by the fixed 2^3 (F8_A_SCALE, azg_tc.cuh): 2^3 x reaches the e4m3 maximum 448 at
    |x| = 56 and 2^14 x_lo (|x_lo| up to half an fp16 ulp) can pass it from |x| = 64; the conversion saturates
    (satfinite) and the element loses (part of) its FP8 correction, never its fp16 part.  Activations of magnitude 0.01, 1, 50 (below 56), 60, 500, 30,000 (above) and rows mixing all of
    them (each element within [0.9, 1] of its magnitude), against the term-by-term float64 model of
    test_nets_gpu.py::test_f16f8_matches_its_exact_emulation whose `_e4m3` clamp is that saturation: the kernel must match
    the model to fp32-accumulation noise, c * sum|terms| with c = 2^-18.  Up to |x| = 50 it also holds 2^-17 * sum|terms|
    against exact float64.  Measured (NVIDIA B200, 1,000 W power limit), the error against exact float64 A W^T + b relative to
    sum|A||W|: 1.8e-6 at |x| ~ 0.01, 1 and 50, 1.7e-6 at 60, 3.2e-5 at 500, 4.1e-5 at 30,000 and 9.5e-5 with the magnitudes
    mixed in a row (DESIGN.md section 4).  fp16 overflows above 65,504: outside the supported range."""
    M, F = 256, 1024
    g = torch.Generator().manual_seed(5)
    levels = torch.tensor([0.01, 1.0, 50.0, 60.0, 500.0, 30000.0])
    if mag == "mixed":
        scale = levels[torch.randint(0, len(levels), (M, F), generator=g)]
    else:
        scale = torch.full((M, F), float(mag))
    sign = torch.randint(0, 2, (M, F), generator=g).float() * 2 - 1
    A = sign * scale * (0.9 + 0.1 * torch.rand(M, F, generator=g))
    W = (torch.rand(F, F, generator=g) * 2 - 1) / F ** 0.5
    b = torch.randn(F, generator=g) * 0.1
    got = _tc_linear(A.cuda(), W.cuda(), b.cuda(), _lib.PREC_F16F8, 0).double().cpu()
    model = _f16f8_model(A, W, b)
    terms = A.double().abs() @ W.double().abs().t() + b.double().abs()
    e_rel = ((got - model).abs() / terms).max().item()
    e_exact = ((got - (A.double() @ W.double().t() + b.double())).abs() / terms).max().item()
    print(f"f16f8 |x| ~ {mag}: |got - emulation| <= {e_rel:.2e} sum|terms|, |got - fp64| <= {e_exact:.2e} sum|terms|")
    assert torch.isfinite(got).all()
    assert e_rel <= 2.0 ** -18
    if mag != "mixed" and mag <= 50:  # below the saturation point nothing is lost
        assert e_exact <= 2.0 ** -17


# ------------------------------------------------------------------------------------ FrozenLake
@pytest.mark.parametrize("n", [4, 8])
@pytest.mark.parametrize("E", [64, 96])
@pytest.mark.parametrize("layers", [2, 3])
def test_frozenlake_embedding_widths(n, E, layers):
    """B200FrozenLakeNet defaults to embedding_dim = 64 (nets.py); the other FrozenLake tests use 128.  E = 64 and 96 (not a
    power of two), L = 2 and 3, n = 4 and 8: every cell's pi and v against oracle.nets.fl_forward in float64, 1e-5."""
    torch.manual_seed(0)
    w = B200FrozenLakeNet(orules.FrozenLakeRules(n), dotdict(dict(lr=1e-3, embedding_dim=E, gnn_layers=layers)))
    cells = torch.zeros(n * n, 2, dtype=torch.int64, device="cuda")
    cells[:, 0] = torch.arange(n * n, device="cuda")
    out = w._forward_cells(cells)
    p = _sd64(w.nnet)
    e_pi = e_v = 0.0
    for cell in range(n * n):
        nodes = onets.fl_node_cells(cell, n)
        nb = torch.zeros(len(nodes), n * n, dtype=torch.float64)
        nb[torch.arange(len(nodes)), torch.tensor(nodes)] = 1.0
        with torch.no_grad():
            pi, v = onets.fl_forward(p, nb.reshape(len(nodes), n, n), layers)
        e_pi = max(e_pi, float((out["pi"][cell].double().cpu() - pi).abs().max()))
        e_v = max(e_v, abs(float(out["v"][cell]) - float(v[0])))
    print(f"frozenlake n={n} E={E} L={layers}: max |dpi| {e_pi:.2e}, max |dv| {e_v:.2e}")
    assert e_pi <= 1e-5 and e_v <= 1e-5
