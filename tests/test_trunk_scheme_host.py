"""Numerics of the fused trunk's tensor-core conv1 (csrc/azg_gemm_tc.cu, c4_trunk2_tc_kernel), restated in torch on the CPU:
the 3x3 neighbourhood of a cell is an exact bf16 operand in {-1, 0, +1}, the fp32 weight is the sum of three bf16 terms,
products are exact and accumulation is fp32 -- so conv1 on the tensor core reproduces Connect4Net.py:45 to fp32 rounding."""
import numpy as np
import torch


def _split3(w):
    hi = w.bfloat16().float()
    mid = (w - hi).bfloat16().float()
    lo = ((w - hi) - mid).bfloat16().float()
    return hi, mid, lo


def test_three_bf16_terms_carry_the_fp32_weight():
    torch.manual_seed(0)
    w = torch.empty(32, 9).uniform_(-1 / 3, 1 / 3)  # conv1 default init range (fan_in = 9)
    w[0, :3] = torch.tensor([1e-8, -3.3e-5, 0.333333])
    hi, mid, lo = _split3(w)
    err = (hi.double() + mid.double() + lo.double() - w.double()).abs()
    assert float((err / w.double().abs().clamp_min(1e-30)).max()) <= 2.0 ** -23


def test_conv1_as_neighbourhood_gemm_matches_conv2d():
    torch.manual_seed(1)
    n, B = 7, 64
    rng = np.random.default_rng(3)
    boards = torch.from_numpy(rng.integers(-1, 2, size=(B, n, n)).astype(np.float32))
    conv = torch.nn.Conv2d(1, 32, 3, padding=1)
    with torch.no_grad():
        want = torch.relu(conv(boards.view(B, 1, n, n)))  # [B, 32, n, n]
    # operand rows: one per (board, cell); K index = kx*3 + ky, taps outside the board are 0 (the kernel reads them as
    # bits of the packed position with a per-row validity mask)
    padded = torch.nn.functional.pad(boards, (1, 1, 1, 1))
    rows = torch.stack([padded[:, kx:kx + n, ky:ky + n] for kx in range(3) for ky in range(3)], dim=-1).reshape(B * n * n, 9)
    assert set(np.unique(rows.numpy())) <= {-1.0, 0.0, 1.0} and torch.equal(rows.bfloat16().float(), rows)
    hi, mid, lo = _split3(conv.weight.detach().reshape(32, 9))
    a3 = torch.cat([rows, rows, rows], dim=1)                      # [A | A | A]
    w3 = torch.cat([hi, mid, lo], dim=1)                           # [w_hi | w_mid | w_lo]
    got = torch.relu((a3 @ w3.T) + conv.bias.detach())             # fp32 accumulation
    got = got.reshape(B, n, n, 32).permute(0, 3, 1, 2)
    assert float((got - want).abs().max()) <= 1e-6
