"""The float64 reference helpers of tests/test_gpu_tensor_tiles_exact.py (oracle/tile_ref.py) on the CPU: operand and G
rounding against torch's own conversions, the shard combination against a one-shot logsumexp, the per-element bound on
hand-made cases."""
import math

import pytest
import torch

from oracle import tile_ref as tr


def test_bf16_operands_are_fixed_points_of_the_bf16_mirror():
    g = torch.Generator().manual_seed(0)
    x = torch.randn(4096, generator=g) * torch.logspace(-20, 20, 4096)
    b = tr.bf16_exact(x)
    assert b.dtype == torch.float32
    assert torch.equal(b, x.bfloat16().float())                   # round to nearest even, as kgeb_to_bf16
    assert torch.equal(tr.bf16_exact(b), b)
    assert torch.equal(b.bfloat16().float(), b)
    assert bool(((b.view(torch.int32) & 0xFFFF) == 0).all())       # 8 significant bits: the low half is clear
    # ties to even: 1 + 2^-8 lies halfway between 1 and 1 + 2^-7
    assert float(tr.bf16_exact(torch.tensor([1.0 + 2.0 ** -8]))) == 1.0
    assert float(tr.bf16_exact(torch.tensor([1.0 + 3 * 2.0 ** -8]))) == 1.0 + 2.0 ** -6


def test_tf32_operands_have_ten_mantissa_bits():
    g = torch.Generator().manual_seed(1)
    x = torch.randn(4096, generator=g) * 3
    t = tr.tf32_exact(x)
    assert bool(((t.view(torch.int32) & 0x1FFF) == 0).all())
    # truncation toward zero of the magnitude: |t| <= |x| < |t| + 2^-10 |t|, same sign, idempotent
    assert bool((t.abs() <= x.abs()).all()) and bool((x.abs() - t.abs() < t.abs() * 2.0 ** -10).all())
    assert bool((torch.sign(t) == torch.sign(x)).all())
    assert torch.equal(tr.tf32_exact(t), t)
    assert float(tr.tf32_exact(torch.tensor([1.0 + 2.0 ** -10]))) == 1.0 + 2.0 ** -10
    assert float(tr.tf32_exact(torch.tensor([1.0 + 2.0 ** -11]))) == 1.0
    # products of two such values are exact in fp32 (22 significant bits)
    a, b = t[:2048], t[2048:]
    assert torch.equal((a.double() * b.double()).float().double(), a.double() * b.double())


def test_g_is_rounded_through_fp32_to_bf16():
    g = torch.Generator().manual_seed(2)
    x = torch.rand(10000, dtype=torch.float64, generator=g) * 1e-3
    r = tr.g_bf16(x)
    assert r.dtype == torch.float64
    assert torch.equal(r, x.float().bfloat16().double())
    assert bool(((r - x).abs() <= x.abs() * 2.0 ** -8).all())       # half an ulp of 8 significant bits
    # double rounding: a value just above a bf16 tie in float64 but on the tie in fp32 goes to even
    tie = 1.0 + 2.0 ** -8 + 2.0 ** -40
    assert float(tr.g_bf16(torch.tensor([tie], dtype=torch.float64))) == 1.0


def test_shard_combination_equals_one_logsumexp():
    g = torch.Generator().manual_seed(3)
    x = torch.randn(50, 1000, dtype=torch.float64, generator=g) * 4
    x[7] -= 300.0                                                  # a row far below 0
    bounds = [(0, 1), (1, 333), (333, 333), (333, 1000)]           # a one-entity and an empty shard
    parts = []
    for lo, hi in bounds:
        s = x[:, lo:hi]
        if hi > lo:
            m = s.max(1).values
            parts.append(torch.stack((m, torch.exp(s - m[:, None]).sum(1), s.sum(1), s[:, :1].sum(1)), 1))
        else:
            parts.append(torch.stack((torch.full((50,), -math.inf, dtype=torch.float64), torch.zeros(50, dtype=torch.float64),
                                      torch.zeros(50, dtype=torch.float64), torch.zeros(50, dtype=torch.float64)), 1))
    st = tr.combine_rowstats(parts, kl=True)
    lse = st[:, 0] + torch.log(st[:, 1])
    assert torch.allclose(lse, torch.logsumexp(x, 1), rtol=1e-14, atol=1e-12)
    assert torch.allclose(st[:, 2], x.sum(1), rtol=1e-12, atol=1e-10)
    assert torch.equal(st[:, 0], x.max(1).values)
    # BCE: plain sums of every column
    assert torch.allclose(tr.combine_rowstats(parts, kl=False), sum(p for p in parts if bool(torch.isfinite(p).all())) +
                          torch.tensor([-math.inf, 0, 0, 0], dtype=torch.float64), equal_nan=True)


def test_dot_bound_on_hand_made_cases():
    a = torch.tensor([[1.0, -2.0, 0.5, 0.0]])
    b = torch.tensor([[3.0, 1.0, -4.0, 7.0], [0.0, 0.0, 0.0, 0.0]])
    bd = tr.dot_bound(a, b, c=1.0)
    assert bd.shape == (1, 2) and bd.dtype == torch.float64
    assert float(bd[0, 0]) == 4 * 2.0 ** -24 * (3 + 2 + 2 + 0)
    assert float(bd[0, 1]) == 0.0                                  # an all-zero row is exact
    assert float(tr.dot_bound(a, b)[0, 0]) == tr.C_TILE * float(bd[0, 0])
    # a real fp32 sequential sum stays inside the c = 1 bound (at most d - 1 roundings of <= u |partial sum|)
    g = torch.Generator().manual_seed(4)
    q, w = tr.bf16_exact(torch.randn(64, 256, generator=g)), tr.bf16_exact(torch.randn(32, 256, generator=g))
    acc = torch.zeros(64, 32)
    for k in range(256):
        acc = acc + q[:, k:k + 1] * w[:, k][None, :]               # products exact in fp32, one rounding per add
    err = (acc.double() - q.double() @ w.double().t()).abs()
    assert bool((err <= tr.dot_bound(q, w, c=1.0)).all())


@pytest.mark.parametrize("kl", [True, False])
def test_label_matrix_and_weights(kl):
    lab_off = torch.tensor([0, 2, 2, 5])
    lab_col = torch.tensor([1, 4, 0, 3, 4, 9])                     # a padding entry past lab_off[-1]
    y = tr.label_matrix(lab_off, lab_col, 3, 5)
    assert torch.equal(y, torch.tensor([[0, 1, 0, 0, 1], [0, 0, 0, 0, 0], [1, 0, 0, 1, 1]], dtype=torch.float64))
    ys = tr.label_matrix(lab_off, lab_col, 3, 2, e_lo=3)           # shard [3, 5)
    assert torch.equal(ys, y[:, 3:5])
    rs = torch.tensor([0.5, 1.0, 2.0], dtype=torch.float64)
    lw = tr.label_weight(y, kl, rs, 0.1)
    t = torch.tensor([0.5, 0.0, 1.0 / 3]) if kl else torch.full((3,), 0.9)
    assert torch.allclose(lw, -(rs * t.double())[:, None] * y)


def test_bf16_flip_marks_only_elements_near_a_rounding_boundary():
    g = torch.tensor([1.0, 1.0 + 2.0 ** -8, 1.0 + 2.0 ** -8 + 2.0 ** -20, 0.75, -(1.0 + 2.0 ** -8)], dtype=torch.float64)
    f = tr.bf16_flip(g, 1e-6)
    # 1 and 0.75 are far from a boundary; 1 + 2^-8 is a tie (either side rounds differently): one ulp of 2^-7
    assert f.tolist() == [0.0, 2.0 ** -7, 2.0 ** -7, 0.0, 2.0 ** -7]
    assert float(tr.bf16_flip(torch.tensor([1.0 + 2.0 ** -8 + 2.0 ** -20], dtype=torch.float64), 1e-7)) == 0.0
