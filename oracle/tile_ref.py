"""Float64 references for the tensor-core tile kernels of the fused all-entity loss (kgeb_fused_fwd / _bwd,
kgeb_fused_flash_fwd / _dq, kgeb_score_all, kgeb_rank_count), for operands the tiles represent exactly.

On such operands every product of the tile GEMMs is exact in fp32 (bf16 x bf16: 16 significant bits, TF32 x TF32: 22), so
a kernel's scores differ from the float64 scores by fp32 accumulation alone.  The references below reproduce the
kernels' own intermediate roundings -- G rounded to bf16 before the second GEMM, P rounded to bf16 for the flash o_sum --
and nothing else, so that what remains of the difference is accumulation error, which `dot_bound` bounds per element.
"""
from __future__ import annotations

from typing import Sequence

import torch

U32 = 2.0 ** -24            # unit roundoff of fp32
# The tensor core adds the exact products of one MMA K-step (8 for TF32, 16 for bf16) before the fp32 accumulator rounds,
# and may truncate while aligning them: at most d / 8 + 1 roundings of at most 2 u each, i.e. <= (d / 4 + 2) u of the
# sum of |products| -- c = 1/4 in dot_bound (plus the constant, which d >= 8 covers twice over).
C_TILE = 0.25


def bf16_exact(x: torch.Tensor) -> torch.Tensor:
    """fp32 values that bf16 represents (round to nearest even): the bf16 mirror of such a table equals the table."""
    return x.float().bfloat16().float()


def tf32_exact(x: torch.Tensor) -> torch.Tensor:
    """fp32 values with the low 13 mantissa bits cleared: exact in TF32 whether the tensor core truncates or rounds."""
    return (x.float().contiguous().view(torch.int32) & -8192).view(torch.float32)


def g_bf16(g: torch.Tensor) -> torch.Tensor:
    """G (float64) as the backward kernels feed it to the second GEMM: rounded to fp32, then to bf16 (cvt.rn)."""
    return g.float().bfloat16().double()


def bf16_flip(g: torch.Tensor, eps) -> torch.Tensor:
    """Largest change of g_bf16(g') over g' within relative eps of g (eps a number or a tensor like g): one bf16 ulp
    (2^-8 of the element) where a perturbation of that size can move g across a rounding boundary, 0 elsewhere."""
    return (g_bf16(g * (1 + eps)) - g_bf16(g * (1 - eps))).abs()


def dot_bound(a: torch.Tensor, b: torch.Tensor, c: float = C_TILE) -> torch.Tensor:
    """Per-element bound on the fp32 accumulation error of a @ b.T with exact products: c * d * 2^-24 * (|a| @ |b|.T)."""
    d = a.shape[1]
    return c * d * U32 * (a.double().abs() @ b.double().abs().t())


def combine_rowstats(parts: Sequence[torch.Tensor], kl: bool) -> torch.Tensor:
    """The shard combination of fused.combine_rowstats (all-reduce of per-shard [B, 4] statistics) in float64: KL takes
    the maximum of column 0 and rescales each shard's column 1 to it (an empty shard, max = -inf, adds nothing); every
    other column, and every column of BCE, is a plain sum."""
    st = torch.stack([p.double() for p in parts])                    # [S, B, 4]
    if not kl:
        return st.sum(0)
    gmax = st[:, :, 0].max(0).values
    scale = torch.where(torch.isneginf(st[:, :, 0]), torch.zeros_like(st[:, :, 0]), torch.exp(st[:, :, 0] - gmax))
    return torch.stack((gmax, (st[:, :, 1] * scale).sum(0), st[:, :, 2].sum(0), st[:, :, 3].sum(0)), dim=1)


def label_matrix(lab_off: torch.Tensor, lab_col: torch.Tensor, b: int, e: int, e_lo: int = 0) -> torch.Tensor:
    """Dense float64 [b, e] count matrix of the label CSR, columns shifted by e_lo (entries outside [0, e) dropped)."""
    n = lab_off[1:] - lab_off[:-1]
    rows = torch.repeat_interleave(torch.arange(b, device=lab_off.device), n)
    cols = lab_col[: int(lab_off[-1])] - e_lo
    keep = (cols >= 0) & (cols < e)
    y = torch.zeros(b, e, dtype=torch.float64, device=lab_off.device)
    y.index_put_((rows[keep], cols[keep]), torch.ones(int(keep.sum()), dtype=torch.float64, device=y.device),
                 accumulate=True)
    return y


def kl_forward(x: torch.Tensor, y: torch.Tensor):
    """(lse, label sum, per-row KL loss) of float64 scores x and label counts y (rows with labels)."""
    lse = torch.logsumexp(x, 1)
    nnz = y.sum(1)
    lab = (x * y).sum(1)
    safe = nnz.clamp(min=1)
    rows = torch.where(nnz > 0, lse - lab / safe - torch.log(safe), torch.zeros_like(lse))
    return lse, lab, rows


def bce_forward(x: torch.Tensor, y: torch.Tensor, offset: float, ls: float, num_entities: int):
    """(sum softplus(x + off), sum (x + off), label sum of (x + off), per-row loss) in float64."""
    z = x + offset
    sp = torch.nn.functional.softplus(z).sum(1)
    xs = z.sum(1)
    lab = (z * y).sum(1)
    add = (1.0 / num_entities) if ls > 0 else 0.0
    return sp, xs, lab, sp - (1.0 - ls) * lab - add * xs


def dense_g(x: torch.Tensor, kl: bool, rs: torch.Tensor, lse32: torch.Tensor = None, offset: float = 0.0,
            ls_add: float = 0.0) -> torch.Tensor:
    """Dense part of G in float64 (KL: rs * exp(x - lse) with the kernel's fp32 lse; BCE: rs * (sigmoid(x + off) - ls_add)),
    before the kernels' bf16 rounding (g_bf16)."""
    if kl:
        return rs[:, None] * torch.exp(x - lse32.double()[:, None])
    return rs[:, None] * (torch.sigmoid(x + offset) - ls_add)


def label_weight(y: torch.Tensor, kl: bool, rs: torch.Tensor, ls: float = 0.0) -> torch.Tensor:
    """The sparse label part of G (exact fp32 kernels): -rs * t * y, t = 1/nnz (KL) or 1 - ls (BCE)."""
    if kl:
        t = torch.where(y.sum(1) > 0, 1.0 / y.sum(1).clamp(min=1), torch.zeros_like(rs))
    else:
        t = torch.full_like(rs, 1.0 - ls)
    return -(rs * t)[:, None] * y
