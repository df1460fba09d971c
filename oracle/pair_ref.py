"""Float64 references for the negative-sampling kernels and the row scorers of rows.cu / ns_segment.cu / update.cu:
query transforms (kgeb_query_build / _bwd), pair scores (kgeb_pairs_score, kgeb_ns_fused), the per-row KL / BCE loss of
[B, 1 + N] score rows with the positive in column 0 (kgeb_ns_loss), the pair backward (kgeb_pairs_bwd, kgeb_ns_bwd_q,
kgeb_ns_cand_grad) and the row sums of the sorted scatter (kgeb_scatter_add_rows).

Everything is computed in float64 on the device of the inputs.  The gradient helpers follow the kernels' zero conventions
explicitly (sign(0) = 0; a zero L2 distance or a zero complex modulus gives a zero gradient) instead of differentiating a
norm.  The bound helpers give first-order per-element bounds on the fp32 error of a kernel: a chain of k roundings moves a
sum by at most k u sum|terms| (u = 2^-24), so every bound is (k + c) u sum|terms| with k the longest chain of roundings in
the kernel's summation order and c the roundings of one term before it enters the sum, plus the documented accuracy of the
MUFU / libdevice functions the kernel calls.
"""
from __future__ import annotations

import math

import torch

U = 2.0 ** -24                 # unit roundoff of fp32
ULP = 2.0 ** -23               # one ulp of an fp32 value v is at most ULP * |v|
LOGF_ABS = 2.0 ** -21.41       # __logf: absolute error on [0.5, 2] (CUDA Programming Guide, intrinsic functions)
TINY = 1e-37                   # results that flush to zero in fp32 (exp overflow in sigmoidf, exp underflow)
FLUSH = 2.0 ** -126            # red / atom .add.f32 flush subnormal inputs and results to zero (PTX ISA): per add
DOT, NEG_L1, NEG_L2, ROT_L1, ROT_L2 = 0, 1, 2, 3, 4
KL, BCE = 0, 1
SP_, _PO = 0, 1
# sincosf without fast math: 2 ulp (Programming Guide) = at most 4 u of |sin| / |cos|
SINCOS_REL = 4 * U
WARP_LEVELS = 5                # butterfly levels of warp_sum
PAIR_BWD_WARPS = 8             # warps of the block-per-row backward kernels, combined in fixed order


def cdiv(a: int, b: int) -> int:
    return -(-a // b)


# ---------------------------------------------------------------------------------------------------------------------
# query transforms (SURVEY.md App. D, as kgeb_query_build documents it)
# ---------------------------------------------------------------------------------------------------------------------
def _combine_mask(combine, n, device):
    """True where a row takes the sp_ form: combine is SP_ / _PO or a per-row int tensor of them (row_combine)."""
    if isinstance(combine, torch.Tensor):
        return (combine.to(device) == SP_).view(n, 1)
    return torch.full((n, 1), combine == SP_, dtype=torch.bool, device=device)


def query(model: str, combine, a: torch.Tensor, p: torch.Tensor, absolute: bool = False) -> torch.Tensor:
    """Q [n, d] of the sp_ form (a = s) or the _po form (a = o) of `model`, in float64.  absolute=True evaluates the same
    terms on |a|, |p| (|cos|, |sin| for RotatE) with every sign +: the sum of |terms| of each element, for the bounds."""
    a, p = a.double(), p.double()
    if absolute:
        a, p = a.abs(), p.abs()
    sg = 1.0 if absolute else -1.0            # the sign of a subtracted term
    n, d = a.shape
    h = d // 2
    sp = _combine_mask(combine, n, a.device)
    z = torch.zeros(n, h, dtype=torch.float64, device=a.device)
    if model == "distmult":
        return a * p
    if model == "transe":
        return torch.where(sp, a + p, a + sg * p)
    if model == "rescal":
        m = p.view(n, d, d)
        return torch.where(sp, torch.einsum("ni,nij->nj", a, m), torch.einsum("nij,nj->ni", m, a))
    ar, ai = a[:, :h], a[:, h:]
    if model == "cp":
        return torch.where(sp, torch.cat((z, ar * p), 1), torch.cat((ai * p, z), 1))
    if model == "simple":
        pf, pb = p[:, :h], p[:, h:]
        return torch.where(sp, 0.5 * torch.cat((ai * pb, ar * pf), 1), 0.5 * torch.cat((ai * pf, ar * pb), 1))
    if model == "complex":
        pr, pi = p[:, :h], p[:, h:]
    elif model == "rotate":
        pr, pi = torch.cos(p), torch.sin(p)
        if absolute:
            pr, pi = pr.abs(), pi.abs()
    else:
        raise ValueError(model)
    q_sp = torch.cat((ar * pr + sg * ai * pi, ai * pr + ar * pi), 1)
    q_po = torch.cat((ar * pr + ai * pi, ai * pr + sg * ar * pi), 1)
    return torch.where(sp, q_sp, q_po)


def query_grads(model: str, combine, a: torch.Tensor, p: torch.Tensor, g: torch.Tensor, absolute: bool = False):
    """(da, dp) of <query(model, combine, a, p), g>: the transforms are (bi)linear in a and in (p or cos p, sin p), so
    autograd through them is exact.  absolute=True: the same on |a|, |p|, |g| with every sign + (the sums of |terms| of
    each element), with RotatE's dp written out because d|cos p| / dp is not |d cos p / dp|."""
    a64 = a.double().clone().requires_grad_(True)
    p64 = p.double().clone().requires_grad_(True)
    g64 = g.double()
    if absolute:
        g64 = g64.abs()
    if absolute and model == "rotate":
        aa, h = a.double().abs(), a.shape[1] // 2
        c, s = torch.cos(p.double()).abs(), torch.sin(p.double()).abs()
        ar, ai, gr, gi = aa[:, :h], aa[:, h:], g64[:, :h], g64[:, h:]
        da = torch.cat((gr * c + gi * s, gr * s + gi * c), 1)
        dp = gr * (ar * s + ai * c) + gi * (ar * c + ai * s)
        return da, dp
    q = query(model, combine, a64.abs() if absolute else a64, p64.abs() if absolute else p64, absolute=absolute)
    da, dp = torch.autograd.grad((q * g64).sum(), (a64, p64), allow_unused=True)
    da = torch.zeros_like(a64) if da is None else da
    dp = torch.zeros_like(p64) if dp is None else dp
    if absolute:
        da, dp = da.abs(), dp.abs()
    return da.detach(), dp.detach()


# roundings per element of the query transforms and their backward, c in c u sum|terms| (query(..., absolute=True)):
# one product (DistMult, CP, TransE, SimplE with its exact 0.5), two (ComplEx: a product and an FMA), RotatE the same
# two plus sincosf's 4u; its dp a sum of two two-term products (4 roundings) plus 4u.  RESCAL: sp_ sums over i in one
# lane (d FMAs), _po a warp sum (ceil(d/32) per lane + 5 levels + 1); its backward the other way round.
C_QUERY = {"distmult": 1, "cp": 1, "transe": 1, "simple": 1, "complex": 2, "rotate": 6}
C_QUERY_BWD = {"distmult": (1, 1), "cp": (1, 1), "transe": (1, 1), "simple": (1, 1), "complex": (2, 2), "rotate": (6, 8)}


def _rescal_c(combine, n, d, device, lane_sum_first: bool):
    sp = _combine_mask(combine, n, device)
    inner, warp = float(d + 1), float(cdiv(d, 32) + WARP_LEVELS + 1)
    a, b = (inner, warp) if lane_sum_first else (warp, inner)
    return torch.where(sp, torch.full(sp.shape, a, dtype=torch.float64, device=device),
                       torch.full(sp.shape, b, dtype=torch.float64, device=device))


def query_bound(model: str, combine, a, p) -> torch.Tensor:
    """Per-element bound on kgeb_query_build: c u sum|terms| (C_QUERY; RESCAL sp_ d + 1, _po ceil(d/32) + 6)."""
    n, d = a.shape
    c = _rescal_c(combine, n, d, a.device, True) if model == "rescal" else C_QUERY[model]
    return c * U * query(model, combine, a, p, absolute=True)


def query_grads_bound(model: str, combine, a, p, g, dg=None):
    """Per-element bounds (da, dp) on kgeb_query_bwd for a dQ g known to dg (absolute, per element): the roundings
    (C_QUERY_BWD; RESCAL da ceil(d/32) + 6 for sp_, d + 1 for _po, dM 1) on the sums of |terms|, plus dg carried through
    the (bi)linear transform, i.e. the same sums of |terms| with |g| replaced by dg."""
    n, d = a.shape
    da_abs, dp_abs = query_grads(model, combine, a, p, g, absolute=True)
    if model == "rescal":
        c_a, c_p = _rescal_c(combine, n, d, a.device, False), 1
    else:
        c_a, c_p = C_QUERY_BWD[model]
    da_b, dp_b = c_a * U * da_abs, c_p * U * dp_abs
    if dg is not None:
        ea, ep = query_grads(model, combine, a, p, dg, absolute=True)
        da_b, dp_b = da_b + ea, dp_b + ep
    return da_b, dp_b


# ---------------------------------------------------------------------------------------------------------------------
# pair scores and their backward
# ---------------------------------------------------------------------------------------------------------------------
def _pair_terms(kind: int, Q, table, cand):
    q = Q.double()[:, None, :]
    c = table.double()[cand.long()]
    return q, c


def modulus(x: torch.Tensor) -> torch.Tensor:
    """|re + i im| per complex coordinate of rows [..., d] = [re | im]."""
    h = x.shape[-1] // 2
    return torch.sqrt(x[..., :h] ** 2 + x[..., h:] ** 2)


def pair_scores(kind: int, Q, table, cand) -> torch.Tensor:
    """Scores [B, M] of the query rows Q [B, d] against table[cand[b, j]], with the kernels' conventions: DOT = q.c,
    NEG_L1 / NEG_L2 = -||q - c||_1 / _2 (no eps: the sp_ / _po form), ROT_L1 / ROT_L2 = +sum / +sqrt of the complex
    moduli |q - c| (RotatE scores the positive distance in this revision)."""
    q, c = _pair_terms(kind, Q, table, cand)
    if kind == DOT:
        return (q * c).sum(-1)
    x = q - c
    if kind == NEG_L1:
        return -x.abs().sum(-1)
    if kind == NEG_L2:
        return -x.square().sum(-1).sqrt()
    if kind == ROT_L1:
        return modulus(x).sum(-1)
    return x.square().sum(-1).sqrt()


def pair_score_bound(kind: int, Q, table, cand, dq=None) -> torch.Tensor:
    """Per-pair bound on |pairs_score - pair_scores| (pair_accumulate_nosum + warp_sum + pair_finish).
    Each lane sums its columns in order: ceil(d/128) float4 groups when d % 4 == 0 -- a term passes through the 3 FMAs
    of its group, the group's add to the lane sum and the later groups' adds: at most ceil(d/128) + 4 roundings -- or
    ceil(d/32) scalar steps (+1 for the product or |q - c|); then 5 butterfly levels.  Before the sum a term carries:
    DOT 0 (the product is counted above), NEG_L1 1 (q - c), L2 2 (q - c, squared), ROT_L1 3 (re, im, re^2 + im^2 and
    the sqrt: 2u + u).  The L2 kinds take a sqrt of the sum S: dsqrt(S) <= dS / (2 sqrt S) + u sqrt S.
    dq [B, d]: the fp32 Q differs from the exact one by at most dq per element; a score moves by at most sum_k dq_k |c_k|
    (DOT) or sum_k dq_k (the distances are 1-Lipschitz in each column: L1, L2 <= L1, a complex modulus)."""
    b = _pair_score_bound(kind, Q, table, cand)
    if dq is None:
        return b
    dq = dq.double()[:, None, :]
    if kind == DOT:
        return b + (dq * table.double()[cand.long()].abs()).sum(-1)
    return b + dq.sum(-1)


def _pair_score_bound(kind: int, Q, table, cand) -> torch.Tensor:
    q, c = _pair_terms(kind, Q, table, cand)
    d = Q.shape[1]
    if kind == ROT_L1:
        k, cc = cdiv(d // 2, 32) + 1 + WARP_LEVELS, 3
    else:
        k = (cdiv(d, 128) + 4 if d % 4 == 0 else cdiv(d, 32) + 1) + WARP_LEVELS
        cc = {DOT: 0, NEG_L1: 1, NEG_L2: 2, ROT_L2: 2}[kind]
    if kind == DOT:
        return (k + cc) * U * (q * c).abs().sum(-1)
    x = q - c
    if kind == NEG_L1:
        return (k + cc) * U * x.abs().sum(-1)
    if kind == ROT_L1:
        return (k + cc) * U * modulus(x).sum(-1)
    dist = x.square().sum(-1).sqrt()
    return ((k + cc) / 2 + 1) * U * dist


def pair_grads(kind: int, Q, table, cand, G):
    """(dQ [B, d], dC [B, M, d]) of sum_j G[b, j] score[b, j]: dC[b, j] is the gradient of the row table[cand[b, j]].
    Zero conventions of the kernels: sign(0) = 0; a zero distance (L2 kinds) or a zero complex modulus (ROT_L1) gives a
    zero term."""
    q, c = _pair_terms(kind, Q, table, cand)
    g = G.double()[..., None]
    if kind == DOT:
        return (g * c).sum(1), (g * q).expand_as(c).clone()
    x = q - c
    if kind == NEG_L1:
        t = -g * torch.sign(x)
    elif kind in (NEG_L2, ROT_L2):
        dist = x.square().sum(-1, keepdim=True).sqrt()
        coef = torch.where(dist == 0, torch.zeros_like(dist), (-g if kind == NEG_L2 else g) / dist.clamp(min=1e-300))
        t = coef * x
    else:
        h = x.shape[-1] // 2
        m = modulus(x)
        inv = torch.where(m == 0, torch.zeros_like(m), g / m.clamp(min=1e-300))
        t = x * torch.cat((inv, inv), -1)
    return t.sum(1), -t


def pair_grad_terms_bound(kind: int, Q, table, cand, G, dG=0.0, dscore=0.0, dq=None):
    """(|t|, err(t), |dC|, err(dC)), all [B, M, d]: the size of each pair's dQ term t and of its candidate-gradient row
    (-t; DOT: g q) and bounds on their fp32 errors, for a G known to dG (absolute, per pair) and -- the L2 kinds, whose
    kernels divide by the fp32 score -- a score known to dscore (absolute, per pair).
    Roundings of one term: DOT g c / g q 1; NEG_L1 0 (the sign of
    q - c is exact); L2 kinds x = q - c, g / dist, coef x: 3, plus the relative error dscore / dist of the divisor;
    ROT_L1 x (1), the modulus (3), g / m (1), the product (1): 6.
    dq [B, d] (a Q known to dq per element) adds: DOT |g| dq to dC; NEG_L1 2|g| where |q - c| <= dq (the sign may flip);
    L2 kinds |g| (dq_k + |x_k| / dist sum dq) / dist (x / dist moves by that); ROT_L1 |g| (dq_re + dq_im) / m."""
    q, c = _pair_terms(kind, Q, table, cand)
    g = G.double()[..., None].abs()
    dg = torch.as_tensor(dG, dtype=torch.float64, device=q.device)
    dg = dg[..., None] if dg.dim() else dg
    dqq = torch.zeros_like(q) if dq is None else dq.double()[:, None, :]
    if kind == DOT:
        tq, tc = g * c.abs(), (g * q.abs()).expand_as(c)
        return tq, dg * c.abs() + U * tq, tc, dg * q.abs() + U * tc + g * dqq
    x = q - c
    if kind == NEG_L1:
        nz = (x != 0).double()
        t = g * nz
        e = dg * nz + torch.where(x.abs() <= dqq, 2 * g, torch.zeros_like(t))
        return t, e, t, e
    if kind in (NEG_L2, ROT_L2):
        dist = x.square().sum(-1, keepdim=True).sqrt()
        ds = torch.as_tensor(dscore, dtype=torch.float64, device=q.device)
        ds = ds[..., None] if ds.dim() else ds
        r = torch.where(dist == 0, torch.zeros_like(dist), x.abs() / dist.clamp(min=1e-300))
        rho = torch.where(dist == 0, torch.zeros_like(dist), ds / dist.clamp(min=1e-300))
        t = g * r
        e = r * (dg + g * (rho + 3 * U))
        if dq is not None:
            e = e + torch.where(dist == 0, torch.zeros_like(x),
                                g * (dqq + r * dqq.sum(-1, keepdim=True)) / dist.clamp(min=1e-300))
        return t, e, t, e
    m = modulus(x)
    m2 = torch.cat((m, m), -1)
    r = torch.where(m2 == 0, torch.zeros_like(m2), x.abs() / m2.clamp(min=1e-300))
    t = g * r
    e = r * (dg + 6 * U * g)
    if dq is not None:
        h = x.shape[-1] // 2
        dm = dqq[..., :h] + dqq[..., h:]
        dm2 = torch.cat((dm, dm), -1)
        e = e + torch.where(m2 == 0, torch.zeros_like(m2), g * dm2 / m2.clamp(min=1e-300))
    return t, e, t, e


def dq_bound(abs_t: torch.Tensor, err_t: torch.Tensor) -> torch.Tensor:
    """Bound on dQ [B, d] = sum_j t[b, j]: the terms' own errors plus the chain of the block-per-row kernels -- warp w adds
    candidates j = w, w + 8, ... in order (ceil(M/8) roundings), then the 8 warp partials are added in fixed order (8)."""
    m = abs_t.shape[1]
    return err_t.sum(1) + (cdiv(m, PAIR_BWD_WARPS) + PAIR_BWD_WARPS) * U * abs_t.sum(1)


# ---------------------------------------------------------------------------------------------------------------------
# negative-sampling loss of [B, M] score rows, column 0 = the positive
# ---------------------------------------------------------------------------------------------------------------------
def ns_rows_and_grad(loss: int, scores, offset: float = 0.0, inv_batch: float = 1.0):
    """(per-row loss [B], dL/dscores [B, M]) in float64, both scaled by inv_batch.  KL: cross entropy with class 0;
    BCE: sum_j softplus(x_j + off) - (x_0 + off)."""
    x = scores.double()
    lab = torch.zeros_like(x)
    lab[:, 0] = 1.0
    if loss == KL:
        lse = torch.logsumexp(x, 1)
        return inv_batch * (lse - x[:, 0]), inv_batch * (torch.softmax(x, 1) - lab)
    z = x + offset
    rows = torch.nn.functional.softplus(z).sum(1) - z[:, 0]
    return inv_batch * rows, inv_batch * (torch.sigmoid(z) - lab)


def _expf_rel(arg: torch.Tensor) -> torch.Tensor:
    """Relative error of __expf(arg): 2 + floor(1.173 |arg|) ulp (Programming Guide), +1 ulp for the rounding of the
    argument the kernel computed."""
    return (3 + 1.173 * arg.abs()) * ULP


def ns_loss_bound(loss: int, scores, offset: float = 0.0, inv_batch: float = 1.0, dscore=0.0):
    """(row bound [B], G bound [B, M]) on the fp32 results of ns_loss_kernel / the loss warp of ns_fused_kernel, for scores
    known to dscore (absolute, per element; 0 when the kernel is given the scores).  The warp sums M columns, ceil(M/32)
    per lane, then 5 butterfly levels: chain ceil(M/32) + 5.
    KL: e_j = __expf(x_j - mx) has relative error rel_j = dscore_j + u|x_j - mx| (the subtraction) + _expf_rel; the sum
    S adds max rel_j and the chain; p_j = e_j (1/S) two more roundings; G_j = inv_batch (p_j - [j == 0]) one rounding of
    the difference and one of the product.  The row loss mx + __logf(S) - x_0 carries dscore_0 + max dscore, the relative
    error of S (an absolute error of log S), __logf's 2^-21.41 absolute or 3 ulp, and the roundings of the two adds.
    BCE: z = x + off (dz = dscore + u|z|); softplusf(z) = max(z, 0) + __logf(1 + __expf(-|z|)): dz, the exp error
    times t = e^-|z|, the rounding of 1 + t (u absolute: it lies in [1, 2]), __logf's 2^-21.41 absolute and the final
    add u|sp|; a saturated term (t < u) is off by about u absolute, so the row bound has an absolute part of about M u.
    sigmoidf = __fdividef(1, 1 + __expf(-z)): sigma(1 - sigma)(dz + exp error) + (u + 2 ulp) sigma; exp overflow gives
    0 for sigma < 1e-38 (TINY)."""
    x = scores.double()
    b, m = x.shape
    ds = torch.as_tensor(dscore, dtype=torch.float64, device=x.device).expand_as(x)
    chain = cdiv(m, 32) + WARP_LEVELS
    onehot = torch.zeros_like(x)
    onehot[:, 0] = 1.0
    rows, g = ns_rows_and_grad(loss, x, offset, 1.0)
    if loss == KL:
        mx = x.max(1, keepdim=True).values
        a = x - mx
        rel_e = ds + U * a.abs() + _expf_rel(a)
        rel_s = rel_e.max(1, keepdim=True).values + (chain + 1) * U
        p = torch.softmax(x, 1)
        under = torch.where(a < -80, p, torch.zeros_like(p))             # __expf underflow to 0 / denormals
        g_b = inv_batch * (p * (rel_e + rel_s + 2 * U) + U * (p - onehot).abs() + under) + U * inv_batch * g.abs() + TINY
        s = torch.exp(a).sum(1)
        logs = torch.log(s)
        row_b = (ds[:, 0] + ds.max(1).values + rel_s[:, 0] + LOGF_ABS + 3 * ULP * logs.abs()
                 + U * (mx[:, 0].abs() + logs.abs() + (mx[:, 0] + logs).abs()) + U * rows.abs())
        return inv_batch * row_b + U * inv_batch * rows.abs(), g_b
    z = x + offset
    dz = ds + U * z.abs()
    t = torch.exp(-z.abs())
    sp = torch.nn.functional.softplus(z)
    term = sp - onehot * z
    term_e = dz + t * _expf_rel(z) + U + LOGF_ABS + U * sp + onehot * (dz + U * term.abs())
    row_b = term_e.sum(1) + (chain + 1) * U * term.abs().sum(1)
    sig = torch.sigmoid(z)
    g_b = (inv_batch * (sig * (1 - sig) * (dz + _expf_rel(z)) + 6 * U * sig + U * (sig - onehot).abs() + TINY)
           + U * inv_batch * g.abs())
    return inv_batch * row_b + U * inv_batch * rows.abs(), g_b


# ---------------------------------------------------------------------------------------------------------------------
# row sums of the scatter
# ---------------------------------------------------------------------------------------------------------------------
def index_add(ids, rows, vocab: int, prefill=None) -> torch.Tensor:
    """float64 dense [vocab, d] = prefill + sum of rows[i] into row ids[i] (ids outside [0, vocab) dropped)."""
    ids = ids.reshape(-1).long()
    rows = rows.reshape(ids.numel(), -1).double()
    keep = (ids >= 0) & (ids < vocab)
    out = torch.zeros(vocab, rows.shape[1], dtype=torch.float64, device=rows.device) if prefill is None \
        else prefill.double().clone()
    return out.index_add_(0, ids[keep], rows[keep])


def run_lengths(ids, vocab: int) -> torch.Tensor:
    ids = ids.reshape(-1).long()
    keep = (ids >= 0) & (ids < vocab)
    return torch.bincount(ids[keep], minlength=vocab)


def sorted_scatter_chain(lengths: torch.Tensor) -> torch.Tensor:
    """Longest chain of roundings of a run of L rows in the sorted scatter (update.cu, packed and segment regimes): at most
    8 adds inside a chunk, then the run's partials (at most ceil(L/8) + 1) added in chunk order, then one add onto the
    dense row."""
    return torch.clamp(lengths, max=8) + torch.div(lengths + 7, 8, rounding_mode="floor") + 2


def one_add(lengths: torch.Tensor) -> torch.Tensor:
    """The sorted scatter adds each run's sum onto the dense row with one atomicAdd (single writer)."""
    return (lengths > 0).long()


def sequential_chain(lengths: torch.Tensor) -> torch.Tensor:
    """A run of L rows added one by one onto the dense row (ns_cand_grad: in position order; ns_fused's vector reductions:
    in any order): L roundings, +1 for the final add of ns_cand_grad's register sum."""
    return lengths + 1


def scatter_bound(ids, abs_rows, vocab: int, chain, err_rows=None, prefill=None, atomic_adds=None) -> torch.Tensor:
    """Per-element bound [vocab, d] on a scatter of rows known to err_rows, whose sizes are abs_rows: the rows' own
    errors plus chain(L) u sum|rows| of each id's run of L rows (plus one rounding onto a nonzero prefill), plus FLUSH
    for each of the atomic_adds(L) float atomics that add into the row (a subnormal operand or result is lost)."""
    lengths = run_lengths(ids, vocab)
    s = index_add(ids, abs_rows, vocab)
    b = chain(lengths).double()[:, None] * U * s
    if atomic_adds is not None:
        b = b + atomic_adds(lengths).double()[:, None] * FLUSH
    if err_rows is not None:
        b = b + index_add(ids, err_rows, vocab)
    if prefill is not None:
        b = b + U * (prefill.double().abs() + s)
    return b


# ---------------------------------------------------------------------------------------------------------------------
# spo scores (the reference is kge_oracle.score_emb in float64) and their bounds
# ---------------------------------------------------------------------------------------------------------------------
def spo_bound(model: str, s, p, o, l_norm: int = 1, eps: float = 1e-6) -> torch.Tensor:
    """Per-row bound on |score_spo - score_emb(..., "spo")| (score_spo_kernel / spo_row).  Lanes stride the columns
    (ceil(w/32) steps, w = d or d/2), then 5 butterfly levels; RESCAL's lanes walk all d rows of M (d ceil(d/32) steps).
    Per-term roundings c: DistMult / CP 2 (two products), SimplE 3 (and the exact 0.5), ComplEx 6 (four triple products
    in one expression); TransE s + p - o + eps 3 roundings of sum|.|; RotatE re / im: sincosf (4u) and 3 roundings of
    |s cos| + |s sin| + |o|, the modulus 3 more.  The L2 forms take a sqrt of the sum (see pair_score_bound)."""
    s, p, o = s.double(), p.double(), o.double()
    n, d = s.shape
    h = d // 2
    if model == "distmult":
        return (cdiv(d, 32) + WARP_LEVELS + 2) * U * (s * p * o).abs().sum(1)
    if model == "cp":
        return (cdiv(h, 32) + WARP_LEVELS + 2) * U * (s[:, :h] * p * o[:, h:]).abs().sum(1)
    if model == "simple":
        t = (s[:, :h] * p[:, :h] * o[:, h:]).abs() + (s[:, h:] * p[:, h:] * o[:, :h]).abs()
        return (cdiv(h, 32) + WARP_LEVELS + 3) * U * 0.5 * t.sum(1)
    if model == "complex":
        sa, pa, oa = s.abs(), p.abs(), o.abs()
        sr, si, pr, pi, orr, oi = sa[:, :h], sa[:, h:], pa[:, :h], pa[:, h:], oa[:, :h], oa[:, h:]
        t = sr * pr * orr + si * pr * oi + sr * pi * oi + si * pi * orr
        return (cdiv(h, 32) + WARP_LEVELS + 6) * U * t.sum(1)
    if model == "rescal":
        t = torch.einsum("ni,nij,nj->n", s.abs(), p.view(n, d, d).abs(), o.abs())
        return (d * cdiv(d, 32) + WARP_LEVELS + 2) * U * t
    chain = (cdiv(d, 32) if model == "transe" else cdiv(h, 32)) + WARP_LEVELS + 1
    if model == "transe":
        x = s + p - o + eps
        ex = 3 * U * (s.abs() + p.abs() + o.abs() + eps)
        if l_norm == 1:
            return ex.sum(1) + chain * U * x.abs().sum(1)
        ssum = x.square().sum(1)
        ds = (2 * x.abs() * ex).sum(1) + (chain + 1) * U * ssum
    else:
        cr, sn = torch.cos(p), torch.sin(p)
        sr, si, orr, oi = s[:, :h], s[:, h:], o[:, :h], o[:, h:]
        re, im = sr * cr - si * sn - orr, sr * sn + si * cr - oi
        e_re = (SINCOS_REL + 3 * U) * ((sr * cr).abs() + (si * sn).abs() + orr.abs())
        e_im = (SINCOS_REL + 3 * U) * ((sr * sn).abs() + (si * cr).abs() + oi.abs())
        m = torch.sqrt(re ** 2 + im ** 2)
        em = e_re + e_im + 3 * U * m
        if l_norm == 1:
            return em.sum(1) + chain * U * m.sum(1)
        ssum = m.square().sum(1)
        ds = (2 * m * em).sum(1) + (chain + 1) * U * ssum
    dist = ssum.sqrt()
    return torch.minimum(ds / (2 * dist).clamp(min=1e-300), ds.sqrt()) + U * dist


def spo_grads(model: str, s, p, o, g, l_norm: int = 1, eps: float = 1e-6):
    """(ds, dp, do) of sum_i g_i score_spo_i in float64, explicit for TransE / RotatE with the kernels' zero conventions
    (sign(0) = 0, a zero distance or modulus gives zero), autograd through score_emb for the (multi)linear models."""
    from oracle.kge_oracle import score_emb
    s64, p64, o64, g64 = s.double(), p.double(), o.double(), g.double()[:, None]
    h = s.shape[1] // 2
    if model == "transe":
        x = s64 + p64 - o64 + eps
        if l_norm == 1:
            dd = -torch.sign(x)
        else:
            dist = x.square().sum(1, keepdim=True).sqrt()
            dd = torch.where(dist == 0, torch.zeros_like(x), -x / dist.clamp(min=1e-300))
        return g64 * dd, g64 * dd, -g64 * dd
    if model == "rotate":
        cr, sn = torch.cos(p64), torch.sin(p64)
        sr, si = s64[:, :h], s64[:, h:]
        re, im = sr * cr - si * sn - o64[:, :h], sr * sn + si * cr - o64[:, h:]
        if l_norm == 1:
            den = torch.sqrt(re ** 2 + im ** 2)
        else:
            den = torch.sqrt((re ** 2 + im ** 2).sum(1, keepdim=True)).expand_as(re)
        inv = torch.where(den == 0, torch.zeros_like(den), 1.0 / den.clamp(min=1e-300))
        dre, dim_ = g64 * re * inv, g64 * im * inv
        ds_ = torch.cat((dre * cr + dim_ * sn, -dre * sn + dim_ * cr), 1)
        do_ = torch.cat((-dre, -dim_), 1)
        dp_ = dre * (-sr * sn - si * cr) + dim_ * (sr * cr - si * sn)
        return ds_, dp_, do_
    t = [x.clone().requires_grad_(True) for x in (s64, p64, o64)]
    out = score_emb(model, t[0], t[1], t[2], "spo").view(-1)
    return tuple(v.detach() for v in torch.autograd.grad((out * g64[:, 0]).sum(), t))


def spo_grad_bound(model: str, s, p, o, g, l_norm: int = 1, eps: float = 1e-6):
    """Per-element bounds (ds, dp, do) on score_spo_bwd_kernel.  The (multi)linear models: each element is a product of
    g and two factors or a short sum of such products (ComplEx: 2 products, 4 roundings; SimplE's 0.5 g is exact), c = 4
    u of the same expression on absolute values; RESCAL's ds_i is a warp sum over j (ceil(d/32) + 5 + 2) and its do_j a
    lane-private sum over i (d + 2).  TransE L1: sign exact, error 0 unless s + p - o + eps rounds to the other sign --
    excluded where |x| exceeds its rounding error 3u sum|.|; L2 and RotatE: the distance / modulus error relative to
    itself plus 6 roundings (sincosf 4u counted once more for RotatE)."""
    s64, p64, o64, ga = s.double(), p.double(), o.double(), g.double().abs()[:, None]
    n, d = s.shape
    h = d // 2
    if model in ("distmult", "cp", "simple", "complex"):
        sa, pa, oa = s64.abs(), p64.abs(), o64.abs()
        if model == "complex":
            sr, si, pr, pi, orr, oi = sa[:, :h], sa[:, h:], pa[:, :h], pa[:, h:], oa[:, :h], oa[:, h:]
            ds_ = torch.cat((pr * orr + pi * oi, pr * oi + pi * orr), 1)
            dp_ = torch.cat((sr * orr + si * oi, sr * oi + si * orr), 1)
            do_ = torch.cat((sr * pr + si * pi, si * pr + sr * pi), 1)
            return tuple(4 * U * ga * t for t in (ds_, dp_, do_))
        # all signs +: the gradient of the score of the absolute values is the sum of |terms|
        return tuple(4 * U * t.abs() for t in spo_grads(model, sa, pa, oa, ga[:, 0]))
    if model == "rescal":
        sa, ma, oa = s64.abs(), p64.abs().view(n, d, d), o64.abs()
        ds_ = (cdiv(d, 32) + WARP_LEVELS + 2) * U * ga * torch.einsum("nij,nj->ni", ma, oa)
        do_ = (d + 2) * U * ga * torch.einsum("ni,nij->nj", sa, ma)
        dp_ = 2 * U * ga[:, :, None] * sa[:, :, None] * oa[:, None, :]
        return ds_, dp_.reshape(n, d * d), do_
    gs, gp, go = spo_grads(model, s, p, o, g, l_norm, eps)
    if model == "transe":
        x = s64 + p64 - o64 + eps
        ex = 3 * U * (s64.abs() + p64.abs() + o64.abs() + eps)
        if l_norm == 1:
            b = torch.where(x.abs() > ex, torch.zeros_like(x), 2 * ga.expand_as(x))
            return b, b, b
        dist = x.square().sum(1, keepdim=True).sqrt()
        dd = spo_bound(model, s, p, o, 2, eps)[:, None]
        rel = torch.where(dist == 0, torch.zeros_like(dist), dd / dist.clamp(min=1e-300))
        b = ga * torch.where(dist == 0, torch.zeros_like(x), (ex + x.abs() * (rel + 3 * U)) / dist.clamp(min=1e-300))
        return b, b, b
    cr, sn = torch.cos(p64), torch.sin(p64)
    sr, si, orr, oi = s64[:, :h], s64[:, h:], o64[:, :h], o64[:, h:]
    re, im = sr * cr - si * sn - orr, sr * sn + si * cr - oi
    e_re = (SINCOS_REL + 3 * U) * ((sr * cr).abs() + (si * sn).abs() + orr.abs())
    e_im = (SINCOS_REL + 3 * U) * ((sr * sn).abs() + (si * cr).abs() + oi.abs())
    m = torch.sqrt(re ** 2 + im ** 2)
    if l_norm == 1:
        den, eden = m, e_re + e_im + 3 * U * m
    else:
        den = torch.sqrt(m.square().sum(1, keepdim=True)).expand_as(m)
        eden = spo_bound(model, s, p, o, 2, eps)[:, None].expand_as(m)
    # dre = g re / den: relative error e_re / |re| + eden / den + 2u -> absolute g (e_re + |re| (eden / den + 2u)) / den
    inv = torch.where(den == 0, torch.zeros_like(den), 1.0 / den.clamp(min=1e-300))
    edre = ga * inv * (e_re + re.abs() * (eden * inv + 2 * U))
    edim = ga * inv * (e_im + im.abs() * (eden * inv + 2 * U))
    adre, adim = ga * re.abs() * inv, ga * im.abs() * inv
    b_s = torch.cat(((edre + edim) + (SINCOS_REL + 3 * U) * (adre + adim),) * 2, 1)
    b_o = torch.cat((edre, edim), 1)
    b_p = ((edre + edim) * (sr.abs() + si.abs())
           + (SINCOS_REL + 4 * U) * (adre + adim) * (sr.abs() + si.abs()))
    return b_s, b_p, b_o


# ---------------------------------------------------------------------------------------------------------------------
# Adagrad (torch.optim semantics: state += g^2; W -= lr g / (sqrt(state) + eps)) and its bound
# ---------------------------------------------------------------------------------------------------------------------
def adagrad(W, state, g, lr: float, eps: float):
    """(W', state') in float64."""
    W, state, g = W.double(), state.double(), g.double()
    s2 = state + g * g
    return W - lr * g / (s2.sqrt() + eps), s2


def adagrad_bound(W, state, g, dg, lr: float, eps: float):
    """Per-element bounds (W', state') on kgeb_adagrad_dense for a gradient known to dg.  state' = fma(g, g, s): 1
    rounding, plus (2|g| + dg) dg.  The update lr g / (sqrt(s') + eps) has slope at most lr / sqrt(s) in g (s the state
    before the step, >= the accumulator floor), so dg moves it by at most lr dg / sqrt(s); its own roundings are the fp32
    rate (1), the product (1), sqrt (1, and half the relative error of s'), + eps (1) and the division (1), and W' one
    more: 5u + rel(s') / 2 of |update| + u |W'|."""
    W64, s64, g64, dg = W.double(), state.double(), g.double(), torch.as_tensor(dg, dtype=torch.float64, device=W.device)
    w2, s2 = adagrad(W64, s64, g64, lr, eps)
    ds2 = (2 * g64.abs() + dg) * dg + U * s2
    upd = (w2 - W64).abs()
    dw = lr * dg / s64.sqrt() + upd * (5 * U + ds2 / (2 * s2)) + U * w2.abs()
    return dw, ds2
