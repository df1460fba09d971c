"""The tensor-core tile kernels of the fused all-entity loss against float64, on operands the tiles represent exactly.

Q and the table hold bf16 values (bf16 cases; the bf16 mirror then equals the fp32 table, and the fp32 label kernels see
the numbers the tiles see) or TF32 values (low 13 mantissa bits clear).  Every product is then exact and the kernels'
scores carry fp32 accumulation error only; the references (oracle/tile_ref.py) add the kernels' own intermediate roundings
-- G to bf16 before the second GEMM, P to bf16 for the flash o_sum -- and nothing else.  Every bound is per element or per
row and says where it comes from; the faults named in the docstrings move a result by more than its bound.

Column 0 of every table is 1 and column 0 of Q holds a per-row score shift (0 unless a test says otherwise); column 1 of Q
is 0.5.  So dQ[:, 0] is the row sum of the dense G and dTable[:, 1] half its column sum: single-signed sums, on which a
relative fault of G (a wrong exponent offset, a scaled weight) shows at full size instead of cancelling.
"""
import numpy as np
import pytest
import torch

from oracle import tile_ref as tr

pytestmark = pytest.mark.gpu

E_FB = 14541            # FB15k-237: 51 padding columns in the last 64-entity tile, 13 valid in its last 32-column part
U = tr.U32


@pytest.fixture(scope="module")
def kb():
    import kgeb200
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return kgeb200


def check(got, ref, tol, what):
    """|got - ref| <= tol element-wise (tol a tensor broadcastable to ref, or a number); NaN fails."""
    got, ref = got.detach().double(), ref.detach().double()
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    tol = torch.as_tensor(tol, dtype=torch.float64, device=ref.device)
    err = (got - ref).abs()
    ratio = torch.where(err == 0, torch.zeros_like(err), err / tol.clamp(min=1e-300))
    ratio = torch.where(torch.isnan(got), torch.full_like(err, float("inf")), ratio)
    worst = float(ratio.max()) if ratio.numel() else 0.0
    i = int(ratio.argmax()) if ratio.numel() else 0
    print(f"ERRBOUND {what}: max err/bound {worst:.3g} (err {float(err.flatten()[i]) if err.numel() else 0:.3e})")
    assert worst <= 1.0, f"{what}: err {float(err.flatten()[i]):.4e} > bound {float(tol.expand_as(err).flatten()[i]):.4e} " \
                         f"at flat index {i} (got {float(got.flatten()[i]):.8e}, ref {float(ref.flatten()[i]):.8e})"


def exact(x, math):
    return tr.bf16_exact(x) if math == "bf16" else tr.tf32_exact(x)


def problem(b, e, d, math="bf16", seed=0, nmax=4, empty_rows=False, shift=None):
    """Exact operands (scores ~ N(0, 1.5^2)) and a label CSR with the last entity in row 0; empty rows for BCE."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    q = torch.randn(b, d, generator=g, device="cuda") * (3.0 / d ** 0.5)
    w = torch.randn(e, d, generator=g, device="cuda") * 0.5
    w[:, 0] = 1.0
    q[:, 0] = 0.0 if shift is None else shift
    if d > 1:
        q[:, 1] = 0.5
    q, w = exact(q, math).contiguous(), exact(w, math).contiguous()
    n = torch.randint(0 if empty_rows else 1, nmax + 1, (b,), generator=g, device="cuda")
    rows = torch.repeat_interleave(torch.arange(b, device="cuda"), n)
    cols = torch.randint(0, e, (rows.numel(),), generator=g, device="cuda")
    rows, cols = torch.cat((rows, torch.zeros(1, dtype=torch.long, device="cuda"))), \
        torch.cat((cols, torch.full((1,), e - 1, dtype=torch.long, device="cuda")))
    key = torch.unique(rows * e + cols)                            # sorted: rows ascending, columns ascending in a row
    if empty_rows and b > 2:
        key = key[key // e != 1]                                   # row 1 has no label (BCE only)
    lab_off = torch.zeros(b + 1, dtype=torch.int64, device="cuda")
    lab_off[1:] = torch.cumsum(torch.bincount(key // e, minlength=b), 0)
    return q, w, lab_off, (key % e).contiguous()


def workspace(kb, b, d, n_ent, nnz):
    return kb.ops._workspace(torch.device("cuda"), kb.lib.load().kgeb_fused_workspace_bytes(b, d, n_ent, nnz))


def fused_fwd(kb, loss, math, q, w, lab_off, lab_col, ls=0.0, offset=0.0, e_lo=0, num_entities=None):
    """kgeb_fused_fwd on the table (slice) w = rows [e_lo, e_lo + len(w)) of a table of num_entities rows."""
    b, d = q.shape
    e_hi = e_lo + w.shape[0]
    st = torch.full((b, 4), float("nan"), device="cuda")
    ws = workspace(kb, b, d, w.shape[0], lab_col.numel())
    mirror = kb.ops.bf16_mirror(w).data_ptr() if math == kb.lib.MATH_BF16 else None
    kb.lib.call("kgeb_fused_fwd", loss, math, q.data_ptr(), b, d, w.data_ptr(), e_lo, e_hi, num_entities or e_hi,
                lab_off.data_ptr(), lab_col.data_ptr(), lab_col.numel(), float(ls), float(offset), mirror, st.data_ptr(),
                ws.data_ptr(), ws.numel(), kb.lib.stream_ptr(q))
    return st


def fused_bwd(kb, loss, q, w, lab_off, lab_col, lse, inv_batch, rs=None, ls=0.0, offset=0.0, e_lo=0, num_entities=None,
              d_table=None, overwrite=False, want_dq=True, want_stats=False):
    """kgeb_fused_bwd on the bf16 tiles: (dQ or None, rowstat_out or None); d_table updated in place."""
    b, d = q.shape
    e_hi = e_lo + w.shape[0]
    dq = torch.full((b, d), float("nan"), device="cuda") if want_dq else None
    st = torch.full((b, 4), float("nan"), device="cuda") if want_stats else None
    ws = workspace(kb, b, d, w.shape[0], lab_col.numel())
    kb.lib.call("kgeb_fused_bwd", loss, kb.lib.MATH_BF16, q.data_ptr(), b, d, w.data_ptr(), e_lo, e_hi,
                num_entities or e_hi, lab_off.data_ptr(), lab_col.data_ptr(), lab_col.numel(), None, float(ls),
                float(offset), None if lse is None else lse.data_ptr(), float(inv_batch),
                None if rs is None else rs.data_ptr(), kb.ops.bf16_mirror(w).data_ptr(),
                None if dq is None else dq.data_ptr(), None if d_table is None else d_table.data_ptr(),
                None if st is None else st.data_ptr(), kb.lib.BWD_OVERWRITE_TABLE if overwrite else 0, ws.data_ptr(),
                ws.numel(), kb.lib.stream_ptr(q))
    return dq, st


def loss_from_rowstat(kb, loss, st, lab_off, ls, e, inv_batch):
    b = st.shape[0]
    rows, lse, total = (torch.empty(b, device="cuda"), torch.empty(b, device="cuda"), torch.empty(1, device="cuda"))
    kb.lib.call("kgeb_loss_from_rowstat", loss, st.data_ptr(), lab_off.data_ptr(), b, float(ls), e, float(inv_batch),
                rows.data_ptr(), lse.data_ptr(), total.data_ptr(), kb.lib.stream_ptr(st))
    return rows, lse, total


# ------------------------------------------------------------------------------------------------------------------
# bounds shared by the tests
# ------------------------------------------------------------------------------------------------------------------
# Sums of E positive fp32 terms (row sums of exp, softplus) in per-thread chains of <= a few hundred terms, combined in
# a fixed order over chunks and column parts, of terms with the 2^-22-relative error of MUFU ex2 / lg2 (or the
# polynomial that stands in for some of them): 2e-6 of the sum covers this with room; the faults these statistics must
# catch -- one phantom entity in a row of 14,541 -- are 7e-5 (KL) and 8e-5 (BCE) of it.
REL_SUM = 2e-6
# MUFU ex2 and the grouped reciprocals of the BCE epilogue: <= 2^-20 relative error of one G or P element, with room.
EX2 = 2.0 ** -20


def acc_rel(e):
    """fp32 accumulation of a second GEMM over e entities: one rounding (<= 2 u with truncation) per 16-deep MMA step of
    a chunk, then a fixed-order sum over <= 148 chunk partials and the label rows."""
    return 2 * U * (-(-e // 16) + 152)


def rounded_gemm_tol(g64, eps, other):
    """Bound on |bf16(G') @ other - bf16(G) @ other| for a kernel G' within relative eps (per element) of the float64 G,
    accumulated in fp32: elements that eps can move across a bf16 rounding boundary change by one ulp (bf16_flip), the
    others by eps of themselves; plus the accumulation (acc_rel) of sum |G| |other|.  The faults the gradient tests must
    catch -- a per-column exponent offset off by 1e-3 log2 units (7e-4 of G), a flash weight scaled by 1 + 1e-3 -- move
    the single-signed columns by 7e-4 and 1e-3 of that sum; eps is ~1e-6 there, acc_rel(14541) = 1.1e-4."""
    a = other.double().abs()
    gb = tr.g_bf16(g64).abs()
    return tr.bf16_flip(g64, eps) @ a + (eps * 1.01 * gb) @ a + acc_rel(g64.shape[1]) * (gb @ a)


def bce_sp_tol(z, sb, sp64):
    """Row sums of softplus(z) on the tiles: d softplus / dz = sigmoid <= 1 weights the score bounds, REL_SUM of the
    (positive) sum, and log(1 + e^-|z|) taken of the fp32 sum 1 + e^-|z|: <= 2 u absolute per element, which loses the
    whole softplus of a score below -17 (2 min(softplus, u) per element)."""
    return (torch.sigmoid(z) * sb).sum(1) + REL_SUM * sp64 + 2 * torch.clamp(torch.nn.functional.softplus(z), max=U).sum(1)


def bce_pad_tol(e, offset):
    """The STATS epilogue of the dQ pass counts the zero-filled padding columns of a row's last tile into its products of
    (1 + e^-|z|) factors and takes n_pad softplus(offset) out afterwards: REL_SUM of that amount on top of the row's."""
    n_pad = -(-e // 64) * 64 - e
    return REL_SUM * n_pad * float(torch.nn.functional.softplus(torch.tensor(offset, dtype=torch.float64)))


def kl_lse_tol(x, sb, lse64):
    """|lse - lse64| <= the softmax-weighted score error bound + REL_SUM (log of a sum: relative -> absolute) + the fp32
    rounding of lse and of its two parts (max + log(sum))."""
    p = torch.softmax(x, 1)
    return (p * sb).sum(1) + REL_SUM + 4 * U * (lse64.abs() + x.max(1).values.abs())


def label_tol(q, w, y):
    """Label sums on the fp32 CUDA cores: a d-term dot of exact products per entry (<= d u sum |q e|) and the sum over
    the row's entries."""
    return (y * tr.dot_bound(q, w, c=1.0)).sum(1) + 2 * U * (y * (q.double() @ w.double().t()).abs()).sum(1)


# ------------------------------------------------------------------------------------------------------------------
# forward statistics and scores (kgeb_fused_fwd, kgeb_score_all, kgeb_loss_from_rowstat)
# ------------------------------------------------------------------------------------------------------------------
FWD_SHAPES = [(1, 1, 32), (257, E_FB, 128), (300, E_FB, 256), (77, 5000, "partial"), (40000, 2000, 32)]
FWD_IDS = ["1x1", "odd-query-blocks", "d256", "partial-k-slab", "multi-wave"]


@pytest.mark.parametrize("shape", FWD_SHAPES, ids=FWD_IDS)
@pytest.mark.parametrize("math", ["tf32", "bf16"])
@pytest.mark.parametrize("loss,ls", [("kl", 0.0), ("bce", 0.0), ("bce", 0.1)])
def test_fused_forward_statistics(kb, shape, math, loss, ls):
    """kgeb_fused_fwd on the TF32 / bf16 tiles (online maximum, ragged tiles, nqb = 1 at d = 256, a partial K slab at
    d = 100 / 72, chunks = 1 with > 148 query groups at B = 40,000) and kgeb_loss_from_rowstat on its statistics, against
    float64.  Smallest fault caught: one phantom zero-score entity in a row (7e-5 of a KL row sum, 8e-5 of a BCE one)."""
    b, e, d = shape
    if d == "partial":
        d = 100 if math == "tf32" else 72
    kl = loss == "kl"
    offset = 0.0 if kl else 0.25
    q, w, lab_off, lab_col = problem(b, e, d, math, seed=b + d, empty_rows=not kl)
    mm = kb.lib.MATH_TF32 if math == "tf32" else kb.lib.MATH_BF16
    st = fused_fwd(kb, kb.lib.LOSS_KL if kl else kb.lib.LOSS_BCE, mm, q, w, lab_off, lab_col, ls, offset)
    x = q.double() @ w.double().t()
    sb = tr.dot_bound(q, w)
    y = tr.label_matrix(lab_off, lab_col, b, e)
    if kl:
        lse64, lab64, rows64 = tr.kl_forward(x, y)
        check(st[:, 0], x.max(1).values, sb.max(1).values + U * x.max(1).values.abs(), f"{math} kl row max")
        lse = st[:, 0].double() + torch.log(st[:, 1].double())
        lse_tol = kl_lse_tol(x, sb, lse64)
        check(lse, lse64, lse_tol, f"{math} kl lse {shape}")
        lab_t = label_tol(q, w, y)
        check(st[:, 3], lab64, lab_t, f"{math} kl label sums")
        nnz = y.sum(1)
        rows, lse_k, _ = loss_from_rowstat(kb, kb.lib.LOSS_KL, st, lab_off, 0.0, e, 1.0 / b)
        check(lse_k, lse64, lse_tol + 2 * U * lse64.abs(), f"{math} kl lse (loss_from_rowstat)")
        check(rows, rows64 / b, (lse_tol + lab_t / nnz + 8 * U * (lse64.abs() + (lab64 / nnz).abs())) / b,
              f"{math} kl row losses")
    else:
        sp64, xs64, lab64, rows64 = tr.bce_forward(x, y, offset, ls, e)
        z = x + offset
        sp_tol = bce_sp_tol(z, sb, sp64)
        check(st[:, 0], sp64, sp_tol, f"{math} bce softplus sums {shape}")
        # signed sum of E terms: the score bounds plus per-chain fp32 rounding, REL_SUM of the sum of |z|
        xs_tol = sb.sum(1) + REL_SUM * z.abs().sum(1)
        check(st[:, 2], xs64, xs_tol, f"{math} bce score sums")
        lab_t = label_tol(q, w, y)
        check(st[:, 3], lab64, lab_t, f"{math} bce label sums")
        rows, _, _ = loss_from_rowstat(kb, kb.lib.LOSS_BCE, st, lab_off, ls, e, 1.0 / b)
        add = 1.0 / e if ls > 0 else 0.0
        check(rows, rows64 / b, (sp_tol + (1 - ls) * lab_t + add * xs_tol + 8 * U * (sp64 + lab64.abs())) / b,
              f"{math} bce row losses (empty rows included)")


@pytest.mark.parametrize("shape", FWD_SHAPES, ids=FWD_IDS)
def test_tf32_score_all_into_a_wider_matrix(kb, shape):
    """kgeb_score_all on the TF32 tiles writing columns [col_off, col_off + m) of a wider, sentinel-filled matrix: every
    score within its per-element accumulation bound and no other element touched.  Smallest fault caught: a score
    off by one fp32 ulp of the sum of |products| beyond the bound, a write one column left or right of the window."""
    b, e, d = shape
    d = 100 if d == "partial" else d
    q, w, _, _ = problem(b, e, d, "tf32", seed=7 + d)
    col_off, ld = 17, e + 17 + 23
    sentinel = 12345.678
    out = torch.full((b, ld), sentinel, device="cuda")
    kb.ops.score_all_into(kb.lib.DOT, q, w, out, col_off, None, kb.lib.MATH_TF32)
    x = q.double() @ w.double().t()
    check(out[:, col_off:col_off + e], x, tr.dot_bound(q, w), f"tf32 scores {shape}")
    assert bool((out[:, :col_off] == sentinel).all()) and bool((out[:, col_off + e:] == sentinel).all()), \
        "kgeb_score_all wrote outside its column window"


# ------------------------------------------------------------------------------------------------------------------
# two-pass backward (kgeb_fused_bwd: dQ, dTable, rowstat_out)
# ------------------------------------------------------------------------------------------------------------------
def bwd_reference(q, w, lab_off, lab_col, kl, lse32, inv_batch, rs_vec, ls, offset, e_total, e_lo=0):
    """(dQ, dTable, dQ bound, dTable bound) in float64 for the shard w = rows [e_lo, e_lo + len(w))."""
    b, e = q.shape[0], w.shape[0]
    x = q.double() @ w.double().t()
    rs = inv_batch * (torch.ones(b, dtype=torch.float64, device="cuda") if rs_vec is None else rs_vec.double())
    ls_add = (1.0 / e_total) if ls > 0 else 0.0
    g64 = tr.dense_g(x, kl, rs, lse32, offset, ls_add)
    gd = tr.g_bf16(g64)
    y = tr.label_matrix(lab_off, lab_col, b, e, e_lo)
    lw = tr.label_weight(y, kl, rs, ls)
    qd, wd = q.double(), w.double()
    dq = (gd + lw) @ wd
    dt = (gd + lw).t() @ qd
    # relative perturbation of a G element before its bf16 rounding: the score's accumulation error (dG / G <= dx),
    # MUFU, and the fp32 rounding of the exponent argument x log2e + (log rs - lse) log2e (KL) / of z (BCE, where
    # sigma - ls_add can be smaller than sigma: scaled by their ratio)
    sb = tr.dot_bound(q, w)
    if kl:
        eps = sb + EX2 + 2 * U * (x.abs() + (lse32.double().abs() + torch.log(rs).abs())[:, None])
    else:
        s_ = torch.sigmoid(x + offset)
        eps = (sb + EX2 + 2 * U * (x + offset).abs()) * s_ / (s_ - ls_add).abs().clamp(min=1e-300)
    # dense part: rounded_gemm_tol; label part: fp32 sums of a few exact-fp32 rows
    dq_tol = rounded_gemm_tol(g64, eps, wd) + 4 * U * (lw.abs() @ wd.abs()) + 1e-30
    dt_tol = rounded_gemm_tol(g64.t(), eps.t(), qd) + 4 * U * (lw.abs().t() @ qd.abs()) + 1e-30
    return dq, dt, dq_tol, dt_tol


def lse32_of(q, w):
    return torch.logsumexp(q.double() @ w.double().t(), 1).float()


BWD_CASES = (
    [(loss, 1000, E_FB, d, False) for loss in ("kl", "bce") for d in (16, 80, 128, 144, 256)]
    + [("kl", b, E_FB, 128, False) for b in (64, 4096, 4097, 8205)]       # colk path (<= 4096 rows) vs shuffle path
    + [("kl", 19000, 3000, 32, True), ("bce", 19000, 3000, 32, False)]     # dQ: > 148 query blocks, chunks = 1
    + [(loss, 300, e, 64, rs) for loss in ("kl", "bce") for e, rs in ((1, True), (63, False), (65, True))]
)


@pytest.mark.parametrize("loss,b,e,d,row_scale", BWD_CASES,
                         ids=[f"{c[0]}-B{c[1]}-E{c[2]}-d{c[3]}{'-rs' if c[4] else ''}" for c in BWD_CASES])
def test_fused_backward_bf16(kb, loss, b, e, d, row_scale):
    """kgeb_fused_bwd on the bf16 tiles against float64 with the kernels' bf16 rounding of G: dQ, the dense table
    gradient (accumulated onto a random prefill, and overwritten over a NaN prefill: every row written) and, for BCE,
    the forward statistics of the dQ pass (rowstat_out: the STATS epilogue and its padding correction).  Covers
    d = 16 / 80 / 144 (partial K slab), d > 128 (no A operand in tensor memory), the KL dTable's per-column exponent
    offsets (B <= 4096) and its shuffle path (B > 4096), > 148 dQ blocks, E = 1 / 63 / 65.  Smallest faults caught: an
    exponent offset off by 1e-3 (log2 units), a padding column counted in a BCE row's statistics."""
    kl = loss == "kl"
    offset, ls = (0.0, 0.0) if kl else (0.25, 0.1 if d == 80 else 0.0)
    q, w, lab_off, lab_col = problem(b, e, d, "bf16", seed=3 * b + d + e, empty_rows=not kl)
    g = torch.Generator(device="cuda").manual_seed(b)
    rs = (torch.rand(b, generator=g, device="cuda") + 0.5) if row_scale else None
    lse32 = lse32_of(q, w) if kl else None
    kind = kb.lib.LOSS_KL if kl else kb.lib.LOSS_BCE
    dq_ref, dt_ref, dq_tol, dt_tol = bwd_reference(q, w, lab_off, lab_col, kl, lse32, 1.0 / b, rs, ls, offset, e)
    prefill = torch.randn(e, d, generator=g, device="cuda")
    dt_acc = prefill.clone()
    dq, st = fused_bwd(kb, kind, q, w, lab_off, lab_col, lse32, 1.0 / b, rs, ls, offset, d_table=dt_acc,
                       want_stats=not kl)
    check(dq, dq_ref, dq_tol, f"{loss} dQ B={b} E={e} d={d}")
    # accumulate mode: prefill + gradient (fp32: the dense part is added in L2, the label rows on top: two roundings)
    check(dt_acc, prefill.double() + dt_ref, dt_tol + 2 * U * (prefill.double().abs() + dt_ref.abs()),
          f"{loss} dTable (accumulate) B={b} E={e} d={d}")
    dt_ovw = torch.full((e, d), float("nan"), device="cuda")
    fused_bwd(kb, kind, q, w, lab_off, lab_col, lse32, 1.0 / b, rs, ls, offset, d_table=dt_ovw, overwrite=True,
              want_dq=False)
    check(dt_ovw, dt_ref, dt_tol, f"{loss} dTable (overwrite) B={b} E={e} d={d}")
    if not kl:
        x = q.double() @ w.double().t()
        y = tr.label_matrix(lab_off, lab_col, b, e)
        sp64, xs64, lab64, _ = tr.bce_forward(x, y, offset, ls, e)
        sb = tr.dot_bound(q, w)
        z = x + offset
        check(st[:, 0], sp64, bce_sp_tol(z, sb, sp64) + bce_pad_tol(e, offset),
              f"bce rowstat_out softplus sums d={d}")
        check(st[:, 2], xs64, sb.sum(1) + REL_SUM * z.abs().sum(1), f"bce rowstat_out score sums d={d}")
        check(st[:, 3], lab64, label_tol(q, w, y), f"bce rowstat_out label sums d={d}")


# ------------------------------------------------------------------------------------------------------------------
# flash pass (kgeb_fused_flash_fwd / _dq)
# ------------------------------------------------------------------------------------------------------------------
def flash_reference(q, w, lab_off, lab_col, mref):
    """(row sums of P = exp(x - mref) in float64, o_sum = bf16(P) @ w, label sums, bounds) against the kernel's mref."""
    b, e = q.shape[0], w.shape[0]
    x = q.double() @ w.double().t()
    p = torch.exp(x - mref.double()[:, None])
    pb = p.float().bfloat16().double()
    y = tr.label_matrix(lab_off, lab_col, b, e)
    sb = tr.dot_bound(q, w)
    l_tol = (p * sb).sum(1) * 1.0001 + REL_SUM * p.sum(1)    # d exp(x) = exp(x) dx, first order
    o = pb @ w.double()
    o_tol = rounded_gemm_tol(p, sb + EX2 + 2 * U * (x.abs() + mref.double().abs()[:, None]), w) + 1e-30
    return x, p.sum(1), l_tol, o, o_tol, y


def check_flash(kb, q, w, lab_off, lab_col, what, shard=None):
    """Runs the flash pass on (q, w) and checks everything against float64; returns (rowstat_local, o_sum)."""
    e = w.shape[0]
    shard = shard or kb.fused.Shard.full(e)
    local, o_sum, status = kb.fused.flash_forward(q, w, lab_off, lab_col, shard)
    assert int(status.item()) == 0, f"{what}: the flash pass reported a score outside its window"
    mref = local[:, 0]
    assert bool(torch.isfinite(mref).all())
    x, l64, l_tol, o64, o_tol, y = flash_reference(q, w, lab_off, lab_col, mref)
    check(local[:, 1], l64, l_tol, f"{what} flash row sums of P")
    check(o_sum, o64, o_tol, f"{what} flash o_sum")
    check(local[:, 3], (x * y).sum(1), label_tol(q, w, y), f"{what} flash label sums")
    return local, o_sum, x, y


def flash_dq_reference(q, w, y, local, o_sum, lse32, inv_batch, nnz):
    """dQ of kgeb_fused_flash_dq on its own inputs (the kernel's mref and o_sum, an fp32 lse): w_q exp(mref - lse) o_sum -
    (w_q / nnz) sum of the row's label rows in this shard (nnz = the row's label count over the whole table); bound: fp32
    exp / products of the first term (8 u + 2^-21 of it; its argument mref - lse, |.| <= 30, rounds to 2e-6 absolute)
    and fp32 sums of the label rows."""
    nnz = nnz.double()
    wq = inv_batch * (nnz > 0).double()
    dense = (wq * torch.exp(local[:, 0].double() - lse32.double()))[:, None] * o_sum.double()
    lab = (wq / nnz.clamp(min=1))[:, None] * (y @ w.double())
    tol = 8e-6 * dense.abs() + 4 * U * (wq / nnz.clamp(min=1))[:, None] * (y @ w.double().abs()) + 1e-30
    return dense - lab, tol


@pytest.mark.parametrize("d", [64, 144, 256])
@pytest.mark.parametrize("e", [65, E_FB])
def test_flash_forward_and_dq(kb, d, e):
    """kgeb_fused_flash_fwd (row sums of P against the kernel's own reference mref, o_sum with P rounded to bf16, label
    sums) and kgeb_fused_flash_dq on its own inputs, against float64; d = 144 / 256 run without the A operand in tensor
    memory.  Smallest faults caught: a padding column's P in the row sum (exp(-mref) against sums of 1e2-1e4), a flash
    dQ weight scaled by 1 + 1e-3."""
    b = 600
    q, w, lab_off, lab_col = problem(b, e, d, "bf16", seed=d + e)
    local, o_sum, x, y = check_flash(kb, q, w, lab_off, lab_col, f"d={d} E={e}")
    lse32 = torch.logsumexp(x, 1).float()
    dq = kb.fused.flash_dq(q, w, lab_off, lab_col, local, lse32, 1.0 / b, None, o_sum, kb.fused.Shard.full(e))
    ref, tol = flash_dq_reference(q, w, y, local, o_sum, lse32, 1.0 / b, y.sum(1))
    check(dq, ref, tol, f"flash dQ d={d} E={e}")


# ------------------------------------------------------------------------------------------------------------------
# rank counts (kgeb_rank_count, TF32 tiles) on dyadic tables: exact in any summation order
# ------------------------------------------------------------------------------------------------------------------
def dyadic(n, d, g):
    return (torch.randint(-4, 5, (n, d), generator=g, device="cuda").float() / 8).contiguous()


def rank_reference(q, w, true_ent):
    x = q.double() @ w.double().t()
    t = x.gather(1, true_ent[:, None]).squeeze(1)
    return (x > t[:, None]).sum(1), (x == t[:, None]).sum(1), t.float()


@pytest.mark.parametrize("nq,e,d", [(300, E_FB, 256), (40000, 2000, 32)], ids=["d256", "multi-wave"])
def test_tf32_rank_counts_exact(kb, nq, e, d):
    """kgeb_rank_count on the TF32 tiles on dyadic tables (entries k/8, |k| <= 4: scores exact in fp32 and TF32 in any
    order, many ties) against exact counting: raw (rank, ties) bit-exact, at d = 256 (one query block per job) and with
    > 148 query groups.  Smallest fault caught: one miscounted candidate."""
    g = torch.Generator(device="cuda").manual_seed(nq + d)
    q, w = dyadic(nq, d, g), dyadic(e, d, g)
    true_ent = torch.randint(0, e, (nq,), generator=g, device="cuda")
    gt, ties, t = rank_reference(q, w, true_ent)
    counts = kb.fused.rank_counts(kb.lib.DOT, q, w, t, true_ent, None, None, kb.lib.MATH_TF32)
    assert torch.equal(counts[:, 0], gt) and torch.equal(counts[:, 1], ties)


# ------------------------------------------------------------------------------------------------------------------
# one table split into shards with e_lo > 0, on one GPU
# ------------------------------------------------------------------------------------------------------------------
SPLIT = [(0, 4097), (4097, 9000), (9000, E_FB)]


def shards_of(kb, w):
    return [(lo, hi, w[lo:hi].clone(), kb.fused.Shard(lo, hi, w.shape[0])) for lo, hi in SPLIT]


def test_sharded_table_statistics_and_gradients(kb):
    """E = 14,541 split at 4097 / 9000 (not multiples of 64 or 128), labels in every shard: per-shard statistics of the
    TF32 and bf16 forward kernels and of the flash pass (each shard's own mref) combined with the shard formula of
    fused.combine_rowstats, summed dQ partials of the two-pass and flash kernels, three shards of rank counts
    accumulating into one buffer -- all against the full-table float64 reference; each shard's dTable rows against
    their slice.  Smallest fault caught: a shard scoring its rows against the wrong entity ids (labels, e_lo)."""
    b, d, e = 700, 128, E_FB
    q, w, lab_off, lab_col = problem(b, e, d, "bf16", seed=91, nmax=6)
    x = q.double() @ w.double().t()
    y = tr.label_matrix(lab_off, lab_col, b, e)
    assert all(bool(y[:, lo:hi].sum() > 0) for lo, hi in SPLIT)
    lse64, lab64, _ = tr.kl_forward(x, y)
    sb = tr.dot_bound(q, w)
    lse_tol = kl_lse_tol(x, sb, lse64) + 4 * U * lse64.abs()
    parts = {"tf32": [], "bf16": [], "flash": []}
    sh = shards_of(kb, w)
    for lo, hi, ws_, shard in sh:
        for math, mm in (("tf32", kb.lib.MATH_TF32), ("bf16", kb.lib.MATH_BF16)):
            parts[math].append(fused_fwd(kb, kb.lib.LOSS_KL, mm, q, ws_, lab_off, lab_col, e_lo=lo, num_entities=e))
        local, o_sum, status = kb.fused.flash_forward(q, ws_, lab_off, lab_col, shard)
        assert int(status.item()) == 0, f"flash pass of shard [{lo}, {hi}) reported a failure"
        parts["flash"].append((local, o_sum))
    for math in ("tf32", "bf16"):
        st = tr.combine_rowstats(parts[math], kl=True)
        check(st[:, 0] + torch.log(st[:, 1]), lse64, lse_tol, f"sharded {math} lse")
        check(st[:, 3], lab64, label_tol(q, w, y), f"sharded {math} label sums")
    stf = tr.combine_rowstats([p[0] for p in parts["flash"]], kl=True)
    check(stf[:, 0] + torch.log(stf[:, 1]), lse64, lse_tol, "sharded flash lse")
    lse32 = lse64.float()
    # two-pass backward: dQ partials summed over the shards, dTable rows per shard
    dq_ref, dt_ref, dq_tol, dt_tol = bwd_reference(q, w, lab_off, lab_col, True, lse32, 1.0 / b, None, 0.0, 0.0, e)
    dq_sum = torch.zeros(b, d, dtype=torch.float64, device="cuda")
    fdq_sum = torch.zeros_like(dq_sum)
    fdq_tol = torch.zeros_like(dq_sum)
    fdq_ref = torch.zeros_like(dq_sum)
    for (lo, hi, ws_, shard), (local, o_sum) in zip(sh, parts["flash"]):
        dt = torch.full((hi - lo, d), float("nan"), device="cuda")
        dq, _ = fused_bwd(kb, kb.lib.LOSS_KL, q, ws_, lab_off, lab_col, lse32, 1.0 / b, e_lo=lo, num_entities=e,
                          d_table=dt, overwrite=True)
        dq_sum += dq.double()
        check(dt, dt_ref[lo:hi], dt_tol[lo:hi], f"sharded dTable rows [{lo}, {hi})")
        fdq = kb.fused.flash_dq(q, ws_, lab_off, lab_col, local, lse32, 1.0 / b, None, o_sum, shard)
        fdq_sum += fdq.double()
        ys = tr.label_matrix(lab_off, lab_col, b, hi - lo, lo)
        ref_s, tol_s = flash_dq_reference(q, ws_, ys, local, o_sum, lse32, 1.0 / b, y.sum(1))
        check(fdq, ref_s, tol_s, f"sharded flash dQ partial [{lo}, {hi})")
        # the same partial from the float64 o_sum of this shard (its own mref, its P rounded to bf16)
        _, _, _, o64, o_tol, _ = flash_reference(q, ws_, lab_off, lab_col, local[:, 0])
        check(o_sum, o64, o_tol, f"sharded flash o_sum [{lo}, {hi})")
        ref64_s, _ = flash_dq_reference(q, ws_, ys, local, o64, lse32, 1.0 / b, y.sum(1))
        fdq_ref += ref64_s
        fdq_tol += tol_s + (1.0 / b) * torch.exp(local[:, 0].double() - lse32.double())[:, None] * o_tol
    check(dq_sum, dq_ref, dq_tol + 2 * U * dq_sum.abs(), "sharded dQ (sum of partials)")
    # flash dQ summed over the shards against float64 o_sums (each shard's P rounded to bf16 against its own mref: the
    # rounding points differ from the two-pass G, so the reference is the flash arithmetic, not dq_ref)
    check(fdq_sum, fdq_ref, fdq_tol + 2 * U * fdq_sum.abs(), "sharded flash dQ (sum of partials)")
    # BCE statistics over the shards: plain sums
    kq, kw, klo, klc = problem(b, e, d, "tf32", seed=92, empty_rows=True)
    st = tr.combine_rowstats([fused_fwd(kb, kb.lib.LOSS_BCE, kb.lib.MATH_TF32, kq, kw[lo:hi].clone(), klo, klc, 0.0,
                                        0.25, e_lo=lo, num_entities=e) for lo, hi in SPLIT], kl=False)
    kx = kq.double() @ kw.double().t()
    ky = tr.label_matrix(klo, klc, b, e)
    sp64, xs64, klab64, _ = tr.bce_forward(kx, ky, 0.25, 0.0, e)
    ksb = tr.dot_bound(kq, kw)
    check(st[:, 0], sp64, bce_sp_tol(kx + 0.25, ksb, sp64), "sharded tf32 bce softplus sums")
    check(st[:, 3], klab64, label_tol(kq, kw, ky), "sharded tf32 bce label sums")
    # rank counts: three shards add into one buffer
    g = torch.Generator(device="cuda").manual_seed(5)
    rq, rw = dyadic(b, 64, g), dyadic(e, 64, g)
    true_ent = torch.randint(0, e, (b,), generator=g, device="cuda")
    gt, ties, t = rank_reference(rq, rw, true_ent)
    counts = torch.zeros(b, 6, dtype=torch.int64, device="cuda")
    for lo, hi in SPLIT:
        kb.fused.rank_counts(kb.lib.DOT, rq, rw[lo:hi].clone(), t, true_ent, None, None, kb.lib.MATH_TF32,
                             kb.fused.Shard(lo, hi, e), counts)
    assert torch.equal(counts[:, 0], gt) and torch.equal(counts[:, 1], ties)


# ------------------------------------------------------------------------------------------------------------------
# rows at any score level (KL is invariant under a per-row shift)
# ------------------------------------------------------------------------------------------------------------------
LEVELS = (0.0, -10.0, -30.0, -120.0)


def shifted(b):
    s = torch.tensor(LEVELS, device="cuda").repeat((b + 3) // 4)[:b].clone()
    s[-1] = -120.0                    # the last row's lse is the one the shuffle path gives the padded query columns
    return s


@pytest.mark.parametrize("b", [4096, 5000])
def test_kl_rows_at_any_score_level(kb, b):
    """Rows whose scores sit at 0, -10, -30 or -120 (exact in bf16) at E = 14,541 (51 padding columns): two-pass KL
    statistics, dQ and dTable (per-column exponent offsets at B = 4096, shuffle path at B = 5000) against float64 -- lse
    moves with the level, the gradients do not, nothing is NaN.  Smallest fault caught: G = rs exp(-lse) of a padding
    column (inf from -89 nats down: NaN in MMA2)."""
    d, e = 128, E_FB
    q, w, lab_off, lab_col = problem(b, e, d, "bf16", seed=b, shift=shifted(b))
    x = q.double() @ w.double().t()
    y = tr.label_matrix(lab_off, lab_col, b, e)
    lse64, lab64, _ = tr.kl_forward(x, y)
    sb = tr.dot_bound(q, w)
    st = fused_fwd(kb, kb.lib.LOSS_KL, kb.lib.MATH_BF16, q, w, lab_off, lab_col)
    check(st[:, 0] + torch.log(st[:, 1].double()), lse64, kl_lse_tol(x, sb, lse64), f"shifted rows: two-pass lse B={b}")
    lse32 = lse64.float()
    dq_ref, dt_ref, dq_tol, dt_tol = bwd_reference(q, w, lab_off, lab_col, True, lse32, 1.0 / b, None, 0.0, 0.0, e)
    dt = torch.full((e, d), float("nan"), device="cuda")
    dq, _ = fused_bwd(kb, kb.lib.LOSS_KL, q, w, lab_off, lab_col, lse32, 1.0 / b, d_table=dt, overwrite=True)
    assert bool(torch.isfinite(dq).all()) and bool(torch.isfinite(dt).all()), "NaN / inf in the KL gradients"
    check(dq, dq_ref, dq_tol, f"shifted rows: dQ B={b}")
    check(dt, dt_ref, dt_tol, f"shifted rows: dTable B={b}")


@pytest.mark.parametrize("levels", [(0.0, -10.0, -30.0), LEVELS], ids=["to-30", "to-120"])
def test_flash_rows_at_any_score_level(kb, levels):
    """The flash pass (kgeb_fused_flash_fwd) on rows at the given score levels, E = 14,541 (51 padding columns): the pass
    must succeed -- mref is each row's own sampled maximum, so no score lies far above it whatever the level -- and its
    row sums, o_sum and lse must match float64.  Smallest faults caught: P = exp(-mref) of a padding column in a row sum
    (swamps the last chunk's share from -20 nats down: the levels down to -30, with no row that could overflow and fail
    the whole call), and the same P overflowing to inf (rows at -120: a failed pass)."""
    b, d, e = 4096, 128, E_FB
    s = torch.tensor(levels, device="cuda").repeat(-(-b // len(levels)))[:b].clone()
    q, w, lab_off, lab_col = problem(b, e, d, "bf16", seed=len(levels), shift=s)
    local, o_sum, status = kb.fused.flash_forward(q, w, lab_off, lab_col, kb.fused.Shard.full(e))
    assert int(status.item()) == 0, "the flash pass failed on rows whose scores lie below 0"
    x, l64, l_tol, o64, o_tol, _ = flash_reference(q, w, lab_off, lab_col, local[:, 0])
    check(local[:, 1], l64, l_tol, f"shifted rows {levels}: flash row sums")
    check(o_sum, o64, o_tol, f"shifted rows {levels}: flash o_sum")
    # lse = mref + log(l) in float64 from the kernel's fp32 mref and l, against float64 with the same mref: the mref
    # terms cancel and the error is that of log(l), <= (1 + 1e-3) l_tol / l to first order; 1e-12 absolute covers the
    # float64 rounding of sums of ~|lse| <= 130
    lf = local[:, 0].double() + torch.log(local[:, 1].double())
    check(lf, torch.logsumexp(x, 1), 1.001 * l_tol / l64 + 1e-12, f"shifted rows {levels}: flash lse")


def test_bce_statistics_at_any_score_level(kb):
    """BCE forward statistics of the dQ pass (rowstat_out) and of the forward kernel for rows at 0 / -10 / -30 / -120:
    against float64, nothing NaN.  Smallest fault caught: a padding column counted in a row's softplus sum."""
    b, d, e = 1000, 128, E_FB
    q, w, lab_off, lab_col = problem(b, e, d, "bf16", seed=17, empty_rows=True, shift=shifted(b))
    x = q.double() @ w.double().t()
    y = tr.label_matrix(lab_off, lab_col, b, e)
    sp64, xs64, lab64, _ = tr.bce_forward(x, y, 0.25, 0.0, e)
    sb = tr.dot_bound(q, w)
    z = x + 0.25
    _, st = fused_bwd(kb, kb.lib.LOSS_BCE, q, w, lab_off, lab_col, None, 1.0 / b, offset=0.25, want_stats=True)
    st2 = fused_fwd(kb, kb.lib.LOSS_BCE, kb.lib.MATH_BF16, q, w, lab_off, lab_col, 0.0, 0.25)
    for name, s, pad in (("rowstat_out", st, bce_pad_tol(e, 0.25)), ("fused_fwd", st2, 0.0)):
        check(s[:, 0], sp64, bce_sp_tol(z, sb, sp64) + pad + 1e-30, f"shifted bce {name} softplus")
        check(s[:, 2], xs64, sb.sum(1) + REL_SUM * z.abs().sum(1), f"shifted bce {name} score sums")
        check(s[:, 3], lab64, label_tol(q, w, y), f"shifted bce {name} label sums")


def test_captured_large_table_step_on_shifted_rows(kb):
    """One captured FusedAllEntityStepper step (1vsAll KL, bf16 tiles, flash pass, Adagrad inside the table-gradient
    kernel) on a DistMult model whose relations shift their rows' scores to 0 / -10 / -30 / -120: the flash pass holds
    (no fallback), and the step equals the autograd flow on the same tiles, everything finite."""
    e, r, d, b = 140_000, 4, 128, 256
    torch.manual_seed(0)
    ref = kb.KgeModel("distmult", e, r, d).cuda()
    with torch.no_grad():
        for t in (ref.get_s_embedder().weight, ref.get_p_embedder().weight):
            t.copy_(tr.bf16_exact(t * 4.0))
        ref.get_s_embedder().weight[:, 0] = 1.0
        ref.get_p_embedder().weight[:, 0] = torch.tensor(LEVELS, device="cuda")
    new = kb.KgeModel("distmult", e, r, d).cuda()
    new.load_state_dict(ref.state_dict())
    mk = lambda m: kb.optim.create("Adagrad", m.parameters(), lr=0.2, initial_accumulator_value=0.1)   # noqa: E731
    jr = kb.TrainingJob1vsAll(ref, mk(ref), kb.KgeLoss.create("kl"), math_mode=kb.lib.MATH_BF16)
    st = kb.trainer.FusedAllEntityStepper(new, mk(new), 2 * b, 2 * b, kb.lib.LOSS_KL, b, math_mode=kb.lib.MATH_BF16)
    assert st.seq and st.fuse_update
    gen = torch.Generator().manual_seed(3)
    t = torch.stack((torch.randint(0, e, (b,), generator=gen), torch.arange(b) % r,
                     torch.randint(0, e, (b,), generator=gen)), 1).cuda()
    z = torch.zeros(b, dtype=torch.int32, device="cuda")
    st.set_inputs(torch.cat((t[:, 0], t[:, 2])), torch.cat((t[:, 1], t[:, 1])), torch.cat((z, z + 1)),
                  torch.arange(2 * b + 1, device="cuda"), torch.cat((t[:, 2], t[:, 0])))
    got = st.step().item()
    a = jr.step(0, {"triples": t})
    # the flash pass must hold on these rows (a fallback would hide a flash fault behind the two-pass kernels)
    assert st.flash_fallbacks == 0, "the captured step fell back to the two-pass kernels"
    assert np.isfinite(got) and got == pytest.approx(a.avg_loss, rel=2e-5)
    for x, y in ((new.get_s_embedder().weight, ref.get_s_embedder().weight), (new.get_p_embedder().weight, ref.get_p_embedder().weight)):
        assert bool(torch.isfinite(x).all())
        # the bound of test_failed_flash_pass_in_the_captured_step_... (same flows, same tiles)
        assert bool(((x - y).abs() <= 0.2 * 1e-3 + 1e-6 * y.abs()).all()), (x - y).abs().max().item()
