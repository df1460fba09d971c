"""The negative-sampling kernels, the row scorers and the sorted scatter against float64 (oracle/pair_ref.py), at the shapes
where their loops run past the first iteration: the WN18RR slot (B = 512, 1 + 256 candidates, d = 128: grid-stride loops
and the 64-bit packed scatter), many candidates per row, d % 4 != 0, both register halves of ns_cand_grad, d up to 512 in
the row scorers and n = 20,000 rows (above the 18,944 warps of one grid).

Each kernel is called through its C entry on fp32 inputs and checked against the float64 result of the same inputs with a
per-element bound derived in pair_ref (a chain of k roundings moves a sum by at most k u sum|terms|, plus the documented
accuracy of __expf / __logf / __fdividef / sincosf).  The candidates include a hub id taking about 5 % of all pairs, the
last id, candidates whose row equals the query row (distance 0) and, for RotatE, rows equal in half the complex coordinates
(modulus 0 there).
"""
import pytest
import torch

from oracle import kge_oracle as ko
from oracle import pair_ref as pr

pytestmark = pytest.mark.gpu

KINDS = {"dot": pr.DOT, "neg_l1": pr.NEG_L1, "neg_l2": pr.NEG_L2, "rot_l1": pr.ROT_L1, "rot_l2": pr.ROT_L2}
E_WN = 40943                       # WN18RR entities: 16 id bits; 512 x 257 pairs take 18 position bits -> 64-bit words
HUB = 17
LOSSES = [("kl", pr.KL, 0.0), ("bce", pr.BCE, 0.0), ("bce_off", pr.BCE, 0.5)]
# (B, M, d): the WN18RR slot; M >> 32 with B not a multiple of 8; d % 4 != 0 (ns_fused refuses, scalar pair loop) with
# 22,500 pairs (grid stride); both halves of ns_cand_grad; ns_cand_grad refuses d > 256; M = 1
SHAPES = [(512, 257, 128), (37, 1001, 64), (2500, 9, 102), (64, 33, 256), (16, 2, 512), (3, 1, 16)]


@pytest.fixture(scope="module")
def kb():
    import kgeb200
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    kgeb200.lib.load()
    return kgeb200


def st():
    return torch.cuda.current_stream().cuda_stream


def check(got, ref, tol, what):
    """|got - ref| <= tol element-wise (tol a tensor broadcastable to ref); NaN fails."""
    got, ref = got.detach().double(), ref.detach().double()
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    tol = torch.as_tensor(tol, dtype=torch.float64, device=ref.device).expand_as(ref)
    err = (got - ref).abs()
    ratio = torch.where(err == 0, torch.zeros_like(err), err / tol.clamp(min=1e-300))
    ratio = torch.where(torch.isnan(got), torch.full_like(err, float("inf")), ratio)
    worst = float(ratio.max()) if ratio.numel() else 0.0
    i = int(ratio.argmax()) if ratio.numel() else 0
    print(f"ERRBOUND {what}: max err/bound {worst:.3g}")
    assert worst <= 1.0, f"{what}: err {float(err.flatten()[i]):.4e} > bound {float(tol.flatten()[i]):.4e} at flat " \
                         f"index {i} (got {float(got.flatten()[i]):.8e}, ref {float(ref.flatten()[i]):.8e})"


def workspace(kb, n, d):
    return torch.empty(kb.lib.load().kgeb_scatter_workspace_bytes(n, d), dtype=torch.uint8, device="cuda")


def scatter(kb, ids, rows, vocab, dense):
    n, d = rows.shape
    ws = workspace(kb, n, d)
    kb.lib.call("kgeb_scatter_add_rows", ids.data_ptr(), int(ids.dtype == torch.int64), rows.data_ptr(), n, d,
                dense.data_ptr(), vocab, ws.data_ptr(), ws.numel(), st())
    return dense


def pair_problem(b, m, d, kind, seed):
    """Q [b, d], table [E, d], target [b], negatives [b, m - 1] with a hub id, the last id, zero-distance pairs and (even
    d) half-equal rows."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    e = E_WN
    table = torch.randn(e, d, generator=g, device="cuda") * 0.5
    q = torch.randn(b, d, generator=g, device="cuda") * 0.5
    cand = torch.randint(0, e, (b, m), generator=g, device="cuda")
    cand[torch.rand(b, m, generator=g, device="cuda") < 0.05] = HUB
    cand[0, m - 1] = e - 1
    cand[b - 1, 0] = e - 1
    h = d // 2
    if m > 1:
        r = torch.arange(1, b, 7, device="cuda")     # pairs (r, 1) have distance 0
        q[r] = table[cand[r, 1]]
        r = torch.arange(4, b, 7, device="cuda")     # pairs (r, m - 1): moduli 0 in half the complex coordinates
        c = table[cand[r, m - 1]]
        q[r, : h // 2] = c[:, : h // 2]
        q[r, h: h + h // 2] = c[:, h: h + h // 2]
    return q.contiguous(), table.contiguous(), cand[:, 0].contiguous(), cand[:, 1:].contiguous()


def ns_loss_call(kb, loss, scores, offset, inv_b):
    b, m = scores.shape
    G = torch.empty_like(scores)
    rows = torch.empty(b, device="cuda")
    kb.lib.call("kgeb_ns_loss", loss, scores.data_ptr(), b, m, offset, inv_b, G.data_ptr(), rows.data_ptr(), st())
    return G, rows


# every shape with KL and BCE at offset 0.5; BCE at offset 0 at the WN18RR shape
PAIR_CASES = [(s, k, l) for s in SHAPES for k in KINDS for l in LOSSES if l[0] != "bce" or s == SHAPES[0]]


@pytest.mark.parametrize("shape,kname,lcase", PAIR_CASES,
                         ids=["x".join(map(str, s)) + f"-{k}-{l[0]}" for s, k, l in PAIR_CASES])
def test_pair_path_against_float64(kb, shape, kname, lcase):
    """kgeb_ns_candidates, kgeb_pairs_score, kgeb_ns_loss, kgeb_pairs_bwd (dC row by row and through the sorted scatter),
    kgeb_ns_fused in both modes (dC rows bit-identical to the three kernels; vector reductions against float64),
    kgeb_ns_bwd_q and kgeb_ns_cand_grad."""
    b, m, d = shape
    kind = KINDS[kname]
    lname, loss, offset = lcase
    lib = kb.lib
    seed = 1000 * SHAPES.index(shape) + 10 * kind + loss
    q, table, target, neg = pair_problem(b, m, d, kind, seed)
    e = table.shape[0]
    inv_b = 1.0 / b
    cand = torch.empty(b, m, dtype=torch.int64, device="cuda")
    lib.call("kgeb_ns_candidates", target.data_ptr(), neg.data_ptr(), b, m - 1, cand.data_ptr(), st())
    assert torch.equal(cand, torch.cat((target[:, None], neg), 1))
    # int32 candidate indexes for pairs_score / pairs_bwd in one shape
    cidx = cand.int().contiguous() if shape == (37, 1001, 64) else cand
    c64 = int(cidx.dtype == torch.int64)

    # ---- three-kernel slot ----
    scores = torch.empty(b, m, device="cuda")
    lib.call("kgeb_pairs_score", kind, q.data_ptr(), table.data_ptr(), cidx.data_ptr(), c64, b, m, d, scores.data_ptr(), st())
    s_ref = pr.pair_scores(kind, q, table, cand)
    s_bound = pr.pair_score_bound(kind, q, table, cand)
    check(scores, s_ref, s_bound, f"pairs_score {kname}")

    G, rows = ns_loss_call(kb, loss, scores, offset, inv_b)
    r_ref, g_ref = pr.ns_rows_and_grad(loss, scores, offset, inv_b)
    r_b, g_b = pr.ns_loss_bound(loss, scores, offset, inv_b)
    check(rows, r_ref, r_b, f"ns_loss rows {lname}")
    check(G, g_ref, g_b, f"ns_loss G {lname}")

    dQ = torch.empty(b, d, device="cuda")
    dC = torch.empty(b * m, d, device="cuda")
    lib.call("kgeb_pairs_bwd", kind, q.data_ptr(), table.data_ptr(), cidx.data_ptr(), c64, b, m, d, G.data_ptr(),
             scores.data_ptr(), dQ.data_ptr(), dC.data_ptr(), st())
    dq_ref, dc_ref = pr.pair_grads(kind, q, table, cand, G)
    at3, et3, ac3, ec3 = pr.pair_grad_terms_bound(kind, q, table, cand, G, 0.0, s_bound)
    check(dQ, dq_ref, pr.dq_bound(at3, et3), f"pairs_bwd dQ {kname}")
    check(dC.view(b, m, d), dc_ref, ec3, f"pairs_bwd dC {kname}")
    prefill = torch.randn(e, d, device="cuda")
    dense = scatter(kb, cand.view(-1), dC, e, prefill.clone())
    check(dense, pr.index_add(cand, dC, e, prefill),
          pr.scatter_bound(cand, dC.abs(), e, pr.sorted_scatter_chain, prefill=prefill, atomic_adds=pr.one_add), "scatter of dC")

    # ---- the fused slot ----
    assert (8 * d + 2 * m) * 4 <= 48 * 1024, "every shape here fits ns_fused's shared memory"
    dQf, rowsf = torch.empty_like(dQ), torch.empty_like(rows)
    dCf = torch.full_like(dC, float("nan"))
    if d % 4:
        with pytest.raises(ValueError, match="multiple of 4"):
            lib.call("kgeb_ns_fused", kind, loss, q.data_ptr(), table.data_ptr(), cand.data_ptr(), b, m, d, offset, inv_b,
                     dQf.data_ptr(), dCf.data_ptr(), None, rowsf.data_ptr(), st())
    else:
        lib.call("kgeb_ns_fused", kind, loss, q.data_ptr(), table.data_ptr(), cand.data_ptr(), b, m, d, offset, inv_b,
                 dQf.data_ptr(), dCf.data_ptr(), None, rowsf.data_ptr(), st())
        assert torch.equal(rowsf, rows) and torch.equal(dQf, dQ) and torch.equal(dCf, dC), "ns_fused != three kernels"
        # vector reductions into a dense gradient, against the float64 slot computed from Q and the table alone
        dense = torch.zeros(e, d, device="cuda")
        lib.call("kgeb_ns_fused", kind, loss, q.data_ptr(), table.data_ptr(), cand.data_ptr(), b, m, d, offset, inv_b,
                 dQf.data_ptr(), None, dense.data_ptr(), rowsf.data_ptr(), st())
        r64, g64 = pr.ns_rows_and_grad(loss, s_ref, offset, inv_b)
        rb64, gb64 = pr.ns_loss_bound(loss, s_ref, offset, inv_b, s_bound)
        check(rowsf, r64, rb64, f"ns_fused rows {lname}")
        dq64, dc64 = pr.pair_grads(kind, q, table, cand, g64)
        at, et, ac, ec = pr.pair_grad_terms_bound(kind, q, table, cand, g64, gb64, s_bound)
        check(dQf, dq64, pr.dq_bound(at, et), f"ns_fused dQ {kname}")
        check(dense, pr.index_add(cand, dc64, e),
              pr.scatter_bound(cand, ac, e, pr.sequential_chain, err_rows=ec, atomic_adds=lambda n: n), f"ns_fused dense {kname}")

    # ---- segment backward: dQ without dC, candidate gradients one warp per distinct candidate ----
    dQs = torch.empty_like(dQ)
    lib.call("kgeb_ns_bwd_q", kind, q.data_ptr(), table.data_ptr(), cand.data_ptr(), b, m, d, G.data_ptr(),
             scores.data_ptr(), dQs.data_ptr(), st())
    check(dQs, dq_ref, pr.dq_bound(at3, et3), f"ns_bwd_q {kname}")
    segws = torch.empty(lib.load().kgeb_ns_segment_workspace_bytes(b * m), dtype=torch.uint8, device="cuda")
    dense = prefill.clone()
    args = (kind, q.data_ptr(), table.data_ptr(), cand.data_ptr(), b, m, d, G.data_ptr(), scores.data_ptr(), e,
            dense.data_ptr(), segws.data_ptr(), segws.numel(), st())
    if d > 256:
        with pytest.raises(ValueError, match="too large"):
            lib.call("kgeb_ns_cand_grad", *args)
        return
    lib.call("kgeb_ns_cand_grad", *args)
    check(dense, pr.index_add(cand, dc_ref, e, prefill),
          pr.scatter_bound(cand, ac3, e, pr.sequential_chain, err_rows=ec3, prefill=prefill), f"ns_cand_grad {kname}")


@pytest.mark.parametrize("lname,loss,offset", LOSSES, ids=[x[0] for x in LOSSES])
def test_ns_loss_on_constructed_rows(kb, lname, loss, offset):
    """Rows whose scores all sit at 0, -30, -120 or +80 (KL: uniform softmax at any shift; BCE: saturated softplus and
    sigmoid), and BCE rows at z = +-40 -- 300 columns, so every lane handles ten."""
    m = 300
    levels = torch.tensor([0.0, -30.0, -120.0, 80.0, 40.0 - offset, -40.0 - offset], device="cuda")
    x = levels[:, None].expand(-1, m).contiguous()
    x2 = torch.randn(6, m, device="cuda") * 3 + levels[:, None]          # the same levels, spread
    x = torch.cat((x, x2)).contiguous()
    G, rows = ns_loss_call(kb, loss, x, offset, 1.0 / 12)
    r_ref, g_ref = pr.ns_rows_and_grad(loss, x, offset, 1.0 / 12)
    r_b, g_b = pr.ns_loss_bound(loss, x, offset, 1.0 / 12)
    check(rows, r_ref, r_b, f"ns_loss rows {lname}")
    check(G, g_ref, g_b, f"ns_loss G {lname}")


# ---------------------------------------------------------------------------------------------------------------------
# row scorers
# ---------------------------------------------------------------------------------------------------------------------
ROW_CASES = [(m, d, l) for m in ("distmult", "complex", "cp", "simple", "transe", "rotate") for d in (16, 102, 256, 512)
             for l in ((1, 2) if m in ("transe", "rotate") else (1,))] + [("rescal", d, 1) for d in (16, 48, 128)]
N_ROWS = (1, 37, 20000)


def row_tables(model, d, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    e, r = 1000, 11
    ent = torch.randn(e, d, generator=g, device="cuda") * 0.5
    dr = ko.relation_dim(model, d)
    if model == "rotate":
        rel = (torch.rand(r, dr, generator=g, device="cuda") * 2 - 1) * 50      # phases far outside [-pi, pi]
    elif model == "rescal":
        rel = torch.randn(r, dr, generator=g, device="cuda") / d ** 0.5
    else:
        rel = torch.randn(r, dr, generator=g, device="cuda") * 0.5
    return ent, rel, g


@pytest.mark.parametrize("model,d,l_norm", ROW_CASES, ids=[f"{m}-d{d}-l{l}" for m, d, l in ROW_CASES])
def test_row_scorers_against_float64(kb, model, d, l_norm):
    """kgeb_query_build / kgeb_query_bwd (sp_, _po, per-row row_combine) and kgeb_score_spo / kgeb_score_spo_bwd at
    n = 1, 37 (int32 indexes) and 20,000 rows (int64, past the grid's 18,944 warps), indexes with repeats."""
    lib = kb.lib
    mid = lib.MODELS[model]
    ent, rel, g = row_tables(model, d, seed=ROW_CASES.index((model, d, l_norm)))
    h = d // 2
    dr = rel.shape[1]
    for n in N_ROWS:
        dt = torch.int32 if n == 37 else torch.int64
        a_idx = torch.randint(0, ent.shape[0], (n,), generator=g, device="cuda").to(dt)
        p_idx = torch.randint(0, rel.shape[0], (n,), generator=g, device="cuda").to(dt)
        o_idx = torch.randint(0, ent.shape[0], (n,), generator=g, device="cuda").to(dt)
        i64 = int(dt == torch.int64)
        a, p, o = ent[a_idx.long()], rel[p_idx.long()], ent[o_idx.long()]
        rc = torch.randint(0, 2, (n,), generator=g, device="cuda").int()
        for combine in (pr.SP_, pr._PO, rc):
            rcp = combine.data_ptr() if isinstance(combine, torch.Tensor) else None
            cflag = 0 if rcp else combine
            Q = torch.empty(n, d, device="cuda")
            lib.call("kgeb_query_build", mid, cflag, rcp, ent.data_ptr(), a_idx.data_ptr(), rel.data_ptr(), p_idx.data_ptr(),
                     i64, n, d, Q.data_ptr(), st())
            what = f"{model} d={d} n={n} combine={'rows' if rcp else combine}"
            check(Q, pr.query(model, combine, a, p), pr.query_bound(model, combine, a, p), f"query_build {what}")
            dQ = torch.randn(n, d, generator=g, device="cuda")
            da, dp = torch.empty(n, d, device="cuda"), torch.empty(n, dr, device="cuda")
            lib.call("kgeb_query_bwd", mid, cflag, rcp, ent.data_ptr(), a_idx.data_ptr(), rel.data_ptr(), p_idx.data_ptr(),
                     i64, n, d, dQ.data_ptr(), da.data_ptr(), dp.data_ptr(), st())
            da_ref, dp_ref = pr.query_grads(model, combine, a, p, dQ)
            da_b, dp_b = pr.query_grads_bound(model, combine, a, p, dQ)
            check(da, da_ref, da_b, f"query_bwd da {what}")
            check(dp, dp_ref, dp_b, f"query_bwd dp {what}")
        out = torch.empty(n, device="cuda")
        lib.call("kgeb_score_spo", mid, l_norm, ent.data_ptr(), a_idx.data_ptr(), rel.data_ptr(), p_idx.data_ptr(),
                 ent.data_ptr(), o_idx.data_ptr(), i64, n, d, out.data_ptr(), st())
        want = ko.score_emb(model, a.double(), p.double(), o.double(), "spo", l_norm).view(-1)
        check(out, want, pr.spo_bound(model, a, p, o, l_norm), f"score_spo {model} d={d} n={n} l{l_norm}")
        gout = torch.randn(n, generator=g, device="cuda")
        ds, dp, do = torch.empty(n, d, device="cuda"), torch.empty(n, dr, device="cuda"), torch.empty(n, d, device="cuda")
        lib.call("kgeb_score_spo_bwd", mid, l_norm, ent.data_ptr(), a_idx.data_ptr(), rel.data_ptr(), p_idx.data_ptr(),
                 ent.data_ptr(), o_idx.data_ptr(), i64, n, d, gout.data_ptr(), ds.data_ptr(), dp.data_ptr(), do.data_ptr(),
                 st())
        refs = pr.spo_grads(model, a, p, o, gout, l_norm)
        bounds = pr.spo_grad_bound(model, a, p, o, gout, l_norm)
        for got, ref, bnd, nm in zip((ds, dp, do), refs, bounds, ("ds", "dp", "do")):
            check(got, ref.reshape(got.shape), bnd.reshape(got.shape), f"score_spo_bwd {nm} {model} d={d} n={n} l{l_norm}")


# ---------------------------------------------------------------------------------------------------------------------
# the sorted scatter
# ---------------------------------------------------------------------------------------------------------------------
def run_ids(n, vocab, g):
    """n ids whose sorted order has runs of 1, 7, 8, 9 and many chunks, starting and ending on 8-row chunk boundaries
    and off them, then random runs; positions shuffled (the sort restores id order, positions ascending in a run)."""
    head = torch.tensor([8, 8, 1, 7, 9, 7, 1, 16, 24, 1000, 1, 8, 9, 3, 5, 8 * 40, 2, 1, 1, 1, 1, 1, 1, 1, 8],
                        device="cuda")
    rest = n - int(head.sum())
    avg = -(-rest // (vocab - head.numel()))
    tail = torch.randint(avg, 2 * avg + 1, (rest // avg + 1,), generator=g, device="cuda")   # <= 2/3 of the ids left
    k = int(torch.searchsorted(tail.cumsum(0), rest)) + 1
    tail = tail[:k]
    tail[-1] -= int(tail.sum()) - rest
    lengths = torch.cat((head, tail))
    assert int(lengths.sum()) == n and int(lengths.min()) >= 1 and lengths.numel() <= vocab
    ids_in_order = torch.randperm(vocab, generator=g, device="cuda")[: lengths.numel()].sort().values
    ids = torch.repeat_interleave(ids_in_order, lengths)
    return ids[torch.randperm(n, generator=g, device="cuda")].contiguous()


# (n, vocab, d): one block (n <= 8192, id + position bits <= 32); 32-bit multi-block; 64-bit words; the segment regime
# (n > 2^26) at d = 4
SCATTER = [(5000, 97, 33), (20000, 1000, 64), (131584, E_WN, 128), ((1 << 26) + 1000, 100000, 4)]


@pytest.mark.parametrize("n,vocab,d", SCATTER, ids=["one_block", "packed32", "packed64", "segment"])
def test_scatter_add_rows_against_index_add(kb, n, vocab, d):
    g = torch.Generator(device="cuda").manual_seed(n % 1000)
    ids = run_ids(n, vocab, g)
    rows = torch.randn(n, d, generator=g, device="cuda")
    prefill = torch.randn(vocab, d, generator=g, device="cuda")
    for idx in ((ids.int(), ids) if n < (1 << 26) else (ids,)):
        dense = scatter(kb, idx.contiguous(), rows, vocab, prefill.clone())
        check(dense, pr.index_add(ids, rows, vocab, prefill),
              pr.scatter_bound(ids, rows.abs(), vocab, pr.sorted_scatter_chain, prefill=prefill, atomic_adds=pr.one_add),
              f"scatter n={n} {idx.dtype}")


def test_segment_reduce_rows_on_hub_heavy_ids(kb):
    """kgeb_segment_reduce_rows: sorted distinct ids and one summed row each, on ids where one hub holds 30 % of 100,000
    rows and a second one 5 %."""
    g = torch.Generator(device="cuda").manual_seed(5)
    n, vocab, d = 100000, 5000, 64
    ids = torch.randint(0, vocab, (n,), generator=g, device="cuda")
    u = torch.rand(n, generator=g, device="cuda")
    ids[u < 0.3] = 11
    ids[(u >= 0.3) & (u < 0.35)] = vocab - 1
    rows = torch.randn(n, d, generator=g, device="cuda")
    ws = workspace(kb, n, d)
    uniq = torch.empty(n, dtype=torch.int64, device="cuda")
    out = torch.empty(n, d, device="cuda")
    nu = torch.empty(1, dtype=torch.int64, device="cuda")
    kb.lib.call("kgeb_segment_reduce_rows", ids.data_ptr(), 1, rows.data_ptr(), n, d, uniq.data_ptr(), out.data_ptr(),
                nu.data_ptr(), ws.data_ptr(), ws.numel(), st())
    want_ids = torch.unique(ids)
    k = int(nu)
    assert k == want_ids.numel()
    assert torch.equal(uniq[:k], want_ids)
    full = pr.index_add(ids, rows, vocab)
    bound = pr.scatter_bound(ids, rows.abs(), vocab, pr.sorted_scatter_chain, atomic_adds=pr.one_add)
    check(out[:k], full[want_ids], bound[want_ids], "segment_reduce_rows")


# ---------------------------------------------------------------------------------------------------------------------
# the captured step end to end
# ---------------------------------------------------------------------------------------------------------------------
R_WN, B_STEP, N_STEP, LR, ACC0 = 11, 512, 256, 0.1, 0.1
# (model, l_norm, d, loss, stepper options): RotatE L1 KL under the default options, the vector reductions and the
# segment backward; RotatE L2 BCE at d = 102 (the three-kernel slot); TransE both norms; ComplEx, DistMult, RESCAL
STEP_CASES = [("rotate", 1, 128, "kl", {}), ("rotate", 1, 128, "kl", {"deterministic": False}),
              ("rotate", 1, 128, "kl", {"segment_bwd": True}), ("rotate", 2, 102, "bce", {}),
              ("transe", 1, 128, "bce", {}), ("transe", 2, 128, "kl", {}), ("complex", 1, 128, "kl", {}),
              ("distmult", 1, 128, "bce", {}), ("rescal", 1, 32, "kl", {})]


def step_reference(model, kind, loss, W, Rw, triples, negs):
    """The float64 restatement of one FusedNegSamplingStepper step and its bounds, slot S (_po query (p, o) against
    subject candidates) and slot O (sp_ query (s, p) against object candidates):
      Q = query(a, p) with query_bound; scores with pair_score_bound carrying Q's error; loss rows / B and G with
      ns_loss_bound carrying the scores' error; dQ / dC with pair_grad_terms_bound carrying G's, the scores' and Q's
      errors; da / dp = query_bwd(dQ) with query_grads_bound carrying dQ's error.
    The entity gradient is four scatters into one buffer (per slot the candidates' rows, then the query-side rows): a
    term passes through at most L_i + 3 roundings in its own scatter (sorted: min(L, 8) + ceil(L/8) + 2; sequential
    orders: L + 1) and one more per later scatter onto its row, so chain <= L + 12 with L the rows added to that entity
    row in the step, plus FLUSH per float atomic (at most L + 4).  The relation gradient: two sorted scatters, L + 6."""
    s, p, o = (triples[:, i] for i in range(3))
    out = {"slots": {}}
    ent = dict(ref=torch.zeros(W.shape, dtype=torch.float64, device="cuda"), abs=0, err=0, n=0)
    rel = dict(ref=torch.zeros(Rw.shape, dtype=torch.float64, device="cuda"), abs=0, err=0, n=0)
    E, Rn = W.shape[0], Rw.shape[0]
    for slot, combine, a_idx, target in ((0, pr._PO, o, s), (2, pr.SP_, s, o)):
        cand = torch.cat((target[:, None], negs[slot]), 1)
        a_rows, p_rows = W[a_idx], Rw[p]
        q64, dq = pr.query(model, combine, a_rows, p_rows), pr.query_bound(model, combine, a_rows, p_rows)
        s64 = pr.pair_scores(kind, q64, W, cand)
        ds = pr.pair_score_bound(kind, q64, W, cand, dq)
        rows64, g64 = pr.ns_rows_and_grad(loss, s64, 0.0, 1.0 / B_STEP)
        rb, gb = pr.ns_loss_bound(loss, s64, 0.0, 1.0 / B_STEP, ds)
        dq64, dc64 = pr.pair_grads(kind, q64, W, cand, g64)
        at, et, ac, ec = pr.pair_grad_terms_bound(kind, q64, W, cand, g64, gb, ds, dq)
        dqb = pr.dq_bound(at, et)
        da64, dp64 = pr.query_grads(model, combine, a_rows, p_rows, dq64)
        dab, dpb = pr.query_grads_bound(model, combine, a_rows, p_rows, dq64, dqb)
        out["slots"][slot] = dict(Q=(q64, dq), scores=(s64, ds), rows=(rows64, rb))
        ent["ref"] += pr.index_add(cand, dc64, E) + pr.index_add(a_idx, da64, E)
        ent["abs"] = ent["abs"] + pr.index_add(cand, ac, E) + pr.index_add(a_idx, da64.abs(), E)
        ent["err"] = ent["err"] + pr.index_add(cand, ec, E) + pr.index_add(a_idx, dab, E)
        ent["n"] = ent["n"] + pr.run_lengths(cand, E) + pr.run_lengths(a_idx, E)
        rel["ref"] += pr.index_add(p, dp64, Rn)
        rel["abs"] = rel["abs"] + pr.index_add(p, dp64.abs(), Rn)
        rel["err"] = rel["err"] + pr.index_add(p, dpb, Rn)
        rel["n"] = rel["n"] + pr.run_lengths(p, Rn)
    ln = ent["n"].double()[:, None]
    out["g_ent"] = (ent["ref"], ent["err"] + (ln + 12) * pr.U * ent["abs"] + (ln + 4) * pr.FLUSH)
    out["g_rel"] = (rel["ref"], rel["err"] + (rel["n"].double()[:, None] + 6) * pr.U * rel["abs"] + 2 * pr.FLUSH)
    rows = torch.cat([out["slots"][k]["rows"][0] for k in (0, 2)])
    rbs = torch.cat([out["slots"][k]["rows"][1] for k in (0, 2)])
    # torch.sum of B rows per slot (any order: at most B - 1 roundings), then the two slot sums (1)
    out["loss"] = (rows.sum(), rbs.sum() + B_STEP * pr.U * rows.abs().sum())
    return out


@pytest.mark.parametrize("model,l_norm,d,lname,opts", STEP_CASES,
                         ids=[f"{m}-l{l}-d{d}-{ls}" + "".join(f"-{k}" for k in o) for m, l, d, ls, o in STEP_CASES])
def test_captured_negative_sampling_step_against_float64(kb, model, l_norm, d, lname, opts):
    """One FusedNegSamplingStepper step (CUDA graph) at the WN18RR shape -- E = 40,943, R = 11, B = 512, 256 negatives
    per slot -- with Adagrad (initial accumulator 0.1): Q, the scores of the three-kernel slots, the loss rows / B, the
    returned loss, g_ent / g_rel (this step's gradient after the replay), W and the Adagrad state against step_reference
    and adagrad_bound (the gradient bound carried through the update with the accumulator floor 0.1)."""
    torch.manual_seed(0)
    g = torch.Generator(device="cuda").manual_seed(STEP_CASES.index((model, l_norm, d, lname, opts)))
    m = kb.KgeModel(model, E_WN, R_WN, d, l_norm=float(l_norm)).cuda()
    ent, rel = m.get_s_embedder().weight, m.get_p_embedder().weight
    with torch.no_grad():
        ent.copy_(torch.randn(ent.shape, generator=g, device="cuda") * 0.5)
        if model == "rotate":
            rel.copy_((torch.rand(rel.shape, generator=g, device="cuda") * 2 - 1) * 50)
        else:
            rel.copy_(torch.randn(rel.shape, generator=g, device="cuda") / (d ** 0.5 if model == "rescal" else 2))
    W0, R0 = ent.detach().clone(), rel.detach().clone()
    opt = kb.optim.create("Adagrad", m.parameters(), lr=LR, initial_accumulator_value=ACC0)
    loss = kb.lib.LOSS_KL if lname == "kl" else kb.lib.LOSS_BCE
    st_ = kb.trainer.FusedNegSamplingStepper(m, opt, B_STEP, N_STEP, N_STEP, loss, **opts)
    assert st_.fused_slot == (d % 4 == 0 and not opts.get("segment_bwd", False))
    triples = torch.stack((torch.randint(0, E_WN, (B_STEP,), generator=g, device="cuda"),
                           torch.randint(0, R_WN, (B_STEP,), generator=g, device="cuda"),
                           torch.randint(0, E_WN, (B_STEP,), generator=g, device="cuda")), 1)
    negs = {}
    for slot in (0, 2):
        n = torch.randint(0, E_WN, (B_STEP, N_STEP), generator=g, device="cuda")
        n[torch.rand(B_STEP, N_STEP, generator=g, device="cuda") < 0.05] = HUB
        negs[slot] = n
    st_.set_inputs(triples, [negs[0], None, negs[2]])
    got_loss = st_.step()
    torch.cuda.synchronize()
    ref = step_reference(model, st_.kind, loss, W0, R0, triples, negs)
    what = f"{model} l{l_norm} d={d} {lname} {opts}"
    for slot in (0, 2):
        b = st_.buf[slot]
        r = ref["slots"][slot]
        check(b["Q"], *r["Q"], f"step Q slot {slot} {what}")
        if not st_.fused_slot:
            check(b["scores"], *r["scores"], f"step scores slot {slot} {what}")
        check(b["rows"], *r["rows"], f"step loss rows slot {slot} {what}")
    check(got_loss.view(1), ref["loss"][0].view(1), ref["loss"][1].view(1), f"step loss {what}")
    ge, geb = ref["g_ent"]
    gr, grb = ref["g_rel"]
    check(st_.g_ent, ge, geb, f"step g_ent {what}")
    check(st_.g_rel, gr, grb, f"step g_rel {what}")
    eps = float(opt.param_groups[0]["eps"])
    for w, w0, s_, gref, gbound, nm in ((ent, W0, opt.state[ent]["sum"], ge, geb, "entities"),
                                        (rel, R0, opt.state[rel]["sum"], gr, grb, "relations")):
        s0 = torch.full_like(w0, ACC0)
        w_ref, s_ref = pr.adagrad(w0, s0, gref, LR, eps)
        dw, ds_ = pr.adagrad_bound(w0, s0, gref, gbound, LR, eps)
        check(w.detach(), w_ref, dw, f"step W {nm} {what}")
        check(s_, s_ref, ds_, f"step Adagrad state {nm} {what}")
