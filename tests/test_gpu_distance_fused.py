"""Fused all-entity KL / BCE training of TransE and RotatE on the fp32 CUDA-core distance tiles (kgeb_fused_fwd_kind /
kgeb_fused_bwd_kind): kernels against a float64 torch restatement and against the materialised fp32 path, the golden
reference steps routed through the fused kernels, the captured step against the autograd flow, and the memory of a
step that never writes the [B, E] score matrix.  Needs a B200: `pytest -m gpu`."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

T = torch.from_numpy


@pytest.fixture(scope="module")
def kb():
    import kgeb200
    assert torch.cuda.is_available(), "these tests need a GPU"
    kgeb200.lib.load()
    return kgeb200


def close(got, ref, rtol, what=""):
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    assert got.shape == ref.shape, f"{what}: shape {tuple(got.shape)} vs {tuple(ref.shape)}"
    if ref.numel() == 0:
        return
    scale = max(ref.abs().max().item(), 1e-30)
    err = (got - ref).abs().max().item()
    assert err <= rtol * scale, f"{what}: max abs err {err:.3e} > {rtol:g} * {scale:.3e}"


def kinds(kb):
    return {"transe_l1": kb.lib.NEG_L1, "transe_l2": kb.lib.NEG_L2, "rotate_l1": kb.lib.ROT_L1, "rotate_l2": kb.lib.ROT_L2}


def ref_scores(kb, kind, q, w):
    """float64 scores of kgeb_score_all: TransE -distance, RotatE +distance (L1 of RotatE: sum of complex moduli)."""
    diff = q[:, None, :] - w[None, :, :]
    if kind == kb.lib.NEG_L1:
        return -diff.abs().sum(-1)
    if kind == kb.lib.ROT_L1:
        h = q.shape[1] // 2
        return (diff[..., :h] ** 2 + diff[..., h:] ** 2).sqrt().sum(-1)
    dist = (diff ** 2).sum(-1).sqrt()
    return -dist if kind == kb.lib.NEG_L2 else dist


def ref_rows(x, y, loss_kl, ls, offset, num_entities):
    """Per-row loss of the reference's losses (loss.py:137-159, 192-213) on scores x and label counts y; label smoothing
    is the reference's (1 - ls) * y + 1 / E (train.py:715-721)."""
    if loss_kl:
        t = y / y.sum(1, keepdim=True)
        return -(t * F.log_softmax(x, 1)).sum(1) + torch.where(t > 0, t * t.log(), torch.zeros_like(t)).sum(1)
    t = (1.0 - ls) * y + (1.0 / num_entities if ls > 0 else 0.0)
    return F.binary_cross_entropy_with_logits(x + offset, t, reduction="none").sum(1)


def make_labels(b, e_lo, e_hi, gen, onehot, empty_rows):
    """CSR (offsets, ascending global columns in [e_lo, e_hi)) of one label per row (1vsAll) or up to 4 (KvsAll);
    `empty_rows`: every fifth row has no label."""
    n_ent = e_hi - e_lo
    cols = []
    for r in range(b):
        if empty_rows and r % 5 == 2:
            k = 0
        else:
            k = 1 if onehot else int(torch.randint(1, 5, (1,), generator=gen))
        k = min(k, n_ent)
        cols.append(torch.randperm(n_ent, generator=gen)[:k].sort().values + e_lo)
    off = torch.zeros(b + 1, dtype=torch.int64)
    off[1:] = torch.cumsum(torch.tensor([len(c) for c in cols]), 0)
    return off.cuda(), torch.cat(cols).long().cuda()


def dense_labels(off, col, b, e_lo, e_hi):
    y = torch.zeros(b, e_hi - e_lo, dtype=torch.float64, device=off.device)
    rows = torch.repeat_interleave(torch.arange(b, device=off.device), off[1:] - off[:-1])
    y[rows, col - e_lo] = 1.0
    return y


def reference(kb, kind, q, w, y, loss_kl, ls, offset, num_entities, rscale, chunk=None):
    """Per-row loss, dQ and dTable in float64 through autograd, in row chunks (bounded [rows, E, d] intermediates)."""
    b, e, d = q.shape[0], w.shape[0], q.shape[1]
    chunk = chunk or max(1, min(b, (1 << 27) // max(1, e * d)))
    qd = q.double().requires_grad_(True)
    wd = w.double().requires_grad_(True)
    rows = []
    for i in range(0, b, chunk):
        x = ref_scores(kb, kind, qd[i:i + chunk], wd)
        r = ref_rows(x, y[i:i + chunk], loss_kl, ls, offset, num_entities)
        (r * rscale[i:i + chunk].double()).sum().div(b).backward()
        rows.append(r.detach())
    return torch.cat(rows), qd.grad, wd.grad


def fused(kb, kind, q, w, off, col, loss, ls, offset, shard, rscale):
    st = kb.fused.fused_rowstats(q, w, off, col, loss, ls, offset, kb.lib.MATH_FP32, shard, kind=kind)
    rows, lse = kb.fused.rows_loss(st, off, loss, ls, shard.num_entities)
    dw = torch.full_like(w, float("nan"))
    dq = kb.fused.fused_backward(q, w, off, col, loss, ls, offset, lse, 1.0 / q.shape[0], rscale, kb.lib.MATH_FP32,
                                 shard, dw, overwrite=True, kind=kind)
    return rows, dq, dw


# (B, E, d, e_lo, e_hi): every B, E and d value of the issue, one sub-range of the table
SHAPES = [(1, 65, 6, 0, 65), (63, 1, 100, 0, 1), (130, 14541, 128, 0, 14541), (2048, 65, 256, 0, 65),
          (63, 14541, 2, 0, 14541), (130, 65, 256, 0, 65), (2048, 14541, 128, 0, 14541), (130, 14541, 100, 4000, 9001)]
LOSSES = [("kl", 0.0, 0.0), ("bce", 0.5, 0.0), ("bce", 0.0, 0.1)]     # (loss, offset, label smoothing)


@pytest.mark.parametrize("tag", ["transe_l1", "transe_l2", "rotate_l1", "rotate_l2"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_fused_kernels_match_float64(kb, tag, shape):
    b, e, d, e_lo, e_hi = shape
    kind = kinds(kb)[tag]
    if tag.startswith("rotate") and d % 2:
        pytest.skip("RotatE needs an even dimension")
    gen = torch.Generator().manual_seed(b * 7 + e + d)
    q = (torch.randn(b, d, generator=gen) * 0.3).cuda()
    w_full = (torch.randn(e, d, generator=gen) * 0.3).cuda()
    w = w_full[e_lo:e_hi].contiguous()
    rscale = (torch.rand(b, generator=gen) + 0.5).cuda()
    shard = kb.fused.Shard(e_lo, e_hi, e)
    for name, offset, ls in LOSSES:
        loss = kb.lib.LOSS_KL if name == "kl" else kb.lib.LOSS_BCE
        for onehot in (True, False):
            # a KL row without labels follows the deviation of DESIGN 2 (loss 0, no gradient): BCE only
            off, col = make_labels(b, e_lo, e_hi, gen, onehot, empty_rows=(loss == kb.lib.LOSS_BCE))
            y = dense_labels(off, col, b, e_lo, e_hi)
            rows, dq, dw = fused(kb, kind, q, w, off, col, loss, ls, offset, shard, rscale)
            want_rows, want_dq, want_dw = reference(kb, kind, q, w, y, loss == kb.lib.LOSS_KL, ls, offset, e, rscale)
            what = f"{tag} {name} off={offset} ls={ls} onehot={onehot} {shape}"
            # BCE with label smoothing gives every entry the same-signed dense part 1/E: at 14,541 entities one fp32
            # accumulator of dQ sums ~1,500 terms that do not cancel, and its rounding grows to ~3e-5 of the result
            gtol = 5e-5 if (ls > 0 and e_hi - e_lo > 4096) else 2e-5
            close(rows, want_rows, 1e-5, "rows " + what)
            close(dq, want_dq, gtol, "dQ " + what)
            close(dw, want_dw, gtol, "dTable " + what)


def materialised(kb, kind, q, w, off, col, loss, ls, offset, rscale):
    """kgeb_score_all + torch's loss + kgeb_score_all_bwd, fp32."""
    qd, wd = q.clone().requires_grad_(True), w.clone().requires_grad_(True)
    x = kb.ops.score_all(kind, qd, wd, kb.lib.MATH_FP32)
    y = dense_labels(off, col, q.shape[0], 0, w.shape[0]).float()
    rows = ref_rows(x, y, loss == kb.lib.LOSS_KL, ls, offset, w.shape[0])
    (rows * rscale).sum().div(q.shape[0]).backward()
    return rows.detach(), qd.grad, wd.grad


@pytest.mark.parametrize("tag", ["transe_l1", "transe_l2", "rotate_l1", "rotate_l2"])
@pytest.mark.parametrize("duplicates", [False, True])
def test_fused_kernels_match_materialised_path(kb, tag, duplicates):
    kind = kinds(kb)[tag]
    b, e, d = 130, 1000, 64
    gen = torch.Generator().manual_seed(11)
    q = (torch.randn(b, d, generator=gen) * 0.3).cuda()
    w = (torch.randn(e, d, generator=gen) * 0.3).cuda()
    if duplicates:    # exact copies of query rows: zero distances, zero-gradient convention of kgeb_score_all_bwd
        dup = torch.arange(0, e, 7, device="cuda")[:b]
        w[dup] = q[: len(dup)]
    rscale = (torch.rand(b, generator=gen) + 0.5).cuda()
    shard = kb.fused.Shard.full(e)
    for name, offset, ls in LOSSES:
        loss = kb.lib.LOSS_KL if name == "kl" else kb.lib.LOSS_BCE
        off, col = make_labels(b, 0, e, gen, onehot=False, empty_rows=False)
        rows, dq, dw = fused(kb, kind, q, w, off, col, loss, ls, offset, shard, rscale)
        want_rows, want_dq, want_dw = materialised(kb, kind, q, w, off, col, loss, ls, offset, rscale)
        what = f"{tag} {name} ls={ls} duplicates={duplicates}"
        assert torch.isfinite(dq).all() and torch.isfinite(dw).all(), what
        close(rows, want_rows, 1e-5, "rows " + what)
        close(dq, want_dq, 2e-5, "dQ " + what)
        close(dw, want_dw, 2e-5, "dTable " + what)


def test_kind_entries_refuse_what_check_fused_refuses(kb):
    q = torch.zeros(4, 6, device="cuda")
    w = torch.zeros(10, 6, device="cuda")
    off = torch.arange(5, dtype=torch.int64, device="cuda")
    col = torch.zeros(4, dtype=torch.int64, device="cuda")
    shard = kb.fused.Shard.full(10)
    with pytest.raises(NotImplementedError):        # KL with label smoothing
        kb.fused.fused_rowstats(q, w, off, col, kb.lib.LOSS_KL, 0.1, 0.0, kb.lib.MATH_FP32, shard, kind=kb.lib.NEG_L1)
    big_q, big_w = torch.zeros(4, 258, device="cuda"), torch.zeros(10, 258, device="cuda")
    with pytest.raises(NotImplementedError):        # d > 256
        kb.fused.fused_rowstats(big_q, big_w, off, col, kb.lib.LOSS_BCE, 0.0, 0.0, kb.lib.MATH_FP32, shard,
                                kind=kb.lib.ROT_L1)
    odd_q, odd_w = torch.zeros(4, 5, device="cuda"), torch.zeros(10, 5, device="cuda")
    with pytest.raises(ValueError):                 # RotatE with an odd dimension
        kb.fused.fused_rowstats(odd_q, odd_w, off, col, kb.lib.LOSS_BCE, 0.0, 0.0, kb.lib.MATH_FP32, shard,
                                kind=kb.lib.ROT_L2)


@pytest.mark.parametrize("case", ["train.1vsAll.transe.kl", "train.KvsAll.rotate.kl"])
def test_golden_distance_cases_run_the_fused_kernels(kb, golden, case, monkeypatch):
    """The reference's own steps of these golden cases, through the fused flow: they reach kgeb_fused_fwd_kind /
    kgeb_fused_bwd_kind (not kgeb_score_all) and still match the golden loss, gradients and parameters."""
    import test_gpu_parity as parity
    assert case in [str(x) for x in golden("train")["train.cases"]]
    calls = []
    real_call = kb.lib.call
    monkeypatch.setattr(kb.lib, "call", lambda name, *a: (calls.append(name), real_call(name, *a))[1])
    parity._run_case(kb, golden, case, fused_path=True)
    assert "kgeb_fused_fwd_kind" in calls and "kgeb_fused_bwd_kind" in calls, case
    assert "kgeb_score_all" not in calls and "kgeb_score_all_bwd" not in calls, case


# ---------------------------------------------------------------------------------------------
# captured step
# ---------------------------------------------------------------------------------------------
def _kvsall_batches(kb, e, r, b, n, seed):
    from oracle import kge_oracle as ko
    g = kb.graph.synthetic_graph("toy", seed=seed)
    idx = [ko.kvsall_index(g["train"], "sp"), ko.kvsall_index(g["train"], "po")]
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        ids = rng.choice(len(idx[0][0]) + len(idx[1][0]), b, replace=False)
        qq, c, qt = ko.kvsall_collate(ids.tolist(), idx)
        out.append({"queries": T(qq), "label_coords": T(c), "query_type_indexes": T(qt)})
    return g, out


def _pair(kb, model, e, r, d, ln, reciprocal=False, penalty=False):
    reg = dict(entity_embedder=dict(regularize_weight=0.01, regularize_p=2),
               relation_embedder=dict(regularize_weight=0.003, regularize_p=2)) if penalty else {}
    cls = kb.model.ReciprocalRelationsModel if reciprocal else kb.KgeModel
    torch.manual_seed(0)
    ref = cls(model, e, r, d, l_norm=ln, **reg).cuda()
    new = cls(model, e, r, d, l_norm=ln, **reg).cuda()
    new.load_state_dict(ref.state_dict())
    return ref, new


def _sync(ref, new, opt_ref, opt_new):
    """Every step starts from the same tables and Adagrad state: Adagrad moves an entry by ~lr * sign(g) where its
    accumulated g^2 is tiny, and L1 / KL gradients have such entries (sums of +-G that cancel exactly in exact
    arithmetic), so a rounding difference between the two flows would otherwise flip them and compound over steps."""
    with torch.no_grad():
        for pr, pn in ((ref.get_s_embedder().weight, new.get_s_embedder().weight),
                       (ref.get_p_embedder().weight, new.get_p_embedder().weight)):
            pn.copy_(pr)
            opt_new.state[pn]["sum"].copy_(opt_ref.state[pr]["sum"])


def _compare(ref, new, opt_ref, opt_new, st, what, penalty):
    """This step's gradients (the stepper's buffers against the autograd flow's .grad; a folded penalty gradient is
    applied inside Adagrad and not in the buffers) and the Adagrad state it produced."""
    pairs = ((ref.get_s_embedder().weight, new.get_s_embedder().weight, "entity"),
             (ref.get_p_embedder().weight, new.get_p_embedder().weight, "relation"))
    if not penalty:
        close(st.g_ent + st.g_q, pairs[0][0].grad, 2e-5, f"entity gradient {what}")
        close(st.g_rel, pairs[1][0].grad, 2e-5, f"relation gradient {what}")
    for pr, pn, name in pairs:
        close(opt_new.state[pn]["sum"], opt_ref.state[pr]["sum"], 1e-5, f"{name} Adagrad state {what}")


CAPTURED = [(m, ln, loss, kind) for m in ("transe", "rotate") for ln in (1.0, 2.0) for loss in ("kl", "bce")
            for kind in ("1vsAll", "KvsAll")]


@pytest.mark.parametrize("use_graph", [False, True], ids=["eager", "graph"])
@pytest.mark.parametrize("case", CAPTURED, ids=lambda c: f"{c[0]}_l{int(c[1])}-{c[2]}-{c[3]}")
def test_captured_step_matches_fused_autograd_flow(kb, case, use_graph):
    model, ln, loss_name, ttype = case
    _run_captured(kb, model, ln, loss_name, ttype, use_graph)


@pytest.mark.parametrize("variant", ["reciprocal_rotate", "penalty_transe"])
def test_captured_step_reciprocal_and_penalty(kb, variant):
    if variant == "reciprocal_rotate":
        _run_captured(kb, "rotate", 1.0, "kl", "KvsAll", True, reciprocal=True)
        _run_captured(kb, "rotate", 1.0, "bce", "1vsAll", True, reciprocal=True)
    else:
        _run_captured(kb, "transe", 2.0, "bce", "KvsAll", True, penalty=True)


def _run_captured(kb, model, ln, loss_name, ttype, use_graph, reciprocal=False, penalty=False):
    d, b = 32, 64
    g, batches = _kvsall_batches(kb, 0, 0, b, 3, seed=3)
    e, r = g["num_entities"], g["num_relations"]
    ref, new = _pair(kb, model, e, r, d, ln, reciprocal, penalty)
    off = 0.25 if loss_name == "bce" else 0.0
    opt_ref = kb.optim.create("Adagrad", ref.parameters(), lr=0.2)
    opt_new = kb.optim.create("Adagrad", new.parameters(), lr=0.2)
    what = f"{model} l{ln} {loss_name} {ttype} graph={use_graph} reciprocal={reciprocal} penalty={penalty}"
    if ttype == "KvsAll":
        jr = kb.TrainingJobKvsAll(ref, opt_ref, kb.KgeLoss.create(loss_name, off), e, r)
        jn = kb.TrainingJobKvsAll(new, opt_new, kb.KgeLoss.create(loss_name, off), e, r)
        st = jn.enable_graph_step(b, max(len(x["label_coords"]) for x in batches), use_graph=use_graph)
        assert st.kind == kinds(kb)[f"{model}_l{int(ln)}"] and st.mirror is None and not st.flash
        for i, batch in enumerate(batches):
            _sync(ref, new, opt_ref, opt_new)
            a, c = jr.step(i, batch), jn.step(i, batch)
            assert c.total_loss == pytest.approx(a.total_loss, rel=1e-5), what
            assert c.avg_loss == pytest.approx(a.avg_loss, rel=1e-5), what
            _compare(ref, new, opt_ref, opt_new, st, f"{what} step {i}", penalty)
        return
    jr = kb.TrainingJob1vsAll(ref, opt_ref, kb.KgeLoss.create(loss_name, off))
    st = kb.trainer.FusedAllEntityStepper(new, opt_new, 2 * b, 2 * b, jr.loss.kind, b, off, 0.0, kb.lib.MATH_BF16,
                                          use_graph=use_graph, onevsall_triples=True, reciprocal=reciprocal)
    assert st.math == kb.lib.MATH_FP32 and st.mirror is None and not st.seq and not st.fuse_update and not st.flash
    rng = np.random.default_rng(5)
    train = g["train"]
    for i in range(3):
        triples = T(train[rng.choice(len(train), b, replace=False)]).long()
        _sync(ref, new, opt_ref, opt_new)
        a = jr.step(i, {"triples": triples})
        st.set_triples(triples.cuda())
        st.step()
        total, _ = st.report.tolist()
        assert total == pytest.approx(a.avg_loss, rel=1e-5), what
        _compare(ref, new, opt_ref, opt_new, st, f"{what} step {i}", penalty)


def test_one_step_at_a_million_entities_never_allocates_the_score_matrix(kb):
    """E = 1,000,000, 2,048 rows, d = 128: one [B, E] fp32 matrix would be 8.2 GB.  The captured step's buffers are
    allocated before the measurement; the step itself may allocate no more than 64 MB."""
    e, r, d, b = 1_000_000, 100, 128, 1024
    torch.manual_seed(0)
    m = kb.KgeModel("transe", e, r, d, l_norm=1.0).cuda()
    opt = kb.optim.create("Adagrad", m.parameters(), lr=0.1)
    st = kb.trainer.FusedAllEntityStepper(m, opt, 2 * b, 2 * b, kb.lib.LOSS_KL, b, use_graph=True, onevsall_triples=True)
    gen = torch.Generator().manual_seed(1)
    triples = torch.stack((torch.randint(0, e, (b,), generator=gen), torch.randint(0, r, (b,), generator=gen),
                           torch.randint(0, e, (b,), generator=gen)), 1)
    st.set_triples(triples.cuda())
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    st.step()
    loss = st.report[0].item()
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated() - base
    assert np.isfinite(loss)
    assert grown <= 64 << 20, f"one step allocated {grown / 2**20:.1f} MB"
    before = m.get_s_embedder().weight[triples[:, 2].cuda()].clone()
    st.step()
    assert not torch.equal(before, m.get_s_embedder().weight[triples[:, 2].cuda()])
