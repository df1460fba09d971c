"""The float64 references of the negative-sampling kernels (oracle/pair_ref.py) on the CPU: query transforms against the
oracle's sp_ / _po scores, the distance kinds against score_emb, the zero conventions of the gradients, and the bounds."""
import math

import pytest
import torch

from oracle import kge_oracle as ko
from oracle import pair_ref as pr

DOT_MODELS = ["distmult", "complex", "cp", "simple", "rescal"]


def tables(model, n, e, d, seed=0):
    g = torch.Generator().manual_seed(seed)
    a = torch.randn(n, d, generator=g, dtype=torch.float64)
    p = torch.randn(n, ko.relation_dim(model, d), generator=g, dtype=torch.float64)
    c = torch.randn(e, d, generator=g, dtype=torch.float64)
    return a, p, c


@pytest.mark.parametrize("model", DOT_MODELS)
@pytest.mark.parametrize("combine", ["sp_", "_po"])
def test_query_then_dot_equals_score_emb(model, combine):
    a, p, c = tables(model, 5, 7, 12)
    q = pr.query(model, pr.SP_ if combine == "sp_" else pr._PO, a, p)
    want = ko.score_emb(model, a, p, c, "sp_") if combine == "sp_" else ko.score_emb(model, c, p, a, "_po")
    assert torch.allclose(q @ c.t(), want, rtol=1e-12, atol=1e-12)
    cand = torch.arange(7).repeat(5, 1)
    assert torch.allclose(pr.pair_scores(pr.DOT, q, c, cand), want, rtol=1e-12, atol=1e-12)


def test_row_combine_mixes_the_two_forms():
    a, p, c = tables("rotate", 6, 4, 10)
    rc = torch.tensor([0, 1, 1, 0, 1, 0], dtype=torch.int32)
    q = pr.query("rotate", rc, a, p)
    for i in range(6):
        want = pr.query("rotate", int(rc[i]), a[i:i + 1], p[i:i + 1])
        assert torch.equal(q[i:i + 1], want)


@pytest.mark.parametrize("l_norm", [1, 2])
def test_distance_kinds_equal_score_emb(l_norm):
    # TransE sp_ / _po through cdist (no eps) and RotatE through the query transform
    a, p, c = tables("transe", 5, 9, 8)
    cand = torch.arange(9).repeat(5, 1)
    kind = pr.NEG_L1 if l_norm == 1 else pr.NEG_L2
    for comb, want in ((pr.SP_, ko.score_emb("transe", a, p, c, "sp_", l_norm)),
                       (pr._PO, ko.score_emb("transe", c, p, a, "_po", l_norm))):
        got = pr.pair_scores(kind, pr.query("transe", comb, a, p), c, cand)
        assert torch.allclose(got, want, rtol=1e-12, atol=1e-12)
    a, p, c = tables("rotate", 5, 9, 8)
    kind = pr.ROT_L1 if l_norm == 1 else pr.ROT_L2
    for comb, want in ((pr.SP_, ko.score_emb("rotate", a, p, c, "sp_", l_norm)),
                       (pr._PO, ko.score_emb("rotate", c, p, a, "_po", l_norm))):
        got = pr.pair_scores(kind, pr.query("rotate", comb, a, p), c, cand)
        assert torch.allclose(got, want, rtol=1e-12, atol=1e-12)


def test_transe_spo_eps_is_the_only_difference_from_the_pair_form():
    # score_emb's spo form is pairwise_distance(s + p, o) with eps 1e-6; the pair kernels use no eps
    a, p, c = tables("transe", 6, 6, 8)
    spo = ko.score_emb("transe", a, p, c, "spo", 1).view(-1)
    pair = pr.pair_scores(pr.NEG_L1, a + p, c, torch.arange(6)[:, None]).view(-1)
    assert not torch.allclose(spo, pair, rtol=0, atol=1e-9)
    pair_eps = pr.pair_scores(pr.NEG_L1, a + p + 1e-6, c, torch.arange(6)[:, None]).view(-1)
    assert torch.allclose(spo, pair_eps, rtol=1e-12, atol=1e-12)


def test_pair_grads_match_autograd_away_from_zero():
    a, p, c = tables("rotate", 4, 6, 8)
    cand = torch.randint(0, 6, (4, 5), generator=torch.Generator().manual_seed(1))
    g = torch.randn(4, 5, dtype=torch.float64)
    for kind in (pr.DOT, pr.NEG_L1, pr.NEG_L2, pr.ROT_L1, pr.ROT_L2):
        q = a.clone().requires_grad_(True)
        t = c.clone().requires_grad_(True)
        (pr.pair_scores(kind, q, t, cand) * g).sum().backward()
        dq, dc = pr.pair_grads(kind, a, c, cand, g)
        assert torch.allclose(dq, q.grad, rtol=1e-12, atol=1e-12), kind
        assert torch.allclose(pr.index_add(cand, dc, 6), t.grad, rtol=1e-12, atol=1e-12), kind


def test_zero_conventions_of_the_gradients():
    q = torch.tensor([[1.0, 2.0, 3.0, 4.0]], dtype=torch.float64)
    table = torch.tensor([[1.0, 2.0, 3.0, 4.0],           # equal: distance 0
                          [1.0, 5.0, 3.0, 4.0],           # q - c = (0, -3 | 0, 0): RotatE moduli (0, 3)
                          [1.0, 2.0, 0.0, 4.0]])          # q - c = (0, 0 | 3, 0): RotatE moduli (3, 0)
    cand = torch.tensor([[0, 1, 2]])
    g = torch.ones(1, 3, dtype=torch.float64)
    for kind in (pr.NEG_L2, pr.ROT_L2, pr.ROT_L1):
        _, dc = pr.pair_grads(kind, q, table, cand, g)
        assert torch.equal(dc[0, 0], torch.zeros(4, dtype=torch.float64)), kind
        assert torch.isfinite(dc).all()
    _, dc = pr.pair_grads(pr.NEG_L1, q, table, cand, g)
    assert torch.equal(dc[0, 0], torch.zeros(4, dtype=torch.float64))
    assert torch.equal(dc[0, 2], torch.tensor([0.0, 0.0, 1.0, 0.0], dtype=torch.float64))
    # ROT_L1: the coordinate of modulus 0 gets a zero gradient, the other one -(q - c) / |q - c|
    _, dc = pr.pair_grads(pr.ROT_L1, q, table, cand, g)
    assert torch.equal(dc[0, 1], torch.tensor([0.0, 1.0, 0.0, 0.0], dtype=torch.float64))
    assert torch.equal(dc[0, 2], torch.tensor([0.0, 0.0, -1.0, 0.0], dtype=torch.float64))
    # spo: TransE sign(0) = 0 (s + p - o + eps = 0), RotatE zero distance
    s = torch.tensor([[0.0, -1e-6]], dtype=torch.float64)
    z = torch.zeros(1, 2, dtype=torch.float64)
    gs, _, _ = pr.spo_grads("transe", s, z, torch.tensor([[1e-6, 0.0]], dtype=torch.float64), torch.ones(1), 1)
    assert torch.equal(gs, torch.zeros(1, 2, dtype=torch.float64))
    gs, gp, go = pr.spo_grads("rotate", s, torch.zeros(1, 1, dtype=torch.float64), s, torch.ones(1), 2)
    assert all(torch.equal(t, torch.zeros_like(t)) for t in (gs, gp, go))


@pytest.mark.parametrize("loss", [pr.KL, pr.BCE])
def test_ns_rows_and_grad_match_autograd(loss):
    x = torch.randn(7, 9, dtype=torch.float64, requires_grad=True)
    rows, g = pr.ns_rows_and_grad(loss, x.detach(), 0.5, 0.25)
    if loss == pr.KL:
        want = torch.nn.functional.cross_entropy(x, torch.zeros(7, dtype=torch.long), reduction="none")
    else:
        y = torch.zeros(7, 9, dtype=torch.float64)
        y[:, 0] = 1
        want = torch.nn.functional.binary_cross_entropy_with_logits(x + 0.5, y, reduction="none").sum(1)
    (0.25 * want).sum().backward()
    assert torch.allclose(rows, 0.25 * want.detach(), rtol=1e-12, atol=1e-12)
    assert torch.allclose(g, x.grad, rtol=1e-12, atol=1e-12)


def test_query_grads_match_a_finite_difference():
    for model in ("complex", "rotate", "rescal"):
        a, p, _ = tables(model, 3, 1, 6)
        g = torch.randn(3, 6, dtype=torch.float64)
        da, dp = pr.query_grads(model, pr._PO, a, p, g)
        h = 1e-6
        p2 = p.clone()
        p2[1, 2] += h
        fd = ((pr.query(model, pr._PO, a, p2) - pr.query(model, pr._PO, a, p)) * g).sum() / h
        assert abs(float(fd) - float(dp[1, 2])) < 1e-5, model


def test_bounds_are_nonnegative_and_grow_with_d():
    torch.manual_seed(0)
    prev = {}
    for d in (16, 64, 256, 1024):
        q = torch.randn(3, d)
        t = torch.randn(5, d)
        cand = torch.randint(0, 5, (3, 4))
        g = torch.randn(3, 4)
        for kind in (pr.DOT, pr.NEG_L1, pr.NEG_L2, pr.ROT_L1, pr.ROT_L2):
            b = pr.pair_score_bound(kind, q, t, cand)
            assert (b >= 0).all()
            # relative to the size of the sums, the bound must not shrink as d grows
            size = pr.pair_scores(kind, q.abs(), t.abs() if kind == pr.DOT else -t.abs(), cand).abs()
            rel = float((b / size).min())
            assert rel >= prev.get(kind, 0.0), (kind, d)
            prev[kind] = rel
            at, et, ac, ec = pr.pair_grad_terms_bound(kind, q, t, cand, g)
            assert all((x >= 0).all() for x in (at, et, ac, ec))
        for model in ("distmult", "complex", "rescal", "transe", "rotate"):
            if model == "rescal" and d > 64:
                continue
            p = torch.randn(3, ko.relation_dim(model, d))
            for l_norm in (1, 2):
                assert (pr.spo_bound(model, q, p, q.flip(0), l_norm) > 0).all()
                assert all((b >= 0).all() for b in pr.spo_grad_bound(model, q, p, q.flip(0), torch.randn(3), l_norm))
    for loss in (pr.KL, pr.BCE):
        x = torch.randn(4, 300) * 10
        rb, gb = pr.ns_loss_bound(loss, x, 0.5, 1 / 4)
        assert (rb > 0).all() and (gb > 0).all()
        # BCE rows: at least an absolute u per column (saturated softplus terms)
        if loss == pr.BCE:
            assert (rb >= 300 * pr.U / 4).all()
    lengths = torch.tensor([0, 1, 7, 8, 9, 1000])
    ch = pr.sorted_scatter_chain(lengths)
    assert (ch[1:] > 0).all() and (ch.diff() >= 0).all()
    assert int(ch[-1]) == 8 + 125 + 2
    assert math.isclose(pr.U, 2.0 ** -24)
