"""GPU tests of reciprocal-relations training in the captured steps (`reciprocal=True`): the *_inv batch builders, the
captured all-entity step against the plain step on the same 2 R-row table fed the rewritten batch (bit for bit), against
the reference's golden step (aux2.npz, `recip.*`), the negative-sampling step against the autograd flow, and -- where the
unmodified reference is installed (baseline/_ref) -- the plug-in's reciprocal model inside the reference's own jobs."""
import os
import sys
import tempfile

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from baseline import ref_env  # noqa: E402
from oracle import kge_oracle as ko  # noqa: E402

pytestmark = pytest.mark.gpu

T = torch.from_numpy


@pytest.fixture(scope="module")
def kb():
    import kgeb200
    assert torch.cuda.is_available(), "these tests need a GPU"
    kgeb200.lib.load()
    return kgeb200


def _triples(e, r, b, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.stack((torch.randint(0, e, (b,), generator=g), torch.randint(0, r, (b,), generator=g),
                        torch.randint(0, e, (b,), generator=g)), 1)


def _inverse_rows(t, r, dev="cuda"):
    """Host form of the reciprocal 1vsAll batch: sp_ rows (s, p), then the _po rows as sp_ rows (o, p + R)."""
    t = t.to(dev)
    s, p, o = t[:, 0], t[:, 1], t[:, 2]
    b = len(t)
    return (torch.cat((s, o)), torch.cat((p, p + r)), torch.zeros(2 * b, dtype=torch.int32, device=dev),
            torch.arange(2 * b + 1, dtype=torch.int64, device=dev), torch.cat((o, s)))


# ---------------------------------------------------------------------------------------------
# 1. batch builders
# ---------------------------------------------------------------------------------------------
def _ova_build(kb, name, t, e, r, *extra):
    b = len(t)
    dev = "cuda"
    out = [torch.full((2 * b,), -1, dtype=torch.int64, device=dev), torch.full((2 * b,), -1, dtype=torch.int64, device=dev),
           torch.full((2 * b,), -1, dtype=torch.int32, device=dev), torch.full((2 * b + 1,), -1, dtype=torch.int64, device=dev),
           torch.full((2 * b,), -1, dtype=torch.int64, device=dev)] + [torch.full((2 * b,), -1, dtype=torch.int32, device=dev)
                                                                       for _ in range(3)]
    tc = t.cuda().contiguous()
    kb.lib.call(name, tc.data_ptr(), b, e, r, *[x.data_ptr() for x in out], *extra, kb.lib.stream_ptr(tc))
    torch.cuda.synchronize()
    return [x.cpu() for x in out]


def test_onevsall_inverse_builder_matches_host_collate(kb):
    e, r, b = 5000, 37, 1000
    t = _triples(e, r, b, 1)
    old = _ova_build(kb, "kgeb_onevsall_batch_build", t, e, r)
    zero = _ova_build(kb, "kgeb_onevsall_batch_build_inv", t, e, r, 0)
    for x, y in zip(old, zero):
        assert torch.equal(x, y)
    got = _ova_build(kb, "kgeb_onevsall_batch_build_inv", t, e, r, r)
    a, p, rc, off, col = (x.cpu() for x in _inverse_rows(t, r, "cpu"))
    sp = kb.trainer.FusedAllEntityStepper.sort_perm
    want = [a, p, rc, off, col, sp(a), sp(p), sp(col, 2 * b)]
    for name, x, y in zip(("a", "p", "combine", "lab_off", "lab_col", "a_perm", "p_perm", "lab_perm"), got, want):
        assert torch.equal(x, y), name


def _kvsall_build(kb, name, sp, po, ids, cap, e, r, *extra):
    dev = "cuda"
    b = len(ids)
    out = [torch.full((b,), -1, dtype=torch.int64, device=dev), torch.full((b,), -1, dtype=torch.int64, device=dev),
           torch.full((b,), -1, dtype=torch.int32, device=dev), torch.full((b + 1,), -1, dtype=torch.int64, device=dev),
           torch.full((cap,), -1, dtype=torch.int64, device=dev), torch.full((b,), -1, dtype=torch.int32, device=dev),
           torch.full((b,), -1, dtype=torch.int32, device=dev), torch.full((cap,), -1, dtype=torch.int32, device=dev),
           torch.full((1,), -1, dtype=torch.int32, device=dev)]
    ws = torch.empty(kb.lib.load().kgeb_kvsall_build_workspace_bytes(b, cap), dtype=torch.uint8, device=dev)
    d_sp, d_po = kb.lib.index_descs([sp.device_arrays(dev)]), kb.lib.index_descs([po.device_arrays(dev)])
    idc = ids.cuda().contiguous()
    kb.lib.call(name, d_sp, d_po, idc.data_ptr(), b, cap, e, r, *[x.data_ptr() for x in out], ws.data_ptr(), ws.numel(),
                *extra, kb.lib.stream_ptr(idc))
    torch.cuda.synchronize()
    return [x.cpu() for x in out]


def test_kvsall_inverse_builder_matches_host_collate(kb):
    g = kb.graph.synthetic_graph("toy", seed=3)
    e, r = g["num_entities"], g["num_relations"]
    idx = [ko.kvsall_index(g["train"], "sp"), ko.kvsall_index(g["train"], "po")]
    sp, po = kb.index.KvsAllIndex(g["train"], "sp"), kb.index.KvsAllIndex(g["train"], "po")
    ids = np.random.default_rng(0).choice(len(idx[0][0]) + len(idx[1][0]), 97, replace=False)
    q, coords, qt = ko.kvsall_collate(ids.tolist(), idx)
    cap = len(coords) + 13
    ids_t = T(ids.astype(np.int64))
    old = _kvsall_build(kb, "kgeb_kvsall_batch_build", sp, po, ids_t, cap, e, r)
    zero = _kvsall_build(kb, "kgeb_kvsall_batch_build_inv", sp, po, ids_t, cap, e, r, 0)
    for x, y in zip(old, zero):
        assert torch.equal(x, y)
    got = _kvsall_build(kb, "kgeb_kvsall_batch_build_inv", sp, po, ids_t, cap, e, r, r)
    a, p, rc = kb.trainer.kvsall_rows(T(q), T(qt), inv_rel_offset=r)
    assert (qt == 1).any() and rc.eq(0).all()
    off, col = kb.fused.csr_from_coords(T(coords), len(ids))
    sp_ = kb.trainer.FusedAllEntityStepper.sort_perm
    col_pad = torch.zeros(cap, dtype=torch.int64)
    col_pad[:len(col)] = col
    want = [a, p, rc, off, col_pad, sp_(a), sp_(p), sp_(col, cap), torch.zeros(1, dtype=torch.int32)]
    for name, x, y in zip(("a", "p", "combine", "lab_off", "lab_col", "a_perm", "p_perm", "lab_perm", "overflow"), got, want):
        assert torch.equal(x, y), name


# ---------------------------------------------------------------------------------------------
# 2. exactness: reciprocal captured step == plain captured step on the rewritten batch
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("no_fused_update", ["0", "1"])
@pytest.mark.parametrize("math", ["bf16", "fp32"])
@pytest.mark.parametrize("loss", ["kl", "bce"])
def test_reciprocal_captured_step_equals_plain_step_on_rewritten_batch(kb, monkeypatch, loss, math, no_fused_update):
    monkeypatch.setenv("KGEB_NO_FUSED_UPDATE", no_fused_update)
    e, r, d, b = 140_000, 20, 128, 64          # 140,000 x 128 fp32 = 72 MB: the large-table flows
    loss_kind = kb.lib.LOSS_KL if loss == "kl" else kb.lib.LOSS_BCE
    math_mode = kb.lib.MATH_BF16 if math == "bf16" else kb.lib.MATH_FP32
    torch.manual_seed(0)
    rec = kb.model.ReciprocalRelationsModel("distmult", e, r, d).cuda()
    plain = kb.KgeModel("distmult", e, 2 * r, d).cuda()
    plain.load_state_dict(rec.state_dict())
    steppers = []
    for m, kw in ((rec, dict(onevsall_triples=True, reciprocal=True)), (plain, {})):
        opt = kb.optim.create("Adagrad", m.parameters(), lr=0.2, initial_accumulator_value=0.1)
        steppers.append(kb.trainer.FusedAllEntityStepper(m, opt, 2 * b, 2 * b, loss_kind, b, math_mode=math_mode, **kw))
    st_r, st_p = steppers
    assert st_r.fuse_update == st_p.fuse_update == (math == "bf16" and no_fused_update == "0")
    assert st_r.seq == (math == "bf16")
    for i in range(3):
        t = _triples(e, r, b, 10 + i)
        st_r.set_triples(t.cuda())
        st_p.set_inputs(*_inverse_rows(t, r))
        lr_, lp_ = st_r.step().clone(), st_p.step().clone()
        assert torch.equal(lr_, lp_), (i, lr_.item(), lp_.item())
        assert torch.equal(st_r.report[0], st_p.report[0])
        # the reported value is that of the _po rows (the last query type, train.py:747)
        assert st_r.report[1].item() == pytest.approx(st_r.loss_rows[b:].sum().item(), rel=1e-5)
    assert st_r.flash_fallbacks == st_p.flash_fallbacks == 0
    for x, y in ((rec.get_s_embedder().weight, plain.get_s_embedder().weight),
                 (rec.get_p_embedder().weight, plain.get_p_embedder().weight),
                 (st_r.opt.state[st_r.ent]["sum"], st_p.opt.state[st_p.ent]["sum"]),
                 (st_r.opt.state[st_r.rel]["sum"], st_p.opt.state[st_p.rel]["sum"])):
        assert torch.equal(x, y)
    # both halves of the relation table moved (sp_ rows on p, inverse rows on p + R)
    moved = (st_r.opt.state[st_r.rel]["sum"] != 0.1).any(1)
    assert moved[:r].any() and moved[r:].any()


# ---------------------------------------------------------------------------------------------
# 3. the reference's reciprocal 1vsAll step (golden)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("onevsall_triples", [True, False])
def test_reciprocal_captured_step_matches_reference_golden(kb, golden, onevsall_triples):
    """aux2.npz `recip.<base>.b0.*`: one TrainingJob1vsAll step (KL, Adagrad lr 0.2) of the reference's
    reciprocal_relations_model; fp32 math, tolerances of DESIGN section 2 (loss / gradient 2e-5)."""
    g = golden("aux2")
    for tag in g["recip.cases"]:
        tag = str(tag)
        base = tag.split(".")[1]
        ent, rel = g[tag + ".ent"], g[tag + ".rel"]
        t = T(g[tag + ".b0.triples"]).long()
        b, r = len(t), rel.shape[0] // 2
        m = kb.ReciprocalRelationsModel(base, ent.shape[0], r, ent.shape[1]).cuda()
        with torch.no_grad():
            m.get_s_embedder().weight.copy_(T(ent))
            m.get_p_embedder().weight.copy_(T(rel))
        opt = kb.optim.create("Adagrad", m.parameters(), lr=0.2)
        st = kb.trainer.FusedAllEntityStepper(m, opt, 2 * b, 2 * b, kb.lib.LOSS_KL, b, math_mode=kb.lib.MATH_FP32,
                                              onevsall_triples=onevsall_triples, reciprocal=True)
        if onevsall_triples:
            st.set_triples(t.cuda())
        else:
            st.set_inputs(*_inverse_rows(t, r))
        loss = st.step().item()
        assert loss == pytest.approx(float(g[tag + ".b0.loss"]), rel=2e-5)
        # Adagrad from a zero accumulator: state = g^2, so |g| is compared through the state.  The parameters moved by
        # lr * g / (|g| + 1e-10), which turns a rounding-level difference of a near-zero g into an O(lr) one: they are
        # compared where |g| >= 1e-4 max |g|
        for w, key, grad in ((m.get_s_embedder().weight, ".b0.ent", ".b0.grad_ent"),
                             (m.get_p_embedder().weight, ".b0.rel", ".b0.grad_rel")):
            gabs = opt.state[w]["sum"].sqrt().cpu().double().numpy()
            want = np.abs(g[tag + grad]).astype(np.float64)
            assert np.abs(gabs - want).max() <= 2e-5 * want.max(), (tag, key)
            sure = want >= 1e-4 * want.max()
            diff = np.abs(w.detach().cpu().double().numpy() - g[tag + key])
            assert sure.any() and diff[sure].max() <= 1e-5, (tag, key, diff[sure].max())


# ---------------------------------------------------------------------------------------------
# 4. negative sampling
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model", ["distmult", "complex", "rotate", "transe"])
def test_reciprocal_negative_sampling_step_matches_autograd_flow(kb, model):
    """slot S = ReciprocalRelationsModel.score_spo(..., "s"): the sp_ query (o, p + R) against the subject candidates;
    the reference flow (fused_path=False: score_spo on the expanded triples, loss, backward, Adagrad) on the same
    negatives."""
    e, r, d, b, n = 300, 6, 32, 64, 8
    torch.manual_seed(0)
    models = [kb.model.ReciprocalRelationsModel(model, e, r, d).cuda() for _ in range(2)]
    models[1].load_state_dict(models[0].state_dict())
    jobs = []
    for i, m in enumerate(models):
        opt = kb.optim.create("Adagrad", m.parameters(), lr=0.1, initial_accumulator_value=0.1)
        job = kb.TrainingJobNegativeSampling(m, opt, kb.KgeLoss.create("kl"), fused_path=False)
        if i == 1:
            job.enable_graph_step(b, n, n, use_graph=True)
            assert job.stepper.inv_rel == r
        jobs.append(job)
    gen = torch.Generator().manual_seed(5)
    for step in range(3):
        t = _triples(e, r, b, 100 + step)
        negs = [torch.randint(0, e, (b, n), generator=gen), torch.zeros(b, 0, dtype=torch.long),
                torch.randint(0, e, (b, n), generator=gen)]
        a = jobs[0].step(step, {"triples": t, "negative_samples": negs})
        c = jobs[1].step(step, {"triples": t, "negative_samples": negs})
        assert c.avg_loss == pytest.approx(a.avg_loss, rel=2e-5)
    for x, y in ((models[0].get_s_embedder().weight, models[1].get_s_embedder().weight),
                 (models[0].get_p_embedder().weight, models[1].get_p_embedder().weight)):
        assert (x - y).abs().max().item() <= 2e-5 * max(1.0, x.abs().max().item())
        sx, sy = jobs[0].optimizer.state[x]["sum"], jobs[1].optimizer.state[y]["sum"]
        assert (sx - sy).abs().max().item() <= 2e-5 * sx.abs().max().item()
    # the inverse relation rows p + R received gradient
    assert (jobs[1].optimizer.state[models[1].get_p_embedder().weight]["sum"][r:] != 0.1).any()


# ---------------------------------------------------------------------------------------------
# 5. the plug-in inside the reference's own jobs
# ---------------------------------------------------------------------------------------------
BASE = {"train.max_epochs": 1, "valid.every": 1, "train.optimizer": "Adagrad",
        "train.optimizer_args": {"lr": 0.1, "initial_accumulator_value": 0.1}, "eval.batch_size": 64,
        "train.batch_size": 512, "train.num_workers": 0, "eval.num_workers": 0}


def _reciprocal_job(base, graph, e, r, dim, options, device, plugin, plugin_args=None, seed=0):
    """ref_env.make_job for the reciprocal relations model: the reference's own (CPU) or the plug-in's (cuda)."""
    ref_env.install()
    from kge import Config, Dataset
    from kge.job import Job
    folder = tempfile.mkdtemp(prefix="kgeb200_ref_")
    c = Config(folder=folder)
    c.set("job.device", device)
    for k, v in options.items():
        if k.startswith("train.optimizer"):
            c.set(k, v, create=True)
    if plugin:
        import kgeb200
        kgeb200.libkge_plugin.register()
        kgeb200.libkge_plugin.configure_reciprocal(c, base, **(plugin_args or {}))
    else:
        c.set("model", "reciprocal_relations_model")
        c._import("reciprocal_relations_model")
        c._import(base)
        c.set("reciprocal_relations_model.base_model.type", base)
    c.set("dataset.num_entities", e)
    c.set("dataset.num_relations", r)
    c.set("dataset.pickle", False)
    c.set("lookup_embedder.dim", dim)
    for k, v in options.items():
        if not k.startswith("train.optimizer"):
            c.set(k, v, create=True)
    ds = Dataset(c, folder=folder)
    for split, arr in graph.items():
        ds._triples[split] = torch.from_numpy(arr.copy())
    torch.manual_seed(seed)
    job = Job.create(c, ds)
    job.epoch_entries = []
    job.post_epoch_hooks.append(ref_env._keep_epoch_entry)
    c.log = ref_env._quiet
    c.print = ref_env._quiet
    return job


@pytest.mark.skipif(not ref_env.available(), reason="baseline/_ref is not installed")
@pytest.mark.parametrize("captured", [False, True])
@pytest.mark.parametrize("train_type,base,loss", [("1vsAll", "distmult", "kl"), ("KvsAll", "complex", "bce")])
def test_reference_reciprocal_job_on_plugin_matches_cpu_reference(kb, train_type, base, loss, captured):
    g = kb.graph.synthetic_graph("toy", seed=1)
    graph = {k: g[k].astype(np.int32) for k in ("train", "valid", "test")}
    e, r = g["num_entities"], g["num_relations"]
    opts = dict(BASE, **{"train.type": train_type, "train.loss": loss})
    jobs = []
    for plugin in (False, True):
        job = _reciprocal_job(base, graph, e, r, 32, opts, "cuda" if plugin else "cpu", plugin,
                              {"captured_step": captured}, seed=0)
        torch.manual_seed(1)
        job.run()
        jobs.append(job)
    ref, new = jobs
    import kge.model as km
    assert type(new.model) is km.B200ReciprocalRelationsModel
    if captured:
        assert getattr(new.model, "_b200_stepper", None) is not None and new.model._b200_stepper.inv_rel == r
    a, c = ref.epoch_entries[-1], new.epoch_entries[-1]
    assert c["avg_loss"] == pytest.approx(a["avg_loss"], rel=5e-5)
    for (ka, wa), (kc, wc) in zip(ref.model.state_dict().items(), new.model.state_dict().items()):
        assert ka == kc
        assert (wa - wc.cpu()).abs().max().item() <= 0.1 * 2e-3, ka
    va, vc = ref.valid_trace[-1], new.valid_trace[-1]
    for k in ("mean_reciprocal_rank", "mean_reciprocal_rank_filtered", "hits_at_1_filtered", "hits_at_10_filtered"):
        assert abs(va[k] - vc[k]) <= 1e-3, (k, va[k], vc[k])


@pytest.mark.skipif(not ref_env.available(), reason="baseline/_ref is not installed")
@pytest.mark.parametrize("captured", [False, True])
def test_reference_reciprocal_job_on_plugin_never_builds_the_score_matrix(kb, captured):
    """200,000 entities, 512 triples per batch: a [1024, E] fp32 score matrix would be 819 MB, the tables 26 MB each."""
    e, r, n = 200_000, 10, 2048
    rng = np.random.default_rng(0)
    tr = np.stack([rng.integers(0, e, n), rng.integers(0, r, n), rng.integers(0, e, n)], 1).astype(np.int32)
    graph = {"train": tr, "valid": tr[:64], "test": tr[64:128]}
    opts = dict(BASE, **{"train.type": "1vsAll", "train.loss": "kl", "valid.every": 0})
    job = _reciprocal_job("distmult", graph, e, r, 32, opts, "cuda", True, {"captured_step": captured})
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    torch.manual_seed(1)
    job.run()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    assert peak < 400 << 20, peak
