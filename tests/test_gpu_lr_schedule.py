"""Learning-rate schedules in the graph-captured steps (B200).

1. The _sched entries (rate read from a device word) give the bits of the by-value entries, and refuse a NULL word.
2. A captured step follows lr changes between steps: after every step its tables, optimizer state and bf16 mirror equal,
   bit for bit, those of a twin that builds a fresh stepper (a fresh capture) at every change.
3. With real torch lr schedulers, and with lr_decay, the captured step matches the autograd flow within the bounds of the
   existing parity tests; state["step"] and the state_dict match as well.
4. A failed flash pass after an lr change repeats the step at the new rate.
5. Entity and relation tables in separate parameter groups get their own rates.
6. The reference's own job with train.lr_scheduler = ReduceLROnPlateau behind b200.captured_step (needs baseline/_ref)."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from baseline import ref_env  # noqa: E402
import oracle.kge_oracle as ko  # noqa: E402

pytestmark = pytest.mark.gpu
T = torch.from_numpy
LRS = [0.2, 0.2, 0.05, 0.05, 0.0125]      # the lr of each step


@pytest.fixture(scope="module")
def kb():
    import kgeb200
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return kgeb200


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _word(x):
    return torch.tensor([x], dtype=torch.float32, device="cuda")


# ---------------------------------------------------------------------------------------------
# 1. the _sched entries
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("grad2,mirror", [(False, False), (True, False), (False, True), (True, True)])
def test_adagrad_dense_sched_equals_by_value(kb, grad2, mirror):
    n, clr, eps = 1_000_003, 0.0371, 1e-10           # odd size: the tail loop reads the word too
    g = torch.Generator(device="cuda").manual_seed(1)
    w0 = torch.randn(n, device="cuda", generator=g)
    s0 = torch.rand(n, device="cuda", generator=g)
    gr = torch.randn(n, device="cuda", generator=g)
    g2 = torch.randn(n, device="cuda", generator=g) if grad2 else None
    word = _word(clr)
    out = []
    for sched in (False, True):
        w, s = w0.clone(), s0.clone()
        m = torch.zeros(n, dtype=torch.bfloat16, device="cuda") if mirror else None
        args = (w.data_ptr(), s.data_ptr(), gr.data_ptr(), None if g2 is None else g2.data_ptr(), n)
        tail = (eps, 0.0, None if m is None else m.data_ptr(), _stream())
        if sched:
            kb.lib.call("kgeb_adagrad_dense_sched", *args, word.data_ptr(), *tail)
        else:
            kb.lib.call("kgeb_adagrad_dense", *args, clr, *tail)
        out.append((w, s, m))
    assert not torch.equal(out[0][0], w0)
    for a, b in zip(*out):
        assert (a is None and b is None) or torch.equal(a, b)
    with pytest.raises(ValueError, match="NULL"):
        kb.lib.call("kgeb_adagrad_dense_sched", w0.data_ptr(), s0.data_ptr(), gr.data_ptr(), None, n, None, eps, 0.0, None,
                    _stream())


@pytest.mark.parametrize("p", [2, 3])
def test_adagrad_dense_lp_sched_equals_by_value(kb, p):
    n, clr, eps = 300_001, 0.11, 1e-10
    g = torch.Generator(device="cuda").manual_seed(2)
    w0, s0 = torch.randn(n, device="cuda", generator=g), torch.rand(n, device="cuda", generator=g)
    gr, g2 = torch.randn(n, device="cuda", generator=g), torch.randn(n, device="cuda", generator=g)
    ws = torch.empty(kb.lib.load().kgeb_penalty_workspace_bytes(0, n), dtype=torch.uint8, device="cuda")
    word = _word(clr)
    out = []
    for sched in (False, True):
        w, s = w0.clone(), s0.clone()
        m = torch.zeros(n, dtype=torch.bfloat16, device="cuda")
        val = torch.zeros(1, device="cuda")
        name, rate = ("kgeb_adagrad_dense_lp_sched", word.data_ptr()) if sched else ("kgeb_adagrad_dense_lp", clr)
        kb.lib.call(name, w.data_ptr(), s.data_ptr(), gr.data_ptr(), g2.data_ptr(), n, rate, eps, 0.0, p, 0.01, m.data_ptr(),
                    val.data_ptr(), ws.data_ptr(), ws.numel(), _stream())
        out.append((w, s, m, val))
    for a, b in zip(*out):
        assert torch.equal(a, b)


def test_touched_update_sched_equals_by_value(kb):
    n_rows, d, n_a, n_b, clr, eps = 5000, 64, 700, 900, 0.07, 1e-10
    gen = torch.Generator(device="cuda").manual_seed(3)
    ids_a = torch.randint(0, n_rows, (n_a,), device="cuda", generator=gen)
    ids_b = torch.randint(0, n_rows, (n_b,), device="cuda", generator=gen)
    w0 = torch.randn(n_rows, d, device="cuda", generator=gen)
    s0 = torch.rand(n_rows, d, device="cuda", generator=gen)
    gd = torch.randn(n_a + n_b, d, device="cuda", generator=gen)
    gs = torch.randn(n_a + n_b + 1, d, device="cuda", generator=gen)
    word = _word(clr)
    out = []
    for sched in (False, True):
        t = kb.trainer._TouchedRows(n_rows, n_a + n_b, d, n_a, n_b, torch.device("cuda"))
        t.build(ids_a, ids_b, None, 0, n_rows, _stream())
        t.g_dense.copy_(gd)
        t.g_sparse.copy_(gs)
        t.g_sparse[int(t.num.item()):t.cap] = 0           # slots past the touched count are never written by a step
        w, s, m = w0.clone(), s0.clone(), w0.bfloat16()
        args = (w.data_ptr(), s.data_ptr(), m.data_ptr(), t.slot_of.data_ptr(), t.uniq.data_ptr(), t.num.data_ptr(), t.cap,
                t.g_dense.data_ptr(), t.g_sparse.data_ptr(), d)
        if sched:
            kb.lib.call("kgeb_touched_update_sched", *args, word.data_ptr(), eps, None, _stream())
        else:
            kb.lib.call("kgeb_touched_update", *args, clr, eps, None, _stream())
        assert int((t.slot_of != -1).sum()) == 0 and float(t.g_sparse.abs().max()) == 0.0
        out.append((w, s, m))
    assert not torch.equal(out[0][0], w0)
    for a, b in zip(*out):
        assert torch.equal(a, b)


@pytest.mark.parametrize("skip", [0, 1])
def test_fused_bwd_update_sched_equals_by_value(kb, skip):
    """The table-gradient tile kernel with Adagrad in its flush, d = 128 on a 72 MB table; skip = 1 (failed flash pass):
    neither entry touches anything."""
    e, d, b, clr, eps = 140_000, 128, 256, 0.2, 1e-10
    gen = torch.Generator(device="cuda").manual_seed(4)
    w0 = torch.randn(e, d, device="cuda", generator=gen) * 0.1
    s0 = torch.full((e, d), 0.1, device="cuda")
    q = torch.randn(b, d, device="cuda", generator=gen) * 0.5
    lab_off = torch.arange(b + 1, device="cuda")
    slots = torch.randint(0, e, (64,), device="cuda", generator=gen).unique()
    ws = torch.empty(kb.lib.load().kgeb_fused_workspace_bytes(b, d, e, 0), dtype=torch.uint8, device="cuda")
    flag = torch.tensor([skip], dtype=torch.int32, device="cuda")
    word = _word(clr)
    out = []
    for sched in (False, True):
        w, s, m = w0.clone(), s0.clone(), w0.bfloat16()
        slot_of = torch.full((e,), -1, dtype=torch.int32, device="cuda")
        slot_of[slots] = torch.arange(slots.numel(), dtype=torch.int32, device="cuda")
        gbuf = torch.zeros(slots.numel(), d, device="cuda")
        name, rate = ("kgeb_fused_bwd_update_sched", word.data_ptr()) if sched else ("kgeb_fused_bwd_update", clr)
        kb.lib.call(name, kb.lib.LOSS_BCE, q.data_ptr(), b, d, w.data_ptr(), 0, e, e, lab_off.data_ptr(), 0.0, 0.0, None,
                    1.0 / b, None, m.data_ptr(), s.data_ptr(), rate, eps, slot_of.data_ptr(), gbuf.data_ptr(),
                    flag.data_ptr(), ws.data_ptr(), ws.numel(), _stream())
        out.append((w, s, m, gbuf))
    torch.cuda.synchronize()
    if skip:
        assert torch.equal(out[0][0], w0) and torch.equal(out[0][1], s0)
    else:
        assert not torch.equal(out[0][0], w0)
    for a, b_ in zip(*out):
        assert torch.equal(a, b_)


# ---------------------------------------------------------------------------------------------
# 2. a captured step follows lr changes: the same bits as a fresh capture at every change
# ---------------------------------------------------------------------------------------------
def _set_lr(opt, lr):
    for g in opt.param_groups:
        g["lr"] = lr


def _snapshot(m, opt, mirror):
    ent, rel = m.get_s_embedder().weight, m.get_p_embedder().weight
    out = [ent, rel, opt.state[ent]["sum"], opt.state[rel]["sum"]]
    return [x.detach().clone() for x in out] + ([mirror.clone()] if mirror is not None else [])


def _follow(kb, make_model, make_opt, build, run, steps=LRS):
    """build(model, opt) -> stepper-like object; run(obj, k) -> loss of step k.  Twin A: one object, lr edited between
    steps.  Twin B: a fresh object whenever the lr changes."""
    ma, mb = make_model(), make_model()
    mb.load_state_dict(ma.state_dict())
    oa, ob = make_opt(ma, steps[0]), make_opt(mb, steps[0])
    a = build(ma, oa)
    bobj, cur = None, None
    for k, lr in enumerate(steps):
        _set_lr(oa, lr)
        _set_lr(ob, lr)
        if lr != cur:
            bobj = None
            bobj = build(mb, ob)
            cur = lr
        la, lb = run(a, k), run(bobj, k)
        assert la == lb, (k, la, lb)
        sa = _snapshot(ma, oa, getattr(_stepper(a), "mirror", None))
        sb = _snapshot(mb, ob, getattr(_stepper(bobj), "mirror", None))
        for i, (x, y) in enumerate(zip(sa, sb)):
            assert torch.equal(x, y), (k, i, (x.float() - y.float()).abs().max().item())
    st = _stepper(a)
    assert st.rate.values[0] == kb.optim.adagrad_clr(steps[-1], 0.0, len(steps))
    return ma, oa


def _stepper(obj):
    return getattr(obj, "stepper", obj)


def _kvsall_batches(kb, b, n, seed):
    g = kb.graph.synthetic_graph("toy", seed=3)
    idx = [ko.kvsall_index(g["train"], "sp"), ko.kvsall_index(g["train"], "po")]
    rng = np.random.default_rng(seed)
    batches = []
    for _ in range(n):
        ids = rng.choice(len(idx[0][0]) + len(idx[1][0]), b, replace=False)
        q, c, qt = ko.kvsall_collate(ids.tolist(), idx)
        batches.append({"queries": T(q), "label_coords": T(c), "query_type_indexes": T(qt)})
    return g["num_entities"], g["num_relations"], batches


@pytest.mark.parametrize("penalty", [False, True])
def test_captured_kvsall_step_follows_lr_changes(kb, penalty):
    """KvsAll + BCE on the fp32 CUDA-core path of a small table; penalty=True: Lp penalties folded into the Adagrad kernels."""
    b = 64
    e, r, batches = _kvsall_batches(kb, b, len(LRS), seed=1)
    nnz_max = max(len(x["label_coords"]) for x in batches)
    reg = dict(entity_embedder=dict(regularize_weight=0.01, regularize_p=2),
               relation_embedder=dict(regularize_weight=0.003, regularize_p=2)) if penalty else {}
    torch.manual_seed(0)
    make_model = lambda: kb.KgeModel("complex", e, r, 32, **reg).cuda()   # noqa: E731
    make_opt = lambda m, lr: kb.optim.create("Adagrad", m.parameters(), lr=lr, initial_accumulator_value=0.1)  # noqa: E731

    def build(m, opt):
        job = kb.TrainingJobKvsAll(m, opt, kb.KgeLoss.create("bce"), e, r, math_mode=kb.lib.MATH_FP32)
        job.enable_graph_step(b, nnz_max)
        assert (job.stepper.pen is not None) == penalty
        return job

    _follow(kb, make_model, make_opt, build, lambda job, k: job.step(k, batches[k]).total_loss)


def _ova_inputs(t):
    b = t.shape[0]
    z = torch.zeros(b, dtype=torch.int32, device="cuda")
    return (torch.cat((t[:, 0], t[:, 2])), torch.cat((t[:, 1], t[:, 1])), torch.cat((z, z + 1)),
            torch.arange(2 * b + 1, device="cuda"), torch.cat((t[:, 2], t[:, 0])))


def _triples(e, r, b, seed):
    gen = torch.Generator().manual_seed(seed)
    return torch.stack((torch.randint(0, e, (b,), generator=gen), torch.randint(0, r, (b,), generator=gen),
                        torch.randint(0, e, (b,), generator=gen)), 1).cuda()


def test_captured_large_table_1vsall_kl_bf16_step_follows_lr_changes(kb):
    """1vsAll + KL on the bf16 tiles of a 72 MB table: flash forward, Adagrad in the flush of the table-gradient kernel
    (kgeb_fused_bwd_update_sched) and the touched-row kernel."""
    e, r, d, b = 140_000, 50, 128, 256
    torch.manual_seed(0)
    make_model = lambda: kb.KgeModel("distmult", e, r, d).cuda()   # noqa: E731
    make_opt = lambda m, lr: kb.optim.create("Adagrad", m.parameters(), lr=lr, initial_accumulator_value=0.1)  # noqa: E731
    batches = [_triples(e, r, b, 10 + k) for k in range(len(LRS))]

    def build(m, opt):
        st = kb.trainer.FusedAllEntityStepper(m, opt, 2 * b, 2 * b, kb.lib.LOSS_KL, b, math_mode=kb.lib.MATH_BF16)
        assert st.seq and st.fuse_update and st.flash
        return st

    def run(st, k):
        st.set_inputs(*_ova_inputs(batches[k]))
        loss = st.step().item()
        assert st.flash_fallbacks == 0
        return loss

    _follow(kb, make_model, make_opt, build, run)


@pytest.mark.parametrize("model", ["rotate", "complex"])
def test_captured_negative_sampling_step_follows_lr_changes(kb, model):
    e, r, d, b, n = 300, 6, 32, 64, 8
    torch.manual_seed(0)
    make_model = lambda: kb.KgeModel(model, e, r, d).cuda()   # noqa: E731
    make_opt = lambda m, lr: kb.optim.create("Adagrad", m.parameters(), lr=lr, initial_accumulator_value=0.1)  # noqa: E731
    gen = torch.Generator().manual_seed(5)
    data = []
    for k in range(len(LRS)):
        gt = torch.Generator().manual_seed(100 + k)
        t = torch.stack((torch.randint(0, e, (b,), generator=gt), torch.randint(0, r, (b,), generator=gt),
                         torch.randint(0, e, (b,), generator=gt)), 1)
        data.append({"triples": t, "negative_samples": [torch.randint(0, e, (b, n), generator=gen),
                                                        torch.zeros(b, 0, dtype=torch.long),
                                                        torch.randint(0, e, (b, n), generator=gen)]})

    def build(m, opt):
        job = kb.TrainingJobNegativeSampling(m, opt, kb.KgeLoss.create("kl"))
        job.enable_graph_step(b, n, n)
        return job

    _follow(kb, make_model, make_opt, build, lambda job, k: job.step(k, data[k]).avg_loss)


# ---------------------------------------------------------------------------------------------
# 3. torch lr schedulers and lr_decay against the autograd flow
# ---------------------------------------------------------------------------------------------
PLATEAU_METRICS = [0.30, 0.28, 0.31, 0.31, 0.25, 0.2]


@pytest.mark.filterwarnings("ignore:Detected call of `lr_scheduler.step\\(\\)` before")   # the captured step never calls optimizer.step()
@pytest.mark.parametrize("kind", ["plateau", "step", "lambda", "lr_decay"])
def test_captured_step_with_torch_schedulers_matches_autograd_flow(kb, kind):
    b, n = 64, 8
    e, r, batches = _kvsall_batches(kb, b, n, seed=2)
    nnz_max = max(len(x["label_coords"]) for x in batches)
    torch.manual_seed(0)
    ref = kb.KgeModel("complex", e, r, 32).cuda()
    new = kb.KgeModel("complex", e, r, 32).cuda()
    new.load_state_dict(ref.state_dict())
    kw = dict(lr=0.2, initial_accumulator_value=0.1, lr_decay=0.05 if kind == "lr_decay" else 0.0)
    jobs, scheds = [], []
    for m in (ref, new):
        opt = kb.optim.create("Adagrad", m.parameters(), **kw)
        jobs.append(kb.TrainingJobKvsAll(m, opt, kb.KgeLoss.create("bce"), e, r))
        scheds.append({"plateau": lambda o: torch.optim.lr_scheduler.ReduceLROnPlateau(o, mode="max", factor=0.5, patience=0),
                       "step": lambda o: torch.optim.lr_scheduler.StepLR(o, step_size=2, gamma=0.3),
                       "lambda": lambda o: torch.optim.lr_scheduler.LambdaLR(o, lambda i: 1.0 / (1.0 + i)),
                       "lr_decay": lambda o: None}[kind](opt))
    jr, jn = jobs
    jn.enable_graph_step(b, nnz_max)
    lrs = []
    for i, batch in enumerate(batches):
        a, c = jr.step(i, batch), jn.step(i, batch)
        assert c.total_loss == pytest.approx(a.total_loss, rel=1e-5), i
        assert c.avg_loss == pytest.approx(a.avg_loss, rel=1e-5), i
        for got, want in ((new.get_s_embedder().weight, ref.get_s_embedder().weight),
                          (new.get_p_embedder().weight, ref.get_p_embedder().weight)):
            err = (got - want).abs().max().item()
            assert err <= 1e-5 * want.abs().max().item(), (kind, i, err)
        for s in scheds:
            if kind == "plateau" and i % 2 == 1:          # "after each validation" (train.py:212-214)
                s.step(PLATEAU_METRICS[i // 2])
            elif kind in ("step", "lambda"):
                s.step()
        lrs.append(jn.optimizer.param_groups[0]["lr"])
    if kind != "lr_decay":
        assert len(set(lrs)) >= 3, lrs          # the schedule did change the rate
    sa, sc = jr.optimizer.state_dict(), jn.optimizer.state_dict()
    assert [g["lr"] for g in sa["param_groups"]] == [g["lr"] for g in sc["param_groups"]]
    for k in sa["state"]:
        assert float(sa["state"][k]["step"]) == float(sc["state"][k]["step"]) == n
        x, y = sa["state"][k]["sum"], sc["state"][k]["sum"]
        assert (x - y).abs().max().item() <= 1e-5 * x.abs().max().item()


# ---------------------------------------------------------------------------------------------
# 4. a failed flash pass after an lr change
# ---------------------------------------------------------------------------------------------
def test_flash_fallback_after_an_lr_change_repeats_the_step_at_the_new_rate(kb):
    """The hot-entity table of test_failed_flash_pass_in_the_captured_step_...: every step's flash pass fails and the
    two-pass graph repeats it.  After the lr changes, both graphs must read the new rate: the result equals, bit for
    bit, a stepper captured at the new rate."""
    e, r, d, b = 140_000, 20, 128, 128
    torch.manual_seed(0)
    hot = torch.tensor([11, 70_001, 139_001], device="cuda")

    def make_model():
        m = kb.KgeModel("distmult", e, r, d).cuda()
        with torch.no_grad():
            m.get_s_embedder().weight[hot] *= 3.0e4
        return m

    make_opt = lambda m, lr: kb.optim.create("Adagrad", m.parameters(), lr=lr, initial_accumulator_value=0.1)  # noqa: E731
    batches = []
    for k in range(3):
        t = _triples(e, r, b, 2 + k)
        assert not torch.isin(hot, t[:, [0, 2]].flatten()).any()
        batches.append(t)

    def build(m, opt):
        st = kb.trainer.FusedAllEntityStepper(m, opt, 2 * b, 2 * b, kb.lib.LOSS_KL, b, math_mode=kb.lib.MATH_BF16)
        assert st.seq and st.fuse_update and st.flash
        return st

    def run(st, k):
        before = st.flash_fallbacks
        st.set_inputs(*_ova_inputs(batches[k]))
        loss = st.step().item()
        assert st.flash_fallbacks == before + 1, "the flash pass did not fail"
        return loss

    _follow(kb, make_model, make_opt, build, run, steps=[0.2, 0.05, 0.05])


# ---------------------------------------------------------------------------------------------
# 5. separate parameter groups
# ---------------------------------------------------------------------------------------------
def _grouped(kb, m, lr_decay=0.0):
    ent, rel = m.get_s_embedder().weight, m.get_p_embedder().weight
    return kb.optim.Adagrad([{"params": [rel], "lr": 0.02, "eps": 1e-8},
                             {"params": [ent], "lr": 0.3, "lr_decay": lr_decay}], initial_accumulator_value=0.1)


def test_entity_and_relation_groups_keep_their_own_rates(kb):
    b, n = 64, 4
    e, r, batches = _kvsall_batches(kb, b, n, seed=3)
    nnz_max = max(len(x["label_coords"]) for x in batches)
    torch.manual_seed(0)
    ref = kb.KgeModel("complex", e, r, 32).cuda()
    new = kb.KgeModel("complex", e, r, 32).cuda()
    new.load_state_dict(ref.state_dict())
    jr = kb.TrainingJobKvsAll(ref, _grouped(kb, ref, 0.1), kb.KgeLoss.create("bce"), e, r)
    jn = kb.TrainingJobKvsAll(new, _grouped(kb, new, 0.1), kb.KgeLoss.create("bce"), e, r)
    jn.enable_graph_step(b, nnz_max)
    assert (jn.stepper.eps_ent, jn.stepper.eps_rel) == (1e-10, 1e-8)
    for i, batch in enumerate(batches):
        if i == 2:
            for j in (jr, jn):
                j.optimizer.param_groups[0]["lr"] = 0.005       # the relation group only
        a, c = jr.step(i, batch), jn.step(i, batch)
        assert c.total_loss == pytest.approx(a.total_loss, rel=1e-5), i
        for got, want in ((new.get_s_embedder().weight, ref.get_s_embedder().weight),
                          (new.get_p_embedder().weight, ref.get_p_embedder().weight)):
            err = (got - want).abs().max().item()
            assert err <= 1e-5 * want.abs().max().item(), (i, err)
    assert jn.stepper.rate.values == [kb.optim.adagrad_clr(0.3, 0.1, n), 0.005]


# ---------------------------------------------------------------------------------------------
# 6. the reference's own job with its lr scheduler behind b200.captured_step
# ---------------------------------------------------------------------------------------------
@pytest.mark.skipif(not ref_env.available(), reason="baseline/_ref is not installed")
def test_reference_job_with_reduce_lr_on_plateau_behind_the_captured_step(kb):
    g = kb.graph.synthetic_graph("toy", seed=1)
    graph = {k: g[k].astype(np.int32) for k in ("train", "valid", "test")}
    opts = {"train.max_epochs": 3, "valid.every": 1, "train.optimizer": "Adagrad",
            "train.optimizer_args": {"lr": 0.1, "initial_accumulator_value": 0.1}, "eval.batch_size": 64,
            "train.batch_size": 512, "train.num_workers": 0, "eval.num_workers": 0, "train.type": "KvsAll",
            "train.loss": "kl", "train.lr_scheduler": "ReduceLROnPlateau",
            "train.lr_scheduler_args": {"patience": 0, "factor": 0.5}}
    jobs = []
    for plugin in (False, True):
        job = ref_env.make_job("distmult", graph, g["num_entities"], g["num_relations"], 32, opts,
                               device="cuda" if plugin else "cpu", plugin=plugin,
                               plugin_args={"captured_step": True} if plugin else None, seed=0)
        torch.manual_seed(1)
        job.run()
        jobs.append(job)
    ref, new = jobs
    assert getattr(new.model, "_b200_stepper", None) is not None, "the captured step never ran"
    assert [g_["lr"] for g_ in new.optimizer.param_groups] == [g_["lr"] for g_ in ref.optimizer.param_groups]
    for (ka, wa), (kc, wc) in zip(ref.model.state_dict().items(), new.model.state_dict().items()):
        assert ka == kc
        assert (wa - wc.cpu()).abs().max().item() <= 0.1 * 2e-3, ka
