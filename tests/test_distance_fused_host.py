"""CPU tests of the fused all-entity path for TransE / RotatE: the captured step refuses the distance models with data
parallelism, a distributed shard and the row-sharded step (tests/test_gpu_distance_fused.py runs them on one GPU); the jobs and the plug-in's loss route every kind to the fused kernels except d > 256 and KL with
label smoothing; the ctypes signatures of the two new entries.  No GPU needed: nothing here launches a kernel."""
import os
import sys
import types

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import kgeb200 as kb  # noqa: E402

E, R = 40, 5
MODELS = [("transe", 1.0, kb.lib.NEG_L1), ("transe", 2.0, kb.lib.NEG_L2), ("rotate", 1.0, kb.lib.ROT_L1),
          ("rotate", 2.0, kb.lib.ROT_L2)]


def _opt(m):
    return kb.optim.create("Adagrad", m.parameters(), lr=0.1)


def _distributed_shard():
    return types.SimpleNamespace(e_lo=0, e_hi=E // 2, num_entities=E, group=None, distributed=True)


@pytest.mark.parametrize("model,ln,kind", MODELS)
def test_stepper_refuses_distance_models_beyond_one_gpu(model, ln, kind):
    m = kb.KgeModel(model, E, R, 16, l_norm=ln)
    with pytest.raises(NotImplementedError):
        kb.trainer.FusedAllEntityStepper(m, _opt(m), 8, 8, kb.lib.LOSS_KL, 4, use_graph=False, dp_group=object())
    with pytest.raises(NotImplementedError):
        kb.trainer.FusedAllEntityStepper(m, _opt(m), 8, 8, kb.lib.LOSS_KL, 4, use_graph=False, shard=_distributed_shard())
    with pytest.raises(NotImplementedError):
        kb.trainer.RowShardedAllEntityStepper(m, _opt(m), 8, 8, kb.lib.LOSS_KL, 4, _distributed_shard(), use_graph=False)


class _Fused(Exception):
    pass


class _Materialised(Exception):
    pass


@pytest.fixture
def spies(monkeypatch):
    """fused.all_entity_loss and the materialised scores raise markers (recording the kind) instead of launching."""
    seen = {}

    def fused_loss(*a, **kw):
        seen["kind"] = kw.get("kind", kb.lib.DOT)
        raise _Fused()

    def materialised(*a, **kw):
        raise _Materialised()

    monkeypatch.setattr(kb.fused, "all_entity_loss", fused_loss)
    monkeypatch.setattr(kb.model.KgeModel, "score_sp", materialised)
    monkeypatch.setattr(kb.model.KgeModel, "queries", lambda self, c, a, p: torch.zeros(len(a), self.get_s_embedder().dim))
    return seen


def _kvsall_batch():
    return {"queries": torch.tensor([[1, 0], [2, 1]]), "label_coords": torch.tensor([[0, 3], [1, 4]]),
            "query_type_indexes": torch.tensor([0, 0])}


@pytest.mark.parametrize("model,ln,kind", MODELS + [("distmult", 1.0, kb.lib.DOT)])
def test_jobs_route_every_kind_to_the_fused_kernels(spies, model, ln, kind):
    m = kb.KgeModel(model, E, R, 16, l_norm=ln)
    job = kb.TrainingJob1vsAll(m, _opt(m), kb.KgeLoss.create("kl"))
    assert job._use_fused()
    with pytest.raises(_Fused):
        job._process_batch(0, {"triples": torch.tensor([[1, 0, 2], [3, 1, 4]])})
    assert spies["kind"] == kind
    job = kb.TrainingJobKvsAll(m, _opt(m), kb.KgeLoss.create("bce"), E, R, label_smoothing=0.1)
    with pytest.raises(_Fused):
        job._process_batch(0, _kvsall_batch())
    assert spies["kind"] == kind


@pytest.mark.parametrize("model,ln,kind", MODELS)
def test_jobs_keep_the_materialised_path_beyond_the_fused_kernels(spies, model, ln, kind):
    wide = kb.KgeModel(model, E, R, 258, l_norm=ln)
    assert not kb.TrainingJob1vsAll(wide, _opt(wide), kb.KgeLoss.create("kl"))._use_fused()
    m = kb.KgeModel(model, E, R, 16, l_norm=ln)
    job = kb.TrainingJobKvsAll(m, _opt(m), kb.KgeLoss.create("kl"), E, R, label_smoothing=0.1)
    with pytest.raises(_Materialised):        # KL with label smoothing
        job._process_batch(0, _kvsall_batch())


@pytest.mark.parametrize("kind", [kb.lib.DOT, kb.lib.NEG_L1, kb.lib.NEG_L2, kb.lib.ROT_L1, kb.lib.ROT_L2])
def test_plugin_loss_routes_lazy_scores_by_kind(spies, monkeypatch, kind):
    inner_calls = []
    monkeypatch.setattr(kb.libkge_jobs.LazyScores, "materialize", lambda self: torch.zeros(self.shape))
    job = types.SimpleNamespace(label_smoothing=0.0)
    loss = kb.libkge_jobs.FusedKgeLoss(lambda s, y, **kw: inner_calls.append(s.shape) or torch.zeros(()), job,
                                       kb.lib.LOSS_KL, 0.0)
    idx = torch.tensor([1, 2])
    with pytest.raises(_Fused):
        loss(kb.libkge_jobs.LazyScores(kind, torch.zeros(2, 16), torch.zeros(E, 16), kb.lib.MATH_FP32), idx)
    assert spies["kind"] == kind and not inner_calls
    loss(kb.libkge_jobs.LazyScores(kind, torch.zeros(2, 258), torch.zeros(E, 258), kb.lib.MATH_FP32), idx)   # d > 256
    job.label_smoothing = 0.1
    loss(kb.libkge_jobs.LazyScores(kind, torch.zeros(2, 16), torch.zeros(E, 16), kb.lib.MATH_FP32),
         torch.zeros(2, E))                                                                             # KL + smoothing
    assert inner_calls == [torch.Size((2, E)), torch.Size((2, E))]


def test_kind_entry_signatures():
    _p, _i, _l, _f = kb.lib._p, kb.lib._i, kb.lib._l, kb.lib._f
    assert kb.lib.SIGNATURES["kgeb_fused_fwd_kind"] == [_i, _i, _p, _l, _i, _p, _l, _l, _l, _p, _p, _l, _f, _f, _p, _p,
                                                         _l, _p]
    assert kb.lib.SIGNATURES["kgeb_fused_bwd_kind"] == [_i, _i, _p, _l, _i, _p, _l, _l, _l, _p, _p, _l, _f, _f, _p, _f,
                                                         _p, _p, _p, _i, _p, _l, _p]
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "kgeb200.h")).read()
    assert "int kgeb_fused_fwd_kind(int kind, int loss," in header
    assert "int kgeb_fused_bwd_kind(int kind, int loss," in header
    lib = kb.lib.load()
    assert lib.kgeb_fused_fwd_kind.argtypes == kb.lib.SIGNATURES["kgeb_fused_fwd_kind"]
    assert lib.kgeb_fused_bwd_kind.argtypes == kb.lib.SIGNATURES["kgeb_fused_bwd_kind"]
