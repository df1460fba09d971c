"""CPU tests of the reciprocal-relations opt-in of the captured steps: the refusal without `reciprocal=True` stays, a
plain model with it is a ValueError, the host collate maps _po queries to sp_ rows on relation p + R, and -- where the
unmodified reference is installed (baseline/_ref) -- the plug-in's reciprocal model keeps the reference's checkpoint
keys.  No GPU needed: every refusal comes before anything touches a device."""
import os
import sys
import tempfile
import types

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import kgeb200 as kb  # noqa: E402
from baseline import ref_env  # noqa: E402

E, R, D = 50, 5, 16


def _opt(m):
    return kb.optim.create("Adagrad", m.parameters(), lr=0.1)


def test_reciprocal_model_is_refused_without_the_opt_in():
    m = kb.model.ReciprocalRelationsModel("distmult", E, R, D)
    with pytest.raises(NotImplementedError):
        kb.trainer.FusedAllEntityStepper(m, _opt(m), 8, 8, kb.lib.LOSS_KL, 4, use_graph=False, reciprocal=False)
    with pytest.raises(NotImplementedError):
        kb.trainer.FusedNegSamplingStepper(m, _opt(m), 4, 2, 2, kb.lib.LOSS_KL, use_graph=False, reciprocal=False)
    with pytest.raises(NotImplementedError):
        kb.trainer.RowShardedAllEntityStepper(m, _opt(m), 8, 8, kb.lib.LOSS_KL, 4, _distributed_shard(), use_graph=False)


def _distributed_shard():
    """What RowShardedAllEntityStepper reads of a shard before its refusals (fused.Shard.distributed needs a process group)."""
    return types.SimpleNamespace(e_lo=0, e_hi=E // 2, num_entities=E, group=None, distributed=True)


def test_opt_in_on_a_plain_model_is_a_value_error():
    m = kb.KgeModel("distmult", E, 2 * R, D)
    with pytest.raises(ValueError):
        kb.trainer.FusedAllEntityStepper(m, _opt(m), 8, 8, kb.lib.LOSS_KL, 4, use_graph=False, reciprocal=True)
    with pytest.raises(ValueError):
        kb.trainer.FusedNegSamplingStepper(m, _opt(m), 4, 2, 2, kb.lib.LOSS_KL, use_graph=False, reciprocal=True)
    with pytest.raises(ValueError):
        kb.trainer.RowShardedAllEntityStepper(m, _opt(m), 8, 8, kb.lib.LOSS_KL, 4, _distributed_shard(), use_graph=False,
                                              reciprocal=True)


def test_sharded_negative_sampling_keeps_refusing():
    m = kb.model.ReciprocalRelationsModel("distmult", E, R, D)
    with pytest.raises(NotImplementedError):
        kb.trainer.ShardedNegSamplingStepper(m, _opt(m), 4, 2, 2, kb.lib.LOSS_KL)


def _batch():
    queries = torch.tensor([[3, 1], [2, 7], [4, 0], [0, 9], [1, 1], [11, 2]])
    qtype = torch.tensor([0, 1, 0, 1, 1, 0])
    coords = torch.tensor([[0, 5], [1, 3], [1, 8], [2, 2], [3, 4], [4, 6], [4, 0], [5, 1]])
    return {"queries": queries, "query_type_indexes": qtype, "label_coords": coords}


def test_kvsall_rows_maps_po_queries_to_inverse_sp_rows():
    b = _batch()
    a0, p0, rc0 = kb.trainer.kvsall_rows(b["queries"], b["query_type_indexes"])
    a, p, rc = kb.trainer.kvsall_rows(b["queries"], b["query_type_indexes"], inv_rel_offset=R)
    # sp_ rows (s, p) = (q0, q1) unchanged; _po rows (p, o) = (q0, q1) -> sp_ (o, p + R)
    assert a.tolist() == [3, 7, 4, 9, 1, 11] == a0.tolist()
    assert p.tolist() == [1, 2 + R, 0, 0 + R, 1 + R, 2]
    assert p0.tolist() == [1, 2, 0, 0, 1, 2]
    assert rc.tolist() == [0] * 6 and rc.dtype == torch.int32
    assert rc0.tolist() == [0, 1, 0, 1, 1, 0]
    # offset 0 is the plain collate
    for x, y in zip(kb.trainer.kvsall_rows(b["queries"], b["query_type_indexes"], 0), (a0, p0, rc0)):
        assert torch.equal(x, y)


def test_collate_packed_of_a_reciprocal_job_gives_inverse_rows_and_permutations():
    b = _batch()
    m = kb.model.ReciprocalRelationsModel("distmult", E, R, D)
    job = kb.TrainingJobKvsAll(m, _opt(m), kb.KgeLoss.create("kl"), E, R)
    captured = {}

    class Stepper:
        nnz_max = 8

        def pack_host_batch(self, a, p, rc, lab_off, lab_col):
            captured.update(a=a, p=p, rc=rc, lab_off=lab_off, lab_col=lab_col)
            return kb.trainer.FusedAllEntityStepper.sort_perm(a), kb.trainer.FusedAllEntityStepper.sort_perm(p)

    job.stepper = Stepper()
    out = job.collate_packed(b)
    assert out["size"] == 6
    assert captured["a"].tolist() == [3, 7, 4, 9, 1, 11]
    assert captured["p"].tolist() == [1, 2 + R, 0, 0 + R, 1 + R, 2]
    assert captured["rc"].tolist() == [0] * 6
    assert captured["lab_off"].tolist() == [0, 1, 3, 4, 5, 7, 8]
    assert captured["lab_col"].tolist() == [5, 3, 8, 2, 4, 0, 6, 1]
    a_perm, p_perm = out["packed"]
    # stable argsorts of the mapped ids: the order of the deterministic scatters into the 2 R-row relation table
    assert p_perm.tolist() == [2, 0, 5, 3, 4, 1]
    assert a_perm.tolist() == [4, 0, 2, 1, 3, 5]
    plain = kb.TrainingJobKvsAll(kb.KgeModel("distmult", E, R, D), _opt(m), kb.KgeLoss.create("kl"), E, R)
    plain.stepper = Stepper()
    plain.collate_packed(b)
    assert captured["p"].tolist() == [1, 2, 0, 0, 1, 2] and captured["rc"].tolist() == [0, 1, 0, 1, 1, 0]


@pytest.mark.skipif(not ref_env.available(), reason="baseline/_ref is not installed")
@pytest.mark.parametrize("base", ["distmult", "complex"])
def test_plugin_reciprocal_model_keeps_the_reference_checkpoint_keys(base):
    ref_env.install()
    kb.libkge_plugin.register()
    from kge import Config, Dataset
    from kge.model import KgeModel
    import kge.model as km

    def make(plugin):
        tmp = tempfile.mkdtemp()
        c = Config(folder=tmp)
        if plugin:
            name = kb.libkge_plugin.configure_reciprocal(c, base)
            assert name == c.get("model") and c.get(name + ".base_model.type") == f"b200_{base}"
        else:
            c.set("model", "reciprocal_relations_model")
            c._import("reciprocal_relations_model")
            c._import(base)
            c.set("reciprocal_relations_model.base_model.type", base)
        c.set("dataset.num_entities", 31)
        c.set("dataset.num_relations", 5)
        c.set("dataset.pickle", False)
        c.set("job.device", "cpu")
        c.set("lookup_embedder.dim", 8)
        c.log = lambda *a, **k: None
        ds = Dataset(c, folder=tmp)
        rng = np.random.default_rng(0)
        t = np.stack([rng.integers(0, 31, 60), rng.integers(0, 5, 60), rng.integers(0, 31, 60)], 1).astype(np.int32)
        ds._triples["train"] = torch.from_numpy(t)
        torch.manual_seed(0)
        return KgeModel.create(c, ds)

    new, ref = make(True), make(False)
    from kge.model.reciprocal_relations_model import ReciprocalRelationsModel
    assert type(new) is km.B200ReciprocalRelationsModel and isinstance(new, ReciprocalRelationsModel)
    assert new._b200_reciprocal and new._b200_base == base
    sd_new, sd_ref = new.state_dict(), ref.state_dict()
    assert list(sd_new.keys()) == list(sd_ref.keys())
    for k in sd_ref:
        assert sd_new[k].shape == sd_ref[k].shape, k
    assert new.get_p_embedder()._embeddings.weight.shape[0] == 10
    new.load_state_dict(sd_ref)           # checkpoints load both ways
    ref.load_state_dict(new.state_dict())
