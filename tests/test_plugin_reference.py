"""The reference-side plug-in (kge-1_b200/libkge_plugin.py) against the real reference, the unmodified LibKGE fork that
baseline/install_ref.sh installs into the git-ignored baseline/_ref (skipped where it is not installed).  CPU: checks
discovery through the reference's own factories, the class contract, checkpoint-key compatibility and that the CUDA path
fails loudly without a GPU."""
import os
import sys
import tempfile

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from baseline import ref_env  # noqa: E402

pytestmark = pytest.mark.skipif(not ref_env.available(), reason="baseline/_ref is not installed")


@pytest.fixture(scope="module")
def ref():
    ref_env.install()
    import kgeb200
    kgeb200.libkge_plugin.register()
    kgeb200.libkge_plugin.register()      # idempotent
    return kgeb200


def _config_and_dataset(ref, base, model_name=None, **options):
    from kge import Config, Dataset
    tmp = tempfile.mkdtemp()
    c = Config(folder=tmp)
    if model_name is None:
        ref.libkge_plugin.configure(c, base)
    else:
        c.set("model", base)
        c._import(base)
    c.set("dataset.num_entities", 31)
    c.set("dataset.num_relations", 5)
    c.set("dataset.pickle", False)
    c.set("job.device", "cpu")
    c.set("lookup_embedder.dim", 8)
    for k, v in options.items():
        c.set(k, v, create=True)
    c.log = lambda *a, **k: None
    ds = Dataset(c, folder=tmp)
    rng = np.random.default_rng(0)
    t = np.unique(np.stack([rng.integers(0, 31, 200), rng.integers(0, 5, 200), rng.integers(0, 31, 200)], 1), axis=0).astype(np.int32)
    ds._triples["train"], ds._triples["valid"], ds._triples["test"] = (torch.from_numpy(x.copy()) for x in (t[:150], t[150:170], t[170:]))
    return c, ds


@pytest.mark.parametrize("base", ["distmult", "complex", "cp", "simple", "rescal", "transe", "rotate"])
def test_plugin_models_are_created_by_the_reference_factory(ref, base):
    from kge.model.kge_model import KgeModel, RelationalScorer
    import kge.model as km
    c, ds = _config_and_dataset(ref, base)
    assert c.get("model") == f"b200_{base}"
    model = KgeModel.create(c, ds)                                   # kge_model.py:469-487
    assert isinstance(model, KgeModel) and type(model) is getattr(km, c.get(f"b200_{base}.class_name"))
    assert isinstance(model.get_scorer(), RelationalScorer) and isinstance(model.get_scorer(), km.B200Scorer)
    # checkpoint format: identical parameter names and shapes as the reference's own model
    c2, ds2 = _config_and_dataset(ref, base, model_name=base)
    theirs = KgeModel.create(c2, ds2)
    ours_sd, their_sd = model.state_dict(), theirs.state_dict()
    assert list(ours_sd.keys()) == list(their_sd.keys())
    assert [tuple(v.shape) for v in ours_sd.values()] == [tuple(v.shape) for v in their_sd.values()]
    model.load_state_dict(their_sd)                                  # a reference checkpoint loads into the plug-in
    # no CPU path: the kernels refuse host tensors instead of silently falling back
    s, p, o = torch.tensor([1, 2]), torch.tensor([0, 1]), torch.tensor([3, 4])
    with pytest.raises(ValueError, match="CUDA"):
        model.score_spo(s, p, o)
    with pytest.raises(ValueError):
        model.get_scorer().score_emb(torch.zeros(2, 8), torch.zeros(2, model.get_p_embedder().dim), torch.zeros(2, 8), "nope")


def test_reference_jobs_accept_the_plugin_model(ref):
    """Job.create -> TrainingJobKvsAll with the plug-in model and its embedded EntityRankingJob (train.py:82-84):
    the reference's job code is used unmodified."""
    from kge.job import Job
    from kge.job.train import TrainingJobKvsAll
    c, ds = _config_and_dataset(ref, "complex", **{"train.type": "KvsAll", "train.batch_size": 16,
                                                    "complex.entity_embedder.regularize_weight": 0.1})
    # options set on the base tree before configure() are copied; options of the plug-in tree can be set directly as well
    c.set("b200_complex.entity_embedder.regularize_weight", 0.1)
    torch.manual_seed(0)
    job = Job.create(c, ds)
    assert isinstance(job, TrainingJobKvsAll)
    assert type(job.model).__name__ == "B200ComplEx"
    assert type(job.valid_job.model) is type(job.model)
    pen = job.model.penalty(epoch=1, batch_index=0, num_batches=1)     # the reference's own penalty code on our model
    # entity table penalised by the s- and the o-embedder (kge_model.py:598-606); the relation embedder's weight is 0 here
    assert [k for k, _ in pen] == ["b200_complex.entity_embedder.L2_penalty", "b200_complex.entity_embedder.L2_penalty"]
    assert all(float(v) > 0 for _, v in pen)
