"""Reference-side registration of the B200 path: what a maintainer of LibKGE (Nzteb/kge-1) adds so that the UNMODIFIED
job code (TrainingJob1vsAll / KvsAll / NegativeSampling, EntityRankingJob) runs on the CUDA kernels of this repo.

    import kgeb200
    kgeb200.libkge_plugin.register()                       # once per process, after `import kge`
    kgeb200.libkge_plugin.configure(config, "complex")     # config.model = "b200_complex"
    job = Job.create(config, dataset)                      # the reference's own factory

    kgeb200.libkge_plugin.configure_reciprocal(config, "distmult")   # reciprocal_relations_model over b200_distmult

How the reference discovers a model (SURVEY.md 8b): `config.get("model")` -> `<model>.class_name` -> attribute of module
`kge.model` (kge_model.py:469-487).  `register()` therefore puts the classes on `kge.model`; `configure()` copies the base
model's option tree to `b200_<base>` (same embedder options, dims, initialisation, penalties) and points `class_name` at
the plug-in class.  The plug-in model IS a reference `KgeModel` (its embedders are the reference's own `LookupEmbedder`s,
so `state_dict()` keys, checkpoints, penalties, hooks are untouched); what changes is underneath:

  * the scorer is a `kge.model.kge_model.RelationalScorer` whose `score_emb(s_emb, p_emb, o_emb, combine)` calls the
    kernels behind include/kgeb200.h (`kgeb_score_spo`, `kgeb_query_build` + `kgeb_score_all`), same argument meaning,
    same `ValueError` for an unknown `combine`;
  * `LookupEmbedder.embed` keeps its signature; the gather runs in `kgeb_gather_rows`, and `embed_all()` returns the
    weight in place instead of an arange-gather copy (lookup_embedder.py:102-107).

Nothing here imports the reference at module import time: `kge` must already be importable by the caller.
"""
from __future__ import annotations

import copy

import torch

from . import lib as _lib
from . import libkge_jobs as _jobs
from . import model as _model
from . import ops as _ops

BASES = ("distmult", "complex", "cp", "simple", "rescal", "transe", "rotate")


def _class_name(base: str) -> str:
    return "B200" + {"distmult": "DistMult", "complex": "ComplEx", "cp": "CP", "simple": "SimplE", "rescal": "Rescal",
                     "transe": "TransE", "rotate": "RotatE"}[base]


def register():
    """Defines the plug-in classes against the caller's `kge` package and hangs them on `kge.model`; idempotent."""
    import kge.model as km
    from kge.model.kge_model import KgeModel as RefKgeModel, RelationalScorer as RefScorer
    from kge.model.reciprocal_relations_model import ReciprocalRelationsModel as RefReciprocal

    if getattr(km, "_b200_registered", False):
        return km

    class B200Scorer(RefScorer):
        """RelationalScorer.score_emb (kge_model.py:120-182) on the CUDA kernels."""

        def __init__(self, config, dataset, configuration_key=None, base="complex"):
            super().__init__(config, dataset, configuration_key)
            l_norm = float(self.get_option("l_norm")) if base in ("transe", "rotate") else 1.0
            self._impl = _model.RelationalScorer(base, l_norm)

        def score_emb(self, s_emb, p_emb, o_emb, combine: str):
            return self._impl.score_emb(s_emb, p_emb, o_emb, combine)

    def patch_embedder(emb):
        """LookupEmbedder.embed / embed_all (lookup_embedder.py:91-107) through kgeb_gather_rows, in place."""
        def embed(indexes):
            return emb._postprocess(_ops.gather_rows(emb._embeddings.weight, indexes, emb._embeddings.sparse))

        def embed_all():
            return emb._postprocess(emb._embeddings.weight)

        emb.embed, emb.embed_all = embed, embed_all
        return emb

    def _lazy_scores(self) -> bool:
        """score_sp / score_po hand out a LazyScores handle only inside a training job whose loss was wrapped by
        FusedKgeLoss (libkge_jobs.prepare_training_job), in training mode with autograd on (every scorer: the DOT
        scorers, TransE and RotatE), without embedder dropout (lookup_embedder.py:97-100 applies it to the whole table)."""
        return (getattr(self, "_b200_lazy_jobs", 0) > 0 and self.training and torch.is_grad_enabled()
                and self._entity_embedder.dropout.p == 0 and self._relation_embedder.dropout.p == 0)

    def make(base):
        class Model(RefKgeModel):
            __doc__ = f"{_class_name(base)}: the reference's {base} model on the B200 kernels (same constructor contract)."

            def __init__(self, config, dataset, configuration_key=None, init_for_load_only=False):
                self._init_configuration(config, configuration_key)
                # the base model's own option rules: even entity dims (cp.py:45-49, simple.py:48-52, rotate.py:77-81),
                # derived relation dims (cp.py:50-55 and rotate.py:82-87: d/2; rescal.py:79-96: d^2)
                d = self.get_option("entity_embedder.dim")
                if base in ("cp", "simple", "rotate") and d % 2 != 0:
                    raise ValueError(f"{_class_name(base)[4:]} requires embeddings of even dimensionality (got {d})")
                rel_key = self.configuration_key + ".relation_embedder.dim"
                if base in ("cp", "rotate", "rescal") and config.get_default(rel_key) < 0:
                    config.set(rel_key, d // 2 if base != "rescal" else d ** 2, log=True)
                scorer = B200Scorer(config, dataset, self.configuration_key, base=base)
                super().__init__(config=config, dataset=dataset, scorer=scorer, configuration_key=self.configuration_key,
                                 init_for_load_only=init_for_load_only)
                patch_embedder(self._entity_embedder)
                patch_embedder(self._relation_embedder)
                self._b200_base = base
                self._b200_eval_math = _jobs.MATH_MODES[self._b200_options().get("eval_math", "fp32")]

            def _b200_options(self) -> dict:
                """`<model>.b200.*` (configure() creates the keys): math = fp32 | tf32 | bf16 for the fused training
                kernels, eval_math = fp32 | tf32 for the ranking tiles, captured_step = graph-captured training step."""
                out = {}
                for k, default in (("math", "fp32"), ("eval_math", "fp32"), ("captured_step", False)):
                    try:
                        out[k] = self.get_option("b200." + k)
                    except Exception:
                        out[k] = default
                return out

            _b200_lazy = _lazy_scores

            def score_sp(self, s, p, o=None):
                if o is None and self._b200_lazy():
                    q = _ops.query_build(base, _lib.SP_, self.get_s_embedder().embed(s), self.get_p_embedder().embed(p))
                    return _jobs.LazyScores(self._scorer._impl.kind, q, self.get_o_embedder()._embeddings.weight, self._b200_math)
                return super().score_sp(s, p, o)

            def score_po(self, p, o, s=None):
                if s is None and self._b200_lazy():
                    q = _ops.query_build(base, _lib._PO, self.get_o_embedder().embed(o), self.get_p_embedder().embed(p))
                    return _jobs.LazyScores(self._scorer._impl.kind, q, self.get_s_embedder()._embeddings.weight, self._b200_math)
                return super().score_po(p, o, s)

            def prepare_job(self, job, **kwargs):
                """kge_model.py:583-586 + the fused seams of this path (idempotent: re-run at every validation)."""
                super().prepare_job(job, **kwargs)
                from kge.job.train import TrainingJob
                if isinstance(job, TrainingJob):
                    _jobs.prepare_training_job(job, self, base, self._b200_options())

            def penalty(self, **kwargs):
                return _jobs.captured_penalties(self, super().penalty, **kwargs)

        Model.__name__ = Model.__qualname__ = _class_name(base)
        return Model

    class B200ReciprocalRelationsModel(RefReciprocal):
        """The reference's reciprocal_relations_model (its constructor, modules, state_dict keys, score_spo / score_sp_po)
        over a `b200_<base>` base model (configure_reciprocal), with the fused seams of the plug-in: score_sp / score_po
        hand out LazyScores in training -- score_po as the sp_ query (o, p + R) of reciprocal_relations_model.py:70-83 --,
        1vsAll / KvsAll jobs get the captured step with `reciprocal=True`, the fused evaluation ranks the _po side as
        sp_ queries on p + R."""

        def __init__(self, config, dataset, configuration_key=None, init_for_load_only=False):
            super().__init__(config=config, dataset=dataset, configuration_key=configuration_key,
                             init_for_load_only=init_for_load_only)
            base = getattr(self._base_model, "_b200_base", None)
            if base is None:
                raise ValueError("B200ReciprocalRelationsModel needs a b200_<base> base model (configure_reciprocal)")
            self._b200_base = base
            self._b200_reciprocal = True
            self._b200_eval_math = self._base_model._b200_eval_math

        _b200_lazy = _lazy_scores

        def score_sp(self, s, p, o=None):
            if o is None and self._b200_lazy():
                q = _ops.query_build(self._b200_base, _lib.SP_, self.get_s_embedder().embed(s), self.get_p_embedder().embed(p))
                return _jobs.LazyScores(self._scorer._impl.kind, q, self.get_o_embedder()._embeddings.weight, self._b200_math)
            return super().score_sp(s, p, o)

        def score_po(self, p, o, s=None):
            if s is None and self._b200_lazy():
                p_inv = self.get_p_embedder().embed(p + self.dataset.num_relations())
                q = _ops.query_build(self._b200_base, _lib.SP_, self.get_o_embedder().embed(o), p_inv)
                return _jobs.LazyScores(self._scorer._impl.kind, q, self.get_s_embedder()._embeddings.weight, self._b200_math)
            return super().score_po(p, o, s)

        def prepare_job(self, job, **kwargs):
            """The fused seams are installed for THIS model first: the base model's own installation, reached through the
            reference's prepare_job, then finds the job prepared and leaves it alone (it would treat _po as _po)."""
            from kge.job.train import TrainingJob
            if isinstance(job, TrainingJob):
                _jobs.prepare_training_job(job, self, self._b200_base, self._base_model._b200_options(), reciprocal=True)
            super().prepare_job(job, **kwargs)

        def penalty(self, **kwargs):
            return _jobs.captured_penalties(self, super().penalty, **kwargs)

    for base in BASES:
        setattr(km, _class_name(base), make(base))
    km.B200ReciprocalRelationsModel = B200ReciprocalRelationsModel
    km.B200Scorer = B200Scorer
    km._b200_registered = True
    _jobs.register_jobs()
    return km


def configure(config, base: str, math: str = "fp32", eval_math: str = "fp32", captured_step: bool = False,
              kernel_optimizer: bool = True) -> str:
    """Points `config` at the plug-in model of `base`: imports the base model's defaults, copies its option tree to
    `b200_<base>` with `class_name` replaced, sets `model`; adds the `b200_<base>.b200.*` options (arithmetic of the fused
    kernels, captured step) and, with `kernel_optimizer`, rewrites `train.optimizer` Adagrad | Adam to the kernel-backed
    classes registered on torch.optim.  Call it AFTER setting `train.optimizer`.  Returns the model name."""
    if base not in BASES:
        raise ValueError(f"no B200 plug-in for model {base!r}")
    name = f"b200_{base}"
    config._import(base)
    tree = copy.deepcopy(config.options[base])
    tree["class_name"] = _class_name(base)
    tree["b200"] = {"math": math, "eval_math": eval_math, "captured_step": bool(captured_step)}
    config.options[name] = tree
    config.set("model", name)
    if kernel_optimizer and config.get("train.optimizer") in ("Adagrad", "Adam"):
        config.set("train.optimizer", "B200" + config.get("train.optimizer"))     # torch.optim.B200Adagrad / B200Adam
    return name


def configure_reciprocal(config, base: str, math: str = "fp32", eval_math: str = "fp32", captured_step: bool = False,
                         kernel_optimizer: bool = True) -> str:
    """Points `config` at the reference's reciprocal relations model over the plug-in model of `base`: configure() builds
    the `b200_<base>` tree (and rewrites the optimizer); the option tree of `reciprocal_relations_model` is copied to
    `b200_reciprocal_relations_model` with `base_model.type: b200_<base>` and `class_name` B200ReciprocalRelationsModel, and
    `model` is set to it.  The `b200.*` options are read from the base model's tree.  Returns the model name."""
    configure(config, base, math=math, eval_math=eval_math, captured_step=captured_step, kernel_optimizer=kernel_optimizer)
    name = "b200_reciprocal_relations_model"
    config._import("reciprocal_relations_model")
    tree = copy.deepcopy(config.options["reciprocal_relations_model"])
    tree["class_name"] = "B200ReciprocalRelationsModel"
    tree["base_model"] = dict(tree.get("base_model") or {}, type=f"b200_{base}")
    config.options[name] = tree
    config.set("model", name)
    return name
