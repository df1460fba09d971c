"""Reference-side JOB integration of the B200 path: what `libkge_plugin.register()` installs so that the reference's own,
unmodified job code (kge/job/train.py, kge/job/entity_ranking.py) reaches the FUSED kernels -- not only the materialised
`[B, E]` score path -- through the seams SURVEY.md 8(b) lists.  Nothing in the reference is edited.

Three levels, all installed from `model.prepare_job(job)` (called by every job, train.py:474, entity_ranking.py:50;
`Job._is_prepared` is never set, job.py:52,153-154, so installation is idempotent per job object):

1. **fused loss** (any TrainingJob1vsAll / TrainingJobKvsAll with `train.loss` kl | bce; TransE / RotatE on fp32 tiles).  The job keeps
   running its own `_process_batch` (train.py:679-756, 1032-1062).  `model.score_sp / score_po` return a `LazyScores`
   handle instead of the `[B, E]` matrix; `job.loss` (a plain attribute, train.py:67) is wrapped by `FusedKgeLoss`, which
   recognises the handle and calls the fused score+loss kernels (kgeb_fused_fwd / kgeb_fused_bwd behind an
   autograd.Function): the job's `loss_value = self.loss(scores, labels) / batch_size; loss_value.item();
   loss_value.backward()` lines run as written, the score matrix is never materialised.
2. **captured step** (`<model>.b200.captured_step: true`; 1vsAll and KvsAll with dense Adagrad).  `job._process_batch` is
   overridden ON THE JOB OBJECT by a function that feeds the batch to the graph-captured stepper (trainer.py): gather ->
   fused forward/backward -> scatter -> Adagrad in one CUDA-graph replay.  The update has been applied when it returns, the
   parameters' `.grad` stay None, so the job's `optimizer.step()` (train.py:375) finds nothing to do; penalty terms are
   folded into the Adagrad kernels and reported through `model.penalty()` as leaf tensors.  Batches of another size (the
   last one of an epoch) run the reference's own `_process_batch` with the fused loss of level 1.
3. **fused evaluation**: `kge.job.EntityRankingJob` is rebound to a subclass (the factories bind late, eval.py:75-79) whose
   `_run` keeps the reference's loader, hooks, histograms and trace entries but ranks every batch with the fused
   score-and-count kernel (kgeb_rank_count) on a filter CSR built on the device from the dataset's own indexes; the
   Python-loop histogram hooks (eval.py:138-224) are replaced by their device forms.

Optimizer: `torch.optim.B200Adagrad` / `B200Adam` are registered (KgeOptimizer.create does `getattr(torch.optim, name)`,
optimizer.py:10-17); `configure()` rewrites `train.optimizer` accordingly.  Same state keys as torch's.
"""
from __future__ import annotations

import math
import time
import types
from typing import Dict, List, Optional

import torch

from . import fused, lib, metrics as dm, ops
from .index import KvsAllIndex, filter_csr

MATH_MODES = {"fp32": lib.MATH_FP32, "tf32": lib.MATH_TF32, "bf16": lib.MATH_BF16}


# ---------------------------------------------------------------------------------------------
# level 1: lazy score handle + fused loss
# ---------------------------------------------------------------------------------------------
class LazyScores:
    """What `score_sp` / `score_po` of a plug-in model return inside a training job whose loss is a `FusedKgeLoss`: the
    query vectors (with autograd through the embedding gathers) and the candidate table, NOT the `[n, E]` matrix.
    Anything that treats it as a tensor gets the materialised matrix (`materialize()`), so foreign code keeps working."""

    def __init__(self, kind: int, q: torch.Tensor, table: torch.Tensor, math_mode: int):
        self.kind, self.q, self.table, self.math_mode = kind, q, table, math_mode

    def materialize(self) -> torch.Tensor:
        m = self.math_mode if (self.math_mode == lib.MATH_TF32 and self.kind == lib.DOT) else lib.MATH_FP32
        return ops.score_all(self.kind, self.q, self.table, m)

    @property
    def shape(self):
        return torch.Size((self.q.shape[0], self.table.shape[0]))

    def size(self, dim=None):
        return self.shape if dim is None else self.shape[dim]

    def __getattr__(self, name):          # view / to / detach / ... : whatever a tensor offers, on the real matrix
        return getattr(self.materialize(), name)


def labels_to_csr(labels: torch.Tensor, n: int, label_smoothing: float, num_entities: int):
    """The label argument the reference's jobs pass to `self.loss` -> CSR over the batch rows.
    1-D: class indexes (1vsAll, train.py:1042,1052).  2-D: the dense `[n, E]` 0/1 matrix of KvsAll, possibly smoothed as
    `(1 - ls) * y + 1 / E` (train.py:698-721); duplicate coordinates were summed by `to_dense()` and come back as repeated
    columns."""
    dev = labels.device
    if labels.dim() == 1:
        return torch.arange(n + 1, dtype=torch.int64, device=dev), labels.long().contiguous()
    y = labels
    if label_smoothing > 0.0:
        y = (labels - 1.0 / num_entities) / (1.0 - label_smoothing)
    nz = (y > 0.5).nonzero()                       # row-major, i.e. ascending columns within a row
    cnt = y[nz[:, 0], nz[:, 1]].round().long()
    rows, cols = nz[:, 0].repeat_interleave(cnt), nz[:, 1].repeat_interleave(cnt)
    off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    off[1:] = torch.cumsum(torch.bincount(rows, minlength=n), 0)
    return off, cols.contiguous()


class FusedKgeLoss:
    """Wraps the job's KgeLoss (kge/util/loss.py).  Called exactly like it -- `loss(scores, labels, **kw)`, result NOT
    divided by the batch size -- and delegates to it unless `scores` is a LazyScores handle."""

    def __init__(self, inner, job, loss_kind: int, offset: float):
        self._inner, self._job, self.kind, self.offset = inner, job, loss_kind, float(offset)

    def __getattr__(self, name):
        return getattr(self._inner, name)

    def __call__(self, scores, labels, **kwargs):
        if not isinstance(scores, LazyScores):
            return self._inner(scores, labels, **kwargs)
        ls = float(getattr(self._job, "label_smoothing", 0.0) or 0.0) if labels.dim() == 2 else 0.0
        d = scores.q.shape[1]
        if d > 256 or (self.kind == lib.LOSS_KL and ls > 0.0 and labels.dim() == 2):
            return self._inner(scores.materialize(), labels, **kwargs)
        n, e = scores.q.shape[0], scores.table.shape[0]
        lab_off, lab_col = labels_to_csr(labels, n, ls, e)
        # batch_size = 1: the reference's losses return the un-normalised sum, the caller divides (train.py:745,1042)
        rows = fused.all_entity_loss(scores.q, scores.table, lab_off, lab_col, self.kind, 1, ls, self.offset,
                                     scores.math_mode, kind=scores.kind)
        return rows.sum()


# ---------------------------------------------------------------------------------------------
# adapters: the reference's model / embedder objects seen through the attributes trainer.py reads
# ---------------------------------------------------------------------------------------------
class _EmbedderView:
    def __init__(self, emb):
        self._e = emb
        self.dim = emb.dim
        self.normalize_p = emb.normalize_p
        self.regularize = emb.regularize
        self.dropout = emb.dropout
        self.sparse = emb.sparse
        self.regularize_weight = float(emb.get_option("regularize_weight")) if emb.regularize != "" else 0.0
        self.regularize_weighted = bool(emb.get_option("regularize_args.weighted")) if emb.regularize != "" else False
        self.regularize_p = emb.get_option("regularize_args.p") if emb.regularize == "lp" else 2

    @property
    def weight(self):
        return self._e._embeddings.weight

    def embed_all(self):
        return self._e._embeddings.weight


class _ModelView:
    """A reference KgeModel (plug-in class) as trainer.FusedAllEntityStepper / jobs.EntityRankingJob see a model.
    For the reciprocal relations model (`reciprocal`) the view declares the wrapper (`reciprocal_relations`) and its R =
    the dataset's relation count; the relation table it exposes is the base model's 2 R-row table."""

    def __init__(self, ref_model, base: str, reciprocal: bool = False):
        self.ref, self.model = ref_model, base
        self._ent = _EmbedderView(ref_model.get_s_embedder())
        self._rel = _EmbedderView(ref_model.get_p_embedder())
        self.reciprocal_relations = bool(reciprocal)
        if reciprocal:
            self.num_relations = ref_model.dataset.num_relations()

    def get_s_embedder(self): return self._ent
    def get_o_embedder(self): return self._ent
    def get_p_embedder(self): return self._rel
    def get_scorer(self): return self.ref.get_scorer()._impl


# ---------------------------------------------------------------------------------------------
# level 2: captured step on the job object
# ---------------------------------------------------------------------------------------------
def _install_captured_step(job, model, base: str, loss_kind: int, offset: float, math_mode: int, reciprocal: bool = False):
    from kge.job.train import TrainingJob, TrainingJob1vsAll, TrainingJobKvsAll
    from .trainer import FusedAllEntityStepper, kvsall_rows
    view = _ModelView(model, base, reciprocal)
    inv_rel = view.num_relations if reciprocal else 0         # _po queries -> sp_ rows on relation p + R
    dev = view.get_s_embedder().weight.device
    ref_body = type(job)._process_batch            # the reference's own batch body (other batch sizes)
    state = {"stepper": None}
    label_smoothing = float(getattr(job, "label_smoothing", 0.0) or 0.0)
    is_1vsall = isinstance(job, TrainingJob1vsAll)
    if not (is_1vsall or isinstance(job, TrainingJobKvsAll)):
        raise NotImplementedError("b200.captured_step serves train.type 1vsAll and KvsAll")
    # (job.query_types is set by _prepare AFTER it called model.prepare_job: read the option it is built from, train.py:549-553)
    if not is_1vsall and [k for k, on in job.config.get("KvsAll.query_types").items() if on] != ["sp_", "_po"]:
        raise NotImplementedError("b200.captured_step: KvsAll.query_types must be sp_ and _po (s_o is served by the "
                                  "reference's own path)")

    def stepper_for(rows: int, nnz_max: int):
        st = state["stepper"]
        if st is None:
            st = FusedAllEntityStepper(view, job.optimizer, rows, nnz_max, loss_kind, job.batch_size if not is_1vsall else rows // 2,
                                       offset, label_smoothing, math_mode, use_graph=True,
                                       onevsall_triples=is_1vsall and rows <= 8192, reciprocal=reciprocal)
            state["stepper"] = st
            model._b200_stepper = st
        return st

    def process_batch(self, batch_index, batch):
        t0 = time.time()
        if is_1vsall:
            triples = batch["triples"]
            b = len(triples)
            if b != self.batch_size:
                model._b200_captured_batch = False
                return ref_body(self, batch_index, batch)
            st = stepper_for(2 * b, 2 * b)
            if st.triples is not None:
                # the batch (queries, labels, scatter permutations) is built by the first kernel of the captured step
                st.set_triples(triples if triples.dtype == torch.int64 else triples.long())
            else:
                t = triples.to(dev, non_blocking=True)
                s, p, o = t[:, 0], t[:, 1], t[:, 2]
                zeros = torch.zeros(b, dtype=torch.int32, device=dev)
                st.set_inputs(torch.cat((s, o)), torch.cat((p, p + inv_rel)), torch.cat((zeros, zeros + (0 if inv_rel else 1))),
                              torch.arange(2 * b + 1, dtype=torch.int64, device=dev), torch.cat((o, s)))
            size = b
        else:
            q = batch["queries"]
            size = len(q)
            nnz = len(batch["label_coords"])
            st = state["stepper"]
            if size != self.batch_size or (st is not None and nnz > st.nnz_max):
                model._b200_captured_batch = False
                return ref_body(self, batch_index, batch)
            if st is None:   # label capacity from the first full batch with head room; larger batches take the autograd path
                st = stepper_for(size, max(2 * nnz, 4 * size))
            qd = q.to(dev, non_blocking=True)
            a, p, rc = kvsall_rows(qd, batch["query_type_indexes"].to(dev, non_blocking=True), inv_rel)
            lab_off, lab_col = fused.csr_from_coords(batch["label_coords"].to(dev, non_blocking=True), size)
            st.set_inputs(a, p, rc, lab_off, lab_col)
        prepare = time.time() - t0
        t1 = time.time()
        st.step()
        total, reported = st.report.tolist()          # one D2H read, as train.py:747 / 1043
        model._b200_captured_batch = True
        return TrainingJob._ProcessBatchResult(reported if not is_1vsall else total, size, prepare, time.time() - t1, 0.0)

    job._process_batch = types.MethodType(process_batch, job)


def captured_penalties(model, base_penalty, **kwargs):
    """`model.penalty()` while the captured step is active: its Adagrad kernels applied the (unweighted Lp) penalty
    gradients already and left the values on the device; they are reported as leaf tensors in the order of
    kge_model.py:588-606 (s-embedder, p-embedder, o-embedder) so that the job's `.backward()` / `.item()` lines run."""
    st = getattr(model, "_b200_stepper", None)
    if st is None or not getattr(model, "_b200_captured_batch", False) or st.pen is None:
        return base_penalty(**kwargs)
    ent_v, rel_v = st.penalty_values[0] * 0.5, st.penalty_values[1]
    e_key = f"{model.get_s_embedder().configuration_key}.L{st.pen['ent'][0]}_penalty"
    r_key = f"{model.get_p_embedder().configuration_key}.L{st.pen['rel'][0]}_penalty"
    out = []
    leaf = lambda v: v.detach().clone().requires_grad_(True)   # noqa: E731
    if st.pen["ent"][1] != 0.0:
        out.append((e_key, leaf(ent_v)))
    if st.pen["rel"][1] != 0.0:
        out.append((r_key, leaf(rel_v)))
    if st.pen["ent"][1] != 0.0:
        out.append((e_key, leaf(ent_v)))
    return out


def prepare_training_job(job, model, base: str, options: dict, reciprocal: bool = False):
    """Called from the plug-in model's prepare_job for training jobs (`reciprocal`: from the reciprocal relations model,
    whose base model's own prepare_job must not install anything).  Idempotent."""
    from kge.job.train import TrainingJob1vsAll, TrainingJobKvsAll
    if getattr(job, "_b200_installed", False):
        return
    job._b200_installed = True
    if not isinstance(job, (TrainingJob1vsAll, TrainingJobKvsAll)):
        return                                  # negative sampling: score_spo is the fused gather+score kernel already
    name = job.config.get("train.loss")
    if name not in ("kl", "bce"):
        return
    loss_kind = lib.LOSS_KL if name == "kl" else lib.LOSS_BCE
    offset = float(job.config.get("train.loss_arg")) if name == "bce" else 0.0
    if math.isnan(offset):
        offset = 0.0
    math_mode = MATH_MODES[options.get("math", "fp32")]
    if not isinstance(job.loss, FusedKgeLoss):
        job.loss = FusedKgeLoss(job.loss, job, loss_kind, offset)
    model._b200_lazy_jobs = getattr(model, "_b200_lazy_jobs", 0) + 1
    model._b200_math = math_mode
    if options.get("captured_step", False):
        _install_captured_step(job, model, base, loss_kind, offset, math_mode, reciprocal)


# ---------------------------------------------------------------------------------------------
# level 3: fused evaluation job
# ---------------------------------------------------------------------------------------------
def make_entity_ranking_job(RefEntityRankingJob):
    import kge.job.eval as ref_eval

    def hist_all(hists, s, p, o, s_ranks, o_ranks, job, **kw):
        """eval.py:138-171 without the Python loop per rank."""
        e = job.dataset.num_entities()
        new = lambda: torch.zeros(e, dtype=torch.float32, device=s.device)   # noqa: E731
        h = hists.setdefault("all", new())
        dm.rank_hist(o_ranks, e, h)
        dm.rank_hist(s_ranks, e, h)
        if job.head_and_tail:
            dm.rank_hist(o_ranks, e, hists.setdefault("tail", new()))
            dm.rank_hist(s_ranks, e, hists.setdefault("head", new()))

    def hist_per_relation_type(hists, s, p, o, s_ranks, o_ranks, job, **kw):
        """eval.py:173-198."""
        e = job.dataset.num_entities()
        new = lambda: torch.zeros(e, dtype=torch.float32, device=s.device)   # noqa: E731
        for rel_type, rels in job.dataset.index("relations_per_type").items():
            ids = torch.as_tensor(sorted(int(r) for r in rels), dtype=torch.int64, device=s.device)
            m = dm.isin_sorted(p, ids)
            h = hists.setdefault(rel_type, new())
            dm.rank_hist(o_ranks, e, h, mask=m)
            dm.rank_hist(s_ranks, e, h, mask=m)
            if job.head_and_tail:
                dm.rank_hist(o_ranks, e, hists.setdefault(f"{rel_type}_tail", new()), mask=m)
                dm.rank_hist(s_ranks, e, hists.setdefault(f"{rel_type}_head", new()), mask=m)

    def hist_per_frequency_percentile(hists, s, p, o, s_ranks, o_ranks, job, **kw):
        """eval.py:201-224."""
        e = job.dataset.num_entities()
        new = lambda: torch.zeros(e, dtype=torch.float32, device=s.device)   # noqa: E731
        percs = job.dataset.index("frequency_percentiles")
        as_set = lambda ids: torch.as_tensor(sorted(int(x) for x in ids), dtype=torch.int64, device=s.device)  # noqa: E731
        for arg in percs:
            for perc in percs[arg]:
                hists.setdefault(f"{arg}_{perc}", new())
        for perc in percs["subject"].keys():
            m_s, m_r, m_o = (dm.isin_sorted(x, as_set(percs[a][perc])) for x, a in ((s, "subject"), (p, "relation"), (o, "object")))
            dm.rank_hist(s_ranks, e, hists[f"subject_{perc}"], mask=m_s)
            dm.rank_hist(s_ranks, e, hists[f"relation_{perc}"], mask=m_r)
            dm.rank_hist(o_ranks, e, hists[f"object_{perc}"], mask=m_o)
            dm.rank_hist(o_ranks, e, hists[f"relation_{perc}"], mask=m_r)

    device_hooks = {ref_eval.hist_all: hist_all, ref_eval.hist_per_relation_type: hist_per_relation_type,
                    ref_eval.hist_per_frequency_percentile: hist_per_frequency_percentile}

    class B200EntityRankingJob(RefEntityRankingJob):
        """EntityRankingJob (kge/job/entity_ranking.py) with `_run`'s chunk loop -- score_sp_po, three dense label
        passes, `_filter_and_rank` (entity_ranking.py:150-217, 428-551) -- replaced by the fused score-and-count kernel.
        Loader, hooks, histograms, metric names and trace entries are the reference's.  Models that are not B200
        plug-in models run the reference's own `_run`."""

        def __init__(self, config, dataset, parent_job, model):
            super().__init__(config, dataset, parent_job, model)
            self._b200 = getattr(model, "_b200_base", None) is not None and str(self.device).startswith("cuda")
            if self._b200:
                self.hist_hooks = [device_hooks.get(f, f) for f in self.hist_hooks]
            if self.__class__ == B200EntityRankingJob:
                for f in RefEntityRankingJob.job_created_hooks:
                    f(self)

        def _collate(self, batch):
            if not self._b200:
                return super()._collate(batch)
            # the filter coordinates are looked up on the device (kgeb_filter_csr_*), not by dict lookups per triple
            return torch.cat(batch).reshape((-1, 3)), None, None

        def _b200_indexes(self, split):
            cache = self.__dict__.setdefault("_b200_index_cache", {})
            if split not in cache:
                sp, po = self.dataset.index(f"{split}_sp_to_o"), self.dataset.index(f"{split}_po_to_s")
                cache[split] = (KvsAllIndex.from_arrays(sp._keys, sp._values_offset, sp._values, "sp"),
                                KvsAllIndex.from_arrays(po._keys, po._values_offset, po._values, "po"))
            return cache[split]

        def _compute_metrics(self, rank_hist, suffix=""):
            if not self._b200:
                return super()._compute_metrics(rank_hist, suffix)
            return dm.rank_metrics(rank_hist, self.hits_at_k_s, suffix)

        @torch.no_grad()
        def _run(self) -> dict:
            if not self._b200:
                return super()._run()
            model = self.model
            was_training = model.training
            model.eval()
            self.config.log("Evaluating on " + self.eval_split + " data (epoch {})...".format(self.epoch))
            filter_with_test = "test" not in self.filter_splits and self.filter_with_test
            view = _ModelView(model, model._b200_base, getattr(model, "_b200_reciprocal", False))
            scorer = view.get_scorer()
            math_mode = getattr(model, "_b200_eval_math", lib.MATH_FP32)
            filt_idx = [self._b200_indexes(split) for split in self.filter_splits]
            test_idx = filt_idx + [self._b200_indexes("test")] if filter_with_test else None
            num_rel = self.dataset.num_relations()
            reciprocal = getattr(model, "_b200_reciprocal", False)
            hists, hists_filt, hists_filt_test = dict(), dict(), dict()
            metrics: Dict[str, float] = {}
            epoch_time = -time.time()
            dev = torch.device(self.device)
            for batch_number, batch_coords in enumerate(self.loader):
                batch = batch_coords[0].to(dev).long()
                s, p, o = batch[:, 0].contiguous(), batch[:, 1].contiguous(), batch[:, 2].contiguous()
                b = len(batch)
                o_true = model.score_spo(s, p, o, "o").view(-1)           # entity_ranking.py:139-140
                s_true = model.score_spo(s, p, o, "s").view(-1)
                ent_w, rel_w = view.get_s_embedder().weight, view.get_p_embedder().weight
                q_sp = ops.query_build(view.model, lib.SP_, ops.gather_rows(ent_w, s), ops.gather_rows(rel_w, p))
                if reciprocal:
                    q_po = ops.query_build(view.model, lib.SP_, ops.gather_rows(ent_w, o), ops.gather_rows(rel_w, p + num_rel))
                else:
                    q_po = ops.query_build(view.model, lib._PO, ops.gather_rows(ent_w, o), ops.gather_rows(rel_w, p))
                q = torch.cat((q_sp, q_po)).contiguous()
                filt = filter_csr([a for a, _ in filt_idx], [c for _, c in filt_idx], s, p, o)
                filt_test = filter_csr([a for a, _ in test_idx], [c for _, c in test_idx], s, p, o) if test_idx else None
                m = scorer._math(ent_w) if math_mode == lib.MATH_TF32 else lib.MATH_FP32
                counts = fused.rank_counts(scorer.kind, q, ent_w.detach(), torch.cat((o_true, s_true)).contiguous(),
                                           torch.cat((o, s)).contiguous(), filt, filt_test, m)
                rk = lambda j: self._get_ranks(counts[:, 2 * j], counts[:, 2 * j + 1])     # noqa: E731
                raw, flt = rk(0), rk(1)
                o_ranks, s_ranks, o_ranks_filt, s_ranks_filt = raw[:b], raw[b:], flt[:b], flt[b:]
                batch_hists, batch_hists_filt, batch_hists_filt_test = dict(), dict(), dict()
                for f in self.hist_hooks:
                    f(batch_hists, s, p, o, s_ranks, o_ranks, job=self)
                    f(batch_hists_filt, s, p, o, s_ranks_filt, o_ranks_filt, job=self)
                if filter_with_test:
                    ft = rk(2)
                    o_ranks_filt_test, s_ranks_filt_test = ft[:b], ft[b:]
                    for f in self.hist_hooks:
                        f(batch_hists_filt_test, s, p, o, s_ranks_filt_test, o_ranks_filt_test, job=self)
                if self.trace_examples:
                    entry = {"type": "entity_ranking", "scope": "example", "split": self.eval_split,
                             "filter_splits": self.filter_splits, "size": b, "batches": len(self.loader),
                             "epoch": self.epoch}
                    cols = [x.tolist() for x in (s, p, o, o_ranks, o_ranks_filt, s_ranks, s_ranks_filt)]
                    tcols = [x.tolist() for x in (o_ranks_filt_test, s_ranks_filt_test)] if filter_with_test else None
                    for i in range(b):
                        entry["batch"] = i
                        entry["s"], entry["p"], entry["o"] = cols[0][i], cols[1][i], cols[2][i]
                        if filter_with_test:
                            entry["rank_filtered_with_test"] = tcols[0][i] + 1
                        self.trace(event="example_rank", task="sp", rank=cols[3][i] + 1, rank_filtered=cols[4][i] + 1, **entry)
                        if filter_with_test:
                            entry["rank_filtered_with_test"] = tcols[1][i] + 1
                        self.trace(event="example_rank", task="po", rank=cols[5][i] + 1, rank_filtered=cols[6][i] + 1, **entry)
                if self.trace_batch:
                    metrics = self._compute_metrics(batch_hists["all"])
                    metrics.update(self._compute_metrics(batch_hists_filt["all"], suffix="_filtered"))
                    if filter_with_test:
                        metrics.update(self._compute_metrics(batch_hists_filt_test["all"], suffix="_filtered_with_test"))
                    self.trace(event="batch_completed", type="entity_ranking", scope="batch", split=self.eval_split,
                               filter_splits=self.filter_splits, epoch=self.epoch, batch=batch_number, size=b,
                               batches=len(self.loader), **metrics)
                for target, source in ((hists, batch_hists), (hists_filt, batch_hists_filt),
                                       (hists_filt_test, batch_hists_filt_test)):
                    for key, h in source.items():
                        target[key] = target[key] + h if key in target else h
            metrics = {}
            for key in hists:
                name = "_" + key if key != "all" else ""
                metrics.update(self._compute_metrics(hists[key], suffix=name))
                metrics.update(self._compute_metrics(hists_filt[key], suffix="_filtered" + name))
                if filter_with_test:
                    metrics.update(self._compute_metrics(hists_filt_test[key], suffix="_filtered_with_test" + name))
            epoch_time += time.time()
            trace_entry = dict(type="entity_ranking", scope="epoch", split=self.eval_split, filter_splits=self.filter_splits,
                               epoch=self.epoch, batches=len(self.loader), size=len(self.triples), epoch_time=epoch_time,
                               event="eval_completed", **metrics)
            for f in self.post_epoch_trace_hooks:
                f(self, trace_entry)
            metric_name = self.config.get("valid.metric")
            if metric_name not in trace_entry:
                trace_entry[metric_name] = eval(self.config.get("valid.metric_expr"), None,
                                                dict(config=self.config, **trace_entry))
            trace_entry = self.trace(**trace_entry, echo=True, echo_prefix="  ", log=True)
            if was_training:
                model.train()
            self.config.log("Finished evaluating on " + self.eval_split + " split.")
            for f in self.post_valid_hooks:
                f(self, trace_entry)
            return trace_entry

    B200EntityRankingJob.__name__ = B200EntityRankingJob.__qualname__ = "EntityRankingJob"
    return B200EntityRankingJob


def register_jobs():
    """Rebinds kge.job.EntityRankingJob (looked up at call time by EvaluationJob.create, eval.py:75-79) and registers the
    kernel-backed optimizers under torch.optim (KgeOptimizer.create, optimizer.py:10-17).  Idempotent."""
    import kge.job as kj
    from . import optim
    if not getattr(kj, "_b200_jobs_registered", False):
        ref_cls = kj.EntityRankingJob
        kj.RefEntityRankingJob = ref_cls
        kj.EntityRankingJob = make_entity_ranking_job(ref_cls)
        import kge.job.entity_ranking as er
        er.B200EntityRankingJob = kj.EntityRankingJob
        kj._b200_jobs_registered = True
    if not hasattr(torch.optim, "B200Adagrad"):
        torch.optim.B200Adagrad = optim.Adagrad
        torch.optim.B200Adam = optim.Adam
