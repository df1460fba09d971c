"""Batch bodies of the reference's training jobs and the entity-ranking evaluation, on top of the
CUDA path.  Two forms of each:

* the reference's own flow (`fused=False`): `model.score_sp/po/spo` -> `loss(scores, labels) / batch_size`
  -> `.backward()`, line for line as kge/job/train.py:679-756, 823-999, 1032-1062 -- this is what the
  unmodified reference jobs execute when the drop-in model classes are registered (INTEGRATION.md);
* the fused flow (`fused=True`): query vectors -> fused score+loss kernels; the [B,E] matrix is never
  materialised, both 1vsAll directions / both KvsAll query types go through one launch.
Evaluation (`EntityRankingJob`) follows kge/job/entity_ranking.py:79-426 with the chunk loop and the
three dense filter passes replaced by the fused score-and-count kernel.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence

import torch
import torch.nn.functional as F

from . import fused, lib, ops
from .index import KvsAllIndex, filter_csr, gather_csr_rows, merge_sorted_csr
from .model import KgeModel, ReciprocalRelationsModel

S, P, O = 0, 1, 2


# ---------------------------------------------------------------------------------------------
# losses on materialised scores (kge/util/loss.py:137-159, 192-213)
# ---------------------------------------------------------------------------------------------
class KgeLoss:
    def __init__(self, name: str, offset: float = 0.0):
        if name not in ("kl", "bce"):
            raise ValueError(f"train.loss={name} is not on the hot path (built: kl, bce)")
        self.name = name
        self.offset = 0.0 if (offset is None or (isinstance(offset, float) and math.isnan(offset))) else float(offset)
        self.kind = lib.LOSS_KL if name == "kl" else lib.LOSS_BCE

    @staticmethod
    def create(name: str, loss_arg: float = float("nan")) -> "KgeLoss":
        return KgeLoss(name, loss_arg)

    def __call__(self, scores, labels, **kwargs):
        if self.name == "kl":
            if labels.dim() == 1:
                return F.cross_entropy(scores, labels.long(), reduction="sum")
            return F.kl_div(F.log_softmax(scores, dim=1), F.normalize(labels.float(), p=1, dim=1), reduction="sum")
        if labels.dim() == 1:
            m = torch.zeros(scores.shape, device=scores.device, dtype=torch.float)
            m[torch.arange(len(scores), device=scores.device), labels.long()] = 1.0
            labels = m
        if self.offset != 0.0:
            scores = scores + self.offset
        return F.binary_cross_entropy_with_logits(scores.reshape(-1), labels.reshape(-1), reduction="sum")


class ProcessBatchResult:
    def __init__(self, avg_loss, size, total_loss=None):
        self.avg_loss, self.size = avg_loss, size
        self.total_loss = avg_loss if total_loss is None else total_loss


# ---------------------------------------------------------------------------------------------
# training jobs
# ---------------------------------------------------------------------------------------------
class TrainingJob:
    """run_epoch's step skeleton (train.py:309-376): zero_grad -> batch -> penalties -> optimizer.step."""

    def __init__(self, model: KgeModel, optimizer, loss: KgeLoss, fused_path: bool = True,
                 math_mode: int = lib.MATH_FP32, shard: Optional[fused.Shard] = None):
        self.model, self.optimizer, self.loss = model, optimizer, loss
        self.fused_path, self.math_mode, self.shard = fused_path, math_mode, shard
        self.device = model.get_s_embedder().weight.device
        self.pre_batch_hooks: List = []
        self.abort_on_nan = True          # train.abort_on_nan (config-default.yaml:211)
        model.prepare_job(self)

    def _check_cost(self, res: "ProcessBatchResult") -> "ProcessBatchResult":
        """train.py:341-345: cost = batch loss + penalties; a NaN cost aborts the job (before optimizer.step() on the
        autograd path; the captured steps have applied their update by the time the loss is read back)."""
        cost = res.avg_loss + getattr(res, "penalty", 0.0)
        if self.abort_on_nan and math.isnan(cost):
            raise FloatingPointError("Cost became nan, aborting training job")
        return res

    def step(self, batch_index: int, batch: dict) -> ProcessBatchResult:
        for f in self.pre_batch_hooks:
            f(self)
        self.optimizer.zero_grad()
        res = self._process_batch(batch_index, batch)
        penalty = 0.0
        for _, value in self.model.penalty(batch=batch):
            value.backward()
            penalty += value.item()
        res.penalty = penalty
        self._check_cost(res)
        self.optimizer.step()
        return res

    def _use_fused(self) -> bool:
        """Fused score + loss kernels: every pair kind (DOT scorers, TransE, RotatE) up to d = 256."""
        return self.fused_path and self.model.get_s_embedder().dim <= 256


class TrainingJob1vsAll(TrainingJob):
    def _process_batch(self, batch_index, batch) -> ProcessBatchResult:
        triples = batch["triples"].to(self.device)
        b = len(triples)
        if self._use_fused():
            # both directions as 2B queries in one launch (gradients accumulate before one step, train.py:375)
            if isinstance(self.model, ReciprocalRelationsModel):
                q_po = self.model.queries(lib.SP_, triples[:, 2], triples[:, 1] + self.model.num_relations)
            else:
                q_po = self.model.queries(lib._PO, triples[:, 2], triples[:, 1])
            q = torch.cat((self.model.queries(lib.SP_, triples[:, 0], triples[:, 1]), q_po))
            lab_off = torch.arange(2 * b + 1, dtype=torch.int64, device=self.device)
            lab_col = torch.cat((triples[:, 2], triples[:, 0])).long().contiguous()
            rows = fused.all_entity_loss(q, self.model.get_o_embedder().embed_all(), lab_off, lab_col,
                                         self.loss.kind, b, 0.0, self.loss.offset, self.math_mode, self.shard,
                                         kind=self.model.get_scorer().kind)
            loss_value = rows.sum()
            loss_value.backward()
            return ProcessBatchResult(loss_value.item(), b)
        scores_sp = self.model.score_sp(triples[:, 0], triples[:, 1])
        loss_value_sp = self.loss(scores_sp, triples[:, 2]) / b
        loss_value = loss_value_sp.item()
        loss_value_sp.backward()
        scores_po = self.model.score_po(triples[:, 1], triples[:, 2])
        loss_value_po = self.loss(scores_po, triples[:, 0]) / b
        loss_value += loss_value_po.item()
        loss_value_po.backward()
        return ProcessBatchResult(loss_value, b)


class TrainingJobKvsAll(TrainingJob):
    """Query types sp_ and _po (config-default.yaml KvsAll.query_types; s_o stays on the reference's own path)."""

    def __init__(self, model, optimizer, loss, num_entities: int, num_relations: int, label_smoothing: float = 0.0,
                 **kw):
        super().__init__(model, optimizer, loss, **kw)
        self.num_entities, self.num_relations = num_entities, num_relations
        self.label_smoothing = label_smoothing
        self.stepper = None

    # -- static-shape, graph-captured step (trainer.py) ---------------------------------------------------
    def enable_graph_step(self, batch_size: int, nnz_max: int, use_graph: bool = True, dp_group=None,
                          dp_p2p: bool = False):
        """Routes step() through FusedAllEntityStepper for batches of exactly `batch_size` queries with at most
        `nnz_max` labels (no autograd, one CUDA-graph replay per step).  Needs dense Adagrad (TransE / RotatE: one GPU);
        unweighted Lp penalties are folded into the Adagrad kernels (the toy config's regularize_weight)."""
        from .trainer import FusedAllEntityStepper
        if any(e.normalize_p > 0 for e in (self.model.get_s_embedder(), self.model.get_p_embedder())):
            # the hook of lookup_embedder.py:58-75 REPLACES the weight tensor every batch; the captured step reads fixed
            # addresses
            raise NotImplementedError("per-batch renormalisation (normalize_p) is served by the autograd path only")
        self.stepper = FusedAllEntityStepper(self.model, self.optimizer, batch_size, nnz_max, self.loss.kind,
                                             batch_size, self.loss.offset, self.label_smoothing, self.math_mode,
                                             use_graph, self.shard, dp_group, dp_p2p,
                                             reciprocal=isinstance(self.model, ReciprocalRelationsModel))
        return self.stepper

    def _inv_rel(self) -> int:
        """R for a reciprocal relations model (its _po queries become sp_ rows on relation p + R), else 0."""
        return self.model.num_relations if isinstance(self.model, ReciprocalRelationsModel) else 0

    # -- on-device batch construction (SURVEY.md 8f-1): the host sends example ids only ----------------------------
    def enable_device_collate(self, sp_index: KvsAllIndex, po_index: KvsAllIndex):
        """KvsAll batches are built on the device from the device-resident indexes (kgeb_kvsall_batch_*, three stable
        sorts for the scatter permutations) on a collate stream, double-buffered so that batch i+1 is built while step
        i runs; step_ids() then costs one 8*B-byte H2D copy and one small D2D copy on top of the graph replay."""
        st = self.stepper
        if st is None:
            raise RuntimeError("enable_graph_step() first")
        dev = self.device
        self._dc = {"sp": sp_index, "po": po_index, "stream": torch.cuda.Stream(device=dev), "slot": 0, "pending": [],
                    "staging": [torch.zeros_like(st.input_bytes) for _ in range(2)],
                    "ids": [torch.zeros(st.rows, dtype=torch.int64, device=dev) for _ in range(2)],
                    "overflow": [torch.zeros(1, dtype=torch.int32, device=dev) for _ in range(2)],
                    "built": [torch.cuda.Event() for _ in range(2)], "consumed": [torch.cuda.Event() for _ in range(2)],
                    "descs": (lib.index_descs([sp_index.device_arrays(dev)]), lib.index_descs([po_index.device_arrays(dev)])),
                    "ws": torch.empty(lib.load().kgeb_kvsall_build_workspace_bytes(st.rows, max(st.nnz_max, 1)),
                                      dtype=torch.uint8, device=dev)}
        for ev in self._dc["consumed"]:
            ev.record()
        # one CUDA graph per staging slot: the build is ~25 small launches (CUB scan / radix sorts), far more host time
        # than device time when issued one by one
        dc = self._dc
        dc["graphs"] = []
        cs = dc["stream"]
        cs.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(cs):
            for slot in range(2):
                self._build_batch(slot)          # warm-up outside capture
        cs.synchronize()
        for slot in range(2):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=cs):
                self._build_batch(slot)
            dc["graphs"].append(g)
        torch.cuda.synchronize()

    def _build_batch(self, slot: int):
        dc, st = self._dc, self.stepper
        v = st.input_views(dc["staging"][slot])
        lib.call("kgeb_kvsall_batch_build_inv", dc["descs"][0], dc["descs"][1], dc["ids"][slot].data_ptr(), st.rows,
                 max(st.nnz_max, 1), self.num_entities, self.num_relations, v["a_idx"].data_ptr(), v["p_idx"].data_ptr(),
                 v["row_combine"].data_ptr(), v["lab_off"].data_ptr(), v["lab_col"].data_ptr(), v["a_perm"].data_ptr(),
                 v["p_perm"].data_ptr(), v["lab_perm"].data_ptr(), dc["overflow"][slot].data_ptr(),
                 dc["ws"].data_ptr(), dc["ws"].numel(), self._inv_rel(), torch.cuda.current_stream().cuda_stream)

    def prefetch_ids(self, example_ids: torch.Tensor):
        """Enqueues the construction of the batch with these example ids (host pinned or device int64 [batch_size])."""
        dc = self._dc
        if len(dc["pending"]) >= 2:
            raise RuntimeError("two batches are already in flight")
        slot = dc["slot"]
        dc["slot"] ^= 1
        cs = dc["stream"]
        with torch.cuda.stream(cs):
            cs.wait_event(dc["consumed"][slot])          # the step that used this staging buffer has copied it
            dc["ids"][slot].copy_(example_ids, non_blocking=True)
            dc["graphs"][slot].replay()
            dc["built"][slot].record(cs)
        dc["pending"].append(slot)

    def step_ids(self, example_ids: Optional[torch.Tensor] = None) -> ProcessBatchResult:
        """One training step on the oldest prefetched batch (or on `example_ids`, built now)."""
        dc, st = self._dc, self.stepper
        if example_ids is not None:
            self.prefetch_ids(example_ids)
        slot = dc["pending"].pop(0)
        for f in self.pre_batch_hooks:
            f(self)
        cur = torch.cuda.current_stream()
        cur.wait_event(dc["built"][slot])
        st.input_bytes.copy_(dc["staging"][slot], non_blocking=True)
        dc["consumed"][slot].record(cur)
        loss = st.step()
        total, reported, overflow = torch.cat((st.report, dc["overflow"][slot].float())).tolist()   # one D2H read, as train.py:747
        if overflow:
            raise ValueError(f"batch has more than {st.nnz_max} labels (enable_graph_step(nnz_max=...))")
        return self._check_cost(ProcessBatchResult(reported, st.rows, total))

    def device_inputs(self, batch):
        """Host (pinned) KvsAll batch -> device tensors (a_idx, p_idx, row_combine, lab_off, lab_col, perms)."""
        from .trainer import kvsall_rows
        q = batch["queries"].to(self.device, non_blocking=True)
        qt = batch["query_type_indexes"].to(self.device, non_blocking=True)
        coords = batch["label_coords"].to(self.device, non_blocking=True)
        a, p, rc = kvsall_rows(q, qt, self._inv_rel())
        lab_off, lab_col = fused.csr_from_coords(coords, len(q))
        return a, p, rc, lab_off, lab_col, self.stepper.batch_perms(a, p, lab_col)

    def collate_packed(self, batch: dict) -> dict:
        """Host-side collate for the graph-captured step (what a DataLoader worker does instead of train.py:590-677's
        tensors): query rows, per-row combine flags and the label CSR laid out in one pinned buffer."""
        from .trainer import kvsall_rows
        q, qt = batch["queries"], batch["query_type_indexes"]
        a, p, rc = kvsall_rows(q, qt, self._inv_rel())
        lab_off, lab_col = fused.csr_from_coords(batch["label_coords"], len(q))
        return {"packed": self.stepper.pack_host_batch(a, p, rc, lab_off, lab_col), "size": len(q)}

    def prefetch_packed(self, batch: dict):
        """Starts the H2D copy of a packed (pinned) batch on a copy stream into one of two device staging buffers, so
        that it runs underneath the step in flight -- what pinned DataLoader batches with non_blocking copies give the
        reference's loop.  step() recognises the batch and takes it from the staging buffer (one D2D copy)."""
        st = self.stepper
        pf = getattr(self, "_pf", None)
        if pf is None:
            dev = st.input_bytes.device
            pf = self._pf = dict(stream=torch.cuda.Stream(device=dev), staging=[torch.empty_like(st.input_bytes) for _ in range(2)],
                                 ready=[torch.cuda.Event(), torch.cuda.Event()],
                                 consumed=[torch.cuda.Event(), torch.cuda.Event()], slot=0, pending=[])
            for ev in pf["consumed"]:
                ev.record()
        if len(pf["pending"]) >= 2:
            raise RuntimeError("two batches are already in flight")
        slot = pf["slot"]
        pf["slot"] ^= 1
        cs = pf["stream"]
        with torch.cuda.stream(cs):
            cs.wait_event(pf["consumed"][slot])          # the step that used this staging buffer has copied it
            pf["staging"][slot].copy_(batch["packed"], non_blocking=True)
            pf["ready"][slot].record(cs)
        pf["pending"].append((batch["packed"].data_ptr(), slot))

    def step(self, batch_index: int, batch: dict) -> ProcessBatchResult:
        size = batch["size"] if "packed" in batch else len(batch["queries"])
        if self.stepper is None or size != self.stepper.rows:
            return super().step(batch_index, batch)
        for f in self.pre_batch_hooks:
            f(self)
        pf = getattr(self, "_pf", None)
        if "packed" in batch and pf is not None and pf["pending"] and pf["pending"][0][0] == batch["packed"].data_ptr():
            _, slot = pf["pending"].pop(0)
            cur = torch.cuda.current_stream()
            cur.wait_event(pf["ready"][slot])
            self.stepper.input_bytes.copy_(pf["staging"][slot], non_blocking=True)
            pf["consumed"][slot].record(cur)
        elif "packed" in batch:
            self.stepper.set_packed(batch["packed"])
        else:
            self.stepper.set_inputs(*self.device_inputs(batch))
        loss = self.stepper.step()
        if self.stepper.p2p is None and self.stepper.dp_world == 1:
            # one D2H read, as train.py:747; avg_loss = value of the last non-empty query type (the reference overwrites
            # it per type), total_loss = what was back-propagated
            total, reported = self.stepper.report.tolist()
        elif self.stepper.p2p is not None:
            # the peer-memory barriers' timeout flag rides along with the loss read-back (one D2H)
            total, timed_out = torch.stack((loss, self.stepper.p2p_timeout[0].float())).tolist()
            if timed_out:
                raise RuntimeError("a peer did not arrive at a peer-memory barrier; the update of this step was skipped")
            reported = total
        else:
            total = reported = loss.item()
        res = ProcessBatchResult(reported, self.stepper.rows, total)
        if self.stepper.pen is not None:
            res.penalty = float(self.stepper.penalty_values.sum().item())   # train.py:320-338 (sum of the terms)
        return self._check_cost(res)

    def _process_batch(self, batch_index, batch) -> ProcessBatchResult:
        queries = batch["queries"].to(self.device)
        b = len(queries)
        coords = batch["label_coords"].to(self.device)
        qt = batch["query_type_indexes"]  # stays on the host, as in train.py:685
        rows_of = [(qt == t).nonzero().view(-1) for t in (0, 1)]
        if self._use_fused() and not (self.loss.kind == lib.LOSS_KL and self.label_smoothing > 0):
            order = torch.cat(rows_of).to(self.device)                 # fused row order: sp_ rows then _po rows
            n_sp = len(rows_of[0])
            inv = torch.empty_like(order)
            inv[order] = torch.arange(b, device=self.device)
            lab_off, lab_col = fused.csr_from_coords(torch.stack((inv[coords[:, 0].long()], coords[:, 1].long()), 1), b)
            qs = queries[order]
            parts = []
            if n_sp > 0:
                parts.append(self.model.queries(lib.SP_, qs[:n_sp, 0], qs[:n_sp, 1]))
            if n_sp < b:
                if isinstance(self.model, ReciprocalRelationsModel):
                    parts.append(self.model.queries(lib.SP_, qs[n_sp:, 1], qs[n_sp:, 0] + self.model.num_relations))
                else:
                    parts.append(self.model.queries(lib._PO, qs[n_sp:, 1], qs[n_sp:, 0]))
            q = torch.cat(parts) if len(parts) > 1 else parts[0]
            rows = fused.all_entity_loss(q, self.model.get_o_embedder().embed_all(), lab_off, lab_col, self.loss.kind,
                                         b, self.label_smoothing, self.loss.offset, self.math_mode, self.shard,
                                         kind=self.model.get_scorer().kind)
            total = rows.sum()
            total.backward()
            # train.py:747 reports the value of the last non-empty query type only
            reported = rows[n_sp:].sum() if n_sp < b else rows.sum()
            return ProcessBatchResult(reported.item(), b, total.item())

        labels = torch.zeros(b, max(self.num_entities, self.num_relations), device=self.device)
        labels.index_put_((coords[:, 0].long(), coords[:, 1].long()),
                          torch.ones(len(coords), device=self.device), accumulate=True)
        reported, total = 0.0, 0.0
        for t, rows in enumerate(rows_of):
            if len(rows) == 0:
                continue
            rows = rows.to(self.device)
            lab = labels[rows, : self.num_entities]
            if self.label_smoothing > 0.0:
                lab = (1.0 - self.label_smoothing) * lab + 1.0 / lab.size(1)
            if t == 0:
                scores = self.model.score_sp(queries[rows, 0], queries[rows, 1])
            else:
                scores = self.model.score_po(queries[rows, 0], queries[rows, 1])
            loss_value = self.loss(scores, lab) / b
            reported = loss_value.item()
            total += reported
            loss_value.backward()
        return ProcessBatchResult(reported, b, total)


class TrainingJobNegativeSampling(TrainingJob):
    """train.py:823-999.  fused: each positive's query vector is built once and scored against its
    1+N candidates (no B*(1+N) triple expansion); otherwise implementation "triple" as in the reference."""

    stepper = None

    def enable_graph_step(self, batch_size: int, num_neg_s: int, num_neg_o: int, use_graph: bool = True, dp_group=None,
                          segment_bwd: bool = False, fused_slot: bool = True, deterministic: bool = True):
        """Routes step() through FusedNegSamplingStepper (no autograd, one CUDA-graph replay per step) for batches of
        exactly `batch_size` triples with these negative counts for the S and O slots (no relation negatives).
        `dp_group`: data-parallel replicas with the peer-memory gradient exchange (trainer.PeerExchange)."""
        from .trainer import FusedNegSamplingStepper
        self.stepper = FusedNegSamplingStepper(self.model, self.optimizer, batch_size, num_neg_s, num_neg_o,
                                               self.loss.kind, self.loss.offset, use_graph, dp_group, segment_bwd,
                                               fused_slot, deterministic,
                                               reciprocal=isinstance(self.model, ReciprocalRelationsModel))
        return self.stepper

    def enable_device_sampling(self, sampler):
        """Negatives are drawn on the device (sampler.KgeSampler, SURVEY.md 8f-2) straight into the static inputs of
        the captured step: the host then ships only the positive triples (24 B each) -- see step_triples()."""
        if self.stepper is None:
            raise ValueError("enable_graph_step() first")
        self.sampler = sampler
        return sampler

    def step_triples(self, triples: torch.Tensor) -> ProcessBatchResult:
        """One step from positive triples alone ([B,3] int64, host or device): H2D copy, on-device sampling of the S
        and O negatives (train.py:801-821 does this on the CPU in the collate), graph replay."""
        st = self.stepper
        if len(triples) != st.B:
            raise ValueError(f"the captured step serves batches of exactly {st.B} triples")
        for f in self.pre_batch_hooks:
            f(self)
        t = triples.to(self.device, non_blocking=True).long()
        st.triples.copy_(t.t(), non_blocking=True)
        for slot in st.slots:
            self.sampler.sample(t, slot, out=st.neg[slot])
        value = st.step().item()
        return self._check_cost(ProcessBatchResult(value, st.B))

    def step(self, batch_index: int, batch: dict) -> ProcessBatchResult:
        st = self.stepper
        negs = batch["negative_samples"]
        if (st is None or len(batch["triples"]) != st.B or (negs[1].dim() == 2 and negs[1].shape[1] > 0)
                or any(negs[s].shape[1] != st.N[s] for s in (0, 2))):
            return super().step(batch_index, batch)
        for f in self.pre_batch_hooks:
            f(self)
        st.set_inputs(batch["triples"], negs)
        loss = st.step()
        if st.px is not None:
            value, timed_out = torch.stack((loss, st.px.timeout[0].float())).tolist()
            if timed_out:
                raise RuntimeError("a peer did not arrive at a peer-memory barrier; the update of this step was skipped")
        else:
            value = loss.item()
        return self._check_cost(ProcessBatchResult(value, st.B))

    def _process_batch(self, batch_index, batch) -> ProcessBatchResult:
        triples = batch["triples"].to(self.device)
        negs = [ns.to(self.device) for ns in batch["negative_samples"]]
        b = len(triples)
        total = 0.0
        for slot in (S, P, O):
            n = negs[slot].shape[1] if negs[slot].dim() == 2 else 0
            if n <= 0:
                continue
            labels = torch.zeros(b, 1 + n, device=self.device)
            labels[:, 0] = 1
            if self.fused_path and slot != P and not isinstance(self.model, ReciprocalRelationsModel):
                if slot == O:
                    q = self.model.queries(lib.SP_, triples[:, S], triples[:, P])
                else:
                    q = self.model.queries(lib._PO, triples[:, O], triples[:, P])
                cand = torch.cat((triples[:, [slot]], negs[slot].long()), 1).contiguous()
                emb = self.model.get_o_embedder()
                scores = ops.pairs_score(self.model.get_scorer().kind, q, emb.embed_all(), cand, emb.sparse)
            else:
                rep = triples.repeat(1, 1 + n).view(-1, 3)
                rep[:, slot] = torch.cat((triples[:, [slot]], negs[slot].long()), 1).view(-1)
                scores = self.model.score_spo(rep[:, 0], rep[:, 1], rep[:, 2],
                                              direction="s" if slot == S else ("o" if slot == O else "p")).view(b, -1)
            loss_value = self.loss(scores, labels, num_negatives=n) / b
            total += loss_value.item()
            loss_value.backward()
        return ProcessBatchResult(total, b)


# ---------------------------------------------------------------------------------------------
# evaluation
# ---------------------------------------------------------------------------------------------
class EntityRankingJob:
    """Filtered entity ranking (kge/job/entity_ranking.py), fused score-and-count form."""

    def __init__(self, model: KgeModel, num_entities: int, filter_splits: Sequence, test_split=None,
                 batch_size: int = 100, tie_handling: str = "rounded_mean_rank", hits_at_k_s=(1, 3, 10, 50, 100, 200, 300, 400, 500, 1000),
                 math_mode: int = lib.MATH_FP32, shard: Optional[fused.Shard] = None):
        if tie_handling not in ("rounded_mean_rank", "best_rank", "worst_rank"):
            raise ValueError(f"entity_ranking.tie_handling={tie_handling}")
        self.model, self.num_entities = model, num_entities
        self.batch_size, self.tie_handling = batch_size, tie_handling
        self.hits_at_k_s = [k for k in hits_at_k_s if k <= num_entities]  # eval.py:19-24
        self.math_mode, self.shard = math_mode, shard
        self.device = model.get_s_embedder().weight.device
        # _prepare (entity_ranking.py:27-51): sp->o and po->s indexes per filter split (+ test)
        self.filter_indexes = [(KvsAllIndex(t, "sp"), KvsAllIndex(t, "po")) for t in filter_splits]
        self.test_indexes = (KvsAllIndex(test_split, "sp"), KvsAllIndex(test_split, "po")) if test_split is not None else None

    def _filter_csr(self, indexes, s, p, o):
        """Device-side replacement of _collate / get_sp_po_coords_from_spo_batch (job/util.py:5-38): one merged CSR
        over the given (sp, po) index pairs; rows 0..B-1 = known objects of (s,p); rows B..2B-1 = known subjects of (p,o)."""
        return filter_csr([sp for sp, _ in indexes], [po for _, po in indexes], s, p, o)

    def _get_ranks(self, rank, ties):
        if self.tie_handling == "rounded_mean_rank":
            return rank + ties // 2
        if self.tie_handling == "best_rank":
            return rank
        return rank + ties - 1

    @torch.no_grad()
    def rank_batch(self, batch: torch.Tensor) -> Dict[str, torch.Tensor]:
        """One batch [B,3] -> 0-based ranks per name s_raw, o_raw, s_filt, o_filt (, s_filt_test, o_filt_test)."""
        model = self.model
        t = batch.to(self.device).long()
        s, p, o = t[:, 0].contiguous(), t[:, 1].contiguous(), t[:, 2].contiguous()
        b = len(t)
        o_true = model.score_spo(s, p, o, "o").view(-1)   # entity_ranking.py:139-140
        s_true = model.score_spo(s, p, o, "s").view(-1)
        if isinstance(model, ReciprocalRelationsModel):
            q_po = model.queries(lib.SP_, o, p + model.num_relations)
        else:
            q_po = model.queries(lib._PO, o, p)
        q = torch.cat((model.queries(lib.SP_, s, p), q_po)).contiguous()
        true_ent = torch.cat((o, s)).contiguous()
        true_score = torch.cat((o_true, s_true)).contiguous()
        filt = self._filter_csr(self.filter_indexes, s, p, o) if self.filter_indexes else None
        filt_test = None
        if self.test_indexes is not None:
            filt_test = self._filter_csr(list(self.filter_indexes) + [self.test_indexes], s, p, o)
        scorer = model.get_scorer()
        table = model.get_o_embedder().embed_all()
        if self.shard is not None:  # this rank scores its own entity rows; counts are all-reduced (exact integers)
            table = table[self.shard.e_lo:self.shard.e_hi]
        counts = fused.rank_counts(scorer.kind, q, table, true_score, true_ent, filt, filt_test,
                                   scorer._math(table) if self.math_mode == lib.MATH_TF32 else lib.MATH_FP32,
                                   self.shard)
        out = {}
        for j, name in enumerate(("_raw", "_filt", "_filt_test")):
            if name == "_filt_test" and filt_test is None:
                continue
            ranks = self._get_ranks(counts[:, 2 * j], counts[:, 2 * j + 1])
            out["o" + name], out["s" + name] = ranks[:b], ranks[b:]
        return out

    def _compute_metrics(self, hist: torch.Tensor, suffix="") -> Dict[str, float]:
        """entity_ranking.py:553-577, reduced on the device (csrc/metrics.cu)."""
        from . import metrics as dm
        return dm.rank_metrics(hist, self.hits_at_k_s, suffix)

    @torch.no_grad()
    def run(self, triples, head_and_tail: bool = False,
            relations_per_type: Optional[Dict[str, Sequence[int]]] = None,
            frequency_percentiles: Optional[Dict[str, Dict[str, Sequence[int]]]] = None) -> Dict[str, object]:
        """Ranks every triple and reduces the ranks to histograms + metrics on the device.  `head_and_tail` adds the
        "head" / "tail" histograms of eval.py:151-171, `relations_per_type` ({type: relation ids}) the drill-down of
        hist_per_relation_type (eval.py:173-198), `frequency_percentiles` ({"subject" | "relation" | "object": {perc:
        ids}}, index.frequency_percentiles) that of hist_per_frequency_percentile (eval.py:201-224); metric names follow
        entity_ranking.py:370-381 ("mean_rank_filtered_head", "hits_at_10_1-N_tail", "hits_at_1_subject_25%", ...)."""
        from . import metrics as dm
        was_training = self.model.training
        self.model.eval()
        triples = torch.as_tensor(triples)
        names = ["_raw", "_filt"] + (["_filt_test"] if self.test_indexes is not None else [])
        E = self.num_entities
        zeros = lambda: torch.zeros(E, dtype=torch.float32, device=self.device)  # noqa: E731
        hists = {n: {"all": zeros()} for n in names}
        rel_sets = {t: torch.as_tensor(sorted(set(int(r) for r in rels)), dtype=torch.int64, device=self.device)
                    for t, rels in (relations_per_type or {}).items()}
        as_set = lambda ids: torch.as_tensor(sorted(set(int(x) for x in ids)), dtype=torch.int64, device=self.device)  # noqa: E731
        freq_sets = {arg: {perc: as_set(ids) for perc, ids in percs.items()}
                     for arg, percs in (frequency_percentiles or {}).items()}
        status = torch.zeros(1, dtype=torch.int32, device=self.device)
        all_ranks: Dict[str, List[torch.Tensor]] = {}
        for lo in range(0, len(triples), self.batch_size):
            batch = triples[lo:lo + self.batch_size]
            res = self.rank_batch(batch)
            masks = {t: dm.isin_sorted(batch[:, P].to(self.device), rs) for t, rs in rel_sets.items()}
            # eval.py:201-224: subject ranks count for the subject's percentile, object ranks for the object's, both for
            # the relation's
            fmask = {(arg, perc): dm.isin_sorted(batch[:, {"subject": S, "relation": P, "object": O}[arg]].to(self.device), ids)
                     for arg, percs in freq_sets.items() for perc, ids in percs.items()}
            for k, v in res.items():
                all_ranks.setdefault(k, []).append(v)
                side, name = k[0], k[1:]               # "o_raw" -> tail ranks of the raw setting
                h = hists[name]
                # hist_all (eval.py:138-171): one kernel per histogram instead of the Python loop over ranks
                dm.rank_hist(v, E, h["all"], status=status)
                if head_and_tail:
                    dm.rank_hist(v, E, h.setdefault("tail" if side == "o" else "head", zeros()), status=status)
                for (arg, perc), m in fmask.items():
                    if arg == "relation" or arg == ("object" if side == "o" else "subject"):
                        dm.rank_hist(v, E, h.setdefault(f"{arg}_{perc}", zeros()), mask=m, status=status)
                for t, m in masks.items():
                    dm.rank_hist(v, E, h.setdefault(t, zeros()), mask=m, status=status)
                    if head_and_tail:
                        dm.rank_hist(v, E, h.setdefault(f"{t}_{'tail' if side == 'o' else 'head'}", zeros()), mask=m,
                                     status=status)
        if int(status.item()) != 0:
            raise RuntimeError("a rank outside [0, num_entities) reached the histogram")
        suffix = {"_raw": "", "_filt": "_filtered", "_filt_test": "_filtered_with_test"}
        metrics = {}
        for n in names:
            for key, h in hists[n].items():      # entity_ranking.py:370-381: "<metric><suffix>[_<group>]"
                metrics.update(self._compute_metrics(h, suffix[n] + ("" if key == "all" else "_" + key)))
        if was_training:
            self.model.train()
        self.hists = hists
        return {"metrics": metrics, "ranks": {k: torch.cat(v) for k, v in all_ranks.items()}}
