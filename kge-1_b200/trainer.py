"""Static-shape fused training step for the all-entity jobs (1vsAll, KvsAll) of the DOT scorers.

One step = the reference's run_epoch body for one batch (train.py:309-376 with _process_batch of
train.py:679-756 / 1032-1062) without autograd and without host round trips:

    gather + query transform -> fused score+loss statistics -> loss -> fused backward (dQ, dense table
    gradient) -> query-transform backward -> sorted scatter of the query-side rows -> Adagrad on both tables

Every buffer has a fixed address and size (rows, nnz_max), so the whole step can be replayed as one CUDA
graph; the per-batch inputs are copied into the static input buffers before each replay.
"""
from __future__ import annotations

from typing import Optional

import os

import torch

from . import fused, lib, ops, optim
from .model import KgeModel


def p2p_slice(numel: int, world: int, rank: int):
    """[lo, hi) of a table's elements that `rank` owns in the peer-memory exchange (csrc/p2p.cu, slice_of): equal
    slices whose bounds are multiples of 4 elements (float4 accesses), the last ones possibly short or empty."""
    per = ((numel + 4 * world - 1) // (4 * world)) * 4
    lo = min(numel, per * rank)
    return lo, min(numel, lo + per)


def gather_owner_slices(flat: torch.Tensor, group) -> torch.Tensor:
    """Every rank broadcasts the slice of `flat` it owns in the peer-memory exchange (p2p_slice): afterwards all ranks hold
    the owners' values everywhere.  Used for the optimizer state, which that mode updates on the owner only."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    ranks = dist.get_process_group_ranks(group)
    n = flat.numel()
    for r in range(world):
        lo, hi = p2p_slice(n, world, r)
        if hi > lo:
            dist.broadcast(flat[lo:hi], src=ranks[r], group=group)
    return flat


def _require_plain_model(model: KgeModel, what: str, allow_penalty: bool = False, allow_normalize: bool = False,
                         allow_reciprocal: bool = False):
    """The captured steps read the raw tables at fixed addresses without autograd.  Options whose effect they would
    silently drop raise here instead (the autograd paths of jobs.py serve them): embedder dropout in training
    (lookup_embedder.py:97-100), the reciprocal-relations wrapper unless the stepper was asked to map it (its _po queries
    are sp_ queries on relation p + R, reciprocal_relations_model.py:70-83; `reciprocal=True`), per-batch renormalisation
    (replaces the weight tensor, lookup_embedder.py:58-75) and penalty terms (train.py:320-338)."""
    from .model import ReciprocalRelationsModel
    if isinstance(model, ReciprocalRelationsModel) and not allow_reciprocal:
        raise NotImplementedError(f"{what}: ReciprocalRelationsModel is served by the autograd path (fused_path=True, no "
                                  "captured step)")
    embs = (model.get_s_embedder(), model.get_p_embedder())
    if any(e.dropout.p > 0 for e in embs):
        raise NotImplementedError(f"{what}: embedder dropout > 0 is served by the autograd path only")
    if not allow_normalize and any(e.normalize_p > 0 for e in embs):
        raise NotImplementedError(f"{what}: per-batch renormalisation (normalize_p) is served by the autograd path only")
    if not allow_penalty and any(e.regularize != "" and e.regularize_weight != 0.0 for e in embs):
        raise NotImplementedError(f"{what}: penalty terms (regularize_weight != 0) are served by the autograd path only")


def _inverse_relation_offset(model, reciprocal: bool, what: str) -> int:
    """R of a reciprocal relations model (relation table of 2 R rows; a _po query (p, o) is the sp_ query (o, p + R)) when
    the stepper is built with `reciprocal=True`, 0 without it.  A model view of the plug-in (libkge_jobs._ModelView)
    declares the wrapper with `reciprocal_relations = True`."""
    if not reciprocal:
        return 0
    from .model import ReciprocalRelationsModel
    if not (isinstance(model, ReciprocalRelationsModel) or getattr(model, "reciprocal_relations", False)):
        raise ValueError(f"{what}: reciprocal=True needs a reciprocal relations model")
    r = int(model.num_relations)
    if model.get_p_embedder().weight.shape[0] != 2 * r:
        raise ValueError(f"{what}: a reciprocal relations model has 2 * {r} relation rows "
                         f"(got {model.get_p_embedder().weight.shape[0]})")
    return r


def _adagrad_groups(optimizer, params, what: str) -> list:
    """The parameter group of each table (by identity, not param_groups[0]).  The captured steps apply Adagrad with
    lr and lr_decay; weight_decay is served by the autograd paths only."""
    groups = [optim.group_of(optimizer, p) for p in params]
    if any(g.get("weight_decay", 0.0) != 0.0 for g in groups):
        raise NotImplementedError(f"{what}: weight_decay != 0 is served by the autograd path only")
    return groups


def adagrad_rates(optimizer, params) -> list:
    """Effective Adagrad rate of each table for the step the optimizer takes next: optim.adagrad_clr with the lr and
    lr_decay of the group that holds the table (looked up now, so that an lr scheduler's edits count) at state["step"] + 1
    -- the value optim.Adagrad.step uses after its increment."""
    out = []
    for p in params:
        g = optim.group_of(optimizer, p)
        out.append(optim.adagrad_clr(float(g["lr"]), float(g.get("lr_decay", 0.0)), float(optimizer.state[p]["step"]) + 1))
    return out


class _RateWords:
    """The learning rate of a captured step in device memory: one float32 word per table, read by the _sched kernels the
    step's CUDA graph launches (include/kgeb200.h).  refresh() runs before every replay: it computes each table's rate
    (adagrad_rates) and rewrites a word only when its value changed, with fill_ on the current stream -- no allocation, no
    host sync.  At a constant rate a step issues nothing extra; with lr_decay one tiny fill per table and step.  A rate
    change therefore needs no re-capture (which would cost a warm-up step and table copies, and is collective for the
    sharded graphs).  Ranks of a sharded or replicated run must compute the same rates (the same scheduler on the same
    metric): nothing here checks that they do."""

    def __init__(self, optimizer, params, what: str, dev):
        self.opt, self.params = optimizer, tuple(params)
        self.eps = [float(g["eps"]) for g in _adagrad_groups(optimizer, self.params, what)]
        self.words = torch.zeros(len(self.params), dtype=torch.float32, device=dev)
        self._word = [self.words[i] for i in range(len(self.params))]
        self.values = [None] * len(self.params)
        self.refresh()

    def ptr(self, i: int) -> int:
        return self.words.data_ptr() + 4 * i

    def refresh(self):
        for i, r in enumerate(adagrad_rates(self.opt, self.params)):
            if r != self.values[i]:
                self._word[i].fill_(r)
                self.values[i] = r


class PeerExchange:
    """The symmetric-memory side of csrc/p2p.cu for a stepper whose gradients live in ONE flat buffer
    [g_table0 (n0) | g_table1 (n1) | loss]: allocates that buffer, the staging buffer [W_table0 | W_table1] and the signal
    pads in torch symmetric memory, and issues the two kernels (exchange, apply).  FusedAllEntityStepper carries its own
    copy of this logic (validated on 2 / 4 / 8 GPUs); this class serves the negative-sampling stepper and has NOT yet run
    on hardware."""

    def __init__(self, group, n0: int, n1: int, device):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        if n0 % 4 or n1 % 4:
            raise NotImplementedError("peer-memory exchange needs table sizes that are multiples of 4 elements")
        self.group, self.n0, self.n1 = group, n0, n1
        self.flat = symm.empty(n0 + n1 + 4, dtype=torch.float32, device=device)     # loss at [n0 + n1]
        hg = symm.rendezvous(self.flat, group)
        self.stage = symm.empty(n0 + n1, dtype=torch.float32, device=device)
        hs = symm.rendezvous(self.stage, group)
        self.pad = symm.empty(64, dtype=torch.int32, device=device)
        hp = symm.rendezvous(self.pad, group)
        self.flat.zero_(); self.stage.zero_(); self.pad.zero_()
        torch.cuda.synchronize()
        dist.barrier(group)                 # nobody signals before every pad is zero
        self.rank, self.world, self.handles = hg.rank, hg.world_size, (hg, hs, hp)
        self.p_flat = lib.ptr_array([int(x) for x in hg.buffer_ptrs])
        self.p_stage = lib.ptr_array([int(x) for x in hs.buffer_ptrs])
        self.p_pads = lib.ptr_array([int(x) for x in hp.buffer_ptrs])
        self.ctr = torch.zeros(2, dtype=torch.int32, device=device)         # [completed steps, block ticket]
        self.timeout = torch.zeros(1, dtype=torch.int32, device=device)
        self.loss_global = torch.zeros((), dtype=torch.float32, device=device)

    def exchange_and_update(self, w0, state0, mirror, w1, state1, rates: int, eps: float, stream: int):
        """`rates`: device address of two float32 words, the learning rates of table 0 and table 1 (_RateWords)."""
        lib.call("kgeb_p2p_exchange_sched", self.p_pads, self.p_flat, self.p_stage, self.rank, self.world,
                 self.ctr.data_ptr(), self.timeout.data_ptr(), w0.data_ptr(), state0.data_ptr(), mirror, w0.numel(),
                 w1.data_ptr(), state1.data_ptr(), w1.numel(), self.loss_global.data_ptr(), rates, eps, stream)
        lib.call("kgeb_p2p_apply", self.p_pads, self.stage.data_ptr(), self.rank, self.world, self.ctr.data_ptr(),
                 self.ctr[1:].data_ptr(), self.timeout.data_ptr(), w0.data_ptr(), mirror, w0.numel(), w1.data_ptr(),
                 w1.numel(), stream)

    def check(self):
        if int(self.timeout.item()) != 0:
            raise RuntimeError("a peer did not arrive at a peer-memory barrier")


class _TouchedRows:
    """Device state of the fused table update (include/kgeb200.h, kgeb_touched_build / kgeb_fused_bwd_update /
    kgeb_touched_update) for one table shard of `n_rows` rows: the rows that receive sparse gradient rows in a step are
    numbered (slots), their dense gradient is parked in g_dense, their sparse rows are summed in g_sparse."""

    def __init__(self, n_rows: int, cap: int, d: int, n_a: int, n_b: int, dev):
        self.cap, self.d = cap, d
        self.slot_of = torch.full((max(n_rows, 1),), -1, dtype=torch.int32, device=dev)
        self.uniq = torch.zeros(cap, dtype=torch.int64, device=dev)
        self.num = torch.zeros(1, dtype=torch.int64, device=dev)
        self.slot_a = torch.zeros(n_a, dtype=torch.int64, device=dev)
        self.slot_b = torch.zeros(n_b, dtype=torch.int64, device=dev)
        self.g_dense = torch.zeros(cap, d, dtype=torch.float32, device=dev)
        self.g_sparse = torch.zeros(cap + 1, d, dtype=torch.float32, device=dev)      # last row: rows of other shards

    def build(self, ids_a, ids_b, n_b_real, e_lo: int, e_hi: int, stream):
        assert ids_a.numel() + ids_b.numel() == self.cap
        lib.call("kgeb_touched_build", ids_a.data_ptr(), ids_a.numel(), ids_b.data_ptr(), ids_b.numel(),
                 None if n_b_real is None else n_b_real.data_ptr(), e_lo, e_hi, self.slot_of.data_ptr(), self.uniq.data_ptr(),
                 self.num.data_ptr(), self.slot_a.data_ptr(), self.slot_b.data_ptr(), stream)

    def update(self, w, state, mirror, rate: int, eps: float, skip, stream):
        """`rate`: device address of the float32 learning-rate word (_RateWords.ptr)."""
        lib.call("kgeb_touched_update_sched", w.data_ptr(), state.data_ptr(), None if mirror is None else mirror.data_ptr(),
                 self.slot_of.data_ptr(), self.uniq.data_ptr(), self.num.data_ptr(), self.cap, self.g_dense.data_ptr(),
                 self.g_sparse.data_ptr(), self.d, rate, eps, None if skip is None else skip.data_ptr(), stream)


class FusedAllEntityStepper:
    def __init__(self, model: KgeModel, optimizer, rows: int, nnz_max: int, loss_kind: int, batch_size: int,
                 offset: float = 0.0, label_smoothing: float = 0.0, math_mode: int = lib.MATH_BF16,
                 use_graph: bool = True, shard: Optional[fused.Shard] = None, dp_group=None, dp_p2p: bool = False,
                 onevsall_triples: bool = False, reciprocal: bool = False):
        """`onevsall_triples`: the step starts from a static [rows / 2, 3] int64 buffer of TRIPLES (`set_triples`): its first
        kernel builds the 1vsAll batch -- queries, one label per row, the three scatter permutations -- on the device
        (kgeb_onevsall_batch_build), so a step costs the host one copy and one graph launch.
        `reciprocal`: the model is a reciprocal relations model (2 R relation rows).  Every query of the step is an sp_
        query: the _po queries of a batch arrive as sp_ rows on relation p + R -- built so by kgeb_onevsall_batch_build_inv
        (onevsall_triples) or by the caller (`kvsall_rows(..., inv_rel_offset=R)` for set_inputs / pack_host_batch).
        Kernels, launches and the update are those of the plain step on a 2 R-row relation table."""
        if model.get_scorer().kind != lib.DOT:
            raise NotImplementedError("the fused all-entity step serves the DOT scorers")
        self.inv_rel = _inverse_relation_offset(model, reciprocal, "FusedAllEntityStepper")
        _require_plain_model(model, "FusedAllEntityStepper", allow_penalty=True, allow_reciprocal=reciprocal)
        self.model, self.opt = model, optimizer
        self.rows, self.nnz_max, self.loss_kind, self.batch_size = rows, nnz_max, loss_kind, batch_size
        self.offset, self.ls, self.math = float(offset), float(label_smoothing), math_mode
        self.ent = model.get_s_embedder().weight
        self.rel = model.get_p_embedder().weight
        dev = self.ent.device
        self.E, self.d = self.ent.shape
        self.dr = self.rel.shape[1]
        # the learning rates live in device words (_RateWords): step() follows lr schedulers and lr_decay
        self.rate = _RateWords(optimizer, (self.ent, self.rel), "FusedAllEntityStepper", dev)
        self.eps_ent, self.eps_rel = self.rate.eps
        if dp_group is not None and dp_p2p and self.eps_ent != self.eps_rel:
            raise NotImplementedError("the peer-memory exchange applies one eps to both tables")
        f32 = dict(dtype=torch.float32, device=dev)
        i64 = dict(dtype=torch.int64, device=dev)
        # Unweighted Lp penalties (lookup_embedder.py:126-134) are folded into the Adagrad kernels (SURVEY.md 8f-3):
        # the entity table is penalised by the s- and the o-embedder (kge_model.py:588-606), i.e. twice.
        self.pen = None
        e_emb, r_emb = model.get_s_embedder(), model.get_p_embedder()
        active = [e for e in (e_emb, r_emb) if e.regularize != "" and e.regularize_weight != 0.0]
        if active:
            if any(e.regularize_weighted for e in active):
                raise NotImplementedError("weighted penalties need the triples of the batch; not part of this step")
            if dp_group is not None or (shard is not None and shard.distributed):
                raise NotImplementedError("penalty terms are built for the single-GPU captured step")
            self.pen = dict(ent=(int(e_emb.regularize_p), 2.0 * e_emb.regularize_weight if e_emb in active else 0.0),
                            rel=(int(r_emb.regularize_p), r_emb.regularize_weight if r_emb in active else 0.0))
            self.penalty_values = torch.zeros(2, **f32)          # [entity terms (s + o), relation term]
            nb = lib.load().kgeb_penalty_workspace_bytes(0, max(self.ent.numel(), self.rel.numel()))
            self.pen_ws = [torch.empty(nb, dtype=torch.uint8, device=dev) for _ in range(2)]
        # static inputs: ONE contiguous byte buffer so that a packed host batch arrives with a single H2D copy
        #   int64 [a_idx (rows) | p_idx (rows) | lab_off (rows+1) | lab_col (nnz_max)]
        #   int32 [row_combine (rows) | a_perm (rows) | p_perm (rows) | lab_perm (nnz_max)]
        # The three permutations are stable argsorts of a_idx, p_idx and the label entities (padding counts as entity
        # 0): the collate knows all ids of the batch, so the sorts of the three deterministic scatters are done there,
        # once per batch, off the step's critical path (kgeb_scatter_add_rows_perm)
        nz = max(nnz_max, 1)
        self.n_i64 = 3 * rows + 1 + nz
        self.input_bytes = torch.zeros(self.n_i64 * 8 + (3 * rows + nz) * 4, dtype=torch.uint8, device=dev)
        iv = self.input_views(self.input_bytes)
        self.a_idx, self.p_idx, self.lab_off, self.lab_col = iv["a_idx"], iv["p_idx"], iv["lab_off"], iv["lab_col"]
        self.row_combine, self.a_perm, self.p_perm, self.lab_perm = (iv["row_combine"], iv["a_perm"], iv["p_perm"],
                                                                     iv["lab_perm"])
        # static intermediates / outputs
        self.Q = torch.empty(rows, self.d, **f32)
        self.dQ = torch.empty(rows, self.d, **f32)
        self.da = torch.empty(rows, self.d, **f32)
        self.dp = torch.empty(rows, self.dr, **f32)
        # gradients and the loss live in ONE flat buffer so that data-parallel replicas need a single all-reduce
        n_e, n_r = self.E * self.d, self.rel.shape[0] * self.dr
        # layout [g_q | g_ent | g_rel | loss]: data-parallel replicas fold g_q into g_ent and all-reduce the tail only
        self.p2p = None
        # Large tables (Wikidata5M: 2.4 GB per [E,d] buffer): ONE gradient buffer that is never cleared.  The dense dTable
        # tile kernel STORES its rows (KGEB_BWD_OVERWRITE_TABLE), the sparse parts (label rows, query-side rows) are
        # scattered on top afterwards, Adagrad reads one buffer: per step 2 x E*d*4 bytes of clears and one E*d*4 read
        # less than the overlapped two-buffer flow that small tables (FB15k-237: 7.4 MB, latency-bound) keep.
        self.seq = (math_mode == lib.MATH_BF16 and self.d % 16 == 0 and self.d <= 256 and dp_group is None
                    and not (shard is not None and shard.distributed) and self.pen is None and nnz_max > 0
                    and n_e * 4 >= (64 << 20))
        # ... and NO gradient buffer at all when the step's sparse rows fit the touched-row machinery: Adagrad runs in the
        # flush of the dTable tile kernel (kgeb_fused_bwd_update), the <= 8192 rows that also get label / query-side rows
        # are parked and updated by a row kernel.  Saves the store and the read-back of an [E, d] gradient per step.
        # (d % 32 == 0: whole 32-column boxes only -- the dimensions this flow has been run at: 64, 128, 256)
        self.fuse_update = (self.seq and self.d % 32 == 0 and rows + max(nnz_max, 1) <= lib.load().kgeb_touched_capacity()
                            and os.environ.get("KGEB_NO_FUSED_UPDATE", "0") in ("", "0"))
        if dp_group is not None and dp_p2p:
            self._setup_p2p(dp_group, n_e, n_r, dev)      # gradients live in peer-mapped (symmetric) memory
        elif self.fuse_update:
            self.gflat = torch.zeros(n_r + 1, **f32)
        elif self.seq:
            self.gflat = torch.zeros(n_e + n_r + 1, **f32)
        else:
            self.gflat = torch.zeros(2 * n_e + n_r + 1, **f32)
        if self.fuse_update:
            cap = rows + max(nnz_max, 1)
            self.touched = _TouchedRows(self.E, cap, self.d, rows, max(nnz_max, 1), dev)
            self.g_q = self.g_ent = None
            self.g_rel = self.gflat[:n_r].view(self.rel.shape[0], self.dr)
            self.loss = self.gflat[n_r:].view(())
        else:
            g0 = 0 if self.seq else n_e
            self.g_q = self.gflat[:n_e].view(self.E, self.d)              # query-side rows (da scattered by entity id)
            self.g_ent = self.gflat[g0:g0 + n_e].view(self.E, self.d)     # dense part (G^T Q) + label rows (side stream)
            self.g_rel = self.gflat[g0 + n_e:g0 + n_e + n_r].view(self.rel.shape[0], self.dr)
            self.loss = self.gflat[g0 + n_e + n_r:].view(())
            self.dp_flat = self.gflat[n_e:]                               # what the replicas exchange
        self.rowstat = torch.empty(rows, 4, **f32)
        # KL on the bf16 tiles: forward statistics and dQ from ONE table pass (kgeb_fused_flash_fwd / _dq)
        # (single GPU, no folded penalty: a failed flash pass is undone by clearing the gradients -- Adagrad is then a no-op --
        # and the step repeats on the two-pass graph; with a penalty gradient folded into Adagrad that is not a no-op)
        self.flash = (fused.flash_supported(loss_kind, math_mode, self.d, self.ls) and dp_group is None
                      and not (shard is not None and shard.distributed) and self.pen is None)
        self._use_flash = self.flash          # which forward / backward the stage functions issue (graph capture toggles it)
        self.flash_fallbacks = 0              # steps that had to be repeated on the two-pass kernels
        if self.flash:
            self.rowstat_local = torch.empty(rows, 4, **f32)      # this shard's statistics (its mref) before the combine
            self.o_sum = torch.empty(rows, self.d, **f32)
            self.flash_status = torch.zeros(4, dtype=torch.int32, device=dev)
        self.loss_rows = torch.zeros(rows, **f32)      # per-row loss values (kgeb_loss_from_rowstat rows_out)
        self.report = torch.zeros(2, **f32)            # [total, value of the last non-empty query type] (train.py:747)
        # Data parallelism for graphs too small to shard (SURVEY.md 8e "replicas" row): every rank trains on its own
        # batch against its full replica; one all-reduce sums gradients and loss; loss terms are divided by the global
        # batch size so all replicas apply the identical update.
        self.dp_group = dp_group
        self.dp_world = 1
        if dp_group is not None:
            import torch.distributed as dist
            self.dp_world = dist.get_world_size(dp_group)
        self.global_batch = batch_size * self.dp_world
        self.lse = torch.zeros(rows, **f32)
        # Multi-GPU (SURVEY.md 8e): every rank sees the whole batch and scores it against its own entity range
        # [e_lo, e_hi); row statistics, dQ and the dense table gradient are all-reduced over NVLink.  The (small)
        # tables and the optimizer state are replicated, so every rank applies the identical update.
        self.shard = shard or fused.Shard.full(self.E)
        self.ws = torch.empty(lib.load().kgeb_fused_workspace_bytes(rows, self.d, self.E, max(nnz_max, 1)),
                              dtype=torch.uint8, device=dev)
        self.sws = torch.empty(lib.load().kgeb_scatter_workspace_bytes(rows, max(self.d, self.dr)), dtype=torch.uint8,
                               device=dev)
        self.ws2 = torch.empty_like(self.ws)   # workspace of the dTable half of the backward (runs on a second stream)
        self.sws2 = torch.empty_like(self.sws)  # scatter workspace of the relation-side chain (third stream)
        self.ws3 = torch.empty_like(self.ws)   # workspace of the dense-only dTable kernel when the label rows go to g_q
        self.side = torch.cuda.Stream(device=dev)
        self.side2 = torch.cuda.Stream(device=dev)
        self.ev_clear, self.ev_q = torch.cuda.Event(), torch.cuda.Event()
        self.mirror = None
        if math_mode == lib.MATH_BF16 and self.d % 16 == 0 and self.d <= 256:
            self.mirror = torch.empty(self.E, self.d, dtype=torch.bfloat16, device=dev)
            lib.call("kgeb_to_bf16", lib.f32(self.ent.detach(), "table"), self.mirror.data_ptr(), self.ent.numel(),
                     lib.stream_ptr(self.ent))
        self.triples = None
        if onevsall_triples:
            if rows % 2 != 0 or nnz_max != rows or rows > 8192:
                raise ValueError("onevsall_triples: rows = nnz_max = 2 * batch <= 8192")
            self.triples = torch.zeros(rows // 2, 3, **i64)
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        if use_graph:
            self._capture()

    def set_triples(self, triples: torch.Tensor):
        """One copy (host pinned or device, non-blocking) of the batch's [batch, 3] int64 triples; see onevsall_triples."""
        self.triples.copy_(triples, non_blocking=True)

    def input_views(self, buf: torch.Tensor) -> dict:
        """Typed views into a byte buffer with the layout of the static inputs (see __init__)."""
        rows, nz = self.rows, max(self.nnz_max, 1)
        v64 = buf[: self.n_i64 * 8].view(torch.int64)
        v32 = buf[self.n_i64 * 8:].view(torch.int32)
        return {"a_idx": v64[:rows], "p_idx": v64[rows:2 * rows], "lab_off": v64[2 * rows:3 * rows + 1],
                "lab_col": v64[3 * rows + 1:], "row_combine": v32[:rows], "a_perm": v32[rows:2 * rows],
                "p_perm": v32[2 * rows:3 * rows], "lab_perm": v32[3 * rows:3 * rows + nz]}

    # -- one step on the current stream, in three stages separated by the (optional) collectives ----------------
    def _fused_stats_in_backward(self) -> bool:
        """BCE on the bf16 tiles: the backward dQ kernel evaluates sigmoid and softplus from the same exponential, so the
        forward statistics (only needed for the loss value) come out of the backward pass and the forward kernel is skipped."""
        return self.loss_kind == lib.LOSS_BCE and self.mirror is not None

    def _stage_forward(self):
        st = lib.stream_ptr(self.ent)
        model_id = lib.MODELS[self.model.model]
        ent, rel = self.ent.detach(), self.rel.detach()
        sh = self.shard
        if self.triples is not None:
            lib.call("kgeb_onevsall_batch_build_inv", self.triples.data_ptr(), self.rows // 2, self.E,
                     self.rel.shape[0] - self.inv_rel, self.a_idx.data_ptr(), self.p_idx.data_ptr(),
                     self.row_combine.data_ptr(), self.lab_off.data_ptr(), self.lab_col.data_ptr(), self.a_perm.data_ptr(),
                     self.p_perm.data_ptr(), self.lab_perm.data_ptr(), self.inv_rel, st)
        # the gradient buffers are cleared on the third stream, beside the query build (joined where they are first used)
        cur = torch.cuda.current_stream()
        self.side2.wait_stream(cur)
        with torch.cuda.stream(self.side2):
            if self.fuse_update:
                self.gflat.zero_()                        # relation gradient + loss
                self.touched.build(self.a_idx, self.lab_col, self.lab_off[self.rows:], 0, self.E, lib.stream_ptr(self.ent))
            elif self.seq:
                self.gflat[self.E * self.d:].zero_()      # relation gradient + loss only
            else:
                self.gflat.zero_()
            self.ev_clear.record()
        lib.call("kgeb_query_build", model_id, 0, self.row_combine.data_ptr(), ent.data_ptr(), self.a_idx.data_ptr(),
                 rel.data_ptr(), self.p_idx.data_ptr(), 1, self.rows, self.d, self.Q.data_ptr(), st)
        if self._split_label_rows() and not self.seq:
            # Label rows of the dense table gradient go to g_q (the optimizer adds g_ent + g_q), on the third stream
            # and underneath the dQ tile kernel: the dTable tile kernel then depends on nothing but the cleared g_ent
            # and starts the moment dQ releases the SMs.  (Scattered into g_ent in front of the tile kernel, as
            # kgeb_fused_bwd does on its own, this chain -- starved of SMs by the persistent dQ CTAs -- ended ~14 us after
            # dQ and delayed dTable by as much: profiles/README.md, step timeline.)
            self.ev_q.record()
            with torch.cuda.stream(self.side2):
                self.side2.wait_event(self.ev_q)
                lib.call("kgeb_fused_label_rows", self.loss_kind, self.Q.data_ptr(), self.rows, self.d, ent.data_ptr(), 0,
                         self.E, self.lab_off.data_ptr(), self.lab_col.data_ptr(), self.nnz_max, self.lab_perm.data_ptr(),
                         self.ls, 1.0 / self.global_batch, None, self.g_q.data_ptr(), self.ws2.data_ptr(),
                         self.ws2.numel(), lib.stream_ptr(self.ent))
        if self._use_flash:
            self.flash_status.zero_()
            lib.call("kgeb_fused_flash_fwd", self.Q.data_ptr(), self.rows, self.d, ent[sh.e_lo:sh.e_hi].data_ptr(), sh.e_lo,
                     sh.e_hi, self.E, self.lab_off.data_ptr(), self.lab_col.data_ptr(), self.nnz_max, self._mirror_ptr(),
                     self.rowstat.data_ptr(), self.o_sum.data_ptr(), self.flash_status.data_ptr(), self.ws.data_ptr(),
                     self.ws.numel(), st)
            self.rowstat_local.copy_(self.rowstat)
        elif not self._fused_stats_in_backward():
            lib.call("kgeb_fused_fwd", self.loss_kind, self.math, self.Q.data_ptr(), self.rows, self.d,
                     ent[sh.e_lo:sh.e_hi].data_ptr(), sh.e_lo, sh.e_hi, self.E, self.lab_off.data_ptr(),
                     self.lab_col.data_ptr(), self.nnz_max, self.ls, self.offset, self._mirror_ptr(),
                     self.rowstat.data_ptr(), self.ws.data_ptr(), self.ws.numel(), st)
        if sh.distributed:
            cur.wait_stream(self.side2)       # the stages are separate graphs there: nothing may stay forked

    def _loss_kernel(self):
        lib.call("kgeb_loss_from_rowstat", self.loss_kind, self.rowstat.data_ptr(), self.lab_off.data_ptr(), self.rows,
                 self.ls, self.E, 1.0 / self.global_batch, self.loss_rows.data_ptr(), self.lse.data_ptr(),
                 self.loss.data_ptr(), lib.stream_ptr(self.ent))
        lib.call("kgeb_loss_report_inv", self.loss_rows.data_ptr(), self.row_combine.data_ptr(), self.p_idx.data_ptr(),
                 self.inv_rel, self.rows, self.report.data_ptr(), lib.stream_ptr(self.ent))

    def _stage_backward(self):
        st = lib.stream_ptr(self.ent)
        ent = self.ent.detach()
        sh = self.shard
        late_stats = self._fused_stats_in_backward()
        if not late_stats:
            self._loss_kernel()   # KL needs the log-sum-exp before the backward
        lse = self.lse.data_ptr() if self.loss_kind == lib.LOSS_KL else None
        common = (self.loss_kind, self.math, self.Q.data_ptr(), self.rows, self.d, ent[sh.e_lo:sh.e_hi].data_ptr(),
                  sh.e_lo, sh.e_hi, self.E, self.lab_off.data_ptr(), self.lab_col.data_ptr(), self.nnz_max,
                  self.lab_perm.data_ptr() if self.nnz_max > 0 else None, self.ls, self.offset, lse,
                  1.0 / self.global_batch, None, self._mirror_ptr())
        # The two halves of the backward are independent: the dense table gradient (+ its label rows) goes to a second
        # stream, so that the chain of small latency-bound kernels that follows dQ on this stream (partial reduce, label
        # scatter, query-transform backward, sorted scatters) runs underneath the dTable tile kernel.
        cur = torch.cuda.current_stream()
        if self._use_flash:
            # the log-sum-exp is known (loss kernel above): the dense table gradient -- the only remaining table pass -- goes
            # to the second stream; dQ = rescaled o_sum + label rows is a [rows, d] elementwise kernel on this one
            self.ev_q.record()
            split = self._split_label_rows()
            with torch.cuda.stream(self.side):
                self.side.wait_event(self.ev_q)
                if split and self.fuse_update:
                    self._dense_update(lse)
                elif split:
                    dense = list(common)
                    dense[11], dense[12] = 0, None          # nnz, lab_perm: label rows are scattered separately
                    if not self.seq:
                        self.side.wait_event(self.ev_clear)
                    lib.call("kgeb_fused_bwd", *dense, None, self.g_ent.data_ptr(), None,
                             lib.BWD_OVERWRITE_TABLE if self.seq else 0, self.ws3.data_ptr(), self.ws3.numel(),
                             lib.stream_ptr(self.ent))
                else:
                    if not sh.distributed:
                        self.side.wait_stream(self.side2)     # cleared gradient buffers
                    lib.call("kgeb_fused_bwd", *common, None, self.g_ent[sh.e_lo:sh.e_hi].data_ptr(), None, 0,
                             self.ws2.data_ptr(), self.ws2.numel(), lib.stream_ptr(self.ent))
            lib.call("kgeb_fused_flash_dq", self.Q.data_ptr(), self.rows, self.d, ent[sh.e_lo:sh.e_hi].data_ptr(), sh.e_lo,
                     sh.e_hi, self.lab_off.data_ptr(), self.lab_col.data_ptr(), self.nnz_max, self.rowstat_local.data_ptr(),
                     self.lse.data_ptr(), 1.0 / self.global_batch, None, self.o_sum.data_ptr(), self.dQ.data_ptr(),
                     self.ws.data_ptr(), self.ws.numel(), st)
            if sh.distributed:
                self._join_side()
            return
        if self._split_label_rows():
            # dQ first; the dense-only dTable kernel (nnz = 0: no label part) queues behind it on the second stream
            lib.call("kgeb_fused_bwd", *common, self.dQ.data_ptr(), None, self.rowstat.data_ptr() if late_stats else None,
                     0, self.ws.data_ptr(), self.ws.numel(), st)
            dense = list(common)
            dense[11], dense[12] = 0, None          # nnz, lab_perm
            with torch.cuda.stream(self.side):
                lib.call("kgeb_fused_bwd_wait_tiles", lib.stream_ptr(self.ent))   # the dQ tile kernel, not its reductions
                if self.fuse_update:
                    self._dense_update(lse)
                else:
                    if not self.seq:
                        self.side.wait_event(self.ev_clear)
                    lib.call("kgeb_fused_bwd", *dense, None, self.g_ent.data_ptr(), None,
                             lib.BWD_OVERWRITE_TABLE if self.seq else 0, self.ws3.data_ptr(), self.ws3.numel(),
                             lib.stream_ptr(self.ent))
            return
        self.side.wait_stream(cur)
        if not sh.distributed:
            self.side.wait_stream(self.side2)     # cleared gradient buffers
        with torch.cuda.stream(self.side):
            lib.call("kgeb_fused_bwd", *common, None, self.g_ent[sh.e_lo:sh.e_hi].data_ptr(), None, 0, self.ws2.data_ptr(),
                     self.ws2.numel(), lib.stream_ptr(self.ent))
        lib.call("kgeb_fused_bwd", *common, self.dQ.data_ptr(), None, self.rowstat.data_ptr() if late_stats else None,
                 0, self.ws.data_ptr(), self.ws.numel(), st)
        if sh.distributed:
            self._join_side()     # the collectives that follow need the complete dense gradient

    def _dense_update(self, lse):
        """(current stream = the dTable stream) Dense table gradient + Adagrad in the tile kernel's flush.  Reads of the fp32
        table that run beside it -- query backward, label rows of dQ -- touch only rows of the touched set, which this kernel
        leaves alone."""
        self.side.wait_event(self.ev_clear)           # slot_of is built on the third stream
        t = self.touched
        lib.call("kgeb_fused_bwd_update_sched", self.loss_kind, self.Q.data_ptr(), self.rows, self.d,
                 self.ent.detach().data_ptr(), 0, self.E, self.E, self.lab_off.data_ptr(), self.ls, self.offset, lse,
                 1.0 / self.global_batch, None, self.mirror.data_ptr(), self.opt.state[self.ent]["sum"].data_ptr(),
                 self.rate.ptr(0), self.eps_ent, t.slot_of.data_ptr(),
                 t.g_dense.data_ptr(), self.flash_status.data_ptr() if self._use_flash else None, self.ws3.data_ptr(),
                 self.ws3.numel(), lib.stream_ptr(self.ent))

    def _join_side(self):
        torch.cuda.current_stream().wait_stream(self.side)

    def _split_label_rows(self) -> bool:
        """bf16 tile path on an unsharded table with labels: see _stage_forward."""
        return self.mirror is not None and not self.shard.distributed and self.nnz_max > 0

    def _guard_flash(self, buf: torch.Tensor):
        """A failed flash pass (flash_status != 0) left garbage in the gradients: clear `buf` right before its Adagrad
        kernel, which then is an exact no-op; step() sees the status and repeats the step on the two-pass graph."""
        if self._use_flash:
            lib.call("kgeb_zero_if", self.flash_status.data_ptr(), buf.data_ptr(), buf.numel(), lib.stream_ptr(self.ent))

    def _stage_update(self):
        st = lib.stream_ptr(self.ent)
        model_id = lib.MODELS[self.model.model]
        ent, rel = self.ent.detach(), self.rel.detach()
        lib.call("kgeb_query_bwd", model_id, 0, self.row_combine.data_ptr(), ent.data_ptr(), self.a_idx.data_ptr(),
                 rel.data_ptr(), self.p_idx.data_ptr(), 1, self.rows, self.d, self.dQ.data_ptr(), self.da.data_ptr(),
                 self.dp.data_ptr(), st)
        # relation-side chain (loss value, dp scatter, relation Adagrad) on a third stream, entity-side scatter here
        cur = torch.cuda.current_stream()
        if not self.shard.distributed:
            cur.wait_stream(self.side2)       # cleared gradient buffers
        self.side2.wait_stream(cur)
        with torch.cuda.stream(self.side2):
            st2 = lib.stream_ptr(self.ent)
            if self._fused_stats_in_backward():
                self._loss_kernel()
            lib.call("kgeb_scatter_add_rows_perm", self.p_idx.data_ptr(), 1, self.p_perm.data_ptr(), self.dp.data_ptr(),
                     self.rows, self.dr, self.g_rel.data_ptr(), self.rel.shape[0], self.sws2.data_ptr(),
                     self.sws2.numel(), st2)
            if self.dp_world == 1:
                s_rel = self.opt.state[self.rel]["sum"]
                if self.pen is not None:
                    lib.call("kgeb_adagrad_dense_lp_sched", rel.data_ptr(), s_rel.data_ptr(), self.g_rel.data_ptr(), None,
                             rel.numel(), self.rate.ptr(1), self.eps_rel, 0.0, self.pen["rel"][0], self.pen["rel"][1], None,
                             self.penalty_values[1:].data_ptr(), self.pen_ws[1].data_ptr(), self.pen_ws[1].numel(), st2)
                else:
                    self._guard_flash(self.g_rel)
                    lib.call("kgeb_adagrad_dense_sched", rel.data_ptr(), s_rel.data_ptr(), self.g_rel.data_ptr(), None,
                             rel.numel(), self.rate.ptr(1), self.eps_rel, 0.0, None, st2)
        if self.fuse_update:
            # the sparse rows (label rows, then query-side rows) are summed per touched row underneath the dTable kernel;
            # the row kernel adds the dense part that kernel parked and applies Adagrad to the touched rows
            t = self.touched
            cur.wait_event(self.ev_clear)
            lib.call("kgeb_fused_label_rows_to", self.loss_kind, self.Q.data_ptr(), self.rows, self.d, ent.data_ptr(), 0,
                     self.E, self.lab_off.data_ptr(), self.lab_col.data_ptr(), self.nnz_max, self.lab_perm.data_ptr(),
                     self.ls, 1.0 / self.global_batch, None, t.slot_b.data_ptr(), t.cap + 1, t.g_sparse.data_ptr(),
                     self.ws2.data_ptr(), self.ws2.numel(), st)
            lib.call("kgeb_scatter_add_rows_perm", t.slot_a.data_ptr(), 1, self.a_perm.data_ptr(), self.da.data_ptr(),
                     self.rows, self.d, t.g_sparse.data_ptr(), t.cap + 1, self.sws.data_ptr(), self.sws.numel(), st)
            self._join_side()
            t.update(ent, self.opt.state[self.ent]["sum"], self.mirror, self.rate.ptr(0), self.eps_ent,
                     self.flash_status if self._use_flash else None, st)
            cur.wait_stream(self.side2)
            return
        if self.seq:
            # the dense part has been STORED into the one gradient buffer: label rows and query-side rows go on top
            self._join_side()
            lib.call("kgeb_fused_label_rows", self.loss_kind, self.Q.data_ptr(), self.rows, self.d, ent.data_ptr(), 0,
                     self.E, self.lab_off.data_ptr(), self.lab_col.data_ptr(), self.nnz_max, self.lab_perm.data_ptr(),
                     self.ls, 1.0 / self.global_batch, None, self.g_ent.data_ptr(), self.ws2.data_ptr(),
                     self.ws2.numel(), st)
        lib.call("kgeb_scatter_add_rows_perm", self.a_idx.data_ptr(), 1, self.a_perm.data_ptr(), self.da.data_ptr(),
                 self.rows, self.d, self.g_q.data_ptr(), self.E, self.sws.data_ptr(), self.sws.numel(), st)
        if self.dp_world > 1:
            cur.wait_stream(self.side2)      # gradients complete on this stream before the all-reduce
            self._join_side()
            self.g_ent.add_(self.g_q)        # one table-sized buffer on the wire instead of two
            return
        if not self.shard.distributed:
            self._join_side()     # dense table gradient from the side stream
        s_ent = self.opt.state[self.ent]["sum"]
        mirror = None if self.mirror is None else self.mirror.data_ptr()
        if self.pen is not None:
            lib.call("kgeb_adagrad_dense_lp_sched", ent.data_ptr(), s_ent.data_ptr(), self.g_ent.data_ptr(),
                     self.g_q.data_ptr(), ent.numel(), self.rate.ptr(0), self.eps_ent, 0.0, self.pen["ent"][0],
                     self.pen["ent"][1], mirror,
                     self.penalty_values.data_ptr(), self.pen_ws[0].data_ptr(), self.pen_ws[0].numel(), st)
        else:
            self._guard_flash(self.gflat[:(1 if self.seq else 2) * self.E * self.d])       # g_ent (and g_q)
            lib.call("kgeb_adagrad_dense_sched", ent.data_ptr(), s_ent.data_ptr(), self.g_ent.data_ptr(),
                     None if self.seq else self.g_q.data_ptr(), ent.numel(), self.rate.ptr(0), self.eps_ent, 0.0, mirror, st)
        cur.wait_stream(self.side2)

    # -- data-parallel exchange fused with the update over NVLink peer memory (csrc/p2p.cu) ---------------------------
    def _setup_p2p(self, group, n_e: int, n_r: int, dev):
        """Gradient buffer, staging buffer (updated weights pushed by the slice owners) and signal pads in torch symmetric
        memory: cuMem allocations that every process of the node maps, so kernels address the peers' copies directly."""
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        if n_e % 4 or n_r % 4:
            raise NotImplementedError("peer-memory exchange needs table sizes that are multiples of 4 elements")
        self.gflat = symm.empty(2 * n_e + n_r + 1, dtype=torch.float32, device=dev)
        hg = symm.rendezvous(self.gflat, group)
        self.p2p_stage = symm.empty(n_e + n_r, dtype=torch.float32, device=dev)
        hs = symm.rendezvous(self.p2p_stage, group)
        self.p2p_pad = symm.empty(64, dtype=torch.int32, device=dev)
        hp = symm.rendezvous(self.p2p_pad, group)
        self.gflat.zero_(); self.p2p_stage.zero_(); self.p2p_pad.zero_()
        torch.cuda.synchronize()
        dist.barrier(group)                 # nobody signals before every pad is zero
        world = hg.world_size
        self.p2p = dict(rank=hg.rank, world=world, handles=(hg, hs, hp),
                        flat=lib.ptr_array([int(x) + 4 * n_e for x in hg.buffer_ptrs]),     # [g_ent | g_rel | loss]
                        stage=lib.ptr_array([int(x) for x in hs.buffer_ptrs]),              # [W_ent | W_rel]
                        pads=lib.ptr_array([int(x) for x in hp.buffer_ptrs]))
        self.p2p_ctr = torch.zeros(2, dtype=torch.int32, device=dev)        # [completed steps, block ticket]
        self.p2p_timeout = torch.zeros(1, dtype=torch.int32, device=dev)
        self.loss_global = torch.zeros((), dtype=torch.float32, device=dev)

    def _stage_exchange_p2p(self):
        """Two kernels on peer pointers, captured in the same CUDA graph as the compute stages:
        exchange = barrier ; reduce the owned slice over all ranks ; Adagrad ; push the new weights to the peers' staging
        apply    = barrier ; copy the other owners' slices into the tables (+ bf16 mirror)."""
        st = lib.stream_ptr(self.ent)
        x = self.p2p
        ent, rel = self.ent.detach(), self.rel.detach()
        s_ent, s_rel = self.opt.state[self.ent]["sum"], self.opt.state[self.rel]["sum"]
        mirror = None if self.mirror is None else self.mirror.data_ptr()
        lib.call("kgeb_p2p_exchange_sched", x["pads"], x["flat"], x["stage"], x["rank"], x["world"],
                 self.p2p_ctr.data_ptr(), self.p2p_timeout.data_ptr(), ent.data_ptr(), s_ent.data_ptr(), mirror, ent.numel(),
                 rel.data_ptr(), s_rel.data_ptr(), rel.numel(), self.loss_global.data_ptr(), self.rate.words.data_ptr(),
                 self.eps_ent, st)
        lib.call("kgeb_p2p_apply", x["pads"], self.p2p_stage.data_ptr(), x["rank"], x["world"], self.p2p_ctr.data_ptr(),
                 self.p2p_ctr[1:].data_ptr(), self.p2p_timeout.data_ptr(), ent.data_ptr(), mirror, ent.numel(),
                 rel.data_ptr(), rel.numel(), st)

    def check_p2p(self):
        """Host check (one sync): no peer-memory barrier ran into its timeout."""
        if self.p2p is not None and int(self.p2p_timeout.item()) != 0:
            raise RuntimeError("a peer did not arrive at a peer-memory barrier")

    def sync_optimizer_state(self):
        """Peer-memory mode shards the Adagrad state by slice owner: gather the slices so that every rank holds the
        complete accumulators again (checkpoints; switching modes)."""
        if self.p2p is None:
            return
        for t in (self.opt.state[self.ent]["sum"], self.opt.state[self.rel]["sum"]):
            gather_owner_slices(t.view(-1), self.dp_group)

    def _stage_apply_dp(self):
        """Data-parallel mode: both Adagrad steps after the gradient all-reduce."""
        st = lib.stream_ptr(self.ent)
        ent, rel = self.ent.detach(), self.rel.detach()
        s_ent, s_rel = self.opt.state[self.ent]["sum"], self.opt.state[self.rel]["sum"]
        lib.call("kgeb_adagrad_dense_sched", rel.data_ptr(), s_rel.data_ptr(), self.g_rel.data_ptr(), None, rel.numel(),
                 self.rate.ptr(1), self.eps_rel, 0.0, None, st)
        lib.call("kgeb_adagrad_dense_sched", ent.data_ptr(), s_ent.data_ptr(), self.g_ent.data_ptr(), None,
                 ent.numel(), self.rate.ptr(0), self.eps_ent, 0.0, None if self.mirror is None else self.mirror.data_ptr(), st)

    def _exchange_dp(self):
        import torch.distributed as dist
        dist.all_reduce(self.dp_flat, group=self.dp_group)   # gradients of both tables and the loss in one collective

    def _mirror_ptr(self):
        return None if self.mirror is None else self.mirror[self.shard.e_lo:self.shard.e_hi].data_ptr()

    def _exchange_stats(self):
        # per-row statistics of the shards -> global (max + rescaled sums for KL)
        if self.shard.distributed and not self._fused_stats_in_backward():
            self.rowstat.copy_(fused.combine_rowstats(self.rowstat, self.loss_kind, self.shard))

    def _exchange_grads(self):
        if self.shard.distributed:
            import torch.distributed as dist
            if self._fused_stats_in_backward():
                self.rowstat.copy_(fused.combine_rowstats(self.rowstat, self.loss_kind, self.shard))
            dist.all_reduce(self.dQ, group=self.shard.group)      # sum of the per-shard partial query gradients
            dist.all_reduce(self.g_ent, group=self.shard.group)   # dense table gradient: each rank filled its rows

    def _launch(self):
        self._stage_forward()
        self._exchange_stats()
        self._stage_backward()
        self._exchange_grads()
        self._stage_update()
        if self.p2p is not None:
            self._stage_exchange_p2p()
        elif self.dp_world > 1:
            self._exchange_dp()
            self._stage_apply_dp()

    @property
    def kernel_launches_per_step(self) -> int:
        """Kernels of this library per step (bench.py gpu_launches), counted from the step timeline under profiles/
        (timeline_bench_r1s2.txt: 31 launches, 29 of them this library's -- the other two are the gradient clear and a
        memset): query build 1; label rows of the table gradient 5 (label weights, label rows, permutation pack, 2
        segment-sum phases); dQ half 10 (label weights, bf16(Q), label rows, key pack, 2 segment-sum phases, label row
        sums, tile kernel, partial reduce, statistics reduce); dense dTable half 3 (label weights, bf16(Q), tile kernel);
        loss 1; query backward 1; two scatters 6 (permutation pack + 2 phases each); Adagrad 2 (or the exchange and
        apply kernels of the peer-memory mode).  KL (or fp32 math) adds the 5 forward-statistics kernels."""
        return 29 + (0 if self._fused_stats_in_backward() else 5)

    def _capture(self):
        """CUDA graphs of the three stages; NCCL collectives (sharded mode) stay outside the graphs."""
        keep = [t.detach().clone() for t in (self.ent, self.rel, self.opt.state[self.ent]["sum"],
                                             self.opt.state[self.rel]["sum"])]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):   # warm-up on a side stream (PyTorch's capture protocol)
            self._launch()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graphs = []
        whole = lambda: (self._stage_forward(), self._stage_backward(), self._stage_update())
        if self.p2p is not None:
            stages = [lambda: (whole(), self._stage_exchange_p2p())]     # compute + exchange + update: ONE graph
        elif self.shard.distributed:
            stages = [self._stage_forward, self._stage_backward, self._stage_update]
        elif self.dp_world > 1:
            stages = [whole, self._stage_apply_dp]
        else:
            stages = [whole]
        for fn in stages:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                fn()
            self.graphs.append(g)
        self.graph = self.graphs[0]
        self.graph_two_pass = None
        if self.flash:        # the same step on the two-pass kernels (online maximum): replayed when the flash pass failed
            self._use_flash = False
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                whole()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            self.graph_two_pass = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph_two_pass):
                whole()
            self._use_flash = True
        torch.cuda.synchronize()
        with torch.no_grad():   # the warm-up / capture runs must not count as training steps
            for dst, src in zip((self.ent, self.rel, self.opt.state[self.ent]["sum"], self.opt.state[self.rel]["sum"]),
                                keep):
                dst.copy_(src)
        if self.mirror is not None:
            lib.call("kgeb_to_bf16", lib.f32(self.ent.detach(), "table"), self.mirror.data_ptr(), self.ent.numel(),
                     lib.stream_ptr(self.ent))
        torch.cuda.synchronize()

    # -- public -------------------------------------------------------------------------------------
    @staticmethod
    def sort_perm(ids: torch.Tensor, size: int = 0) -> torch.Tensor:
        """Stable argsort (int32) of ids, zero-padded to `size` entries -- the order in which a deterministic scatter
        sums its rows.  Works on host or device tensors; part of the batch collate."""
        n = max(size, ids.numel(), 1)
        padded = torch.zeros(n, dtype=torch.int64, device=ids.device)
        padded[: ids.numel()] = ids
        return torch.sort(padded, stable=True).indices.to(torch.int32)

    def batch_perms(self, a_idx, p_idx, lab_col):
        """(a_perm, p_perm, lab_perm) of a batch, see __init__."""
        if lab_col.numel() > self.nnz_max:
            raise ValueError(f"batch has {lab_col.numel()} labels, stepper was built for at most {self.nnz_max}")
        return self.sort_perm(a_idx), self.sort_perm(p_idx), self.sort_perm(lab_col, self.nnz_max)

    def set_inputs(self, a_idx, p_idx, row_combine, lab_off, lab_col, perms=None):
        """Copies one batch into the static input buffers (host pinned or device tensors; non-blocking)."""
        if self.triples is not None:
            raise RuntimeError("this stepper builds its batch from triples inside the captured step: use set_triples()")
        if perms is None:
            perms = self.batch_perms(a_idx, p_idx, lab_col)
        self.a_perm.copy_(perms[0], non_blocking=True)
        self.p_perm.copy_(perms[1], non_blocking=True)
        self.lab_perm.copy_(perms[2], non_blocking=True)
        self.a_idx.copy_(a_idx, non_blocking=True)
        self.p_idx.copy_(p_idx, non_blocking=True)
        self.row_combine.copy_(row_combine, non_blocking=True)
        self.lab_off.copy_(lab_off, non_blocking=True)
        k = lab_col.numel()
        if k > self.nnz_max:
            raise ValueError(f"batch has {k} labels, stepper was built for at most {self.nnz_max}")
        self.lab_col[:k].copy_(lab_col, non_blocking=True)

    def pack_host_batch(self, a_idx, p_idx, row_combine, lab_off, lab_col) -> torch.Tensor:
        """Collate-side helper: one pinned byte buffer in the layout of the static inputs (see __init__)."""
        buf = torch.zeros(self.input_bytes.numel(), dtype=torch.uint8).pin_memory()
        v64 = buf[: self.n_i64 * 8].view(torch.int64)
        r = self.rows
        v64[:r] = a_idx
        v64[r:2 * r] = p_idx
        v64[2 * r:3 * r + 1] = lab_off
        k = lab_col.numel()
        if k > self.nnz_max:
            raise ValueError(f"batch has {k} labels, stepper was built for at most {self.nnz_max}")
        v64[3 * r + 1:3 * r + 1 + k] = lab_col
        v32 = buf[self.n_i64 * 8:].view(torch.int32)
        v32[:r] = row_combine
        v32[r:2 * r], v32[2 * r:3 * r], v32[3 * r:] = self.batch_perms(torch.as_tensor(a_idx), torch.as_tensor(p_idx),
                                                                      torch.as_tensor(lab_col))
        return buf

    def set_packed(self, packed: torch.Tensor):
        """One H2D copy of a packed (pinned) host batch into the static inputs."""
        if self.triples is not None:
            raise RuntimeError("this stepper builds its batch from triples inside the captured step: use set_triples()")
        self.input_bytes.copy_(packed, non_blocking=True)

    def step(self) -> torch.Tensor:
        """Runs one training step; returns the (device) loss tensor of this batch."""
        self.rate.refresh()       # the optimizer's current rates (the two-pass graph of a failed flash pass reads the same)
        if self.graph is None:
            self._launch()
            if self.flash and int(self.flash_status[0].item()) != 0:
                self.flash_fallbacks += 1
                self._use_flash = False
                self._launch()
                self._use_flash = True
        elif len(self.graphs) == 1:
            self.graphs[0].replay()
            # flash pass: one 4-byte read-back per step (the job reads the loss back every step as well, train.py:747,
            # 1043); a failed pass cleared its gradients, so nothing was updated and the step repeats on the two-pass graph
            if self.flash and int(self.flash_status[0].item()) != 0:
                self.flash_fallbacks += 1
                self.graph_two_pass.replay()
        elif self.dp_world > 1:
            self.graphs[0].replay()
            self._exchange_dp()
            self.graphs[1].replay()
        else:
            self.graphs[0].replay()
            self._exchange_stats()
            self.graphs[1].replay()
            self._exchange_grads()
            self.graphs[2].replay()
        for st in (self.opt.state[self.ent], self.opt.state[self.rel]):
            st["step"] += 1
        torch.autograd.graph.increment_version(self.ent)
        torch.autograd.graph.increment_version(self.rel)
        return self.loss if self.p2p is None else self.loss_global


class RowShardedAllEntityStepper:
    """All-entity training step (1vsAll / KvsAll, DOT scorers) with the entity table sharded BY ROW over the ranks of
    `shard.group` (SURVEY.md 8e, first row): rank g owns the rows [e_lo, e_hi) -- parameters, Adagrad state, bf16
    mirror and gradient -- and every rank sees the whole batch.  Per step the ranks exchange only

        all-reduce  [rows, d]   query-side entity rows (owners contribute theirs, zeros elsewhere)
        all-reduce  [rows, 4]   row statistics (max + rescaled sums for KL; plain sums for BCE)
        all-reduce  [rows, d]   partial dQ of the shards

    i.e. O(batch * d) bytes, independent of the table size; the dense table gradient, the label scatter and the Adagrad
    update stay local to the owner, the (small) relation table is replicated and updated identically everywhere.
    The model object keeps its full-size table: rows outside the shard go stale during training and are refreshed by
    sync_tables() (broadcast of every owner's rows) before evaluation or checkpointing.  The compute stages between
    the collectives are CUDA graphs; the collectives are plain NCCL calls."""

    def __init__(self, model: KgeModel, optimizer, rows: int, nnz_max: int, loss_kind: int, batch_size: int,
                 shard: fused.Shard, offset: float = 0.0, label_smoothing: float = 0.0, math_mode: int = lib.MATH_BF16,
                 use_graph: bool = True, peer_memory: bool = True, reciprocal: bool = False):
        """`peer_memory`: the three exchanges run as one-shot all-reduce KERNELS over torch symmetric memory
        (kgeb_p2p_allreduce, csrc/p2p.cu) inside ONE CUDA graph with the compute stages; where symmetric memory cannot be
        set up (or peer_memory=False) they are NCCL all-reduces between four separately captured graphs.
        `reciprocal`: as FusedAllEntityStepper -- the batch's _po queries arrive as sp_ rows on relation p + R
        (`kvsall_rows(..., inv_rel_offset=R)`); the 2 R-row relation table is replicated."""
        if model.get_scorer().kind != lib.DOT:
            raise NotImplementedError("the fused all-entity step serves the DOT scorers")
        if not shard.distributed:
            raise ValueError("RowShardedAllEntityStepper needs a distributed Shard (fused.Shard.of_rank)")
        self.inv_rel = _inverse_relation_offset(model, reciprocal, "RowShardedAllEntityStepper")
        _require_plain_model(model, "RowShardedAllEntityStepper", allow_reciprocal=reciprocal)
        self.model, self.opt, self.shard = model, optimizer, shard
        self.rows, self.nnz_max, self.loss_kind, self.batch_size = rows, nnz_max, loss_kind, batch_size
        self.offset, self.ls, self.math = float(offset), float(label_smoothing), math_mode
        self.ent = model.get_s_embedder().weight
        self.rel = model.get_p_embedder().weight
        dev = self.ent.device
        self.E, self.d = self.ent.shape
        self.dr = self.rel.shape[1]
        self.rate = _RateWords(optimizer, (self.ent, self.rel), "RowShardedAllEntityStepper", dev)
        self.eps_ent, self.eps_rel = self.rate.eps
        self.e_lo, self.e_hi = shard.e_lo, shard.e_hi
        self.n_loc = self.e_hi - self.e_lo
        f32 = dict(dtype=torch.float32, device=dev)
        i64 = dict(dtype=torch.int64, device=dev)
        nz = max(nnz_max, 1)
        self.a_idx, self.p_idx = torch.zeros(rows, **i64), torch.zeros(rows, **i64)
        self.row_combine = torch.zeros(rows, dtype=torch.int32, device=dev)
        self.lab_off, self.lab_col = torch.zeros(rows + 1, **i64), torch.zeros(nz, **i64)
        self.iota = torch.arange(rows, **i64)
        self.loc_ids = torch.zeros(rows, **i64)
        self.A = torch.zeros(rows, self.d, **f32)          # query-side entity rows, assembled by all-reduce
        self.Q, self.dQ = torch.empty(rows, self.d, **f32), torch.empty(rows, self.d, **f32)
        self.px = None
        if peer_memory:
            try:
                self._setup_peer(rows, dev)
            except (RuntimeError, ImportError, AttributeError) as exc:      # no symmetric memory on this box / build
                import sys
                print(f"[kgeb200] peer-memory exchange unavailable ({type(exc).__name__}: {exc}); using NCCL", file=sys.stderr)
                self.px = None
        self.da, self.dp = torch.empty(rows, self.d, **f32), torch.empty(rows, self.dr, **f32)
        # bf16 tiles: ONE gradient buffer [n_loc + 1, d] that is never cleared -- the tile kernel stores the dense part
        # (KGEB_BWD_OVERWRITE_TABLE), label rows and query-side rows are scattered on top; row n_loc collects the
        # query-side rows of other owners ("not mine") and is the only row zeroed per step.  fp32 tiles: two cleared buffers.
        self.one_buffer = math_mode == lib.MATH_BF16 and self.d % 16 == 0 and self.d <= 256
        # ... or none: Adagrad in the flush of the tile kernel, touched rows by a row kernel (see FusedAllEntityStepper)
        self.fuse_update = (self.one_buffer and self.d % 32 == 0 and self.n_loc > 0
                            and rows + nz <= lib.load().kgeb_touched_capacity()
                            and os.environ.get("KGEB_NO_FUSED_UPDATE", "0") in ("", "0"))
        if self.fuse_update:
            self.touched = _TouchedRows(self.n_loc, rows + nz, self.d, rows, nz, dev)
            self.g_all = self.g_ent = self.g_q = None
        else:
            self.g_all = torch.zeros(self.n_loc + 1, self.d, **f32)
            self.g_ent = self.g_all[:max(self.n_loc, 1)]                      # dense part + label rows, local rows only
            self.g_q = self.g_all if self.one_buffer else torch.zeros(self.n_loc + 1, self.d, **f32)   # last row = "not mine"
        self.g_rel = torch.zeros(self.rel.shape[0], self.dr, **f32)
        self.loss = torch.zeros((), **f32)
        self.rowstat = torch.empty(rows, 4, **f32)
        # flash pass (KL, bf16 tiles) in the peer-memory mode only: its status must be agreed on by all ranks inside the graph
        self.flash = fused.flash_supported(loss_kind, math_mode, self.d, self.ls) and self.px is not None
        self._use_flash = self.flash
        self.flash_fallbacks = 0
        if self.flash:
            self.rowstat_local = torch.empty(rows, 4, **f32)
            self.o_sum = torch.empty(rows, self.d, **f32)
            self.flash_status = torch.zeros(4, dtype=torch.int32, device=dev)      # reduced over the ranks (non-zero = failed)
        self.lse = torch.zeros(rows, **f32)
        L = lib.load()
        self.ws = torch.empty(L.kgeb_fused_workspace_bytes(rows, self.d, max(self.n_loc, 1), nz), dtype=torch.uint8, device=dev)
        self.ws2 = torch.empty_like(self.ws)
        self.sws = torch.empty(L.kgeb_scatter_workspace_bytes(rows, max(self.d, self.dr)), dtype=torch.uint8, device=dev)
        self.sws2 = torch.empty_like(self.sws)
        self.side = torch.cuda.Stream(device=dev)
        self.ev_touched = torch.cuda.Event()
        self.mirror = None
        if math_mode == lib.MATH_BF16 and self.d % 16 == 0 and self.d <= 256:
            self.mirror = torch.empty(max(self.n_loc, 1), self.d, dtype=torch.bfloat16, device=dev)
            self._refresh_mirror()
        self.graphs = None
        if use_graph:
            self._capture()

    # -- helpers -------------------------------------------------------------------------------------
    def _dst(self, which: str) -> torch.Tensor:
        """Where a producer writes this rank's PARTIAL of an exchanged quantity: the symmetric buffer the peers read
        (peer-memory mode) or the tensor NCCL reduces in place."""
        if self.px is not None:
            return {"A": self.A_part, "stat": self.stat_part, "dQ": self.dQ_part}[which]
        return {"A": self.A, "stat": self.rowstat, "dQ": self.dQ}[which]

    def _guard_flash(self, buf: torch.Tensor):
        """A failed flash pass on ANY rank: clear `buf` right before its Adagrad kernel (an exact no-op then)."""
        if self._use_flash:
            lib.call("kgeb_zero_if", self.flash_status.data_ptr(), buf.data_ptr(), buf.numel(), lib.stream_ptr(self.ent))

    def _ent_loc(self):
        return self.ent.detach()[self.e_lo:self.e_hi]

    def _refresh_mirror(self):
        if self.mirror is not None and self.n_loc > 0:
            lib.call("kgeb_to_bf16", self._ent_loc().data_ptr(), self.mirror.data_ptr(), self.n_loc * self.d,
                     lib.stream_ptr(self.ent))

    def _late_stats(self) -> bool:
        return self.loss_kind == lib.LOSS_BCE and self.mirror is not None

    def _loss_kernel(self):
        lib.call("kgeb_loss_from_rowstat", self.loss_kind, self.rowstat.data_ptr(), self.lab_off.data_ptr(), self.rows,
                 self.ls, self.E, 1.0 / self.batch_size, None, self.lse.data_ptr(), self.loss.data_ptr(),
                 lib.stream_ptr(self.ent))

    # -- compute stages (each one CUDA graph) and the collectives between them ----------------------------------
    def _stage_gather(self):
        st = lib.stream_ptr(self.ent)
        if self.fuse_update:
            # numbering of the touched rows: needed by the dTable kernel (second stream) and by the sparse scatters of the
            # update stage only -- off the critical path (a one-block sort: 27 us)
            cur = torch.cuda.current_stream()
            self.side.wait_stream(cur)
            with torch.cuda.stream(self.side):
                self.touched.build(self.a_idx, self.lab_col, self.lab_off[self.rows:], self.e_lo, self.e_hi,
                                   lib.stream_ptr(self.ent))
                self.ev_touched.record()
            if self.px is None:
                cur.wait_stream(self.side)         # separately captured stage graphs: nothing may stay forked
        elif self.one_buffer:
            self.g_all[self.n_loc:].zero_()
        else:
            self.g_ent.zero_(); self.g_q.zero_()
        self.g_rel.zero_()
        lib.call("kgeb_gather_rows_shard", self._ent_loc().data_ptr(), self.e_lo, self.e_hi, self.d, self.a_idx.data_ptr(),
                 1, self.rows, self._dst("A").data_ptr(), self.loc_ids.data_ptr(), st)

    def _stage_forward(self):
        st = lib.stream_ptr(self.ent)
        model_id = lib.MODELS[self.model.model]
        rel = self.rel.detach()
        lib.call("kgeb_query_build", model_id, 0, self.row_combine.data_ptr(), self.A.data_ptr(), self.iota.data_ptr(),
                 rel.data_ptr(), self.p_idx.data_ptr(), 1, self.rows, self.d, self.Q.data_ptr(), st)
        if self._use_flash:
            self.status_part.zero_()
            lib.call("kgeb_fused_flash_fwd", self.Q.data_ptr(), self.rows, self.d, self._ent_loc().data_ptr(), self.e_lo,
                     self.e_hi, self.E, self.lab_off.data_ptr(), self.lab_col.data_ptr(), self.nnz_max,
                     self.mirror.data_ptr(), self._dst("stat").data_ptr(), self.o_sum.data_ptr(), self.status_part.data_ptr(),
                     self.ws.data_ptr(), self.ws.numel(), st)
            self.rowstat_local.copy_(self._dst("stat"))
            # every rank learns whether ANY rank's pass failed (sum of the status words; an int 1 read as a float is a
            # non-zero denormal, the guard tests the 32-bit word)
            self._peer_allreduce("status", 4, 0, self.flash_status)
        elif not self._late_stats():
            lib.call("kgeb_fused_fwd", self.loss_kind, self.math, self.Q.data_ptr(), self.rows, self.d,
                     self._ent_loc().data_ptr(), self.e_lo, self.e_hi, self.E, self.lab_off.data_ptr(),
                     self.lab_col.data_ptr(), self.nnz_max, self.ls, self.offset,
                     None if self.mirror is None else self.mirror.data_ptr(), self._dst("stat").data_ptr(),
                     self.ws.data_ptr(), self.ws.numel(), st)

    def _stage_backward(self):
        st = lib.stream_ptr(self.ent)
        late = self._late_stats()
        if not late:
            self._loss_kernel()          # KL needs the global log-sum-exp before the backward
        lse = self.lse.data_ptr() if self.loss_kind == lib.LOSS_KL else None
        common = (self.loss_kind, self.math, self.Q.data_ptr(), self.rows, self.d, self._ent_loc().data_ptr(), self.e_lo,
                  self.e_hi, self.E, self.lab_off.data_ptr(), self.lab_col.data_ptr(), self.nnz_max, None, self.ls,
                  self.offset, lse, 1.0 / self.batch_size, None, None if self.mirror is None else self.mirror.data_ptr())
        cur = torch.cuda.current_stream()
        self.side.wait_stream(cur)
        dq_first = self.fuse_update and not self._use_flash
        if dq_first:
            # the fused update rewrites the bf16 mirror, which the dQ tile kernel reads: dQ first, the update kernel behind
            # its TILE kernel (kgeb_fused_bwd_wait_tiles), beside its small reduction kernels
            lib.call("kgeb_fused_bwd", *common, self._dst("dQ").data_ptr(), None,
                     self._dst("stat").data_ptr() if late else None, 0, self.ws.data_ptr(), self.ws.numel(), st)
        with torch.cuda.stream(self.side):
            if dq_first:
                lib.call("kgeb_fused_bwd_wait_tiles", lib.stream_ptr(self.ent))
            if self.fuse_update:
                # dense part + Adagrad in the tile kernel's flush; rows of the touched set are parked for _stage_update
                lib.call("kgeb_fused_bwd_update_sched", self.loss_kind, self.Q.data_ptr(), self.rows, self.d,
                         self._ent_loc().data_ptr(), self.e_lo, self.e_hi, self.E, self.lab_off.data_ptr(), self.ls, self.offset,
                         lse, 1.0 / self.batch_size, None, self.mirror.data_ptr(),
                         self.opt.state[self.ent]["sum"][self.e_lo:self.e_hi].data_ptr(), self.rate.ptr(0), self.eps_ent,
                         self.touched.slot_of.data_ptr(), self.touched.g_dense.data_ptr(),
                         self.flash_status.data_ptr() if self._use_flash else None, self.ws2.data_ptr(), self.ws2.numel(),
                         lib.stream_ptr(self.ent))
            else:
                # the dense part is stored (no cleared buffer), the label rows of this shard are scattered on top by the call
                lib.call("kgeb_fused_bwd", *common, None, self.g_ent.data_ptr(), None,
                         lib.BWD_OVERWRITE_TABLE if self.mirror is not None else 0, self.ws2.data_ptr(), self.ws2.numel(),
                         lib.stream_ptr(self.ent))
        if self._use_flash:      # dQ partial of this shard from o_sum and the GLOBAL log-sum-exp: no second table pass
            lib.call("kgeb_fused_flash_dq", self.Q.data_ptr(), self.rows, self.d, self._ent_loc().data_ptr(), self.e_lo,
                     self.e_hi, self.lab_off.data_ptr(), self.lab_col.data_ptr(), self.nnz_max,
                     self.rowstat_local.data_ptr(), self.lse.data_ptr(), 1.0 / self.batch_size, None, self.o_sum.data_ptr(),
                     self._dst("dQ").data_ptr(), self.ws.data_ptr(), self.ws.numel(), st)
        elif not dq_first:
            lib.call("kgeb_fused_bwd", *common, self._dst("dQ").data_ptr(), None,
                     self._dst("stat").data_ptr() if late else None, 0, self.ws.data_ptr(), self.ws.numel(), st)
        if self.px is None:      # separately captured stage graphs: nothing may stay forked at the end of one
            cur.wait_stream(self.side)

    def _stage_update(self):
        st = lib.stream_ptr(self.ent)
        model_id = lib.MODELS[self.model.model]
        rel = self.rel.detach()
        if self._late_stats():
            self._loss_kernel()
        lib.call("kgeb_query_bwd", model_id, 0, self.row_combine.data_ptr(), self.A.data_ptr(), self.iota.data_ptr(),
                 rel.data_ptr(), self.p_idx.data_ptr(), 1, self.rows, self.d, self.dQ.data_ptr(), self.da.data_ptr(),
                 self.dp.data_ptr(), st)
        lib.call("kgeb_scatter_add_rows", self.p_idx.data_ptr(), 1, self.dp.data_ptr(), self.rows, self.dr,
                 self.g_rel.data_ptr(), self.rel.shape[0], self.sws2.data_ptr(), self.sws2.numel(), st)
        self._guard_flash(self.g_rel)
        lib.call("kgeb_adagrad_dense_sched", rel.data_ptr(), self.opt.state[self.rel]["sum"].data_ptr(),
                 self.g_rel.data_ptr(), None, rel.numel(), self.rate.ptr(1), self.eps_rel, 0.0, None, st)
        if self.fuse_update:
            # label rows of this shard and the query-side rows it owns, summed per touched row (rows of other owners go to the
            # dummy slot) -- still underneath the dTable kernel; then the row kernel finishes the touched rows
            t = self.touched
            if self.px is not None:
                torch.cuda.current_stream().wait_event(self.ev_touched)
            lib.call("kgeb_fused_label_rows_to", self.loss_kind, self.Q.data_ptr(), self.rows, self.d,
                     self._ent_loc().data_ptr(), self.e_lo, self.e_hi, self.lab_off.data_ptr(), self.lab_col.data_ptr(),
                     self.nnz_max, None, self.ls, 1.0 / self.batch_size, None, t.slot_b.data_ptr(), t.cap + 1,
                     t.g_sparse.data_ptr(), self.ws.data_ptr(), self.ws.numel(), st)
            lib.call("kgeb_scatter_add_rows", t.slot_a.data_ptr(), 1, self.da.data_ptr(), self.rows, self.d,
                     t.g_sparse.data_ptr(), t.cap + 1, self.sws.data_ptr(), self.sws.numel(), st)
            if self.px is not None:
                torch.cuda.current_stream().wait_stream(self.side)
            t.update(self._ent_loc(), self.opt.state[self.ent]["sum"][self.e_lo:self.e_hi], self.mirror, self.rate.ptr(0),
                     self.eps_ent,
                     self.flash_status if self._use_flash else None, st)
            return
        if self.px is not None:
            # one graph for the whole step: the dense table gradient (second stream) is joined only here -- the dQ exchange,
            # the query-transform backward and the relation chain ran underneath the dTable tile kernel.  The query-side
            # rows below go ON TOP of what that kernel stored, so they must follow it.
            torch.cuda.current_stream().wait_stream(self.side)
        # query-side rows: every rank has the same da (dQ was all-reduced); each adds the rows it owns, the others go
        # to the dummy row n_loc
        lib.call("kgeb_scatter_add_rows", self.loc_ids.data_ptr(), 1, self.da.data_ptr(), self.rows, self.d,
                 self.g_q.data_ptr(), self.n_loc + 1, self.sws.data_ptr(), self.sws.numel(), st)
        if self.n_loc > 0:
            self._guard_flash(self.g_all[:self.n_loc])
            s_loc = self.opt.state[self.ent]["sum"][self.e_lo:self.e_hi]
            lib.call("kgeb_adagrad_dense_sched", self._ent_loc().data_ptr(), s_loc.data_ptr(), self.g_ent.data_ptr(),
                     None if self.one_buffer else self.g_q.data_ptr(), self.n_loc * self.d, self.rate.ptr(0), self.eps_ent, 0.0,
                     None if self.mirror is None else self.mirror.data_ptr(), st)

    def _setup_peer(self, rows: int, dev):
        """Partials of the three exchanges in ONE symmetric allocation [A_part | dQ_part | rowstat_part] + signal pad."""
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        n_a, n_s = rows * self.d, rows * 4
        flat = symm.empty(2 * n_a + n_s + 4, dtype=torch.float32, device=dev)
        hf = symm.rendezvous(flat, self.shard.group)
        pad = symm.empty(64, dtype=torch.int32, device=dev)
        hp = symm.rendezvous(pad, self.shard.group)
        flat.zero_(); pad.zero_()
        torch.cuda.synchronize()
        dist.barrier(self.shard.group)             # nobody signals before every pad is zero
        ptrs = [int(x) for x in hf.buffer_ptrs]
        self.px = dict(rank=hf.rank, world=hf.world_size, handles=(hf, hp), flat=flat, pad=pad,
                       pads=lib.ptr_array([int(x) for x in hp.buffer_ptrs]),
                       A=lib.ptr_array(ptrs), dQ=lib.ptr_array([x + 4 * n_a for x in ptrs]),
                       stat=lib.ptr_array([x + 8 * n_a for x in ptrs]),
                       status=lib.ptr_array([x + 8 * n_a + 4 * n_s for x in ptrs]),
                       epoch=torch.zeros(2, dtype=torch.int32, device=dev),
                       timeout=torch.zeros(1, dtype=torch.int32, device=dev))
        self.A_part = flat[:n_a].view(rows, self.d)
        self.dQ_part = flat[n_a:2 * n_a].view(rows, self.d)
        self.stat_part = flat[2 * n_a:2 * n_a + n_s].view(rows, 4)
        self.status_part = flat[2 * n_a + n_s:].view(torch.int32)       # this rank's flash status (4 words)

    def _peer_allreduce(self, which: str, numel: int, mode: int, out: torch.Tensor):
        x = self.px
        lib.call("kgeb_p2p_allreduce", x["pads"], x[which], x["rank"], x["world"], x["epoch"].data_ptr(),
                 x["timeout"].data_ptr(), numel, mode, out.data_ptr(), lib.stream_ptr(self.ent))

    def check_peer(self):
        """Host check (one sync): no peer-memory barrier ran into its timeout."""
        if self.px is not None and int(self.px["timeout"].item()) != 0:
            raise RuntimeError("a peer did not arrive at a peer-memory barrier")

    def _exchange(self, which: int):
        import torch.distributed as dist
        grp = self.shard.group
        if self.px is not None:
            # producers wrote their partials into the symmetric buffers (A_part / stat_part / dQ_part); results land in the
            # local tensors the next stage reads
            if which == 0:
                self._peer_allreduce("A", self.A.numel(), 0, self.A)
            elif which == 1:
                if not self._late_stats():
                    self._peer_allreduce("stat", self.rowstat.numel(), 1 if self.loss_kind == lib.LOSS_KL else 0, self.rowstat)
            else:
                self._peer_allreduce("dQ", self.dQ.numel(), 0, self.dQ)
                if self._late_stats():
                    self._peer_allreduce("stat", self.rowstat.numel(), 0, self.rowstat)
            return
        if which == 0:
            dist.all_reduce(self.A, group=grp)
        elif which == 1:
            if not self._late_stats():
                self.rowstat.copy_(fused.combine_rowstats(self.rowstat, self.loss_kind, self.shard))
        else:
            dist.all_reduce(self.dQ, group=grp)
            if self._late_stats():
                self.rowstat.copy_(fused.combine_rowstats(self.rowstat, self.loss_kind, self.shard))

    def _stages(self):
        return [self._stage_gather, self._stage_forward, self._stage_backward, self._stage_update]

    def _launch(self):
        for i, fn in enumerate(self._stages()):
            fn()
            if i < 3:
                self._exchange(i)

    def _capture(self):
        keep = [t.detach().clone() for t in (self.ent, self.rel, self.opt.state[self.ent]["sum"],
                                             self.opt.state[self.rel]["sum"])]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            self._launch()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graphs = []
        if self.px is not None:
            # compute stages AND exchanges in one graph.  The capture itself launches nothing, but every rank must replay
            # the same number of collectives: the warm-up above ran exactly one step on every rank.
            import torch.distributed as dist
            dist.barrier(self.shard.group)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._launch()
            self.graphs.append(g)
            self.graph_two_pass = None
            if self.flash:     # the same step on the two-pass kernels, replayed by every rank when any rank's flash pass failed
                self._use_flash = False
                with torch.cuda.stream(side):
                    self._launch()
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize()
                dist.barrier(self.shard.group)
                self.graph_two_pass = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.graph_two_pass):
                    self._launch()
                self._use_flash = True
        else:
            for fn in self._stages():
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    fn()
                self.graphs.append(g)
        torch.cuda.synchronize()
        with torch.no_grad():
            for dst, src in zip((self.ent, self.rel, self.opt.state[self.ent]["sum"], self.opt.state[self.rel]["sum"]), keep):
                dst.copy_(src)
        self._refresh_mirror()
        torch.cuda.synchronize()

    # -- public -------------------------------------------------------------------------------------
    def set_inputs(self, a_idx, p_idx, row_combine, lab_off, lab_col, perms=None):
        if lab_col.numel() > self.nnz_max:
            raise ValueError(f"batch has {lab_col.numel()} labels, stepper was built for at most {self.nnz_max}")
        self.a_idx.copy_(a_idx, non_blocking=True)
        self.p_idx.copy_(p_idx, non_blocking=True)
        self.row_combine.copy_(row_combine, non_blocking=True)
        self.lab_off.copy_(lab_off, non_blocking=True)
        self.lab_col[: lab_col.numel()].copy_(lab_col, non_blocking=True)

    def step(self) -> torch.Tensor:
        self.rate.refresh()
        if self.graphs is None:
            self._launch()
            if self.flash and int(self.flash_status[0].item()) != 0:
                self.flash_fallbacks += 1
                self._use_flash = False
                self._launch()
                self._use_flash = True
        elif len(self.graphs) == 1:
            self.graphs[0].replay()
            if self.flash and int(self.flash_status[0].item()) != 0:       # the same on every rank
                self.flash_fallbacks += 1
                self.graph_two_pass.replay()
        else:
            for i, g in enumerate(self.graphs):
                g.replay()
                if i < 3:
                    self._exchange(i)
        for st in (self.opt.state[self.ent], self.opt.state[self.rel]):
            st["step"] += 1
        torch.autograd.graph.increment_version(self.ent)
        torch.autograd.graph.increment_version(self.rel)
        return self.loss

    def sync_tables(self):
        """Every owner broadcasts its rows of the entity table and of the Adagrad state: afterwards all ranks hold the
        complete, current table (evaluation, checkpoints)."""
        import torch.distributed as dist
        world = dist.get_world_size(self.shard.group)
        ranks = dist.get_process_group_ranks(self.shard.group)
        with torch.no_grad():
            for r in range(world):
                sh = fused.Shard.of_rank(self.E, r, world, self.shard.group)
                if sh.e_hi > sh.e_lo:
                    dist.broadcast(self.ent.data[sh.e_lo:sh.e_hi], src=ranks[r], group=self.shard.group)
                    dist.broadcast(self.opt.state[self.ent]["sum"][sh.e_lo:sh.e_hi], src=ranks[r], group=self.shard.group)
        torch.autograd.graph.increment_version(self.ent)


def kvsall_rows(queries: torch.Tensor, query_type: torch.Tensor, inv_rel_offset: int = 0):
    """KvsAll batch -> (a_idx, p_idx, row_combine): sp_ rows use (s,p) = (q0,q1); _po rows (p,o) = (q0,q1).
    inv_rel_offset = R > 0 (reciprocal relations model): a _po row (p,o) becomes the sp_ row (o, p + R)."""
    qt = query_type.to(torch.int32)
    a = torch.where(qt == 0, queries[:, 0], queries[:, 1])
    p = torch.where(qt == 0, queries[:, 1], queries[:, 0])
    if inv_rel_offset > 0:
        p = torch.where(qt == 0, p, p + inv_rel_offset)
        qt = torch.zeros_like(qt)
    return a.contiguous(), p.contiguous(), qt.contiguous()


class FusedNegSamplingStepper:
    """Static-shape negative-sampling step (train.py:823-999, implementation "triple", slots S and O) for all seven
    scorers: per slot   query vector of the positive -> pair scores against its 1+N candidates -> loss + dL/dscores ->
    pair backward (dQ, candidate gradient rows) -> query-transform backward;   then the sorted scatters of the candidate /
    query-side rows and Adagrad on both tables.  No autograd, no B*(1+N) triple expansion; replayed as one CUDA graph.
    """

    def __init__(self, model: KgeModel, optimizer, batch_size: int, num_neg_s: int, num_neg_o: int, loss_kind: int,
                 offset: float = 0.0, use_graph: bool = True, dp_group=None, segment_bwd: bool = False,
                 fused_slot: bool = True, deterministic: bool = True, reciprocal: bool = False):
        """`segment_bwd`: candidate gradients without materialised rows (csrc/ns_segment.cu: pairs sorted by candidate, one
        warp per distinct candidate) instead of pairs_bwd's dC rows + the sorted scatter; measured slower than the sort it
        replaces (0.509 vs 0.414 ms per C3 step, DESIGN.md section 8): kept as a tuning path.
        `dp_group`: data-parallel replicas (every rank its own batch of `batch_size` triples; SURVEY.md 8e, second row):
        gradients of both tables are exchanged and applied by the peer-memory kernels of csrc/p2p.cu inside the same CUDA
        graph; loss terms are scaled by the global batch so that all replicas apply the identical update
        (tests/p2p_ns_check.py; profiles/r2/p2p_ns_check_2.log).
        `reciprocal`: reciprocal relations model (2 R relation rows): slot S scores the sp_ query (o, p + R) against its
        subject candidates (ReciprocalRelationsModel.score_spo(..., "s")), its relation gradient rows go to p + R; the
        shifted ids are computed inside the captured graph."""
        self.inv_rel = _inverse_relation_offset(model, reciprocal, "FusedNegSamplingStepper")
        _require_plain_model(model, "FusedNegSamplingStepper", allow_reciprocal=reciprocal)
        # fused_slot: scores, loss, dQ and the candidate gradient of a slot in ONE kernel (kgeb_ns_fused) instead of
        # kgeb_pairs_score + kgeb_ns_loss + kgeb_pairs_bwd -- same sums in the same order, bit-identical results.
        # deterministic=False (opt-in): that kernel adds the candidate gradients straight into the dense gradient with
        # vector reductions -- no materialised gradient rows, no sort -- at the price of order-dependent rounding.
        self.model, self.opt = model, optimizer
        self.fused_slot = bool(fused_slot) and not segment_bwd and model.get_s_embedder().weight.shape[1] % 4 == 0
        self.deterministic = bool(deterministic) or not self.fused_slot
        self.B, self.N = batch_size, {0: int(num_neg_s), 2: int(num_neg_o)}
        self.loss_kind, self.offset = loss_kind, float(offset)
        self.kind = model.get_scorer().kind
        self.ent, self.rel = model.get_s_embedder().weight, model.get_p_embedder().weight
        dev = self.ent.device
        self.E, self.d = self.ent.shape
        self.dr = self.rel.shape[1]
        self.rate = _RateWords(optimizer, (self.ent, self.rel), "FusedNegSamplingStepper", dev)
        self.eps_ent, self.eps_rel = self.rate.eps
        if dp_group is not None and self.eps_ent != self.eps_rel:
            raise NotImplementedError("the peer-memory exchange applies one eps to both tables")
        f32 = dict(dtype=torch.float32, device=dev)
        i64 = dict(dtype=torch.int64, device=dev)
        B = batch_size
        self.triples = torch.zeros(3, B, **i64)            # static inputs: rows s, p, o
        self.p_inv = torch.zeros(B, **i64) if self.inv_rel else None       # p + R: relation ids of slot S
        self.neg = {slot: torch.zeros(B, n, **i64) for slot, n in self.N.items() if n > 0}
        self.slots = [slot for slot in (0, 2) if self.N[slot] > 0]
        self.buf = {}
        for slot in self.slots:
            m = 1 + self.N[slot]
            self.buf[slot] = dict(cand=torch.zeros(B, m, **i64), scores=torch.empty(B, m, **f32), G=torch.empty(B, m, **f32),
                                  rows=torch.empty(B, **f32), Q=torch.empty(B, self.d, **f32), dQ=torch.empty(B, self.d, **f32),
                                  dC=torch.empty(B * m, self.d, **f32), da=torch.empty(B, self.d, **f32),
                                  dp=torch.empty(B, self.dr, **f32))
        self.segment_bwd = bool(segment_bwd)
        if self.segment_bwd:
            nseg = B * (1 + max(self.N.values()))
            self.segws = torch.empty(lib.load().kgeb_ns_segment_workspace_bytes(nseg), dtype=torch.uint8, device=dev)
        self.px = None
        self.global_batch = B
        if dp_group is not None:
            n_e, n_r = self.E * self.d, self.rel.shape[0] * self.dr
            self.px = PeerExchange(dp_group, n_e, n_r, dev)
            self.global_batch = B * self.px.world
            self.g_ent = self.px.flat[:n_e].view(self.E, self.d)
            self.g_rel = self.px.flat[n_e:n_e + n_r].view(self.rel.shape[0], self.dr)
            self.loss = self.px.flat[n_e + n_r:n_e + n_r + 1].view(())
        else:
            self.g_ent = torch.zeros(self.E, self.d, **f32)
            self.g_rel = torch.zeros(self.rel.shape[0], self.dr, **f32)
            self.loss = torch.zeros((), **f32)
        nmax = B * (1 + max(self.N.values()))
        self.sws = torch.empty(lib.load().kgeb_scatter_workspace_bytes(nmax, max(self.d, self.dr)), dtype=torch.uint8,
                               device=dev)
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        if use_graph:
            self._capture()

    def _launch(self):
        st = lib.stream_ptr(self.ent)
        model_id = lib.MODELS[self.model.model]
        ent, rel = self.ent.detach(), self.rel.detach()
        B, d = self.B, self.d
        s_idx, p_fwd, o_idx = self.triples[0], self.triples[1], self.triples[2]
        self.g_ent.zero_(); self.g_rel.zero_()
        if self.inv_rel:
            torch.add(p_fwd, self.inv_rel, out=self.p_inv)
        for slot in self.slots:
            b = self.buf[slot]
            m = 1 + self.N[slot]
            # slot O: query (s,p) against object candidates; slot S: query (p,o) against subject candidates -- for a
            # reciprocal model the sp_ query (o, p + R)
            combine, a_idx, target, p_idx = (lib.SP_, s_idx, o_idx, p_fwd) if slot == 2 else (
                (lib.SP_, o_idx, s_idx, self.p_inv) if self.inv_rel else (lib._PO, o_idx, s_idx, p_fwd))
            lib.call("kgeb_query_build", model_id, combine, None, ent.data_ptr(), a_idx.data_ptr(), rel.data_ptr(),
                     p_idx.data_ptr(), 1, B, d, b["Q"].data_ptr(), st)
            lib.call("kgeb_ns_candidates", target.data_ptr(), self.neg[slot].data_ptr(), B, self.N[slot],
                     b["cand"].data_ptr(), st)
            if self.fused_slot:
                lib.call("kgeb_ns_fused", self.kind, self.loss_kind, b["Q"].data_ptr(), ent.data_ptr(), b["cand"].data_ptr(), B, m,
                         d, self.offset, 1.0 / self.global_batch, b["dQ"].data_ptr(),
                         b["dC"].data_ptr() if self.deterministic else None,
                         None if self.deterministic else self.g_ent.data_ptr(), b["rows"].data_ptr(), st)
                lib.call("kgeb_query_bwd", model_id, combine, None, ent.data_ptr(), a_idx.data_ptr(), rel.data_ptr(),
                         p_idx.data_ptr(), 1, B, d, b["dQ"].data_ptr(), b["da"].data_ptr(), b["dp"].data_ptr(), st)
                if self.deterministic:
                    lib.call("kgeb_scatter_add_rows", b["cand"].data_ptr(), 1, b["dC"].data_ptr(), B * m, d,
                             self.g_ent.data_ptr(), self.E, self.sws.data_ptr(), self.sws.numel(), st)
                lib.call("kgeb_scatter_add_rows", a_idx.data_ptr(), 1, b["da"].data_ptr(), B, d, self.g_ent.data_ptr(),
                         self.E, self.sws.data_ptr(), self.sws.numel(), st)
                lib.call("kgeb_scatter_add_rows", p_idx.data_ptr(), 1, b["dp"].data_ptr(), B, self.dr,
                         self.g_rel.data_ptr(), self.rel.shape[0], self.sws.data_ptr(), self.sws.numel(), st)
                continue
            lib.call("kgeb_pairs_score", self.kind, b["Q"].data_ptr(), ent.data_ptr(), b["cand"].data_ptr(), 1, B, m, d,
                     b["scores"].data_ptr(), st)
            lib.call("kgeb_ns_loss", self.loss_kind, b["scores"].data_ptr(), B, m, self.offset, 1.0 / self.global_batch,
                     b["G"].data_ptr(), b["rows"].data_ptr(), st)
            if self.segment_bwd:
                lib.call("kgeb_ns_bwd_q", self.kind, b["Q"].data_ptr(), ent.data_ptr(), b["cand"].data_ptr(), B, m, d,
                         b["G"].data_ptr(), b["scores"].data_ptr(), b["dQ"].data_ptr(), st)
                lib.call("kgeb_query_bwd", model_id, combine, None, ent.data_ptr(), a_idx.data_ptr(), rel.data_ptr(),
                         p_idx.data_ptr(), 1, B, d, b["dQ"].data_ptr(), b["da"].data_ptr(), b["dp"].data_ptr(), st)
                lib.call("kgeb_ns_cand_grad", self.kind, b["Q"].data_ptr(), ent.data_ptr(), b["cand"].data_ptr(), B, m, d,
                         b["G"].data_ptr(), b["scores"].data_ptr(), self.E, self.g_ent.data_ptr(), self.segws.data_ptr(),
                         self.segws.numel(), st)
            else:
                lib.call("kgeb_pairs_bwd", self.kind, b["Q"].data_ptr(), ent.data_ptr(), b["cand"].data_ptr(), 1, B, m, d,
                         b["G"].data_ptr(), b["scores"].data_ptr(), b["dQ"].data_ptr(), b["dC"].data_ptr(), st)
                lib.call("kgeb_query_bwd", model_id, combine, None, ent.data_ptr(), a_idx.data_ptr(), rel.data_ptr(),
                         p_idx.data_ptr(), 1, B, d, b["dQ"].data_ptr(), b["da"].data_ptr(), b["dp"].data_ptr(), st)
                lib.call("kgeb_scatter_add_rows", b["cand"].data_ptr(), 1, b["dC"].data_ptr(), B * m, d,
                         self.g_ent.data_ptr(), self.E, self.sws.data_ptr(), self.sws.numel(), st)
            lib.call("kgeb_scatter_add_rows", a_idx.data_ptr(), 1, b["da"].data_ptr(), B, d, self.g_ent.data_ptr(),
                     self.E, self.sws.data_ptr(), self.sws.numel(), st)
            lib.call("kgeb_scatter_add_rows", p_idx.data_ptr(), 1, b["dp"].data_ptr(), B, self.dr,
                     self.g_rel.data_ptr(), self.rel.shape[0], self.sws.data_ptr(), self.sws.numel(), st)
        torch.sum(torch.stack([self.buf[s]["rows"].sum() for s in self.slots]), dim=0, out=self.loss)
        s_ent, s_rel = self.opt.state[self.ent]["sum"], self.opt.state[self.rel]["sum"]
        if self.px is not None:     # exchange + update of the owned slices + gather of the new weights, in this graph
            self.px.exchange_and_update(ent, s_ent, None, rel, s_rel, self.rate.words.data_ptr(), self.eps_ent, st)
            return
        lib.call("kgeb_adagrad_dense_sched", ent.data_ptr(), s_ent.data_ptr(), self.g_ent.data_ptr(), None, ent.numel(),
                 self.rate.ptr(0), self.eps_ent, 0.0, None, st)
        lib.call("kgeb_adagrad_dense_sched", rel.data_ptr(), s_rel.data_ptr(), self.g_rel.data_ptr(), None, rel.numel(),
                 self.rate.ptr(1), self.eps_rel, 0.0, None, st)

    def _capture(self):
        keep = [t.detach().clone() for t in (self.ent, self.rel, self.opt.state[self.ent]["sum"],
                                             self.opt.state[self.rel]["sum"])]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            self._launch()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self._launch()
        torch.cuda.synchronize()
        with torch.no_grad():
            for dst, src in zip((self.ent, self.rel, self.opt.state[self.ent]["sum"], self.opt.state[self.rel]["sum"]),
                                keep):
                dst.copy_(src)
        torch.cuda.synchronize()

    def set_inputs(self, triples: torch.Tensor, negative_samples):
        """triples [B,3]; negative_samples = list of [B,N_slot] for slots S, P, O (as the reference's collate emits)."""
        self.triples.copy_(triples.t(), non_blocking=True)
        for slot in self.slots:
            self.neg[slot].copy_(negative_samples[slot], non_blocking=True)

    def step(self) -> torch.Tensor:
        self.rate.refresh()
        if self.graph is not None:
            self.graph.replay()
        else:
            self._launch()
        for st in (self.opt.state[self.ent], self.opt.state[self.rel]):
            st["step"] += 1
        torch.autograd.graph.increment_version(self.ent)
        torch.autograd.graph.increment_version(self.rel)
        return self.loss if self.px is None else self.px.loss_global


# ---------------------------------------------------------------------------------------------
# SURVEY.md 8(e), second row: negative sampling, data-parallel over triples with ROW-SHARDED embedding tables
# ---------------------------------------------------------------------------------------------
class RowExchange:
    """Routing of embedding-row requests to their owners and of row gradients back (all-to-all-v over the process group).
    Rank g owns the rows [g * per, (g + 1) * per) of a table of `num_rows` rows, per = ceil(num_rows / world).
    Works on CPU tensors with gloo as well (tests/test_host_logic.py) -- it is index arithmetic plus three collectives."""

    def __init__(self, num_rows: int, group=None):
        import torch.distributed as dist
        self.group = group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.per = (num_rows + self.world - 1) // self.world
        self.lo = min(self.rank * self.per, num_rows)
        self.hi = min(self.lo + self.per, num_rows)

    def _a2a(self, x: torch.Tensor, send: list, recv: list) -> torch.Tensor:
        import torch.distributed as dist
        out = torch.empty((sum(recv),) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
        dist.all_to_all_single(out, x.contiguous(), output_split_sizes=recv, input_split_sizes=send, group=self.group)
        return out

    def plan(self, ids: torch.Tensor) -> dict:
        """ids int64 [n] (duplicates allowed) -> routing plan.  One host sync (the split sizes)."""
        import torch.distributed as dist
        owner = torch.div(ids, self.per, rounding_mode="floor")
        order = torch.sort(owner, stable=True).indices           # requests grouped by owner, original order within one
        send = torch.bincount(owner, minlength=self.world)
        recv = torch.empty_like(send)
        dist.all_to_all_single(recv, send, group=self.group)
        send_l, recv_l = send.tolist(), recv.tolist()
        wanted = self._a2a(ids[order], send_l, recv_l) - self.lo     # local row numbers other ranks ask me for
        return {"order": order, "send": send_l, "recv": recv_l, "wanted": wanted, "n": ids.numel()}

    def fetch(self, plan: dict, gather) -> torch.Tensor:
        """rows [n, d] of the requested ids; `gather(local_rows int64) -> [m, d]` reads this rank's shard."""
        back = self._a2a(gather(plan["wanted"]), plan["recv"], plan["send"])
        rows = torch.empty_like(back)
        rows[plan["order"]] = back
        return rows

    def push(self, plan: dict, grad_rows: torch.Tensor):
        """Row gradients [n, d] (one per requested id) -> (local row numbers, rows) at their owners, ordered by
        (sender rank, position in the sender's request list): a deterministic order for the owner's segment sums."""
        return plan["wanted"], self._a2a(grad_rows[plan["order"]], plan["send"], plan["recv"])


class ShardedNegSamplingStepper:
    """Negative-sampling training step (train.py:823-999, implementation "triple", slots S and O) data-parallel over the
    triples of a batch with the ENTITY TABLE SHARDED BY ROW over the ranks (SURVEY.md 8e, second row):

        every rank: its share of the batch -> ids of all rows it needs (positives' s / o, negatives of both slots)
        all-to-all-v   ids to the row owners, rows back                                  (RowExchange.fetch)
        local          query vectors -> pair scores -> loss -> pair backward on the fetched rows (the kernels of
                       FusedNegSamplingStepper, the fetched rows being the "table")
        all-to-all-v   one gradient row per requested row back to its owner               (RowExchange.push)
        owner          sorted, deterministic segment sum into its rows' gradient + Adagrad on its rows + state
        relation table replicated: its (small) gradient and the loss are all-reduced, every rank applies the same update

    The model object keeps a full-size table whose foreign rows go stale; sync_tables() gathers the owners' rows.
    Eager (the all-to-all sizes change per batch); the single-GPU step stays FusedNegSamplingStepper."""

    def __init__(self, model: KgeModel, optimizer, batch_size: int, num_neg_s: int, num_neg_o: int, loss_kind: int,
                 group=None, offset: float = 0.0):
        import torch.distributed as dist
        _require_plain_model(model, "ShardedNegSamplingStepper")
        self.model, self.opt, self.group = model, optimizer, group
        self.B, self.N = batch_size, {0: int(num_neg_s), 2: int(num_neg_o)}
        self.loss_kind, self.offset = loss_kind, float(offset)
        self.kind = model.get_scorer().kind
        self.ent, self.rel = model.get_s_embedder().weight, model.get_p_embedder().weight
        self.E, self.d = self.ent.shape
        self.dr = self.rel.shape[1]
        # eager: the rates are read from the optimizer's groups and passed by value every step (adagrad_rates)
        self.eps_ent, self.eps_rel = [float(g["eps"]) for g in
                                      _adagrad_groups(optimizer, (self.ent, self.rel), "ShardedNegSamplingStepper")]
        self.ex = RowExchange(self.E, group)
        self.world = self.ex.world
        self.global_batch = batch_size * self.world
        dev = self.ent.device
        self.n_loc = self.ex.hi - self.ex.lo
        self.g_loc = torch.zeros(max(self.n_loc, 1), self.d, dtype=torch.float32, device=dev)
        self.g_rel = torch.zeros_like(self.rel)
        self.loss = torch.zeros((), dtype=torch.float32, device=dev)
        self.slots = [s for s in (0, 2) if self.N[s] > 0]

    def _ws(self, n: int) -> torch.Tensor:
        return ops._workspace(self.ent.device, lib.load().kgeb_scatter_workspace_bytes(max(n, 1), max(self.d, self.dr)))

    def step(self, triples: torch.Tensor, negative_samples) -> torch.Tensor:
        """triples [B,3] and negative_samples (list per slot S, P, O of [B, N_slot]) of THIS rank's share of the batch."""
        import torch.distributed as dist
        dev, B, d = self.ent.device, self.B, self.d
        st = lib.stream_ptr(self.ent)
        model_id = lib.MODELS[self.model.model]
        ent, rel = self.ent.detach(), self.rel.detach()
        t = triples.to(dev).long()
        s_idx, p_idx, o_idx = t[:, 0].contiguous(), t[:, 1].contiguous(), t[:, 2].contiguous()
        negs = {slot: negative_samples[slot].to(dev).long().contiguous() for slot in self.slots}
        # requested rows: [s (B) | o (B) | negatives of slot S (B*N_S) | negatives of slot O (B*N_O)]
        parts, base = [s_idx, o_idx], {}
        off = 2 * B
        for slot in self.slots:
            base[slot] = off
            parts.append(negs[slot].view(-1))
            off += B * self.N[slot]
        ids = torch.cat(parts)
        plan = self.ex.plan(ids)
        loc = ent[self.ex.lo:self.ex.hi]
        rows = self.ex.fetch(plan, lambda w: ops.gather_rows(loc, w) if w.numel() else loc.new_zeros(0, d))
        g_rows = torch.zeros_like(rows)                    # gradient of every fetched row (each is referenced by position)
        self.g_rel.zero_()
        ar = torch.arange(B, dtype=torch.int64, device=dev)
        slot_loss = []
        for slot in self.slots:
            m = 1 + self.N[slot]
            # slot O: query (s,p) against [o | negatives]; slot S: query (p,o) against [s | negatives]
            combine, a_pos, tgt_pos = (lib.SP_, ar, ar + B) if slot == 2 else (lib._PO, ar + B, ar)
            Q = torch.empty(B, d, dtype=torch.float32, device=dev)
            lib.call("kgeb_query_build", model_id, combine, None, rows.data_ptr(), a_pos.data_ptr(), rel.data_ptr(),
                     p_idx.data_ptr(), 1, B, d, Q.data_ptr(), st)
            cand = torch.cat((tgt_pos[:, None], base[slot] + torch.arange(B * self.N[slot], device=dev).view(B, -1)), 1).contiguous()
            scores = torch.empty(B, m, dtype=torch.float32, device=dev)
            G, lrows = torch.empty_like(scores), torch.empty(B, dtype=torch.float32, device=dev)
            lib.call("kgeb_pairs_score", self.kind, Q.data_ptr(), rows.data_ptr(), cand.data_ptr(), 1, B, m, d,
                     scores.data_ptr(), st)
            lib.call("kgeb_ns_loss", self.loss_kind, scores.data_ptr(), B, m, self.offset, 1.0 / self.global_batch,
                     G.data_ptr(), lrows.data_ptr(), st)
            dQ, dC = torch.empty_like(Q), torch.empty(B * m, d, dtype=torch.float32, device=dev)
            lib.call("kgeb_pairs_bwd", self.kind, Q.data_ptr(), rows.data_ptr(), cand.data_ptr(), 1, B, m, d, G.data_ptr(),
                     scores.data_ptr(), dQ.data_ptr(), dC.data_ptr(), st)
            da, dp = torch.empty_like(Q), torch.empty(B, self.dr, dtype=torch.float32, device=dev)
            lib.call("kgeb_query_bwd", model_id, combine, None, rows.data_ptr(), a_pos.data_ptr(), rel.data_ptr(),
                     p_idx.data_ptr(), 1, B, d, dQ.data_ptr(), da.data_ptr(), dp.data_ptr(), st)
            g_rows.index_add_(0, cand.view(-1), dC)          # positions are distinct within a slot: a plain placement
            g_rows.index_add_(0, a_pos, da)
            lib.call("kgeb_scatter_add_rows", p_idx.data_ptr(), 1, dp.data_ptr(), B, self.dr, self.g_rel.data_ptr(),
                     self.rel.shape[0], self._ws(B).data_ptr(), self._ws(B).numel(), st)
            slot_loss.append(lrows.sum())
        # gradient rows to their owners; the owners' deterministic segment sums + update of the local rows
        wanted, recv = self.ex.push(plan, g_rows)
        self.g_loc.zero_()
        if wanted.numel() and self.n_loc > 0:
            ws = self._ws(wanted.numel())
            lib.call("kgeb_scatter_add_rows", wanted.contiguous().data_ptr(), 1, recv.data_ptr(), wanted.numel(), d,
                     self.g_loc.data_ptr(), self.n_loc, ws.data_ptr(), ws.numel(), st)
        flat = torch.cat((self.g_rel.view(-1), torch.stack(slot_loss).sum().view(1)))
        dist.all_reduce(flat, group=self.group)
        self.g_rel.copy_(flat[:-1].view_as(self.g_rel))
        self.loss.copy_(flat[-1])
        s_ent, s_rel = self.opt.state[self.ent]["sum"], self.opt.state[self.rel]["sum"]
        lr_ent, lr_rel = adagrad_rates(self.opt, (self.ent, self.rel))
        if self.n_loc > 0:
            lib.call("kgeb_adagrad_dense", loc.data_ptr(), s_ent[self.ex.lo:self.ex.hi].data_ptr(), self.g_loc.data_ptr(), None,
                     self.n_loc * d, lr_ent, self.eps_ent, 0.0, None, st)
        lib.call("kgeb_adagrad_dense", rel.data_ptr(), s_rel.data_ptr(), self.g_rel.data_ptr(), None, rel.numel(), lr_rel,
                 self.eps_rel, 0.0, None, st)
        for stt in (self.opt.state[self.ent], self.opt.state[self.rel]):
            stt["step"] += 1
        torch.autograd.graph.increment_version(self.ent)
        torch.autograd.graph.increment_version(self.rel)
        return self.loss

    def sync_tables(self):
        """Every owner broadcasts its rows of the entity table and of the Adagrad state (evaluation, checkpoints)."""
        import torch.distributed as dist
        ranks = dist.get_process_group_ranks(self.group) if self.group is not None else list(range(self.world))
        with torch.no_grad():
            for r in range(self.world):
                lo = min(r * self.ex.per, self.E)
                hi = min(lo + self.ex.per, self.E)
                if hi > lo:
                    dist.broadcast(self.ent.data[lo:hi], src=ranks[r], group=self.group)
                    dist.broadcast(self.opt.state[self.ent]["sum"][lo:hi], src=ranks[r], group=self.group)
        torch.autograd.graph.increment_version(self.ent)
