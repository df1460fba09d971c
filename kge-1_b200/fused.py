"""Fused all-entity score + loss (forward and backward) and fused filtered rank counting.

`AllEntityLoss` replaces the reference's  scores = model.score_sp/po(...) ; loss(scores, labels) / batch_size ;
.backward()  chain (train.py:732-750, 1040-1057 with loss.py:137-159, 192-213) for the DOT scorers and, on the fp32
CUDA-core tiles, for TransE and RotatE (`kind`): the [B, E] score matrix is never written; labels are a CSR over the batch rows.  With an entity-sharded
table (`shard`), per-row statistics and the query gradient are all-reduced over the process group
(SURVEY.md 8e); integer rank counts are exact under sharding.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
import torch.distributed as dist

from . import lib, ops


class Shard:
    """Contiguous entity range [e_lo, e_hi) of a table of E rows held by this rank."""

    def __init__(self, e_lo: int, e_hi: int, num_entities: int, group=None):
        self.e_lo, self.e_hi, self.num_entities, self.group = int(e_lo), int(e_hi), int(num_entities), group

    @staticmethod
    def full(num_entities: int) -> "Shard":
        return Shard(0, num_entities, num_entities, None)

    @staticmethod
    def of_rank(num_entities: int, rank: int, world: int, group=None) -> "Shard":
        per = (num_entities + world - 1) // world
        return Shard(min(rank * per, num_entities), min((rank + 1) * per, num_entities), num_entities, group)

    @property
    def distributed(self) -> bool:
        return self.group is not None and dist.is_initialized() and dist.get_world_size(self.group) > 1


def csr_from_coords(label_coords: torch.Tensor, num_rows: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """[nnz,2] (row, column) coordinates -> (offsets [num_rows+1], columns ascending within a row), on device."""
    c = label_coords.long()
    if c.numel() == 0:
        return (torch.zeros(num_rows + 1, dtype=torch.int64, device=c.device),
                torch.zeros(0, dtype=torch.int64, device=c.device))
    key = (c[:, 0] << 32) + c[:, 1]  # columns < 2^32, rows < 2^31: no host sync, no overflow
    order = torch.argsort(key)
    c = c[order]
    counts = torch.bincount(c[:, 0], minlength=num_rows)
    off = torch.zeros(num_rows + 1, dtype=torch.int64, device=c.device)
    off[1:] = torch.cumsum(counts, 0)
    return off, c[:, 1].contiguous()


def combine_rowstats(rowstat: torch.Tensor, loss: int, shard: Shard) -> torch.Tensor:
    """All-reduce of the per-shard row statistics (max + rescaled sums for KL, plain sums otherwise)."""
    if not shard.distributed:
        return rowstat
    if loss == lib.LOSS_KL:
        gmax = rowstat[:, 0].clone()
        dist.all_reduce(gmax, op=dist.ReduceOp.MAX, group=shard.group)
        scale = torch.where(torch.isinf(rowstat[:, 0]) & (rowstat[:, 0] < 0), torch.zeros_like(gmax),
                            torch.exp(rowstat[:, 0] - gmax))
        packed = torch.stack((rowstat[:, 1] * scale, rowstat[:, 2], rowstat[:, 3]), dim=1).contiguous()
        dist.all_reduce(packed, op=dist.ReduceOp.SUM, group=shard.group)
        return torch.stack((gmax, packed[:, 0], packed[:, 1], packed[:, 2]), dim=1)
    out = rowstat.clone()
    dist.all_reduce(out, op=dist.ReduceOp.SUM, group=shard.group)
    return out


def fused_rowstats(q, table, lab_off, lab_col, loss, label_smoothing, offset, math, shard: Shard,
                   kind: int = lib.DOT) -> torch.Tensor:
    """Per-row forward statistics [B, 4] of this shard; a distance `kind` runs the fp32 tiles whatever `math` says."""
    b, d = q.shape
    rowstat = torch.empty(b, 4, dtype=torch.float32, device=q.device)
    n_ent = shard.e_hi - shard.e_lo
    ws = ops._workspace(q.device, lib.load().kgeb_fused_workspace_bytes(b, d, n_ent, lab_col.numel()))
    if kind != lib.DOT:
        lib.call("kgeb_fused_fwd_kind", kind, loss, lib.f32(q, "queries"), b, d, lib.f32(table, "table"), shard.e_lo,
                 shard.e_hi, shard.num_entities, lib.i64(lab_off, "label offsets"), lib.i64(lab_col, "label columns"),
                 lab_col.numel(), float(label_smoothing), float(offset), rowstat.data_ptr(), ws.data_ptr(), ws.numel(),
                 lib.stream_ptr(q))
        return rowstat
    lib.call("kgeb_fused_fwd", loss, math, lib.f32(q, "queries"), b, d, lib.f32(table, "table"), shard.e_lo,
             shard.e_hi, shard.num_entities, lib.i64(lab_off, "label offsets"), lib.i64(lab_col, "label columns"),
             lab_col.numel(), float(label_smoothing), float(offset), _mirror_ptr(table, math, b, d), rowstat.data_ptr(), ws.data_ptr(),
             ws.numel(), lib.stream_ptr(q))
    return rowstat


def flash_supported(loss: int, math: int, d: int, label_smoothing: float) -> bool:
    """KL on the bf16 tiles: forward statistics + query gradient in one table pass (kgeb_fused_flash_fwd)."""
    return loss == lib.LOSS_KL and math == lib.MATH_BF16 and d % 16 == 0 and d <= 256 and label_smoothing == 0.0


def flash_forward(q, table, lab_off, lab_col, shard: Shard):
    """(rowstat_local [B,4] = (mref, sum exp(x - mref), 0, label dot), o_sum [B,d], status int32 [1]) of this shard.
    status != 0: a score lay more than ~88 nats above the row's reference -- the results are invalid, use the two-pass
    kernels (fused_rowstats / fused_backward)."""
    b, d = q.shape
    rowstat = torch.empty(b, 4, dtype=torch.float32, device=q.device)
    o_sum = torch.empty(b, d, dtype=torch.float32, device=q.device)
    status = torch.zeros(1, dtype=torch.int32, device=q.device)
    n_ent = shard.e_hi - shard.e_lo
    ws = ops._workspace(q.device, lib.load().kgeb_fused_workspace_bytes(b, d, n_ent, lab_col.numel()))
    lib.call("kgeb_fused_flash_fwd", lib.f32(q, "queries"), b, d, lib.f32(table, "table"), shard.e_lo, shard.e_hi,
             shard.num_entities, lib.i64(lab_off), lib.i64(lab_col), lab_col.numel(),
             _mirror_ptr(table, lib.MATH_BF16, b, d), rowstat.data_ptr(), o_sum.data_ptr(), status.data_ptr(), ws.data_ptr(),
             ws.numel(), lib.stream_ptr(q))
    return rowstat, o_sum, status


def flash_dq(q, table, lab_off, lab_col, rowstat_local, lse, inv_batch, grad_scale, o_sum, shard: Shard) -> torch.Tensor:
    """dQ from the flash forward's o_sum (no table pass); summed over the shards."""
    b, d = q.shape
    n_ent = shard.e_hi - shard.e_lo
    dq = torch.empty(b, d, dtype=torch.float32, device=q.device)
    ws = ops._workspace(q.device, lib.load().kgeb_fused_workspace_bytes(b, d, n_ent, lab_col.numel()))
    lib.call("kgeb_fused_flash_dq", lib.f32(q, "queries"), b, d, lib.f32(table, "table"), shard.e_lo, shard.e_hi,
             lib.i64(lab_off), lib.i64(lab_col), lab_col.numel(), lib.f32(rowstat_local), lib.f32(lse, "lse"),
             float(inv_batch), None if grad_scale is None else lib.f32(grad_scale, "grad scale"), lib.f32(o_sum),
             dq.data_ptr(), ws.data_ptr(), ws.numel(), lib.stream_ptr(q))
    if shard.distributed:
        dist.all_reduce(dq, op=dist.ReduceOp.SUM, group=shard.group)
    return dq


def _mirror_ptr(table, math, b, d):
    """bf16 mirror of the table for KGEB_MATH_BF16 (None when the tensor tiles will not be used)."""
    if math != lib.MATH_BF16 or d % 16 != 0 or d > 256:
        return None
    return ops.bf16_mirror(table).data_ptr()


def rows_loss(rowstat: torch.Tensor, lab_off: torch.Tensor, loss: int, label_smoothing: float,
              num_entities: int) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """Per-row loss values (un-normalised sums as in the reference) and, for KL, the log-sum-exp."""
    nnz = (lab_off[1:] - lab_off[:-1]).float()
    if loss == lib.LOSS_KL:
        lse = rowstat[:, 0] + torch.log(rowstat[:, 1])
        # sum_j t (log t - log_softmax_j), t = y/nnz:  -log(nnz) - labeldot/nnz + lse   (loss.py:199-213)
        has = nnz > 0
        safe = torch.where(has, nnz, torch.ones_like(nnz))
        per_row = torch.where(has, lse - rowstat[:, 3] / safe - torch.log(safe), torch.zeros_like(lse))
        return per_row, lse
    keep = 1.0 - label_smoothing
    add = (1.0 / num_entities) if label_smoothing > 0 else 0.0
    # sum_j softplus(x) - t x with t = keep*y + add   (loss.py:153-159, train.py:715-721)
    return rowstat[:, 0] - keep * rowstat[:, 3] - add * rowstat[:, 2], None


def fused_backward(q, table, lab_off, lab_col, loss, label_smoothing, offset, lse, inv_batch, grad_scale, math,
                   shard: Shard, d_table: Optional[torch.Tensor], want_dq: bool = True,
                   lab_perm: Optional[torch.Tensor] = None, overwrite: bool = False,
                   kind: int = lib.DOT) -> Optional[torch.Tensor]:
    """dQ (returned, all-reduced over shards) and d_table += G^T Q for the rows of this shard (`overwrite`: d_table = ...,
    KGEB_BWD_OVERWRITE_TABLE -- the buffer need not be cleared).  lab_perm (int32, optional): stable argsort of lab_col
    from the collate (spares the device sort of the label scatter).  A distance `kind` runs the fp32 tiles."""
    b, d = q.shape
    n_ent = shard.e_hi - shard.e_lo
    dq = torch.empty(b, d, dtype=torch.float32, device=q.device) if want_dq else None
    ws = ops._workspace(q.device, lib.load().kgeb_fused_workspace_bytes(b, d, n_ent, lab_col.numel()))
    if kind != lib.DOT:
        lib.call("kgeb_fused_bwd_kind", kind, loss, lib.f32(q, "queries"), b, d, lib.f32(table, "table"), shard.e_lo,
                 shard.e_hi, shard.num_entities, lib.i64(lab_off), lib.i64(lab_col), lab_col.numel(),
                 float(label_smoothing), float(offset), None if lse is None else lib.f32(lse, "lse"), float(inv_batch),
                 None if grad_scale is None else lib.f32(grad_scale, "grad scale"), None if dq is None else dq.data_ptr(),
                 None if d_table is None else lib.f32(d_table, "table gradient"),
                 lib.BWD_OVERWRITE_TABLE if (overwrite and d_table is not None) else 0, ws.data_ptr(), ws.numel(),
                 lib.stream_ptr(q))
    else:
        lib.call("kgeb_fused_bwd", loss, math, lib.f32(q, "queries"), b, d, lib.f32(table, "table"), shard.e_lo,
                 shard.e_hi, shard.num_entities, lib.i64(lab_off), lib.i64(lab_col), lab_col.numel(),
                 None if lab_perm is None else lab_perm.data_ptr(), float(label_smoothing), float(offset), None if lse is None else lib.f32(lse, "lse"), float(inv_batch),
                 None if grad_scale is None else lib.f32(grad_scale, "grad scale"), _mirror_ptr(table, math, b, d),
                 None if dq is None else dq.data_ptr(), None if d_table is None else lib.f32(d_table, "table gradient"),
                 None, lib.BWD_OVERWRITE_TABLE if (overwrite and d_table is not None) else 0, ws.data_ptr(), ws.numel(),
                 lib.stream_ptr(q))
    if dq is not None and n_ent == 0:
        dq.zero_()
    if dq is not None and shard.distributed:
        dist.all_reduce(dq, op=dist.ReduceOp.SUM, group=shard.group)
    return dq


class AllEntityLoss(torch.autograd.Function):
    """Per-row loss(score(Q, table), labels) / batch_size  [B]  with autograd to Q and the table.
    (Summing the rows gives the reference's batch loss; row sub-sums give its per-query-type values.)"""

    @staticmethod
    def forward(ctx, q, table, lab_off, lab_col, loss, label_smoothing, offset, batch_size, math, shard, kind):
        qd, td = q.detach().contiguous(), table.detach()
        flash = kind == lib.DOT and flash_supported(loss, math, qd.shape[1], label_smoothing) and qd.shape[0] > 0
        if flash:
            local, o_sum, status = flash_forward(qd, td, lab_off, lab_col, shard)
            if shard.distributed:      # every rank must take the same path
                dist.all_reduce(status, op=dist.ReduceOp.MAX, group=shard.group)
            flash = int(status.item()) == 0     # (the job reads the loss back every batch anyway, train.py:747, 1043)
        if flash:
            rowstat = combine_rowstats(local, loss, shard)
        else:
            local = o_sum = None
            rowstat = combine_rowstats(
                fused_rowstats(qd, td, lab_off, lab_col, loss, label_smoothing, offset, math, shard, kind), loss, shard)
        per_row, lse = rows_loss(rowstat, lab_off, loss, label_smoothing, shard.num_entities)
        ctx.save_for_backward(qd, td, lab_off, lab_col, lse, local, o_sum)
        ctx.cfg = (loss, label_smoothing, offset, 1.0 / batch_size, math, shard, kind)
        return per_row / batch_size

    @staticmethod
    def backward(ctx, g):
        qd, td, lab_off, lab_col, lse, local, o_sum = ctx.saved_tensors
        loss, ls, offset, inv_batch, math, shard, kind = ctx.cfg
        # a table-sized gradient: written once by the kernels (no zero-fill pass) when this rank scores every row
        whole = shard.e_lo == 0 and shard.e_hi == td.shape[0]
        d_table = None
        if ctx.needs_input_grad[1]:
            d_table = torch.empty_like(td) if whole else torch.zeros_like(td)
        gs = g.detach().float().contiguous()  # upstream gradient per row; stays on the device
        if local is not None:     # flash forward: dQ needs no table pass, only the table gradient recomputes the scores
            dq = flash_dq(qd, td, lab_off, lab_col, local, lse, inv_batch, gs, o_sum, shard) if ctx.needs_input_grad[0] else None
            if d_table is not None:
                fused_backward(qd, td, lab_off, lab_col, loss, ls, offset, lse, inv_batch, gs, math, shard, d_table,
                               want_dq=False, overwrite=whole)
        else:
            dq = fused_backward(qd, td, lab_off, lab_col, loss, ls, offset, lse, inv_batch, gs, math, shard, d_table,
                                want_dq=ctx.needs_input_grad[0], overwrite=whole, kind=kind)
        return dq, d_table, None, None, None, None, None, None, None, None, None


def all_entity_loss(q, table, lab_off, lab_col, loss: int, batch_size: int, label_smoothing: float = 0.0,
                    offset: float = 0.0, math: int = lib.MATH_FP32, shard: Optional[Shard] = None,
                    kind: int = lib.DOT) -> torch.Tensor:
    """`kind`: pair kind of the scorer (lib.DOT, or TransE / RotatE's distance kinds, which run the fp32 CUDA-core
    tiles with no flash pass whatever `math` says)."""
    shard = shard or Shard.full(table.shape[0])
    return AllEntityLoss.apply(q, table, lab_off, lab_col, loss, float(label_smoothing), float(offset),
                               int(batch_size), math, shard, int(kind))


# ---------------------------------------------------------------------------------------------
# fused filtered ranking
# ---------------------------------------------------------------------------------------------
def rank_counts(kind: int, q, table, true_score, true_ent, filt: Optional[Tuple[torch.Tensor, torch.Tensor]],
                filt_test: Optional[Tuple[torch.Tensor, torch.Tensor]], math: int = lib.MATH_FP32,
                shard: Optional[Shard] = None, counts: Optional[torch.Tensor] = None) -> torch.Tensor:
    """counts[nq, 6] int64 = (rank, ties) x (raw, filtered, filtered-with-test); see kgeb_rank_count."""
    shard = shard or Shard.full(table.shape[0])
    nq, d = q.shape
    if counts is None:
        counts = torch.zeros(nq, 6, dtype=torch.int64, device=q.device)
    tp, t64 = lib.idx(true_ent.contiguous(), "true entities")
    f_off, f_col = filt if filt is not None else (None, None)
    u_off, u_col = filt_test if filt_test is not None else (None, None)
    lib.call("kgeb_rank_count", kind, math, lib.f32(q.contiguous(), "queries"), nq, d, lib.f32(table, "table"),
             shard.e_lo, shard.e_hi, lib.f32(true_score.contiguous(), "true scores"), tp, t64, lib.i64(f_off),
             lib.i64(f_col), lib.i64(u_off), lib.i64(u_col), counts.data_ptr(), lib.stream_ptr(q))
    if shard.distributed:
        dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=shard.group)
    return counts
