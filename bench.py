#!/usr/bin/env python
"""Benchmark of the hot path on the workload the north star scales over GPUs (BASELINE.json configs[3]):

    DistMult 1vsAll + KL, dim 128, synthetic Wikidata5M-shaped graph (4,600,000 entities, 822 relations),
    Adagrad lr 0.2, 1,024 triples (= 2,048 sp_ / _po queries) per step -- the SAME batch at every GPU count.

A step = TrainingJob1vsAll's batch body + optimizer step (train.py:1032-1062, 309-376): gather -> query transform ->
fused score + log-sum-exp -> backward (dQ, dense table gradient) -> scatter of the query-side / label rows -> Adagrad
on both tables.  Metric: training triples/s.  The table (2.36 GB fp32 + 1.18 GB bf16 mirror + 2.36 GB Adagrad state)
fits one GPU, so N = 1 runs the same workload; for N > 1 the entity table, its optimizer state and its gradient are
sharded BY ROW over the ranks (trainer.RowShardedAllEntityStepper: three O(batch * d) all-reduces per step) and the
per-step batch stays 1,024 triples: strong scaling.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Prints ONE JSON line.  `value`: batches resident in HBM, CUDA-event timed, max over ranks.  `e2e`: the same step through
the REFERENCE's own job object (baseline/_ref, unmodified `TrainingJob1vsAll` created by `Job.create` with the B200
plug-in model: `job._process_batch(...)` + `job.optimizer.step()`), pinned host batches, H2D copy and loss read-back
inside the timed region (N > 1: this repo's sharded stepper fed from pinned host batches).  `roofline`: the dominant
tile kernel timed alone + the whole step against SURVEY.md 8(d)'s 12*E*d FLOP per triple.  `cpu_baseline` /
`--impl reference`: the unmodified reference (`kge` from baseline/_ref, model distmult, job.device cpu) on the box's host
cores.  `parity`: loss of the same batch from the same tables on both arms.  `extra.fb15k237`: round 1's line
(ComplEx KvsAll + BCE, bench_fb237.py), N = 1 only.
"""
import argparse
import contextlib
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import bench_fb237  # noqa: E402  (ClockSampler, peaks, the configs[1] workload)

E, R, DIM, LR, B = 4_600_000, 822, 128, 0.2, 1024
E = int(os.environ.get("KGEB_BENCH_ENTITIES", E))      # dry runs of this script on a small table; never set by the driver
WORKLOAD = (f"DistMult 1vsAll+KL d=128, synthetic Wikidata5M shape (E={E}, R=822), 1024 triples "
            "(2048 sp_/_po queries) per step")


def config(world: int, math: str) -> dict:
    """The `config` object of both arms' JSON lines (same keys, same workload string)."""
    return {"workload": WORKLOAD, "batch": B, "global_batch": B, "optimizer": f"Adagrad lr {LR}",
            "entities": E, "relations": R, "dim": DIM, "loss": "kl", "train_type": "1vsAll",
            "parallelism": "1 GPU" if world == 1 else
            f"entity table, Adagrad state and gradient row-sharded over {world} GPUs; every rank sees the whole batch; "
            "all-reduce of the query-side rows, the row statistics and dQ ([2048,128] fp32 each) per step",
            "l2": "inputs larger than L2 (bf16 table 1.18 GB vs 126 MB): no flush between timed steps"}


def make_batches(n: int, seed: int = 7):
    """n batches of B synthetic triples: s, o from a truncated Zipf over a permutation of the entity ids, p from a Zipf
    over the relations (SURVEY.md Appendix C); int64 [B,3] pinned host tensors, as the reference's collate emits them
    (train.py:1016-1020)."""
    rng = np.random.default_rng(seed)
    perm = rng.permutation(E)
    zipf = lambda m, size: np.minimum((np.exp(rng.random(size) * np.log(m + 1.0)) - 1.0).astype(np.int64), m - 1)  # noqa: E731
    out = []
    for _ in range(n):
        t = np.stack([perm[zipf(E, B)], zipf(R, B), perm[zipf(E, B)]], 1).astype(np.int64)
        out.append(torch.from_numpy(t))
    return out


def quiet():
    """The reference logs to stdout; this program's stdout carries exactly one JSON line."""
    return contextlib.redirect_stdout(sys.stderr)


# ---------------------------------------------------------------------------------------------
# reference arm: the unmodified reference on the host cores
# ---------------------------------------------------------------------------------------------
def cpu_batch_size() -> int:
    """Largest batch (<= B) whose [batch, E] fp32 score / softmax / gradient matrices (train.py:1040-1057, ~3 live copies
    per direction) plus the table-sized tensors (parameters, gradients, Adagrad state, embed_all copies: ~8 x 2.36 GB)
    fit in 70 % of the host's available memory."""
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 64 << 30
    b = B
    while b > 16 and (3 * b * E * 4 + 8 * E * DIM * 4) > 0.7 * avail:
        b //= 2
    return b


def reference_job(device="cpu", plugin=False, plugin_args=None, batch=B):
    from baseline import ref_env
    graph = {"train": np.zeros((8, 3), dtype=np.int32), "valid": np.zeros((8, 3), dtype=np.int32),
             "test": np.zeros((8, 3), dtype=np.int32)}
    opts = {"train.type": "1vsAll", "train.loss": "kl", "train.batch_size": batch, "train.optimizer": "Adagrad",
            "train.optimizer_args": {"lr": LR}, "train.num_workers": 0,
            # SURVEY.md 8(d): tables normal_(0, 0.1) as in examples/toy-complex-train.yaml:17-21
            "lookup_embedder.initialize_args.normal_.std": 0.1}
    with quiet():
        job = ref_env.make_job("distmult", graph, E, R, DIM, opts, device=device, plugin=plugin, plugin_args=plugin_args,
                               seed=0)
        job._prepare()
    return job


def reference_step(job, i, triples):
    """run_epoch's body for one batch (train.py:309-376) on the reference's own objects."""
    job.optimizer.zero_grad()
    res = job._process_batch(i, {"triples": triples})
    for _, v in job.model.penalty(epoch=1, batch_index=i, num_batches=1, batch={"triples": triples}):
        v.backward()
    job.optimizer.step()
    return res.avg_loss


def run_cpu_reference(batches, steps, warmup, job=None):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    bc = cpu_batch_size()
    if job is None:
        job = reference_job("cpu", batch=bc)
    losses, times = [], []
    with quiet():
        for i in range(warmup + steps):
            t = batches[i % len(batches)][:bc]
            t0 = time.perf_counter()
            losses.append(reference_step(job, i, t))
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    ms = 1e3 * float(np.mean(times))
    sample = (f"{steps} step(s) + {warmup} warm-up of kge.job.train.TrainingJob1vsAll._process_batch + optimizer.step() from "
              f"baseline/_ref (unmodified reference, model distmult, job.device cpu, {cores} threads) on {bc} triples per step")
    if bc < B:
        sample += (f" -- the first {bc} of the step's {B} triples: the reference materialises [batch, E] fp32 score, "
                   f"softmax and gradient matrices and {B} triples do not fit this host's memory; its per-step cost has a "
                   "batch-independent part (table-sized gradient + dense Adagrad), so triples/s at the full batch would be "
                   "higher than this figure by up to the batch ratio")
    return {"value": bc / (ms / 1e3), "ms_per_step": ms, "cores": cores, "sample": sample, "batch": bc,
            "loss_step0": losses[0], "job": job}


def reference_cuda(batches, local_rank, steps, warmup=2):
    """SURVEY.md 8(d), last paragraph: the reference's own CUDA path -- the UNMODIFIED reference with its stock model and
    torch.optim.Adagrad, job.device cuda -- on the same GPU, same config and batches: 'same API, stock kernels'.  Timed like
    the e2e figure (pinned host triples in, loss read back by the job) with CUDA events around the steps."""
    try:
        job = reference_job(f"cuda:{local_rank}")
        torch.cuda.synchronize()
        with quiet():
            for i in range(warmup):
                reference_step(job, i, batches[i % len(batches)])
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            for i in range(steps):
                loss = reference_step(job, warmup + i, batches[(warmup + i) % len(batches)])
            b.record()
            torch.cuda.synchronize()
        ms = a.elapsed_time(b) / steps
        peak = torch.cuda.max_memory_allocated() / 2 ** 30
        del job
        torch.cuda.empty_cache()
        return {"value": B / (ms * 1e-3), "unit": "triples/s", "ms_per_step": ms, "steps": steps, "warmup": warmup,
                "last_loss": float(loss), "peak_memory_gib": round(peak, 1),
                "what": ("kge.job.train.TrainingJob1vsAll from baseline/_ref, model distmult (stock scorer / LookupEmbedder), "
                         "torch.optim.Adagrad, job.device cuda: zero_grad + _process_batch + optimizer.step() per step; fp32 "
                         "(torch's default matmul precision), [batch, E] score matrices materialised")}
    except Exception as exc:      # e.g. out of memory next to this arm's own allocations
        torch.cuda.empty_cache()
        return {"value": None, "unavailable": f"{type(exc).__name__}: {str(exc)[:200]}"}


def reference_arm(args):
    from baseline import ref_env
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if not ref_env.available():
        print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref is not installed (baseline/install_ref.sh)"}))
        return
    # a reference step at this shape takes tens of seconds on the host: --steps 20 runs for several minutes
    steps, warm = args.steps, min(args.warmup, 1)
    batches = make_batches(steps + warm)
    res = run_cpu_reference(batches, steps, warm)
    print(json.dumps({
        "impl": "reference", "metric": "training triples/s", "value": res["value"], "unit": "triples/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "steps_requested": args.steps, "warmup_requested": args.warmup,
        "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config(args.gpus, "fp32"),
        "cpu_baseline": {"value": res["value"], "unit": "triples/s", "cores": res["cores"], "kind": "reference",
                         "sample": res["sample"]},
        "e2e": {"value": res["value"], "unit": "triples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "loss_step0": res["loss_step0"], "gpu_launches": 0}))


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
def count_library_launches(fn) -> int:
    """Kernels of libkgeb200.so launched by one call of fn (CUPTI activity records; not inside a timed region)."""
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = ("kgeb", "label_weight_kernel", "loss_rows_kernel", "loss_report_kernel")
    return sum(1 for ev in prof.events()
               if ev.device_type == torch.autograd.DeviceType.CUDA and any(n in ev.name for n in names))


def device_batch(t: torch.Tensor, dev):
    """[B,3] triples -> the stepper's static inputs: rows 0..B-1 = sp_ queries, B..2B-1 = _po queries (both directions
    of 1vsAll in one launch; their gradients accumulate before one step, train.py:1041-1057, 375)."""
    t = t.to(dev, non_blocking=True)
    s, p, o = t[:, 0], t[:, 1], t[:, 2]
    z = torch.zeros(len(t), dtype=torch.int32, device=dev)
    return (torch.cat((s, o)), torch.cat((p, p)), torch.cat((z, z + 1)),
            torch.arange(2 * len(t) + 1, dtype=torch.int64, device=dev), torch.cat((o, s)))


DUMP_SAMPLE_ROWS, DUMP_SAMPLE_SEED = 32768, 11
# where the tables the timed steps start from come from (index = initial_tables.npy of --dump-outputs)
INITIAL_TABLES = ("KgeModel under torch.manual_seed(0)",
                  "the reference's TrainingJob1vsAll with the plug-in model on the GPU (baseline/_ref), after one step "
                  "that captures the stepper",
                  "as 1, with the CPU reference job's tables loaded first (--cpu-steps > 0)")


def dump_outputs(out_dir, st, loss, last_batch, initial_tables, rank, world):
    """Writes what the timed step hands its caller after the last timed step as float32 .npy files under out_dir (about
    36 MB): the batch's loss, the relation table and its Adagrad state, and rows of the entity table and of its Adagrad
    state -- the rows of the step's own entities (`*_batch`) and a fixed, seeded sample of all rows (`*_sample`; the
    whole table is 2.36 GB).  The row ids go along as float64, and initial_tables.npy holds the index into INITIAL_TABLES
    of the path that made the starting tables: that path depends on whether baseline/_ref is installed.  Runs of two
    builds on the same arguments and the same path start from the same tables and batches, so their files can be compared
    array by array."""
    if world > 1:
        st.sync_tables()          # every rank then holds the whole, current entity table and its state
    if rank != 0:
        return
    ent, rel = st.ent.detach(), st.rel.detach()
    s_ent, s_rel = st.opt.state[st.ent]["sum"], st.opt.state[st.rel]["sum"]
    batch_ids = torch.unique(torch.cat((last_batch[:, 0], last_batch[:, 2]))).to(ent.device)
    rng = np.random.default_rng(DUMP_SAMPLE_SEED)
    sample_ids = np.sort(rng.choice(E, min(E, DUMP_SAMPLE_ROWS), replace=False))
    sample_ids = torch.from_numpy(sample_ids).to(ent.device)
    arrays = {"loss": loss.detach().reshape(()), "relation_table": rel, "relation_adagrad_sum": s_rel,
              "initial_tables": torch.tensor(float(initial_tables), dtype=torch.float64)}
    for tag, ids in (("batch", batch_ids), ("sample", sample_ids)):
        arrays[f"entity_ids_{tag}"] = ids.double()
        arrays[f"entity_rows_{tag}"] = ent[ids]
        arrays[f"entity_adagrad_sum_{tag}"] = s_ent[ids]
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def kernel_roofline(kb, st, rows, n_ent, step_ms, world):
    """The tile kernels of the step timed alone (CUDA events on the launching stream, empty label CSR so that only the
    tile kernel and its tiny pre / post kernels run; the operands are far larger than L2) and the whole step against
    SURVEY.md 8(d)'s algorithmic count."""
    pk = bench_fb237.peaks()
    L, d, dev = kb.lib, st.d, st.ent.device
    table = st.ent.detach() if not hasattr(st, "e_lo") else st.ent.detach()[st.e_lo:st.e_hi]
    e_lo, e_hi = (0, st.E) if not hasattr(st, "e_lo") else (st.e_lo, st.e_hi)
    mp = st.mirror.data_ptr()
    off0 = torch.zeros(rows + 1, dtype=torch.int64, device=dev)
    lse = torch.full((rows,), 15.3, device=dev)
    gtmp = torch.empty(n_ent, d, device=dev)
    rowstat = torch.empty(rows, 4, device=dev)
    dq = torch.empty(rows, d, device=dev)
    ws = st.ws

    def fwd():
        L.call("kgeb_fused_fwd", L.LOSS_KL, L.MATH_BF16, st.Q.data_ptr(), rows, d, table.data_ptr(), e_lo, e_hi, st.E,
               off0.data_ptr(), st.lab_col.data_ptr(), 0, 0.0, 0.0, mp, rowstat.data_ptr(), ws.data_ptr(), ws.numel(),
               L.stream_ptr(table))

    def bwd(want_dq, want_dt):
        L.call("kgeb_fused_bwd", L.LOSS_KL, L.MATH_BF16, st.Q.data_ptr(), rows, d, table.data_ptr(), e_lo, e_hi, st.E,
               off0.data_ptr(), st.lab_col.data_ptr(), 0, None, 0.0, 0.0, lse.data_ptr(), 1.0 / B, None, mp,
               dq.data_ptr() if want_dq else None, gtmp.data_ptr() if want_dt else None, None,
               L.BWD_OVERWRITE_TABLE if want_dt else 0, ws.data_ptr(), ws.numel(), L.stream_ptr(table))

    # name -> (launcher, GEMMs the launch EXECUTES, GEMMs of the algorithm it stands for, ncu kernel name)
    cases = {"tc_tiles_kernel<stats> (kgeb_fused_fwd: scores + online log-sum-exp)": (fwd, 1, 1, "tc_tiles_kernel<1, 2, 1>"),
             "tc_bwd_kernel<dQ> (kgeb_fused_bwd: S recomputed, dQ += G*T)": (lambda: bwd(True, False), 2, 1, "tc_bwd4_kernel<1, 0, 0, 0, 0, 0>"),
             "tc_bwd_kernel<dTable> (kgeb_fused_bwd: S recomputed, dT = G^T*Q)": (lambda: bwd(False, True), 2, 1, "tc_bwd4_kernel<0, 0, 0, 0, 0, 0>")}
    if getattr(st, "flash", False):
        # forward statistics and dQ come out of ONE table pass (kgeb_fused_flash_fwd): two GEMMs executed, both algorithmic
        o_sum = torch.empty(rows, d, device=dev)
        status = torch.zeros(4, dtype=torch.int32, device=dev)

        def flash():
            L.call("kgeb_fused_flash_fwd", st.Q.data_ptr(), rows, d, table.data_ptr(), e_lo, e_hi, st.E, off0.data_ptr(),
                   st.lab_col.data_ptr(), 0, mp, rowstat.data_ptr(), o_sum.data_ptr(), status.data_ptr(), ws.data_ptr(),
                   ws.numel(), L.stream_ptr(table))

        dt = [v for k, v in cases.items() if "dTable" in k][0]
        cases = {"tc_bwd_kernel<flash> (kgeb_fused_flash_fwd: scores + log-sum-exp + o_sum for dQ, one pass)":
                 (flash, 2, 2, "tc_bwd4_kernel<1, 0, 0, 0, 1, 0>"),
                 "tc_bwd_kernel<dTable> (kgeb_fused_bwd: S recomputed, dT = G^T*Q)": dt}
    if getattr(st, "fuse_update", False):
        # what the step runs instead of the storing dTable kernel + kgeb_adagrad_dense: Adagrad applied by that kernel's
        # update warps (lr 0 here: W and the mirror are written back unchanged; scratch state; no touched rows)
        gtmp.fill_(0.1)
        t = st.touched

        def upd():
            L.call("kgeb_fused_bwd_update", L.LOSS_KL, st.Q.data_ptr(), rows, d, table.data_ptr(), e_lo, e_hi, st.E,
                   off0.data_ptr(), 0.0, 0.0, lse.data_ptr(), 1.0 / B, None, mp, gtmp.data_ptr(), 0.0, 1e-10,
                   t.slot_of.data_ptr(), t.g_dense.data_ptr(), None, ws.data_ptr(), ws.numel(), L.stream_ptr(table))

        state2 = None

        def adagrad():      # the pass the fused kernel replaces (reads the stored gradient; lr 0)
            L.call("kgeb_adagrad_dense", table.data_ptr(), state2.data_ptr(), gtmp.data_ptr(), None, table.numel(), 0.0, 1e-10,
                   0.0, mp, L.stream_ptr(table))

        cases["tc_bwd_kernel<dTable + Adagrad> (kgeb_fused_bwd_update: dT = G^T*Q applied to W / state / bf16 mirror by "
              "update warps)"] = (upd, 2, 1, "tc_bwd4_kernel<0, 0, 0, 0, 0, 1>")
        try:
            state2 = torch.full_like(gtmp, 0.1)
            cases["kgeb_adagrad_dense (separate pass, for comparison: not part of the step)"] = (adagrad, 0, 0, "adagrad_dense_kernel")
        except torch.OutOfMemoryError:
            pass
    res = {}
    for name, (fn, executed, algorithmic, _) in cases.items():
        ts = []
        for i in range(5):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record()
            torch.cuda.synchronize()
            if i >= 2:
                ts.append(a.elapsed_time(b))
        res[name] = float(np.mean(ts))
    in_step = {k: v for k, v in res.items() if "for comparison" not in k and not (getattr(st, "fuse_update", False) and
                                                                                   "dTable>" in k)}
    name = max(in_step, key=in_step.get)
    ms = res[name]
    gemm = 2.0 * rows * n_ent * d
    achieved = cases[name][2] * gemm / (ms * 1e-3) / 1e12
    # the whole step: 12*E*d FLOP per triple (3 GEMMs of 2*(2B)*E*d: forward, dQ, dTable), SURVEY.md 8(d) C4
    step_flops = 12.0 * E * DIM * B
    step_achieved = step_flops / (step_ms * 1e-3) / 1e12 / world
    traffic = None
    path = os.path.join(ROOT, "profiles", "ncu_full_latest_summary.json")
    if os.path.exists(path):
        summ = json.load(open(path))
        k = summ.get("wd5m " + cases[name][3]) or summ.get("wd5m " + cases[name][3].replace(", 0>", ">"))
        if k:
            traffic = k["dram_bytes_read"] + k["dram_bytes_write"]
    return {"kernel": name, "bound": "tensor", "achieved": achieved, "peak": pk["bf16_burst"], "unit": "TFLOP/s",
            "frac": achieved / pk["bf16_burst"], "traffic": traffic,
            "executed_tflops": cases[name][1] * gemm / (ms * 1e-3) / 1e12,
            "step": {"achieved": step_achieved, "peak": pk["bf16_sustained"], "frac": step_achieved / pk["bf16_sustained"],
                     "unit": "TFLOP/s per GPU", "flops_per_triple": 12.0 * E * DIM},
            "note": ("achieved = ALGORITHMIC FLOPs of the launch (one GEMM of 2*rows*E*d: the score tile a backward kernel "
                     "recomputes is not counted; executed_tflops counts it; the Adagrad update the dTable kernel applies -- "
                     "9 bytes read + 9 written per table element -- is not counted either) / CUDA-event time of the kernel run alone incl. "
                     "its bf16(Q) / reduce helpers; peak = %s dense bf16 burst.  step = 12*E*d FLOP per triple / step time "
                     "(per GPU) against the sustained bf16 figure.  rows = %d, shard entities = %d" % (pk["source"], rows, n_ent)),
            "all_ms": res}


def our_arm(args):
    import kgeb200 as kb
    from baseline import ref_env
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    steps, warm = args.steps, max(args.warmup, 3)
    batches = [b.pin_memory() for b in make_batches(steps + warm)]
    math_mode = kb.lib.MATH_BF16

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    ref_job, parity, cpu = None, None, None
    use_ref = world == 1 and ref_env.available() and not args.no_reference_job
    initial_tables = 0 if not use_ref else (2 if args.cpu_steps > 0 else 1)
    if use_ref:
        # the reference's own TrainingJob1vsAll, created by its factories with the plug-in model on cuda
        ref_job = reference_job(f"cuda:{local_rank}", plugin=True, plugin_args={"math": "bf16", "captured_step": True})
        model_ent = ref_job.model.get_s_embedder()._embeddings.weight
    else:
        torch.manual_seed(0)
        model = kb.KgeModel("distmult", E, R, DIM).to(dev)
        opt = kb.optim.create("Adagrad", model.parameters(), lr=LR)

    # ---------------- cpu baseline + parity (N = 1, rank 0): same tables, same batch, both arms ----------------------
    if use_ref and args.cpu_steps > 0:
        cpu_job = reference_job("cpu", batch=cpu_batch_size())
        with torch.no_grad():                         # both arms start from the CPU reference's tables
            ref_job.model.load_state_dict(cpu_job.model.state_dict())
        bc = cpu_batch_size()
        with torch.no_grad(), quiet():
            t = batches[0][:bc].to(dev)
            q = torch.cat((kb.ops.query_build("distmult", kb.lib.SP_, ref_job.model.get_s_embedder().embed(t[:, 0]),
                                              ref_job.model.get_p_embedder().embed(t[:, 1])),
                           kb.ops.query_build("distmult", kb.lib._PO, ref_job.model.get_o_embedder().embed(t[:, 2]),
                                              ref_job.model.get_p_embedder().embed(t[:, 1]))))
            rows = kb.fused.all_entity_loss(q, model_ent.detach(), torch.arange(2 * bc + 1, device=dev),
                                            torch.cat((t[:, 2], t[:, 0])).contiguous(), kb.lib.LOSS_KL, bc, 0.0, 0.0, math_mode)
            loss_gpu = float(rows.sum().item())
        cpu = run_cpu_reference(batches, args.cpu_steps, 1, job=cpu_job)
        cpu.pop("job")
        del cpu_job
        rel = abs(loss_gpu - cpu["loss_step0"]) / abs(cpu["loss_step0"])
        parity = {"what": f"loss of batch 0 (first {bc} triples) from the same initial tables: unmodified reference on the "
                          "CPU vs the fused bf16-tile kernels", "loss_cpu": cpu["loss_step0"], "loss_gpu": loss_gpu,
                  "rel_diff": rel, "bound": 1e-3, "ok": bool(rel <= 1e-3)}

    # ---------------- the stepper --------------------------------------------------------------------------------------
    if use_ref:
        with quiet():
            reference_step(ref_job, 0, batches[0])       # builds + captures the stepper inside the reference's job
        st = ref_job.model._b200_stepper
        n_ent = E
    elif world == 1:
        st = kb.trainer.FusedAllEntityStepper(model, opt, 2 * B, 2 * B, kb.lib.LOSS_KL, B, math_mode=math_mode)
        n_ent = E
    else:
        sh = kb.fused.Shard.of_rank(E, rank, world, dist.group.WORLD)
        st = kb.trainer.RowShardedAllEntityStepper(model, opt, 2 * B, 2 * B, kb.lib.LOSS_KL, B, sh, math_mode=math_mode,
                                                   peer_memory=not os.environ.get("KGEB_NO_PEER"))
        n_ent = sh.e_hi - sh.e_lo

    # ---------------- value: batches resident in HBM, CUDA events ---------------------------------------------------
    if getattr(st, "triples", None) is not None:
        # the stepper builds its batch from the triples inside the captured step (kgeb_onevsall_batch_build): the resident
        # inputs are the triples themselves
        dev_triples = [b.to(dev) for b in batches]
        set_batch = lambda i: st.set_triples(dev_triples[i])       # noqa: E731
        dev_inputs = None
    else:
        dev_inputs = [device_batch(b, dev) for b in batches]
        set_batch = lambda i: st.set_inputs(*dev_inputs[i])        # noqa: E731
    for i in range(warm):
        set_batch(i)
        st.step()
    barrier()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    with bench_fb237.ClockSampler(local_rank) as clocks:
        barrier()
        for i in range(steps):
            set_batch(warm + i)
            evs[i][0].record()
            loss = st.step()
            evs[i][1].record()
        barrier()
    if args.dump_outputs:
        # here: the e2e leg below trains the tables further
        dump_outputs(args.dump_outputs, st, loss, batches[warm + steps - 1], initial_tables, rank, world)
    total_ms = float(np.sum([a.elapsed_time(b) for a, b in evs]))
    if world > 1:
        t = torch.tensor([total_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = t.item()
    value = B * steps / (total_ms / 1e3)
    final_loss = float(st.loss.item())
    if hasattr(st, "check_peer"):
        st.check_peer()          # no peer-memory barrier timed out

    # ---------------- e2e: host batches, H2D + step + loss read-back inside the timed region ------------------------
    e2e_s = 0.0
    for i in range(0 if args.skip_e2e else warm + steps):
        b = batches[i]
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        if use_ref:
            with quiet():
                reference_step(ref_job, i, b)           # copies the triples to the device, replays the step, reads the loss
        else:
            st.set_inputs(*device_batch(b, dev))
            st.step().item()
        torch.cuda.synchronize()
        if i >= warm:
            e2e_s += time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = t.item()
    e2e_value = None if args.skip_e2e else B * steps / e2e_s

    launches = count_library_launches(lambda: (set_batch(0), st.step()))
    roof = kernel_roofline(kb, st, 2 * B, n_ent, total_ms / steps, world)

    extra = None
    if world == 1 and not args.skip_extra:
        del dev_inputs
        fb_args = bench_fb237.parser().parse_args(["--steps", str(steps), "--warmup", "5", "--cpu-steps", "3"])
        with quiet():
            extra = {"fb15k237": bench_fb237.run(fb_args)}
        if use_ref and not args.skip_reference_cuda:
            extra["reference_cuda"] = reference_cuda(batches, local_rank, steps=steps)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    out = {
        "metric": "training triples/s", "value": value, "unit": "triples/s", "n_gpus": world, "steps": steps, "warmup": warm,
        "ms_per_step": total_ms / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": config(world, "bf16"),
        "details": {"math": "bf16 tensor tiles (tcgen05, bf16 mirror of the table), fp32 accumulate, fp32 master tables "
                            "and optimizer", "cuda_graph": True, "final_loss": final_loss,
                    "flash_fallbacks": getattr(st, "flash_fallbacks", None),
                    "initial_tables": INITIAL_TABLES[initial_tables],
                    "stepper": type(st).__name__ + (" inside the reference's TrainingJob1vsAll" if use_ref else ""),
                    "exchange": (None if world == 1 else ("one-shot all-reduce kernels over NVLink peer memory inside the "
                                 "step's CUDA graph (kgeb_p2p_allreduce)" if getattr(st, "px", None) is not None else
                                 "NCCL all-reduces between four CUDA graphs"))},
        "clocks": clocks.summary(),
        "e2e": {"value": e2e_value, "unit": "triples/s", "h2d_bytes_per_step": int(batches[0].numel() * 8),
                "d2h_bytes_per_step": 8,
                "note": ("the reference's own TrainingJob1vsAll from baseline/_ref (Job.create, plug-in model b200_distmult, "
                         "b200.captured_step): zero_grad + job._process_batch(pinned [1024,3] int64 triples) + penalties + "
                         "job.optimizer.step() per timed step" if use_ref else
                         "this repo's stepper fed from pinned host batches: H2D copy of the triples, step, loss.item() per "
                         "timed step")},
        "gpu_launches": int(launches * steps), "gpu_launches_per_step": launches,
        "roofline": roof,
        "cpu_baseline": ({"value": cpu["value"], "unit": "triples/s", "cores": cpu["cores"], "kind": "reference",
                          "sample": cpu["sample"], "ms_per_step": cpu["ms_per_step"]} if cpu else
                         {"value": None, "unit": "triples/s", "cores": 0, "kind": "reference",
                          "sample": "not run (N > 1, --cpu-steps 0 or baseline/_ref missing)"}),
        "parity": parity,
        "extra": extra,
    }
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed training steps of each workload and arm (the CPU sample inside a GPU run: --cpu-steps; "
                         "the roofline times single kernels separately)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-steps", type=int, default=1, help="timed steps of the bounded CPU-baseline sample (N = 1)")
    ap.add_argument("--skip-reference-cuda", action="store_true", help="do not time the reference's stock CUDA path (N = 1)")
    ap.add_argument("--skip-e2e", action="store_true", help="tuning runs: device-resident value + kernel roofline only")
    ap.add_argument("--skip-extra", action="store_true", help="do not run the FB15k-237 workload (extra key)")
    ap.add_argument("--no-reference-job", action="store_true", help="e2e through this repo's stepper instead of the reference's job object")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss, tables and Adagrad state after the last timed step as .npy files to DIR "
                         "(entity rows: the step's own and a fixed, seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        reference_arm(args)
    else:
        our_arm(args)


if __name__ == "__main__":
    main()
