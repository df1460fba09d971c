#!/usr/bin/env python
"""Measurements of the other BASELINE.json configurations (SURVEY.md 8d: C3, C4, C5) on one B200.  These are
parity-test shapes, not the bench line (bench.py is the contract's benchmark); results are appended as JSON lines to
profiles/extra_workloads_r1.jsonl and summarised in DESIGN.md.

    python bench_extra.py --workload wd5m-1vsall | wnrr-rotate-ns | wd5m-eval-transe | wd5m-eval-complex [--scale F]
    python bench_extra.py --workload wd5m-1vsall-reciprocal --batch 1024
    python bench_extra.py --workload wd5m-1vsall-lr-schedule --batch 1024
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import kgeb200 as kb  # noqa: E402


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def kernel_table(fn, steps, tag):
    """Per-kernel device times of `steps` calls of fn through CUPTI activity tracing (torch.profiler); written to
    gpurun_out/kernels_<tag>.txt.  Diagnostic only: the numbers reported as results are timed without it."""
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
    rows = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            r = rows.setdefault(ev.name, [0, 0.0])
            r[0] += 1
            r[1] += ev.device_time
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    total = sum(r[1] for r in rows.values())
    with open(os.path.join(ROOT, "gpurun_out", f"kernels_{tag}.txt"), "w") as f:
        f.write(f"# {tag}: {steps} steps, {total / steps:.1f} us of kernel time per step\n")
        for name, (cnt, us) in sorted(rows.items(), key=lambda kv: -kv[1][1]):
            f.write(f"{us / steps:10.1f} us/step  {cnt / steps:6.1f} launches/step  {us / cnt:9.1f} us avg  {name[:150]}\n")


def peaks():
    p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    return p.get("hbm_gbs", 6650.0), p.get("bf16_tflops_sustained", 1400.0)


def wd5m_1vsall(args):
    """C4: DistMult 1vsAll + KL, d=128, E=4.6M (scaled by --scale), B triples -> 2B query rows per step."""
    E, R, d, B = int(4_600_000 * args.scale), 822, 128, args.batch
    dev = torch.device("cuda")
    torch.manual_seed(0)
    model = kb.KgeModel("distmult", E, R, d).to(dev)
    opt = kb.optim.create("Adagrad", model.parameters(), lr=0.2)
    math_mode = {"bf16": kb.lib.MATH_BF16, "tf32": kb.lib.MATH_TF32, "fp32": kb.lib.MATH_FP32}[args.math]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:   # entity table sharded by row over the ranks; every rank sees the whole batch (SURVEY.md 8e)
        import torch.distributed as dist
        sh = kb.fused.Shard.of_rank(E, int(os.environ["RANK"]), world, dist.group.WORLD)
        st = kb.trainer.RowShardedAllEntityStepper(model, opt, 2 * B, 2 * B, kb.lib.LOSS_KL, B, sh, math_mode=math_mode)
    else:
        st = kb.trainer.FusedAllEntityStepper(model, opt, 2 * B, 2 * B, kb.lib.LOSS_KL, B, math_mode=math_mode, use_graph=True)
    gen = torch.Generator(device=dev).manual_seed(1)

    def new_batch():
        s = torch.randint(0, E, (B,), device=dev, generator=gen)
        o = torch.randint(0, E, (B,), device=dev, generator=gen)
        p = torch.randint(0, R, (B,), device=dev, generator=gen)
        st.set_inputs(torch.cat((s, o)), torch.cat((p, p)),
                      torch.cat((torch.zeros(B, dtype=torch.int32, device=dev), torch.ones(B, dtype=torch.int32, device=dev))),
                      torch.arange(2 * B + 1, device=dev), torch.cat((o, s)))

    def step():
        new_batch()
        st.step()

    ms = timed(step, args.steps, args.warmup)
    if args.kernels:
        kernel_table(step, 3, f"wd5m_1vsall_B{B}")
    hbm, tf = peaks()
    flops = 5 * 2.0 * (2 * B) * E * d   # 1 forward + 2x2 backward GEMMs (S recomputed per output)
    # bytes this implementation moves per step: 3 bf16 table reads (fwd, dQ, dTable), gradient zero + RMW,
    # Adagrad read W/state/grad + write W/state/mirror
    bytes_step = E * d * (3 * 2 + 4 + 8 + 12 + 10)
    return {"workload": f"DistMult 1vsAll+KL d=128 E={E} B={B} triples ({2 * B} query rows) {args.math}"
                        + (f", entity table row-sharded over {world} GPUs (same batch on every rank)" if world > 1 else ""),
            "metric": "training triples/s", "value": B / (ms * 1e-3), "ms_per_step": ms, "n_gpus": world,
            "loss": st.loss.item(),
            "roofline": {"tensor_tflops": flops / (ms * 1e-3) / 1e12, "tensor_frac_of_bf16_sustained": flops / (ms * 1e-3) / 1e12 / tf,
                         "hbm_gbs": bytes_step / (ms * 1e-3) / 1e9, "hbm_frac": bytes_step / (ms * 1e-3) / 1e9 / hbm,
                         "algorithmic_bytes_per_step": bytes_step, "algorithmic_flops_per_step": flops}}


def wd5m_1vsall_reciprocal(args):
    """DistMult with reciprocal relations (2 R relation rows, _po queries as sp_ queries on p + R), 1vsAll + KL, d=128,
    E=4.6M (scaled by --scale), --batch triples per step, against plain DistMult in the same process: both captured steps
    build their batch from the triples on the device (onevsall_triples), so the two differ only in the batch builder
    (kgeb_onevsall_batch_build_inv with R vs 0) and in the relation table's row count.  The two steppers are timed in
    alternating rounds of --steps steps; the medians are reported."""
    E, R, d, B = int(4_600_000 * args.scale), 822, 128, args.batch
    dev = torch.device("cuda")
    math_mode = {"bf16": kb.lib.MATH_BF16, "tf32": kb.lib.MATH_TF32, "fp32": kb.lib.MATH_FP32}[args.math]
    arms = {}
    for name in ("plain", "reciprocal"):
        torch.manual_seed(0)
        if name == "plain":
            model = kb.KgeModel("distmult", E, R, d).to(dev)
        else:
            model = kb.model.ReciprocalRelationsModel("distmult", E, R, d).to(dev)
        opt = kb.optim.create("Adagrad", model.parameters(), lr=0.2)
        st = kb.trainer.FusedAllEntityStepper(model, opt, 2 * B, 2 * B, kb.lib.LOSS_KL, B, math_mode=math_mode,
                                              onevsall_triples=True, reciprocal=name == "reciprocal")
        gen = torch.Generator(device=dev).manual_seed(1)
        batches = [torch.stack((torch.randint(0, E, (B,), device=dev, generator=gen),
                                torch.randint(0, R, (B,), device=dev, generator=gen),
                                torch.randint(0, E, (B,), device=dev, generator=gen)), 1) for _ in range(8)]
        arms[name] = dict(st=st, batches=batches, i=0, ms=[])

    def stepper_fn(arm):
        def step():
            arm["st"].set_triples(arm["batches"][arm["i"] % len(arm["batches"])])
            arm["i"] += 1
            arm["st"].step()
        return step

    fns = {name: stepper_fn(arm) for name, arm in arms.items()}
    for _ in range(5):
        for name in ("plain", "reciprocal"):
            arms[name]["ms"].append(timed(fns[name], args.steps, args.warmup))
    med = {name: float(np.median(arm["ms"])) for name, arm in arms.items()}
    gpu = torch.cuda.get_device_properties(dev).name
    return {"workload": f"DistMult reciprocal relations 1vsAll+KL d=128 E={E} R={R} (2R={2 * R} relation rows) B={B} "
                        f"triples ({2 * B} query rows) {args.math}, captured step with the batch built on the device; "
                        "plain DistMult in the same process, alternating rounds",
            "metric": "training triples/s", "value": B / (med["reciprocal"] * 1e-3), "ms_per_step": med["reciprocal"],
            "ms_per_step_plain": med["plain"], "ratio_reciprocal_over_plain": med["reciprocal"] / med["plain"],
            "ms_rounds": {name: arm["ms"] for name, arm in arms.items()},
            "flash_fallbacks": {name: arm["st"].flash_fallbacks for name, arm in arms.items()},
            "loss": {name: arm["st"].loss.item() for name, arm in arms.items()}, "gpu": gpu}


def gpu_info() -> dict:
    """Card name and power limit of this run (a read-only nvidia-smi query): part of every number measured here."""
    import subprocess
    out = {"gpu": torch.cuda.get_device_properties(0).name}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
        out["nvidia_smi"] = q
    except (OSError, subprocess.SubprocessError):
        out["nvidia_smi"] = "unavailable"
    return out


def wd5m_1vsall_lr_schedule(args):
    """The Wikidata5M 1vsAll + KL captured step (DistMult, d=128, batch built on the device) at a constant learning rate
    and with the rate changed before every step (one 4-byte fill of the rate word per step), in alternating rounds of
    --steps steps on one stepper; the medians are reported.  Then a one-process A/B of the table-gradient + Adagrad
    kernel alone: kgeb_fused_bwd_update (rate by value) against kgeb_fused_bwd_update_sched (rate read from a device word)
    on the same inputs, alternating rounds of --steps launches each."""
    E, R, d, B = int(4_600_000 * args.scale), 822, 128, args.batch
    dev = torch.device("cuda")
    torch.manual_seed(0)
    model = kb.KgeModel("distmult", E, R, d).to(dev)
    opt = kb.optim.create("Adagrad", model.parameters(), lr=0.2)
    st = kb.trainer.FusedAllEntityStepper(model, opt, 2 * B, 2 * B, kb.lib.LOSS_KL, B, math_mode=kb.lib.MATH_BF16,
                                          onevsall_triples=True)
    gen = torch.Generator(device=dev).manual_seed(1)
    batches = [torch.stack((torch.randint(0, E, (B,), device=dev, generator=gen),
                            torch.randint(0, R, (B,), device=dev, generator=gen),
                            torch.randint(0, E, (B,), device=dev, generator=gen)), 1) for _ in range(8)]
    state = {"i": 0}

    def step_fn(changing):
        def step():
            if changing:        # a new rate every step, as lr_decay or a per-batch scheduler gives
                opt.param_groups[0]["lr"] = 0.2 / (1.0 + 1e-4 * state["i"])
            st.set_triples(batches[state["i"] % len(batches)])
            state["i"] += 1
            st.step()
        return step

    ms = {"constant": [], "changing": []}
    for _ in range(5):
        for name in ("constant", "changing"):
            ms[name].append(timed(step_fn(name == "changing"), args.steps, args.warmup))
    med = {name: float(np.median(v)) for name, v in ms.items()}

    # kernel A/B on the step's shapes: [2B, d] queries against the E-row table, BCE (no log-sum-exp needed), no touched rows
    lib = kb.lib
    n = 2 * B
    q = torch.randn(n, d, device=dev, generator=gen) * 0.05
    w = model.get_s_embedder().weight.detach()
    s_ = opt.state[model.get_s_embedder().weight]["sum"]
    mirror = w.bfloat16()
    lab_off = torch.arange(n + 1, device=dev)
    slot_of = torch.full((E,), -1, dtype=torch.int32, device=dev)
    gbuf = torch.zeros(1, d, device=dev)
    ws = torch.empty(lib.load().kgeb_fused_workspace_bytes(n, d, E, 0), dtype=torch.uint8, device=dev)
    word = torch.tensor([1e-6], dtype=torch.float32, device=dev)       # a tiny rate: the table barely moves

    def kernel_fn(sched):
        rate = word.data_ptr() if sched else 1e-6
        name = "kgeb_fused_bwd_update_sched" if sched else "kgeb_fused_bwd_update"

        def call():
            lib.call(name, lib.LOSS_BCE, q.data_ptr(), n, d, w.data_ptr(), 0, E, E, lab_off.data_ptr(), 0.0, 0.0, None,
                     1.0 / n, None, mirror.data_ptr(), s_.data_ptr(), rate, 1e-10, slot_of.data_ptr(), gbuf.data_ptr(), None,
                     ws.data_ptr(), ws.numel(), lib.stream_ptr(w))
        return call

    kms = {"by_value": [], "sched": []}
    for _ in range(5):
        for name in ("by_value", "sched"):
            kms[name].append(timed(kernel_fn(name == "sched"), args.steps, args.warmup))
    kmed = {name: float(np.median(v)) for name, v in kms.items()}
    return {"workload": f"DistMult 1vsAll+KL d=128 E={E} B={B} triples ({2 * B} query rows) bf16, captured step with the "
                        "batch built on the device: constant lr vs lr changed before every step, alternating rounds on one "
                        "stepper; kernel A/B kgeb_fused_bwd_update vs _sched (BCE, same inputs), alternating rounds",
            "metric": "ms per step", "value": med["changing"], "ms_per_step_constant_lr": med["constant"],
            "ms_per_step_changing_lr": med["changing"], "ratio_changing_over_constant": med["changing"] / med["constant"],
            "ms_rounds": ms, "kernel_ms_by_value": kmed["by_value"], "kernel_ms_sched": kmed["sched"],
            "kernel_ratio_sched_over_by_value": kmed["sched"] / kmed["by_value"], "kernel_ms_rounds": kms,
            "flash_fallbacks": st.flash_fallbacks, "loss": st.loss.item(), "lr_words": st.rate.words.tolist(),
            **gpu_info()}


def wnrr_rotate_ns(args):
    """C3: RotatE negative sampling, 256 negatives for s and o, E=40943, R=11, B=512."""
    E, R, d, B, N = 40943, 11, 128, args.batch, 256
    dev = torch.device("cuda")
    torch.manual_seed(0)
    model = kb.KgeModel("rotate", E, R, d).to(dev)
    opt = kb.optim.create("Adagrad", model.parameters(), lr=0.2)
    job = kb.TrainingJobNegativeSampling(model, opt, kb.KgeLoss.create("kl"), fused_path=not args.reference_flow)
    if args.graph_step:
        job.enable_graph_step(B, N, N, segment_bwd=args.segment_bwd, fused_slot=not args.no_fused_slot,
                              deterministic=not args.atomic)
    gen = torch.Generator().manual_seed(1)
    batches = []
    for _ in range(8):
        t = torch.stack((torch.randint(0, E, (B,), generator=gen), torch.randint(0, R, (B,), generator=gen),
                         torch.randint(0, E, (B,), generator=gen)), 1)
        negs = [torch.randint(0, E, (B, N), generator=gen), torch.zeros(B, 0, dtype=torch.long),
                torch.randint(0, E, (B, N), generator=gen)]
        batches.append({"triples": t.to(dev), "negative_samples": [n.to(dev) for n in negs]})
    i = [0]

    def step():
        job.step(i[0], batches[i[0] % len(batches)])
        i[0] += 1

    ms = timed(step, args.steps, args.warmup)
    if args.kernels:
        kernel_table(step, 3, "wnrr_rotate_ns" + ("_graph" if args.graph_step else "") + ("_seg" if args.segment_bwd else "")
                     + ("_3k" if args.no_fused_slot else "") + ("_atomic" if args.atomic else ""))
    hbm, _ = peaks()
    bytes_step = B * 2 * (1 + N) * d * 4 * 2   # gather of each candidate row + write of its gradient row (SURVEY.md 8d C3)
    return {"workload": f"RotatE NS 2x{N} negatives d=128 E={E} B={B} ({'reference flow' if args.reference_flow else ('graph-captured fused step' + (', segment backward' if args.segment_bwd else '') + (', three kernels per slot' if args.no_fused_slot else ', one kernel per slot') + (', vector-reduction candidate gradients (not bit-reproducible)' if args.atomic else ', deterministic sorted scatter') if args.graph_step else 'fused pairs, autograd')})",
            "metric": "training triples/s", "value": B / (ms * 1e-3), "ms_per_step": ms,
            "roofline": {"hbm_gbs": bytes_step / (ms * 1e-3) / 1e9, "hbm_frac": bytes_step / (ms * 1e-3) / 1e9 / hbm,
                         "algorithmic_bytes_per_step": bytes_step}}


def wd5m_eval(args, model_name):
    """C5: filtered entity ranking on the Wikidata5M shape: B triples -> 2B queries per batch."""
    E, R, d, B = int(4_600_000 * args.scale), 822, 128, args.batch
    dev = torch.device("cuda")
    torch.manual_seed(0)
    math_mode = kb.lib.MATH_TF32 if (model_name == "complex" and args.math != "fp32") else kb.lib.MATH_FP32
    model = kb.KgeModel(model_name, E, R, d, math_mode=math_mode).to(dev)
    rng = np.random.default_rng(0)
    known = np.stack([rng.integers(0, E, 20000), rng.integers(0, R, 20000), rng.integers(0, E, 20000)], 1).astype(np.int32)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    shard = None
    if world > 1:   # every rank scores the whole batch against its own entity rows; int64 counts are all-reduced
        import torch.distributed as dist
        shard = kb.fused.Shard.of_rank(E, int(os.environ["RANK"]), world, dist.group.WORLD)
    if args.real_filter:
        # SURVEY.md 8(d) C5 as specified: the synthetic Wikidata5M-shaped graph (App. C generator, 20 M train + 5,000 valid +
        # 5,000 test triples), filter = train + valid (+ test for the filtered_with_test numbers) over the FULL splits,
        # every one of the 5,000 validation triples ranked once (10,000 queries), histograms and metrics included
        t0 = time.time()
        g = kb.graph.synthetic_graph("wikidata5m", seed=0, scale=args.scale)
        t1 = time.time()
        job = kb.EntityRankingJob(model, E, [g["train"], g["valid"]], g["test"], batch_size=B, math_mode=math_mode,
                                  hits_at_k_s=(1, 3, 10), shard=shard)
        t2 = time.time()
        job.run(g["valid"][:2 * B])                      # warm-up (index arrays to the device, kernels loaded)
        torch.cuda.synchronize()
        a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        res = job.run(g["valid"])
        b_.record()
        torch.cuda.synchronize()
        total_ms = a.elapsed_time(b_)
        nq = 2 * len(g["valid"])
        ops = 2.0 * nq * E * d
        hbm, tf = peaks()
        return {"workload": f"filtered ranking {model_name} d=128 E={E}, ALL {len(g['valid'])} validation triples ({nq} queries) in "
                            f"batches of {B}, filter = full train ({len(g['train'])}) + valid + test splits, "
                            f"{'tf32 tcgen05 tiles' if math_mode == kb.lib.MATH_TF32 else 'fp32 CUDA-core tiles'}"
                            + (f", scoring sharded by entity over {world} GPUs" if world > 1 else ""),
                "metric": "eval queries/s", "value": nq / (total_ms * 1e-3), "ms_per_batch": total_ms / (len(g["valid"]) / B),
                "n_gpus": world, "mrr_filtered": res["metrics"]["mean_reciprocal_rank_filtered"],
                "host_seconds": {"graph": t1 - t0, "indexes": t2 - t1},
                "roofline": {"ops_per_s_T": ops / (total_ms * 1e-3) / 1e12,
                             "frac_of_fp32_alu_nominal_37T": ops / (total_ms * 1e-3) / 1e12 / 37.2 if math_mode == kb.lib.MATH_FP32 else None,
                             "frac_of_bf16_sustained": ops / (total_ms * 1e-3) / 1e12 / tf if math_mode != kb.lib.MATH_FP32 else None}}
    job = kb.EntityRankingJob(model, E, [known], None, batch_size=B, math_mode=math_mode, hits_at_k_s=(1, 3, 10),
                              shard=shard)
    batch = torch.from_numpy(known[:B].copy())

    def step():
        job.rank_batch(batch)

    ms = timed(step, args.steps, args.warmup)
    if args.kernels:
        kernel_table(step, 3, f"wd5m_eval_{model_name}_B{B}")
    hbm, tf = peaks()
    ops = 2.0 * (2 * B) * E * d
    return {"workload": f"filtered ranking {model_name} d=128 E={E} B={B} triples ({2 * B} queries) "
                        f"{'tf32 tcgen05 tiles' if math_mode == kb.lib.MATH_TF32 else 'fp32 CUDA-core tiles'}"
                        + (f", scoring sharded by entity over {world} GPUs" if world > 1 else ""),
            "metric": "eval queries/s", "value": 2 * B / (ms * 1e-3), "ms_per_batch": ms, "n_gpus": world,
            "roofline": {"ops_per_s_T": ops / (ms * 1e-3) / 1e12,
                         "frac_of_fp32_alu_nominal_37T": ops / (ms * 1e-3) / 1e12 / 37.2 if math_mode == kb.lib.MATH_FP32 else None,
                         "frac_of_bf16_sustained": ops / (ms * 1e-3) / 1e12 / tf if math_mode != kb.lib.MATH_FP32 else None,
                         "table_read_gbs": E * d * 4 / (ms * 1e-3) / 1e9}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", required=True)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the 4.6M entities (memory / time bound runs)")
    ap.add_argument("--math", default="bf16")
    ap.add_argument("--reference-flow", action="store_true")
    ap.add_argument("--graph-step", action="store_true")
    ap.add_argument("--segment-bwd", action="store_true", help="negative sampling: candidate gradients by segment (ns_segment.cu)")
    ap.add_argument("--no-fused-slot", action="store_true", help="negative sampling: the three-kernel slot of round 1")
    ap.add_argument("--atomic", action="store_true", help="negative sampling: candidate gradients by vector reductions (not bit-reproducible)")
    ap.add_argument("--real-filter", action="store_true", help="eval workloads: the full synthetic graph as filter, all 5,000 validation triples")
    ap.add_argument("--kernels", action="store_true", help="also write a per-kernel time table (CUPTI) to gpurun_out/")
    args = ap.parse_args()
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
        dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
    if args.workload == "wd5m-1vsall":
        res = wd5m_1vsall(args)
    elif args.workload == "wd5m-1vsall-reciprocal":
        res = wd5m_1vsall_reciprocal(args)
    elif args.workload == "wd5m-1vsall-lr-schedule":
        res = wd5m_1vsall_lr_schedule(args)
    elif args.workload == "wnrr-rotate-ns":
        res = wnrr_rotate_ns(args)
    elif args.workload == "wd5m-eval-transe":
        res = wd5m_eval(args, "transe")
    elif args.workload == "wd5m-eval-complex":
        res = wd5m_eval(args, "complex")
    else:
        raise SystemExit(f"unknown workload {args.workload}")
    res.setdefault("n_gpus", 1)
    if int(os.environ.get("RANK", "0")) != 0:
        return
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    with open(os.path.join(ROOT, "gpurun_out", "extra_workloads.jsonl"), "a") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
