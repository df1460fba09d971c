"""Run under torchrun on >= 2 GPUs (not collected by pytest):
    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tests/lr_schedule_multi_gpu_check.py
The sharded and replicated captured steps under a learning-rate schedule -- lr edited between steps, then an lr_decay
phase -- against the single-GPU step under the same schedule, with the tolerances of tests/multi_gpu_check.py,
tests/p2p_check.py and tests/p2p_ns_check.py:
  * RowShardedAllEntityStepper (peer-memory exchange kernels and NCCL) vs FusedAllEntityStepper on the whole batch;
  * data-parallel replicas with the peer-memory exchange (dp_p2p, kgeb_p2p_exchange_sched) vs the NCCL replicas;
  * data-parallel negative sampling (PeerExchange) vs FusedNegSamplingStepper on the global batch.
Every rank runs the same schedule, as ranks that run the same scheduler on the same metric do."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import kgeb200 as kb  # noqa: E402
from oracle import kge_oracle as ko  # noqa: E402

# (lr, lr_decay) of each step
SCHEDULE = [(0.2, 0.0), (0.2, 0.0), (0.05, 0.0), (0.05, 0.05), (0.05, 0.05)]


def _apply(opts, k):
    lr, decay = SCHEDULE[k]
    for o in opts:
        for g in o.param_groups:
            g["lr"], g["lr_decay"] = lr, decay


def row_sharded(rank, world, dev):
    e, r, d, b = 20_000, 12, 64, 128
    gen = torch.Generator().manual_seed(4)
    batches = [torch.stack((torch.randint(0, e, (b,), generator=gen), torch.randint(0, r, (b,), generator=gen),
                            torch.randint(0, e, (b,), generator=gen)), 1) for _ in SCHEDULE]
    for peer in (True, False):
        torch.manual_seed(0)
        ref = kb.KgeModel("distmult", e, r, d).to(dev)
        new = kb.KgeModel("distmult", e, r, d).to(dev)
        new.load_state_dict(ref.state_dict())
        opt_ref = kb.optim.create("Adagrad", ref.parameters(), lr=0.2)
        opt_new = kb.optim.create("Adagrad", new.parameters(), lr=0.2)
        single = kb.trainer.FusedAllEntityStepper(ref, opt_ref, 2 * b, 2 * b, kb.lib.LOSS_BCE, b, math_mode=kb.lib.MATH_BF16)
        sh = kb.fused.Shard.of_rank(e, rank, world, dist.group.WORLD)
        st = kb.trainer.RowShardedAllEntityStepper(new, opt_new, 2 * b, 2 * b, kb.lib.LOSS_BCE, b, sh,
                                                   math_mode=kb.lib.MATH_BF16, peer_memory=peer)
        for k, t in enumerate(batches):
            _apply((opt_ref, opt_new), k)
            tc = t.to(dev)
            s, p, o = tc[:, 0], tc[:, 1], tc[:, 2]
            z = torch.zeros(b, dtype=torch.int32, device=dev)
            args = (torch.cat((s, o)), torch.cat((p, p)), torch.cat((z, z + 1)), torch.arange(2 * b + 1, device=dev),
                    torch.cat((o, s)))
            single.set_inputs(*args)
            st.set_inputs(*args)
            a, c = single.step().item(), st.step().item()
            assert abs(a - c) <= 1e-3 * abs(a), (peer, k, a, c)
            assert st.rate.values == single.rate.values, (peer, k, st.rate.values, single.rate.values)
        st.check_peer()
        st.sync_tables()
        for x, y in ((ref.get_s_embedder().weight, new.get_s_embedder().weight),
                     (ref.get_p_embedder().weight, new.get_p_embedder().weight),
                     (opt_ref.state[ref.get_s_embedder().weight]["sum"], opt_new.state[new.get_s_embedder().weight]["sum"])):
            err = (x - y).abs().max().item()
            assert err <= 5e-3, (peer, err)
        if rank == 0:
            print(f"row-sharded step == single-GPU step under the schedule (world {world}, exchange="
                  f"{'peer-memory kernels' if st.px is not None else 'NCCL'}); rates {st.rate.values}", flush=True)
        del single, st


def replicas(rank, world, dev):
    g = kb.graph.synthetic_graph("toy", seed=3)
    e, r, d, b = g["num_entities"], g["num_relations"], 64, 96
    idx = [ko.kvsall_index(g["train"], "sp"), ko.kvsall_index(g["train"], "po")]
    rng = np.random.default_rng(100 + rank)
    batches = []
    for _ in SCHEDULE:
        ids = rng.choice(len(idx[0][0]) + len(idx[1][0]), b, replace=False)
        q, c, qt = ko.kvsall_collate(ids.tolist(), idx)
        batches.append({"queries": torch.from_numpy(q), "label_coords": torch.from_numpy(c),
                        "query_type_indexes": torch.from_numpy(qt)})
    t = torch.tensor([max(len(x["label_coords"]) for x in batches)], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    nnz_max = int(t.item())
    torch.manual_seed(0)
    models = [kb.KgeModel("complex", e, r, d).to(dev) for _ in range(2)]
    models[1].load_state_dict(models[0].state_dict())
    jobs = []
    for m, p2p in zip(models, (False, True)):
        job = kb.TrainingJobKvsAll(m, kb.optim.create("Adagrad", m.parameters(), lr=0.2), kb.KgeLoss.create("bce"), e, r,
                                   math_mode=kb.lib.MATH_BF16)
        job.enable_graph_step(b, nnz_max, use_graph=True, dp_group=dist.group.WORLD, dp_p2p=p2p)
        jobs.append(job)
    for k, batch in enumerate(batches):
        _apply([j.optimizer for j in jobs], k)
        a, c = jobs[0].step(k, batch), jobs[1].step(k, batch)
        jobs[1].stepper.check_p2p()
        tol = 0.0 if world == 2 else 2e-5 * abs(a.avg_loss)
        assert abs(a.avg_loss - c.avg_loss) <= tol, (k, a.avg_loss, c.avg_loss)
        for x, y in ((models[0].get_s_embedder().weight, models[1].get_s_embedder().weight),
                     (models[0].get_p_embedder().weight, models[1].get_p_embedder().weight)):
            err = (x - y).abs().max().item()
            assert err == 0.0 if world == 2 else err <= 2e-3, (k, err)
    w = models[1].get_s_embedder().weight.detach().contiguous()
    ws = [torch.empty_like(w) for _ in range(world)]
    dist.all_gather(ws, w)
    assert all(torch.equal(ws[0], x) for x in ws), "replicas diverged"
    if rank == 0:
        print(f"peer-memory replicas == NCCL replicas under the schedule (world {world}); rates "
              f"{jobs[1].stepper.rate.values}", flush=True)


def negative_sampling(rank, world, dev):
    g = kb.graph.synthetic_graph("toy", seed=3)
    e, r, d, b, n = g["num_entities"], g["num_relations"], 64, 32, 8
    rng = np.random.default_rng(7)
    steps = len(SCHEDULE)
    triples = [[torch.from_numpy(g["train"][(s * world + k) * b:(s * world + k + 1) * b].astype(np.int64)) for k in range(world)]
               for s in range(steps)]
    negs = [[[torch.from_numpy(rng.integers(0, e, (b, n))), torch.zeros(b, 0, dtype=torch.long),
              torch.from_numpy(rng.integers(0, e, (b, n)))] for _ in range(world)] for _ in range(steps)]
    torch.manual_seed(0)
    ref = kb.KgeModel("complex", e, r, d).to(dev)
    new = kb.KgeModel("complex", e, r, d).to(dev)
    new.load_state_dict(ref.state_dict())
    mk = lambda m: kb.optim.create("Adagrad", m.parameters(), lr=0.1, initial_accumulator_value=0.1)  # noqa: E731
    jr = kb.TrainingJobNegativeSampling(ref, mk(ref), kb.KgeLoss.create("kl"))
    jr.enable_graph_step(b * world, n, n, use_graph=True)
    jn = kb.TrainingJobNegativeSampling(new, mk(new), kb.KgeLoss.create("kl"))
    jn.enable_graph_step(b, n, n, use_graph=True, dp_group=dist.group.WORLD)
    for s in range(steps):
        _apply((jr.optimizer, jn.optimizer), s)
        glob = {"triples": torch.cat(triples[s]),
                "negative_samples": [torch.cat([negs[s][k][slot] for k in range(world)]) for slot in range(3)]}
        mine = {"triples": triples[s][rank], "negative_samples": negs[s][rank]}
        a, c = jr.step(s, glob), jn.step(s, mine)
        jn.stepper.px.check()
        assert abs(a.avg_loss - c.avg_loss) <= 1e-5 * abs(a.avg_loss), (s, a.avg_loss, c.avg_loss)
        for x, y in ((ref.get_s_embedder().weight, new.get_s_embedder().weight),
                     (ref.get_p_embedder().weight, new.get_p_embedder().weight)):
            err = (x - y).abs().max().item()
            assert err <= 1e-5, (s, err)
    if rank == 0:
        print(f"data-parallel negative-sampling step == single-GPU step under the schedule (world {world}); rates "
              f"{jn.stepper.rate.values}", flush=True)


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    dev = torch.device("cuda", torch.cuda.current_device())
    dist.init_process_group("nccl", device_id=dev)
    row_sharded(rank, world, dev)
    replicas(rank, world, dev)
    negative_sampling(rank, world, dev)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
