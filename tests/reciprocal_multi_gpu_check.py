"""Run under torchrun on >= 2 GPUs (not collected by pytest):
    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tests/reciprocal_multi_gpu_check.py
Checks that the row-sharded training step of a reciprocal relations model (RowShardedAllEntityStepper(reciprocal=True):
_po queries as sp_ rows on relation p + R, 2 R-row relation table replicated) equals the single-GPU reciprocal step
(FusedAllEntityStepper(reciprocal=True), batch built on the device from the triples), with the tolerances of
tests/multi_gpu_check.py."""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import kgeb200 as kb  # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl", device_id=dev)
    e, r, d, b = 20_000, 12, 64, 128
    gen = torch.Generator().manual_seed(4)
    batches = [torch.stack((torch.randint(0, e, (b,), generator=gen), torch.randint(0, r, (b,), generator=gen),
                            torch.randint(0, e, (b,), generator=gen)), 1) for _ in range(3)]
    for loss_name, loss_kind, math_mode, use_graph, peer in (("bce", kb.lib.LOSS_BCE, kb.lib.MATH_BF16, True, True),
                                                             ("kl", kb.lib.LOSS_KL, kb.lib.MATH_BF16, True, True),
                                                             ("bce", kb.lib.LOSS_BCE, kb.lib.MATH_BF16, True, False),
                                                             ("kl", kb.lib.LOSS_KL, kb.lib.MATH_FP32, False, True),
                                                             ("kl", kb.lib.LOSS_KL, kb.lib.MATH_FP32, False, False)):
        torch.manual_seed(0)
        ref = kb.model.ReciprocalRelationsModel("distmult", e, r, d).to(dev)
        new = kb.model.ReciprocalRelationsModel("distmult", e, r, d).to(dev)
        new.load_state_dict(ref.state_dict())
        opt_ref = kb.optim.create("Adagrad", ref.parameters(), lr=0.2)
        opt_new = kb.optim.create("Adagrad", new.parameters(), lr=0.2)
        single = kb.trainer.FusedAllEntityStepper(ref, opt_ref, 2 * b, 2 * b, loss_kind, b, math_mode=math_mode,
                                                  onevsall_triples=True, reciprocal=True)
        sh = kb.fused.Shard.of_rank(e, rank, world, dist.group.WORLD)
        st = kb.trainer.RowShardedAllEntityStepper(new, opt_new, 2 * b, 2 * b, loss_kind, b, sh, math_mode=math_mode,
                                                   use_graph=use_graph, peer_memory=peer, reciprocal=True)
        if peer and st.px is None and rank == 0:
            print("  (symmetric memory unavailable: this case ran over NCCL)")
        # KL on the bf16 tiles: one step only (see multi_gpu_check.py: a flipped sign of a ~1e-9 gradient moves a weight
        # by 2 * lr, after which the runs are different trajectories)
        for i, t in enumerate(batches[:1] if (loss_name == "kl" and math_mode == kb.lib.MATH_BF16) else batches):
            tc = t.to(dev)
            s, p, o = tc[:, 0], tc[:, 1], tc[:, 2]
            st.set_inputs(torch.cat((s, o)), torch.cat((p, p + r)), torch.zeros(2 * b, dtype=torch.int32, device=dev),
                          torch.arange(2 * b + 1, dtype=torch.int64, device=dev), torch.cat((o, s)))
            single.set_triples(tc)
            a, c = single.step().item(), st.step().item()
            ltol = 1e-3 if math_mode == kb.lib.MATH_BF16 else 1e-4
            assert abs(a - c) <= ltol * abs(a), (loss_name, math_mode, i, a, c)
        st.check_peer()
        st.sync_tables()
        for x, y in ((ref.get_s_embedder().weight, new.get_s_embedder().weight),
                     (ref.get_p_embedder().weight, new.get_p_embedder().weight),
                     (opt_ref.state[ref.get_s_embedder().weight]["sum"], opt_new.state[new.get_s_embedder().weight]["sum"]),
                     (opt_ref.state[ref.get_p_embedder().weight]["sum"], opt_new.state[new.get_p_embedder().weight]["sum"])):
            diff = (x - y).abs()
            if loss_name == "bce":
                assert diff.max().item() <= 5e-3, (loss_name, math_mode, diff.max().item())
            else:
                frac = (diff > 5e-3).float().mean().item()
                assert frac <= 5e-3, (loss_name, math_mode, frac, diff.max().item())
        moved = (opt_new.state[new.get_p_embedder().weight]["sum"] != 0).any(1)
        assert moved[:r].any() and moved[r:].any()        # sp_ rows on p and inverse rows on p + R
        if rank == 0:
            print(f"row-sharded reciprocal step == single-GPU reciprocal step ({loss_name}, math={math_mode}, "
                  f"graph={use_graph}, exchange={'peer-memory kernels' if st.px is not None else 'NCCL'})")
        del single, st
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
