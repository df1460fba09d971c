"""CPU tests of the learning-rate handling of the captured steps: the one rate formula (optim.adagrad_clr) that
optim.Adagrad and the steppers share, the lookup of each table's own parameter group, and the refusals (weight_decay
still refused, lr_decay no longer).  No GPU needed: the negative-sampling stepper builds on CPU tensors without its graph,
and every refusal comes before anything touches a device."""
import os
import sys
import types

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import kgeb200 as kb  # noqa: E402

E, R, D = 50, 5, 16


@pytest.mark.parametrize("lr", [0.2, 0.05, 1e-3])
@pytest.mark.parametrize("lr_decay", [0.0, 0.05, 0.3])
def test_rate_formula_equals_torch_adagrad(lr, lr_decay):
    """torch.optim.Adagrad on a scalar parameter with gradient 1 and a zero accumulator moves it by exactly clr / (1 + eps)
    -- in double precision the formula must reproduce torch's rate to the last bits."""
    for step in range(1, 8):
        p = torch.zeros(1, dtype=torch.float64, requires_grad=True)
        opt = torch.optim.Adagrad([p], lr=lr, lr_decay=lr_decay, eps=0.0)
        opt.state[p]["step"] = torch.tensor(float(step - 1))
        p.grad = torch.ones(1, dtype=torch.float64)
        opt.step()
        assert -p.item() == pytest.approx(kb.optim.adagrad_clr(lr, lr_decay, step), rel=1e-15, abs=0), (lr, lr_decay, step)
    assert kb.optim.adagrad_clr(lr, lr_decay, 1) == lr


def test_the_rate_the_steppers_compute_is_the_one_optim_adagrad_applies():
    """adagrad_rates() before a step == the clr optim.Adagrad.step uses for that step (state["step"] + 1)."""
    m = kb.KgeModel("distmult", E, R, D)
    opt = kb.optim.create("Adagrad", m.parameters(), lr=0.3, lr_decay=0.1)
    ent, rel = m.get_s_embedder().weight, m.get_p_embedder().weight
    for k in range(5):
        want = [kb.optim.adagrad_clr(0.3, 0.1, k + 1)] * 2
        assert kb.trainer.adagrad_rates(opt, (ent, rel)) == want
        for p in (ent, rel):
            opt.state[p]["step"] += 1


def test_each_table_takes_its_own_parameter_group():
    m = kb.KgeModel("distmult", E, R, D)
    ent, rel = m.get_s_embedder().weight, m.get_p_embedder().weight
    # relation table in the FIRST group: a lookup of param_groups[0] would hand it to the entity table
    opt = kb.optim.Adagrad([{"params": [rel], "lr": 0.01, "eps": 1e-6},
                            {"params": [ent], "lr": 0.5, "lr_decay": 0.2, "eps": 1e-9}])
    assert kb.optim.group_of(opt, ent) is opt.param_groups[1]
    assert kb.optim.group_of(opt, rel) is opt.param_groups[0]
    for p in (ent, rel):
        opt.state[p]["step"] += 3
    assert kb.trainer.adagrad_rates(opt, (ent, rel)) == [kb.optim.adagrad_clr(0.5, 0.2, 4), 0.01]
    with pytest.raises(ValueError):
        kb.optim.group_of(opt, torch.nn.Parameter(torch.zeros(2)))


def test_negative_sampling_stepper_keeps_one_word_per_table_and_writes_it_on_change():
    """Built on CPU tensors without a graph: the device words hold each table's rate, the eps of each table's group,
    and refresh() follows an edit of param_groups (what an lr scheduler does) and lr_decay."""
    m = kb.KgeModel("distmult", E, R, D)
    ent, rel = m.get_s_embedder().weight, m.get_p_embedder().weight
    opt = kb.optim.Adagrad([{"params": [ent], "lr": 0.2, "eps": 1e-8},
                            {"params": [rel], "lr": 0.05, "lr_decay": 0.5, "eps": 1e-7}])
    st = kb.trainer.FusedNegSamplingStepper(m, opt, 4, 2, 2, kb.lib.LOSS_KL, use_graph=False)
    f32 = lambda x: torch.tensor(x, dtype=torch.float32).item()   # noqa: E731
    assert st.rate.words.dtype == torch.float32 and st.rate.words.numel() == 2
    assert st.rate.words.tolist() == [f32(0.2), f32(0.05)]
    assert (st.eps_ent, st.eps_rel) == (1e-8, 1e-7)
    opt.param_groups[0]["lr"] = 0.0125
    for p in (ent, rel):
        opt.state[p]["step"] += 1
    st.rate.refresh()
    assert st.rate.words.tolist() == [f32(0.0125), f32(kb.optim.adagrad_clr(0.05, 0.5, 2))]
    assert st.rate.values == [0.0125, kb.optim.adagrad_clr(0.05, 0.5, 2)]


def _distributed_shard():
    return types.SimpleNamespace(e_lo=0, e_hi=E // 2, num_entities=E, group=None, distributed=True)


def _steppers(m, opt):
    return [lambda: kb.trainer.FusedAllEntityStepper(m, opt, 8, 8, kb.lib.LOSS_KL, 4, use_graph=False),
            lambda: kb.trainer.RowShardedAllEntityStepper(m, opt, 8, 8, kb.lib.LOSS_KL, 4, _distributed_shard(),
                                                          use_graph=False, peer_memory=False),
            lambda: kb.trainer.FusedNegSamplingStepper(m, opt, 4, 2, 2, kb.lib.LOSS_KL, use_graph=False),
            lambda: kb.trainer.ShardedNegSamplingStepper(m, opt, 4, 2, 2, kb.lib.LOSS_KL)]


def test_weight_decay_is_still_refused_by_every_stepper():
    m = kb.KgeModel("distmult", E, R, D)
    ent, rel = m.get_s_embedder().weight, m.get_p_embedder().weight
    # in the relation table's group only: every table's own group is checked
    opt = kb.optim.Adagrad([{"params": [ent]}, {"params": [rel], "weight_decay": 1e-4}], lr=0.1)
    for make in _steppers(m, opt):
        with pytest.raises(NotImplementedError, match="weight_decay"):
            make()


def test_lr_decay_is_no_longer_refused():
    """Past the optimizer checks, a CPU model fails where the step needs a GPU (streams, process groups) -- with anything
    but the NotImplementedError of a refusal."""
    m = kb.KgeModel("distmult", E, R, D)
    opt = kb.optim.create("Adagrad", m.parameters(), lr=0.1, lr_decay=0.05)
    for make in _steppers(m, opt):
        try:
            make()
        except NotImplementedError as exc:        # pragma: no cover - the failure this test is about
            raise AssertionError(f"lr_decay refused: {exc}")
        except Exception:
            pass
