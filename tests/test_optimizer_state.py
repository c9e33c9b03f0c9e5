"""Host side of SageTrainer.optimizer (no GPU): validation of param groups and loaded state dicts, and the mapping
between the trainer's flat moment buffers and torch.optim.Adam's per-parameter state, on a stand-in trainer that holds
the flat buffers on the CPU."""
import io
from types import SimpleNamespace

import pytest
import torch
import torch.nn.functional as F

import gnn_tableextraction_b200 as gte
from gnn_tableextraction_b200.engine import TrainerAdam, check_adam_group, loaded_adam_step
from oracle import sage_oracle as so

CFG = (13, 24, 9, 3)


def _model(seed=0):
    torch.manual_seed(seed)
    return so.OracleGcnSAGE(*CFG, F.relu, 0)


def _flat_trainer(model):
    """what TrainerAdam reads of a SageTrainer: flat moment buffers with every tensor on a 4-float boundary, the
    offsets, and the device step counter"""
    offs, o = [], 0
    for p in model.parameters():
        offs.append(o)
        o += (p.numel() + 3) // 4 * 4
    return SimpleNamespace(exp_avg=torch.zeros(o), exp_avg_sq=torch.zeros(o), step_dev=torch.zeros(1, dtype=torch.int64),
                           _offs=offs)


def _adam_after(model, steps, lr=0.01):
    """a plain torch.optim.Adam over ``model`` after ``steps`` steps with seeded gradients"""
    opt = torch.optim.Adam(model.parameters(), lr=lr, weight_decay=5e-4)
    gen = torch.Generator().manual_seed(5)
    for _ in range(steps):
        for p in model.parameters():
            p.grad = torch.randn(p.shape, generator=gen)
        opt.step()
    return opt


def _trainer_adam(model):
    tr = _flat_trainer(model)
    return tr, TrainerAdam(tr, model.parameters(), 0.01, (0.9, 0.999), 1e-8, 5e-4)


def test_check_adam_group_accepts_torch_defaults_and_refuses_what_the_kernels_cannot_run():
    group = dict(torch.optim.Adam(_model().parameters(), lr=0.02, weight_decay=1e-4).param_groups[0])
    assert check_adam_group(group, "t") == (0.02, 0.9, 0.999, 1e-8, 1e-4)
    assert check_adam_group({**group, "lr": 0}, "t")[0] == 0.0
    for change, match in (({"amsgrad": True}, "amsgrad"), ({"maximize": True}, "maximize"),
                          ({"decoupled_weight_decay": True}, "decoupled_weight_decay"),
                          ({"lr": torch.tensor(0.01)}, "tensor"), ({"betas": (torch.tensor(0.9), 0.999)}, "tensor"),
                          ({"lr": -1.0}, "learning rate"), ({"lr": float("nan")}, "learning rate"),
                          ({"eps": -1e-8}, "epsilon"), ({"betas": (1.0, 0.999)}, "beta"), ({"betas": (0.9,)}, "pair"),
                          ({"weight_decay": -1.0}, "weight_decay"), ({"lr": "0.01"}, "number")):
        with pytest.raises(gte.GteError, match=match):
            check_adam_group({**group, **change}, "t")


def test_loaded_adam_step_reads_the_step_of_a_plain_adam_state_dict():
    model = _model()
    shapes = [p.shape for p in model.parameters()]
    assert loaded_adam_step(torch.optim.Adam(model.parameters()).state_dict(), shapes) == 0
    sd = _adam_after(model, 3).state_dict()
    assert loaded_adam_step(sd, shapes) == 3
    for st in sd["state"].values():  # torch before 1.12 saved the step as a Python number
        st["step"] = 3
    assert loaded_adam_step(sd, shapes) == 3


def _state_dict_refusals(model):
    def sd():
        return _adam_after(_model(), 2).state_dict()

    out = []
    s = sd()
    s["param_groups"].append(dict(s["param_groups"][0], params=[]))
    out.append((s, "one param group"))
    s = sd()
    s["param_groups"][0]["amsgrad"] = True
    out.append((s, "amsgrad"))
    s = sd()
    s["param_groups"][0]["lr"] = torch.tensor(0.01)
    out.append((s, "tensor"))
    s = sd()
    s["param_groups"][0]["params"] = s["param_groups"][0]["params"][:-1]
    out.append((s, "parameters, the model has"))
    s = sd()
    s["state"][1]["exp_avg"] = s["state"][1]["exp_avg"][:-1]
    out.append((s, "exp_avg of shape"))
    s = sd()
    s["state"][2]["step"] = torch.tensor(1.0)
    out.append((s, "different step counts"))
    s = sd()
    del s["state"][0]
    out.append((s, "no state"))
    return out


def test_loaded_adam_step_refuses_state_dicts_that_do_not_match_the_model():
    model = _model()
    shapes = [p.shape for p in model.parameters()]
    for sd, match in _state_dict_refusals(model):
        with pytest.raises(gte.GteError, match=match):
            loaded_adam_step(sd, shapes)


def test_trainer_adam_state_dict_has_the_format_of_a_plain_adam():
    m1, m2 = _model(), _model()
    ref = _adam_after(m1, 1).state_dict()
    tr, opt = _trainer_adam(m2)
    assert isinstance(opt, torch.optim.Optimizer) and len(opt.param_groups) == 1
    assert opt.state_dict()["state"] == {}  # before the first step, as torch
    tr.step_dev.fill_(1)
    sd = opt.state_dict()
    assert sd["param_groups"][0].keys() == ref["param_groups"][0].keys()
    assert sd["param_groups"][0] == ref["param_groups"][0]
    assert sd["state"].keys() == ref["state"].keys()
    for k, st in sd["state"].items():
        assert list(st.keys()) == list(ref["state"][k].keys())
        assert st["step"].dtype == ref["state"][k]["step"].dtype == torch.float32
        assert st["step"].device == ref["state"][k]["step"].device and st["step"].item() == 1
        assert st["exp_avg"].shape == ref["state"][k]["exp_avg"].shape


def test_trainer_adam_loads_a_plain_adam_checkpoint_into_the_flat_buffers_and_back():
    src = _model()
    ref = _adam_after(src, 4, lr=0.003)
    buf = io.BytesIO()
    torch.save(ref.state_dict(), buf)
    buf.seek(0)
    m = _model(1)
    tr, opt = _trainer_adam(m)
    exp_avg_ptr = tr.exp_avg.data_ptr()
    opt.load_state_dict(torch.load(buf))
    assert tr.exp_avg.data_ptr() == exp_avg_ptr and int(tr.step_dev.item()) == 4  # copied in place
    assert opt.param_groups[0]["lr"] == 0.003
    for p, q, off in zip(m.parameters(), src.parameters(), tr._offs):
        n = p.numel()
        assert torch.equal(tr.exp_avg[off:off + n].view_as(p), ref.state[q]["exp_avg"])
        assert torch.equal(tr.exp_avg_sq[off:off + n].view_as(p), ref.state[q]["exp_avg_sq"])
        # the optimizer's per-parameter state is a view of the flat buffers again
        assert opt.state[p]["exp_avg"].data_ptr() == tr.exp_avg[off:].data_ptr()
    pad = torch.ones(tr.exp_avg.numel(), dtype=torch.bool)
    for p, off in zip(m.parameters(), tr._offs):
        pad[off:off + p.numel()] = False
    assert (tr.exp_avg[pad] == 0).all()
    # and back into a plain Adam: the same state dict
    back = torch.optim.Adam(_model(2).parameters())
    back.load_state_dict(opt.state_dict())
    for k, st in back.state_dict()["state"].items():
        r = ref.state_dict()["state"][k]
        assert torch.equal(st["exp_avg"], r["exp_avg"]) and torch.equal(st["exp_avg_sq"], r["exp_avg_sq"])
        assert torch.equal(st["step"], r["step"])
    # an empty state dict: zero moments, step 0
    opt.load_state_dict(torch.optim.Adam(_model().parameters()).state_dict())
    assert int(tr.step_dev.item()) == 0 and not tr.exp_avg.any() and not tr.exp_avg_sq.any()
    assert opt.state_dict()["state"] == {}


def test_trainer_adam_refuses_bad_checkpoints_before_touching_its_state():
    m = _model()
    tr, opt = _trainer_adam(m)
    opt.load_state_dict(_adam_after(_model(), 2).state_dict())
    before = (tr.exp_avg.clone(), tr.exp_avg_sq.clone(), tr.step_dev.clone(), dict(opt.param_groups[0]))
    for sd, match in _state_dict_refusals(m):
        with pytest.raises(gte.GteError, match=match):
            opt.load_state_dict(sd)
        assert torch.equal(tr.exp_avg, before[0]) and torch.equal(tr.exp_avg_sq, before[1])
        assert torch.equal(tr.step_dev, before[2]) and opt.param_groups[0] == before[3]


def test_trainer_adam_refuses_step_zero_grad_and_a_second_group():
    m = _model()
    _, opt = _trainer_adam(m)
    grads = [p.grad for p in m.parameters()]
    for call in (opt.step, opt.zero_grad, lambda: opt.zero_grad(set_to_none=False)):
        with pytest.raises(gte.GteError):
            call()
    assert [p.grad for p in m.parameters()] == grads
    with pytest.raises(gte.GteError, match="one param group"):
        opt.add_param_group({"params": [torch.nn.Parameter(torch.zeros(3))]})
    # a scheduler wraps step(); the wrapped call is refused too
    sched = torch.optim.lr_scheduler.StepLR(opt, step_size=1, gamma=0.5)
    with pytest.raises(gte.GteError):
        opt.step()
    sched.step()
    assert opt.param_groups[0]["lr"] == 0.005
