"""
Host side of FusedAdam / FusedAdamW (utils/optim_util.py), without a GPU: get_optimizer resolution, torch's
constructor defaults, the options that are refused, the exported C symbol and state_dict conversion.
"""
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _model():
    return torch.nn.Sequential(torch.nn.Conv2d(3, 8, 3), torch.nn.Linear(8, 4))


@pytest.mark.parametrize("name,cls_name,base", [("SGD", "FusedSGD", torch.optim.SGD),
                                                ("Adam", "FusedAdam", torch.optim.Adam),
                                                ("AdamW", "FusedAdamW", torch.optim.AdamW)])
def test_get_optimizer_resolves_fused_classes(name, cls_name, base):
    from pytorch_ddp_resnet_b200.utils import optim_util
    args = dict(lr=0.1, momentum=0.9) if name == "SGD" else dict(lr=1e-3)
    opt = optim_util.get_optimizer(name, _model(), args)
    assert type(opt) is getattr(optim_util, cls_name)
    assert isinstance(opt, base)
    assert opt._step_supports_amp_scaling


def test_other_names_still_resolve_to_torch():
    from pytorch_ddp_resnet_b200.utils.optim_util import get_optimizer
    opt = get_optimizer("RMSprop", _model(), dict(lr=1e-3))
    assert type(opt) is torch.optim.RMSprop
    opt = get_optimizer("Adagrad", _model(), dict(lr=1e-2))
    assert type(opt) is torch.optim.Adagrad


@pytest.mark.parametrize("cls_name,base", [("FusedAdam", torch.optim.Adam), ("FusedAdamW", torch.optim.AdamW)])
def test_constructor_defaults_match_torch(cls_name, base):
    from pytorch_ddp_resnet_b200.utils import optim_util
    mine = getattr(optim_util, cls_name)(_model().parameters())
    theirs = base(_model().parameters())
    assert mine.defaults == theirs.defaults
    keys = ("lr", "betas", "eps", "weight_decay", "amsgrad", "maximize", "capturable", "differentiable",
            "decoupled_weight_decay", "foreach", "fused")
    for g1, g2 in zip(mine.param_groups, theirs.param_groups):
        assert {k: g1[k] for k in keys} == {k: g2[k] for k in keys}
    assert theirs.defaults["weight_decay"] == (0.01 if base is torch.optim.AdamW else 0.0)
    assert mine.defaults["decoupled_weight_decay"] == (base is torch.optim.AdamW)


@pytest.mark.parametrize("cls_name", ["FusedAdam", "FusedAdamW"])
def test_every_torch_hyperparameter_is_accepted(cls_name):
    from pytorch_ddp_resnet_b200.utils import optim_util
    cls = getattr(optim_util, cls_name)
    extra = dict(decoupled_weight_decay=True) if cls_name == "FusedAdam" else {}
    opt = cls(_model().parameters(), lr=3e-4, betas=(0.8, 0.99), eps=1e-6, weight_decay=5e-4, amsgrad=True,
              foreach=True, fused=True, capturable=True, **extra)   # the last three are accepted and ignored
    g = opt.param_groups[0]
    assert (g["lr"], g["betas"], g["eps"], g["weight_decay"], g["amsgrad"]) == (3e-4, (0.8, 0.99), 1e-6, 5e-4, True)
    assert g["decoupled_weight_decay"] is True
    assert not g["fused"] and not g["capturable"]


def test_param_groups_keep_their_own_hyperparameters():
    from pytorch_ddp_resnet_b200.utils.optim_util import FusedAdamW
    m = _model()
    opt = FusedAdamW([{"params": m[0].parameters(), "lr": 1e-2, "weight_decay": 0.0},
                      {"params": m[1].parameters()}], lr=1e-3)
    assert [(g["lr"], g["weight_decay"]) for g in opt.param_groups] == [(1e-2, 0.0), (1e-3, 0.01)]


@pytest.mark.parametrize("cls_name", ["FusedAdam", "FusedAdamW"])
@pytest.mark.parametrize("flag", ["maximize", "differentiable"])
def test_unsupported_options_raise(cls_name, flag):
    from pytorch_ddp_resnet_b200.utils import optim_util
    with pytest.raises(NotImplementedError, match=flag):
        getattr(optim_util, cls_name)(_model().parameters(), **{flag: True})


def test_cpu_parameters_are_refused_at_step():
    from pytorch_ddp_resnet_b200.utils.optim_util import FusedAdamW
    w = torch.nn.Parameter(torch.randn(4, 4))
    opt = FusedAdamW([w])
    w.grad = torch.ones_like(w)
    with pytest.raises(RuntimeError, match="fp32 CUDA parameters"):
        opt.step()


def test_header_declares_and_library_exports_adam_step():
    from pytorch_ddp_resnet_b200 import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "b200resnet.h")).read()
    assert "int b200_adam_step(" in header
    assert "b200_adam_step" in _lib.SIGNATURES
    restype, argtypes = _lib.SIGNATURES["b200_adam_step"]
    assert len(argtypes) == 21
    assert hasattr(_lib.load(), "b200_adam_step")


@pytest.mark.parametrize("step", [3, torch.tensor(3.0), torch.tensor(3, dtype=torch.int64)])
def test_prepare_state_converts_step_and_relayouts_moments(step):
    """What load_state_dict does to each parameter's state (shown on host tensors): the step becomes a 0-d fp32
    tensor on the parameter's device, NCHW-contiguous moments take a channels_last parameter's layout."""
    from pytorch_ddp_resnet_b200.utils.optim_util import _FusedAdamBase, _same_layout
    p = torch.randn(8, 3, 3, 3).contiguous(memory_format=torch.channels_last)
    m = torch.randn(8, 3, 3, 3)
    state = {"step": step, "exp_avg": m.clone(), "exp_avg_sq": m.abs()}
    _FusedAdamBase._prepare_state(p, state)
    assert torch.is_tensor(state["step"]) and state["step"].dtype == torch.float32 and state["step"].dim() == 0
    assert float(state["step"]) == 3.0
    for k in ("exp_avg", "exp_avg_sq"):
        assert _same_layout(state[k], p)
    assert torch.equal(state["exp_avg"], m) and torch.equal(state["exp_avg_sq"], m.abs())
