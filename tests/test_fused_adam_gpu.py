"""
FusedAdam / FusedAdamW (utils/optim_util.py) and b200_adam_step (csrc/head_sgd.cuh) on the GPU.

Error bound. Every comparison starts from the SAME fp32 state (params, moments, step) and checks one step, so
errors never compound. For one element, with eps32 = 2^-24 (the largest relative error of one fp32 rounding to
nearest) and the fp64 restatement of torch's formula

    g = grad * inv_scale;  wd: decoupled ? p *= 1 - lr*wd : g += wd*p
    m' = m + (1-b1)(g - m);  v' = b2 v + (1-b2) g^2;  vv = amsgrad ? max(vmax, v') : v'
    D = sqrt(vv) / sqrt(1 - b2^t) + eps;  u = (lr / (1 - b1^t)) m' / D;  p' = p - u

the kernel's fp32 evaluation stays within the first-order worst case W, the sum of one eps32 per rounding:
    W(m')  = 4 eps32 (|m| + |g|~)                 |g|~ = |g| + wd|p| (coupled decay): rounded g, g - m, the fma
    W(v')  = 6 eps32 (b2 |v| + (1-b2) |g|~^2)     rounded g (twice in g^2), 1-b2, (1-b2) g, b2 v, the fma
    W(D)   = min(sqrt(W(vv)), W(vv) / (2 sqrt(vv))) / sqrt(bc2) + 4 eps32 D      sqrt, sqrt(bc2), /, + eps
    W(u)   = (lr/bc1) W(m') / D + |u| (W(D) / D + 4 eps32)                      lr/bc1, m'/D, the fma product
    W(p')  = eps32 |p'| + [decoupled] 2 eps32 |p| + W(u)                         the parameter's own rounding
The bound is 2 W: a result within the worst case scores at most 0.5, which every check requires. The parameter's
own rounding (half an ulp, up to eps32 |p'| at the bottom of a binade) can take it close to 0.5 by itself, so
parameter ratios just under 0.5 are expected. Against torch.optim, whose fp32 evaluation has its own error of the
same kind, the bound is 2 (W + W) = 4 W.
"""
import io
import os
import subprocess
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests.kernel_check import kernels_launched  # noqa: E402

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS32 = 2.0 ** -24
STATE_KEYS = ("exp_avg", "exp_avg_sq", "max_exp_avg_sq")


def _ops():
    from pytorch_ddp_resnet_b200 import ops
    return ops


# ---------------------------------------------------------------------------------------------------------
# fp64 reference and its bound
# ---------------------------------------------------------------------------------------------------------
def _reference(p, g, m, v, vmax, t, hp, lr_exact=True):
    """fp64 result of one step from fp32 state at step t (1-based) and the worst-case fp32 error W of each output.
    hp: lr, betas, eps, weight_decay, decoupled, amsgrad, inv_scale. Returns {name: (ref, W)}."""
    lr, (b1, b2), eps, wd = hp["lr"], hp["betas"], hp["eps"], hp["weight_decay"]
    p, g, m, v = (x.double() for x in (p, g, m, v))
    g = g * hp.get("inv_scale", 1.0)
    gmag = g.abs()
    p_in = p
    if wd != 0:
        if hp["decoupled"]:
            p = p * (1 - lr * wd)
        else:
            g = g + wd * p
            gmag = gmag + wd * p.abs()
    m1 = m + (1 - b1) * (g - m)
    v1 = b2 * v + (1 - b2) * g * g
    w_m = 4 * EPS32 * (m.abs() + gmag)
    w_v = 6 * EPS32 * (b2 * v.abs() + (1 - b2) * gmag * gmag)
    out = {"exp_avg": (m1, w_m), "exp_avg_sq": (v1, w_v)}
    vv = v1
    if hp["amsgrad"]:
        vv = torch.maximum(vmax.double(), v1)
        out["max_exp_avg_sq"] = (vv, w_v)
    bc1, bc2 = 1 - b1 ** t, 1 - b2 ** t
    sv = vv.sqrt()
    d = sv / bc2 ** 0.5 + eps
    w_sqrt = torch.minimum(w_v.sqrt(), w_v / (2 * sv).clamp_min(1e-300))
    w_d = w_sqrt / bc2 ** 0.5 + 4 * EPS32 * d
    u = (lr / bc1) * m1 / d
    w_u = (lr / bc1) * w_m / d + u.abs() * (w_d / d + 4 * EPS32 + (0 if lr_exact else EPS32))
    p1 = p - u
    w_p = EPS32 * p1.abs() + w_u
    if wd != 0 and hp["decoupled"]:
        w_p = w_p + 2 * EPS32 * p_in.abs()
    out["param"] = (p1, w_p)
    return out


def _worst_ratio(got, ref, w, factor):
    """max |got - ref| / (factor * W); W is floored at the smallest fp32 normal (exact zeros stay zero)."""
    err = (got.double() - ref).abs()
    bound = factor * w.clamp_min(2.0 ** -126)
    return float((err / bound).max())


# ---------------------------------------------------------------------------------------------------------
# 1. the kernel, through ops.adam_step, against fp64
# ---------------------------------------------------------------------------------------------------------
SIZES = [1, 3, 4, 4097, 640 * 640 * 3 * 3]   # + one 4097-element set offset by one float (scalar path)


def _tensor_set(n, offset, gen):
    """p, g, m, v, vmax as separate allocations, each starting `offset` floats into its buffer."""
    def make(x):
        buf = torch.empty(n + offset, device="cuda")
        view = buf[offset:]
        view.copy_(x)
        return view
    p = make(torch.randn(n, device="cuda", generator=gen) * 0.1)
    return [p] + [make(torch.zeros(n, device="cuda")) for _ in range(4)]


def _launch(sets, steps, hp, inv_scale=None, found_inf=None, lr_dev=None):
    ops = _ops()
    rows = [[s[k].data_ptr() for s in sets] for k in range(5)]
    rows.append([t.data_ptr() for t in steps])
    rows.append([s[0].numel() for s in sets])
    table = torch.tensor(rows, dtype=torch.int64, device="cuda")
    ops.adam_step(table, len(sets), max(s[0].numel() for s in sets), hp["lr"], hp["betas"][0], hp["betas"][1],
                  hp["eps"], hp["weight_decay"], hp["decoupled"], hp["amsgrad"], inv_scale=inv_scale,
                  found_inf=found_inf, lr_dev=lr_dev)


@pytest.mark.parametrize("decoupled", [False, True], ids=["adam", "adamw"])
@pytest.mark.parametrize("amsgrad", [False, True], ids=["plain", "amsgrad"])
@pytest.mark.parametrize("wd", [0.0, 5e-4])
def test_kernel_against_fp64(decoupled, amsgrad, wd):
    gen = torch.Generator(device="cuda").manual_seed(1)
    sets = [_tensor_set(n, 0, gen) for n in SIZES] + [_tensor_set(4097, 1, gen)]
    assert sets[-1][0].data_ptr() % 16 == 4
    steps = [torch.zeros((), device="cuda") for _ in sets]
    hp = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=wd, decoupled=decoupled, amsgrad=amsgrad)
    worst = {}
    for t in range(1, 21):
        grads = [torch.randn(s[0].numel(), device="cuda", generator=gen) * (1.0 if t % 3 else 1e-3) for s in sets]
        for s, g in zip(sets, grads):
            s[1].copy_(g)
        before = [[x.clone() for x in s] for s in sets]
        _launch(sets, steps, hp)
        for i, (s, b) in enumerate(zip(sets, before)):
            ref = _reference(b[0], b[1], b[2], b[3], b[4], t, hp)
            got = {"param": s[0], "exp_avg": s[2], "exp_avg_sq": s[3], "max_exp_avg_sq": s[4]}
            for k, (r, w) in ref.items():
                worst[k] = max(worst.get(k, 0.0), _worst_ratio(got[k], r, w, 2.0))
            assert float(steps[i]) == float(t)
    print(f"worst ratio to 2W: {worst}")
    assert max(worst.values()) <= 0.5, worst


def test_kernel_device_lr_and_inv_scale():
    """lr from the device scalar overrides the argument; inv_scale multiplies the gradient."""
    gen = torch.Generator(device="cuda").manual_seed(2)
    sets = [_tensor_set(n, 0, gen) for n in (5, 4096)]
    steps = [torch.zeros((), device="cuda") for _ in sets]
    hp = dict(lr=123.0, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, decoupled=True, amsgrad=False)
    lr_dev = torch.full((), 2e-3, device="cuda")
    before = [[x.clone() for x in s] for s in sets]
    for s in sets:
        s[1].copy_(torch.randn(s[0].numel(), device="cuda", generator=gen) * 1024.0)
    grads = [s[1].clone() for s in sets]
    _launch(sets, steps, hp, inv_scale=torch.full((), 1 / 1024.0, device="cuda"), lr_dev=lr_dev)
    for s, b, g in zip(sets, before, grads):
        ref = _reference(b[0], g, b[2], b[3], b[4], 1, dict(hp, lr=2e-3, inv_scale=1 / 1024.0), lr_exact=False)
        r, w = ref["param"]
        assert _worst_ratio(s[0], r, w, 2.0) <= 0.5


# ---------------------------------------------------------------------------------------------------------
# 2. against torch.optim.Adam / AdamW (foreach=False)
# ---------------------------------------------------------------------------------------------------------
def _params(gen):
    shapes = [(160, 160, 3, 3), (640, 10), (10,), (3,), (4097,)]
    ps = []
    for sh in shapes:
        x = torch.randn(sh, device="cuda", generator=gen) * 0.1
        if len(sh) == 4:
            x = x.contiguous(memory_format=torch.channels_last)
        ps.append(torch.nn.Parameter(x))
    return ps


def _sync_torch_from_fused(fused, theirs_opt, mine, theirs):
    """torch's optimizer takes the fused optimizer's exact parameters and state (step as a host tensor)."""
    with torch.no_grad():
        for p, q in zip(mine, theirs):
            q.copy_(p)
            st = fused.state[p]
            if not st:
                continue
            ts = theirs_opt.state[q]
            ts["step"] = torch.tensor(float(st["step"]))
            for k in STATE_KEYS:
                if k in st:
                    ts[k] = st[k].clone()


def _groups(ps, cls_name):
    return [{"params": ps[:2], "lr": 1e-3, "weight_decay": 5e-4},
            {"params": ps[2:], "lr": 3e-3, "weight_decay": 0.0 if cls_name == "Adam" else 0.05}]


@pytest.mark.parametrize("cls_name", ["Adam", "AdamW"])
@pytest.mark.parametrize("amsgrad", [False, True], ids=["plain", "amsgrad"])
def test_against_torch_optim(cls_name, amsgrad):
    from pytorch_ddp_resnet_b200.utils import optim_util
    gen = torch.Generator(device="cuda").manual_seed(3)
    mine = _params(gen)
    theirs = [torch.nn.Parameter(p.detach().clone()) for p in mine]
    fused = getattr(optim_util, "Fused" + cls_name)(_groups(mine, cls_name), amsgrad=amsgrad)
    ref = getattr(torch.optim, cls_name)(_groups(theirs, cls_name), amsgrad=amsgrad, foreach=False)
    worst = 0.0
    for t in range(1, 9):
        if t == 5:   # an lr change between steps, in one group
            fused.param_groups[0]["lr"] = ref.param_groups[0]["lr"] = 4e-4
        _sync_torch_from_fused(fused, ref, mine, theirs)
        before = {id(p): (p.detach().clone(), {k: v.clone() for k, v in fused.state[p].items()}) for p in mine}
        for p, q in zip(mine, theirs):
            g = torch.randn(p.shape, device="cuda", generator=gen).contiguous(memory_format=torch.channels_last) \
                if p.dim() == 4 else torch.randn(p.shape, device="cuda", generator=gen)
            p.grad, q.grad = g, g.clone()
        fused.step()
        ref.step()
        for gi, group in enumerate(fused.param_groups):
            hp = dict(lr=group["lr"], betas=group["betas"], eps=group["eps"], weight_decay=group["weight_decay"],
                      decoupled=group["decoupled_weight_decay"], amsgrad=amsgrad)
            for p, q in zip(group["params"], ref.param_groups[gi]["params"]):
                p0, st0 = before[id(p)]
                z = torch.zeros_like(p0)
                bound = _reference(p0, p.grad, st0.get("exp_avg", z), st0.get("exp_avg_sq", z),
                                   st0.get("max_exp_avg_sq", z), t, hp, lr_exact=False)
                pairs = [("param", p, q)] + [(k, fused.state[p][k], ref.state[q][k]) for k in STATE_KEYS
                                             if k in fused.state[p]]
                for k, a, b in pairs:
                    assert a.stride() == b.stride() or a.dim() < 4
                    worst = max(worst, _worst_ratio(a, b.double(), bound[k][1], 4.0))
                assert float(fused.state[p]["step"]) == float(ref.state[q]["step"]) == t
                assert fused.state[p]["step"].is_cuda and fused.state[p]["step"].dtype == torch.float32
    print(f"{cls_name} amsgrad={amsgrad}: worst ratio to 4W against torch: {worst:.3f}")
    assert worst <= 0.5


# ---------------------------------------------------------------------------------------------------------
# 3. GradScaler contract
# ---------------------------------------------------------------------------------------------------------
def _snapshot(opt, ps):
    return [p.detach().clone() for p in ps] + [v.clone() for p in ps for v in opt.state[p].values()]


@pytest.mark.parametrize("amsgrad", [False, True], ids=["plain", "amsgrad"])
def test_found_inf_skips_everything_and_scaled_grads_equal_unscaled(amsgrad):
    from pytorch_ddp_resnet_b200.utils.optim_util import FusedAdamW
    gen = torch.Generator(device="cuda").manual_seed(4)
    ps = _params(gen)
    twins = [torch.nn.Parameter(p.detach().clone()) for p in ps]
    o1, o2 = FusedAdamW(ps, amsgrad=amsgrad), FusedAdamW(twins, amsgrad=amsgrad)
    for _ in range(2):
        for p, q in zip(ps, twins):
            g = torch.randn(p.shape, device="cuda", generator=gen)
            p.grad, q.grad = g.clone(), g * 65536.0
        o1.step()
        o2.grad_scale = torch.full((), 65536.0, device="cuda")
        o2.found_inf = torch.zeros((), device="cuda")
        o2.step()
        del o2.grad_scale, o2.found_inf
        # scaling by a power of two is exact, so the scaled step is not just within the bound: it is identical
        for a, b in zip(_snapshot(o1, ps), _snapshot(o2, twins)):
            assert torch.equal(a, b)
    before = _snapshot(o2, twins)
    for q in twins:
        q.grad = torch.randn(q.shape, device="cuda", generator=gen)
    o2.found_inf = torch.ones((), device="cuda")
    o2.step()
    del o2.found_inf
    for a, b in zip(before, _snapshot(o2, twins)):
        assert torch.equal(a, b)
    assert all(float(o2.state[q]["step"]) == 2.0 for q in twins)


def test_gradscaler_drives_fused_adamw():
    from pytorch_ddp_resnet_b200.utils.optim_util import get_optimizer
    torch.manual_seed(0)
    w1 = torch.nn.Parameter(torch.randn(64, 33, device="cuda"))
    w2 = torch.nn.Parameter(w1.detach().clone())
    o1 = get_optimizer("AdamW", torch.nn.ParameterList([w1]), dict(lr=1e-2))
    o2 = get_optimizer("AdamW", torch.nn.ParameterList([w2]), dict(lr=1e-2))
    scaler = torch.amp.GradScaler("cuda", init_scale=1024.0)
    for gv in [torch.randn_like(w1) for _ in range(3)]:
        o1.zero_grad(set_to_none=True)
        o2.zero_grad(set_to_none=True)
        (w1 * gv).sum().backward()
        o1.step()
        scaler.scale((w2 * gv).sum()).backward()
        scaler.step(o2)
        scaler.update()
    assert torch.equal(w1, w2)   # power-of-two scale: exact
    before = w2.detach().clone()
    o2.zero_grad(set_to_none=True)
    scaler.scale((w2 * torch.full_like(w2, float("inf"))).sum()).backward()
    scaler.step(o2)
    scaler.update()
    assert torch.equal(w2.detach(), before)
    assert float(o2.state[w2]["step"]) == 3.0
    assert scaler.get_scale() < 1024.0


# ---------------------------------------------------------------------------------------------------------
# 4. whole-step CUDA graph
# ---------------------------------------------------------------------------------------------------------
SPEC = "c3,32,3,1,1 r2 r2 n a ap16,1,0 fc64,10"


def _models(n, seed=0):
    from pytorch_ddp_resnet_b200.architectures.resnet import ResNet
    torch.manual_seed(seed)
    ms = [ResNet(SPEC, True, True, 0.0).cuda().train() for _ in range(n)]
    for m in ms[1:]:
        m.load_state_dict(ms[0].state_dict())
    return ms


def test_graph_replays_equal_eager_steps_bitwise():
    from pytorch_ddp_resnet_b200.algos.metrics import compute_losses_and_metrics
    from pytorch_ddp_resnet_b200.utils.graph_util import GraphedTrainStep
    from pytorch_ddp_resnet_b200.utils.optim_util import get_optimizer
    ops = _ops()
    g = torch.Generator().manual_seed(5)
    batches = [(torch.randn(16, 3, 32, 32, generator=g).cuda(), torch.randint(0, 10, (16,), generator=g).cuda())
               for _ in range(5)]
    m1, m2, m3 = _models(3)
    args = dict(lr=2e-3, weight_decay=5e-4, amsgrad=True)
    o1, o2 = get_optimizer("AdamW", m1, dict(args)), get_optimizer("AdamW", m2, dict(args))
    s1 = torch.optim.lr_scheduler.MultiStepLR(o1, milestones=[2], gamma=0.1)
    s2 = torch.optim.lr_scheduler.MultiStepLR(o2, milestones=[2], gamma=0.1)
    with ops.deterministic():
        l1 = []
        for x, y in batches:
            loss = compute_losses_and_metrics(logits=m1(x), labels=y)["loss"]
            loss.backward(); o1.step(); o1.zero_grad(set_to_none=True); s1.step()
            l1.append(loss.item())
        before = {k: v.clone() for k, v in m2.state_dict().items()}
        step = GraphedTrainStep(m2, o2, *batches[0])
        for k, v in m2.state_dict().items():
            assert torch.equal(v, before[k]), f"GraphedTrainStep construction changed {k}"
        assert all(float(t.abs().max()) == 0 for st in o2.state.values() for t in st.values())   # fresh state
        l2 = []
        for x, y in batches:
            l2.append(step(x, y)["loss"].item())
            s2.step()
        assert not step.eager_first
    assert l1 == l2, (l1, l2)
    for (k, a), (_, b) in zip(m1.state_dict().items(), m2.state_dict().items()):
        assert torch.equal(a, b), k
    for p, q in zip(m1.parameters(), m2.parameters()):
        st1, st2 = o1.state[p], o2.state[q]
        assert sorted(st1) == sorted(st2) == ["exp_avg", "exp_avg_sq", "max_exp_avg_sq", "step"]
        for k in st1:
            assert torch.equal(st1[k], st2[k]), k
        assert float(st2["step"]) == 5.0
    assert o2.param_groups[0]["lr"] == pytest.approx(2e-4)
    # the milestone took effect in the replays: the same five replays at the initial lr end elsewhere
    m4, = _models(1)
    o4 = get_optimizer("AdamW", m4, dict(args))
    with ops.deterministic():
        step4 = GraphedTrainStep(m4, o4, *batches[0])
        for x, y in batches:
            step4(x, y)
    assert any(not torch.equal(a, b) for a, b in zip(m2.parameters(), m4.parameters()))
    # one launch per step replaces the SGD launch: the same number of our kernels per replay
    o3 = get_optimizer("SGD", m3, dict(lr=0.1, momentum=0.9, dampening=0.0, nesterov=True, weight_decay=5e-4))
    with ops.deterministic():
        step3 = GraphedTrainStep(m3, o3, *batches[0])
    assert step.launches_per_step == step3.launches_per_step, (step.launches_per_step, step3.launches_per_step)


# ---------------------------------------------------------------------------------------------------------
# 5. kernel identity
# ---------------------------------------------------------------------------------------------------------
def test_one_step_is_one_adam_kernel():
    from pytorch_ddp_resnet_b200.utils.optim_util import FusedAdamW
    gen = torch.Generator(device="cuda").manual_seed(6)
    ps = _params(gen)
    opt = FusedAdamW(ps)
    for p in ps:
        p.grad = torch.randn_like(p)
    opt.step()   # creates the state (zero fills)
    _, names = kernels_launched(opt.step)
    assert names == ["adam_step_kernel"], names


# ---------------------------------------------------------------------------------------------------------
# 6. state_dict round trips with torch.optim
# ---------------------------------------------------------------------------------------------------------
def _train(opt, ps, grads):
    for gs in grads:
        for p, g in zip(ps, gs):
            p.grad = g.clone()
        opt.step()


def _compare_next_step(o_a, ps_a, o_b, ps_b, grad, hp, t):
    """One more step of both from equal state; every output within 4W of the other."""
    before = [(p.detach().clone(), {k: v.clone() for k, v in o_a.state[p].items()}) for p in ps_a]
    for p, q, g in zip(ps_a, ps_b, grad):
        p.grad, q.grad = g.clone(), g.clone()
    o_a.step()
    o_b.step()
    worst = 0.0
    for (p0, st0), p, q, g in zip(before, ps_a, ps_b, grad):
        bound = _reference(p0, g, st0["exp_avg"].to(p0.device), st0["exp_avg_sq"].to(p0.device), p0, t, hp,
                           lr_exact=False)
        worst = max(worst, _worst_ratio(p, q.detach().double(), bound["param"][1], 4.0))
        for k in ("exp_avg", "exp_avg_sq"):
            worst = max(worst, _worst_ratio(o_a.state[p][k], o_b.state[q][k].double(), bound[k][1], 4.0))
    return worst


@pytest.mark.parametrize("direction", ["fused_to_torch", "torch_to_fused"])
def test_state_dict_round_trip_with_torch_adamw(direction):
    from pytorch_ddp_resnet_b200.utils.optim_util import FusedAdamW
    gen = torch.Generator(device="cuda").manual_seed(7)
    ps = _params(gen)
    grads = [[torch.randn(p.shape, device="cuda", generator=gen) for p in ps] for _ in range(4)]
    twins = [torch.nn.Parameter(p.detach().clone()) for p in ps]
    hp = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01, decoupled=True, amsgrad=False)
    first_cls, second_cls = (FusedAdamW, torch.optim.AdamW) if direction == "fused_to_torch" \
        else (torch.optim.AdamW, FusedAdamW)
    kw = lambda cls: dict(foreach=False) if cls is torch.optim.AdamW else {}   # noqa: E731
    o1 = first_cls(ps, **kw(first_cls))
    _train(o1, ps, grads[:3])
    with torch.no_grad():
        for p, q in zip(ps, twins):
            q.copy_(p)
    o2 = second_cls(twins, **kw(second_cls))
    buf = io.BytesIO()   # through a file, as a checkpoint does (a state_dict holds the live state tensors)
    torch.save(o1.state_dict(), buf)
    buf.seek(0)
    o2.load_state_dict(torch.load(buf, map_location="cuda"))
    for p, q in zip(ps, twins):
        assert float(o2.state[q]["step"]) == 3.0
        if second_cls is FusedAdamW:
            assert o2.state[q]["step"].is_cuda and o2.state[q]["exp_avg"].stride() == q.stride()
    worst = _compare_next_step(o1, ps, o2, twins, grads[3], hp, 4)
    print(f"{direction}: worst ratio to 4W after the loaded step: {worst:.3f}")
    assert worst <= 0.5


def test_torch_1_10_state_dict_with_integer_step_loads():
    """torch 1.10 (the reference's pinned version) saves `step` as a Python int and, for a model that was NCHW
    there, the moments NCHW-contiguous; both load, and the next step matches torch's from the same state."""
    from pytorch_ddp_resnet_b200.utils.optim_util import FusedAdamW
    gen = torch.Generator(device="cuda").manual_seed(8)
    ps = _params(gen)
    twins = [torch.nn.Parameter(p.detach().clone()) for p in ps]
    state = {i: {"step": 7, "exp_avg": torch.randn(p.shape, generator=torch.Generator().manual_seed(i)) * 1e-2,
                 "exp_avg_sq": torch.rand(p.shape, generator=torch.Generator().manual_seed(100 + i)) * 1e-4}
             for i, p in enumerate(ps)}
    groups = [{"lr": 1e-3, "betas": (0.9, 0.999), "eps": 1e-8, "weight_decay": 0.01, "amsgrad": False,
               "params": list(range(len(ps)))}]
    sd = {"state": state, "param_groups": groups}
    o = FusedAdamW(ps)
    o.load_state_dict(sd)
    ref = torch.optim.AdamW(twins, foreach=False)
    ref.load_state_dict(sd)
    for p in ps:
        st = o.state[p]
        assert st["step"].is_cuda and st["step"].dtype == torch.float32 and float(st["step"]) == 7.0
        assert st["exp_avg"].is_cuda and st["exp_avg"].stride() == p.stride()
    grad = [torch.randn(p.shape, device="cuda", generator=gen) for p in ps]
    hp = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01, decoupled=True, amsgrad=False)
    worst = _compare_next_step(o, ps, ref, twins, grad, hp, 8)
    assert worst <= 0.5
    assert all(float(o.state[p]["step"]) == 8.0 for p in ps)


# ---------------------------------------------------------------------------------------------------------
# 7. end to end through script.py
# ---------------------------------------------------------------------------------------------------------
def test_script_adamw_graph_train_resume_eval(tmp_path):
    import yaml
    from tests.test_script_gpu import CONFIG
    cfg = dict(CONFIG, optimizer_cls_name="AdamW", optimizer_args={"lr": 2e-3, "weight_decay": 5e-4},
               master_port="12391", max_steps=20)
    run_dir = tmp_path / "models_dir" / "tiny"
    run_dir.mkdir(parents=True)
    (run_dir / "config.yaml").write_text(yaml.safe_dump(cfg, sort_keys=False))
    common = ["--models_dir", str(tmp_path / "models_dir"), "--run_name", "tiny", "--data_dir", str(tmp_path)]

    def run(args):
        env = dict(os.environ, PYTHONPATH=ROOT)
        return subprocess.run([sys.executable, os.path.join(ROOT, "script.py")] + args, cwd=tmp_path, env=env,
                              capture_output=True, text=True, timeout=600)

    def losses(out):
        return [float(l.split("loss:")[1]) for l in out.splitlines() if l.startswith("global step")]

    r = run(["--mode", "train"] + common)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    l1 = losses(r.stdout)
    assert len(l1) == 20 and all(l == l and l < 10.0 for l in l1), l1
    assert sum(l1[-5:]) < sum(l1[:5]), l1
    assert "optimizer_16.pth" in os.listdir(run_dir / "checkpoints")
    import torch as _t
    osd = _t.load(run_dir / "checkpoints" / "optimizer_16.pth", map_location="cpu")
    assert float(osd["state"][0]["step"]) == 16.0   # saved after the 16th step and "exp_avg_sq" in osd["state"][0]
    # resume from the newest checkpoint with a longer budget: Adam state and step counters come back
    cfg["max_steps"] = 30
    (run_dir / "config.yaml").write_text(yaml.safe_dump(cfg, sort_keys=False))
    r2 = run(["--mode", "train"] + common)
    assert r2.returncode == 0, r2.stdout[-2000:] + r2.stderr[-2000:]
    assert "Loaded classifier checkpoint" in r2.stdout
    l2 = losses(r2.stdout)
    assert l2 and all(l == l and l < 10.0 for l in l2), l2
    assert sum(l2[-5:]) / 5 < sum(l1[:5]) / 5, (l1, l2)
    r3 = run(["--mode", "eval"] + common)
    assert r3.returncode == 0, r3.stderr[-2000:]
    assert "Test metrics:" in r3.stdout


# ---------------------------------------------------------------------------------------------------------
# 8. two ranks
# ---------------------------------------------------------------------------------------------------------
def _ddp_worker(rank, world, port):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    from pytorch_ddp_resnet_b200.utils.ddp_util import prepare_env_for_graphs, wrap_ddp
    prepare_env_for_graphs()
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from pytorch_ddp_resnet_b200.architectures.resnet import ResNet
    from pytorch_ddp_resnet_b200.utils.graph_util import GraphedTrainStep
    from pytorch_ddp_resnet_b200.utils.optim_util import get_optimizer
    torch.manual_seed(0)
    model = ResNet(SPEC, True, True, 0.0).cuda()
    ddp = wrap_ddp(model, torch.device("cuda", rank))
    g = torch.Generator().manual_seed(100 + rank)   # different data per rank
    x = torch.randn(8, 3, 32, 32, generator=g).cuda()
    y = torch.randint(0, 10, (8,), generator=g).cuda()
    opt = get_optimizer("AdamW", ddp, dict(lr=2e-3, weight_decay=5e-4))
    step = GraphedTrainStep(ddp, opt, x, y, bucket_bytes=64 << 10)
    for _ in range(3):
        step(x, y)
    torch.cuda.synchronize()
    for n, p in model.named_parameters():
        ref = p.detach().clone()
        dist.broadcast(ref, 0)
        assert torch.equal(ref, p.detach()), f"replicas diverged at {n}"
        assert float(opt.state[p]["step"]) == 3.0
        for k in ("exp_avg", "exp_avg_sq"):
            buf = opt.state[p][k].clone()
            dist.broadcast(buf, 0)
            assert torch.equal(buf, opt.state[p][k]), f"optimizer state diverged at {n}.{k}"
    step.close()
    dist.barrier()
    dist.destroy_process_group()


def test_ddp_two_ranks_graphed_adamw():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    mp.spawn(_ddp_worker, args=(2, 29500 + os.getpid() % 1000 + 13), nprocs=2, join=True)
