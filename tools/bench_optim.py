"""Optimizer step timing on the WRN-28-10 parameter set (36.5 M fp32 parameters, ~1 GB per Adam step, larger than
the 126 MB L2), after warm-up, arms alternated in blocks of 50 steps:

  * the optimizer step alone: FusedAdamW, torch.optim.AdamW(fused=True), torch.optim.AdamW(foreach=True) and
    FusedSGD (momentum, nesterov, weight decay) as the anchor. An eager step() is bound by its Python host code
    (hundreds of microseconds), so two numbers per arm: the device time of the kernels one step launches
    (torch.profiler, summed per block) with the achieved bytes/s it implies, counting the algorithmic traffic
    (AdamW 28 B / parameter, SGD 20 B) against 7.7 TB/s; and the wall time of back-to-back eager steps (CUDA
    events);
  * the whole captured training step (GraphedTrainStep, WRN-28-10, batch 128): FusedAdamW against FusedSGD.

The GPU's name and power limit are read in the same run. Writes one JSON line to OUT/bench_optim.json.

    python tools/bench_optim.py --out DIR [--opt-steps 400] [--train-steps 400]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SPEC = "c3,160,3,1,1 r4 r4 r4 n a ap8,1,0 fc640,10"   # WRN-28-10
SGD = dict(lr=0.1, momentum=0.9, dampening=0.0, nesterov=True, weight_decay=5e-4)
ADAMW = dict(lr=1e-3, weight_decay=5e-4)
HBM_BPS = 7.7e12
BLOCK = 50   # steps per timed block; the arms take turns block by block


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit",
                        "--format=csv,noheader"], capture_output=True, text=True, check=True).stdout.strip()
    name, power = [s.strip() for s in q.split(",")]
    return {"gpu": name, "power_limit": power}


def _model():
    from pytorch_ddp_resnet_b200.architectures.resnet import ResNet
    torch.manual_seed(0)
    return ResNet(SPEC, True, True, 0.0).cuda().train()


def _time_alternating(arms, steps):
    """arms: {name: fn() doing one step}. Blocks of BLOCK steps, arms in turn, until each has `steps`.
    Returns {name: ms per step} from CUDA events around each block."""
    total = {k: 0.0 for k in arms}
    done = {k: 0 for k in arms}
    while min(done.values()) < steps:
        for name, fn in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(BLOCK):
                fn()
            e1.record()
            e1.synchronize()
            total[name] += e0.elapsed_time(e1)
            done[name] += BLOCK
    return {k: total[k] / done[k] for k in arms}


def _kernel_time_alternating(arms, steps):
    """Like _time_alternating, but sums the device durations of the CUDA kernels each block launched
    (torch.profiler, one session per block; copies and memsets are not counted). Returns {name: ms per step}."""
    from torch.profiler import ProfilerActivity, profile
    total = {k: 0.0 for k in arms}
    done = {k: 0 for k in arms}
    while min(done.values()) < steps:
        for name, fn in arms.items():
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(BLOCK):
                    fn()
                torch.cuda.synchronize()
            us = sum(e.time_range.elapsed_us() for e in prof.events()
                     if e.device_type == torch.autograd.DeviceType.CUDA
                     and not e.name.startswith(("Memset", "Memcpy", "[memory]")))
            total[name] += us * 1e-3
            done[name] += BLOCK
    return {k: total[k] / done[k] for k in arms}


def bench_optimizer_step(steps):
    from pytorch_ddp_resnet_b200.utils.optim_util import FusedAdamW, FusedSGD
    n_params = sum(p.numel() for p in _model().parameters())
    makers = {
        "FusedAdamW": (lambda ps: FusedAdamW(ps, **ADAMW), 28),
        "torch.AdamW(fused=True)": (lambda ps: torch.optim.AdamW(ps, fused=True, **ADAMW), 28),
        "torch.AdamW(foreach=True)": (lambda ps: torch.optim.AdamW(ps, foreach=True, **ADAMW), 28),
        "FusedSGD": (lambda ps: FusedSGD(ps, **SGD), 20),
    }
    arms, bytes_per_param = {}, {}
    torch.manual_seed(1)
    for name, (make, bpp) in makers.items():
        ps = list(_model().parameters())
        for p in ps:
            p.grad = torch.randn_like(p) * 1e-2   # the parameter's layout (channels_last filters)
        opt = make(ps)
        for _ in range(20):   # warm-up: state, tables, algorithm selection
            opt.step()
        arms[name] = opt.step
        bytes_per_param[name] = bpp
    torch.cuda.synchronize()
    kernel_ms = _kernel_time_alternating(arms, steps)
    wall_ms = _time_alternating(arms, steps)
    out = {}
    for name, t in kernel_ms.items():
        bps = bytes_per_param[name] * n_params / (t * 1e-3)
        out[name] = {"kernel_ms_per_step": round(t, 4), "bytes_per_param": bytes_per_param[name],
                     "TBps": round(bps / 1e12, 3), "share_of_7.7TBps": round(bps / HBM_BPS, 3),
                     "eager_wall_ms_per_step": round(wall_ms[name], 4)}
    return n_params, out


def bench_train_step(steps):
    from pytorch_ddp_resnet_b200.utils.graph_util import GraphedTrainStep
    from pytorch_ddp_resnet_b200.utils.optim_util import get_optimizer
    g = torch.Generator().manual_seed(2)
    x = torch.randn(128, 3, 32, 32, generator=g).cuda()
    y = torch.randint(0, 10, (128,), generator=g).cuda()
    arms = {}
    for name, args in (("AdamW", ADAMW), ("SGD", SGD)):
        model = _model()
        opt = get_optimizer(name, model, dict(args))
        step = GraphedTrainStep(model, opt, x, y)
        for _ in range(20):
            step(x, y)
        arms[name] = (lambda s: (lambda: s(x, y)))(step)
    torch.cuda.synchronize()
    return {k: round(v, 4) for k, v in _time_alternating(arms, steps).items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for bench_optim.json")
    ap.add_argument("--opt-steps", type=int, default=400)
    ap.add_argument("--train-steps", type=int, default=400)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_optim.py needs a CUDA device")
    info = gpu_info()
    n_params, opt_ms = bench_optimizer_step(a.opt_steps)
    train_ms = bench_train_step(a.train_steps)
    rec = dict(info, n_params=n_params, optimizer_step=opt_ms, optimizer_steps_per_arm=a.opt_steps,
               train_step_ms=train_ms, train_steps_per_arm=a.train_steps, batch=128, model="WRN-28-10",
               timing="after warm-up, arms alternated in blocks of %d steps; optimizer kernel time from "
                      "torch.profiler, wall times from CUDA events" % BLOCK)
    os.makedirs(a.out, exist_ok=True)
    line = json.dumps(rec)
    with open(os.path.join(a.out, "bench_optim.json"), "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
