#!/usr/bin/env python
"""
bench.py — train img/s of WRN-28-10 (dropout 0.3) on CIFAR-shaped synthetic data, batch 128 per GPU,
bf16, N GPUs of one node (BASELINE.json configs[1]; N > 1 is the DDP weak-scaling run of configs[4],
100 classes). `--config` selects the other BASELINE configs (ResNet-v1-20, ResNet-v2-164, WRN-50-2-like
ImageNet shape); they are parity cases first and secondary bench lines.

    python bench.py --gpus 1 --steps 30 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the UNMODIFIED reference (oracle/_ref) on the host CPU cores
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # + what the last timed step computed

One "step" = forward + mean cross-entropy + backward (+ the bucketed NCCL gradient all-reduce of the
data-parallel ranks, overlapped with backward inside the captured graph) + fused SGD update, through the
public API of pytorch_ddp_resnet_b200 (GraphedTrainStep).
`value`     : images/s with the batch already resident in HBM, CUDA-event timed, max over ranks, over
              exactly --steps steps.
`sustained` : the same measurement over >= 300 further steps (steady state under the power cap).
`e2e`       : the same step fed from pinned host memory (H2D copy of x, y every step) with a device->host
              read of the loss every step, inside the timed region.
`exposed_comm_ms` (N > 1): step time minus the step time of the SAME captured kernels with the collectives
              left out (SURVEY 8d protocol).
`roofline`  : the dominant kernel (tcgen05 implicit-GEMM conv, fprop of the 160->160 3x3 @32x32 layer that
              carries 34.6 % of the FLOPs) timed alone with CUDA events, against the measured bf16 peak in
              MEASURED_PEAKS.json; `traffic` comes from the committed ncu capture under profiles/.
`cpu_baseline`: the unmodified reference's own training_loop (oracle/_ref, kind "reference"; the oracle port
              if oracle/_ref is absent) timed on the box's host cores on a bounded sample.
`gpu_reference`: the unmodified reference modules on the SAME GPU through torch + cuDNN: bf16 autocast and the
              reference's literal default (fp16 autocast + GradScaler), batch 128 — the bar to beat.

--dump-outputs DIR (rank 0): after the --steps timed steps, what the last of them handed back: its metrics
(loss.npy, top1_err.npy, top5_err.npy) and the model state it left (state.<state_dict key>.npy: parameters and
BatchNorm buffers), float32 (integer buffers float64). Model init, batches and dropout seeds are fixed, and the
run uses the deterministic mode (B200_DETERMINISTIC=1: fixed-order reductions), so two runs with the same
arguments write the same arrays and two builds can be compared array for array. The default kernels reduce
with fp32 atomics: every step differs from run to run in the last bits and training amplifies that (35
WRN-28-10 steps at lr 0.1: losses 0.62 and 0.59). The numbers of such a run are those of the deterministic mode
(WRN-28-10, batch 128, one B200 at a 1000 W power limit: 5.21 instead of 4.73 ms/step); time without the flag.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
REF_DIR = os.path.join(ROOT, "oracle", "_ref")

SGD = dict(lr=0.1, momentum=0.9, dampening=0.0, nesterov=True, weight_decay=5e-4)


def sgd_args(cfg):
    """The reference recipe's SGD arguments; a config may carry its own learning rate (the ImageNet-shape net
    diverges at 0.1 on random labels in BOTH implementations: profiles/r02_imagenet_loss_trajectory.txt)."""
    a = dict(SGD)
    a["lr"] = cfg.get("lr", a["lr"])
    return a
METRIC = "train img/s WRN-28-10 CIFAR"

# BASELINE.json configs (SURVEY 8d, App. A). `classes_multi`: head used when N > 1 (config 5: CIFAR-100)
CONFIGS = {
    "wrn28": dict(spec="c3,160,3,1,1 r4 r4 r4 n a ap8,1,0 fc640,{classes}", preact=True, use_proj=True,
                  dropout=0.3, hw=32, batch=128, classes=10, classes_multi=100, metric=METRIC,
                  workload="WRN-28-10 (dropout 0.3) CIFAR-{classes}-shape 32x32 synthetic bf16 training, "
                           "batch 128/GPU"),
    "resnet20": dict(spec="c3,16,3,1,1 n a r3 r3 r3 ap8,1,0 fc64,{classes}", preact=False, use_proj=False,
                     dropout=0.0, hw=32, batch=128, classes=10, classes_multi=10,
                     metric="train img/s ResNet-v1-20 CIFAR",
                     workload="ResNet-v1-20 CIFAR-10-shape 32x32 synthetic bf16 training, batch 128/GPU"),
    "v2-164": dict(spec="c3,64,3,1,1 b18 b18 b18 n a ap8,1,0 fc256,{classes}", preact=True, use_proj=True,
                   dropout=0.0, hw=32, batch=128, classes=10, classes_multi=10,
                   metric="train img/s ResNet-v2-164 CIFAR",
                   workload="ResNet-v2-164 preact-bottleneck CIFAR-10-shape 32x32 synthetic bf16 training, "
                            "batch 128/GPU"),
    "wrn50-imagenet": dict(spec="c3,512,7,2,3 n a mp3,2,1 b3 b4 b6 b3 ap7,1,0 fc4096,{classes}", preact=False,
                           use_proj=True, dropout=0.0, hw=224, batch=256, classes=1000, classes_multi=1000, lr=0.005,
                           metric="train img/s WRN-50-2-like ImageNet",
                           workload="WRN-50-2-like bottleneck ImageNet-shape 224x224 synthetic bf16 training, "
                                    "batch 256/GPU (the true WRN-50-2 is not expressible in the reference's "
                                    "grammar, SURVEY Q7)"),
}


def resolve_config(name: str, world: int):
    c = dict(CONFIGS[name])
    c["classes"] = c["classes_multi"] if world > 1 else c["classes"]
    c["spec"] = c["spec"].format(classes=c["classes"])
    c["workload"] = c["workload"].format(classes=c["classes"])
    c["name"] = name
    return c


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(bf16=p.get("bf16_tflops", 1590.0), bf16_sustained=p.get("bf16_tflops_sustained", 1400.0),
                    hbm=p.get("hbm_gbs", 6650.0), source="measured (MEASURED_PEAKS.json)")
    return dict(bf16=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


# --------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi in the background during the timed regions)
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,utilization.gpu,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int, period_ms: int = 20):
        self.proc, self.lines, self.gpu, self.period = None, [], gpu_index, period_ms
        self.marks = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", str(self.period)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def mark(self):
        """Start / end of a timed region (host clock; the region is bracketed by device syncs)."""
        self.marks.append(time.perf_counter())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(2.5 * self.period / 1e3)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        windows = list(zip(self.marks[0::2], self.marks[1::2]))
        sm, mx, power, reasons = [], None, [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        total = 0
        for t, ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 8:
                continue
            total += 1
            try:
                clk, mxv, util = float(parts[0]), float(parts[1]), float(parts[2])
            except ValueError:
                continue
            mx = mxv
            # a sample is "under load" when it was printed inside a timed window (+ one period of slack)
            if not any(a <= t <= b + 2 * self.period / 1e3 for a, b in windows):
                continue
            sm.append(clk)
            try:
                power.append(float(parts[3]))
            except ValueError:
                pass
            for n, v in zip(names, parts[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None,
                "sm_max_mhz": mx, "power_w_max": max(power) if power else None, "reasons": sorted(reasons),
                "samples": len(sm), "samples_total": total, "period_ms": self.period}


# --------------------------------------------------------------------------------------------------
# the reference itself (oracle/_ref): CPU arm, cpu_baseline, gpu_reference
# --------------------------------------------------------------------------------------------------
def use_all_host_threads() -> int:
    """torchrun exports OMP_NUM_THREADS=1; the CPU arms use every core the process may run on."""
    import torch
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    torch.set_num_threads(max(1, n))
    return torch.get_num_threads()


def have_ref() -> bool:
    return os.path.exists(os.path.join(REF_DIR, "resnet", "algos", "training.py"))


class _TimedLoader:
    """A dataloader of `n` synthetic batches that records when each batch is requested: the interval between
    the request of batch w and the request after batch w+k-1 (or StopIteration) is exactly k loop bodies of
    the reference's training_loop (training.py:92-144). On CUDA the boundaries are device-synchronised."""

    def __init__(self, batches, sync):
        self.batches, self.sync, self.t = batches, sync, []

    def __iter__(self):
        for b in self.batches:
            self.sync()
            self.t.append(time.perf_counter())
            yield b
        self.sync()
        self.t.append(time.perf_counter())

    def __len__(self):
        return len(self.batches)


class _Sampler:
    def set_epoch(self, e):
        pass


def reference_training_loop(cfg, device: str, steps: int, warmup: int, mode: str):
    """Runs the UNMODIFIED reference training_loop from oracle/_ref on synthetic batches and returns
    (img/s, seconds per step) over `steps` optimisation steps after `warmup`.
    mode: 'fp32' (scaler None: the reference's CPU / non-AMP path), 'fp16' (its literal GPU default:
    tc.cuda.amp.autocast() + GradScaler, script.py:63, training.py:95) or 'bf16' (the same code with
    autocast's dtype patched to bfloat16, SURVEY Q1)."""
    import contextlib
    import io
    import torch
    import torch.distributed as dist
    sys.path.insert(0, REF_DIR)
    from resnet.algos import training as ref_training
    from resnet.architectures.resnet import ResNet as RefResNet
    from resnet.utils.checkpoint_util import FrequencyCheckpointStrategy
    from resnet.utils.optim_util import get_optimizer as ref_get_optimizer

    own_pg = not dist.is_initialized()
    if own_pg:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", str(29700 + os.getpid() % 200))
        dist.init_process_group("nccl" if device.startswith("cuda") else "gloo", rank=0, world_size=1)
    torch.manual_seed(0)
    model = RefResNet(architecture_spec=cfg["spec"], preact=cfg["preact"], use_proj=cfg["use_proj"],
                      dropout_prob=cfg["dropout"]).to(device)
    opt = ref_get_optimizer("SGD", model, sgd_args(cfg))
    g = torch.Generator().manual_seed(1234)
    n = warmup + steps
    B, hw = cfg["batch"], cfg["hw"]
    batches = [(torch.randn(B, 3, hw, hw, generator=g), torch.randint(0, cfg["classes"], (B,), generator=g))
               for _ in range(min(n, 4))]
    batches = [batches[i % len(batches)] for i in range(n)]
    sync = torch.cuda.synchronize if device.startswith("cuda") else (lambda: None)
    dl = _TimedLoader(batches, sync)
    dl_test = [(batches[0][0][:2], batches[0][1][:2])]
    scaler = None
    patched = None
    if mode in ("fp16", "bf16"):
        scaler = torch.amp.GradScaler("cuda", enabled=(mode == "fp16"))
        if mode == "bf16":
            patched = ref_training.tc.cuda.amp.autocast
            ref_training.tc.cuda.amp.autocast = lambda: torch.autocast("cuda", dtype=torch.bfloat16)
    strat = FrequencyCheckpointStrategy(unit="batch", frequency=10 ** 9)
    tmp = tempfile.mkdtemp(prefix="b200_ref_")
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            ref_training.training_loop(
                rank=0, world_size=1, device=device, sampler_train=_Sampler(), sampler_test=_Sampler(),
                dl_train=dl, dl_test=dl_test, classifier=model, optimizer=opt, scaler=scaler, scheduler=None,
                scheduler_step_unit="none", checkpoint_strategy=strat, checkpoint_dir=os.path.join(tmp, "ck"),
                num_microbatches=1, global_step=0, max_steps=n, log_dir=os.path.join(tmp, "tb"))
    finally:
        if patched is not None:
            ref_training.tc.cuda.amp.autocast = patched
        if own_pg:
            dist.destroy_process_group()
    dt = dl.t[warmup + steps] - dl.t[warmup] if len(dl.t) > warmup + steps else dl.t[-1] - dl.t[warmup]
    return B * steps / dt, dt / steps


def port_steps(cfg, batch: int, steps: int, warmup: int):
    """Fallback when oracle/_ref is absent: the oracle's restatement of the same step (kind 'port')."""
    import torch
    from oracle import resnet_oracle as O
    state = O.init_state(cfg["spec"], cfg["preact"], cfg["use_proj"], seed=0)
    bufs = {}
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(batch, 3, cfg["hw"], cfg["hw"], generator=g)
    y = torch.randint(0, cfg["classes"], (batch,), generator=g)
    for _ in range(warmup):
        O.train_step(state, bufs, x, y, cfg["spec"], cfg["preact"], cfg["use_proj"], cfg["dropout"], sgd_args(cfg))
    t0 = time.perf_counter()
    for _ in range(steps):
        O.train_step(state, bufs, x, y, cfg["spec"], cfg["preact"], cfg["use_proj"], cfg["dropout"], sgd_args(cfg))
    dt = time.perf_counter() - t0
    return batch * steps / dt, dt / steps


def cpu_reference(cfg, steps: int, warmup: int):
    """(img/s, s/step, kind, sample, cores) of the reference's CPU path on a bounded sample."""
    cores = use_all_host_threads()
    if have_ref():
        ips, sps = reference_training_loop(cfg, "cpu", steps, warmup, "fp32")
        kind = "reference"
        what = "the unmodified reference training_loop (oracle/_ref)"
    else:
        c = dict(cfg, batch=min(cfg["batch"], 16))
        ips, sps = port_steps(c, c["batch"], steps, warmup)
        cfg = c
        kind = "port"
        what = "the oracle port (oracle/_ref not built)"
    sample = (f"{steps} steps (+{warmup} warm-up) of batch {cfg['batch']} of the same workload through {what}, "
              f"fp32, {cores} threads")
    return ips, sps, kind, sample, cores


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = resolve_config(args.config, 1 if args.gpus <= 1 else args.gpus)
    heavy = cfg["name"] in ("wrn28", "wrn50-imagenet")
    steps = max(1, min(args.steps, 3 if heavy else 20))
    warm = 1 if heavy else max(1, min(args.warmup, 3))
    if cfg["name"] == "wrn50-imagenet":
        cfg["batch"] = 16   # a 256-image ImageNet-shape fp32 step takes minutes on the host cores
    ips, sps, kind, sample, cores = cpu_reference(cfg, steps, warm)
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": ips, "unit": "img/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": sps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["workload"], "sample": sample},
        "cpu_baseline": {"value": ips, "unit": "img/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": ips, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
def time_dominant_kernel(torch, ops, _lib, iters=30):
    """Average duration of the dominant kernel launch (conv fprop 160->160 3x3 @32x32, batch 128),
    CUDA events on the launching stream, rotating inputs whose total footprint exceeds L2."""
    N, H, W, C, K = 128, 32, 32, 160, 160
    nb = 6  # 6 x (42 MB in + 42 MB out) > 126 MB L2
    xs = [torch.randn(N, H, W, C, device="cuda").bfloat16() for _ in range(nb)]
    w = (torch.randn(K, 3, 3, C, device="cuda") * 0.02).bfloat16()
    for i in range(3):
        ops.conv_fprop(xs[i % nb], w, 1, 1, algo=_lib.ALGO_TC)
    # capture the launches in a CUDA graph so that host launch latency is not part of the number
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.conv_fprop(xs[0], w, 1, 1, algo=_lib.ALGO_TC)
        with torch.cuda.graph(g, stream=s):
            for i in range(iters):
                ops.conv_fprop(xs[i % nb], w, 1, 1, algo=_lib.ALGO_TC)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g.replay()
    torch.cuda.synchronize()
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    flops = 2.0 * N * H * W * K * C * 9
    return ms, flops


def ncu_record():
    """DRAM traffic / tensor-pipe activity of the dominant kernel from the committed `ncu --set full`
    capture of this round (profiles/dominant_kernel_ncu.json, written by tools/ncu_to_json.py)."""
    path = os.path.join(ROOT, "profiles", "dominant_kernel_ncu.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return None


DUMP_MAX_BYTES = 64 << 20
DUMP_SAMPLE = 1 << 18   # elements kept of a larger tensor (46.7 MB in all for the largest config, wrn50-imagenet)


def dump_outputs(out_dir, metrics, model):
    """Writes the metrics of a step and the model state after it as <out_dir>/<name>.npy. A tensor of more than
    DUMP_SAMPLE elements is reduced to a fixed, seeded sample of its flattened elements (logical order, so the
    memory layout of a build does not move the sample); other tensors keep their shape."""
    import numpy as np
    import torch
    arrays = dict(metrics)
    arrays.update({"state." + k: v for k, v in model.state_dict().items()})
    for name, t in arrays.items():
        t = t.detach()
        t = t.float() if t.is_floating_point() else t.double()
        if t.numel() > DUMP_SAMPLE:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        arrays[name] = t.cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES >> 20} MB limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from pytorch_ddp_resnet_b200 import _lib, ops
    from pytorch_ddp_resnet_b200.algos.metrics import compute_losses_and_metrics
    from pytorch_ddp_resnet_b200.architectures.resnet import ResNet
    from pytorch_ddp_resnet_b200.utils.optim_util import get_optimizer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    cfg = resolve_config(args.config, world)
    B, hw = cfg["batch"], cfg["hw"]
    if world > 1:
        from pytorch_ddp_resnet_b200.utils.ddp_util import prepare_env_for_graphs, wrap_ddp
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        prepare_env_for_graphs()
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)
    _lib.load()

    torch.manual_seed(0)
    model = ResNet(cfg["spec"], cfg["preact"], cfg["use_proj"], cfg["dropout"]).to(device).train()
    classifier = wrap_ddp(model, device) if world > 1 else model
    opt = get_optimizer("SGD", classifier, sgd_args(cfg))

    gen = torch.Generator().manual_seed(1234 + rank)
    nbuf = 4
    xs_host = [torch.randn(B, 3, hw, hw, generator=gen).pin_memory() for _ in range(nbuf)]
    ys_host = [torch.randint(0, cfg["classes"], (B,), generator=gen).pin_memory() for _ in range(nbuf)]
    xs_dev = [x.to(device) for x in xs_host]
    ys_dev = [y.to(device) for y in ys_host]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)

    def timed(run_steps, fn, mark=False):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        if mark:
            sampler.mark()
        e0.record()
        for i in range(run_steps):
            fn(i)
        e1.record()
        barrier()
        if mark:
            sampler.mark()
        ms = torch.tensor([e0.elapsed_time(e1)], device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    launches_per_step = None
    noexch_ms = None
    if args.eager:
        def step(x, y):
            m = compute_losses_and_metrics(logits=classifier(x), labels=y)
            m["loss"].backward()
            opt.step()
            opt.zero_grad(set_to_none=True)
            return m
    else:
        # public API: whole-step CUDA graph (pytorch_ddp_resnet_b200.utils.graph_util.GraphedTrainStep)
        from pytorch_ddp_resnet_b200.utils.graph_util import GraphedTrainStep
        if world > 1:
            # the same captured kernels WITHOUT the collectives: the difference is the exposed communication
            g0 = GraphedTrainStep(classifier, opt, xs_dev[0], ys_dev[0], exchange=False)
            for i in range(args.warmup):
                g0(xs_dev[i % nbuf], ys_dev[i % nbuf])
            noexch_ms = timed(args.steps, lambda i: g0(xs_dev[i % nbuf], ys_dev[i % nbuf])) / args.steps
            g0.reducer.detach()
            del g0
        graphed = GraphedTrainStep(classifier, opt, xs_dev[0], ys_dev[0])
        launches_per_step = graphed.launches_per_step

        def step(x, y):
            return graphed(x, y)

    # ---- device-resident run ---------------------------------------------------------------------
    for i in range(args.warmup):
        step(xs_dev[i % nbuf], ys_dev[i % nbuf])
    if rank == 0:
        sampler.start()
        time.sleep(0.2)
    last = {}

    def resident_step(i):
        last["metrics"] = step(xs_dev[i % nbuf], ys_dev[i % nbuf])

    l0 = _lib.launch_count()
    total_ms = timed(args.steps, resident_step, mark=True)
    launches = _lib.launch_count() - l0
    if args.dump_outputs and rank == 0:   # before later steps overwrite the graph's output buffers
        dump_outputs(args.dump_outputs, last["metrics"], model)
    if launches_per_step is not None:  # replays do not pass through the C ABI: kernels captured per step
        launches = launches_per_step * args.steps
    ms_per_step = total_ms / args.steps
    value = B * world * args.steps / (total_ms / 1e3)

    # ---- steady state: >= 300 further steps (the part settles under its power cap) ----------------
    sus_steps = max(args.sustained, 0)
    sustained = None
    if sus_steps:
        sus_ms = timed(sus_steps, lambda i: step(xs_dev[i % nbuf], ys_dev[i % nbuf]), mark=True)
        sustained = {"steps": sus_steps, "ms_per_step": sus_ms / sus_steps,
                     "value": B * world * sus_steps / (sus_ms / 1e3), "unit": "img/s"}
    clocks = sampler.stop() if rank == 0 else None

    # ---- end to end: pinned host batch -> H2D, step, loss -> host, every step --------------------
    loss_host = [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(nbuf)]

    def e2e_step(i):
        if args.eager:
            x = xs_host[i % nbuf].to(device, non_blocking=True)
            y = ys_host[i % nbuf].to(device, non_blocking=True)
        else:  # GraphedTrainStep copies the pinned host batch into its static device buffers
            x, y = xs_host[i % nbuf], ys_host[i % nbuf]
        loss = step(x, y)["loss"]
        loss_host[i % nbuf].copy_(loss.detach().float(), non_blocking=True)

    for i in range(min(3, args.warmup)):
        e2e_step(i)
    e2e_ms = timed(args.steps, e2e_step)
    e2e_value = B * world * args.steps / (e2e_ms / 1e3)
    last_loss = float(loss_host[(args.steps - 1) % nbuf].item())
    h2d = xs_host[0].numel() * 4 + ys_host[0].numel() * 8
    d2h = 4

    def leave():
        """Multi-rank exit: release the graphs that hold NCCL kernels, meet at a barrier, and leave without
        the process-group destructor (it was seen to hang once captured collectives exist)."""
        if world == 1:
            return
        if not args.eager:
            graphed.close()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)

    if rank != 0:
        leave()
        return

    # ---- roofline + tensor-pipe utilisation (rank 0) ------------------------------------------------
    pk = peaks()
    from oracle import resnet_oracle as O
    _, train_flops = O.conv_train_flops(cfg["spec"], cfg["preact"], cfg["use_proj"], B, hw)
    conv_tflops_in_step = train_flops / (ms_per_step * 1e-3) / 1e12
    line = {
        "metric": cfg["metric"], "value": value, "unit": "img/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": cfg["workload"], "name": cfg["name"], "global_batch": B * world,
                   "deterministic": ops.is_deterministic(),
                   "parallelism": f"dp{world}",
                   "l2": "per-step working set (GBs of saved activations) is far larger than the 126 MB L2; "
                         "4 rotating input batches"},
        "e2e": {"value": e2e_value, "unit": "img/s", "h2d_bytes_per_step": h2d * world,
                "d2h_bytes_per_step": d2h * world, "ms_per_step": e2e_ms / args.steps, "last_loss": last_loss},
        "gpu_launches": launches,
        "clocks": clocks,
    }
    if sustained:
        line["sustained"] = sustained
    if noexch_ms is not None:
        line["exposed_comm_ms"] = ms_per_step - noexch_ms
        line["ms_per_step_without_collectives"] = noexch_ms
    if cfg["name"] == "wrn28":
        kms, kflops = time_dominant_kernel(torch, ops, _lib)
        achieved = kflops / (kms * 1e-3) / 1e12
        rec = ncu_record()
        line["roofline"] = {
            "bound": "tensor", "achieved": achieved, "peak": pk["bf16"], "unit": "TFLOP/s",
            "frac": achieved / pk["bf16"],
            "traffic": rec.get("dram_bytes_per_launch") if rec else None,
            "traffic_source": (rec.get("source") if rec else "no ncu capture committed for this build"),
            "algorithmic_bytes": 84.3e6,
            "kernel": "conv_tc2h_kernel (cta_group::2, halo reuse) fprop 3x3 s1 160->160 @32x32 batch 128 "
                      "(60.4 GFLOP/launch)",
            "kernel_ms": kms, "peak_source": pk["source"] + ", burst figure (kernel timed alone)"}
        line["tensor_pipe_util"] = {
            "dominant_kernel_of_measured_burst_peak": achieved / pk["bf16"],
            "dominant_kernel_of_nominal_2250": achieved / 2250.0,
            "whole_step_conv_tflops": conv_tflops_in_step,
            "whole_step_of_measured_sustained_peak": conv_tflops_in_step / pk["bf16_sustained"],
            "whole_step_of_nominal_2250": conv_tflops_in_step / 2250.0,
            "ncu_pipe_tensor_cycles_active_pct": rec.get("pipe_tensor_cycles_active_pct") if rec else None}
    elif cfg["name"] == "wrn50-imagenet":
        line["roofline"] = {"bound": "tensor", "achieved": conv_tflops_in_step, "peak": pk["bf16_sustained"],
                            "unit": "TFLOP/s", "frac": conv_tflops_in_step / pk["bf16_sustained"], "traffic": None,
                            "kernel": "whole step: conv FLOPs (fprop + dgrad + wgrad) / step time",
                            "peak_source": pk["source"] + ", sustained figure (inside a long step)"}
    else:
        # C <= 64 everywhere: every kernel of these nets is HBM / latency bound (SURVEY 8d); algorithmic bytes =
        # BN-family traffic (16 B per BN input element) + conv activations read + written once per pass
        bn_elems = {"resnet20": 24.1e6, "v2-164": 409.5e6}[cfg["name"]]
        abytes = bn_elems * (16 + 12)
        ach = abytes / (ms_per_step * 1e-3) / 1e9
        line["roofline"] = {"bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s",
                            "frac": ach / pk["hbm"], "traffic": None,
                            "kernel": "whole step: 28 algorithmic bytes per BN-input element (BN family 16 B + "
                                      "conv fprop/dgrad/wgrad activation reads and writes 12 B) / step time",
                            "peak_source": pk["source"]}
    if world == 1 and not args.no_cpu_baseline:
        heavy = cfg["name"] in ("wrn28", "wrn50-imagenet")
        c = dict(cfg)
        if cfg["name"] == "wrn50-imagenet":
            c["batch"] = 16
        ips, _, kind, sample, cores = cpu_reference(c, 2 if heavy else 10, 1)
        line["cpu_baseline"] = {"value": ips, "unit": "img/s", "cores": cores, "kind": kind, "sample": sample}
    if world == 1 and not args.no_gpu_reference and have_ref():
        ref = {}
        for mode in ("bf16", "fp16"):
            try:
                ips, sps = reference_training_loop(cfg, f"cuda:{local_rank}", max(10, min(args.steps, 30)), 5, mode)
                ref[mode] = {"value": ips, "unit": "img/s", "ms_per_step": sps * 1e3}
            except Exception as e:  # the bar is informative; never lose our own line over it
                ref[mode] = {"error": f"{type(e).__name__}: {e}"[:200]}
            torch.cuda.empty_cache()
        ref["what"] = ("the unmodified reference (oracle/_ref: resnet.architectures.resnet.ResNet through "
                       "resnet.algos.training.training_loop) on the same GPU with torch + cuDNN, same batch, "
                       "synthetic batches resident in host memory as its loop expects; bf16 = its autocast "
                       "patched to bfloat16, fp16 = its literal default (autocast + GradScaler)")
        line["gpu_reference"] = ref
    print(json.dumps(line), flush=True)
    leave()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--config", choices=sorted(CONFIGS), default="wrn28")
    ap.add_argument("--sustained", type=int, default=300, help="extra steady-state steps (0 = skip)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true")
    ap.add_argument("--eager", action="store_true", help="launch every kernel from the host (no CUDA graph)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the metrics and model state of the last timed step to DIR/<name>.npy; runs the "
                         "deterministic mode so that runs with the same arguments write the same arrays")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what this implementation's timed step computed (--impl ours)")
    if args.dump_outputs:
        os.environ["B200_DETERMINISTIC"] = "1"   # read when run_ours imports the package
    args.warmup = max(3, args.warmup)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
