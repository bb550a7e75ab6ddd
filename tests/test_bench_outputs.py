"""bench.py --dump-outputs: what the last timed step computed, as <name>.npy files that two builds can compare."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_dump_outputs_fixed_sample_and_size(tmp_path):
    """Every config's dump fits the size limit, and large tensors are sampled at the same indices every time."""
    import bench
    from pytorch_ddp_resnet_b200.architectures.resnet import ResNet
    for name in bench.CONFIGS:
        c = bench.resolve_config(name, 1)
        model = ResNet(c["spec"], c["preact"], c["use_proj"], c["dropout"])
        n = sum(min(v.numel(), bench.DUMP_SAMPLE) for v in model.state_dict().values())
        assert 4 * n <= bench.DUMP_MAX_BYTES, name
    torch.manual_seed(0)
    c = bench.resolve_config("wrn28", 1)
    model = ResNet(c["spec"], c["preact"], c["use_proj"], c["dropout"])
    metrics = {"loss": torch.tensor(2.5), "top1_err": torch.tensor(0.75), "top5_err": torch.tensor(0.25)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), metrics, model)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(os.listdir(tmp_path / "b"))
    assert len(files) == 3 + len(model.state_dict())
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_MAX_BYTES
    sd = model.state_dict()
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert np.array_equal(a, b), f
        assert a.dtype in (np.float32, np.float64), f
        if f.startswith("state."):
            t = sd[f[len("state."):-len(".npy")]]
            if t.numel() > bench.DUMP_SAMPLE:
                assert a.shape == (bench.DUMP_SAMPLE,)
                assert np.isin(a, t.float().reshape(-1).numpy()).all()
            else:
                assert np.array_equal(a, t.double().numpy() if not t.is_floating_point() else t.float().numpy())
    assert float(np.load(tmp_path / "a" / "loss.npy")) == 2.5


def _bench(steps, out):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "3", "--sustained",
           "0", "--no-cpu-baseline", "--no-gpu-reference", "--dump-outputs", str(out)]
    env = {k: v for k, v in os.environ.items() if k != "B200_DETERMINISTIC"}   # the flag alone must make runs equal
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == steps and line["config"]["deterministic"] is True


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(tmp_path):
    """--steps sets how many steps the dumped state has seen (warm-up + timed; BatchNorm counts them), the dump
    holds finite metrics and parameters, and the same arguments give the same arrays."""
    _bench(2, tmp_path / "s2")
    _bench(3, tmp_path / "s3")
    _bench(3, tmp_path / "s3again")
    files = sorted(os.listdir(tmp_path / "s2"))
    assert files == sorted(os.listdir(tmp_path / "s3")) == sorted(os.listdir(tmp_path / "s3again"))
    tracked = [f for f in files if f.endswith("num_batches_tracked.npy")]
    assert tracked
    for f in tracked:
        assert int(np.load(tmp_path / "s2" / f)) == 3 + 2, f
        assert int(np.load(tmp_path / "s3" / f)) == 3 + 3, f
    for f in files:
        a = np.load(tmp_path / "s3" / f)
        assert np.isfinite(a).all(), f
        assert np.array_equal(a, np.load(tmp_path / "s3again" / f)), f
    assert 0.0 < float(np.load(tmp_path / "s3" / "loss.npy")) < 10.0
