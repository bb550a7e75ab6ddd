"""GPU parity of the on-device input pipeline (b200_augment_batch through the C ABI): bit-exact against golden
vectors made from the UNMODIFIED reference transforms and, at CIFAR shape / batch 128, against the numpy
oracle with injected random draws (integer / index work + IEEE fp32 arithmetic => exact equality)."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import transform_oracle as TO  # noqa: E402
from tests.test_transform_cpu import CASES, GOLDEN, case_kwargs  # noqa: E402

pytestmark = pytest.mark.gpu


def _run(data, index, kw, want_f32=True):
    from pytorch_ddp_resnet_b200 import ops
    dev = "cuda"
    t = lambda a, dt: None if a is None else torch.as_tensor(np.ascontiguousarray(a)).to(dt).to(dev)  # noqa: E731
    H, W = data.shape[1:3]
    pad = kw["pad_size"]
    out_hw = (kw["crop_size"],) * 2 if kw["crop_size"] else (H + 2 * pad, W + 2 * pad)
    return ops.augment_batch(
        torch.from_numpy(data).to(dev), t(index, torch.int64), flip=t(kw["flips"], torch.uint8),
        top=t(kw["tops"], torch.int32), left=t(kw["lefts"], torch.int32), mean=t(kw["mean"], torch.float32),
        stddev=t(kw["stddev"], torch.float32), pad=pad, pad_mirror=kw["pad_type"] == "mirror", out_hw=out_hw,
        want_f32=want_f32, want_bf16=True)


@pytest.mark.parametrize("c", CASES)
def test_kernel_bit_exact_vs_reference_golden(c):
    z = np.load(GOLDEN)
    of, ob = _run(z["data"], z[f"{c}/index"], case_kwargs(z, c))
    ref = torch.from_numpy(z[f"{c}/out"]).cuda()
    assert torch.equal(of, ref)
    assert torch.equal(ob.permute(0, 3, 1, 2), ref.bfloat16())   # the NHWC bf16 batch the stem consumes


@pytest.mark.parametrize("pad_type,whiten", [("mirror", "standardize"), ("zero", "zeromean"), ("zero", None)])
def test_kernel_bit_exact_vs_oracle_cifar_shape_batch128(pad_type, whiten):
    rng = np.random.default_rng(7)
    M, B, H = 500, 128, 32
    data = rng.integers(0, 256, size=(M, H, H, 3), dtype=np.uint8)
    mean = rng.random((3, H, H), dtype=np.float32) if whiten else None
    std = (rng.random((3, H, H), dtype=np.float32) + 0.2) if whiten == "standardize" else None
    kw = dict(mean=mean, stddev=std, flips=rng.integers(0, 2, B).astype(np.uint8), pad_size=4, pad_type=pad_type,
              tops=rng.integers(0, 9, B).astype(np.int32), lefts=rng.integers(0, 9, B).astype(np.int32), crop_size=32)
    kw["tops"][:4] = [0, 8, 0, 8]       # the extreme crop positions
    kw["lefts"][:4] = [0, 0, 8, 8]
    index = rng.integers(0, M, B)
    of, ob = _run(data, index, kw)
    ref = torch.from_numpy(TO.pipeline(data, index, **kw)).cuda()
    assert torch.equal(of, ref)
    assert torch.equal(ob.permute(0, 3, 1, 2), ref.bfloat16())


def test_device_loader_feeds_the_model(tmp_path):
    """DeviceDataLoader: one launch per batch, draws made on the device, batches that ResNet.forward takes as
    they are; an epoch visits every sample of the rank's shard once."""
    from pytorch_ddp_resnet_b200.architectures.resnet import ResNet
    from pytorch_ddp_resnet_b200.utils import data_util as D
    aug = {"ToTensorTransform": {}, "StandardizeWhiteningTransform": {}, "FlipTransform": {"p": 0.5},
           "PaddingTransform": {"pad_size": 4, "pad_type": "mirror"}, "RandomCropTransform": {"crop_size": 32}}
    ds = D.get_datasets("SyntheticCIFAR10", str(tmp_path), aug, {"ToTensorTransform": {}, "StandardizeWhiteningTransform": {}},
                        synthetic_train_size=256, synthetic_test_size=64)
    sm = D.get_samplers(0, 1, ds["dataset_train"], ds["dataset_test"])
    dl = D.get_dataloaders(64, 1, 1, ds["dataset_train"], ds["dataset_test"], **sm)
    model = ResNet("c3,16,3,1,1 n a r1 ap32,1,0 fc16,10", False, False, 0.0).cuda().train()
    seen = 0
    for x, y in dl["dl_train"]:
        assert x.is_cuda and x.dtype == torch.bfloat16 and tuple(x.shape) == (64, 3, 32, 32)
        assert x.permute(0, 2, 3, 1).is_contiguous() and y.dtype == torch.int64
        assert model(x).shape == (64, 10)
        seen += y.numel()
    assert seen == 256
    # whitened data: per-pixel statistics ~ (0, 1) over the training set when nothing is augmented
    tr = ds["dataset_train"]
    allx = ds["dataset_test"].pipeline(tr.data, torch.arange(256, device="cuda"), want_f32=True)
    assert allx.mean().abs() < 1e-3 and abs(allx.std().item() - 1.0) < 0.05
    flip, top, left = tr.pipeline.draw(4096, tr.data.device)
    assert abs(flip.float().mean().item() - 0.5) < 0.05 and top.min() >= 0 and top.max() == 8 and left.max() == 8
