"""Record the reference-side values of the host-logic tests in tests/test_host_logic.py -> case_host.npz and
bunny_smoke_config.yaml.  Run once with a checkout of ueda0319/neddf (it is not needed afterwards):

    python tests/golden/make_host_golden.py <path to the ueda0319/neddf checkout>

* ``neus_*``: neddf.network.NeuS(**NEUS_KW) built after torch.manual_seed(7): its state_dict key order, a SHA-256 of
  every tensor's float32 bytes and a seeded sample of 16 values per tensor (the whole state_dict is 2.5 MB).
* ``gather_*``: BaseTrainer.construct_ground_truth on a seeded dataset item and seeded pixel ids.
* ``ckpt_keys``: key order of pretrained/bunny_smoke/models/model_02000.pth, whose tensors are the ones in
  bunny_smoke_weights.npz (checked here); bunny_smoke_config.yaml is that run's saved .hydra/config.yaml.
"""
import hashlib
import json
import os
import shutil
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
NEUS_KW = dict(embed_pos_rank=5, embed_dir_rank=3, sdf_layer_count=6, col_layer_count=3, activation_type="tanhExp",
               init_variance=0.45, skips=[1, 3])
GATHER_KINDS = ["ColorLoss", "MaskBCELoss", "FieldsConstraintLoss"]


def tensor_digest(t: torch.Tensor) -> str:
    return hashlib.sha256(t.detach().to(torch.float32).contiguous().numpy().tobytes()).hexdigest()


def tensor_sample(t: torch.Tensor) -> np.ndarray:
    flat = t.detach().to(torch.float32).reshape(-1).numpy()
    return flat[np.random.default_rng(0).choice(flat.size, min(16, flat.size), replace=False)]


def gather_inputs():
    rng = np.random.default_rng(3)
    rgb = rng.integers(0, 256, (20, 30, 3), dtype=np.uint8)
    mask = rng.integers(0, 256, (20, 30), dtype=np.uint8)
    g = torch.Generator().manual_seed(3)
    us = (torch.rand(64, generator=g) * 29).to(torch.int16)
    vs = (torch.rand(64, generator=g) * 19).to(torch.int16)
    return rgb, mask, us, vs


def main(ref: str) -> None:
    sys.path[:0] = [ref, os.path.join(HERE, "_refstub")]
    sk, m = types.ModuleType("skimage"), types.ModuleType("skimage.metrics")
    m.peak_signal_noise_ratio = m.structural_similarity = None
    sk.metrics = m
    sys.modules.update({"skimage": sk, "skimage.metrics": m})
    from neddf.network import NeuS
    from neddf.trainer.base_trainer import BaseTrainer

    torch.manual_seed(7)
    sd = NeuS(**NEUS_KW).state_dict()
    out = {"neus_keys": json.dumps(list(sd)), "neus_sha256": json.dumps([tensor_digest(v) for v in sd.values()])}
    for i, v in enumerate(sd.values()):
        out[f"neus_sample_{i}"] = tensor_sample(v)

    rgb, mask, us, vs = gather_inputs()
    t = types.SimpleNamespace(device=torch.device("cpu"), dataset=[dict(rgb_images=rgb, mask_images=mask)])
    targets = BaseTrainer.construct_ground_truth(t, 0, us, vs, GATHER_KINDS)
    assert sorted(targets) == ["color", "fields_penalty", "mask"]
    out.update({"gather_" + k: v.numpy() for k, v in targets.items()})

    run = os.path.join(ref, "pretrained", "bunny_smoke")
    ckpt = torch.load(os.path.join(run, "models", "model_02000.pth"), map_location="cpu")
    w = np.load(os.path.join(HERE, "bunny_smoke_weights.npz"))
    for k, v in ckpt.items():
        assert np.array_equal(v.numpy(), w[k.split(".", 1)[1]]), k
    out["ckpt_keys"] = json.dumps(list(ckpt))
    np.savez(os.path.join(HERE, "case_host.npz"), **out)
    shutil.copyfile(os.path.join(run, ".hydra", "config.yaml"), os.path.join(HERE, "bunny_smoke_config.yaml"))


if __name__ == "__main__":
    main(sys.argv[1])
