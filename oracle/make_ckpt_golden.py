"""Fixture for the ONLY artefact the reference ships for this path: its pretrained generator `models/model.pt`
(3.7 MB, 36 fp32 tensors saved from a torch.compile'd module: keys carry `_orig_mod.`, inference.py:27-33).

    python oracle/make_ckpt_golden.py REFERENCE_DIR    # a checkout of the reference; writes tests/golden/checkpoint_golden.npz

A fixture file stays under 1 MB, so the checkpoint is stored with every conv weight quantized to int8 per output
channel (symmetric, fp32 scale; biases and PReLU slopes stay fp32).  The quantized network keeps what the test is
about - trained weights that amplify operand rounding through 17 stacked InstanceNorms: with the oracle's fp16
storage rounding its output error is 3.4e-4 mean-abs, the same as the fp32 checkpoint's.

Imports the UNMODIFIED reference model.py, loads the dequantized weights with the `_orig_mod.` prefix stripped the
way inference.py:27-35 does, runs `Generator.forward` (model.py:112-117) in fp32 on the CPU on frame 0 of the
survey's anchor input (`torch.manual_seed(0); x = torch.rand(2,3,90,160)*2-1`, SURVEY.md 8c), asserts the oracle
restatement reproduces it, and stores: the quantized state dict (original key names, `_orig_mod.` prefix kept - the
loader must strip it) and the reference's output at the N_SAMPLE seeded positions of `sample_idx`.
The tests never read the reference: tests/test_baseline_configs_gpu.py uses the fixture and the helpers below only.
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
import srgan_oracle as O  # noqa: E402

N_SAMPLE = 32768


def anchor_input() -> torch.Tensor:
    """Frame 0 of SURVEY.md 8c's anchor input, 1x3x90x160."""
    return torch.rand((1, 3, 90, 160), generator=torch.Generator().manual_seed(0)) * 2 - 1


def sample_idx(numel: int) -> torch.Tensor:
    """Seeded uniform sample of flat output positions, shared with the test."""
    return torch.randperm(numel, generator=torch.Generator().manual_seed(8))[:N_SAMPLE].sort().values


def state_dict(fix) -> dict:
    """The fixture's generator weights as fp32 tensors (keys keep `_orig_mod.`): int8 conv weights times their scale."""
    sd = {k[3:]: torch.from_numpy(fix[k]) for k in fix if k.startswith("sd/")}
    for k in fix:
        if k.startswith("q/"):
            sd[k[2:]] = torch.from_numpy(fix[k]).float() * torch.from_numpy(fix["scale/" + k[2:]]).view(-1, 1, 1, 1)
    return sd


def main(ref_dir):
    sys.path.insert(0, ref_dir)
    import model  # the reference's model.py, unmodified
    raw = torch.load(os.path.join(ref_dir, "models", "model.pt"), map_location="cpu")
    out = {}
    for k, v in raw.items():
        if v.dim() == 4:
            scale = v.abs().amax(dim=(1, 2, 3)) / 127
            out["q/" + k] = torch.round(v / scale.view(-1, 1, 1, 1)).to(torch.int8).numpy()
            out["scale/" + k] = scale.numpy()
        else:
            out["sd/" + k] = v.numpy()
    weights = {k.replace("_orig_mod.", ""): v for k, v in state_dict(out).items()}   # inference.py:30-33
    g = model.Generator(types.SimpleNamespace(n_filters=64, n_layers=8))
    print(g.load_state_dict(weights))
    g.eval()
    x = anchor_input()
    with torch.no_grad():
        y = g(x)
        yo = O.generator_forward(weights, x)
    err = (y - yo).abs().max().item()
    print(f"oracle vs reference on the quantized checkpoint: max-abs {err:.3e}")
    assert err <= 5e-5
    out["y_sample"] = y.reshape(-1)[sample_idx(y.numel())].numpy()
    path = os.path.join(ROOT, "tests", "golden", "checkpoint_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
