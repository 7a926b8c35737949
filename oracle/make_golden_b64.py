"""Golden fixture for the BASELINE training config (configs[2]: full GAN train_step, 24x24 LR / 96x96 HR, batch 64).

    python oracle/make_golden_b64.py          # ~3 min on 8 cores; writes tests/golden/train_b64_golden.npz

Runs THREE consecutive iterations of the reference GAN loop body (trainer.py:168-196) in fp64 through
oracle/srgan_oracle.py::gan_step - which oracle/make_golden.py pins against a genuine Trainer.train() iteration of
the unmodified reference (fp64: gradients <=2e-16, parameters <=4e-14) - on seeded weights / inputs / label noise
with persistent AdamW state, and also three iterations of the pre-training body (trainer.py:104-111) at batch 16.

A full fp64 gradient set is 45 MB and a fixture file stays under 1 MB, so the fixture keeps per tensor:
  * the full-tensor L2 norm and a seeded uniform random SUBSAMPLE (<= 2048 elements) of the step-1 gradient
    (rel-L2 / cosine over a 2 K uniform subsample estimate the full-tensor figures to ~2 %),
  * the parameter UPDATE of every step on a <= 512-element subsample (sign agreement of the trajectory),
  * the four losses of every step.
tests/test_baseline_configs_gpu.py rebuilds the same inputs from the seeds below and compares the B200 engine with it.
"""
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
import srgan_oracle as O  # noqa: E402

B, STEPS = 64, 3
K_GRAD, K_UPD = 2048, 512
PRE_B = 16


def sub_idx(numel: int, k: int) -> torch.Tensor:
    """Seeded uniform subsample shared with the test (sorted indices; every element when numel <= k).  Random rather
    than strided: a stride that is a multiple of 9 would keep a single tap of every 3x3 kernel."""
    if numel <= k:
        return torch.arange(numel)
    return torch.randperm(numel, generator=torch.Generator().manual_seed(numel))[:k].sort().values


def step_inputs(step: int, b: int = B):
    g = torch.Generator().manual_seed(1000 + step)
    lr = torch.rand((b, 3, 24, 24), generator=g) * 2 - 1
    hr = torch.rand((b, 3, 96, 96), generator=g) * 2 - 1
    noise = {k: torch.rand((b, 1, 6, 6), generator=g) for k in ("d_real", "d_fake", "g_real")}
    return lr, hr, noise


def main():
    torch.set_num_threads(os.cpu_count() or 8)
    out = {}
    c = lambda sd: {k: v.double().clone() for k, v in sd.items()}
    og, od, ov = c(O.make_generator_state(64, 8, 1234)), c(O.make_discriminator_state(64, 4321)), c(O.make_vgg19_state(99))
    opt_g, opt_d = O.AdamWState(og, 1e-4), O.AdamWState(od, 1e-4)
    for s in range(STEPS):
        lr, hr, noise = step_inputs(s)
        before = {"g": {k: v.clone() for k, v in og.items()}, "d": {k: v.clone() for k, v in od.items()}}
        t0 = time.time()
        res = O.gan_step(og, od, ov, lr.double(), hr.double(), {k: v.double() for k, v in noise.items()}, opt_g, opt_d)
        print(f"step {s}: {time.time() - t0:.1f} s  " + "  ".join(f"{k}={res[k].item():.9f}" for k in ("loss_real", "loss_fake", "adv_loss", "content_loss")))
        for k in ("loss_real", "loss_fake", "adv_loss", "content_loss"):
            out[f"s{s}/{k}"] = np.float64(res[k].item())
        for net, after in (("g", og), ("d", od)):
            for k, v in after.items():
                upd = (v - before[net][k]).reshape(-1)
                out[f"s{s}/{net}_upd/{k}"] = upd[sub_idx(upd.numel(), K_UPD)].float().numpy()
        if s == 0:
            for net, grads in (("g", res["g_grads"]), ("d", res["d_grads"])):
                for k, v in grads.items():
                    flat = v.reshape(-1)
                    out[f"s0/{net}_grad_norm/{k}"] = np.float64(flat.norm().item())
                    out[f"s0/{net}_grad/{k}"] = flat[sub_idx(flat.numel(), K_GRAD)].float().numpy()

    # ---- pre-training body (trainer.py:104-111), fp64, 3 steps at batch 16
    pg = c(O.make_generator_state(64, 8, 1234))
    popt = O.AdamWState(pg, 1e-4)
    for s in range(STEPS):
        lr, hr, _ = step_inputs(50 + s, PRE_B)
        before = {k: v.clone() for k, v in pg.items()}
        res = O.pretrain_step(pg, lr.double(), hr.double(), popt)
        out[f"pre{s}/loss"] = np.float64(res["loss"].item())
        print(f"pretrain step {s}: loss {res['loss'].item():.9f}")
        for k, v in pg.items():
            upd = (v - before[k]).reshape(-1)
            out[f"pre{s}/upd/{k}"] = upd[sub_idx(upd.numel(), K_UPD)].float().numpy()
        if s == 0:
            for k, v in res["g_grads"].items():
                flat = v.reshape(-1)
                out[f"pre0/grad_norm/{k}"] = np.float64(flat.norm().item())
                out[f"pre0/grad/{k}"] = flat[sub_idx(flat.numel(), K_GRAD)].float().numpy()
    path = os.path.join(ROOT, "tests", "golden", "train_b64_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
