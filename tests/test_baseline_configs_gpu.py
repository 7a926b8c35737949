"""Parity at the BASELINE.json configurations themselves (VERDICT r01 "what's missing" 1-3):

  configs[1]  one 180x320 frame through Generator.forward, fp16, vs the CPU oracle (model.py:112-117)        <= 1e-3
  configs[2]  THREE consecutive GAN train steps at batch 64 (trainer.py:168-196) vs the fp64 oracle fixture
              tests/golden/train_b64_golden.npz (oracle/make_golden_b64.py): losses, step-1 gradients per tensor,
              sign agreement of every parameter update of the trajectory
  f1          three pre-training steps (trainer.py:104-111) at batch 16 vs the same fixture
  fixture     the reference's shipped checkpoint models/model.pt, conv weights int8 per output channel
              (tests/golden/checkpoint_golden.npz, oracle/make_ckpt_golden.py)

The gradient / update figures are printed per tensor and, when FSR_REPORT_DIR is set, written as a markdown report
(committed as profiles/r02/grad_parity.md).
"""
import os
import sys
import types

import numpy as np
import pytest
import torch

import srgan_oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))


def ns(**k):
    return types.SimpleNamespace(**k)


def seeded(shape, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(shape, generator=g) * 2 - 1


@pytest.fixture(scope="module")
def gold64():
    return np.load(os.path.join(ROOT, "tests", "golden", "train_b64_golden.npz"))


@pytest.fixture(scope="module")
def ckpt():
    return np.load(os.path.join(ROOT, "tests", "golden", "checkpoint_golden.npz"))


def _report(name: str, lines):
    d = os.environ.get("FSR_REPORT_DIR")
    if d:
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, name), "w") as f:
            f.write("\n".join(lines) + "\n")


# ------------------------------------------------------------------------------------------- configs[1]
@pytest.mark.parametrize("dt,tol", [(torch.float16, 1e-3), (torch.float32, 1e-4)])
def test_generator_180x320_frame_vs_oracle(dt, tol):
    """The benchmarked shape (BASELINE configs[1]: 180x320 -> 720x1280), one frame, against the CPU oracle.
    fp16 operands: north_star's 1e-3; compute_dtype=float32 (split-operand precise mode): 1e-4."""
    from fast_srgan_b200.model import Generator
    sd = O.make_generator_state(64, 8, seed=1234)
    g = Generator(ns(n_filters=64, n_layers=8), compute_dtype=dt)
    g.load_state_dict(sd)
    g = g.cuda().eval()
    x = seeded((1, 3, 180, 320), 41)
    with torch.no_grad():
        y = g(x.cuda()).cpu()
        ref = O.generator_forward(sd, x)
    err = (y - ref).abs().max().item()
    print(f"generator 1x3x180x320 {dt}: max-abs vs oracle {err:.3e}")
    assert y.shape == (1, 3, 720, 1280) and err <= tol


# ------------------------------------------------------------------------------------------- shipped checkpoint
@pytest.mark.parametrize("dt,tol", [(torch.float32, 1e-3), (torch.float16, 6e-3), (torch.bfloat16, 6e-2)])
def test_shipped_checkpoint_parity(ckpt, dt, tol):
    """models/model.pt (conv weights int8 per output channel) loaded the way inference.py:27-35 does (`_orig_mod.`
    keys), 90x160 anchor frame of SURVEY 8c, against the output of the UNMODIFIED reference at the fixture's seeded
    sample of output positions.  The trained weights amplify operand rounding through 17 stacked InstanceNorms
    (residual stream |x| up to 17): fp16 operands measure ~3e-3 here (SURVEY 0 predicted 3.2e-3), bf16 ~3e-2;
    north_star's 1e-3 on this fixture needs the precise mode (compute_dtype=torch.float32: fp16 hi+lo split
    operands, fp32 storage)."""
    import make_ckpt_golden as MC
    from fast_srgan_b200.model import Generator
    g = Generator(ns(n_filters=64, n_layers=8), compute_dtype=dt)
    g.load_state_dict(MC.state_dict(ckpt))                                      # keys keep `_orig_mod.`
    g = g.cuda().eval()
    with torch.no_grad():
        y = g(MC.anchor_input().cuda()).cpu()
    assert y.shape == (1, 3, 360, 640)
    got = y.reshape(-1)[MC.sample_idx(y.numel())]
    ref = torch.from_numpy(ckpt["y_sample"])
    err = (got - ref).abs().max().item()
    print(f"shipped checkpoint, 1x3x90x160, {dt}: max-abs vs reference {err:.3e}  mean-abs {(got - ref).abs().mean().item():.3e}"
          f"  ({ref.numel()} sampled outputs)")
    assert err <= tol


# ------------------------------------------------------------------------------------------- configs[2]
def _sub(t: torch.Tensor, k: int) -> torch.Tensor:
    import make_golden_b64 as MG
    flat = t.reshape(-1)
    return flat[MG.sub_idx(flat.numel(), k).to(flat.device)]


def _trainer(dt, lr=1e-4):
    from fast_srgan_b200.trainer import Trainer
    cfg = ns(experiment=ns(name="t", seed=0), generator=ns(n_filters=64, n_layers=8), discriminator=ns(n_filters=64, n_layers=7),
             training=ns(device="cuda", generator_lr=lr, discriminator_lr=lr))
    tr = Trainer(cfg, compute_dtype=dt, vgg_state_dict=O.make_vgg19_state(99))
    tr.generator.load_state_dict(O.make_generator_state(64, 8, 1234))
    tr.discriminator.load_state_dict(O.make_discriminator_state(64, 4321))
    return tr


def _grad_table(title, nets, gold, prefix, S):
    """nets: [(name, FlatParams, key)].  Returns (markdown lines, list of (name, tensor, numel, rel, cos))."""
    import make_golden_b64 as MG
    lines = [f"### {title}", "", "| net | tensor | numel | rel-L2 err (subsample) | cosine | norm engine / norm fp64 |", "|---|---|---|---|---|---|"]
    rows = []
    for name, fp, key in nets:
        for k in fp.names:
            gk = f"{prefix}{key}_grad/{k}" if key else f"{prefix}grad/{k}"
            nk = f"{prefix}{key}_grad_norm/{k}" if key else f"{prefix}grad_norm/{k}"
            if gk not in gold.files:
                continue
            ref = torch.from_numpy(gold[gk]).double()
            got_full = fp.g[k].double() / S
            got = _sub(got_full, MG.K_GRAD).cpu()
            rel = ((got - ref).norm() / ref.norm().clamp_min(1e-30)).item()
            cos = (got @ ref / (got.norm() * ref.norm()).clamp_min(1e-30)).item()
            nr = got_full.norm().item() / max(float(gold[nk]), 1e-30)
            rows.append((name, k, got_full.numel(), rel, cos, nr))
            lines.append(f"| {name} | {k} | {got_full.numel()} | {rel:.3e} | {cos:.4f} | {nr:.4f} |")
    return lines, rows


@pytest.mark.parametrize("dt,ltol", [(torch.bfloat16, 5e-3), (torch.float16, 1.5e-3)])
def test_train_step_b64_three_steps_vs_fp64_oracle(gold64, dt, ltol):
    """BASELINE configs[2] (batch 64, 24x24 LR / 96x96 HR), three consecutive steps with persistent AdamW state:
    steps 1-2 run eagerly, step 3 is the captured CUDA graph.  Asserted: the four losses of every step against the
    fp64 oracle; step-1 gradients per tensor (rel-L2 and cosine over a seeded 2 K-element subsample, full-tensor norm ratio);
    sign agreement of every parameter update."""
    import make_golden_b64 as MG
    tr = _trainer(dt)
    e = tr.engine
    tag = "bf16" if dt == torch.bfloat16 else "fp16"
    report = [f"## GAN train step, batch 64, {tag} operands / fp32 accumulate, vs the fp64 oracle (trainer.py:168-196)", ""]
    prev = {"g": {k: v.clone() for k, v in e.gp.p.items()}, "d": {k: v.clone() for k, v in e.dp.p.items()}}
    for s in range(MG.STEPS):
        lr_img, hr_img, noise = MG.step_inputs(s)
        out = tr.train_step(lr_img, hr_img, noise=noise)
        torch.cuda.synchronize()
        report.append(f"step {s + 1} losses (engine / fp64 oracle): " + ", ".join(
            f"{k} {out[k].item():.6f} / {float(gold64[f's{s}/{k}']):.6f}" for k in ("loss_real", "loss_fake", "adv_loss", "content_loss")))
        print(report[-1])
        for k in ("loss_real", "loss_fake", "adv_loss", "content_loss"):
            ref = float(gold64[f"s{s}/{k}"])
            assert abs(out[k].item() - ref) <= ltol * max(1.0, abs(ref)) * (1 + s), (s, k, out[k].item(), ref)
        if s == 0:
            lines, rows = _grad_table("step-1 gradients", [("D", e.dp, "d"), ("G", e.gp, "g")], gold64, "s0/", e.S)
            report += [""] + lines + [""]
            print("\n".join(lines))
            for name, k, numel, rel, cos, nr in rows:
                if numel > 1:
                    # measured on B200 (profiles/r02/grad_parity.md); the 16-bit-storage floor of these ill-conditioned
                    # gradients is DESIGN.md section 5
                    assert cos >= (0.90 if dt == torch.bfloat16 else 0.97), (name, k, cos)
                    assert rel <= (0.45 if dt == torch.bfloat16 else 0.25), (name, k, rel)
                    assert 0.8 <= nr <= 1.25, (name, k, nr)
        agree_lines = []
        for net, fp in (("g", e.gp), ("d", e.dp)):
            for k in fp.names:
                upd = _sub(fp.p[k] - prev[net][k], MG.K_UPD).double().cpu()
                ref = torch.from_numpy(gold64[f"s{s}/{net}_upd/{k}"]).double()
                agree = (torch.sign(upd) == torch.sign(ref)).double().mean().item()
                maxd = (upd - ref).abs().max().item()
                agree_lines.append((net, k, upd.numel(), agree, maxd))
                assert maxd <= 2.05e-4 * (s + 1), (s, net, k, maxd)           # |update| <= lr (+wd) per step
                if upd.numel() > 1:
                    assert agree >= 0.80, (s, net, k, agree)
                prev[net][k] = fp.p[k].clone()
        worst = min(a for _, _, n, a, _ in agree_lines if n > 1)
        mean = float(np.mean([a for _, _, n, a, _ in agree_lines if n > 1]))
        report.append(f"step {s + 1} update-sign agreement over {len(agree_lines)} tensors: mean {mean:.4f}, worst {worst:.4f}")
        print(report[-1])
    assert e.gp.step_count == MG.STEPS and int(e.dp.step_dev.item()) == MG.STEPS
    _report(f"grad_parity_train_b64_{tag}.md", report)


@pytest.mark.parametrize("dt,ltol", [(torch.bfloat16, 5e-3), (torch.float16, 1e-3)])
def test_pretrain_three_steps_vs_fp64_oracle(gold64, dt, ltol):
    """SURVEY 8 row f1: Trainer.pretrain's loop body (trainer.py:104-111: SmoothL1(G(lr), hr), backward, AdamW) at
    batch 16, three steps, against the fp64 oracle restatement (oracle/srgan_oracle.py::pretrain_step)."""
    import make_golden_b64 as MG
    tr = _trainer(dt)
    e = tr.engine
    tag = "bf16" if dt == torch.bfloat16 else "fp16"
    report = [f"## pre-training step, batch {MG.PRE_B}, {tag} operands, vs the fp64 oracle (trainer.py:104-111)", ""]
    prev = {k: v.clone() for k, v in e.gp.p.items()}
    for s in range(MG.STEPS):
        lr_img, hr_img, _ = MG.step_inputs(50 + s, MG.PRE_B)
        out = tr.pretrain_step(lr_img, hr_img)
        torch.cuda.synchronize()
        ref = float(gold64[f"pre{s}/loss"])
        report.append(f"step {s + 1} loss (engine / fp64 oracle): {out['loss'].item():.6f} / {ref:.6f}")
        print(report[-1])
        assert abs(out["loss"].item() - ref) <= ltol * max(1.0, abs(ref))
        if s == 0:
            lines, rows = _grad_table("step-1 gradients", [("G", e.gp, "")], gold64, "pre0/", e.S)
            report += [""] + lines + [""]
            print("\n".join(lines))
            for name, k, numel, rel, cos, nr in rows:
                if numel > 1:
                    assert cos >= (0.90 if dt == torch.bfloat16 else 0.97), (k, cos)
                    assert rel <= (0.45 if dt == torch.bfloat16 else 0.25), (k, rel)
        agrees = []
        for k in e.gp.names:
            upd = _sub(e.gp.p[k] - prev[k], MG.K_UPD).double().cpu()
            refu = torch.from_numpy(gold64[f"pre{s}/upd/{k}"]).double()
            assert (upd - refu).abs().max().item() <= 2.05e-4 * (s + 1), (s, k)
            if upd.numel() > 1:
                agrees.append((torch.sign(upd) == torch.sign(refu)).double().mean().item())
            prev[k] = e.gp.p[k].clone()
        report.append(f"step {s + 1} update-sign agreement: mean {float(np.mean(agrees)):.4f}, worst {min(agrees):.4f}")
        print(report[-1])
        assert min(agrees) >= 0.80
    _report(f"grad_parity_pretrain_{tag}.md", report)
