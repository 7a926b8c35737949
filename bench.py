#!/usr/bin/env python
"""bench.py - headline benchmark of the Fast-SRGAN B200 engine (driver contract, see DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): generator-only 4x super-resolution, 180x320 -> 720x1280,
batch 32 frames per GPU per step, L=8 residual blocks, F=64, synthetic frames, random-init weights.
One "step" = one pass of Generator.forward over one batch.  Metric: SR frames/s (whole job).

  value : inputs resident in HBM, device-timed (CUDA events, max over ranks), Generator.forward.
  e2e   : same metric through the public API with HOST buffers: pinned uint8 frames -> H2D ->
          Generator.super_resolve_u8 (the inference.py:48-56 pipeline) -> D2H uint8 frames, every step.
  roofline     : dominant kernel (the 64->256 upsampling conv at 360x640), timed per launch inside the
                 timed region with CUDA events on its launch stream (fsr_profile_* hooks).
  cpu_baseline : the oracle port of the reference generator on the host cores, bounded sample.
  --impl reference : the reference CPU path (the oracle port of the reference generator).
  --dump-outputs DIR : after the timed steps, rank 0 writes what its last step returned to the caller, as float32
          .npy files (56 MB in all): value's Generator.forward output (frame 0 in full + a seeded sample of the batch)
          and e2e's uint8 frames (the same).  Inputs and weights are seeded, so two builds can be compared file by file.
Multi-GPU: frames are independent -> one replica per rank, no data-path collective ("weak" scaling).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

BATCH, H, W, NF, NL = 32, 180, 320, 64, 8
METRIC = "4x SR frames/sec at 180x320->720p, batch 32"
UNIT = "frames/s"


def gen_flops_per_frame(h, w, F=NF, L=NL):
    """SURVEY.md 8(d): conv FLOPs (MAC = 2) per LR pixel of the generator."""
    return float(h * w) * (2 * 27 * F + 2 * 9 * F * F * (2 * L + 1) + 2 * 9 * F * 4 * F * (1 + 4) + 16 * 2 * 9 * F * 3)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1425.0), d.get("hbm_gbs", 6566.7), "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clock / throttle-reason samples DURING the timed region."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for nme, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except (ValueError, IndexError):
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def _host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


class _CpuGenerator:
    """The reference's CPU implementation of the path, as the oracle port of model.py:112-117 - kind "port"."""

    def __init__(self):
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import srgan_oracle as O
        self.sd = O.make_generator_state(NF, NL, seed=1234)
        self.kind, self.what = "port", "oracle port of model.py:112-117 (oracle/srgan_oracle.py), fp32 oneDNN"
        self.fn = lambda x: O.generator_forward(self.sd, x)


def _cpu_setup():
    c = _CpuGenerator()
    return c, c.sd


def _time_cpu(O, sd, rows, iters):
    g = torch.Generator().manual_seed(0)
    x = torch.rand((1, 3, rows, W), generator=g) * 2 - 1
    with torch.no_grad():
        t0 = time.perf_counter()
        for _ in range(iters):
            O.fn(x)
    return (time.perf_counter() - t0) / iters


def pick_cpu_threads(O, sd):
    """Give the reference CPU path its best thread count (oversubscribed boxes are slower with all cores)."""
    avail = _host_threads()
    best, best_t = None, None
    for th in sorted({avail, min(avail, 64), min(avail, 32), min(avail, 16)}, reverse=True):
        torch.set_num_threads(th)
        _time_cpu(O, sd, 24, 1)
        t = _time_cpu(O, sd, 24, 2)
        if best_t is None or t < best_t:
            best, best_t = th, t
    torch.set_num_threads(best)
    return best


def cpu_generator_fps(budget_s=20.0):
    """Reference CPU path (oracle port of model.py:112-117) on the host cores, bounded sample:
    full-width row bands of a 180x320 frame (the net is fully convolutional: cost/pixel is uniform)."""
    O, sd = _cpu_setup()
    threads = pick_cpu_threads(O, sd)
    t_probe = _time_cpu(O, sd, 45, 1)                      # quarter frame
    rows = int(max(9, min(H, H * (budget_s / 3.0) / (t_probe * 4.0))))
    _time_cpu(O, sd, rows, 1)
    t = _time_cpu(O, sd, rows, 2)
    return (rows / H) / t, threads, f"2 x 1 band of {rows}x{W} px of a {H}x{W} frame ({2 * t:.1f} s), fps = (rows/{H})/t; {O.what}", O.kind


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (the oracle port), rank 0 only."""
    if rank != 0:
        return
    O, sd = _cpu_setup()
    threads = pick_cpu_threads(O, sd)
    t_probe = _time_cpu(O, sd, 45, 1)
    budget = 150.0
    rows = int(max(9, min(H, H * budget / ((args.steps + args.warmup) * t_probe * 4.0))))
    for _ in range(args.warmup):
        _time_cpu(O, sd, rows, 1)
    t = _time_cpu(O, sd, rows, args.steps)
    fps = (rows / H) / t
    sample = f"{args.steps} steps x 1 band of {rows}x{W} px of a {H}x{W} frame; fps = (rows/{H}) / step time; {O.what}"
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"generator-only 4x SR {H}x{W}->{4*H}x{4*W}, L={NL} F={NF} (BASELINE configs[1]); CPU sample: {sample}"},
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": threads, "kind": O.kind, "sample": sample},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


K_NAMES = {0: "neck_conv3x3", 1: "conv3x3_c64<64,RAW_STATS> (64->64 res-block convs, incl. fused-input variants)", 2: "instnorm_apply",
           3: "conv3x3_up (64->256 + PixelShuffle + PReLU)", 4: "conv3x3_head", 5: "conv3x3_c64<64,BIAS_ACT> (64->64 dgrad)",
           6: "conv3x3_gen_ws (general conv: VGG19 / discriminator forward + data gradient)", 7: "conv3x3_wgrad"}


def read_profile(lib):
    """-> {kernel id: [(ms, flops), ...]} of the launches timed since fsr_profile_enable_mask."""
    import ctypes
    cap = 8192
    ms, ids, fl = (ctypes.c_float * cap)(), (ctypes.c_int * cap)(), (ctypes.c_double * cap)()
    n = lib.fsr_profile_read_ex(ms, ids, fl, cap)
    out = {}
    for i in range(n):
        out.setdefault(ids[i], []).append((ms[i], fl[i]))
    return out


def load_traffic():
    """DRAM bytes per launch of the profiled kernels, written by tools/ncu_summary.py from the committed `ncu --set full`
    capture (profiles/r02/traffic.json); None when no capture of this round's kernels is committed."""
    for rnd in ("r02",):
        path = os.path.join(ROOT, "profiles", rnd, "traffic.json")
        if os.path.exists(path):
            try:
                d = json.load(open(path))
                d["_source"] = f"profiles/{rnd}/traffic.json"
                return d
            except ValueError:
                pass
    return {}


DUMP_SAMPLE = 1 << 22


def output_sample(name, t):
    """{<name>_frame0: frame 0 in full, <name>_sample: DUMP_SAMPLE values of the whole tensor at seeded positions},
    float32 host arrays; t is a caller's output, batch first."""
    idx = torch.randint(0, t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
    return {f"{name}_frame0": t[0].float().cpu().numpy(), f"{name}_sample": t.reshape(-1)[idx.to(t.device)].float().cpu().numpy()}


def _time_steps(fn, n, dev, dist):
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    if dist is not None:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    return ms


def bench_train_step(args, rank, world, dev, dist, lib):
    """GAN train step (trainer.py:168-196): G + D + VGG19 perceptual, 24x24 LR / 96x96 HR synthetic pairs, bf16 operands,
    random-init weights (VGG19 too: no ImageNet download).  Measured at 32 samples per GPU for EVERY N (BASELINE
    configs[3]: global batch 256 on 8 GPUs; the same shape at N=1 is the weak-scaling anchor) and, at N=1, also at batch
    64 (configs[2]).  N>1: gradients are summed with libfsr_b200's NCCL all-reduce inside the step's CUDA graph; the
    same run also times the step WITHOUT the exchange (world forced to 1 on every rank) -> efficiency_vs_n1, times the
    two all-reduces alone, and checks that all replicas hold identical parameters after the timed steps."""
    import types
    import warnings
    from fast_srgan_b200.trainer import Trainer
    ns = types.SimpleNamespace
    steps = args.steps
    FLOPS_B64 = 2636e9                                 # SURVEY.md 8(a10)/(d): needed conv FLOPs of one step at batch 64

    def make(B, standalone):
        cfg = ns(experiment=ns(name="bench", seed=0), generator=ns(n_filters=NF, n_layers=NL), discriminator=ns(n_filters=64, n_layers=7),
                 training=ns(device=str(dev), generator_lr=1e-4, discriminator_lr=1e-4))
        torch.manual_seed(1234)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")               # random-init VGG19 is stated in `data`
            tr = Trainer(cfg, compute_dtype=torch.bfloat16)
        e = tr.engine
        if standalone:
            e.world = 1                                   # no exchange: this GPU alone on its 32 samples
        g = torch.Generator().manual_seed(7 + rank)
        lr = (torch.rand((B, 3, 24, 24), generator=g) * 2 - 1).to(dev)
        hr = (torch.rand((B, 3, 96, 96), generator=g) * 2 - 1).to(dev)
        noise = {k: torch.rand((B, 1, 6, 6), generator=g).to(dev) for k in ("d_real", "d_fake", "g_real")}
        return tr, (lambda: tr.train_step(lr, hr, noise=noise))

    def run(B, standalone):
        tr, step = make(B, standalone)
        for _ in range(4):                                # 2 eager + graph capture + 1 replay
            out = step()
        ms = _time_steps(step, steps, dev, None if standalone else dist)
        if standalone and dist is not None:               # anchor: slowest rank, like the sharded run
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return tr, step, ms, float(out["content_loss"])

    res = {"metric": "GAN train-step ms", "dtype": "bf16 operands, fp32 accumulate", "steps": steps,
           "data": "synthetic 24x24 LR / 96x96 HR pairs, random-init G / D / VGG19"}
    tr, step, ms32, closs = run(32, standalone=False)
    res["b32_per_gpu"] = {"ms_per_step": ms32, "per_gpu_batch": 32, "global_batch": 32 * world, "samples_per_s": 32 * world / (ms32 / 1e3),
                          "needed_tflops_per_gpu": FLOPS_B64 * 0.5 / (ms32 * 1e-3) / 1e12, "content_loss": closs}
    if world > 1:
        e = tr.engine
        # every replica must hold the same parameters after the timed steps (the only multi-GPU correctness number that
        # reaches the SCALE record): max over ranks - min over ranks, element-wise, summed over both networks
        diff = 0.0
        for fp in (e.gp, e.dp):
            hi, lo = fp.flat.clone(), fp.flat.clone()
            dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            dist.all_reduce(lo, op=dist.ReduceOp.MIN)
            diff = max(diff, (hi - lo).abs().max().item())
        res["replica_max_diff"] = diff
        res["exchange"] = "fsr_nccl_allreduce (libfsr_b200, captured in the step graph)" if e.comm.native else "torch.distributed.all_reduce"
        res["overlap"] = bool(e.overlap)
        # the two exchanges alone (flat fp32 gradient buffers: D 18.7 MB, G 3.7 MB), device-timed, max over ranks
        ar = {}
        for name, fp in (("d_grads", e.dp), ("g_grads", e.gp)):
            buf = torch.zeros_like(fp.grad)
            for _ in range(3):
                e.comm.allreduce(buf)
            ar[name + "_us"] = _time_steps(lambda: e.comm.allreduce(buf), 20, dev, dist) * 1e3
            ar[name + "_bytes"] = buf.numel() * 4
        res["allreduce"] = ar
        del tr, step
        _, _, ms_anchor, _ = run(32, standalone=True)
        res["n1_anchor_b32_ms"] = ms_anchor
        res["efficiency_vs_n1"] = ms_anchor / ms32
    else:
        # in-situ roofline of the training kernels: ONE eager step (launches are event-bracketed; a graph replay is not)
        e = tr.engine
        e.use_graph = False
        lib.fsr_profile_enable_mask((1 << 6) | (1 << 7) | (1 << 1) | (1 << 5) | (1 << 3))
        step()
        torch.cuda.synchronize()
        prof = read_profile(lib)
        lib.fsr_profile_enable_mask(0)
        tf_peak, _, peak_src = load_peaks()
        kern = {}
        for kid, recs in prof.items():
            t = sum(r[0] for r in recs) * 1e-3
            f = sum(r[1] for r in recs)
            kern[K_NAMES.get(kid, str(kid))] = {"launches": len(recs), "ms": t * 1e3, "achieved_tflops": f / t / 1e12 if t > 0 else None,
                                              "frac_of_peak": f / t / 1e12 / tf_peak if t > 0 else None}
        res["kernels_b32_eager_step"] = kern
        if 6 in prof:
            t = sum(r[0] for r in prof[6]) * 1e-3
            f = sum(r[1] for r in prof[6])
            res["roofline"] = {"bound": "tensor", "kernel": K_NAMES[6], "achieved": f / t / 1e12, "peak": tf_peak, "unit": "TFLOP/s",
                               "frac": f / t / 1e12 / tf_peak, "launches_timed": len(prof[6]), "flops": f, "peak_source": peak_src,
                               "traffic": None, "how": "sum of algorithmic FLOPs / sum of per-launch CUDA-event times over one eager b32 step"}
        del tr, step
        _, _, ms64, closs64 = run(64, standalone=False)
        res["b64"] = {"ms_per_step": ms64, "per_gpu_batch": 64, "global_batch": 64, "samples_per_s": 64 / (ms64 / 1e3),
                      "needed_tflops_per_gpu": FLOPS_B64 / (ms64 * 1e-3) / 1e12, "content_loss": closs64}
    res["ms_per_step"] = res["b64"]["ms_per_step"] if world == 1 else ms32
    return res


_REAL_STDOUT = None


def quiet_stdout():
    """Route fd 1 to stderr while working (NCCL prints its version banner on stdout); emit() restores it so that the
    ONE JSON line is the only thing on stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(line), flush=True)


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dtype", default=os.environ.get("FSR_DTYPE", "fp16"), choices=["fp16", "bf16"])
    ap.add_argument("--l2-group", type=int, default=int(os.environ.get("FSR_L2_GROUP", "0")))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the auxiliary GAN train-step measurement")
    ap.add_argument("--streams", type=int, default=int(os.environ.get("FSR_STREAMS", "1")),
                    help="sub-batches of the forward run concurrently on internal side streams (1 = single stream)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR as .npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA (B200) device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    import types
    from fast_srgan_b200 import _lib as L
    from fast_srgan_b200.model import Generator
    dt = torch.float16 if args.dtype == "fp16" else torch.bfloat16
    torch.manual_seed(1234)                       # reference configs/config.yaml:3; random-init weights (torch default init)
    gen = Generator(types.SimpleNamespace(n_filters=NF, n_layers=NL), compute_dtype=dt)
    gen = gen.to(dev).eval()
    gen.l2_group = args.l2_group
    lib = L.load()
    lib.fsr_set_overlap_streams(args.streams)

    g = torch.Generator().manual_seed(100 + rank)
    x_dev = (torch.rand((BATCH, 3, H, W), generator=g) * 2 - 1).to(dev)
    frames_u8 = torch.randint(0, 256, (BATCH, H, W, 3), generator=g, dtype=torch.uint8)
    h_in = [frames_u8.clone().pin_memory() for _ in range(2)]
    h_out = [torch.empty((BATCH, 4 * H, 4 * W, 3), dtype=torch.uint8).pin_memory() for _ in range(2)]
    d_in = [torch.empty((BATCH, H, W, 3), dtype=torch.uint8, device=dev) for _ in range(2)]
    d_out = [torch.empty((BATCH, 4 * H, 4 * W, 3), dtype=torch.uint8, device=dev) for _ in range(2)]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if dist is None:
            return ms
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    # ---------------- value: device-resident inputs, Generator.forward (fp32 NCHW in/out)
    with torch.no_grad():
        for _ in range(args.warmup):
            y = gen(x_dev)
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        lib.fsr_profile_enable_mask((1 << L.K_CONV_UP) | (1 << L.K_CONV_RES))
        launches0 = lib.fsr_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            y = gen(x_dev)
        e1.record()
        barrier()
        ms_total = max_over_ranks(e0.elapsed_time(e1))
        launches = lib.fsr_launch_count() - launches0
        clocks = sampler.stop() if rank == 0 else None
        prof = read_profile(lib)
        lib.fsr_profile_enable_mask(0)
        dumps = output_sample("sr", y) if args.dump_outputs else {}
    up1_flops = 2.0 * BATCH * (2 * H) * (2 * W) * 64 * 256 * 9
    # two upsampling convs per step: the 360x640 launches are the ones tagged with up1's FLOPs
    up1 = [ms for ms, fl in prof.get(L.K_CONV_UP, []) if abs(fl - up1_flops) < 1e-3 * up1_flops]
    res_ms = [ms for ms, fl in prof.get(L.K_CONV_RES, [])]
    ms_step = ms_total / args.steps
    fps = world * BATCH * args.steps / (ms_total / 1e3)

    # ---------------- e2e: pinned host uint8 frames -> H2D -> super_resolve_u8 -> D2H, double buffered
    copy_in, copy_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    main_s = torch.cuda.current_stream(dev)

    def e2e_loop(n):
        ev_in = [torch.cuda.Event() for _ in range(2)]
        ev_done = [torch.cuda.Event() for _ in range(2)]
        ev_out = [None, None]
        for i in range(n):
            b = i & 1
            with torch.cuda.stream(copy_in):
                if ev_out[b] is not None:
                    copy_in.wait_event(ev_done[b])      # d_in[b] free once compute i-2 finished
                d_in[b].copy_(h_in[b], non_blocking=True)
                ev_in[b].record(copy_in)
            main_s.wait_event(ev_in[b])
            if ev_out[b] is not None:
                main_s.wait_event(ev_out[b])            # d_out[b] drained by D2H of step i-2
            gen.super_resolve_u8(d_in[b], out=d_out[b])
            ev_done[b].record(main_s)
            with torch.cuda.stream(copy_out):
                copy_out.wait_event(ev_done[b])
                h_out[b].copy_(d_out[b], non_blocking=True)
                ev_out[b] = torch.cuda.Event()
                ev_out[b].record(copy_out)
        copy_out.synchronize()

    e2e_loop(max(2, args.warmup))
    barrier()
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record(main_s)
    wall0 = time.perf_counter()
    e2e_loop(args.steps)
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - wall0) * 1e3
    if args.dump_outputs:
        dumps.update(output_sample("sr_u8", h_out[(args.steps - 1) & 1]))
    barrier()
    e2e_ms = max_over_ranks(wall_ms)    # host-visible completion of the last D2H, max over ranks
    e2e_fps = world * BATCH * args.steps / (e2e_ms / 1e3)

    # ---------------- auxiliary: GAN train-step ms (second half of BASELINE's metric string; configs[2]/[3])
    train_aux = None
    if not args.no_train:
        try:
            train_aux = bench_train_step(args, rank, world, dev, dist, lib)
        except Exception as exc:                     # never let the auxiliary number break the headline line
            train_aux = {"error": repr(exc)[:200]}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    tf_peak, hbm_peak, peak_src = load_peaks()
    traffic = load_traffic()
    roof = roof_res = None
    if up1:
        avg = sum(up1) / len(up1)
        ach = up1_flops / (avg * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": "conv3x3_up_2cta_kernel (upsampling.1.conv, 360x640, 64->256, tcgen05 cta_group::2)"
                if os.environ.get("FSR_UP_2CTA", "1") != "0" else "conv3x3_c64_kernel<128,EPI_PS_PRELU> (upsampling.1.conv, 360x640, 64->256)",
                "achieved": ach, "peak": tf_peak, "unit": "TFLOP/s", "frac": ach / tf_peak,
                "traffic": traffic.get("conv_up1_bytes_per_launch"), "traffic_source": traffic.get("_source"),
                "algorithmic_bytes": BATCH * (2 * H) * (2 * W) * 64 * 2 * 5 + 9 * 256 * 64 * 2,
                "avg_launch_ms": avg, "launches_timed": len(up1), "flops_per_launch": up1_flops, "peak_source": peak_src}
    if res_ms:
        # the north_star's 70 % kernel: the 64->64 residual-block convs (17 per forward: plain, fused bn1+relu1 input,
        # fused bn2+skip input), all launches of the timed region
        res_flops = 2.0 * BATCH * H * W * 64 * 64 * 9
        avg = sum(res_ms) / len(res_ms)
        ach = res_flops / (avg * 1e-3) / 1e12
        roof_res = {"bound": "tensor", "kernel": "conv3x3_c64_kernel<64,RAW_STATS,XF=0|1|2> (17 residual-chain convs per forward, 180x320, 64->64)",
                    "achieved": ach, "peak": tf_peak, "unit": "TFLOP/s", "frac": ach / tf_peak,
                    "traffic": traffic.get("conv_res_bytes_per_launch"), "traffic_source": traffic.get("_source"),
                    "avg_launch_ms": avg, "launches_timed": len(res_ms), "flops_per_launch": res_flops, "peak_source": peak_src,
                    "note": "the fused variants also do the InstanceNorm(+PReLU | +skip) pass of their input inside this time"}
    total_flops = gen_flops_per_frame(H, W) * BATCH
    line = {
        "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": args.dtype + " operands, fp32 accumulate", "data": "synthetic",
        "config": {"workload": f"generator-only 4x SR {H}x{W}->{4*H}x{4*W}, batch {BATCH}/GPU, L={NL} F={NF} (BASELINE configs[1])",
                   "parallelism": f"{world} independent replicas (frames shard, no collective)",
                   "l2": "activations streamed per step (>5 GB) exceed the 126 MB L2; no explicit flush",
                   "l2_group": args.l2_group, "overlap_streams": args.streams,
                   "switches": {k: os.environ.get(k, "default") for k in ("FSR_FUSE_IN", "FSR_FUSE_RES", "FSR_UP_2CTA", "FSR_GEN_WS", "FSR_SMALL_MMA", "FSR_WS", "FSR_HALO1")}},
        "whole_model_tflops": total_flops / (ms_step * 1e-3) / 1e12 * 1.0,
        "clocks": clocks, "gpu_launches": int(launches),
        "e2e": {"value": e2e_fps, "unit": UNIT, "h2d_bytes_per_step": BATCH * H * W * 3,
                "d2h_bytes_per_step": BATCH * 16 * H * W * 3, "api": "Generator.super_resolve_u8 (uint8 NHWC host frames in/out)",
                "ms_per_step": e2e_ms / args.steps},
        "roofline": roof,
        "roofline_resblock_conv": roof_res,
        "train_step": train_aux,
    }
    if not args.no_cpu_baseline and world == 1:
        cfps, cthreads, csample, ckind = cpu_generator_fps()
        line["cpu_baseline"] = {"value": cfps, "unit": UNIT, "cores": cthreads, "kind": ckind, "sample": csample}
    if dist is not None:
        dist.destroy_process_group()
    if args.dump_outputs:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumps.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    emit(line)


if __name__ == "__main__":
    main()
