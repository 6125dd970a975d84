#!/usr/bin/env python
"""bench.py -- images/sec of the Theia distillation step (BASELINE.json metric) on N B200 GPUs.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the UNMODIFIED reference (oracle/_ref) on the host cores
    python bench.py --impl eager ...          # the same reference modules through torch eager on one B200

One step = train_rvfm.py:116-133 on one synthetic batch: forward (pre-process, DeiT student, lconv
translator heads) -> get_loss -> main_loss = 0.9 cos + 0.1 smooth-l1 -> backward -> AdamW step,
through the public `RobotVisionFM` API.  Prints ONE JSON line (rank 0).  --dump-outputs DIR also writes what the
last timed step computed as DIR/*.npy (see dump_outputs), to compare two builds on identical seeded inputs.
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "images/sec (224^2, bf16) Theia-base cdiv distill step"
BACKBONES = {"tiny": "facebook/deit-tiny-patch16-224", "small": "facebook/deit-small-patch16-224",
             "base": "facebook/deit-base-patch16-224"}


def fwd_gflop_per_image(D: int, teachers: dict) -> tuple[float, float]:
    """SURVEY section 8d algorithmic forward FLOPs per image: (total, attention-only part)."""
    N, P = 197, 196
    attn = 12 * 4 * N * N * D
    back = 2 * P * 768 * D + 12 * 24 * N * D * D + attn
    tr = 0
    for c, h, w in teachers.values():
        if h == 16:
            tr += 2 * 196 * 9 * D * D + 2 * (2 * 256 * 9 * D * D) + 2 * 256 * D * c
        else:
            tr += 2 * 196 * 9 * D * D + 2 * 256 * 9 * D * D + 2 * 961 * 9 * D * D + 2 * 4096 * D * c
    return (back + tr) / 1e9, attn / 1e9


def measured_peaks() -> tuple[dict, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "200", "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self) -> dict:
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def usable_cpus():
    """Logical CPUs this process may run on (affinity mask and cgroup quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q = open("/sys/fs/cgroup/cpu.max").read().split()
        if q[0] != "max":
            n = min(n, max(1, int(float(q[0]) / float(q[1]))))
    except (OSError, ValueError, IndexError):
        try:
            quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota > 0:
                n = min(n, max(1, quota // period))
        except (OSError, ValueError):
            pass
    return max(1, n)


def pick_cpu_threads(probe):
    """The thread count the CPU arm runs with: the fastest of {all, 1/2, 1/4, 1/8 of the usable CPUs} on a
    one-image probe step.  On a shared two-socket hyper-threaded host "all logical CPUs" can be an order of
    magnitude slower than the physical cores of one socket; the reference gets the best of them.
    Returns (threads, seconds of the best probe, {threads: seconds})."""
    n = usable_cpus()
    cand = sorted({max(1, n // d) for d in (1, 2, 4, 8)}, reverse=True)
    timings = {}
    for t in cand:
        torch.set_num_threads(t)
        probe()  # warm this thread count (pool start-up, first-touch)
        t0 = time.perf_counter()
        probe()
        timings[t] = time.perf_counter() - t0
    best = min(timings, key=timings.get)
    torch.set_num_threads(best)
    return best, timings[best], timings


def build_reference_module(cfgO, O, backbone, device):
    """The UNMODIFIED reference `RobotVisionFM` (oracle/_ref, the pip-installed copy build() makes) with the
    oracle's deterministic weights, or None when that copy is absent."""
    try:
        from baseline import ref_shim
        Ref = ref_shim.import_reference()
    except Exception:
        return None
    ref = Ref(backbone=backbone, pretrained=False, translator="lconv", target_feature_sizes=dict(cfgO.teachers),
              translator_kwargs={"hidden_size_factor": 1.0})
    ref.load_state_dict(O.init_params(cfgO, seed=0))
    return ref.to(device).train()


def reference_step_fn(ref, cfgO, O, B, device, autocast=False, lr=1e-4):
    """train_rvfm.py:101-133 on one synthetic batch with the reference's own module, loss and torch AdamW
    (two weight-decay groups of optimizers/utils.py:8-35)."""
    decay, no_decay = [], []
    for n, p in ref.named_parameters():
        (no_decay if (p.ndim <= 1 or n.endswith(".bias")) else decay).append(p)
    opt = torch.optim.AdamW([{"params": no_decay, "weight_decay": 0.0}, {"params": decay, "weight_decay": 0.01}],
                            lr=lr, betas=(0.9, 0.999))
    images, targets = O.synthetic_batch(cfgO, B, seed=0)
    tb = {t: v.to(torch.bfloat16) for t, v in targets.items()}

    def step():
        im = images.to(device)                                    # train_rvfm.py:101
        tg = {t: v.to(device).float() for t, v in tb.items()}    # :107-114
        with torch.autocast(device_type="cuda", dtype=torch.bfloat16, enabled=autocast):
            pred = ref(im, do_resize=False)                       # :116
            losses = ref.get_loss(pred, tg)                       # :117
            ml = 0.9 * losses["cos_loss"] + 0.1 * losses["l1_loss"]  # :119-122
        opt.zero_grad()
        ml.backward()
        opt.step()
        return float(ml.detach())
    return step


def run_reference(args, cfgO, O):
    """The reference's own CPU implementation of the step on the host cores: the UNMODIFIED reference modules from
    oracle/_ref (kind "reference"); the oracle port only when that copy is absent (kind "port")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    backbone = BACKBONES[args.backbone]
    ref = build_reference_module(cfgO, O, backbone, "cpu")
    kind = "reference" if ref is not None else "port"
    if ref is not None:
        def make_step(B):
            return reference_step_fn(ref, cfgO, O, B, "cpu")
    else:
        P = O.init_params(cfgO, seed=0)
        params = {k: v.clone().requires_grad_(True) for k, v in P.items()}
        opt = torch.optim.AdamW(list(params.values()), lr=1e-4, weight_decay=0.01)

        def make_step(B):
            images, targets = O.synthetic_batch(cfgO, B, seed=0)

            def step():
                preds = O.forward(params, images, cfgO, do_resize=False)
                losses = O.get_loss(preds, targets)
                ml = O.main_loss(losses)
                opt.zero_grad()
                ml.backward()
                opt.step()
                return float(ml.detach())
            return step

    # Bounded sample: the per-step batch is sized from a one-image probe step so that the whole
    # --steps K --warmup W run stays within THEIA_REF_BUDGET_S seconds (default 240) on this host.
    budget = float(os.environ.get("THEIA_REF_BUDGET_S", "240"))
    probe = make_step(1)
    cores, t1, thread_timings = pick_cpu_threads(probe)
    B = max(1, min(args.cpu_batch, int(budget / (max(args.steps + args.warmup, 1) * t1))))
    step = make_step(B)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    val = B / dt
    what = ("UNMODIFIED reference RobotVisionFM (oracle/_ref) + torch AdamW, fp32 CPU" if kind == "reference"
            else "oracle port (torch fp32 CPU; oracle/_ref absent)")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "images/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, B),
            "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": kind,
                             "sample": f"{what}: fwd+loss+bwd+AdamW, batch {B} per step (sized from a 1-image probe of "
                                       f"{t1:.2f} s for a {budget:.0f} s budget), {args.steps} timed steps; threads chosen from "
                                       f"{ {k: round(v, 2) for k, v in thread_timings.items()} } s/probe"},
            "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def gpu_eager_leg(args, cfgO, O, dev, steps=3):
    """The meaningful GPU comparator (SURVEY 8d / BASELINE.md section 3): the reference's own modules run by torch
    eager (cuBLAS / cuDNN / ATen) on the SAME B200, same replayed step and batch, in fp32 (as the reference trains)
    and under autocast(bfloat16).  Returns None when oracle/_ref is absent."""
    out = {}
    for mode in ("fp32", "autocast_bf16"):
        ref = build_reference_module(cfgO, O, BACKBONES[args.backbone], dev)
        if ref is None:
            return None
        B = args.batch
        try:
            step = reference_step_fn(ref, cfgO, O, B, dev, autocast=(mode == "autocast_bf16"))
            for _ in range(2):
                step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[mode] = {"value": B / (ms / 1e3), "unit": "images/s", "ms_per_step": ms, "batch": B, "steps": steps}
        except torch.cuda.OutOfMemoryError:
            out[mode] = {"value": None, "note": f"out of memory at batch {B}"}
        del ref
        torch.cuda.empty_cache()
    out["what"] = ("UNMODIFIED reference RobotVisionFM (oracle/_ref) on this GPU through torch eager "
                   "(cuBLAS/cuDNN/ATen), fwd+get_loss+bwd+torch AdamW; inputs copied from host each step as "
                   "train_rvfm.py:101-114 does; matmul TF32 off (torch default), cuDNN conv TF32 on (torch default)")
    return out


def cpu_baseline_leg(args, cfgO, O):
    """`cpu_baseline` of the GPU arm: the reference's CPU path timed on the host cores on a bounded sample
    (full steps -- forward, loss, backward, AdamW -- at --cpu-batch images)."""
    Bc = args.cpu_batch
    ref = build_reference_module(cfgO, O, BACKBONES[args.backbone], "cpu")
    kind = "reference" if ref is not None else "port"
    if ref is not None:
        probe = reference_step_fn(ref, cfgO, O, 1, "cpu")
        step = reference_step_fn(ref, cfgO, O, Bc, "cpu")
    else:
        Pc = O.init_params(cfgO, seed=0)
        i1, t1_ = O.synthetic_batch(cfgO, 1, seed=0)
        ic, tc = O.synthetic_batch(cfgO, Bc, seed=0)
        probe = lambda: O.distill_step(Pc, i1, t1_, cfgO, do_resize=False)  # noqa: E731
        step = lambda: O.distill_step(Pc, ic, tc, cfgO, do_resize=False)  # noqa: E731
    cores, _, thread_timings = pick_cpu_threads(probe)
    step()  # warm-up
    nrep = 3
    t0 = time.perf_counter()
    for _ in range(nrep):
        step()
    dt = (time.perf_counter() - t0) / nrep
    what = ("UNMODIFIED reference RobotVisionFM (oracle/_ref), fp32 CPU: fwd+loss+bwd+AdamW" if kind == "reference"
            else "oracle port (torch fp32 CPU): fwd+loss+bwd")
    return {"value": Bc / dt, "unit": "images/s", "cores": cores, "kind": kind,
            "sample": f"{what}, batch {Bc}, {nrep} timed steps; threads chosen from "
                      f"{ {k: round(v, 2) for k, v in thread_timings.items()} } s per 1-image probe"}


def parity_check(model, cfgO, O, d_images, d_targets, dev, n=4):
    """Step-0 check of the benchmarked configuration against the fp32 oracle (same weights, first n images of the
    batch, oracle run on this GPU in fp32): the three loss scalars and the predictions.  Raises on a miss."""
    P = {k: v.detach().clone() for k, v in model.state_dict().items()}
    im = d_images[:n]
    tg = {t: v[:n].float() for t, v in d_targets.items()}
    with torch.no_grad():
        pred = model(im, do_resize=False)
        losses = model.get_loss(pred, tg)
        pred_o = O.forward(P, im, cfgO, do_resize=False)
        losses_o = O.get_loss(pred_o, tg)
    out = {"images": n, "against": "oracle (torch fp32 on this GPU, TF32 off), identical weights and inputs"}
    worst = 0.0
    for k in ("mse_loss", "cos_loss", "l1_loss"):
        a, b = float(losses[k]), float(losses_o[k])
        out[k] = {"ours": a, "oracle": b, "rel": abs(a - b) / abs(b)}
        worst = max(worst, out[k]["rel"])
    pr = 0.0
    for t in pred:
        pr = max(pr, ((pred[t].double() - pred_o[t].double()).norm() / pred_o[t].double().norm()).item())
    out["pred_rel_l2_max"] = pr
    out["loss_rel_max"] = worst
    out["tolerance"] = {"loss_rel": 1e-3, "pred_rel_l2": 3e-2}
    out["ok"] = bool(worst <= 1e-3 and pr <= 3e-2)
    if not out["ok"]:
        raise SystemExit("bench.py parity check FAILED: " + json.dumps(out))
    return out


DUMP_SAMPLE = 1 << 20  # elements kept of each large array (4 MiB each, 20 MiB for the three cdiv teachers)


def dump_outputs(out_dir, model, last):
    """What the last timed step handed its caller, as float32 / float64 .npy files: pred_<teacher> (predictions),
    main_loss / mse_loss / cos_loss / l1_loss, loss_<teacher> (that teacher's mse, cos and l1 loss), grads (the
    step's parameter gradients) and params (the parameters after the AdamW update), both in model.parameters() order.
    That step starts from the seeded initial weights and optimizer state (see timed_step in main).
    Arrays above DUMP_SAMPLE elements keep the same seeded sample of positions on every run, so that two builds can
    be compared element by element."""
    import numpy as np

    def sample(t):
        f = t.detach().flatten()
        if f.numel() > DUMP_SAMPLE:
            idx = torch.randint(0, f.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0))
            f = f[idx.sort().values.to(f.device)]
        return f.float().cpu().numpy()

    def fname(t):
        return t.replace("/", "_")

    losses = last["losses"]
    arrays = {"pred_" + fname(t): sample(v) for t, v in last["pred"].items()}
    for k in ("main_loss", "mse_loss", "cos_loss", "l1_loss"):
        arrays[k] = np.array(float(last["main_loss"] if k == "main_loss" else losses[k]), dtype=np.float64)
    for t in last["pred"]:
        arrays["loss_" + fname(t)] = np.array([losses[k + "_losses_per_model"][t] for k in ("mse", "cos", "l1")],
                                              dtype=np.float64)
    params = list(model.parameters())
    arrays["grads"] = sample(torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).flatten()
                                        for p in params]))
    arrays["params"] = sample(torch.cat([p.detach().flatten() for p in params]))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_config(args, B):
    return {"workload": f"theia-{args.backbone} {args.teachers} distill step (fwd+loss+bwd+AdamW), per-GPU batch {B}, "
                        f"224x224x3 uint8 -> {args.teachers} teacher targets",
            "backbone": BACKBONES[args.backbone], "teachers": args.teachers, "per_gpu_batch": B,
            "global_batch": B * args.gpus, "main_loss": "cos_l1", "optimizer": "AdamW (" + getattr(args, "optimizer", "flat") + ")",
            "preprocess": "rescale+normalize in-kernel, do_resize=False on both arms",
            "l2_policy": "per-step working set (>10 GB of activations at batch 256) far exceeds the 126 MB L2",
            "parallelism": f"dp{args.gpus}" + ("" if args.gpus == 1 else
                                               (" (one flat-buffer NCCL all-reduce per step)" if getattr(args, "dp_mode", "flat") == "flat"
                                                else " (torch DDP wrapper, bucketed all-reduce)"))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "eager"])
    ap.add_argument("--backbone", default="base", choices=list(BACKBONES))
    ap.add_argument("--teachers", default="cdiv")
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--cpu-batch", type=int, default=8)
    ap.add_argument("--no-eager", action="store_true", help="skip the torch-eager-on-this-GPU comparator leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the step-0 parity check against the oracle")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dp-mode", default="flat", choices=["flat", "ddp"],
                    help="N>1: one flat-buffer NCCL all-reduce issued by the module (default) or the reference's DDP wrapper")
    ap.add_argument("--optimizer", default="flat", choices=["flat", "torch"],
                    help="flat = theia_b200.optim.FlatAdamW (one fused pass over the flat buffers); torch = torch.optim.AdamW(fused=True)")
    ap.add_argument("--gemm-csv", default=None, help="dump per-launch GEMM timings of the timed region")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step computed (predictions, losses, gradients, updated "
                         "parameters; fixed seeded samples of the large arrays) as DIR/<name>.npy; that step "
                         "starts from the seeded initial weights and optimizer state")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the CUDA path computed: it needs --impl ours")

    from oracle import theia_oracle as O  # checker / CPU baseline only
    cfgO = O.make_config(BACKBONES[args.backbone], args.teachers)
    if args.impl == "reference":
        args.warmup = min(args.warmup, 1)
        run_reference(args, cfgO, O)
        return
    if args.impl == "eager":
        if int(os.environ.get("RANK", "0")) == 0:
            torch.cuda.set_device(0)
            eg = gpu_eager_leg(args, cfgO, O, torch.device("cuda", 0), steps=args.steps)
            print(json.dumps({"impl": "eager", "metric": METRIC, "unit": "images/s", "n_gpus": 1,
                              "config": workload_config(args, args.batch), "gpu_eager_baseline": eg}), flush=True)
        return

    import torch.distributed as dist
    from theia_b200 import RobotVisionFM, _lib
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"  # keep stdout to the one JSON line (the image sets NCCL_DEBUG=VERSION)
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.lib()

    B = args.batch
    torch.manual_seed(0)
    model = RobotVisionFM(backbone=BACKBONES[args.backbone], translator="lconv",
                          target_feature_sizes=dict(cfgO.teachers), translator_kwargs={"hidden_size_factor": 1.0},
                          max_batch=B).to(dev)
    model.train()
    net = model
    if world > 1 and args.dp_mode == "ddp":
        from torch.nn.parallel import DistributedDataParallel as DDP
        net = DDP(model, device_ids=[local], find_unused_parameters=False)  # train_rvfm.py:258
    elif world > 1:
        dist.broadcast(model._flat, 0)  # what DDP's constructor does: rank 0's parameters everywhere
        model.sync_gradients(True)      # single all-reduce (avg) over the flat gradient buffer inside backward()
    # lr rule of train_rvfm.py:299-301
    lr = 2e-3 * (B * world) / (64 * 8)
    decay, no_decay = [], []
    for n, p in model.named_parameters():  # optimizers/utils.py:26-33
        (no_decay if (p.ndim <= 1 or n.endswith(".bias")) else decay).append(p)
    if args.optimizer == "flat":
        from theia_b200.optim import FlatAdamW
        opt = FlatAdamW(model, lr=lr, betas=(0.9, 0.999), weight_decay=0.01)  # same two decay groups, fused pass
    else:
        opt = torch.optim.AdamW([{"params": no_decay, "weight_decay": 0.0}, {"params": decay, "weight_decay": 0.01}],
                                lr=lr, betas=(0.9, 0.999), fused=True)

    # synthetic data (SURVEY 8d): pinned host copies for the e2e leg, device copies for `value`
    g = torch.Generator().manual_seed(1000 + rank)
    h_images = torch.randint(0, 256, (B, 224, 224, 3), dtype=torch.uint8, generator=g).pin_memory()
    g2 = torch.Generator().manual_seed(2000 + rank)
    h_targets = {t: torch.randn((B, h * w, c), generator=g2).to(torch.bfloat16).pin_memory()
                 for t, (c, h, w) in cfgO.teachers.items()}  # bf16, as the reference's dataloader yields them
    d_images = h_images.to(dev)
    d_targets = {t: v.to(dev) for t, v in h_targets.items()}

    last = {}  # the last step's results, kept only for --dump-outputs

    def step(images, targets):
        pred = net(images, do_resize=False)
        losses = model.get_loss(pred, targets)  # returns python floats per teacher (one D2H), like the reference
        main_loss = 0.9 * losses["cos_loss"] + 0.1 * losses["l1_loss"]
        opt.zero_grad(set_to_none=True)
        main_loss.backward()
        opt.step()
        if args.dump_outputs:
            last.update(pred=pred, losses=losses, main_loss=main_loss)
        return losses

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms

    start = None
    if args.dump_outputs:  # the state the first step starts from
        start = (model._flat.detach().clone(), copy.deepcopy(opt.state_dict()))
    parity = None
    if rank == 0 and not args.no_parity:
        parity = parity_check(model, cfgO, O, d_images, d_targets, dev)
    for _ in range(max(args.warmup, 3)):
        step(d_images, d_targets)
    # ---- device-resident timed region (value) with per-GEMM-launch events for the roofline ----
    sampler = ClockSampler(local) if rank == 0 else None
    n0 = lib.theia_launch_count()
    _lib.check(lib.theia_prof_enable(1))

    reset = []

    def timed_step(i):
        if start is not None and i == args.steps - 1:
            # the fp32 atomics of the CUDA path sum in a different order on each run and every AdamW step on the
            # synthetic batch amplifies that noise, so the step whose outputs are dumped starts again from the
            # seeded initial weights and a fresh optimizer: its inputs are then identical from run to run.  The
            # restore and the re-pack of the restored weights are timed apart and left out of `value`.
            reset[:] = [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)]
            reset[0].record()
            with torch.no_grad():
                model._flat.copy_(start[0])
            opt.load_state_dict(start[1])
            model._ensure(B)
            reset[1].record()
        step(d_images, d_targets)

    ms = timed(timed_step, args.steps)
    reset_ms = reset[0].elapsed_time(reset[1]) if reset else 0.0  # timed() ended in a synchronize
    if world > 1:
        t = torch.tensor([reset_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        reset_ms = float(t)
    ms -= reset_ms
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model, last)  # before the e2e leg steps the model further
    import ctypes as C
    pm, pf, pn = C.c_double(), C.c_double(), C.c_longlong()
    if args.gemm_csv and rank == 0:
        torch.cuda.synchronize()
        with open(args.gemm_csv, "w") as f:
            f.write("idx,ms,M,N,K,a_mode,b_mode,epi,splits_z,BN,tflops\n")
            i = 0
            ms1, meta = C.c_double(), (C.c_int * 8)()
            while lib.theia_prof_record(i, C.byref(ms1), meta) == 0:
                z = meta[6] % 1000
                fl = 2.0 * meta[0] * meta[1] * meta[2] * z
                f.write(f"{i},{ms1.value:.5f},{meta[0]},{meta[1]},{meta[2]},{meta[3]},{meta[4]},{meta[5]},{meta[6]},"
                        f"{meta[7]},{fl / (ms1.value * 1e-3) / 1e12 if ms1.value > 0 else 0:.1f}\n")
                i += 1
    _lib.check(lib.theia_prof_collect(C.byref(pm), C.byref(pf), C.byref(pn)))
    _lib.check(lib.theia_prof_enable(0))
    launches = lib.theia_launch_count() - n0
    clocks = sampler.stop() if sampler else None
    ms_step = ms / args.steps
    value = B * world / (ms_step / 1e3)

    # ---- end-to-end: pinned host buffers -> H2D on a copy stream (prefetched one step ahead) ----
    e2e = None
    if not args.no_e2e:
        copy_stream = torch.cuda.Stream()
        bufs = [None, None]

        def prefetch(slot):
            with torch.cuda.stream(copy_stream):
                im = h_images.to(dev, non_blocking=True)
                tg = {t: v.to(dev, non_blocking=True) for t, v in h_targets.items()}
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            bufs[slot] = (im, tg, ev)

        def e2e_step(i):
            if bufs[i % 2] is None:
                prefetch(i % 2)
            im, tg, ev = bufs[i % 2]
            bufs[i % 2] = None
            prefetch((i + 1) % 2)  # next step's inputs travel while this step computes
            torch.cuda.current_stream().wait_event(ev)
            losses = step(im, tg)
            for t_ in tg.values():
                t_.record_stream(torch.cuda.current_stream())
            im.record_stream(torch.cuda.current_stream())
            return losses  # per-teacher python floats were read back (D2H) inside get_loss

        for i in range(2):
            e2e_step(i)
        bufs = [None, None]
        ms2 = timed(e2e_step, args.steps) / args.steps
        h2d = h_images.numel() + sum(v.numel() * 2 for v in h_targets.values())
        e2e = {"value": B * world / (ms2 / 1e3), "unit": "images/s", "ms_per_step": ms2,
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(len(h_targets) * 3 * 4),
               "note": "pinned host uint8 images + bf16 targets copied every step on a copy stream, prefetched "
                       "one step ahead; loss scalars read back to host every step"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    fwd_g, attn_g = fwd_gflop_per_image(cfgO.hidden, cfgO.teachers)
    peaks, peak_src = measured_peaks()
    gemm_ms_step = pm.value / args.steps
    gemm_alg_tflop = 3.0 * (fwd_g - attn_g) * B / 1e3  # algorithmic GEMM/conv FLOPs of one step (3x forward)
    achieved = gemm_alg_tflop / (gemm_ms_step / 1e3) if gemm_ms_step > 0 else 0.0
    peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if not os.path.exists(tpath):
        tpath = os.path.join(ROOT, "profiles", "r01_traffic.json")
    if os.path.exists(tpath) and args.backbone == "base":
        traffic = json.load(open(tpath)).get("traffic_bytes_per_launch_mean")  # ncu --set full capture, see profiles/
    roofline = {"bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05 GEMM / implicit-GEMM conv, all instances)",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic,
                "peak_source": peak_src + ", sustained figure (kernel timed inside a long step)",
                "launches_per_step": pn.value / args.steps, "kernel_ms_per_step": gemm_ms_step,
                "kernel_share_of_step": gemm_ms_step / ms_step,
                "executed_tflops": pf.value / args.steps / 1e12 / (gemm_ms_step / 1e3) if gemm_ms_step > 0 else 0.0,
                "step_tflops_all_kernels": 3.0 * fwd_g * B / 1e3 / (ms_step / 1e3),
                "step_frac_of_peak": 3.0 * fwd_g * B / 1e3 / (ms_step / 1e3) / peak}

    cpu = cpu_baseline_leg(args, cfgO, O) if (world == 1 and not args.no_cpu_baseline) else None
    eager = None
    if world == 1 and not args.no_eager:
        del model, net, opt
        torch.cuda.empty_cache()
        eager = gpu_eager_leg(args, cfgO, O, dev)

    line = {"metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": workload_config(args, B),
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
            "gpu_eager_baseline": eager, "parity_check": parity}
    if args.dump_outputs:
        line["dump_outputs"] = {"dir": args.dump_outputs, "reset_ms_excluded": reset_ms,
                                "note": "the last timed step started from the seeded initial weights and optimizer "
                                        "state; restoring them took reset_ms_excluded, left out of value"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
