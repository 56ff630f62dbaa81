#!/usr/bin/env python
"""bench.py -- FNO2d train samples/sec on B200 (BASELINE.json metric), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B_per_gpu] [--impl ours|reference] [--config 1..5]

--config selects the BASELINE.json configuration (default 1 = configs[0], the workload the metric is quoted on):
  1  FNO2d m12 w20, 2-D diffusion-reaction 128x128x2ch                      (per-GPU batch 128)
  2  fno_aux two-head FNO2d, joint step: primary + 3 auxiliary samples per item, loss = p + 0.7 a, three Adam groups
  3  FNO2d m16 w64, 2-D incompressible NS 256x256x3ch                         (per-GPU batch 32)
  4  FNO3d m12 w20, 3-D compressible NS 64^3 x 5ch                            (per-GPU batch 4)
  5  config-3 model, data-parallel GLOBAL batch sweep 64..1024 + autoregressive rollout evaluation (rollout_test 5)

Workload (config.workload): BASELINE.json configs[0] -- FNO2d(modes 12, width 20, initial_step 10,
2 channels) on 2-D diffusion-reaction-shaped 128x128 fields, one full training step exactly as
fno/train.py:264-278 (forward, nRMSE loss, backward, adaptive grad-norm clip, Adam(wd 1e-4),
cosine LR), synthetic data, random-init weights (seed 16).  fp32 end to end.

Keys beyond the base contract:
  value     whole-job samples/s with inputs already resident in HBM (device-timed, max over ranks)
  e2e       same metric through the public module API with HOST pinned inputs: per step an H2D
            copy of (xx, yy, grid) and a D2H read of the loss, copies prefetched on a side stream
  roofline  the dominant libfno_sm100 kernel: algorithmic bytes per launch / its mean launch time
            (CUDA events on the launching stream, measured live in a separate instrumented pass)
            against MEASURED_PEAKS.json's HBM copy bandwidth
  cpu_baseline  the oracle port of the reference step (oracle/fno_port.py) on the host cores
  --impl reference: times that CPU port alone (rank 0 only under torchrun).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
for _p in (ROOT, ROOT / "sciml-pde_b200"):
    if str(_p) not in sys.path:
        sys.path.insert(0, str(_p))

import torch  # noqa: E402

WORKLOADS = {
    1: dict(kind="fno2d", ctor=dict(num_channels=2, modes1=12, modes2=12, width=20, initial_step=10), res=128, nd=2, batch=128,
            name="FNO2d m12 w20 init10, 2D diffusion-reaction 128x128x2ch (BASELINE configs[0]), full train step"),
    2: dict(kind="aux2d", ctor=dict(num_channels=2, modes1=12, modes2=12, width=20, initial_step=10), res=128, nd=2, batch=32,
            num_aux=3, aux_w=0.7, lr_share=1e-3, lr_fc2=2e-3,
            name="fno_aux FNO2d m12 w20 joint step: 128x128x2ch primary + 3 auxiliary samples per item, loss = p + 0.7 a "
                 "(BASELINE configs[1]); samples = primary items"),
    3: dict(kind="fno2d", ctor=dict(num_channels=3, modes1=16, modes2=16, width=64, initial_step=10), res=256, nd=2, batch=32,
            name="FNO2d m16 w64 init10, 2D incompressible NS 256x256x3ch (BASELINE configs[2]), full train step"),
    4: dict(kind="fno3d", ctor=dict(num_channels=5, modes1=12, modes2=12, modes3=12, width=20, initial_step=10), res=64, nd=3,
            batch=4, name="FNO3d m12 w20 init10, 3D compressible NS 64^3x5ch (BASELINE configs[3]), full train step"),
}
WORKLOADS[5] = dict(WORKLOADS[3], name="FNO2d m16 w64 256x256x3ch, data-parallel global-batch sweep 64..1024 + rollout eval "
                                       "(BASELINE configs[4])")
WL = WORKLOADS[1]
CFG = WL["ctor"]
RES = WL["res"]
WORKLOAD = WL["name"]
METRIC = "FNO2d train samples/sec"


def select_workload(n: int):
    global WL, CFG, RES, WORKLOAD
    WL = WORKLOADS[n]
    CFG, RES, WORKLOAD = WL["ctor"], WL["res"], WL["name"]


def make_model():
    from fno_b200 import fno, fno_aux
    return {"fno2d": fno.FNO2d, "fno3d": fno.FNO3d, "aux2d": fno_aux.FNO2d}[WL["kind"]](**CFG)


def make_batch(batch: int, seed: int):
    """One batch in the loaders' layout: (xx, yy, grid) or, for the joint step, (xx, yy, grid, xx_aux, yy_aux, grid_aux)
    with the auxiliary tensors already flattened to [B * num_aux, ...] (fno_train_aux.py:251-256)."""
    from fno_b200 import data
    xx, yy, grid = data.synthetic_batch(batch, RES, CFG["initial_step"], CFG["num_channels"], seed=seed, nd=WL["nd"])
    if WL["kind"] != "aux2d":
        return xx, yy, grid
    na = WL["num_aux"]
    xa, ya, ga = data.synthetic_batch(batch * na, RES, CFG["initial_step"], CFG["num_channels"], seed=seed + 500, nd=2)
    return xx, yy, grid, xa, ya, ga


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (weak scaling); 0 = the configuration's default")
    ap.add_argument("--config", type=int, default=1, choices=[1, 2, 3, 4, 5], help="BASELINE.json configuration (see above)")
    ap.add_argument("--dp-eager", action="store_true",
                    help="data-parallel runs: eager step with hook-issued, overlapped all-reduces instead of two CUDA "
                         "graphs around inline bucket all-reduces")
    ap.add_argument("--no-torch-gpu", action="store_true", help="skip the stock-PyTorch-on-the-same-GPU baseline")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-batch", type=int, default=0,
                    help="batch of the bounded CPU sample (0 = the GPU arm's per-GPU batch, capped so that the CPU leg "
                         "stays within ~30 s)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--tail", default="graph", choices=["torch", "fused", "graph"],
                    help="step tail: torch library ops / fused device-side tail / fused + whole step in one CUDA graph "
                         "(graph applies to single-GPU runs; data-parallel runs use the fused eager tail)")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference training step
# ------------------------------------------------------------------------------------------------
def _ref_modules():
    """The reference's own model classes from the verbatim copies under oracle/_ref (oracle/build_ref.py), or None."""
    ref = ROOT / "oracle" / "_ref"
    if not (ref / "fno" / "fno.py").exists():
        return None
    if str(ref) not in sys.path:
        sys.path.insert(0, str(ref))
    import importlib
    return importlib.import_module("fno.fno"), importlib.import_module("fno_aux.fno_aux")


def reference_step_fn(device, batch: int):
    """(step(), kind): one full training step of the REFERENCE algorithm on `device` through stock PyTorch -- the
    reference's own nn.Module (oracle/_ref, kind "reference") when its files are there, else the functional port
    (oracle/fno_port.py, kind "port"); nRMSE loss and the train.py:271-278 tail in both cases.  TF32 off."""
    from oracle import fno_port as P

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.manual_seed(16)
    mods = _ref_modules()
    batch_t = tuple(t.to(device) for t in make_batch(batch, 0))
    if mods is not None:
        cls = {"fno2d": mods[0].FNO2d, "fno3d": mods[0].FNO3d, "aux2d": mods[1].FNO2d}[WL["kind"]]
        model = cls(**CFG).to(device)
        leaves = list(model.parameters())
        fwd = lambda *a: model(*a)                                          # noqa: E731
        kind = "reference"
    else:
        if WL["kind"] == "aux2d":
            raise RuntimeError("the joint-step baseline needs oracle/_ref (python oracle/build_ref.py)")
        modes = tuple(CFG[k] for k in ("modes1", "modes2", "modes3") if k in CFG)
        params = P.as_leaves(P.init_params(WL["nd"], CFG["num_channels"], modes, CFG["width"], CFG["initial_step"]))
        params = {k: v.to(device).detach().requires_grad_(v.requires_grad) for k, v in params.items()}
        leaves = [v for v in params.values() if v.requires_grad]
        fwd = lambda x, g: P.fno_forward(params, x, g)                      # noqa: E731
        kind = "port"
    opt = torch.optim.Adam(leaves, lr=1e-3, weight_decay=1e-4)
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=1000)

    def step():
        if WL["kind"] == "aux2d":
            xx, yy, grid, xa, ya, ga = batch_t
            op, oa = fwd(xx, grid, xa, ga)
            loss = P.nrmse(op, yy).mean() + WL["aux_w"] * P.nrmse(oa, ya).mean()
        else:
            xx, yy, grid = batch_t
            loss = P.nrmse(fwd(xx, grid), yy).mean()
        P.train_step_tail(loss, leaves, opt, sched)
        return loss.detach()

    return step, kind


def cpu_batch_for(args, gpu_batch: int, steps: int) -> int:
    """Per-step batch of the CPU leg: the GPU arm's per-GPU batch when the whole leg (steps + warm-up) stays bounded
    (about 90 samples/s on 16 host cores at config 1), else the largest batch that does."""
    if args.cpu_batch > 0:
        return args.cpu_batch
    budget = {1: 4000, 2: 500, 3: 200, 4: 40, 5: 200}[args.config]           # samples for the whole leg (~30-60 s)
    return max(1, min(gpu_batch, budget // max(1, steps)))


def cpu_port_run(batch: int, steps: int, warmup: int):
    """Times the reference algorithm on the host cores.  Returns (samples_per_s, ms_per_step, cores, kind)."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step, kind = reference_step_fn(torch.device("cpu"), batch)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return batch * steps / dt, 1e3 * dt / steps, torch.get_num_threads(), kind


def torch_gpu_run(device, batch: int, steps: int = 10, warmup: int = 3):
    """The same reference step on the SAME B200 through stock PyTorch (cuFFT / cuBLAS, TF32 off): "what a user of the
    reference gets today" (SURVEY 8d).  Device-timed.  Returns a dict or {"unavailable": why}."""
    try:
        step, kind = reference_step_fn(device, batch)
        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        return {"value": round(batch / (ms / 1e3), 2), "unit": "samples/s", "ms_per_step": round(ms, 3), "batch": batch,
                "kind": kind, "steps": steps, "how": "stock PyTorch eager on the same GPU, fp32 (TF32 off), full step"}
    except Exception as exc:  # noqa: BLE001
        torch.cuda.empty_cache()
        return {"unavailable": f"{type(exc).__name__}: {str(exc)[:160]}"}


def bench_config(args, world: int, batch: int) -> dict:
    """`config` object shared by both arms (ours / reference): the same workload, batch and parallelism."""
    return {"workload": WORKLOAD, "baseline_config": args.config, "per_gpu_batch": batch, "global_batch": batch * world,
            "parallelism": f"dp{world}" if world > 1 else "single"}


def run_reference(args, rank):
    if rank != 0:
        return
    steps, warmup = args.steps, args.warmup
    gpu_batch = args.batch or WL["batch"]
    cb = cpu_batch_for(args, gpu_batch, steps + warmup)
    v, ms, cores, kind = cpu_port_run(cb, steps, warmup)
    sample = (f"{steps} timed + {warmup} warm-up full training steps of batch {cb} on the host CPU "
              f"({'oracle/_ref reference modules' if kind == 'reference' else 'oracle/fno_port.py'}, torch {torch.__version__})")
    cfg = bench_config(args, args.gpus, gpu_batch)
    cfg["cpu_per_step_batch"] = cb
    line = {
        "impl": "reference", "metric": METRIC, "value": round(v, 3), "unit": "samples/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": round(ms, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": round(v, 3), "unit": "samples/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": round(v, 3), "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return None
        if not self.lines:                      # nothing delivered yet: one synchronous query right after the timed region
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
                self.lines.extend(ln.strip() for ln in out.splitlines() if ln.strip())
            except Exception:
                pass
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# per-kernel event timing (roofline)
# ------------------------------------------------------------------------------------------------
class KernelTimer:
    """Wraps the fno_b200.lib call wrappers with CUDA events on the current stream."""

    NAMES = ["fwd_transform", "inv_transform", "layer_inv_fused", "mix_fwd", "mix_bwd", "pointwise_fwd", "pointwise_wgrad", "pointwise_bwd",
             "lift_stats", "lift_fwd", "lift_bwd", "head_fwd", "head_bwd"]

    def __init__(self, lib):
        self.lib = lib
        self.records = []
        self.saved = {}

    def __enter__(self):
        for name in self.NAMES:
            fn = getattr(self.lib, name)
            self.saved[name] = fn
            setattr(self.lib, name, self._wrap(name, fn))
        return self

    def __exit__(self, *exc):
        for name, fn in self.saved.items():
            setattr(self.lib, name, fn)

    def _wrap(self, name, fn):
        def inner(*a, **k):
            tag = name
            if name == "fwd_transform" and k.get("preact") is not None:
                tag = "fwd_transform+gelu_grad"
            if name == "inv_transform":
                tag = "inv_transform+bypass" + ("+gelu" if k.get("apply_gelu") else "") if k.get("addend") is not None else "inv_transform"
                if k.get("s_out") is not None:
                    tag += "+preact"
            if name == "layer_inv_fused":
                # K3 + 1x1-conv bypass (+ bias, GELU, pre-activation store) in one tcgen05 kernel (+ its strided-axis
                # pre-kernel): same algorithmic bytes as the r1 pair inv_transform(+addend) -- `lin` no longer exists
                tag = "inv_transform+bypass" + ("+gelu" if k.get("apply_gelu") else "") + ("+preact" if k.get("s_out") is not None else "")
                tag += " [tcgen05 fused]"
            if name == "pointwise_fwd" and k.get("transpose"):
                tag = "pointwise_bwd_data"
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn(*a, **k)
            e1.record()
            self.records.append((tag, e0, e1))
            return out
        return inner

    def summary(self):
        torch.cuda.synchronize()
        agg = {}
        for tag, e0, e1 in self.records:
            d = agg.setdefault(tag, [0.0, 0])
            d[0] += e0.elapsed_time(e1)
            d[1] += 1
        return {k: {"ms_total": v[0], "launches": v[1], "ms_avg": v[0] / v[1]} for k, v in agg.items()}


# FMA per valid pixel of the FP32-bound kernels (DESIGN.md 3.2): head forward 128 x (20 + 2), head backward
# 128 x (20 + 20 + 20 + 2 + 2 + 1), lift forward / backward 20 x 22 (+ bias)
FP32_BOUND = ("head_fwd", "head_bwd", "lift_fwd", "lift_bwd")


def fp32_bound_fma(tag: str) -> int:
    C, V, F = CFG["width"], CFG["num_channels"], CFG["initial_step"] * CFG["num_channels"] + WL["nd"]
    return {"head_fwd": 128 * (C + V), "head_bwd": 128 * (3 * C + 2 * V + 1), "lift_fwd": C * F, "lift_bwd": C * (F + 1)}[tag]


def algorithmic_bytes(tag: str, B: int) -> int:
    """Per-launch algorithmic bytes of each kernel at the bench workload (DESIGN.md section 4):
    every input read once, every output written once, weights once per launch."""
    C = CFG["width"]
    if WL["nd"] == 2:
        N, M = (RES + 2) * (RES + 2), 2 * CFG["modes1"] * CFG["modes2"]
    else:                                   # only the last axis is padded, by 6 (fno/fno.py:360); 4 corners
        N, M = RES * RES * (RES + 6), 4 * CFG["modes1"] * CFG["modes2"] * CFG["modes3"]
    pix = RES ** WL["nd"]
    act, spec, wts = 4 * C * N * B, 8 * C * M * B, 8 * C * C * M
    table = {
        "fwd_transform": act + spec,
        "fwd_transform+gelu_grad": 3 * act + spec,                 # reads g, s; writes dS; + gY
        "inv_transform": spec + act,
        "inv_transform+bypass": spec + 2 * act,                    # layer 3 fwd / layer bwd: read addend, write out
        "inv_transform+bypass+gelu": spec + 2 * act,
        "inv_transform+bypass+gelu+preact": spec + 3 * act,        # + store of the pre-activation
        "inv_transform+bypass+preact": spec + 3 * act,
        "mix_fwd": 2 * spec + wts,
        "mix_bwd": 4 * spec + 2 * wts,                             # data-grad + weight-grad launches together
        "pointwise_fwd": 2 * act,
        "pointwise_bwd_data": 2 * act,
        "pointwise_wgrad": 2 * act,
        "pointwise_bwd": 3 * act,                                  # reads ds, a; writes dx (weight + data gradient)
        # lift / head: x = [B,128,128,10,2] (+grid [..,2]) in, h = act out; out/dout = [B,128,128,2]
        "lift_stats": 4 * B * pix * CFG["initial_step"] * CFG["num_channels"],
        "lift_fwd": 4 * B * pix * (CFG["initial_step"] * CFG["num_channels"] + WL["nd"]) + act,
        "lift_bwd": 4 * B * pix * (CFG["initial_step"] * CFG["num_channels"] + WL["nd"] + C),
        "head_fwd": 4 * B * pix * (C + CFG["num_channels"]),
        "head_bwd": 4 * B * pix * (C + CFG["num_channels"]) + act,
    }
    return table[tag.replace(" [tcgen05 fused]", "")]


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist

    from fno_b200 import data, lib
    from fno_b200.dp import BucketedGradAllReduce
    from fno_b200.train import FusedTrainStep, TrainStep

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device: libfno_sm100 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib.load()
    B, K, W = (args.batch or WL["batch"]), args.steps, max(args.warmup, 3)
    aux = WL["kind"] == "aux2d"

    torch.manual_seed(16)
    model = make_model().to(dev)
    dp = BucketedGradAllReduce(model) if world > 1 else None
    if aux:
        # the joint loop's optimizer (fno_aux/fno_train_aux.py:175-179): three Adam groups, two learning rates
        groups = [{"params": model.shared_layers.parameters(), "lr": WL["lr_share"]},
                  {"params": model.fc2_primary.parameters(), "lr": WL["lr_fc2"]},
                  {"params": model.fc2_auxiliary.parameters(), "lr": WL["lr_fc2"]}]
        step = FusedTrainStep(model, lr=WL["lr_share"], weight_decay=1e-4, t_max=100000, dp=dp,
                              graph=(args.tail == "graph" and (world == 1 or not args.dp_eager)), alias_inputs=True,
                              max_graphs=4, auxiliary_weight=WL["aux_w"], param_groups=groups)
        eager_step = step._eager
    elif args.tail == "torch":
        opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=1e-4)
        sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=100000)
        step = TrainStep(model, opt, sched, dp=dp)
        eager_step = step
    else:
        # the graph reads the input buffers in place (one captured graph per buffer set: the two HBM-resident
        # batches and the two end-to-end staging sets) -- no 201 MB device copy per step
        step = FusedTrainStep(model, lr=1e-3, weight_decay=1e-4, t_max=100000, dp=dp,
                              graph=(args.tail == "graph" and (world == 1 or not args.dp_eager)), alias_inputs=True, max_graphs=4)
        eager_step = step._eager
    graphed = args.tail == "graph" and (world == 1 or not args.dp_eager)

    # two distinct host batches per rank (pinned); device copies for the HBM-resident measurement
    host = []
    for i in range(2):
        host.append(tuple(t.pin_memory() for t in make_batch(B, 1000 * rank + i)))
    devb = [tuple(t.to(dev) for t in hb) for hb in host]
    h2d_bytes = sum(t.numel() * t.element_size() for t in host[0])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident throughput ---------------------------------------------------------
    l0 = lib.launch_count()
    eager_step(*devb[0])                      # also counts this library's launches per (eager) step
    launches_per_step = lib.launch_count() - l0
    # the clock sampler starts before the warm-up steps (same load as the timed steps): nvidia-smi needs ~100 ms to
    # deliver its first line and the timed region of a short run is shorter than that
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for i in range(max(W, 3)):                # graph mode: calls 1-2 eager, call 3 captures
        step(*devb[i % 2])
    barrier()
    l0 = lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        loss = step(*devb[i % 2])
    e1.record()
    torch.cuda.synchronize()
    launches = (lib.launch_count() - l0) if not graphed else launches_per_step * K   # replays do not pass the counter
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    final_loss = float(loss.flatten()[0])

    # ---- end to end: host-pinned inputs, prefetch on a copy stream, loss read back every step ----
    e2e = None
    if not args.no_e2e:
        copy_stream = torch.cuda.Stream()
        bufs = [tuple(torch.empty_like(t, device=dev) for t in host[0]) for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]

        def prefetch(i):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[i % 2])
                for dst, src in zip(bufs[i % 2], host[i % 2]):
                    dst.copy_(src, non_blocking=True)
                ready[i % 2].record(copy_stream)

        def e2e_loop(n):
            cur = torch.cuda.current_stream()
            for s in range(2):
                consumed[s].record(cur)
            prefetch(0)
            last = 0.0
            for i in range(n):
                if i + 1 < n:
                    prefetch(i + 1)
                cur.wait_event(ready[i % 2])
                loss_i = step(*bufs[i % 2])
                consumed[i % 2].record(cur)
                last = float(loss_i.flatten()[0])   # D2H read of the step's loss (4 bytes) -> host sync
            return last

        e2e_loop(W)
        barrier()
        t0 = torch.cuda.Event(enable_timing=True)
        t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        e2e_loop(K)
        t1.record()
        torch.cuda.synchronize()
        ms_e2e = max_over_ranks(t0.elapsed_time(t1))
        barrier()
        e2e = {"value": round(world * B * K / (ms_e2e / 1e3), 2), "unit": "samples/s",
               "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4, "ms_per_step": round(ms_e2e / K, 3)}

    # ---- end to end through the streaming device-resident dataset (SURVEY 8f row f4): the declared `e2e` at config 1 ----
    # The reference loaders read a whole trajectory per item (fno/utils_2d_rd_baseline.py:74-86) and consecutive windows
    # share 9 of their 10 input frames, so shipping assembled (xx, yy) batches moves every frame ~11 times (201 MB per
    # step at batch 128: the PCIe link, not the GPU, then sets the rate, and 8 ranks saturate the host).  Here every
    # trajectory FRAME crosses the link once: trajectories live in HBM in the loaders' own order, each step uploads --
    # inside the timed region, from pinned host memory, on a copy stream -- the share of fresh trajectory data its B
    # windows consume (B * T / n_windows frames) plus the B item indices, gathers its windows on the device
    # (fno_window_gather) and reads the loss back.
    e2e_dev = None
    if not args.no_e2e and WL["kind"] == "fno2d":
        T_traj = CFG["initial_step"] + 91                      # 101 frames -> 91 windows per trajectory, as in PDEBench
        n_traj = 8
        traj = data.diffusion_trajectories(n_traj, RES, T_traj, CFG["num_channels"], seed=5 + rank)
        ds = data.DeviceWindows(traj, CFG["initial_step"], 1, device=dev)
        h_store = ds.traj.detach().cpu().pin_memory()          # the store's own layout [n, pixels, T, V]
        flat_dev, flat_host = ds.traj.view(-1), h_store.view(-1)
        frame_floats = RES ** WL["nd"] * CFG["num_channels"]
        chunk = min(flat_dev.numel(), ((B * T_traj + ds.n_windows - 1) // ds.n_windows) * frame_floats)   # floats per step
        gi = torch.Generator().manual_seed(7 + rank)
        items_host = [ds.split_items(torch.randint(0, len(ds), (B,), generator=gi, dtype=torch.int64)) for _ in range(2)]
        npx = RES ** WL["nd"]
        outs = [(torch.empty(B, npx, CFG["initial_step"], CFG["num_channels"], device=dev),
                 torch.empty(B, npx, 1, CFG["num_channels"], device=dev)) for _ in range(2)]   # fixed addresses: aliased graphs
        up_stream = torch.cuda.Stream()
        up_done = [torch.cuda.Event() for _ in range(2)]
        state = {"off": 0}

        def upload(i):                                         # step i's share of fresh trajectory frames (rotating region
            with torch.cuda.stream(up_stream):                 # of the store, values unchanged), one step ahead of its use
                if state["off"] + chunk > flat_dev.numel():
                    state["off"] = 0
                o = state["off"]
                flat_dev[o:o + chunk].copy_(flat_host[o:o + chunk], non_blocking=True)
                up_done[i % 2].record(up_stream)
                state["off"] = o + chunk

        loss_host = torch.zeros(2, dtype=torch.float32).pin_memory()
        loss_ev = [torch.cuda.Event() for _ in range(2)]

        def dev_loop(n):
            # host-side software pipeline: the next batch is gathered (queued behind the running step) BEFORE the host
            # blocks on this step's loss, so the GPU never waits for the host between steps; the loss of every step is
            # still copied to pinned host memory and read
            last = 0.0
            cur = torch.cuda.current_stream()
            upload(0)
            cur.wait_event(up_done[0])
            nxt = ds.batch(items_host[0], out=outs[0])
            for i in range(n):
                loss_i = step(*nxt)
                loss_host[i % 2:i % 2 + 1].copy_(loss_i.flatten()[:1], non_blocking=True)
                loss_ev[i % 2].record(cur)
                if i + 1 < n:
                    upload(i + 1)
                    cur.wait_event(up_done[(i + 1) % 2])
                    nxt = ds.batch(items_host[(i + 1) % 2], out=outs[(i + 1) % 2])
                loss_ev[i % 2].synchronize()
                last = float(loss_host[i % 2])                 # D2H read of the step's loss (4 bytes)
            return last

        dev_loop(W)
        barrier()
        t0 = torch.cuda.Event(enable_timing=True)
        t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        dev_loop(K)
        t1.record()
        torch.cuda.synchronize()
        ms_dev = max_over_ranks(t0.elapsed_time(t1))
        barrier()
        e2e_dev = {"value": round(world * B * K / (ms_dev / 1e3), 2), "unit": "samples/s",
                   "h2d_bytes_per_step": 4 * chunk + 8 * B, "d2h_bytes_per_step": 4, "ms_per_step": round(ms_dev / K, 3),
                   "how": f"streaming device-resident dataset (fno_b200.data.DeviceWindows): per step {4 * chunk / 1e6:.1f} MB of "
                          f"fresh trajectory frames ({T_traj}/{ds.n_windows} frames per window consumed) + {8 * B} B of item "
                          "indices H2D from pinned memory inside the timed region, windows gathered on the device, loss read "
                          "back every step"}
        del ds, traj, h_store

    # ---- instrumented pass: per-kernel CUDA events (never used for `value`) -------------------
    roofline, kernels = None, None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    nprof = min(K, 5)
    for i in range(2):                     # let the caching allocator settle outside the graph's private pool
        eager_step(*devb[i % 2])
    torch.cuda.synchronize()
    with KernelTimer(lib) as kt:
        for i in range(nprof):
            eager_step(*devb[i % 2])
        ksum = kt.summary()
    barrier()
    if rank == 0:
        kernels = {}
        traffic = {}
        try:   # dram__bytes_read+write per launch from the committed `ncu --set full` capture of this workload
            tj = json.loads((ROOT / "profiles" / "traffic_cfg1_b128.json").read_text())
            if tj.get("batch") == B:
                traffic = tj["bytes_per_launch"]
        except Exception:
            pass
        for tag, r in sorted(ksum.items(), key=lambda kv: -kv[1]["ms_total"]):
            # trunk kernels of the joint step see the primary and the auxiliary stream in one batch; its two heads
            # see B and num_aux * B (the mean is used)
            Bk = B if not aux else (B * (1 + WL["num_aux"]) // (2 if tag.startswith("head") else 1))
            nbytes = algorithmic_bytes(tag, Bk)
            entry = {"ms_avg": round(r["ms_avg"], 4), "launches_per_step": r["launches"] / nprof,
                     "gbs": round(nbytes / (r["ms_avg"] * 1e-3) / 1e9, 1),
                     "ms_per_step": round(r["ms_total"] / nprof, 3), "bound": "hbm",
                     "hbm_frac": round(nbytes / (r["ms_avg"] * 1e-3) / 1e9 / peak, 4)}
            if tag in FP32_BOUND:   # FMA/issue-bound kernels (DESIGN.md section 5): report the useful-FLOP rate too
                fma = fp32_bound_fma(tag) * Bk * RES ** WL["nd"]
                # the projection head runs its dense contractions on tcgen05 (3xTF32) and is bound by the CUDA-core
                # epilogue (GELU) and the shared-memory pipe; the lift kernels are FP32 CUDA-core kernels
                entry["bound"] = "tcgen05-3xtf32+epilogue-issue" if tag.startswith("head") else "fp32-issue"
                entry["fp32_tflops"] = round(2 * fma / (r["ms_avg"] * 1e-3) / 1e12, 2)
                entry["fp32_frac_of_74"] = round(2 * fma / (r["ms_avg"] * 1e-3) / 1e12 / 74.4, 3)
            kernels[tag] = entry
        # BASELINE.json's second metric is "spectral-conv HBM GB/s vs peak": the roofline object is the
        # spectral-convolution kernel (K1 / K2 / K3 families) with the largest share of the step; every
        # other kernel, including the FP32-bound projection head, is listed under "kernels".
        spectral = [t for t in kernels if t.startswith(("fwd_transform", "inv_transform", "mix_"))]
        top = max(spectral, key=lambda t: kernels[t]["ms_per_step"])
        roofline = {"bound": "hbm", "kernel": top, "kernel_class": "spectral-conv (K1/K2/K3), largest step share",
                    "achieved": kernels[top]["gbs"], "peak": peak, "unit": "GB/s",
                    "frac": round(kernels[top]["gbs"] / peak, 4),
                    "traffic": traffic.get(top), "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": algorithmic_bytes(top, B),
                    "step_share": round(kernels[top]["ms_per_step"] / (ms_total / K), 3),
                    "largest_kernel_overall": next(iter(kernels))}

    # ---- CPU baseline (rank 0, N = 1 only) ------------------------------------------------------
    # ---- the reference step on the same GPU through stock PyTorch (rank 0, N = 1 only) --------------
    torch_gpu = None
    if rank == 0 and world == 1 and not args.no_torch_gpu:
        del devb, host
        torch.cuda.empty_cache()
        torch_gpu = torch_gpu_run(dev, B)
        torch.cuda.empty_cache()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cb = cpu_batch_for(args, B, 8)
        v, ms, cores, kind = cpu_port_run(cb, 6, 2)
        cpu = {"value": round(v, 3), "unit": "samples/s", "cores": cores, "kind": kind,
               "sample": f"6 timed + 2 warm-up full training steps of batch {cb} on the host CPU "
                         f"({'oracle/_ref reference modules' if kind == 'reference' else 'oracle/fno_port.py'}, "
                         f"torch {torch.__version__})", "ms_per_step": round(ms, 2)}

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    value = world * B * K / (ms_total / 1e3)
    line = {
        "metric": METRIC, "value": round(value, 2), "unit": "samples/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": round(ms_total / K, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": dict(bench_config(args, world, B),
                       step_tail=args.tail if (world == 1 or args.tail == "torch" or graphed) else "fused",
                       l2_policy=f"inputs larger than L2: two alternating {h2d_bytes / 1e6:.0f} MB input batches, activation "
                                 f"tensors of {algorithmic_bytes('pointwise_fwd', B * (1 + WL.get('num_aux', 0))) / 2e6:.0f} MB"),
        # declared end-to-end number: the streaming device-resident dataset where the workload has one (2-D single-head
        # configs); `e2e_host_batches` ships fully assembled (xx, yy, grid) batches every step (round 1's `e2e`)
        "e2e": e2e_dev if e2e_dev is not None else e2e, "e2e_host_batches": e2e, "gpu_launches": int(launches),
        "clocks": clocks, "roofline": roofline,
        "cpu_baseline": cpu, "torch_gpu_baseline": torch_gpu,
        "kernels": kernels, "final_loss": round(final_loss, 6),
    }
    print(json.dumps(line), flush=True)


def run_sweep(args):
    """BASELINE configs[4]: the config-3 model under data parallelism at GLOBAL batch 64..1024 (split evenly over the
    ranks) plus the autoregressive rollout evaluation (rollout_test = 5, metrics.py:337-344) on a sharded validation set.
    One JSON line; `value` is the throughput at the largest global batch that fits, `sweep` holds every point."""
    import torch.distributed as dist

    from fno_b200 import data, evaluate, lib
    from fno_b200.dp import BucketedGradAllReduce
    from fno_b200.train import FusedTrainStep

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib.load()
    K, W = args.steps, max(args.warmup, 3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def maxr(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    points = []
    model = None
    for G in (64, 128, 256, 512, 1024):
        b = G // world
        if b < 1 or b * world != G or b > 256:          # > 256 samples of 256x256 w64 per GPU exceed the 180 GB of HBM3e
            points.append({"global_batch": G, "per_gpu_batch": b, "skipped": "does not fit / not divisible"})
            continue
        torch.manual_seed(16)
        model = make_model().to(dev)
        dp = BucketedGradAllReduce(model) if world > 1 else None
        step = FusedTrainStep(model, lr=1e-3, weight_decay=1e-4, t_max=100000, dp=dp, graph=True, alias_inputs=True,
                              max_graphs=2)
        devb = [tuple(t.to(dev) for t in make_batch(b, 1000 * rank + i)) for i in range(2)]
        for i in range(W):
            step(*devb[i % 2])
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            step(*devb[i % 2])
        e1.record()
        torch.cuda.synchronize()
        ms = maxr(e0.elapsed_time(e1))
        barrier()
        points.append({"global_batch": G, "per_gpu_batch": b, "samples_per_s": round(G * K / (ms / 1e3), 1),
                       "ms_per_step": round(ms / K, 3), "step": "cuda-graph" if world == 1 else "two cuda graphs around the bucket all-reduces"})
        del step, dp, devb
        torch.cuda.empty_cache()
    # rollout evaluation: 5 autoregressive steps on this rank's shard of a 64-item validation set
    rollout = None
    if model is not None:
        nval = max(1, 64 // world)
        vb = min(8, nval)
        traj = data.diffusion_trajectories(nval, RES, CFG["initial_step"] + 5, CFG["num_channels"], seed=77 + rank)
        xx, yy = data.windows(traj, CFG["initial_step"], 5)
        grid = data.cell_centre_grid(RES).unsqueeze(0)
        batches = [(xx[i:i + vb].to(dev), yy[i:i + vb].to(dev), grid.expand(min(vb, nval - i), -1, -1, -1).contiguous().to(dev))
                   for i in range(0, nval, vb)]
        model.eval()
        evaluate.evaluate_rollout(model, batches[:1], 5)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = evaluate.evaluate_rollout(model, batches, 5)
        e1.record()
        torch.cuda.synchronize()
        ms = maxr(e0.elapsed_time(e1))
        rollout = dict(res, rollout_test=5, val_items=nval * world, ms=round(ms, 2),
                       rollout_steps_per_s=round(nval * world * 5 / (ms / 1e3), 1))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    done = [p for p in points if "samples_per_s" in p]
    top = done[-1]
    line = {"metric": METRIC, "value": top["samples_per_s"], "unit": "samples/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": top["ms_per_step"], "higher_is_better": True, "scaling": "strong (global batch fixed per point)",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(bench_config(args, world, top["per_gpu_batch"]), sweep="global batch 64..1024"),
            "sweep": points, "rollout_eval": rollout, "e2e": None, "gpu_launches": None}
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    select_workload(args.config)
    if args.config == 5 and args.impl == "ours":
        run_sweep(args)
        return
    if args.impl == "reference":
        run_reference(args, rank)
        return
    run_ours(args)


if __name__ == "__main__":
    main()
