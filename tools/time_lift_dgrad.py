"""Times the input-gradient kernels and the graphed rollout training step on one GPU.

  * fno_lift_dgrad (dx only, the training path) and fno_window_shift_bwd at config 1 (B = 128, 128x128, width 20,
    T*V = 20) and config 3 (B = 32, 256x256, width 64, T*V = 30): CUDA events around each launch, a 256 MB buffer
    rewritten between launches (L2 flush), mean over many launches.  Algorithmic bytes: the valid region of dh read once
    and dx written once; g read once and gxx + gpred written once.  Fraction of 6544 GB/s, the HBM rate this project
    measured on a B200 (DESIGN.md section 4).
  * FusedTrainStep(graph=True, alias_inputs=True, rollout_steps=K) at config 1, B = 128, for K = 1, 2, 4: ms per step
    over graph replays (events, synchronised).

usage: python tools/time_lift_dgrad.py [--json OUT.json] [--launches N] [--steps N]"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "sciml-pde_b200")]
from fno_b200 import lib  # noqa: E402

HBM_GBS = 6544.0
CONFIGS = {1: dict(B=128, spatial=(128, 128), C=20, T=10, V=2, G=2, pad=2),
           3: dict(B=32, spatial=(256, 256), C=64, T=10, V=3, G=2, pad=2)}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return f"{name}, power limit / max SM clock: {out}"


def time_launches(fn, n, flush):
    for _ in range(3):
        fn()
    tot = 0.0
    for _ in range(n):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    return 1e3 * tot / n                                       # us


def kernels(cfg_id, n, flush):
    c = CONFIGS[cfg_id]
    B, C, T, V, G = c["B"], c["C"], c["T"], c["V"], c["G"]
    geo = lib.TrunkGeo(c["spatial"], c["pad"])
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(0)
    dh = torch.randn((B, C) + geo.padded, device=dev, generator=gen)
    W0 = torch.randn(C, T * V + G, device=dev, generator=gen)
    stats = torch.rand(B, 2, V, device=dev, generator=gen) + 0.5
    dx = torch.empty(B, geo.npix, T, V, device=dev)
    g = torch.randn(B, geo.npix, T, V, device=dev, generator=gen)
    gxx, gpred = torch.empty_like(g), torch.empty(B, geo.npix, 1, V, device=dev)
    L = lib.load()
    st = torch.cuda.current_stream().cuda_stream

    def dgrad():
        lib._check(L.fno_lift_dgrad(dh.data_ptr(), W0.data_ptr(), stats.data_ptr(), dx.data_ptr(), None, B, *geo.ints,
                                    T, V, G, C, st), "fno_lift_dgrad")

    def shift_bwd():
        lib._check(L.fno_window_shift_bwd(g.data_ptr(), gxx.data_ptr(), gpred.data_ptr(), B * geo.npix, T, V, st),
                   "fno_window_shift_bwd")

    rows = []
    for name, fn, nbytes in (("fno_lift_dgrad", dgrad, 4 * B * geo.npix * (C + T * V)),
                             ("fno_window_shift_bwd", shift_bwd, 4 * B * geo.npix * (2 * T * V + V))):
        us = time_launches(fn, n, flush)
        gbs = nbytes / (us * 1e-6) / 1e9
        rows.append(dict(config=cfg_id, kernel=name, B=B, us=round(us, 1), bytes=nbytes, TBps=round(gbs / 1e3, 3),
                         frac_hbm=round(gbs / HBM_GBS, 3)))
        print(f"  cfg {cfg_id} {name:22s} {us:8.1f} us  {nbytes / 1e6:7.1f} MB  {gbs / 1e3:5.2f} TB/s  "
              f"{gbs / HBM_GBS:5.2f} of {HBM_GBS:.0f} GB/s", flush=True)
    return rows


def rollout_steps(K, steps):
    from fno_b200.fno import FNO2d
    from fno_b200.train import FusedTrainStep

    dev = torch.device("cuda", 0)
    B, X = 128, 128
    torch.manual_seed(0)
    model = FNO2d(num_channels=2, modes1=12, modes2=12, width=20, initial_step=10).to(dev)
    step = FusedTrainStep(model, lr=1e-3, weight_decay=1e-4, t_max=100000, graph=True, alias_inputs=True,
                          rollout_steps=K)
    gen = torch.Generator(device=dev).manual_seed(1)
    xx = torch.randn(B, X, X, 10, 2, device=dev, generator=gen)
    yy = torch.randn(B, X, X, K, 2, device=dev, generator=gen)
    lin = torch.linspace(0, 1, X, device=dev)
    grid = torch.stack(torch.meshgrid(lin, lin, indexing="ij"), dim=-1).unsqueeze(0).repeat(B, 1, 1, 1).contiguous()
    for _ in range(5):                                          # eager warm-up, capture, first replays
        step(xx, yy, grid)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = step(xx, yy, grid)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    assert torch.isfinite(out).all()
    print(f"  cfg 1 B={B} rollout_steps={K}: {ms:7.2f} ms/step  ({B / ms * 1e3:7.0f} samples/s)", flush=True)
    del step, model
    torch.cuda.empty_cache()
    return dict(K=K, B=B, ms_per_step=round(ms, 3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json", default="")
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_lift_dgrad needs a CUDA device")
    info = card()
    print(info, flush=True)
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")
    res = dict(card=info, kernels=[], rollout=[])
    for cfg_id in (1, 3):
        res["kernels"] += kernels(cfg_id, args.launches, flush)
    del flush
    torch.cuda.empty_cache()
    for K in (1, 2, 4):
        res["rollout"].append(rollout_steps(K, args.steps))
    if args.json:
        Path(args.json).parent.mkdir(parents=True, exist_ok=True)
        Path(args.json).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
