"""Times rollout training of the two-head joint model on one GPU at config 2 (fno_aux FNO2d, modes 12, width 20,
initial_step 10, 128x128x2, B = 32 primary items + 3 auxiliary samples each: a joined batch of 128).

  * fno_window_shift_split and fno_window_shift_split_bwd on the joined window [128, 128x128, 10, 2] (168 MB), primary
    rows first: CUDA events around each launch, a 256 MB buffer rewritten between launches (L2 flush), mean over many
    launches.  Byte floor: the bytes each launch has to move (shift: the window read once with the new frames in place
    of the dropped one, the window written once; adjoint: g read once, gxx and both gpred written once) at 6544 GB/s,
    the HBM rate this project measured on a B200 (DESIGN.md section 4).
  * The joint heads' forward + backward on the trunk activation [128, 20, 130, 130] (173 MB): ops.TwoHeadFn against the
    per-head form on slices of h that it replaced, whose backward zero-fills one trunk-sized gradient per head and adds
    the two.  Same timing method.
  * FusedTrainStep(graph=True, alias_inputs=True, auxiliary_weight=0.7, the joint loop's three Adam groups,
    rollout_steps=K) for K = 1, 2, 4: ms per step over graph replays (events, synchronised).  Then `bench.py --config 2`
    runs in a subprocess of the same call, so its step time stands next to K = 1.

usage: python tools/time_joint_rollout.py [--json OUT.json] [--launches N] [--steps N] [--no-bench]"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "sciml-pde_b200")]
from fno_b200 import lib, ops  # noqa: E402

HBM_GBS = 6544.0
B, NUM_AUX, X, T, V, C = 32, 3, 128, 10, 2, 20
N = B * (1 + NUM_AUX)
AUX_W = 0.7


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


def row(name, us, nbytes):
    gbs = nbytes / (us * 1e-6) / 1e9
    floor = nbytes / (HBM_GBS * 1e9) * 1e6
    print(f"  {name:28s} {us:8.1f} us  {nbytes / 1e6:7.1f} MB  {gbs / 1e3:5.2f} TB/s  {gbs / HBM_GBS:5.2f} of "
          f"{HBM_GBS:.0f} GB/s  (byte floor {floor:6.1f} us)", flush=True)
    return dict(kernel=name, us=round(us, 1), bytes=nbytes, TBps=round(gbs / 1e3, 3), frac_hbm=round(gbs / HBM_GBS, 3),
                floor_us=round(floor, 1))


def shift_kernels(n, flush):
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(0)
    xj = torch.randn(N, X * X, T, V, device=dev, generator=gen)
    pa, pb = torch.randn(B, X * X, 1, V, device=dev, generator=gen), torch.randn(N - B, X * X, 1, V, device=dev,
                                                                                  generator=gen)
    out, g = torch.empty_like(xj), torch.randn_like(xj)
    gxx, ga, gb = torch.empty_like(xj), torch.empty_like(pa), torch.empty_like(pb)
    L = lib.load()
    st = torch.cuda.current_stream().cuda_stream
    points, points_a = N * X * X, B * X * X

    def fwd():
        lib._check(L.fno_window_shift_split(xj.data_ptr(), pa.data_ptr(), pb.data_ptr(), out.data_ptr(), points_a,
                                            points, T, V, st), "fno_window_shift_split")

    def bwd():
        lib._check(L.fno_window_shift_split_bwd(g.data_ptr(), gxx.data_ptr(), ga.data_ptr(), gb.data_ptr(), points_a,
                                                points, T, V, st), "fno_window_shift_split_bwd")

    rows = [row("fno_window_shift_split", time_launches(fwd, n, flush), 4 * points * 2 * T * V),
            row("fno_window_shift_split_bwd", time_launches(bwd, n, flush), 4 * points * (2 * T * V + V))]
    torch.cuda.synchronize()
    assert torch.equal(out, torch.cat((xj[..., 1:, :], torch.cat((pa, pb))), dim=-2))
    return rows


def heads(n, flush):
    """Forward + backward of the two heads at config 2: TwoHeadFn against the per-head form on slices of h."""
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(2)
    geo = lib.TrunkGeo((X, X), 2)
    h = torch.randn((N, C) + geo.padded, device=dev, generator=gen).requires_grad_(True)
    stats = torch.stack((torch.randn(N, V, device=dev, generator=gen), 0.5 + torch.rand(N, V, device=dev, generator=gen)),
                        dim=1)
    W1 = (torch.randn(128, C, device=dev, generator=gen) / C ** 0.5).requires_grad_(True)
    b1 = torch.zeros(128, device=dev).requires_grad_(True)
    W2 = [(torch.randn(V, 128, device=dev, generator=gen) / 128 ** 0.5).requires_grad_(True) for _ in range(2)]
    b2 = [torch.zeros(V, device=dev).requires_grad_(True) for _ in range(2)]
    dout = [torch.randn((k, X, X, V), device=dev, generator=gen) for k in (B, N - B)]
    sa, sb = stats[:B].contiguous(), stats[B:].contiguous()

    leaves = [h, W1, b1, W2[0], b2[0], W2[1], b2[1]]

    def per_head():
        outs = (ops.head(h[:B], W1, b1, W2[0], b2[0], sa, geo), ops.head(h[B:], W1, b1, W2[1], b2[1], sb, geo))
        torch.autograd.grad(outs, leaves, dout)

    def two_head():
        outs = ops.TwoHeadFn.apply(h, W1, b1, W2[0], b2[0], W2[1], b2[1], stats, geo, B)
        torch.autograd.grad(outs, leaves, dout)

    res = []
    for name, fn in (("heads fwd+bwd, per-head", per_head), ("heads fwd+bwd, TwoHeadFn", two_head)):
        us = time_launches(fn, n, flush)
        print(f"  {name:28s} {us:8.1f} us", flush=True)
        res.append(dict(path=name, us=round(us, 1)))
    trunk = 4 * h.numel()
    print(f"  extra traffic of the per-head backward: 2 trunk-sized zero fills + the two slices copied in (read + "
          f"write) + one add (2 reads, 1 write) = 7 x {trunk / 1e6:.0f} MB = {7 * trunk / 1e9:.2f} GB", flush=True)
    res.append(dict(extra_bytes_per_head_backward=7 * trunk))
    return res


def joint_step(K, steps):
    from fno_b200.fno_aux import FNO2d
    from fno_b200.train import FusedTrainStep

    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    model = FNO2d(num_channels=V, modes1=12, modes2=12, width=C, initial_step=T).to(dev)
    groups = [{"params": model.shared_layers.parameters(), "lr": 1e-3},
              {"params": model.fc2_primary.parameters(), "lr": 2e-3},
              {"params": model.fc2_auxiliary.parameters(), "lr": 2e-3}]
    step = FusedTrainStep(model, lr=1e-3, weight_decay=1e-4, t_max=100000, graph=True, alias_inputs=True,
                          auxiliary_weight=AUX_W, param_groups=groups, rollout_steps=K)
    gen = torch.Generator(device=dev).manual_seed(1)
    lin = torch.linspace(0, 1, X, device=dev)
    grid1 = torch.stack(torch.meshgrid(lin, lin, indexing="ij"), dim=-1).unsqueeze(0)
    batch = []
    for nb in (B, B * NUM_AUX):
        batch += [torch.randn(nb, X, X, T, V, device=dev, generator=gen), torch.randn(nb, X, X, K, V, device=dev,
                                                                                      generator=gen),
                  grid1.repeat(nb, 1, 1, 1).contiguous()]
    for _ in range(5):                                          # eager warm-up, capture, first replays
        step(*batch)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = step(*batch)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    assert torch.isfinite(out).all()
    print(f"  cfg 2 B={B}+{B * NUM_AUX} rollout_steps={K}: {ms:7.2f} ms/step  ({B / ms * 1e3:7.0f} primary samples/s)",
          flush=True)
    del step, model, batch
    torch.cuda.empty_cache()
    return dict(K=K, B=B, ms_per_step=round(ms, 3))


def bench_config2(steps):
    cmd = [sys.executable, str(ROOT / "bench.py"), "--config", "2", "--steps", str(steps), "--warmup", "5",
           "--no-cpu-baseline", "--no-torch-gpu", "--no-e2e"]
    out = subprocess.run(cmd, capture_output=True, text=True, cwd=str(ROOT))
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    if out.returncode != 0 or not lines:
        raise SystemExit(f"bench.py --config 2 failed ({out.returncode}):\n{out.stderr[-2000:]}")
    line = json.loads(lines[-1])
    print(f"  bench.py --config 2 --steps {steps}: {line['ms_per_step']:7.2f} ms/step  ({line['value']:7.0f} samples/s)",
          flush=True)
    return dict(ms_per_step=line["ms_per_step"], value=line["value"], steps=steps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json", default="")
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--no-bench", action="store_true", help="skip the bench.py --config 2 run")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_joint_rollout needs a CUDA device")
    info = card()
    print(info, flush=True)
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")
    res = dict(card=info, kernels=shift_kernels(args.launches, flush), heads=heads(args.launches, flush), rollout=[])
    del flush
    torch.cuda.empty_cache()
    for K in (1, 2, 4):
        res["rollout"].append(joint_step(K, args.steps))
    if not args.no_bench:
        res["bench_config2"] = bench_config2(max(args.steps, 20))
    if args.json:
        Path(args.json).parent.mkdir(parents=True, exist_ok=True)
        Path(args.json).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
