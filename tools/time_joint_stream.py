"""Times the streaming data path of the two-head joint model on one GPU at config 2 (fno_aux FNO2d, modes 12, width 20,
initial_step 10, 128x128x2, B = 32 primary items + 3 auxiliary samples each: a trunk batch of 128).

  * fno_window_gather_joint at config 2 (A = 3, the joined window [128, 128x128, 10, 2] plus both targets) and
    fno_window_gather at config 1 (A = 0, B = 128): CUDA events around each launch, a 256 MB buffer rewritten between
    launches (L2 flush), mean over many launches.  The stores hold 8 trajectories of 101 frames (91 windows each, as
    bench.py's streamed e2e) and the items are random.  Byte floor: the window and targets read once and written once,
    2 * rows * pixels * (T0 + R) * V * 4 bytes, at 6544 GB/s, the HBM rate this project measured on a B200 (DESIGN.md
    section 4).  With --parent-lib, the A = 0 gather of that library is timed in the same process, alternated.
  * The graphed config-2 joint step (FusedTrainStep, graph=True, alias_inputs=True, the joint loop's three Adam
    groups, auxiliary_weight 0.7) on joined views (xx / xx_aux and grid / grid_aux adjacent in one buffer, as
    data.DeviceJointWindows yields them) against the same tensors as separate allocations, which the forward
    concatenates: ms per step over graph replays, alternated.
  * Streamed config-2 end to end (data.DeviceJointWindows): every step uploads, from pinned host memory on a copy
    stream, the share of fresh trajectory frames its B windows consume on both stores, plus the item indices, gathers
    the joined batch into one of two double-buffered out= sets and reads the loss back -- the upload model of bench.py's
    config-1 `e2e`.  Next to it, host-batch shipping: the assembled 6-tuple copied from pinned memory on a copy stream
    into double buffers, loss read back every step.  Samples/s (primary items) and H2D bytes per step for each.

usage: python tools/time_joint_stream.py [--json OUT.json] [--launches N] [--steps N] [--rounds N] [--parent-lib SO]"""
import argparse
import ctypes
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "sciml-pde_b200")]
from fno_b200 import data, fno_aux, lib  # noqa: E402
from fno_b200.train import FusedTrainStep  # noqa: E402

HBM_GBS = 6544.0
B2, B1, NUM_AUX, X, T0, V = 32, 128, 3, 128, 10, 2
T_TRAJ, N_TRAJ = T0 + 91, 8
AUX_W = 0.7


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return f"{name}, power limit / max SM clock: {out}"


def time_launch(fn, flush):
    flush.zero_()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1)                          # us


def row(name, us, nbytes):
    gbs = nbytes / (us * 1e-6) / 1e9
    print(f"  {name:34s} {us:8.1f} us  {nbytes / 1e6:7.1f} MB  {gbs / 1e3:5.2f} TB/s  {gbs / HBM_GBS:5.2f} of "
          f"{HBM_GBS:.0f} GB/s  (byte floor {nbytes / (HBM_GBS * 1e9) * 1e6:6.1f} us)", flush=True)
    return dict(kernel=name, us=round(us, 1), bytes=nbytes, TBps=round(gbs / 1e3, 3), frac_hbm=round(gbs / HBM_GBS, 3))


def stores(seed):
    g = torch.Generator().manual_seed(seed)
    traj = torch.randn(N_TRAJ, T_TRAJ, X, X, V, generator=g)
    traj_aux = torch.randn(N_TRAJ, NUM_AUX, T_TRAJ, X, X, V, generator=g)
    return traj, traj_aux


def gather_kernels(ds, n, rounds, parent_lib, flush):
    npix = X * X
    st = torch.cuda.current_stream().cuda_stream
    gi = torch.Generator().manual_seed(3)
    res = {}
    # config 2: the joined gather
    ti2, ts2 = (t.cuda() for t in ds.split_items(torch.randint(0, len(ds), (B2,), generator=gi)))
    out2 = ds.joined_buffers(B2)
    fn2 = lambda: lib.window_gather_joint(ds.traj, ds.traj_aux, ti2, ts2, T0, 1, out=out2)   # noqa: E731
    # config 1: A = 0, this build and (optionally) the parent build on the same buffers
    ti1, ts1 = (t.cuda() for t in ds.split_items(torch.randint(0, len(ds), (B1,), generator=gi)))
    xx1, yy1 = torch.empty(B1, npix, T0, V, device="cuda"), torch.empty(B1, npix, 1, V, device="cuda")
    args1 = (ds.traj.data_ptr(), ti1.data_ptr(), ts1.data_ptr(), xx1.data_ptr(), yy1.data_ptr(), B1, npix, T_TRAJ, V,
             T0, 1, st)
    L = lib.load()
    forms = {"fno_window_gather_joint cfg2 A=3": (fn2, 2 * B2 * (1 + NUM_AUX) * npix * (T0 + 1) * V * 4),
             "fno_window_gather cfg1 A=0": (lambda: lib._check(L.fno_window_gather(*args1), "gather"),
                                            2 * B1 * npix * (T0 + 1) * V * 4)}
    if parent_lib:
        P = ctypes.CDLL(parent_lib)
        P.fno_window_gather.restype = ctypes.c_int
        P.fno_window_gather.argtypes = L.fno_window_gather.argtypes
        forms["parent fno_window_gather cfg1 A=0"] = (lambda: P.fno_window_gather(*args1), forms[
            "fno_window_gather cfg1 A=0"][1])
    tot = {k: 0.0 for k in forms}
    for name, (fn, _) in forms.items():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    if parent_lib:                                             # same items, same outputs
        forms["fno_window_gather cfg1 A=0"][0]()
        a = xx1.clone(), yy1.clone()
        forms["parent fno_window_gather cfg1 A=0"][0]()
        assert torch.equal(a[0], xx1) and torch.equal(a[1], yy1), "parent and this build gather different windows"
    for _ in range(rounds):
        for name, (fn, _) in forms.items():                    # alternated
            tot[name] += sum(time_launch(fn, flush) for _ in range(n))
    for name, (fn, nbytes) in forms.items():
        res[name] = row(name, tot[name] / (n * rounds), nbytes)
    return res


def joint_model():
    torch.manual_seed(16)
    model = fno_aux.FNO2d(num_channels=V, modes1=12, modes2=12, width=20, initial_step=T0).cuda()
    groups = [{"params": model.shared_layers.parameters(), "lr": 1e-3},
              {"params": model.fc2_primary.parameters(), "lr": 2e-3},
              {"params": model.fc2_auxiliary.parameters(), "lr": 2e-3}]
    step = FusedTrainStep(model, lr=1e-3, weight_decay=1e-4, t_max=100000, graph=True, alias_inputs=True, max_graphs=4,
                          auxiliary_weight=AUX_W, param_groups=groups)
    return model, step


def joined_vs_separate(ds, steps, rounds):
    joint = ds.batch(torch.arange(B2))
    separate = tuple(t.clone() for t in joint)
    assert fno_aux.is_joined(joint[0], joint[3]) and not fno_aux.is_joined(separate[0], separate[3])
    runs = {"joined views": (joint, joint_model()[1]), "separate tensors": (separate, joint_model()[1])}
    tot = {k: 0.0 for k in runs}
    for batch, step in runs.values():
        for _ in range(5):
            step(*batch)
    torch.cuda.synchronize()
    for _ in range(rounds):
        for name, (batch, step) in runs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                out = step(*batch)
            e1.record()
            torch.cuda.synchronize()
            tot[name] += e0.elapsed_time(e1)
            assert torch.isfinite(out).all()
    res = {}
    for name in runs:
        ms = tot[name] / (steps * rounds)
        print(f"  graphed cfg-2 step on {name:16s}: {ms:7.3f} ms/step", flush=True)
        res[name] = round(ms, 4)
    return res


def streamed(ds, steps, rounds):
    """Returns (streamed, host-batch) dicts: samples/s of primary items and H2D bytes per step."""
    h_traj, h_aux = ds.traj.cpu().pin_memory(), ds.traj_aux.cpu().pin_memory()
    stores = [(ds.traj.view(-1), h_traj.view(-1)), (ds.traj_aux.view(-1), h_aux.view(-1))]
    frames = (B2 * T_TRAJ + ds.n_windows - 1) // ds.n_windows                  # fresh frames per step, per stream
    chunks = [min(d.numel(), frames * X * X * V * m) for (d, _), m in zip(stores, (1, NUM_AUX))]
    gi = torch.Generator().manual_seed(7)
    items_host = [ds.split_items(torch.randint(0, len(ds), (B2,), generator=gi)) for _ in range(2)]
    outs = [ds.joined_buffers(B2) for _ in range(2)]
    up_stream = torch.cuda.Stream()
    up_done = [torch.cuda.Event() for _ in range(2)]
    off = [0, 0]
    loss_host = torch.zeros(2, dtype=torch.float32).pin_memory()
    loss_ev = [torch.cuda.Event() for _ in range(2)]
    _, step = joint_model()

    def upload(i):
        with torch.cuda.stream(up_stream):
            for s, ((d, h), c) in enumerate(zip(stores, chunks)):
                if off[s] + c > d.numel():
                    off[s] = 0
                d[off[s]:off[s] + c].copy_(h[off[s]:off[s] + c], non_blocking=True)
                off[s] += c
            up_done[i % 2].record(up_stream)

    def dev_loop(n):
        cur = torch.cuda.current_stream()
        upload(0)
        cur.wait_event(up_done[0])
        nxt = ds.batch(items_host[0], out=outs[0])
        last = 0.0
        for i in range(n):
            loss_i = step(*nxt)
            loss_host[i % 2:i % 2 + 1].copy_(loss_i.flatten()[:1], non_blocking=True)
            loss_ev[i % 2].record(cur)
            if i + 1 < n:
                upload(i + 1)
                cur.wait_event(up_done[(i + 1) % 2])
                nxt = ds.batch(items_host[(i + 1) % 2], out=outs[(i + 1) % 2])
            loss_ev[i % 2].synchronize()
            last = float(loss_host[i % 2])
        return last

    # host-batch shipping: the assembled tuple (the joint batch itself) from pinned memory
    _, hstep = joint_model()
    host = [tuple(t.cpu().pin_memory() for t in ds.batch(items_host[s])) for s in range(2)]
    h2d_host = sum(t.numel() * t.element_size() for t in host[0])
    bufs = [tuple(torch.empty_like(t, device="cuda") for t in host[0]) for _ in range(2)]
    copy_stream = torch.cuda.Stream()
    ready, consumed = [torch.cuda.Event() for _ in range(2)], [torch.cuda.Event() for _ in range(2)]

    def prefetch(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[i % 2])
            for dst, src in zip(bufs[i % 2], host[i % 2]):
                dst.copy_(src, non_blocking=True)
            ready[i % 2].record(copy_stream)

    def host_loop(n):
        cur = torch.cuda.current_stream()
        for s in range(2):
            consumed[s].record(cur)
        prefetch(0)
        last = 0.0
        for i in range(n):
            if i + 1 < n:
                prefetch(i + 1)
            cur.wait_event(ready[i % 2])
            loss_i = hstep(*bufs[i % 2])
            consumed[i % 2].record(cur)
            last = float(loss_i.flatten()[0])
        return last

    loops = {"streamed (DeviceJointWindows)": dev_loop, "host batches": host_loop}
    tot = {k: 0.0 for k in loops}
    for fn in loops.values():
        fn(6)
    torch.cuda.synchronize()
    for _ in range(rounds):
        for name, fn in loops.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn(steps)
            e1.record()
            torch.cuda.synchronize()
            tot[name] += e0.elapsed_time(e1)
    h2d = {"streamed (DeviceJointWindows)": 4 * sum(chunks) + 12 * B2, "host batches": h2d_host}
    res = {}
    for name in loops:
        ms = tot[name] / (steps * rounds)
        res[name] = dict(samples_per_s=round(B2 / ms * 1e3, 1), ms_per_step=round(ms, 3), h2d_bytes_per_step=h2d[name],
                         d2h_bytes_per_step=4)
        print(f"  cfg-2 e2e {name:30s}: {B2 / ms * 1e3:8.0f} samples/s  {ms:7.3f} ms/step  "
              f"H2D {h2d[name] / 1e6:7.1f} MB/step", flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json", default="")
    ap.add_argument("--launches", type=int, default=30)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--parent-lib", default="", help="libfno_sm100.so of another build: its fno_window_gather is timed "
                                                      "alternated with this build's")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_joint_stream needs a CUDA device")
    info = card()
    print(info, flush=True)
    traj, traj_aux = stores(0)
    ds = data.DeviceJointWindows(traj, traj_aux, T0, 1, device="cuda")
    del traj, traj_aux
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")
    res = dict(card=info, gather=gather_kernels(ds, args.launches, args.rounds, args.parent_lib, flush))
    del flush
    torch.cuda.empty_cache()
    res["graphed_step"] = joined_vs_separate(ds, args.steps, args.rounds)
    torch.cuda.empty_cache()
    res["e2e"] = streamed(ds, args.steps, args.rounds)
    if args.json:
        Path(args.json).parent.mkdir(parents=True, exist_ok=True)
        Path(args.json).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
