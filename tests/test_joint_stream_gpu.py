"""Streaming data for the two-head joint model: fno_window_gather_joint and data.DeviceJointWindows against host-side
windows and the reference-layout joint dataset, the zero-copy joined forward (fno_aux.joined), and FusedTrainStep fed
from the device-resident joint dataset against the same step fed host-assembled separate tensors."""
import json

import pytest
import torch


gpu = pytest.mark.gpu
AUX_W = 0.7


def _stores(n, T, spatial, V, A, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn((n, T) + spatial + (V,), generator=g), torch.randn((n, A, T) + spatial + (V,), generator=g)


def _host_joint(traj, traj_aux, T0, R, items):
    """Host-side windows per stream, the auxiliary ones flattened [B * A, ...] item-major as the joint loop has them."""
    from fno_b200 import data

    xx, yy = data.windows(traj, T0, R)
    per = [data.windows(traj_aux[:, k], T0, R) for k in range(traj_aux.shape[1])]
    xa, ya = torch.stack([p[0] for p in per], dim=1), torch.stack([p[1] for p in per], dim=1)
    return xx[items], yy[items], xa[items].flatten(0, 1), ya[items].flatten(0, 1)


# ---- 1. the gather ---------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("spatial,V,T,T0", [((16, 12), 2, 9, 4), ((13, 11), 3, 10, 3), ((6, 5, 3), 2, 8, 4)])
@pytest.mark.parametrize("A", [1, 3])
@pytest.mark.parametrize("R", [1, 3])
def test_joint_gather_matches_host_windows(spatial, V, T, T0, A, R):
    """Bitwise against data.windows per stream (16-byte-store and scalar forms of the kernel), and the single-stream
    gather (its A = 0 case) bitwise on the same cases."""
    from fno_b200 import data

    traj, traj_aux = _stores(5, T, spatial, V, A, 11 * A + R)
    ds = data.DeviceJointWindows(traj, traj_aux, T0, R, device="cuda")
    assert len(ds) == 5 * (T - T0 - R + 1) and ds.A == A
    items = torch.randperm(len(ds), generator=torch.Generator().manual_seed(2))[:7]
    xx, yy, grid, xa, ya, ga = ds.batch(items)
    ref = _host_joint(traj, traj_aux, T0, R, items)
    for got, want in zip((xx, yy, xa, ya), ref):
        assert got.shape == want.shape and torch.equal(got.cpu(), want)
    assert xa.data_ptr() == xx.data_ptr() + xx.numel() * 4 and ga.data_ptr() == grid.data_ptr() + grid.numel() * 4
    assert tuple(grid.shape) == (7,) + spatial + (len(spatial),) and tuple(ga.shape) == (7 * A,) + spatial + (len(spatial),)
    assert torch.equal(ga.cpu(), grid.cpu()[:1].expand_as(ga)) and torch.equal(grid.cpu(), ds.grid.cpu().expand_as(grid))
    sx, sy, _ = data.DeviceWindows(traj, T0, R, device="cuda").batch(items)
    assert torch.equal(sx.cpu(), ref[0]) and torch.equal(sy.cpu(), ref[1])
    # caller-owned buffers and the (ti, ts) form of the items give the same batch
    bufs = ds.joined_buffers(7)
    again = ds.batch(ds.split_items(items), out=bufs)
    assert again[0].data_ptr() == bufs[0].data_ptr() and again[4].data_ptr() == bufs[2].data_ptr()
    for got, want in zip(again, (xx, yy, grid, xa, ya, ga)):
        assert torch.equal(got, want)


@gpu
def test_joint_items_pair_like_the_reference_dataset(monkeypatch):
    """Item i is AuxFNODatasetMult[i] (the dataset of the golden joint-loop fixture): the auxiliary windows of an item come
    from the auxiliary trajectories of the item's own trajectory, at the same start."""
    from fno_b200 import data
    from oracle import ref_datasets

    cfg = {"train_traj": 3, "val_traj": 1, "n": 16, "windows": 4, "initial_step": 5, "num_channels": 2,
           "train_seed": 21, "val_seed": 22, "aux_seed": 23}
    monkeypatch.setenv("FNO_REF_DATA", json.dumps(cfg))
    A, T = 3, cfg["initial_step"] + 1 + cfg["windows"] - 1
    ref = ref_datasets.AuxFNODatasetMult(num_aux_samples=A)
    traj = data.diffusion_trajectories(cfg["train_traj"], cfg["n"], T, cfg["num_channels"], cfg["train_seed"])
    traj_aux = torch.stack([data.diffusion_trajectories(cfg["train_traj"], cfg["n"], T, cfg["num_channels"],
                                                        cfg["aux_seed"] + 17 * k, diffusivity=(3e-3 * (k + 1), 3e-2 * (k + 1)))
                            for k in range(A)], dim=1)
    ds = data.DeviceJointWindows(traj, traj_aux, cfg["initial_step"], 1, device="cuda")
    assert len(ds) == len(ref)
    items = torch.arange(len(ds))
    xx, yy, grid, xa, ya, ga = (t.cpu() for t in ds.batch(items))
    for i in range(len(ref)):
        r = ref[i]
        assert torch.equal(xx[i], r[0]) and torch.equal(yy[i], r[1])
        assert torch.equal(xa[i * A:(i + 1) * A], r[2]) and torch.equal(ya[i * A:(i + 1) * A], r[3])
        assert torch.allclose(grid[i], r[4], rtol=0, atol=1e-6) and torch.allclose(ga[i * A], r[5], rtol=0, atol=1e-6)


# ---- 2. rejections ---------------------------------------------------------------------------------------------------
@gpu
def test_joint_gather_rejections():
    from fno_b200 import lib

    L = lib.load()
    B, A, npix, T, V, T0, R = 2, 3, 64, 8, 2, 4, 1
    traj = torch.zeros(4, npix, T, V, device="cuda")
    traj_aux = torch.zeros(4, A, npix, T, V, device="cuda")
    ti = torch.zeros(B, dtype=torch.int64, device="cuda")
    ts = torch.zeros(B, dtype=torch.int32, device="cuda")
    xj = torch.empty(B * (1 + A), npix, T0, V, device="cuda")
    yy, ya = torch.empty(B, npix, R, V, device="cuda"), torch.empty(B * A, npix, R, V, device="cuda")
    st = torch.cuda.current_stream().cuda_stream

    def call(traj_p=traj.data_ptr(), aux_p=traj_aux.data_ptr(), xj_p=xj.data_ptr(), yy_p=yy.data_ptr(),
             ya_p=ya.data_ptr(), b=B, a=A, n=npix, t=T, t0=T0):
        return L.fno_window_gather_joint(traj_p, aux_p, ti.data_ptr(), ts.data_ptr(), xj_p, yy_p, ya_p, b, a, n, t, V,
                                         t0, R, st)

    assert call() == 0
    torch.cuda.synchronize()
    cases = {"A = -1": dict(a=-1), "needs traj_aux": dict(aux_p=None), "longer than": dict(t0=T),
             "32 bits": dict(b=2000, n=1 << 20, t0=10, t=20), "aliases": dict(xj_p=traj.data_ptr()),
             "aliases ": dict(ya_p=traj_aux.data_ptr() + 64)}
    for msg, kw in cases.items():
        assert call(**kw) == -1, msg
        assert msg.strip().encode() in L.fno_last_error(), (msg, L.fno_last_error())
    # the single-stream entry point keeps its checks
    assert L.fno_window_gather(traj.data_ptr(), ti.data_ptr(), ts.data_ptr(), traj.data_ptr(), yy.data_ptr(), B, npix,
                               T, V, T0, R, st) == -1
    assert L.fno_window_gather(traj.data_ptr(), ti.data_ptr(), ts.data_ptr(), xj.data_ptr(), yy.data_ptr(), B, npix,
                               T, V, T, R, st) == -1
    # the Python wrapper checks shapes and caller-owned buffers against the whole store
    with pytest.raises(lib.FnoError):
        lib.window_gather_joint(traj, traj_aux[:3], ti, ts, T0, R)
    with pytest.raises(lib.FnoError, match="aliases"):
        lib.window_gather_joint(traj, traj_aux, ti, ts, T0, R, out=(traj_aux.view(-1)[-xj.numel():], yy, ya))
    with pytest.raises(lib.FnoError, match="wrong|needs"):
        lib.window_gather_joint(traj, traj_aux, ti, ts, T0, R, out=(xj[1:], yy, ya))


def test_joint_dataset_constructor_rejections():
    """Checked before anything reaches the device."""
    from fno_b200 import data

    traj, traj_aux = _stores(3, 6, (8, 8), 2, 2, 0)
    data.DeviceJointWindows(traj, traj_aux, 4, 1, device="cpu")
    with pytest.raises(ValueError, match="shorter"):
        data.DeviceJointWindows(traj, traj_aux, 5, 2, device="cpu")
    bad = {"trajectory count": traj_aux[:2], "frame count": traj_aux[:, :, :5], "channel count": traj_aux[..., :1],
           "spatial shape": traj_aux[:, :, :, :7], "A >= 1": traj_aux[:, :0], "must be": traj_aux[:, 0]}
    for msg, aux in bad.items():
        with pytest.raises(ValueError, match=msg):
            data.DeviceJointWindows(traj, aux, 4, 1, device="cpu")


# ---- 3. the zero-copy joined forward ---------------------------------------------------------------------------------
def _model():
    from fno_b200 import fno_aux as FA

    torch.manual_seed(16)
    return FA.FNO2d(num_channels=2, modes1=4, modes2=4, width=8, initial_step=3).cuda()


def _dataset(R, A=3, spatial=(12, 10), seed=5):
    from fno_b200 import data

    traj, traj_aux = _stores(3, 9, spatial, 2, A, seed)
    return data.DeviceJointWindows(traj, traj_aux, 3, R, device="cuda")


def _fwd_bwd(model, batch):
    from fno_b200.steptail import nrmse_loss

    model.zero_grad(set_to_none=True)
    xx, yy, grid, xa, ya, ga = batch
    p, a = model(xx, grid, xa, ga)
    loss = nrmse_loss(p, yy) + AUX_W * nrmse_loss(a, ya)
    loss.backward()
    return p.detach().clone(), a.detach().clone(), {k: q.grad.clone() for k, q in model.named_parameters()}


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


@gpu
def test_joined_forward_is_bitwise_and_copies_nothing():
    from fno_b200 import fno_aux

    model, ds = _model(), _dataset(1)
    joint = ds.batch(torch.tensor([0, 4, 9, 13]))
    separate = tuple(t.cpu().cuda() for t in joint)              # host-assembled: one allocation per tensor
    assert fno_aux.is_joined(joint[0], joint[3]) and fno_aux.is_joined(joint[2], joint[5])
    assert not fno_aux.is_joined(separate[0], separate[3])
    assert fno_aux.joined(joint[0], joint[3]).data_ptr() == joint[0].data_ptr()
    a, b = _fwd_bwd(model, joint), _fwd_bwd(model, separate)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    for k in a[2]:
        assert torch.equal(a[2][k], b[2][k]), k

    def copies(names):
        return [n for n in names if "CatArray" in n or "copy" in n.lower()]      # torch.cat, copy_ / .contiguous(), memcpy

    assert copies(_kernels(lambda: _fwd_bwd(model, separate))), "the separate inputs are concatenated"
    assert not copies(_kernels(lambda: _fwd_bwd(model, joint)))
    # an input that requires grad takes the concatenating path, with the same results and gradients
    grads = []
    for batch in (joint, separate):
        x = batch[0].clone().requires_grad_()
        assert not fno_aux.is_joined(x, batch[3])
        _fwd_bwd(model, (x,) + batch[1:])
        grads.append(x.grad)
    assert grads[0] is not None and torch.equal(grads[0], grads[1])


# ---- 4. training through the dataset ---------------------------------------------------------------------------------
def _groups(model):
    # the joint loop's three Adam groups (fno_train_aux.py:175-179)
    return [{"params": model.shared_layers.parameters(), "lr": 1e-3},
            {"params": model.fc2_primary.parameters(), "lr": 2e-3},
            {"params": model.fc2_auxiliary.parameters(), "lr": 2e-3}]


def _train(ds, plan, K, joined):
    from fno_b200.train import FusedTrainStep

    model = _model()
    step = FusedTrainStep(model, lr=1e-3, weight_decay=1e-4, t_max=100, graph=True, alias_inputs=True,
                          auxiliary_weight=AUX_W, param_groups=_groups(model), rollout_steps=K)
    outs = [ds.joined_buffers(len(plan[0])) for _ in range(2)]        # double-buffered, fixed addresses
    losses = []
    for i, items in enumerate(plan):
        batch = ds.batch(items, out=outs[i % 2])
        if not joined:
            batch = tuple(t.cpu().cuda() for t in batch)
        losses.append(step(*batch).clone())
    torch.cuda.synchronize()
    return torch.stack(losses), {k: v.detach().clone() for k, v in model.state_dict().items()}, step


@gpu
@pytest.mark.parametrize("R", [1, 2])
def test_fused_step_fed_by_joint_dataset(R):
    """Graphed, aliased FusedTrainStep on DeviceJointWindows batches (two double-buffered out= sets) is bitwise the same
    step fed the same items as separate host-assembled tensors; R = 2 trains a two-step rollout."""
    ds = _dataset(R)
    g = torch.Generator().manual_seed(R)
    plan = [torch.randperm(len(ds), generator=g)[:3] for _ in range(7)]
    a_loss, a_sd, step = _train(ds, plan, R, True)
    b_loss, b_sd, _ = _train(ds, plan, R, False)
    assert a_loss.shape == ((7, 2) if R == 1 else (7, R, 2)) and torch.isfinite(a_loss).all()
    assert len(step._aliased) == 2                               # one graph per out= set, replayed in place
    assert torch.equal(a_loss, b_loss)
    for k in a_sd:
        assert torch.equal(a_sd[k], b_sd[k]), k


@gpu
def test_copying_graph_keeps_joined_inputs_joined():
    """Without alias_inputs the graph's static inputs are one joined buffer per pair when the call's inputs are joined,
    so the captured forward does not concatenate."""
    from fno_b200 import fno_aux
    from fno_b200.train import FusedTrainStep

    ds = _dataset(1)
    model = _model()
    step = FusedTrainStep(model, graph=True, auxiliary_weight=AUX_W, param_groups=_groups(model))
    for i in range(4):
        step(*ds.batch(torch.arange(i, i + 3)))
    s = step._static_in
    assert fno_aux.is_joined(s[0], s[3]) and fno_aux.is_joined(s[2], s[5])
    step2 = FusedTrainStep(_model(), graph=True, auxiliary_weight=AUX_W)
    for i in range(3):
        step2(*(t.cpu().cuda() for t in ds.batch(torch.arange(i, i + 3))))
    assert not fno_aux.is_joined(step2._static_in[0], step2._static_in[3])


# ---- 5. epochs -------------------------------------------------------------------------------------------------------
@gpu
def test_joint_epoch_over_two_ranks():
    from fno_b200 import data

    ds = _dataset(1, A=3)                                        # trunk batch <= 3 * (1 + 3) = 12
    n, batch, world = len(ds), 5, 2                             # 18 items: the last global batch is ragged
    seen = []
    for r in range(world):
        plan = data.epoch_plan(n, batch, True, 16, 0, r, world)
        got = list(ds.epoch(batch, rank=r, world=world, with_weight=True))
        assert len(got) == len(plan)
        for (items, w), b in zip(plan, got):
            assert len(b) == 7 and b[6] == w
            want = ds.batch(items)
            for x, y in zip(b[:6], want):
                assert torch.equal(x, y)
            if w > 0:
                seen += items.tolist()
    assert sorted(seen) == list(range(n))
    with pytest.raises(ValueError, match="DeviceJointWindows.epoch"):
            list(ds.epoch(batch, rank=0, world=world))
