"""Gradients through the model input on a B200: the lift data gradient (fno_lift_dgrad) against a numpy restatement of
its formula, the modules' x.grad / grid.grad against the fp64 torch port of the reference on the CPU, the launch cost of
asking for them, and rollout training (rollout_loss, FusedTrainStep(rollout_steps=K)) against the port unrolled with a
torch.cat shift."""
import numpy as np
import pytest
import torch

from oracle import dft_oracle as O
from oracle import fno_port as P
from oracle.make_golden import seeded

pytestmark = pytest.mark.gpu
TOL = 1e-5


# ---- 1. the kernel -------------------------------------------------------------------------------------------------
def _dgrad_reference(dh, W0, stats, geo, T, V, G):
    """fp64 numpy: dx[b,p,t,v] = (1/sd[b,v]) sum_c W0[c,tV+v] dh[b,c,off(p)], dgrid[b,p,g] = sum_c W0[c,TV+g] dh[..]."""
    B, C = dh.shape[:2]
    dhv = dh.reshape(B, C, geo.R_out, geo.Wp)[:, :, :geo.R_in, :geo.W_in].reshape(B, C, -1).astype(np.float64)
    W = W0.astype(np.float64)
    F1 = T * V
    sd = stats[:, 1, :].astype(np.float64)                                  # [B, V], already + 1e-7
    rs = (1.0 / sd)[:, np.tile(np.arange(V), T)]                            # [B, F1]: 1 / sd[b, f % V]
    dx = np.einsum("bcp,cf->bpf", dhv, W[:, :F1]) * rs[:, None, :]
    dgrid = np.einsum("bcp,cf->bpf", dhv, W[:, F1:])
    return dx.reshape(B, -1, T, V), dgrid


@pytest.mark.parametrize("TV", [(10, 2), (3, 3), (1, 1), (10, 3)])
@pytest.mark.parametrize("C", [8, 20, 24, 64])
@pytest.mark.parametrize("G", [2, 3])
@pytest.mark.parametrize("nd", [2, 3])
def test_lift_dgrad_kernel_vs_numpy(nd, G, C, TV):
    """Odd W_in with a partial second row tile (2-D) / the 3-D rows-of-(X, Y) geometry; NaN in the padding of dh proves
    it is never read; dx-only, dgrid-only and both; a dx that is not 16-byte aligned."""
    from fno_b200 import lib

    T, V = TV
    B = 2
    spatial = (5, 67) if nd == 2 else (3, 4, 9)
    geo = lib.TrunkGeo(spatial, 2 if nd == 2 else 6)
    rng = np.random.default_rng(1000 * nd + 100 * G + C + 10 * T + V)
    dh = np.full((B, C) + geo.padded, np.nan, dtype=np.float32)
    valid = rng.standard_normal((B, C, geo.R_in, geo.W_in)).astype(np.float32)
    dh.reshape(B, C, geo.R_out, geo.Wp)[:, :, :geo.R_in, :geo.W_in] = valid
    W0 = (rng.standard_normal((C, T * V + G)) / np.sqrt(T * V + G)).astype(np.float32)
    stats = np.stack([rng.standard_normal((B, V)), 0.1 + rng.random((B, V))], axis=1).astype(np.float32)
    ref_dx, ref_dg = _dgrad_reference(dh, W0, stats, geo, T, V, G)
    dht, W0t, st = (torch.from_numpy(a).cuda() for a in (dh, W0, stats))
    npix = geo.npix
    L = lib.load()
    for need_dx, need_dg, offset in ((True, True, 0), (True, False, 1), (False, True, 0), (True, True, 1)):
        dx_buf = torch.full((B * npix * T * V + offset,), float("nan"), device="cuda")
        dg_buf = torch.full((B * npix * G + offset,), float("nan"), device="cuda")
        dx_ptr = dx_buf.data_ptr() + 4 * offset if need_dx else None
        dg_ptr = dg_buf.data_ptr() + 4 * offset if need_dg else None
        rc = L.fno_lift_dgrad(dht.data_ptr(), W0t.data_ptr(), st.data_ptr(), dx_ptr, dg_ptr, B, *geo.ints, T, V, G, C,
                              torch.cuda.current_stream().cuda_stream)
        assert rc == 0, L.fno_last_error()
        torch.cuda.synchronize()
        if need_dx:
            got = dx_buf[offset:].cpu().numpy().reshape(ref_dx.shape)
            assert np.isfinite(got).all()
            assert O.rel_err(got, ref_dx) < TOL
        else:
            assert torch.isnan(dx_buf).all()
        if need_dg:
            got = dg_buf[offset:].cpu().numpy().reshape(ref_dg.shape)
            assert np.isfinite(got).all()
            assert O.rel_err(got, ref_dg) < TOL
        else:
            assert torch.isnan(dg_buf).all()
    # both outputs NULL is an argument error, not a silent no-op
    assert L.fno_lift_dgrad(dht.data_ptr(), W0t.data_ptr(), st.data_ptr(), None, None, B, *geo.ints, T, V, G, C,
                            None) < 0


def test_window_shift_bwd_kernel():
    from fno_b200 import lib

    g = torch.randn(3, 7, 5, 4, 2, device="cuda")
    gxx, gpred = lib.window_shift_bwd(g)
    ref = torch.zeros_like(g)
    ref[..., 1:, :] = g[..., :-1, :]
    assert torch.equal(gxx, ref) and torch.equal(gpred, g[..., -1:, :])
    assert lib.window_shift_bwd(g, need_xx=False)[0] is None and torch.equal(lib.window_shift_bwd(g, need_xx=False)[1],
                                                                             gpred)
    assert torch.equal(lib.window_shift_bwd(g, need_pred=False)[0], ref)
    with pytest.raises(lib.FnoError):
        lib.window_shift_bwd(g, need_xx=False, need_pred=False)
    # the adjoint of the forward: <shift(xx, pred), g> = <xx, gxx> + <pred, gpred>
    xx, pred = torch.randn_like(g), torch.randn(3, 7, 5, 1, 2, device="cuda")
    lhs = (lib.window_shift(xx, pred).double() * g.double()).sum()
    rhs = (xx.double() * gxx.double()).sum() + (pred.double() * gpred.double()).sum()
    assert abs(float(lhs - rhs)) < 1e-9 * float(g.double().abs().sum())


# ---- 2. the modules ------------------------------------------------------------------------------------------------
def _model(name):
    from fno_b200 import fno as F
    from fno_b200 import fno_aux as FA

    torch.manual_seed(16)
    if name == "fno2d":
        return F.FNO2d(num_channels=2, modes1=4, modes2=4, width=8, initial_step=3), (2, 12, 10, 3, 2)
    if name == "fno3d":
        return F.FNO3d(num_channels=3, modes1=3, modes2=3, modes3=3, width=6, initial_step=2), (2, 8, 6, 10, 2, 3)
    if name == "aux2d":
        return FA.FNO2d(num_channels=2, modes1=4, modes2=4, width=8, initial_step=3), (2, 12, 10, 3, 2)
    if name == "aux3d":
        return FA.FNO3d(num_channels=2, modes1=3, modes2=3, modes3=3, width=6, initial_step=2), (1, 8, 6, 10, 2, 2)
    return F.FNO2d(num_channels=2, modes1=12, modes2=12, width=20, initial_step=10), (2, 128, 128, 10, 2)   # cfg 1


@pytest.mark.parametrize("grid_grad", [False, True])
@pytest.mark.parametrize("name", ["fno2d", "fno3d", "aux2d", "aux3d", "cfg1"])
def test_module_input_grad_vs_cpu_port(name, grid_grad):
    model, xshape = _model(name)
    aux = name.startswith("aux")
    nd = len(xshape) - 3
    gshape = xshape[:-2] + (nd,)
    oshape = xshape[:-2] + (1, xshape[-1])
    inputs = [seeded(xshape, 70), torch.rand(gshape, generator=torch.Generator().manual_seed(71))]
    if aux:
        inputs += [seeded(xshape, 72), torch.rand(gshape, generator=torch.Generator().manual_seed(73))]
    gouts = [seeded(oshape, 74 + k) for k in range(2 if aux else 1)]
    needs = [True, grid_grad] * (2 if aux else 1)

    p = P.as_leaves(model.state_dict(), dtype=torch.float64)
    ref_in = [t.double().requires_grad_(n) for t, n in zip(inputs, needs)]
    ref = P.fno_aux_forward(p, *ref_in) if aux else (P.fno_forward(p, *ref_in),)
    sum((o * g.double()).sum() for o, g in zip(ref, gouts)).backward()

    model = model.cuda()

    def run(want_input_grad):
        dev_in = [t.cuda().requires_grad_(n and want_input_grad) for t, n in zip(inputs, needs)]
        model.zero_grad(set_to_none=True)
        outs = model(*dev_in)
        outs = outs if aux else (outs,)
        sum((o * g.cuda()).sum() for o, g in zip(outs, gouts)).backward()
        return dev_in, {k: q.grad.clone() for k, q in model.named_parameters() if q.grad is not None}

    dev_in, grads = run(True)
    for t, r, n in zip(dev_in, ref_in, needs):
        if n:
            assert t.grad is not None
            assert O.rel_err(t.grad.cpu().numpy(), r.grad.numpy()) < TOL
        else:
            assert t.grad is None
    # the weight-gradient path is untouched: asking for input gradients changes no parameter gradient
    _, plain = run(False)
    assert grads.keys() == plain.keys()
    for k in grads:
        assert torch.equal(grads[k], plain[k]), k


def test_input_grad_costs_exactly_one_launch():
    """The first layer's adjoint already produces dh for the fc0 gradient: x.grad adds the fno_lift_dgrad call and
    nothing else, and a plain x launches exactly what it did before."""
    from fno_b200 import lib

    model, xshape = _model("fno2d")
    model = model.cuda()
    x = seeded(xshape, 80).cuda()
    grid = torch.rand(xshape[:-2] + (2,), device="cuda")

    def launches(req):
        xi = x.clone().requires_grad_(req)
        model.zero_grad(set_to_none=True)
        l0 = lib.launch_count()
        model(xi, grid).square().sum().backward()
        n = lib.launch_count() - l0
        assert (xi.grad is not None) == req
        return n

    launches(True), launches(False)          # warm-up
    assert launches(True) - launches(False) == 1


# ---- 3. rollout training -------------------------------------------------------------------------------------------
def _rollout_data(B=2, K=3, X=16, Y=12, T=3, V=2, seed=90):
    xx = seeded((B, X, Y, T, V), seed)
    yy = seeded((B, X, Y, K, V), seed + 1)
    lin_x, lin_y = torch.linspace(0, 1, X), torch.linspace(0, 1, Y)
    gx, gy = torch.meshgrid(lin_x, lin_y, indexing="ij")
    grid = torch.stack((gx, gy), dim=-1).unsqueeze(0).repeat(B, 1, 1, 1)
    return xx, yy, grid


def test_rollout_loss_vs_port():
    from fno_b200 import fno as F
    from fno_b200.train import rollout_loss

    K = 3
    torch.manual_seed(16)
    model = F.FNO2d(num_channels=2, modes1=4, modes2=4, width=8, initial_step=3)
    p = P.as_leaves(model.state_dict(), dtype=torch.float64)
    xx, yy, grid = _rollout_data(K=K)
    x, ref_losses = xx.double(), []
    for k in range(K):
        pred = P.fno_forward(p, x, grid.double())
        ref_losses.append(P.nrmse(pred, yy[..., k:k + 1, :].double()).mean())
        if k + 1 < K:
            x = torch.cat((x[..., 1:, :], pred), dim=-2)
    ref = torch.stack(ref_losses)
    ref.mean().backward()

    model = model.cuda()
    loss, per_step = rollout_loss(model, xx.cuda(), yy.cuda(), grid.cuda(), K)
    loss.backward()
    assert per_step.shape == (K,)
    assert abs(loss.item() - ref.mean().item()) <= TOL * abs(ref.mean().item())
    assert O.rel_err(per_step.detach().cpu().numpy(), ref.detach().numpy()) < TOL
    for k, q in model.named_parameters():
        assert O.rel_err(q.grad.cpu().numpy(), p[k].grad.numpy()) < 2e-5, k


def _step_run(rollout_steps, graph, n, data, **kw):
    """n FusedTrainSteps from the same seeded model; rollout_steps=None constructs the step without the argument."""
    from fno_b200 import fno as F
    from fno_b200.train import FusedTrainStep

    torch.manual_seed(16)
    model = F.FNO2d(num_channels=2, modes1=4, modes2=4, width=8, initial_step=3).cuda()
    if rollout_steps is not None:
        kw["rollout_steps"] = rollout_steps
    step = FusedTrainStep(model, lr=1e-3, weight_decay=1e-4, t_max=100, graph=graph, **kw)
    outs = []
    for i in range(n):
        xx, yy, grid = data(i)
        outs.append(step(xx.cuda(), yy.cuda(), grid.cuda()).clone())
    torch.cuda.synchronize()
    return torch.stack(outs), {k: v.detach().clone() for k, v in model.state_dict().items()}


def test_fused_step_rollout_one_is_todays_step():
    """rollout_steps=1 is bitwise today's single-step FusedTrainStep over three steps, and so is a step on
    rollout_loss(steps=1): the mean over one step is the single-step loss."""
    from fno_b200 import fno as F
    from fno_b200.steptail import FusedClipAdam
    from fno_b200.train import rollout_loss

    data = lambda i: _rollout_data(K=1, seed=100 + 10 * i)          # noqa: E731
    a_loss, a_sd = _step_run(None, False, 3, data)
    b_loss, b_sd = _step_run(1, False, 3, data)
    assert torch.equal(a_loss, b_loss)
    for k in a_sd:
        assert torch.equal(a_sd[k], b_sd[k]), k
    torch.manual_seed(16)
    model = F.FNO2d(num_channels=2, modes1=4, modes2=4, width=8, initial_step=3).cuda()
    opt = FusedClipAdam(model.parameters(), lr=1e-3, weight_decay=1e-4, t_max=100)
    losses = []
    for i in range(3):
        xx, yy, grid = (t.cuda() for t in data(i))
        loss, per_step = rollout_loss(model, xx, yy, grid, 1)
        opt.zero_grad()
        loss.backward()
        opt.step()
        losses.append(per_step.detach()[0].clone())
    assert torch.equal(torch.stack(losses), a_loss)
    for k, v in model.state_dict().items():
        assert torch.equal(v, a_sd[k]), k


def test_fused_step_rollout_graph_equals_eager():
    """rollout_steps=3: two eager warm-up steps, the capture step, then three replays -- copying and aliasing forms --
    are bitwise the eager steps."""
    K, n = 3, 6
    data = lambda i: _rollout_data(K=K, seed=200 + 10 * i)          # noqa: E731
    e_loss, e_sd = _step_run(K, False, n, data)
    assert e_loss.shape == (n, K) and torch.isfinite(e_loss).all()
    for kw in ({}, {"alias_inputs": True}):
        g_loss, g_sd = _step_run(K, True, n, data, **kw)
        assert torch.equal(e_loss, g_loss), kw
        for k in e_sd:
            assert torch.equal(e_sd[k], g_sd[k]), (k, kw)


def test_fused_step_rollout_rejections():
    from fno_b200 import fno as F
    from fno_b200 import lib
    from fno_b200.train import FusedTrainStep, rollout_loss

    model = F.FNO2d(num_channels=2, modes1=4, modes2=4, width=8, initial_step=3).cuda()
    xx, yy, grid = (t.cuda() for t in _rollout_data(K=2))
    step = FusedTrainStep(model, rollout_steps=3)
    with pytest.raises(lib.FnoError):
        step(xx, yy, grid)                                   # 2 target frames for 3 steps
    with pytest.raises(lib.FnoError):
        rollout_loss(model, xx, yy, grid, 3)
    with pytest.raises(lib.FnoError):
        FusedTrainStep(model, rollout_steps=2, auxiliary_weight=0.5)
    with pytest.raises(lib.FnoError):
        FusedTrainStep(model, rollout_steps=0)
