"""Rollout training of the two-head joint model on a B200: the split window shift (fno_window_shift_split and its adjoint)
against a torch.cat restatement, the two heads on one trunk activation (ops.TwoHeadFn) against the per-head path it
replaces, joint_rollout_loss against the fp64 torch port unrolled with torch.cat on both streams, its launch count, and
FusedTrainStep(rollout_steps=K, auxiliary_weight=w) in the eager, graphed and aliased forms."""
import pytest
import torch

from oracle import dft_oracle as O
from oracle import fno_port as P
from oracle.make_golden import seeded

pytestmark = pytest.mark.gpu
TOL = 1e-5
NUM_AUX = 3
AUX_W = 0.7


# ---- 1. the kernels ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("na", [0, 2, 5])
def test_window_shift_split_kernel_vs_cat(na):
    """A pure copy: bitwise equal to torch.cat at points_a = 0, mid and all points, odd T0 and V."""
    from fno_b200 import lib

    N, T0, V = 5, 7, 3
    xx = torch.randn(N, 9, 5, T0, V, device="cuda")
    pa = torch.randn(na, 9, 5, 1, V, device="cuda")
    pb = torch.randn(N - na, 9, 5, 1, V, device="cuda")
    out = lib.window_shift_split(xx, pa, pb)
    assert torch.equal(out, torch.cat((xx[..., 1:, :], torch.cat((pa, pb))), dim=-2))

    g = torch.randn_like(xx)
    gxx, ga, gb = lib.window_shift_split_bwd(g, na)
    ref = torch.zeros_like(g)
    ref[..., 1:, :] = g[..., :-1, :]
    assert torch.equal(gxx, ref)
    assert torch.equal(ga, g[:na, ..., -1:, :]) and torch.equal(gb, g[na:, ..., -1:, :])
    for need in ((False, True, True), (True, False, False), (False, False, True)):
        got = lib.window_shift_split_bwd(g, na, need_xx=need[0], need_a=need[1], need_b=need[2])
        for t, r, n in zip(got, (gxx, ga, gb), need):
            assert (t is None) if not n else torch.equal(t, r)
    # the adjoint of the forward: <shift(xx, pa, pb), g> = <xx, gxx> + <pa, gpa> + <pb, gpb>
    lhs = (out.double() * g.double()).sum()
    rhs = sum((a.double() * b.double()).sum() for a, b in ((xx, gxx), (pa, ga), (pb, gb)))
    assert abs(float(lhs - rhs)) < 1e-9 * float(g.double().abs().sum())


def test_window_shift_split_rejections():
    from fno_b200 import lib

    L = lib.load()
    N, T0, V, na = 4, 5, 3, 1
    xx = torch.randn(N, 6, T0, V, device="cuda")
    pa, pb = torch.randn(na, 6, 1, V, device="cuda"), torch.randn(N - na, 6, 1, V, device="cuda")
    out, g = torch.empty_like(xx), torch.randn_like(xx)
    gxx, ga, gb = torch.empty_like(xx), torch.empty_like(pa), torch.empty_like(pb)
    pts = N * 6
    args = lambda pa_pts: (pa_pts, pts, T0, V, None)               # noqa: E731
    ok = L.fno_window_shift_split(xx.data_ptr(), pa.data_ptr(), pb.data_ptr(), out.data_ptr(), *args(na * 6))
    assert ok == 0, L.fno_last_error()
    for bad in (-1, pts + 1):                                      # points_a outside [0, points]
        assert L.fno_window_shift_split(xx.data_ptr(), pa.data_ptr(), pb.data_ptr(), out.data_ptr(), *args(bad)) < 0
        assert L.fno_window_shift_split_bwd(g.data_ptr(), gxx.data_ptr(), ga.data_ptr(), gb.data_ptr(), *args(bad)) < 0
    for dst in (xx, pa, pb):                                       # in place
        assert L.fno_window_shift_split(xx.data_ptr(), pa.data_ptr(), pb.data_ptr(), dst.data_ptr(), *args(na * 6)) < 0
    assert L.fno_window_shift_split(xx.data_ptr(), None, pb.data_ptr(), out.data_ptr(), *args(na * 6)) < 0
    assert L.fno_window_shift_split_bwd(g.data_ptr(), g.data_ptr(), None, None, *args(na * 6)) < 0
    assert L.fno_window_shift_split_bwd(g.data_ptr(), None, None, None, *args(na * 6)) < 0      # nothing to write
    with pytest.raises(lib.FnoError):
        lib.window_shift_split_bwd(g, na, need_xx=False, need_a=False, need_b=False)
    with pytest.raises(lib.FnoError):
        lib.window_shift_split(xx, pa, pb[1:])                     # predictions do not cover the window
    torch.cuda.synchronize()
    assert torch.equal(out, torch.cat((xx[..., 1:, :], torch.cat((pa, pb))), dim=-2))


# ---- 2. the two heads ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C,spatial,V", [(20, (12, 10), 2), (64, (12, 10), 3), (24, (11, 9), 2), (20, (4, 6, 5), 2)])
def test_two_head_fn_equals_per_head_path(C, spatial, V):
    """TwoHeadFn is bitwise the per-head path on slices of h it replaces (outputs, dh and every parameter gradient) for
    the tensor-core head backward (C <= 23), the wide form (C = 64) and the FP32 form (C = 24, padded plane % 4 != 0),
    in 2-D and 3-D."""
    from fno_b200 import lib, ops

    torch.manual_seed(5)
    nb, nt = 2, 2 + 2 * NUM_AUX
    geo = lib.TrunkGeo(spatial, 2 if len(spatial) == 2 else 6)
    h0 = torch.randn((nt, C) + geo.padded, device="cuda")
    stats = torch.stack((torch.randn(nt, V), 0.5 + torch.rand(nt, V)), dim=1).cuda()
    W1, b1 = torch.randn(128, C, device="cuda") / C ** 0.5, torch.randn(128, device="cuda") * 0.1
    W2s = [torch.randn(V, 128, device="cuda") / 128 ** 0.5 for _ in range(2)]
    b2s = [torch.randn(V, device="cuda") * 0.1 for _ in range(2)]
    douts = [torch.randn((n,) + geo.spatial + (V,), device="cuda") for n in (nb, nt - nb)]

    def leaves():
        return [t.clone().requires_grad_(True) for t in (h0, W1, b1, W2s[0], b2s[0], W2s[1], b2s[1])]

    old = leaves()
    h, w1, bb1, w2a, b2a, w2b, b2b = old
    outs_old = (ops.head(h[:nb], w1, bb1, w2a, b2a, stats[:nb].contiguous(), geo),
                ops.head(h[nb:], w1, bb1, w2b, b2b, stats[nb:].contiguous(), geo))
    sum((o * d).sum() for o, d in zip(outs_old, douts)).backward()

    new = leaves()
    outs_new = ops.TwoHeadFn.apply(*new, stats, geo, nb)
    sum((o * d).sum() for o, d in zip(outs_new, douts)).backward()
    for a, b in zip(outs_old, outs_new):
        assert torch.equal(a, b)
    for i, (a, b) in enumerate(zip(old, new)):
        assert torch.equal(a.grad, b.grad), i


def _walk(outs):
    seen, stack, names = set(), [o.grad_fn for o in outs], []
    while stack:
        fn = stack.pop()
        if fn is None or fn in seen:
            continue
        seen.add(fn)
        names.append(fn)
        stack += [n for n, _ in fn.next_functions]
    return names


def test_joint_forward_has_no_slice_backward():
    """Neither head output reaches a SliceBackward0 or a CatBackward0 over the trunk activation; the only CatBackward0
    is the input join when the inputs require grad."""
    model, xshape = _model("aux2d")
    model = model.cuda()
    x, grid, xa, ga = (t.cuda() for t in _joint_inputs(xshape, 300))
    fns = _walk(model(x, grid, xa, ga))
    assert not [f for f in fns if type(f).__name__ in ("SliceBackward0", "CatBackward0")]
    assert any(type(f).__name__ == "TwoHeadFnBackward" for f in fns)
    x.requires_grad_(True)
    xa.requires_grad_(True)
    fns = _walk(model(x, grid, xa, ga))
    assert not [f for f in fns if type(f).__name__ == "SliceBackward0"]
    cats = [f for f in fns if type(f).__name__ == "CatBackward0"]
    assert len(cats) == 1
    assert {id(getattr(n, "variable", None)) for n, _ in cats[0].next_functions} == {id(x), id(xa)}


# ---- 3. joint rollout training -------------------------------------------------------------------------------------
def _model(name):
    from fno_b200 import fno_aux as FA

    torch.manual_seed(16)
    if name == "aux2d":
        return FA.FNO2d(num_channels=2, modes1=4, modes2=4, width=8, initial_step=3), (2, 12, 10, 3, 2)
    return FA.FNO3d(num_channels=2, modes1=3, modes2=3, modes3=3, width=6, initial_step=2), (1, 8, 6, 10, 2, 2)


def _joint_inputs(xshape, seed):
    B, nd = xshape[0], len(xshape) - 3
    ashape = (B * NUM_AUX,) + xshape[1:]
    gen = torch.Generator().manual_seed(seed + 1)
    return (seeded(xshape, seed), torch.rand(xshape[:-2] + (nd,), generator=gen), seeded(ashape, seed + 2),
            torch.rand(ashape[:-2] + (nd,), generator=gen))


def _joint_data(xshape, K, seed):
    """(xx, yy, grid, xx_aux, yy_aux, grid_aux) with K target frames on both streams."""
    x, grid, xa, ga = _joint_inputs(xshape, seed)
    yy = seeded(xshape[:-2] + (K, xshape[-1]), seed + 3)
    ya = seeded(xa.shape[:-2] + (K, xshape[-1]), seed + 4)
    return x, yy, grid, xa, ya, ga


@pytest.mark.parametrize("name", ["aux2d", "aux3d"])
def test_joint_rollout_loss_vs_port(name):
    from fno_b200.train import joint_rollout_loss

    K = 3
    model, xshape = _model(name)
    p = P.as_leaves(model.state_dict(), dtype=torch.float64)
    xx, yy, grid, xa, ya, ga = _joint_data(xshape, K, 400)
    x, xa_ref, ref = xx.double(), xa.double(), []
    for k in range(K):
        op, oa = P.fno_aux_forward(p, x, grid.double(), xa_ref, ga.double())
        ref.append(torch.stack((P.nrmse(op, yy[..., k:k + 1, :].double()).mean(),
                                P.nrmse(oa, ya[..., k:k + 1, :].double()).mean())))
        if k + 1 < K:
            x = torch.cat((x[..., 1:, :], op), dim=-2)
            xa_ref = torch.cat((xa_ref[..., 1:, :], oa), dim=-2)
    ref = torch.stack(ref)
    ref_loss = (ref[:, 0] + AUX_W * ref[:, 1]).mean()
    ref_loss.backward()

    model = model.cuda()
    loss, per_step = joint_rollout_loss(model, *(t.cuda() for t in (xx, yy, grid, xa, ya, ga)), K, AUX_W)
    loss.backward()
    assert per_step.shape == (K, 2)
    assert abs(loss.item() - ref_loss.item()) <= TOL * abs(ref_loss.item())
    assert O.rel_err(per_step.detach().cpu().numpy(), ref.detach().numpy()) < TOL
    n = 0
    for k, q in model.named_parameters():
        if q.grad is None:                                   # FNO3d's never-called bn*
            assert p[k].grad is None, k
            continue
        assert O.rel_err(q.grad.cpu().numpy(), p[k].grad.numpy()) < 2e-5, k
        n += 1
    assert n >= 20


def _groups(model):
    # the joint loop's three Adam groups (fno_train_aux.py:175-179)
    return [{"params": model.shared_layers.parameters(), "lr": 1e-3},
            {"params": model.fc2_primary.parameters(), "lr": 2e-3},
            {"params": model.fc2_auxiliary.parameters(), "lr": 2e-3}]


def _step_run(rollout_steps, graph, n, data, **kw):
    """n joint FusedTrainSteps from the same seeded model; rollout_steps=None constructs the step without it."""
    from fno_b200.train import FusedTrainStep

    model, _ = _model("aux2d")
    model = model.cuda()
    if rollout_steps is not None:
        kw["rollout_steps"] = rollout_steps
    step = FusedTrainStep(model, lr=1e-3, weight_decay=1e-4, t_max=100, graph=graph, auxiliary_weight=AUX_W,
                          param_groups=_groups(model), **kw)
    outs = []
    for i in range(n):
        outs.append(step(*(t.cuda() for t in data(i))).clone())
    torch.cuda.synchronize()
    return torch.stack(outs), {k: v.detach().clone() for k, v in model.state_dict().items()}


def test_fused_joint_step_rollout_one_is_todays_step():
    """rollout_steps=1 is bitwise today's joint FusedTrainStep over three steps, and so is a step on
    joint_rollout_loss(steps=1): the mean over one step is the single-step joint loss lp + w la."""
    from fno_b200.steptail import FusedClipAdam
    from fno_b200.train import joint_rollout_loss

    xshape = _model("aux2d")[1]
    data = lambda i: _joint_data(xshape, 1, 500 + 10 * i)          # noqa: E731
    a_loss, a_sd = _step_run(None, False, 3, data)
    b_loss, b_sd = _step_run(1, False, 3, data)
    assert a_loss.shape == (3, 2)
    assert torch.equal(a_loss, b_loss)
    for k in a_sd:
        assert torch.equal(a_sd[k], b_sd[k]), k
    model, _ = _model("aux2d")
    model = model.cuda()
    opt = FusedClipAdam(_groups(model), lr=1e-3, weight_decay=1e-4, t_max=100)
    losses = []
    for i in range(3):
        loss, per_step = joint_rollout_loss(model, *(t.cuda() for t in data(i)), 1, AUX_W)
        opt.zero_grad()
        loss.backward()
        opt.step()
        losses.append(per_step.detach()[0].clone())
    assert torch.equal(torch.stack(losses), a_loss)
    for k, v in model.state_dict().items():
        assert torch.equal(v, a_sd[k]), k


def test_fused_joint_step_rollout_graph_equals_eager():
    """rollout_steps=3: two eager warm-up steps, the capture step, then three replays -- copying and aliasing forms --
    are bitwise the eager steps."""
    K, n = 3, 6
    xshape = _model("aux2d")[1]
    data = lambda i: _joint_data(xshape, K, 600 + 10 * i)          # noqa: E731
    e_loss, e_sd = _step_run(K, False, n, data)
    assert e_loss.shape == (n, K, 2) and torch.isfinite(e_loss).all()
    for kw in ({}, {"alias_inputs": True}):
        g_loss, g_sd = _step_run(K, True, n, data, **kw)
        assert torch.equal(e_loss, g_loss), kw
        for k in e_sd:
            assert torch.equal(e_sd[k], g_sd[k]), (k, kw)


def test_joint_rollout_launch_count():
    """Each fed-back step adds exactly one split shift, its adjoint and one fno_lift_dgrad to K copies of the
    single-step loss + backward."""
    from fno_b200 import lib
    from fno_b200.train import joint_rollout_loss

    model, xshape = _model("aux2d")
    model = model.cuda()
    batch = [t.cuda() for t in _joint_data(xshape, 4, 700)]

    def launches(K):
        model.zero_grad(set_to_none=True)
        l0 = lib.launch_count()
        joint_rollout_loss(model, *batch, K, AUX_W)[0].backward()
        return lib.launch_count() - l0

    for K in (1, 2, 4):                                      # warm-up
        launches(K)
    L1 = launches(1)
    for K in (2, 3, 4):
        assert launches(K) == K * L1 + 3 * (K - 1), K


def test_joint_rollout_rejections():
    from fno_b200 import lib
    from fno_b200.train import FusedTrainStep, joint_rollout_loss

    model, xshape = _model("aux2d")
    model = model.cuda()
    xx, yy, grid, xa, ya, ga = (t.cuda() for t in _joint_data(xshape, 3, 800))
    short = ya[..., :2, :].contiguous()
    with pytest.raises(lib.FnoError):
        joint_rollout_loss(model, xx, yy, grid, xa, short, ga, 3, AUX_W)
    with pytest.raises(lib.FnoError):
        joint_rollout_loss(model, xx, yy[..., :2, :], grid, xa, ya, ga, 3, AUX_W)
    with pytest.raises(lib.FnoError):
        joint_rollout_loss(model, xx, yy, grid, xa, ya, ga, 0, AUX_W)
    step = FusedTrainStep(model, rollout_steps=3, auxiliary_weight=AUX_W)     # the two-head model has a rollout form
    with pytest.raises(lib.FnoError):
        step(xx, yy, grid, xa, short, ga)
    with pytest.raises(lib.FnoError):
        step(xx, yy[..., :2, :].contiguous(), grid, xa, ya, ga)
