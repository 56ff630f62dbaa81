"""torch.autograd glue for the sm_100a kernels: the spectral convolution operator and the fused
Fourier layer.  Each Function's forward/backward is a fixed sequence of C-ABI launches on the
current stream (no host sync, no Python arithmetic on tensor values), so a whole trunk can be
captured in a CUDA graph.

Math (SURVEY.md 8a; checked by tests against oracle/dft_oracle.py):
    forward   X = K1(x);  Y = K2(X, W);  y = K3(Y)
    backward  gY = (c/N) K1(g);  gX, gW = K2'(X, gY, W);  gx = K3(gX; c = 1, scale = 1)
"""
from __future__ import annotations

from typing import Sequence

import torch

from . import lib

def _plan_for(x: torch.Tensor, weights: Sequence[torch.Tensor]) -> lib.Plan:
    modes = tuple(weights[0].shape[2:])
    nd = len(modes)
    if nd not in (2, 3) or len(weights) != (2 if nd == 2 else 4):
        raise lib.FnoError("expected 2 corner weights [Ci,Co,m1,m2] (2-D) or 4 [Ci,Co,m1,m2,m3] (3-D)")
    if x.dim() != nd + 2:
        raise lib.FnoError(f"input must be [B, C, {'H, W' if nd == 2 else 'D1, D2, D3'}], got {tuple(x.shape)}")
    return lib.get_plan(x.device, tuple(x.shape[-nd:]), modes)


class SpectralConvFn(torch.autograd.Function):
    """y = irfftn(scatter(einsum(rfftn(x)[corners], W)))  -- fno/fno.py:70-92, :259-288."""

    @staticmethod
    def forward(ctx, x, *weights):
        x = x.contiguous()
        weights = tuple(w.contiguous() for w in weights)
        plan = _plan_for(x, weights)
        X = lib.fwd_transform(plan, x)
        Y = lib.mix_fwd(plan, X, weights)
        y = lib.inv_transform(plan, Y, cmode=1)
        ctx.plan = plan
        ctx.save_for_backward(X, *weights)
        return y

    @staticmethod
    def backward(ctx, g):
        X, *weights = ctx.saved_tensors
        plan = ctx.plan
        g = g.contiguous()
        need_gx = ctx.needs_input_grad[0]
        need_gw = any(ctx.needs_input_grad[1:])
        gY = lib.fwd_transform(plan, g, cmode=1, scale=1.0 / plan.npix)
        gX, gws = lib.mix_bwd(plan, X, gY, weights, need_gx=need_gx, need_gw=need_gw)
        gx = lib.inv_transform(plan, gX, cmode=0, scale=1.0) if need_gx else None
        if gws is None:
            gws = [None] * len(weights)
        return (gx, *gws)


def spectral_conv(x: torch.Tensor, weights: Sequence[torch.Tensor]) -> torch.Tensor:
    return SpectralConvFn.apply(x, *weights)


class FourierLayerFn(torch.autograd.Function):
    """a' = act(SpectralConv(a) + Conv1x1(a)),  act = exact GELU or identity (fno/fno.py:161-178).

    Forward launches: bypass -> K1 -> K2 -> K3(+bypass, +GELU).  Saved for backward: a, the
    pre-activation s (exact-erf GELU is not invertible from its output), the spectrum X.
    Backward launches: K1(g * gelu'(s)) [stores dS] -> bypass weight/bias gradient ->
    K2' -> bypass^T(dS) -> K3(gX) + bypass^T.
    """

    @staticmethod
    def forward(ctx, a, wl, bl, apply_gelu, *weights):
        a = a.contiguous()
        weights = tuple(w.contiguous() for w in weights)
        wl = wl.contiguous()
        plan = _plan_for(a, weights)
        training = any(ctx.needs_input_grad)
        fused = lib.layer_fused_supported(plan, a.shape[1]) and wl.shape[0] == wl.shape[1] == a.shape[1]
        if fused:
            # K1 -> K2 -> one tensor-core pass: K3 + bypass + bias + GELU (layer2d_tc.cu); `lin` never exists
            X = lib.fwd_transform(plan, a)
            Y = lib.mix_fwd(plan, X, weights)
            s = torch.empty_like(a) if (training and apply_gelu) else None
            out = lib.layer_inv_fused(plan, Y, a, wl, bl, s_out=s, cmode=1, apply_gelu=bool(apply_gelu))
        else:
            lin = lib.pointwise_fwd(a, wl, bl)
            X = lib.fwd_transform(plan, a)
            Y = lib.mix_fwd(plan, X, weights)
            s = torch.empty_like(lin) if (training and apply_gelu) else None
            out = lib.inv_transform(plan, Y, addend=lin, s_out=s, out=lin, cmode=1, apply_gelu=apply_gelu)
        if training:
            ctx.plan = plan
            ctx.apply_gelu = bool(apply_gelu)
            ctx.has_bias = bl is not None
            ctx.fused = fused
            ctx.save_for_backward(a, wl, X, s if s is not None else a.new_empty(0), *weights)
        return out

    @staticmethod
    def backward(ctx, g):
        a, wl, X, s, *weights = ctx.saved_tensors
        plan = ctx.plan
        g = g.contiguous()
        need_ga, need_wl, need_bl = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        need_gw = any(ctx.needs_input_grad[4:])
        inv_n = 1.0 / plan.npix
        if ctx.apply_gelu:
            ds = torch.empty_like(g)
            gY = lib.fwd_transform(plan, g, preact=s, ds_out=ds, cmode=1, scale=inv_n)
        else:
            ds = g
            gY = lib.fwd_transform(plan, g, cmode=1, scale=inv_n)
        gwl = gbl = None
        ga_lin = None
        if ctx.fused:
            # bypass weight / bias gradient, then K2', then the data gradient K3(gX) + Wl^T dS in one tensor-core pass
            if need_wl or (need_bl and ctx.has_bias):
                gwl, gbl = lib.pointwise_wgrad(ds, a, wl.shape, need_bias=ctx.has_bias)
            gX, gws = lib.mix_bwd(plan, X, gY, weights, need_gx=need_ga, need_gw=need_gw)
            ga = lib.layer_inv_fused(plan, gX, ds, wl, None, cmode=0, scale=1.0, transpose=True) if need_ga else None
            if gws is None:
                gws = [None] * len(weights)
            return (ga, gwl if need_wl else None, gbl if (need_bl and ctx.has_bias) else None, None, *gws)
        if need_ga and need_wl:
            # weight, bias and data gradient of the bypass in one pass over ds (fno_pointwise_bwd)
            ga_lin, gwl, gbl = lib.pointwise_bwd(ds, a, wl, need_bias=ctx.has_bias)
        elif need_wl or (need_bl and ctx.has_bias):
            gwl, gbl = lib.pointwise_wgrad(ds, a, wl.shape, need_bias=ctx.has_bias)
        gX, gws = lib.mix_bwd(plan, X, gY, weights, need_gx=need_ga, need_gw=need_gw)
        ga = None
        if need_ga:
            ga = ga_lin if ga_lin is not None else lib.pointwise_fwd(ds, wl, None, transpose=True)
            lib.inv_transform(plan, gX, addend=ga, out=ga, cmode=0, scale=1.0)
        if gws is None:
            gws = [None] * len(weights)
        return (ga, gwl if need_wl else None, gbl if (need_bl and ctx.has_bias) else None, None, *gws)


def fourier_layer(a, wl, bl, apply_gelu: bool, weights: Sequence[torch.Tensor]) -> torch.Tensor:
    return FourierLayerFn.apply(a, wl, bl, apply_gelu, *weights)


class LiftFn(torch.autograd.Function):
    """h = pad(permute(fc0(cat(normalise(x), grid))))  -- fno/fno.py:140-159, :343-360.

    One kernel writes the trunk layout directly.  Backward is the fc0 weight/bias gradient and, when x or grid
    requires grad, their gradient from one more kernel (fno_lift_dgrad).  Only the statistics are constants: the
    reference computes them under no_grad, while the normalisation, the grid concat and fc0 are differentiated, so a
    prediction fed back as the next input (rollout training) or a loss taken w.r.t. the input field gets its full
    gradient."""

    @staticmethod
    def forward(ctx, x, grid, stats, W0, b0, geo):
        x, grid = x.contiguous(), grid.contiguous()
        W0, b0 = W0.contiguous(), b0.contiguous()
        h = lib.lift_fwd(geo, x, grid, stats, W0, b0)
        ctx.geo = geo
        ctx.w_shape = W0.shape
        ctx.in_shapes = (x.shape, grid.shape)
        need_data = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        ctx.save_for_backward(x, grid, stats, W0 if need_data else None)
        return h

    @staticmethod
    def backward(ctx, dh):
        x, grid, stats, W0 = ctx.saved_tensors
        dh = dh.contiguous()
        gW0, gb0 = lib.lift_bwd(ctx.geo, x, grid, stats, dh, ctx.w_shape)
        dx = dgrid = None
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
            dx, dgrid = lib.lift_dgrad(ctx.geo, dh, W0, stats, *ctx.in_shapes, need_dx=ctx.needs_input_grad[0],
                                       need_dgrid=ctx.needs_input_grad[1])
        return dx, dgrid, None, gW0, gb0, None


class HeadFn(torch.autograd.Function):
    """out = fc2(gelu(fc1(unpad(h)))) * std + mean  -- fno/fno.py:180-187, :381-389.

    Saves only h: the 128-wide hidden layer is recomputed in backward."""

    @staticmethod
    def forward(ctx, h, W1, b1, W2, b2, stats, geo):
        h = h.contiguous()
        W1, b1, W2, b2 = W1.contiguous(), b1.contiguous(), W2.contiguous(), b2.contiguous()
        out = lib.head_fwd(geo, h, W1, b1, W2, b2, stats)
        ctx.geo = geo
        ctx.save_for_backward(h, W1, b1, W2, stats)
        return out

    @staticmethod
    def backward(ctx, dout):
        h, W1, b1, W2, stats = ctx.saved_tensors
        dh, gW1, gb1, gW2, gb2 = lib.head_bwd(ctx.geo, h, dout.contiguous(), W1, b1, W2, stats)
        return dh, gW1, gb1, gW2, gb2, None, None


class TwoHeadFn(torch.autograd.Function):
    """The two-head joint model's heads on one trunk activation h [Na + Nb, C, ...] (fno_aux.py:187, 216): samples
    [0, Na) through fc1 -> fc2_primary, samples [Na, Na + Nb) through fc1 -> fc2_auxiliary.

    The sample ranges of h are contiguous views, so the head kernels read them in place.  Backward writes both heads'
    dh into one trunk-sized tensor (each head kernel writes its range whole, zero padding included), so no zero-filled
    full-size gradient per head and no add of the two exist; the shared fc1 gradient is the sum of the two heads'
    [128, C] contributions."""

    @staticmethod
    def forward(ctx, h, W1, b1, W2a, b2a, W2b, b2b, stats, geo, na):
        h = h.contiguous()
        W1, b1 = W1.contiguous(), b1.contiguous()
        W2a, b2a, W2b, b2b = W2a.contiguous(), b2a.contiguous(), W2b.contiguous(), b2b.contiguous()
        out_a = lib.head_fwd(geo, h[:na], W1, b1, W2a, b2a, stats[:na])
        out_b = lib.head_fwd(geo, h[na:], W1, b1, W2b, b2b, stats[na:])
        ctx.geo, ctx.na = geo, na
        ctx.save_for_backward(h, W1, b1, W2a, W2b, stats)
        return out_a, out_b

    @staticmethod
    def backward(ctx, dout_a, dout_b):
        h, W1, b1, W2a, W2b, stats = ctx.saved_tensors
        geo, na = ctx.geo, ctx.na
        dh = torch.empty_like(h)
        _, gW1a, gb1a, gW2a, gb2a = lib.head_bwd(geo, h[:na], dout_a.contiguous(), W1, b1, W2a, stats[:na],
                                                  dh_out=dh[:na])
        _, gW1b, gb1b, gW2b, gb2b = lib.head_bwd(geo, h[na:], dout_b.contiguous(), W1, b1, W2b, stats[na:],
                                                  dh_out=dh[na:])
        return dh, gW1a + gW1b, gb1a + gb1b, gW2a, gb2a, gW2b, gb2b, None, None, None


def lift(x, grid, W0, b0, padding: int):
    """Returns (h in trunk layout, stats [B, 2, V], geometry)."""
    geo = lib.TrunkGeo(x.shape[1:-2], padding)
    with torch.no_grad():
        stats = lib.lift_stats(x.contiguous())
    return LiftFn.apply(x, grid, stats, W0, b0, geo), stats, geo


def head(h, W1, b1, W2, b2, stats, geo):
    return HeadFn.apply(h, W1, b1, W2, b2, stats, geo)


class WindowShiftFn(torch.autograd.Function):
    """xx' = cat(xx[..., 1:, :], pred) along the time axis (metrics.py:344) with its adjoint, so that a rollout can be
    trained through: forward fno_window_shift, backward fno_window_shift_bwd (one launch each)."""

    @staticmethod
    def forward(ctx, xx, pred):
        return lib.window_shift(xx.contiguous(), pred.contiguous())

    @staticmethod
    def backward(ctx, g):
        return lib.window_shift_bwd(g.contiguous(), need_xx=ctx.needs_input_grad[0], need_pred=ctx.needs_input_grad[1])


class JointWindowShiftFn(torch.autograd.Function):
    """The rollout shift of the two-head model's joined window xj = cat(xx, xx_aux):
    cat(xj[..., 1:, :], cat(pred, pred_aux)) with its adjoint, one launch each (fno_window_shift_split(_bwd)).  Both
    streams are fed back without splitting the window or joining the predictions."""

    @staticmethod
    def forward(ctx, xj, pred_a, pred_b):
        ctx.na = pred_a.shape[0]
        return lib.window_shift_split(xj.contiguous(), pred_a.contiguous(), pred_b.contiguous())

    @staticmethod
    def backward(ctx, g):
        need = ctx.needs_input_grad
        return lib.window_shift_split_bwd(g.contiguous(), ctx.na, need_xx=need[0], need_a=need[1], need_b=need[2])


class SpectralConv1dFn(torch.autograd.Function):
    """y = irfft(pad(einsum(rfft(x)[..., :m], W)), n = N) for x [B, Ci, N], W [Ci, Co, m] complex64 (the 2-D layer's
    convention, fno/fno.py:70-92, one dimension down).  Backward mirrors each kernel: K1' = c_k / N * pruned rfft of g,
    K2' = the two mixing gradients, K3' = unweighted inverse of gX."""

    @staticmethod
    def forward(ctx, x, w):
        x, w = x.contiguous(), w.contiguous()
        m = w.shape[2]
        X = lib.fwd_transform1d(x, m)
        Y = lib.mix1d_fwd(X, w)
        ctx.save_for_backward(X, w)
        ctx.n = x.shape[-1]
        return lib.inv_transform1d(Y, x.shape[-1])

    @staticmethod
    def backward(ctx, g):
        X, w = ctx.saved_tensors
        n = ctx.n
        gY = lib.fwd_transform1d(g.contiguous(), w.shape[2], cmode=1, scale=1.0 / n)
        gX, gW = lib.mix1d_bwd(X, gY, w, need_gx=ctx.needs_input_grad[0], need_gw=ctx.needs_input_grad[1])
        gx = lib.inv_transform1d(gX, n, cmode=0, scale=1.0) if gX is not None else None
        return gx, gW


def spectral_conv1d(x: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    if x.dim() != 3 or w.dim() != 3 or x.shape[1] != w.shape[0]:
        raise lib.FnoError(f"spectral_conv1d: expected x [B, Ci, N] and W [Ci, Co, m], got {tuple(x.shape)}, {tuple(w.shape)}")
    if w.shape[2] > x.shape[-1] // 2 + 1:
        raise lib.FnoError(f"spectral_conv1d: modes1 = {w.shape[2]} exceeds N/2 + 1 = {x.shape[-1] // 2 + 1}")
    return SpectralConv1dFn.apply(x, w)
