"""The reference's training step (fno/train.py:264-278, fno_aux/fno_train_aux.py:308-329) without
host synchronisation, plus its data-parallel form.

    im = model(xx, grid); loss = nrmse(im, yy).mean()
    zero_grad; backward; total_norm; clip = max(5, 0.1 * total_norm); clip_grad_norm_; Adam; sched

The reference evaluates ``max(5, 0.1 * total_norm)`` in Python (a device->host sync per step);
here it is a device-side clamp, numerically identical.  Under data parallelism the gradient
all-reduce (fno_b200.dp) completes before the norm is taken, so every rank clips and steps
identically.
"""
from __future__ import annotations

from typing import Optional

import torch

from .dp import BucketedGradAllReduce


def nrmse(output: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """fno/train.py:34-40: per-sample MSE over dims 1..3, normalised by the target's mean square."""
    dims = tuple(range(output.ndim))[1:4]
    num = (output - target).pow(2).mean(dims, keepdim=True)
    den = 1e-7 + target.pow(2).mean(dims, keepdim=True)
    return num / den


def global_grad_norm(params) -> torch.Tensor:
    norms = [torch.linalg.vector_norm(torch.view_as_real(p.grad) if p.grad.is_complex() else p.grad)
             for p in params if p.grad is not None]
    return torch.linalg.vector_norm(torch.stack(norms))


def rollout_loss(model, xx: torch.Tensor, yy: torch.Tensor, grid: torch.Tensor, steps: int):
    """Multi-step ("pushforward" / unrolled autoregressive) loss, upstream PDEBench's ``training_type="autoregressive"``:
    for k < steps, ``pred_k = model(xx_k, grid)``, ``loss_k = nrmse(pred_k, yy[..., k:k+1, :]).mean()`` and
    ``xx_{k+1} = cat(xx_k[..., 1:, :], pred_k)``, no shift after the last step.  The gradient flows through every fed-back
    prediction (fno_lift_dgrad, fno_window_shift_bwd).  Returns ``(mean_k loss_k, stacked per-step losses [steps])``.

    The mean, not upstream's sum, so that ``steps=1`` is exactly the single-step loss and the adaptive clip
    ``max(5, 0.1 * total_norm)`` keeps its scale as ``steps`` grows.

    Torch arithmetic in the step: the mean of the ``steps`` losses and, in the backward, the adds with which autograd sums
    two gradients into every fed-back prediction (``steps - 1``) and every intermediate window (``steps - 2``).  A
    target frame ``yy[..., k:k+1, :]`` that is not contiguous is copied before the fused loss reads it."""
    from . import lib, ops
    from .steptail import nrmse_loss

    if steps < 1:
        raise lib.FnoError(f"rollout_loss: steps must be >= 1, got {steps}")
    if yy.shape[-2] < steps:
        raise lib.FnoError(f"rollout_loss: yy has {yy.shape[-2]} target frames, {steps} rollout steps need {steps}")
    losses = []
    for k in range(steps):
        pred = model(xx, grid)
        losses.append(nrmse_loss(pred, yy[..., k:k + 1, :]))
        if k + 1 < steps:
            xx = ops.WindowShiftFn.apply(xx, pred)
    per_step = torch.stack(losses)
    return per_step.mean(), per_step


def joint_rollout_loss(model, xx: torch.Tensor, yy: torch.Tensor, grid: torch.Tensor, xx_aux: torch.Tensor,
                       yy_aux: torch.Tensor, grid_aux: torch.Tensor, steps: int, auxiliary_weight: float):
    """``rollout_loss`` for the two-head joint model (fno_b200.fno_aux), the auxiliary tensors flattened to
    ``[B * num_aux, ...]`` as the joint loop has them (fno_train_aux.py:251-256).  For k < steps:
    ``(p_k, a_k) = model(xx_k, grid, xx_aux_k, grid_aux)``, ``lp_k = nrmse(p_k, yy[..., k:k+1, :]).mean()``,
    ``la_k = nrmse(a_k, yy_aux[..., k:k+1, :]).mean()``, and both streams are fed back,
    ``xx_{k+1} = cat(xx_k[..., 1:, :], p_k)``, ``xx_aux_{k+1} = cat(xx_aux_k[..., 1:, :], a_k)``, no shift after the last
    step.  Returns ``(mean_k (lp_k + auxiliary_weight * la_k), per-step losses [steps, 2] with rows (lp_k, la_k))``;
    ``steps=1`` is the single-step joint loss ``lp + w * la``.

    The streams are joined once at entry (a view, no copy, when they are adjacent in memory: ``fno_aux.joined``).  After that one shift of the joined window feeds both predictions back
    (ops.JointWindowShiftFn: one launch forward, one backward), so no step joins or splits the window again."""
    from . import fno_aux, lib, ops
    from .fno import _check_cuda
    from .steptail import nrmse_loss

    if steps < 1:
        raise lib.FnoError(f"joint_rollout_loss: steps must be >= 1, got {steps}")
    for t, n in ((yy, "yy"), (yy_aux, "yy_aux")):
        if t.shape[-2] < steps:
            raise lib.FnoError(f"joint_rollout_loss: {n} has {t.shape[-2]} target frames, {steps} rollout steps need "
                               f"{steps}")
    _check_cuda(model, xx)
    nb = xx.shape[0]
    xj, gridj = fno_aux.joined(xx, xx_aux), fno_aux.joined(grid, grid_aux)
    lps, las = [], []
    for k in range(steps):
        p, a = fno_aux._joint_forward(model, xj, gridj, nb)
        lps.append(nrmse_loss(p, yy[..., k:k + 1, :]))
        las.append(nrmse_loss(a, yy_aux[..., k:k + 1, :]))
        if k + 1 < steps:
            xj = ops.JointWindowShiftFn.apply(xj, p, a)
    per_step = torch.stack((torch.stack(lps), torch.stack(las)), dim=1)
    return (per_step[:, 0] + auxiliary_weight * per_step[:, 1]).mean(), per_step


class TrainStep:
    """One optimisation step of FNO2d/FNO3d (``aux=False``) or the two-head joint model."""

    def __init__(self, model, optimizer, scheduler=None, dp: Optional[BucketedGradAllReduce] = None,
                 auxiliary_weight: float = 0.0):
        self.model = model
        self.optimizer = optimizer
        self.scheduler = scheduler
        self.dp = dp
        self.auxiliary_weight = auxiliary_weight
        self.params = [p for p in model.parameters()]

    def _backward_and_update(self, loss):
        if self.dp is not None:
            self.dp.zero_grad()
        else:
            self.optimizer.zero_grad()
        loss.backward()
        if self.dp is not None:
            self.dp.finish()
        total_norm = global_grad_norm(self.params)
        clip_value = torch.clamp(0.1 * total_norm, min=5.0)
        torch.nn.utils.clip_grad_norm_(self.params, clip_value)
        self.optimizer.step()
        if self.scheduler is not None:
            self.scheduler.step()
        return total_norm

    def __call__(self, xx, yy, grid, weight: Optional[float] = None):
        """``weight``: data parallelism with unequal local batches (fno_b200.data.epoch_plan): the local mean loss is
        scaled by local_b * world / global_b so that the AVERAGED gradient is the global-batch-mean gradient."""
        loss = nrmse(self.model(xx, grid), yy).mean()
        self._backward_and_update(loss if weight is None else loss * weight)
        return loss.detach()

    def joint(self, xx, yy, grid, xx_aux, yy_aux, grid_aux):
        """fno_train_aux.py:308-329: loss = primary + auxiliary_weight * auxiliary."""
        out_p, out_a = self.model(xx, grid, xx_aux, grid_aux)
        lp = nrmse(out_p, yy).mean()
        la = nrmse(out_a, yy_aux).mean()
        loss = lp + self.auxiliary_weight * la
        self._backward_and_update(loss)
        return lp.detach(), la.detach()


class FusedTrainStep:
    """The same step with the device-side tail (fno_b200.steptail): fused nRMSE loss, and norm +
    clip + Adam + cosine LR in three launches with no host round trip.

        step = FusedTrainStep(model, lr=1e-3, weight_decay=1e-4, t_max=T, dp=None, graph=True)
        loss = step(xx, yy, grid)            # 0-dim device tensor; never synchronises

    ``graph=True`` captures forward + loss + backward + update in ONE CUDA graph after two eager
    warm-up steps (the first discovers which parameters receive gradients); inputs are copied
    into static buffers, so a replay is a single launch -- at the reference's own batch sizes
    (2-16) the eager step is bound by ~150 kernel launches, not by the GPU.  With
    ``alias_inputs=True`` the graph reads the caller's tensors in place instead (no 200 MB device copy
    per step at batch 128): one graph is captured per distinct set of input addresses (up to
    ``max_graphs``; a double-buffered input pipeline needs two), the caller keeps those tensors alive
    and refills them between steps; other inputs fall back to the copying graph.  Under data
    parallelism (``dp``) the optimizer reads the reduced bucket views in place (``own_grads=False``); with
    ``graph=True`` the step is two graph replays around the bucket all-reduces (issued in ``dp.finish()`` on the same
    stream); without it they are issued from autograd hooks and overlap the rest of the backward pass.

    ``rollout_steps=K > 1`` trains on the K-step rollout loss (``rollout_loss``): ``yy`` carries at least K target frames
    and the step returns the K per-step losses.  With ``auxiliary_weight`` (the two-head joint model) it is
    ``joint_rollout_loss``: ``yy`` and ``yy_aux`` carry at least K frames and the step returns ``[K, 2]``, rows (primary,
    auxiliary).  Eager, graph and ``alias_inputs`` steps work as for K = 1."""

    def __init__(self, model, lr: float = 1e-3, weight_decay: float = 1e-4, t_max: float = 0.0, betas=(0.9, 0.999),
                 eps: float = 1e-8, dp: Optional[BucketedGradAllReduce] = None, graph: bool = False,
                 auxiliary_weight: Optional[float] = None, alias_inputs: bool = False, max_graphs: int = 2,
                 param_groups=None, rollout_steps: int = 1):
        from . import lib
        from .steptail import FusedClipAdam

        if rollout_steps < 1:
            raise lib.FnoError(f"FusedTrainStep: rollout_steps must be >= 1, got {rollout_steps}")
        if rollout_steps > 1 and auxiliary_weight is not None and not hasattr(model, "fc2_auxiliary"):
            raise lib.FnoError("FusedTrainStep: a rollout with auxiliary_weight needs the two-head joint model "
                               "(fno_b200.fno_aux)")
        self.rollout_steps = rollout_steps
        self.model = model
        self.dp = dp
        self.aux_w = auxiliary_weight
        # param_groups: torch.optim-style group dicts, e.g. the joint loop's three groups (fno_train_aux.py:175-179)
        self.opt = FusedClipAdam(param_groups if param_groups is not None else model.parameters(), lr=lr, betas=betas,
                                 eps=eps, weight_decay=weight_decay, t_max=t_max, own_grads=dp is None)
        # data parallelism + graph: two graphs around the (eager, inline) bucket all-reduces -- see _capture
        self.use_graph = graph
        if graph and dp is not None:
            dp.set_inline(True)
        self._calls = 0
        self._graph = None
        self._static_in = None
        self._static_out = None
        self.alias_inputs = alias_inputs
        self.max_graphs = max_graphs
        self._aliased = {}                      # input addresses -> (graph, inputs kept alive, static output)

    def _fwd_bwd(self, *batch, weight=None):
        from .steptail import nrmse_loss

        if self.rollout_steps > 1 and self.aux_w is not None:
            loss, ret = joint_rollout_loss(self.model, *batch, self.rollout_steps, self.aux_w)
        elif self.rollout_steps > 1:
            xx, yy, grid = batch
            loss, ret = rollout_loss(self.model, xx, yy, grid, self.rollout_steps)
        elif self.aux_w is None:
            xx, yy, grid = batch
            loss = nrmse_loss(self.model(xx, grid), yy)
            ret = loss
        else:
            xx, yy, grid, xx_aux, yy_aux, grid_aux = batch
            out_p, out_a = self.model(xx, grid, xx_aux, grid_aux)
            lp, la = nrmse_loss(out_p, yy), nrmse_loss(out_a, yy_aux)
            loss = lp + self.aux_w * la
            ret = torch.stack((lp.detach(), la.detach()))
        if self.dp is not None:
            self.dp.zero_grad()
        else:
            self.opt.zero_grad()
        (loss if weight is None else loss * weight).backward()
        return ret.detach()

    def _eager(self, *batch, weight=None):
        ret = self._fwd_bwd(*batch, weight=weight)
        if self.dp is not None:
            self.dp.finish()
        self.opt.step()
        return ret

    def _capture(self, batch):
        """Returns (replay, static output).  Single GPU: forward + loss + backward + update in ONE graph.  Data parallel:
        TWO graphs around the gradient exchange -- forward + loss + backward, then (eagerly, on the same stream) one NCCL
        all-reduce per bucket, then the optimizer graph.  (Capturing the collectives themselves was tried on 2 B200s in
        rounds 1 and 2 and hung during capture; with 2 graph launches + 5 NCCL calls the step no longer pays for ~150
        kernel launches.)"""
        if self.dp is None:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                out = self._eager(*batch)
            return g.replay, out
        g1, g2 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(g1):
            out = self._fwd_bwd(*batch)
        with torch.cuda.graph(g2, pool=g1.pool()):
            self.opt.step()

        def replay():
            g1.replay()
            self.dp.finish()
            g2.replay()
        return replay, out

    def _static_inputs(self, batch):
        """The copying graph's input buffers.  Joint-model inputs that arrive joined (``xx_aux`` continuing ``xx``, or
        ``grid_aux`` continuing ``grid``, as ``data.DeviceJointWindows`` yields them) get one joined buffer per pair, so
        the captured forward reads the joined window in place instead of concatenating it in the graph."""
        from .fno_aux import is_joined

        static = [torch.empty_like(t) for t in batch]
        if self.aux_w is not None and len(batch) == 6:
            for i, j in ((0, 3), (2, 5)):
                if is_joined(batch[i], batch[j]):
                    whole = torch.empty((batch[i].shape[0] + batch[j].shape[0],) + tuple(batch[i].shape[1:]),
                                        dtype=batch[i].dtype, device=batch[i].device)
                    static[i], static[j] = whole[:batch[i].shape[0]], whole[batch[i].shape[0]:]
        return tuple(static)

    def __call__(self, *batch, weight=None):
        """``weight`` (data parallelism, eager only): see TrainStep.__call__."""
        if self.rollout_steps > 1:
            targets = ((1, "yy"), (4, "yy_aux")) if self.aux_w is not None else ((1, "yy"),)
            for i, n in targets:
                if batch[i].shape[-2] < self.rollout_steps:
                    from . import lib
                    raise lib.FnoError(f"FusedTrainStep: {n} has {batch[i].shape[-2]} target frames, rollout_steps="
                                       f"{self.rollout_steps} needs {self.rollout_steps}")
        if not self.use_graph:
            return self._eager(*batch, weight=weight)
        if weight is not None:
            raise ValueError("FusedTrainStep: a loss weight needs the eager step (graph=False)")
        if self._graph is None:
            if self._calls < 2:                       # eager warm-up: plans, attributes, gradient discovery
                self._calls += 1
                return self._eager(*batch)
            # third call: this batch's step runs eagerly on a side stream (the stream-capture warm-up
            # PyTorch asks for), then the same sequence is captured -- capture records, it does not
            # execute -- and every later call is a graph replay
            self._static_in = self._static_inputs(batch)
            for dst, src in zip(self._static_in, batch):
                dst.copy_(src)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                ret = self._eager(*self._static_in)
            torch.cuda.current_stream().wait_stream(side)
            self._graph, self._static_out = self._capture(self._static_in)
            return ret
        elif self.alias_inputs and all(t.is_contiguous() for t in batch):
            key = tuple((t.data_ptr(), tuple(t.shape)) for t in batch)
            hit = self._aliased.get(key)
            if hit is None and len(self._aliased) < self.max_graphs:
                # same parameters, optimizer state and step counter; only the input addresses differ.  Capture
                # records, it does not execute: the replay below runs this batch's step.
                replay, out = self._capture(batch)
                hit = self._aliased[key] = (replay, batch, out)
            if hit is not None:
                hit[0]()
                return hit[2]
            for dst, src in zip(self._static_in, batch):
                dst.copy_(src, non_blocking=True)
        else:
            for dst, src in zip(self._static_in, batch):
                dst.copy_(src, non_blocking=True)
        self._graph()
        return self._static_out
