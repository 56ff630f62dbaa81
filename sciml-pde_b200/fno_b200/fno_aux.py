"""Drop-in two-head FNO2d / FNO3d of the multiphysics joint-training path (reference:
pdebench/models/fno_aux/fno_aux.py:70-222, :325-475).

Differences from fno_b200.fno: ``fc2`` is replaced by ``fc2_primary`` / ``fc2_auxiliary``,
``shared_layers`` aliases the trunk modules (adding the duplicate ``shared_layers.N.*``
state_dict keys the reference has), and ``forward(x, grid, x_aux, grid_aux)`` returns
``(out_primary, out_auxiliary)``.  The reference runs the shared trunk twice, once per stream;
no op in the trunk couples samples, so here both streams go through ONE batched pass over
``cat([x, x_aux])`` -- half the kernel launches, identical results per sample.  When ``x_aux`` continues ``x`` in
memory (``fno_b200.data.DeviceJointWindows`` gathers them so) that joined window is a view and nothing is copied.
"""
from __future__ import annotations

import torch
from torch import nn

from . import fno as _base
from . import ops


class FNO2d(_base.FNO2d):
    def __init__(self, num_channels, modes1=12, modes2=12, width=20, initial_step=10):
        super().__init__(num_channels, modes1, modes2, width, initial_step)
        self.shared_layers = nn.ModuleList([
            self.fc0, self.conv0, self.conv1, self.conv2, self.conv3,
            self.w0, self.w1, self.w2, self.w3, self.fc1,
        ])

    def _make_heads(self, num_channels):
        # same RNG position as the reference: right after fc1 (fno_aux.py:113-116)
        self.fc2_primary = nn.Linear(128, num_channels)
        self.fc2_auxiliary = nn.Linear(128, num_channels)

    def forward(self, x, grid, x_aux, grid_aux):
        return _two_head_forward(self, x, grid, x_aux, grid_aux)


class FNO3d(_base.FNO3d):
    def __init__(self, num_channels, modes1=8, modes2=8, modes3=8, width=20, initial_step=10):
        super().__init__(num_channels, modes1, modes2, modes3, width, initial_step)
        self.shared_layers = nn.ModuleList([
            self.fc0, self.conv0, self.conv1, self.conv2, self.conv3,
            self.w0, self.w1, self.w2, self.w3, self.fc1,
            self.bn0, self.bn1, self.bn2, self.bn3,
        ])

    def _make_heads(self, num_channels):
        self.fc2_primary = nn.Linear(128, num_channels)
        self.fc2_auxiliary = nn.Linear(128, num_channels)

    def forward(self, x, grid, x_aux, grid_aux):
        return _two_head_forward(self, x, grid, x_aux, grid_aux)


def is_joined(a: torch.Tensor, b: torch.Tensor) -> bool:
    """True when ``b`` continues ``a`` in the same storage (both contiguous, neither requiring grad), so that
    ``cat((a, b))`` is a view, e.g. ``xx`` / ``xx_aux`` from ``fno_b200.data.DeviceJointWindows``."""
    return (not a.requires_grad and not b.requires_grad and a.is_contiguous() and b.is_contiguous()
            and a.dtype == b.dtype and a.device == b.device and a.dim() == b.dim() and a.shape[1:] == b.shape[1:]
            and a.untyped_storage().data_ptr() == b.untyped_storage().data_ptr()
            and b.data_ptr() == a.data_ptr() + a.numel() * a.element_size())


def joined(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """``torch.cat((a, b), dim=0)``: the joined view when ``is_joined(a, b)``, no copy; a concatenation otherwise."""
    if not is_joined(a, b):
        return torch.cat((a, b), dim=0)
    shape = (a.shape[0] + b.shape[0],) + tuple(a.shape[1:])
    return a.as_strided(shape, torch.empty(shape, device="meta").stride(), a.storage_offset())


def _two_head_forward(model, x, grid, x_aux, grid_aux):
    _base._check_cuda(model, x)
    return _joint_forward(model, joined(x, x_aux), joined(grid, grid_aux), x.shape[0])


def _joint_forward(model, xj, gridj, nb):
    """The joint forward on an already joined window xj = cat(x, x_aux), gridj = cat(grid, grid_aux); rows [0, nb) are
    the primary stream.  A rollout joins once and feeds both predictions back into xj (ops.JointWindowShiftFn)."""
    h, stats, geo = _base._lift(model, xj, gridj)
    h = _base._trunk(model, h)
    out_p, out_a = ops.TwoHeadFn.apply(h, model.fc1.weight, model.fc1.bias, model.fc2_primary.weight,
                                       model.fc2_primary.bias, model.fc2_auxiliary.weight, model.fc2_auxiliary.bias,
                                       stats, geo, nb)
    return out_p.unsqueeze(-2), out_a.unsqueeze(-2)
