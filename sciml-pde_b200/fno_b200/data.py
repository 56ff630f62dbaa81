"""Synthetic PDEBench-shaped fields for benchmarks and loop-level parity (SURVEY.md 8d).

The reference loaders (fno/utils_2d_rd_baseline.py:59-102 and friends) read HDF5 trajectories
``[t, x, y, v]`` and emit sliding windows ``xx [X, Y, initial_step, v]``, ``yy [X, Y, 1, v]`` plus a
cell-centre ``grid [X, Y, 2]``.  No datasets (and no h5py) exist here, so trajectories are
generated: a band-limited Gaussian random field per channel, evolved by exact spectral
diffusion u_hat(t) = u_hat(0) exp(-D |k|^2 t) -- the reference's own ``sim_type="diff"`` physics
(data_gen/src/sim_diff_react.py:165-167).  Generation is host-side utility code, not part of the
measured path.
"""
from __future__ import annotations

import math

import torch
import torch.utils.data


def cell_centre_grid(n: int, lo: float = -1.0, hi: float = 1.0, nd: int = 2) -> torch.Tensor:
    """meshgrid(ij) of cell centres, as the loaders build it -> [n, ..., n, nd]."""
    dx = (hi - lo) / n
    lin = torch.linspace(lo + dx / 2, hi - dx / 2, n)
    return torch.stack(torch.meshgrid(*([lin] * nd), indexing="ij"), dim=-1)


def diffusion_trajectories(n_traj: int, n: int, steps: int, channels: int, seed: int, nd: int = 2,
                           kmax: int = 16, t_end: float = 5.0, diffusivity=(1e-3, 1e-1)) -> torch.Tensor:
    """[n_traj, steps, n, (n,) n, channels] float32 trajectories with O(1) values."""
    g = torch.Generator().manual_seed(seed)
    k1 = torch.fft.fftfreq(n, d=1.0 / n)
    ks = torch.meshgrid(*([k1] * nd), indexing="ij")
    k2 = sum(k * k for k in ks)
    band = (k2 <= kmax * kmax).float() / (1.0 + k2)
    t = torch.linspace(0.0, t_end, steps)
    out = []
    for c in range(channels):
        d = diffusivity[c % len(diffusivity)]
        noise = torch.randn((n_traj,) + (n,) * nd, generator=g)
        u0 = torch.fft.fftn(noise, dim=tuple(range(1, nd + 1))) * band
        decay = torch.exp(-d * (2 * math.pi / 2.0) ** 2 * k2[None, None] * t.view(1, -1, *([1] * nd)))
        u = torch.fft.ifftn(u0[:, None] * decay, dim=tuple(range(2, nd + 2))).real
        u = u / u[:, :1].std(dim=tuple(range(2, nd + 2)), keepdim=True).clamp_min(1e-6)
        out.append(u)
    return torch.stack(out, dim=-1).float()


def windows(traj: torch.Tensor, initial_step: int, rollout: int = 1):
    """All sliding windows of a trajectory batch -> (xx [N, *sp, initial_step, v], yy [N, *sp, rollout, v])."""
    nt = traj.shape[1]
    nd = traj.dim() - 3
    xs, ys = [], []
    for s in range(nt - initial_step - rollout + 1):
        xs.append(traj[:, s:s + initial_step])
        ys.append(traj[:, s + initial_step:s + initial_step + rollout])
    xx = torch.stack(xs, dim=1).flatten(0, 1)
    yy = torch.stack(ys, dim=1).flatten(0, 1)
    perm = (0,) + tuple(range(2, 2 + nd)) + (1, 2 + nd)
    return xx.permute(*perm).contiguous(), yy.permute(*perm).contiguous()


def synthetic_batch(batch: int, n: int = 128, initial_step: int = 10, channels: int = 2, seed: int = 0, nd: int = 2):
    """One batch in the loaders' layout: (xx, yy, grid)."""
    traj = diffusion_trajectories(batch, n, initial_step + 1, channels, seed, nd=nd)
    xx, yy = windows(traj, initial_step)
    grid = cell_centre_grid(n, nd=nd).unsqueeze(0).expand(batch, *([-1] * (nd + 1))).contiguous()
    return xx, yy, grid


class SyntheticWindows(torch.utils.data.Dataset):
    """Map-style dataset with the sample layout of the reference loaders (fno/utils_2d_rd_baseline.py:
    59-102): item i -> (xx [X, Y, initial_step, v], yy [X, Y, rollout, v], grid [X, Y, 2]), sliding
    windows over synthetic diffusion trajectories.  Deterministic in (seed, sizes); used by the
    loop-level parity fixtures (oracle/make_golden_loop.py, tests/test_loop_parity*.py)."""

    def __init__(self, n_traj: int, n: int, windows: int, initial_step: int = 10, channels: int = 2, seed: int = 0,
                 rollout: int = 1):
        steps = initial_step + rollout + windows - 1
        traj = diffusion_trajectories(n_traj, n, steps, channels, seed)
        self.xx, self.yy = windows_of(traj, initial_step, rollout)
        self.grid = cell_centre_grid(n)

    def __len__(self):
        return self.xx.shape[0]

    def __getitem__(self, i):
        return self.xx[i], self.yy[i], self.grid


def windows_of(traj, initial_step, rollout=1):
    return windows(traj, initial_step, rollout)


# ---------------------------------------------------------------------------------------------------
# Device-resident windowed dataset (SURVEY 8f row f4)
# ---------------------------------------------------------------------------------------------------
def epoch_indices(n_items: int, batch: int, shuffle: bool, seed: int, epoch: int = 0, rank: int = 0, world: int = 1):
    """Host-side index plan of one epoch: the global order (a seeded ``torch.randperm`` when shuffling, as a
    ``DataLoader(shuffle=True)`` with a seeded generator draws it), cut into global batches of ``batch`` items
    with the last one ragged (``drop_last=False``, fno/train.py:95-97); under data parallelism rank r takes the
    rank-strided slice of every global batch (SURVEY 8e), so the union over ranks is the single-GPU batch.
    Returns a list of 1-D int64 tensors (this rank's items per step; possibly empty for a ragged tail)."""
    if n_items <= 0 or batch <= 0 or world <= 0 or not 0 <= rank < world:
        raise ValueError("epoch_indices: bad arguments")
    if shuffle:
        g = torch.Generator().manual_seed(seed + epoch)
        order = torch.randperm(n_items, generator=g)
    else:
        order = torch.arange(n_items)
    return [order[s:s + batch][rank::world].contiguous() for s in range(0, n_items, batch)]


def epoch_plan(n_items: int, batch: int, shuffle: bool, seed: int, epoch: int = 0, rank: int = 0, world: int = 1):
    """``epoch_indices`` made safe for data parallelism: EVERY rank gets a non-empty batch for EVERY step (so the
    gradient all-reduces pair up), together with the weight its mean loss must be multiplied by so that the averaged
    gradient is the gradient of the GLOBAL batch mean (the reference's DataLoader has ``drop_last=False``,
    fno/train.py:95-97, so the last global batch is ragged: ranks hold unequal, possibly empty, slices).

    Returns [(items, weight)]: weight = local_b * world / global_b; a rank whose slice of a ragged tail is empty gets the
    first item of that global batch with weight 0 (its gradient contributes nothing, every hook still fires)."""
    out = []
    plans = [epoch_indices(n_items, batch, shuffle, seed, epoch, r, world) for r in range(world)] if world > 1 else None
    mine = epoch_indices(n_items, batch, shuffle, seed, epoch, rank, world)
    for step, items in enumerate(mine):
        if world == 1:
            out.append((items, 1.0))
            continue
        global_b = sum(int(pl[step].numel()) for pl in plans)
        if items.numel() == 0:
            out.append((plans[0][step][:1].clone(), 0.0))
        else:
            out.append((items, items.numel() * world / global_b))
    return out


class DeviceWindows:
    """Trajectories cached on the GPU, sliding windows gathered on the device (one copy kernel per batch).

    Replaces ``FNODatasetMult`` + ``DataLoader`` of the reference (fno/utils_2d_rd_baseline.py:59-102,
    fno/train.py:95-97): item ``i`` is window ``i % n_windows`` of trajectory ``i // n_windows`` -- the order
    ``SyntheticWindows`` / the reference loaders use -- and yields ``xx [*sp, initial_step, V]``,
    ``yy [*sp, rollout, V]``, ``grid [*sp, nd]``.  ``traj`` is ``[n_traj, T, *spatial, V]`` (PDEBench layout);
    it is stored once, time-inner, in device memory (180 GB of HBM3e holds ~270 full cfg-1 trajectories
    per GPU; shard trajectories across ranks beyond that)."""

    def __init__(self, traj: torch.Tensor, initial_step: int = 10, rollout: int = 1, device=None,
                 grid_lo: float = -1.0, grid_hi: float = 1.0):
        name = type(self).__name__
        if traj.dim() < 4:
            raise ValueError(f"{name}: traj must be [n_traj, T, *spatial, V]")
        device = torch.device(device if device is not None else "cuda")
        self.spatial = tuple(traj.shape[2:-1])
        self.nd = len(self.spatial)
        self.T, self.V = traj.shape[1], traj.shape[-1]
        self.initial_step, self.rollout = initial_step, rollout
        self.n_windows = self.T - initial_step - rollout + 1
        if self.n_windows <= 0:
            raise ValueError(f"{name}: trajectories shorter than initial_step + rollout")
        self.traj = self._store(traj, device)
        lins = [torch.linspace(grid_lo + (grid_hi - grid_lo) / (2 * n), grid_hi - (grid_hi - grid_lo) / (2 * n), n)
                for n in self.spatial]                                           # cell centres per axis
        self.grid = torch.stack(torch.meshgrid(*lins, indexing="ij"), dim=-1).to(device)
        self.device = device

    def _store(self, traj: torch.Tensor, device) -> torch.Tensor:
        """[n, *lead, T, *spatial, V] -> the time-inner device store [n, *lead, pixels, T, V]."""
        lead = traj.dim() - self.nd - 2                                          # 1, or 2 with the auxiliary axis
        perm = tuple(range(lead)) + tuple(range(lead + 1, lead + 1 + self.nd)) + (lead, lead + 1 + self.nd)
        store = traj.to(device=device, dtype=torch.float32).permute(*perm).contiguous()
        return store.view(tuple(traj.shape[:lead]) + (-1, self.T, self.V))

    def __len__(self):
        return self.traj.shape[0] * self.n_windows

    def split_items(self, items: torch.Tensor):
        """Host-side index arithmetic of a batch: item -> (trajectory index int64, window start int32), pinned."""
        items = items.to(dtype=torch.int64, device="cpu")
        ti = torch.div(items, self.n_windows, rounding_mode="floor")
        ts = (items - ti * self.n_windows).to(torch.int32)
        return ti.contiguous().pin_memory(), ts.contiguous().pin_memory()

    def _device_items(self, items):
        """items (1-D int64, host or device) or the (ti, ts) pair of ``split_items`` -> (ti, ts, B) on the device."""
        if isinstance(items, tuple):
            ti, ts = (t.to(self.device, non_blocking=True) for t in items)
            return ti, ts, ti.numel()
        items = items.to(device=self.device, dtype=torch.int64)
        ti = torch.div(items, self.n_windows, rounding_mode="floor").contiguous()
        ts = (items - ti * self.n_windows).to(torch.int32).contiguous()
        return ti, ts, items.numel()

    def batch(self, items, out=None):
        """items: 1-D int64 (host or device), or the (ti, ts) pair of ``split_items`` -> (xx [B,*sp,T0,V], yy [B,*sp,R,V],
        grid [B,*sp,nd]) on the device.  ``out = (xx, yy)``: gather into caller-owned buffers (fixed addresses)."""
        from . import lib

        ti, ts, B = self._device_items(items)
        xx, yy = lib.window_gather(self.traj, ti, ts, self.initial_step, self.rollout, out=out)
        xx = xx.view((B,) + self.spatial + (self.initial_step, self.V))
        yy = yy.view((B,) + self.spatial + (self.rollout, self.V))
        if getattr(self, "_grid_b", None) is None or self._grid_b.shape[0] != B:
            self._grid_b = self.grid.unsqueeze(0).expand(B, *([-1] * (self.nd + 1))).contiguous()   # same tensor every step
        return xx, yy, self._grid_b

    def epoch(self, batch: int, shuffle: bool = True, seed: int = 16, epoch: int = 0, rank: int = 0, world: int = 1,
              with_weight: bool = False):
        """Iterates this rank's batches of one epoch (see ``epoch_plan``).  Under data parallelism every rank yields a
        batch for every step; ``with_weight=True`` appends the loss weight of ``epoch_plan`` (pass it to the train
        step: ``step(xx, yy, grid, weight=w)``) -- required whenever ``len(self) % (batch * world) != 0``."""
        for items, w in epoch_plan(len(self), batch, shuffle, seed, epoch, rank, world):
            if world > 1 and not with_weight and w != 1.0:
                raise ValueError(f"{type(self).__name__}.epoch: ragged global batch under data parallelism -- iterate with "
                                 "with_weight=True and pass the weight to the train step")
            yield (self.batch(items) + (w,)) if with_weight else self.batch(items)


class DeviceJointWindows(DeviceWindows):
    """``DeviceWindows`` for the two-head joint model (fno_b200.fno_aux): each item also carries the windows of its ``A``
    auxiliary trajectories, as ``fno_aux/utils_2d_rd.py`` yields them (``oracle/ref_datasets.AuxFNODatasetMult``).

    ``traj [n, T, *spatial, V]`` and ``traj_aux [n, A, T, *spatial, V]`` (PDEBench layout; ``traj_aux[i, k]`` is the k-th
    auxiliary trajectory of trajectory i) are stored once, time-inner, in device memory.  Item ``i`` is window
    ``i % n_windows`` of trajectory ``i // n_windows`` on every stream.  ``batch`` gathers the primary and auxiliary
    windows with ONE kernel (fno_window_gather_joint) into one joined buffer ``xj [B + B*A, *spatial, T0, V]``, so
    ``xx = xj[:B]`` and ``xx_aux = xj[B:]`` (flattened ``[B*A, ...]`` in the joint loop's order, fno_train_aux.py:251-256)
    reach the joint forward as adjacent views and it runs on ``xj`` without concatenating.  The trunk batch is
    ``B * (1 + A)``."""

    def __init__(self, traj: torch.Tensor, traj_aux: torch.Tensor, initial_step: int = 10, rollout: int = 1, device=None,
                 grid_lo: float = -1.0, grid_hi: float = 1.0):
        super().__init__(traj, initial_step, rollout, device, grid_lo, grid_hi)
        if traj_aux.dim() != traj.dim() + 1 or traj_aux.shape[1] < 1:
            raise ValueError(f"DeviceJointWindows: traj_aux must be [n_traj, A >= 1, T, *spatial, V], got "
                             f"{tuple(traj_aux.shape)}")
        for what, a, p in (("trajectory count n", traj_aux.shape[0], traj.shape[0]), ("frame count T", traj_aux.shape[2],
                           self.T), ("spatial shape", tuple(traj_aux.shape[3:-1]), self.spatial),
                           ("channel count V", traj_aux.shape[-1], self.V)):
            if a != p:
                raise ValueError(f"DeviceJointWindows: traj_aux {what} {a} does not match traj's {p}")
        self.A = traj_aux.shape[1]
        self.traj_aux = self._store(traj_aux, self.device)
        self._gridj = None

    def batch(self, items, out=None):
        """items: as ``DeviceWindows.batch`` -> (xx [B,*sp,T0,V], yy [B,*sp,R,V], grid [B,*sp,nd], xx_aux [B*A,*sp,T0,V],
        yy_aux [B*A,*sp,R,V], grid_aux [B*A,*sp,nd]) on the device; xx / xx_aux are views of one gathered buffer and
        grid / grid_aux views of one constant joined grid (built once per batch size).  ``out = (xj, yy, yy_aux)``: gather
        into caller-owned buffers (fixed addresses, for CUDA-graph steps that alias them)."""
        from . import lib

        ti, ts, B = self._device_items(items)
        xj, yy, yy_aux = lib.window_gather_joint(self.traj, self.traj_aux, ti, ts, self.initial_step, self.rollout,
                                                 out=out)
        rows = B * (1 + self.A)
        xj = xj.view((rows,) + self.spatial + (self.initial_step, self.V))
        yy = yy.view((B,) + self.spatial + (self.rollout, self.V))
        yy_aux = yy_aux.view((B * self.A,) + self.spatial + (self.rollout, self.V))
        if self._gridj is None or self._gridj.shape[0] != rows:
            self._gridj = self.grid.unsqueeze(0).expand(rows, *([-1] * (self.nd + 1))).contiguous()
        return xj[:B], yy, self._gridj[:B], xj[B:], yy_aux, self._gridj[B:]

    def joined_buffers(self, batch: int):
        """Freshly allocated ``out=`` buffers (xj, yy, yy_aux) for batches of ``batch`` items."""
        rows, sp = batch * (1 + self.A), self.spatial
        return (torch.empty((rows,) + sp + (self.initial_step, self.V), device=self.device),
                torch.empty((batch,) + sp + (self.rollout, self.V), device=self.device),
                torch.empty((batch * self.A,) + sp + (self.rollout, self.V), device=self.device))
