"""ctypes binding of libfno_sm100.so (include/fno_sm100.h) for torch CUDA tensors.

PyTorch is plumbing here: it owns device memory and streams.  Every function below passes raw
device pointers plus the caller's *current* CUDA stream to the C ABI; nothing is computed in
Python and there is no CPU / eager fallback -- a missing library or a non-CUDA tensor raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from pathlib import Path
from typing import Optional, Sequence

import torch

_LIB_PATH = Path(__file__).resolve().parent / "libfno_sm100.so"
_lib = None
_lib_lock = threading.Lock()

c_float_p = C.POINTER(C.c_float)


class FnoError(RuntimeError):
    pass


def lib_path() -> Path:
    return _LIB_PATH


def load():
    """Loads the shared library (once).  Raises FnoError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        if not _LIB_PATH.exists():
            raise FnoError(
                f"{_LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  There is no CPU fallback for the FNO spectral-convolution path."
            )
        lib = C.CDLL(str(_LIB_PATH))
        vp, i, l, f = C.c_void_p, C.c_int, C.c_long, C.c_float
        vpp = C.POINTER(C.c_void_p)
        sig = {
            "fno_version": (i, []),
            "fno_sm_arch": (i, []),
            "fno_last_error": (C.c_char_p, []),
            "fno_launch_count": (C.c_ulonglong, []),
            "fno_shutdown": (None, []),
            "fno_plan2d_create": (i, [i, i, i, i, i, vpp]),
            "fno_plan3d_create": (i, [i, i, i, i, i, i, i, vpp]),
            "fno_window_gather": (i, [vp, vp, vp, vp, vp, i, l, i, i, i, i, vp]),
            "fno_window_gather_joint": (i, [vp, vp, vp, vp, vp, vp, vp, i, i, l, i, i, i, i, vp]),
            "fno_sc1d_fwd_transform": (i, [vp, vp, l, i, i, i, f, vp]),
            "fno_sc1d_inv_transform": (i, [vp, vp, vp, l, i, i, i, f, vp]),
            "fno_mix1d_fwd": (i, [vp, vp, vp, i, i, i, i, vp]),
            "fno_mix1d_bwd": (i, [vp, vp, vp, vp, vp, i, i, i, i, vp]),
            "fno_metric_workspace_bytes": (C.c_size_t, [i, i, i, i, i, i]),
            "fno_metric_func": (i, [vp, vp, vp, vp, i, i, i, i, i, i, f, f, f, i, i, vp]),
            "fno_window_shift": (i, [vp, vp, vp, l, i, i, vp]),
            "fno_window_shift_bwd": (i, [vp, vp, vp, l, i, i, vp]),
            "fno_window_shift_split": (i, [vp, vp, vp, vp, l, l, i, i, vp]),
            "fno_window_shift_split_bwd": (i, [vp, vp, vp, vp, l, l, i, i, vp]),
            "fno_set_math_mode": (i, [i]),
            "fno_get_math_mode": (i, []),
            "fno_plan_destroy": (i, [vp]),
            "fno_plan_workspace_bytes": (C.c_size_t, [vp, l]),
            "fno_sc2d_fwd_transform": (i, [vp, vp, vp, vp, vp, l, i, f, vp]),
            "fno_sc2d_fwd_workspace_bytes": (C.c_size_t, [vp, l]),
            "fno_sc2d_fwd_transform_ws": (i, [vp, vp, vp, vp, vp, vp, l, i, f, vp]),
            "fno_sc3d_fwd_transform": (i, [vp, vp, vp, vp, vp, vp, l, i, f, vp]),
            "fno_mix_fwd": (i, [vp, vp, vpp, vp, i, i, i, vp]),
            "fno_mix_bwd": (i, [vp, vp, vp, vpp, vp, vpp, i, i, i, vp]),
            "fno_mix_tc_supported": (i, [vp, i, i]),
            "fno_sc2d_inv_transform": (i, [vp, vp, vp, vp, vp, l, i, f, i, vp]),
            "fno_sc3d_inv_transform": (i, [vp, vp, vp, vp, vp, vp, l, i, f, i, vp]),
            "fno_layer2d_fused_supported": (i, [vp, i]),
            "fno_layer2d_fused_workspace_bytes": (C.c_size_t, [vp, i, i]),
            "fno_layer2d_inv_fused": (i, [vp, vp, vp, vp, vp, vp, vp, vp, i, i, i, f, i, i, vp]),
            "fno_pointwise_fwd": (i, [vp, vp, vp, vp, i, i, i, l, i, vp]),
            "fno_pointwise_wgrad_workspace_bytes": (C.c_size_t, [i, i, i, l]),
            "fno_pointwise_wgrad": (i, [vp, vp, vp, vp, vp, i, i, i, l, vp]),
            "fno_pointwise_bwd": (i, [vp, vp, vp, vp, vp, vp, vp, i, i, i, l, vp]),
            "fno_lift_stats_workspace_bytes": (C.c_size_t, [i, i]),
            "fno_lift_stats": (i, [vp, vp, vp, i, l, i, vp]),
            "fno_lift_fwd": (i, [vp, vp, vp, vp, vp, vp, i, i, i, i, i, i, i, i, i, vp]),
            "fno_lift_bwd_workspace_bytes": (C.c_size_t, [i, i, i, i]),
            "fno_lift_bwd": (i, [vp, vp, vp, vp, vp, vp, vp, i, i, i, i, i, i, i, i, i, vp]),
            "fno_lift_dgrad": (i, [vp, vp, vp, vp, vp, i, i, i, i, i, i, i, i, i, vp]),
            "fno_head_fwd": (i, [vp, vp, vp, vp, vp, vp, vp, i, i, i, i, i, i, i, i, vp]),
            "fno_head_fwd_tc": (i, [vp, vp, vp, vp, vp, vp, vp, i, i, i, i, i, i, i, i, vp]),
            "fno_head_bwd_workspace_bytes": (C.c_size_t, [i, i, i]),
            "fno_head_bwd": (i, [vp] * 12 + [i] * 8 + [vp]),
            "fno_head_bwd_tc": (i, [vp] * 12 + [i] * 8 + [vp]),
            "fno_head_fwd_wide_tc": (i, [vp] * 7 + [i] * 8 + [vp]),
            "fno_head_bwd_wide_supported": (i, [i, i, i, i, i]),
            "fno_head_bwd_wide_workspace_bytes": (C.c_size_t, [i, i, i, i, i]),
            "fno_head_bwd_wide_tc": (i, [vp] * 12 + [i] * 8 + [vp]),
            "fno_nrmse_workspace_bytes": (C.c_size_t, [i, i]),
            "fno_nrmse_fwd": (i, [vp, vp, vp, vp, i, l, i, vp]),
            "fno_nrmse_bwd": (i, [vp, vp, vp, vp, vp, i, l, i, vp]),
            "fno_opt_chunk_floats": (i, []),
            "fno_opt_chunk_bytes": (C.c_size_t, []),
            "fno_clip_adam_step": (i, [vp, i, vp, vp, vp, vp]),
        }
        for name, (res, args) in sig.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


# K1 with its contiguous-axis half as a tcgen05 truncated-DFT GEMM (transform2d_tc.cu, A operand through
# TMEM, 3xTF32: fp32-mode accuracy) followed by the FP32 strided-axis fold.  FNO_K1_TC=0 selects the all-FP32 kernel.
K1_TENSOR_CORES = os.environ.get("FNO_K1_TC", "1") != "0"

EXPORTED_SYMBOLS = (
    "fno_version", "fno_sm_arch", "fno_last_error", "fno_launch_count", "fno_shutdown",
    "fno_set_math_mode", "fno_get_math_mode", "fno_window_gather", "fno_window_gather_joint",
    "fno_plan2d_create", "fno_plan3d_create", "fno_plan_destroy", "fno_plan_workspace_bytes",
    "fno_sc2d_fwd_transform", "fno_sc2d_fwd_workspace_bytes", "fno_sc2d_fwd_transform_ws",
    "fno_sc3d_fwd_transform", "fno_mix_fwd", "fno_mix_bwd", "fno_mix_tc_supported",
    "fno_sc2d_inv_transform", "fno_sc3d_inv_transform", "fno_layer2d_fused_supported",
    "fno_layer2d_fused_workspace_bytes", "fno_layer2d_inv_fused", "fno_pointwise_fwd",
    "fno_pointwise_wgrad_workspace_bytes", "fno_pointwise_wgrad", "fno_pointwise_bwd",
    "fno_lift_stats_workspace_bytes", "fno_lift_stats", "fno_lift_fwd", "fno_lift_bwd_workspace_bytes",
    "fno_lift_bwd", "fno_lift_dgrad", "fno_head_fwd", "fno_head_fwd_tc", "fno_head_bwd_workspace_bytes", "fno_head_bwd", "fno_head_bwd_tc",
    "fno_head_fwd_wide_tc", "fno_head_bwd_wide_supported", "fno_head_bwd_wide_workspace_bytes", "fno_head_bwd_wide_tc",
    "fno_nrmse_workspace_bytes", "fno_nrmse_fwd", "fno_nrmse_bwd", "fno_opt_chunk_floats",
    "fno_opt_chunk_bytes", "fno_clip_adam_step",
    "fno_metric_workspace_bytes", "fno_metric_func", "fno_window_shift", "fno_window_shift_bwd",
    "fno_window_shift_split", "fno_window_shift_split_bwd",
    "fno_sc1d_fwd_transform", "fno_sc1d_inv_transform", "fno_mix1d_fwd", "fno_mix1d_bwd",
)


def _check(rc: int, what: str):
    if rc != 0:
        msg = load().fno_last_error().decode("utf-8", "replace")
        raise FnoError(f"{what} failed (code {rc}): {msg}")


def launch_count() -> int:
    return int(load().fno_launch_count())


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _on_tensor_device(fn):
    """Runs a wrapper with the CUDA device of its first tensor argument current: the launch then goes to that device's
    current stream, per-device kernel attributes apply to the right context, and a plan created for another device is
    refused instead of being launched with foreign pointers (single-process multi-GPU use)."""
    import functools

    @functools.wraps(fn)
    def inner(*args, **kwargs):
        dev = None
        plan = None
        for a in list(args) + list(kwargs.values()):
            if isinstance(a, Plan) and plan is None:
                plan = a
            elif isinstance(a, torch.Tensor) and a.is_cuda and dev is None:
                dev = a.device
            elif isinstance(a, (list, tuple)) and dev is None and a and isinstance(a[0], torch.Tensor) and a[0].is_cuda:
                dev = a[0].device
        if dev is None:
            return fn(*args, **kwargs)
        if plan is not None and plan.device != dev.index:
            raise FnoError(f"plan was created for cuda:{plan.device}, tensors live on {dev}")
        if dev.index == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)
    return inner


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _require(t: torch.Tensor, dtype, name: str):
    if not t.is_cuda:
        raise FnoError(f"{name} must be a CUDA tensor (libfno_sm100 has no CPU path); got device {t.device}")
    if t.dtype != dtype:
        raise FnoError(f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise FnoError(f"{name} must be contiguous")


# ---------------------------------------------------------------------------------------------
# plans (cached per device / geometry; immutable, thread-safe once created)
# ---------------------------------------------------------------------------------------------
class Plan:
    def __init__(self, handle: int, device: int, spatial: Sequence[int], modes: Sequence[int]):
        self.handle = handle
        self.device = device
        self.spatial = tuple(spatial)
        self.modes = tuple(modes)
        self.nd = len(spatial)

    @property
    def spec_shape(self):
        """Retained-spectrum extents: (2*m1, m2) or (2*m1, 2*m2, m3)."""
        return tuple(2 * m for m in self.modes[:-1]) + (self.modes[-1],)

    @property
    def num_modes(self) -> int:
        n = 1
        for s in self.spec_shape:
            n *= s
        return n

    @property
    def npix(self) -> int:
        n = 1
        for s in self.spatial:
            n *= s
        return n

    def workspace(self, planes: int, device) -> Optional[torch.Tensor]:
        if self.nd == 2:
            return None
        nbytes = load().fno_plan_workspace_bytes(self.handle, planes)
        return torch.empty(nbytes // 4, dtype=torch.float32, device=device)


_plans: dict = {}
_plans_lock = threading.Lock()


def get_plan(device: torch.device, spatial: Sequence[int], modes: Sequence[int]) -> Plan:
    if device.type != "cuda":
        raise FnoError(f"the FNO spectral path runs on CUDA (sm_100a) only, got device {device}")
    idx = device.index if device.index is not None else torch.cuda.current_device()
    key = (idx, tuple(int(s) for s in spatial), tuple(int(m) for m in modes))
    plan = _plans.get(key)
    if plan is not None:
        return plan
    with _plans_lock:
        plan = _plans.get(key)
        if plan is not None:
            return plan
        lib = load()
        h = C.c_void_p()
        if len(spatial) == 2:
            rc = lib.fno_plan2d_create(idx, int(spatial[0]), int(spatial[1]), int(modes[0]), int(modes[1]), C.byref(h))
        elif len(spatial) == 3:
            rc = lib.fno_plan3d_create(idx, *[int(s) for s in spatial], *[int(m) for m in modes], C.byref(h))
        else:
            raise FnoError("only 2-D and 3-D spectral convolutions exist in the reference")
        _check(rc, "fno_plan_create")
        plan = Plan(h.value, idx, spatial, modes)
        _plans[key] = plan
    return plan


def shutdown():
    with _plans_lock:
        _plans.clear()
        if _lib is not None:
            _lib.fno_shutdown()


# ---------------------------------------------------------------------------------------------
# thin call wrappers (shape bookkeeping only)
# ---------------------------------------------------------------------------------------------
@_on_tensor_device
def fwd_transform(plan: Plan, x: torch.Tensor, *, preact: Optional[torch.Tensor] = None,
                  ds_out: Optional[torch.Tensor] = None, cmode: int = 0, scale: float = 1.0) -> torch.Tensor:
    """x [B, C, *spatial] f32 -> retained spectrum [B, C, *spec_shape] complex64."""
    _require(x, torch.float32, "x")
    if tuple(x.shape[-plan.nd:]) != plan.spatial:
        raise FnoError(f"x spatial dims {tuple(x.shape[-plan.nd:])} do not match plan {plan.spatial}")
    planes = x.numel() // plan.npix
    if preact is not None:
        _require(preact, torch.float32, "preact")
    if ds_out is not None:
        _require(ds_out, torch.float32, "ds_out")
    X = torch.empty(tuple(x.shape[:-plan.nd]) + plan.spec_shape, dtype=torch.complex64, device=x.device)
    lib = load()
    if plan.nd == 2:
        nbytes = lib.fno_sc2d_fwd_workspace_bytes(plan.handle, planes) if K1_TENSOR_CORES else 0
        if nbytes:
            work = torch.empty(nbytes // 4, dtype=torch.float32, device=x.device)
            rc = lib.fno_sc2d_fwd_transform_ws(plan.handle, x.data_ptr(), _ptr(preact), _ptr(ds_out), X.data_ptr(),
                                               work.data_ptr(), planes, cmode, scale, _stream())
        else:
            rc = lib.fno_sc2d_fwd_transform(plan.handle, x.data_ptr(), _ptr(preact), _ptr(ds_out), X.data_ptr(), planes,
                                            cmode, scale, _stream())
    else:
        work = plan.workspace(planes, x.device)
        rc = lib.fno_sc3d_fwd_transform(plan.handle, x.data_ptr(), _ptr(preact), _ptr(ds_out), X.data_ptr(),
                                        work.data_ptr(), planes, cmode, scale, _stream())
    _check(rc, "fno_fwd_transform")
    return X


@_on_tensor_device
def inv_transform(plan: Plan, Y: torch.Tensor, *, addend: Optional[torch.Tensor] = None,
                  s_out: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None, cmode: int = 1,
                  scale: Optional[float] = None, apply_gelu: bool = False) -> torch.Tensor:
    """Y [B, C, *spec_shape] complex64 -> [B, C, *spatial] f32 (+addend, optional GELU)."""
    _require(Y, torch.complex64, "Y")
    if tuple(Y.shape[-plan.nd:]) != plan.spec_shape:
        raise FnoError(f"Y mode dims {tuple(Y.shape[-plan.nd:])} do not match plan {plan.spec_shape}")
    lead = tuple(Y.shape[:-plan.nd])
    planes = Y.numel() // plan.num_modes
    if scale is None:
        scale = 1.0 / plan.npix
    if out is None:
        out = torch.empty(lead + plan.spatial, dtype=torch.float32, device=Y.device)
    _require(out, torch.float32, "out")
    if addend is not None:
        _require(addend, torch.float32, "addend")
    if s_out is not None:
        _require(s_out, torch.float32, "s_out")
    lib = load()
    if plan.nd == 2:
        rc = lib.fno_sc2d_inv_transform(plan.handle, Y.data_ptr(), _ptr(addend), _ptr(s_out), out.data_ptr(), planes,
                                        cmode, scale, int(apply_gelu), _stream())
    else:
        work = plan.workspace(planes, Y.device)
        rc = lib.fno_sc3d_inv_transform(plan.handle, Y.data_ptr(), _ptr(addend), _ptr(s_out), out.data_ptr(),
                                        work.data_ptr(), planes, cmode, scale, int(apply_gelu), _stream())
    _check(rc, "fno_inv_transform")
    return out


# K3 with the 1x1-conv bypass folded into one tcgen05 GEMM per row (layer2d_tc.cu).  FNO_LAYER_TC=0 selects the
# round-1 path (pointwise kernel + FP32 inverse transform).
LAYER_TENSOR_CORES = os.environ.get("FNO_LAYER_TC", "1") != "0"


def layer_fused_supported(plan: Plan, width: int) -> bool:
    return bool(LAYER_TENSOR_CORES and plan.nd == 2 and load().fno_layer2d_fused_supported(plan.handle, int(width)))


@_on_tensor_device
def layer_inv_fused(plan: Plan, Y: torch.Tensor, a: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], *,
                    s_out: Optional[torch.Tensor] = None, cmode: int = 1, scale: Optional[float] = None,
                    apply_gelu: bool = False, transpose: bool = False) -> torch.Tensor:
    """act(K3(Y) + W a + bias) in one tensor-core pass over a (fno_layer2d_inv_fused).  a [B, C, H, W] f32,
    Y [B, C, 2*m1, m2] c64, weight = the 1x1-conv weight [C, C, 1, 1]; transpose: W^T a (the layer's data gradient)."""
    _require(Y, torch.complex64, "Y")
    _require(a, torch.float32, "a")
    _require(weight, torch.float32, "weight")
    B, Cw = a.shape[0], a.shape[1]
    if tuple(a.shape[2:]) != plan.spatial or tuple(Y.shape) != (B, Cw) + plan.spec_shape:
        raise FnoError(f"layer_inv_fused: a {tuple(a.shape)} / Y {tuple(Y.shape)} do not match plan {plan.spatial} {plan.spec_shape}")
    if weight.shape[0] != Cw or weight.shape[1] != Cw:
        raise FnoError(f"layer_inv_fused: weight {tuple(weight.shape)} is not [{Cw}, {Cw}, ...]")
    if bias is not None:
        _require(bias, torch.float32, "bias")
    if s_out is not None:
        _require(s_out, torch.float32, "s_out")
    if scale is None:
        scale = 1.0 / plan.npix
    lib = load()
    nbytes = lib.fno_layer2d_fused_workspace_bytes(plan.handle, B, Cw)
    if nbytes == 0:
        raise FnoError("layer_inv_fused: geometry not supported by the tensor-core layer kernel")
    work = torch.empty(nbytes // 4, dtype=torch.float32, device=a.device)
    out = torch.empty_like(a)
    rc = lib.fno_layer2d_inv_fused(plan.handle, Y.data_ptr(), a.data_ptr(), weight.data_ptr(), _ptr(bias), _ptr(s_out),
                                   out.data_ptr(), work.data_ptr(), B, Cw, cmode, scale, int(apply_gelu), int(transpose),
                                   _stream())
    _check(rc, "fno_layer2d_inv_fused")
    return out


def _ptr_array(tensors: Sequence[torch.Tensor]):
    arr = (C.c_void_p * len(tensors))()
    for k, t in enumerate(tensors):
        arr[k] = t.data_ptr()
    return arr


def mix_tc_supported(plan: Plan, Ci: int, Co: int) -> bool:
    """True when K2 (mix_fwd / mix_bwd) runs this shape on the tensor cores (width 33..64, even innermost mode count)."""
    return bool(load().fno_mix_tc_supported(plan.handle, int(Ci), int(Co)))


@_on_tensor_device
def mix_fwd(plan: Plan, X: torch.Tensor, weights: Sequence[torch.Tensor]) -> torch.Tensor:
    _require(X, torch.complex64, "X")
    B, Ci = X.shape[0], X.shape[1]
    Co = weights[0].shape[1]
    for k, w in enumerate(weights):
        _require(w, torch.complex64, f"weights{k + 1}")
        if tuple(w.shape) != (Ci, Co) + plan.modes:
            raise FnoError(f"weights{k + 1} shape {tuple(w.shape)} != {(Ci, Co) + plan.modes}")
    Y = torch.empty((B, Co) + plan.spec_shape, dtype=torch.complex64, device=X.device)
    rc = load().fno_mix_fwd(plan.handle, X.data_ptr(), _ptr_array(weights), Y.data_ptr(), B, Ci, Co, _stream())
    _check(rc, "fno_mix_fwd")
    return Y


@_on_tensor_device
def mix_bwd(plan: Plan, X: Optional[torch.Tensor], gY: torch.Tensor, weights: Sequence[torch.Tensor], *,
            need_gx: bool = True, need_gw: bool = True):
    _require(gY, torch.complex64, "gY")
    B, Co = gY.shape[0], gY.shape[1]
    Ci = weights[0].shape[0]
    gX = torch.empty((B, Ci) + plan.spec_shape, dtype=torch.complex64, device=gY.device) if need_gx else None
    gws = [torch.empty_like(w) for w in weights] if need_gw else None
    if need_gw:
        _require(X, torch.complex64, "X")
    rc = load().fno_mix_bwd(plan.handle, _ptr(X), gY.data_ptr(), _ptr_array(weights), _ptr(gX),
                            _ptr_array(gws) if need_gw else None, B, Ci, Co, _stream())
    _check(rc, "fno_mix_bwd")
    return gX, gws


@_on_tensor_device
def pointwise_fwd(a: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], *, transpose: bool = False,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """1x1 conv on channel-first [B, C, *spatial]; weight is the conv weight [Co, Ci, 1, 1(, 1)]."""
    _require(a, torch.float32, "a")
    _require(weight, torch.float32, "weight")
    Co, Ci = weight.shape[0], weight.shape[1]
    B = a.shape[0]
    N = a.numel() // (B * a.shape[1])
    cin, cout = (Co, Ci) if transpose else (Ci, Co)
    if a.shape[1] != cin:
        raise FnoError(f"pointwise: input has {a.shape[1]} channels, expected {cin}")
    if out is None:
        out = torch.empty((B, cout) + tuple(a.shape[2:]), dtype=torch.float32, device=a.device)
    if bias is not None:
        _require(bias, torch.float32, "bias")
    rc = load().fno_pointwise_fwd(a.data_ptr(), weight.data_ptr(), _ptr(bias), out.data_ptr(), B, Co, Ci, N,
                                  int(transpose), _stream())
    _check(rc, "fno_pointwise_fwd")
    return out


@_on_tensor_device
def pointwise_wgrad_buffers(ds: torch.Tensor, a: torch.Tensor, weight_shape, *, need_bias: bool = True):
    """Allocates (gw, gb, work) for pointwise_wgrad on the CURRENT stream (so that the launch itself
    may run on a side stream without handing the caching allocator cross-stream blocks)."""
    B, Co, Ci = ds.shape[0], ds.shape[1], a.shape[1]
    N = ds.numel() // (B * Co)
    nbytes = load().fno_pointwise_wgrad_workspace_bytes(B, Co, Ci, N)
    work = torch.empty(nbytes // 4, dtype=torch.float32, device=ds.device)
    gw = torch.empty(tuple(weight_shape), dtype=torch.float32, device=ds.device)
    gb = torch.empty(Co, dtype=torch.float32, device=ds.device) if need_bias else None
    return gw, gb, work


@_on_tensor_device
def pointwise_bwd(ds: torch.Tensor, a: torch.Tensor, weight: torch.Tensor, *, need_bias: bool = True):
    """Autograd of the 1x1 convolution in one call: (dx = W^T ds, gW, gb).  ds is read once when the TMA-fed
    weight-gradient kernel can carry the data gradient (fno_pointwise_bwd)."""
    for t, n in ((ds, "ds"), (a, "a"), (weight, "weight")):
        _require(t, torch.float32, n)
    gw, gb, work = pointwise_wgrad_buffers(ds, a, weight.shape, need_bias=need_bias)
    B, Co, Ci = ds.shape[0], ds.shape[1], a.shape[1]
    N = ds.numel() // (B * Co)
    dx = torch.empty_like(a)
    rc = load().fno_pointwise_bwd(ds.data_ptr(), a.data_ptr(), weight.data_ptr(), dx.data_ptr(), gw.data_ptr(), _ptr(gb),
                                  work.data_ptr(), B, Co, Ci, N, _stream())
    _check(rc, "fno_pointwise_bwd")
    return dx, gw, gb


@_on_tensor_device
def pointwise_wgrad(ds: torch.Tensor, a: torch.Tensor, weight_shape, *, need_bias: bool = True, buffers=None):
    _require(ds, torch.float32, "ds")
    _require(a, torch.float32, "a")
    B, Co, Ci = ds.shape[0], ds.shape[1], a.shape[1]
    N = ds.numel() // (B * Co)
    gw, gb, work = buffers if buffers is not None else pointwise_wgrad_buffers(ds, a, weight_shape, need_bias=need_bias)
    rc = load().fno_pointwise_wgrad(ds.data_ptr(), a.data_ptr(), gw.data_ptr(), _ptr(gb), work.data_ptr(), B, Co, Ci, N,
                                    _stream())
    _check(rc, "fno_pointwise_wgrad")
    return gw, gb


# ---------------------------------------------------------------------------------------------
# lift / projection head (trunk layout h[B, C, R_out, Wp], see include/fno_sm100.h)
# ---------------------------------------------------------------------------------------------
import os as _os

HEAD_TC = _os.environ.get("FNO_HEAD_TC", "1") != "0"
HEAD_BWD_TC = _os.environ.get("FNO_HEAD_BWD_TC", "1") != "0"


class TrunkGeo:
    """Geometry of the channel-first padded trunk activation for inputs [B, *spatial, ...]."""

    def __init__(self, spatial: Sequence[int], padding: int):
        self.spatial = tuple(int(s) for s in spatial)
        self.padding = int(padding)
        if len(self.spatial) == 2:      # F.pad(x, [0, p, 0, p]): both axes (fno.py:159)
            self.R_in, self.W_in = self.spatial
            self.R_out, self.Wp = self.R_in + padding, self.W_in + padding
            self.padded = (self.R_out, self.Wp)
        elif len(self.spatial) == 3:    # F.pad(x, [0, p]): last axis only (fno.py:360)
            self.R_in, self.W_in = self.spatial[0] * self.spatial[1], self.spatial[2]
            self.R_out, self.Wp = self.R_in, self.W_in + padding
            self.padded = (self.spatial[0], self.spatial[1], self.Wp)
        else:
            raise FnoError("only 2-D and 3-D models exist in the reference")
        self.npix = self.R_in * self.W_in

    @property
    def ints(self):
        return self.R_in, self.W_in, self.R_out, self.Wp


@_on_tensor_device
def lift_stats(x: torch.Tensor) -> torch.Tensor:
    """x [B, *spatial, T, V] -> [B, 2, V] (mean, std + 1e-7) over everything but batch and variable."""
    _require(x, torch.float32, "x")
    B, V = x.shape[0], x.shape[-1]
    entries = x.numel() // (B * V)
    lib = load()
    work = torch.empty(lib.fno_lift_stats_workspace_bytes(B, V) // 4, dtype=torch.float32, device=x.device)
    stats = torch.empty((B, 2, V), dtype=torch.float32, device=x.device)
    _check(lib.fno_lift_stats(x.data_ptr(), stats.data_ptr(), work.data_ptr(), B, entries, V, _stream()),
           "fno_lift_stats")
    return stats


@_on_tensor_device
def lift_fwd(geo: TrunkGeo, x, grid, stats, W0, b0) -> torch.Tensor:
    for t, n in ((x, "x"), (grid, "grid"), (stats, "stats"), (W0, "fc0.weight"), (b0, "fc0.bias")):
        _require(t, torch.float32, n)
    B, T, V, G, C = x.shape[0], x.shape[-2], x.shape[-1], grid.shape[-1], W0.shape[0]
    if W0.shape[1] != T * V + G:
        raise FnoError(f"fc0.weight has {W0.shape[1]} inputs, expected {T * V + G}")
    h = torch.empty((B, C) + geo.padded, dtype=torch.float32, device=x.device)
    _check(load().fno_lift_fwd(x.data_ptr(), grid.data_ptr(), stats.data_ptr(), W0.data_ptr(), b0.data_ptr(),
                               h.data_ptr(), B, *geo.ints, T, V, G, C, _stream()), "fno_lift_fwd")
    return h


@_on_tensor_device
def lift_bwd(geo: TrunkGeo, x, grid, stats, dh, W0_shape):
    _require(dh, torch.float32, "dh")
    B, T, V, G, C = x.shape[0], x.shape[-2], x.shape[-1], grid.shape[-1], W0_shape[0]
    lib = load()
    work = torch.empty(lib.fno_lift_bwd_workspace_bytes(T, V, G, C) // 4, dtype=torch.float32, device=x.device)
    gW0 = torch.empty(tuple(W0_shape), dtype=torch.float32, device=x.device)
    gb0 = torch.empty(C, dtype=torch.float32, device=x.device)
    _check(lib.fno_lift_bwd(x.data_ptr(), grid.data_ptr(), stats.data_ptr(), dh.data_ptr(), gW0.data_ptr(),
                            gb0.data_ptr(), work.data_ptr(), B, *geo.ints, T, V, G, C, _stream()), "fno_lift_bwd")
    return gW0, gb0


@_on_tensor_device
def lift_dgrad(geo: TrunkGeo, dh, W0, stats, x_shape, grid_shape, *, need_dx: bool = True, need_dgrid: bool = False):
    """Gradient of lift_fwd w.r.t. x [B, *spatial, T, V] and grid [B, *spatial, G] (statistics held constant), from
    dh in trunk layout.  Returns (dx or None, dgrid or None)."""
    for t, n in ((dh, "dh"), (W0, "fc0.weight"), (stats, "stats")):
        _require(t, torch.float32, n)
    B, T, V, G, C = x_shape[0], x_shape[-2], x_shape[-1], grid_shape[-1], W0.shape[0]
    if tuple(dh.shape) != (B, C) + geo.padded or W0.shape[1] != T * V + G:
        raise FnoError(f"lift_dgrad: dh {tuple(dh.shape)} / fc0.weight {tuple(W0.shape)} do not match x {tuple(x_shape)}")
    dx = torch.empty(tuple(x_shape), dtype=torch.float32, device=dh.device) if need_dx else None
    dgrid = torch.empty(tuple(grid_shape), dtype=torch.float32, device=dh.device) if need_dgrid else None
    _check(load().fno_lift_dgrad(dh.data_ptr(), W0.data_ptr(), stats.data_ptr(), _ptr(dx), _ptr(dgrid), B, *geo.ints,
                                 T, V, G, C, _stream()), "fno_lift_dgrad")
    return dx, dgrid


MATH_MODES = {"fp32": 0, "tf32": 1, "bf16": 2}


def set_math_mode(mode: str) -> str:
    """Arithmetic mode of the tensor-core kernels: "fp32" (3xTF32 split, <= 1e-5 relative; default), "tf32" (single
    kind::tf32 pass, stated bound <= 2e-3 relative) or "bf16" (operands rounded to bfloat16, single pass, fp32 accumulate,
    stated bound <= 2e-2).  Returns the previous mode."""
    if mode not in MATH_MODES:
        raise FnoError(f"unknown math mode {mode!r} (expected one of {sorted(MATH_MODES)})")
    prev = load().fno_set_math_mode(MATH_MODES[mode])
    if prev < 0:
        _check(prev, "fno_set_math_mode")
    return {v: k for k, v in MATH_MODES.items()}[prev]


def get_math_mode() -> str:
    return {v: k for k, v in MATH_MODES.items()}[load().fno_get_math_mode()]


@_on_tensor_device
def head_fwd(geo: TrunkGeo, h, W1, b1, W2, b2, stats) -> torch.Tensor:
    for t, n in ((h, "h"), (W1, "fc1.weight"), (b1, "fc1.bias"), (W2, "fc2.weight"), (b2, "fc2.bias"),
                 (stats, "stats")):
        _require(t, torch.float32, n)
    B, C, HID, V = h.shape[0], h.shape[1], W1.shape[0], W2.shape[0]
    if tuple(h.shape[2:]) != geo.padded or W1.shape[1] != C or W2.shape[1] != HID:
        raise FnoError(f"head: inconsistent shapes h {tuple(h.shape)}, fc1 {tuple(W1.shape)}, fc2 {tuple(W2.shape)}")
    out = torch.empty((B,) + geo.spatial + (V,), dtype=torch.float32, device=h.device)
    if HEAD_TC and HID == 128 and C <= 32 and V <= 8:
        # tensor-core path (tcgen05 kind::tf32, 3xTF32 split: fp32-mode accuracy)
        _check(load().fno_head_fwd_tc(h.data_ptr(), W1.data_ptr(), b1.data_ptr(), W2.data_ptr(), b2.data_ptr(),
                                      stats.data_ptr(), out.data_ptr(), B, *geo.ints, C, HID, V, _stream()),
               "fno_head_fwd_tc")
        return out
    if HEAD_TC and HID == 128 and C <= 64 and V <= 4:
        # wide trunks (cfg 3): h through tensor memory as the A operand (head_wide_tc.cu)
        _check(load().fno_head_fwd_wide_tc(h.data_ptr(), W1.data_ptr(), b1.data_ptr(), W2.data_ptr(), b2.data_ptr(),
                                           stats.data_ptr(), out.data_ptr(), B, *geo.ints, C, HID, V, _stream()),
               "fno_head_fwd_wide_tc")
        return out
    _check(load().fno_head_fwd(h.data_ptr(), W1.data_ptr(), b1.data_ptr(), W2.data_ptr(), b2.data_ptr(),
                               stats.data_ptr(), out.data_ptr(), B, *geo.ints, C, HID, V, _stream()), "fno_head_fwd")
    return out


@_on_tensor_device
def head_bwd(geo: TrunkGeo, h, dout, W1, b1, W2, stats, dh_out: Optional[torch.Tensor] = None):
    """Returns (dh, gW1, gb1, gW2, gb2).  ``dh_out``: where to write dh (shape of h, e.g. this head's sample range of
    a larger trunk gradient); every form writes it whole, zero in the padding."""
    _require(dout, torch.float32, "dout")
    B, C, HID, V = h.shape[0], h.shape[1], W1.shape[0], W2.shape[0]
    lib = load()
    if dh_out is not None:
        _require(dh_out, torch.float32, "dh_out")
        if dh_out.shape != h.shape:
            raise FnoError(f"head_bwd: dh_out {tuple(dh_out.shape)} must have the shape of h {tuple(h.shape)}")
    dh = torch.empty_like(h) if dh_out is None else dh_out
    gW1, gb1 = torch.empty_like(W1), torch.empty(HID, dtype=torch.float32, device=h.device)
    gW2, gb2 = torch.empty_like(W2), torch.empty(V, dtype=torch.float32, device=h.device)
    tc = HEAD_BWD_TC and HID == 128 and C <= 23 and V <= 8
    # wide trunks (24 <= C <= 64, cfg 3): two tcgen05 launches with the hidden-layer gradient passing through HBM
    wide = HEAD_BWD_TC and not tc and bool(lib.fno_head_bwd_wide_supported(geo.R_out, geo.Wp, C, HID, V))
    if wide:
        nbytes, fn, name = lib.fno_head_bwd_wide_workspace_bytes(B, geo.R_out, geo.Wp, C, V), lib.fno_head_bwd_wide_tc, "fno_head_bwd_wide_tc"
    else:
        nbytes = lib.fno_head_bwd_workspace_bytes(C, HID, V)
        fn, name = (lib.fno_head_bwd_tc, "fno_head_bwd_tc") if tc else (lib.fno_head_bwd, "fno_head_bwd")   # tcgen05 3xTF32 / FP32
    work = torch.empty(nbytes // 4, dtype=torch.float32, device=h.device)
    _check(fn(h.data_ptr(), dout.data_ptr(), W1.data_ptr(), b1.data_ptr(), W2.data_ptr(),
              stats.data_ptr(), dh.data_ptr(), gW1.data_ptr(), gb1.data_ptr(), gW2.data_ptr(),
              gb2.data_ptr(), work.data_ptr(), B, *geo.ints, C, HID, V, _stream()), name)
    return dh, gW1, gb1, gW2, gb2


@_on_tensor_device
def window_gather(traj: torch.Tensor, traj_idx: torch.Tensor, t_start: torch.Tensor, initial_step: int, rollout: int,
                  out=None):
    """traj [n_traj, pixels, T, V] (device, time-inner) -> xx [B, pixels, initial_step, V], yy [B, pixels, rollout, V]
    for the items (traj_idx[b], t_start[b]); one copy kernel, nothing touches the host."""
    _require(traj, torch.float32, "traj")
    if traj.dim() != 4 or traj_idx.dtype != torch.int64 or t_start.dtype != torch.int32 or \
            traj_idx.device != traj.device or t_start.device != traj.device or traj_idx.shape != t_start.shape:
        raise FnoError("window_gather: traj [n, pixels, T, V] f32, traj_idx int64 [B], t_start int32 [B], one device")
    n, npix, T, V = traj.shape
    B = traj_idx.numel()
    if out is not None:                      # caller-owned (xx, yy): fixed addresses for CUDA-graph steps that alias them
        xx, yy = out
        _require(xx, torch.float32, "xx")
        _require(yy, torch.float32, "yy")
        if xx.numel() != B * npix * initial_step * V or yy.numel() != B * npix * rollout * V:
            raise FnoError("window_gather: out buffers have the wrong size")
    else:
        xx = torch.empty((B, npix, initial_step, V), dtype=torch.float32, device=traj.device)
        yy = torch.empty((B, npix, rollout, V), dtype=torch.float32, device=traj.device)
    _check(load().fno_window_gather(traj.data_ptr(), traj_idx.data_ptr(), t_start.data_ptr(), xx.data_ptr(),
                                    yy.data_ptr(), B, npix, T, V, initial_step, rollout, _stream()),
           "fno_window_gather")
    return xx, yy


def _overlaps(a: torch.Tensor, b: torch.Tensor) -> bool:
    a0, b0 = a.data_ptr(), b.data_ptr()
    return a0 < b0 + b.numel() * b.element_size() and b0 < a0 + a.numel() * a.element_size()


@_on_tensor_device
def window_gather_joint(traj: torch.Tensor, traj_aux: torch.Tensor, traj_idx: torch.Tensor, t_start: torch.Tensor,
                        initial_step: int, rollout: int, out=None):
    """traj [n, pixels, T, V], traj_aux [n, A, pixels, T, V] (device, time-inner) -> xj [B + B*A, pixels, initial_step, V]
    (primary rows, then item b's auxiliary stream k at row B + b*A + k), yy [B, pixels, rollout, V],
    yy_aux [B*A, pixels, rollout, V]; one copy kernel.  ``out = (xj, yy, yy_aux)``: caller-owned buffers."""
    _require(traj, torch.float32, "traj")
    _require(traj_aux, torch.float32, "traj_aux")
    if traj.dim() != 4 or traj_aux.dim() != 5 or traj_idx.dtype != torch.int64 or t_start.dtype != torch.int32 or \
            traj_idx.device != traj.device or t_start.device != traj.device or traj_aux.device != traj.device or \
            traj_idx.shape != t_start.shape:
        raise FnoError("window_gather_joint: traj [n, pixels, T, V] and traj_aux [n, A, pixels, T, V] f32, traj_idx "
                       "int64 [B], t_start int32 [B], one device")
    n, npix, T, V = traj.shape
    if traj_aux.shape[0] != n or tuple(traj_aux.shape[2:]) != (npix, T, V):
        raise FnoError(f"window_gather_joint: traj_aux {tuple(traj_aux.shape)} does not match traj {tuple(traj.shape)}")
    A, B = traj_aux.shape[1], traj_idx.numel()
    shapes = ((B * (1 + A), npix, initial_step, V), (B, npix, rollout, V), (B * A, npix, rollout, V))
    if out is not None:                      # caller-owned: fixed addresses for CUDA-graph steps that alias them
        for t, s, name in zip(out, shapes, ("xj", "yy", "yy_aux")):
            _require(t, torch.float32, name)
            if t.numel() != s[0] * s[1] * s[2] * s[3]:
                raise FnoError(f"window_gather_joint: out buffer {name} has {t.numel()} elements, needs {s}")
            if _overlaps(t, traj) or _overlaps(t, traj_aux):
                raise FnoError(f"window_gather_joint: out buffer {name} aliases a trajectory store")
        xj, yy, yy_aux = out
    else:
        xj, yy, yy_aux = (torch.empty(s, dtype=torch.float32, device=traj.device) for s in shapes)
    _check(load().fno_window_gather_joint(traj.data_ptr(), traj_aux.data_ptr(), traj_idx.data_ptr(), t_start.data_ptr(),
                                          xj.data_ptr(), yy.data_ptr(), yy_aux.data_ptr(), B, A, npix, T, V,
                                          initial_step, rollout, _stream()),
           "fno_window_gather_joint")
    return xj, yy, yy_aux


@_on_tensor_device
def metric_func(pred: torch.Tensor, target: torch.Tensor, Lx: float = 1.0, Ly: float = 1.0, Lz: float = 1.0,
                iLow: int = 4, iHigh: int = 12) -> torch.Tensor:
    """pred, target [B, nx, ny(, nz), T, V] f32 -> device tensor [8 + T]: RMSE, nRMSE, CSV, Max, BD, F_low, F_mid, F_high,
    then the per-time-step RMSE (metrics.py:164-306 with if_mean=True, :386-393).  No host synchronisation."""
    _require(pred, torch.float32, "pred")
    _require(target, torch.float32, "target")
    if pred.shape != target.shape or pred.dim() not in (5, 6):
        raise FnoError(f"metric_func: pred / target must be equal-shaped [B, nx, ny(, nz), T, V], got {tuple(pred.shape)} / {tuple(target.shape)}")
    B, nx, ny = pred.shape[:3]
    nz = pred.shape[3] if pred.dim() == 6 else 1
    T, V = pred.shape[-2:]
    L = load()
    nbytes = L.fno_metric_workspace_bytes(B, nx, ny, nz, T, V)
    work = torch.empty(nbytes, dtype=torch.uint8, device=pred.device)
    out = torch.empty(8 + T, dtype=torch.float32, device=pred.device)
    _check(L.fno_metric_func(pred.data_ptr(), target.data_ptr(), work.data_ptr(), out.data_ptr(), B, nx, ny, nz, T, V,
                             float(Lx), float(Ly), float(Lz), int(iLow), int(iHigh), _stream()), "fno_metric_func")
    return out


@_on_tensor_device
def window_shift(xx: torch.Tensor, pred: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """xx [..., T0, V], pred [..., 1, V] -> cat(xx[..., 1:, :], pred) (metrics.py:344) in one kernel."""
    _require(xx, torch.float32, "xx")
    _require(pred, torch.float32, "pred")
    T0, V = xx.shape[-2:]
    if tuple(pred.shape) != tuple(xx.shape[:-2]) + (1, V):
        raise FnoError(f"window_shift: pred must be {tuple(xx.shape[:-2]) + (1, V)}, got {tuple(pred.shape)}")
    if out is None:
        out = torch.empty_like(xx)
    _require(out, torch.float32, "out")
    points = xx.numel() // (T0 * V)
    _check(load().fno_window_shift(xx.data_ptr(), pred.data_ptr(), out.data_ptr(), points, T0, V, _stream()),
           "fno_window_shift")
    return out


@_on_tensor_device
def window_shift_bwd(g: torch.Tensor, *, need_xx: bool = True, need_pred: bool = True):
    """Adjoint of window_shift: g [..., T0, V] -> (gxx [..., T0, V] or None, gpred [..., 1, V] or None)."""
    _require(g, torch.float32, "g")
    T0, V = g.shape[-2:]
    gxx = torch.empty_like(g) if need_xx else None
    gpred = torch.empty(tuple(g.shape[:-2]) + (1, V), dtype=torch.float32, device=g.device) if need_pred else None
    _check(load().fno_window_shift_bwd(g.data_ptr(), _ptr(gxx), _ptr(gpred), g.numel() // (T0 * V), T0, V, _stream()),
           "fno_window_shift_bwd")
    return gxx, gpred


@_on_tensor_device
def window_shift_split(xx: torch.Tensor, pred_a: torch.Tensor, pred_b: torch.Tensor) -> torch.Tensor:
    """Joined window xx [Na + Nb, *spatial, T0, V] (the rows of pred_a's stream first), pred_a [Na, *spatial, 1, V],
    pred_b [Nb, *spatial, 1, V] -> cat(xx[..., 1:, :], cat(pred_a, pred_b)) in one kernel, without joining the two
    predictions."""
    for t, n in ((xx, "xx"), (pred_a, "pred_a"), (pred_b, "pred_b")):
        _require(t, torch.float32, n)
    T0, V = xx.shape[-2:]
    tail = tuple(xx.shape[1:-2]) + (1, V)
    if (tuple(pred_a.shape[1:]) != tail or tuple(pred_b.shape[1:]) != tail
            or pred_a.shape[0] + pred_b.shape[0] != xx.shape[0]):
        raise FnoError(f"window_shift_split: predictions {tuple(pred_a.shape)} + {tuple(pred_b.shape)} do not fill the "
                       f"last frame of {tuple(xx.shape)}")
    out = torch.empty_like(xx)
    points = xx.numel() // (T0 * V)
    _check(load().fno_window_shift_split(xx.data_ptr(), pred_a.data_ptr(), pred_b.data_ptr(), out.data_ptr(),
                                         pred_a.numel() // V, points, T0, V, _stream()), "fno_window_shift_split")
    return out


@_on_tensor_device
def window_shift_split_bwd(g: torch.Tensor, n_a: int, *, need_xx: bool = True, need_a: bool = True,
                           need_b: bool = True):
    """Adjoint of window_shift_split: g [N, *spatial, T0, V] -> (gxx or None, gpred_a [n_a, *spatial, 1, V] or None,
    gpred_b [N - n_a, *spatial, 1, V] or None)."""
    _require(g, torch.float32, "g")
    if not 0 <= n_a <= g.shape[0]:
        raise FnoError(f"window_shift_split_bwd: n_a = {n_a} outside [0, {g.shape[0]}]")
    if not (need_xx or need_a or need_b):
        raise FnoError("window_shift_split_bwd: no output requested")
    T0, V = g.shape[-2:]
    tail = tuple(g.shape[1:-2]) + (1, V)
    gxx = torch.empty_like(g) if need_xx else None
    ga = torch.empty((n_a,) + tail, dtype=torch.float32, device=g.device) if need_a else None
    gb = torch.empty((g.shape[0] - n_a,) + tail, dtype=torch.float32, device=g.device) if need_b else None
    if not any(t is not None and t.numel() > 0 for t in (gxx, ga, gb)):
        return gxx, ga, gb                   # only the gradient of an empty stream was asked for
    points = g.numel() // (T0 * V)
    _check(load().fno_window_shift_split_bwd(g.data_ptr(), _ptr(gxx), _ptr(ga), _ptr(gb), points // g.shape[0] * n_a,
                                             points, T0, V, _stream()), "fno_window_shift_split_bwd")
    return gxx, ga, gb


# ---- SpectralConv1d ------------------------------------------------------------------------------------------
@_on_tensor_device
def fwd_transform1d(x: torch.Tensor, modes: int, *, cmode: int = 0, scale: float = 1.0) -> torch.Tensor:
    """x [..., N] f32 -> [..., modes] complex64 (pruned rfft; cmode=1, scale=1/N: backward of inv_transform1d)."""
    _require(x, torch.float32, "x")
    N = x.shape[-1]
    X = torch.empty(tuple(x.shape[:-1]) + (modes,), dtype=torch.complex64, device=x.device)
    _check(load().fno_sc1d_fwd_transform(x.data_ptr(), X.data_ptr(), x.numel() // N, N, modes, cmode, scale, _stream()),
           "fno_sc1d_fwd_transform")
    return X


@_on_tensor_device
def inv_transform1d(Y: torch.Tensor, n: int, *, addend: Optional[torch.Tensor] = None, cmode: int = 1,
                    scale: Optional[float] = None) -> torch.Tensor:
    """Y [..., modes] complex64 -> [..., n] f32 (zero-padded irfft; cmode=0, scale=1: backward of fwd_transform1d)."""
    _require(Y, torch.complex64, "Y")
    m = Y.shape[-1]
    y = torch.empty(tuple(Y.shape[:-1]) + (n,), dtype=torch.float32, device=Y.device)
    if addend is not None:
        _require(addend, torch.float32, "addend")
        if addend.shape != y.shape:
            raise FnoError("inv_transform1d: addend shape mismatch")
    _check(load().fno_sc1d_inv_transform(Y.data_ptr(), _ptr(addend), y.data_ptr(), Y.numel() // m, n, m, cmode,
                                         1.0 / n if scale is None else scale, _stream()), "fno_sc1d_inv_transform")
    return y


@_on_tensor_device
def mix1d_fwd(X: torch.Tensor, W: torch.Tensor) -> torch.Tensor:
    _require(X, torch.complex64, "X")
    _require(W, torch.complex64, "W")
    B, Ci, m = X.shape
    if W.shape[0] != Ci or W.shape[2] != m:
        raise FnoError(f"mix1d: X {tuple(X.shape)} does not match W {tuple(W.shape)}")
    Y = torch.empty((B, W.shape[1], m), dtype=torch.complex64, device=X.device)
    _check(load().fno_mix1d_fwd(X.data_ptr(), W.data_ptr(), Y.data_ptr(), B, Ci, W.shape[1], m, _stream()), "fno_mix1d_fwd")
    return Y


@_on_tensor_device
def mix1d_bwd(X: torch.Tensor, gY: torch.Tensor, W: torch.Tensor, need_gx: bool = True, need_gw: bool = True):
    _require(gY, torch.complex64, "gY")
    _require(X, torch.complex64, "X")
    _require(W, torch.complex64, "W")
    B, Ci, m = X.shape
    Co = W.shape[1]
    gX = torch.empty_like(X) if need_gx else None
    gW = torch.empty_like(W) if need_gw else None
    _check(load().fno_mix1d_bwd(X.data_ptr(), gY.data_ptr(), W.data_ptr(), _ptr(gX), _ptr(gW), B, Ci, Co, m, _stream()),
           "fno_mix1d_bwd")
    return gX, gW
