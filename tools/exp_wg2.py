#!/usr/bin/env python
"""Bypass weight gradient (csrc/pointwise.cu, wgrad2_partial_kernel) at the cfg-1 layer geometry: parity against an fp64 einsum on
ragged cases (with and without the fused data gradient), then event-timed launches with L2 flushed in between
(profiles/r2g_wgrad_forms.md has the sweep over operand feeds and ring shapes that led to the tensor-map feed)."""
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
for p in (ROOT, ROOT / "sciml-pde_b200"):
    sys.path.insert(0, str(p))

import torch  # noqa: E402

from fno_b200 import lib  # noqa: E402

dev = torch.device("cuda", 0)
torch.manual_seed(0)
flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)


def ref(ds, a):
    d64, a64 = ds.double().flatten(2), a.double().flatten(2)
    return torch.einsum("bop,bip->oi", d64, a64), d64.sum((0, 2))


def check(B, C, n):
    ds = torch.randn(B, C, n, n, device=dev)
    a = torch.randn(B, C, n, n, device=dev) + 0.5
    gw, gb = lib.pointwise_wgrad(ds, a, (C, C, 1, 1))
    rw, rb = ref(ds, a)
    ew = float((gw.double().view(C, C) - rw).abs().max() / rw.abs().max())
    eb = float((gb.double() - rb).abs().max() / rb.abs().max())
    return ew, eb


def timeit(B, C, n, iters=20):
    ds = torch.randn(B, C, n, n, device=dev)
    a = torch.randn(B, C, n, n, device=dev)
    bufs = lib.pointwise_wgrad_buffers(ds, a, (C, C, 1, 1))
    for _ in range(3):
        lib.pointwise_wgrad(ds, a, (C, C, 1, 1), buffers=bufs)
    ts = []
    for _ in range(iters):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        lib.pointwise_wgrad(ds, a, (C, C, 1, 1), buffers=bufs)
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    ts.sort()
    med = ts[len(ts) // 2]
    nbytes = 8.0 * B * C * n * n
    return med, ts[0], nbytes / med * 1e-3


for (B, C, n) in ((3, 20, 34), (2, 12, 130), (5, 20, 66), (16, 20, 130), (2, 30, 34), (2, 8, 66)):
    ew, eb = check(B, C, n)
    print(f"parity B={B} C={C} n={n}: gW {ew:.2e} gb {eb:.2e}", "OK" if max(ew, eb) < 1e-5 else "FAIL", flush=True)
# the fused data gradient (cfg 4's unfused layers): dx = W^T ds from the same slabs
for (B, C, n) in ((3, 20, 34), (4, 20, 130), (2, 12, 66)):
    ds = torch.randn(B, C, n, n, device=dev)
    a = torch.randn(B, C, n, n, device=dev)
    w = torch.randn(C, C, 1, 1, device=dev) / C
    dx, gw, gb = lib.pointwise_bwd(ds, a, w)
    rdx = torch.einsum("oi,bop->bip", w.double().view(C, C), ds.double().flatten(2)).view_as(dx)
    rw, rb = ref(ds, a)
    e = [float((dx.double() - rdx).abs().max() / rdx.abs().max()), float((gw.double().view(C, C) - rw).abs().max() / rw.abs().max()),
         float((gb.double() - rb).abs().max() / rb.abs().max())]
    print(f"bwd (dgrad) B={B} C={C} n={n}: dx {e[0]:.2e} gW {e[1]:.2e} gb {e[2]:.2e}", "OK" if max(e) < 1e-5 else "FAIL", flush=True)
for B in (128, 32):
    med, best, gbs = timeit(B, 20, 130)
    print(f"B={B}: median {med:.1f} us, best {best:.1f} us, {gbs:.0f} GB/s (wgrad2 + reduce)", flush=True)
