"""Kernel-level parity: every C-ABI entry point of libfno_sm100.so against the fp64 dense-DFT
oracle (oracle/dft_oracle.py) on seeded inputs, plus the reference's own golden vectors.

Tolerance (BASELINE.json north_star, fp32 mode): max-abs-err / max-abs-ref <= 1e-5.
"""
import numpy as np
import pytest
import torch

from oracle import dft_oracle as O

pytestmark = pytest.mark.gpu
TOL = 1e-5


@pytest.fixture(scope="module")
def lib():
    from fno_b200 import lib as L

    L.load()
    return L


@pytest.fixture(autouse=True)
def fp32_mode(lib):
    """The math mode is library-global state: every test starts in fp32 mode and leaves it there, even when it fails."""
    assert lib.get_math_mode() == "fp32"
    try:
        yield
    finally:
        lib.set_math_mode("fp32")


def run_modes(lib, low, fn):
    """{mode: fn()} for fp32, tf32 and -- when ``low`` is bf16 -- bf16 mode, each on the same inputs."""
    errs = {}
    for mode in ("fp32", "tf32", "bf16")[:3 if low == "bf16" else 2]:
        lib.set_math_mode(mode)
        errs[mode] = fn()
        torch.cuda.synchronize()
    lib.set_math_mode("fp32")
    return errs


def check_mode_errors(errs, low, what, shows_mode=None):
    """errs[mode]: {result name: rel_err vs fp64}.  Every result is within its mode's bound; the results named in
    ``shows_mode`` (default: all) are more than 4x less accurate than in fp32 mode -- the mode reached the kernel -- and,
    in bf16 mode, more than 2x less accurate than in tf32 mode -- bf16 rounding reached it too."""
    print(f"{what} errors:", {m: {k: f"{v:.2e}" for k, v in e.items()} for m, e in errs.items()})
    assert max(errs["fp32"].values()) <= TOL, errs["fp32"]
    assert max(errs[low].values()) < MODE_TOL[low], errs[low]
    for k in shows_mode or errs[low]:
        assert errs[low][k] > 4 * errs["fp32"][k], (k, errs)
        if low == "bf16":
            assert errs["bf16"][k] > 2 * errs["tf32"][k], (k, errs)


def mode_params(names, cases):
    """(low, *case) parameter sets for tf32 and bf16.  The first case keeps the bare mode as its id; ``names`` label the
    cases after it."""
    assert len(names) == len(cases) - 1
    return [pytest.param(low, *case, id=f"{low}-{names[i - 1]}" if i else low)
            for i, case in enumerate(cases) for low in ("tf32", "bf16")]


def dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda()


def cplx(rng, shape, scale=1.0):
    return (scale * (rng.standard_normal(shape) + 1j * rng.standard_normal(shape))).astype(np.complex64)


PLANES_2D = [
    # B, C, H, W, m1, m2
    (2, 3, 10, 9, 3, 4),        # odd W
    (1, 2, 7, 16, 2, 5),        # odd H
    (2, 4, 12, 12, 6, 7),       # 2*m1 == H (corners touch), m2 == W/2+1 (Nyquist column)
    (3, 5, 34, 34, 12, 12),
    (2, 3, 130, 130, 12, 12),   # cfg 1 padded plane
    (1, 2, 258, 258, 16, 16),   # cfg 3 padded plane
    (1, 3, 64, 70, 12, 12),     # a 3-D slice of cfg 4
    (5, 1, 20, 6, 1, 1),        # single mode
    (1, 1, 66, 40, 32, 20),     # max supported modes1
    (7, 3, 33, 31, 5, 9),       # ragged plane count vs planes-per-CTA
]


@pytest.mark.parametrize("B,C,H,W,m1,m2", PLANES_2D)
@pytest.mark.parametrize("cmode", [0, 1])
def test_fwd_transform_2d(lib, B, C, H, W, m1, m2, cmode):
    rng = np.random.default_rng(H * 1000 + W)
    x = rng.standard_normal((B, C, H, W)).astype(np.float32)
    scale = 1.0 if cmode == 0 else 1.0 / (H * W)
    plan = lib.get_plan(torch.device("cuda", 0), (H, W), (m1, m2))
    X = lib.fwd_transform(plan, dev(x), cmode=cmode, scale=scale).cpu().numpy()
    ref = O.fwd_transform(x, (m1, m2), cmode=cmode, scale=scale)
    assert X.shape == ref.shape
    assert O.rel_err(X, ref) < TOL


@pytest.mark.parametrize("B,C,H,W,m1,m2", PLANES_2D)
@pytest.mark.parametrize("cmode", [0, 1])
def test_inv_transform_2d(lib, B, C, H, W, m1, m2, cmode):
    rng = np.random.default_rng(H * 1000 + W + 7)
    Y = cplx(rng, (B, C, 2 * m1, m2))
    scale = 1.0 if cmode == 0 else 1.0 / (H * W)
    plan = lib.get_plan(torch.device("cuda", 0), (H, W), (m1, m2))
    y = lib.inv_transform(plan, dev(Y), cmode=cmode, scale=scale).cpu().numpy()
    ref = O.inv_transform(Y, (H, W), cmode=cmode, scale=scale)
    assert O.rel_err(y, ref) < TOL


@pytest.mark.parametrize("B,C,H,W,m1,m2", [(2, 3, 10, 9, 3, 4), (2, 3, 130, 130, 12, 12), (1, 2, 64, 70, 12, 12)])
@pytest.mark.parametrize("gelu", [False, True])
def test_inv_transform_fused_epilogue(lib, B, C, H, W, m1, m2, gelu):
    rng = np.random.default_rng(11)
    Y = cplx(rng, (B, C, 2 * m1, m2), scale=30.0)
    add = rng.standard_normal((B, C, H, W)).astype(np.float32)
    plan = lib.get_plan(torch.device("cuda", 0), (H, W), (m1, m2))
    addt = dev(add)
    s_out = torch.empty_like(addt)
    out = lib.inv_transform(plan, dev(Y), addend=addt, s_out=s_out, out=addt, cmode=1, apply_gelu=gelu)
    assert out.data_ptr() == addt.data_ptr()  # in place over the addend
    s_ref = O.inv_transform(Y, (H, W), cmode=1) + add
    assert O.rel_err(s_out.cpu().numpy(), s_ref) < TOL
    ref = O.gelu(s_ref) if gelu else s_ref
    assert O.rel_err(out.cpu().numpy(), ref) < TOL


LAYER_TC_CASES = [
    # B, C, H, W, m1, m2
    (2, 3, 10, 9, 3, 4),          # odd W, partial lane tile
    (2, 4, 12, 12, 6, 7),         # touching corners, Nyquist column
    (3, 5, 34, 34, 12, 12),
    (7, 3, 33, 31, 5, 9),         # odd H and W, 2*m2 = 18 -> padded K
    (2, 20, 130, 130, 12, 12),    # cfg 1: 128 lanes + 2 edge columns, width 20
    (1, 8, 16, 132, 4, 16),       # 4 edge columns, K padding of the bypass part
    (1, 31, 20, 64, 5, 8),        # widest supported layer
    (1, 5, 64, 70, 12, 12),       # a 3-D slice of cfg 4
]


@pytest.mark.parametrize("B,C,H,W,m1,m2", LAYER_TC_CASES)
@pytest.mark.parametrize("gelu", [False, True])
def test_layer_inv_fused_tensor_core(lib, B, C, H, W, m1, m2, gelu):
    """fno_layer2d_inv_fused: K3 + 1x1-conv bypass + bias (+ GELU) as one tcgen05 GEMM per row vs the fp64 oracle
    (fno/fno.py:161-164)."""
    rng = np.random.default_rng(H * 100 + W + C)
    Y = cplx(rng, (B, C, 2 * m1, m2), scale=30.0)
    a = rng.standard_normal((B, C, H, W)).astype(np.float32)
    wl = (rng.standard_normal((C, C, 1, 1)) / np.sqrt(C)).astype(np.float32)
    bl = rng.standard_normal(C).astype(np.float32)
    plan = lib.get_plan(torch.device("cuda", 0), (H, W), (m1, m2))
    assert lib.layer_fused_supported(plan, C)
    at = dev(a)
    s_out = torch.empty_like(at)
    out = lib.layer_inv_fused(plan, dev(Y), at, dev(wl), dev(bl), s_out=s_out, cmode=1, apply_gelu=gelu)
    s_ref = O.inv_transform(Y, (H, W), cmode=1) + O.pointwise_conv(a, wl, bl)
    assert O.rel_err(s_out.cpu().numpy(), s_ref) < TOL
    ref = O.gelu(s_ref) if gelu else s_ref
    assert O.rel_err(out.cpu().numpy(), ref) < TOL
    assert torch.equal(at.cpu(), torch.from_numpy(a))          # the input is read only


@pytest.mark.parametrize("B,C,H,W,m1,m2", LAYER_TC_CASES)
def test_layer_inv_fused_adjoint(lib, B, C, H, W, m1, m2):
    """Data gradient of a Fourier layer in one pass: K3(gX; c = 1, no 1/HW) + Wl^T dS."""
    rng = np.random.default_rng(H * 100 + W + C + 1)
    gX = cplx(rng, (B, C, 2 * m1, m2))
    ds = rng.standard_normal((B, C, H, W)).astype(np.float32)
    wl = (rng.standard_normal((C, C, 1, 1)) / np.sqrt(C)).astype(np.float32)
    plan = lib.get_plan(torch.device("cuda", 0), (H, W), (m1, m2))
    ga = lib.layer_inv_fused(plan, dev(gX), dev(ds), dev(wl), None, cmode=0, scale=1.0, transpose=True)
    ref = O.inv_transform(gX, (H, W), cmode=0, scale=1.0) + np.einsum("oi,bohw->bihw", wl[:, :, 0, 0].astype(np.float64), ds)
    assert O.rel_err(ga.cpu().numpy(), ref) < TOL


def test_layer_inv_fused_rejects_bad_arguments(lib):
    plan = lib.get_plan(torch.device("cuda", 0), (300, 300), (12, 12))
    assert not lib.layer_fused_supported(plan, 20)                # W = 300 does not fit one lane tile
    plan = lib.get_plan(torch.device("cuda", 0), (34, 34), (12, 12))
    assert not lib.layer_fused_supported(plan, 40)                # width + bias column > 32
    a = torch.zeros(1, 5, 34, 34, device="cuda")
    with pytest.raises(lib.FnoError):
        lib.layer_inv_fused(plan, torch.zeros(1, 5, 24, 11, dtype=torch.complex64, device="cuda"), a,
                            torch.zeros(5, 5, 1, 1, device="cuda"), None)


@pytest.mark.parametrize("B,C,H,W,m1,m2", [(2, 3, 10, 9, 3, 4), (2, 3, 130, 130, 12, 12)])
def test_fwd_transform_gelu_grad_prologue(lib, B, C, H, W, m1, m2):
    """bwd_pre: transform of g * gelu'(s), storing dS."""
    rng = np.random.default_rng(12)
    g = rng.standard_normal((B, C, H, W)).astype(np.float32)
    s = (2.0 * rng.standard_normal((B, C, H, W))).astype(np.float32)
    plan = lib.get_plan(torch.device("cuda", 0), (H, W), (m1, m2))
    ds = torch.empty(B, C, H, W, device="cuda")
    gY = lib.fwd_transform(plan, dev(g), preact=dev(s), ds_out=ds, cmode=1, scale=1.0 / (H * W))
    ds_ref = g.astype(np.float64) * O.gelu_grad(s)
    assert O.rel_err(ds.cpu().numpy(), ds_ref) < TOL
    assert O.rel_err(gY.cpu().numpy(), O.fwd_transform(ds_ref, (m1, m2), cmode=1, scale=1.0 / (H * W))) < TOL


VOLUMES_3D = [
    # B, C, D1, D2, D3, m1, m2, m3
    (2, 2, 8, 6, 10, 3, 2, 4),
    (1, 3, 8, 8, 8, 4, 4, 5),     # touching corners on both full axes + Nyquist
    (1, 2, 12, 10, 14, 4, 3, 4),
    (1, 2, 64, 64, 70, 12, 12, 12),  # cfg 4 padded volume
]


@pytest.mark.parametrize("B,C,D1,D2,D3,m1,m2,m3", VOLUMES_3D)
def test_transforms_3d(lib, B, C, D1, D2, D3, m1, m2, m3):
    rng = np.random.default_rng(D1 + D2 + D3)
    x = rng.standard_normal((B, C, D1, D2, D3)).astype(np.float32)
    plan = lib.get_plan(torch.device("cuda", 0), (D1, D2, D3), (m1, m2, m3))
    X = lib.fwd_transform(plan, dev(x)).cpu().numpy()
    assert O.rel_err(X, O.fwd_transform(x, (m1, m2, m3))) < TOL
    n = D1 * D2 * D3
    Xs = lib.fwd_transform(plan, dev(x), cmode=1, scale=1.0 / n).cpu().numpy()
    assert O.rel_err(Xs, O.fwd_transform(x, (m1, m2, m3), cmode=1, scale=1.0 / n)) < TOL
    Y = cplx(rng, (B, C, 2 * m1, 2 * m2, m3))
    y = lib.inv_transform(plan, dev(Y), cmode=1).cpu().numpy()
    assert O.rel_err(y, O.inv_transform(Y, (D1, D2, D3), cmode=1)) < TOL
    y0 = lib.inv_transform(plan, dev(Y), cmode=0, scale=1.0).cpu().numpy()
    assert O.rel_err(y0, O.inv_transform(Y, (D1, D2, D3), cmode=0, scale=1.0)) < TOL


@pytest.mark.parametrize("B,Ci,Co,spatial,modes", [
    (2, 3, 4, (10, 9), (3, 4)),
    (5, 20, 20, (130, 130), (12, 12)),
    (3, 7, 5, (34, 34), (6, 9)),
    (2, 64, 64, (66, 66), (16, 16)),
    (2, 3, 2, (8, 6, 10), (3, 2, 4)),
    (1, 20, 20, (24, 24, 24), (12, 12, 12)),
    (9, 4, 6, (12, 10, 14), (4, 3, 4)),
])
def test_mix_fwd_bwd(lib, B, Ci, Co, spatial, modes):
    rng = np.random.default_rng(B * 100 + Ci)
    nd = len(spatial)
    plan = lib.get_plan(torch.device("cuda", 0), spatial, modes)
    ws = [cplx(rng, (Ci, Co) + tuple(modes), scale=0.5) for _ in range(2 if nd == 2 else 4)]
    X = cplx(rng, (B, Ci) + plan.spec_shape)
    gY = cplx(rng, (B, Co) + plan.spec_shape)
    wt = [dev(w) for w in ws]
    Y = lib.mix_fwd(plan, dev(X), wt).cpu().numpy()
    wcat = O.cat_corner_weights(ws)
    assert O.rel_err(Y, O.mix_fwd(X.astype(np.complex128), wcat)) < TOL
    gX, gws = lib.mix_bwd(plan, dev(X), dev(gY), wt)
    gx_ref, gw_ref = O.mix_bwd(X.astype(np.complex128), gY.astype(np.complex128), wcat)
    assert O.rel_err(gX.cpu().numpy(), gx_ref) < TOL
    for got, ref in zip(gws, O.split_corner_grads(gw_ref, len(ws))):
        assert O.rel_err(got.cpu().numpy(), ref) < TOL


# K2 on the tensor cores (mix_tc_kernel / mix_wgrad_tc_kernel): width 33..64 with an even innermost mode count.
# BASELINE configs[2] shape first; then ragged batches (one chunk of 32 partly filled, several chunks), channel counts
# that are not multiples of 8, Ci != Co, a 3-D spectrum, and shapes just outside the envelope (FP32 kernels).
@pytest.mark.parametrize("B,Ci,Co,spatial,modes,tc", [
    (32, 64, 64, (66, 66), (16, 16), True),        # cfg 3: m 16 x 16, width 64, per-GPU batch 32
    (5, 64, 64, (40, 40), (4, 6), True),           # partly filled batch chunk
    (70, 48, 64, (40, 40), (3, 4), True),          # three batch chunks (32 + 32 + 6), Ci != Co
    (33, 64, 40, (40, 40), (5, 2), True),
    (3, 37, 61, (24, 24), (2, 8), True),           # channel counts that are not multiples of 4 / 8
    (4, 64, 64, (12, 12, 14), (2, 3, 4), True),    # 3-D corners
    (3, 64, 64, (40, 40), (4, 5), False),          # odd innermost mode count -> FP32 kernel
    (3, 32, 32, (40, 40), (4, 4), False),          # width 32 -> FP32 kernel
])
def test_mix_tensor_core(lib, B, Ci, Co, spatial, modes, tc):
    rng = np.random.default_rng(B * 1000 + Ci * 7 + Co)
    nd = len(spatial)
    plan = lib.get_plan(torch.device("cuda", 0), spatial, modes)
    assert lib.mix_tc_supported(plan, Ci, Co) == tc
    ws = [cplx(rng, (Ci, Co) + tuple(modes), scale=0.5) for _ in range(2 if nd == 2 else 4)]
    X = cplx(rng, (B, Ci) + plan.spec_shape)
    gY = cplx(rng, (B, Co) + plan.spec_shape)
    wt = [dev(w) for w in ws]
    wcat = O.cat_corner_weights(ws)
    Y = lib.mix_fwd(plan, dev(X), wt).cpu().numpy()
    assert O.rel_err(Y, O.mix_fwd(X.astype(np.complex128), wcat)) < TOL
    gX, gws = lib.mix_bwd(plan, dev(X), dev(gY), wt)
    gx_ref, gw_ref = O.mix_bwd(X.astype(np.complex128), gY.astype(np.complex128), wcat)
    assert O.rel_err(gX.cpu().numpy(), gx_ref) < TOL
    for got, ref in zip(gws, O.split_corner_grads(gw_ref, len(ws))):
        assert O.rel_err(got.cpu().numpy(), ref) < TOL
    # per-mode errors too: a wrong mode pair / corner would hide behind a global max
    err = np.abs(Y - O.mix_fwd(X.astype(np.complex128), wcat)).reshape(B, Co, -1).max(axis=(0, 1))
    assert err.max() < 1e-5 * np.abs(Y).max()


@pytest.mark.parametrize("low,B,spatial", mode_params(
    ["cfg3"], [(2, (66, 66)),
               (3, (258, 258))]))             # cfg-3 plane: wgrad_tc_kernel<64, 64> with a ragged last slab
def test_pointwise_tensor_core_math_modes(lib, low, B, spatial):
    """The width-64 bypass kernels (pointwise_tc.cu: product, data gradient, weight gradient) follow the math mode."""
    rng = np.random.default_rng(3)
    C = 64
    a = rng.standard_normal((B, C) + spatial).astype(np.float32)
    w = rng.standard_normal((C, C, 1, 1)).astype(np.float32) / 8
    b = rng.standard_normal(C).astype(np.float32)
    ds = rng.standard_normal((B, C) + spatial).astype(np.float32)
    w2 = w.reshape(C, C).astype(np.float64)
    a2, ds2 = a.reshape(B, C, -1).astype(np.float64), ds.reshape(B, C, -1).astype(np.float64)
    refs = {"out": O.pointwise_conv(a, w, b), "d a": np.einsum("oi,bo...->bi...", w2, ds.astype(np.float64)),
            "d W": np.einsum("bop,bip->oi", ds2, a2)}
    da, dsd, wd, bd = dev(a), dev(ds), dev(w), dev(b)

    def errors():
        got = {"out": lib.pointwise_fwd(da, wd, bd), "d a": lib.pointwise_fwd(dsd, wd, None, transpose=True),
               "d W": lib.pointwise_wgrad(dsd, da, w.shape)[0]}
        return {k: O.rel_err(t.cpu().numpy().reshape(refs[k].shape), refs[k]) for k, t in got.items()}

    check_mode_errors(run_modes(lib, low, errors), low, f"bypass {spatial}")


MIX_MODE_CASES = [
    # B, C, spatial, modes
    (16, 64, (34, 34), (8, 8)),
    (4, 64, (16, 16, 18), (4, 4, 6)),       # 3-D: four corners, three spatial modes
    (32, 64, (66, 66), (16, 16)),           # cfg 3 (per-GPU batch 32)
]


@pytest.mark.parametrize("low,B,C,spatial,modes", mode_params(["3d", "cfg3"], MIX_MODE_CASES))
def test_mix_tensor_core_math_modes(lib, low, B, C, spatial, modes):
    """tf32 / bf16 modes reach K2's tensor-core kernels: single pass, stated bounds 2e-3 / 2e-2, visibly worse than fp32."""
    rng = np.random.default_rng(5)
    plan = lib.get_plan(torch.device("cuda", 0), spatial, modes)
    assert lib.mix_tc_supported(plan, C, C)
    ws = [cplx(rng, (C, C) + modes, scale=0.5) for _ in range(2 if len(spatial) == 2 else 4)]
    X, gY = cplx(rng, (B, C) + plan.spec_shape), cplx(rng, (B, C) + plan.spec_shape)
    wcat = O.cat_corner_weights(ws)
    y_ref = O.mix_fwd(X.astype(np.complex128), wcat)
    gx_ref, gw_ref = O.mix_bwd(X.astype(np.complex128), gY.astype(np.complex128), wcat)
    gw_refs = O.split_corner_grads(gw_ref, len(ws))
    Xd, gYd, wsd = dev(X), dev(gY), [dev(w) for w in ws]

    def errors():
        Y = lib.mix_fwd(plan, Xd, wsd)
        gX, gws = lib.mix_bwd(plan, Xd, gYd, wsd)
        e = {"Y": O.rel_err(Y.cpu().numpy(), y_ref), "d X": O.rel_err(gX.cpu().numpy(), gx_ref)}
        e.update({f"d W{k}": O.rel_err(g.cpu().numpy(), r) for k, (g, r) in enumerate(zip(gws, gw_refs))})
        return e

    check_mode_errors(run_modes(lib, low, errors), low, f"K2 {spatial} m {modes}")


@pytest.mark.parametrize("B,Co,Ci,spatial", [
    (2, 20, 20, (130, 130)),
    (3, 8, 8, (13, 11)),         # N not a multiple of 4 -> scalar path
    (2, 6, 10, (16, 16)),        # Co != Ci
    (1, 64, 64, (66, 66)),
    (3, 64, 64, (258, 258)),     # cfg-3 planes: tcgen05 weight gradient (wgrad_tc_kernel<64, 64>), ragged last slab
    (2, 48, 33, (30, 34)),       # wide, Co != Ci, channel counts that are not multiples of 8
    (2, 24, 24, (20, 20)),       # FP32 wide-channel weight gradient (one CTA owns the whole output)
    (2, 20, 20, (16, 16, 22)),
    (1, 5, 3, (9, 7)),           # channel counts that are not tile multiples
])
def test_pointwise_fwd_transpose_wgrad(lib, B, Co, Ci, spatial):
    rng = np.random.default_rng(Co * 10 + Ci)
    a = rng.standard_normal((B, Ci) + spatial).astype(np.float32)
    w = rng.standard_normal((Co, Ci) + (1,) * len(spatial)).astype(np.float32)
    b = rng.standard_normal(Co).astype(np.float32)
    ds = rng.standard_normal((B, Co) + spatial).astype(np.float32)
    out = lib.pointwise_fwd(dev(a), dev(w), dev(b)).cpu().numpy()
    assert O.rel_err(out, O.pointwise_conv(a, w, b)) < TOL
    w2 = w.reshape(Co, Ci).astype(np.float64)
    back = lib.pointwise_fwd(dev(ds), dev(w), None, transpose=True).cpu().numpy()
    assert O.rel_err(back, np.einsum("oi,bo...->bi...", w2, ds.astype(np.float64))) < TOL
    gw, gb = lib.pointwise_wgrad(dev(ds), dev(a), w.shape)
    ds2 = ds.reshape(B, Co, -1).astype(np.float64)
    a2 = a.reshape(B, Ci, -1).astype(np.float64)
    assert O.rel_err(gw.cpu().numpy().reshape(Co, Ci), np.einsum("bop,bip->oi", ds2, a2)) < TOL
    assert O.rel_err(gb.cpu().numpy(), ds2.sum(axis=(0, 2))) < TOL
    # fused autograd (fno_pointwise_bwd): data, weight and bias gradient in one pass over ds when eligible
    dx, gw3, gb3 = lib.pointwise_bwd(dev(ds), dev(a), dev(w))
    assert O.rel_err(dx.cpu().numpy(), np.einsum("oi,bo...->bi...", w2, ds.astype(np.float64))) < TOL
    assert O.rel_err(gw3.cpu().numpy().reshape(Co, Ci), np.einsum("bop,bip->oi", ds2, a2)) < TOL
    assert O.rel_err(gb3.cpu().numpy(), ds2.sum(axis=(0, 2))) < TOL


def test_transform_properties_full_size(lib):
    """Size-independent properties at the BASELINE cfg-1 plane size and a bench-sized batch:
    linearity, adjointness <K1 x, Y> = <x, K1^H Y>, and exact recovery of a band-limited field."""
    B, C, H, W, m = 16, 20, 130, 130, 12
    plan = lib.get_plan(torch.device("cuda", 0), (H, W), (m, m))
    g = torch.Generator(device="cuda").manual_seed(0)
    x1 = torch.randn(B, C, H, W, device="cuda", generator=g)
    x2 = torch.randn(B, C, H, W, device="cuda", generator=g)
    X1, X2 = lib.fwd_transform(plan, x1), lib.fwd_transform(plan, x2)
    X12 = lib.fwd_transform(plan, 0.5 * x1 - 2.0 * x2)
    lin = (X12 - (0.5 * X1 - 2.0 * X2)).abs().max() / X12.abs().max()
    assert lin.item() < TOL
    Y = torch.randn(B, C, 2 * m, m, device="cuda", generator=g, dtype=torch.float32).to(torch.complex64)
    Y = Y + 1j * torch.randn(B, C, 2 * m, m, device="cuda", generator=g)
    lhs = (X1.to(torch.complex128) * Y.conj().to(torch.complex128)).real.sum()
    rhs = (x1.double() * lib.inv_transform(plan, Y, cmode=0, scale=1.0).double()).sum()
    assert abs(lhs.item() - rhs.item()) < 1e-5 * abs(lhs.item())
    # A real field made only of retained modes is a fixed point of inverse(forward(.)).  The one
    # retained mode whose Hermitian partner is NOT retained is (k1 = -m1, k2 = 0) (row m1 of the
    # kept spectrum; +m1 is outside the low block), so it is zeroed before building the field.
    Y[:, :, m, 0] = 0
    band = lib.inv_transform(plan, Y, cmode=1)
    again = lib.inv_transform(plan, lib.fwd_transform(plan, band), cmode=1)
    assert ((again - band).abs().max() / band.abs().max()).item() < TOL


def test_golden_spectral_kernels(lib, golden_spectral):
    """The reference's own outputs (tests/golden/spectral_small.npz) through the raw kernels."""
    from oracle.make_golden import SC2D_CASES

    g = golden_spectral
    for ci, (B, Ci, Co, H, W, m1, m2) in enumerate(SC2D_CASES):
        pre = f"sc2d_{ci}_"
        plan = lib.get_plan(torch.device("cuda", 0), (H, W), (m1, m2))
        ws = [dev(g[pre + "w1"]), dev(g[pre + "w2"])]
        X = lib.fwd_transform(plan, dev(g[pre + "x"]))
        y = lib.inv_transform(plan, lib.mix_fwd(plan, X, ws), cmode=1)
        assert O.rel_err(y.cpu().numpy(), g[pre + "y"]) < TOL


def test_errors_are_loud(lib):
    with pytest.raises(lib.FnoError):
        lib.get_plan(torch.device("cuda", 0), (8, 8), (5, 3))       # 2*m1 > H
    with pytest.raises(lib.FnoError):
        lib.get_plan(torch.device("cuda", 0), (8, 8), (2, 6))       # m2 > W/2+1
    with pytest.raises(lib.FnoError):
        lib.get_plan(torch.device("cpu"), (8, 8), (2, 2))
    plan = lib.get_plan(torch.device("cuda", 0), (8, 8), (2, 2))
    with pytest.raises(lib.FnoError):
        lib.fwd_transform(plan, torch.zeros(1, 1, 8, 8))            # CPU tensor
    with pytest.raises(lib.FnoError):
        lib.fwd_transform(plan, torch.zeros(1, 1, 8, 9, device="cuda"))
    with pytest.raises(lib.FnoError):
        lib.fwd_transform(plan, torch.zeros(1, 1, 8, 8, device="cuda", dtype=torch.float64))


# ---------------------------------------------------------------------------------------------
# lift (statistics + normalise + fc0 + pad) and projection head (fc1 + GELU + fc2 + de-normalise)
# checked against the fp64 oracle port (oracle/fno_port.py: _normalise / _lift / _project)
# ---------------------------------------------------------------------------------------------
LIFT_CASES = [
    # spatial, T, V, C          (2-D: pad 2 on both axes; 3-D: pad 6 on the last axis)
    ((9, 7), 3, 2, 8),
    ((16, 16), 10, 2, 20),
    ((5, 66), 2, 3, 6),          # W_in > one 64-pixel tile, width not a multiple of 4
    ((4, 5, 6), 2, 3, 6),
    ((6, 6, 10), 3, 5, 20),      # V = 5 (cfg 4 channel count)
    ((12, 10), 2, 1, 32),
    # T * V % 4 == 0: the register-tiled backward (lift_bwd2_kernel)
    ((8, 128), 10, 2, 20),       # cfg-1 row: two full 64-pixel tiles per row
    ((13, 70), 4, 2, 20),        # ragged second tile (6 valid pixels)
    ((4, 4, 64), 4, 3, 12),      # 3-D: three grid features, 12 channels
    ((20, 40), 2, 2, 40),        # two items per lane
    ((10, 10), 8, 4, 64),        # output tile too large for the register-tiled form: first form
]


def _lift_inputs(spatial, T, V, C, seed):
    g = torch.Generator().manual_seed(seed)
    B, nd = 3, len(spatial)
    x = torch.randn((B,) + spatial + (T, V), generator=g) * torch.tensor([0.5, 3.0, 0.01, 1.0, 2.0][:V]) \
        + torch.tensor([10.0, -2.0, 1.0, 0.0, 100.0][:V])       # |mean| >> std in some variables
    grid = torch.rand((B,) + spatial + (nd,), generator=g)
    W0 = torch.randn(C, T * V + nd, generator=g) / 4
    b0 = torch.randn(C, generator=g)
    return x, grid, W0, b0


@pytest.mark.parametrize("spatial,T,V,C", LIFT_CASES)
def test_lift_stats(lib, spatial, T, V, C):
    x, _, _, _ = _lift_inputs(spatial, T, V, C, 1)
    nd = len(spatial)
    stats = lib.lift_stats(x.cuda()).cpu().double()
    std, mean = torch.std_mean(x.double(), dim=tuple(range(1, nd + 2)))
    assert float((stats[:, 0] - mean).abs().max() / mean.abs().max()) < 1e-6
    assert float(((stats[:, 1] - (std + 1e-7)) / std).abs().max()) < 1e-5


@pytest.mark.parametrize("spatial,T,V,C", LIFT_CASES)
def test_lift_forward_backward(lib, spatial, T, V, C):
    from fno_b200 import ops
    from oracle import fno_port as P

    x, grid, W0, b0 = _lift_inputs(spatial, T, V, C, 2)
    nd = len(spatial)
    pad = 2 if nd == 2 else 6
    # oracle, fp64 autograd
    p = {"fc0.weight": W0.double().requires_grad_(), "fc0.bias": b0.double().requires_grad_()}
    xn, _, _ = P._normalise(x.double(), nd)
    h_ref = P._lift(p, xn, grid.double(), nd)
    gh = torch.randn(h_ref.shape, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    h_ref.backward(gh)
    # CUDA
    W0c, b0c = W0.cuda().requires_grad_(), b0.cuda().requires_grad_()
    h, stats, geo = ops.lift(x.cuda(), grid.cuda(), W0c, b0c, pad)
    assert tuple(h.shape) == tuple(h_ref.shape)
    assert O.rel_err(h.detach().cpu().numpy(), h_ref.detach().numpy()) < TOL
    h.backward(gh.float().cuda())
    assert O.rel_err(W0c.grad.cpu().numpy(), p["fc0.weight"].grad.numpy()) < TOL
    assert O.rel_err(b0c.grad.cpu().numpy(), p["fc0.bias"].grad.numpy()) < TOL


HEAD_CASES = [
    # spatial, C, V, B
    ((9, 7), 8, 2, 2),
    ((16, 16), 20, 2, 3),
    ((5, 66), 6, 3, 2),
    ((3, 130), 20, 1, 1),
    ((4, 5, 6), 6, 3, 2),
    ((6, 6, 10), 20, 5, 2),
    ((12, 10), 32, 4, 2),
    ((8, 8), 64, 3, 1),
    ((64, 64), 20, 2, 5),       # 320 64-pixel tiles: several pipelined tiles per persistent CTA (tensor-core backward)
    ((40, 50), 23, 4, 3),       # widest tensor-core case (C + bias column = 24), ragged last tile, V = 4
    ((128, 128), 20, 2, 2),     # cfg-1 plane
    ((16, 16, 22), 20, 5, 2),   # cfg-4 shape class: 5 variables (tensor-core heads with 8-wide variable rows), many tiles
    ((30, 34), 12, 8, 2),       # V = 8: the widest tensor-core case
    ((20, 20), 8, 7, 1),
    # wide trunks (24 <= C <= 64): head_bwd_wide_kernel + wgrad_tc_kernel<128, 32> when the padded plane is a multiple of 4
    ((256, 256), 64, 3, 1),     # cfg-3 plane: 521 position tiles per sample, 2081 pixel slabs
    ((40, 50), 48, 2, 3),       # C not a multiple of 16, several samples, ragged last tile
    ((30, 33), 24, 4, 2),       # narrowest wide case, V = 4
    ((6, 6, 10), 40, 3, 2),     # 3-D trunk layout (rows = X * Y, last axis padded by 6)
    ((9, 11), 64, 3, 2),        # padded plane 11 x 13: not a multiple of 4 -> FP32 kernels
]


@pytest.mark.parametrize("bwd_tc", [True, False], ids=["tcgen05", "fp32"])
@pytest.mark.parametrize("spatial,C,V,B", HEAD_CASES)
def test_head_forward_backward(lib, monkeypatch, spatial, C, V, B, bwd_tc):
    monkeypatch.setattr(lib, "HEAD_BWD_TC", bwd_tc)
    nd = len(spatial)
    pad = 2 if nd == 2 else 6
    geo = lib.TrunkGeo(spatial, pad)
    wide = bool(lib.load().fno_head_bwd_wide_supported(geo.R_out, geo.Wp, C, 128, V))
    assert wide == (24 <= C <= 64 and V <= 4 and (geo.R_out * geo.Wp) % 4 == 0)
    if bwd_tc and (C > 23 or V > 8) and not wide:
        pytest.skip("outside the tensor-core backward's envelopes (FP32 path covers it)")
    from fno_b200 import ops
    from oracle import fno_port as P

    g = torch.Generator().manual_seed(5)
    h = torch.randn((B, C) + geo.padded, generator=g) * 1.5
    W1 = torch.randn(128, C, generator=g) / C ** 0.5
    b1 = torch.randn(128, generator=g) * 0.3
    W2 = torch.randn(V, 128, generator=g) / 11
    b2 = torch.randn(V, generator=g)
    mean = torch.randn(B, V, generator=g)
    std = torch.rand(B, V, generator=g) + 0.5
    stats = torch.stack((mean, std), dim=1).contiguous()
    # oracle, fp64 autograd
    p = {"fc1.weight": W1.double().requires_grad_(), "fc1.bias": b1.double().requires_grad_(),
         "fc2.weight": W2.double().requires_grad_(), "fc2.bias": b2.double().requires_grad_()}
    h64 = h.double().requires_grad_()
    bshape = (B,) + (1,) * nd + (V,)
    out_ref = P._project(p, h64, nd, "fc2") * std.double().view(bshape) + mean.double().view(bshape)
    gout = torch.randn(out_ref.shape, generator=g, dtype=torch.float64)
    out_ref.backward(gout)
    # CUDA
    hc = h.cuda().requires_grad_()
    leaves = [t.cuda().requires_grad_() for t in (W1, b1, W2, b2)]
    out = ops.head(hc, *leaves, stats.cuda(), geo)
    assert tuple(out.shape) == tuple(out_ref.shape)
    assert O.rel_err(out.detach().cpu().numpy(), out_ref.detach().numpy()) < TOL
    out.backward(gout.float().cuda())
    assert O.rel_err(hc.grad.cpu().numpy(), h64.grad.numpy()) < TOL
    # the padding of dh must be exactly zero (F.pad backward drops it; layer 3 reads all of dh)
    pad_mask = torch.ones_like(h, dtype=torch.bool)
    pad_mask[(Ellipsis,) + tuple(slice(0, s) for s in (spatial if nd == 2 else (spatial[0], spatial[1], spatial[2])))] = False
    assert float(hc.grad.cpu()[pad_mask].abs().max()) == 0.0
    for t, name in zip(leaves, ("fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias")):
        assert O.rel_err(t.grad.cpu().numpy(), p[name].grad.numpy()) < TOL, name


# ---------------------------------------------------------------------------------------------
# tensor-core W-axis stage of K1 (transform2d_tc.cu, tcgen05 kind::tf32 with 3xTF32 split) + FP32
# H-axis fold: opt-in (lib.K1_TENSOR_CORES); taken when planes * H >= 4096 rows, W even and <= 136, 2 * m2 <= 32
# ---------------------------------------------------------------------------------------------
TC_PLANES = [
    # B, C, H, W, m1, m2
    (4, 20, 130, 130, 12, 12),      # cfg 1 plane; 80 planes = 81.25 row tiles (ragged last tile)
    (3, 16, 96, 70, 12, 12),        # a 3-D slice width (W = 70: 18 chunks, last chunk half valid)
    (2, 24, 100, 136, 16, 16),      # widest supported row, 2 * m2 = 32 accumulator columns
    (5, 9, 129, 66, 5, 7),          # odd H, modes below the padded template sizes
]


@pytest.mark.parametrize("B,C,H,W,m1,m2", TC_PLANES)
@pytest.mark.parametrize("cmode", [0, 1])
def test_fwd_transform_tensor_core_path(lib, monkeypatch, B, C, H, W, m1, m2, cmode):
    monkeypatch.setattr(lib, "K1_TENSOR_CORES", True)
    rng = np.random.default_rng(H * 7 + W)
    x = (rng.standard_normal((B, C, H, W)) * 3 + 0.5).astype(np.float32)
    scale = 1.0 if cmode == 0 else 1.0 / (H * W)
    plan = lib.get_plan(torch.device("cuda", 0), (H, W), (m1, m2))
    assert lib.load().fno_sc2d_fwd_workspace_bytes(plan.handle, B * C) == 4 * B * C * H * ((2 * m2 + 3) // 4 * 4)
    X = lib.fwd_transform(plan, dev(x), cmode=cmode, scale=scale).cpu().numpy()
    ref = O.fwd_transform(x, (m1, m2), cmode=cmode, scale=scale)
    assert O.rel_err(X, ref) < TOL


@pytest.mark.parametrize("B,C,H,W,m1,m2", TC_PLANES[:2])
def test_fwd_transform_tensor_core_path_with_gelu_grad(lib, monkeypatch, B, C, H, W, m1, m2):
    monkeypatch.setattr(lib, "K1_TENSOR_CORES", True)
    rng = np.random.default_rng(99)
    g = rng.standard_normal((B, C, H, W)).astype(np.float32)
    s = (rng.standard_normal((B, C, H, W)) * 1.5).astype(np.float32)
    plan = lib.get_plan(torch.device("cuda", 0), (H, W), (m1, m2))
    ds = torch.empty(B, C, H, W, device="cuda")
    X = lib.fwd_transform(plan, dev(g), preact=dev(s), ds_out=ds, cmode=1, scale=1.0 / (H * W)).cpu().numpy()
    ds_ref = g.astype(np.float64) * O.gelu_grad(s.astype(np.float64))
    assert O.rel_err(ds.cpu().numpy(), ds_ref) < TOL
    ref = O.fwd_transform(ds_ref, (m1, m2), cmode=1, scale=1.0 / (H * W))
    assert O.rel_err(X, ref) < TOL


# ---------------------------------------------------------------------------------------------
# tf32 math mode (north_star: "a separately stated bound for tf32/bf16 modes"): the projection head's
# tcgen05 kernels run a single kind::tf32 pass instead of the 3xTF32 split.  Stated bound: <= 2e-3
# relative (max |err| / max |ref|) on outputs and gradients; fp32 mode stays <= 1e-5.
# ---------------------------------------------------------------------------------------------
TF32_TOL = 2e-3
# bf16 math mode: every MMA operand rounded to bfloat16 (8-bit significand), one pass, fp32 accumulation.  Stated bound
# <= 2e-2 relative (max-norm); measured 2e-3 .. 6e-3.
BF16_TOL = 2e-2
MODE_TOL = {"tf32": TF32_TOL, "bf16": BF16_TOL}


@pytest.mark.parametrize("low", ["tf32", "bf16"])
@pytest.mark.parametrize("spatial,C,V,B", [((64, 64), 20, 2, 3), ((40, 50), 23, 4, 2),
                                           ((62, 62), 64, 3, 2),         # wide trunk: head_wide_tc.cu kernels
                                           ((64, 64, 64), 20, 5, 1),     # cfg-4 head: 3-D trunk, V = 5
                                           ((16, 16, 22), 40, 3, 2)])    # 3-D wide trunk: + wgrad_tc_kernel<128, 32>
def test_head_tf32_mode(lib, spatial, C, V, B, low):
    from fno_b200 import ops
    from oracle import fno_port as P

    g = torch.Generator().manual_seed(11)
    nd = len(spatial)
    geo = lib.TrunkGeo(spatial, 2 if nd == 2 else 6)
    narrow = C <= 23
    wide = bool(lib.load().fno_head_bwd_wide_supported(geo.R_out, geo.Wp, C, 128, V))
    assert narrow != wide                                   # a tensor-core backward either way
    h = torch.randn((B, C) + geo.padded, generator=g) * 1.5
    W1 = torch.randn(128, C, generator=g) / C ** 0.5
    b1 = torch.randn(128, generator=g) * 0.3
    W2 = torch.randn(V, 128, generator=g) / 11
    b2 = torch.randn(V, generator=g)
    mean = torch.randn(B, V, generator=g)
    std = torch.rand(B, V, generator=g) + 0.5
    stats = torch.stack((mean, std), dim=1).contiguous()
    p = {"fc1.weight": W1.double().requires_grad_(), "fc1.bias": b1.double().requires_grad_(),
         "fc2.weight": W2.double().requires_grad_(), "fc2.bias": b2.double().requires_grad_()}
    h64 = h.double().requires_grad_()
    bshape = (B,) + (1,) * nd + (V,)
    out_ref = P._project(p, h64, nd, "fc2") * std.double().view(bshape) + mean.double().view(bshape)
    gout = torch.randn(out_ref.shape, generator=g, dtype=torch.float64)
    out_ref.backward(gout)
    names = ("fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias")

    def errors():
        hc = h.cuda().requires_grad_()
        leaves = [t.cuda().requires_grad_() for t in (W1, b1, W2, b2)]
        out = ops.head(hc, *leaves, stats.cuda(), geo)
        out.backward(gout.float().cuda())
        e = {"out": O.rel_err(out.detach().cpu().numpy(), out_ref.detach().numpy()),
             "dh": O.rel_err(hc.grad.cpu().numpy(), h64.grad.numpy())}
        e.update({n: O.rel_err(t.grad.cpu().numpy(), p[n].grad.numpy()) for t, n in zip(leaves, names)})
        return e

    # fc2.bias's gradient is a plain sum of the output gradient: no MMA, the same in every mode
    check_mode_errors(run_modes(lib, low, errors), low, f"head {spatial} C {C} V {V}",
                      shows_mode=("out", "dh", "fc1.weight", "fc1.bias", "fc2.weight"))


# ---------------------------------------------------------------------------------------------
# device-resident windowed dataset (SURVEY 8f row f4): bit-exact against the host-side windows
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("spatial,T,V,T0,R", [((16, 16), 15, 2, 10, 1), ((12, 10), 9, 3, 4, 2), ((6, 5, 4), 8, 5, 3, 1)])
def test_device_windows_match_host_windows(lib, spatial, T, V, T0, R):
    from fno_b200 import data

    g = torch.Generator().manual_seed(3)
    traj = torch.randn((5, T) + spatial + (V,), generator=g)
    xx_ref, yy_ref = data.windows(traj, T0, R)                      # item order: trajectory-major, window-minor
    ds = data.DeviceWindows(traj, T0, R, device="cuda")
    assert len(ds) == xx_ref.shape[0]
    items = torch.randperm(len(ds), generator=g)[:17]
    xx, yy, grid = ds.batch(items)
    assert torch.equal(xx.cpu(), xx_ref[items]) and torch.equal(yy.cpu(), yy_ref[items])
    assert tuple(grid.shape) == (17,) + spatial + (len(spatial),)
    # one epoch over two ranks covers every item exactly once
    seen = torch.cat([torch.cat(data.epoch_indices(len(ds), 8, True, 16, 0, r, 2)) for r in range(2)])
    assert sorted(seen.tolist()) == list(range(len(ds)))


@pytest.mark.parametrize("low,B,C,spatial,modes", mode_params(
    ["cfg4"], [(4, 20, (130, 130), (12, 12)),
               (4, 20, (64, 64, 70), (12, 12, 12))]))   # cfg-4 volume: K1's tensor-core stage on the inner planes
def test_fwd_transform_tf32_mode(lib, monkeypatch, low, B, C, spatial, modes):
    """tf32 / bf16 math modes on the K1 tensor-core kernels (plain and GELU'-premultiply forms): single pass, stated
    bound <= 2e-3 (tf32) / 2e-2 (bf16) relative; fp32 mode (3xTF32) <= 1e-5 on the same inputs."""
    monkeypatch.setattr(lib, "K1_TENSOR_CORES", True)
    rng = np.random.default_rng(5)
    shape = (B, C) + spatial
    g = rng.standard_normal(shape).astype(np.float32)
    s_ = (rng.standard_normal(shape) * 1.5).astype(np.float32)
    plan = lib.get_plan(torch.device("cuda", 0), spatial, modes)
    L = lib.load()
    if len(spatial) == 2:
        assert L.fno_sc2d_fwd_workspace_bytes(plan.handle, B * C) > 0
    else:       # the 3-D workspace carries the W-axis GEMM's scratch only when the inner planes take the tensor cores
        inner = B * C * spatial[0]
        assert inner * spatial[1] >= 4096 and L.fno_sc2d_fwd_workspace_bytes(plan.handle, inner) > 0
        spectra = (8 * B * C * spatial[0] * 2 * modes[1] * modes[2] + 255) // 256 * 256
        assert L.fno_plan_workspace_bytes(plan.handle, B * C) == spectra + L.fno_sc2d_fwd_workspace_bytes(plan.handle, inner)
    npix = int(np.prod(spatial))
    ref_plain = O.fwd_transform(g, modes, cmode=0, scale=1.0)
    ds_ref = g.astype(np.float64) * O.gelu_grad(s_.astype(np.float64))
    ref_pre = O.fwd_transform(ds_ref, modes, cmode=1, scale=1.0 / npix)
    gd, sd = dev(g), dev(s_)

    def errors():
        X = lib.fwd_transform(plan, gd, cmode=0, scale=1.0)
        ds = torch.empty_like(gd)
        Xp = lib.fwd_transform(plan, gd, preact=sd, ds_out=ds, cmode=1, scale=1.0 / npix)
        return {"plain": O.rel_err(X.cpu().numpy(), ref_plain), "premultiply": O.rel_err(Xp.cpu().numpy(), ref_pre),
                "dS": O.rel_err(ds.cpu().numpy(), ds_ref)}

    errs = run_modes(lib, low, errors)
    assert max(e["dS"] for e in errs.values()) <= TOL, errs          # dS itself is computed in fp32 in every mode
    check_mode_errors(errs, low, f"K1 {spatial}", shows_mode=("plain", "premultiply"))


LAYER_MODE_CASES = [
    # B, C, n, m
    (2, 20, 66, 12),
    (2, 20, 130, 12),     # cfg-1 plane: 128 lanes + 2 edge columns, K1 on the tensor cores
    (2, 31, 66, 12),      # widest fused layer (31 channels + the bias column)
]


@pytest.mark.parametrize("low,B,C,n,m", mode_params(["cfg1", "width31"], LAYER_MODE_CASES))
def test_fourier_layer_reduced_precision_modes(lib, low, B, C, n, m):
    """One whole Fourier layer (K1 -> K2 -> fused tcgen05 K3 + bypass + GELU, forward and backward) in tf32 / bf16 mode
    against the fp64 oracle: stated bounds 2e-3 / 2e-2; fp32 mode <= 1e-5 on the same inputs."""
    from fno_b200 import ops

    assert lib.layer_fused_supported(lib.get_plan(torch.device("cuda", 0), (n, n), (m, m)), C)
    rng = np.random.default_rng(21)
    a = rng.standard_normal((B, C, n, n)).astype(np.float32)
    wl = (rng.standard_normal((C, C, 1, 1)) / C ** 0.5).astype(np.float32)
    bl = rng.standard_normal(C).astype(np.float32)
    ws = [((rng.random((C, C, m, m)) + 1j * rng.random((C, C, m, m))) / C).astype(np.complex64) for _ in range(2)]
    g = rng.standard_normal((B, C, n, n)).astype(np.float32)
    ref, _ = O.fourier_layer_forward(a, ws, wl, bl, True)
    ga, gws, gwl, gbl = O.fourier_layer_backward(a, ws, wl, bl, True, g)

    def errors():
        ad = dev(a).requires_grad_()
        wld, bld = dev(wl).requires_grad_(), dev(bl).requires_grad_()
        wsd = [dev(w).requires_grad_() for w in ws]
        out = ops.fourier_layer(ad, wld, bld, True, wsd)
        out.backward(dev(g))
        got = {"out": (out.detach(), ref), "d a": (ad.grad, ga), "d W0": (wsd[0].grad, gws[0]),
               "d W1": (wsd[1].grad, gws[1]), "d Wl": (wld.grad, gwl), "d bias": (bld.grad, gbl)}
        return {k: O.rel_err(t.cpu().numpy().reshape(np.shape(r)), r) for k, (t, r) in got.items()}

    check_mode_errors(run_modes(lib, low, errors), low, f"Fourier layer B {B} C {C} n {n} m {m}")


def _k1_fp32_form(lib, rng, B, C, H, W):
    plan = lib.get_plan(torch.device("cuda", 0), (H, W), (12, 12))
    g, s = dev(rng.standard_normal((B, C, H, W)).astype(np.float32)), dev(rng.standard_normal((B, C, H, W)).astype(np.float32))

    def run():
        ds = torch.empty_like(g)
        return lib.fwd_transform(plan, g), lib.fwd_transform(plan, g, preact=s, ds_out=ds, cmode=1, scale=0.1), ds
    return run


def _k2_fp32_form(lib, rng, B, C, spatial, modes):
    plan = lib.get_plan(torch.device("cuda", 0), spatial, modes)
    assert not lib.mix_tc_supported(plan, C, C)
    ws = [dev(cplx(rng, (C, C) + modes)) for _ in range(2)]
    X, gY = dev(cplx(rng, (B, C) + plan.spec_shape)), dev(cplx(rng, (B, C) + plan.spec_shape))

    def run():
        gX, gws = lib.mix_bwd(plan, X, gY, ws)
        return [lib.mix_fwd(plan, X, ws), gX] + gws
    return run


def _bypass_fp32_form(lib, rng, B, C, spatial):
    a, ds = (dev(rng.standard_normal((B, C) + spatial).astype(np.float32)) for _ in range(2))
    w, b = dev(rng.standard_normal((C, C, 1, 1)).astype(np.float32)), dev(rng.standard_normal(C).astype(np.float32))
    return lambda: (lib.pointwise_fwd(a, w, b), lib.pointwise_fwd(ds, w, None, transpose=True),
                    *lib.pointwise_wgrad(ds, a, w.shape), *lib.pointwise_bwd(ds, a, w))


def _head_fp32_form(lib, rng, spatial, C, V, B, fwd):
    geo = lib.TrunkGeo(spatial, 2 if len(spatial) == 2 else 6)
    h = dev(rng.standard_normal((B, C) + geo.padded).astype(np.float32))
    W1, b1 = dev(rng.standard_normal((128, C)).astype(np.float32) / C ** 0.5), dev(rng.standard_normal(128).astype(np.float32))
    W2, b2 = dev(rng.standard_normal((V, 128)).astype(np.float32) / 11), dev(rng.standard_normal(V).astype(np.float32))
    stats = dev(np.stack((rng.standard_normal((B, V)), rng.random((B, V)) + 0.5), axis=1).astype(np.float32))
    dout = dev(rng.standard_normal((B,) + geo.spatial + (V,)).astype(np.float32))
    return lambda: ((lib.head_fwd(geo, h, W1, b1, W2, b2, stats),) if fwd else ()) + \
        lib.head_bwd(geo, h, dout, W1, b1, W2, stats)


def _inv_epilogue_form(lib, rng, B, C, H, W):
    plan = lib.get_plan(torch.device("cuda", 0), (H, W), (12, 12))
    Y, add = dev(cplx(rng, (B, C, 24, 12))), dev(rng.standard_normal((B, C, H, W)).astype(np.float32))

    def run():
        s_out = torch.empty_like(add)
        return lib.inv_transform(plan, Y, addend=add, s_out=s_out, apply_gelu=True), s_out
    return run


FP32_FORMS = {
    "k1_below_envelope": lambda lib, rng: _k1_fp32_form(lib, rng, 1, 20, 130, 130),     # planes * H = 2600 < 4096
    "k1_odd_w": lambda lib, rng: _k1_fp32_form(lib, rng, 2, 20, 130, 129),
    "k2_width20": lambda lib, rng: _k2_fp32_form(lib, rng, 4, 20, (34, 34), (12, 12)),
    "k2_odd_modes": lambda lib, rng: _k2_fp32_form(lib, rng, 3, 64, (40, 40), (4, 5)),
    "bypass_width20": lambda lib, rng: _bypass_fp32_form(lib, rng, 2, 20, (130, 130)),
    "head_bwd_fp32": lambda lib, rng: _head_fp32_form(lib, rng, (64, 64), 20, 2, 2, fwd=False),
    "head_outside_envelopes": lambda lib, rng: _head_fp32_form(lib, rng, (12, 10), 40, 5, 2, fwd=True),
    "inv_fused_epilogue": lambda lib, rng: _inv_epilogue_form(lib, rng, 2, 20, 130, 130),
}


@pytest.mark.parametrize("form", list(FP32_FORMS))
def test_fp32_forms_ignore_math_mode(lib, monkeypatch, form):
    """Kernels that run in FP32 -- shapes outside a tensor-core envelope, or files that have no tensor-core form -- give
    bitwise the same results in all three math modes: only a tensor-core launch may read the mode."""
    monkeypatch.setattr(lib, "K1_TENSOR_CORES", True)
    monkeypatch.setattr(lib, "HEAD_BWD_TC", form != "head_bwd_fp32")
    run = FP32_FORMS[form](lib, np.random.default_rng(31))
    results = {}
    for mode in ("fp32", "tf32", "bf16"):
        lib.set_math_mode(mode)
        results[mode] = [t.clone() for t in run() if t is not None]
        torch.cuda.synchronize()
    for mode in ("tf32", "bf16"):
        for k, (a, b) in enumerate(zip(results["fp32"], results[mode])):
            assert torch.equal(a, b), (mode, k)


def test_new_entry_points_reject_bad_arguments(lib):
    """C-ABI error behaviour of the entry points added for the tensor-core / dataset paths: a negative code and a
    message, never a silent fallback."""
    L = lib.load()
    z = torch.zeros(1 << 16, device="cuda")
    p = z.data_ptr()
    st = 0
    # tcgen05 head backward: hidden width must be 128, C + bias column <= 24, V <= 4
    assert L.fno_head_bwd_tc(p, p, p, p, p, p, p, p, p, p, p, p, 1, 8, 8, 10, 10, 24, 128, 2, st) < 0
    assert b"C <= 23" in L.fno_last_error()
    assert L.fno_head_bwd_tc(p, p, p, p, p, p, p, p, p, p, p, p, 1, 8, 8, 10, 10, 20, 64, 2, st) < 0
    assert L.fno_head_bwd_tc(p, p, p, p, p, p, p, p, p, p, p, None, 1, 8, 8, 10, 10, 20, 128, 2, st) < 0   # no workspace
    # fused bypass backward: needs the weights and the output tensor
    assert L.fno_pointwise_bwd(p, p, None, p, p, p, p, 1, 20, 20, 64, st) < 0
    # window gather: window longer than the trajectory
    assert L.fno_window_gather(p, p, p, p, p, 2, 16, 5, 2, 5, 1, st) < 0
    # math mode
    assert L.fno_set_math_mode(7) < 0
    assert lib.get_math_mode() == "fp32"
    with pytest.raises(lib.FnoError):
        lib.set_math_mode("fp8")          # only fp32 / tf32 / bf16 exist
    assert lib.get_math_mode() == "fp32"
    # device-resident dataset: trajectories shorter than a window
    from fno_b200 import data
    with pytest.raises(ValueError):
        data.DeviceWindows(torch.zeros(2, 5, 8, 8, 2), initial_step=5, rollout=1, device="cuda")
