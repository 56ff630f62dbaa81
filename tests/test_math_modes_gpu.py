"""The tf32 and bf16 math modes (fno_b200.lib.set_math_mode) on whole models and in captured CUDA graphs.

Whole models: BASELINE configs 1-4 through the drop-in modules in fp32, tf32 and bf16 mode on the same seeded inputs and
weights, against the fp64 port of the reference (oracle/fno_port.py): output, nRMSE loss and every parameter gradient,
one tensor at a time, as max|err| / max|ref|.  fp32 mode keeps the tolerances of test_configs_gpu.py (1e-5 outputs,
2e-5 gradients).  The low modes are held to the per-kernel bounds (tf32 2e-3, bf16 2e-2): errors do not compound past
them through four Fourier layers, the lift and the head.

Graphs: the mode is read on the host at each launch, so a captured training step keeps the mode it was captured in
whatever the global mode is at replay."""
import copy

import pytest
import torch

from oracle import dft_oracle as O
from oracle import fno_port as P

pytestmark = pytest.mark.gpu
MODEL_TOL = {"fp32": (1e-5, 2e-5), "tf32": (2e-3, 2e-3), "bf16": (2e-2, 2e-2)}     # (outputs and loss, gradients)


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


def seeded(shape, seed, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return scale * torch.randn(shape, generator=g)


def _grid(n, nd, lo=0.0, hi=1.0):
    lin = torch.linspace(lo, hi, n)
    return torch.stack(torch.meshgrid(*(lin,) * nd, indexing="ij"), dim=-1).unsqueeze(0)


def _cfg1():
    from fno_b200.fno import FNO2d

    torch.manual_seed(16)
    model = FNO2d(num_channels=2, modes1=12, modes2=12, width=20, initial_step=10)
    x, yy = seeded((2, 128, 128, 10, 2), 100), seeded((2, 128, 128, 1, 2), 101)
    return model, (x, _grid(128, 2).repeat(2, 1, 1, 1)), (yy,), True


def _cfg2():
    from fno_b200.fno_aux import FNO2d

    torch.manual_seed(16)
    model = FNO2d(num_channels=2, modes1=12, modes2=12, width=20, initial_step=10)
    B, A = 2, 3
    g1 = _grid(128, 2, -1 + 1 / 128, 1 - 1 / 128)
    inputs = (seeded((B, 128, 128, 10, 2), 500), g1.repeat(B, 1, 1, 1),
              seeded((B * A, 128, 128, 10, 2), 501, scale=0.5), g1.repeat(B * A, 1, 1, 1))
    return model, inputs, (seeded((B, 128, 128, 1, 2), 502), seeded((B * A, 128, 128, 1, 2), 503)), False


def _cfg3():
    from fno_b200.fno import FNO2d

    torch.manual_seed(16)
    model = FNO2d(num_channels=3, modes1=16, modes2=16, width=64, initial_step=10)
    return model, (seeded((1, 256, 256, 10, 3), 300), _grid(256, 2)), (seeded((1, 256, 256, 1, 3), 301),), False


def _cfg4():
    from fno_b200.fno import FNO3d

    torch.manual_seed(16)
    model = FNO3d(num_channels=5, modes1=12, modes2=12, modes3=12, width=20, initial_step=10)
    return model, (seeded((1, 64, 64, 64, 10, 5), 400), _grid(64, 3)), (seeded((1, 64, 64, 64, 1, 5), 401),), False


CASES = {"cfg1": _cfg1, "cfg2": _cfg2, "cfg3": _cfg3, "cfg4": _cfg4}


def _loss(outs, targets):
    """nRMSE training loss (the joint model's: primary + 0.7 * auxiliary)."""
    return sum(w * P.nrmse(o, t).mean() for w, o, t in zip((1.0, 0.7), outs, targets))


class ModelCase:
    """The fp64 port's forward, loss and gradients, computed once; the drop-in model's errors against them per mode."""

    def __init__(self, name):
        model, self.inputs, self.targets, self.input_grad = CASES[name]()
        self.name = name
        self.state = {k: v.clone() for k, v in model.state_dict().items()}
        self.model = model
        skip = () if name != "cfg2" else ("shared_layers",)           # aliases of the trunk's parameters
        p = P.as_leaves({k: v for k, v in self.state.items() if not k.startswith(skip)}, dtype=torch.float64)
        x64 = [t.double().requires_grad_(self.input_grad and i == 0) for i, t in enumerate(self.inputs)]
        outs = P.fno_aux_forward(p, *x64) if name == "cfg2" else (P.fno_forward(p, *x64),)
        loss = _loss(outs, [t.double() for t in self.targets])
        loss.backward()
        self.ref_outs = [o.detach() for o in outs]
        self.ref_loss = loss.detach()
        self.ref_grads = {k: q.grad for k, q in p.items() if q.grad is not None}
        self.ref_xgrad = x64[0].grad
        self.errs = {}

    def run(self, lib, mode):
        """{tensor: rel_err} for the drop-in model in ``mode`` (memoised: the bf16 test compares with tf32)."""
        if mode in self.errs:
            return self.errs[mode]
        model = copy.deepcopy(self.model)
        model.load_state_dict(self.state)
        model = model.cuda()
        inputs = [t.cuda().requires_grad_(self.input_grad and i == 0) for i, t in enumerate(self.inputs)]
        lib.set_math_mode(mode)
        try:
            outs = model(*inputs)
            outs = outs if isinstance(outs, tuple) else (outs,)
            loss = _loss(outs, [t.cuda() for t in self.targets])
            loss.backward()
            torch.cuda.synchronize()
        finally:
            lib.set_math_mode("fp32")
        e = {f"out{k}": O.rel_err(o.detach().cpu().numpy(), r.numpy()) for k, (o, r) in enumerate(zip(outs, self.ref_outs))}
        e["loss"] = abs(float(loss.detach()) - float(self.ref_loss)) / abs(float(self.ref_loss))
        grads = {}
        for k, q in model.named_parameters():
            assert q.grad is not None or k.startswith("bn"), k
            if q.grad is not None:
                grads[k] = q.grad
        assert grads.keys() == self.ref_grads.keys()
        for k, g in grads.items():
            r = self.ref_grads[k]
            g, r = (torch.view_as_real(t) if t.is_complex() else t for t in (g, r))
            e[f"d {k}"] = O.rel_err(g.cpu().numpy(), r.numpy())
        if self.input_grad:
            e["d x"] = O.rel_err(inputs[0].grad.cpu().numpy(), self.ref_xgrad.numpy())
        self.errs[mode] = e
        return e


@pytest.fixture(scope="module", params=list(CASES))
def case(request):
    return ModelCase(request.param)


def _maxima(e):
    out = max(v for k, v in e.items() if not k.startswith("d "))
    grad = max(v for k, v in e.items() if k.startswith("d "))
    return out, grad


@pytest.mark.parametrize("mode", ["fp32", "tf32", "bf16"])
def test_model_math_modes(lib, case, mode):
    e = case.run(lib, mode)
    out, grad = _maxima(e)
    worst = max(e, key=e.get)
    print(f"\n{case.name} {mode}: outputs/loss max {out:.2e}, gradients max {grad:.2e} (worst: {worst} {e[worst]:.2e})")
    print("   ", {k: f"{v:.1e}" for k, v in e.items()})
    otol, gtol = MODEL_TOL[mode]
    assert out <= otol and grad <= gtol, e
    if mode == "bf16":                  # the mode reached the model: bf16 is coarser than tf32, tf32 than fp32
        t32, f32 = _maxima(case.run(lib, "tf32")), _maxima(case.run(lib, "fp32"))
        assert f32[0] < t32[0] < out and f32[1] < t32[1] < grad, (f32, t32, (out, grad))


# ---------------------------------------------------------------------------------------------------------------------
# a captured graph keeps its mode
# ---------------------------------------------------------------------------------------------------------------------
def _graph_run(lib, graph, modes, alias=False):
    """len(modes) FusedTrainSteps of one seeded width-8 model, step i in global math mode modes[i].  The aliasing run
    refills one set of input tensors in place, so that its aliased graph is captured on the fourth call."""
    from fno_b200 import data
    from fno_b200.fno import FNO2d
    from fno_b200.train import FusedTrainStep

    torch.manual_seed(16)
    model = FNO2d(num_channels=2, modes1=4, modes2=4, width=8, initial_step=3).cuda()
    plan = lib.get_plan(torch.device("cuda", 0), (18, 18), (4, 4))
    assert lib.layer_fused_supported(plan, 8) and lib.HEAD_TC and lib.HEAD_BWD_TC     # tcgen05 layers and head
    step = FusedTrainStep(model, lr=1e-3, weight_decay=1e-4, t_max=50, graph=graph, alias_inputs=alias)
    batches = [tuple(t.cuda() for t in data.synthetic_batch(4, 16, 3, 2, seed=s)) for s in range(3)]
    held = tuple(torch.empty_like(t) for t in batches[0])
    losses = []
    for i, mode in enumerate(modes):
        lib.set_math_mode(mode)
        batch = batches[i % 3]
        if alias:
            for dst, src in zip(held, batch):
                dst.copy_(src)
            batch = held
        losses.append(step(*batch).clone())
    torch.cuda.synchronize()
    lib.set_math_mode("fp32")
    return torch.stack(losses), {k: v.detach().clone() for k, v in model.state_dict().items()}


def _same(a, b):
    return torch.equal(a[0], b[0]) and all(torch.equal(a[1][k], b[1][k]) for k in a[1])


@pytest.mark.parametrize("captured,replayed,alias", [("tf32", "fp32", False), ("fp32", "bf16", False),
                                                      ("tf32", "fp32", True)], ids=["tf32-fp32", "fp32-bf16", "alias"])
def test_captured_graph_keeps_its_mode(lib, captured, replayed, alias):
    """The copying graph is captured on the third call, the aliased one on the fourth; the global mode changes after that
    and three more steps are replayed.  They are bitwise the eager steps in the capture mode, and differ from eager
    steps in the mode set at replay."""
    n_cap = 4 if alias else 3
    switched = [captured] * n_cap + [replayed] * 3
    graphed = _graph_run(lib, True, switched, alias)
    kept = _graph_run(lib, False, [captured] * len(switched))
    followed = _graph_run(lib, False, switched)
    assert torch.isfinite(graphed[0]).all()
    assert _same(graphed, kept)
    assert not torch.equal(graphed[0][n_cap:], followed[0][n_cap:])
    assert not _same(graphed, followed)
