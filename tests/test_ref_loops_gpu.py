"""The reference's UNMODIFIED training loops on the B200 (SURVEY.md 8c, oracle stack item 3): `fno.train.run_training`
(fno/train.py:43-347) and `fno_aux.fno_train_aux.run_training` (fno_aux/fno_train_aux.py:43-430), imported from the verbatim
copies under oracle/_ref/ (oracle/build_ref.py), driven through oracle/run_ref_loop.py in a subprocess each (the loops seed
the RNG at import and pick their device at module level).

* `--model dropin`: `fno.fno` / `fno_aux.fno_aux` shadowed by the sm_100a drop-in (INTEGRATION.md) -- the loops, their
  DataLoaders, torch.optim.Adam over three parameter groups, CosineAnnealingLR, clip and checkpointing are the reference's;
* `--model reference`: the reference's own modules on the same GPU through stock PyTorch.
Both must reproduce the per-epoch numbers the reference printed on the CPU (tests/golden/loop_cfg1.json,
loop_aux_cfg2.json; 1e-4 relative, SURVEY 8c), and the checkpoint the loop wrote must hold the reference's keys."""
import json
import subprocess
import sys
from pathlib import Path

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
GOLDEN = ROOT / "tests" / "golden"
TOL = 1e-4


def _run(loop, model, workdir=None):
    if not (ROOT / "oracle" / "_ref" / "fno" / "train.py").exists():
        pytest.skip("needs the reference's own training loops in oracle/_ref/ (build() with PDEBENCH_MODELS set)")
    cmd = [sys.executable, str(ROOT / "oracle" / "run_ref_loop.py"), "--loop", loop, "--model", model]
    if workdir is not None:
        cmd += ["--workdir", str(workdir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("REFLOOP_JSON ")][-1]
    return json.loads(line[len("REFLOOP_JSON "):])


def _check(got, gold, names, tol=TOL):
    assert got["config"] == gold["config"]
    assert len(got["epochs"]) == len(gold["epochs"])
    for a, b in zip(got["epochs"], gold["epochs"]):
        for n in names:
            assert abs(a[n] - b[n]) <= tol * abs(b[n]) + 6e-6, (b["epoch"], n, a[n], b[n])


@pytest.mark.parametrize("model", ["dropin", "reference"])
def test_unmodified_fno_loop(model, tmp_path):
    gold = json.loads((GOLDEN / "loop_cfg1.json").read_text())
    got = _run("fno", model, tmp_path)
    assert got["device"] == "cuda"
    _check(got, gold, ("loss", "trainL2", "testL2"))
    # the checkpoint the loop wrote (fno/train.py:319-329)
    ck = torch.load(tmp_path / "refloop_FNO.pt", map_location="cpu", weights_only=False)
    assert sorted(ck) == ["epoch", "loss", "model_state_dict", "optimizer_state_dict"]
    assert len(ck["model_state_dict"]) == 22
    if model == "dropin":
        # ... loads strict into the reference's own module and vice versa
        sys.path.insert(0, str(ROOT / "sciml-pde_b200"))
        from fno_b200.fno import FNO2d
        c = gold["config"]
        m = FNO2d(num_channels=c["num_channels"], modes1=c["modes"], modes2=c["modes"], width=c["width"],
                  initial_step=c["initial_step"])
        m.load_state_dict(ck["model_state_dict"], strict=True)


@pytest.mark.parametrize("model", ["dropin", "reference"])
def test_unmodified_joint_loop(model, tmp_path):
    """config 2: two-head model, B * (1 + 3) trunk batch, loss = primary + 0.7 auxiliary, three Adam groups."""
    gold = json.loads((GOLDEN / "loop_aux_cfg2.json").read_text())
    got = _run("aux", model, tmp_path)
    assert got["device"] == "cuda"
    _check(got, gold, ("loss", "trainL2", "trainL2_AUX", "testL2", "testL2_AUX"))
    ck = torch.load(tmp_path / "refloop_aux_FNO.pt", map_location="cpu", weights_only=False)
    assert sorted(ck) == ["epoch", "loss", "model_state_dict", "optimizer_state_dict"]
    assert len(ck["model_state_dict"]) == 44
    assert len(ck["optimizer_state_dict"]["param_groups"]) == 3
