"""Runs one of the reference's UNMODIFIED training loops and prints the per-epoch numbers it printed as JSON.

    python oracle/run_ref_loop.py --loop fno|aux --model reference|dropin [--cfg '{...}'] [--golden out.json] [--workdir d]

--model reference : the reference's own FNO2d (fno/fno.py or fno_aux/fno_aux.py), on whatever device the loop picks
                    (`cuda` if available, fno/train.py:32) -- on the GPU box this is "the reference on the same B200"
--model dropin    : `fno.fno` / `fno_aux.fno_aux` are shadowed in sys.modules by fno_b200.fno / fno_b200.fno_aux before the
                    loop is imported (INTEGRATION.md): the loop itself is untouched and drives the sm_100a kernels
The reference files are taken from oracle/_ref/ (oracle/build_ref.py).
Recipe of SURVEY.md appendix B: stub h5py / matplotlib, register the synthetic datasets under the loader module names, disable
wandb, call run_training(**kwargs).  TEST INFRASTRUCTURE ONLY.
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import os
import re
import sys
import tempfile
import types
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
DEFAULT_CFG = {
    "fno": dict(n=128, modes=12, width=20, initial_step=10, num_channels=2, batch_size=4, epochs=3, train_traj=3, val_traj=1,
                windows=8, train_seed=0, val_seed=1, learning_rate=1e-3),
    # config 2 (fno_aux multiphysics joint training): batch 2, 3 auxiliary samples per item, auxiliary_weight 0.7
    # (config_dr.yaml:20,36-37), two learning rates
    "aux": dict(n=128, modes=12, width=20, initial_step=10, num_channels=2, batch_size=2, epochs=3, train_traj=2, val_traj=1,
                windows=8, train_seed=0, val_seed=1, aux_seed=2, learning_rate_share=1e-3, learning_rate_fc2=2e-3,
                num_aux_samples=3, auxiliary_weight=0.7),
}


def ref_root() -> Path:
    ref = ROOT / "oracle" / "_ref"
    if not (ref / "fno" / "train.py").exists():
        raise SystemExit("reference files not found: build() with PDEBENCH_MODELS=<pdebench>/pdebench/models, or "
                         "python oracle/build_ref.py <pdebench>/pdebench/models")
    return ref


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--loop", choices=["fno", "aux"], required=True)
    ap.add_argument("--model", choices=["reference", "dropin"], required=True)
    ap.add_argument("--cfg", default="{}")
    ap.add_argument("--golden", default=None, help="also write the result as a golden fixture to this path")
    ap.add_argument("--workdir", default=None, help="directory the loop writes its checkpoint into (default: a temp dir)")
    args = ap.parse_args()
    cfg = dict(DEFAULT_CFG[args.loop], **json.loads(args.cfg))
    os.environ["WANDB_MODE"] = "disabled"
    os.environ["FNO_REF_DATA"] = json.dumps(cfg)
    ref = ref_root()
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(ROOT / "sciml-pde_b200"))
    sys.path.insert(0, str(ref))
    import torch

    for name in ["h5py", "matplotlib", "matplotlib.pyplot", "mpl_toolkits", "mpl_toolkits.axes_grid1"]:
        sys.modules[name] = types.ModuleType(name)
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.modules["mpl_toolkits.axes_grid1"].make_axes_locatable = lambda *a, **k: None
    from oracle import ref_datasets

    import fno  # noqa: F401  (namespace packages of the reference tree)
    import fno_aux  # noqa: F401
    stub = types.ModuleType("fno.utils_2d_ns_baseline_lie")
    stub.FNODatasetMult = ref_datasets.FNODatasetMult
    sys.modules["fno.utils_2d_ns_baseline_lie"] = stub
    stub = types.ModuleType("fno_aux.utils_2d_ns")
    stub.FNODatasetMult = ref_datasets.AuxFNODatasetMult
    sys.modules["fno_aux.utils_2d_ns"] = stub
    if args.model == "dropin":
        import fno_b200.fno
        import fno_b200.fno_aux
        sys.modules["fno.fno"] = fno_b200.fno
        sys.modules["fno_aux.fno_aux"] = fno_b200.fno_aux
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    common = dict(if_training=True, continue_training=False, rollout_test=1, modes=cfg["modes"], width=cfg["width"],
                  initial_step=cfg["initial_step"], t_train=101, num_channels=cfg["num_channels"], batch_size=cfg["batch_size"],
                  epochs=cfg["epochs"], train_subsample=[8, 4, 12], scheduler_step=100, scheduler_gamma=0.5, model_update=1,
                  plot=False, channel_plot=0, x_min=-1, x_max=1, y_min=-1, y_max=1, t_min=0, t_max=5, base_path="unused",
                  training_type="single", scheduler="cosine")
    if args.loop == "fno":
        from fno.train import run_training
        kwargs = dict(common, num_workers=0, learning_rate=cfg["learning_rate"], FNO_model_flmn="refloop")
        pat = r"epoch: (\d+), loss: ([\d.eE+-]+),\s+trainL2: ([\d.eE+-]+), testL2: ([\d.eE+-]+)"
        names = ("loss", "trainL2", "testL2")
    else:
        from fno_aux.fno_train_aux import run_training
        kwargs = dict(common, num_workers=1, if_downsample=False, learning_rate_share=cfg["learning_rate_share"],
                      learning_rate_fc2=cfg["learning_rate_fc2"], num_aux_samples=cfg["num_aux_samples"],
                      auxiliary_weight=cfg["auxiliary_weight"], model_flmn="refloop", aux_path="unused")
        pat = (r"epoch: (\d+), loss: ([\d.eE+-]+),\s+trainL2: ([\d.eE+-]+), trainL2_AUX: ([\d.eE+-]+), "
               r"testL2: ([\d.eE+-]+), testL2_AUX: ([\d.eE+-]+)")
        names = ("loss", "trainL2", "trainL2_AUX", "testL2", "testL2_AUX")
    buf = io.StringIO()
    cwd = os.getcwd()
    tmp = None
    if args.workdir is None:
        tmp = tempfile.TemporaryDirectory()
        workdir = tmp.name
    else:
        workdir = args.workdir
        os.makedirs(workdir, exist_ok=True)
    os.chdir(workdir)                      # the loop writes <name>_FNO.pt into cwd
    try:
        with contextlib.redirect_stdout(buf):
            run_training(**kwargs)
    finally:
        os.chdir(cwd)
    text = buf.getvalue()
    rows = re.findall(pat, text)
    if len(rows) != cfg["epochs"]:
        sys.stderr.write(text)
        raise SystemExit("could not parse the reference loop's per-epoch lines")
    import torch as _t
    dev = "cuda" if _t.cuda.is_available() else "cpu"
    out = {"loop": args.loop, "model": args.model, "device": dev, "config": cfg, "seed": 16, "torch": torch.__version__,
           "reference_files": str(ref),
           "source": "stdout of the unmodified run_training (%s)" % ("fno/train.py" if args.loop == "fno" else "fno_aux/fno_train_aux.py"),
           "printed_precision": "5 decimals",
           "epochs": [dict(epoch=int(r[0]), **{n: float(v) for n, v in zip(names, r[1:])}) for r in rows],
           "checkpoints": sorted(p.name for p in Path(workdir).glob("*.pt"))}
    if args.golden:
        Path(args.golden).write_text(json.dumps(out, indent=1))
    print("REFLOOP_JSON " + json.dumps(out))
    if tmp is not None:
        tmp.cleanup()


if __name__ == "__main__":
    main()
