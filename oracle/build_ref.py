"""Recipe for oracle/_ref/: the reference's own files for the training path, copied VERBATIM from a PDEBench checkout so
that tests/test_ref_loops_gpu.py can run the UNMODIFIED loops -- `fno.train.run_training` (fno/train.py:43-347) and
`fno_aux.fno_train_aux.run_training` (fno_aux/fno_train_aux.py:43-430) -- against either the reference models or the
shadowed drop-in.

    PDEBENCH_MODELS=<pdebench checkout>/pdebench/models python -c "import __graft_entry__ as g; g.build()"
    python oracle/build_ref.py [<pdebench checkout>/pdebench/models]

__graft_entry__.build() calls build() and so refreshes the copy whenever $PDEBENCH_MODELS names a readable reference
tree; an unset, absent or unreadable source leaves oracle/_ref/ as it is.  TEST INFRASTRUCTURE ONLY.  oracle/_ref/ is
listed in .gitignore: no reference source enters the history.  Nothing in the product imports it; without it the
unmodified-loop tests skip.
"""
from __future__ import annotations

import hashlib
import json
import os
import shutil
import sys
from pathlib import Path
from typing import Optional

ROOT = Path(__file__).resolve().parent.parent
DST = ROOT / "oracle" / "_ref"
FILES = ["fno/fno.py", "fno/train.py", "fno_aux/fno_aux.py", "fno_aux/fno_train_aux.py", "metrics.py", "metrics_aux.py"]
ENV = "PDEBENCH_MODELS"


def build(src: Optional[Path] = None, verbose: bool = True) -> bool:
    """Copies FILES from `src` (default: $PDEBENCH_MODELS) into oracle/_ref/.  Returns whether oracle/_ref/ holds a
    copy afterwards; a source that is unset, absent or unreadable (PermissionError included) is skipped, not raised."""
    if src is None and os.environ.get(ENV):
        src = Path(os.environ[ENV])
    if src is None:
        return (DST / FILES[1]).exists()
    try:
        data = {rel: (src / rel).read_bytes() for rel in FILES}
    except OSError as exc:
        if verbose:
            print(f"[oracle/_ref] reference tree {src} not readable ({exc.strerror}); left as it is", file=sys.stderr)
        return (DST / FILES[1]).exists()
    for rel, blob in data.items():
        dst = DST / rel
        dst.parent.mkdir(parents=True, exist_ok=True)
        dst.write_bytes(blob)
    manifest = {rel: hashlib.sha256(blob).hexdigest() for rel, blob in data.items()}
    (DST / "MANIFEST.json").write_text(json.dumps({"source": str(src), "sha256": manifest}, indent=1))
    if verbose:
        print(f"[oracle/_ref] copied {len(FILES)} reference files", file=sys.stderr)
    return True


if __name__ == "__main__":
    if len(sys.argv) > 2 or (len(sys.argv) == 1 and not os.environ.get(ENV)):
        raise SystemExit(__doc__)
    if not build(Path(sys.argv[1]) if len(sys.argv) == 2 else None):
        raise SystemExit(1)
