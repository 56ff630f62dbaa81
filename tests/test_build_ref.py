"""oracle/build_ref.py, which build() calls: it copies the reference's training-loop files into oracle/_ref/ when
$PDEBENCH_MODELS names a readable tree, and skips an unset, absent or unreadable source instead of failing the build."""
import json
from pathlib import Path

import pytest

from oracle import build_ref


@pytest.fixture
def dst(tmp_path, monkeypatch):
    d = tmp_path / "_ref"
    monkeypatch.setattr(build_ref, "DST", d)
    return d


def _reference_tree(root: Path) -> Path:
    for rel in build_ref.FILES:
        (root / rel).parent.mkdir(parents=True, exist_ok=True)
        (root / rel).write_text(f"# {rel}\n")
    return root


def test_copies_the_tree_named_by_the_environment(tmp_path, dst, monkeypatch):
    monkeypatch.setenv(build_ref.ENV, str(_reference_tree(tmp_path / "models")))
    assert build_ref.build(verbose=False)
    for rel in build_ref.FILES:
        assert (dst / rel).read_text() == f"# {rel}\n"
    assert sorted(json.loads((dst / "MANIFEST.json").read_text())["sha256"]) == sorted(build_ref.FILES)


def test_unset_absent_or_unreadable_source_is_skipped(tmp_path, dst, monkeypatch):
    monkeypatch.delenv(build_ref.ENV, raising=False)
    assert not build_ref.build(verbose=False)
    monkeypatch.setenv(build_ref.ENV, str(tmp_path / "missing"))
    assert not build_ref.build(verbose=False)
    src = _reference_tree(tmp_path / "models")

    def denied(self):
        raise PermissionError(13, "Permission denied", str(self))

    monkeypatch.setattr(Path, "read_bytes", denied)
    assert not build_ref.build(src, verbose=False)
    assert not dst.exists()
