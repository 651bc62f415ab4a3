"""Imports the UNMODIFIED reference (`open_clip` + `training` of UCSC-VLAA/CLIPA clipa_torch) for
measurement and drop-in tests.  Never imported by the product path (clipa_b200/).

Where it comes from: `oracle/_ref/`, filled from a clipa_torch checkout by `oracle/install_reference.sh`
(git-ignored).  Nothing else is searched: tests compare against the committed vectors under tests/golden.

The reference's tokenizer / data modules import ftfy, tensorflow(_text), webdataset, braceexpand
unconditionally (open_clip/tokenizer.py:11-18, training/data.py:9,17-22); none of them is on the
hot path and none is installed, so they are stubbed.  The wheel does not carry the JSON model
configs (setup.py has no package_data): they are registered through the reference's own
`add_model_config` from clipa_b200's size table, which tests pin against the reference's JSON files.
"""
from __future__ import annotations

import importlib.machinery
import json
import sys
import tempfile
from pathlib import Path
from unittest.mock import MagicMock

ROOT = Path(__file__).resolve().parent.parent
REF_DIR = ROOT / "oracle" / "_ref"
_STUBS = ("ftfy", "tensorflow", "tensorflow_text", "webdataset", "webdataset.filters",
          "webdataset.tariterators", "braceexpand", "fsspec", "timm", "horovod", "horovod.torch")


def reference_root():
    return REF_DIR if (REF_DIR / "open_clip" / "factory.py").exists() else None


def available() -> bool:
    return reference_root() is not None


def import_reference(register_configs: bool = True):
    """Returns the reference's `open_clip` module (its `training` package becomes importable too)."""
    root = reference_root()
    if root is None:
        raise RuntimeError(f"reference not installed in {REF_DIR}: run oracle/install_reference.sh <clipa_torch dir>")
    for n in _STUBS:
        if n not in sys.modules:
            try:
                __import__(n)
            except Exception:
                m = MagicMock()
                m.__spec__ = importlib.machinery.ModuleSpec(n, None)
                m.__path__ = []
                sys.modules[n] = m
    if str(root) not in sys.path:
        sys.path.insert(0, str(root))
    import open_clip  # noqa: the reference's, top-level
    assert Path(open_clip.__file__).resolve().is_relative_to(root.resolve()), open_clip.__file__
    if register_configs:
        from clipa_b200.open_clip.model_configs import _MODEL_CONFIGS
        tmp = Path(tempfile.mkdtemp(prefix="clipa_ref_cfg_"))
        for name, cfg in _MODEL_CONFIGS.items():
            if open_clip.get_model_config(name) is None:
                (tmp / f"{name}.json").write_text(json.dumps(cfg))
        open_clip.add_model_config(tmp)
    return open_clip
