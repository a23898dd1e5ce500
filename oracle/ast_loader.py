"""ORACLE — test infrastructure only. Loads the reference's own model classes WITHOUT copying them.

The reference scripts cannot be imported (they np.load absent Features/*.npz at import time and import librosa /
allennlp / tensorflow, audio_gru_whole.py:19-20, fuse_net_whole.py:10-16), but their model classes are
self-contained: this module parses a script, extracts the wanted ``ClassDef`` nodes and executes just those
with torch in scope. Works only where a checkout of the reference is at ``B200RNN_REFERENCE_ROOT``; the tests never
need it (they compare against what oracle/make_golden.py recorded from it under tests/golden/).
"""
from __future__ import annotations

import ast
import os
from typing import Dict, Iterable

import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.autograd import Variable

REFERENCE_ROOT = os.environ.get("B200RNN_REFERENCE_ROOT", "")

FILES = {
    "audio_clf": "Classification/audio_gru_whole.py",
    "text_clf": "Classification/text_bilstm_whole.py",
    "fuse_clf": "Classification/fuse_net_whole.py",
    "audio_reg": "Regression/audio_bilstm_perm.py",
    "text_reg": "Regression/text_bilstm_perm.py",
    "fuse_reg": "Regression/fuse_net.py",
}


def available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isdir(REFERENCE_ROOT)


def load_classes(key: str, names: Iterable[str], extra_globals: Dict | None = None) -> Dict[str, type]:
    """Execute the ``ClassDef``s called ``names`` from the reference script ``FILES[key]``."""
    path = os.path.join(REFERENCE_ROOT, FILES[key])
    with open(path, "r", encoding="utf-8") as fh:
        tree = ast.parse(fh.read(), filename=path)
    wanted = set(names)
    nodes = [n for n in tree.body if isinstance(n, ast.ClassDef) and n.name in wanted]
    missing = wanted - {n.name for n in nodes}
    if missing:
        raise KeyError(f"{path}: no class {sorted(missing)}")
    scope = {"torch": torch, "nn": nn, "F": F, "Variable": Variable, "__name__": f"reference_{key}"}
    if extra_globals:
        scope.update(extra_globals)
    module = ast.Module(body=nodes, type_ignores=[])
    exec(compile(module, path, "exec"), scope)  # noqa: S102 - executing the read-only reference on purpose
    return {n: scope[n] for n in wanted}
