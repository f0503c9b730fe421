"""Loads the reference's UNMODIFIED stack Python op files, ``pcdet/ops/pointnet2/pointnet2_stack/pointnet2_utils.py``
and ``pointnet2_modules.py`` (test infrastructure), straight from the reference tree (``oracle/build_ref.REF_ROOT``) over
THIS repo's pybind-name shim, as INTEGRATION.md section 1 wires them:
``pcdet.ops.pointnet2.pointnet2_stack.pointnet2_stack_cuda`` resolves to ``tsmdet_b200.pointnet2_stack.pointnet2_stack_cuda``.
Nothing is copied, edited or written (no bytecode cache)."""
from __future__ import annotations

import importlib.util
import os
import sys

from ref_py import _alias, _stub

_PKG = "pcdet.ops.pointnet2.pointnet2_stack"


def _load_source(name: str, path: str):
    if name in sys.modules:
        return sys.modules[name]
    parent, _, leaf = name.rpartition(".")
    _stub(parent)
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    mod.__package__ = parent
    sys.modules[name] = mod
    old = sys.dont_write_bytecode
    sys.dont_write_bytecode = True
    try:
        spec.loader.exec_module(mod)
    finally:
        sys.dont_write_bytecode = old
    setattr(sys.modules[parent], leaf, mod)
    return mod


def load_reference_stack_python():
    """Returns (pointnet2_utils, pointnet2_modules) of the reference's pointnet2_stack, or None without the reference
    tree."""
    from oracle import build_ref
    from tsmdet_b200.pointnet2_stack import pointnet2_stack_cuda

    src = os.path.join(build_ref.REF_ROOT, *_PKG.split("."))
    paths = [os.path.join(src, f) for f in ("pointnet2_utils.py", "pointnet2_modules.py")]
    if not all(os.path.exists(p) for p in paths):
        return None
    _alias(f"{_PKG}.pointnet2_stack_cuda", pointnet2_stack_cuda)
    return tuple(_load_source(f"{_PKG}.{os.path.basename(p)[:-3]}", p) for p in paths)
