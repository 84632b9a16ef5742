"""Import the UNMODIFIED reference (UCSD-Comp-Imaging/Nerf-Simple) as a live oracle / CPU baseline.
TEST INFRASTRUCTURE ONLY: used by oracle/gen_golden.py, bench.py's reference arm and tests/.

Where the reference comes from, in order: $NERF_REFERENCE, the checkout BASELINE.json's reference_path
names, baseline/_ref (staged from one of those by __graft_entry__.build() / scripts/stage_reference.sh;
git-ignored).  Without any of them, callers skip or fall back as they document.

Two shims, both outside the reference's files (SURVEY.md 8c):
  * cpu=True: `Tensor.cuda` / `Module.cuda` become no-ops, because the reference hard-codes `.cuda()`
    (utils/rendering.py:30,68,...) and the CPU arm has to run without a device.  Process-wide, so
    callers that also use a GPU run this in a process of its own.
  * a `natsort` stand-in (natsort_keygen / ns.IGNORECASE) when the package is missing:
    utils/dataload.py:8 imports it and it is not installed in this image.
"""
from __future__ import annotations

import importlib
import json
import os
import re
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _is_checkout(path):
    return bool(path) and os.path.isfile(os.path.join(path, "utils", "rendering.py"))


def checkout_root():
    """A reference checkout outside the tree: $NERF_REFERENCE, else BASELINE.json's reference_path; None if neither
    holds one."""
    cands = [os.environ.get("NERF_REFERENCE")]
    try:
        with open(os.path.join(ROOT, "BASELINE.json")) as fh:
            cands.append(json.load(fh).get("reference_path"))
    except (OSError, ValueError):
        pass
    return next((c for c in cands if _is_checkout(c)), None)


def reference_root():
    staged = os.path.join(ROOT, "baseline", "_ref")
    return checkout_root() or (staged if _is_checkout(staged) else None)


def install_natsort_stub():
    try:
        import natsort  # noqa: F401
        return False
    except ImportError:
        pass
    mod = types.ModuleType("natsort")

    class ns:  # noqa: N801
        IGNORECASE = 1

    def natsort_keygen(alg=0):
        def key(s):
            s = str(s)
            return [int(t) if t.isdigit() else (t.lower() if alg & ns.IGNORECASE else t) for t in re.split(r"(\d+)", s)]
        return key

    mod.ns, mod.natsort_keygen = ns, natsort_keygen
    sys.modules["natsort"] = mod
    return True


def cuda_noop_shim():
    import torch
    torch.Tensor.cuda = lambda self, *a, **k: self
    torch.nn.Module.cuda = lambda self, *a, **k: self


def import_reference(cpu=True, root=None, with_dataload=False):
    """Returns (nets, rendering, xyz[, dataload]) modules of the reference, imported from `root`."""
    root = root or reference_root()
    if root is None:
        raise FileNotFoundError("reference checkout not found (set NERF_REFERENCE or run scripts/stage_reference.sh)")
    if cpu:
        cuda_noop_shim()
    install_natsort_stub()
    for name in [m for m in sys.modules if m == "utils" or m.startswith("utils.")]:
        del sys.modules[name]
    sys.path.insert(0, root)
    try:
        nets = importlib.import_module("utils.nets")
        rendering = importlib.import_module("utils.rendering")
        xyz = importlib.import_module("utils.xyz")
        mods = [nets, rendering, xyz]
        if with_dataload:
            mods.append(importlib.import_module("utils.dataload"))
    finally:
        sys.path.remove(root)
    assert os.path.samefile(os.path.dirname(nets.__file__), os.path.join(root, "utils")), nets.__file__
    return tuple(mods)
