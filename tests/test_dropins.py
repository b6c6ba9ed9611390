"""CPU: goliath_b200.install_dropins() against the interface the reference's own Python wrappers expect —
extensions/sgutils/sgutils.py, extensions/utils/utils.py, extensions/mvpraymarch/mvpraymarch.py and
ca_code/utils/render_gsplat.py.  That interface (imported names, every call into an extension module with its
positional count and keywords, the argument names of the public functions) is stored as data in
tests/golden/reference_interface.json, written by tests/golden/make_reference_interface_golden.py."""
import importlib
import inspect
import json
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
IFACE = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_interface.json")))
OURS = {"extensions/sgutils/sgutils.py": "goliath_b200.sgutils", "extensions/utils/utils.py": "goliath_b200.utils",
        "extensions/mvpraymarch/mvpraymarch.py": "goliath_b200.mvpraymarch"}


def _calls():
    return [c for w in IFACE.values() for c in w["calls"]]


def test_reference_wrappers_bind_to_our_modules():
    import goliath_b200

    goliath_b200.install_dropins()
    imported = {n for w in IFACE.values() for n in w["imports"]}
    assert imported == {"sgutilslib", "utilslib", "mvpraymarchlib", "gsplat"}
    for name in imported:  # what the wrappers' `import X` / `from X import ...` now resolve to
        assert importlib.import_module(name) is importlib.import_module("goliath_b200." + name), name
    assert sys.modules["gsplat"] is importlib.import_module("goliath_b200.gsplat")
    gsplat = importlib.import_module("gsplat")
    for w in IFACE.values():
        for n in w["imported_names"]:
            assert callable(getattr(gsplat, n)), n
    # every call the wrappers make into an extension module binds to the drop-in's signature
    for c in _calls():
        fn = getattr(importlib.import_module(c["module"]), c["function"])
        inspect.signature(fn).bind(*([None] * c["positional"]), **{k: None for k in c["keywords"]})
    # our mirrors of the wrappers' public functions take the same argument names
    for path, mod in OURS.items():
        for fname, names in IFACE[path]["functions"].items():
            ours = getattr(importlib.import_module(mod), fname)
            assert list(inspect.signature(ours).parameters) == names, (path, fname)
    # render_raymarcher.py:59 introspects the Python function's co_varnames: it must stay a Python function with them
    from goliath_b200.mvpraymarch import mvpraymarch
    names = mvpraymarch.__code__.co_varnames
    assert {"raypos", "raydir", "stepsize", "tminmax", "primtransf", "template", "warp", "usebvh", "fadescale"} <= set(names)
    assert set(names[:mvpraymarch.__code__.co_argcount]) == set(IFACE["extensions/mvpraymarch/mvpraymarch.py"]["functions"]["mvpraymarch"])


def test_reference_wrappers_reach_our_abi_on_cpu_tensors():
    """No GPU here: each call the reference's wrappers make into sgutilslib / utilslib / mvpraymarchlib, made with CPU
    tensors, must arrive at our shim, which refuses it (build_tree: a path the reference cannot run either)."""
    import goliath_b200

    goliath_b200.install_dropins()
    t = torch.zeros(1, 4, 3)
    for c in _calls():
        if c["module"] == "gsplat":
            continue
        fn = getattr(importlib.import_module(c["module"]), c["function"])
        with pytest.raises(RuntimeError, match="CUDA" if c["function"] != "build_tree" else "reference"):
            fn(*([t] * c["positional"]), **{k: t for k in c["keywords"]})
