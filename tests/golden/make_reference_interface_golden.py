"""Generate tests/golden/reference_interface.json: the interface the reference's own Python wrappers expect of the
extension modules that goliath_b200.install_dropins() replaces, read from the wrappers' syntax trees (no source text is
stored).  Per wrapper file: the extension names it imports, every call into an extension module (function, number of
positional arguments, keyword names) and the argument names of its public functions.  tests/test_dropins.py checks the
drop-ins against it.

Needs a checkout of the reference (facebookresearch/goliath), found as oracle/build_ref.py finds it; the .json is
committed.   Usage: [GOLIATH_REFERENCE=<goliath checkout>] python tests/golden/make_reference_interface_golden.py
"""
import ast
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
OUT = os.path.join(HERE, "reference_interface.json")
EXT = ("sgutilslib", "utilslib", "mvpraymarchlib", "gsplat")
WRAPPERS = {  # wrapper file -> its public functions
    "extensions/sgutils/sgutils.py": ("evaluate_gaussian",),
    "extensions/utils/utils.py": ("compute_raydirs",),
    "extensions/mvpraymarch/mvpraymarch.py": ("mvpraymarch", "build_accel"),
    "ca_code/utils/render_gsplat.py": (),
}
# a starred argument of a call into an extension unpacks the tuple last assigned to that name in the same function;
# without such an assignment it is a parameter: build_accel's `primtransfin`, documented as tuple[tensor, tensor, tensor]
STARRED_PARAM = {"primtransfin": 3}


def arg_names(fn):
    a = fn.args
    return [x.arg for x in a.posonlyargs + a.args + a.kwonlyargs]


def scan(path, public):
    tree = ast.parse(open(path).read())
    imports, from_gsplat, calls, funcs = set(), set(), [], {}
    for node in ast.walk(tree):
        if isinstance(node, ast.Import):
            imports.update(a.name for a in node.names if a.name in EXT)
        elif isinstance(node, ast.ImportFrom) and node.module in EXT:
            imports.add(node.module)
            from_gsplat.update(a.name for a in node.names)
        elif isinstance(node, ast.FunctionDef) and node.name in public:
            funcs[node.name] = arg_names(node)
    tuples = {}  # call -> {name: length of the tuple assigned to it before the call in the enclosing function}
    for fn in ast.walk(tree):
        if not isinstance(fn, ast.FunctionDef):
            continue
        assigns = [(n.lineno, t.id, len(n.value.elts)) for n in ast.walk(fn) if isinstance(n, ast.Assign)
                   and isinstance(n.value, ast.Tuple) for t in n.targets if isinstance(t, ast.Name)]
        for call in ast.walk(fn):
            if isinstance(call, ast.Call):
                tuples[call] = {name: k for line, name, k in sorted(assigns) if line < call.lineno}
    for node in ast.walk(tree):
        if not isinstance(node, ast.Call):
            continue
        f = node.func
        if isinstance(f, ast.Attribute) and isinstance(f.value, ast.Name) and f.value.id in EXT:
            module, name = f.value.id, f.attr
        elif isinstance(f, ast.Name) and f.id in from_gsplat:
            module, name = "gsplat", f.id
        else:
            continue
        n = 0
        for a in node.args:
            if isinstance(a, ast.Starred):
                n += tuples.get(node, {}).get(a.value.id) or STARRED_PARAM[a.value.id]
            else:
                n += 1
        calls.append({"module": module, "function": name, "positional": n,
                      "keywords": sorted(k.arg for k in node.keywords if k.arg is not None)})
    calls = [dict(t) for t in sorted({tuple((k, tuple(v) if isinstance(v, list) else v) for k, v in c.items())
                                      for c in calls})]
    for c in calls:
        c["keywords"] = list(c["keywords"])
    return {"imports": sorted(imports), "imported_names": sorted(from_gsplat), "calls": calls, "functions": funcs}


def main():
    from oracle.build_ref import reference_dir

    ref = reference_dir()
    if not os.path.isdir(ref):
        sys.exit("no reference checkout at %s: set GOLIATH_REFERENCE to a checkout of facebookresearch/goliath" % ref)
    out = {f: scan(os.path.join(ref, f), pub) for f, pub in WRAPPERS.items()}
    with open(OUT, "w") as fh:
        json.dump(out, fh, indent=1, sort_keys=True)
        fh.write("\n")
    print("wrote", OUT)


if __name__ == "__main__":
    main()
