"""Generate tests/golden/reference_surface.json: the plugin surface of ray_lightning (ray-project/ray_lightning
@ 24f5922), read from its source by AST (the package cannot be imported without ray / pytorch_lightning).
tests/test_surface_conformance.py checks this package's classes against it.

    python -m oracle.make_surface_golden PATH/TO/ray_lightning      # the package directory of a checkout

A signature is stored as [[[name, default], ...], vararg, kwarg, [kwonly, ...]]: positional parameters with
their defaults (None when there is none, "<expr>" when the default is not a literal).
"""
import ast
import json
import os
import sys

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                      "reference_surface.json")


def _tree(ref, path):
    with open(os.path.join(ref, path)) as f:
        return ast.parse(f.read())


def _cls(ref, path, name):
    for node in ast.walk(_tree(ref, path)):
        if isinstance(node, ast.ClassDef) and node.name == name:
            return node
    raise KeyError(name)


def _sig(fn):
    a = fn.args
    names = [x.arg for x in a.args]
    defaults = [None] * (len(names) - len(a.defaults)) + [ast.literal_eval(d) if isinstance(d, ast.Constant) else "<expr>" for d in a.defaults]
    return [list(zip(names, defaults)), (a.vararg.arg if a.vararg else None), (a.kwarg.arg if a.kwarg else None),
            [k.arg for k in a.kwonlyargs]]


def _methods(ref, path, name):
    return {n.name: _sig(n) for n in _cls(ref, path, name).body if isinstance(n, ast.FunctionDef)}


def surface(ref):
    init = _tree(ref, "__init__.py")
    out = {
        "RayStrategy": _methods(ref, "ray_ddp.py", "RayStrategy"),
        "HorovodRayStrategy": _methods(ref, "ray_horovod.py", "HorovodRayStrategy"),
        "RayLauncher": _methods(ref, "launchers/ray_launcher.py", "RayLauncher"),
        "RayExecutor": _methods(ref, "launchers/utils.py", "RayExecutor"),
        "RayHorovodLauncher": _methods(ref, "launchers/ray_horovod_launcher.py", "RayHorovodLauncher"),
        "_RayOutput_fields": [n.target.id for n in _cls(ref, "launchers/utils.py", "_RayOutput").body
                              if isinstance(n, ast.AnnAssign)],
        "__all__": next(ast.literal_eval(n.value) for n in init.body
                        if isinstance(n, ast.Assign) and n.targets[0].id == "__all__"),
    }
    for mod in ("session", "util"):
        out[mod + "_names"] = [n.name for n in _tree(ref, mod + ".py").body
                               if isinstance(n, (ast.FunctionDef, ast.ClassDef))]
    return out


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    s = surface(sys.argv[1])
    # one method (or one list) per line, so that a change of the reference reads as a small diff
    body = []
    for key in sorted(s):
        v = s[key]
        if isinstance(v, dict):
            inner = ",\n".join("  %s: %s" % (json.dumps(m), json.dumps(v[m])) for m in sorted(v))
            body.append(" %s: {\n%s\n }" % (json.dumps(key), inner))
        else:
            body.append(" %s: %s" % (json.dumps(key), json.dumps(v)))
    with open(GOLDEN, "w") as f:
        f.write("{\n" + ",\n".join(body) + "\n}\n")
    print(GOLDEN, os.path.getsize(GOLDEN))
