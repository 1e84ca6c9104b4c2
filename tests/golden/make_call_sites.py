"""Record how DreamScene calls the rasterizer and simple_knn, from the AST of its own sources, into
tests/golden/ref_call_sites.json (read by tests/test_reference_call_sites.py).

Only the call-site facts the drop-in contract depends on are stored: imported names, keyword names,
positional-argument counts and the names the results are unpacked into, each with its line number.

    python tests/golden/make_call_sites.py <DreamScene checkout>
"""
import ast
import json
import os
import sys


def _name(f):
    return f.id if isinstance(f, ast.Name) else (f.attr if isinstance(f, ast.Attribute) else None)


def _call(n):
    return {"line": n.lineno, "n_args": len(n.args), "keywords": [k.arg for k in n.keywords]}


def rasterizer_sites(src):
    """scene_gaussian.py: the import of diff_gaussian_rasterization, every GaussianRasterizationSettings(...),
    GaussianRasterizer(...) and rasterizer(...) call, and every tuple the rasterizer's results are unpacked into."""
    tree = ast.parse(src)
    out = {"imports": [], "settings": [], "ctor": [], "call": [], "unpack": []}
    for n in ast.walk(tree):
        if isinstance(n, ast.ImportFrom) and n.module == "diff_gaussian_rasterization":
            out["imports"] += [a.name for a in n.names]
        elif isinstance(n, ast.Call):
            key = {"GaussianRasterizationSettings": "settings", "GaussianRasterizer": "ctor",
                   "rasterizer": "call"}.get(_name(n.func))
            if key:
                out[key].append(_call(n))
        if isinstance(n, ast.Assign) and isinstance(n.value, ast.Call):
            f = n.value.func
            if isinstance(f, ast.Name) and f.id == "rasterizer" and isinstance(n.targets[0], ast.Tuple):
                out["unpack"].append({"line": n.lineno, "targets": [getattr(e, "id", None) for e in n.targets[0].elts]})
    for k in ("settings", "ctor", "call", "unpack"):
        out[k].sort(key=lambda d: d["line"])
    return out


def knn_sites(src):
    """gs_renderer.py: the import from simple_knn._C and every distCUDA2(...) call."""
    tree = ast.parse(src)
    imports = [n for n in ast.walk(tree) if isinstance(n, ast.ImportFrom) and n.module == "simple_knn._C"]
    calls = [n for n in ast.walk(tree) if isinstance(n, ast.Call) and isinstance(n.func, ast.Name)
             and n.func.id == "distCUDA2"]
    return {"imports": [[a.name for a in n.names] for n in imports],
            "call": sorted((_call(n) for n in calls), key=lambda d: d["line"])}


def main(ref):
    out = {"scene_gaussian.py": rasterizer_sites(open(os.path.join(ref, "scene_gaussian.py")).read()),
           "gs_renderer.py": knn_sites(open(os.path.join(ref, "gs_renderer.py")).read())}
    dst = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_call_sites.json")
    with open(dst, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("wrote", dst)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
