"""Writes ``tests/golden/reference_api_surface.json``: the public module-level names of the reference's packages
(long-context-attention / yunchang) that ``tests/test_api_surface_cpu.py`` requires under the same names here.
The reference tree is parsed, never imported.

    python tools/reference_api_surface.py <path to long-context-attention checkout>
"""
import ast
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_api_surface.json")
PACKAGES = ["yunchang", "yunchang.ring", "yunchang.hybrid", "yunchang.ulysses", "yunchang.comm", "yunchang.kernels",
            "yunchang.globals"]


def module_level_names(path):
    names = set()
    def visit(body):
        for n in body:
            if isinstance(n, ast.ImportFrom):
                names.update(a.asname or a.name for a in n.names)
            elif isinstance(n, (ast.FunctionDef, ast.ClassDef)):
                names.add(n.name)
            elif isinstance(n, ast.Assign):
                names.update(t.id for t in n.targets if isinstance(t, ast.Name))
            elif isinstance(n, (ast.Try, ast.If)):          # guarded optional imports
                visit(n.body)
                for h in getattr(n, "handlers", []):
                    visit(h.body)
                visit(n.orelse)
    visit(ast.parse(open(path).read()).body)
    return {n for n in names if not n.startswith("_") and n != "*"}


def public_defs(path):
    tree = ast.parse(open(path).read())
    return {n.name for n in tree.body if isinstance(n, (ast.FunctionDef, ast.ClassDef)) and not n.name.startswith("_")}


def read_reference(ref):
    """``packages``: every public module-level name of each package / ``globals`` module (imports included);
    ``modules``: the public top-level functions and classes of every other module."""
    packages = {}
    for mod in PACKAGES:
        rel = mod.replace(".", "/")
        path = os.path.join(ref, rel, "__init__.py") if os.path.isdir(os.path.join(ref, rel)) else os.path.join(ref, rel + ".py")
        packages[mod] = sorted(module_level_names(path))
    modules = {}
    for d, _, files in os.walk(os.path.join(ref, "yunchang")):
        for f in files:
            if f.endswith(".py") and f != "__init__.py":
                path = os.path.join(d, f)
                modules[os.path.relpath(path, ref)[:-3].replace(os.sep, ".")] = sorted(public_defs(path))
    return {"packages": packages, "modules": dict(sorted(modules.items()))}


if __name__ == "__main__":
    with open(GOLDEN, "w") as f:
        json.dump(read_reference(sys.argv[1]), f, indent=1)
        f.write("\n")
