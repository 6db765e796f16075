"""Generates tests/golden/reference_signatures.json. Run with a checkout of the reference:

    python tests/golden/make_signature_golden.py <reference checkout>

Parameter names, order and default values of the reference's public Python surface, read with `ast` from
multimodars/_processing.py, multimodars/_converters.py (functions) and multimodars/multimodars.pyi (classes, methods,
properties) — the names a user's code depends on. tests/test_signatures_cpu.py holds this package against it."""
import ast
import json
import sys
from pathlib import Path

REF = Path(sys.argv[1]) / "multimodars"
OUT = Path(__file__).resolve().parent / "reference_signatures.json"


def params(fn):
    a = fn.args
    pos = [x.arg for x in a.posonlyargs + a.args]
    defaults = [None] * (len(pos) - len(a.defaults)) + [ast.unparse(d) for d in a.defaults]
    out = [[n, d] for n, d in zip(pos, defaults) if n not in ("self", "cls")]
    out += [[x.arg, ast.unparse(d) if d is not None else None] for x, d in zip(a.kwonlyargs, a.kw_defaults)]
    return out


sig = {"functions": {}, "classes": {}}
for mod in ("_processing", "_converters"):
    for node in ast.parse((REF / f"{mod}.py").read_text()).body:
        if isinstance(node, ast.FunctionDef) and not node.name.startswith("_"):
            sig["functions"][node.name] = {"module": mod, "params": params(node)}
for node in ast.parse((REF / "multimodars.pyi").read_text()).body:
    if isinstance(node, ast.ClassDef):
        c = {"methods": {}, "properties": [], "attributes": []}
        for it in node.body:
            if isinstance(it, ast.FunctionDef):
                decos = [ast.unparse(d) for d in it.decorator_list]
                if "property" in decos:
                    c["properties"].append(it.name)
                elif not any(d.endswith(".setter") for d in decos):
                    c["methods"][it.name] = {"params": params(it), "static": "staticmethod" in decos}
            elif isinstance(it, ast.AnnAssign) and isinstance(it.target, ast.Name):
                c["attributes"].append(it.target.id)
        sig["classes"][node.name] = c
OUT.write_text(json.dumps(sig, indent=1, sort_keys=True) + "\n")
print(len(sig["functions"]), "functions,", len(sig["classes"]), "classes")
