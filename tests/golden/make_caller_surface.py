#!/usr/bin/env python
"""Extracts, from the reference's own caller (datagen/generate.py of a namanxkumar/fea-diffusion
checkout), every use it makes of the classes the drop-in replaces: constructor keywords, methods
with their positional counts and keywords, attributes read.  The result is committed as
tests/golden/caller_surface.json so that the GPU box (which has no reference checkout) can check
the drop-in against it; tests/test_caller_surface.py re-derives it when the checkout is present.

    python tests/golden/make_caller_surface.py <reference checkout> > tests/golden/caller_surface.json
"""
import ast
import json
import sys


def surface(source: str) -> dict:
    tree = ast.parse(source)
    out = {"imports": {}, "FEAnalysis": {"init": None, "methods": {}, "attributes": []},
           "MeshGenerator": {"init": None, "methods": {}, "attributes": []}, "functions": {}}
    var_class = {}
    for node in ast.walk(tree):
        if isinstance(node, ast.ImportFrom) and node.level == 1:
            out["imports"][node.module] = sorted(a.name for a in node.names)
        if isinstance(node, ast.Assign) and isinstance(node.value, ast.Call) and isinstance(node.value.func, ast.Name) \
                and node.value.func.id in ("FEAnalysis", "MeshGenerator"):
            for t in node.targets:
                if isinstance(t, ast.Name):
                    var_class[t.id] = node.value.func.id

    def call_sig(c):
        return {"n_pos": len(c.args), "keywords": sorted(k.arg for k in c.keywords if k.arg)}

    def merge(d, name, sig):
        old = d.get(name)
        if old is None:
            d[name] = sig
        else:
            old["n_pos"] = max(old["n_pos"], sig["n_pos"])
            old["keywords"] = sorted(set(old["keywords"]) | set(sig["keywords"]))

    called_attrs = set()
    for node in ast.walk(tree):
        if isinstance(node, ast.Call):
            f = node.func
            if isinstance(f, ast.Name) and f.id in ("FEAnalysis", "MeshGenerator"):
                sig = call_sig(node)
                cur = out[f.id]["init"]
                out[f.id]["init"] = sig if cur is None else {"n_pos": max(cur["n_pos"], sig["n_pos"]),
                                                             "keywords": sorted(set(cur["keywords"]) | set(sig["keywords"]))}
            elif isinstance(f, ast.Name) and f.id in ("find_image_bounds", "verify_directory"):
                merge(out["functions"], f.id, call_sig(node))
            elif isinstance(f, ast.Attribute) and isinstance(f.value, ast.Name) and f.value.id in var_class:
                merge(out[var_class[f.value.id]]["methods"], f.attr, call_sig(node))
                called_attrs.add(id(f))
    for node in ast.walk(tree):
        if isinstance(node, ast.Attribute) and isinstance(node.value, ast.Name) and node.value.id in var_class \
                and id(node) not in called_attrs:
            a = out[var_class[node.value.id]]["attributes"]
            if node.attr not in a:
                a.append(node.attr)
    for k in ("FEAnalysis", "MeshGenerator"):
        out[k]["attributes"].sort()
    return out


if __name__ == "__main__":
    root = sys.argv[1]
    with open(root + "/datagen/generate.py") as f:
        print(json.dumps(surface(f.read()), indent=1, sort_keys=True))
