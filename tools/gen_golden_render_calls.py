"""Record how the reference's own caller, `gaussian_renderer.render()` (reference gaussian_renderer/__init__.py), uses
`diff_gaussian_rasterization`: the names it imports, the keywords of every `GaussianRasterizationSettings(...)`,
`rasterizer(...)` and `.integrate(...)` call, and how many outputs it unpacks from `rasterizer(...)`.

    python tools/gen_golden_render_calls.py REFERENCE_CHECKOUT > tests/golden/render_call_sites.json

tests/test_dropin_static.py checks this package against the recorded call sites.
"""
from __future__ import annotations

import ast
import json
import os
import sys


def call_sites(source: str) -> dict:
    tree = ast.parse(source)
    rec = {"imports": [a.name for n in ast.walk(tree) if isinstance(n, ast.ImportFrom) and n.module == "diff_gaussian_rasterization" for a in n.names],
           "settings_calls": [], "rasterizer_calls": [], "integrate_calls": [], "rasterizer_unpack": []}
    for node in ast.walk(tree):
        if isinstance(node, ast.Call) and isinstance(node.func, ast.Name) and node.func.id == "GaussianRasterizationSettings":
            rec["settings_calls"].append(sorted(k.arg for k in node.keywords))
        if isinstance(node, ast.Call) and isinstance(node.func, ast.Name) and node.func.id == "rasterizer":
            rec["rasterizer_calls"].append(sorted(k.arg for k in node.keywords))
        if isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute) and node.func.attr == "integrate":
            rec["integrate_calls"].append(sorted(k.arg for k in node.keywords))
        if (isinstance(node, ast.Assign) and isinstance(node.targets[0], ast.Tuple) and isinstance(node.value, ast.Call)
                and isinstance(node.value.func, ast.Name) and node.value.func.id == "rasterizer"):
            rec["rasterizer_unpack"].append(len(node.targets[0].elts))
    return rec


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    with open(os.path.join(sys.argv[1], "gaussian_renderer", "__init__.py")) as f:
        print(json.dumps(call_sites(f.read()), indent=1))
