"""Static drop-in check against the reference's own caller, `gaussian_renderer.render()` (reference
gaussian_renderer/__init__.py:19-95): every name it imports from `diff_gaussian_rasterization`, every keyword it passes to
`GaussianRasterizationSettings(...)` and to `rasterizer(...)`, and the 8-tuple it unpacks must exist in this repo's package.
The call sites are recorded in tests/golden/render_call_sites.json (tools/gen_golden_render_calls.py)."""
import inspect
import json
import os

from conftest import GOLDEN_DIR


def test_render_call_sites_fit_our_package():
    import diff_gaussian_rasterization as dgr
    with open(os.path.join(GOLDEN_DIR, "render_call_sites.json")) as f:
        sites = json.load(f)
    imported = sites["imports"]
    assert imported and all(hasattr(dgr, name) for name in imported), imported
    fields = set(dgr.GaussianRasterizationSettings._fields)
    fwd_params = set(inspect.signature(dgr.GaussianRasterizer.forward).parameters) - {"self"}
    integ_params = set(inspect.signature(dgr.GaussianRasterizer.integrate).parameters) - {"self"}
    for kws in map(set, sites["settings_calls"]):
        assert kws <= fields, kws - fields
        assert fields - kws == set() or kws, "render() must be able to build the settings tuple"
    for kws in map(set, sites["rasterizer_calls"]):
        assert kws <= fwd_params, kws - fwd_params
    for kws in map(set, sites["integrate_calls"]):
        assert kws <= integ_params, kws - integ_params
    assert len(sites["settings_calls"]) >= 1 and len(sites["rasterizer_calls"]) >= 1
    # render() unpacks 8 outputs from the rasterizer call (reference :71)
    assert sites["rasterizer_unpack"] and sites["rasterizer_unpack"][0] == 8
