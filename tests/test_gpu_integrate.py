"""`GaussianRasterizer.integrate` (SURVEY.md 8f row 3) on the GPU against (1) the fixtures produced by the unmodified reference
build, (2) the CPU oracle on fresh scenes, (3) what the reference build computed on a larger load (hashed or sampled).

Tolerances as in tests/test_oracle_integrate.py: integers, radii, projected coordinates and the points-per-pixel channel
exact; float results 1e-4 (+1e-4 relative) with at most 1e-3 of the elements across an alpha threshold."""
import os
import sys

import numpy as np
import pytest
import torch

from conftest import INTEGRATE_CASES, ROOT, integrate_oracle_inputs, load_golden
from test_oracle_integrate import close_with_outliers

sys.path.insert(0, os.path.join(ROOT, "tools"))
pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NAMES = ("color", "alpha_integrated", "color_integrated", "point_coordinate", "point_sdf", "radii")


def _settings(dgr, d=None, sc=None, deg=3):
    if d is not None:
        t = lambda k: torch.from_numpy(d["in_" + k]).to(DEV)  # noqa: E731
        return dgr.GaussianRasterizationSettings(
            image_height=int(d["meta_H"]), image_width=int(d["meta_W"]), tanfovx=float(d["in_tanfov"][0]), tanfovy=float(d["in_tanfov"][1]),
            kernel_size=0.0, bg=t("bg"), scale_modifier=1.0, viewmatrix=t("viewmatrix"), projmatrix=t("projmatrix"), sh_degree=int(d["meta_deg"]),
            campos=t("campos"), prefiltered=False, require_depth=True, require_coord=True, debug=False)
    return dgr.GaussianRasterizationSettings(
        image_height=sc.height, image_width=sc.width, tanfovx=sc.tanfovx, tanfovy=sc.tanfovy, kernel_size=0.0, bg=sc.bg, scale_modifier=1.0,
        viewmatrix=sc.viewmatrix, projmatrix=sc.projmatrix, sh_degree=deg, campos=sc.campos, prefiltered=False, require_depth=True,
        require_coord=True, debug=False)


def _check(ours, ref, name):
    assert np.array_equal(ours["radii"], ref["radii"]), name
    assert np.array_equal(ours["point_coordinate"], ref["point_coordinate"]), name
    assert np.array_equal(ours["color"][8], ref["color"][8]), name
    assert not ours["color"][5].any()
    for ch in (0, 1, 2, 3, 4, 6, 7):
        close_with_outliers(ours["color"][ch], ref["color"][ch], f"{name}/color[{ch}]")
    for k in ("alpha_integrated", "color_integrated", "point_sdf"):
        close_with_outliers(ours[k], ref[k], f"{name}/{k}")
    untouched = ref["point_sdf"] == -1000.0
    assert np.array_equal(untouched, ours["point_sdf"] == -1000.0)
    assert (ours["alpha_integrated"][untouched] == 1.0).all()


@pytest.mark.parametrize("case", INTEGRATE_CASES)
def test_integrate_matches_reference_fixture(case):
    import diff_gaussian_rasterization as dgr
    d = load_golden(case)
    t = lambda k: torch.from_numpy(d["in_" + k]).to(DEV)  # noqa: E731
    M = (int(d["meta_deg"]) + 1) ** 2
    rast = dgr.GaussianRasterizer(_settings(dgr, d=d))
    out = rast.integrate(points3D=t("points3D"), means3D=t("means3D"), means2D=None, opacities=t("opacities"), shs=t("shs")[:, :M].contiguous(),
                         scales=t("scales"), rotations=t("rotations"))
    ours = {k: v.cpu().numpy() for k, v in zip(NAMES, out)}
    _check(ours, {k: d["out_" + k] for k in NAMES}, case)


def _fresh_scene(P, W, H, focal, mu, seed, PN):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from gen_golden_integrate import make_points
    from rade_gs_b200 import scenes
    sc = scenes.make_scene(P, W, H, focal, mu, seed=seed, view=scenes.look_at_view((0.3, 0.2, -0.4), (0.0, 0.1, 6.0)), bg=(0.3, 0.1, 0.2))
    return sc, make_points(sc, PN, seed + 1)


def _run_ours(sc, pts, deg=3):
    import diff_gaussian_rasterization as dgr
    scd, M = sc.to(DEV), (deg + 1) ** 2
    out = dgr.GaussianRasterizer(_settings(dgr, sc=scd, deg=deg)).integrate(
        points3D=pts.to(DEV), means3D=scd.means3D, means2D=None, opacities=scd.opacities, shs=scd.shs[:, :M].contiguous(), scales=scd.scales,
        rotations=scd.rotations)
    return {k: v.cpu().numpy() for k, v in zip(NAMES, out)}


def test_integrate_matches_oracle_on_a_fresh_scene():
    import oracle
    sc, pts = _fresh_scene(6000, 160, 112, 130.0, -2.3, 77, 30000)
    ours = _run_ours(sc, pts)
    inp = oracle.Inputs(sc.means3D.numpy(), sc.opacities.numpy(), sc.viewmatrix.numpy(), sc.projmatrix.numpy(), sc.campos.numpy(), sc.bg.numpy(),
                        sc.width, sc.height, sc.tanfovx, sc.tanfovy, sh_degree=3, kernel_size=0.0, require_coord=True, require_depth=True,
                        shs=sc.shs.numpy(), scales=sc.scales.numpy(), rotations=sc.rotations.numpy())
    ref = oracle.integrate(inp, pts.numpy())
    assert ref["overflowed"] == 0
    _check(ours, ref, "fresh")


def test_integrate_many_points_in_one_pixel_and_empty_inputs():
    """More points in a pixel than the reference's per-thread batch of 256 (it loops; we have no batch), and the fill values
    for P == 0 / PN == 0 (rasterize_points.cu:310-316,341)."""
    import diff_gaussian_rasterization as dgr
    import oracle
    sc, pts = _fresh_scene(1500, 64, 48, 60.0, -2.0, 5, 2000)
    # 700 points along one camera ray (same pixel, different depths)
    vm = sc.viewmatrix.t()
    z = torch.linspace(1.0, 9.0, 700)
    ray = torch.stack([0.013 * z, -0.021 * z, z], 1)
    pts = torch.cat([pts, (ray - vm[:3, 3]) @ vm[:3, :3]]).contiguous()
    ours = _run_ours(sc, pts)
    assert ours["color"][8].max() >= 700
    inp = oracle.Inputs(sc.means3D.numpy(), sc.opacities.numpy(), sc.viewmatrix.numpy(), sc.projmatrix.numpy(), sc.campos.numpy(), sc.bg.numpy(),
                        sc.width, sc.height, sc.tanfovx, sc.tanfovy, sh_degree=3, kernel_size=0.0, require_coord=True, require_depth=True,
                        shs=sc.shs.numpy(), scales=sc.scales.numpy(), rotations=sc.rotations.numpy())
    _check(ours, oracle.integrate(inp, pts.numpy()), "one-pixel")
    # alpha along a ray is non-decreasing in depth while the point is in front of the splats it passes (monotone occupancy)
    scd = sc.to(DEV)
    rast = dgr.GaussianRasterizer(_settings(dgr, sc=scd))
    empty_pts = torch.zeros(0, 3, device=DEV)
    o = rast.integrate(points3D=empty_pts, means3D=scd.means3D, means2D=None, opacities=scd.opacities, shs=scd.shs, scales=scd.scales,
                       rotations=scd.rotations)
    assert o[0].shape == (9, 48, 64) and not o[0].any() and o[1].numel() == 0 and not o[5].any()
    o = rast.integrate(points3D=pts.to(DEV), means3D=scd.means3D[:0], means2D=None, opacities=scd.opacities[:0], shs=scd.shs[:0],
                       scales=scd.scales[:0], rotations=scd.rotations[:0])
    assert (o[1] == 1.0).all() and (o[4] == -1000.0).all() and not o[2].any() and not o[0].any()


def reference_build_scene():
    """Mesh-extraction-like load: 50k splats, 9 points per splat (CPU tensors)."""
    from gen_golden_refbuild import one_thread
    with one_thread():
        return _fresh_scene(50_000, 400, 304, 330.0, -3.0, 9, 450_000)


def test_integrate_next_to_the_reference_build():
    """The mesh-extraction-like load against what the reference's own kernel computed on it (tests/golden/refbuild/integrate_50k.npz):
    arrays compared bit for bit through their SHA-256, the others on a fixed sample of pixels and points."""
    from gen_golden_refbuild import digest, scene_digest
    sc, pts = reference_build_scene()
    d = load_golden("refbuild/integrate_50k")
    assert scene_digest(sc, pts) == str(d["inputs_sha256"]), "the scene recipe no longer makes the fixture's inputs"
    ours = _run_ours(sc, pts)
    assert digest(ours["radii"]) == str(d["sha256_radii"])
    assert digest(ours["point_coordinate"]) == str(d["sha256_point_coordinate"])
    assert digest(ours["color"][8]) == str(d["sha256_points_per_pixel"])
    assert not ours["color"][5].any()
    color = ours["color"].reshape(9, -1)[:, d["pix"]]
    for ch in (0, 1, 2, 3, 4, 6, 7):
        close_with_outliers(color[ch], d["color"][ch], f"ref-50k/color[{ch}]")
    for k in ("alpha_integrated", "color_integrated", "point_sdf"):
        close_with_outliers(ours[k][d["pts"]], d[k], f"ref-50k/{k}")
    untouched = ours["point_sdf"] == -1000.0
    assert digest(untouched) == str(d["sha256_untouched"])
    assert (ours["alpha_integrated"][untouched] == 1.0).all()
