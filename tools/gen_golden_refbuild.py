"""Fixtures that pin the large-scene comparisons with the UNMODIFIED reference build (oracle/_ref/ref_dgr_C.so).

Must run where a GPU is:   python tools/gen_golden_refbuild.py OUT_DIR
and writes OUT_DIR/*.npz; copy them to tests/golden/refbuild/ and commit them with this script.

The scenes of these tests (BASELINE configs C1..C4 at up to 10M splats and 4096x4096, a C1 scene with a pile of splats on
one spot, a 50k-splat integrate load) are far too large to store, so a fixture keeps what the test compares, shrunk:
  * the SHA-256 of every array the test compares bit for bit (radii, sorted instance list, keys, tile ranges, ...),
  * the values at a fixed, seeded sample of pixels / points / Gaussian rows for everything compared within a tolerance,
    with the full-tensor scale the gradient check needs,
  * the SHA-256 of the inputs, so that a change of the scene recipe shows up as such rather than as a parity failure.
The tests rebuild the inputs from the same seeded recipes (tests/test_gpu_parity.py, tests/test_gpu_integrate.py), on one CPU
thread (see one_thread).
The reference's backward uses float atomics: both of its runs are stored, as grad_close_vs_reference_runs expects.
"""
from __future__ import annotations

import contextlib
import hashlib
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (os.path.join(ROOT, "rade-gs_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

RASTER_CASES = [("C1", 0.0), ("C1", 0.1), ("C2", 0.0), ("C3", 0.0), ("C4", 0.0)]
IMG_KEYS = ("color", "alpha", "depth", "mdepth", "normal", "coord", "mcoord")
SCENE_KEYS = ("means3D", "scales", "rotations", "opacities", "shs", "viewmatrix", "projmatrix", "campos", "bg")
N_PIX, N_CONTRIB, N_ROWS, N_ROWS_ANY, N_POINTS = 2048, 8192, 448, 64, 8192


@contextlib.contextmanager
def one_thread():
    """Synthesise scenes on one CPU thread.  torch splits a large elementwise op (sigmoid, exp) into one chunk per thread, and
    the scalar tail of a chunk rounds differently from its vectorised body, so on several threads the seeded inputs would
    depend on the machine's core count."""
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        yield
    finally:
        torch.set_num_threads(n)


def config_inputs(cfg):
    """BASELINE config `cfg` and the default upstream gradients, as CPU tensors: (scene, coord, depth, grads)."""
    from rade_gs_b200 import scenes
    with one_thread():
        sc, coord, depth = scenes.make_config(cfg)
        return sc, coord, depth, scenes.make_upstream_grads(sc.height, sc.width)


def raster_name(cfg, ks):
    return f"{cfg}_ks{str(ks).replace('.', '')}"


def digest(*arrays) -> str:
    """SHA-256 over the raw bytes of tensors / arrays (dtype and layout as given: callers compare like with like)."""
    h = hashlib.sha256()
    for a in arrays:
        if isinstance(a, torch.Tensor):
            a = a.detach().contiguous().cpu().numpy()
        a = np.ascontiguousarray(a)
        h.update(str(a.dtype).encode() + str(a.shape).encode())
        h.update(a.tobytes())
    return h.hexdigest()


def scene_digest(sc, *extra) -> str:
    return digest(*[getattr(sc, k) for k in SCENE_KEYS], np.array([sc.width, sc.height]), np.array([sc.tanfovx, sc.tanfovy]), *extra)


def sample(n, k, seed):
    """k distinct indices of range(n), sorted; the same for the same (n, k, seed)."""
    return np.sort(np.random.default_rng(seed).choice(n, size=min(k, n), replace=False))


def pixel_samples(f, idx, keys=IMG_KEYS):
    return {"img_" + k: f[k].reshape(f[k].shape[0], -1)[:, torch.from_numpy(idx).to(f[k].device)].cpu().numpy() for k in keys}


def gradient_rows(b, seed):
    """Rows of the gradient tensors to keep: mostly rows that received a gradient (most visible splats of these dense scenes
    receive none), plus a few uniformly drawn rows, which are mostly zero and must stay so."""
    got = torch.zeros_like(b["means2D"][:, 0], dtype=torch.bool)
    for v in b.values():
        got |= (v.reshape(v.shape[0], -1) != 0).any(1)
    live = torch.nonzero(got).squeeze(1).cpu().numpy()
    P = got.shape[0]
    rows = np.union1d(live[sample(len(live), N_ROWS, seed)], sample(P, N_ROWS_ANY, seed + 1))
    return rows


def raster_record(ref, cfg, ks, dev):
    from rade_gs_b200 import rawapi
    from tolerances import grad_close_vs_reference_runs
    sc_cpu, coord, depth, grads_cpu = config_inputs(cfg)
    sc = sc_cpu.to(dev)
    grads = {k: v.to(dev) for k, v in grads_cpu.items()}
    fr = rawapi.forward(ref, sc, coord, depth, kernel_size=ks)
    vr = rawapi.ref_views(fr, sc)
    H, W = sc.height, sc.width
    rec = {"meta_cfg": np.array(cfg), "meta_ks": np.array(ks), "inputs_sha256": np.array(scene_digest(sc_cpu, *grads_cpu.values())),
           "num_rendered": np.array(int(fr["num_rendered"])), "sha256_radii": np.array(digest(fr["radii"]))}
    for k in ("point_list", "keys", "ranges"):
        rec["sha256_" + k] = np.array(digest(vr[k]))
    rec["pix"] = sample(H * W, N_PIX, 11)
    rec.update(pixel_samples(fr, rec["pix"]))
    rec["nc_idx"] = sample(2 * H * W, N_CONTRIB, 12)
    rec["nc"] = vr["n_contrib"].reshape(-1)[torch.from_numpy(rec["nc_idx"]).to(dev)].cpu().numpy()
    del vr
    b1 = rawapi.backward(ref, sc, fr, grads)
    b2 = rawapi.backward(ref, sc, fr, grads)
    rows = gradient_rows(b1, 13)
    rec["rows"] = rows
    r = torch.from_numpy(rows).to(dev)
    for k in rawapi.BWD_KEYS:
        rec["grad1_" + k] = b1[k][r].cpu().numpy()
        rec["grad2_" + k] = b2[k][r].cpu().numpy()
        rec["scale_" + k] = np.array((0.5 * (b1[k].double() + b2[k].double())).abs().max().item() if b1[k].numel() else 0.0)
        # the sample must be a fair test of the reference against itself before it can test anything else
        grad_close_vs_reference_runs(rec["grad1_" + k], rec["grad1_" + k], rec["grad2_" + k], k, scale=float(rec["scale_" + k]))
    return rec


def pile_record(ref, dev):
    from rade_gs_b200 import rawapi
    from test_gpu_parity import pile_scene
    _, big_cpu, coord, depth = pile_scene()
    big = big_cpu.to(dev)
    fr = rawapi.forward(ref, big, coord, depth)
    vr = rawapi.ref_views(fr, big)
    rec = {"inputs_sha256": np.array(scene_digest(big_cpu)), "num_rendered": np.array(int(fr["num_rendered"]))}
    for k in ("point_list", "keys", "ranges"):
        rec["sha256_" + k] = np.array(digest(vr[k]))
    rec["pix"] = sample(big.height * big.width, N_PIX, 21)
    rec.update(pixel_samples(fr, rec["pix"]))
    return rec


def integrate_record(ref, dev):
    from gen_golden_integrate import call_reference
    from test_gpu_integrate import NAMES, reference_build_scene
    sc_cpu, pts_cpu = reference_build_scene()
    r1 = call_reference(ref, sc_cpu.to(dev), pts_cpu.to(dev), 3)
    r2 = call_reference(ref, sc_cpu.to(dev), pts_cpu.to(dev), 3)
    for k, a, b in zip(NAMES, r1[1:7], r2[1:7]):
        assert torch.equal(a, b), f"reference output {k} differs between two runs"
    out = {k: v.cpu().numpy() for k, v in zip(NAMES, r1[1:7])}
    rec = {"inputs_sha256": np.array(scene_digest(sc_cpu, pts_cpu)), "num_rendered": np.array(int(r1[0])),
           "sha256_radii": np.array(digest(out["radii"])), "sha256_point_coordinate": np.array(digest(out["point_coordinate"])),
           "sha256_points_per_pixel": np.array(digest(out["color"][8])), "sha256_untouched": np.array(digest(out["point_sdf"] == -1000.0))}
    rec["pix"] = sample(sc_cpu.height * sc_cpu.width, N_PIX, 31)
    rec["color"] = out["color"].reshape(9, -1)[:, rec["pix"]]
    rec["pts"] = sample(pts_cpu.shape[0], N_POINTS, 32)
    for k in ("alpha_integrated", "color_integrated", "point_sdf"):
        rec[k] = out[k][rec["pts"]]
    return rec


def main():
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    out_dir = sys.argv[1]
    import build_ref
    ref = build_ref.load()
    dev = torch.device("cuda:0")
    os.makedirs(out_dir, exist_ok=True)
    jobs = [(raster_name(cfg, ks), lambda cfg=cfg, ks=ks: raster_record(ref, cfg, ks, dev)) for cfg, ks in RASTER_CASES]
    jobs += [("C1_pile", lambda: pile_record(ref, dev)), ("integrate_50k", lambda: integrate_record(ref, dev))]
    for name, make in jobs:
        rec = make()
        torch.cuda.synchronize()
        path = os.path.join(out_dir, name + ".npz")
        np.savez_compressed(path, **rec)
        print(f"{name}: R={int(rec['num_rendered'])} -> {path} ({os.path.getsize(path) / 1024:.0f} KiB)", flush=True)
        assert os.path.getsize(path) < 1_000_000, path
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
