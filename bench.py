#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 rasterizer (BASELINE.json: Mpix/s fwd+bwd @ 1M splats, 1600x1200).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config C2] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step is one pass of the hot path over one synthetic camera: `_C.rasterize_gaussians` followed by
`_C.rasterize_gaussians_backward` with fixed upstream gradients (SURVEY.md 8d).  Prints ONE JSON line (rank 0).

Protocol (SURVEY.md 8d: median of >= 20 timed iterations after >= 5 warm-ups; the defaults):
  * each measured quantity is timed over EXACTLY `--steps` iterations, bracketed by barrier + torch.cuda.synchronize() on both
    sides, with a CUDA event between consecutive iterations (on the launching stream); per iteration the time is the MAX over ranks;
  * `ms_per_step` = MEDIAN of the per-iteration times, `value` = W*H / that; min / median / max are in `timing` so a perturbed
    iteration is visible instead of being averaged in;
  * SM clocks / throttle reasons are sampled by a separate PROCESS (NVML, no GIL contention with the timed loop) that
    runs during every timed phase of the run.
  value        inputs resident in HBM
  e2e          same metric through the public autograd API (`GaussianRasterizer`, what render() calls) with the
               step's host inputs -- camera matrices and the 8-bit ground-truth image -- copied from pinned host
               memory inside the timed region and the loss read back to the host every step; same protocol
  roofline     dominant kernel (backward render): algorithmic bytes (SURVEY.md 8d) / its average launch duration,
               measured live with CUDA events the library records on the launching stream; `traffic` and the
               instruction count behind `roofline_issue` are REPLAYED from the committed ncu capture (labelled so)
  cpu_baseline the CPU oracle port (oracle/oracle.c, 1 thread) on a bounded sample of the same workload, plus the
               pure-torch config[0] plumbing timing -- reported, not a target
`--impl reference` times the reference's own CUDA rasterizer (oracle/_ref/ref_dgr_C.so, built from /root/reference
by oracle/build_ref.py) on the same config through the same harness: the reference has NO CPU implementation of
this path (BASELINE.md section 2), so its arm runs where it can -- on the GPU (see DESIGN.md "Measurement").  That arm
never imports the product's extension modules.
N > 1: tile rows of the one image are sharded over the ranks (strong scaling); the screen-space gradient rows are
exchanged once per backward.
`--dump-outputs DIR` writes, after the timed steps, what the last timed step of the resident path returned to its caller
(see dump_outputs); the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(ROOT, "rade-gs_b200"), os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

METRIC = "Mpix/s fwd+bwd @1M splats 1600x1200"
SM_COUNT = 148


# ---- clocks ----------------------------------------------------------------------------------------------------

_SAMPLER_SRC = r"""
import sys, time
idx, path = int(sys.argv[1]), sys.argv[2]
import pynvml as n
n.nvmlInit()
h = n.nvmlDeviceGetHandleByIndex(idx)
get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons")
mx = n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)
with open(path, "w", buffering=1) as f:
    f.write("nvml\n")
    while True:
        try:
            pw = n.nvmlDeviceGetPowerUsage(h) / 1000.0
        except Exception:
            pw = 0.0
        f.write("%d,%d,%.1f,%d\n" % (n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM), mx, pw, int(get(h))))
        time.sleep(0.01)
"""


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed regions by a separate process (B200_PROFILING.md 'clocks'
    line): NVML every 10 ms in a helper python process; `nvidia-smi -lms` as the fallback.  Nothing of it runs in this
    process, so the timed loop does not share the GIL with it."""
    REASON_BITS = (("sw_power_cap", 0x4), ("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        phys = index
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        if vis and all(v.strip().isdigit() for v in vis.split(",")) and index < len(vis.split(",")):
            phys = int(vis.split(",")[index])
        self.index, self.proc, self.source = phys, None, None
        fd, self.path = tempfile.mkstemp(prefix="rgs_clocks_", suffix=".csv")
        os.close(fd)

    def __enter__(self):
        try:
            self.proc = subprocess.Popen([sys.executable, "-c", _SAMPLER_SRC, str(self.index), self.path], stdout=subprocess.DEVNULL,
                                         stderr=subprocess.DEVNULL)
            t0 = time.time()
            while time.time() - t0 < 10.0 and self.proc.poll() is None and os.path.getsize(self.path) == 0:
                time.sleep(0.02)
            if self.proc.poll() is not None or os.path.getsize(self.path) == 0:
                raise RuntimeError("nvml sampler did not start")
            self.source = "nvml (separate process, 10 ms)"
        except Exception:
            if self.proc is not None and self.proc.poll() is None:
                self.proc.kill()
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
            self.source = "nvidia-smi -lms 50 (separate process)"
        return self

    def __exit__(self, *a):
        if self.proc is not None and self.proc.poll() is None:
            self.proc.terminate()           # the exact PID we started
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons, n = [], [], set(), 0
        try:
            for ln in open(self.path):
                c = [x.strip() for x in ln.strip().split(",")]
                if len(c) < 4 or not c[0].replace(".", "").isdigit():
                    continue
                n += 1
                sm.append(float(c[0]))
                mx.append(float(c[1]))
                if len(c) == 4:     # nvml helper: bit mask
                    bits = int(c[3])
                    reasons |= {name for name, mask in self.REASON_BITS if bits & mask}
                else:               # nvidia-smi: Active / Not Active columns
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[3:7]):
                        if v.lower().startswith("active"):
                            reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_min_mhz": min(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": n, "source": self.source}


# ---- implementations under test ----------------------------------------------------------------------------------

def load_impl(name):
    if name == "ours":
        import diff_gaussian_rasterization as dgr
        return dgr._C
    import build_ref
    return build_ref.load()


class _RefFunction(torch.autograd.Function):
    """Autograd adapter around a reference-style `_C` (same call sequence as the reference's Python wrapper,
    diff_gaussian_rasterization/__init__.py:44-169); used for the reference arm's e2e number."""

    @staticmethod
    def forward(ctx, C, sc, coord, depth, ks, means3D, means2D, sh, opac, scales, rots):
        E = torch.Tensor([])
        out = C.rasterize_gaussians(sc["bg"], means3D, E, opac, scales, rots, 1.0, E, sc["view"], sc["proj"], sc["tanx"], sc["tany"], ks,
                                    sc["H"], sc["W"], sh, 3, sc["campos"], False, coord, depth, False)
        n, color, co, mco, alpha, normal, dep, mdep, radii, gb, bb, ib = out
        ctx.C, ctx.sc, ctx.coord, ctx.depth, ctx.ks, ctx.n = C, sc, coord, depth, ks, n
        ctx.save_for_backward(means3D, scales, rots, normal, radii, sh, gb, bb, ib, alpha)
        return color, radii, co, mco, dep, mdep, alpha, normal

    @staticmethod
    def backward(ctx, g_color, g_radii, g_co, g_mco, g_dep, g_mdep, g_alpha, g_normal):
        means3D, scales, rots, normal, radii, sh, gb, bb, ib, alpha = ctx.saved_tensors
        sc, E = ctx.sc, torch.Tensor([])
        g = ctx.C.rasterize_gaussians_backward(sc["bg"], means3D, radii, E, scales, rots, 1.0, E, sc["view"], sc["proj"], sc["tanx"], sc["tany"], ctx.ks,
                                               g_color, g_co, g_mco, g_dep, g_mdep, g_alpha, g_normal, normal, sh, 3, sc["campos"], gb, ctx.n, bb, ib,
                                               alpha, ctx.coord, ctx.depth, False)
        g_means2D, g_colors, g_opac, g_means3D, g_cov, g_sh, g_scales, g_rots = g
        return None, None, None, None, None, g_means3D, g_means2D, g_sh, g_opac, g_scales, g_rots


def cpu_baseline():
    """Bounded CPU work (about 10-20 s): the oracle port on a C2-density sample + config[0] torch plumbing."""
    import oracle
    from rade_gs_b200 import scenes
    Wd, Hd, P = 400, 300, 62_500   # 1/16 of C2's pixels and splats, same focal-per-pixel density (f scaled by 1/4)
    sc = scenes.make_scene(P, Wd, Hd, 350.0, -4.6, seed=1234)
    g = scenes.make_upstream_grads(Hd, Wd, seed=4321)
    inp = oracle.Inputs(sc.means3D.numpy(), sc.opacities.numpy(), sc.viewmatrix.numpy(), sc.projmatrix.numpy(), sc.campos.numpy(), sc.bg.numpy(),
                        Wd, Hd, sc.tanfovx, sc.tanfovy, shs=sc.shs.numpy(), scales=sc.scales.numpy(), rotations=sc.rotations.numpy(), sh_degree=3,
                        require_depth=True)
    oracle.lib()
    t0 = time.perf_counter()
    reps = 0
    while True:
        f = oracle.forward(inp)
        oracle.backward(inp, f, {k: v.numpy() for k, v in g.items()})
        reps += 1
        if time.perf_counter() - t0 > 10.0 or reps >= 50:
            break
    dt = (time.perf_counter() - t0) / reps
    res = {"value": Wd * Hd / dt / 1e6, "unit": "Mpix/s", "cores": 1, "kind": "port",
           "sample": f"oracle/oracle.c fwd+bwd, {P} splats {Wd}x{Hd} (C2 scaled 1/16: same splats per pixel), {reps} reps, R={f['num_rendered']}"}
    # config[0]: 1k Gaussians, torch-CPU cov3D (L L^T) + SH degree-0 colour + projection (plumbing only)
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    s0 = scenes.make_scene(1000, 1600, 1200, 1400.0, -4.6)
    t0 = time.perf_counter()
    n0 = 200
    for _ in range(n0):
        r, x, y, z = s0.rotations.unbind(1)
        R = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y), 2 * (x * y + r * z), 1 - 2 * (x * x + z * z),
                         2 * (y * z - r * x), 2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)], 1).view(-1, 3, 3)
        L = R * s0.scales[:, None, :]
        cov = L @ L.transpose(1, 2)
        col = (0.28209479177387814 * s0.shs[:, 0] + 0.5).clamp_min(0)
        ph = torch.cat([s0.means3D, torch.ones(1000, 1)], 1) @ s0.projmatrix
        ndc = ph[:, :3] / (ph[:, 3:] + 1e-7)
        _ = cov.sum() + col.sum() + ndc.sum()
    res["config0_torch_cpu"] = {"us_per_call": (time.perf_counter() - t0) / n0 * 1e6, "threads": torch.get_num_threads(),
                                "what": "1k Gaussians: cov3D + SH deg-0 + projection in pure torch on CPU"}
    return res


# SURVEY.md 8d per-variant constants: (A_v gather bytes per instance, O_v fwd bytes per pixel, I_v bwd bytes per pixel, G_v grad floats per Gaussian)
VARIANT_BYTES = {(False, False): (36, 24, 28, 10), (False, True): (60, 52, 68, 16), (True, False): (84, 76, 92, 22), (True, True): (96, 88, 104, 25)}


def algorithmic_bytes(P, Pv, R, N, T, M, coord, depth):
    """SURVEY.md 8d, per stage, for one step."""
    A, O, I, G = VARIANT_BYTES[(coord, depth)]
    tiles_bits = max(1, math.ceil(math.log2(max(T, 2))))
    sort = math.ceil((32 + tiles_bits) / 8) * 2 * 12 * R
    return {
        "preprocess_forward": P * (44 + 12 * M + 4) + Pv * (A + 35),
        "binning": 8 * P + 12 * R + sort,
        "render_forward": R * (A + 4) + N * O + 8 * T,
        "render_backward": R * (A + 4) + N * I + 8 * T + 4 * G * Pv,
        "preprocess_backward": Pv * (12 + 24 + 28 + 4 * G + 12 * M + 12 * M + 12 + 12 + 16 + 24),
    }


DUMP_PIXELS, DUMP_ROWS = 1 << 18, 1 << 16   # 15 image channels and 72 floats per Gaussian row: about 37 MB with the indices


def dump_outputs(out_dir, fwd, grads, H, W, P):
    """Write what one step of the resident path returned to its caller as out_dir/<name>.npy (float32; float64 for counts and
    indices): the image maps (`color`, `alpha`, `depth`, ... as [C, pixels]), `radii` and `grad_<name>` for each gradient tensor.
    Larger outputs are sampled: the same seeded DUMP_PIXELS pixels and DUMP_ROWS Gaussian rows every run, whose flat indices
    are written as `pixel_index` and `row_index`.  The private state buffers are left out: their layout is the build's own."""
    import numpy as np

    def pick(n, k, seed):
        return np.arange(n) if n <= k else np.sort(np.random.default_rng(seed).choice(n, size=k, replace=False))

    pix, rows = pick(H * W, DUMP_PIXELS, 1), pick(P, DUMP_ROWS, 2)
    out = {"num_rendered": np.array(int(fwd["num_rendered"]), np.float64), "pixel_index": pix.astype(np.float64), "row_index": rows.astype(np.float64)}
    for k in ("color", "coord", "mcoord", "alpha", "normal", "depth", "mdepth"):
        if k in fwd:
            t = fwd[k]
            out[k] = t.reshape(t.shape[0], -1)[:, torch.from_numpy(pix).to(t.device)].float().cpu().numpy()
    per_row = {"radii": fwd["radii"]} if "radii" in fwd else {}
    per_row.update({"grad_" + k: v for k, v in grads.items()})
    for k, t in per_row.items():
        out[k] = (t[torch.from_numpy(rows).to(t.device)] if t.shape[0] == P else t).float().cpu().numpy()
    assert sum(v.nbytes for v in out.values()) <= 64 << 20
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    a = ap.parse_args()
    a.warmup = max(a.warmup, 3)
    a.steps = max(a.steps, 1)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference" and rank != 0:
        return  # single-GPU reference: rank 0 alone runs it
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the rasterizer has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    ours = a.impl == "ours"
    multi = world > 1 and ours
    if multi:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"   # keep NCCL's version banner off stdout: rank 0 prints exactly one JSON line
        dist.init_process_group("nccl", device_id=dev)

    from rade_gs_b200 import rawapi, scenes   # pure-Python helpers (scene synthesis, the two raw _C calls): no extension is loaded by them
    C = load_impl(a.impl)
    dgr = multigpu = None
    if ours:
        import diff_gaussian_rasterization as dgr
        from rade_gs_b200 import multigpu
    sc_cpu, coord, depth = scenes.make_config(a.config)
    sc = sc_cpu.to(dev)
    if multi:
        sc = multigpu.broadcast_scene_(sc)   # replicated model state: rank 0's bits everywhere
    W, H, P = sc.width, sc.height, sc.means3D.shape[0]
    grads = scenes.make_upstream_grads(H, W, device=dev)
    grid_y = (H + 15) // 16
    tiles = ((W + 15) // 16) * grid_y
    slab = multigpu.partition_tile_rows(grid_y, world)[rank] if multi else (0, grid_y)
    E = torch.Tensor([])
    exchange = multigpu.GradExchange(P, C.grad_stride(coord, depth), dev) if multi else None
    # multi-GPU: the maps are compact ([C, slab rows, W]); the upstream gradients of a rank are the rows of its slab
    sgrads = {k: v[:, min(slab[0] * 16, H):min(slab[1] * 16, H)].contiguous() for k, v in grads.items()} if multi else grads

    def step_resident():
        if not multi:
            f = rawapi.forward(C, sc, coord, depth)
            return f, rawapi.backward(C, sc, f, grads)
        out = C.rasterize_gaussians_slab(sc.bg, sc.means3D, E, sc.opacities, sc.scales, sc.rotations, 1.0, E, sc.viewmatrix, sc.projmatrix,
                                         sc.tanfovx, sc.tanfovy, 0.0, H, W, sc.shs, 3, sc.campos, False, coord, depth, False, slab[0], slab[1], True)
        acc = exchange.backward_render(C, sc.bg, sc.means3D, out[8], E, sc.scales, sc.rotations, 1.0, E, sc.viewmatrix, sc.projmatrix,
                                       sc.tanfovx, sc.tanfovy, 0.0, sgrads["color"], sgrads["coord"], sgrads["mcoord"], sgrads["depth"],
                                       sgrads["mdepth"], sgrads["alpha"], sgrads["normal"], out[5], sc.shs, 3, sc.campos, out[9], out[0],
                                       out[10], out[11], out[4], coord, depth, False, slab[0], slab[1], True, H)
        g = C.rasterize_gaussians_backward_preprocess(acc, sc.bg, sc.means3D, out[8], E, sc.opacities, sc.scales, sc.rotations, 1.0, E, sc.viewmatrix,
                                                      sc.projmatrix, sc.tanfovx, sc.tanfovy, 0.0, H, W, sc.shs, 3, sc.campos, out[9], coord, depth, False)
        return {"num_rendered": out[0]}, dict(zip(rawapi.BWD_KEYS, g))

    def barrier():
        if multi:
            dist.barrier()
        torch.cuda.synchronize()

    def measure(fn):
        """Exactly --steps iterations (barrier + synchronize on both sides, CUDA events between iterations on the launching
        stream, max over ranks per iteration); returns their statistics and what the last one returned."""
        fn()                      # one more untimed step: the first call after a phase change pays one-off allocator / event set-up
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(a.steps + 1)]
        barrier()
        ev[0].record()
        for i in range(a.steps):
            last = fn()
            ev[i + 1].record()
        barrier()
        t = torch.tensor([ev[i].elapsed_time(ev[i + 1]) for i in range(a.steps)] + [ev[0].elapsed_time(ev[a.steps])], device=dev, dtype=torch.float64)
        if multi:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t = t.tolist()
        iters = t[:-1]
        return {"ms": statistics.median(iters), "min_ms": min(iters), "max_ms": max(iters), "iterations": len(iters), "timed_s": t[-1] * 1e-3}, last

    import contextlib
    with (ClockSampler(local) if rank == 0 else contextlib.nullcontext()) as clk:
        # ---- resident-input number ----
        for _ in range(a.warmup):
            last = step_resident()
        launches0 = C.launch_count() if ours else 0
        t_res, last = measure(step_resident)
        launches = (C.launch_count() - launches0) if ours else None
        ms_per_step = t_res["ms"]
        value = W * H / (ms_per_step * 1e-3) / 1e6
        R = int(last[0]["num_rendered"])
        if a.dump_outputs and rank == 0:
            dump_outputs(a.dump_outputs, *last, H, W, P)
        del last

        # ---- end-to-end number: public autograd API, host inputs copied in, loss copied out ----
        # Host inputs of one training step, as train.py has them: the camera (matrices, position, background) and the
        # ground-truth photograph, 8 bits per channel like every dataset the reference reads (PNG/JPEG).  Depth / normal
        # supervision in RaDe-GS is self-consistency between rendered maps, so no ground truth is shipped for them.
        r0, r1 = min(slab[0] * 16, H), min(slab[1] * 16, H)
        # multi-GPU: a rank's loss needs the ground-truth rows of its own slab only, so that is what it copies in
        host = {"view": sc_cpu.viewmatrix.pin_memory(), "proj": sc_cpu.projmatrix.pin_memory(), "campos": sc_cpu.campos.pin_memory(),
                "bg": sc_cpu.bg.pin_memory(),
                "gt_color": (torch.rand(3, H, W, generator=torch.Generator().manual_seed(5678)) * 255).to(torch.uint8)[:, r0:r1].contiguous().pin_memory()}
        h2d = sum(v.numel() * v.element_size() for v in host.values())
        dbuf = {k: torch.empty_like(v, device=dev) for k, v in host.items()}
        leaves = {k: getattr(sc, k).clone().requires_grad_(True) for k in ("means3D", "scales", "rotations", "opacities", "shs")}
        copy_stream = torch.cuda.Stream(device=dev)

        def step_e2e():
            for k in ("view", "proj", "campos", "bg"):                 # camera: needed by forward, current stream
                dbuf[k].copy_(host[k], non_blocking=True)
            copy_stream.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(copy_stream):                        # ground truth: needed by the loss only -> overlaps forward
                dbuf["gt_color"].copy_(host["gt_color"], non_blocking=True)
            for t in leaves.values():
                t.grad = None
            means2D = torch.zeros_like(leaves["means3D"], requires_grad=True)
            if ours:
                st = dgr.GaussianRasterizationSettings(H, W, sc.tanfovx, sc.tanfovy, 0.0, dbuf["bg"], 1.0, dbuf["view"], dbuf["proj"], 3, dbuf["campos"],
                                                       False, depth, coord, False)
                rast = multigpu.ShardedGaussianRasterizer(st, rank=rank, world_size=world, exchange=exchange, compact=True) if multi else dgr.GaussianRasterizer(st)
                color, radii, co, mco, dep, mdep, alpha, normal = rast(leaves["means3D"], means2D, leaves["opacities"], shs=leaves["shs"],
                                                                        scales=leaves["scales"], rotations=leaves["rotations"])
            else:
                scd = {"bg": dbuf["bg"], "view": dbuf["view"], "proj": dbuf["proj"], "campos": dbuf["campos"], "tanx": sc.tanfovx, "tany": sc.tanfovy,
                       "H": H, "W": W}
                color, radii, co, mco, dep, mdep, alpha, normal = _RefFunction.apply(C, scd, coord, depth, 0.0, leaves["means3D"], means2D, leaves["shs"],
                                                                                     leaves["opacities"], leaves["scales"], leaves["rotations"])
            torch.cuda.current_stream().wait_stream(copy_stream)
            sl = slice(0, r1 - r0) if multi else slice(r0, r1)   # compact maps start at the slab's first row
            gsl = slice(0, r1 - r0)                                 # the ground truth held on the device is this rank's rows
            # photometric L1 against the 8-bit ground truth + small regularisers that keep the depth / normal / alpha gradient
            # paths live (stand-ins for train.py's depth-normal consistency terms, which also need no ground truth)
            loss = (color[:, sl] - dbuf["gt_color"][:, gsl].float() * (1.0 / 255.0)).abs().mean() + 0.01 * alpha[:, sl].mean()
            if depth:
                loss = loss + 0.05 * dep[:, sl].mean()
            if coord:
                loss = loss + 0.05 * co[2, sl].mean()
            if depth or coord:
                loss = loss + 0.05 * (1 - normal[2, sl]).mean()
            loss.backward()
            return float(loss.item())                                   # D2H read of the step's result

        for _ in range(a.warmup):
            step_e2e()
        t_e2e, _ = measure(step_e2e)
        e2e_value = W * H / (t_e2e["ms"] * 1e-3) / 1e6
    clocks = clk.summary() if clk is not None else {}

    # ---- per-stage device times (separate pass, events recorded by the library on the launching stream) ----
    roofline = roofline_issue = stages = step_hbm = None
    if ours and hasattr(C, "stage_timing"):
        C.stage_timing(True)
        for _ in range(a.steps):
            step_resident()
        torch.cuda.synchronize()
        stages = C.stage_times()          # {name: (total_ms, launches)}
        C.stage_timing(False)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_source = "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        if not multi:
            Pv = int((rawapi.forward(C, sc, coord, depth)["radii"] > 0).sum().item())
            alg = algorithmic_bytes(P, Pv, R, W * H, tiles, 16, coord, depth)
            stage_of = {"preprocess_forward": "preprocess_forward", "scan": "binning", "binning_sort": "binning", "render_forward": "render_forward",
                        "render_backward": "render_backward", "preprocess_backward": "preprocess_backward"}
            tot, n = stages.get("render_backward", (0.0, 0))
            if n:
                dur = tot / n * 1e-3
                prof, prof_name = None, f"profiles/r02_ncu_render_backward_{a.config}.json"
                try:
                    prof = json.load(open(os.path.join(ROOT, prof_name)))
                except Exception:
                    pass
                traffic = None
                if prof:
                    traffic = float(prof["dram__bytes_read.sum"]["value"]) * {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}.get(prof["dram__bytes_read.sum"].get("unit", "Mbyte"), 1e6) + \
                        float(prof["dram__bytes_write.sum"]["value"]) * {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}.get(prof["dram__bytes_write.sum"].get("unit", "Mbyte"), 1e6)
                roofline = {"kernel": "render_backward_kernel", "bound": "hbm", "achieved": alg["render_backward"] / dur / 1e9, "peak": peak, "unit": "GB/s",
                            "frac": alg["render_backward"] / dur / 1e9 / peak, "traffic": traffic,
                            "traffic_source": (f"REPLAYED from {prof_name} (one `ncu --set full` capture of this kernel on this config), not measured in this run"
                                               if traffic is not None else None),
                            "algorithmic_bytes": alg["render_backward"], "avg_launch_ms": tot / n, "peak_source": peak_source,
                            "note": "this kernel is warp-instruction-issue bound, not HBM bound (records are L2-resident); see roofline_issue and DESIGN.md section 4"}
                if prof and "smsp__inst_executed.sum" in prof:
                    inst = float(prof["smsp__inst_executed.sum"]["value"])
                    clk_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6
                    floor = inst / (SM_COUNT * 4 * clk_hz)
                    roofline_issue = {"kernel": "render_backward_kernel", "bound": "warp-instruction issue (4 schedulers/SM, 1 inst/clk each)",
                                      "warp_instructions": inst, "warp_instructions_source": f"REPLAYED from {prof_name}",
                                      "sm_clock_mhz": clk_hz / 1e6, "floor_ms": floor * 1e3, "avg_launch_ms": tot / n, "frac": floor / dur}
            step_alg = sum(alg.values())
            step_hbm = {"algorithmic_bytes": step_alg, "achieved": step_alg / (ms_per_step * 1e-3) / 1e9, "unit": "GB/s", "peak": peak, "frac": step_alg / (ms_per_step * 1e-3) / 1e9 / peak,
                        "per_stage": {}}
            agg = {}
            for k, (t_ms, n) in stages.items():
                if n:
                    agg[stage_of[k]] = agg.get(stage_of[k], 0.0) + t_ms / n
            for k, t_ms in agg.items():
                step_hbm["per_stage"][k] = {"ms": t_ms, "algorithmic_bytes": alg[k], "GBps": alg[k] / (t_ms * 1e-3) / 1e9, "frac": alg[k] / (t_ms * 1e-3) / 1e9 / peak}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "Mpix/s", "n_gpus": world if multi else 1, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "impl": a.impl,
            "config": {"workload": f"{a.config}: {P} random-init Gaussians (SURVEY app. C seed 1234), {W}x{H}, SH deg 3, "
                                   f"require_depth={depth} require_coord={coord}, fwd+bwd at the _C boundary, num_rendered={R if not multi else 'per-slab'}",
                       "parallelism": (f"tile-row slabs x{world}, gradient-row exchange: {exchange.mode}" + (f" over {exchange.window}" if exchange.window else "") + (f" (peer self-check failed: {exchange.fallback_reason})" if exchange.fallback_reason else "")
                                       if multi else "single GPU"),
                       "l2": "per-step working set (192 MB SH + 248 MB SH grads + 64 MB records + sort buffers) exceeds the 126 MB L2; no explicit flush",
                       "protocol": f"median of {t_res['iterations']} per-iteration CUDA-event times (one window of {a.steps} steps, barrier+synchronize around it, max over ranks per iteration)"},
            "timing": t_res,
            "e2e": {"value": e2e_value, "unit": "Mpix/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "ms_per_step": t_e2e["ms"], "timing": t_e2e,
                    "api": "GaussianRasterizer autograd module (what render() calls) + L1 vs 8-bit GT image + depth/normal/alpha regularisers; camera + GT image H2D from pinned memory every step (GT on a side stream), loss.item() D2H"},
            "gpu_launches": launches, "clocks": clocks,
        }
        if stages:
            line["stage_ms"] = {k: v[0] / max(v[1], 1) for k, v in stages.items()}
        if roofline:
            line["roofline"] = roofline
        if roofline_issue:
            line["roofline_issue"] = roofline_issue
        if step_hbm:
            line["step_hbm"] = step_hbm
        if a.impl == "reference":
            line["cpu_baseline"] = {"value": value, "unit": "Mpix/s", "cores": 0, "kind": "reference",
                                    "sample": "reference CUDA rasterizer (oracle/_ref, sm_100a build of /root/reference) on 1xB200; the reference has no CPU rasterizer"}
            line["e2e"] = {"value": e2e_value, "unit": "Mpix/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "ms_per_step": t_e2e["ms"], "timing": t_e2e}
        elif not a.no_cpu_baseline and not multi:
            line["cpu_baseline"] = cpu_baseline()
        print(json.dumps(line), flush=True)
    if multi:
        exchange.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
