"""tools/rigid_bench.py -- rigid motion of whole meshes: refit against rebuild, and the scene-wide LBVH against the per-mesh one.

One process on one GPU.  The scene is 64 meshes of 2^20 hash-soup triangles each (scenes.hash_soup_torch, generated on the device from a
seed), one per cell of a 4 x 4 x 4 grid over [-1, 1]^3, under a constant environment light.  Every mesh is moved rigidly: rotated about
its centre by a seeded random angle of up to 45 degrees and translated by 0, 0.1, 1 or 4 cell sizes in a seeded random direction.  Arms:
  (a) KZ_BUILD_LBVH at rest, then kzgpu_mesh_transform x 64 + kzgpu_accel_refit
  (b) KZ_BUILD_LBVH_MESHES at rest, then transform x 64 + refit
  (c) a fresh KZ_BUILD_LBVH of the moved scene
  (d) a fresh KZ_BUILD_LBVH_MESHES of the moved scene
For each: Mpaths/s of one 4K x 64 spp render_device step (one warm-up step, then `--steps` timed with CUDA events) and Mrays/s of 2^24
incoherent trace_device rays (one warm-up batch, then `--steps` timed).  Per-frame cost, host clock around the synchronous calls, median of
`--reps` alternated runs: transform x 64 + refit, mesh_update x 64 from host arrays + refit, and a rebuild with either builder.
Prints the card's name and power limit, one line per measurement and a JSON summary; --out FILE also writes the summary there.

    python tools/rigid_bench.py [--reps 5] [--steps 2] [--out results.json]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "nano-kazen_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import pykazen as pk  # noqa: E402
import scenes  # noqa: E402
from refit_bench import card  # noqa: E402


def rigid(centre, axis, deg, t):
    """float32 row-major 4x4 of p -> R (p - centre) + centre + t, composed in float64"""
    a = np.asarray(axis, np.float64); a /= np.linalg.norm(a)
    th = np.radians(deg)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    R = np.eye(3) + np.sin(th) * K + (1 - np.cos(th)) * K @ K
    M = np.eye(4)
    M[:3, :3] = R
    M[:3, 3] = centre - R @ centre + t
    return M.astype(np.float32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", type=int, default=4)
    ap.add_argument("--tris", type=int, default=1 << 20, help="triangles per mesh")
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--rays", type=int, default=1 << 24)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("rigid_bench.py: no CUDA device")
    dev = torch.device("cuda", 0)
    info = card(0)
    print(f"card: {info}", flush=True)
    k, n, W, H, spp = args.grid ** 3, args.tris, args.width, args.height, 64
    cell = 2.0 / args.grid
    centres = np.array([[-1 + cell * (i % args.grid + 0.5), -1 + cell * (i // args.grid % args.grid + 0.5), -1 + cell * (i // args.grid ** 2 + 0.5)]
                        for i in range(k)])
    # rest pose: the n-triangle hash soup (in [-1, 1]^3 plus its offsets) shrunk to half a cell around each cell's centre
    P, F = scenes.hash_soup_torch(n, seed=0x5EED, device=dev)
    rest = [(P * (0.25 * cell) + torch.tensor(centres[i], dtype=torch.float32, device=dev)).contiguous() for i in range(k)]
    del P
    sb = pk.SceneBuilder()
    bs = sb.bsdf_diffuse((0.5, 0.5, 0.5))
    for i in range(k):
        m = pk.MeshDesc()
        m.positions = C.cast(rest[i].data_ptr(), pk.c_float_p); m.indices = C.cast(F.data_ptr(), pk.c_u32_p)
        m.n_vertices, m.n_triangles, m.bsdf, m.light = 3 * n, n, bs, -1
        sb.meshes.append(m)
    sb.background = sb.tex_background(1.0, sb.tex_constant((0.8, 0.9, 1.0)))
    sb.set_camera(W, H, 40.0, pk.lookat((0, 0, -3.5), (0, 0, 0), (0, 1, 0)))
    sb.set_sampler("stratified", 1024)
    sb.set_filter("gaussian")
    sb.set_integrator(max_depth=5)
    G = pk.Gpu(sb.desc(), devices=(0,), builder=pk.BUILD_LBVH)
    del F
    rest_host = [r.cpu().numpy() for r in rest]          # the host arrays of the mesh_update arm
    del rest
    torch.cuda.empty_cache()
    stream = torch.cuda.current_stream().cuda_stream
    eye = np.eye(4, dtype=np.float32)

    def build(builder):
        torch.cuda.synchronize()
        t = time.perf_counter(); G._call("accel_build", G.h, C.c_int(builder)); return (time.perf_counter() - t) * 1e3

    def transform_all(mats):
        for i in range(k):
            G.mesh_transform(i, mats[i])

    def transform_refit(mats):
        torch.cuda.synchronize()
        t = time.perf_counter(); transform_all(mats); G.refit(); return (time.perf_counter() - t) * 1e3

    def update_refit():
        torch.cuda.synchronize()
        t = time.perf_counter()
        for i in range(k):
            G.mesh_update(i, rest_host[i])
        G.refit()
        return (time.perf_counter() - t) * 1e3

    frame = torch.zeros(G.frame_shape()[:2] + (4,), dtype=torch.float32, device=dev)
    gen = torch.Generator(device=dev).manual_seed(args.seed)
    rays = torch.zeros((args.rays, 8), dtype=torch.float32, device=dev)
    rays[:, 0:3] = torch.rand((args.rays, 3), device=dev, generator=gen) * 2.4 - 1.2
    dirs = torch.randn((args.rays, 3), device=dev, generator=gen)
    rays[:, 4:7] = dirs / dirs.norm(dim=1, keepdim=True)
    rays[:, 3] = 1e-4; rays[:, 7] = float("inf")
    hits = torch.empty((args.rays, 5), dtype=torch.float32, device=dev)

    def rates():
        G.render_device(0, spp, device=0, clear=True, stream=stream, frame_ptr=frame.data_ptr())
        G.trace_device(rays.data_ptr(), args.rays, hits.data_ptr(), stream=stream)
        torch.cuda.synchronize()
        e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        e[0].record()
        for s in range(args.steps):
            s0 = ((s + 1) % 16) * spp
            G.render_device(s0, s0 + spp, device=0, clear=True, stream=stream, frame_ptr=frame.data_ptr())
        e[1].record(); e[2].record()
        for _ in range(args.steps):
            G.trace_device(rays.data_ptr(), args.rays, hits.data_ptr(), stream=stream)
        e[3].record()
        torch.cuda.synchronize()
        return (W * H * spp / (e[0].elapsed_time(e[1]) / args.steps * 1e-3) / 1e6, args.rays / (e[2].elapsed_time(e[3]) / args.steps * 1e-3) / 1e6)

    rng = np.random.default_rng(args.seed)
    axes, angles, dirs_t = rng.normal(size=(k, 3)), rng.uniform(0, 45, k), rng.normal(size=(k, 3))
    dirs_t /= np.linalg.norm(dirs_t, axis=1, keepdims=True)
    arms = {"a_lbvh_refit": (pk.BUILD_LBVH, True), "b_lbvh_meshes_refit": (pk.BUILD_LBVH_MESHES, True),
            "c_lbvh_fresh": (pk.BUILD_LBVH, False), "d_lbvh_meshes_fresh": (pk.BUILD_LBVH_MESHES, False)}
    quality = []
    for cells in (0.0, 0.1, 1.0, 4.0):
        mats = [rigid(centres[i], axes[i], angles[i], dirs_t[i] * cells * cell) for i in range(k)]
        row = {"translate_cells": cells}
        for name, (builder, refit) in arms.items():
            if refit:
                transform_all([eye] * k)            # the rest pose, built ...
                build(builder)
                transform_all(mats); G.refit()      # ... and refitted to the moved one
            else:
                transform_all(mats)
                build(builder)
            row[name] = dict(zip(("mpaths", "mrays"), rates()))
        quality.append(row)
        print(f"translate {cells:3.1f} cells + rotate <= 45 deg: " + ", ".join(f"{a} {v['mpaths']:7.1f} Mpaths/s {v['mrays']:7.1f} Mrays/s"
                                                                          for a, v in row.items() if a != "translate_cells"), flush=True)
    # per-frame cost, alternated
    mats = [rigid(centres[i], axes[i], angles[i], dirs_t[i] * cell) for i in range(k)]
    timing = {"transform_refit_ms": [], "update_host_refit_ms": [], "build_lbvh_ms": [], "build_lbvh_meshes_ms": []}
    build(pk.BUILD_LBVH_MESHES)
    transform_refit(mats)                          # the first refit after a build checks the level layout: not timed
    for _ in range(args.reps):
        timing["transform_refit_ms"].append(transform_refit(mats))
        timing["update_host_refit_ms"].append(update_refit())
        timing["build_lbvh_ms"].append(build(pk.BUILD_LBVH))
        timing["build_lbvh_meshes_ms"].append(build(pk.BUILD_LBVH_MESHES))
        transform_refit(mats)
    for key, v in timing.items():
        v = np.array(v)
        print(f"{key:24s} median {np.median(v):8.1f}  min {v.min():8.1f}  max {v.max():8.1f}  ({len(v)} runs)", flush=True)
    G.close()
    out = {"card": info, "meshes": k, "tris_per_mesh": n, "film": [W, H], "spp_per_step": spp, "rays": args.rays, "steps": args.steps,
           "timing": timing, "timing_median_ms": {key: float(np.median(v)) for key, v in timing.items()}, "trace_quality": quality}
    print(json.dumps(out), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
