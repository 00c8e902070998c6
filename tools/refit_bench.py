"""tools/refit_bench.py -- animation on the headline scene: what a refit costs against a rebuild, and what it costs the traversal.

One process on one GPU.  The 10^8-triangle hash soup of the headline (configs[4]) is generated on the device (scenes.hash_soup_torch)
and built with the LBVH.  Then:
  1. time: kzgpu_mesh_update from the device tensor + kzgpu_accel_refit against kzgpu_accel_build(LBVH) over the same positions, host
     clock around the synchronous calls, alternated `--reps` times.  The first refit after a build also checks the accel's level layout
     (once per build and device), so it is reported apart from the refits that follow it;
  2. trace quality: Mpaths/s of one headline step (4K, 64 spp; one warm-up step, then `--steps` timed with CUDA events) on a fresh build
     and after a refit of the unmoved build, for no motion and for per-vertex jitter of 0.1, 1 and 10 mean edge lengths.
Prints the card's name and power limit, one line per measurement and a JSON summary; --out FILE also writes the summary there.

    python tools/refit_bench.py [--tris 100000000] [--reps 5] [--steps 2] [--out results.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "nano-kazen_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import pykazen as pk  # noqa: E402
import scenes  # noqa: E402


def card(index):
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown (nvidia-smi unavailable)"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tris", type=int, default=100_000_000)
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("refit_bench.py: no CUDA device")
    dev = torch.device("cuda", 0)
    info = card(0)
    print(f"card: {info}", flush=True)
    n, W, H, spp = args.tris, args.width, args.height, 64
    P0, F = scenes.hash_soup_torch(n, device=dev)
    sb = scenes.big_scene(n, W, H, 1024, positions=P0.data_ptr(), indices=F.data_ptr(), keep=(P0, F))
    G = pk.Gpu(sb.desc(), devices=(0,), builder=pk.BUILD_LBVH)
    del F
    sb._keep.clear()
    torch.cuda.empty_cache()
    stream = torch.cuda.current_stream().cuda_stream

    def build():
        torch.cuda.synchronize()
        t = time.perf_counter(); G._call("accel_build", G.h, C.c_int(pk.BUILD_LBVH)); return (time.perf_counter() - t) * 1e3

    def update_refit(P):
        torch.cuda.synchronize()
        t = time.perf_counter(); G.mesh_update(0, P.data_ptr()); G.refit(); return (time.perf_counter() - t) * 1e3

    # ---- 1. refit vs rebuild, alternated
    t_build, t_first, t_next = [], [], []
    for _ in range(args.reps):
        t_build.append(build())
        t_first.append(update_refit(P0))
        t_next.append(update_refit(P0))
    st = G.stats()
    timing = {"build_ms": t_build, "update_refit_first_after_build_ms": t_first, "update_refit_ms": t_next,
              "bvh_nodes": st["bvh_nodes"], "bvh_bytes": st["bvh_bytes"]}
    for k in ("build_ms", "update_refit_first_after_build_ms", "update_refit_ms"):
        v = np.array(timing[k])
        print(f"{k:36s} median {np.median(v):8.1f}  min {v.min():8.1f}  max {v.max():8.1f}  ({len(v)} runs)", flush=True)

    # ---- 2. trace quality after a refit
    frame = torch.zeros(G.frame_shape()[:2] + (4,), dtype=torch.float32, device=dev)

    def mpaths():
        G.render_device(0, spp, device=0, clear=True, stream=stream, frame_ptr=frame.data_ptr())
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(args.steps):
            s0 = ((k + 1) % 16) * spp
            G.render_device(s0, s0 + spp, device=0, clear=True, stream=stream, frame_ptr=frame.data_ptr())
        e1.record()
        torch.cuda.synchronize()
        return W * H * spp / (e0.elapsed_time(e1) / args.steps * 1e-3) / 1e6

    # mean edge length of the soup, from a sample of its triangles
    idx = torch.arange(0, n, max(1, n // (1 << 20)), device=dev)
    T = P0.view(n, 3, 3)[idx]
    edge = float(((T[:, 1] - T[:, 0]).norm(dim=1) + (T[:, 2] - T[:, 1]).norm(dim=1) + (T[:, 0] - T[:, 2]).norm(dim=1)).mean() / 3)
    del T
    quality = []
    gen = torch.Generator(device=dev)
    for amp in (0.0, 0.1, 1.0, 10.0):
        if amp == 0.0:
            P = P0
        else:
            gen.manual_seed(int(amp * 1000) + 7)
            P = P0.clone()
            for first in range(0, P.shape[0], 1 << 25):
                blk = P[first: first + (1 << 25)]
                blk += torch.randn(blk.shape, device=dev, generator=gen) * (amp * edge)
        G.mesh_update(0, P0.data_ptr())
        build()                                   # the tree of the unmoved soup ...
        update_refit(P)                           # ... refitted to the moved one
        refit_rate = mpaths()
        build()                                   # the moved soup's own tree
        fresh_rate = mpaths()
        row = {"jitter_edges": amp, "mpaths_fresh_build": fresh_rate, "mpaths_after_refit": refit_rate, "ratio": refit_rate / fresh_rate}
        quality.append(row)
        print(f"jitter {amp:5.1f} mean edges ({amp * edge:.2e}): fresh build {fresh_rate:7.1f} Mpaths/s, after refit {refit_rate:7.1f} Mpaths/s "
              f"({100 * row['ratio']:.1f} %)", flush=True)
        del P
        torch.cuda.empty_cache()
    G.close()
    out = {"card": info, "tris": n, "film": [W, H], "spp_per_step": spp, "steps": args.steps, "mean_edge": edge, "timing": timing, "trace_quality": quality}
    print(json.dumps(out), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
