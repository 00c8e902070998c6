#!/usr/bin/env python
"""Texture filtering (path_mis textureFiltering) on one GPU, in one process.

Scene: the BASELINE configs[2] stand-in of tests/data/make_configs.py (look-dev material ball in the studio, thin-lens camera,
3840x2160) with its three 4096^2 textures, rendered with the independent sampler.  For sample_count 1, 4, 16 and 64 the flag off and
on are uploaded side by side and their renders alternated (--reps times each): Mpaths/s from the host clock around a synchronous
kzgpu_render, the relative MSE against a flag-off reference of --ref-spp samples per pixel, the upload time, and the HBM the pyramids
add.  Prints one JSON object, card name and power limit included.

    python tools/texture_filtering_bench.py [--ref-spp 1024] [--reps 3] [--tex-res 4096]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "nano-kazen_b200"), os.path.join(ROOT, "tests", "data")):
    sys.path.insert(0, p)
import make_configs  # noqa: E402
import pykazen as pk  # noqa: E402


def rel_mse(a, ref):
    return float((((a - ref) ** 2) / (ref ** 2 + 1e-2)).mean())


def pyramid_texels(w, h):
    n = 0
    while w > 1 or h > 1:
        w, h = max(1, w >> 1), max(1, h >> 1)
        n += w * h
    return n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref-spp", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--tex-res", type=int, default=4096)
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    out = {"gpu": gpu[0] if gpu else "unknown"}
    with tempfile.TemporaryDirectory() as td:
        make_configs.generate(td, args.tex_res)
        hs = pk.HostScene(os.path.join(td, "c3_lookdev_4k.xml"))
        d = hs.desc
        W, H = d.camera.width, d.camera.height
        out["scene"] = {"size": [W, H], "images": [[d.images[i].width, d.images[i].height] for i in range(d.n_images)]}
        out["pyramid_extra_MiB"] = sum(pyramid_texels(d.images[i].width, d.images[i].height) for i in range(d.n_images)) * 16 / 2 ** 20
        d.sampler.type, d.sampler.res_x, d.sampler.res_y = pk.SAMPLER_INDEPENDENT, 0, 0

        def context(on, spp):
            d.integrator.texture_filtering = int(on)
            d.sampler.sample_count = spp
            return pk.Gpu(d, builder=pk.BUILD_LBVH)

        G = context(False, 1)
        ref = G.resolve(G.render(1 << 20, (1 << 20) + args.ref_spp))[0]
        G.close()
        res = {}
        for spp in (1, 4, 16, 64):
            G = {on: context(on, spp) for on in (False, True)}
            r = {}
            for on in (False, True):
                G[on].render(0, spp)                     # warm-up
                r["on" if on else "off"] = {"ms_upload": G[on].stats()["ms_upload"], "Mpaths_s": [], "rel_mse": None}
            for _ in range(args.reps):
                for on in (False, True):
                    t0 = time.perf_counter()
                    f = G[on].render(spp, 2 * spp)
                    sec = time.perf_counter() - t0
                    k = r["on" if on else "off"]
                    k["Mpaths_s"].append(W * H * spp / sec / 1e6)
                    if k["rel_mse"] is None:
                        k["rel_mse"] = rel_mse(G[on].resolve(f)[0], ref)
            for on in (False, True):
                G[on].close()
            res[str(spp)] = r
        out["sample_count"] = res
        hs.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
