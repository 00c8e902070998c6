#!/usr/bin/env python
"""Environment importance sampling (path_mis envSampling) on one GPU, in one process:

  * the sun studio (tests/env_scenes.py) at 960x540: Mpaths/s with the flag off and on, the relative MSE against a converged reference
    at 16, 64 and 256 spp, and the efficiency 1 / (relMSE * time) of each;
  * the headline scene (BASELINE configs[4]: hash soup, constant sky) at 3840x2160 x 64 spp with the flag off and on: what the flag
    costs where importance sampling cannot help.

Prints one JSON object (card name and power limit included).  Usage: python tools/env_sampling_bench.py [--ref-spp 16384] [--tris 100000000]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "nano-kazen_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import env_scenes  # noqa: E402
import pykazen as pk  # noqa: E402
import scenes  # noqa: E402


def timed_render(G, s0, s1):
    t0 = time.perf_counter()
    f = G.render(s0, s1)
    return f, time.perf_counter() - t0


def rel_mse(a, ref):
    return float((((a - ref) ** 2) / (ref ** 2 + 1e-2)).mean())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--width", type=int, default=960)
    ap.add_argument("--height", type=int, default=540)
    ap.add_argument("--ref-spp", type=int, default=16384, help="samples per pixel of each method's half of the reference")
    ap.add_argument("--tris", type=int, default=100_000_000, help="triangles of the headline scene")
    args = ap.parse_args()
    import torch
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    out = {"gpu": gpu[0] if gpu else "unknown", "studio": {"size": [args.width, args.height]}}
    spp_total = max(args.ref_spp, 1 << 15)
    sbs = {on: env_scenes.sun_studio(args.width, args.height, spp_total, env_sampling=on) for on in (False, True)}      # own the arrays the scenes point at
    G = {on: pk.Gpu(sbs[on].desc()) for on in (False, True)}
    b = G[False].frame_shape()[2]
    for on in (False, True):
        G[on].render(0, 16)      # warm-up
    # converged reference: both methods, sample indices none of the measured renders use
    ref = 0.5 * sum(env_scenes.resolve(G[on].render(1 << 20, (1 << 20) + args.ref_spp), b) for on in (False, True))
    npx = args.width * args.height
    for on in (False, True):
        key = "on" if on else "off"
        res = {}
        for spp in (16, 64, 256):
            f, sec = timed_render(G[on], 0, spp)
            e = rel_mse(env_scenes.resolve(f, b), ref)
            res[str(spp)] = {"seconds": sec, "Mpaths_s": npx * spp / sec / 1e6, "rel_mse": e, "efficiency": 1.0 / (e * sec)}
        out["studio"][key] = res
    for spp in ("16", "64", "256"):
        out["studio"].setdefault("efficiency_ratio_on_over_off", {})[spp] = out["studio"]["on"][spp]["efficiency"] / out["studio"]["off"][spp]["efficiency"]
    for g in G.values():
        g.close()
    # headline scene: constant sky, 4K x 64 spp
    P, F = scenes.hash_soup_torch(args.tris, device="cuda")
    torch.cuda.synchronize()
    head = {}
    for on in (False, True, False, True):
        sb = scenes.big_scene(args.tris, 3840, 2160, 1024, positions=P.data_ptr(), indices=F.data_ptr(), keep=(P, F))
        sb.set_integrator(max_depth=5, env_sampling=on)
        g = pk.Gpu(sb.desc(), builder=pk.BUILD_LBVH)
        g.render_device(0, 64)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        g.render_device(64, 128)
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        head.setdefault("on" if on else "off", []).append(3840 * 2160 * 64 / sec / 1e6)
        g.close()
    out["headline_4k_64spp_Mpaths_s"] = head
    print(json.dumps(out))


if __name__ == "__main__":
    main()
