#!/usr/bin/env python
"""A/B of the primary-hit hints (kzgpu_configure "primary_hint" 0 against 2 = always) in one process, on the GPU.

For every scene: steps with the hints off and on, alternating, timed with CUDA events (default lanes, as bench.py times its steps);
one step of each with a single lane under torch.profiler for the per-kernel device time (k_extend<true> = primary rays); the seeded
fraction of the primary rays (kz_stats.rays_seeded / paths); and the frames of the same sample range rendered off and on, which must
agree to float rounding (only the order of the atomic splats differs).  Prints one JSON object; --out FILE also writes it there.

usage: primary_hint_ab.py [--scenes headline,warm,c2,c3] [--tris N] [--width W --height H] [--rounds R] [--out FILE]"""
import argparse, json, os, shutil, sys, tempfile, time
R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
[sys.path.insert(0, os.path.join(R, p)) for p in ("tests", "nano-kazen_b200")]
import numpy as np, torch
import scenes, pykazen as pk

WARM_XML = os.path.join(R, "tests", "data", "kazen_scenes", "2022_q1", "WarmStudio", "WarmStudio.xml")


def kernel_ms(G, render):
    """device time per kernel name of one render with a single lane (serial kernels), from torch.profiler"""
    G.configure("lanes", 1)
    render(); torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        render(); torch.cuda.synchronize()
    G.configure("lanes", int(os.environ.get("KZGPU_LANES", 3)))
    out = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            name = e.name.replace("void ", "").split("(")[0]
            out[name] = out.get(name, 0.0) + e.device_time_total / 1e3
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def ab(G, W, H, spp, rounds, steps_per_round):
    stream = torch.cuda.current_stream().cuda_stream
    fh, fw, _ = G.frame_shape()
    frame = torch.zeros((fh, fw, 4), dtype=torch.float32, device="cuda")
    n_frames = max(1, G._desc.sampler.sample_count // spp)
    k = [0]

    def step():
        base = (k[0] % n_frames) * spp; k[0] += 1
        G.render_device(base, base + spp, device=0, clear=True, stream=stream, frame_ptr=frame.data_ptr())

    for on in (1, 0, 1):
        G.configure("primary_hint", 2 * on); step(); step()
    torch.cuda.synchronize()
    ms = {0: [], 1: []}
    for _ in range(rounds):
        for on in (0, 1):
            G.configure("primary_hint", 2 * on)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps_per_round):
                step()
            e1.record(); torch.cuda.synchronize()
            ms[on].append(e0.elapsed_time(e1) / steps_per_round)
    res = {"paths_per_step": W * H * spp, "step_ms": {"off": ms[0], "on": ms[1]},
           "mpaths_s": {"off": W * H * spp / (np.median(ms[0]) * 1e3), "on": W * H * spp / (np.median(ms[1]) * 1e3)}}
    res["speedup_median"] = float(np.median(ms[0]) / np.median(ms[1]))
    # per-kernel device time and counters of one step each
    res["kernels_ms"] = {}
    for on in (0, 1):
        G.configure("primary_hint", 2 * on)
        res["kernels_ms"]["on" if on else "off"] = kernel_ms(G, step)
        G.stats(reset=True); step(); torch.cuda.synchronize()
        st = G.stats(reset=True)
        res["stats_" + ("on" if on else "off")] = {k_: st[k_] for k_ in ("paths", "rays_extension", "rays_shadow", "vertices", "rays_seeded")}
    res["seeded_fraction_of_primary_rays"] = res["stats_on"]["rays_seeded"] / max(1, res["stats_on"]["paths"])
    # the same sample range off and on
    frames = {}
    for on in (0, 1, 0, 1):
        G.configure("primary_hint", 2 * on)
        G.render_device(0, spp, device=0, clear=True, stream=stream, frame_ptr=frame.data_ptr()); torch.cuda.synchronize()
        frames.setdefault(on, []).append(frame.double().cpu().numpy())
    a, b = frames[0][1], frames[1][1]
    scale = float(np.abs(a).max())
    res["frame"] = {"mean_off": float(a[..., :3].mean()), "mean_on": float(b[..., :3].mean()),
                    "mean_rel_diff": float(abs(b[..., :3].mean() / a[..., :3].mean() - 1.0)),
                    "max_abs_diff_over_max": float(np.abs(a - b).max() / scale),
                    "off_vs_off_max_abs_diff_over_max": float(np.abs(a - frames[0][0]).max() / scale),
                    "weights_equal": bool(np.array_equal(a[..., 3] != 0, b[..., 3] != 0))}
    G.configure("primary_hint", 1)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", default="headline")
    ap.add_argument("--tris", type=int, default=100_000_000)
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()
    props = torch.cuda.get_device_properties(0)
    out = {"device": props.name}
    try:
        import subprocess
        out["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    except OSError:
        out["power_limit"] = None
    cfg = None
    for name in args.scenes.split(","):
        t0 = time.perf_counter()
        if name == "headline":
            P, F = scenes.hash_soup_torch(args.tris)
            sb = scenes.big_scene(args.tris, args.width, args.height, 1024, positions=P.data_ptr(), indices=F.data_ptr(), keep=(P, F))
            G = pk.Gpu(sb.desc(), builder=pk.BUILD_LBVH)
            del P, F; sb._keep.clear(); torch.cuda.empty_cache()
            W, H, spp, steps = args.width, args.height, 64, 2
        else:
            if name == "warm":
                hs = pk.HostScene(WARM_XML, {"camera.width": "i:512", "camera.height": "i:512", "sampler.type": "s:stratified", "sampler.sampleCount": "i:64"})
            else:
                if cfg is None:
                    import importlib.util
                    spec = importlib.util.spec_from_file_location("make_configs", os.path.join(R, "tests", "data", "make_configs.py"))
                    mc = importlib.util.module_from_spec(spec); spec.loader.exec_module(mc)
                    cfg = tempfile.mkdtemp(prefix="kz_hint_cfg_")
                    mc.generate(cfg, tex_res=4096)
                hs = pk.HostScene(os.path.join(cfg, {"c2": "c3_lookdev_4k.xml", "c3": "c4_pmj02bn_1080p.xml"}[name]), {})
            G = pk.Gpu(hs.desc, builder=pk.BUILD_HOST_SAH)
            W, H, spp, steps = hs.desc.camera.width, hs.desc.camera.height, 64, 3
        out[name] = ab(G, W, H, spp, args.rounds, steps)
        out[name]["wall_s"] = time.perf_counter() - t0
        G.close()
        torch.cuda.empty_cache()
        print(name, json.dumps({k: out[name][k] for k in ("mpaths_s", "speedup_median", "seeded_fraction_of_primary_rays", "frame")}), flush=True)
    if cfg:
        shutil.rmtree(cfg, ignore_errors=True)
    js = json.dumps(out, indent=1)
    print(js)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        open(args.out, "w").write(js)


if __name__ == "__main__":
    main()
