#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric (Mpaths/s and Mrays/s at 1/2/4/8 B200, time-to-image) on the render hot path.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...        # the CPU port of the reference path on the host cores
    python bench.py ... --dump-outputs DIR      # also write the headline's last timed frame to DIR/frame.npy

Headline (every N): BASELINE configs[4] AT SPEC -- a procedural 10^8-triangle scene with an environment light, 3840x2160,
stratified sampler with 1024 samples per pixel, path_mis maxDepth 5 (SURVEY 8d-5).  The scene is generated on the device from a
seed (tests/scenes.py hash soup), ingested and its LBVH accel built through the C ABI.  A STEP = one pass of the whole wavefront
(raygen, extend, material-sorted shade, accumulate) over 64 consecutive sample indices of all 8.3 M pixels = 530.8 M paths; 16
steps are the full 1024-spp frame.  Multi-GPU is STRONG scaling: the step's 64 sample indices are sharded over the ranks (scene
replicated), and every step ends with the ONE collective of the path, the NCCL reduce of the bordered frame to rank 0
(ImageBlock merge, block.cpp:87-96) -- inside the timed region.

Further legs (N = 1; `--legs` selects): the triangle-soup intersection microbench of configs[1] at 2^20 and 10^7 triangles
(k_trace roofline with its ncu DRAM traffic), kazen's own WarmStudio.xml at 512x512x64 spp (configs[0]), and the configs[2] /
configs[3] stand-in XML scenes at full resolution; each path-tracing leg reports Mpaths/s, Mrays/s, rays per path, the SURVEY 8(d)
per-path roofline fraction, an end-to-end number through kzgpu_render (host frame out) and a time-to-image that INCLUDES
kzgpu_scene_upload + kzgpu_accel_build.
"""
import argparse
import json
import math
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(ROOT, "nano-kazen_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

SPP_TOTAL = 1024          # configs[4]
SPP_PER_STEP = 64
WARM_XML = os.path.join(ROOT, "tests", "data", "kazen_scenes", "2022_q1", "WarmStudio", "WarmStudio.xml")
DUMP_MAX_PIXELS = 1 << 21     # 32 MiB of RGBW float32
DUMP_SEED = 0


def dump_frame(frame, out_dir):
    """Writes a (H+2b, W+2b, 4) float32 device frame to out_dir/frame.npy: the whole frame when it has at most DUMP_MAX_PIXELS
    pixels, else a (DUMP_MAX_PIXELS, 4) sample of its pixels, chosen with DUMP_SEED and kept in row-major order, so that two
    builds run with the same arguments write the same pixels.  The path contributions are summed into the frame by atomic adds in
    no fixed order, so two runs of one build agree to float rounding, not bit for bit: compare with a relative tolerance."""
    import torch
    fh, fw, _ = frame.shape
    if fh * fw <= DUMP_MAX_PIXELS:
        out = frame.cpu().numpy()
    else:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(fh * fw, DUMP_MAX_PIXELS, replace=False))
        out = frame.reshape(-1, 4).index_select(0, torch.from_numpy(idx).to(frame.device)).cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "frame.npy"), np.ascontiguousarray(out, np.float32))


def b_ray(n_tris, shadow=False):
    """SURVEY 8(d): algorithmic bytes per ray = ray in + hit out + one root-to-leaf descent of
    80-byte 8-wide nodes + one 4-triangle leaf of 48-byte triangles."""
    return 32 + (8 if shadow else 20) + 80 * math.ceil(math.log(max(n_tris, 8) / 4.0, 8)) + 4 * 48


def b_path(n_tris, n_ext, n_sh, n_vtx):
    """SURVEY 8(d): B_path = n_ext*B_ray + n_sh*(B_ray - 12) + n_vtx*512 + 256 with the MEASURED per-path counts."""
    br = b_ray(n_tris)
    return n_ext * br + n_sh * (br - 12) + n_vtx * 512 + 256


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def committed_traffic(**match):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu capture of the same workload, else None"""
    try:
        with open(os.path.join(ROOT, "profiles", "r7_traffic.json")) as f:
            for tj in json.load(f)["workloads"]:
                if all(tj.get(k) == v for k, v in match.items()):
                    return tj["dram_bytes_per_launch_mean"]
    except Exception:
        pass
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.lines, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for k, nme in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


_JSON_FD = None


def claim_stdout():
    """Everything that libraries print on stdout (NCCL's version banner, ...) is sent to stderr; the ONE JSON line is
    written to the original stdout by emit()."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_JSON_FD if _JSON_FD is not None else 1, (json.dumps(line) + "\n").encode())


def headline_config(args, world):
    return {"workload": f"BASELINE configs[4]: procedural {args.tris}-triangle scene + environment light, {args.width}x{args.height}, "
                        f"{SPP_TOTAL} spp stratified, path_mis maxDepth 5; one step = {SPP_PER_STEP} sample indices of every pixel",
            "tris": args.tris, "width": args.width, "height": args.height, "spp_total": SPP_TOTAL, "spp_per_step": SPP_PER_STEP,
            "paths_per_step": args.width * args.height * SPP_PER_STEP, "steps_per_frame": SPP_TOTAL // SPP_PER_STEP,
            "accel": "LBVH built on the GPU", "parallelism": f"sample-index shards x{world} + one NCCL reduce of the frame per step",
            "l2": "scene (accel + shading geometry) and path state are far larger than the 126 MB L2"}


def find_embree():
    """BASELINE.md section 4 step 1: the reference's own CPU path needs Embree 3.13 + TBB + OpenImageIO; report what this box has"""
    found = {"libembree3": None, "libOpenImageIO": None, "libtbb": None}
    for top in ("/usr/lib", "/usr/lib64", "/usr/local/lib", "/opt"):
        if not os.path.isdir(top):
            continue
        for root, dirs, files in os.walk(top):
            if root.count(os.sep) - top.count(os.sep) >= 3:
                dirs[:] = []
            for name in found:
                if found[name] is None and any(f.startswith(name) and ".so" in f for f in files):
                    found[name] = root
    return found


# =================================================================================================== the reference arm (CPU)
def run_reference(args):
    """The reference arm: the CPU port (oracle) of the same path -- Scene::rayIntersect + PathMisIntegrator::Li + ImageBlock::put --
    on all host cores, on the headline scene.  Each step renders a bounded sample of the step the GPU arm times: one of its 64
    sample indices on the central quarter of the frame."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import kzo_py
    import scenes
    kzo_py.build()
    cores = os.cpu_count() or 1
    libs = find_embree()
    t0 = time.perf_counter()
    sb = scenes.big_scene(args.tris, args.width, args.height, SPP_TOTAL)
    O = kzo_py.Oracle(sb.desc())
    setup_s = time.perf_counter() - t0
    W, H = args.width, args.height
    rect = (W // 4, H // 4, W // 4 + W // 2, H // 4 + H // 2) if args.tris > 100000 else (0, 0, W, H)
    npaths = (rect[2] - rect[0]) * (rect[3] - rect[1])
    frame = np.zeros(O.frame_shape()[:2] + (4,), np.float32)
    for k in range(min(args.warmup, 1)):
        O.render(0, 1, rect=(rect[0], rect[1], rect[0] + 64, rect[1] + 64), frame=frame)
    t0 = time.perf_counter()
    for k in range(args.steps):
        s = (SPP_PER_STEP * k) % SPP_TOTAL
        O.render(s, s + 1, rect=rect, frame=frame)
    dt = time.perf_counter() - t0
    st = O.stats()
    val = args.steps * npaths / dt / 1e6
    sample = f"per step: sample index 64*k of the {rect[2] - rect[0]}x{rect[3] - rect[1]} central pixels of the same frame ({npaths} paths)"
    line = {"impl": "reference", "metric": "Mpaths/s", "value": val, "unit": "Mpaths/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": headline_config(args, args.gpus),
            "cpu_baseline": {"value": val, "unit": "Mpaths/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "Mpaths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "mrays_per_s": (st["rays_extension"] + st["rays_shadow"]) / dt / 1e6, "setup_s": setup_s,
            "reference_libraries_found": libs,
            "note": "CPU port of the reference path (oracle: median-split BVH2 + Embree-robust Pluecker test + restated Li, std::thread over all cores); "
                    "the reference itself (Embree 3.13 + TBB + OpenImageIO) cannot be built in this image" +
                    ("" if not all(libs.values()) else " -- its libraries ARE present on this box, see reference_libraries_found")}
    O.close()
    emit(line)


# =================================================================================================== the GPU arm
def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--tris", type=int, default=100_000_000, help="triangles of the headline scene (configs[4]: 10^8)")
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--legs", default="auto", help="comma list of headline,soup1m,soup10m,c0,c2,c3 (auto: all at N=1, headline+c0 at N>1)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--cfg-dir", default=None, help="directory for the generated configs[2] / configs[3] scenes (default: a temporary one, removed at exit)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the frame of the headline's last timed step to DIR/frame.npy (float32, see dump_frame)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's frame; it does not apply to --impl reference")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if rank == 0:
            run_reference(args)
        return 0
    legs = set(args.legs.split(",")) if args.legs != "auto" else ({"headline", "soup1m", "soup10m", "c0", "c2", "c3"} if world == 1 else {"headline", "c0"})

    import torch
    import torch.distributed as dist
    import pykazen as pk
    import scenes
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU path; use --impl reference for the CPU port)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    stream = torch.cuda.current_stream().cuda_stream
    peak, peak_kind = measured_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_scalar(v, op):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t.item())

    def rmax(v): return reduce_scalar(v, dist.ReduceOp.MAX) if world > 1 else v
    def rsum(v): return reduce_scalar(v, dist.ReduceOp.SUM) if world > 1 else v

    # ------------------------------------------------------------------------------------------ a path-tracing leg
    def path_leg(G, n_tris, W, H, spp_step, spp_total, steps, warmup, label, upload_ms, build_ms, oracle_desc=None, cpu_rect=None, clocks_on=False,
                 dump_dir=None):
        """Times `steps` steps of spp_step sample indices each (strong scaling: this rank's shard + the NCCL reduce), then the same
        through the host-frame C ABI call, then (rank 0, N = 1) a bounded sample on the CPU port.  dump_dir: rank 0 writes the frame
        of the last timed step there (dump_frame)."""
        fh, fw, _ = G.frame_shape()
        frame = torch.zeros((fh, fw, 4), dtype=torch.float32, device=dev)
        host_frame = torch.zeros((fh, fw, 4), dtype=torch.float32).pin_memory() if rank == 0 else None
        n_steps_frame = max(1, spp_total // spp_step)

        def pstep(k):
            base = (k % n_steps_frame) * spp_step
            s0, s1 = pk.shard_range(base, base + spp_step, rank, world)
            G.render_device(s0, s1, device=0, clear=True, stream=stream, frame_ptr=frame.data_ptr())
            if world > 1:
                dist.reduce(frame, dst=0, op=dist.ReduceOp.SUM)      # the only collective of the path: ImageBlock merge (block.cpp:87-96)
        for k in range(warmup):
            pstep(k)
        barrier(); G.stats(reset=True)
        clocks = ClockSampler(local) if (rank == 0 and clocks_on) else None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        prof = clocks_on and os.environ.get("KZ_PROFILE_STEP") == "1"      # ncu --profile-from-start off: the timed steps of the headline only
        if prof:
            torch.cuda.profiler.start()
        e0.record()
        for k in range(steps):
            pstep(k)
        e1.record()
        barrier()
        if prof:
            torch.cuda.profiler.stop()
        ms = rmax(e0.elapsed_time(e1)) / steps
        clk = clocks.stop() if clocks else None
        if dump_dir and rank == 0:
            dump_frame(frame, dump_dir)
        st = G.stats(reset=True)
        npaths = W * H * spp_step
        n_ext = rsum(st["rays_extension"]) / steps / npaths
        n_sh = rsum(st["rays_shadow"]) / steps / npaths
        n_vtx = rsum(st["vertices"]) / steps / npaths
        launches = int(rsum(st["kernel_launches"]))
        bp = b_path(n_tris, n_ext, n_sh, n_vtx)
        ach = npaths * bp / (ms * 1e-3) / 1e9 / world           # per GPU, against one GPU's HBM
        out = {"value": npaths / (ms * 1e-3) / 1e6, "unit": "Mpaths/s", "mrays_per_s": npaths * (n_ext + n_sh) / (ms * 1e-3) / 1e6, "ms_per_step": ms,
               "scene": label, "steps": steps, "paths_per_step": npaths, "rays_per_path": n_ext + n_sh, "gpu_launches": launches,
               "path_roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "bytes_per_path": bp, "bytes_per_ray": b_ray(n_tris),
                                 "tris": n_tris, "n_ext": n_ext, "n_sh": n_sh, "n_vtx": n_vtx,
                                 "note": "SURVEY 8(d) B_path with the measured per-path counts; whole wavefront, per GPU"}}
        if clk is not None:
            out["clocks"] = clk
        # single-lane pass: kernels of one chunk run strictly one after the other, so the library's CUDA-event times are per-kernel
        # times (with two lanes in flight the kernels of both lanes overlap and their event times add up to more than the wall time)
        G.configure("lanes", 1)
        pstep(0); barrier(); G.stats(reset=True)
        pstep(0); barrier()
        s1 = G.stats(reset=True)
        G.configure("lanes", int(os.environ.get("KZGPU_LANES", 3)))
        ext_bytes = s1["rays_extension"] * b_ray(n_tris) + s1["rays_shadow"] * b_ray(n_tris, shadow=True)
        tr_ach = ext_bytes / (s1["ms_trace"] * 1e-3) / 1e9 if s1["ms_trace"] > 0 else 0.0
        out["roofline"] = {"bound": "hbm", "kernel": "k_extend + k_shadow (closest-hit traversal inside the wavefront)", "achieved": tr_ach, "peak": peak, "unit": "GB/s",
                           "frac": tr_ach / peak, "traffic": None, "peak_kind": peak_kind,
                           "algorithmic_bytes_per_step": ext_bytes, "kernel_ms_per_step": s1["ms_trace"], "other_kernels_ms_per_step": s1["ms_shade"],
                           "share_of_device_time": s1["ms_trace"] / max(1e-9, s1["ms_trace"] + s1["ms_shade"]),
                           "how": "one step with a single lane (serial kernels): CUDA events of the library around every traversal launch, this rank"}
        # ---- end to end through the C ABI: host frame out (N > 1: shard + NCCL reduce + one D2H on rank 0)
        def estep(k):
            base = (k % n_steps_frame) * spp_step
            if world == 1:
                G.render_host_ptr(base, base + spp_step, host_frame.data_ptr(), clear=True)
            else:
                pstep(k)
                if rank == 0:
                    host_frame.copy_(frame, non_blocking=True)
        estep(0); barrier()
        esteps = max(2, min(steps, 4))
        t0 = time.perf_counter()
        for k in range(esteps):
            estep(k)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        es = rmax(time.perf_counter() - t0) / esteps
        out["e2e"] = {"value": npaths / es / 1e6, "unit": "Mpaths/s", "h2d_bytes_per_step": 28, "d2h_bytes_per_step": fh * fw * 16, "steps": esteps,
                      "api": "kzgpu_render (request in, host frame out)" if world == 1 else "kzgpu_render_device + NCCL reduce + D2H of the frame on rank 0",
                      "note": "the scene is resident; a step's input is the 28-byte kz_render_req"}
        render_s = n_steps_frame * ms * 1e-3
        readback_s = fh * fw * 16 / 50e9
        if rank == 0:            # the D2H copy of the finished frame into pinned memory, measured
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            host_frame.copy_(frame, non_blocking=True); torch.cuda.synchronize()
            ev0.record(); host_frame.copy_(frame, non_blocking=True); ev1.record(); torch.cuda.synchronize()
            readback_s = ev0.elapsed_time(ev1) * 1e-3
        out["time_to_image_s"] = {"scene_upload": upload_ms * 1e-3, "accel_build": build_ms * 1e-3, "render": render_s, "frame_readback": readback_s,
                                  "total": upload_ms * 1e-3 + build_ms * 1e-3 + render_s + readback_s,
                                  "spans": f"kzgpu_scene_upload + kzgpu_accel_build + {n_steps_frame} step(s) = {spp_total} spp + D2H (renderer.cpp:72-153 without XML/OBJ parsing)"}
        if rank == 0:
            fr = host_frame.numpy()
            wsum = float(fr[..., 3].sum())
            out["mean_rgb"] = float(fr[..., :3].sum() / max(wsum, 1e-9))
        # ---- CPU port beside it: a bounded sample of the same frame on all host cores
        if rank == 0 and world == 1 and not args.no_cpu and oracle_desc is not None:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import kzo_py
            t0 = time.perf_counter()
            OP = kzo_py.Oracle(oracle_desc)
            setup = time.perf_counter() - t0
            rect = cpu_rect or (0, 0, W, H)
            cn = (rect[2] - rect[0]) * (rect[3] - rect[1])
            cs = max(1, min(spp_step, int(2.0e6 // cn)))
            t0 = time.perf_counter()
            OP.render(0, cs, rect=rect)
            dt = time.perf_counter() - t0
            OP.close()
            cmp_ = cs * cn / dt / 1e6
            out["cpu_baseline"] = {"value": cmp_, "unit": "Mpaths/s", "cores": os.cpu_count() or 1, "kind": "port",
                                   "sample": f"sample indices 0..{cs - 1} of the {rect[2] - rect[0]}x{rect[3] - rect[1]} pixel rectangle at ({rect[0]},{rect[1]}) of the same frame ({cs * cn} paths)",
                                   "setup_s": setup, "time_to_image_s_extrapolated": W * H * spp_total / (cmp_ * 1e6)}
        return out

    def xml_leg(xml, overrides, builder, label, spp, steps=3, warmup=2, with_cpu=True, cpu_rect=None):
        hs = pk.HostScene(xml, overrides)
        d = hs.desc
        G = pk.Gpu(d, devices=(local,), builder=builder)
        st = G.stats()
        n_tris = sum(d.meshes[i].n_triangles for i in range(d.n_meshes))
        out = path_leg(G, n_tris, d.camera.width, d.camera.height, spp, spp, steps, warmup,
                       label + f", {d.camera.width}x{d.camera.height}, {spp} spp", st["ms_upload"], st["ms_build"],
                       oracle_desc=d if with_cpu else None, cpu_rect=cpu_rect)
        out["accel"] = {"builder": "sah" if builder == pk.BUILD_HOST_SAH else "lbvh", "nodes": st["bvh_nodes"], "bytes": st["bvh_bytes"]}
        out["roofline"]["traffic"] = committed_traffic(tris=n_tris, kernel="k_extend+k_shadow")
        G.close(); hs.close()
        return out

    # ------------------------------------------------------------------------------------------ the soup microbench (configs[1])
    def soup_leg(n_tris, builder, steps, with_cpu):
        sb = scenes.soup_scene(n_tris)
        prim = scenes.primary_rays(4096); inc = scenes.incoherent_rays(1 << 24, seed=0xBEEF + rank)
        d = sb.desc()
        G = pk.Gpu(d, devices=(local,), builder=builder)
        st0 = G.stats()
        batches = []
        for r in (prim, inc):
            host = torch.from_numpy(r.view(np.float32).reshape(-1, 8)).pin_memory()
            batches.append({"n": r.shape[0], "host": host, "dev": host.to(dev), "hits": torch.empty((r.shape[0], 5), dtype=torch.float32, device=dev),
                            "host_hits": torch.empty((r.shape[0], 5), dtype=torch.float32).pin_memory()})
        rays_per_step = sum(b["n"] for b in batches)

        def step():
            for k, b in enumerate(batches):
                G.trace_device(b["dev"].data_ptr(), b["n"], b["hits"].data_ptr(), shadow=(k == 1), device=0, stream=stream)
        for _ in range(3):
            step()
        barrier(); G.stats(reset=True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        st = G.stats(reset=True)
        kernel_ms = st["ms_trace"] / (steps * len(batches))
        bytes_per_launch = batches[0]["n"] * b_ray(n_tris)            # both batches hold 2^24 rays and return 20-byte hits
        ach = bytes_per_launch / (kernel_ms * 1e-3) / 1e9
        bname = "sah" if builder == pk.BUILD_HOST_SAH else "lbvh"
        out = {"value": steps * rays_per_step / (ms * 1e-3) / 1e6, "unit": "Mrays/s", "tris": n_tris, "builder": bname, "rays_per_step": rays_per_step,
               "ms_per_step": ms / steps, "accel_build_ms": st0["ms_build"], "scene_upload_ms": st0["ms_upload"], "accel_bytes": st0["bvh_bytes"],
               "primary_hit_fraction": float((batches[0]["hits"][:, 4].view(torch.int32) != -1).float().mean().item()),
               "roofline": {"bound": "hbm", "kernel": "k_trace", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                            "traffic": committed_traffic(tris=n_tris, builder=bname, kernel="k_trace"), "algorithmic_bytes_per_launch": bytes_per_launch,
                            "kernel_ms": kernel_ms, "bytes_per_ray": b_ray(n_tris), "peak_kind": peak_kind}}
        # end to end through the host-buffer C ABI (H2D + trace + D2H inside the call)
        for k, b in enumerate(batches):
            G.trace_host_ptr(b["host"].data_ptr(), b["n"], b["host_hits"].data_ptr(), shadow=(k == 1))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(2):
            for k, b in enumerate(batches):
                G.trace_host_ptr(b["host"].data_ptr(), b["n"], b["host_hits"].data_ptr(), shadow=(k == 1))
        torch.cuda.synchronize()
        es = (time.perf_counter() - t0) / 2
        out["e2e"] = {"value": rays_per_step / es / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": rays_per_step * 32, "d2h_bytes_per_step": rays_per_step * 20,
                      "api": "kzgpu_trace (pinned host buffers)",
                      "matches_device": bool(torch.equal(batches[1]["host_hits"].view(torch.int32), batches[1]["hits"].cpu().view(torch.int32)))}
        if with_cpu and rank == 0 and not args.no_cpu:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import kzo_py
            O = kzo_py.Oracle(d)
            # the SAME rays as the GPU arm: the first 2^18 of each of its two batches
            cp, ci = prim[: 1 << 18], inc[: 1 << 18]
            t0 = time.perf_counter()
            ho_p = O.trace(cp); ho_i = O.trace(ci, shadow=True)
            dt = time.perf_counter() - t0
            ok = ho_p.tobytes() == batches[0]["hits"][: 1 << 18].cpu().numpy().reshape(-1).view(pk.HIT_DTYPE).tobytes() and \
                ho_i.tobytes() == batches[1]["hits"][: 1 << 18].cpu().numpy().reshape(-1).view(pk.HIT_DTYPE).tobytes()
            out["cpu_baseline"] = {"value": (cp.shape[0] + ci.shape[0]) / dt / 1e6, "unit": "Mrays/s", "cores": os.cpu_count() or 1, "kind": "port",
                                   "sample": "the first 2^18 rays of each of the two GPU batches (identical ray arrays), once", "hits_match_gpu": bool(ok)}
            O.close()
        G.close()
        return out

    # ------------------------------------------------------------------------------------------ headline: configs[4]
    t0 = time.perf_counter()
    P, F = scenes.hash_soup_torch(args.tris, device=dev)
    torch.cuda.synchronize()
    gen_s = time.perf_counter() - t0
    sb = scenes.big_scene(args.tris, args.width, args.height, SPP_TOTAL, positions=P.data_ptr(), indices=F.data_ptr(), keep=(P, F))
    G = pk.Gpu(sb.desc(), devices=(local,), builder=pk.BUILD_LBVH)
    st0 = G.stats()
    oracle_desc = None
    if rank == 0 and world == 1 and not args.no_cpu:
        # the CPU port needs the triangles in host memory: copy them back (they were generated on the device)
        Ph = P.cpu().numpy(); Fh = F.cpu().numpy().view(np.uint32)
        sbo = scenes.big_scene(args.tris, args.width, args.height, SPP_TOTAL, positions=Ph, indices=Fh)
        oracle_desc = sbo.desc()
    del P, F
    sb._keep.clear()          # the library copied what it needs (records + accel live in HBM): free the generator's arrays
    torch.cuda.empty_cache()
    W, H = args.width, args.height
    head = path_leg(G, args.tris, W, H, SPP_PER_STEP, SPP_TOTAL, args.steps, args.warmup, headline_config(args, world)["workload"], st0["ms_upload"], st0["ms_build"],
                    oracle_desc=oracle_desc, cpu_rect=(W // 4, H // 4, W // 4 + W // 2, H // 4 + H // 2) if args.tris > 100000 else None, clocks_on=True,
                    dump_dir=args.dump_outputs)
    head["roofline"]["traffic"] = committed_traffic(tris=args.tris, kernel="k_extend")
    G.close()
    oracle_desc = None
    torch.cuda.empty_cache()

    extra = {}
    if "c0" in legs:
        extra["warmstudio"] = xml_leg(WARM_XML, {"camera.width": "i:512", "camera.height": "i:512", "sampler.type": "s:stratified", "sampler.sampleCount": "i:64"},
                                      pk.BUILD_HOST_SAH, "BASELINE configs[0]: scene/2022_q1/WarmStudio/WarmStudio.xml (17952 triangles, kiss + diffuse + mesh light)", 64)
    if "c2" in legs or "c3" in legs:
        import importlib.util
        spec = importlib.util.spec_from_file_location("make_configs", os.path.join(ROOT, "tests", "data", "make_configs.py"))
        mc = importlib.util.module_from_spec(spec); spec.loader.exec_module(mc)
        cfg = args.cfg_dir or tempfile.mkdtemp(prefix="kz_bench_cfg_")       # the tree may be read-only
        try:
            mc.generate(cfg, tex_res=4096)
            if "c2" in legs:
                extra["lookdev_4k"] = xml_leg(os.path.join(cfg, "c3_lookdev_4k.xml"), {}, pk.BUILD_HOST_SAH,
                                              "BASELINE configs[2] stand-in: normalmap + kiss + 4096^2 image textures through blend, thin lens", 64,
                                              cpu_rect=(1440, 810, 2400, 1350))
            if "c3" in legs:
                extra["pmj02bn_1080p"] = xml_leg(os.path.join(cfg, "c4_pmj02bn_1080p.xml"), {}, pk.BUILD_HOST_SAH,
                                                 "BASELINE configs[3] stand-in: pmj02bn sampler, traceBias 1e-3, regularization, low-poly smooth sphere", 64,
                                                 cpu_rect=(480, 270, 1440, 810))
        finally:
            if not args.cfg_dir:
                shutil.rmtree(cfg, ignore_errors=True)
    if "soup1m" in legs:
        extra["soup_1m"] = soup_leg(1 << 20, pk.BUILD_HOST_SAH, 6, True)
    if "soup10m" in legs:
        extra["soup_10m"] = soup_leg(10_000_000, pk.BUILD_LBVH, 6, True)

    if rank == 0:
        line = {"metric": "Mpaths/s", "value": head["value"], "unit": "Mpaths/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": headline_config(args, world),            # identical, key by key, to the reference arm's
                "scene": {"generation_on_device_s": gen_s, "upload_ms": st0["ms_upload"], "accel_build_ms": st0["ms_build"], "accel_nodes": st0["bvh_nodes"], "accel_bytes": st0["bvh_bytes"]},
                "mrays_per_s": head["mrays_per_s"], "rays_per_path": head["rays_per_path"],
                "roofline": head["roofline"], "path_roofline": head["path_roofline"], "cpu_baseline": head.get("cpu_baseline"), "e2e": head["e2e"],
                "time_to_image_s": head["time_to_image_s"], "mean_rgb": head.get("mean_rgb"),
                "gpu_launches": head["gpu_launches"], "clocks": head.get("clocks"), "legs": extra}
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
