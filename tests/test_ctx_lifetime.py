"""Context lifetime: a context gives back every device resource it made, after a full create -> destroy cycle and after a failed
kzgpu_create, and a failed create leaves nothing behind that later contexts could trip over."""
import ctypes as C

import numpy as np
import pytest

import scenes
import pykazen as pk

N_TRIS = 1 << 20
LEAK_TOL = 64 << 20       # bytes of free device memory that three cycles may lose (one cycle holds gigabytes)


def _cycle(torch, P, F, Pm, rays):
    """create, upload, SAH build, render, LBVH build, mesh_update + refit, trace, render_device into a torch tensor, destroy"""
    sb = scenes.big_scene(N_TRIS, width=512, height=512, spp=64, positions=P, indices=F)     # keeps the desc's arrays alive
    d = sb.desc()
    G = pk.Gpu(d, builder=pk.BUILD_HOST_SAH)
    try:
        G.render(0, 64)                                               # 2^24 paths: two lanes of path pools, primary-hit hints
        assert G.lib.kzgpu_accel_build(G.h, C.c_int(pk.BUILD_LBVH)) == 0
        G.mesh_update(0, Pm)
        G.refit()
        hits = G.trace(rays)
        assert (hits["geom_id"] != pk.KZ_INVALID_ID).mean() > 0.5
        H, W, _ = G.frame_shape()
        frame = torch.empty((H, W, 4), dtype=torch.float32, device="cuda")
        stream = torch.cuda.Stream()
        assert G.render_device(0, 16, stream=stream.cuda_stream, frame_ptr=frame.data_ptr()) == frame.data_ptr()
        stream.synchronize()
        assert G.stats()["paths"] == 512 * 512 * (64 + 16)
        del frame
    finally:
        G.close()


@pytest.mark.gpu
def test_full_cycles_release_device_memory(gpu_lib):
    torch = pytest.importorskip("torch")
    P = scenes.hash_soup_numpy(N_TRIS)
    F = np.arange(3 * N_TRIS, dtype=np.uint32).reshape(-1, 3)
    Pm = P + np.random.default_rng(5).normal(0.0, 1e-3, P.shape).astype(np.float32)
    rays = scenes.incoherent_rays(1 << 16)

    def free():
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        return torch.cuda.mem_get_info()[0]

    _cycle(torch, P, F, Pm, rays)                                     # warm-up: CUDA context, module load, torch allocator
    before = free()
    for _ in range(3):
        _cycle(torch, P, F, Pm, rays)
    after = free()
    assert before - after < LEAK_TOL, f"three create -> destroy cycles lost {(before - after) / 2**20:.1f} MiB"


@pytest.mark.gpu
def test_failed_create_leaves_no_context(kzo, gpu_lib):
    torch = pytest.importorskip("torch")
    lib = C.CDLL(gpu_lib)
    lib.kzgpu_last_error.restype = C.c_char_p
    for ids, code, msg in (((0, 0), -1, b"listed twice"), ((0, torch.cuda.device_count()), -2, b"out of range")):
        h = C.c_void_p(1)
        arr = (C.c_int * 2)(*ids)
        assert lib.kzgpu_create(arr, 2, C.byref(h)) == code, ids
        assert h.value is None, ids
        assert msg in lib.kzgpu_last_error(None), ids
    # a context created afterwards works: hits bit for bit and the image as the oracle's
    sb = scenes.cornell_scene(64, 64, 16, "stratified")
    d = sb.desc()
    G, O = pk.Gpu(d, builder=pk.BUILD_LBVH), kzo.Oracle(d)
    rays = np.concatenate([scenes.primary_rays(64, 39.0, (0, 0, -3.4)), scenes.incoherent_rays(20000, extent=0.95)])
    assert G.trace(rays).tobytes() == O.trace(rays).tobytes()
    rg, _ = G.resolve(G.render())
    ro, _ = O.resolve(O.render())
    assert scenes.rel_mse(rg, ro).max() < 2e-4
    G.close(); O.close()
