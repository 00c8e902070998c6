"""The benchmarked render path against the oracle: the headline's 4K camera, 1024-spp stratified sampler, gaussian filter,
constant environment light and integrator (scenes.big_scene) with a smaller soup; the on-device soup generator; and the
entry points a timed step goes through (kzgpu_render_device on a torch stream into a torch frame, kzgpu_render into pinned
host memory), including the sample ranges past 0, the primary-hit hints and the three lanes that only a frame of this size
turns on."""
import numpy as np
import pytest

import scenes
import pykazen as pk

W4K, H4K, SPP = 3840, 2160, 1024
RANGES = ((0, 64), (960, 1024))                                # the first and the last 64-index step of a frame
RECTS = ((3808, 2144, 3840, 2160), (1904, 1072, 1936, 1088))   # 32 x 16 at the far corner (x > 2048) and at the centre
IMAGE_RELMSE_TOL = 2e-4                                        # as test_gpu_parity: GPU vs oracle at equal samples


def _divide(f):
    f = np.asarray(f, np.float64)
    w = f[..., 3:]
    return np.where(w != 0, f[..., :3] / np.where(w != 0, w, 1), 0)


def _crop(frame, rect, b):
    """resolved rgb of the rectangle and of the texels its filter footprint reaches (frame coordinates: pixel + border)"""
    x0, y0, x1, y1 = rect
    return _divide(frame[y0: y1 + 2 * b, x0: x1 + 2 * b])


# ------------------------------------------------------------------------------------------------ CPU: generator, sampler, render
def test_hash_soup_torch_matches_numpy():
    """the headline's scene (torch generator) is the scene of the CPU reference and of every soup test (numpy generator): bit
    for bit, with both chunk loops crossing chunk boundaries and ending on a ragged chunk"""
    import torch
    n = 3 * (1 << 20) + 5
    P, F = scenes.hash_soup_torch(n, device="cpu", chunk=1 << 20)
    Pn = scenes.hash_soup_numpy(n, chunk=1 << 20)
    assert P.dtype == torch.float32 and P.shape == (3 * n, 3)
    assert P.numpy().tobytes() == Pn.tobytes()
    assert F.numpy().astype(np.uint32).tobytes() == np.arange(3 * n, dtype=np.uint32).tobytes()
    # a window of the numpy generator is the same slice of the whole
    assert scenes.hash_soup_numpy(n, first=(1 << 20) - 7, count=19).tobytes() == Pn[3 * ((1 << 20) - 7): 3 * ((1 << 20) + 12)].tobytes()


def _sampler_triples(sample_count, rng):
    pix = [(W4K - 1, H4K - 1), (0, H4K - 1), (W4K - 1, 0), (0, 0), (2048, 1080), (2047, 2047)]
    idx = sorted({0, 63, 64, 960, 1023, sample_count - 1} & set(range(sample_count)))
    tr = [(x, y, j) for (x, y) in pix for j in idx]
    r = np.stack([rng.integers(0, W4K, 2000), rng.integers(0, H4K, 2000), rng.integers(0, sample_count, 2000)], 1)
    return np.concatenate([np.array(tr), r]).astype(np.int32)


@pytest.mark.parametrize("spp", [1024, 4096, 900])
def test_sampler_headline_sizes_cpu(kzo, emu, spp):
    """the stratified sampler at the headline's 1024 spp (and 4096, and the non-power-of-two square 900), 4K pixel coordinates:
    the device routines compiled for the host draw the oracle's sequences bit for bit"""
    sb = scenes.big_scene(16, W4K, H4K, spp)
    assert sb.sampler.sample_count == spp
    d = sb.desc()
    O, E = kzo.Oracle(d), emu.Emu(d)
    tr = _sampler_triples(spp, np.random.default_rng(spp))
    pat = "P2" + "1111" * 2 + "12" * 3 + "1"
    assert O.sample_dump(tr, pat).tobytes() == E.sample_dump(tr, pat).tobytes()
    O.close(); E.close()


@pytest.fixture(scope="module")
def small_headline(kzo, emu):
    sb = scenes.big_scene(1 << 14, W4K, H4K, SPP)      # owns the arrays the desc points to
    d = sb.desc()
    O, E = kzo.Oracle(d), emu.Emu(d)
    yield O, E
    O.close(); E.close()


@pytest.mark.parametrize("rect", RECTS)
@pytest.mark.parametrize("spp_range", RANGES)
def test_render_headline_rects_cpu(small_headline, rect, spp_range):
    """rectangles of the 4K film, first and last step of the 1024-spp frame, 2^14-triangle soup: host-compiled device routines
    vs oracle at the bars of test_hostemu.test_render_matches_oracle"""
    O, E = small_headline
    s0, s1 = spp_range
    keys = ("paths", "rays_extension", "vertices")
    before = [(O.stats()[k], E.stats()[k]) for k in keys]
    fo, fe = O.render(s0, s1, rect=rect), E.render(s0, s1, rect=rect)
    assert fo[..., 3].any()
    assert np.allclose(fo[..., 3], fe[..., 3], rtol=1e-5, atol=1e-6)
    b = O.frame_shape()[2]
    assert scenes.rel_mse(_crop(fe, rect, b), _crop(fo, rect, b)).max() < 1e-6
    so, se = O.stats(), E.stats()
    delta = [(so[k] - o, se[k] - e) for k, (o, e) in zip(keys, before)]
    assert delta[0] == (32 * 16 * 64, 32 * 16 * 64) and all(o == e for o, e in delta), delta


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_hash_soup_torch_on_device(gpu_lib):
    """hash_soup_torch(10^8) on the GPU (the headline scene) against the numpy generator on sampled windows: both ends, the
    middle, and across every boundary of the torch generator's 2^24-triangle chunks"""
    import torch
    n, win = 10 ** 8, 1 << 16
    P, F = scenes.hash_soup_torch(n, device="cuda")
    starts = [0, n - win, n // 2 - win // 2] + [(k << 24) - win // 2 for k in range(1, (n >> 24) + 1)]
    for first in starts:
        got = P[3 * first: 3 * (first + win)].cpu().numpy()
        assert got.tobytes() == scenes.hash_soup_numpy(n, first=first, count=win).tobytes(), first
    assert torch.equal(F[-2:].cpu(), torch.tensor([[3 * n - 6, 3 * n - 5, 3 * n - 4], [3 * n - 3, 3 * n - 2, 3 * n - 1]], dtype=torch.int32))
    del P, F
    torch.cuda.empty_cache()


@pytest.fixture(scope="module")
def headline(kzo, gpu_lib):
    """the headline scene at 2^20 triangles: LBVH, default options (primary_hint 1 turns the hints on at this size)"""
    sb = scenes.big_scene(1 << 20, W4K, H4K, SPP)
    d = sb.desc()
    G = pk.Gpu(d, builder=pk.BUILD_LBVH)
    O = kzo.Oracle(d)
    yield G, O
    G.close(); O.close()


@pytest.mark.gpu
def test_headline_rects_match_oracle(headline):
    """render_device into a torch frame on a non-default torch stream, as a timed step does, vs the oracle; the second range
    starts past 0 and is seeded with the hints the first one left"""
    import torch
    G, O = headline
    H, W, b = G.frame_shape()
    stream = torch.cuda.Stream()
    frame = torch.empty((H, W, 4), dtype=torch.float32, device="cuda")
    for rect in RECTS:
        for s0, s1 in RANGES:
            G.stats(reset=True)
            G.render_device(s0, s1, clear=True, stream=stream.cuda_stream, frame_ptr=frame.data_ptr(), rect=rect)
            stream.synchronize()
            fg = frame.cpu().numpy()
            st = G.stats(reset=True)
            fo = O.render(s0, s1, rect=rect)
            assert np.allclose(fo[..., 3], fg[..., 3], rtol=1e-4, atol=1e-5)
            err = scenes.rel_mse(_crop(fg, rect, b), _crop(fo, rect, b))
            assert err.max() < IMAGE_RELMSE_TOL, (rect, s0, err)
            assert st["paths"] == 32 * 16 * 64
            if s0 == 960:
                assert st["rays_seeded"] > 0


def _render_stats(G):
    st = G.stats(reset=True)
    return st["paths"], st["rays_extension"], st["rays_shadow"], st["vertices"]


@pytest.mark.gpu
def test_render_device_semantics(gpu_lib):
    """kzgpu_render_device against kzgpu_render on one context, 4.2 M paths (two lanes): clear = 1 clears the caller's frame on
    the caller's stream; clear = 0 adds to what the stream wrote just before (the second lane must wait for it); nothing carries
    over into the next clear = 1 request; rectangles; kzgpu_render into pinned host memory with and without clear"""
    import torch
    sb = scenes.cornell_scene(256, 256, 64, "stratified")
    G = pk.Gpu(sb.desc())
    H, W, b = G.frame_shape()
    G.stats(reset=True)
    ref = G.render(0, 64)
    st_ref = _render_stats(G)
    close = dict(rtol=1e-4, atol=1e-5)
    stream = torch.cuda.Stream()
    frame = torch.empty((H, W, 4), dtype=torch.float32, device="cuda")
    fill = torch.rand((H, W, 4), dtype=torch.float32, device="cuda", generator=torch.Generator("cuda").manual_seed(5))
    torch.cuda.synchronize()
    with torch.cuda.stream(stream):
        torch.cuda._sleep(20_000_000)                  # the stream is still busy when the request is enqueued
        frame.fill_(7.0)
    G.render_device(0, 64, clear=True, stream=stream.cuda_stream, frame_ptr=frame.data_ptr())
    stream.synchronize()
    assert np.allclose(frame.cpu().numpy(), ref, **close)
    assert _render_stats(G) == st_ref
    with torch.cuda.stream(stream):
        torch.cuda._sleep(20_000_000)
        frame.copy_(fill)
    G.render_device(0, 64, clear=False, stream=stream.cuda_stream, frame_ptr=frame.data_ptr())
    stream.synchronize()
    assert np.allclose(frame.cpu().numpy(), fill.cpu().numpy() + ref, **close)
    G.render_device(0, 64, clear=True, stream=stream.cuda_stream, frame_ptr=frame.data_ptr())
    stream.synchronize()
    assert np.allclose(frame.cpu().numpy(), ref, **close)
    G.stats(reset=True)
    rect = (37, 5, 203, 250)
    G.render_device(0, 64, clear=True, stream=stream.cuda_stream, frame_ptr=frame.data_ptr(), rect=rect)
    stream.synchronize()
    st_rect = _render_stats(G)
    assert st_rect[0] == 166 * 245 * 64
    assert np.allclose(frame.cpu().numpy(), G.render(0, 64, rect=rect), **close)
    assert _render_stats(G) == st_rect
    # kzgpu_render into pinned torch host memory
    host = torch.full((H, W, 4), 3.0, dtype=torch.float32).pin_memory()
    G.render_host_ptr(0, 64, host.data_ptr(), clear=True)
    assert np.allclose(host.numpy(), ref, **close)
    host.copy_(fill.cpu())
    G.render_host_ptr(0, 64, host.data_ptr(), clear=False)
    assert np.allclose(host.numpy(), fill.cpu().numpy() + ref, **close)
    G.close()


@pytest.mark.gpu
def test_headline_shards_sum_to_the_step(headline):
    """the strong-scaling decomposition of a timed step: the eight shards of [960, 1024) add up to the whole step"""
    import torch
    G, _ = headline
    H, W, _ = G.frame_shape()
    stream = torch.cuda.Stream()
    whole = torch.empty((H, W, 4), dtype=torch.float32, device="cuda")
    part = torch.empty_like(whole)
    acc = torch.zeros((H, W, 4), dtype=torch.float64, device="cuda")
    G.render_device(960, 1024, clear=True, stream=stream.cuda_stream, frame_ptr=whole.data_ptr())
    paths = 0
    for r in range(8):
        s0, s1 = pk.shard_range(960, 1024, r, 8)
        G.render_device(s0, s1, clear=True, stream=stream.cuda_stream, frame_ptr=part.data_ptr())
        with torch.cuda.stream(stream):
            acc += part
        paths += W4K * H4K * (s1 - s0)
    stream.synchronize()
    assert paths == W4K * H4K * 64
    assert torch.allclose(acc.float(), whole, rtol=1e-4, atol=1e-5)


@pytest.mark.gpu
def test_headline_step_three_lanes(headline):
    """one whole 4K step [960, 1024) of the 2^20 soup: 530 M paths, enough for three lanes, against one lane with 2^22-path
    pools (identical counters, images equal up to the order of the float sums), and against three rectangles that tile the
    film (every texel's weight: no path dropped or repeated)"""
    import torch
    G, _ = headline
    H, W, b = G.frame_shape()
    stream = torch.cuda.Stream()

    def step(rect=None):
        f = torch.empty((H, W, 4), dtype=torch.float32, device="cuda")
        G.render_device(960, 1024, clear=True, stream=stream.cuda_stream, frame_ptr=f.data_ptr(), rect=rect)
        stream.synchronize()
        return f.cpu().numpy(), G.stats(reset=True)

    G.stats(reset=True)
    f3, st3 = step()
    G.configure("lanes", 1); G.configure("pool_log2", 22)
    try:
        f1, st1 = step()
    finally:
        G.configure("lanes", 3); G.configure("pool_log2", 24)
    keys = ("paths", "rays_extension", "rays_shadow", "vertices")
    assert st3["paths"] == W4K * H4K * 64
    assert [st3[k] for k in keys] == [st1[k] for k in keys]
    assert scenes.rel_mse(_divide(f3[b: b + H4K, b: b + W4K]), _divide(f1[b: b + H4K, b: b + W4K])).max() < 1e-9
    tiles = [(0, 0, 1000, H4K), (1000, 0, W4K, 1234), (1000, 1234, W4K, H4K)]
    wsum = np.zeros(f3.shape[:2], np.float64)
    paths = 0
    for t in tiles:
        ft, st = step(t)
        wsum += ft[..., 3]
        paths += st["paths"]
    assert paths == st3["paths"]
    assert np.allclose(wsum, f3[..., 3], rtol=1e-4, atol=1e-5)
    assert abs(wsum.sum() - f3[..., 3].astype(np.float64).sum()) <= 1e-6 * wsum.sum()
