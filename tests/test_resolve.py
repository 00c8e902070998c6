"""The resolve (k_resolve: film / weight, then Bitmap::savePNG's 8-bit sRGB conversion) against the oracle's kzo_resolve, bit for
bit on adversarial frames: every float of the sRGB power branch, the floats on either side of each 8-bit code boundary, and
special weights and values, on films whose sizes leave ragged edges in the kernel's 32 x 8 thread blocks.  A mean over random
frames cannot see a resolve that is one code off for a few hundred linear values; these inputs can."""
import numpy as np
import pytest

import scenes
import pykazen as pk

pytestmark = pytest.mark.gpu

SRGB_LO = np.float32(0.0031308)            # toSRGB (color.h): v <= 0.0031308f takes the linear branch
FILTERS = ("box", "gaussian")              # border 0 (radius 0.5) and border 2 (radius 2)
SHAPES = ((1, 1), (7, 5), (3840, 2160))


def _bits(x):
    return int(np.float32(x).view(np.int32))


def _open(kzo, width, height, filt):
    """oracle + product on one scene desc: the film size comes from the camera, the border from the filter"""
    sb = pk.SceneBuilder()
    sb.mesh(*scenes.quad((-1, -1, 0), (1, -1, 0), (1, 1, 0), (-1, 1, 0)), sb.bsdf_diffuse())
    sb.set_camera(width, height, 40.0, pk.lookat((0, 0, -3), (0, 0, 0), (0, 1, 0)))
    sb.set_filter(filt)
    d = sb.desc()
    O, G = kzo.Oracle(d), pk.Gpu(d)
    O.sb = G.sb = sb                       # the desc points into arrays the builder owns
    return O, G


def _frames(G, texels):
    """bordered frames holding `texels` (n, 4) in row-major order, as many as needed (the last one padded with (0, 0, 0, 1));
    the border holds random bit patterns (NaNs, infinities, huge values) that the resolve must never read"""
    H, W, b = G.frame_shape()
    w, h = W - 2 * b, H - 2 * b
    rng = np.random.default_rng(len(texels))
    for s in range(0, len(texels), w * h):
        f = rng.integers(-2 ** 31, 2 ** 31, (H, W, 4), dtype=np.int64).astype(np.int32).view(np.float32)
        inner = np.zeros((w * h, 4), np.float32); inner[:, 3] = 1.0
        part = texels[s: s + w * h]
        inner[: len(part)] = part
        f[b: b + h, b: b + w] = inner.reshape(h, w, 4)
        yield s, len(part), f


def _canonical_bits(x):
    """int32 view with every NaN mapped to one pattern: IEEE 754 leaves the NaN payload of a division open, and x86 (0/0 ->
    0xffc00000, NaN operands propagated) and the GPU (0x7fffffff) fill it differently.  Everything else compares bit for bit,
    signed zeros and subnormals included."""
    v = np.ascontiguousarray(x, np.float32).reshape(-1).view(np.int32).copy()
    v[np.isnan(x.reshape(-1))] = 0x7FC00000
    return v


def _resolve_both(O, G, texels):
    """oracle rgb, oracle codes, product rgb, product codes of the texels: (n, 3) float32 / uint8 each"""
    n = len(texels)
    ro, so, rg, sg = (np.empty((n, 3), np.float32), np.empty((n, 3), np.uint8), np.empty((n, 3), np.float32), np.empty((n, 3), np.uint8))
    for s, m, f in _frames(G, texels):
        a, b = O.resolve(f), G.resolve(f)
        ro[s: s + m], so[s: s + m] = a[0].reshape(-1, 3)[:m], a[1].reshape(-1, 3)[:m]
        rg[s: s + m], sg[s: s + m] = b[0].reshape(-1, 3)[:m], b[1].reshape(-1, 3)[:m]
    return ro, so, rg, sg


def _assert_same(texels, ro, so, rg, sg):
    bad_rgb = _canonical_bits(ro) != _canonical_bits(rg)
    bad_code = (so != sg).reshape(-1)
    where = np.flatnonzero(bad_rgb | bad_code)[:8]
    show = [(texels[i // 3].tolist(), float(ro.reshape(-1)[i]), float(rg.reshape(-1)[i]), int(so.reshape(-1)[i]), int(sg.reshape(-1)[i]))
            for i in where]
    assert not bad_rgb.any() and not bad_code.any(), \
        f"{int(bad_rgb.sum())} rgb values and {int(bad_code.sum())} 8-bit codes differ; (texel, oracle rgb, gpu rgb, oracle code, gpu code): {show}"


def _power_branch_texels(first, count):
    """floats first .. first+count-1 of (0.0031308f, 1], three per texel, weight 1"""
    lo = _bits(SRGB_LO) + 1
    v = np.arange(lo + first, lo + first + count, dtype=np.int64).astype(np.int32).view(np.float32)
    v = np.concatenate([v, np.full((-count) % 3, 0.5, np.float32)]).reshape(-1, 3)
    return np.concatenate([v, np.ones((len(v), 1), np.float32)], 1)


@pytest.mark.parametrize("filt", FILTERS)
def test_resolve_every_float_of_the_power_branch(kzo, gpu_lib, filt):
    """all 70 439 396 floats in (0.0031308, 1] as rgb with w = 1, 3 x 3840 x 2160 of them per frame: every input on which the
    8-bit code depends on how powf, the multiply by 1.055 and the subtraction of 0.055 round"""
    O, G = _open(kzo, 3840, 2160, filt)
    total = _bits(1.0) - _bits(SRGB_LO)
    assert total == 70_439_396
    per = 3 * 3840 * 2160
    n_bad_rgb = n_bad_code = 0
    examples = []
    for first in range(0, total, per):
        t = _power_branch_texels(first, min(per, total - first))
        ro, so, rg, sg = _resolve_both(O, G, t)
        bad_rgb = _canonical_bits(ro) != _canonical_bits(rg)
        bad_code = (so != sg).reshape(-1)
        n_bad_rgb += int(bad_rgb.sum()); n_bad_code += int(bad_code.sum())
        for i in np.flatnonzero(bad_code)[: 8 - len(examples)]:
            examples.append((float(t[:, :3].reshape(-1)[i]), int(so.reshape(-1)[i]), int(sg.reshape(-1)[i])))
    assert n_bad_rgb == 0 and n_bad_code == 0, f"{n_bad_rgb} rgb values and {n_bad_code} 8-bit codes differ; (linear, oracle, gpu): {examples}"
    O.close(); G.close()


def _srgb_code_f32(x):
    """toSRGB + savePNG's scale and truncation restated in float32 (powf as the double power rounded once), for locating the
    code boundaries; the test compares the two libraries, not this function"""
    x = np.asarray(x, np.float32)
    with np.errstate(invalid="ignore"):
        p = (np.asarray(x, np.float64) ** np.float64(np.float32(1.0) / np.float32(2.4))).astype(np.float32)
    s = np.where(x <= SRGB_LO, np.float32(12.92) * x, (np.float32(1.055) * p).astype(np.float32) - np.float32(0.055)).astype(np.float32)
    return np.clip(np.float32(255) * s, 0, 255).astype(np.int32)


def _boundary_values(half=64):
    """for each 8-bit code k in 1..255 the `half` floats on either side of the smallest linear value whose code is k
    (found by bisection over float bit patterns, above 1 for k = 255): (255, 2 * half) float32"""
    k = np.arange(1, 256)
    lo = np.zeros(255, np.int64); hi = np.full(255, _bits(4.0), np.int64)
    while np.any(hi - lo > 1):
        mid = (lo + hi) // 2
        up = _srgb_code_f32(mid.astype(np.int32).view(np.float32)) >= k
        hi = np.where(up, mid, hi); lo = np.where(up, lo, mid)
    return (hi[:, None] + np.arange(-half, half)[None, :]).astype(np.int32).view(np.float32)


def _special_texels(seed=17):
    f32 = np.float32
    tiny, sub = np.finfo(np.float32).tiny, f32(1e-40)
    values = np.array([0.0, -0.0, 1e-45, sub, tiny, 1e-20, 1e-4, 0.001, np.nextafter(SRGB_LO, f32(0)), SRGB_LO,
                       np.nextafter(SRGB_LO, f32(1)), 0.04045, 0.2, 0.5, np.nextafter(f32(1), f32(0)), 1.0, np.nextafter(f32(1), f32(2)),
                       1.0001, 1.5, 10.0, 1e30, 3.4028235e38, -1e-30, -0.001, -0.5, -1.0, -3e38, np.inf, -np.inf, np.nan], np.float32)
    weights = np.array([1.0, 0.0, -0.0, -1.0, -0.25, 1e-45, sub, tiny, 1e-30, 0.3, 1.0 / 3.0, 0.7, 2.0, 3.0, 17.25, 1e6, 1e30,
                        3.4028235e38, np.inf, -np.inf, np.nan], np.float32)
    n = len(values)
    rows = []
    for j, w in enumerate(weights):                      # every value under every weight, the channels rotated against each other
        for i in range(n):
            rows.append((values[i], values[(i + 7 + j) % n], values[(i + 13 + 2 * j) % n], w))
    rng = np.random.default_rng(seed)
    m = 4096                                             # accumulated splat sums: rgb = colour * weight, w a sum of filter taps
    w = rng.uniform(0.01, 40.0, m).astype(np.float32)
    c = (rng.uniform(0, 1.3, (m, 3)) * w[:, None]).astype(np.float32)
    return np.concatenate([np.array(rows, np.float32), np.concatenate([c, w[:, None]], 1)])


@pytest.mark.parametrize("filt", FILTERS)
@pytest.mark.parametrize("shape", SHAPES[1:])
def test_resolve_code_boundaries(kzo, gpu_lib, filt, shape):
    """the 64 floats on either side of every 8-bit code boundary, linear branch, branch point and power branch (w = 1)"""
    v = _boundary_values().reshape(-1)
    v = np.concatenate([v, np.full((-len(v)) % 3, 0.5, np.float32)]).reshape(-1, 3)
    t = np.concatenate([v, np.ones((len(v), 1), np.float32)], 1)
    O, G = _open(kzo, *shape, filt)
    ro, so, rg, sg = _resolve_both(O, G, t)
    _assert_same(t, ro, so, rg, sg)
    codes = so.reshape(-1)[: 255 * 128].reshape(255, 128).astype(int)
    k = np.arange(1, 256)
    assert np.all(codes.min(1) <= k - 1) and np.all(codes.max(1) >= k), "the windows do not straddle their code boundaries"
    O.close(); G.close()


@pytest.mark.parametrize("filt", FILTERS)
@pytest.mark.parametrize("shape", SHAPES)
def test_resolve_weights_and_specials(kzo, gpu_lib, filt, shape):
    """zero, negative, subnormal, huge, infinite and NaN weights; values at and around the branch point, above 1, signed zeros,
    subnormals, infinities and NaN; and accumulated sums with non-unit weights (the division rounds)"""
    t = _special_texels()
    O, G = _open(kzo, *shape, filt)
    _assert_same(t, *_resolve_both(O, G, t))
    O.close(); G.close()
