"""Environment importance sampling in path_mis (kz_integrator_desc::env_sampling, kz_env.h).

CPU: the luminance table of the host-compiled bodies equals a numpy restatement byte for byte; the chain classification agrees with
kz_background; the density is positive where the background is, integrates to 1, and the sampler draws cells with the table's
probabilities; the C++ host parses envSampling.
GPU: the probe matches the host emulation; on the sun studio the estimate with the flag on agrees with the reference estimator within
the shards' spread and is less noisy; without a counted environment the flag changes nothing."""
import math
import os

import numpy as np
import pytest

import env_scenes
import pykazen as pk

C0, C1, C2 = (np.float64(np.float32(c)) for c in (0.212671, 0.715160, 0.072169))


# ------------------------------------------------------------------------------------------------ numpy restatement of the table
def table_numpy(img=None, const_hw=(32, 64)):
    """(row CDFs, marginal, cell probabilities, total) of kz_env.h's rules; img None: a constant chain"""
    if img is None:
        H, W = const_hw
        m = np.ones((H, W))
    else:
        img = np.asarray(img, np.float32)
        H, W = img.shape[:2]
        x = img.astype(np.float64)
        lum = np.abs(x[..., 0] * C0 + x[..., 1] * C1 + x[..., 2] * C2)
        m = np.zeros((H, W))
        for j in range(-2, 3):
            for i in range(-2, 3):
                yy = (np.arange(H) + j) % H; xx = (np.arange(W) + i) % W
                m = np.maximum(m, lum[yy][:, xx])
    sines = np.array([math.sin(math.pi * (r + 0.5) / H) for r in range(H)])
    w = m * sines[:, None]
    acc = np.cumsum(w, axis=1)                  # sequential, as one thread per row sums
    rsum = acc[:, -1]
    cdf = np.zeros((H, W + 1), np.float32)
    uni = (np.arange(1, W + 1) / W).astype(np.float32)
    for r in range(H):
        cdf[r, 1:] = (acc[r] / rsum[r]).astype(np.float32) if rsum[r] > 0 else uni
    cdf[:, W] = 1
    macc = np.cumsum(rsum)
    total = macc[-1]
    marg = np.zeros(H + 1, np.float32)
    marg[1:] = (macc / total).astype(np.float32) if total > 0 else (np.arange(1, H + 1) / H).astype(np.float32)
    marg[H] = 1
    prob = (w / total).astype(np.float32) if total > 0 else np.zeros((H, W), np.float32)
    return cdf, marg, prob, total


def sky_scene(img=None, chain=None, env_sampling=True, kind="path_mis"):
    sb = pk.SceneBuilder()
    P, F = np.array([[0, -1, -1], [0, -1, 1], [0, 1, 1]], np.float32), np.array([[0, 1, 2]], np.uint32)
    sb.mesh(P, F, sb.bsdf_diffuse())
    if chain is not None:
        chain(sb)
    elif img is not None:
        env_scenes.sky_background(sb, img)
    sb.set_camera(16, 16, 40.0, pk.lookat((-3, 0, 0), (0, 0, 0), (0, 1, 0)))
    sb.set_integrator(env_sampling=env_sampling, kind=kind)
    return sb


def gpu(sb, **kw):
    """pykazen.Gpu over `sb`'s scene; the context keeps `sb` (which owns the arrays the scene points at) alive"""
    g = pk.Gpu(sb.desc(), **kw)
    g.builder = sb
    return g


def emu(env, sb):
    e = env.EnvEmu(sb.desc())
    e.builder = sb
    return e


@pytest.fixture(scope="module")
def env():
    import env_emu
    env_emu.build()
    return env_emu


def _one_texel(h=8, w=16):
    img = np.zeros((h, w, 3), np.float32); img[5, 3] = (0.0, 2.0, 0.0)
    return img


TABLE_CASES = {
    "sun256x128": lambda: env_scenes.sun_sky(),
    "1x1": lambda: np.array([[[0.5, 0.25, 2.0]]], np.float32),
    "3x2": lambda: np.random.default_rng(1).uniform(0, 3, (2, 3, 3)).astype(np.float32),
    "5x7": lambda: np.random.default_rng(2).uniform(-1, 3, (7, 5, 3)).astype(np.float32),
    "one_texel": _one_texel,
    "constant": None,
}


@pytest.mark.parametrize("case", sorted(TABLE_CASES))
def test_table_matches_numpy_restatement(env, case):
    make = TABLE_CASES[case]
    img = make() if make else None
    if img is None:
        sb = sky_scene(chain=lambda sb: setattr(sb, "background", sb.tex_background(2.0, sb.tex_constant((0.3, 0.4, 0.5)))))
    else:
        sb = sky_scene(img)
    e = emu(env, sb)
    cdf, marg, prob = e.table()
    rc, rm, rp, total = table_numpy(img)
    assert e.kind == (env.ENV_CONSTANT if img is None else env.ENV_IMAGE) and e.counted
    assert cdf.tobytes() == rc.tobytes() and marg.tobytes() == rm.tobytes() and prob.tobytes() == rp.tobytes()
    assert e.total == total
    e.close()


def _dirs(n, seed):
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(n, 3))
    return (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)


def _image_tex(sb, img=None):
    return sb.tex_image(env_scenes.sun_sky(32, 16) if img is None else img, srgb=False)


CHAINS = {   # name -> (builder, expected kind)
    "image": (lambda sb: setattr(sb, "background", sb.tex_background(1.5, _image_tex(sb))), 2),
    "image_root": (lambda sb: setattr(sb, "background", _image_tex(sb)), 2),
    "constant": (lambda sb: setattr(sb, "background", sb.tex_background(1.0, sb.tex_constant((0.2, 0.3, 0.4)))), 1),
    "black_constant": (lambda sb: setattr(sb, "background", sb.tex_background(1.0, sb.tex_constant((0, 0, 0)))), 0),
    "zero_intensity": (lambda sb: setattr(sb, "background", sb.tex_background(0.0, _image_tex(sb))), 0),
    "colorramp": (lambda sb: setattr(sb, "background", sb.tex_background(1.0, sb.tex_colorramp(0.2, 0.8, _image_tex(sb)))), 0),
    "blend": (lambda sb: setattr(sb, "background", sb.tex_background(1.0, sb.tex_blend("mix", -1, _image_tex(sb), sb.tex_constant((1, 1, 1))))), 0),
    "nested_at_limit": (lambda sb: setattr(sb, "background", sb.tex_background(1.0, sb.tex_background(2.0, sb.tex_background(0.5, _image_tex(sb))))), 2),
    "nested_constant": (lambda sb: setattr(sb, "background", sb.tex_background(1.0, sb.tex_background(2.0, sb.tex_background(0.5, sb.tex_constant((1, 2, 3)))))), 1),
    "missing_child_at_limit": (lambda sb: setattr(sb, "background", sb.tex_background(1.0, sb.tex_background(2.0, sb.tex_background(0.5, sb.tex_background(1.0, -1))))), 0),
    "missing_child": (lambda sb: setattr(sb, "background", sb.tex_background(1.0, -1)), 0),
    "none": (lambda sb: None, 0),
}


@pytest.mark.parametrize("name", sorted(CHAINS))
def test_chain_classification_agrees_with_background(env, name):
    build, kind = CHAINS[name]
    e = emu(env, sky_scene(chain=build))
    rgb, _ = e.eval(_dirs(10000, 3))
    assert e.kind == kind
    zero = not rgb.any()
    constant = not zero and (rgb == rgb[0]).all()
    assert zero == (kind == env.ENV_ZERO)
    assert constant == (kind == env.ENV_CONSTANT)
    e.close()


def test_chain_deeper_than_the_limit_is_rejected(env):
    """a chain deeper than kz_tex_eval_tree's stack never reaches the classification: the upload refuses it"""
    sb = sky_scene(chain=lambda sb: setattr(sb, "background", sb.tex_background(1.0, sb.tex_background(1.0, sb.tex_background(1.0, sb.tex_background(1.0, _image_tex(sb)))))))
    with pytest.raises(RuntimeError):
        emu(env, sb)


@pytest.fixture(scope="module")
def sun(env):
    img = env_scenes.sun_sky()
    e = emu(env, sky_scene(img))
    yield e, img
    e.close()


def test_density_positive_where_background_is(sun):
    e, img = sun
    sd = np.array([-0.5, 0.7, -0.45]); sd /= np.linalg.norm(sd)
    near = sd + 0.05 * np.random.default_rng(9).normal(size=(100000, 3))
    d = np.concatenate([_dirs(900000, 4), (near / np.linalg.norm(near, axis=1, keepdims=True)).astype(np.float32)])
    rgb, pdf = e.eval(d)
    lit = (rgb != 0).any(axis=1)
    assert lit.sum() > 990000
    assert (pdf[lit] > 0).all() and np.isfinite(pdf).all()


def test_density_integrates_to_one(sun):
    """midpoint quadrature over the lat-long square, d(omega) = 2 pi^2 cos(elevation) ds dt, 16 x 16 points per table cell"""
    e, _ = sun
    ns, nt = 16 * e.w, 16 * e.h_
    s = (np.arange(ns) + 0.5) / ns
    total = 0.0
    for k in range(0, nt, 256):
        t = (np.arange(k, min(nt, k + 256)) + 0.5) / nt
        tt, ss = np.meshgrid(t, s, indexing="ij")
        _, pdf = e.eval(env_scenes.st_to_dir(ss, tt).reshape(-1, 3).astype(np.float32))
        jac = 2 * np.pi ** 2 * np.cos((0.5 - tt) * np.pi).reshape(-1)
        total += (pdf.astype(np.float64) * jac).sum() / (ns * nt)
    assert abs(total - 1) < 1e-3, total


def _cells(d, w, h):
    s = np.arctan2(-d[:, 0].astype(np.float64), d[:, 2]) / (2 * np.pi) + 0.5
    t = 0.5 - np.arctan2(d[:, 1].astype(np.float64), np.hypot(d[:, 2], d[:, 0])) / np.pi
    return np.clip((t * h).astype(np.int64), 0, h - 1), np.clip((s * w).astype(np.int64), 0, w - 1), s * w, t * h


def test_samples_follow_the_cell_probabilities(sun):
    from scipy import stats
    e, _ = sun
    _, _, prob = e.table()
    n = 10 ** 7
    u = np.random.default_rng(12345).random((n, 2), dtype=np.float32)
    out = e.sample(u)
    r, c, _, _ = _cells(out[:, :3], e.w, e.h_)
    counts = np.bincount(r * e.w + c, minlength=e.w * e.h_).astype(np.float64)
    p = prob.reshape(-1).astype(np.float64); p /= p.sum()
    expct = n * p
    big = expct >= 5
    obs = np.append(counts[big], counts[~big].sum()); exp = np.append(expct[big], expct[~big].sum())
    keep = exp > 0
    chi2 = ((obs[keep] - exp[keep]) ** 2 / exp[keep]).sum()
    pval = stats.chi2.sf(chi2, keep.sum() - 1)
    assert pval > 1e-3, (chi2, keep.sum(), pval)


def test_returned_density_is_the_sampled_cells(sun):
    """the density returned with a sample is kz_env_pdf of its direction; it is the density of the cell the table inversion picked
    except where the direction rounds across a cell boundary"""
    e, _ = sun
    cdf, marg, prob = e.table()
    n = 10 ** 6
    u = np.random.default_rng(77).random((n, 2), dtype=np.float32)
    out = e.sample(u)
    _, pdf = e.eval(out[:, :3])
    assert out[:, 3].tobytes() == pdf.tobytes()
    r = np.clip(np.searchsorted(marg, u[:, 0], "left") - 1, 0, e.h_ - 1)
    c = np.array([min(max(np.searchsorted(cdf[ri], ui, "left") - 1, 0), e.w - 1) for ri, ui in zip(r, u[:, 1])])
    d = out[:, :3].astype(np.float64)
    cl = np.hypot(d[:, 2], d[:, 0]) / np.linalg.norm(d, axis=1)
    want = prob[r, c].astype(np.float64) * e.w * e.h_ / (2 * np.pi ** 2 * cl)
    ok = np.isclose(out[:, 3], want, rtol=1e-4)
    assert ok.mean() >= 0.9999, ok.mean()


def test_host_parses_env_sampling(tmp_path):
    import subprocess
    subprocess.check_call(["make", "-s", "-C", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "nano-kazen_b200", "host")])
    (tmp_path / "q.obj").write_text("v -1 -1 0\nv 1 -1 0\nv 1 1 0\nv -1 1 0\nf 1 2 3 4\n")
    mesh = "<camera type='perspective'/><mesh type='obj'><string name='filename' value='q.obj'/><bsdf type='diffuse'/></mesh></scene>"
    for integ, want in (("<integrator type='path_mis'><boolean name='envSampling' value='true'/></integrator>", 1),
                        ("<integrator type='path_mis'/>", 0), ("<integrator type='ao'/>", 0)):
        (tmp_path / "s.xml").write_text("<scene>" + integ + mesh)
        hs = pk.HostScene(str(tmp_path / "s.xml"))
        assert hs.desc.integrator.env_sampling == want
        assert f"envSampling={want}]" in hs.describe()
        hs.close()


# ------------------------------------------------------------------------------------------------ GPU
def _gpu_count():
    import torch
    return torch.cuda.device_count()


@pytest.mark.gpu
def test_probe_matches_host_emulation(gpu_lib, sun):
    e, img = sun
    G = gpu(sky_scene(img))
    u = np.random.default_rng(31).random((200000, 2), dtype=np.float32)
    g, h = G.env_sample_dump(u), e.sample(u)
    np.testing.assert_allclose(g[:, :3], h[:, :3], rtol=4e-6, atol=2e-7)
    _, _, sw, th = _cells(h[:, :3], e.w, e.h_)
    inside = (np.abs(sw - np.round(sw)) > 1e-3) & (np.abs(th - np.round(th)) > 1e-3)
    assert inside.mean() > 0.99
    np.testing.assert_allclose(g[inside, 3], h[inside, 3], rtol=1e-5)
    np.testing.assert_allclose(g[inside, 4:7], h[inside, 4:7], rtol=1e-3, atol=1e-5)
    if _gpu_count() >= 2:
        G2 = gpu(sky_scene(img), devices=(0, 1))
        assert G2.env_sample_dump(u, 0).tobytes() == G2.env_sample_dump(u, 1).tobytes()
        G2.close()
    G.close()
    G = gpu(sky_scene(img, env_sampling=False))
    with pytest.raises(RuntimeError, match="env_sample_dump failed \\(-4\\)"):
        G.env_sample_dump(u[:4])
    G.close()


VARIANTS = {"plain": dict(), "regularized": dict(regularization=True), "no_emitters": dict(emitters=False)}
SHARDS = 16


def _shards(G, per, b):
    out = []
    for k in range(SHARDS):
        out.append(env_scenes.resolve(G.render(k * per, (k + 1) * per), b))
    return np.stack(out)


def _blocks(img):
    h, w = img.shape[:2]
    return img[:h - h % 8, :w - w % 8].reshape(h // 8, 8, w // 8, 8, 3).mean(axis=(1, 3, 4))


@pytest.fixture(scope="module")
def studio_runs(gpu_lib):
    res = {}
    for name, kw in VARIANTS.items():
        runs = {}
        for on, per in ((False, 4096), (True, 256)):
            G = gpu(env_scenes.sun_studio(env_sampling=on, **kw))
            _, _, b = G.frame_shape()
            runs[on] = _shards(G, per, b)
            runs[(on, 64)] = env_scenes.resolve(G.render(1 << 17, (1 << 17) + 64), b)       # sample indices no shard used
            G.close()
        res[name] = runs
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_env_sampling_is_unbiased(studio_runs, variant):
    """|mean_on - mean_off| <= 5 sigma for the frame mean and every 8x8 block.  With regularisation only the frame mean: the reference's
    regularised kiss sampler draws from the unregularised lobe but reports the regularised density (bsdf.cpp:1323), so its BSDF-sampled
    estimate is not an estimate of the regularised BSDF's integral and the sum depends on the strategy it is combined with; where the sun
    reflects in a regularised lobe a block differs by more than the shards' spread, and that is regularisation's bias, not this estimator's"""
    runs = studio_runs[variant]
    stats = [lambda im: np.array([im.mean()])] + ([] if variant == "regularized" else [lambda im: _blocks(im).reshape(-1)])
    for stat in stats:
        off = np.stack([stat(x) for x in runs[False]]); on = np.stack([stat(x) for x in runs[True]])
        se = np.sqrt(off.var(axis=0, ddof=1) / SHARDS + on.var(axis=0, ddof=1) / SHARDS)
        diff = np.abs(on.mean(axis=0) - off.mean(axis=0))
        assert (diff <= 5 * se).all(), (variant, diff.max(), (diff / np.maximum(se, 1e-30)).max())


@pytest.mark.gpu
@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_env_sampling_reduces_noise(studio_runs, variant):
    runs = studio_runs[variant]
    ref = 0.5 * (runs[False].mean(axis=0) + runs[True].mean(axis=0))
    rel = lambda a: float((((a - ref) ** 2) / (ref ** 2 + 1e-2)).mean())
    assert rel(runs[(True, 64)]) <= 0.5 * rel(runs[(False, 64)]), (rel(runs[(True, 64)]), rel(runs[(False, 64)]))


def _no_env_cases():
    black = np.zeros((16, 32, 3), np.float32)
    yield "no_background", lambda on: sky_scene(None, env_sampling=on)
    yield "zero_intensity", lambda on: sky_scene(chain=lambda sb: env_scenes.sky_background(sb, env_scenes.sun_sky(64, 32), intensity=0.0), env_sampling=on)
    yield "black_image", lambda on: sky_scene(black, env_sampling=on)
    for kind in ("normals", "ao", "whitted", "path_mats"):
        yield kind, (lambda k: lambda on: sky_scene(env_scenes.sun_sky(64, 32), env_sampling=on, kind=k))(kind)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c, _ in _no_env_cases()])
def test_no_counted_environment_changes_nothing(gpu_lib, case):
    make = dict(_no_env_cases())[case]
    frames, counters = [], []
    for on in (False, True):
        sb = make(on)
        sb.set_sampler("independent", 64)
        G = gpu(sb)
        frames.append(G.render())
        s = G.stats()
        counters.append((s["paths"], s["rays_extension"], s["rays_shadow"], s["vertices"]))
        G.close()
    np.testing.assert_allclose(frames[1], frames[0], rtol=1e-4, atol=1e-5)
    assert counters[0] == counters[1]


@pytest.mark.gpu
def test_two_devices_render_like_one(gpu_lib):
    if _gpu_count() < 2:
        pytest.skip("needs two GPUs")
    sb = env_scenes.sun_studio(env_sampling=True, spp=64)
    a = gpu(sb).render(); b = gpu(sb, devices=(0, 1)).render()
    np.testing.assert_allclose(b, a, rtol=1e-4, atol=1e-5)
