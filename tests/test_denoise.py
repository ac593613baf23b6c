"""First-hit AOVs (mox_set_aovs, mox_read_aovs) and the a-trous denoiser (mox_denoise).

The filter is restated here in numpy float32, operation by operation in the order include/mox.h writes it, and fed
with what the ABI returns: read_accum / read_sample_counts / read_aovs.  The only freedom the implementations have is
the library's exp: each weight may differ by a few ulps, so outputs are compared within EXP_RTOL (relative, with a
floor for values near 0)."""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from minimaloptix_b200 import MoxError, structs as S
import adaptive_model as M
import refcases as R

ERR_INVALID, ERR_STATE = -1, -4
# A few ulps of expf per weight, carried through up to 10 iterations of normalised sums.
EXP_RTOL, EXP_ATOL = 2e-4, 1e-6
COUNTS = ("rays_primary", "rays_bounce", "rays_shadow", "rays_shadow_traced", "nonfinite_samples", "rays_depth",
          "shadow_traced_depth", "launches")
# Cornell, 64 x 64, 16 spp, default parameters: the RMSE against 1024 spp must fall by more than this factor.
QUALITY_RATIO = 1.75
H_TAPS = np.array([1 / 16, 1 / 4, 3 / 8, 1 / 4, 1 / 16], np.float32)


def atrous(color, albedo, normal, depth, iterations, sigma_color, sigma_normal, sigma_depth):
    """mox_denoise in numpy float32: every product, sum and division rounded on its own, in the header's order."""
    f = np.float32
    H, W, _ = color.shape
    m = albedo + f(0.001)
    e = color / m
    sn, sd = f(sigma_normal), f(sigma_depth)
    for i in range(iterations):
        s = 1 << i
        sigma = f(sigma_color) * f(2.0 ** -i)
        sig2 = sigma * sigma
        sx = np.zeros((H, W), np.float32)
        sy, sz, sw = sx.copy(), sx.copy(), sx.copy()
        for dy in range(-2, 3):
            for dx in range(-2, 3):
                # q = p + s (dx, dy); taps outside the image are skipped
                ys, xs = np.arange(H) + s * dy, np.arange(W) + s * dx
                vy, vx = (ys >= 0) & (ys < H), (xs >= 0) & (xs < W)
                if not vy.any() or not vx.any():
                    continue
                py, px = np.nonzero(vy)[0], np.nonzero(vx)[0]
                P = np.ix_(py, px)
                Q = np.ix_(ys[py], xs[px])
                eq = e[Q]
                if dx == 0 and dy == 0:
                    w = np.ones(eq.shape[:2], np.float32)
                else:
                    ep, npp, nq, zp, zq = e[P], normal[P], normal[Q], depth[P], depth[Q]
                    d = ep - eq
                    tc = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1] + d[..., 2] * d[..., 2]) / sig2
                    dot = npp[..., 0] * nq[..., 0] + npp[..., 1] * nq[..., 1] + npp[..., 2] * nq[..., 2]
                    tn = np.maximum(f(0), f(1) - dot) / sn
                    tz = np.abs(zp - zq) / (sd * np.maximum(zp, zq) + f(1e-30))
                    w = np.exp(-(tc + tn + tz)).astype(np.float32)
                k = H_TAPS[dx + 2] * H_TAPS[dy + 2] * w
                sx[P] += k * eq[..., 0]
                sy[P] += k * eq[..., 1]
                sz[P] += k * eq[..., 2]
                sw[P] += k
        e = np.stack([sx / sw, sy / sw, sz / sw], axis=-1)
    return e * m


def restated(ctx, iterations, sc, sn, sd):
    """atrous() fed with the context's own read-backs."""
    n = ctx.read_sample_counts().astype(np.float32)
    acc = ctx.read_accum()
    with np.errstate(invalid="ignore", divide="ignore"):
        color = np.where(n[..., None] > 0, acc / n[..., None], np.float32(0)).astype(np.float32)
    a, nr, z = ctx.read_aovs()
    return atrous(color, a, nr, z, iterations, sc, sn, sd)


def assert_close(got, want):
    err = np.abs(got - want)
    bad = err > EXP_ATOL + EXP_RTOL * np.abs(want)
    assert not bad.any(), (int(bad.sum()), float((err / (np.abs(want) + EXP_ATOL)).max()))


def rmse(a, b):
    return float(np.sqrt(np.mean((np.clip(a, 0, 1) - np.clip(b, 0, 1)) ** 2)))


# ---- scenes

def two_planes(ctx, host, w, h, depth=5):
    """A floor and a wall behind it: a hard normal edge where they meet, and a depth step at the wall's top edge
    against a far backdrop."""
    ctx.set_globals(w, h, depth, bg=(0.6, 0.7, 0.9))
    ctx.set_camera(host.set_cam_params((0.0, 1.5, 5.0), (0, 0.8, 0), (0, 1, 0), 45, w / h, 0.0, 5.0))
    lam = S.LambertianParams(S.float3(0.7, 0.6, 0.5))
    ctx.add_quad(host.set_quad_params((-4, 0, 4), (8, 0, 0), (0, 0, -8)), S.MAT_LAMBERTIAN, lam)      # floor
    ctx.add_quad(host.set_quad_params((-4, 0, -2), (8, 0, 0), (0, 1.6, 0)), S.MAT_LAMBERTIAN,
                 S.LambertianParams(S.float3(0.3, 0.5, 0.8)))                                      # wall
    ctx.add_quad(host.set_quad_params((-9, -1, -9), (18, 0, 0), (0, 9, 0)), S.MAT_LAMBERTIAN,
                 S.LambertianParams(S.float3(0.9, 0.9, 0.9)))                                      # far backdrop
    ctx.add_sphere(S.SphereParams(1.0, S.float3(0, 5, 2)), S.MAT_LIGHT, S.LightParams(emission=S.float3(6, 6, 6)))


def quads(ctx, host, w, h):
    """Axis-aligned quads facing the camera, which looks along -z: per material an exact albedo, normals of exactly
    +z / +y, and a miss where a clamped background shows."""
    ctx.set_globals(w, h, 3, bg=(2.0, 0.5, -1.0))
    ctx.set_camera(host.set_cam_params((0.0, 0.0, 0.0), (0, 0, -1), (0, 1, 0), 60, w / h, 0.0, 1.0))
    lam = S.LambertianParams(S.float3(0.25, 0.5, 0.75))
    dis = R._disney(color=(0.5, 0.125, 1.0))
    # edge vectors of power-of-two length: the normalised cross products are exact
    ctx.add_quad(host.set_quad_params((-3, -1, -4), (4, 0, 0), (0, 4, 0)), S.MAT_LAMBERTIAN, lam)      # left, z = -4
    ctx.add_quad(host.set_quad_params((0, 3, -6), (4, 0, 0), (0, -4, 0)), S.MAT_DISNEY, dis)           # right, z = -6, facing -z
    ctx.add_quad(host.set_quad_params((-4, -1.5, 0), (8, 0, 0), (0, 0, -8)), S.MAT_METAL,
                 S.MetalParams(S.float3(0.125, 0.25, 0.5), 0.0))                                       # floor, y = -1.5
    ctx.add_quad(host.set_quad_params((-0.5, 1.5, -3), (0.5, 0, 0), (0, 0.5, 0)), S.MAT_LIGHT,
                 S.LightParams(emission=S.float3(4.0, 0.25, 0.0)))                                  # small light, z = -3


# The oracle keys its AOV state by context address (oracle/denoise.cpp): the contexts of this file stay alive, so no
# later context inherits one's switch.
_ORACLE_CONTEXTS = []


def new_oracle(orc):
    _ORACLE_CONTEXTS.append(orc.context())
    return _ORACLE_CONTEXTS[-1]


def oracle_ctx(orc, api_tables, host, build, *args):
    o = new_oracle(orc)
    if build is None:
        M.load_cornell(host).upload(api_tables.oracle, o, *args)
    else:
        build(o, host, *args)
    o.build_accel()
    return o


# ---- CPU: the oracle

def test_oracle_aovs_of_axis_aligned_quads(orc, host):
    w, h = 64, 48
    o = new_oracle(orc)
    quads(o, host, w, h)
    o.build_accel()
    o.set_aovs(True)
    o.render(1, 0xA0F)
    a, n, z = o.read_aovs()
    mats = {(0.25, 0.5, 0.75): ((0, 0, 1), -4.0), (0.5, 0.125, 1.0): ((0, 0, 1), -6.0), (0.125, 0.25, 0.5): ((0, 1, 0), None),
            (1.0, 0.25, 0.0): ((0, 0, 1), -3.0), (1.0, 0.5, 0.0): ((0, 0, 0), None)}
    seen = set()
    for y in range(h):
        for x in range(w):
            key = tuple(float(v) for v in a[y, x])
            assert key in mats, (x, y, key)
            seen.add(key)
            N, plane = mats[key]
            assert tuple(n[y, x]) == N, (x, y, n[y, x])
            if key == (1.0, 0.5, 0.0):
                assert z[y, x] == 0
                continue
            # depth: the pixel's camera ray (inside its footprint, pinhole at the origin) meets the plane
            corners = []
            for cx in (x - 0.5, x + 1.5):
                for cy in (y - 0.5, y + 1.5):
                    t = np.tan(np.radians(30))
                    d = np.array([(2 * cx / w - 1) * t * w / h, (2 * cy / h - 1) * t, -1.0])
                    d /= np.linalg.norm(d)
                    corners.append(plane / d[2] if plane is not None else -1.5 / d[1])
            corners = [c for c in corners if c > 0] or [np.inf]
            assert min(corners) * 0.999 <= z[y, x] <= max(corners) * 1.001, (x, y, z[y, x], corners)
    assert len(seen) == 5


@pytest.mark.parametrize("scene,size,iterations", [("two_planes", (37, 23), 10), ("two_planes", (64, 40), 3),
                                                   ("random_spheres", (45, 31), 5), ("random_spheres", (37, 23), 1)])
def test_oracle_denoise_matches_numpy(orc, host, api_tables, scene, size, iterations):
    w, h = size
    o = new_oracle(orc)
    if scene == "two_planes":
        two_planes(o, host, w, h)
    else:
        host.Scene.builtin("random_spheres").upload(api_tables.oracle, o, w, h, 5)
    o.build_accel()
    o.set_aovs(True)
    o.render(4, 0xD0)
    for sc, sn, sd in ((4.0, 0.1, 0.1), (0.5, 0.02, 0.05)):
        got, _ = o.denoise(iterations, sc, sn, sd)
        assert_close(got, restated(o, iterations, sc, sn, sd))


def test_oracle_aovs_reset_and_partial(orc, host):
    o = new_oracle(orc)
    two_planes(o, host, 32, 24)
    o.build_accel()
    o.render(2, 1)
    o.set_aovs(True)           # on after two samples: the AOVs count only their own
    o.render(2, 1)
    a2, n2, z2 = o.read_aovs()
    o.clear_accum()
    assert not any(v.any() for v in o.read_aovs())
    o.set_accum(np.zeros((24, 32, 3), np.float32), 2)
    with pytest.raises(MoxError, match="rendered"):
        o.denoise()            # a loaded buffer alone has no guides
    o.render(2, 1)             # the same two launches as above
    for u, v in zip(o.read_aovs(), (a2, n2, z2)):
        assert np.array_equal(u, v)


def test_oracle_quality_cornell(orc, host, api_tables):
    """Denoised 16 spp against 1024 spp with the default parameters.  Measured on the oracle: RMSE ratio noisy / denoised
    2.2."""
    w = h = 64
    ref = oracle_ctx(orc, api_tables, host, None, w, h, 5)
    ref.render(1024, 77)
    truth = ref.read_accum() / 1024
    o = oracle_ctx(orc, api_tables, host, None, w, h, 5)
    o.set_aovs(True)
    o.render(16, 5)
    noisy = o.read_accum() / 16
    den, _ = o.denoise()
    ratio = rmse(noisy, truth) / rmse(den, truth)
    print("oracle cornell 16 spp: noisy", rmse(noisy, truth), "denoised", rmse(den, truth), "ratio", ratio)
    assert ratio > QUALITY_RATIO, ratio


# ---- GPU

def gpu_ctx(gpu_backend, api_tables, host, scene, w, h, depth=5, device=0, aovs=False):
    g = gpu_backend.context(device)
    if scene == "cornell":
        M.load_cornell(host).upload(api_tables.gpu, g, w, h, depth)
    elif scene == "zoo":
        R.build_zoo(g, host, w, h, depth, textured=True)
    elif scene == "zoo_flat":
        R.build_zoo(g, host, w, h, depth, textured=False)
    elif scene == "interior":
        host.Scene.builtin("interior", 30000).upload(api_tables.gpu, g, w, h, depth)
    elif scene == "two_planes":
        two_planes(g, host, w, h, depth)
    g.build_accel()
    if aovs:
        g.set_aovs(True)
    return g


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["cornell", "zoo", "interior"])
@pytest.mark.parametrize("mode", ["render", "adaptive", "depth0"])
def test_aovs_leave_the_image_unchanged(host, api_tables, gpu_backend, scene, mode):
    w, h = 96, 64
    out = []
    for aovs in (False, True):
        g = gpu_ctx(gpu_backend, api_tables, host, scene, w, h, 0 if mode == "depth0" else 5, aovs=aovs)
        if mode == "adaptive":
            g.render_adaptive(16, 9, 0.05, 1e-3, min_spp=4, round_spp=4)
        else:
            g.render(6, 9)
            g.launch(1234)
        st = g.stats()
        out.append((bits(g.read_accum()), g.read_sample_counts(), {k: st[k] for k in COUNTS}, st["kernel_launches"]))
    (a0, n0, s0, k0), (a1, n1, s1, k1) = out
    assert np.array_equal(a0, a1) and np.array_equal(n0, n1) and s0 == s1
    assert k1 > k0


@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["cornell", "zoo", "zoo_flat"])
def test_gpu_aovs_match_the_oracle(host, api_tables, orc, gpu_backend, scene):
    w, h = 80, 60
    g = gpu_ctx(gpu_backend, api_tables, host, scene, w, h, aovs=True)
    o = new_oracle(orc)
    if scene == "cornell":
        M.load_cornell(host).upload(api_tables.oracle, o, w, h, 5)
    else:
        R.build_zoo(o, host, w, h, 5, textured=scene == "zoo")
    o.build_accel()
    o.set_aovs(True)
    for c in (g, o):
        c.render(1, 0x5EED)   # one sample per pixel: a pixel's record is one hit, or one miss
    (ag, ng, zg), (ao, no, zo) = g.read_aovs(), o.read_aovs()
    hit_g, hit_o = zg > 0, zo > 0
    assert hit_g.mean() == hit_o.mean()
    same = hit_g == hit_o
    assert same.mean() >= 0.999, same.mean()
    hit = hit_g & same
    # the same primitive where the albedos agree; elsewhere the two picked different primitives at a tie
    agree = np.all(ag == ao, axis=2)
    if scene != "zoo":
        assert agree.mean() >= 0.999, agree.mean()
    else:   # the texture filter's 8-bit weights (test_shading_math.py)
        assert np.abs(ag - ao).max() <= 1 / 256 + 1e-6
    sel = hit & np.all(np.abs(ag - ao) <= 1 / 256 + 1e-6, axis=2)
    assert np.abs(zg - zo)[sel].max() <= 1e-5 * zo[sel].max()
    assert np.abs(ng - no)[sel].max() <= 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("scene,size,iterations", [("two_planes", (37, 23), 10), ("cornell", (61, 45), 1),
                                                   ("cornell", (61, 45), 10), ("zoo", (75, 49), 5)])
def test_gpu_denoise_matches_numpy(host, api_tables, gpu_backend, scene, size, iterations):
    g = gpu_ctx(gpu_backend, api_tables, host, scene, *size, aovs=True)
    g.render(8, 3)
    for sc, sn, sd in ((1.0, 0.5, 0.05), (4.0, 0.1, 0.1)):
        got, ms = g.denoise(iterations, sc, sn, sd)
        assert ms > 0
        assert_close(got, restated(g, iterations, sc, sn, sd))
        again, _ = g.denoise(iterations, sc, sn, sd)
        assert np.array_equal(bits(got), bits(again))


@pytest.mark.gpu
def test_gpu_denoise_tall_image(host, api_tables, gpu_backend):
    """Taller than 65535 blocks of 16 rows: each iteration takes two launches, and the filter crosses their seam."""
    w, h = 2, 65535 * 16 + 301
    g = gpu_ctx(gpu_backend, api_tables, host, "two_planes", w, h, aovs=True)
    g.render(1, 8)
    got, _ = g.denoise(3)
    d = S.DENOISE_DEFAULTS
    assert_close(got, restated(g, 3, d["sigma_color"], d["sigma_normal"], d["sigma_depth"]))


@pytest.mark.gpu
def test_gpu_denoise_adaptive(host, api_tables, gpu_backend):
    g = gpu_ctx(gpu_backend, api_tables, host, "cornell", 64, 48, aovs=True)
    g.render_adaptive(32, 4, 0.05, 1e-3, min_spp=4, round_spp=4)
    n = g.read_sample_counts()
    assert (n < 32).any() and (n == 32).any()
    got, _ = g.denoise()
    d = S.DENOISE_DEFAULTS
    assert_close(got, restated(g, d["iterations"], d["sigma_color"], d["sigma_normal"], d["sigma_depth"]))


@pytest.mark.gpu
def test_gpu_errors_and_resets(host, api_tables, gpu_backend):
    w, h = 40, 30
    g = gpu_ctx(gpu_backend, api_tables, host, "cornell", w, h)
    out = np.empty((h, w, 3), np.float32)

    def rc(p=None, ctx=g):
        return ctx.b.denoise(ctx.h, None if p is None else C.byref(p), out.ctypes.data_as(C.c_void_p), None)
    assert rc() == ERR_STATE                                        # AOVs off
    assert g.b.read_aovs(g.h, None, None, None) == ERR_STATE
    g.set_aovs(True)
    assert rc() == ERR_STATE                                        # nothing rendered
    g.render(2, 1)
    assert rc() == 0
    for p in (S.DenoiseParams(0, 1, 1, 1), S.DenoiseParams(11, 1, 1, 1), S.DenoiseParams(5, 0, 1, 1),
              S.DenoiseParams(5, 1, -1, 1), S.DenoiseParams(5, 1, 1, float("nan")), S.DenoiseParams(5, float("inf"), 1, 1)):
        assert rc(p) == ERR_INVALID
    assert rc(S.DenoiseParams(10, 1, 1, 1)) == 0
    part = gpu_ctx(gpu_backend, api_tables, host, "cornell", w, h, aovs=True)
    part.set_partition(0, 2, 16)
    part.render(2, 1)
    assert rc(ctx=part) == ERR_STATE                                # needs the whole frame
    # the resets: clear, set_accum, a size change
    a2 = g.read_aovs()
    assert a2[2].any()
    g.clear_accum()
    assert not any(v.any() for v in g.read_aovs())
    g.set_accum(np.zeros((h, w, 3), np.float32), 0)
    g.render(2, 1)
    assert all(np.array_equal(bits(u), bits(v)) for u, v in zip(g.read_aovs(), a2))
    g.set_accum(np.zeros((h, w, 3), np.float32), 7)
    assert not any(v.any() for v in g.read_aovs())
    assert rc() == ERR_STATE                                        # a loaded buffer alone has no guides
    g.render(1, 1)
    assert rc() == 0
    g.set_globals(w // 2, h // 2, 5)
    assert [v.shape[:2] for v in g.read_aovs()] == [(h // 2, w // 2)] * 3 and not any(v.any() for v in g.read_aovs())
    g.set_aovs(False)
    assert g.b.read_aovs(g.h, None, None, None) == ERR_STATE


@pytest.mark.gpu
def test_multi_handle_denoise_equals_one_device(host, api_tables, gpu_backend):
    import torch
    n = min(torch.cuda.device_count(), 4)
    one = gpu_ctx(gpu_backend, api_tables, host, "cornell", 96, 80, aovs=True)
    one.render(8, 2)
    want, _ = one.denoise(5)
    aovs = one.read_aovs()
    for devices in ([0], list(range(n))) if n >= 2 else ([0],):
        m = gpu_ctx(gpu_backend, api_tables, host, "cornell", 96, 80, device=devices, aovs=True)
        m.render(8, 2)
        got, _ = m.denoise(5)
        assert np.array_equal(bits(got), bits(want)), devices
        assert all(np.array_equal(bits(u), bits(v)) for u, v in zip(m.read_aovs(), aovs))
    if n < 2:
        pytest.skip("one device: the one-device handle was checked, the split over several was not")


@pytest.mark.gpu
def test_cli_denoise(tmp_path):
    from PIL import Image
    cli = os.path.join(ROOT, "minimaloptix_b200", "mox_cli")
    out = str(tmp_path / "cb")
    base = [cli, "--scene", "cornell", "--scene-dir", os.path.join(ROOT, "scenes"), "--width", "64", "--height", "48",
            "--max-depth", "5", "--spp", "8", "--out", out]
    for extra in (["--denoise"], ["--denoise", "3", "--adaptive", "0.05"]):
        r = subprocess.run(base + extra, capture_output=True, text=True, timeout=120)
        assert r.returncode == 0, r.stderr
        stats = json.loads(r.stdout.strip().splitlines()[-1])
        assert stats["ms_denoise"] > 0 and stats["denoise_iterations"] == (5 if len(extra) == 1 else 3)
        for suffix in ("_denoised", "_albedo", "_normal"):
            img = np.asarray(Image.open(out + suffix + ".png"))
            assert img.shape == (48, 64, 3) and img.std() > 3
    r = subprocess.run(base, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "ms_denoise" not in r.stdout


@pytest.mark.gpu
def test_gpu_quality_cornell(host, api_tables, gpu_backend):
    """The CPU quality check on the GPU: Cornell, 64 x 64, 16 spp, default parameters, against 1024 spp."""
    ref = gpu_ctx(gpu_backend, api_tables, host, "cornell", 64, 64)
    ref.render(1024, 77)
    truth = ref.read_accum() / 1024
    g = gpu_ctx(gpu_backend, api_tables, host, "cornell", 64, 64, aovs=True)
    g.render(16, 5)
    den, _ = g.denoise()
    ratio = rmse(g.read_accum() / 16, truth) / rmse(den, truth)
    print("gpu cornell 16 spp ratio", ratio)
    assert ratio > QUALITY_RATIO, ratio
