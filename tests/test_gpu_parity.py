"""GPU parity tests: the CUDA path (through the C ABI of libmox.so) against the CPU oracle on
the same seeded inputs.  Run on a B200: python -m pytest tests -m gpu."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import ROOT, random_rays
from minimaloptix_b200 import structs as S

pytestmark = pytest.mark.gpu


def both(host, api_tables, orc, gpu_backend, scene, w, h, depth, brute=False, flags=0):
    o = orc.context(brute_force=brute)
    g = gpu_backend.context(0)
    scene.upload(api_tables.oracle, o, w, h, depth)
    scene.upload(api_tables.gpu, g, w, h, depth)
    o.build_accel()
    g.build_accel(flags)
    return o, g


def check_ids(o, g, rays, name):
    """Primitive ids must be bit-exact except epsilon ties (SURVEY.md §8d tolerances):
    runner-up within |dt| <= 1e-5 t, an edge graze min(b, g, 1-b-g) < 1e-5, or t within 1e-5 t of tmin."""
    to, io, bo, go = o.trace_closest(rays)
    tg, ig, bg, gg = g.trace_closest(rays)
    same = io == ig
    # where ids agree every reported number is bit-identical
    assert np.array_equal(to[same].view(np.uint32), tg[same].view(np.uint32)), name
    hitmask = same & (io >= 0)
    assert np.array_equal(bo[hitmask].view(np.uint32), bg[hitmask].view(np.uint32)), name
    assert np.array_equal(go[hitmask].view(np.uint32), gg[hitmask].view(np.uint32)), name
    bad = np.nonzero(~same)[0]
    for k in bad:
        t1, t2 = float(to[k]), float(tg[k])
        tie_t = abs(t1 - t2) <= 1e-5 * max(abs(t1), abs(t2))
        graze = False
        for (b_, g_, i_) in ((bo[k], go[k], io[k]), (bg[k], gg[k], ig[k])):
            if i_ >= 0 and min(b_, g_, 1 - b_ - g_) < 1e-5:
                graze = True
        near_tmin = min(t1, t2) <= rays[k, 3] * (1 + 1e-5)
        assert tie_t or graze or near_tmin, (name, k, io[k], ig[k], t1, t2)
    return len(bad), int((io >= 0).sum())


def _sort_keys(rng, n, kind):
    if kind == "morton":   # 30-bit Morton-like keys with heavy duplication in the low bits
        return (rng.integers(0, 1 << 30, size=n, dtype=np.uint32) & np.uint32(0x3FFF00FF)).astype(np.uint32)
    if kind == "full32":   # every digit of every pass, 0 and 0xFFFFFFFF included
        keys = rng.integers(0, 1 << 32, size=n, dtype=np.uint64).astype(np.uint32)
        keys[rng.integers(0, n, size=min(n, 8))] = 0xFFFFFFFF
        keys[rng.integers(0, n, size=min(n, 8))] = 0
        return keys
    if kind == "invalid":  # Morton codes with k_morton's key of an invalid primitive mixed in
        keys = rng.integers(0, 1 << 30, size=n, dtype=np.uint32)
        keys[rng.random(n) < 0.2] = 0x40000000
        return keys
    if kind == "equal":
        return np.full(n, 0x2AAAAAAA, np.uint32)
    if kind == "descending":
        return (np.uint32(0xFFFFFFFF) - np.arange(n, dtype=np.uint32) * np.uint32(977)).astype(np.uint32)
    raise ValueError(kind)


# n at the edges of the 4096-key sort tile (256 threads x 16 keys)
@pytest.mark.parametrize("n, kind", [pytest.param(n, "morton", id=str(n)) for n in [1, 31, 4096, 4097, 100000, (1 << 20) + 17]]
                         + [pytest.param(n, k, id=f"{k}-{n}") for k, n in [("full32", 4095), ("full32", 8193), ("full32", (1 << 20) + 17),
                                                                          ("invalid", 4096), ("invalid", 100000), ("equal", 1), ("equal", 8192),
                                                                          ("equal", 12289), ("descending", 4097), ("descending", 65536),
                                                                          ("morton", 4095), ("morton", 8191), ("morton", 8192)]])
def test_radix_sort_matches_stable_sort(gpu_backend, n, kind):
    g = gpu_backend.context(0)
    rng = np.random.default_rng(n)
    keys = _sort_keys(rng, n, kind)
    vals = np.arange(n, dtype=np.uint32)
    k, v = g.debug_radix_sort(keys, vals)
    order = np.argsort(keys, kind="stable")
    assert np.array_equal(k, keys[order])
    assert np.array_equal(v, vals[order])  # stability: equal keys keep input order


def test_closest_hit_spheres_and_quads(host, api_tables, orc, gpu_backend):
    sc = host.Scene.builtin("random_spheres")
    o, g = both(host, api_tables, orc, gpu_backend, sc, 64, 64, 5, brute=True)
    rays = random_rays(200000, [-30, -1, -30], [30, 20, 30], 1)
    nbad, nhit = check_ids(o, g, rays, "random_spheres")
    assert nhit > 50000
    assert nbad == 0


def test_closest_hit_cornell(host, api_tables, orc, gpu_backend):
    sc = host.Scene.load(os.path.join(ROOT, "scenes", "cornell"), "cornell")
    o, g = both(host, api_tables, orc, gpu_backend, sc, 64, 64, 5, brute=True)
    rays = random_rays(300000, [0.1, 0.1, 0.1], [5.4, 5.3, 5.4], 2)
    nbad, nhit = check_ids(o, g, rays, "cornell")
    assert nhit > 0.8 * len(rays)  # origins inside the box; the open front lets some rays out
    assert nbad <= 3


def test_closest_hit_cornell_open_front(host, api_tables, orc, gpu_backend):
    sc = host.Scene.load(os.path.join(ROOT, "scenes", "cornell"), "cornell")
    o, g = both(host, api_tables, orc, gpu_backend, sc, 64, 64, 5, brute=True)
    rays = random_rays(100000, [-2, -2, -8], [8, 8, 0], 3)
    nbad, nhit = check_ids(o, g, rays, "cornell-outside")
    assert 0 < nhit < len(rays)
    assert nbad <= 3


@pytest.mark.parametrize("flags", [S.ACCEL_DEFAULT, S.ACCEL_BINARY, S.ACCEL_LBVH], ids=["wide", "binary-ploc", "binary-lbvh"])
def test_closest_hit_interior_mesh(host, api_tables, orc, gpu_backend, flags):
    sc = host.Scene.builtin("interior", 60000)
    info = sc.info()
    assert 40000 < info.n_triangles < 90000
    o, g = both(host, api_tables, orc, gpu_backend, sc, 64, 64, 5, flags=flags)  # oracle BVH for speed
    rays = random_rays(400000, [0.05, 0.05, 0.05], [9.95, 3.95, 7.95], 4)
    nbad, nhit = check_ids(o, g, rays, "interior")
    assert nhit == len(rays)
    assert nbad <= 8
    # and against brute force on a subset (the id ground truth)
    ob = orc.context(brute_force=True)
    sc.upload(api_tables.oracle, ob, 64, 64, 5)
    ob.build_accel()
    nbad, _ = check_ids(ob, g, rays[:20000], "interior-brute")
    assert nbad <= 2


@pytest.mark.parametrize("flags", [S.ACCEL_DEFAULT, S.ACCEL_BINARY, S.ACCEL_LBVH], ids=["wide", "binary-ploc", "binary-lbvh"])
def test_closest_hit_soup(host, api_tables, orc, gpu_backend, flags):
    sc = host.Scene.builtin("soup", 200000, 7)
    o, g = both(host, api_tables, orc, gpu_backend, sc, 64, 64, 5, flags=flags)
    rays = random_rays(300000, [0, 0, 0], [1, 1, 1], 5)
    nbad, nhit = check_ids(o, g, rays, "soup")
    assert nhit > 150000
    assert nbad <= 6


def test_full_size_soup_two_builders_agree(host, api_tables, gpu_backend):
    """BASELINE config 5 at full size (10 M triangles, 2^22 incoherent rays): the oracle cannot
    finish this in seconds, so the check is a size-independent property — two different
    hierarchies (the compressed 8-wide BVH collapsed from PLOC, and the binary Karras radix tree)
    over the same primitives must report the same closest hit, bit for bit, for every ray; and re-tracing is idempotent."""
    import torch
    sc = host.Scene.builtin("soup", 10_000_000)
    a, b = gpu_backend.context(0), gpu_backend.context(0)
    sc.upload(api_tables.gpu, a, 64, 64, 5)
    sc.upload(api_tables.gpu, b, 64, 64, 5)
    ms_a = a.build_accel(S.ACCEL_DEFAULT)
    ms_b = b.build_accel(S.ACCEL_LBVH)
    assert a.stats()["n_triangles"] == 10_000_000
    n = 1 << 22
    gen = torch.Generator(device="cuda").manual_seed(12345)
    r = torch.empty((n, 8), device="cuda")
    r[:, 0:3] = torch.rand((n, 3), generator=gen, device="cuda")
    d = torch.randn((n, 3), generator=gen, device="cuda")
    r[:, 4:7] = d / d.norm(dim=1, keepdim=True)
    r[:, 3], r[:, 7] = 1e-3, 1e27
    ha, hb, ha2 = (torch.empty((n, 4), device="cuda") for _ in range(3))
    torch.cuda.synchronize()
    a.trace_closest_device(r.data_ptr(), n, ha.data_ptr())
    b.trace_closest_device(r.data_ptr(), n, hb.data_ptr())
    a.trace_closest_device(r.data_ptr(), n, ha2.data_ptr())
    ia, ib = ha.view(torch.int32), hb.view(torch.int32)
    diff = int((ia != ib).any(dim=1).sum())
    print("10M soup: build ms ploc", ms_a, "lbvh", ms_b, "rays differing", diff, "hit fraction", float((ia[:, 1] >= 0).float().mean()))
    assert torch.equal(ia, ha2.view(torch.int32))
    assert diff <= 4  # only exact-tie / slab-graze cases may differ between hierarchies
    assert float((ia[:, 1] >= 0).float().mean()) > 0.8


def test_full_size_interior_wide_equals_binary_and_split(host, api_tables, gpu_backend):
    """BASELINE config 4 at full size (≈1 M triangles, 3840x2160, depth 5): size-independent properties instead
    of the oracle — (1) the 8-wide BVH and the binary BVH give the same image and the same ray counts; (2) the
    frame rendered as two interleaved tile partitions (what two GPUs do) is the 1-partition frame bit for bit
    where each partition owns the pixel, and zero elsewhere."""
    sc = host.Scene.builtin("interior", 1_000_000)
    W, H = 3840, 2160
    ref = None
    for flags in (S.ACCEL_DEFAULT, S.ACCEL_BINARY):
        g = gpu_backend.context(0)
        sc.upload(api_tables.gpu, g, W, H, 5)
        g.build_accel(flags)
        g.render(1, 77)
        st = g.stats()
        img = g.read_accum()
        assert st["n_triangles"] > 950_000 and st["nonfinite_samples"] == 0
        if ref is None:
            ref = (img, st["rays_bounce"], st["rays_shadow"])
            assert st["rays_primary"] == W * H and st["rays_bounce"] > W * H
        else:
            # A closest hit may differ between two hierarchies only on exact ties / slab grazes (the 10 M soup test
            # bounds that at one ray per million); such a path then continues differently, so allow a few pixels
            # per million to differ and the ray counts to move by the same fraction.  GLASS attenuation is a
            # product in traversal order: last-bit differences only there.
            differing = int((np.abs(img - ref[0]).max(axis=-1) > 1e-5).sum())
            drift = abs(st["rays_bounce"] - ref[1]) / ref[1], abs(st["rays_shadow"] - ref[2]) / ref[2]
            print("4K interior, wide vs binary: pixels differing", differing, "of", W * H, "ray count drift", drift)
            assert differing <= 1e-6 * W * H and max(drift) <= 1e-6   # measured: 1 pixel of 8.3 M, drift 3e-8
        del g
    union = np.zeros_like(ref[0])
    for rank in range(2):
        g = gpu_backend.context(0)
        sc.upload(api_tables.gpu, g, W, H, 5)
        g.set_partition(rank, 2, 32)
        g.build_accel()
        g.render(1, 77)
        part = g.read_accum()
        assert not (union != 0)[part != 0].any()   # partitions are disjoint
        union += part
        del g
    assert np.array_equal(union, ref[0])


def test_degenerate_and_tiny_scenes(host, api_tables, orc, gpu_backend):
    """Empty scene, one primitive, zero-area triangles (excluded from the BVH, Geometry.cu:169-174)."""
    g = gpu_backend.context(0)
    o = orc.context(brute_force=True)
    lam = S.LambertianParams(S.float3(0.5, 0.5, 0.5))
    for ctx in (o, g):
        ctx.set_globals(16, 16, 5, bg=(0.25, 0.5, 0.75))
        ctx.set_camera(host.set_cam_params((0, 0, 5), (0, 0, 0), (0, 1, 0), 40, 1.0, 0.0, 1.0))
        ctx.build_accel()
        ctx.render(2, 1)
        img = ctx.read_accum()
        assert np.allclose(img, np.array([0.5, 1.0, 1.5], dtype=np.float32))  # 2 x bg, every pixel
    rays = random_rays(1000, [-1, -1, 2], [1, 1, 3], 6)
    rays[:, 4:7] = [0, 0, -1]
    for ctx in (o, g):
        ctx.clear_accum()
        verts = np.array([[-1, -1, 0], [1, -1, 0], [0, 1, 0], [2, 2, 0], [2, 2, 0], [3, 3, 0]], dtype=np.float32)
        ctx.add_mesh(verts, np.array([[0, 1, 2], [3, 4, 5]], dtype=np.int32), S.MAT_LAMBERTIAN, lam)  # 2nd is degenerate
        ctx.build_accel()
    to, io, _, _ = o.trace_closest(rays)
    tg, ig, _, _ = g.trace_closest(rays)
    assert np.array_equal(io, ig) and np.array_equal(to.view(np.uint32), tg.view(np.uint32))
    assert set(np.unique(ig)) <= {-1, 0} and (ig == 0).any()


def test_shadow_transmittance(host, api_tables, orc, gpu_backend):
    sc = host.Scene.builtin("interior", 30000)  # has Disney NORMAL and GLASS meshes
    o, g = both(host, api_tables, orc, gpu_backend, sc, 64, 64, 5)
    rays = random_rays(100000, [0.05, 0.05, 0.05], [9.95, 3.95, 7.95], 8, tmax=3.0)
    ao = o.trace_shadow(rays)
    ag = g.trace_shadow(rays)
    mism = np.any(ao != ag, axis=1).sum()
    assert (ao == 0).all(axis=1).any() and (ao == 1).all(axis=1).any()
    assert mism <= 5, mism


def image_metrics(a, b, n):
    a = a / n
    b = b / n
    rmse = float(np.sqrt(np.mean((np.clip(a, 0, 1) - np.clip(b, 0, 1)) ** 2)))
    from minimaloptix_b200 import host as H
    qa = H.accum_to_rgb8(a, 1).astype(np.int32)
    qb = H.accum_to_rgb8(b, 1).astype(np.int32)
    within = float(np.mean(np.all(np.abs(qa - qb) <= 1, axis=2)))
    lum = lambda x: float((0.3 * x[..., 0] + 0.6 * x[..., 1] + 0.1 * x[..., 2]).mean())
    rel = abs(lum(a) - lum(b)) / max(lum(b), 1e-6)
    return rmse, within, rel


# (scene kind, loader, w, h, spp, depth): rng=ref, equal seeds.  SURVEY.md §8d tolerance (ii) allows RMSE <= 2e-3;
# measured values are 4e-10 ... 1.3e-6 with equal ray counts, so the assertions hold the suite to RMSE <= 1e-5 and
# to equal counts up to the few Disney paths whose branch decision flips on a 1-ulp libm difference.
RENDER_CASES = [
    ("spheres_lens", None, 160, 90, 8, 5, 0xC0FFEE),
    ("spheres_pinhole", None, 160, 90, 8, 5, 0xC0FFEE),
    ("random_spheres", None, 192, 108, 4, 5, 0x5EED),
    ("cornell", "cornell", 128, 128, 16, 5, 0xC0FFEE),
    ("interior", 20000, 160, 90, 4, 5, 0xD1A1A6),
]


@pytest.mark.parametrize("case", RENDER_CASES, ids=[c[0] for c in RENDER_CASES])
def test_render_matches_oracle_ref_rng(host, api_tables, orc, gpu_backend, case):
    kind, arg, w, h, spp, depth, seed = case
    if arg == "cornell":
        sc = host.Scene.load(os.path.join(ROOT, "scenes", "cornell"), "cornell")
    elif isinstance(arg, int):
        sc = host.Scene.builtin(kind, arg)
    else:
        sc = host.Scene.builtin(kind)
    o, g = both(host, api_tables, orc, gpu_backend, sc, w, h, depth)
    o.render(spp, seed)
    g.render(spp, seed)
    a, b = g.read_accum(), o.read_accum()
    so, sg = o.stats(), g.stats()
    rmse, within, rel = image_metrics(a, b, spp)
    print(kind, "rmse", rmse, "within1", within, "rel-lum", rel, "rays", sg["rays_primary"], sg["rays_bounce"], sg["rays_shadow"],
          "oracle", so["rays_primary"], so["rays_bounce"], so["rays_shadow"])
    assert sg["nonfinite_samples"] == so["nonfinite_samples"] == 0
    assert sg["rays_primary"] == so["rays_primary"] == w * h * spp
    assert abs(sg["rays_bounce"] - so["rays_bounce"]) <= 1e-5 * so["rays_bounce"] + 1
    assert abs(sg["rays_shadow"] - so["rays_shadow"]) <= 1e-5 * so["rays_shadow"] + 1
    if so["rays_shadow"] == 0:
        assert sg["rays_bounce"] == so["rays_bounce"]   # no Disney shading: IEEE-exact operations only
    assert rmse <= 1e-5
    assert within >= 0.9999
    assert rel <= 1e-5


@pytest.mark.parametrize("kind", ["cornell", "interior"])
def test_brdf_ieee_mode_follows_the_oracle_operation_for_operation(host, api_tables, orc, gpu_backend, monkeypatch, kind):
    """BRDF values use the hardware reciprocal / square-root approximations by default (shading.cuh::bdiv, ~2 ulp);
    MOX_BRDF_IEEE=1 (read by mox_create) keeps every division and square root IEEE, i.e. the oracle's operations —
    what is left then is libm (powf / logf / sinf / cosf).  Directions never use the approximations, so both modes
    trace the same rays; the images of the two modes and the oracle agree far inside the 1e-5 the suite asserts."""
    sc = host.Scene.load(os.path.join(ROOT, "scenes", "cornell"), "cornell") if kind == "cornell" else host.Scene.builtin("interior", 20000)
    w, h, spp, seed = (128, 128, 16, 0xC0FFEE) if kind == "cornell" else (160, 90, 4, 0xD1A1A6)
    o = orc.context()
    sc.upload(api_tables.oracle, o, w, h, 5)
    o.build_accel()
    o.render(spp, seed)
    ref, so = o.read_accum(), o.stats()
    res = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("MOX_BRDF_IEEE", mode)
        g = gpu_backend.context(0)
        sc.upload(api_tables.gpu, g, w, h, 5)
        g.build_accel()
        g.render(spp, seed)
        st = g.stats()
        res[mode] = (g.read_accum(), st["rays_bounce"], st["rays_shadow"], image_metrics(g.read_accum(), ref, spp))
    print(kind, "ieee rmse/within/rel", res["1"][3], "fast", res["0"][3], "fast vs ieee", image_metrics(res["0"][0], res["1"][0], spp))
    assert res["1"][1:3] == res["0"][1:3]                          # the same rays in both modes
    assert abs(res["1"][1] - so["rays_bounce"]) <= 1e-5 * so["rays_bounce"] + 1
    assert res["1"][3][0] <= 2e-6 and res["0"][3][0] <= 1e-5        # RMSE against the oracle
    assert image_metrics(res["0"][0], res["1"][0], spp)[0] <= 2e-6  # the approximations themselves


@pytest.mark.skipif(not os.path.exists(os.path.join(ROOT, "scenes", "coffee", "coffee.scene")), reason="scenes/coffee not fetched")
def test_render_coffee_matches_oracle(host, api_tables, orc, gpu_backend):
    """BASELINE config 3 at reduced size.  The coffee materials have roughness 0.001-0.01: GTR2 is
    so peaked that 1-ulp differences between the CUDA and glibc sinf/cosf/powf move individual
    highlight samples, so pixels are compared with the stated tolerance, and ray counts may differ
    by the few paths whose `N.L > 0` / `pdf > 0` decision flips."""
    sc = host.Scene.load(os.path.join(ROOT, "scenes", "coffee"), "coffee")
    o, g = both(host, api_tables, orc, gpu_backend, sc, 480, 270, 5)
    o.render(2, 0xC0FFEE)
    g.render(2, 0xC0FFEE)
    so, sg = o.stats(), g.stats()
    rmse, within, rel = image_metrics(g.read_accum(), o.read_accum(), 2)
    print("coffee rmse", rmse, "within1", within, "rel", rel, "rays", sg["rays_bounce"], so["rays_bounce"], "shadow", sg["rays_shadow"], so["rays_shadow"])
    assert sg["rays_primary"] == so["rays_primary"]
    assert abs(sg["rays_bounce"] - so["rays_bounce"]) <= 1e-3 * so["rays_bounce"]
    assert abs(sg["rays_shadow"] - so["rays_shadow"]) <= 1e-3 * so["rays_shadow"]
    assert rmse <= 2e-3 and within >= 0.999 and rel <= 5e-3


def test_textured_disney_matches_oracle(host, api_tables, orc, gpu_backend):
    """§8 f-1: Disney albedo texture (bilinear, REPEAT, normalized coords).  The GPU uses the
    hardware filter (9-bit weights) like OptiX did; the oracle filters in float."""
    import tempfile
    from test_host import _textured_scene
    with tempfile.TemporaryDirectory() as tmp:
        sc = host.Scene.load(_textured_scene(tmp), "tex")
        o, g = both(host, api_tables, orc, gpu_backend, sc, 128, 128, 3)
        cam = host.set_cam_params((0, 1.5, 2.5), (0, 0, 0), (0, 1, 0), 40, 1.0, 0.0, 1.0)
        for ctx in (o, g):
            ctx.set_camera(cam)
            ctx.render(8, 11)
        a, b = g.read_accum(), o.read_accum()
        rmse, within, rel = image_metrics(a, b, 8)
        print("textured rmse", rmse, "within1", within, "rel", rel)
        img = a / 8
        assert (img[..., 0] > 2 * img[..., 1] + 0.02).any() and (img[..., 1] > 2 * img[..., 0] + 0.02).any()
        assert rmse <= 2e-3 and within >= 0.995 and rel <= 5e-3


# BASELINE configs 1-3 at THEIR resolution (spp reduced where the config's spp would take the oracle minutes):
# (name, width, height, spp, seed, Disney?)  Non-Disney scenes use only IEEE-exact operations (+ - * / sqrt), so
# every branch decision is the oracle's and the ray counts must be EQUAL; Disney shading calls sinf/cosf/powf/logf,
# where CUDA and glibc differ by an ulp, so a handful of `N.L > 0` / `pdf > 0` decisions per million paths may flip.
FULL_SIZE_CASES = [
    ("cornell", 512, 512, 16, 0xC0FFEE, True),          # config 1 exactly: 512x512, 16 spp, depth 5
    ("random_spheres", 1920, 1080, 2, 0x5EED, False),   # config 2 at 1920x1080, thin lens
    ("coffee", 1920, 1080, 1, 0xC0FFEE, True),          # config 3 at 1080p
]


@pytest.mark.parametrize("case", FULL_SIZE_CASES, ids=[c[0] for c in FULL_SIZE_CASES])
def test_baseline_configs_at_full_resolution(host, api_tables, orc, gpu_backend, case):
    name, w, h, spp, seed, is_disney = case
    if name == "random_spheres":
        sc = host.Scene.builtin(name)
    else:
        d = os.path.join(ROOT, "scenes", name)
        if not os.path.exists(os.path.join(d, name + ".scene")):
            pytest.skip(f"scenes/{name} not present")
        sc = host.Scene.load(d, name)
    o, g = both(host, api_tables, orc, gpu_backend, sc, w, h, 5)
    o.render(spp, seed)
    g.render(spp, seed)
    so, sg = o.stats(), g.stats()
    rmse, within, rel = image_metrics(g.read_accum(), o.read_accum(), spp)
    print(name, f"{w}x{h}x{spp}", "rmse", rmse, "within1", within, "rel", rel, "bounce", sg["rays_bounce"], so["rays_bounce"],
          "shadow", sg["rays_shadow"], so["rays_shadow"])
    assert sg["nonfinite_samples"] == so["nonfinite_samples"] == 0
    assert sg["rays_primary"] == so["rays_primary"] == w * h * spp
    if not is_disney:
        assert sg["rays_bounce"] == so["rays_bounce"]
        assert rmse <= 1e-5 and within == 1.0
    elif name == "cornell":
        assert abs(sg["rays_bounce"] - so["rays_bounce"]) <= 4e-6 * so["rays_bounce"]
        assert abs(sg["rays_shadow"] - so["rays_shadow"]) <= 4e-6 * so["rays_shadow"]
        assert rmse <= 1e-5 and within >= 0.99999
    else:
        # coffee: roughness 0.001-0.01 makes GTR2 so peaked that 1-ulp differences in sinf/cosf/powf move
        # individual highlight samples (stated tolerance of SURVEY §8d ii)
        assert abs(sg["rays_bounce"] - so["rays_bounce"]) <= 1e-3 * so["rays_bounce"]
        assert abs(sg["rays_shadow"] - so["rays_shadow"]) <= 1e-3 * so["rays_shadow"]
        assert rmse <= 1e-3 and within >= 0.999 and rel <= 5e-3


@pytest.mark.parametrize("mode", [S.RNG_REF, S.RNG_PHILOX], ids=["ref", "philox"])
@pytest.mark.parametrize("textured", [False, True], ids=["plain", "textured"])
def test_zoo_every_program_matches_oracle(host, orc, gpu_backend, mode, textured):
    """The scene of tests/refcases.py that runs every program — Disney NORMAL with all lobes, Disney GLASS, a
    SPHERE light (volume sampling, Material.cu:177-179; corrected sphere box, Geometry.cu:57-63) next to a QUAD
    light, lambertian / metal / glass — on the GPU against the oracle, in both RNG modes (Philox x Disney)."""
    import refcases as R
    o, g = orc.context(), gpu_backend.context(0)
    for ctx in (o, g):
        R.build_zoo(ctx, host, 240, 160, 5, textured=textured)
        ctx.set_rng_mode(mode)
        ctx.render(8, 0xD15EA5E)
    so, sg = o.stats(), g.stats()
    rmse, within, rel = image_metrics(g.read_accum(), o.read_accum(), 8)
    print("zoo", mode, textured, "rmse", rmse, "within1", within, "rel", rel, sg["rays_bounce"], so["rays_bounce"], sg["rays_shadow"], so["rays_shadow"])
    assert sg["nonfinite_samples"] == so["nonfinite_samples"] == 0
    assert sg["rays_primary"] == so["rays_primary"]
    assert sg["rays_shadow"] > 0.5 * sg["rays_primary"]      # two lights, most first hits are Disney
    assert abs(sg["rays_bounce"] - so["rays_bounce"]) <= 1e-5 * so["rays_bounce"] + 2
    assert abs(sg["rays_shadow"] - so["rays_shadow"]) <= 1e-5 * so["rays_shadow"] + 2
    if textured:   # hardware bilinear filter (9-bit weights) vs float filter in the oracle
        assert rmse <= 2e-3 and within >= 0.995
    else:
        # Glossy Disney lobes: a 1-ulp difference between CUDA's and glibc's sinf/cosf/powf flips the branch
        # decision of a few paths per million (measured: 0-3 of 373 k), and one flipped path moves one pixel of
        # this small image by up to 1/spp.  So: at most a handful of outlier pixels, everything else to 1e-5.
        d = np.abs(g.read_accum() - o.read_accum()).max(axis=-1) / 8
        outliers = d > 1e-4
        assert outliers.sum() <= 6, int(outliers.sum())
        assert float(np.sqrt(np.mean(d[~outliers] ** 2))) <= 1e-5 and within >= 0.9999
    # primitive ids, t, beta, gamma against brute force on incoherent rays through the zoo
    ob = orc.context(brute_force=True)
    R.build_zoo(ob, host, 16, 16, 5, textured=textured)
    nbad, nhit = check_ids(ob, g, random_rays(100000, [-4, 0.01, -4], [4, 4, 4], 12), "zoo")
    assert nhit > 30000 and nbad <= 2
    # shadow transmittance incl. the tinting GLASS sphere
    rays = random_rays(50000, [-4, 0.01, -4], [4, 4, 4], 13, tmax=3.0)
    assert np.any(ob.trace_shadow(rays) != g.trace_shadow(rays), axis=1).sum() <= 2


def test_disney_with_more_than_32_lights(host, orc, gpu_backend):
    """The Disney kernel reserves its shadow-queue slots once per group of 32 lights (one bit per light): 40 quad lights
    and one sphere light cross the group boundary.  Equal ray counts — one shadow ray per light and hit that faces it —
    and the image of the oracle."""
    d = S.DisneyParams()
    d.color = S.float3(0.7, 0.6, 0.5); d.specular = d.roughness = d.sheenTint = 0.5; d.clearcoatGloss = 1.0; d.metallic = 0.2
    floor = S.DisneyParams()
    floor.color = S.float3(0.4, 0.5, 0.6); floor.specular = floor.roughness = floor.sheenTint = 0.5; floor.clearcoatGloss = 1.0
    lights = []
    for k in range(40):
        lq = S.LightParams()
        x, z = -3.0 + 0.75 * (k % 8), -2.0 + 0.9 * (k // 8)
        lq.position, lq.u, lq.v, lq.normal = S.float3(x, 3.0, z), S.float3(0.3, 0, 0), S.float3(0, 0, 0.3), S.float3(0, -1, 0)
        lq.area, lq.emission, lq.shape = 0.09, S.float3(3, 3, 3), S.QUAD
        lights.append(lq)
    ls = S.LightParams()
    ls.position, ls.radius, ls.area, ls.emission, ls.shape = S.float3(2.5, 1.0, 1.5), 0.2, 4 * 3.14159265 * 0.04, S.float3(6, 5, 4), S.SPHERE
    lights.append(ls)
    out = []
    for ctx in (orc.context(), gpu_backend.context(0)):
        ctx.set_globals(96, 64, 4, bg=(0.05, 0.05, 0.05))
        ctx.set_camera(host.set_cam_params((0, 1.5, 5), (0, 0.5, 0), (0, 1, 0), 40, 1.5, 0.0, 1.0))
        ctx.add_sphere(S.SphereParams(0.8, S.float3(0, 0.8, 0), S.float3()), S.MAT_DISNEY, d)
        ctx.add_quad(host.set_quad_params((-6, 0, -6), (12, 0, 0), (0, 0, 12)), S.MAT_DISNEY, floor)
        for lq in lights[:40]:
            ctx.add_quad(host.set_quad_params((lq.position.x, lq.position.y, lq.position.z), (0.3, 0, 0), (0, 0, 0.3)), S.MAT_LIGHT, lq)
        ctx.add_sphere(S.SphereParams(0.2, S.float3(2.5, 1.0, 1.5), S.float3()), S.MAT_LIGHT, ls)
        ctx.set_lights(lights)
        ctx.build_accel()
        ctx.render(3, 41)
        st = ctx.stats()
        out.append((ctx.read_accum(), st["rays_bounce"], st["rays_shadow"], st["nonfinite_samples"]))
    assert out[0][1:] == out[1][1:]
    assert out[1][2] > 41 * 1000
    rmse, within, rel = image_metrics(out[1][0], out[0][0], 3)
    print("41 lights: rmse", rmse, "shadow rays", out[1][2])
    assert rmse <= 1e-5 and within >= 0.9999


def test_nonfinite_samples_become_bad_color(host, orc, gpu_backend):
    """Exception.cu:10-12 / MinimalOptiX.cpp:149-151: badColor is what the reference paints when a launch index
    fails.  Here a NaN/Inf sample is that failure: a Disney material with a negative colour (pow(c, 2.2) = NaN) and a NaN emission.
    Custom badColor; oracle and GPU agree, count the same samples, and a pixel fully covered by the bad sphere is
    exactly spp x badColor."""
    bad = (0.25, 0.5, 0.75)
    d = S.DisneyParams()
    d.color = S.float3(-1.0, 0.5, 0.5); d.specular = d.roughness = d.sheenTint = 0.5; d.clearcoatGloss = 1.0
    d.emission = S.float3(float("nan"), 0.0, 0.0)     # every hit of this material is non-finite, whatever the path does next
    lq = S.LightParams()
    lq.position, lq.u, lq.v, lq.normal = S.float3(-1, 3, -1), S.float3(2, 0, 0), S.float3(0, 0, 2), S.float3(0, -1, 0)
    lq.area, lq.emission, lq.shape = 4.0, S.float3(5, 5, 5), S.QUAD
    imgs, stats = [], []
    for ctx in (orc.context(), gpu_backend.context(0)):
        ctx.set_globals(64, 64, 5, bad=bad, bg=(0.1, 0.1, 0.1))
        ctx.set_camera(host.set_cam_params((0, 0, 4), (0, 0, 0), (0, 1, 0), 30, 1.0, 0.0, 1.0))
        ctx.add_sphere(S.SphereParams(0.7, S.float3(0, 0, 0), S.float3()), S.MAT_DISNEY, d)
        ctx.add_quad(host.set_quad_params((-1, 3, -1), (2, 0, 0), (0, 0, 2)), S.MAT_LIGHT, lq)
        ctx.set_lights([lq])
        ctx.build_accel()
        ctx.render(4, 3)
        imgs.append(ctx.read_accum()); stats.append(ctx.stats())
    assert stats[0]["nonfinite_samples"] == stats[1]["nonfinite_samples"] > 1000
    assert np.allclose(imgs[0], imgs[1], atol=1e-5)
    assert np.array_equal(imgs[1][32, 32], 4 * np.array(bad, np.float32))      # centre pixel: every sample hits the sphere
    assert np.allclose(imgs[1][1, 1], 4 * 0.1)                                # corner: background only


def test_scheduling_variants_are_bit_identical(host, api_tables, gpu_backend, monkeypatch):
    """How a render is scheduled must not show in the result: shadow rays on a second stream or in line, and all
    samples in one batch or one sample per batch (MOX_MAX_BATCH_PATHS = the pixel count: three batches, whose
    samples k_accumulate adds in launch order) — same image bit for bit, same ray counts (all read by mox_create)."""
    sc = host.Scene.builtin("interior", 30000)
    out = []
    for overlap, batch_paths in (("1", None), ("0", None), ("1", str(400 * 300))):
        monkeypatch.setenv("MOX_OVERLAP_SHADOW", overlap)
        if batch_paths is None:
            monkeypatch.delenv("MOX_MAX_BATCH_PATHS", raising=False)
        else:
            monkeypatch.setenv("MOX_MAX_BATCH_PATHS", batch_paths)
        g = gpu_backend.context(0)
        sc.upload(api_tables.gpu, g, 400, 300, 5)
        g.build_accel()
        g.render(3, 77)
        st = g.stats()
        out.append((g.read_accum(), st["rays_bounce"], st["rays_shadow"], st["extend_launches"]))
    for o in out[1:]:
        assert o[1:3] == out[0][1:3]
        assert np.array_equal(o[0].view(np.uint32), out[0][0].view(np.uint32))
    assert out[2][3] > out[0][3]    # three batches: the bounce loop ran once per batch


def test_wide_and_binary_traversal_render_identically(host, api_tables, gpu_backend):
    """The acceleration structure must not influence the image: 8-wide vs binary BVH, bit for bit
    (including the order-independent shadow transmittance through GLASS)."""
    sc = host.Scene.builtin("interior", 30000)
    imgs = []
    for flags in (S.ACCEL_DEFAULT, S.ACCEL_BINARY, S.ACCEL_LBVH):
        g = gpu_backend.context(0)
        sc.upload(api_tables.gpu, g, 160, 90, 5)
        g.build_accel(flags)
        g.render(3, 9)
        st = g.stats()
        imgs.append((g.read_accum(), st["rays_bounce"], st["rays_shadow"], st["node_bytes"]))
    assert imgs[0][3] == 80 and imgs[1][3] == 64
    assert imgs[0][1:3] == imgs[1][1:3] == imgs[2][1:3]
    # GLASS attenuation is a product over hits in traversal order: allow last-bit differences only there
    assert np.allclose(imgs[0][0], imgs[1][0], rtol=0, atol=1e-5) and np.allclose(imgs[0][0], imgs[2][0], rtol=0, atol=1e-5)
    assert np.mean(imgs[0][0] == imgs[1][0]) > 0.999


def test_shading_records_equal_the_gather_path(host, api_tables, gpu_backend, monkeypatch):
    """The per-triangle 128-byte shading records hold exactly what the index gather reads (positions,
    normals, uvs): images are bit-identical with `MOX_SHADE_RECORDS=0`, on a mesh scene with normals and on a
    textured mesh with uvs."""
    import tempfile
    from test_host import _textured_scene

    def render(sc, w, h, spp, cam=None):
        out = []
        for rec in ("1", "0"):
            monkeypatch.setenv("MOX_SHADE_RECORDS", rec)   # read by mox_build_accel
            g = gpu_backend.context(0)
            sc.upload(api_tables.gpu, g, w, h, 5)
            g.build_accel()
            if cam is not None:
                g.set_camera(cam)
            g.render(spp, 21)
            out.append((g.read_accum(), g.stats()["rays_bounce"], g.stats()["rays_shadow"]))
        return out

    a, b = render(host.Scene.builtin("interior", 30000), 160, 90, 3)
    assert a[1:] == b[1:] and np.array_equal(a[0], b[0])
    with tempfile.TemporaryDirectory() as tmp:
        sc = host.Scene.load(_textured_scene(tmp), "tex")
        cam = host.set_cam_params((0, 1.5, 2.5), (0, 0, 0), (0, 1, 0), 40, 1.0, 0.0, 1.0)
        a, b = render(sc, 96, 96, 4, cam)
        assert a[1:] == b[1:] and np.array_equal(a[0], b[0])
        assert a[0].max() > 0


def test_render_matches_oracle_philox(host, api_tables, orc, gpu_backend):
    sc = host.Scene.builtin("random_spheres")
    o, g = both(host, api_tables, orc, gpu_backend, sc, 160, 90, 5, 5)
    for ctx in (o, g):
        ctx.set_rng_mode(S.RNG_PHILOX)
        ctx.render(4, 99)
    rmse, within, rel = image_metrics(g.read_accum(), o.read_accum(), 4)
    assert o.stats()["rays_bounce"] == g.stats()["rays_bounce"]
    assert rmse <= 1e-5 and within >= 0.9999


def test_batched_render_equals_single_launches(host, api_tables, gpu_backend):
    sc = host.Scene.builtin("spheres_lens")
    g1, g2 = gpu_backend.context(0), gpu_backend.context(0)
    for g in (g1, g2):
        sc.upload(api_tables.gpu, g, 96, 54, 5)
        g.build_accel()
    g1.render(6, 123)
    for k in range(6):
        g2.launch(host.launch_seed(k, 123))
    assert np.array_equal(g1.read_accum().view(np.uint32), g2.read_accum().view(np.uint32))
    assert np.array_equal(g1.map_accum(), g1.read_accum())  # map() view == copied read
    # progressive: two renders continue the seed schedule
    g2.clear_accum()
    g2.render(2, 123)
    g2.render(4, 123)
    assert np.array_equal(g1.read_accum().view(np.uint32), g2.read_accum().view(np.uint32))


def test_tile_partition_union_is_bit_identical(host, api_tables, gpu_backend):
    """Virtual ranks on one GPU: rendering the tile sets of 3 ranks and gathering them through
    pack/unpack must reproduce the 1-rank accumulation buffer bit for bit (seeds depend only on
    the global pixel index)."""
    import torch
    sc = host.Scene.builtin("random_spheres")
    w, h, world = 200, 120, 3  # ragged tiles on both axes
    full = gpu_backend.context(0)
    sc.upload(api_tables.gpu, full, w, h, 5)
    full.build_accel()
    full.render(3, 77)
    want = full.read_accum()
    root = gpu_backend.context(0)
    sc.upload(api_tables.gpu, root, w, h, 5)
    root.set_partition(0, world, 32)
    root.build_accel()
    total = 0
    for r in range(world):
        ctx = gpu_backend.context(0)
        sc.upload(api_tables.gpu, ctx, w, h, 5)
        ctx.set_partition(r, world, 32)
        ctx.build_accel()
        ctx.render(3, 77)
        n = ctx.owned_pixels(r)
        total += n
        buf = torch.empty(n * 3, dtype=torch.float32, device="cuda:0")
        ctx.pack_owned(buf.data_ptr())
        torch.cuda.synchronize()
        root.unpack_owned(r, buf.data_ptr())
    assert total == w * h
    got = root.read_accum()
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def test_animated_spheres_rebuild_and_resume(host, api_tables, orc, gpu_backend):
    """§8 f-2/f-3: move the spheres (reference animate()), update + rebuild on both sides, images
    still agree; then dump / set_accum resumes the seed schedule bit-exactly."""
    sc = host.Scene.builtin("random_spheres")
    o, g = both(host, api_tables, orc, gpu_backend, sc, 160, 90, 5)
    for _ in range(5):
        sc.animate(0.002)
    sc.apply_spheres(api_tables.oracle, o)
    sc.apply_spheres(api_tables.gpu, g)
    from minimaloptix_b200 import MoxError
    with pytest.raises(MoxError):
        g.launch(1)  # accel is stale after update_sphere
    o.build_accel(); g.build_accel()
    o.render(4, 5); g.render(4, 5)
    rmse, within, rel = image_metrics(g.read_accum(), o.read_accum(), 4)
    assert rmse <= 2e-3 and within >= 0.999
    # the moved scene differs from the static one
    s2 = host.Scene.builtin("random_spheres")
    g2 = gpu_backend.context(0)
    s2.upload(api_tables.gpu, g2, 160, 90, 5)
    g2.build_accel(); g2.render(4, 5)
    assert not np.array_equal(g2.read_accum(), g.read_accum())
    # resume: 2 spp, dump, reload into a fresh context, 2 more == 4 spp in one go
    g3 = gpu_backend.context(0)
    s2.upload(api_tables.gpu, g3, 160, 90, 5)
    g3.build_accel(); g3.render(2, 5)
    half = g3.read_accum()
    g4 = gpu_backend.context(0)
    s2.upload(api_tables.gpu, g4, 160, 90, 5)
    g4.build_accel()
    g4.set_accum(half, 2)
    g4.render(2, 5)
    assert np.array_equal(g4.read_accum().view(np.uint32), g2.read_accum().view(np.uint32))


def test_deep_paths_default_depth_and_philox(host, api_tables, orc, gpu_backend):
    """rayMaxDepth = 256 (the reference default, MinimalOptiX.h:85): the wavefront loop runs until
    every path has terminated; both RNG modes."""
    sc = host.Scene.builtin("spheres_pinhole")
    for mode in (S.RNG_REF, S.RNG_PHILOX):
        o, g = both(host, api_tables, orc, gpu_backend, sc, 96, 54, 256)
        for ctx in (o, g):
            ctx.set_rng_mode(mode)
            ctx.render(2, 77)
        so, sg = o.stats(), g.stats()
        rmse, within, rel = image_metrics(g.read_accum(), o.read_accum(), 2)
        assert sg["rays_bounce"] == so["rays_bounce"] and sg["rays_bounce"] > sg["rays_primary"]
        assert rmse <= 2e-3 and within >= 0.999


def test_headless_cli_snapshots_and_resume(tmp_path):
    """mox_cli replaces the Qt app: power-of-two snapshots (MinimalOptiX.cpp:543-553), final PNG,
    JSON stats line, accumulator dump and --resume."""
    import json, subprocess
    from PIL import Image
    cli = os.path.join(ROOT, "minimaloptix_b200", "mox_cli")
    out = str(tmp_path / "cb")
    cmd = [cli, "--scene", "cornell", "--scene-dir", os.path.join(ROOT, "scenes"), "--width", "96", "--height", "96", "--max-depth", "5",
           "--seed", "0xC0FFEE", "--out", out]
    r = subprocess.run(cmd + ["--spp", "8", "--snapshots", "--dump-accum"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    stats = json.loads(r.stdout.strip().splitlines()[-1])
    assert stats["spp"] == 8 and stats["triangles"] == 30 and stats["mrays_per_s"] > 0 and stats["nonfinite"] == 0
    for n in (1, 2, 4, 8):
        assert os.path.exists(f"{out}_{n}.png")
    full = np.asarray(Image.open(out + ".png"))
    assert full.shape == (96, 96, 3) and full.std() > 5
    # 4 spp, dump, then resume to 8 spp: same pixels as the 8 spp run
    out2 = str(tmp_path / "half")
    r = subprocess.run([c if c != out else out2 for c in cmd] + ["--spp", "4", "--dump-accum"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    out3 = str(tmp_path / "resumed")
    r = subprocess.run([c if c != out else out3 for c in cmd] + ["--spp", "8", "--resume", out2 + ".moxa"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert np.array_equal(np.asarray(Image.open(out3 + ".png")), full)


def test_error_paths(host, api_tables, gpu_backend):
    from minimaloptix_b200 import MoxError
    g = gpu_backend.context(0)
    with pytest.raises(MoxError):
        g.launch(1)  # no accel yet
    g.set_globals(8, 8, 5)
    g.build_accel()
    with pytest.raises(MoxError):
        g.launch(1)  # no camera
    with pytest.raises(MoxError):
        g.add_mesh(np.zeros((3, 3), np.float32), np.array([[0, 1, 7]], np.int32), S.MAT_LAMBERTIAN,
                   S.LambertianParams(S.float3(1, 1, 1)))
    with pytest.raises(MoxError):
        g.set_partition(3, 2, 32)


# ---------------------------------------------------------------------------------------------- multi-GPU handle
def _render_image(ctx, sc, api, w, h, spp, seed):
    sc.upload(api, ctx, w, h, 5)
    ctx.build_accel()
    ctx.render(spp, seed)
    return ctx.read_accum(), ctx.stats()


def test_multi_handle_on_one_device_equals_plain_context(host, api_tables, gpu_backend):
    """mox_create_multi with a single device goes through the whole group machinery (forwarded scene calls, worker
    thread, push into the gather buffer, asynchronous read-back) and must give the plain context's image bit for bit."""
    sc = host.Scene.builtin("interior", 20000)
    want, st0 = _render_image(gpu_backend.context(0), sc, api_tables.gpu, 200, 120, 3, 17)
    m = gpu_backend.multi_context([0])
    assert m.device_count() == 1
    got, st1 = _render_image(m, sc, api_tables.gpu, 200, 120, 3, 17)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert (st0["rays_bounce"], st0["rays_shadow"]) == (st1["rays_bounce"], st1["rays_shadow"])
    from minimaloptix_b200 import MoxError
    with pytest.raises(MoxError):
        m.set_partition(0, 2, 32)     # the handle owns the partition
    # raw queries go to device 0
    rays = random_rays(5000, [0.05, 0.05, 0.05], [9.95, 3.95, 7.95], 3)
    g = gpu_backend.context(0)
    sc.upload(api_tables.gpu, g, 64, 64, 5); g.build_accel()
    assert all(np.array_equal(a, b) for a, b in zip(m.trace_closest(rays), g.trace_closest(rays)))


def test_asynchronous_readback_double_buffer(host, api_tables, gpu_backend):
    """mox_read_accum_begin/_end: the snapshot is taken at _begin, rendering continues, two host images alternate."""
    sc = host.Scene.builtin("spheres_lens")
    g = gpu_backend.context(0)
    sc.upload(api_tables.gpu, g, 160, 90, 5)
    g.build_accel()
    g.render(2, 5)
    a2 = g.read_accum()
    g.read_accum_begin()            # snapshot of the 2-spp image ...
    g.render(2, 5)                  # ... while 2 more samples are rendered
    img2 = g.read_accum_end().copy()
    a4 = g.read_accum()
    g.read_accum_begin()
    img4 = g.read_accum_end()
    assert np.array_equal(img2, a2) and np.array_equal(img4, a4) and not np.array_equal(a2, a4)
    from minimaloptix_b200 import MoxError
    with pytest.raises(MoxError):
        g.read_accum_end()          # nothing pending


def _n_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.skipif("_n_gpus() < 2", reason="needs two GPUs")
def test_multi_handle_two_devices_bit_identical_and_cli(host, api_tables, gpu_backend, tmp_path):
    """Two devices behind one handle (C++ threads, tiles pushed over NVLink into device 0): the image equals the
    one-device image bit for bit; and the headless C++ driver does the same without any Python (mox_cli --gpus 2)."""
    import json, subprocess
    from PIL import Image
    sc = host.Scene.builtin("interior", 60000)
    want, st0 = _render_image(gpu_backend.context(0), sc, api_tables.gpu, 400, 240, 4, 29)
    m = gpu_backend.multi_context([0, 1])
    got, st1 = _render_image(m, sc, api_tables.gpu, 400, 240, 4, 29)
    assert m.device_count() == 2
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert (st0["rays_primary"], st0["rays_bounce"], st0["rays_shadow"]) == (st1["rays_primary"], st1["rays_bounce"], st1["rays_shadow"])
    # progressive: a second render continues the seed schedule on every device
    m.render(2, 29)
    g = gpu_backend.context(1)     # and a plain context on the OTHER device agrees too
    sc.upload(api_tables.gpu, g, 400, 240, 5); g.build_accel(); g.render(6, 29)
    assert np.array_equal(m.read_accum().view(np.uint32), g.read_accum().view(np.uint32))
    cli = os.path.join(ROOT, "minimaloptix_b200", "mox_cli")
    outs = []
    for extra, name in ((["--device", "0"], "one"), (["--gpus", "2"], "two")):
        out = str(tmp_path / name)
        r = subprocess.run([cli, "--scene", "cornell", "--scene-dir", os.path.join(ROOT, "scenes"), "--width", "256", "--height", "256",
                            "--max-depth", "5", "--spp", "8", "--seed", "7", "--out", out] + extra, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
        outs.append((np.asarray(Image.open(out + ".png")), json.loads(r.stdout.strip().splitlines()[-1])))
    assert np.array_equal(outs[0][0], outs[1][0])
    assert outs[1][1]["gpus"] == 2 and outs[0][1]["rays_bounce"] == outs[1][1]["rays_bounce"]


@pytest.mark.skipif("_n_gpus() < 2", reason="needs two GPUs")
def test_peer_memory_gather_across_processes():
    """One process per GPU (the bench.py / torchrun arrangement): every rank pushes its tiles into rank 0's gather
    buffer through a CUDA IPC mapping; rank 0's frame equals the 1-rank frame bit for bit."""
    import socket, subprocess, sys
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), LOCAL_RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "_mp_gpu_worker.py")], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=300)[0] for p in procs]
    for r, p in enumerate(procs):
        assert p.returncode == 0, f"rank {r} failed:\n{outs[r]}"
    assert "bit-identical: True" in outs[0] and "peer-memory" in outs[0]
