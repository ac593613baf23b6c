"""The terminal bounce (the one past rayMaxDepth) resolved from the light list and an any-hit query.

k_classify ends every path of that bounce, and k_accumulate adds one term chosen by the hit record alone: miss,
light or anything else.  The library answers it with the closest light and an any-hit traversal bounded by it;
MOX_TERMINAL_CLOSEST=1 (read by mox_create) runs the closest-hit traversal instead.  Both must render the same
accumulation buffer bit for bit, with the same ray counts.  A context that uses the terminal query skips one
k_classify launch per batch, which is how these tests see that it ran."""
import numpy as np
import pytest

from minimaloptix_b200 import structs as S

pytestmark = pytest.mark.gpu

COUNTS = ("rays_primary", "rays_bounce", "rays_shadow", "rays_shadow_traced", "rays_shadow_blocked", "rays_shadow_tinted",
          "nonfinite_samples", "rays_depth", "shadow_traced_depth")


def render_both(monkeypatch, gpu_backend, setup, spp, seed):
    """[(accumulation buffer, stats)] with the terminal query, then with the closest-hit traversal."""
    out = []
    for closest in ("0", "1"):
        monkeypatch.setenv("MOX_TERMINAL_CLOSEST", closest)
        g = gpu_backend.context(0)
        setup(g)
        g.render(spp, seed)
        out.append((g.read_accum(), g.stats()))
    return out


def assert_same(out, terminal_ran=True):
    (ia, sa), (ib, sb) = out
    assert np.array_equal(ia.view(np.uint32), ib.view(np.uint32))
    for k in COUNTS:
        assert sa[k] == sb[k], k
    assert sa["rays_primary"] > 0
    if terminal_ran:
        assert sa["kernel_launches"] < sb["kernel_launches"]
    else:
        assert sa["kernel_launches"] == sb["kernel_launches"]


def upload(api_tables, scene, w, h, depth, flags=0, **globals_):
    def setup(g):
        scene.upload(api_tables.gpu, g, w, h, depth)
        if globals_:
            g.set_globals(w, h, depth, **globals_)
        g.build_accel(flags)
    return setup


@pytest.mark.parametrize("flags", [S.ACCEL_DEFAULT, S.ACCEL_WATERTIGHT, S.ACCEL_COUNTERS], ids=["wide", "watertight", "counters"])
def test_interior(host, api_tables, gpu_backend, monkeypatch, flags):
    sc = host.Scene.builtin("interior", 30000)
    out = render_both(monkeypatch, gpu_backend, upload(api_tables, sc, 160, 120, 5, flags), 3, 77)
    assert_same(out)
    if flags == S.ACCEL_COUNTERS:   # the any-hit query visits fewer nodes than the closest-hit traversal
        assert 0 < out[0][1]["node_visits"] < out[1][1]["node_visits"]


def test_interior_absorb_differs_from_background(host, api_tables, gpu_backend, monkeypatch):
    """With absorbColor != bgColor a ray that hits no light still needs the any-hit query."""
    sc = host.Scene.builtin("interior", 30000)
    setup = upload(api_tables, sc, 160, 120, 5, absorb=(0.25, 0.5, 0.125), bg=(0.0625, 0.125, 0.375))
    assert_same(render_both(monkeypatch, gpu_backend, setup, 3, 78))


@pytest.mark.parametrize("depth", [0, 1])
def test_interior_shallow(host, api_tables, gpu_backend, monkeypatch, depth):
    sc = host.Scene.builtin("interior", 30000)
    setup = upload(api_tables, sc, 96, 72, depth, absorb=(0.5, 0.25, 0.125), bg=(0.125, 0.25, 0.5))
    assert_same(render_both(monkeypatch, gpu_backend, setup, 2, 79))


def test_cornell(host, api_tables, gpu_backend, monkeypatch):
    import os
    sc = host.Scene.load(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scenes", "cornell"), "cornell")
    assert_same(render_both(monkeypatch, gpu_backend, upload(api_tables, sc, 96, 96, 5), 4, 80))


def test_random_spheres(host, api_tables, gpu_backend, monkeypatch):
    """bgColor 0.2, absorbColor 0: every terminal ray runs the any-hit query."""
    sc = host.Scene.builtin("random_spheres")
    assert_same(render_both(monkeypatch, gpu_backend, upload(api_tables, sc, 128, 72, 5), 3, 81))


@pytest.mark.parametrize("mode", [S.RNG_REF, S.RNG_PHILOX], ids=["ref", "philox"])
def test_zoo_sphere_light(host, gpu_backend, monkeypatch, mode):
    import refcases as R

    def setup(g):
        R.build_zoo(g, host, 120, 80, 5, textured=False)
        g.set_rng_mode(mode)
    assert_same(render_both(monkeypatch, gpu_backend, setup, 4, 0xD15EA5E))


def test_zoo_refit_after_moving_the_light_sphere(host, gpu_backend, monkeypatch):
    import refcases as R

    def setup(g):
        R.build_zoo(g, host, 120, 80, 5, textured=False)
        light_sphere = g.stats()["n_prims"] - 2      # build_zoo adds the light sphere, then the light quad
        g.update_sphere(light_sphere, S.SphereParams(0.5, S.float3(0.3, 1.9, 1.0), S.float3()))
        g.build_accel(S.ACCEL_REFIT)
    assert_same(render_both(monkeypatch, gpu_backend, setup, 4, 82))


def light(pos, u, v, emission):
    lq = S.LightParams()
    n = np.cross(u, v)
    lq.position, lq.u, lq.v = S.float3(*pos), S.float3(*u), S.float3(*v)
    lq.area = float(np.linalg.norm(n)); lq.normal = S.float3(*(n / np.linalg.norm(n)))
    lq.emission, lq.shape = S.float3(*emission), S.QUAD
    return lq


def test_coplanar_light_and_blockers(host, gpu_backend, monkeypatch):
    """A light quad between two non-light quads in the same plane: a camera ray meets all of them at the same t, and
    the lower id wins.  Left half of the light: the quad before it (absorbColor); right half: the light itself, ahead
    of the quad after it."""
    absorb, bg, emission = (0.5, 0.25, 0.125), (0.125, 0.25, 0.5), (0.875, 0.75, 0.625)
    lq = light((-0.5, -0.5, 0.0), (1.0, 0.0, 0.0), (0.0, 1.0, 0.0), emission)

    def scene(depth):
        def setup(g):
            g.set_globals(64, 64, depth, absorb=absorb, bg=bg)
            g.set_camera(host.set_cam_params((0, 0, 4), (0, 0, 0), (0, 1, 0), 40, 1.0, 0.0, 1.0))
            lam = S.LambertianParams(S.float3(0.5, 0.5, 0.5))
            assert g.add_quad(host.set_quad_params((-1.0, -1.0, 0.0), (1.0, 0.0, 0.0), (0.0, 2.0, 0.0)), S.MAT_LAMBERTIAN, lam) == 0
            assert g.add_quad(host.set_quad_params((-0.5, -0.5, 0.0), (1.0, 0.0, 0.0), (0.0, 1.0, 0.0)), S.MAT_LIGHT, lq) == 1
            assert g.add_quad(host.set_quad_params((0.0, -1.0, 0.0), (1.0, 0.0, 0.0), (0.0, 2.0, 0.0)), S.MAT_LAMBERTIAN, lam) == 2
            g.add_quad(host.set_quad_params((-3.0, -1.5, 3.0), (6.0, 0.0, 0.0), (0.0, 0.0, -6.0)), S.MAT_LAMBERTIAN, lam)
            g.set_lights([lq])
            g.build_accel()
        return setup
    for depth in (0, 1):
        out = render_both(monkeypatch, gpu_backend, scene(depth), 1, 83)
        assert_same(out)
        if depth == 0:
            px = out[0][0].reshape(-1, 3)
            assert (px == np.float32(absorb)).all(axis=1).sum() > 100
            assert (px == np.float32(emission)).all(axis=1).sum() > 100


def test_triangle_mesh_light_keeps_closest_hit(host, gpu_backend, monkeypatch):
    lq = light((-0.5, 2.0, -0.5), (1.0, 0.0, 0.0), (0.0, 0.0, 1.0), (4.0, 4.0, 4.0))

    def setup(g):
        g.set_globals(64, 48, 3, bg=(0.1, 0.1, 0.1))
        g.set_camera(host.set_cam_params((0, 1, 4), (0, 0.5, 0), (0, 1, 0), 45, 64 / 48, 0.0, 1.0))
        g.add_quad(host.set_quad_params((-3, 0, -3), (6, 0, 0), (0, 0, 6)), S.MAT_LAMBERTIAN, S.LambertianParams(S.float3(0.6, 0.6, 0.6)))
        v = np.array([[-0.5, 2.0, -0.5], [0.5, 2.0, -0.5], [0.5, 2.0, 0.5], [-0.5, 2.0, 0.5]], np.float32)
        g.add_mesh(v, np.array([[0, 1, 2], [0, 2, 3]], np.int32), S.MAT_LIGHT, lq)
        g.set_lights([lq])
        g.build_accel()
    assert_same(render_both(monkeypatch, gpu_backend, setup, 4, 84), terminal_ran=False)


@pytest.mark.parametrize("depth", [0, 1])
def test_degenerate_light_quad_is_not_found(host, gpu_backend, monkeypatch, depth):
    """A light quad with a zero edge is left out of the BVH (zero area); its quad test alone would still report hits
    along an infinite strip in front of the camera, so the light list must leave it out too.  Depth 0: the camera rays
    are the terminal bounce; depth 1: the rays off the floor."""
    lq = light((-0.5, 2.0, -0.5), (1.0, 0.0, 0.0), (0.0, 0.0, 1.0), (4.0, 4.0, 4.0))

    def setup(g):
        g.set_globals(64, 48, depth, bg=(0.1, 0.2, 0.3))
        g.set_camera(host.set_cam_params((0, 1, 4), (0, 0.5, 0), (0, 1, 0), 45, 64 / 48, 0.0, 1.0))
        g.add_quad(host.set_quad_params((-3, 0, -3), (6, 0, 0), (0, 0, 6)), S.MAT_LAMBERTIAN, S.LambertianParams(S.float3(0.6, 0.6, 0.6)))
        g.add_quad(host.set_quad_params((-0.5, 2.0, -0.5), (1.0, 0.0, 0.0), (0.0, 0.0, 1.0)), S.MAT_LIGHT, lq)
        bad = host.set_quad_params((-2.0, -1.0, 0.0), (4.0, 0.0, 0.0), (0.0, 4.0, 0.0))   # the plane z = 0, facing the camera
        bad.v1 = S.float3(0.0, 0.0, 0.0)
        g.add_quad(bad, S.MAT_LIGHT, light((-2.0, -1.0, 0.0), (4.0, 0.0, 0.0), (0.0, 4.0, 0.0), (9.0, 9.0, 9.0)))
        g.set_lights([lq])
        g.build_accel()
    assert_same(render_both(monkeypatch, gpu_backend, setup, 4, 85))
