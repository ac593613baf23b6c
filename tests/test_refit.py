"""Mesh vertex updates (mox_update_mesh) and the in-place BVH refit (MOX_ACCEL_REFIT).

Scene: the 30 k-triangle interior.  buildInterior adds the room's meshes first (six walls, the table top and its four
legs), then the blobs and tori, then the quad lights, so a mesh's first primitive id is the running sum of the face
counts before it.  The blobs and tori move: a rigid offset plus a small sinusoidal displacement, which leaves every
triangle non-degenerate."""
import numpy as np
import pytest

from conftest import random_rays
from minimaloptix_b200 import MoxError
from minimaloptix_b200 import structs as S

ERR_INVALID, ERR_STATE = -1, -4
ROOM_MESHES = 11
ARRAYS = ("nodes", "nodes8", "packed", "packed8")
FLAGS = [S.ACCEL_DEFAULT, S.ACCEL_BINARY, S.ACCEL_LBVH]
FLAG_IDS = ["wide", "binary-ploc", "binary-lbvh"]


def interior(host, n_tris=30000):
    """The scene and its movers: (first primitive id, vertices, normal count) of every blob and torus."""
    sc = host.Scene.builtin("interior", n_tris)
    first, movers = 0, []
    for m in range(sc.info().n_meshes):
        info = sc.mesh_info(m)
        if m >= ROOM_MESHES:
            movers.append((first, sc.mesh_arrays(m)[0], info["normals"]))
        first += info["faces"]
    return sc, movers


def moved(verts, k, t):
    off = np.array([0.06 * np.sin(1.3 * t + k), 0.02 * t, 0.06 * np.cos(0.7 * t + k)], np.float32)
    return (verts + off + 0.004 * np.sin(7.0 * verts[:, [1, 2, 0]] + t)).astype(np.float32)


def radial_normals(verts):
    d = verts - verts.mean(axis=0)
    return (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)


def set_pose(ctx, movers, t, with_normals=False):
    """Pose t > 0 moves every mover; t = 0 puts the original vertices back."""
    for k, (first, verts, n_normals) in enumerate(movers):
        v = verts if t == 0 else moved(verts, k, t)
        normals = radial_normals(v) if with_normals and n_normals == len(v) and k % 2 == 0 else None
        ctx.update_mesh(first, v, normals)


def build_rc(ctx, flags):
    return ctx.b.build_accel(ctx.h, flags, None)


def accel_arrays(ctx):
    return {k: ctx.debug_read_accel(k) for k in ARRAYS}


def assert_images_agree(a, b):
    """The rule between two hierarchies (test_wide_and_binary_traversal_render_identically)."""
    (ia, sa), (ib, sb) = a, b
    assert (sa["rays_primary"], sa["rays_bounce"], sa["rays_shadow"]) == (sb["rays_primary"], sb["rays_bounce"], sb["rays_shadow"])
    assert np.allclose(ia, ib, rtol=0, atol=1e-5)
    assert np.mean(ia == ib) > 0.999


def render(ctx, spp=3, seed=9):
    ctx.render(spp, seed)
    return ctx.read_accum(), ctx.stats()


# ---------------------------------------------------------------------------------------------- oracle (no GPU)
def test_oracle_refit_renders_like_a_build_at_the_new_pose(host, api_tables, orc):
    sc, movers = interior(host)
    imgs = []
    for refit in (True, False):
        o = orc.context()
        sc.upload(api_tables.oracle, o, 48, 27, 4)
        if refit:
            o.build_accel()
            set_pose(o, movers, 1.0, with_normals=True)
            with pytest.raises(MoxError):
                o.launch(1)   # stale until the refit
            o.build_accel(S.ACCEL_REFIT)
        else:
            set_pose(o, movers, 1.0, with_normals=True)
            o.build_accel()
        imgs.append(render(o, 2, 7))
    assert np.array_equal(imgs[0][0].view(np.uint32), imgs[1][0].view(np.uint32))
    assert imgs[0][1]["rays_bounce"] == imgs[1][1]["rays_bounce"] and imgs[0][1]["rays_shadow"] == imgs[1][1]["rays_shadow"]
    # the moved scene renders differently from the static one
    s = orc.context()
    sc.upload(api_tables.oracle, s, 48, 27, 4)
    s.build_accel()
    assert not np.array_equal(render(s, 2, 7)[0], imgs[0][0])


def test_oracle_refit_and_update_errors(host, api_tables, orc):
    sc, movers = interior(host)
    o = orc.context()
    sc.upload(api_tables.oracle, o, 32, 32, 3)
    assert build_rc(o, S.ACCEL_REFIT) == ERR_STATE            # no build yet
    o.build_accel(S.ACCEL_WATERTIGHT)
    assert build_rc(o, S.ACCEL_REFIT) == ERR_INVALID          # flags differ from the build's
    assert build_rc(o, S.ACCEL_REFIT | S.ACCEL_WATERTIGHT) == 0
    first, verts, n_normals = movers[0]
    with pytest.raises(MoxError):
        o.update_mesh(first, verts[:-1])                      # vertex count
    with pytest.raises(MoxError):
        o.update_mesh(first, verts, np.zeros((n_normals + 1, 3), np.float32))   # normal count
    with pytest.raises(MoxError):
        o.update_mesh(first + 1, verts)                       # not the first primitive of a mesh
    with pytest.raises(MoxError):
        o.update_mesh(0, np.zeros((sc.mesh_info(0)["vertices"], 3), np.float32), np.zeros((sc.mesh_info(0)["vertices"], 3), np.float32))
        # the floor was added without normals
    o.add_sphere(S.SphereParams(0.1, S.float3(5, 2, 4)), S.MAT_LAMBERTIAN, S.LambertianParams(S.float3(1, 1, 1)))
    assert build_rc(o, S.ACCEL_REFIT | S.ACCEL_WATERTIGHT) == ERR_STATE   # primitives added since the build
    o.build_accel(S.ACCEL_WATERTIGHT)
    assert build_rc(o, S.ACCEL_REFIT | S.ACCEL_WATERTIGHT) == 0


# ---------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("watertight", [0, S.ACCEL_WATERTIGHT], ids=["sdk", "watertight"])
@pytest.mark.parametrize("flags", FLAGS, ids=FLAG_IDS)
def test_refit_round_trip_is_byte_identical(host, api_tables, gpu_backend, flags, watertight):
    sc, movers = interior(host)
    g = gpu_backend.context(0)
    sc.upload(api_tables.gpu, g, 64, 64, 5)
    f = flags | watertight
    g.build_accel(f)
    want = accel_arrays(g)
    assert want["packed"].size > 0 and (want["nodes8"].size > 0) == (flags == S.ACCEL_DEFAULT)
    g.build_accel(f | S.ACCEL_REFIT)                          # nothing moved
    got = accel_arrays(g)
    for k in ARRAYS:
        assert np.array_equal(got[k], want[k]), k
    set_pose(g, movers, 1.0)
    g.build_accel(f | S.ACCEL_REFIT)
    assert not np.array_equal(g.debug_read_accel("nodes"), want["nodes"])
    set_pose(g, movers, 0)
    g.build_accel(f | S.ACCEL_REFIT)
    got = accel_arrays(g)
    for k in ARRAYS:
        assert np.array_equal(got[k], want[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("flags", FLAGS, ids=FLAG_IDS)
def test_hits_after_refit_match_the_oracle(host, api_tables, orc, gpu_backend, flags):
    from test_gpu_parity import check_ids
    sc, movers = interior(host)
    g = gpu_backend.context(0)
    sc.upload(api_tables.gpu, g, 64, 64, 5)
    g.build_accel(flags)
    set_pose(g, movers, 1.0)
    g.build_accel(flags | S.ACCEL_REFIT)
    o = orc.context()
    sc.upload(api_tables.oracle, o, 64, 64, 5)
    set_pose(o, movers, 1.0)
    o.build_accel()
    rays = random_rays(400000, [0.05, 0.05, 0.05], [9.95, 3.95, 7.95], 4)
    nbad, nhit = check_ids(o, g, rays, "interior-refit")
    assert nhit == len(rays)
    assert nbad <= 8
    rays = random_rays(100000, [0.05, 0.05, 0.05], [9.95, 3.95, 7.95], 8, tmax=3.0)
    ao, ag = o.trace_shadow(rays), g.trace_shadow(rays)
    assert (ao == 0).all(axis=1).any() and (ao == 1).all(axis=1).any()
    assert np.any(ao != ag, axis=1).sum() <= 5


@pytest.mark.gpu
@pytest.mark.parametrize("flags", FLAGS, ids=FLAG_IDS)
def test_render_after_refit_equals_a_full_build(host, api_tables, gpu_backend, flags):
    sc, movers = interior(host)
    imgs = []
    for refit in (True, False):
        g = gpu_backend.context(0)
        sc.upload(api_tables.gpu, g, 160, 90, 5)
        if refit:
            g.build_accel(flags)
            set_pose(g, movers, 1.0, with_normals=True)
            g.build_accel(flags | S.ACCEL_REFIT)
        else:
            set_pose(g, movers, 1.0, with_normals=True)
            g.build_accel(flags)
        imgs.append(render(g))
    assert_images_agree(imgs[0], imgs[1])


@pytest.mark.gpu
def test_refit_of_animated_spheres_equals_a_full_build(host, api_tables, gpu_backend):
    sc = host.Scene.builtin("random_spheres")
    g = gpu_backend.context(0)
    sc.upload(api_tables.gpu, g, 160, 90, 5)
    g.build_accel()
    for _ in range(5):
        sc.animate(0.002)
    sc.apply_spheres(api_tables.gpu, g)
    g.build_accel(S.ACCEL_REFIT)
    fresh = gpu_backend.context(0)
    sc.upload(api_tables.gpu, fresh, 160, 90, 5)
    sc.apply_spheres(api_tables.gpu, fresh)
    fresh.build_accel()
    assert_images_agree(render(g, 4, 5), render(fresh, 4, 5))


@pytest.mark.gpu
def test_validity_change_and_staleness(host, api_tables, gpu_backend):
    sc, movers = interior(host)
    g = gpu_backend.context(0)
    sc.upload(api_tables.gpu, g, 32, 32, 3)
    g.build_accel()
    n_packed = g.debug_read_accel("packed").size
    g.launch(1)
    first, verts, _ = movers[0]
    set_pose(g, movers, 1.0)
    with pytest.raises(MoxError):
        g.launch(2)                       # stale after update_mesh
    g.build_accel(S.ACCEL_REFIT)
    g.launch(2)
    # collapse face 0 of the first mover to a point: it (and the faces sharing two of its vertices) leave the BVH
    idx = sc.mesh_arrays(ROOM_MESHES)[1]
    v = verts.copy()
    v[idx[0, 1]] = v[idx[0, 2]] = v[idx[0, 0]]
    g.update_mesh(first, v)
    assert build_rc(g, S.ACCEL_REFIT) == ERR_STATE
    assert "ACCEL_REFIT" in g.b.last_error(g.h).decode()
    with pytest.raises(MoxError):
        g.launch(3)
    assert build_rc(g, S.ACCEL_REFIT) == ERR_STATE        # a failed refit leaves no structure to refit
    g.build_accel()
    assert g.debug_read_accel("packed").size < n_packed
    g.launch(3)


@pytest.mark.gpu
def test_refit_on_a_multi_gpu_handle_equals_a_plain_context(host, api_tables, gpu_backend):
    sc, movers = interior(host)
    imgs = []
    for ctx in (gpu_backend.context(0), gpu_backend.multi_context([0])):
        sc.upload(api_tables.gpu, ctx, 200, 120, 5)
        ctx.build_accel()
        set_pose(ctx, movers, 1.0)
        ctx.build_accel(S.ACCEL_REFIT)
        imgs.append(render(ctx, 3, 17))
    assert np.array_equal(imgs[0][0].view(np.uint32), imgs[1][0].view(np.uint32))
    assert (imgs[0][1]["rays_bounce"], imgs[0][1]["rays_shadow"]) == (imgs[1][1]["rays_bounce"], imgs[1][1]["rays_shadow"])
