"""The built acceleration structure itself, checked by the numpy validator in bvh_check.py after every build: primitive
boxes, binary nodes, packed records, wide nodes and their quantised planes, for every builder and for the shapes where
builders go wrong (no or only invalid primitives, the PLOC tail and tile edges, flat, offset and uneven geometry, the
greedy collapse above 4 M primitives, a refit, many primitives with the same box).  The parity tests compare hits,
which forgive a few wrong primitives; these compare the structure."""
import os

import numpy as np
import pytest

import bvh_check as B
from conftest import ROOT
from minimaloptix_b200 import structs as S

pytestmark = pytest.mark.gpu

# (id, accel flags, environment): every way the library builds a hierarchy
BUILDERS = [("default", S.ACCEL_DEFAULT, {}), ("binary", S.ACCEL_BINARY, {}), ("lbvh", S.ACCEL_LBVH, {}),
            ("watertight", S.ACCEL_WATERTIGHT, {}), ("greedy", S.ACCEL_DEFAULT, {"MOX_WIDE_GREEDY": "1"}),
            ("radius1", S.ACCEL_DEFAULT, {"MOX_PLOC_RADIUS": "1"}), ("radius200", S.ACCEL_DEFAULT, {"MOX_PLOC_RADIUS": "200"})]
BUILDER_IDS = [b[0] for b in BUILDERS]


@pytest.fixture(scope="module")
def mats(host):
    dn = host.init_disney_params()
    dg = host.init_disney_params()
    dg.brdfType = S.GLASS
    light = S.LightParams()
    light.emission = S.float3(4, 4, 4)
    return [(S.MAT_LAMBERTIAN, S.LambertianParams(S.float3(0.5, 0.5, 0.5))), (S.MAT_METAL, S.MetalParams(S.float3(0.6, 0.6, 0.6), 0.1)),
            (S.MAT_GLASS, S.GlassParams(S.float3(1, 1, 1), 1.5)), (S.MAT_DISNEY, dn), (S.MAT_DISNEY, dg), (S.MAT_LIGHT, light)]


@pytest.fixture
def build(gpu_backend, monkeypatch):
    """build(scene_fn, builder) -> (context, SceneData, validator summary): a fresh context, the scene added, built."""
    def run(scene_fn, builder=BUILDERS[0], ctx=None):
        _, flags, env = builder
        for k in ("MOX_WIDE_GREEDY", "MOX_PLOC_RADIUS"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        g = ctx or gpu_backend.context(0)
        g.set_globals(16, 16, 5)
        sd = B.SceneData(g)
        scene_fn(sd)
        g.build_accel(flags)
        return g, sd, B.check(g, sd, watertight=bool(flags & S.ACCEL_WATERTIGHT))
    return run


# ------------------------------------------------------------------------------------------------------- scenes
def soup(rng, n, lo=0.0, hi=1.0, size=None, sizes=None):
    """n random triangles with centres in [lo, hi]^3: (vertices (3n, 3), faces (n, 3))."""
    size = size if size is not None else 0.5 * (hi - lo) * max(n, 1) ** (-1 / 3)
    c = rng.uniform(lo, hi, size=(n, 1, 3))
    s = size if sizes is None else sizes[:, None, None]
    v = (c + rng.uniform(-1, 1, size=(n, 3, 3)) * s).astype(np.float32).reshape(-1, 3)
    return v, np.arange(3 * n, dtype=np.int32).reshape(-1, 3)


def add_soup(sd, mats, v, f, pieces=3):
    """The faces as `pieces` meshes with different materials."""
    for k, part in enumerate(np.array_split(np.arange(len(f)), pieces)):
        if len(part):
            idx = f[part]
            used = np.unique(idx)
            remap = np.searchsorted(used, idx).astype(np.int32)
            sd.add_mesh(v[used], remap, *mats[k % len(mats)])


def add_invalid(sd, host, mats, k):
    """One primitive the builder must leave out, exactly degenerate: a repeated vertex, a NaN / infinite radius, a zero v1."""
    kind, params = mats[k % len(mats)]
    if k % 4 == 0:
        sd.add_mesh(np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32), [[0, 1, 0]], kind, params)
    elif k % 4 == 1:
        sd.add_sphere(S.SphereParams(float("nan"), S.float3(0.5, 0.5, 0.5)), kind, params)
    elif k % 4 == 2:
        sd.add_sphere(S.SphereParams(float("inf"), S.float3(0.2, 0.5, 0.5)), kind, params)
    else:
        sd.add_quad(host.set_quad_params((0.1, 0.2, 0.3), (0, 0, 0), (0, 0, 0.5)), kind, params)


def mixed(host, mats, n_valid, seed, quads=True):
    """n_valid primitives of all three types (some spheres with negative radii) between invalid ones first, in the
    middle and last."""
    def fn(sd):
        rng = np.random.default_rng(seed)
        add_invalid(sd, host, mats, 0)
        add_invalid(sd, host, mats, 1)
        for i in range(n_valid):
            if i == n_valid // 2:
                for k in (2, 3, 0):
                    add_invalid(sd, host, mats, k)
            c = rng.uniform(-1, 1, 3)
            kind, params = mats[i % len(mats)]
            t = i % 3 if quads else i % 2
            if t == 0:
                v = (c + rng.uniform(-0.2, 0.2, (3, 3))).astype(np.float32)
                if i % 4 == 0:   # a mesh with a degenerate face among valid ones
                    sd.add_mesh(np.vstack([v, v[:1]]), [[0, 1, 3], [0, 1, 2]], kind, params)
                else:
                    sd.add_mesh(v, [[0, 1, 2]], kind, params)
            elif t == 1:
                r = float(rng.uniform(0.01, 0.3)) * (-1 if i % 5 == 1 else 1)
                sd.add_sphere(S.SphereParams(r, S.float3(*c)), kind, params)
            else:
                sd.add_quad(host.set_quad_params(tuple(c), tuple(rng.uniform(-0.3, 0.3, 3)), tuple(rng.uniform(-0.3, 0.3, 3))), kind, params)
        for k in (1, 3, 2):
            add_invalid(sd, host, mats, k)
    return fn


def replica(host_scene):
    """The meshes of a host scene (Disney materials, as its loader gives them), then its quad lights: the order in
    which the interior builder adds them."""
    def fn(sd):
        info = host_scene.info()
        for m in range(info.n_meshes):
            d = host_scene.mesh_info(m)["disney"]
            d.albedoID = 0
            v, f = host_scene.mesh_arrays(m)
            sd.add_mesh(v, f, S.MAT_DISNEY, d)
        for i in range(info.n_lights):
            lt = host_scene.light(i)
            if lt.shape == S.QUAD:
                sd.add_quad(_quad_of_light(lt), S.MAT_LIGHT, lt)
    return fn


def _quad_of_light(lt):
    from minimaloptix_b200 import host
    return host.set_quad_params(lt.position.tuple(), lt.u.tuple(), lt.v.tuple())


# ------------------------------------------------------------------------------------------------------- shapes
@pytest.mark.parametrize("builder", BUILDERS, ids=BUILDER_IDS)
def test_empty_and_invalid_only(build, host, mats, builder):
    _, _, got = build(lambda sd: None, builder)
    assert got["n_valid"] == 0 and got["n_nodes"] == 1

    def invalid(sd):
        for k in range(9):
            add_invalid(sd, host, mats, k)
    _, sd, got = build(invalid, builder)
    assert sd.n == 9 and got["n_valid"] == 0 and got["n_nodes"] == 1


@pytest.mark.parametrize("builder", BUILDERS, ids=BUILDER_IDS)
@pytest.mark.parametrize("n_valid", [1, 2, 3, 8, 9, 17, 33])
def test_small_mixed_scenes(build, host, mats, builder, n_valid):
    _, _, got = build(mixed(host, mats, n_valid, n_valid), builder)
    assert got["n_valid"] == n_valid


@pytest.mark.parametrize("builder", BUILDERS, ids=BUILDER_IDS)
@pytest.mark.parametrize("n_valid", [1024, 1025, 2049])
def test_ploc_tail_and_tile_edges(build, host, mats, builder, n_valid):
    _, _, got = build(mixed(host, mats, n_valid, n_valid, quads=False), builder)
    assert got["n_valid"] == n_valid
    if builder[0] == "default":
        assert got["n_nodes8"] > 0 and got["exact_wide_nodes"] == got["n_nodes8"]


SHAPES = {
    "flat": lambda rng: (lambda v, f: (np.column_stack([v[:, :2], np.full(len(v), 0.5, np.float32)]), f))(*soup(rng, 5000)),
    "offset": lambda rng: soup(rng, 5000, 1e5, 1e5 + 10.0),
    "straddle": lambda rng: soup(rng, 5000, -1.0, 1.0),
    "uneven": lambda rng: soup(rng, 5000, 0.0, 10.0, sizes=10.0 ** rng.uniform(-4, 1, 5000)),
}


@pytest.mark.parametrize("builder", BUILDERS, ids=BUILDER_IDS)
@pytest.mark.parametrize("shape", list(SHAPES))
def test_geometry_shapes(build, mats, builder, shape):
    v, f = SHAPES[shape](np.random.default_rng(len(shape)))
    _, _, got = build(lambda sd: add_soup(sd, mats, np.ascontiguousarray(v, np.float32), f), builder)
    assert got["n_valid"] > 0.99 * len(f)
    if builder[0] == "default":
        assert got["n_nodes8"] > 0 and got["exact_wide_nodes"] == got["n_nodes8"]


@pytest.mark.parametrize("builder", BUILDERS, ids=BUILDER_IDS)
def test_soup_200k(build, mats, builder):
    v, f = soup(np.random.default_rng(200), 200_000)
    _, _, got = build(lambda sd: add_soup(sd, mats, v, f, pieces=6), builder)
    assert got["n_valid"] == 200_000


@pytest.mark.parametrize("builder", BUILDERS[:4], ids=BUILDER_IDS[:4])
def test_interior_1m(build, host, builder):
    g, _, got = build(replica(host.Scene.builtin("interior", 1_000_000)), builder)
    print(f"\ninterior 1M {builder[0]}: binary depth {got['binary_depth']}, wide depth {got['wide_depth']}, "
          f"{got['n_nodes']} binary / {got['n_nodes8']} wide nodes")
    if builder[0] in ("default", "watertight"):
        assert g.stats()["node_bytes"] == 80   # PLOC + wide, not the radix-tree fallback


@pytest.mark.skipif(not os.path.exists(os.path.join(ROOT, "scenes", "coffee", "coffee.scene")), reason="scenes/coffee not fetched")
def test_coffee(build, host):
    _, _, got = build(replica(host.Scene.load(os.path.join(ROOT, "scenes", "coffee"), "coffee")))
    print(f"\ncoffee: binary depth {got['binary_depth']}, wide depth {got['wide_depth']}")


def test_greedy_collapse_above_4m(build, mats):
    """4 000 001 primitives: the collapse switches from the dynamic programme to the greedy one."""
    v, f = soup(np.random.default_rng(4), 4_000_001)
    g, _, got = build(lambda sd: add_soup(sd, mats, v, f, pieces=2))
    assert got["n_valid"] == 4_000_001 and g.stats()["node_bytes"] == 80
    print(f"\n4 M soup: binary depth {got['binary_depth']}, wide depth {got['wide_depth']}")


@pytest.mark.parametrize("builder", BUILDERS[:4], ids=BUILDER_IDS[:4])
def test_after_refit(build, host, builder):
    """A refit to a moved pose: the boxes must be those of the new pose (the movers of test_refit.py)."""
    from test_refit import ROOM_MESHES, moved
    sc = host.Scene.builtin("interior", 30000)
    g, sd, _ = build(replica(sc), builder)
    first = 0
    for m in range(sc.info().n_meshes):
        if m >= ROOM_MESHES:
            sd.update_mesh(first, moved(sc.mesh_arrays(m)[0], m - ROOM_MESHES, 1.0))
        first += sc.mesh_info(m)["faces"]
    g.build_accel(builder[1] | S.ACCEL_REFIT)
    B.check(g, sd, watertight=bool(builder[1] & S.ACCEL_WATERTIGHT))


# ------------------------------------------------------------------------------------------------------- the validator
def test_validator_rejects_corrupted_copies(build, mats):
    """Corrupt host copies of a real structure, one defect at a time: each must be rejected."""
    v, f = soup(np.random.default_rng(9), 3000)
    g, sd, _ = build(lambda sd: add_soup(sd, mats, v, f))
    arrays, stats = B.read_arrays(g), g.stats()
    B.check_arrays(arrays, stats, sd)

    def corrupt(name, fn):
        a = {k: x.copy() for k, x in arrays.items()}
        fn(a)
        with pytest.raises(B.BvhError) as e:
            B.check_arrays(a, stats, sd)
        print(f"\n{name}: {e.value}")

    def plane_inward(a):   # the first non-empty slot of node 3: its qlo.x one step up (or qhi.x one down)
        q = a["nodes8"].reshape(-1, 80)[3, 32:80].reshape(6, 8)
        s = int(np.flatnonzero(~((q[0] == 255) & (q[3] == 0)))[0])
        if q[0, s] < q[3, s]:
            q[0, s] += 1
        else:
            q[3, s] -= 1
    corrupt("plane byte inward", plane_inward)

    def duplicate_ref(a):  # a binary node with two inner children refers twice to the first
        ref = a["nodes"].view(np.int32).reshape(-1, 16)[:, 12:14]
        k = int(np.flatnonzero((ref[:, 0] >= 0) & (ref[:, 1] >= 0))[0])
        ref[k, 1] = ref[k, 0]
    corrupt("duplicated child ref", duplicate_ref)

    def drop_binary(a):    # a two-primitive binary leaf loses its second primitive
        ref = a["nodes"].view(np.int32).reshape(-1, 16)[:, 12:14]
        k = np.argwhere((ref < 0) & ((~ref & 7) == 1))[0]
        ref[k[0], k[1]] = ~(~ref[k[0], k[1]] & ~7)
    corrupt("dropped primitive (binary leaf)", drop_binary)

    def drop_wide(a):      # a two-primitive wide leaf slot loses its second primitive, in valid and group alike
        u = a["nodes8"].view(np.uint32).reshape(-1, 20)
        for w in range(len(u)):
            s = [s for s in range(8) if (u[w, 6] >> (2 * s)) & 3 == 3]
            if s:
                u[w, 6] &= ~np.uint32(2 << (2 * s[0]))
                u[w, 7] &= ~np.uint32(2 << (2 * s[0] + 8))
                return
        raise AssertionError("no two-primitive wide leaf")
    corrupt("dropped primitive (wide leaf)", drop_wide)

    def class_bit(a):      # the shade class of one packed record
        a["packed"].view(np.uint32).reshape(-1, 12)[len(f) // 2, 7] ^= np.uint32(1 << 2)
    corrupt("flipped class bit", class_bit)


# ------------------------------------------------------------------------------------------------------- coincident primitives
def _rays_at(rng, tri, n):
    """Rays from random origins towards random points of the triangle, plus incoherent ones."""
    o = rng.uniform(-1.5, 2.5, size=(n, 3))
    b = rng.dirichlet([1, 1, 1], size=n)
    d = b @ tri.astype(np.float64) - o
    d[n // 2:] = rng.normal(size=(n - n // 2, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays = np.empty((n, 8), np.float32)
    rays[:, 0:3], rays[:, 3], rays[:, 4:7], rays[:, 7] = o, 1e-3, d, 1e27
    return rays


@pytest.mark.parametrize("with_soup", [False, True], ids=["alone", "in-20k-soup"])
@pytest.mark.parametrize("n_same", [200, 1300, 5000])
def test_coincident_primitives(gpu_backend, orc, mats, n_same, with_soup):
    """Many triangles with the same box: PLOC merges one pair of them per iteration, so its tree gets too deep or it
    runs out of iterations; the build must fall through to the radix tree instead of failing, and find what brute
    force finds."""
    from test_gpu_parity import check_ids
    g, o = gpu_backend.context(0), orc.context(brute_force=True)
    for c in (g, o):
        c.set_globals(16, 16, 5)
    sd = B.SceneData(g, o)
    rng = np.random.default_rng(n_same)
    tri = np.array([[0.2, 0.3, 0.4], [0.8, 0.35, 0.5], [0.45, 0.9, 0.6]], np.float32)
    if with_soup:
        v, f = soup(rng, 10_000)
        add_soup(sd, mats, v, f, pieces=2)
    sd.add_mesh(np.tile(tri, (n_same, 1)), np.arange(3 * n_same, dtype=np.int32).reshape(-1, 3), *mats[3])
    if with_soup:
        v, f = soup(rng, 10_000)
        add_soup(sd, mats, v, f, pieces=2)
    g.build_accel()
    o.build_accel()
    got = B.check(g, sd)
    assert got["n_valid"] == sd.n
    if not with_soup:
        # the radix tree: 200 coincident triangles give a PLOC tree deeper than the traversal stack, 1300 and 5000 run
        # PLOC out of iterations
        assert g.stats()["node_bytes"] == 64
    nbad, nhit = check_ids(o, g, _rays_at(rng, tri, 20000), f"coincident-{n_same}")
    assert nhit > 5000
    assert nbad == 0
