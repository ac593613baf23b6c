"""Traversal against brute force on the rays where slab arithmetic goes wrong: direction components of exactly +0 or
-0, below the 1e-30 threshold or just above it, origins on primitive-box planes, rays along walls, rays aimed exactly
at vertices and edge midpoints, far origins, non-unit directions, and tmin / tmax cut exactly at a hit.  The random
rays of the parity tests almost never have any of these.

The criterion is bit for bit, with no graze or tie excuse.  Closest hit: t, id, beta and gamma equal brute force's.  A
ray may differ only where, in float64, the brute-force winner's hit point lies outside that primitive's own box by
more than the slab tests' slack (1e-5 of t), and then only towards a miss: the traversal's (t, id) is never
lexicographically smaller than brute force's, because a traversal can lose a hit but never invent one.  Any hit:
transmittance equals brute force's on every ray (the glass tints are powers of two, so their product does not depend
on the order of the hits).

The GPU half runs every traversal kernel through the public flags; the CPU half runs the oracle's own BVH (brute force
off) through the same generators and criterion.  Each test prints one line per ray family: rays, hits, exceptions."""
import os

import numpy as np
import pytest

import bvh_check as B
from conftest import ROOT
from minimaloptix_b200 import structs as S

F32, F64, U32 = np.float32, np.float64, np.uint32
TINY = 1e-30        # a direction component of at most this magnitude counts as zero (traverse.cuh::prepRay, oracle.cpp::slab)
SLACK = 1e-5        # relative slack of the slab tests in t
INF32 = F32(np.inf)


# ------------------------------------------------------------------------------------------------------------ scenes
def _materials(host):
    """Disney NORMAL (blocks shadow rays) and three Disney GLASS materials whose tints are powers of two."""
    normal = host.init_disney_params()
    mats = [(S.MAT_DISNEY, normal)]
    for tint in ((0.5, 0.25, 0.125), (0.25, 1.0, 0.5), (1.0, 0.125, 0.5)):
        g = host.init_disney_params()
        g.brdfType, g.color = S.GLASS, S.float3(*tint)
        mats.append((S.MAT_DISNEY, g))
    return mats


def _add_triangles(sd, mats, tri):
    """(n, 3, 3) triangles as four meshes, half of them glass."""
    order = (0, 1, 0, 2)
    for k, part in enumerate(np.array_split(np.arange(len(tri)), 4)):
        if len(part):
            sd.add_mesh(tri[part].reshape(-1, 3), np.arange(3 * len(part), dtype=np.int32).reshape(-1, 3), *mats[order[k]])


def lattice_triangles(n, seed, flat=False):
    """n triangles with vertices on the 0.5 lattice of [0, 8.5]^3; a third of them perpendicular to an axis, many
    sharing edges and vertices.  flat: every vertex in the plane z = 2."""
    rng = np.random.default_rng(seed)
    v = rng.integers(0, 15, size=(n, 1, 3)) + rng.integers(-2, 3, size=(n, 3, 3))
    for i in np.flatnonzero(rng.random(n) < 0.35):
        a = rng.integers(0, 3)
        v[i, :, a] = v[i, 0, a]
    v = np.clip(v, 0, 17).astype(F64) * 0.5
    if flat:
        v[:, :, 2] = 2.0
    c = np.cross(v[:, 1] - v[:, 0], v[:, 2] - v[:, 0])
    return v[np.any(c != 0, axis=1)].astype(F32)


def lattice(n=1300, seed=1, offset=0.0, scale=1.0):
    def fn(sd, host, mats):
        tri = lattice_triangles(n, seed)
        _add_triangles(sd, mats, (tri.astype(F64) * scale + offset).astype(F32))
    return fn


def flat(sd, host, mats):
    _add_triangles(sd, mats, lattice_triangles(1500, 2, flat=True))


def cornell(sd, host, mats):
    """scenes/cornell: axis-aligned walls and blocks, and its quad light."""
    sc = host.Scene.load(os.path.join(ROOT, "scenes", "cornell"), "cornell")
    info = sc.info()
    for m in range(info.n_meshes):
        v, f = sc.mesh_arrays(m)
        sd.add_mesh(v, f, *mats[m % 2])
    for i in range(info.n_lights):
        lt = sc.light(i)
        if lt.shape == S.QUAD:
            sd.add_quad(host.set_quad_params(lt.position.tuple(), lt.u.tuple(), lt.v.tuple()), S.MAT_LIGHT, lt)


def room(sd, host, mats):
    """A 4 x 4 x 4 box room of axis-aligned quads, two shelves against its walls and spheres touching one, two or
    three walls."""
    q = host.set_quad_params
    walls = [((0, 0, 0), (4, 0, 0), (0, 0, 4)), ((0, 4, 0), (4, 0, 0), (0, 0, 4)), ((0, 0, 0), (0, 4, 0), (0, 0, 4)),
             ((4, 0, 0), (0, 4, 0), (0, 0, 4)), ((0, 0, 0), (4, 0, 0), (0, 4, 0)), ((0, 0, 4), (4, 0, 0), (0, 4, 0)),
             ((0, 2, 0), (2, 0, 0), (0, 0, 4)), ((2, 1, 4), (2, 0, 0), (0, 0, -1.5))]
    for k, w in enumerate(walls):
        sd.add_quad(q(*w), *mats[k % 4])
    for k, (c, r) in enumerate((((0.5, 1.0, 1.5), 0.5), ((3.5, 0.5, 3.0), 0.5), ((2.0, 3.25, 2.0), 0.75),
                                ((0.5, 0.5, 0.5), 0.5), ((2.0, 2.5, 0.25), 0.25), ((1.0, 2.5, 3.0), 0.5))):
        sd.add_sphere(S.SphereParams(r, S.float3(*c), S.float3()), *mats[(k + 1) % 4])


# name -> (scene, rays per family, spheres in it)
SCENES = {"lattice": (lattice(), 6000, False), "cornell": (cornell, 6000, False), "room": (room, 6000, True),
          "flat": (flat, 5000, False)}
for _off in (0.0, 1e3, 1e5):
    for _sc in (1e-3, 1.0, 1e4):
        if (_off, _sc) != (0.0, 1.0):
            SCENES[f"lattice-{_off:g}+{_sc:g}x"] = (lattice(600, 3, _off, _sc), 1500, False)


# ------------------------------------------------------------------------------------------------------ ray families
class Geometry:
    """What the generators aim at and the criterion measures: primitive boxes, box planes, vertices and edge midpoints
    of the valid primitives."""

    def __init__(self, sd):
        valid, lo, hi, slack = B.prim_bounds(sd)
        b = B._Boxes.of_prims(lo, hi, slack)
        # the criterion uses the smallest box the builder can have made (a quad's is known to one ulp), the
        # generators the planes of the computed one
        self.lo, self.hi = b.lo_up.astype(F64), b.hi_dn.astype(F64)
        self.plo, self.phi = lo.astype(F64), hi.astype(F64)
        a = sd.arrays()
        self.word = a["word"]
        v = self.lo[valid], self.hi[valid]
        self.blo, self.bhi = v[0].min(axis=0), v[1].max(axis=0)
        self.size = float((self.bhi - self.blo).max())
        self.planes = [np.unique(np.concatenate([lo[valid, k], hi[valid, k]])) for k in range(3)]
        self.valid = np.flatnonzero(valid)
        pts, mids = [], []
        tri = a["tri"][valid & (a["type"] == B.PT_TRI)]
        if len(tri):
            pts.append(tri.reshape(-1, 3))
            mids.append(((tri + np.roll(tri, 1, axis=1)) * F32(0.5)).reshape(-1, 3))
        quad = a["quad"][valid & (a["type"] == B.PT_QUAD)]
        if len(quad):
            v1, v2, an = quad[:, 0:3], quad[:, 3:6], quad[:, 6:9]
            tv1 = v1 * (F32(1) / (v1 * v1).sum(axis=1))[:, None]
            tv2 = v2 * (F32(1) / (v2 * v2).sum(axis=1))[:, None]
            c = np.stack([an, an + tv1, an + tv1 + tv2, an + tv2], axis=1)
            pts.append(c.reshape(-1, 3))
            mids.append(((c + np.roll(c, 1, axis=1)) * F32(0.5)).reshape(-1, 3))
        sph = a["sph"][valid & (a["type"] == B.PT_SPHERE)]
        for k in range(3):   # the points where a sphere touches its box
            for s in (-1, 1):
                p = sph[:, :3].copy()
                p[:, k] += s * sph[:, 3]
                pts.append(p)
        self.points = np.concatenate(pts).astype(F32)
        self.mids = np.concatenate(mids).astype(F32) if mids else self.points
        self.tmin = F32(1e-4 * self.size)

    def origins(self, rng, n, on_plane=0.7):
        """Origins in the scene box grown by a tenth; each coordinate on a primitive-box plane with probability on_plane."""
        o = rng.uniform(self.blo - 0.1 * self.size, self.bhi + 0.1 * self.size, size=(n, 3))
        for k in range(3):
            m = rng.random(n) < on_plane
            o[m, k] = rng.choice(self.planes[k], size=int(m.sum()))
        return o.astype(F32)


def _unit(d):
    """Float32 unit directions, renormalised the way random_rays does (exact zeros keep their sign)."""
    d = d.astype(F32)
    inv = (F32(1.0) / np.sqrt((d * d).sum(axis=1, dtype=F32))).astype(F32)
    return (d * inv[:, None]).astype(F32)


def _rays(o, d, tmin, tmax=1e27):
    r = np.empty((len(o), 8), F32)
    r[:, 0:3], r[:, 3], r[:, 4:7], r[:, 7] = o, tmin, d, tmax
    return r


def _zero_some(rng, d, value):
    """Set one or two components of each direction to +-value (value 0: exactly +0 or -0)."""
    d = d.copy()
    n = len(d)
    first = rng.integers(0, 3, n)
    second = np.where(rng.random(n) < 0.5, (first + rng.integers(1, 3, n)) % 3, first)
    for axis in (first, second):
        sign = np.where(rng.random(n) < 0.5, F32(-1), F32(1))
        mag = value if np.isscalar(value) else rng.choice(value, size=n)
        d[np.arange(n), axis] = np.copysign(np.asarray(mag, F32), sign)
    return d


def fam_zero(g, rng, n):
    """One or two direction components exactly +0 or -0; origins on primitive-box planes."""
    return _rays(g.origins(rng, n), _unit(_zero_some(rng, rng.normal(size=(n, 3)).astype(F32), 0.0)), g.tmin)


def fam_wall(g, rng, n):
    """Rays in the plane of a face of a primitive's box, running along it (that component +0 or -0)."""
    p = rng.choice(g.valid, size=n)
    axis = rng.integers(0, 3, n)
    lo, hi = g.plo[p], g.phi[p]
    ext = np.maximum(hi - lo, 1e-3 * g.size)
    o = rng.uniform(lo - ext, hi + ext)
    face = np.where((rng.random(n) < 0.5)[:, None], lo, hi)
    o[np.arange(n), axis] = face[np.arange(n), axis]
    d = rng.normal(size=(n, 3))
    d[np.arange(n), axis] = np.where(rng.random(n) < 0.5, -0.0, 0.0)
    return _rays(o.astype(F32), _unit(d), g.tmin)


def fam_vertex(g, rng, n):
    """Rays aimed exactly at vertices and at edge midpoints, from origins that are often on box planes."""
    o = g.origins(rng, n, on_plane=0.5)
    target = np.where((rng.random(n) < 0.5)[:, None], g.points[rng.integers(0, len(g.points), n)],
                      g.mids[rng.integers(0, len(g.mids), n)])
    d = (target - o).astype(F32)
    z = ~np.any(d != 0, axis=1)
    d[z] = rng.normal(size=(int(z.sum()), 3))
    return _rays(o, _unit(d), g.tmin)


def fam_tiny(g, rng, n):
    """One or two components of +-1e-35 or +-1e-31: below the 1e-30 clamp, not zero."""
    return _rays(g.origins(rng, n), _zero_some(rng, _unit(rng.normal(size=(n, 3))), np.array([1e-35, 1e-31], F32)), g.tmin)


def fam_small(g, rng, n):
    """One or two components of +-1e-29, 1e-25 or 1e-20: just above the 1e-30 threshold, where 1/d is finite and huge."""
    return _rays(g.origins(rng, n), _zero_some(rng, _unit(rng.normal(size=(n, 3))), np.array([1e-29, 1e-25, 1e-20], F32)),
                 g.tmin)


def fam_far(g, rng, n):
    """Origins 1e4 to 1e6 scene sizes away, aimed at points of the scene (triangles and quads only)."""
    u = _unit(rng.normal(size=(n, 3))).astype(F64)
    c = 0.5 * (g.blo + g.bhi)
    o = (c + u * g.size * 10.0 ** rng.uniform(4, 6, size=(n, 1))).astype(F32)
    target = np.where((rng.random(n) < 0.5)[:, None], g.points[rng.integers(0, len(g.points), n)],
                      rng.uniform(g.blo, g.bhi, size=(n, 3)).astype(F32))
    return _rays(o, _unit(target - o), g.tmin)


def fam_nonunit(g, rng, n):
    """Zero-component and vertex rays with directions of length 1e-3 and 1e3 (triangles and quads only)."""
    r = np.concatenate([fam_zero(g, rng, n - n // 2), fam_vertex(g, rng, n // 2)])
    s = np.where(rng.random(n) < 0.5, F32(1e-3), F32(1e3))
    r[:, 4:7] *= s[:, None]
    r[:, 3] /= s
    return r


FAMILIES = {"zero": fam_zero, "wall": fam_wall, "vertex": fam_vertex, "tiny": fam_tiny, "small": fam_small, "far": fam_far,
            "nonunit": fam_nonunit}
CUTS = ("cut-tmax", "cut-tmax-next", "cut-tmin")


# ------------------------------------------------------------------------------------------------------ references
class Case:
    """A scene added to a brute-force oracle context, its rays by family and brute force's answers."""

    def __init__(self, host, orc, name, watertight):
        fn, n, spheres = SCENES[name]
        self.name, self.watertight, self.flags = name, watertight, S.ACCEL_WATERTIGHT if watertight else 0
        self.mats = _materials(host)
        ob = orc.context(brute_force=True)
        ob.set_globals(16, 16, 5)
        self.sd = B.SceneData(ob)
        fn(self.sd, host, self.mats)
        ob.build_accel(self.flags)
        self.ob = ob
        g = self.geometry = Geometry(self.sd)
        rng = np.random.default_rng(sum(map(ord, name)))
        # the sphere test assumes unit directions, and from 1e4 scene sizes away its c = |o - center|^2 - r^2 has an
        # error far above r^2 (it reports hits metres off the sphere): both families are for triangles and quads
        self.rays = {k: f(g, rng, n) for k, f in FAMILIES.items() if not (spheres and k in ("nonunit", "far"))}
        # cuts at the first brute-force hit of zero-component and vertex rays
        base = np.concatenate([self.rays["zero"], self.rays["vertex"]])
        t, i, _, _ = ob.trace_closest(base)
        hit = i >= 0
        base, t, i = base[hit], t[hit], i[hit]
        self.cut_of = {}
        for k in CUTS:
            r = base.copy()
            if k == "cut-tmin":
                r[:, 3] = t
            else:
                r[:, 7] = t if k == "cut-tmax" else np.nextafter(t, INF32)
            self.rays[k] = r
            self.cut_of[k] = (t, i)
        self.all = np.concatenate(list(self.rays.values()))
        self.split = np.cumsum([len(r) for r in self.rays.values()])[:-1]
        self.closest = ob.trace_closest(self.all)
        self.shadow = ob.trace_shadow(self.all)
        self._check_cuts()

    def _check_cuts(self):
        """Brute force itself honours the open interval (tmin, tmax)."""
        for k, (tr, ir, _, _) in self.by_family(self.closest).items():
            if k not in CUTS:
                continue
            t0, i0 = self.cut_of[k]
            if k == "cut-tmax":
                assert np.all((tr < t0) | (ir < 0)), k
            elif k == "cut-tmax-next":
                assert np.array_equal(ir, i0) and np.array_equal(tr.view(U32), t0.view(U32)), k
            else:
                assert np.all((tr > t0) | (ir < 0)), k
        # a blocker's own t as tmax lets the ray pass it; one ulp more and it is blocked
        sh = self.by_family(self.shadow)
        blocks = (self.geometry.word[self.cut_of["cut-tmax-next"][1]] & 3) == 1
        assert np.all(sh["cut-tmax-next"][blocks] == 0)

    def hits_along(self, rays):
        """Brute force's hits (t, id) along each ray in (tmin, tmax), by repeated closest hits (of hits at one t, only
        the lowest id)."""
        out = [[] for _ in rays]
        r, live = rays.copy(), np.arange(len(rays))
        while len(live):
            t, i, _, _ = self.ob.trace_closest(r[live])
            h = i >= 0
            for k, tk, ik in zip(live[h], t[h], i[h]):
                out[k].append((tk, ik))
            live = live[h]
            r[live, 3] = t[h]
        return out

    def by_family(self, arrays):
        """Split the per-ray results (a tuple of arrays or one array) by family."""
        if isinstance(arrays, tuple):
            parts = [np.split(a, self.split) for a in arrays]
            return {k: tuple(p[j] for p in parts) for j, k in enumerate(self.rays)}
        return dict(zip(self.rays, np.split(arrays, self.split)))


_CASES = {}


def get_case(host, orc, name, watertight):
    if (name, watertight) not in _CASES:
        _CASES[name, watertight] = Case(host, orc, name, watertight)
    return _CASES[name, watertight]


def outside_own_box(g, rays, t, ids):
    """Rays whose hit point at t lies outside primitive ids' box by more than the slab slack, computed in float64 with
    the zero-component rule: such a component keeps the ray in the slab for every t when lo <= o <= hi."""
    o, d = rays[:, 0:3].astype(F64), rays[:, 4:7].astype(F64)
    lo, hi = g.lo[ids], g.hi[ids]
    zero = np.abs(d) <= TINY
    inside = (lo <= o) & (o <= hi)
    with np.errstate(divide="ignore", invalid="ignore"):
        dd = np.where(zero, 1.0, d)
        t0, t1 = (lo - o) / dd, (hi - o) / dd
    tn = np.where(zero, np.where(inside, -np.inf, np.inf), np.minimum(t0, t1)).max(axis=1)
    tf = np.where(zero, np.where(inside, np.inf, -np.inf), np.maximum(t0, t1)).min(axis=1)
    t = t.astype(F64)
    return (t < tn - SLACK * np.abs(t)) | (t > tf + SLACK * np.abs(t))


def compare_closest(g, rays, ref, got):
    """(number of excused rays, indices of wrong rays) of one family."""
    tr, ir, br, gr = ref
    tg, ig, bg, gg = got
    diff = (ir != ig) | (tr.view(U32) != tg.view(U32)) | (br.view(U32) != bg.view(U32)) | (gr.view(U32) != gg.view(U32))
    k = np.flatnonzero(diff)
    excused = np.zeros(len(k), bool)
    h = ir[k] >= 0
    excused[h] = outside_own_box(g, rays[k[h]], tr[k[h]], ir[k[h]])
    big = np.iinfo(np.int64).max
    idr, idg = np.where(ir[k] < 0, big, ir[k].astype(np.int64)), np.where(ig[k] < 0, big, ig[k].astype(np.int64))
    not_smaller = (tg[k] > tr[k]) | ((tg[k] == tr[k]) & (idg >= idr))
    ok = excused & not_smaller
    return int(ok.sum()), k[~ok]


def compare_shadow(case, rays, ref, got):
    """(number of excused rays, indices of wrong rays) of one family: a transmittance may differ only where one of
    brute force's occluding hits lies outside its primitive's box by more than the slack, and then only upwards
    (fewer occluders: every factor is at most 1)."""
    k = np.flatnonzero(np.any(ref.view(U32) != got.view(U32), axis=1))
    if not len(k):
        return 0, k
    g = case.geometry
    # A component just above the threshold has a finite, huge 1/d: a ray that starts on a face of a box and points out
    # of it by such a component leaves the box at t = 0, so any of its hits may be lost.  The list of brute force's hits
    # below shows only the lowest id of hits at one t, so for these rays only the direction of the change is checked.
    dk = np.abs(rays[k, 4:7])
    excused = np.any((dk > TINY) & (dk < 1e-15), axis=1)
    for j, hl in enumerate(case.hits_along(rays[k])):
        if excused[j]:
            continue
        hl = [(t, i) for t, i in hl if g.word[i] & 3]          # shadow class: only Disney primitives occlude
        if hl:
            t, i = np.array([h[0] for h in hl], F32), np.array([h[1] for h in hl])
            excused[j] = outside_own_box(g, np.repeat(rays[k[j]][None], len(hl), axis=0), t, i).any()
    ok = excused & np.all(got[k] >= ref[k], axis=1)
    return int(ok.sum()), k[~ok]


def check_against_brute(case, variant, closest, shadow):
    """Compare one traversal's answers on every family with brute force's; print a line per family and query."""
    g = case.geometry
    wrong = []
    ref_c, got_c = case.by_family(case.closest), case.by_family(closest)
    ref_s, got_s = case.by_family(case.shadow), case.by_family(shadow)
    for fam, rays in case.rays.items():
        n_exc, bad = compare_closest(g, rays, ref_c[fam], got_c[fam])
        print(f"{case.name:24s} {fam:14s} {variant:22s} closest rays {len(rays):6d} hits {int((ref_c[fam][1] >= 0).sum()):6d} "
              f"exceptions {n_exc:5d} wrong {len(bad)}")
        if len(bad):
            k = bad[0]
            wrong.append(f"{fam} closest: {len(bad)} rays, first {rays[k].tolist()}: brute force (t, id) "
                         f"({ref_c[fam][0][k]!r}, {ref_c[fam][1][k]}), {variant} ({got_c[fam][0][k]!r}, {got_c[fam][1][k]})")
        n_exc, bad = compare_shadow(case, rays, ref_s[fam], got_s[fam])
        print(f"{case.name:24s} {fam:14s} {variant:22s} shadow  rays {len(rays):6d} hits {int(np.any(ref_s[fam] != 1, axis=1).sum()):6d} "
              f"exceptions {n_exc:5d} wrong {len(bad)}")
        if len(bad):
            k = bad[0]
            wrong.append(f"{fam} shadow: {len(bad)} rays, first {rays[k].tolist()}: brute force {ref_s[fam][k].tolist()}, "
                         f"{variant} {got_s[fam][k].tolist()}")
    assert not wrong, f"{case.name}, {variant}:\n" + "\n".join(wrong)


# ------------------------------------------------------------------------------------------------------------ CPU half
@pytest.mark.parametrize("watertight", [False, True], ids=["sdk", "watertight"])
@pytest.mark.parametrize("scene", list(SCENES))
def test_oracle_bvh_matches_brute_force(host, orc, scene, watertight):
    case = get_case(host, orc, scene, watertight)
    o = orc.context()
    o.set_globals(16, 16, 5)
    SCENES[scene][0](B.SceneData(o), host, case.mats)
    o.build_accel(case.flags)
    check_against_brute(case, "oracle-bvh" + ("-watertight" if watertight else ""), o.trace_closest(case.all), o.trace_shadow(case.all))


# ------------------------------------------------------------------------------------------------------------ GPU half
VARIANTS = [("wide", S.ACCEL_DEFAULT), ("wide-counters", S.ACCEL_COUNTERS), ("binary", S.ACCEL_BINARY),
            ("lbvh", S.ACCEL_LBVH), ("wide-watertight", S.ACCEL_WATERTIGHT),
            ("binary-watertight", S.ACCEL_WATERTIGHT | S.ACCEL_BINARY)]


def gpu_context(gpu_backend, host, case, flags):
    g = gpu_backend.context(0)
    g.set_globals(16, 16, 5)
    SCENES[case.name][0](B.SceneData(g), host, case.mats)
    g.build_accel(flags)
    return g


@pytest.mark.gpu
@pytest.mark.parametrize("variant", VARIANTS, ids=[v[0] for v in VARIANTS])
@pytest.mark.parametrize("scene", list(SCENES))
def test_traversal_matches_brute_force(host, orc, gpu_backend, scene, variant):
    name, flags = variant
    case = get_case(host, orc, scene, bool(flags & S.ACCEL_WATERTIGHT))
    g = gpu_context(gpu_backend, host, case, flags)
    check_against_brute(case, name, g.trace_closest(case.all), g.trace_shadow(case.all))
    if flags & S.ACCEL_COUNTERS:
        assert g.stats()["node_visits"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [S.ACCEL_COUNTERS, S.ACCEL_COUNTERS | S.ACCEL_BINARY], ids=["wide", "binary"])
def test_zero_components_keep_culling(host, orc, gpu_backend, flags):
    """A zero direction component must not switch the slab test of its axis off (which would still give the right
    hits): rays with exact zeros visit about as many nodes, and test about as many primitives, as the same rays with
    those components at +-1e-20, where 1/d is finite and every plane culls."""
    case = get_case(host, orc, "lattice", False)
    g = gpu_context(gpu_backend, host, case, flags)
    zero = np.concatenate([case.rays["zero"], case.rays["wall"]])
    small = zero.copy()
    d = small[:, 4:7]
    d[d == 0] = np.copysign(F32(1e-20), d[d == 0])
    work = []
    for rays in (zero, small):
        before = g.stats()
        g.trace_closest(rays)
        after = g.stats()
        work.append((after["node_visits"] - before["node_visits"], after["prim_tests"] - before["prim_tests"]))
    print(f"\n{len(zero)} rays, node visits / primitive tests: zero components {work[0]}, +-1e-20 {work[1]}")
    assert work[1][0] > len(zero)
    assert work[0][0] <= 1.5 * work[1][0] and work[0][1] <= 1.5 * work[1][1]


@pytest.mark.gpu
@pytest.mark.parametrize("variant", VARIANTS, ids=[v[0] for v in VARIANTS])
def test_ray_counts_around_the_claim_granularity(host, orc, gpu_backend, variant):
    """Lanes claim rays one refill at a time (closest hit) or 32 at a time (shadow rays): counts on both sides of 32
    and of a 4096-ray block, and 65 537, all on edge rays of the lattice.  The 65 537 answers meet the criterion, and
    every shorter launch returns their prefix bit for bit."""
    import torch
    name, flags = variant
    case = get_case(host, orc, "lattice", bool(flags & S.ACCEL_WATERTIGHT))
    g = gpu_context(gpu_backend, host, case, flags)
    reps = -(-65537 // len(case.all))
    rays = np.tile(case.all, (reps, 1))[:65537]
    full_c, full_s = g.trace_closest(rays), g.trace_shadow(rays)
    _, bad = compare_closest(case.geometry, rays, tuple(np.tile(a, reps)[:65537] for a in case.closest), full_c)
    assert not len(bad), (name, len(bad))
    _, bad = compare_shadow(case, rays, np.tile(case.shadow, (reps, 1))[:65537], full_s)
    assert not len(bad), (name, len(bad))
    for n in (1, 31, 32, 33, 4095):
        for a, b in zip(full_c, g.trace_closest(rays[:n])):
            assert np.array_equal(a[:n].view(U32), b.view(U32)), (name, n)
        assert np.array_equal(full_s[:n].view(U32), g.trace_shadow(rays[:n]).view(U32)), (name, n)
    if flags == S.ACCEL_DEFAULT:
        dev = torch.from_numpy(rays).cuda()
        hits = torch.empty((65537, 4), device="cuda")
        g.trace_closest_device(dev.data_ptr(), 65537, hits.data_ptr())
        torch.cuda.synchronize()
        h = hits.cpu().numpy()
        for k, a in enumerate(full_c):
            assert np.array_equal(a.view(U32), h[:, k].view(U32)), k
