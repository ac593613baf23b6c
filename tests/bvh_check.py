"""A numpy validator of a built acceleration structure: the four arrays mox_debug_read_accel returns (binary nodes, wide
nodes, and the two leaf-ordered packed primitive arrays) against the primitives the test added.

It restates what the builder must produce, not how:
  * primitive boxes and validity as bvh_build.cu::primBounds computes them (float32, the same operation order; the
    library is compiled with -fmad=false, so triangles and spheres match bit for bit; quads are given one ulp);
  * binary nodes (gpu_types.h::BvhNode2): a tree from node 0, leaf ranges that partition [0, nValid), child boxes that
    are the exact unions of what lies below, depth within the traversal stack;
  * packed records as bvh_build.cu::k_pack writes them, class bits included;
  * wide nodes (gpu_types.h::BvhNode8): header words, a tree over [0, nNodes8), every packed8 record referenced once,
    the node origin and the grid exponents and plane bytes of the quantiser model in test_wide_node_bits.py.
Every check raises BvhError naming the node, slot or primitive at fault."""
import numpy as np

from test_wide_node_bits import _grid_exponent, _quantise

LEAF_MAX = 2                      # gpu_types.h MOX_LEAF_MAX (binary leaves) and MOX_WIDE_LEAF_MAX
TRAVERSAL_STACK = 128             # gpu_types.h MOX_TRAVERSAL_STACK
DEPTH_MAX = TRAVERSAL_STACK - 2
EMPTY_CHILD = -0x80000000
FAR = np.float32(3.0e38)
PT_TRI, PT_SPHERE, PT_QUAD = 0, 1, 2
MAT_LAMBERTIAN, MAT_METAL, MAT_GLASS, MAT_DISNEY, MAT_LIGHT = range(5)
BRDF_GLASS = 1
ID_MASK = 0x3FFFFFFF
F32 = np.float32


class BvhError(AssertionError):
    pass


def _fail(msg):
    raise BvhError(msg)


def class_word(kind, brdf_type=0):
    """Word 1 .w of a packed record: shadow class | shade class << 2 (gpu_types.h MOX_SHADOW_* / MOX_CLASS_*)."""
    shadow, cls = 0, 0
    if kind == MAT_DISNEY:
        shadow, cls = (2, 2) if brdf_type == BRDF_GLASS else (1, 3)
    elif kind == MAT_METAL:
        cls = 1
    elif kind == MAT_GLASS:
        cls = 2
    elif kind == MAT_LIGHT:
        cls = 4
    return shadow | cls << 2


class SceneData:
    """The primitives of a scene in id order, mirrored on the host while add_* forwards them to every context."""

    def __init__(self, *ctxs):
        self.ctxs = list(ctxs)
        self.chunks = []          # (type, first id, count, class word, payload)
        self.n = 0
        self._cache = None

    def _mat_word(self, kind, params):
        return class_word(kind, getattr(params, "brdfType", 0) if kind == MAT_DISNEY else 0)

    def add_mesh(self, verts, idx, kind, params):
        verts = np.ascontiguousarray(verts, np.float32).reshape(-1, 3)
        idx = np.ascontiguousarray(idx, np.int32).reshape(-1, 3)
        first = None
        for c in self.ctxs:
            got = c.add_mesh(verts, idx, kind, params)
            assert first is None or got == first
            first = got
        assert first in (None, self.n), (first, self.n)
        self.chunks.append([PT_TRI, self.n, len(idx), self._mat_word(kind, params), [verts, idx]])
        self.n += len(idx)
        self._cache = None
        return self.n - len(idx)

    def update_mesh(self, first, verts):
        verts = np.ascontiguousarray(verts, np.float32).reshape(-1, 3)
        for c in self.ctxs:
            c.update_mesh(first, verts)
        ch = next(ch for ch in self.chunks if ch[0] == PT_TRI and ch[1] == first)
        assert ch[4][0].shape == verts.shape
        ch[4][0] = verts
        self._cache = None

    def add_sphere(self, sphere, kind, params):
        for c in self.ctxs:
            c.add_sphere(sphere, kind, params)
        cr = np.array([[sphere.center.x, sphere.center.y, sphere.center.z, sphere.radius]], np.float32)
        self.chunks.append([PT_SPHERE, self.n, 1, self._mat_word(kind, params), cr])
        self.n += 1
        self._cache = None

    def add_quad(self, quad, kind, params):
        for c in self.ctxs:
            c.add_quad(quad, kind, params)
        q = np.array([[quad.v1.x, quad.v1.y, quad.v1.z, quad.v2.x, quad.v2.y, quad.v2.z,
                       quad.anchor.x, quad.anchor.y, quad.anchor.z]], np.float32)
        self.chunks.append([PT_QUAD, self.n, 1, self._mat_word(kind, params), q])
        self.n += 1
        self._cache = None

    def arrays(self):
        """Per primitive id: type, class word, analytic index, triangle vertices (n, 3, 3), spheres (n, 4), quads (n, 9)."""
        if self._cache is not None:
            return self._cache
        n = self.n
        typ = np.zeros(n, np.uint32)
        word = np.zeros(n, np.uint32)
        geom = np.zeros(n, np.int64)
        tri = np.zeros((n, 3, 3), np.float32)
        sph = np.zeros((n, 4), np.float32)
        quad = np.zeros((n, 9), np.float32)
        n_analytic = 0
        for t, first, cnt, w, payload in self.chunks:
            sl = slice(first, first + cnt)
            typ[sl], word[sl] = t, w
            if t == PT_TRI:
                verts, idx = payload
                tri[sl] = verts[idx]
            else:
                geom[sl] = n_analytic
                n_analytic += 1
                (sph if t == PT_SPHERE else quad)[sl] = payload
        self._cache = dict(type=typ, word=word, geom=geom, tri=tri, sph=sph, quad=quad)
        return self._cache


# ------------------------------------------------------------------------------------------------ primitive boxes
def _cross(a, b):
    return np.stack([a[..., 1] * b[..., 2] - a[..., 2] * b[..., 1],
                     a[..., 2] * b[..., 0] - a[..., 0] * b[..., 2],
                     a[..., 0] * b[..., 1] - a[..., 1] * b[..., 0]], axis=-1)


def _dot(a, b):
    return a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1] + a[..., 2] * b[..., 2]


def prim_bounds(scene):
    """primBounds of every primitive: (valid, lo, hi, slack) with float32 boxes; slack = one ulp (quads), else 0."""
    a = scene.arrays()
    typ, n = a["type"], scene.n
    lo = np.full((n, 3), np.inf, np.float32)
    hi = np.full((n, 3), -np.inf, np.float32)
    valid = np.zeros(n, bool)
    with np.errstate(all="ignore"):
        m = typ == PT_TRI
        if m.any():
            v0, v1, v2 = (a["tri"][m, k] for k in range(3))
            area = np.sqrt(_dot(c := _cross(v1 - v0, v2 - v0), c))
            valid[m] = (area > 0) & ~np.isinf(area)
            lo[m] = np.fmin(np.fmin(v0, v1), v2)
            hi[m] = np.fmax(np.fmax(v0, v1), v2)
        m = typ == PT_SPHERE
        if m.any():
            c, r = a["sph"][m, :3], a["sph"][m, 3:4]
            l, h = c + (-r), c + r
            neg = r < 0
            lo[m], hi[m] = np.where(neg, h, l), np.where(neg, l, h)
            valid[m] = (r[:, 0] == r[:, 0]) & ~np.isinf(r[:, 0])
        m = typ == PT_QUAD
        if m.any():
            q = a["quad"][m]
            v1, v2, an = q[:, 0:3], q[:, 3:6], q[:, 6:9]
            tv1 = v1 * (F32(1) / _dot(v1, v1))[:, None]
            tv2 = v2 * (F32(1) / _dot(v2, v2))[:, None]
            p01, p10, p11 = an + tv1, an + tv2, an + tv1 + tv2
            area = np.sqrt(_dot(c := _cross(tv1, tv2), c))
            valid[m] = (area > 0) & ~np.isinf(area)
            lo[m] = np.fmin(np.fmin(an, p01), np.fmin(p10, p11))
            hi[m] = np.fmax(np.fmax(an, p01), np.fmax(p10, p11))
    lo[~valid], hi[~valid] = np.inf, -np.inf
    return valid, lo, hi, (typ == PT_QUAD) & valid


class _Boxes:
    """Box bounds per entry: the true box lies in lo [lo_dn, lo_up], hi [hi_dn, hi_up] (equal bounds: exact)."""

    def __init__(self, lo_dn, lo_up, hi_dn, hi_up):
        self.lo_dn, self.lo_up, self.hi_dn, self.hi_up = lo_dn, lo_up, hi_dn, hi_up

    @classmethod
    def of_prims(cls, lo, hi, slack):
        s = slack[:, None]
        return cls(np.where(s, np.nextafter(lo, F32(-np.inf)), lo), np.where(s, np.nextafter(lo, F32(np.inf)), lo),
                   np.where(s, np.nextafter(hi, F32(-np.inf)), hi), np.where(s, np.nextafter(hi, F32(np.inf)), hi))

    def take(self, i):
        return _Boxes(self.lo_dn[i], self.lo_up[i], self.hi_dn[i], self.hi_up[i])

    def exact(self):
        return np.all(self.lo_dn == self.lo_up, axis=-1) & np.all(self.hi_dn == self.hi_up, axis=-1)

    def holds(self, lo, hi):
        """Rows whose stored box (lo, hi) is not within the bounds."""
        return ~(np.all((self.lo_dn <= lo) & (lo <= self.lo_up) & (self.hi_dn <= hi) & (hi <= self.hi_up), axis=-1))


def _union(boxes, axis):
    return _Boxes(boxes.lo_dn.min(axis=axis), boxes.lo_up.min(axis=axis), boxes.hi_dn.max(axis=axis), boxes.hi_up.max(axis=axis))


# ------------------------------------------------------------------------------------------------ packed records
def expected_records(scene, ids, watertight):
    """k_pack's 48-byte record of each primitive id, as (len(ids), 12) uint32."""
    a = scene.arrays()
    typ, word, geom = a["type"][ids], a["word"][ids], a["geom"][ids]
    rec = np.zeros((len(ids), 12), np.uint32)
    f = rec.view(np.float32)
    rec[:, 3] = ids.astype(np.uint32) | (typ << 30)
    rec[:, 7] = word
    rec[:, 11] = typ
    m = typ == PT_TRI
    t = a["tri"][ids[m]]
    p0, p1, p2 = t[:, 0], t[:, 1], t[:, 2]
    f[m, 0:3] = p0
    f[m, 4:7] = p1 if watertight else p1 - p0
    f[m, 8:11] = p2 if watertight else p0 - p2
    m = typ != PT_TRI
    rec[m, 0] = geom[m].astype(np.uint32)
    m = typ == PT_SPHERE
    s = a["sph"][ids[m]]
    f[m, 4:7] = s[:, :3]
    f[m, 8] = s[:, 3]
    return rec


def _check_packed(name, packed, scene, valid, watertight):
    rec = packed.view(np.uint32).reshape(-1, 12)
    n_valid = int(valid.sum())
    if len(rec) != n_valid:
        _fail(f"{name}: {len(rec)} records for {n_valid} valid primitives")
    ids = (rec[:, 3] & ID_MASK).astype(np.int64)
    bad = np.flatnonzero(ids >= scene.n)
    if len(bad):
        _fail(f"{name}: slot {bad[0]} holds primitive id {ids[bad[0]]} of {scene.n}")
    bad = np.flatnonzero(~valid[ids])
    if len(bad):
        _fail(f"{name}: slot {bad[0]} holds the invalid primitive {ids[bad[0]]}")
    count = np.bincount(ids, minlength=scene.n)
    if (count > 1).any():
        p = int(np.flatnonzero(count > 1)[0])
        _fail(f"{name}: primitive {p} is in slots {np.flatnonzero(ids == p).tolist()}")
    want = expected_records(scene, ids, watertight)
    bad = np.flatnonzero(np.any(want != rec, axis=1))
    if len(bad):
        k = int(bad[0])
        _fail(f"{name}: slot {k} (primitive {ids[k]}): record {rec[k].tolist()} != k_pack's {want[k].tolist()}")
    return ids


# ------------------------------------------------------------------------------------------------ binary nodes
def _binary_slots(nodes):
    f = nodes.view(np.float32).reshape(-1, 16)
    lo = np.stack([np.stack([f[:, 4 * k], f[:, 4 * k + 2], f[:, 8 + 2 * k]], axis=-1) for k in range(2)], axis=1)
    hi = np.stack([np.stack([f[:, 4 * k + 1], f[:, 4 * k + 3], f[:, 9 + 2 * k]], axis=-1) for k in range(2)], axis=1)
    ref = nodes.view(np.int32).reshape(-1, 16)[:, 12:14]
    return lo, hi, ref


def _check_binary(nodes, packed_ids, prim_boxes, n_valid):
    n_nodes = nodes.size // 64
    lo, hi, ref = _binary_slots(nodes)
    if n_valid <= 1:
        if n_nodes != 1:
            _fail(f"binary: {n_nodes} nodes for {n_valid} valid primitives")
        far = np.full(3, FAR, np.float32)
        if ref[0, 1] != EMPTY_CHILD or not (np.array_equal(lo[0, 1], far) and np.array_equal(hi[0, 1], far)):
            _fail("binary: root slot 1 is not an empty child with MOX_FAR planes")
        if n_valid == 0:
            if ref[0, 0] != EMPTY_CHILD or not (np.array_equal(lo[0, 0], far) and np.array_equal(hi[0, 0], far)):
                _fail("binary: root slot 0 of an empty structure is not an empty child with MOX_FAR planes")
        else:
            if ref[0, 0] != ~0:
                _fail(f"binary: root slot 0 ref {ref[0, 0]} is not the one-primitive leaf ~0")
            if prim_boxes.take(packed_ids[:1]).holds(lo[0, :1], hi[0, :1]).any():
                _fail(f"binary: root box {lo[0, 0]} {hi[0, 0]} is not the box of primitive {packed_ids[0]}")
        return 1
    if n_nodes != n_valid - 1:
        _fail(f"binary: {n_nodes} nodes for {n_valid} valid primitives")
    refcount = np.zeros(n_nodes, np.int64)
    frontier, depth, reached = np.array([0]), 0, 1
    leaves = []                                          # (node, slot, first, count)
    while len(frontier):
        depth += 1
        if depth > DEPTH_MAX:
            _fail(f"binary: depth {depth} > {DEPTH_MAX} at nodes {frontier[:4].tolist()}")
        r = ref[frontier]
        inner = r >= 0
        kids = r[inner]
        if (kids >= n_nodes).any():
            k = np.argwhere(inner & (r >= n_nodes))[0]
            _fail(f"binary: node {frontier[k[0]]} slot {k[1]} refers to node {r[k[0], k[1]]} of {n_nodes}")
        if (kids == 0).any() or len(np.unique(kids)) != len(kids) or (refcount[kids] > 0).any():
            dup = kids[(kids == 0) | (refcount[kids] > 0) | (np.bincount(kids, minlength=n_nodes)[kids] > 1)][0]
            _fail(f"binary: node {dup} is referenced more than once (or is the root)")
        refcount[kids] += 1
        # child box = union of the child's two stored boxes
        pn, ps = np.nonzero(inner)
        if len(pn):
            c = r[pn, ps]
            ulo, uhi = np.minimum(lo[c, 0], lo[c, 1]), np.maximum(hi[c, 0], hi[c, 1])
            bad = np.flatnonzero(np.any((lo[frontier[pn], ps] != ulo) | (hi[frontier[pn], ps] != uhi), axis=1))
            if len(bad):
                k = bad[0]
                _fail(f"binary: node {frontier[pn[k]]} slot {ps[k]} box {lo[frontier[pn[k]], ps[k]]} {hi[frontier[pn[k]], ps[k]]}"
                      f" != union of node {c[k]}'s boxes {ulo[k]} {uhi[k]}")
        ln, ls = np.nonzero(~inner)
        if len(ln):
            v = ~r[ln, ls]
            if (r[ln, ls] == EMPTY_CHILD).any():
                k = np.flatnonzero(r[ln, ls] == EMPTY_CHILD)[0]
                _fail(f"binary: node {frontier[ln[k]]} slot {ls[k]} is empty in a tree of {n_valid} primitives")
            leaves.append(np.stack([frontier[ln], ls, v >> 3, (v & 7) + 1], axis=1))
        frontier = kids
        reached += len(kids)
    leaves = np.concatenate(leaves)
    node, slot, first, count = leaves.T
    bad = np.flatnonzero((count > LEAF_MAX) | (first + count > n_valid))
    if len(bad):
        k = bad[0]
        _fail(f"binary: node {node[k]} slot {slot[k]} leaf [{first[k]}, +{count[k]}) (leaf max {LEAF_MAX}, {n_valid} records)")
    cover = np.zeros(n_valid + 1, np.int64)
    for c in range(1, LEAF_MAX + 1):
        for j in range(c):
            np.add.at(cover, first[count == c] + j, 1)
    if (cover[:n_valid] != 1).any():
        p = int(np.flatnonzero(cover[:n_valid] != 1)[0])
        _fail(f"binary: packed record {p} is covered by {cover[p]} leaves")
    # a leaf of c primitives stands for c - 1 folded inner nodes: the reachable nodes and the folded ones are all nodes
    if reached + int((count - 1).sum()) != n_nodes:
        _fail(f"binary: {reached} reachable nodes + {int((count - 1).sum())} folded != {n_nodes}")
    # leaf box = union of its primitives' boxes
    pid = packed_ids[np.stack([first, np.minimum(first + 1, n_valid - 1)], axis=1)]
    b = prim_boxes.take(pid)
    one = count == 1
    for arr in (b.lo_dn, b.lo_up, b.hi_dn, b.hi_up):
        arr[one, 1] = arr[one, 0]
    bad = np.flatnonzero(_union(b, 1).holds(lo[node, slot], hi[node, slot]))
    if len(bad):
        k = bad[0]
        _fail(f"binary: node {node[k]} slot {slot[k]} leaf box {lo[node[k], slot[k]]} {hi[node[k], slot[k]]} != the union of "
              f"primitives {pid[k, :count[k]].tolist()}")
    return depth


# ------------------------------------------------------------------------------------------------ wide nodes
def _check_wide(nodes8, packed_ids, prim_boxes, n_valid, rec_packed, rec_packed8):
    m = nodes8.size // 80
    u = nodes8.view(np.uint32).reshape(m, 20)
    f = nodes8.view(np.float32).reshape(m, 20)
    q = nodes8.reshape(m, 80)[:, 32:80].reshape(m, 6, 8).astype(np.int64)     # qlx qly qlz qhx qhy qhz, 8 slots each
    ql, qh = q[:, 0:3].transpose(0, 2, 1), q[:, 3:6].transpose(0, 2, 1)       # (m, 8 slots, 3 axes)
    p = f[:, 0:3]
    e = np.stack([u[:, 3] & 255, (u[:, 3] >> 8) & 255, (u[:, 3] >> 16) & 255], axis=1).astype(np.int64)
    imask, child_base, prim_base, valid, group = u[:, 3] >> 24, u[:, 4].astype(np.int64), u[:, 5].astype(np.int64), u[:, 6], u[:, 7]
    vbits = valid & 0xFFFF
    for name, bad in (("n0.w and valid disagree on imask", (valid >> 24) != imask),
                      ("valid bits 16..23 are set", (valid >> 16) & 0xFF != 0),
                      ("group != V << 8 | imask", group != ((vbits << 8) | imask))):
        if bad.any():
            _fail(f"wide: node {np.flatnonzero(bad)[0]}: {name}")
    slot_v = np.stack([(vbits >> (2 * s)) & 3 for s in range(8)], axis=1).astype(np.int64)      # (m, 8)
    slot_inner = np.stack([(imask >> s) & 1 for s in range(8)], axis=1).astype(bool)
    for name, bad in (("primitive bits 10", slot_v == 2), ("both an inner and a leaf child", slot_inner & (slot_v != 0))):
        if bad.any():
            w, s = np.argwhere(bad)[0]
            _fail(f"wide: node {w} slot {s}: {name}")
    empty = ~slot_inner & (slot_v == 0)
    bad = empty & ~(np.all(ql == 255, axis=2) & np.all(qh == 0, axis=2))
    if bad.any():
        w, s = np.argwhere(bad)[0]
        _fail(f"wide: node {w} slot {s} is empty but its planes are {ql[w, s].tolist()} {qh[w, s].tolist()}")
    # children: inner ones at childBase + rank, primitives at primBase + rank of their V bit
    inner_rank = np.cumsum(slot_inner, axis=1) - slot_inner
    child = np.where(slot_inner, child_base[:, None] + inner_rank, -1)
    slot_cnt = np.where(slot_v == 3, 2, slot_v)
    prim_off = prim_base[:, None] + np.cumsum(slot_cnt, axis=1) - slot_cnt
    refcount = np.zeros(m, np.int64)
    levels, frontier, depth = [], np.array([0]), 0
    while len(frontier):
        depth += 1
        if depth > DEPTH_MAX:
            _fail(f"wide: depth {depth} > {DEPTH_MAX} at nodes {frontier[:4].tolist()}")
        levels.append(frontier)
        kids = child[frontier][slot_inner[frontier]]
        if (kids >= m).any():
            _fail(f"wide: a child of nodes {frontier[:4].tolist()} refers to node {kids[kids >= m][0]} of {m}")
        if (kids == 0).any() or len(np.unique(kids)) != len(kids) or (refcount[kids] > 0).any():
            dup = kids[(kids == 0) | (refcount[kids] > 0) | (np.bincount(kids, minlength=m)[kids] > 1)][0]
            _fail(f"wide: node {dup} is referenced more than once (or is the root)")
        refcount[kids] += 1
        frontier = kids
    if refcount[1:].min(initial=1) != 1:
        _fail(f"wide: node {1 + int(np.argmin(refcount[1:]))} of {m} is not reached from the root")
    lw, ls = np.nonzero(slot_cnt)
    first, cnt = prim_off[lw, ls], slot_cnt[lw, ls]
    if (first + cnt > n_valid).any():
        k = np.flatnonzero(first + cnt > n_valid)[0]
        _fail(f"wide: node {lw[k]} slot {ls[k]} refers to packed8 [{first[k]}, +{cnt[k]}) of {n_valid}")
    cover = np.zeros(n_valid, np.int64)
    np.add.at(cover, first, 1)
    np.add.at(cover, first[cnt == 2] + 1, 1)
    if (cover != 1).any():
        k = int(np.flatnonzero(cover != 1)[0])
        _fail(f"wide: packed8 record {k} is referenced by {cover[k]} leaf slots")
    # packed8 is a permutation of packed (both hold each valid primitive once, checked by the caller)
    ids8 = (rec_packed8[:, 3] & ID_MASK).astype(np.int64)
    o, o8 = np.argsort(packed_ids), np.argsort(ids8)
    if not np.array_equal(packed_ids[o], ids8[o8]) or not np.array_equal(rec_packed[o], rec_packed8[o8]):
        _fail("wide: packed8 is not a permutation of packed's records")
    # subtree boxes, bottom-up: leaf slots from their primitives, inner slots from the child's union
    inf = np.full((m, 8, 3), np.inf, np.float32)
    slots = _Boxes(inf.copy(), inf.copy(), -inf, -inf)
    pb = prim_boxes.take(ids8)
    for k in range(2):
        sel = cnt > k
        idx = first[sel] + k
        for a, b, red in ((slots.lo_dn, pb.lo_dn, np.minimum), (slots.lo_up, pb.lo_up, np.minimum),
                          (slots.hi_dn, pb.hi_dn, np.maximum), (slots.hi_up, pb.hi_up, np.maximum)):
            a[lw[sel], ls[sel]] = red(a[lw[sel], ls[sel]], b[idx])
    fields = ("lo_dn", "lo_up", "hi_dn", "hi_up")
    node_box = {a: np.zeros((m, 3), np.float32) for a in fields}
    exact_nodes = 0
    for level in reversed(levels):
        iw, is_ = np.nonzero(slot_inner[level])
        c = child[level[iw], is_]
        for a in fields:
            getattr(slots, a)[level[iw], is_] = node_box[a][c]
        occ = ~empty[level]
        sb = slots.take(level)
        nb = _union(sb, 1)
        # origin = the minimum over the slots
        bad = np.flatnonzero(~np.all((nb.lo_dn <= p[level]) & (p[level] <= nb.lo_up), axis=1))
        if len(bad):
            _fail(f"wide: node {level[bad[0]]} origin {p[level[bad[0]]]} != the minimum over its slots {nb.lo_dn[bad[0]]}")
        exact = np.all(sb.exact() | ~occ, axis=1)
        exact_nodes += int(exact.sum())
        ex = level[exact]
        if len(ex):
            blo, bhi = nb.lo_dn[exact], nb.hi_dn[exact]
            want_e = _grid_exponent((bhi - blo).astype(np.float32))
            bad = np.flatnonzero(np.any(want_e != e[ex], axis=1))
            if len(bad):
                _fail(f"wide: node {ex[bad[0]]} exponents {e[ex[bad[0]]].tolist()} != {want_e[bad[0]].tolist()}")
            s = np.ldexp(F32(1.0), e[ex] - 127).astype(np.float32)[:, None, :]
            wl, wh = _quantise(p[ex][:, None, :], s, sb.lo_dn[exact], sb.hi_dn[exact])
            bad = np.argwhere(occ[exact][:, :, None] & ((wl != ql[ex]) | (wh != qh[ex])))
            if len(bad):
                w, sl, ax = bad[0]
                _fail(f"wide: node {ex[w]} slot {sl} axis {ax}: planes ({ql[ex[w], sl, ax]}, {qh[ex[w], sl, ax]}) != the "
                      f"quantiser's ({wl[w, sl, ax]}, {wh[w, sl, ax]})")
        nx = level[~exact]
        if len(nx):   # one-ulp boxes: the planes contain the box and lie at most two grid steps outside it
            s = np.ldexp(F32(1.0), e[nx] - 127).astype(np.float32)[:, None, :]
            pl = (p[nx][:, None, :] + ql[nx].astype(np.float32) * s).astype(np.float32)
            ph = (p[nx][:, None, :] + qh[nx].astype(np.float32) * s).astype(np.float32)
            b = slots.take(nx)
            with np.errstate(invalid="ignore"):
                ok = (pl <= b.lo_up) & (ph >= b.hi_dn) & (pl >= b.lo_dn - 2 * s) & (ph <= b.hi_up + 2 * s)
            bad = np.argwhere(occ[~exact][:, :, None] & ~ok)
            if len(bad):
                w, sl, ax = bad[0]
                _fail(f"wide: node {nx[w]} slot {sl} axis {ax}: planes [{pl[w, sl, ax]}, {ph[w, sl, ax]}] do not hold the box "
                      f"[{b.lo_dn[w, sl, ax]}, {b.hi_up[w, sl, ax]}] within two grid steps")
        for a in fields:
            node_box[a][level] = getattr(nb, a)
    return depth, exact_nodes


def check_arrays(arrays, stats, scene, watertight=False):
    """Validate the host copies of the four arrays (uint8, as Context.debug_read_accel returns them) against the
    scene and the stats record (n_nodes, node_bytes).  Returns a summary: valid primitives, node counts, depths."""
    valid, lo, hi, slack = prim_bounds(scene)
    boxes = _Boxes.of_prims(lo, hi, slack)
    n_valid = int(valid.sum())
    ids = _check_packed("packed", arrays["packed"], scene, valid, watertight)
    depth = _check_binary(arrays["nodes"], ids, boxes, n_valid)
    out = dict(n_valid=n_valid, n_nodes=arrays["nodes"].size // 64, binary_depth=depth, n_nodes8=0, wide_depth=0)
    wide = arrays["nodes8"].size > 0
    if stats["node_bytes"] != (80 if wide else 64):
        _fail(f"stats: node_bytes {stats['node_bytes']} with {arrays['nodes8'].size} bytes of wide nodes")
    if stats["n_nodes"] != (arrays["nodes8"].size // 80 if wide else out["n_nodes"]):
        _fail(f"stats: n_nodes {stats['n_nodes']} != the {'wide' if wide else 'binary'} node count")
    if wide:
        _check_packed("packed8", arrays["packed8"], scene, valid, watertight)
        rec = arrays["packed"].view(np.uint32).reshape(-1, 12)
        rec8 = arrays["packed8"].view(np.uint32).reshape(-1, 12)
        out["wide_depth"], out["exact_wide_nodes"] = _check_wide(arrays["nodes8"], ids, boxes, n_valid, rec, rec8)
        out["n_nodes8"] = arrays["nodes8"].size // 80
    elif arrays["packed8"].size:
        _fail("packed8 holds records without wide nodes")
    return out


ARRAYS = ("nodes", "nodes8", "packed", "packed8")


def read_arrays(ctx):
    return {k: ctx.debug_read_accel(k) for k in ARRAYS}


def check(ctx, scene, watertight=False):
    """Read the built structure of ctx and validate it against scene; returns check_arrays' summary."""
    return check_arrays(read_arrays(ctx), ctx.stats(), scene, watertight)
