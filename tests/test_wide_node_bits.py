"""The bit arithmetic of the fixed-slot wide-BVH node (gpu_types.h::BvhNode8, traverse_wide.cuh), restated with Python
integers and checked exhaustively where the domain is small.  The GPU kernels are covered by the parity tests (the
8-wide, the binary and the brute-force traversals must agree bit for bit); these tests pin the identities the node
step relies on, so that a change of the layout fails here first, on the CPU:
  * the three branch-free conditional swaps move hit bit 24 + s to 24 + (s ^ octinv) for every mask and octant;
  * the rank of a primitive bit among the bits that exist is its offset from primBase;
  * subtracting a missed child's constant from the all-hit mask (the IMAD form) equals OR-ing the hit children's
    constants (the select form), and masking with the node's valid word leaves exactly the children that exist;
  * the byte -> float conversion by PRMT (m = 1 + b * 2^-15) folded into the plane FMA is the affine map it replaces,
    with the addends rounded away from the box."""
import itertools
import struct

import numpy as np
import pytest

M32 = 0xFFFFFFFF


def bit_select(a, b, m):
    """lop3 0xE4: (a & m) | (b & ~m)"""
    return ((a & m) | (b & ~m)) & M32


def octant_order(hitmask, octinv):
    """traverse_wide.cuh: the inner byte of the hit mask brought into front-to-back order."""
    s4, s2, s1 = octinv & 4, octinv & 2, octinv & 1
    x = hitmask
    x = bit_select((x << s4) & M32, x >> s4, 0xF0000000)
    x = bit_select((x << s2) & M32, x >> s2, 0xCC000000)
    x = bit_select((x << s1) & M32, x >> s1, 0xAA000000)
    return x & 0xFF000000


def child_constant(slot):
    return (1 << (24 + slot)) | (3 << (2 * slot))


@pytest.mark.parametrize("octinv", range(8))
def test_conditional_swaps_are_the_xor_permutation(octinv):
    rng = np.random.default_rng(octinv)
    for inner in range(256):
        low = int(rng.integers(0, 1 << 24))               # primitive bits and whatever else sits below: must not leak
        want = 0
        for s in range(8):
            if inner >> s & 1:
                want |= 1 << (24 + (s ^ octinv))
        assert octant_order((inner << 24) | low, octinv) == want


def test_front_most_child_is_the_highest_bit():
    # slots are assigned by centroid octant; a ray with octant mask o visits slot (7 ^ o) ^ ... first: popping the highest
    # bit of the permuted byte and XOR-ing back gives the slot, as the kernel does
    for octinv, inner in itertools.product(range(8), range(1, 256)):
        g = octant_order(inner << 24, octinv)
        bit = g.bit_length() - 1
        slot = (bit - 24) ^ octinv
        assert inner >> slot & 1
        assert all((s ^ octinv) <= (slot ^ octinv) for s in range(8) if inner >> s & 1)


def test_primitive_rank_is_the_offset_from_prim_base():
    rng = np.random.default_rng(7)
    for _ in range(2000):
        counts = rng.integers(0, 3, 8)                    # 0 = inner or empty slot, 1..2 primitives of a leaf child
        valid, offsets, off = 0, {}, 0
        for s, c in enumerate(counts):                    # bvh_wide.cu: primitives stored in slot order
            for k in range(int(c)):
                valid |= 1 << (2 * s + k)
                offsets[2 * s + k] = off
                off += 1
        g_bits = (int(rng.integers(0, 256)) << 24) | (valid << 8) | int(rng.integers(0, 256))   # hit byte | V | imask
        for k, o in offsets.items():
            rank = bin((g_bits >> 8) & ~(M32 << k) & M32).count("1")
            assert rank == o


def test_imad_form_equals_select_form_and_valid_mask():
    rng = np.random.default_rng(11)
    assert sum(child_constant(s) for s in range(8)) == 0xFF00FFFF
    for _ in range(2000):
        hit = rng.integers(0, 2, 8)
        selected = 0
        imad = 0xFF00FFFF
        for s in range(8):
            if hit[s]:
                selected |= child_constant(s)
            else:
                imad = (imad + (1 * ((0 - child_constant(s)) & M32))) & M32   # mad.lo.u32: miss bit * -K + mask
        assert imad == selected
        # the node's valid word keeps inner children (imask) and existing primitives (V) only
        kinds = rng.integers(0, 4, 8)                     # 0 empty, 1 inner, 2 leaf with 1, 3 leaf with 2 primitives
        imask = sum(1 << s for s in range(8) if kinds[s] == 1)
        v = sum(((1 << (int(kinds[s]) - 1)) - 1) << (2 * s) for s in range(8) if kinds[s] >= 2)
        got = selected & ((imask << 24) | v)
        for s in range(8):
            assert (got >> (24 + s) & 1) == int(bool(hit[s]) and kinds[s] == 1)
            assert (got >> (2 * s) & 3) == ((1 << (int(kinds[s]) - 1)) - 1 if hit[s] and kinds[s] >= 2 else 0)


def f32(x):
    return struct.unpack("<f", struct.pack("<f", x))[0]


def test_prmt_byte_conversion_is_the_affine_map_within_the_stated_bound():
    # stated bound: the I2F addends' 2^-21 of the origin term, then the subtraction of 2^15 ia rounded away from the box
    rng = np.random.default_rng(3)
    one = 0x3F800000
    for _ in range(4000):
        b = int(rng.integers(0, 256))
        m = struct.unpack("<f", struct.pack("<I", one | (b << 8)))[0]      # prmt: byte b into mantissa bits 8..15
        assert m == 1.0 + b * 2.0 ** -15
        ia = f32(float(rng.normal()) * 2.0 ** int(rng.integers(-12, 6)))   # grid scale * 1/d
        oa = f32(float(rng.normal()) * 2.0 ** int(rng.integers(-6, 12)))   # (node origin - ray origin) * 1/d
        k = f32(ia * 32768.0)
        exact = b * ia + oa
        an0, af0 = f32(oa - 2.0 ** -21 * abs(oa)), f32(oa + 2.0 ** -21 * abs(oa))   # one FMA each (the product is exact)
        near = f32(m * k + float(_round_directed(np.float64(an0) - k, up=False)))   # one FMA on the GPU: compare with its exact value
        far = f32(m * k + float(_round_directed(np.float64(af0) - k, up=True)))
        slack = 2.0 ** -23 * (abs(near) + abs(far)) + 1e-30  # the FMA's own rounding, covered by the 1e-5 far-side widening
        assert near <= exact + slack and far >= exact - slack


# ---------------------------------------------------------------------------------------------------------------------
# The node test itself: quantisation as bvh_wide.cu::k_collapse_level does it, the plane arithmetic as
# traverse_wide.cuh does it (float32, fused multiply-adds emulated through float64), against the exact slab test of the
# child's true box in float64.  The traversal may visit too much, never too little: exact hit => kernel hit.
def _fma(a, b, c):
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def _grid_exponent(extent):
    v = np.maximum(extent, np.float32(1e-30)) * np.float32(1.0 / 255.0)
    _, k = np.frexp(v)
    e = np.clip(k + 127, 1, 254)
    for _ in range(3):   # guard against rounding in the division above
        bump = (e < 254) & (np.float32(255.0) * np.ldexp(np.float32(1.0), e - 127).astype(np.float32) < extent)
        e = e + bump
    return e


def _quantise(blo, s, lo, hi):
    ql = np.clip(np.floor((lo - blo) / s), 0, 255).astype(np.int64)
    qh = np.clip(np.ceil((hi - blo) / s), 0, 255).astype(np.int64)
    for _ in range(3):   # outward rounding, verified against the planes the traversal will reconstruct
        ql -= (ql > 0) & ((blo + ql.astype(np.float32) * s).astype(np.float32) > lo)
        qh += (qh < 255) & ((blo + qh.astype(np.float32) * s).astype(np.float32) < hi)
    return ql, qh


def _round_directed(x64, up):
    """float64 -> float32 rounded towards +inf (up) or -inf, as FADD.RP / FADD.RM do."""
    r = x64.astype(np.float32)
    if up:
        return np.where(r.astype(np.float64) < x64, np.nextafter(r, np.float32(np.inf)), r).astype(np.float32)
    return np.where(r.astype(np.float64) > x64, np.nextafter(r, np.float32(-np.inf)), r).astype(np.float32)


@pytest.mark.parametrize("mix", [0x00, 0x10, 0x18, 0x30, 0x33, 0x38, 0x39, 0x3F])
def test_quantised_box_test_is_conservative(mix):
    rng = np.random.default_rng(1000 + mix)
    n = 200000
    f = np.float32
    blo = (rng.normal(size=(n, 3)) * 50).astype(f)
    ext = (10.0 ** rng.uniform(-3, 2, size=(n, 3))).astype(f)
    ext[rng.random((n, 3)) < 0.05] = 0.0                                     # flat node boxes (walls, floors)
    bhi = (blo + ext).astype(f)
    ext = (bhi - blo).astype(f)
    a, b = rng.random((n, 3)), rng.random((n, 3))
    lo = (blo + np.minimum(a, b).astype(f) * ext).astype(f)
    hi = (blo + np.maximum(a, b).astype(f) * ext).astype(f)
    flat = rng.random((n, 3)) < 0.1
    hi[flat] = lo[flat]                                                      # flat child boxes
    lo, hi = np.clip(lo, blo, bhi), np.clip(hi, blo, bhi)
    e = _grid_exponent(ext)
    s = np.ldexp(f(1.0), e - 127).astype(f)
    ql, qh = _quantise(blo, s, lo, hi)
    assert np.all((blo + ql.astype(f) * s).astype(f) <= lo) and np.all((blo + qh.astype(f) * s).astype(f) >= hi)

    # rays: aimed at a point of the child box (so that many of them hit), some axis-aligned, some far away
    target = lo + rng.random((n, 3)).astype(f) * (hi - lo)
    o = (target + rng.normal(size=(n, 3)).astype(f) * (10.0 ** rng.uniform(-2, 3, size=(n, 1))).astype(f)).astype(f)
    d = (target - o).astype(np.float64)
    d += rng.normal(size=(n, 3)) * 1e-3 * np.linalg.norm(d, axis=1, keepdims=True)   # graze: not all through the centre
    d /= np.maximum(np.linalg.norm(d, axis=1, keepdims=True), 1e-30)
    d = d.astype(f)
    axis_aligned = rng.random((n, 3)) < 0.02
    d[axis_aligned] = 0.0
    d[np.all(d == 0, axis=1)] = f(1.0)
    tmin = f(1e-3)
    tbest = np.where(rng.random(n) < 0.5, f(1e27), (10.0 ** rng.uniform(-2, 4, size=n)).astype(f)).astype(f)

    # ---- exact slab test of the true child box (float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        o64, d64 = o.astype(np.float64), d.astype(np.float64)
        t1, t2 = (lo - o64) / d64, (hi - o64) / d64
        zero = d64 == 0
        inside = (lo <= o64) & (o64 <= hi)
        near = np.where(zero, np.where(inside, -np.inf, np.inf), np.minimum(t1, t2))   # a ray parallel to a slab is
        far = np.where(zero, np.where(inside, np.inf, -np.inf), np.maximum(t1, t2))    # inside it for all t or for none
    tn_true = np.maximum(near.max(axis=1), tmin)
    tf_true = np.minimum(far.min(axis=1), tbest)
    hit_true = tn_true <= tf_true

    # ---- the kernel's arithmetic (float32)
    dd = np.where(np.abs(d) > f(1e-30), d, np.copysign(f(1e-30), d)).astype(f)
    idir = (f(1.0) / dd).astype(f)
    ulp = rng.integers(-1, 2, size=idir.shape)                               # rcp.approx: 1 ulp
    idir = np.where(ulp > 0, np.nextafter(idir, f(np.inf)), np.where(ulp < 0, np.nextafter(idir, f(-np.inf)), idir)).astype(f)
    ia = (s * idir).astype(f)
    oa = ((blo - o).astype(f) * idir).astype(f)
    neg = idir < 0
    nb, fb = np.where(neg, qh, ql), np.where(neg, ql, qh)
    c21 = f(4.76837158203125e-07)
    k = (ia * f(32768.0)).astype(f)
    tn_ax, tf_ax = np.empty_like(oa), np.empty_like(oa)
    for ax in range(3):
        for far in (False, True):
            byte = (fb if far else nb)[:, ax].astype(f)
            if mix >> (ax + (3 if far else 0)) & 1:                          # PRMT form
                m = (f(1.0) + byte * f(2.0 ** -15)).astype(f)
                # the I2F addend minus 2^15 ia, rounded away from the box
                add0 = _fma(np.full(n, c21 if far else -c21, f), np.abs(oa[:, ax]), oa[:, ax])
                add = _round_directed(add0.astype(np.float64) - k[:, ax].astype(np.float64), up=far)
                t = _fma(m, k[:, ax], add)
            else:                                                            # I2F form
                add = _fma(np.full(n, c21 if far else -c21, f), np.abs(oa[:, ax]), oa[:, ax])
                t = _fma(byte, ia[:, ax], add)
            (tf_ax if far else tn_ax)[:, ax] = t
    tn = np.maximum(tn_ax.max(axis=1), tmin)
    tf = np.minimum(tf_ax.min(axis=1), tbest)
    diff = _fma(tf, np.full(n, f(1.00001)), -tn)                             # the sign bit decides
    hit_kernel = ~np.signbit(diff)
    assert hit_true.sum() > n // 10                                          # the sample does exercise hits
    missed = hit_true & ~hit_kernel
    assert not missed.any(), f"{missed.sum()} exact hits culled, e.g. index {np.flatnonzero(missed)[:5]}"
    # and it is a box test, not a constant: most exact misses stay misses
    assert (hit_kernel & ~hit_true).sum() < 0.5 * (~hit_true).sum()
