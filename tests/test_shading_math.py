"""The shading math, value by value, against a float64 restatement of the reference (tests/disney_ref.py).

The image tests hold the render path to the oracle through whole images, where k_accumulate clamps every sample
to [0, 1] and a few image-wide tolerances hide errors confined to thin bands of pixels.  Here:
  * the float64 reference against the oracle's float32 functions over an edge grid (CPU), which pins the
    reference to the formulas the oracle states;
  * the device functions of shading.cuh, compiled into tests/probe/libshading_probe.so with the flags of
    libmox.so, over the same grid: DisneyHit in IEEE mode bit for bit against the oracle, in the default fast mode
    against the float64 reference within the documented error bounds of the approximate instructions;
    disneySample; refract3 / fresnelDielectric;
  * the hardware texture filter per pixel through the product, and the Disney light loop per pixel at depth 1.
Tolerances are stated against a conditioning scale: a first-order bound on the error of a float32 evaluation of the
same operations (disney_ref.X), so that cancelling sums are held to the error of their terms.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import disney_ref as R
from conftest import ROOT
from minimaloptix_b200 import structs as S

EPS = R.EPS
PROBE_LIB = os.path.join(ROOT, "tests", "probe", "libshading_probe.so")
# First-order bounds are exceeded only by second-order terms; the factor covers those, nothing else.
C_BOUND = 2.0
PARAM_NAMES = ("metallic", "subsurface", "specular", "roughness", "specularTint", "anisotropic", "sheen", "sheenTint",
               "clearcoat", "clearcoatGloss")


# ---------------------------------------------------------------------------------------------- the edge grid
def _unit(v):
    v = np.asarray(v, np.float64)
    return (v / np.linalg.norm(v, axis=-1, keepdims=True)).astype(np.float32)


def _frame(n):
    """Two float64 unit vectors orthogonal to each row of n."""
    a = np.where(np.abs(n[:, :1]) < 0.9, [[1.0, 0, 0]], [[0, 1.0, 0]])
    t = np.cross(n, a)
    t /= np.linalg.norm(t, axis=1, keepdims=True)
    return t, np.cross(n, t)


def _direction(n, cos_theta, rng):
    """Unit vectors at the given cosine to n (float64 n), random azimuth."""
    t, b = _frame(n)
    phi = rng.uniform(0, 2 * np.pi, len(n))
    s = np.sqrt(np.maximum(0.0, 1 - cos_theta ** 2))
    return cos_theta[:, None] * n + s[:, None] * (np.cos(phi)[:, None] * t + np.sin(phi)[:, None] * b)


def make_grid(seed=20261022, n_random=3000):
    """Cases of (params, baseColor, N, V, L, kind).  Parameters each in {0, 1, random}, the roughness corners around
    the 0.001 clamps, anisotropic = 1, clearcoatGloss = 1, metallic = 1; base colours 0, 1, primaries, 1e-6, random;
    normals on the axes, on the |n.x| == |n.z| tie of the Onb, random; directions random in the hemisphere, grazing
    (N.V, N.L in {1e-7, 1e-4}), the mirror direction (H = N), L ~ -V and N.V < 0 < N.L."""
    rng = np.random.default_rng(seed)
    normals = [[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1], [1, 0.3, 1], [-0.7, 0.2, 0.7]]
    colours = [[0, 0, 0], [1, 1, 1], [1, 0, 0], [0, 1, 0], [0, 0, 1], [1e-6, 1e-6, 1e-6]]
    kinds = ["random", "graze_v", "graze_l", "graze_both", "mirror", "opposite", "backside"]
    n = n_random + 64 * len(kinds)
    P = np.where(rng.random((n, 10)) < 0.5, rng.integers(0, 2, (n, 10)).astype(np.float64), rng.random((n, 10)))
    corner = rng.random(n)
    rough = rng.choice([1e-4, 0.001, 0.0316, 1.0], n)
    P[:, 3] = np.where(corner < 0.3, rough, P[:, 3])
    P[:, 5] = np.where(rng.random(n) < 0.15, 1.0, P[:, 5])
    P[:, 9] = np.where(rng.random(n) < 0.15, 1.0, P[:, 9])
    P[:, 0] = np.where(rng.random(n) < 0.15, 1.0, P[:, 0])
    pick = rng.random(n)
    base = np.where((pick < 0.5)[:, None], rng.random((n, 3)), np.array(colours)[rng.integers(0, len(colours), n)])
    Nn = np.where((rng.random(n) < 0.4)[:, None], np.array(normals, np.float64)[rng.integers(0, len(normals), n)],
                  rng.normal(size=(n, 3)))
    N = _unit(Nn)
    n64 = N.astype(np.float64)
    kind = np.array(kinds)[np.concatenate([np.zeros(n_random, int), np.repeat(np.arange(len(kinds)), 64)])]
    graze = rng.choice([1e-7, 1e-4], n)
    cv = np.where(np.isin(kind, ["graze_v", "graze_both"]), graze, rng.uniform(0.02, 1, n))
    cl = np.where(np.isin(kind, ["graze_l", "graze_both"]), rng.choice([1e-7, 1e-4], n), rng.uniform(0.02, 1, n))
    cv = np.where(kind == "backside", -rng.uniform(0.001, 0.5, n), cv)
    V = _direction(n64, cv, rng)
    L = _direction(n64, cl, rng)
    mirror = kind == "mirror"
    L[mirror] = 2 * np.sum(n64[mirror] * V[mirror], axis=1, keepdims=True) * n64[mirror] - V[mirror]
    opp = kind == "opposite"    # L within a few ulps of -V; V below the shading normal, L above it
    V[opp] = _direction(n64[opp], -rng.uniform(0.05, 0.9, opp.sum()), rng)
    L[opp] = -V[opp] + rng.normal(scale=1e-6, size=(opp.sum(), 3))
    V, L = _unit(V), _unit(L)
    params = (S.DisneyParams * n)()
    for i in range(n):
        d = params[i]
        for k, name in enumerate(PARAM_NAMES):
            setattr(d, name, float(P[i, k]))
        d.color = S.float3(*base[i]); d.brdfType = S.NORMAL
    return params, base.astype(np.float32), N, V, L, kind


def dot32(a, b):
    """The device's dot product (-fmad=false): ((x*x + y*y) + z*z), each step rounded to float32."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return (a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1]) + a[:, 2] * b[:, 2]


def normalize32(v):
    """IEEE normalize as the SDK spells it: v * (1 / sqrt(dot(v, v)))."""
    v = np.asarray(v, np.float32)
    inv = np.float32(1.0) / np.sqrt(dot32(v, v))
    return v * inv[:, None]


def well_conditioned(N, V, L, H):
    return (dot32(N, V) >= 1e-3) & (dot32(N, L) >= 1e-3) & (np.abs(dot32(L, H)) >= 1e-3)


@pytest.fixture(scope="module")
def grid():
    return make_grid()


def _oracle_pdf_eval(orc, params, base, N, V, L, H):
    b = orc.backend()
    f3 = C.c_float * 3
    n = len(N)
    pdf, ev = np.empty(n, np.float32), np.empty((n, 3), np.float32)
    out = f3()
    for i in range(n):
        args = [f3(*N[i]), f3(*L[i]), f3(*V[i]), f3(*H[i])]
        pdf[i] = b.disney_pdf(C.byref(params[i]), *args)
        b.disney_eval(C.byref(params[i]), f3(*base[i]), *args, out)
        ev[i] = out[:]
    return pdf, ev


def _ratio(got, ref, bound):
    """|got - ref| in units of the conditioning bound; 0 where both agree exactly."""
    got = np.asarray(got, np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.abs(got - ref) / (EPS * bound)
    return np.where(got == ref, 0.0, r)


def _finite(*a):
    m = np.ones(a[0].shape[0], bool)
    for x in a:
        m &= np.all(np.isfinite(x.reshape(len(x), -1)), axis=1)
    return m


# ---------------------------------------------------------------------------------------------- CPU: the reference
def test_reference_states_the_oracle_formulas(orc, grid):
    """The float64 reference against the oracle's float32 disneyPdf / disneyEval, which test_ref_render.py pins bit for
    bit to the compiled reference sources: one bound factor for the whole grid."""
    params, base, N, V, L, kind = grid
    H = normalize32(L + V)
    pdf, ev = _oracle_pdf_eval(orc, params, base, N, V, L, H)
    rp, _, re = R.pdf_eval(params, base, N, V, L, H, R.IEEE)
    ok = _finite(rp.v, rp.e, R.vals(re), R.errs(re))
    assert ok.mean() > 0.9
    rpdf = _ratio(pdf, rp.v, rp.e)[ok]
    rev = _ratio(ev, R.vals(re), R.errs(re))[ok]
    print(f"oracle vs float64 reference over {ok.sum()} cases: max |err| / (2^-23 scale): pdf {rpdf.max():.3f}, "
          f"eval {rev.max():.3f}")
    assert rpdf.max() <= C_BOUND and rev.max() <= C_BOUND
    # where the reference is finite with a meaningful bound, so is the oracle
    meaningful = ok & (rp.e * EPS < 0.5 * np.abs(rp.v))
    assert np.isfinite(pdf[meaningful]).all()


def test_reference_sample_states_the_oracle_formulas(orc, grid):
    """disneySample with the oracle's own LCG draws, replayed into the reference."""
    params, base, N, V, L, kind = grid
    b = orc.backend()
    f3 = C.c_float * 3
    n = 1500
    draws = np.zeros((n, 4), np.float32)
    Lo, Ho = np.empty((n, 3), np.float32), np.empty((n, 3), np.float32)
    lo, ho = f3(), f3()
    V1 = np.where((dot32(N, V) > 0)[:, None], V, -V)[:n]
    for i in range(n):
        s = C.c_int32(0x5EED + 7919 * i)
        t = C.c_int32(s.value)
        draws[i, :3] = [b.rand(C.byref(t)) for _ in range(3)]
        b.disney_sample(C.byref(s), C.byref(params[i]), f3(*N[i]), f3(*V1[i]), lo, ho)
        Lo[i], Ho[i] = lo[:], ho[:]
        assert s.value == t.value                     # three draws
    RL, RH, _ = R.sample(params[:n], N[:n], V1, draws, R.IEEE)
    ok = _finite(R.vals(RL), R.errs(RL), R.vals(RH), R.errs(RH))
    rl = _ratio(Lo, R.vals(RL), R.errs(RL))[ok]
    rh = _ratio(Ho, R.vals(RH), R.errs(RH))[ok]
    print(f"oracle disneySample vs reference: max ratio L {rl.max():.3f}, H {rh.max():.3f}")
    assert ok.mean() > 0.99 and rl.max() <= C_BOUND and rh.max() <= C_BOUND


def test_reference_refraction_states_the_oracle_formulas(orc):
    d, Ns, ior = _refraction_cases()
    b = orc.backend()
    f3 = C.c_float * 3
    out = f3()
    r32 = np.empty_like(d)
    fr = np.ones(len(d), np.float32)
    tir = np.empty(len(d), bool)
    for i in range(len(d)):   # the oracle's dielectric(): orientation, refract(), fresnel()
        cosI = -dot32(d[i:i + 1], Ns[i:i + 1])[0]
        nrm, ri = (Ns[i], ior[i]) if cosI > 0 else (-Ns[i], np.float32(1) / ior[i])
        tir[i] = not b.refract(f3(*d[i]), f3(*nrm), float(ri), out)
        r32[i] = out[:]
        if not tir[i]:
            fr[i] = b.fresnel(float(abs(cosI)), float(-dot32(nrm[None], r32[i:i + 1])[0]), float(ri))
    rr, k, rf = R.refract_fresnel(d, Ns, ior)
    clear = np.abs(k.v) > C_BOUND * EPS * k.e
    assert (tir[clear] == (k.v[clear] < 0)).all()
    m = clear & ~tir
    ratio = _ratio(r32[m], R.vals(rr)[m], R.errs(rr)[m])
    rfr = _ratio(fr[m], rf.v[m], rf.e[m])
    print(f"oracle refract vs reference: max ratio {ratio.max():.3f}, fresnel {rfr.max():.3f}, TIR {tir.sum()} of {len(d)}")
    assert ratio.max() <= C_BOUND and rfr.max() <= C_BOUND


def _refraction_cases(seed=5, n=4000):
    rng = np.random.default_rng(seed)
    Ns = _unit(rng.normal(size=(n, 3)))
    d = _unit(rng.normal(size=(n, 3)))
    d[:200] = _unit(_direction(Ns[:200].astype(np.float64), rng.choice([1e-7, 1e-4, 0.999, 1.0], 200), rng)) * -1
    ior = rng.choice([1.45, 1.0, 1.5, 2.4, 1.0001], n).astype(np.float32)
    # grazing from inside near the critical angle of 1.45
    crit = np.sqrt(1 - 1 / 1.45 ** 2)
    d[200:400] = _unit(_direction(Ns[200:400].astype(np.float64), crit + rng.normal(scale=1e-6, size=200), rng))
    ior[200:400] = 1.45
    return d, Ns, ior


# ---------------------------------------------------------------------------------------------- the device probe
class Probe:
    def __init__(self, path):
        self.lib = C.CDLL(path)
        fp, ip = C.POINTER(C.c_float), C.POINTER(C.c_int)
        self.lib.probe_disney_hit_eval.argtypes = [C.c_int, C.c_int, C.c_void_p] + [fp] * 9
        self.lib.probe_disney_sample.argtypes = [C.c_int, C.c_void_p, fp, fp, fp, fp, fp, ip]
        self.lib.probe_refract_fresnel.argtypes = [C.c_int, fp, fp, fp, fp, ip, fp]
        self.lib.probe_libm.argtypes = [C.c_int, fp, fp, fp]

    @staticmethod
    def _p(a):
        return None if a is None else a.ctypes.data_as(C.POINTER(C.c_int if a.dtype == np.int32 else C.c_float))

    def _call(self, fn, *args):
        rc = fn(*[self._p(a) if isinstance(a, np.ndarray) or a is None else a for a in args])
        assert rc == 0, f"CUDA error {rc}"

    def hit_eval(self, fast, params, base, N, V, L, H=None):
        n = len(N)
        c = lambda a: np.ascontiguousarray(a, np.float32)
        pdf, dr, ev, h = np.empty(n, np.float32), np.empty(n, np.float32), np.empty((n, 3), np.float32), np.empty((n, 3), np.float32)
        self._call(self.lib.probe_disney_hit_eval, int(fast), n, C.cast(params, C.c_void_p), c(base), c(N), c(V), c(L),
                   None if H is None else c(H), pdf, dr, ev, h)
        return pdf, dr, ev, h

    def sample(self, params, N, V, draws):
        n = len(N)
        c = lambda a: np.ascontiguousarray(a, np.float32)
        L, H, used = np.empty((n, 3), np.float32), np.empty((n, 3), np.float32), np.empty(n, np.int32)
        self._call(self.lib.probe_disney_sample, n, C.cast(params, C.c_void_p), c(N), c(V), c(draws), L, H, used)
        return L, H, used

    def refract_fresnel(self, d, Ns, ior):
        n = len(d)
        c = lambda a: np.ascontiguousarray(a, np.float32)
        r, tir, fr = np.empty((n, 3), np.float32), np.empty(n, np.int32), np.empty(n, np.float32)
        self._call(self.lib.probe_refract_fresnel, n, c(d), c(Ns), c(ior), r, tir, fr)
        return r, tir.astype(bool), fr

    def libm(self, x):
        x = np.ascontiguousarray(x, np.float32).ravel()
        p, lg = np.empty_like(x), np.empty_like(x)
        self._call(self.lib.probe_libm, len(x), x, p, lg)
        return p, lg


@pytest.fixture(scope="module")
def probe():
    subprocess.check_call(["make", "-C", ROOT, "probe"], stdout=subprocess.DEVNULL)
    return Probe(PROBE_LIB)


def _glibc():
    m = C.CDLL("libm.so.6")
    m.powf.restype = m.logf.restype = C.c_float
    m.powf.argtypes, m.logf.argtypes = [C.c_float, C.c_float], [C.c_float]
    return m


def _clearcoat_a2(params):
    g = np.array([p.clearcoatGloss for p in params], np.float32)
    a = np.float32(0.1) + g * (np.float32(0.001) - np.float32(0.1))
    return a * a


@pytest.mark.gpu
def test_ieee_mode_is_the_oracle_bit_for_bit(orc, probe, grid):
    """DisneyHit<false> (hoisted setView terms, GTR1 shared by pdf and eval) against the oracle's disneyPdf /
    disneyEval given the same float32 H: equal bits wherever CUDA's and glibc's powf(c, 2.2f) and logf(a^2) agree,
    within the bound elsewhere."""
    params, base, N, V, L, kind = grid
    pdf, dr, ev, H = probe.hit_eval(False, params, base, N, V, L)
    assert np.array_equal(H, normalize32(L + V), equal_nan=True)    # bnormalize<false> is the IEEE normalize
    opdf, oev = _oracle_pdf_eval(orc, params, base, N, V, L, H)
    m = _glibc()
    a2 = _clearcoat_a2(params)
    cpow, clog = probe.libm(np.concatenate([base.ravel(), a2]))
    gpow = np.array([m.powf(float(x), 2.2) for x in base.ravel()], np.float32)
    glog = np.array([m.logf(float(x)) for x in a2], np.float32)
    same_pow = np.all((cpow[:base.size] == gpow).reshape(-1, 3), axis=1)
    same_log = clog[base.size:] == glog
    same = same_pow & same_log
    print(f"libm inputs equal on {same.sum()} of {len(N)} cases (powf {same_pow.mean():.3f}, logf {same_log.mean():.3f})")
    assert same.sum() > 0.3 * len(N)
    bits = lambda a: np.asarray(a, np.float32).view(np.int32)
    # NaN payloads aside, equal bits
    eq_pdf = (bits(pdf) == bits(opdf)) | (np.isnan(pdf) & np.isnan(opdf))
    eq_ev = np.all((bits(ev) == bits(oev)) | (np.isnan(ev) & np.isnan(oev)), axis=1)
    assert eq_pdf[same_log].all(), np.flatnonzero(~eq_pdf & same_log)[:10]
    assert eq_ev[same].all(), np.flatnonzero(~eq_ev & same)[:10]
    rp, _, re = R.pdf_eval(params, base, N, V, L, H, R.IEEE)
    ok = ~same & _finite(rp.e, R.errs(re), opdf, oev)
    rpdf = np.abs(pdf[ok].astype(float) - opdf[ok]) / (EPS * rp.e[ok] + 1e-300)
    rev = np.abs(ev[ok].astype(float) - oev[ok]) / (EPS * R.errs(re)[ok] + 1e-300)
    print(f"libm-different cases {ok.sum()}: max |gpu - oracle| / (2^-23 scale) pdf {rpdf.max(initial=0):.3f} "
          f"eval {rev.max(initial=0):.3f}")
    assert rpdf.max(initial=0) <= 2 * C_BOUND and rev.max(initial=0) <= 2 * C_BOUND


def _mode_errors(probe, grid, fast, H=None):
    params, base, N, V, L, kind = grid
    pdf, dr, ev, Hu = probe.hit_eval(fast, params, base, N, V, L, H)
    rp, rdr, re = R.pdf_eval(params, base, N, V, L, Hu, R.FAST if fast else R.IEEE)
    return dict(pdf=pdf, ev=ev, H=Hu, rp=rp, re=re,
                r_pdf=_ratio(pdf, rp.v, rp.e), r_ev=_ratio(ev, R.vals(re), R.errs(re)).max(axis=1))


@pytest.mark.gpu
@pytest.mark.parametrize("sampled", [False, True], ids=["light_sample", "given_H"])
def test_fast_mode_within_the_instruction_bounds(probe, grid, sampled):
    """DisneyHit<true> (the default: __fdividef, sqrt.approx, rsqrtf, __powf, __logf) against the float64 reference.
    Well-conditioned cases (N.V, N.L, |L.H| >= 1e-3) within the first-order bound built from the documented error of
    each approximate instruction.  Elsewhere (grazing, N.V < 0, L ~ -V): finite on the same cases as the IEEE mode,
    the same sign decision pdf > 0 (it decides whether a ray is spawned), and an error within a small factor of the
    IEEE mode's own error against the reference."""
    params, base, N, V, L, kind = grid
    H = None
    if sampled:    # the sampled-direction form: H given (the IEEE half vector of L and V)
        H = normalize32(L + V)
    f = _mode_errors(probe, grid, True, H)
    i = _mode_errors(probe, grid, False, f["H"])       # the IEEE mode on the fast mode's H
    good = well_conditioned(N, V, L, f["H"]) & _finite(f["rp"].v, f["rp"].e, R.vals(f["re"]), R.errs(f["re"]))
    fin = _finite(f["rp"].e, R.errs(f["re"]))
    assert good.sum() > 0.5 * len(N)
    wp, we = f["r_pdf"][good].max(), f["r_ev"][good].max()
    print(f"fast mode, well-conditioned ({good.sum()} cases): max |gpu - ref64| / (2^-23 bound_fast): pdf {wp:.3f} "
          f"eval {we:.3f}")
    assert wp <= C_BOUND and we <= C_BOUND
    ill = ~good
    assert np.array_equal(np.isfinite(f["pdf"][ill]), np.isfinite(i["pdf"][ill]))
    assert np.array_equal(np.isfinite(f["ev"][ill]).all(axis=1), np.isfinite(i["ev"][ill]).all(axis=1))
    assert np.array_equal(f["pdf"][ill] > 0, i["pdf"][ill] > 0)
    sc_p, sc_e = f["rp"].e, R.errs(f["re"])
    ok = ill & fin & _finite(f["pdf"], f["ev"])
    fe = lambda d: (np.abs(d["pdf"][ok] - d["rp"].v[ok]) / (EPS * sc_p[ok]),
                    (np.abs(d["ev"][ok] - R.vals(d["re"])[ok]) / (EPS * sc_e[ok])).max(axis=1))
    fp_, fe_ = fe(f)
    ip_, ie_ = fe(i)
    print(f"ill-conditioned ({ok.sum()} finite cases): max error / (2^-23 fast bound): fast pdf {fp_.max():.3f} "
          f"eval {fe_.max():.3f}; IEEE pdf {ip_.max():.3f} eval {ie_.max():.3f}")
    for name in ("backside", "opposite", "graze_v", "graze_both"):
        k = kind[ok] == name
        if k.any():
            print(f"  {name}: fast eval {fe_[k].max():.3f}  IEEE eval {ie_[k].max():.3f}")
    assert fp_.max() <= max(4 * ip_.max(), C_BOUND) and fe_.max() <= max(4 * ie_.max(), C_BOUND)


@pytest.mark.gpu
def test_disney_sample_follows_the_reference(probe, grid):
    """disneySample fed chosen draws: three draws on both branches, the branch r0 < diffuseRatio decided in float32
    (r0 == diffuseRatio included), L and H within the conditioning bound per component (the xi -> 1 and u1 -> 1
    corners, where cos(theta) and the hemisphere's z are square roots of cancellations, are bounded, not excluded)."""
    params, base, N, V, L, kind = grid
    n = len(N)
    rng = np.random.default_rng(17)
    draws = (rng.integers(0, 1 << 24, (n, 4)) / float(1 << 24)).astype(np.float32)
    metallic = np.array([p.metallic for p in params], np.float32)
    ratio = np.float32(0.5) * (np.float32(1) - metallic)
    tie = rng.random(n) < 0.1
    draws[tie, 0] = ratio[tie]                                # r0 == diffuseRatio: the specular branch
    edge = rng.random(n) < 0.1
    draws[edge, 2] = np.float32(1 - 2 ** -24)                 # xi, u2 at the top of the generator's range
    draws[rng.random(n) < 0.05, 1] = np.float32(1 - 2 ** -24)
    draws[rng.random(n) < 0.05, 2] = 0
    V1 = np.where((dot32(N, V) > 0)[:, None], V, -V)
    Lg, Hg, used = probe.sample(params, N, V1, draws)
    assert (used == 3).all()
    RL, RH, diffuse = R.sample(params, N, V1, draws, R.IEEE)
    assert (diffuse == (draws[:, 0] < ratio)).all() and not diffuse[tie].any() and diffuse.any() and (~diffuse).any()
    ok = _finite(R.vals(RL), R.errs(RL), R.vals(RH), R.errs(RH))
    assert ok.mean() > 0.99
    rl = _ratio(Lg, R.vals(RL), R.errs(RL))[ok]
    rh = _ratio(Hg, R.vals(RH), R.errs(RH))[ok]
    print(f"disneySample vs reference: max ratio L {rl.max():.3f}, H {rh.max():.3f}")
    assert rl.max() <= C_BOUND and rh.max() <= C_BOUND
    # the branch is visible in the result: diffuse samples are not reflections about H
    spec = ok & ~diffuse
    refl = 2 * dot32(V1[spec], Hg[spec])[:, None] * Hg[spec] - V1[spec]
    assert np.allclose(normalize32(refl), Lg[spec], atol=1e-5)


@pytest.mark.gpu
def test_refract_and_fresnel_follow_the_reference(probe):
    """refract3 + fresnelDielectric as k_shade_dielectric uses them: the TIR decision equals float64's except within the
    rounding of k = 0, the refracted direction and the reflection probability within the bound."""
    d, Ns, ior = _refraction_cases()
    r, tir, fr = probe.refract_fresnel(d, Ns, ior)
    rr, k, rf = R.refract_fresnel(d, Ns, ior)
    clear = np.abs(k.v) > C_BOUND * EPS * k.e
    assert (tir[clear] == (k.v[clear] < 0)).all()
    assert (fr[tir] == 1).all() and (r[tir] == 0).all()
    m = clear & ~tir
    rd = _ratio(r[m], R.vals(rr)[m], R.errs(rr)[m])
    rp = _ratio(fr[m], rf.v[m], rf.e[m])
    print(f"refract3 vs reference: max ratio {rd.max():.3f}; fresnel {rp.max():.3f}; TIR {tir.sum()} "
          f"ambiguous {(~clear).sum()}")
    assert rd.max() <= C_BOUND and rp.max() <= C_BOUND


# ---------------------------------------------------------------------------------------------- through the product
def _textures():
    rng = np.random.default_rng(3)

    def rgba(rgb):
        t = np.ones(rgb.shape[:2] + (4,), np.float32)
        t[..., :3] = rgb
        return t
    checker = np.zeros((2, 2, 3), np.float32)
    checker[0, 0] = checker[1, 1] = 1
    return {"1x1": rgba(rng.random((1, 1, 3))), "1x7": rgba(rng.random((1, 7, 3))), "7x1": rgba(rng.random((7, 1, 3))),
            "3x5": rgba(rng.random((3, 5, 3))), "checker2x2": rgba(checker), "random64": rgba(rng.random((64, 64, 3)))}


def _filter_bound(tex):
    """Per channel, the largest error of a bilinear filter whose two weights are each off by less than 1/256 (8
    fractional bits): the largest step between texels the REPEAT filter blends along u, plus the same along v."""
    rgb = tex[..., :3].astype(np.float64)
    du = np.abs(rgb - np.roll(rgb, 1, axis=1)).max(axis=(0, 1))
    dv = np.abs(rgb - np.roll(rgb, 1, axis=0)).max(axis=(0, 1))
    return (du + dv) / 256 + 2.0 ** -20


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(_textures()))
def test_texture_filter_per_pixel(host, orc, gpu_backend, name):
    """A Disney GLASS quad that fills the frame, tinted by a texture over several periods of u and v, negative values
    included, in front of a white background: every sample is tint(u, v) exactly (both children miss), and uv is the
    oracle's bit for bit (IEEE camera and triangle arithmetic).  So each pixel of each 1-spp launch differs from the
    oracle's float filter only by the hardware filter's 8-bit fractional weights (_filter_bound).  Wrong wrap mode, row
    order or texel centre shows in whole bands of pixels."""
    tex = _textures()[name]
    w, h = 96, 64
    bound = _filter_bound(tex)
    verts = np.array([[-2, -2, 0], [2, -2, 0], [2, 2, 0], [-2, 2, 0]], np.float32)
    uv = np.array([[-1.25, -0.5], [2.75, -0.5], [2.75, 1.5], [-1.25, 1.5]], np.float32)
    faces = np.array([[0, 1, 2], [0, 2, 3]], np.int32)
    worst = 0.0
    for seed in (1, 2, 3):
        imgs = []
        for ctx in (orc.context(), gpu_backend.context(0)):
            ctx.set_globals(w, h, 2, absorb=(0, 0, 0), bg=(1, 1, 1))
            ctx.set_camera(host.set_cam_params((0, 0, 2.5), (0, 0, 0), (0, 1, 0), 60, w / h, 0.0, 1.0))
            tid = ctx.add_texture(tex)
            mat = host.init_disney_params()
            mat.albedoID, mat.brdfType = tid, S.GLASS
            ctx.add_mesh(verts, faces, S.MAT_DISNEY, mat, texcoords=uv, t_idx=faces)
            ctx.build_accel()
            ctx.render(1, seed)
            imgs.append(ctx.read_accum())
        o, g = imgs
        d = np.abs(g.astype(np.float64) - o)
        assert (d <= bound).all(), (name, seed, d.max(axis=(0, 1)), bound, int((d > bound).any(axis=-1).sum()))
        worst = max(worst, float((d / bound).max()))
    print(f"texture {name}: max |gpu - oracle| per pixel = {worst:.3f} of the bound {bound}")


def _disney_row():
    """Analytic spheres across the parameter corners, left to right."""
    def disney(**kw):
        d = host_disney()
        for k, v in kw.items():
            setattr(d, k, S.float3(*v) if k == "color" else v)
        return d
    return [disney(color=(0.9, 0.7, 0.3), metallic=1.0, roughness=0.001),
            disney(color=(0.2, 0.5, 0.9), roughness=1.0, subsurface=1.0, sheen=1.0, sheenTint=1.0),
            disney(color=(0.8, 0.1, 0.1), clearcoat=1.0, clearcoatGloss=1.0, roughness=0.5),
            disney(color=(0.6, 0.6, 0.6), metallic=0.7, anisotropic=1.0, roughness=0.3, specularTint=1.0),
            disney(color=(1e-6, 1e-6, 1e-6), specular=1.0, roughness=0.0316),
            disney(color=(0.0, 1.0, 0.0), metallic=0.0, roughness=1e-4, clearcoat=0.5, clearcoatGloss=0.0)]


def host_disney():
    from minimaloptix_b200 import host
    d = host.init_disney_params()
    d.brdfType = S.NORMAL
    return d


@pytest.mark.gpu
def test_direct_light_per_pixel(host, orc, gpu_backend, monkeypatch):
    """Depth 1, no background, no absorption: a pixel is the Disney light loop of k_shade_disney (light pdf,
    powerHeuristic, 1 / max(0.001, lightPdf)) plus the sampled direction when it reaches the light.  Per pixel at 1 spp
    against the oracle: the IEEE mode within a few ulps (what is left is libm), the fast mode within the bound of the
    approximate instructions, the same non-finite samples.  Emission is kept low so that most samples stay below the
    [0, 1] clamp of k_accumulate."""
    w, h = 192, 48
    light = S.LightParams()
    light.position, light.u, light.v, light.normal = S.float3(-3, 2.5, -1), S.float3(6, 0, 0), S.float3(0, 0, 2), S.float3(0, -1, 0)
    light.area, light.emission, light.shape = 12.0, S.float3(0.3, 0.3, 0.3), S.QUAD
    row = _disney_row()

    def render(ctx, seed):
        ctx.set_globals(w, h, 1, absorb=(0, 0, 0), bg=(0, 0, 0))
        ctx.set_camera(host.set_cam_params((0, 0.3, 6), (0, 0, 0), (0, 1, 0), 22, w / h, 0.0, 1.0))
        for k, d in enumerate(row):
            ctx.add_sphere(S.SphereParams(0.45, S.float3(-2.5 + k, 0, 0), S.float3()), S.MAT_DISNEY, d)
        ctx.add_quad(host.set_quad_params((-3, 2.5, -1), (6, 0, 0), (0, 0, 2)), S.MAT_LIGHT, light)
        ctx.set_lights([light])
        ctx.build_accel()
        ctx.render(1, seed)
        return ctx.read_accum().astype(np.float64), ctx.stats()["nonfinite_samples"]

    for seed in (5, 6):
        o, onf = render(orc.context(), seed)
        hit = o.max(axis=-1) > 0
        unclamped = float(np.mean(o[hit].max(axis=-1) < 1))
        # IEEE mode: libm ulps only.  Fast mode: the light loop's half vector is bnormalize<true> (rsqrtf, 2 ulp), and at
        # the GTR2 peak of roughness 0.001 and below, t = a^2 + (1 - N.H^2) turns those 2 ulps of N.H into relative
        # changes of the lobe up to ~1e-3 (measured 4.2e-4 on this scene); the instruction bounds themselves are held
        # value by value in test_fast_mode_within_the_instruction_bounds.
        for mode, rel in (("1", 8 * EPS), ("0", 2.0 ** -10)):
            monkeypatch.setenv("MOX_BRDF_IEEE", mode)
            g, gnf = render(gpu_backend.context(0), seed)
            assert gnf == onf
            d = np.abs(g - o)
            over = (d > rel * o + 2.0 ** -20).any(axis=-1)
            print(f"seed {seed} {'IEEE' if mode == '1' else 'fast'}: max rel {float((d / np.maximum(o, 1e-30)).max()):.3e}, "
                  f"pixels over {int(over.sum())} of {int(hit.sum())} lit, unclamped {unclamped:.3f}")
            assert hit.sum() > 500 and unclamped > 0.5
            assert over.sum() <= 2     # a sampled direction that grazes the light's edge may flip on a libm ulp
