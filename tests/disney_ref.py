"""Float64 restatement of the Disney BRDF (disney.h:9-91), the dielectric refraction / Fresnel step
(utils_device.h:63-67, SDK refract) and their helpers, vectorised over cases, as the reference to hold
the float32 implementations to: the CUDA code of shading.cuh and the CPU oracle's oracle/device_spec.h.

The reference's quirks are kept, as device_spec.h states them: sampling uses alpha = roughness while
eval uses roughness^2; no cosine factor; srgb2lin (powf(c, 2.2f)) on the base colour; Cdlum = 0 gives
Ctint = 1; the 0.001 clamps; the SDK Onb's branch on |n.x| > |n.z|.  Every literal is the float32
literal of the source (0.08f, MOX_PI_F, ...), every input is a float32 value; only the arithmetic is
float64 (exact to ~1e-16, far below what is measured).

Alongside each value the evaluation carries a first-order bound on the error of a float32
evaluation that performs the same operations in the same order (the "conditioning scale").  Each
operation contributes its own rounding budget times the magnitude of its result, and the input
errors are propagated through the derivative.  A sum that cancels therefore carries the error of
its terms, not of its small result: that is what makes grazing angles, the GTR peaks and the
N.V < 0 Smith term testable at all.  Bounds are in units of 2^-23 (one ulp of 1.0), absolute.

Budgets (ulps of the operation's result), from the CUDA C++ Programming Guide's accuracy tables and
the PTX ISA for the approximate instructions:
  IEEE + - * / sqrt: 0.5 (correctly rounded); powf 4; logf 1; sinf / cosf 2 (also cover glibc);
  fast mode (shading.cuh, F = true):
    __fdividef 2; rsqrtf 2; sqrt.approx.f32 2 (conservative: PTX states ~1 ulp);
    __logf 3 outside [0.5, 2] (absolute 2^-21.41 inside);
    __powf = ex2.approx(y * lg2.approx(x)): 2 ulps of ex2, plus ln2 * |y| times the error of lg2
    (2^-22 absolute in [0.5, 2], 2 ulps elsewhere), plus ln2 * |y lg2 x| * 0.5 for the product.
"""
import numpy as np

F64 = np.float64
U = 0.5                      # one correctly rounded operation, in ulps of its result
EPS = 2.0 ** -23
PI_F = F64(np.float32(np.pi))  # MOX_PI_F / M_PIf: the float32 literal of the source

IEEE = dict(div=U, sqrt=U, rsqrt=None, pow=4.0, log=1.0, sincos=2.0)
FAST = dict(div=2.0, sqrt=2.0, rsqrt=2.0, pow="approx", log="approx", sincos=2.0)


def f32(c):
    return F64(np.float32(c))


class X:
    """A float64 value and a bound on the absolute error (units of 2^-23) of its float32 evaluation."""
    __slots__ = ("v", "e")

    def __init__(self, v, e=None):
        self.v = np.asarray(v, dtype=F64)
        self.e = np.zeros_like(self.v) if e is None else np.broadcast_to(np.asarray(e, F64), self.v.shape).copy()

    @staticmethod
    def rounded(v, e, budget=U):
        return X(v, e + budget * np.abs(v))

    def __add__(a, b):
        b = cx(b)
        return X.rounded(a.v + b.v, a.e + b.e)
    __radd__ = __add__

    def __sub__(a, b):
        b = cx(b)
        return X.rounded(a.v - b.v, a.e + b.e)

    def __rsub__(a, b):
        return cx(b) - a

    def __neg__(a):
        return X(-a.v, a.e)

    def __mul__(a, b):
        b = cx(b)
        # with the second-order term: a square of a value smaller than its own error (rs^2 of Fresnel at ior = 1);
        # 0 * an unbounded error is NaN: no bound
        with np.errstate(invalid="ignore"):
            return X.rounded(a.v * b.v, np.abs(b.v) * a.e + np.abs(a.v) * b.e + EPS * a.e * b.e)
    __rmul__ = __mul__

    def __truediv__(a, b):
        return div(a, b, U)

    def __rtruediv__(a, b):
        return div(cx(b), a, U)


def cx(c):
    """A float literal of the source: rounded to float32, exact."""
    return c if isinstance(c, X) else X(f32(c))


def where(cond, a, b):
    a, b = cx(a), cx(b)
    return X(np.where(cond, a.v, b.v), np.where(cond, a.e, b.e))


def div(a, b, budget):
    a, b = cx(a), cx(b)
    with np.errstate(divide="ignore", invalid="ignore"):
        v = a.v / b.v
        e = a.e / np.abs(b.v) + np.abs(v / b.v) * b.e
    # a divisor whose error interval holds 0 bounds nothing (the float32 quotient may be inf, and inf * 0 = NaN)
    return X.rounded(v, np.where(np.abs(b.v) <= EPS * b.e, np.inf, e), budget)


def sqrt(a, budget=U):
    with np.errstate(divide="ignore", invalid="ignore"):
        v = np.sqrt(a.v)
        # first order, capped by |sqrt(x + d) - sqrt(x)| <= sqrt(|d|) (the bound that holds at x -> 0)
        e = np.minimum(a.e / (2 * v), np.sqrt(a.e / EPS))
    return X.rounded(v, np.where(a.e == 0, 0.0, e), budget)


def fabs(a):
    return X(np.abs(a.v), a.e)


def fmax(c, a):
    c, a = cx(c), cx(a)
    return where(a.v > c.v, a, c)       # fmaxf(c, a): a where a > c


def clamp(a, lo, hi):
    return fmax(lo, where(a.v < f32(hi), a, hi))


def sin_cos(a, budget):
    s, c = np.sin(a.v), np.cos(a.v)
    return X.rounded(s, np.abs(c) * a.e, budget), X.rounded(c, np.abs(s) * a.e, budget)


def powf(x, y, m):
    """powf(x, y) (IEEE mode, the oracle) or __powf (fast mode) for a float32 literal y."""
    y = f32(y)
    with np.errstate(divide="ignore", invalid="ignore"):
        v = np.power(x.v, y)
        prop = np.where(x.v > 0, np.abs(y * v / np.where(x.v > 0, x.v, 1.0)) * x.e, 0.0)
        if m["pow"] == "approx":
            lg = np.abs(np.log2(np.where(x.v > 0, x.v, 1.0)))
            lg2_err = np.where((x.v >= 0.5) & (x.v <= 2.0), 2.0 ** -22 / EPS, 2.0 * lg)   # ulps of 1.0
            budget = 2.0 + np.log(2.0) * (np.abs(y) * lg2_err + 0.5 * np.abs(y) * lg)
        else:
            budget = m["pow"]
    return X(v, prop + budget * np.abs(v))


def logf(x, m):
    with np.errstate(divide="ignore", invalid="ignore"):
        v = np.log(x.v)
        prop = x.e / np.abs(x.v)
    if m["log"] == "approx":
        inside = (x.v >= 0.5) & (x.v <= 2.0)
        return X(v, prop + np.where(inside, 2.0 ** -21.41 / EPS, 3.0 * np.abs(v)))
    return X(v, prop + m["log"] * np.abs(v))


# ---------------------------------------------------------------- vectors: lists of three X
def v3(a):
    a = np.asarray(a, dtype=np.float32).astype(F64)
    return [X(a[..., 0]), X(a[..., 1]), X(a[..., 2])]


def vals(v):
    return np.stack([c.v for c in v], axis=-1)


def errs(v):
    return np.stack([c.e for c in v], axis=-1)


def add(a, b): return [x + y for x, y in zip(a, b)]
def sub(a, b): return [x - y for x, y in zip(a, b)]
def smul(s, a): return [s * x for x in a]
def dot(a, b): return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]
def cross(a, b): return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]
def lerp(a, b, t): return a + t * (b - a)
def lerp3(a, b, t): return add(a, smul(t, sub(b, a)))
def const3(c): return [cx(c), cx(c), cx(c)]


def normalize(v):
    """IEEE: v * (1 / sqrt(dot(v, v))), the SDK's operator order."""
    inv = 1.0 / sqrt(dot(v, v))
    return smul(inv, v)


def bnormalize(v, m):
    if m["rsqrt"] is None:
        return normalize(v)
    d = dot(v, v)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = 1.0 / np.sqrt(d.v)
        e = np.abs(0.5 * r / d.v) * d.e
    return smul(X.rounded(r, e, m["rsqrt"]), v)


def onb(N):
    """SDK Onb: (tangent, binormal); branch on |n.x| > |n.z| of the float32 normal."""
    br = np.abs(N[0].v) > np.abs(N[2].v)
    b = [where(br, -N[1], X(0.0)), where(br, N[0], -N[2]), where(br, X(0.0), N[1])]
    b = normalize(b)
    return cross(b, N), b


def schlick(u):
    m = clamp(1.0 - u, 0.0, 1.0)
    m2 = m * m
    return m2 * m2 * m


def smith(NdotV, alphaG, m):
    a, b = alphaG * alphaG, NdotV * NdotV
    return div(1.0, NdotV + sqrt(a + b - a * b, m["sqrt"]), m["div"])


def smith_aniso(NdotV, VdotX, VdotY, ax, ay, m):
    s = (VdotX * ax) * (VdotX * ax) + (VdotY * ay) * (VdotY * ay) + NdotV * NdotV
    return div(1.0, NdotV + sqrt(s, m["sqrt"]), m["div"])


def params(mp):
    """DisneyParams rows (a ctypes array or a list) -> dict of float64 arrays of the float32 fields."""
    names = ("metallic", "subsurface", "specular", "roughness", "specularTint", "anisotropic", "sheen", "sheenTint",
             "clearcoat", "clearcoatGloss")
    return {k: X(np.array([getattr(p, k) for p in mp], np.float32).astype(F64)) for k in names}


def pdf_eval(mp, base, N, V, L, H, m=IEEE):
    """disneyPdf and disneyEval (disney.h:32-91) for per-case params and float32 vectors (n x 3).
    Returns (pdf, dr, eval) as X / list of X; dr = GTR1(|N.H|, clearcoatAlpha) as shared by pdf and eval."""
    p = params(mp)
    N, V, L, H = v3(N), v3(V), v3(L), v3(H)
    tangent, _ = onb(N)
    Cdlin = [powf(c, 2.2, m) for c in v3(base)]
    Cdlum = dot(Cdlin, [cx(0.3), cx(0.6), cx(0.1)])
    pos = Cdlum.v > 0
    inv = 1.0 / where(pos, Cdlum, 1.0)
    Ctint = [where(pos, c * inv, 1.0) for c in Cdlin]
    Cspec0 = lerp3(smul(p["specular"] * 0.08, lerp3(const3(1.0), Ctint, p["specularTint"])), Cdlin, p["metallic"])
    Csheen = lerp3(const3(1.0), Ctint, p["sheenTint"])
    aspect = sqrt(1.0 - p["anisotropic"] * 0.9)
    r2 = p["roughness"] * p["roughness"]
    ax = fmax(0.001, r2 / aspect)
    ay = fmax(0.001, r2 * aspect)
    Xv = bnormalize(tangent, m)
    Yv = bnormalize(cross(N, Xv), m)
    ccAlpha = lerp(cx(0.1), cx(0.001), p["clearcoatGloss"])
    specAlpha = fmax(0.001, p["roughness"])
    diffuseRatio = 0.5 * (1.0 - p["metallic"])
    pdfRatio = 1.0 / (1.0 + p["clearcoat"])

    NdotV, NdotL, NdotH, LdotH = dot(N, V), dot(N, L), dot(N, H), dot(L, H)
    a2 = ccAlpha * ccAlpha

    def gtr1(c):
        t = 1.0 + (a2 - 1.0) * c * c
        return div(a2 - 1.0, (PI_F * logf(a2, m)) * t, m["div"])

    def gtr2(c, a):
        aa = a * a
        t = 1.0 + (aa - 1.0) * c * c
        return div(aa, PI_F * t * t, m["div"])

    cosTheta = fabs(NdotH)
    dr = gtr1(cosTheta)
    pdfH = lerp(dr * cosTheta, gtr2(cosTheta, specAlpha) * cosTheta, pdfRatio)
    pdfL = div(pdfH, 4.0 * fabs(LdotH), m["div"])
    pdfDiff = div(fabs(NdotL), PI_F, m["div"])
    pdf = diffuseRatio * pdfDiff + (1.0 - diffuseRatio) * pdfL

    FL, FV = schlick(NdotL), schlick(NdotV)
    Fd90 = 0.5 + 2.0 * LdotH * LdotH * p["roughness"]
    Fd = lerp(cx(1.0), Fd90, FL) * lerp(cx(1.0), Fd90, FV)
    Fss90 = LdotH * LdotH * p["roughness"]
    Fss = lerp(cx(1.0), Fss90, FL) * lerp(cx(1.0), Fss90, FV)
    ss = 1.25 * (Fss * (div(1.0, NdotL + NdotV, m["div"]) - 0.5) + 0.5)
    hx, hy = div(dot(H, Xv), ax, m["div"]), div(dot(H, Yv), ay, m["div"])
    s = hx * hx + hy * hy + NdotH * NdotH
    Ds = div(1.0, (PI_F * ax * ay) * (s * s), m["div"])
    FH = schlick(LdotH)
    Fs = lerp3(Cspec0, const3(1.0), FH)
    Gs = smith_aniso(NdotL, dot(L, Xv), dot(L, Yv), ax, ay, m) * smith_aniso(NdotV, dot(V, Xv), dot(V, Yv), ax, ay, m)
    Fsheen = smul(FH * p["sheen"], Csheen)
    Fr = lerp(cx(0.04), cx(1.0), FH)
    Gr = smith(NdotL, 0.25, m) * smith(NdotV, 0.25, m)
    # the source's order: ((1/pi * lerp * Cdlin + Fsheen) * (1 - metallic) + Gs * Fs * Ds) + 0.25 * cc * Gr * Fr * Dr
    diffuse = smul((1.0 / PI_F) * lerp(Fd, ss, p["subsurface"]), Cdlin)
    spec = [Gs * c * Ds for c in Fs]
    base_t = [(d + sh) * (1.0 - p["metallic"]) for d, sh in zip(diffuse, Fsheen)]
    cc = 0.25 * p["clearcoat"] * Gr * Fr * gtr1(NdotH)
    brdf = [b + s_ + cc for b, s_ in zip(base_t, spec)]
    return pdf, dr, brdf


def sample(mp, N, V, draws, m=IEEE):
    """disneySample (disney.h:9-30) fed the float32 draws r0, then (u1, u2) | (phi, xi).
    Returns (L, H, diffuse branch?)."""
    p = params(mp)
    N, V = v3(N), v3(V)
    d = np.asarray(draws, np.float32)
    metallic32 = np.array([q.metallic for q in mp], np.float32)
    diffuseRatio32 = np.float32(0.5) * (np.float32(1.0) - metallic32)
    diffuse = d[:, 0] < diffuseRatio32           # the branch is decided in float32, as on both sides
    tangent, binormal = onb(N)
    r1, r2 = X(d[:, 1].astype(F64)), X(d[:, 2].astype(F64))

    def to_world(px, py, pz):
        return add(add(smul(px, tangent), smul(py, binormal)), smul(pz, N))

    # diffuse: cosine-weighted hemisphere
    r = sqrt(r1)
    phi = (2.0 * PI_F) * r2
    s, c = sin_cos(phi, m["sincos"])
    px, py = r * c, r * s
    pz = sqrt(fmax(0.0, 1.0 - px * px - py * py))
    Ld = normalize(to_world(px, py, pz))
    Hd = normalize(add(Ld, V))
    # specular: GTR2 half vector with alpha = roughness
    a = fmax(0.001, p["roughness"])
    phi = (r1 * 2.0) * PI_F
    xi = r2
    cosT = sqrt((1.0 - xi) / (1.0 + (a * a - 1.0) * xi))
    sinT = sqrt(1.0 - cosT * cosT)
    s, c = sin_cos(phi, m["sincos"])
    Hs = to_world(sinT * c, sinT * s, cosT)
    Ls = normalize(sub(smul(2.0 * dot(V, Hs), Hs), V))
    Hs = normalize(Hs)
    L = [where(diffuse, x, y) for x, y in zip(Ld, Ls)]
    H = [where(diffuse, x, y) for x, y in zip(Hd, Hs)]
    return L, H, diffuse


def refract_fresnel(d, Ns, ior):
    """k_shade_dielectric up to the coin flip: orientation, SDK refract (TIR when k < 0), Fresnel.
    Returns (refracted, k, reflectProb) with k the TIR discriminant; the branch on the sign of the
    incidence cosine is taken from its float32 value (the dot product below is the device's, bit for bit)."""
    d32, n32 = np.asarray(d, np.float32), np.asarray(Ns, np.float32)
    dot32 = (d32[:, 0] * n32[:, 0] + d32[:, 1] * n32[:, 1]) + d32[:, 2] * n32[:, 2]
    outside = -dot32 > 0
    D, Nn = v3(d), v3(Ns)
    ior = X(np.asarray(ior, np.float32).astype(F64))
    cosI = -dot(D, Nn)
    refIdx = where(outside, ior, 1.0 / ior)
    cosI = where(outside, cosI, -cosI)
    normal = [where(outside, c, -c) for c in Nn]
    # refract3 with the oriented normal: dot(i, n) <= 0, so eta = 1 / refIdx
    negNdotV = dot(D, normal)
    eta = 1.0 / refIdx
    k = 1.0 - eta * eta * (1.0 - negNdotV * negNdotV)
    kk = where(k.v >= 0, k, 0.0)
    r = normalize(sub(smul(eta, D), smul(eta * negNdotV + sqrt(kk), normal)))
    cosTt = -dot(normal, r)
    rs = (cosI - cosTt * refIdx) / (cosI + refIdx * cosTt)
    rp = (cosI * refIdx - cosTt) / (cosI * refIdx + cosTt)
    fr = 0.5 * (rs * rs + rp * rp)
    return r, k, fr
