// shading.cuh — device-side material math: dielectric Fresnel, hit-point refinement, the
// microfacet helpers and the Disney BRDF sample / pdf / eval.
// Semantics: MinimalOptiX/utils_device.h:63-185 and disney.h:9-91 (quirks kept: sampling uses
// alpha = roughness while eval uses roughness^2; no cosine factor; srgb2lin on constants).
// FP32 throughout: the reference's stray double literals ("4.0 *", "1.0 /") round to the same
// floats as the single-precision expressions used here.
#pragma once
#include "mox_structs.h"
#include "rng.cuh"

MOX_D float fresnelDielectric(float cosI, float cosT, float ior) {
  float rs = (cosI - cosT * ior) / (cosI + ior * cosT);
  float rp = (cosI * ior - cosT) / (cosI * ior + cosT);
  return 0.5f * (rs * rs + rp * rp);
}

// Integer-ULP offset along the normal, per coordinate.
MOX_D float offsetCoord(float h, float n) {
  const float epsilon = 1.0e-4f;
  if ((__float_as_int(h) & 0x7fffffff) < __float_as_int(epsilon)) return h + epsilon * n;
  return __int_as_float(__float_as_int(h) + (int)(copysignf(8192.0f, h) * n));
}
MOX_D float3 offsetPoint(const float3& p, const float3& n) {
  return mk3(offsetCoord(p.x, n.x), offsetCoord(p.y, n.y), offsetCoord(p.z, n.z));
}
// Re-project the hit onto the triangle plane through p0, then push it to both sides.
MOX_D void refineHitpoint(const float3& hitPoint, const float3& dir, const float3& normal, const float3& p0,
                          float3& back, float3& front) {
  float refinedT = -(dot(normal, hitPoint - p0)) / dot(normal, dir);
  float3 refined = hitPoint + refinedT * dir;
  if (dot(dir, normal) > 0.0f) { back = offsetPoint(refined, normal); front = offsetPoint(refined, -normal); }
  else { back = offsetPoint(refined, -normal); front = offsetPoint(refined, normal); }
}

MOX_D float sqr(float x) { return x * x; }

// Division and square root inside BRDF *values* (pdf, eval, MIS weights): F = true uses the hardware reciprocal /
// square root approximations (MUFU.RCP + one multiply, ~2 ulp) instead of the IEEE sequences (~8 instructions and a
// slow-path branch each; a light sample holds 16 divisions and 4 square roots).  Directions and hit points never go
// through these: they decide which primitive a ray hits and stay IEEE so that ids match the oracle bit for bit.
// Default F = true (shade stage 49.1 -> 41.8 ms per step, images within 1e-5 RMSE of the oracle as before);
// MOX_BRDF_IEEE=1 selects F = false, whose values follow the oracle's operations one for one.
template <bool F> MOX_D float bdiv(float a, float b) { return F ? __fdividef(a, b) : a / b; }
template <bool F> MOX_D float bpow(float x, float y) { return F ? __powf(x, y) : powf(x, y); }   // ex2(y * lg2(x)): NaN for x < 0 like powf
template <bool F> MOX_D float blog(float x) { return F ? __logf(x) : logf(x); }
// normalize for vectors that only enter BRDF values (half vector of a light sample, tangent frame of the anisotropic lobe)
template <bool F> MOX_D float3 bnormalize(const float3& v) { return F ? v * rsqrtf(dot(v, v)) : normalize(v); }
template <bool F> MOX_D float bsqrt(float x) {
  if (!F) return sqrtf(x);
  float r;
  asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

template <bool F> MOX_D float GTR2(float NdotH, float a) {
  float a2 = a * a;
  float t = 1.f + (a2 - 1.f) * NdotH * NdotH;
  return bdiv<F>(a2, MOX_PI_F * t * t);
}
MOX_D float GTR2Aniso(float NdotH, float HdotX, float HdotY, float ax, float ay) {
  return 1 / (MOX_PI_F * ax * ay * sqr(sqr(HdotX / ax) + sqr(HdotY / ay) + NdotH * NdotH));
}
MOX_D float schlickFresnel(float u) {
  float m = clampf(1.f - u, 0.f, 1.f);
  float m2 = m * m;
  return m2 * m2 * m;
}
template <bool F> MOX_D float smithGGgx(float NdotV, float alphaG) {
  float a = alphaG * alphaG, b = NdotV * NdotV;
  return bdiv<F>(1.f, NdotV + bsqrt<F>(a + b - a * b));
}
template <bool F> MOX_D float smithGGgxAniso(float NdotV, float VdotX, float VdotY, float ax, float ay) {
  return bdiv<F>(1.0f, NdotV + bsqrt<F>(sqr(VdotX * ax) + sqr(VdotY * ay) + sqr(NdotV)));
}
template <bool F> MOX_D float powerHeuristic(float a, float b) { float t = a * a; return bdiv<F>(t, b * b + t); }

// disney.h:9-30; draws: lobe, then (u1,u2) | (phi, xi).
template <class R>
MOX_D void disneySample(R& rng, const DisneyParams& mp, const float3& N, float3& L, const float3& V, float3& H) {
  float diffuseRatio = 0.5f * (1.0f - mp.metallic);
  Onb3 onb(N);
  float r0 = rng.rnd();
  if (r0 < diffuseRatio) {
    float u1 = rng.rnd(), u2 = rng.rnd();
    float r = sqrtf(u1), phi = 2.0f * MOX_PI_F * u2;
    float3 p;
    p.x = r * cosf(phi);
    p.y = r * sinf(phi);
    p.z = sqrtf(fmaxf(0.0f, 1.0f - p.x * p.x - p.y * p.y));
    L = normalize(onb.toWorld(p));
    H = normalize(L + V);
  } else {
    float a = fmaxf(0.001f, mp.roughness);
    float phi = rng.rnd() * 2.0f * MOX_PI_F;
    float xi = rng.rnd();
    float cosTheta = sqrtf((1.f - xi) / (1.0f + (a * a - 1.f) * xi));
    float sinTheta = sqrtf(1.0f - (cosTheta * cosTheta));
    float sinPhi = sinf(phi), cosPhi = cosf(phi);
    H = onb.toWorld(mk3(sinTheta * cosPhi, sinTheta * sinPhi, cosTheta));
    L = normalize(2.0f * dot(V, H) * H - V);
    H = normalize(H);
  }
}

// Everything in disneyPdf / disneyEval that depends only on the material, the base colour and
// the shading normal — evaluated once per hit and reused for every light and for the sampled
// direction.  Same operations in the same order as evaluating the reference functions from
// scratch each time, so the results are bit-identical.
template <bool F>
struct DisneyHit {
  float3 N, X, Y, Cdlin, Cspec0, Csheen;
  float metallic, subsurface, roughness, sheen, clearcoat, ax, ay, clearcoatAlpha, specularAlpha, diffuseRatio, pdfRatio;

  MOX_D DisneyHit(const DisneyParams& mp, const float3& baseColor, const float3& n) {
    N = n;
    Onb3 onb(N);
    Cdlin = mk3(bpow<F>(baseColor.x, 2.2f), bpow<F>(baseColor.y, 2.2f), bpow<F>(baseColor.z, 2.2f));
    float Cdlum = dot(Cdlin, mk3(0.3f, 0.6f, 0.1f));
    float3 Ctint = Cdlum > 0.f ? Cdlin / Cdlum : mk3(1.f);
    Cspec0 = lerp3(mp.specular * 0.08f * lerp3(mk3(1.f), Ctint, mp.specularTint), Cdlin, mp.metallic);
    Csheen = lerp3(mk3(1.f), Ctint, mp.sheenTint);
    float aspect = sqrtf(1 - mp.anisotropic * 0.9f);
    ax = fmaxf(.001f, sqr(mp.roughness) / aspect);
    ay = fmaxf(.001f, sqr(mp.roughness) * aspect);
    X = bnormalize<F>(onb.tangent);
    Y = bnormalize<F>(cross(N, X));
    metallic = mp.metallic; subsurface = mp.subsurface; roughness = mp.roughness; sheen = mp.sheen; clearcoat = mp.clearcoat;
    clearcoatAlpha = lerpf(0.1f, 0.001f, mp.clearcoatGloss);
    specularAlpha = fmaxf(0.001f, mp.roughness);
    diffuseRatio = 0.5f * (1.0f - mp.metallic);
    pdfRatio = 1.0f / (1.0f + mp.clearcoat);
  }

  // Terms of disneyPdf / disneyEval that depend on the view direction only (the same V for every light sample and
  // for the sampled direction of a hit), and products of per-hit constants that the reference expressions
  // evaluate first.  Same operations on the same operands in the same order: bit-identical results.
  float3 V;
  float NdotV, FV, GsV, GrV;
  float specularRatio, ccA2m1, ccPiLog, piAxAy, quarterClearcoat, oneMinusMetallic;
  MOX_D void setView(const float3& v) {
    V = v;
    NdotV = dot(N, V);
    FV = schlickFresnel(NdotV);
    GsV = smithGGgxAniso<F>(NdotV, dot(V, X), dot(V, Y), ax, ay);
    GrV = smithGGgx<F>(NdotV, 0.25f);
    specularRatio = 1.f - diffuseRatio;
    float a2 = clearcoatAlpha * clearcoatAlpha;
    ccA2m1 = a2 - 1.0f;
    ccPiLog = MOX_PI_F * blog<F>(a2);
    piAxAy = MOX_PI_F * ax * ay;
    quarterClearcoat = 0.25f * clearcoat;
    oneMinusMetallic = 1.0f - metallic;
  }
  // GTR1(c, clearcoatAlpha); even in c (each rounding is sign-symmetric), so pdf (|N.H|) and eval (N.H) share it
  MOX_D float gtr1Clearcoat(float c) const {
    if (clearcoatAlpha >= 1.f) return 1.f / MOX_PI_F;
    float t = 1.f + ccA2m1 * c * c;
    return bdiv<F>(ccA2m1, ccPiLog * t);
  }

  // disney.h:32-46; `dr` = GTR1(|N.H|, clearcoatAlpha) for eval()
  MOX_D float pdf(const float3& L, const float3& H, float& dr) const {
    float cosTheta = fabsf(dot(N, H));
    dr = gtr1Clearcoat(cosTheta);
    float pdfGTR1 = dr * cosTheta;
    float pdfGTR2 = GTR2<F>(cosTheta, specularAlpha) * cosTheta;
    float pdfH = lerpf(pdfGTR1, pdfGTR2, pdfRatio);
    float pdfL = bdiv<F>(pdfH, 4.0f * fabsf(dot(L, H)));
    float pdfDiff = bdiv<F>(fabsf(dot(N, L)), MOX_PI_F);
    return diffuseRatio * pdfDiff + specularRatio * pdfL;
  }

  // disney.h:48-91
  MOX_D float3 eval(const float3& L, const float3& H, float Dr) const {
    float NdotL = dot(N, L), NdotH = dot(N, H), LdotH = dot(L, H);
    float FL = schlickFresnel(NdotL);
    float Fd90 = 0.5f + 2.f * LdotH * LdotH * roughness;
    float Fd = lerpf(1.f, Fd90, FL) * lerpf(1.f, Fd90, FV);
    float Fss90 = LdotH * LdotH * roughness;
    float Fss = lerpf(1.0f, Fss90, FL) * lerpf(1.0f, Fss90, FV);
    float ss = 1.25f * (Fss * (bdiv<F>(1.f, NdotL + NdotV) - 0.5f) + 0.5f);
    float Ds = bdiv<F>(1.f, piAxAy * sqr(sqr(bdiv<F>(dot(H, X), ax)) + sqr(bdiv<F>(dot(H, Y), ay)) + NdotH * NdotH));
    float FH = schlickFresnel(LdotH);
    float3 Fs = lerp3(Cspec0, mk3(1.f), FH);
    float Gs = smithGGgxAniso<F>(NdotL, dot(L, X), dot(L, Y), ax, ay) * GsV;
    float3 Fsheen = FH * sheen * Csheen;
    float Fr = lerpf(0.04f, 1.f, FH);
    float Gr = smithGGgx<F>(NdotL, 0.25f) * GrV;
    return ((1.0f / MOX_PI_F) * lerpf(Fd, ss, subsurface) * Cdlin + Fsheen) * oneMinusMetallic + Gs * Fs * Ds +
           mk3(quarterClearcoat * Gr * Fr * Dr);
  }
};

