// oracle/oracle.cpp — TEST INFRASTRUCTURE.  Multi-threaded scalar C++ restatement of the
// reference's render path; the parity anchor and the CPU baseline.  Never linked into or
// loaded by the product library.
//
// PARITY PINNING: pinned to the reference's own text.  `make ref` compiles the reference's
// Camera.cu, Geometry.cu, Material.cu, miss.cu, disney.h and utils_device.h UNCHANGED with g++
// behind an OptiX shim (oracle/ref_shim/) into oracle/_ref/libref_render.so;
// scripts/make_render_golden.py stores its outputs in tests/golden/render_ref.npz and
// tests/test_ref_render.py holds this file to them BIT FOR BIT: every helper function,
// closest hits with all attributes, shadow transmittance, ray counts and whole images of
// five scenes that run every program (and BASELINE config 1 at full size, recorded in
// tests/golden/render_ref.json).  Not pinned by reference text: the OptiX SDK math helpers
// (optixu_math_namespace.h is not vendored; restated twice, here and in the shim) and OptiX's
// closed traversal.  The loader half is pinned by oracle/_ref/libref_loader.so.
//
// What follows what (paths relative to /root/reference/MinimalOptiX/):
//   camera()                 Camera.cu:21-42
//   sphere/quad/mesh tests   Geometry.cu:18-55, 70-91, 121-160   (bounds: :57-63, 93-110, 162-175)
//   miss                     miss.cu:10-12
//   lambertian/metal/glass   Material.cu:28-43, 49-66, 72-110
//   disney (+NEE, any-hit)   Material.cu:118-223, 225-232
//   light                    Material.cu:238-240
//   spp loop / accumulation  MinimalOptiX.cpp:540-560, 43-66
// OptiX's closed traversal (rtTrace) is replaced by (a) a brute-force loop over all
// primitives in id order — the primitive-id ground truth — or (b) a binned-SAH BVH2 with
// the same (t, id) lexicographic tie rule, used for timed runs.
//
// Deliberate deviations (SURVEY.md Appendix C): correct sphere AABB (Q7); order-independent
// shadow transmittance (Q8): over all Disney prims hit in (tmin,tmax): any NORMAL -> 0,
// else product of GLASS colours; light.radius/u/v zero-initialised by the loader (Q11).
#include "oracle.h"
#include "device_spec.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <string>
#include <thread>
#include <vector>

using namespace orc;

namespace {

inline float3 f3(const mox_float3& v) { return {v.x, v.y, v.z}; }

enum PrimType { PT_SPHERE = 0, PT_QUAD = 1, PT_TRI = 2 };

struct Material {
  int kind;
  LambertianParams lam;
  MetalParams met;
  GlassParams gls;
  DisneyParams dis;
  LightParams lgt;
};

struct Prim { int type; int geom; int mat; };
struct Tri { int v[3]; int n[3]; int t[3]; bool hasN, hasT; };
struct Texture { int w, h; std::vector<float> texels; };

struct Box { float3 lo, hi; bool valid; };

struct BvhNode {  // binary node; leaf when count > 0
  float3 lo, hi;
  int left, right;  // children (inner)
  int first, count; // prim range in `order` (leaf)
};

struct HitAttr {
  float t;
  int prim;
  float beta, gamma;
  float3 geoNormal, shadingNormal, front, back, texcoord;
};

struct Counters { uint64_t primary = 0, bounce = 0, shadow = 0, nonfinite = 0; };

}  // namespace

struct orc_ctx {
  std::string err;
  uint32_t W = 0, H = 0, maxDepth = 256;
  float eps = 0.001f, minIntensity = 0.001f;
  float3 absorb{0, 0, 0}, bad{1, 1, 1}, bg{0, 0, 0};
  CamParams cam{};
  int rngMode = 0;
  uint32_t rank = 0, world = 1, tile = 32;
  int nThreads = 0;
  bool brute = false;
  bool built = false;
  bool watertight = false;   // MOX_ACCEL_WATERTIGHT: the twin of the GPU's opt-in watertight triangle test
  int quadLightDrawOrder = 0;

  std::vector<Prim> prims;
  std::vector<SphereParams> spheres;
  std::vector<QuadParams> quads;
  std::vector<Tri> tris;
  std::vector<float3> verts, normals;
  std::vector<float2> uvs;
  std::vector<Material> mats;
  std::vector<LightParams> lights;
  std::vector<Texture> textures;

  std::vector<BvhNode> nodes;
  std::vector<int> order;

  std::vector<float> accu;
  uint64_t launches = 0;
  Counters cnt;
  double msRender = 0, msBuild = 0;
};

namespace {

// ------------------------------------------------------------------ bounds (Geometry.cu bbox programs)
Box primBox(const orc_ctx& c, const Prim& p) {
  Box b{};
  if (p.type == PT_SPHERE) {
    const SphereParams& s = c.spheres[p.geom];
    b.lo = f3(s.center) - s.radius;  // corrected orientation (reference passes (max,min), Geometry.cu:59-62)
    b.hi = f3(s.center) + s.radius;
    b.valid = true;
  } else if (p.type == PT_QUAD) {
    const QuadParams& q = c.quads[p.geom];
    float3 v1 = f3(q.v1), v2 = f3(q.v2), a = f3(q.anchor);
    float3 tv1 = v1 / dot(v1, v1);
    float3 tv2 = v2 / dot(v2, v2);
    float3 p00 = a, p01 = a + tv1, p10 = a + tv2, p11 = a + tv1 + tv2;
    float area = length(cross(tv1, tv2));
    b.valid = area > 0.0f && !std::isinf(area);
    b.lo = fminf3(fminf3(p00, p01), fminf3(p10, p11));
    b.hi = fmaxf3(fmaxf3(p00, p01), fmaxf3(p10, p11));
  } else {
    const Tri& t = c.tris[p.geom];
    float3 v0 = c.verts[t.v[0]], v1 = c.verts[t.v[1]], v2 = c.verts[t.v[2]];
    float area = length(cross(v1 - v0, v2 - v0));
    b.valid = area > 0.0f && !std::isinf(area);
    b.lo = fminf3(fminf3(v0, v1), v2);
    b.hi = fmaxf3(fmaxf3(v0, v1), v2);
  }
  return b;
}

// ------------------------------------------------------------------ primitive tests
// Each returns true and fills `h` when the primitive reports a hit with tmin < t < tmaxCur
// (rtPotentialIntersection semantics).
bool hitSphere(const SphereParams& sp, const Ray& ray, float tmaxCur, HitAttr& h) {  // Geometry.cu:18-55
  float3 oc = ray.origin - f3(sp.center);
  float b = dot(ray.direction, oc);
  float c = dot(oc, oc) - sp.radius * sp.radius;
  float disc = b * b - c;
  if (disc < 0) return false;
  float root = sqrtf(disc);
  float t = -b - root;
  if (!(t > ray.tmin && t < tmaxCur)) {
    t = -b + root;
    if (!(t > ray.tmin && t < tmaxCur)) return false;
  }
  h.t = t;
  h.geoNormal = normalize(ray.origin + t * ray.direction - f3(sp.center));
  h.shadingNormal = h.geoNormal;
  h.front = ray.origin + t * ray.direction;
  h.back = h.front;
  h.texcoord = make_float3(0.f);
  h.beta = h.gamma = 0.f;
  return true;
}

bool hitQuad(const QuadParams& q, const Ray& ray, float tmaxCur, HitAttr& h) {  // Geometry.cu:70-91
  float3 n = make_float3(q.plane.x, q.plane.y, q.plane.z);
  float dt = dot(ray.direction, n);
  float t = (q.plane.w - dot(n, ray.origin)) / dt;
  if (t > ray.tmin && t < ray.tmax) {
    float3 p = ray.origin + ray.direction * t;
    float3 vi = p - f3(q.anchor);
    float a1 = dot(f3(q.v1), vi);
    if (a1 >= 0 && a1 <= 1) {
      float a2 = dot(f3(q.v2), vi);
      if (a2 >= 0 && a2 <= 1) {
        if (t > ray.tmin && t < tmaxCur) {
          h.t = t;
          h.geoNormal = n;
          h.shadingNormal = n;
          h.front = ray.origin + t * ray.direction;
          h.back = h.front;
          h.texcoord = make_float3(0.f);  // left unset by the reference (Q10): defined as 0
          h.beta = a1; h.gamma = a2;
          return true;
        }
      }
    }
  }
  return false;
}

// Watertight ray-triangle test (Woop, Benthin, Wald 2013) — not part of the reference (its mesh program calls the
// SDK's intersect_triangle); the twin of triTestWt in minimaloptix_b200/csrc/gpu/traverse.cuh, operation for
// operation (this file is compiled with -ffp-contract=off, the GPU side with -fmad=false).  The vertices are
// sheared and scaled into a space where the ray is the +z axis; the scaled edge functions U, V, W of two triangles
// sharing an edge are computed from the same operands, so a ray cannot pass between them; exact zeros are decided
// in double.  No backface culling.  beta / gamma weigh p1 / p2.
struct WtRay { int kx, ky, kz; float Sx, Sy, Sz; };
inline float pick3(const float3& v, int k) { return k == 0 ? v.x : (k == 1 ? v.y : v.z); }
inline WtRay wtPrep(const float3& d) {
  WtRay w;
  const float ax = fabsf(d.x), ay = fabsf(d.y), az = fabsf(d.z);
  w.kz = ax > ay ? (ax > az ? 0 : 2) : (ay > az ? 1 : 2);
  w.kx = w.kz == 2 ? 0 : w.kz + 1;
  w.ky = w.kx == 2 ? 0 : w.kx + 1;
  const float dz = pick3(d, w.kz);
  if (dz < 0.f) { const int t = w.kx; w.kx = w.ky; w.ky = t; }
  w.Sx = pick3(d, w.kx) / dz;
  w.Sy = pick3(d, w.ky) / dz;
  w.Sz = 1.0f / dz;
  return w;
}
inline bool watertightTriangle(const Ray& ray, const float3& p0, const float3& p1, const float3& p2, float& t, float& beta,
                               float& gamma) {
  const WtRay w = wtPrep(ray.direction);
  const float3 A = p0 - ray.origin, B = p1 - ray.origin, C = p2 - ray.origin;
  const float Akz = pick3(A, w.kz), Bkz = pick3(B, w.kz), Ckz = pick3(C, w.kz);
  const float Ax = pick3(A, w.kx) - w.Sx * Akz, Ay = pick3(A, w.ky) - w.Sy * Akz;
  const float Bx = pick3(B, w.kx) - w.Sx * Bkz, By = pick3(B, w.ky) - w.Sy * Bkz;
  const float Cx = pick3(C, w.kx) - w.Sx * Ckz, Cy = pick3(C, w.ky) - w.Sy * Ckz;
  float U = Cx * By - Cy * Bx, V = Ax * Cy - Ay * Cx, W = Bx * Ay - By * Ax;
  if (U == 0.f || V == 0.f || W == 0.f) {
    U = (float)((double)Cx * (double)By - (double)Cy * (double)Bx);
    V = (float)((double)Ax * (double)Cy - (double)Ay * (double)Cx);
    W = (float)((double)Bx * (double)Ay - (double)By * (double)Ax);
  }
  if ((U < 0.f || V < 0.f || W < 0.f) && (U > 0.f || V > 0.f || W > 0.f)) return false;
  const float det = U + V + W;
  if (det == 0.f) return false;
  const float T = U * (w.Sz * Akz) + V * (w.Sz * Bkz) + W * (w.Sz * Ckz);
  const float rcp = 1.0f / det;
  t = T * rcp; beta = V * rcp; gamma = W * rcp;
  return t > ray.tmin;
}

// Geometry test only (t, beta, gamma, n); attributes are filled by triAttributes for the winner.
bool hitTriGeom(const orc_ctx& c, const Tri& tr, const Ray& ray, float tmaxCur, float3& n, float& t, float& beta,
                float& gamma) {  // Geometry.cu:121-134
  const float3 &p0 = c.verts[tr.v[0]], &p1 = c.verts[tr.v[1]], &p2 = c.verts[tr.v[2]];
  if (c.watertight) {
    n = cross(p0 - p2, p1 - p0);   // geometric normal as the SDK test leaves it
    return watertightTriangle(ray, p0, p1, p2, t, beta, gamma) && t < tmaxCur;
  }
  if (!intersect_triangle(ray, p0, p1, p2, n, t, beta, gamma)) return false;
  return t > ray.tmin && t < tmaxCur;
}

void triAttributes(const orc_ctx& c, const Tri& tr, const Ray& ray, const float3& n, float t, float beta,
                   float gamma, HitAttr& h) {  // Geometry.cu:135-158
  h.t = t; h.beta = beta; h.gamma = gamma;
  h.geoNormal = normalize(n);
  if (!tr.hasN) {
    h.shadingNormal = h.geoNormal;
  } else {
    h.shadingNormal = normalize(c.normals[tr.n[1]] * beta + c.normals[tr.n[2]] * gamma +
                                c.normals[tr.n[0]] * (1.f - beta - gamma));
  }
  if (!tr.hasT) {
    h.texcoord = make_float3(0.f);
  } else {
    float2 t0 = c.uvs[tr.t[0]], t1 = c.uvs[tr.t[1]], t2 = c.uvs[tr.t[2]];
    float w = 1.0f - beta - gamma;
    h.texcoord = make_float3(t1.x * beta + t2.x * gamma + t0.x * w, t1.y * beta + t2.y * gamma + t0.y * w, 0.f);
  }
  refineHitpoint(ray.origin + t * ray.direction, ray.direction, h.geoNormal, c.verts[tr.v[0]], h.back, h.front);
}

// One primitive against the current best under the (t, id) lexicographic rule.
inline void testPrimClosest(const orc_ctx& c, int id, const Ray& ray, HitAttr& best, float3& bestN) {
  const Prim& p = c.prims[id];
  // Accept t < best.t, or t == best.t with a lower id: implemented by testing against an
  // open upper bound nextafter(best.t) when id < best.prim.
  float bound = best.t;
  if (best.prim >= 0 && id < best.prim) bound = std::nextafterf(best.t, INFINITY);
  if (p.type == PT_TRI) {
    float3 n; float t, be, ga;
    if (hitTriGeom(c, c.tris[p.geom], ray, bound, n, t, be, ga)) {
      best.t = t; best.prim = id; best.beta = be; best.gamma = ga; bestN = n;
    }
  } else {
    HitAttr h;
    bool ok = (p.type == PT_SPHERE) ? hitSphere(c.spheres[p.geom], ray, bound, h)
                                    : hitQuad(c.quads[p.geom], ray, bound, h);
    if (ok) { h.prim = id; best = h; }
  }
}

// One axis of the slab test.  A direction component of magnitude at most 1e-30 (where the GPU's prepRay stops
// taking 1/d) counts as zero: the ray then stays in the slab for every t when lo <= o <= hi, and never otherwise.
// (With 1/d itself, an origin on a plane gives (lo - o) * inf = 0 * inf = NaN; with 1/d clamped, a ray on the far
// plane whose component is "+0 outwards" leaves the slab at t = 0.  Both culled hits on the plane that the
// primitive test accepts.)
inline bool slab(float lo, float hi, float o, float d, float inv, float& tn, float& tf) {
  if (fabsf(d) <= 1e-30f) return lo <= o && o <= hi;
  float t0 = (lo - o) * inv, t1 = (hi - o) * inv;
  tn = fmaxf(tn, fminf(t0, t1));
  tf = fminf(tf, fmaxf(t0, t1));
  return true;
}

// Slab test, padded so it never rejects a box whose primitive test could accept.
inline bool hitBox(const float3& lo, const float3& hi, const float3& o, const float3& d, const float3& inv, float tmin,
                   float tmax) {
  float tn = tmin, tf = tmax;
  if (!slab(lo.x, hi.x, o.x, d.x, inv.x, tn, tf) || !slab(lo.y, hi.y, o.y, d.y, inv.y, tn, tf) ||
      !slab(lo.z, hi.z, o.z, d.z, inv.z, tn, tf))
    return false;
  // tn >= tmin >= 0 here; widen the interval by a relative 1e-5 on both ends (the stated
  // epsilon-tie tolerance) so rounding in the slab arithmetic can never cull a primitive
  // the exact test would accept.
  return tn * 0.99999f <= tf * 1.00001f;
}

bool closestHit(const orc_ctx& c, const Ray& ray, HitAttr& out) {
  HitAttr best{};
  best.t = ray.tmax;
  best.prim = -1;
  float3 bestN{};
  if (c.brute || c.nodes.empty()) {
    for (int id = 0; id < (int)c.prims.size(); ++id) testPrimClosest(c, id, ray, best, bestN);
  } else {
    float3 inv = {1.0f / ray.direction.x, 1.0f / ray.direction.y, 1.0f / ray.direction.z};
    int stack[128];
    int sp = 0;
    stack[sp++] = 0;
    while (sp) {
      const BvhNode& nd = c.nodes[stack[--sp]];
      if (!hitBox(nd.lo, nd.hi, ray.origin, ray.direction, inv, ray.tmin, best.t)) continue;
      if (nd.count > 0) {
        for (int k = 0; k < nd.count; ++k) testPrimClosest(c, c.order[nd.first + k], ray, best, bestN);
      } else {
        stack[sp++] = nd.left;
        stack[sp++] = nd.right;
      }
    }
  }
  if (best.prim < 0) return false;
  const Prim& p = c.prims[best.prim];
  if (p.type == PT_TRI) {
    HitAttr h;
    triAttributes(c, c.tris[p.geom], ray, bestN, best.t, best.beta, best.gamma, h);
    h.prim = best.prim;
    best = h;
  }
  out = best;
  return true;
}

// Shadow-ray transmittance, order-independent rule (SURVEY.md a-11): only Disney prims
// occlude (MinimalOptiX.cpp:183,194,205,516 register no any-hit on the others).
inline void testPrimShadow(const orc_ctx& c, int id, const Ray& ray, float3& atten, bool& blocked) {
  const Prim& p = c.prims[id];
  const Material& m = c.mats[p.mat];
  if (m.kind != MOX_MAT_DISNEY) return;
  bool hit;
  if (p.type == PT_TRI) {
    float3 n; float t, be, ga;
    hit = hitTriGeom(c, c.tris[p.geom], ray, ray.tmax, n, t, be, ga);
  } else {
    HitAttr h;
    hit = (p.type == PT_SPHERE) ? hitSphere(c.spheres[p.geom], ray, ray.tmax, h) : hitQuad(c.quads[p.geom], ray, ray.tmax, h);
  }
  if (!hit) return;
  if (m.dis.brdfType == GLASS) atten *= f3(m.dis.color);  // Material.cu:226-227
  else blocked = true;                                     // Material.cu:229-230
}

float3 shadowTransmittance(const orc_ctx& c, const Ray& ray) {
  float3 atten = make_float3(1.f);
  bool blocked = false;
  if (c.brute || c.nodes.empty()) {
    for (int id = 0; id < (int)c.prims.size() && !blocked; ++id) testPrimShadow(c, id, ray, atten, blocked);
  } else {
    float3 inv = {1.0f / ray.direction.x, 1.0f / ray.direction.y, 1.0f / ray.direction.z};
    int stack[128];
    int sp = 0;
    stack[sp++] = 0;
    while (sp && !blocked) {
      const BvhNode& nd = c.nodes[stack[--sp]];
      if (!hitBox(nd.lo, nd.hi, ray.origin, ray.direction, inv, ray.tmin, ray.tmax)) continue;
      if (nd.count > 0) {
        for (int k = 0; k < nd.count && !blocked; ++k) testPrimShadow(c, c.order[nd.first + k], ray, atten, blocked);
      } else {
        stack[sp++] = nd.left;
        stack[sp++] = nd.right;
      }
    }
  }
  return blocked ? make_float3(0.f) : atten;
}

// ------------------------------------------------------------------ texture (rtTex2D<float4>, bilinear, REPEAT)
float3 sampleTexture(const orc_ctx& c, int id, float u, float v) {
  const Texture& tx = c.textures[id - 1];
  float x = u * tx.w - 0.5f, y = v * tx.h - 0.5f;
  float fx = floorf(x), fy = floorf(y);
  float ax = x - fx, ay = y - fy;
  auto wrap = [](int i, int n) { int m = i % n; return m < 0 ? m + n : m; };
  int x0 = wrap((int)fx, tx.w), x1 = wrap((int)fx + 1, tx.w);
  int y0 = wrap((int)fy, tx.h), y1 = wrap((int)fy + 1, tx.h);
  auto px = [&](int xi, int yi) { const float* p = &tx.texels[4 * ((size_t)yi * tx.w + xi)]; return make_float3(p[0], p[1], p[2]); };
  float3 c00 = px(x0, y0), c10 = px(x1, y0), c01 = px(x0, y1), c11 = px(x1, y1);
  return (c00 * (1 - ax) + c10 * ax) * (1 - ay) + (c01 * (1 - ax) + c11 * ax) * ay;
}

// ------------------------------------------------------------------ integrator (recursive, as the reference)
float3 trace(const orc_ctx& c, const Ray& ray, int depth, Rng rng, Counters& cnt);

// Shared by glass() and disney()/GLASS (Material.cu:79-109, 134-167).
float3 dielectric(const orc_ctx& c, const Ray& ray, const HitAttr& h, int depth, Rng& rng, float ior,
                  const float3& tint, Counters& cnt) {
  float3 normal = h.shadingNormal;
  float cosThetaI = -dot(ray.direction, normal);
  float refIdx;
  if (cosThetaI > 0.f) {
    refIdx = ior;
  } else {
    refIdx = 1.f / ior;
    cosThetaI = -cosThetaI;
    normal = -normal;
  }
  float3 refracted;
  bool totalReflection = !refract(refracted, ray.direction, normal, refIdx);
  float cosThetaT = -dot(normal, refracted);
  float reflectProb = totalReflection ? 1.f : fresnel(cosThetaI, cosThetaT, refIdx);
  Ray nr;
  nr.tmin = c.eps;
  nr.tmax = RT_DEFAULT_MAX;
  Rng child = forkRng(rng, depth + 1);  // child seed BEFORE the coin flip (Material.cu:100-101)
  if (rnd(rng) < reflectProb) {
    nr.origin = h.front;
    nr.direction = reflect(ray.direction, normal);
  } else {
    nr.origin = h.back;
    nr.direction = refracted;
  }
  float3 childColor = trace(c, nr, depth + 1, child, cnt);
  return childColor * tint;
}

float3 shadeDisney(const orc_ctx& c, const Material& m, const Ray& ray, const HitAttr& h, int depth, Rng& rng,
                   Counters& cnt) {  // Material.cu:118-223
  const DisneyParams& dp = m.dis;
  float3 N = faceforward(h.shadingNormal, -ray.direction, h.geoNormal);
  float3 V = -ray.direction;
  float3 L, H;
  float3 baseColor = dp.albedoID == MOX_TEXTURE_ID_NULL ? f3(dp.color) : sampleTexture(c, dp.albedoID, h.texcoord.x, h.texcoord.y);
  if (dp.brdfType == GLASS) return dielectric(c, ray, h, depth, rng, 1.45f, baseColor, cnt);

  float3 direct = make_float3(0.f);
  for (size_t i = 0; i < c.lights.size(); ++i) {
    const LightParams& light = c.lights[i];
    float3 pointOnLight, normalOnLight;
    if (light.shape == SPHERE) {
      pointOnLight = f3(light.position) + randInUnitSphere(rng) * light.radius;
      normalOnLight = normalize(pointOnLight - f3(light.position));
    } else {
      // Material.cu:180 draws both numbers inside one expression, `u * rand(s) + v * rand(s)`:
      // C++ leaves the order open (SURVEY.md F10).  Pinned: first draw scales u (nvcc's order).
      // quadLightDrawOrder = 1 gives the first draw to v instead — what g++ makes of the
      // reference's text; only the differential tests against oracle/_ref set it.
      float r1 = rnd(rng);
      float r2 = rnd(rng);
      if (c.quadLightDrawOrder) std::swap(r1, r2);
      pointOnLight = f3(light.position) + f3(light.u) * r1 + f3(light.v) * r2;
      normalOnLight = normalize(f3(light.normal));
    }
    L = pointOnLight - h.front;
    float lightDst = length(L);
    L = normalize(L);
    if (dot(L, N) > 0.f && dot(L, normalOnLight) < 0.f) {
      Ray sr{h.front, L, c.eps, lightDst - c.eps};
      cnt.shadow++;
      float3 atten = shadowTransmittance(c, sr);
      if (length(atten)) {
        H = normalize(L + V);
        float lightPdf = lightDst * lightDst / light.area / dot(normalOnLight, -L);
        float objPdf = disneyPdf(dp, N, L, V, H);
        if (lightPdf > 0 && objPdf > 0) {
          float3 brdf = disneyEval(dp, baseColor, N, L, V, H);
          direct += powerHeuristic(lightPdf, objPdf) * brdf * f3(light.emission) * atten / fmaxf(0.001f, lightPdf);
        }
      }
    }
  }

  float3 indirect = make_float3(0.f);
  disneySample(rng, dp, N, L, V, H);
  if (dot(N, L) > 0.0f && dot(N, V) > 0.0f) {
    Ray nr{h.front, L, c.eps, RT_DEFAULT_MAX};
    Rng child = forkRng(rng, depth + 1);
    float3 childColor = trace(c, nr, depth + 1, child, cnt);
    float pdf = disneyPdf(dp, N, L, V, H);
    if (pdf > 0) {
      float3 brdf = disneyEval(dp, baseColor, N, L, V, H);
      indirect = brdf * childColor / pdf;
    }
  }
  return indirect + direct + f3(dp.emission);
}

float3 trace(const orc_ctx& c, const Ray& ray, int depth, Rng rng, Counters& cnt) {
  if (depth == 1) cnt.primary++; else cnt.bounce++;
  HitAttr h;
  if (!closestHit(c, ray, h)) return make_float3(1.f) * c.bg;  // miss.cu:10-12 (payload colour starts at 1)
  const Material& m = c.mats[c.prims[h.prim].mat];
  if (m.kind == MOX_MAT_LIGHT) return f3(m.lgt.emission);  // Material.cu:238-240
  // Every scattering program starts with this test (Material.cu:29,50,73,119); the incoming
  // payload colour is always (1,1,1), so the intensity clause never fires for minIntensity < sqrt(3).
  if ((uint32_t)depth > c.maxDepth || length(make_float3(1.f)) < c.minIntensity) return c.absorb;
  switch (m.kind) {
    case MOX_MAT_LAMBERTIAN: {  // Material.cu:28-43
      float3 v = randInUnitSphere(rng);
      Ray nr{ray.origin + h.t * ray.direction, normalize(h.geoNormal + v), c.eps, RT_DEFAULT_MAX};
      Rng child = forkRng(rng, depth + 1);
      return trace(c, nr, depth + 1, child, cnt) * f3(m.lam.albedo);
    }
    case MOX_MAT_METAL: {  // Material.cu:49-66
      float3 v = randInUnitSphere(rng);
      Ray nr{ray.origin + h.t * ray.direction, normalize(reflect(ray.direction, h.geoNormal) + m.met.fuzz * v), c.eps,
             RT_DEFAULT_MAX};
      Rng child = forkRng(rng, depth + 1);
      return f3(m.met.albedo) * trace(c, nr, depth + 1, child, cnt);
    }
    case MOX_MAT_GLASS:  // Material.cu:72-110
      return dielectric(c, ray, h, depth, rng, m.gls.refIdx, f3(m.gls.albedo), cnt);
    case MOX_MAT_DISNEY:
      return shadeDisney(c, m, ray, h, depth, rng, cnt);
  }
  return c.absorb;
}

// Camera.cu:21-42 for pixel (x, y) of launch `launchSeed`; returns the clamped sample.
float3 cameraSample(const orc_ctx& c, uint32_t x, uint32_t y, int32_t launchSeed, Counters& cnt) {
  Rng rng = rngForPixel(c.rngMode, y * c.W + x, (uint32_t)launchSeed);
  const CamParams& cp = c.cam;
  float3 randInLens = cp.lensRadius * randInUnitDisk(rng);
  float3 offset = f3(cp.u) * randInLens.x + f3(cp.v) * randInLens.y;
  float r1 = rnd(rng);
  float r2 = rnd(rng);
  float sx = ((float)x + r1 - 0.5f) / (float)c.W;
  float sy = ((float)y + r2 - 0.5f) / (float)c.H;
  Ray ray;
  ray.origin = f3(cp.origin) + offset;
  ray.direction = normalize(f3(cp.scrLowerLeftCorner) + sx * f3(cp.horizontal) + sy * f3(cp.vertical) - f3(cp.origin) - offset);
  ray.tmin = c.eps;
  ray.tmax = RT_DEFAULT_MAX;
  float3 color = trace(c, ray, 1, rng, cnt);
  // A non-finite sample is this path's "exception": badColor replaces it (Exception.cu:10-12; the
  // reference's clamp would turn NaN into 1 per channel — SURVEY App. A.8, a stated deviation).
  if (!std::isfinite(color.x) || !std::isfinite(color.y) || !std::isfinite(color.z)) { cnt.nonfinite++; return c.bad; }
  return clamp(color, make_float3(0.f), make_float3(1.f));
}

// ------------------------------------------------------------------ binned-SAH BVH2 (oracle's own accel)
struct BuildItem { float3 lo, hi, ctr; int id; };

int buildNode(orc_ctx& c, std::vector<BuildItem>& items, int first, int count) {
  int idx = (int)c.nodes.size();
  c.nodes.push_back({});
  float3 lo = make_float3(INFINITY), hi = make_float3(-INFINITY), clo = lo, chi = hi;
  for (int i = first; i < first + count; ++i) {
    lo = fminf3(lo, items[i].lo); hi = fmaxf3(hi, items[i].hi);
    clo = fminf3(clo, items[i].ctr); chi = fmaxf3(chi, items[i].ctr);
  }
  auto makeLeaf = [&]() {
    BvhNode& n = c.nodes[idx];
    n.lo = lo; n.hi = hi; n.first = first; n.count = count; n.left = n.right = -1;
    return idx;
  };
  if (count <= 2) return makeLeaf();
  float3 ext = chi - clo;
  int axis = ext.x > ext.y ? (ext.x > ext.z ? 0 : 2) : (ext.y > ext.z ? 1 : 2);
  float e = axis == 0 ? ext.x : axis == 1 ? ext.y : ext.z;
  float cmin = axis == 0 ? clo.x : axis == 1 ? clo.y : clo.z;
  if (!(e > 0)) {
    if (count <= 8) return makeLeaf();
    int mid = first + count / 2;  // coincident centroids: split by count
    int l = buildNode(c, items, first, mid - first), r = buildNode(c, items, mid, first + count - mid);
    BvhNode& n = c.nodes[idx];
    n.lo = lo; n.hi = hi; n.count = 0; n.first = 0; n.left = l; n.right = r;
    return idx;
  }
  const int NB = 16;
  struct Bin { float3 lo, hi; int n; } bins[NB];
  for (auto& b : bins) { b.lo = make_float3(INFINITY); b.hi = make_float3(-INFINITY); b.n = 0; }
  auto comp = [&](const float3& v) { return axis == 0 ? v.x : axis == 1 ? v.y : v.z; };
  auto binOf = [&](const BuildItem& it) { int b = (int)((comp(it.ctr) - cmin) / e * NB); return std::min(NB - 1, std::max(0, b)); };
  for (int i = first; i < first + count; ++i) {
    Bin& b = bins[binOf(items[i])];
    b.lo = fminf3(b.lo, items[i].lo); b.hi = fmaxf3(b.hi, items[i].hi); b.n++;
  }
  auto area = [](const float3& l, const float3& h) { float3 d = h - l; return 2.f * (d.x * d.y + d.y * d.z + d.z * d.x); };
  float rightArea[NB]; int rightN[NB];
  float3 rl = make_float3(INFINITY), rh = make_float3(-INFINITY); int rn = 0;
  for (int i = NB - 1; i > 0; --i) {
    rl = fminf3(rl, bins[i].lo); rh = fmaxf3(rh, bins[i].hi); rn += bins[i].n;
    rightArea[i] = rn ? area(rl, rh) : 0.f; rightN[i] = rn;
  }
  float3 ll = make_float3(INFINITY), lh = make_float3(-INFINITY); int ln = 0;
  float bestCost = INFINITY; int bestSplit = -1;
  for (int i = 1; i < NB; ++i) {
    ll = fminf3(ll, bins[i - 1].lo); lh = fmaxf3(lh, bins[i - 1].hi); ln += bins[i - 1].n;
    if (ln == 0 || rightN[i] == 0) continue;
    float cost = area(ll, lh) * ln + rightArea[i] * rightN[i];
    if (cost < bestCost) { bestCost = cost; bestSplit = i; }
  }
  if (bestSplit < 0 || (count <= 4 && bestCost >= area(lo, hi) * count)) {
    if (count <= 8) return makeLeaf();
    bestSplit = NB / 2;
  }
  auto midIt = std::partition(items.begin() + first, items.begin() + first + count,
                              [&](const BuildItem& it) { return binOf(it) < bestSplit; });
  int mid = (int)(midIt - items.begin());
  if (mid == first || mid == first + count) mid = first + count / 2;
  int l = buildNode(c, items, first, mid - first), r = buildNode(c, items, mid, first + count - mid);
  BvhNode& n = c.nodes[idx];
  n.lo = lo; n.hi = hi; n.count = 0; n.first = 0; n.left = l; n.right = r;
  return idx;
}

void buildBvh(orc_ctx& c) {
  c.nodes.clear();
  c.order.clear();
  std::vector<BuildItem> items;
  items.reserve(c.prims.size());
  for (int id = 0; id < (int)c.prims.size(); ++id) {
    Box b = primBox(c, c.prims[id]);
    if (!b.valid) continue;  // invalid boxes are excluded from the accel (Geometry.cu:104-109,169-174)
    items.push_back({b.lo, b.hi, (b.lo + b.hi) * 0.5f, id});
  }
  if (items.empty()) return;
  c.nodes.reserve(items.size() * 2);
  buildNode(c, items, 0, (int)items.size());
  c.order.resize(items.size());
  for (size_t i = 0; i < items.size(); ++i) c.order[i] = items[i].id;
}

inline bool owns(const orc_ctx& c, uint32_t rank, uint32_t x, uint32_t y) {
  return ((x / c.tile) + (y / c.tile)) % c.world == rank;
}

// Owned pixels of `rank` in tile order (tiles by ascending index, row-major inside a tile).
void ownedList(const orc_ctx& c, uint32_t rank, std::vector<uint32_t>& out) {
  out.clear();
  uint32_t tx = (c.W + c.tile - 1) / c.tile, ty = (c.H + c.tile - 1) / c.tile;
  for (uint32_t j = 0; j < ty; ++j)
    for (uint32_t i = 0; i < tx; ++i) {
      if ((i + j) % c.world != rank) continue;
      for (uint32_t y = j * c.tile; y < std::min(c.H, (j + 1) * c.tile); ++y)
        for (uint32_t x = i * c.tile; x < std::min(c.W, (i + 1) * c.tile); ++x) out.push_back(y * c.W + x);
    }
}

int launchSeeds(orc_ctx* c, const std::vector<int32_t>& seeds) {
  if (!c->built) { c->err = "launch before build_accel"; return MOX_ERR_STATE; }
  if (c->W == 0 || c->H == 0) { c->err = "launch before set_globals"; return MOX_ERR_STATE; }
  auto t0 = std::chrono::steady_clock::now();
  int nt = c->nThreads > 0 ? c->nThreads : (int)std::thread::hardware_concurrency();
  if (nt < 1) nt = 1;
  const uint32_t T = 32;
  uint32_t tilesX = (c->W + T - 1) / T, tilesY = (c->H + T - 1) / T;
  std::atomic<uint32_t> next{0};
  std::vector<Counters> cnts(nt);
  auto worker = [&](int tid) {
    Counters& cnt = cnts[tid];
    for (;;) {
      uint32_t t = next.fetch_add(1);
      if (t >= tilesX * tilesY) break;
      uint32_t x0 = (t % tilesX) * T, y0 = (t / tilesX) * T;
      for (uint32_t y = y0; y < std::min(c->H, y0 + T); ++y)
        for (uint32_t x = x0; x < std::min(c->W, x0 + T); ++x) {
          if (!owns(*c, c->rank, x, y)) continue;
          float* a = &c->accu[3 * ((size_t)y * c->W + x)];
          for (int32_t s : seeds) {  // samples accumulate in launch order, as successive launches do
            float3 col = cameraSample(*c, x, y, s, cnt);
            a[0] += col.x; a[1] += col.y; a[2] += col.z;  // Camera.cu:41
          }
        }
    }
  };
  std::vector<std::thread> th;
  for (int i = 1; i < nt; ++i) th.emplace_back(worker, i);
  worker(0);
  for (auto& t : th) t.join();
  for (auto& k : cnts) {
    c->cnt.primary += k.primary; c->cnt.bounce += k.bounce; c->cnt.shadow += k.shadow; c->cnt.nonfinite += k.nonfinite;
  }
  c->launches += seeds.size();
  c->msRender += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return MOX_OK;
}

int addMaterial(orc_ctx* c, int kind, const void* params) {
  Material m{};
  m.kind = kind;
  switch (kind) {
    case MOX_MAT_LAMBERTIAN: m.lam = *(const LambertianParams*)params; break;
    case MOX_MAT_METAL: m.met = *(const MetalParams*)params; break;
    case MOX_MAT_GLASS: m.gls = *(const GlassParams*)params; break;
    case MOX_MAT_DISNEY: m.dis = *(const DisneyParams*)params; break;
    case MOX_MAT_LIGHT: m.lgt = *(const LightParams*)params; break;
    default: return -1;
  }
  c->mats.push_back(m);
  return (int)c->mats.size() - 1;
}

}  // namespace

// ====================================================================== C ABI
extern "C" {

int orc_abi_version(void) { return MOX_ABI_VERSION; }

int orc_create(orc_ctx** out, int) {
  if (!out) return MOX_ERR_INVALID;
  *out = new orc_ctx();
  return MOX_OK;
}
void orc_destroy(orc_ctx* c) { delete c; }
const char* orc_last_error(const orc_ctx* c) { return c ? c->err.c_str() : ""; }

int orc_set_globals(orc_ctx* c, uint32_t w, uint32_t h, uint32_t maxDepth, float eps, float minI, const float absorb[3],
                    const float bad[3], const float bg[3]) {
  if (!c || w == 0 || h == 0) return MOX_ERR_INVALID;
  if (w != c->W || h != c->H) c->accu.assign((size_t)w * h * 3, 0.f), c->launches = 0;
  c->W = w; c->H = h; c->maxDepth = maxDepth; c->eps = eps; c->minIntensity = minI;
  c->absorb = {absorb[0], absorb[1], absorb[2]};
  c->bad = {bad[0], bad[1], bad[2]};
  c->bg = {bg[0], bg[1], bg[2]};
  return MOX_OK;
}
int orc_set_camera(orc_ctx* c, const CamParams* p) { if (!c || !p) return MOX_ERR_INVALID; c->cam = *p; return MOX_OK; }
int orc_set_rng_mode(orc_ctx* c, int m) { if (!c || m < 0 || m > 1) return MOX_ERR_INVALID; c->rngMode = m; return MOX_OK; }
int orc_set_partition(orc_ctx* c, uint32_t rank, uint32_t world, uint32_t tile) {
  if (!c || world == 0 || rank >= world || tile == 0) return MOX_ERR_INVALID;
  c->rank = rank; c->world = world; c->tile = tile;
  return MOX_OK;
}
int orc_set_threads(orc_ctx* c, int n) { if (!c) return MOX_ERR_INVALID; c->nThreads = n; return MOX_OK; }
int orc_set_quad_light_draw_order(orc_ctx* c, int order) { if (!c || order < 0 || order > 1) return MOX_ERR_INVALID; c->quadLightDrawOrder = order; return MOX_OK; }
int orc_set_brute_force(orc_ctx* c, int on) { if (!c) return MOX_ERR_INVALID; c->brute = on != 0; return MOX_OK; }

int orc_add_texture_rgba32f(orc_ctx* c, const float* texels, int w, int h, int* out_id) {
  if (!c || !texels || w <= 0 || h <= 0) return MOX_ERR_INVALID;
  Texture t; t.w = w; t.h = h; t.texels.assign(texels, texels + (size_t)w * h * 4);
  c->textures.push_back(std::move(t));
  if (out_id) *out_id = (int)c->textures.size();
  return MOX_OK;
}

int orc_add_sphere(orc_ctx* c, const SphereParams* s, int kind, const void* params, uint32_t* out_id) {
  if (!c || !s || !params) return MOX_ERR_INVALID;
  int m = addMaterial(c, kind, params);
  if (m < 0) { c->err = "bad material kind"; return MOX_ERR_INVALID; }
  c->spheres.push_back(*s);
  c->prims.push_back({PT_SPHERE, (int)c->spheres.size() - 1, m});
  if (out_id) *out_id = (uint32_t)c->prims.size() - 1;
  c->built = false;
  return MOX_OK;
}
int orc_add_quad(orc_ctx* c, const QuadParams* q, int kind, const void* params, uint32_t* out_id) {
  if (!c || !q || !params) return MOX_ERR_INVALID;
  int m = addMaterial(c, kind, params);
  if (m < 0) { c->err = "bad material kind"; return MOX_ERR_INVALID; }
  c->quads.push_back(*q);
  c->prims.push_back({PT_QUAD, (int)c->quads.size() - 1, m});
  if (out_id) *out_id = (uint32_t)c->prims.size() - 1;
  c->built = false;
  return MOX_OK;
}
int orc_add_mesh(orc_ctx* c, const float* v, size_t nv, const float* n, size_t nn, const float* uv, size_t nt,
                 const int32_t* vIdx, const int32_t* nIdx, const int32_t* tIdx, size_t nFaces, int kind,
                 const void* params, uint32_t* out_first) {
  if (!c || !params || (nFaces && (!v || !vIdx))) return MOX_ERR_INVALID;
  int m = addMaterial(c, kind, params);
  if (m < 0) { c->err = "bad material kind"; return MOX_ERR_INVALID; }
  bool hasN = nn > 0 && n && nIdx, hasT = nt > 0 && uv && tIdx;
  for (size_t f = 0; f < nFaces * 3; ++f) {
    if (vIdx[f] < 0 || (size_t)vIdx[f] >= nv) { c->err = "vertex index out of range"; return MOX_ERR_INVALID; }
    if (hasN && (nIdx[f] < 0 || (size_t)nIdx[f] >= nn)) hasN = false;   // any missing index: mesh treated as normal-less
    if (hasT && (tIdx[f] < 0 || (size_t)tIdx[f] >= nt)) hasT = false;
  }
  int vb = (int)c->verts.size(), nb = (int)c->normals.size(), tb = (int)c->uvs.size();
  for (size_t i = 0; i < nv; ++i) c->verts.push_back({v[3 * i], v[3 * i + 1], v[3 * i + 2]});
  if (hasN) for (size_t i = 0; i < nn; ++i) c->normals.push_back({n[3 * i], n[3 * i + 1], n[3 * i + 2]});
  if (hasT) for (size_t i = 0; i < nt; ++i) c->uvs.push_back({uv[2 * i], uv[2 * i + 1]});
  if (out_first) *out_first = (uint32_t)c->prims.size();
  for (size_t f = 0; f < nFaces; ++f) {
    Tri t{};
    t.hasN = hasN; t.hasT = hasT;
    for (int k = 0; k < 3; ++k) {
      t.v[k] = vb + vIdx[3 * f + k];
      t.n[k] = hasN ? nb + nIdx[3 * f + k] : -1;
      t.t[k] = hasT ? tb + tIdx[3 * f + k] : -1;
    }
    c->tris.push_back(t);
    c->prims.push_back({PT_TRI, (int)c->tris.size() - 1, m});
  }
  c->built = false;
  return MOX_OK;
}
int orc_set_lights(orc_ctx* c, const LightParams* l, size_t n) {
  if (!c || (n && !l)) return MOX_ERR_INVALID;
  c->lights.assign(l, l + n);
  return MOX_OK;
}
int orc_clear_scene(orc_ctx* c) {
  if (!c) return MOX_ERR_INVALID;
  c->prims.clear(); c->spheres.clear(); c->quads.clear(); c->tris.clear(); c->verts.clear(); c->normals.clear();
  c->uvs.clear(); c->mats.clear(); c->lights.clear(); c->textures.clear(); c->nodes.clear(); c->order.clear();
  c->built = false;
  return MOX_OK;
}
int orc_build_accel(orc_ctx* c, uint32_t flags, float* out_ms) {
  if (!c) return MOX_ERR_INVALID;
  c->watertight = (flags & MOX_ACCEL_WATERTIGHT) != 0;
  auto t0 = std::chrono::steady_clock::now();
  buildBvh(*c);
  c->msBuild = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  if (out_ms) *out_ms = (float)c->msBuild;
  c->built = true;
  return MOX_OK;
}
int orc_launch(orc_ctx* c, int32_t seed) {
  if (!c) return MOX_ERR_INVALID;
  return launchSeeds(c, std::vector<int32_t>{seed});
}
int orc_render(orc_ctx* c, uint32_t spp, uint32_t seed) {
  if (!c) return MOX_ERR_INVALID;
  std::vector<int32_t> seeds(spp);
  for (uint32_t i = 0; i < spp; ++i) seeds[i] = (int32_t)tea<16>((uint32_t)(c->launches + i), seed);
  return launchSeeds(c, seeds);
}
int orc_read_accum(orc_ctx* c, float* dst) {
  if (!c || !dst) return MOX_ERR_INVALID;
  std::copy(c->accu.begin(), c->accu.end(), dst);
  return MOX_OK;
}
int orc_map_accum(orc_ctx* c, const float** out) { if (!c || !out) return MOX_ERR_INVALID; *out = c->accu.data(); return MOX_OK; }
int orc_unmap_accum(orc_ctx* c) { return c ? MOX_OK : MOX_ERR_INVALID; }
int orc_device_count(const orc_ctx* c) { return c ? 1 : 0; }
int orc_get_device_stats(orc_ctx* c, int index, mox_stats* s) { return index == 0 ? orc_get_stats(c, s) : MOX_ERR_INVALID; }
// host memory already: begin is a no-op, end hands out the accumulation buffer
int orc_read_accum_begin(orc_ctx* c) { return c ? MOX_OK : MOX_ERR_INVALID; }
int orc_read_accum_end(orc_ctx* c, const float** out) { return orc_map_accum(c, out); }
int orc_clear_accum(orc_ctx* c) {
  if (!c) return MOX_ERR_INVALID;
  std::fill(c->accu.begin(), c->accu.end(), 0.f);
  c->launches = 0; c->cnt = Counters{}; c->msRender = 0;
  return MOX_OK;
}
int orc_set_accum(orc_ctx* c, const float* src, uint64_t launches) {
  if (!c || !src || c->accu.empty()) return MOX_ERR_INVALID;
  std::copy(src, src + c->accu.size(), c->accu.begin());
  c->launches = launches;
  return MOX_OK;
}
int orc_update_sphere(orc_ctx* c, uint32_t prim, const SphereParams* s) {
  if (!c || !s || prim >= c->prims.size() || c->prims[prim].type != PT_SPHERE) return MOX_ERR_INVALID;
  c->spheres[c->prims[prim].geom] = *s;
  c->built = false;
  return MOX_OK;
}
int orc_owned_pixels(orc_ctx* c, uint32_t rank, uint64_t* out_n) {
  if (!c || !out_n || rank >= c->world) return MOX_ERR_INVALID;
  std::vector<uint32_t> l; ownedList(*c, rank, l); *out_n = l.size();
  return MOX_OK;
}
int orc_pack_owned(orc_ctx* c, void* dst) {
  if (!c || !dst) return MOX_ERR_INVALID;
  std::vector<uint32_t> l; ownedList(*c, c->rank, l);
  float* d = (float*)dst;
  for (size_t i = 0; i < l.size(); ++i) for (int k = 0; k < 3; ++k) d[3 * i + k] = c->accu[3 * (size_t)l[i] + k];
  return MOX_OK;
}
int orc_unpack_owned(orc_ctx* c, uint32_t rank, const void* src) {
  if (!c || !src || rank >= c->world) return MOX_ERR_INVALID;
  std::vector<uint32_t> l; ownedList(*c, rank, l);
  const float* s = (const float*)src;
  for (size_t i = 0; i < l.size(); ++i) for (int k = 0; k < 3; ++k) c->accu[3 * (size_t)l[i] + k] = s[3 * i + k];
  return MOX_OK;
}
int orc_get_stats(orc_ctx* c, mox_stats* s) {
  if (!c || !s) return MOX_ERR_INVALID;
  *s = mox_stats{};
  s->rays_primary = c->cnt.primary; s->rays_bounce = c->cnt.bounce; s->rays_shadow = c->cnt.shadow;
  s->nonfinite_samples = c->cnt.nonfinite; s->launches = c->launches;
  s->ms_render = c->msRender; s->ms_build = c->msBuild;
  s->n_prims = (uint32_t)c->prims.size(); s->n_triangles = (uint32_t)c->tris.size();
  s->n_spheres = (uint32_t)c->spheres.size(); s->n_quads = (uint32_t)c->quads.size();
  s->n_nodes = (uint32_t)c->nodes.size(); s->node_bytes = sizeof(BvhNode); s->prim_bytes = 36;
  s->n_lights = (uint32_t)c->lights.size();
  return MOX_OK;
}

int orc_trace_closest(orc_ctx* c, const float* rays, size_t n, void* hits) {
  if (!c || (n && (!rays || !hits))) return MOX_ERR_INVALID;
  if (!c->built) { c->err = "trace before build_accel"; return MOX_ERR_STATE; }
  int nt = c->nThreads > 0 ? c->nThreads : (int)std::thread::hardware_concurrency();
  if (nt < 1) nt = 1;
  std::atomic<size_t> next{0};
  auto worker = [&]() {
    for (;;) {
      size_t b = next.fetch_add(4096);
      if (b >= n) break;
      for (size_t i = b; i < std::min(n, b + 4096); ++i) {
        const float* r = rays + 8 * i;
        Ray ray{{r[0], r[1], r[2]}, {r[4], r[5], r[6]}, r[3], r[7]};
        HitAttr h;
        float* ho = (float*)hits + 4 * i;
        int32_t* hi = (int32_t*)hits + 4 * i;
        if (closestHit(*c, ray, h)) { ho[0] = h.t; hi[1] = h.prim; ho[2] = h.beta; ho[3] = h.gamma; }
        else { ho[0] = ray.tmax; hi[1] = -1; ho[2] = 0; ho[3] = 0; }
      }
    }
  };
  std::vector<std::thread> th;
  for (int i = 1; i < nt; ++i) th.emplace_back(worker);
  worker();
  for (auto& t : th) t.join();
  return MOX_OK;
}
int orc_trace_shadow(orc_ctx* c, const float* rays, size_t n, float* out) {
  if (!c || (n && (!rays || !out))) return MOX_ERR_INVALID;
  if (!c->built) { c->err = "trace before build_accel"; return MOX_ERR_STATE; }
  for (size_t i = 0; i < n; ++i) {
    const float* r = rays + 8 * i;
    Ray ray{{r[0], r[1], r[2]}, {r[4], r[5], r[6]}, r[3], r[7]};
    float3 a = shadowTransmittance(*c, ray);
    out[3 * i] = a.x; out[3 * i + 1] = a.y; out[3 * i + 2] = a.z;
  }
  return MOX_OK;
}

// Closest hit with the five attributes the intersection programs write (Geometry.cu:8-12):
// attrs: n x 15 floats geoNormal, shadingNormal, frontHitPoint, backHitPoint, texcoord.
int orc_trace_closest_attrs(orc_ctx* c, const float* rays, size_t n, void* hits, float* attrs) {
  if (!c || (n && (!rays || !hits || !attrs))) return MOX_ERR_INVALID;
  if (!c->built) { c->err = "trace before build_accel"; return MOX_ERR_STATE; }
  for (size_t i = 0; i < n; ++i) {
    const float* r = rays + 8 * i;
    Ray ray{{r[0], r[1], r[2]}, {r[4], r[5], r[6]}, r[3], r[7]};
    HitAttr h;
    float* ho = (float*)hits + 4 * i;
    int32_t* hi = (int32_t*)hits + 4 * i;
    float* a = attrs + 15 * i;
    if (closestHit(*c, ray, h)) {
      ho[0] = h.t; hi[1] = h.prim;
      bool tri = c->prims[h.prim].type == PT_TRI;
      ho[2] = tri ? h.beta : 0.f; ho[3] = tri ? h.gamma : 0.f;
      const float3* v[5] = {&h.geoNormal, &h.shadingNormal, &h.front, &h.back, &h.texcoord};
      for (int k = 0; k < 5; ++k) { a[3 * k] = v[k]->x; a[3 * k + 1] = v[k]->y; a[3 * k + 2] = v[k]->z; }
    } else {
      ho[0] = ray.tmax; hi[1] = -1; ho[2] = 0; ho[3] = 0;
      for (int k = 0; k < 15; ++k) a[k] = 0.f;
    }
  }
  return MOX_OK;
}
// Bounds as the bbox programs define them (Geometry.cu:57-63,93-110,162-175): out = min, max;
// returns 1 in *valid when the primitive enters the acceleration structure.
int orc_prim_bounds(orc_ctx* c, uint32_t prim, float out[6], int* valid) {
  if (!c || prim >= c->prims.size() || !out) return MOX_ERR_INVALID;
  Box b = primBox(*c, c->prims[prim]);
  out[0] = b.lo.x; out[1] = b.lo.y; out[2] = b.lo.z; out[3] = b.hi.x; out[4] = b.hi.y; out[5] = b.hi.z;
  if (valid) *valid = b.valid ? 1 : 0;
  return MOX_OK;
}

// ---- unit-test hooks
uint32_t orc_tea16(uint32_t a, uint32_t b) { return tea<16>(a, b); }
uint32_t orc_lcg(int32_t* seed) { Rng r; r.seed = *seed; uint32_t v = lcg(r); *seed = r.seed; return v; }
float orc_rand(int32_t* seed) { Rng r; r.seed = *seed; float v = rnd(r); *seed = r.seed; return v; }
void orc_philox(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  philox4x32_10(ctr[0], ctr[1], ctr[2], ctr[3], key[0], key[1], out);
}
static float3 a3(const float* p) { return {p[0], p[1], p[2]}; }
static void s3(float* p, const float3& v) { p[0] = v.x; p[1] = v.y; p[2] = v.z; }
void orc_disney_eval(const DisneyParams* mp, const float bc[3], const float N[3], const float L[3], const float V[3],
                     const float H[3], float out[3]) {
  s3(out, disneyEval(*mp, a3(bc), a3(N), a3(L), a3(V), a3(H)));
}
float orc_disney_pdf(const DisneyParams* mp, const float N[3], const float L[3], const float V[3], const float H[3]) {
  return disneyPdf(*mp, a3(N), a3(L), a3(V), a3(H));
}
void orc_disney_sample(int32_t* seed, const DisneyParams* mp, const float N[3], const float V[3], float L[3], float H[3]) {
  Rng r; r.seed = *seed;
  float3 l{}, h{};
  disneySample(r, *mp, a3(N), l, a3(V), h);
  *seed = r.seed; s3(L, l); s3(H, h);
}
void orc_refine_hitpoint(const float hit[3], const float dir[3], const float n[3], const float p[3], float back[3],
                         float front[3]) {
  float3 b, f;
  refineHitpoint(a3(hit), a3(dir), a3(n), a3(p), b, f);
  s3(back, b); s3(front, f);
}
int orc_refract(const float i[3], const float n[3], float ior, float out[3]) {
  float3 r; bool ok = refract(r, a3(i), a3(n), ior); s3(out, r); return ok ? 1 : 0;
}
float orc_fresnel(float ci, float ct, float ior) { return fresnel(ci, ct, ior); }
void orc_rand_in_unit_sphere(int32_t* seed, float out[3]) { Rng r; r.seed = *seed; s3(out, randInUnitSphere(r)); *seed = r.seed; }
void orc_rand_in_unit_disk(int32_t* seed, float out[3]) { Rng r; r.seed = *seed; s3(out, randInUnitDisk(r)); *seed = r.seed; }
int32_t orc_fork_seed(int32_t parentSeed, int32_t parentDepth) { Rng r; r.seed = parentSeed; return forkRng(r, parentDepth + 1).seed; }
void orc_offset(const float hit[3], const float n[3], float out[3]) { s3(out, offsetPoint(a3(hit), a3(n))); }
float orc_gtr1(float ndh, float a) { return GTR1(ndh, a); }
float orc_gtr2(float ndh, float a) { return GTR2(ndh, a); }
float orc_gtr2_aniso(float ndh, float hx, float hy, float ax, float ay) { return GTR2Aniso(ndh, hx, hy, ax, ay); }
float orc_schlick_fresnel(float u) { return schlickFresnel(u); }
float orc_smith_ggx(float ndv, float a) { return smithGGgx(ndv, a); }
float orc_smith_ggx_aniso(float ndv, float vx, float vy, float ax, float ay) { return smithGGgxAniso(ndv, vx, vy, ax, ay); }
float orc_power_heuristic(float a, float b) { return powerHeuristic(a, b); }
void orc_srgb2lin(const float v[3], float out[3]) { s3(out, srgb2lin(a3(v))); }

}  // extern "C"
