// wavefront.cu — the render kernels.  The reference is a recursive OptiX megakernel
// (camera() -> rtTrace -> closest-hit program -> rtTrace ...); here one sample of every pixel
// is a path in a wavefront, advanced one bounce per iteration:
//
//   k_generate   camera()                      Camera.cu:21-36
//   k_traverse   rtTrace: persistent-thread traversal, closest hit (extend rays) or shadow
//                transmittance (disneyAnyHit, Material.cu:225-232) — traverse.cuh
//   k_classify   the depth test every scattering program starts with (Material.cu:29,50,73,119); surviving
//                paths are binned into per-material queues by the shade class the traversal kernel left in
//                the hit record.  Paths that end here — miss (miss.cu:10-12), light() (Material.cu:238-240),
//                depth exceeded — are not touched again: k_accumulate adds their last term.
//   k_shade_*    lambertian / metal / glass / disney   Material.cu:28-223, disney.h
//   k_apply      adds the NEE terms to the path radiance in light order (deterministic)
//   k_accumulate clamp + accuBuffer +=                 Camera.cu:39-41
//
// Every reference program is affine in the child radiance (colour = A * child + B), so a path
// carries throughput T and radiance R: R += T*B, T *= A (SURVEY.md Appendix A.7).
#include "wavefront.h"

#include <atomic>
#include <cstdlib>

#include "shading.cuh"
#include "traverse.cuh"
#include "traverse_wide.cuh"

namespace {

constexpr int TPB = 256;

__device__ __forceinline__ uint32_t queuePush(uint32_t* counter) {
  // warp-aggregated atomic increment
  uint32_t mask = __activemask();
  int leader = __ffs(mask) - 1;
  int lane = threadIdx.x & 31;
  uint32_t base = 0;
  if (lane == leader) base = atomicAdd(counter, (uint32_t)__popc(mask));
  base = __shfl_sync(mask, base, leader);
  return base + __popc(mask & ((1u << lane) - 1u));
}

struct PathCtx {
  uint32_t path, pixel;
  int32_t launchSeed;
};

__device__ __forceinline__ PathCtx pathCtx(const LaunchCtx& c, uint32_t path) {
  PathCtx p;
  p.path = path;
  uint32_t s = path / c.nOwned, j = path - s * c.nOwned;
  p.pixel = __ldg(&c.ownedPix[j]);
  p.launchSeed = __ldg(&c.pb.seeds[s]);
  return p;
}

// ------------------------------------------------------------------ generate (Camera.cu:21-36)
template <int RM>
__global__ void __launch_bounds__(TPB) k_generate(LaunchCtx c, uint32_t nPaths) {
  uint32_t p = blockIdx.x * TPB + threadIdx.x;
  if (p >= nPaths) return;
  PathCtx pc = pathCtx(c, p);
  const RenderParams& rp = c.rp;
  uint32_t x = pc.pixel % rp.W, y = pc.pixel / rp.W;
  int st = RM == 0 ? (int)tea16(pc.pixel, (uint32_t)pc.launchSeed) : 0;
  RngT<RM> rng = makeRng<RM>(st, pc.pixel, (uint32_t)pc.launchSeed, 1u);
  const CamParams& cp = rp.cam;
  float3 lens = cp.lensRadius * randInUnitDisk(rng);
  float3 offset = f3(cp.u) * lens.x + f3(cp.v) * lens.y;
  float r1 = rng.rnd();
  float r2 = rng.rnd();
  float sx = ((float)x + r1 - 0.5f) / (float)rp.W;
  float sy = ((float)y + r2 - 0.5f) / (float)rp.H;
  float3 o = f3(cp.origin) + offset;
  float3 d = normalize(f3(cp.scrLowerLeftCorner) + sx * f3(cp.horizontal) + sy * f3(cp.vertical) - f3(cp.origin) - offset);
  c.pb.rayO[p] = make_float4(o.x, o.y, o.z, rp.eps);
  c.pb.rayD[p] = make_float4(d.x, d.y, d.z, MOX_RAY_TMAX);
  c.pb.thr[p] = make_float4(1.f, 1.f, 1.f, 0.f);
  c.pb.rad[p] = make_float4(0.f, 0.f, 0.f, 0.f);
  c.pb.state[p] = rng.state;
  c.pb.qCur[p] = p;
}

// ------------------------------------------------------------------ traversal + classify
constexpr int TRAV_TPB = MOX_TRAV_TPB;
#ifndef MOX_TRAV_MINBLOCKS
#define MOX_TRAV_MINBLOCKS 10  // caps the kernel at 48 registers: measured 983 (55 regs) -> 1022 Mrays/s; 12 blocks (40 regs): 1005
#endif

template <bool ANYHIT, bool COUNT, bool CLASSIFY>
__global__ void __launch_bounds__(TRAV_TPB, MOX_TRAV_MINBLOCKS) k_traverse(SceneView s, TraceJob job) {
  traverseWarpPersistent<ANYHIT, COUNT, CLASSIFY>(s, job);
}
// Watertight variants (MOX_ACCEL_WATERTIGHT): six more per-ray values (shear axes and scales), so one CTA less per SM
// than the default kernels instead of spills.
template <bool ANYHIT, bool COUNT, bool CLASSIFY>
__global__ void __launch_bounds__(TRAV_TPB, 8) k_traverse_wt(SceneView s, TraceJob job) {
  traverseWarpPersistent<ANYHIT, COUNT, CLASSIFY, true>(s, job);
}
template <bool ANYHIT, bool COUNT, bool CLASSIFY>
__global__ void __launch_bounds__(TRAV_TPB, 8) k_traverse_wide_wt(SceneView s, TraceJob job) {
  traverseWidePersistent<ANYHIT, COUNT, CLASSIFY, true>(s, job);
}

#ifndef MOX_WIDE_MINBLOCKS
#define MOX_WIDE_MINBLOCKS 9   // 56 registers, no spills: measured 8 -> 1229, 9 -> 1258, 10 -> 1240 Mrays/s (before the weighted vote: 1064 / 1090 / 1069)
#endif
template <bool ANYHIT, bool COUNT, bool CLASSIFY>
__global__ void __launch_bounds__(TRAV_TPB, MOX_WIDE_MINBLOCKS) k_traverse_wide(SceneView s, TraceJob job) {
  traverseWidePersistent<ANYHIT, COUNT, CLASSIFY>(s, job);
}
// The terminal bounce: closest light, then an any-hit query bounded by it (traverse_wide.cuh, TERMINAL).
template <bool COUNT>
__global__ void __launch_bounds__(TRAV_TPB, MOX_WIDE_MINBLOCKS) k_traverse_wide_terminal(SceneView s, TraceJob job, TerminalLights tl) {
  traverseWidePersistent<false, COUNT, true, false, true>(s, job, tl);
}
template <bool COUNT>
__global__ void __launch_bounds__(TRAV_TPB, 8) k_traverse_wide_wt_terminal(SceneView s, TraceJob job, TerminalLights tl) {
  traverseWidePersistent<false, COUNT, true, true, true>(s, job, tl);
}

// Bins the paths of the current queue by the shade class in their hit record.  A miss, a light and a path
// beyond rayMaxDepth end here without a write: their last term is added by k_accumulate from the same record.
// Queue slots are reserved once per block and class: a push per warp is a million atomics on one address per
// launch at 4K x 4 spp, and same-address atomics retire about one per nanosecond — the kernel ran at 6-8 % issue
// utilisation waiting for them (ncu, profiles/r2a_*).
__global__ void __launch_bounds__(TPB) k_classify(LaunchCtx c, const uint32_t* __restrict__ queue, uint32_t count,
                                                  const uint32_t* __restrict__ countPtr, uint32_t depth) {
  __shared__ uint32_t sCount[TPB / 32][Q_COUNT];   // per warp and class: lanes that push
  __shared__ uint32_t sBase[Q_COUNT];
  const uint32_t i = blockIdx.x * TPB + threadIdx.x;
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  if (countPtr) count = __ldg(countPtr);
  uint32_t cls = Q_COUNT, path = 0;    // Q_COUNT: nothing to push
  if (i < count) {
    path = queue[i];
    const int bits = __float_as_int(c.pb.hit[path].y);
    const RenderParams& rp = c.rp;
    // miss: bits < 0; light(): terminal; the incoming payload colour is always (1,1,1): |colour| = sqrt(3)
    if (bits >= 0 && ((uint32_t)bits >> MOX_HIT_ID_BITS) < MOX_CLASS_LIGHT && !(depth > rp.maxDepth || length(mk3(1.f)) < rp.minIntensity))
      cls = (uint32_t)bits >> MOX_HIT_ID_BITS;   // classes 0..3 are the queue indices
  }
  uint32_t rankInWarp = 0;
#pragma unroll
  for (uint32_t k = 0; k < Q_COUNT; ++k) {
    const unsigned m = __ballot_sync(0xffffffffu, cls == k);
    if (lane == 0) sCount[warp][k] = (uint32_t)__popc(m);
    if (cls == k) rankInWarp = (uint32_t)__popc(m & ((1u << lane) - 1u));
  }
  __syncthreads();
  if (threadIdx.x < Q_COUNT) {
    uint32_t total = 0;
    for (int w = 0; w < TPB / 32; ++w) { const uint32_t n = sCount[w][threadIdx.x]; sCount[w][threadIdx.x] = total; total += n; }
    sBase[threadIdx.x] = total ? atomicAdd(c.bc + C_MAT0 + threadIdx.x, total) : 0u;
  }
  __syncthreads();
  if (cls < Q_COUNT) c.pb.qMat[cls][sBase[cls] + sCount[warp][cls] + rankInWarp] = path;
}

// ------------------------------------------------------------------ hit attributes (Geometry.cu)
struct Attr { float3 Ng, Ns, front, back, hitPoint; float u, v; };

__device__ __forceinline__ float3 ld3(const float* p, int i) { return mk3(__ldg(p + 3 * i), __ldg(p + 3 * i + 1), __ldg(p + 3 * i + 2)); }

// beta / gamma of a triangle hit are not stored by the traversal kernel: they are recomputed here with the
// operation sequence of the primitive test (triTest) on the same operands — bit-identical values.
__device__ __forceinline__ void triBarycentrics(bool watertight, const float3& o, const float3& d, const float3& p0, const float3& p1,
                                                const float3& p2, float& beta, float& gamma) {
  float t;
  if (watertight) triTestWt(wtPrep(d), o, 0.f, p0, p1, p2, t, beta, gamma);
  else triTest(o, d, 0.f, p0, p1 - p0, p0 - p2, t, beta, gamma);
}

__device__ __forceinline__ Attr hitAttributes(const SceneView& s, const PrimDesc& pd, const float3& o, const float3& d,
                                               float t, bool needShading) {
  Attr a;
  float beta = 0.f, gamma = 0.f;
  uint32_t type = pd.typeMat & 3u;
  a.hitPoint = o + t * d;
  a.u = a.v = 0.f;
  if (type == PT_SPHERE) {
    float4 cr = __ldg(&s.analytic[pd.geom].a);
    a.Ng = normalize(o + t * d - mk3(cr));
    a.Ns = a.Ng;
    a.front = a.back = a.hitPoint;
  } else if (type == PT_QUAD) {
    a.Ng = mk3(__ldg(&s.analytic[pd.geom].a));
    a.Ns = a.Ng;
    a.front = a.back = a.hitPoint;
  } else if (s.shadeRec) {
    const float4* r = s.shadeRec + (size_t)pd.geom * MOX_SHADE_REC_F4;
    const float4 r0 = __ldg(r), r1 = __ldg(r + 1), r2 = __ldg(r + 2);
    const float3 p0 = mk3(r0), p1 = mk3(r1), p2 = mk3(r2);
    float3 e0 = p1 - p0, e1 = p0 - p2;
    a.Ng = normalize(cross(e1, e0));
    a.Ns = a.Ng;
    a.front = a.back = a.hitPoint;
    if (needShading) {
      const uint32_t flags = __float_as_uint(r0.w);
      if (flags) {
        const float4 r3 = __ldg(r + 3), r4 = __ldg(r + 4), r5 = __ldg(r + 5);
        triBarycentrics(s.watertight != 0, o, d, p0, p1, p2, beta, gamma);
        if (flags & 1u) a.Ns = normalize(mk3(r4) * beta + mk3(r5) * gamma + mk3(r3) * (1.f - beta - gamma));
        if (flags & 2u) {
          float w = 1.0f - beta - gamma;
          a.u = r3.w * beta + r5.w * gamma + r1.w * w;
          a.v = r4.w * beta + __ldg(&r[6].x) * gamma + r2.w * w;
        }
      }
      refineHitpoint(a.hitPoint, d, a.Ng, p0, a.back, a.front);
    }
  } else {
    const TriIdx* ti = s.tris + pd.geom;
    int v0 = __ldg(&ti->v[0]), v1 = __ldg(&ti->v[1]), v2 = __ldg(&ti->v[2]);
    float3 p0 = ld3(s.verts, v0), p1 = ld3(s.verts, v1), p2 = ld3(s.verts, v2);
    float3 e0 = p1 - p0, e1 = p0 - p2;
    a.Ng = normalize(cross(e1, e0));
    a.Ns = a.Ng;
    a.front = a.back = a.hitPoint;
    if (needShading) {
      int n0 = __ldg(&ti->n[0]);
      if (n0 >= 0 || __ldg(&ti->t[0]) >= 0) triBarycentrics(s.watertight != 0, o, d, p0, p1, p2, beta, gamma);
      if (n0 >= 0) {
        int n1 = __ldg(&ti->n[1]), n2 = __ldg(&ti->n[2]);
        a.Ns = normalize(ld3(s.normals, n1) * beta + ld3(s.normals, n2) * gamma + ld3(s.normals, n0) * (1.f - beta - gamma));
      }
      int t0 = __ldg(&ti->t[0]);
      if (t0 >= 0) {
        int t1 = __ldg(&ti->t[1]), t2 = __ldg(&ti->t[2]);
        float w = 1.0f - beta - gamma;
        a.u = __ldg(s.uvs + 2 * t1) * beta + __ldg(s.uvs + 2 * t2) * gamma + __ldg(s.uvs + 2 * t0) * w;
        a.v = __ldg(s.uvs + 2 * t1 + 1) * beta + __ldg(s.uvs + 2 * t2 + 1) * gamma + __ldg(s.uvs + 2 * t0 + 1) * w;
      }
      refineHitpoint(a.hitPoint, d, a.Ng, p0, a.back, a.front);
    }
  }
  return a;
}

// Material.cu:126-132: constant colour, or rtTex2D<float4>(albedoID, u, v).rgb
__device__ __forceinline__ float3 disneyBaseColor(const SceneView& s, const DisneyParams& dp, float u, float v) {
  if (dp.albedoID == MOX_TEXTURE_ID_NULL) return f3(dp.color);
  float4 t = tex2D<float4>(s.textures[dp.albedoID - 1], u, v);
  return mk3(t.x, t.y, t.z);
}

template <int RM>
struct ShadeIn {
  uint32_t path;
  float3 o, d;
  float t;
  PrimDesc pd;
  const GpuMaterial* m;
  RngT<RM> rng;
};

template <int RM>
__device__ __forceinline__ ShadeIn<RM> loadShadeIn(const LaunchCtx& c, uint32_t path, uint32_t depth) {
  ShadeIn<RM> s;
  s.path = path;
  float4 ro = c.pb.rayO[path], rd = c.pb.rayD[path];
  float2 h = c.pb.hit[path];
  s.o = mk3(ro); s.d = mk3(rd);
  s.t = h.x;
  s.pd = c.scene.prims[__float_as_uint(h.y) & MOX_HIT_ID_MASK];
  s.m = c.scene.mats + (s.pd.typeMat >> 2);
  if (RM == 0) {
    s.rng = makeRng<RM>(c.pb.state[path], 0u, 0u, depth);
  } else {
    PathCtx pc = pathCtx(c, path);
    s.rng = makeRng<RM>(c.pb.state[path], pc.pixel, (uint32_t)pc.launchSeed, depth);
  }
  return s;
}

// Writes the spawned ray, the new throughput and RNG state, and queues the path at slot `pos` of the next queue.
__device__ __forceinline__ void spawnAt(const LaunchCtx& c, uint32_t path, const float3& o, const float3& d, const float3& A,
                                        int childState, uint32_t pos) {
  c.pb.rayO[path] = make_float4(o.x, o.y, o.z, c.rp.eps);
  c.pb.rayD[path] = make_float4(d.x, d.y, d.z, MOX_RAY_TMAX);
  float4 T = c.pb.thr[path];
  float3 t = mk3(T) * A;
  c.pb.thr[path] = make_float4(t.x, t.y, t.z, 0.f);
  c.pb.state[path] = childState;
  c.pb.qNext[pos] = path;
}
__device__ __forceinline__ void spawn(const LaunchCtx& c, uint32_t path, const float3& o, const float3& d, const float3& A,
                                      int childState) {
  spawnAt(c, path, o, d, A, childState, queuePush(c.bc + C_NEXT));
}

// lambertian (Material.cu:28-43) and metal (:49-66)
template <bool METAL, int RM>
__global__ void __launch_bounds__(TPB) k_shade_diffuse(LaunchCtx c, uint32_t count, uint32_t depth) {
  uint32_t i = blockIdx.x * TPB + threadIdx.x;
  if (i >= count) return;
  ShadeIn<RM> s = loadShadeIn<RM>(c, c.pb.qMat[METAL ? Q_METAL : Q_LAMBERT][i], depth);
  Attr a = hitAttributes(c.scene, s.pd, s.o, s.d, s.t, false);
  float3 v = randInUnitSphere(s.rng);
  float3 dir, albedo;
  if (METAL) {
    dir = normalize(reflect3(s.d, a.Ng) + s.m->met.fuzz * v);
    albedo = f3(s.m->met.albedo);
  } else {
    dir = normalize(a.Ng + v);
    albedo = f3(s.m->lam.albedo);
  }
  spawn(c, s.path, a.hitPoint, dir, albedo, s.rng.forkState((int)depth + 1));
}

// glass (Material.cu:72-110) and disney/GLASS (:134-168)
template <int RM>
__global__ void __launch_bounds__(TPB) k_shade_dielectric(LaunchCtx c, uint32_t count, uint32_t depth) {
  uint32_t i = blockIdx.x * TPB + threadIdx.x;
  if (i >= count) return;
  ShadeIn<RM> s = loadShadeIn<RM>(c, c.pb.qMat[Q_DIELECTRIC][i], depth);
  Attr a = hitAttributes(c.scene, s.pd, s.o, s.d, s.t, true);
  float ior;
  float3 tint;
  if (s.m->kind == MOX_MAT_GLASS) { ior = s.m->gls.refIdx; tint = f3(s.m->gls.albedo); }
  else { ior = 1.45f; tint = disneyBaseColor(c.scene, s.m->dis, a.u, a.v); }
  float3 normal = a.Ns;
  float cosI = -dot(s.d, normal);
  float refIdx;
  if (cosI > 0.f) { refIdx = ior; }
  else { refIdx = 1.f / ior; cosI = -cosI; normal = -normal; }
  float3 refracted;
  bool tir = !refract3(refracted, s.d, normal, refIdx);
  float cosT = -dot(normal, refracted);
  float reflectProb = tir ? 1.f : fresnelDielectric(cosI, cosT, refIdx);
  int childState = s.rng.forkState((int)depth + 1);  // forked BEFORE the coin flip (Material.cu:100-101)
  float3 o, dir;
  if (s.rng.rnd() < reflectProb) { o = a.front; dir = reflect3(s.d, normal); }
  else { o = a.back; dir = refracted; }
  spawn(c, s.path, o, dir, tint, childState);
}

// disney/NORMAL (Material.cu:170-222)
constexpr int DISNEY_TPB = 128;
#ifndef MOX_DISNEY_MINBLOCKS
#define MOX_DISNEY_MINBLOCKS 6
#endif

// One reservation of `n` consecutive queue slots per thread with ONE atomic per block: warp scan, per-warp totals in
// shared memory, thread 0 adds the block total to the counter.  Every thread of the block must call it.  Returns the
// first slot of the calling thread.  (A push per warp and light is ~5 M atomics on two addresses per Disney launch
// at 4K x 4 spp; same-address atomics retire about one per nanosecond.)
__device__ __forceinline__ uint32_t blockReserve(uint32_t n, uint32_t* counter, uint32_t (&sWarp)[DISNEY_TPB / 32], uint32_t& sBase) {
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  uint32_t incl = n;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= (uint32_t)o) incl += t; }
  if (lane == 31u) sWarp[warp] = incl;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t total = 0;
#pragma unroll
    for (int w = 0; w < DISNEY_TPB / 32; ++w) { const uint32_t t = sWarp[w]; sWarp[w] = total; total += t; }
    sBase = total ? atomicAdd(counter, total) : 0u;
  }
  __syncthreads();
  const uint32_t first = sBase + sWarp[warp] + incl - n;
  __syncthreads();   // the shared words are reused by the next reservation
  return first;
}

template <int RM, bool F>
__global__ void __launch_bounds__(DISNEY_TPB, MOX_DISNEY_MINBLOCKS) k_shade_disney(LaunchCtx c, uint32_t count, uint32_t depth) {
  __shared__ uint32_t sWarp[DISNEY_TPB / 32];
  __shared__ uint32_t sBase;
  const uint32_t i = blockIdx.x * DISNEY_TPB + threadIdx.x;
  const bool live = i < count;          // no early return: the block reserves its queue slots together
  const uint32_t iq = live ? i : count - 1u;
  ShadeIn<RM> s = loadShadeIn<RM>(c, c.pb.qMat[Q_DISNEY][iq], depth);
  Attr a = hitAttributes(c.scene, s.pd, s.o, s.d, s.t, true);
  const DisneyParams dp = s.m->dis;
  float3 N = faceforward3(a.Ns, -s.d, a.Ng);
  float3 V = -s.d;
  float3 baseColor = disneyBaseColor(c.scene, dp, a.u, a.v);
  DisneyHit<F> dh(dp, baseColor, N);
  dh.setView(V);
  float3 Tprev = mk3(c.pb.thr[s.path]);
  float3 L, H;
  const int nL = c.scene.nLights;
  uint32_t shadowCount = 0;
  for (int g0 = 0; g0 < nL; g0 += 32) {   // lights in groups of 32: one bit per light that needs a shadow ray
    uint32_t traceMask = 0;
    const int g1 = min(nL, g0 + 32);
    for (int li = g0; li < g1; ++li) {
      const LightParams* lp = c.scene.lights + li;
      float3 lpos = mk3(__ldg(&lp->position.x), __ldg(&lp->position.y), __ldg(&lp->position.z));
      float3 pointOnLight, normalOnLight;
      if (__ldg((const int*)&lp->shape) == SPHERE) {
        pointOnLight = lpos + randInUnitSphere(s.rng) * __ldg(&lp->radius);
        normalOnLight = normalize(pointOnLight - lpos);
      } else {
        float r1 = s.rng.rnd();
        float r2 = s.rng.rnd();
        pointOnLight = lpos + f3(lp->u) * r1 + f3(lp->v) * r2;
        normalOnLight = mk3(__ldg(c.scene.lightN + li));
      }
      L = pointOnLight - a.front;
      float lightDst = length(L);
      L = normalize(L);
      size_t slot = (size_t)li * count + i;  // light-major: neighbouring lanes aim at the same light
      float3 contrib = mk3(0.f);
      if (dot(L, N) > 0.f && dot(L, normalOnLight) < 0.f) {
        shadowCount++;
        H = bnormalize<F>(L + V);
        float lightPdf = bdiv<F>(bdiv<F>(lightDst * lightDst, __ldg(&lp->area)), dot(normalOnLight, -L));
        float dr;
        float objPdf = dh.pdf(L, H, dr);
        if (lightPdf > 0 && objPdf > 0) {
          float3 brdf = dh.eval(L, H, dr);
          contrib = powerHeuristic<F>(lightPdf, objPdf) * brdf * f3(lp->emission) * bdiv<F>(1.0f, fmaxf(0.001f, lightPdf));
        }
      }
      float3 pc = Tprev * contrib;
      // a zero contribution needs no shadow ray (it is still counted, as the reference traces it)
      if (live) {
        c.pb.shC[slot] = make_float4(pc.x, pc.y, pc.z, 0.f);
        if (pc.x != 0.f || pc.y != 0.f || pc.z != 0.f) {
          c.pb.shD[slot] = make_float4(L.x, L.y, L.z, lightDst - c.rp.eps);
          traceMask |= 1u << (li - g0);
        }
      }
    }
    uint32_t pos = blockReserve((uint32_t)__popc(traceMask), c.bc + C_SHQ, sWarp, sBase);
    while (traceMask) {
      const int b = __ffs(traceMask) - 1;
      traceMask &= traceMask - 1u;
      c.pb.shQueue[pos++] = (uint32_t)((size_t)(g0 + b) * count + i);
    }
  }
  if (nL && live) c.pb.shO[i] = make_float4(a.front.x, a.front.y, a.front.z, c.rp.eps);  // one origin for all lights of this hit
  if (live) {  // + emission
    float3 e = f3(dp.emission);
    if (e.x != 0.f || e.y != 0.f || e.z != 0.f) {
      float3 r = mk3(c.pb.rad[s.path]) + Tprev * e;
      c.pb.rad[s.path] = make_float4(r.x, r.y, r.z, 0.f);
    }
  }
  disneySample(s.rng, dp, N, L, V, H);
  bool spawned = false;
  float3 A = mk3(0.f);
  if (live && dot(N, L) > 0.0f && dot(N, V) > 0.0f) {
    float dr;
    float pdf = dh.pdf(L, H, dr);
    if (pdf > 0) {
      float3 brdf = dh.eval(L, H, dr);
      A = brdf * bdiv<F>(1.0f, pdf);
      spawned = true;
    }
  }
  // shadow-ray statistics ride in the high half of the same reservation: one more atomic per block, not per warp
  const uint32_t nextPos = blockReserve(spawned ? 1u : 0u, c.bc + C_NEXT, sWarp, sBase);
  {
    uint32_t sc = live ? shadowCount : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sc += __shfl_xor_sync(0xffffffffu, sc, o);
    if ((threadIdx.x & 31u) == 0u && sc) atomicAdd(c.pb.counters + C_SHADOW, sc);
  }
  if (spawned) spawnAt(c, s.path, a.front, L, A, s.rng.forkState((int)depth + 1), nextPos);
  // no indirect ray: the path ends with what it has; its (stale) hit record must not be read as a terminal hit
  else if (live) c.pb.hit[s.path].y = __int_as_float(MOX_HIT_DEAD);
}

__global__ void __launch_bounds__(TPB) k_apply(LaunchCtx c, uint32_t count) {
  uint32_t i = blockIdx.x * TPB + threadIdx.x;
  if (i >= count) return;
  uint32_t path = c.pb.qMat[Q_DISNEY][i];
  const int nL = c.scene.nLights;
  float3 direct = mk3(0.f);
  for (int li = 0; li < nL; ++li) direct += mk3(c.pb.shC[(size_t)li * count + i]);
  float3 r = mk3(c.pb.rad[path]) + direct;
  c.pb.rad[path] = make_float4(r.x, r.y, r.z, 0.f);
}

// The luminance sums of adaptive sampling for one pixel: y = 0.2126 r + 0.7152 g + 0.0722 b rounded step by step in
// float32 (no contraction, so a host model reproduces it), y and y^2 summed in float64 in launch order.
template <bool ADAPTIVE>
struct LumSums {
  __device__ __forceinline__ LumSums(const PixelStats&, uint32_t) {}
  __device__ __forceinline__ void add(float, float, float) {}
  __device__ __forceinline__ void store(const PixelStats&, uint32_t, uint32_t) {}
};
template <>
struct LumSums<true> {
  double s1, s2;
  __device__ __forceinline__ LumSums(const PixelStats& ps, uint32_t pix) : s1(ps.s1[pix]), s2(ps.s2[pix]) {}
  __device__ __forceinline__ void add(float r, float g, float b) {
    const float y = __fadd_rn(__fadd_rn(__fmul_rn(0.2126f, r), __fmul_rn(0.7152f, g)), __fmul_rn(0.0722f, b));
    s1 = __dadd_rn(s1, (double)y);
    s2 = __dadd_rn(s2, __dmul_rn((double)y, (double)y));
  }
  __device__ __forceinline__ void store(const PixelStats& ps, uint32_t pix, uint32_t nSamples) {
    ps.s1[pix] = s1; ps.s2[pix] = s2; ps.n[pix] += nSamples;
  }
};

// Camera.cu:39-41 — samples of one pixel are added in launch order, so a batch of S samples
// gives bit-identical sums to S successive launches.  ADAPTIVE also adds every sample's luminance to ps; the image
// is the same.  (The body stays in the kernel: moved into an inlined helper, the plain kernel compiled to different
// instructions.)
template <bool ADAPTIVE>
__global__ void __launch_bounds__(TPB) k_accumulate(LaunchCtx c, uint32_t nSamples, PixelStats ps) {
  uint32_t j = blockIdx.x * TPB + threadIdx.x;
  if (j >= c.nOwned) return;
  uint32_t pix = c.ownedPix[j];
  float* a = c.accu + 3 * (size_t)pix;
  float3 acc = mk3(a[0], a[1], a[2]);
  LumSums<ADAPTIVE> lum(ps, pix);
  uint32_t bad = 0;
  for (uint32_t s = 0; s < nSamples; ++s) {
    const size_t p = (size_t)s * c.nOwned + j;
    float4 r = c.pb.rad[p];
    {
      // The path's last term.  Its final hit record says how it ended: miss -> payload colour (1,1,1) * bgColor
      // (miss.cu:10-12); a light -> emission (Material.cu:238-240); a scattering material -> the depth test failed,
      // absorbColor (Material.cu:29,50,73,119); MOX_HIT_DEAD -> shaded without an indirect ray, nothing to add.
      const int bits = __float_as_int(c.pb.hit[p].y);
      if (bits != MOX_HIT_DEAD) {
        float3 B;
        if (bits < 0) B = mk3(1.f) * c.rp.bg;
        else if (((uint32_t)bits >> MOX_HIT_ID_BITS) >= MOX_CLASS_LIGHT) {
          const GpuMaterial* m = c.scene.mats + (__ldg(&c.scene.prims[(uint32_t)bits & MOX_HIT_ID_MASK].typeMat) >> 2);
          B = mk3(__ldg(&m->lgt.emission.x), __ldg(&m->lgt.emission.y), __ldg(&m->lgt.emission.z));
        } else B = c.rp.absorb;
        const float3 rr = mk3(r) + mk3(c.pb.thr[p]) * B;
        r = make_float4(rr.x, rr.y, rr.z, 0.f);
      }
    }
    if (!isfinite(r.x) || !isfinite(r.y) || !isfinite(r.z)) {
      // The reference paints badColor when a launch index raises an OptiX exception (Exception.cu:10-12,
      // MinimalOptiX.cpp:149-151).  A NaN/Inf sample is this path's exception: badColor instead of the
      // sample, counted in mox_stats.nonfinite_samples (SURVEY App. A.8).
      bad++;
      acc.x += c.rp.bad.x; acc.y += c.rp.bad.y; acc.z += c.rp.bad.z;
      lum.add(c.rp.bad.x, c.rp.bad.y, c.rp.bad.z);
      continue;
    }
    const float cx = clampf(r.x, 0.f, 1.f), cy = clampf(r.y, 0.f, 1.f), cz = clampf(r.z, 0.f, 1.f);
    acc.x += cx;
    acc.y += cy;
    acc.z += cz;
    lum.add(cx, cy, cz);
  }
  a[0] = acc.x; a[1] = acc.y; a[2] = acc.z;
  lum.store(ps, pix, nSamples);
  if (bad) atomicAdd(c.pb.counters + C_NONFINITE, bad);
}

// ------------------------------------------------------------------ first-hit AOVs (mox_set_aovs)
// One thread per pixel of the batch's list: its samples s * nOwned + j are added in launch order, so the sums do not
// depend on the batching.  Runs at depth 1 after k_classify, when rayO / rayD still hold the camera rays and hit their
// closest hits; the shade kernels overwrite both.
__global__ void __launch_bounds__(TPB) k_aov(LaunchCtx c, uint32_t nSamples, AovBuffers aov) {
  const uint32_t j = blockIdx.x * TPB + threadIdx.x;
  if (j >= c.nOwned) return;
  const uint32_t pix = c.ownedPix[j];
  float3 alb = mk3(aov.albedo[3 * (size_t)pix], aov.albedo[3 * (size_t)pix + 1], aov.albedo[3 * (size_t)pix + 2]);
  float3 nrm = mk3(aov.normal[3 * (size_t)pix], aov.normal[3 * (size_t)pix + 1], aov.normal[3 * (size_t)pix + 2]);
  float depth = aov.depth[pix];
  uint32_t hits = aov.hits[pix];
  const float3 bg = mk3(fmaxf(0.f, fminf(c.rp.bg.x, 1.f)), fmaxf(0.f, fminf(c.rp.bg.y, 1.f)), fmaxf(0.f, fminf(c.rp.bg.z, 1.f)));
  for (uint32_t s = 0; s < nSamples; ++s) {
    const size_t p = (size_t)s * c.nOwned + j;
    const float2 h = c.pb.hit[p];
    const int bits = __float_as_int(h.y);
    if (bits < 0) { alb = alb + bg; continue; }   // miss: normal 0, no depth
    const PrimDesc pd = c.scene.prims[(uint32_t)bits & MOX_HIT_ID_MASK];
    const GpuMaterial* m = c.scene.mats + (pd.typeMat >> 2);
    const float3 o = mk3(c.pb.rayO[p]), d = mk3(c.pb.rayD[p]);
    const Attr a = hitAttributes(c.scene, pd, o, d, h.x, true);
    float3 A;
    switch (m->kind) {
      case MOX_MAT_LAMBERTIAN: A = f3(m->lam.albedo); break;
      case MOX_MAT_METAL: A = f3(m->met.albedo); break;
      case MOX_MAT_GLASS: A = f3(m->gls.albedo); break;
      case MOX_MAT_DISNEY: A = disneyBaseColor(c.scene, m->dis, a.u, a.v); break;
      default: {
        const float3 e = f3(m->lgt.emission);
        A = mk3(fmaxf(0.f, fminf(e.x, 1.f)), fmaxf(0.f, fminf(e.y, 1.f)), fmaxf(0.f, fminf(e.z, 1.f)));
      }
    }
    alb = alb + A;
    nrm = nrm + faceforward3(a.Ns, -d, a.Ng);
    depth += h.x;
    hits++;
  }
  aov.albedo[3 * (size_t)pix] = alb.x; aov.albedo[3 * (size_t)pix + 1] = alb.y; aov.albedo[3 * (size_t)pix + 2] = alb.z;
  aov.normal[3 * (size_t)pix] = nrm.x; aov.normal[3 * (size_t)pix + 1] = nrm.y; aov.normal[3 * (size_t)pix + 2] = nrm.z;
  aov.depth[pix] = depth;
  aov.hits[pix] = hits;
  aov.n[pix] += nSamples;
}

// ------------------------------------------------------------------ adaptive sampling: the active-pixel list
// One tile of the list per block: SEL_ITEMS consecutive entries per thread, so the survivors of a thread, a warp and
// a block keep their order.
constexpr int SEL_ITEMS = 8;
constexpr int SEL_TILE = TPB * SEL_ITEMS;

// The stopping rule of mox_render_adaptive (include/mox.h), rounded step by step in float64.
__device__ __forceinline__ bool pixelConverged(const PixelStats& ps, const AdaptiveRule& rule, uint32_t pix) {
  const uint32_t n = ps.n[pix];
  if (n < rule.minSpp) return false;
  const double dn = (double)n, s1 = ps.s1[pix], s2 = ps.s2[pix];
  const double m = __ddiv_rn(s1, dn);
  const double var = fmax(0.0, __ddiv_rn(__dsub_rn(s2, __dmul_rn(s1, m)), __dsub_rn(dn, 1.0)));
  const double err = __dsqrt_rn(__ddiv_rn(var, dn));
  return err < fmax(__dmul_rn(rule.rel, m), rule.abs);
}

__device__ __forceinline__ uint32_t blockSum(uint32_t v, uint32_t* sh) {
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if (lane == 0) sh[warp] = v;
  __syncthreads();
  uint32_t t = 0;
#pragma unroll
  for (int w = 0; w < TPB / 32; ++w) t += sh[w];
  return t;
}

// Evaluates the rule for the tile's pixels, adds `remaining` to the skipped launches of the converged ones and counts
// the survivors of the tile.
__global__ void __launch_bounds__(TPB) k_adaptive_select(PixelStats ps, AdaptiveRule rule, const uint32_t* __restrict__ list,
                                                         uint32_t count, uint32_t remaining, uint32_t* __restrict__ tileSums) {
  __shared__ uint32_t sh[TPB / 32];
  const uint32_t base = blockIdx.x * SEL_TILE + threadIdx.x * SEL_ITEMS;
  uint32_t keep = 0;
#pragma unroll
  for (int k = 0; k < SEL_ITEMS; ++k) {
    const uint32_t i = base + k;
    if (i >= count) break;
    const uint32_t pix = list[i];
    if (pixelConverged(ps, rule, pix)) ps.skipped[pix] += remaining;
    else keep++;
  }
  const uint32_t t = blockSum(keep, sh);
  if (threadIdx.x == 0) tileSums[blockIdx.x] = t;
}

// Writes the survivors in list order: the tile's offset is the sum of the tile counts in front of it (a few thousand
// words at most, L2-resident), the offset inside the tile a block scan.  The last tile writes the total.
__global__ void __launch_bounds__(TPB) k_adaptive_compact(PixelStats ps, AdaptiveRule rule, const uint32_t* __restrict__ list,
                                                          uint32_t count, const uint32_t* __restrict__ tileSums,
                                                          uint32_t* __restrict__ out, uint32_t* __restrict__ survivors) {
  __shared__ uint32_t sh[TPB / 32];
  __shared__ uint32_t warpOff[TPB / 32];
  uint32_t part = 0;
  for (uint32_t t = threadIdx.x; t < blockIdx.x; t += TPB) part += tileSums[t];
  const uint32_t tileOffset = blockSum(part, sh);
  __syncthreads();   // sh is reused below
  const uint32_t base = blockIdx.x * SEL_TILE + threadIdx.x * SEL_ITEMS;
  uint32_t keepMask = 0, v = 0;
#pragma unroll
  for (int k = 0; k < SEL_ITEMS; ++k) {
    const uint32_t i = base + k;
    if (i < count && !pixelConverged(ps, rule, list[i])) { keepMask |= 1u << k; v++; }
  }
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= (uint32_t)o) incl += t; }
  if (lane == 31) sh[warp] = incl;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t run = 0;
    for (int w = 0; w < TPB / 32; ++w) { warpOff[w] = run; run += sh[w]; }
    if (blockIdx.x == gridDim.x - 1) *survivors = tileOffset + run;
  }
  __syncthreads();
  uint32_t pos = tileOffset + warpOff[warp] + incl - v;
  while (keepMask) {
    const int k = __ffs(keepMask) - 1;
    keepMask &= keepMask - 1u;
    out[pos++] = list[base + k];
  }
}

// ------------------------------------------------------------------ raw ray queries
// out[i] = transmittance (the shC buffer is pre-set to 1)
// scene upload: gathers each triangle's vertices, normals and uvs into one 128-byte record (gpu_types.h)
__global__ void k_build_shade_records(const TriIdx* __restrict__ tris, const float* __restrict__ verts, const float* __restrict__ normals,
                                      const float* __restrict__ uvs, uint32_t n, float4* __restrict__ out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const TriIdx t = tris[i];
  const bool hasN = t.n[0] >= 0, hasT = t.t[0] >= 0;
  float3 p[3], nn[3];
  float2 uv[3];
  for (int k = 0; k < 3; ++k) {
    p[k] = ld3(verts, t.v[k]);
    nn[k] = hasN ? ld3(normals, t.n[k]) : mk3(0.f);
    uv[k] = hasT ? make_float2(uvs[2 * t.t[k]], uvs[2 * t.t[k] + 1]) : make_float2(0.f, 0.f);
  }
  float4* r = out + (size_t)i * MOX_SHADE_REC_F4;
  r[0] = make_float4(p[0].x, p[0].y, p[0].z, __uint_as_float((hasN ? 1u : 0u) | (hasT ? 2u : 0u)));
  r[1] = make_float4(p[1].x, p[1].y, p[1].z, uv[0].x);
  r[2] = make_float4(p[2].x, p[2].y, p[2].z, uv[0].y);
  r[3] = make_float4(nn[0].x, nn[0].y, nn[0].z, uv[1].x);
  r[4] = make_float4(nn[1].x, nn[1].y, nn[1].z, uv[1].y);
  r[5] = make_float4(nn[2].x, nn[2].y, nn[2].z, uv[2].x);
  r[6] = make_float4(uv[2].y, 0.f, 0.f, 0.f);
  r[7] = make_float4(0.f, 0.f, 0.f, 0.f);
}

__global__ void k_fill_ones(float4* __restrict__ p, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = make_float4(1.f, 1.f, 1.f, 0.f);
}
__global__ void k_copy_rgb(const float4* __restrict__ src, float* __restrict__ dst, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { float4 v = src[i]; dst[3 * i] = v.x; dst[3 * i + 1] = v.y; dst[3 * i + 2] = v.z; }
}
// split interleaved (o,tmin,d,tmax) rays into the two arrays the traversal kernel reads
__global__ void k_split_rays(const float4* __restrict__ rays, float4* __restrict__ o, float4* __restrict__ d, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { o[i] = rays[2 * i]; d[i] = rays[2 * i + 1]; }
}

__global__ void k_pack_owned(const float* __restrict__ accu, const uint32_t* __restrict__ ownedPix, uint32_t nOwned, float* __restrict__ dst) {
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= nOwned) return;
  uint32_t pix = ownedPix[j];
  dst[3 * (size_t)j] = accu[3 * (size_t)pix];
  dst[3 * (size_t)j + 1] = accu[3 * (size_t)pix + 1];
  dst[3 * (size_t)j + 2] = accu[3 * (size_t)pix + 2];
}
__global__ void k_unpack_owned(float* __restrict__ accu, const uint32_t* __restrict__ ownedPix, uint32_t nOwned, const float* __restrict__ src) {
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= nOwned) return;
  uint32_t pix = ownedPix[j];
  accu[3 * (size_t)pix] = src[3 * (size_t)j];
  accu[3 * (size_t)pix + 1] = src[3 * (size_t)j + 1];
  accu[3 * (size_t)pix + 2] = src[3 * (size_t)j + 2];
}

// Tile gather without staging: every owned pixel goes straight to its place in the full-size destination, which
// may be peer memory (another GPU's gather buffer, mapped with P2P or CUDA IPC).  One thread per float; the owned
// list is in tile order, so a warp writes runs of 96 contiguous floats.
__global__ void k_push_owned(const float* __restrict__ accu, const uint32_t* __restrict__ ownedPix, uint32_t nOwned, float* __restrict__ dstFull) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)nOwned * 3) return;
  uint32_t j = (uint32_t)(i / 3), k = (uint32_t)(i - (size_t)j * 3);
  size_t at = 3 * (size_t)ownedPix[j] + k;
  dstFull[at] = accu[at];
}

inline unsigned grid(size_t n) { return (unsigned)((n + TPB - 1) / TPB); }

}  // namespace

void launchGenerate(const LaunchCtx& c, uint32_t nSamples) {
  uint32_t n = nSamples * c.nOwned;
  if (!n) return;
  if (c.rp.rngMode == 0) k_generate<0><<<grid(n), TPB, 0, c.stream>>>(c, n);
  else k_generate<1><<<grid(n), TPB, 0, c.stream>>>(c, n);
}
// Launch geometry of the persistent kernels.  Called from several host threads (one per device of a multi-GPU
// handle): the cached values are written once each, atomically; every device of a box is the same GPU model.
template <class K>
static unsigned persistentGridFor(K kernel, uint32_t count, std::atomic<int>& blocksPerSm) {
  static std::atomic<int> numSms{0};
  int sms = numSms.load(std::memory_order_relaxed);
  if (!sms) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); numSms.store(sms, std::memory_order_relaxed); }
  int bps = blocksPerSm.load(std::memory_order_relaxed);
  if (!bps) {
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kernel, TRAV_TPB, 0);
    if (bps < 1) bps = 1;
    blocksPerSm.store(bps, std::memory_order_relaxed);
  }
  unsigned full = (unsigned)(sms * bps);
  unsigned need = (count + TRAV_TPB - 1) / TRAV_TPB;
  return need < full ? need : full;
}

// Busy lanes below which a warp refills.  Closest hit: 24 (20: 70.2, 24: 69.1, 28: 71.0 ms of extend per step).
// Shadow rays on the wide BVH claim their ray ids in chunks, which makes a refill cheap (one memory level): 24 there
// too (16: 93.9, 20: 89.8, 24: 86.7, 26: 86.9, 28: 88.2, 32: 100.6 ms of shadow per step); the binary kernel, which
// pays an atomic and a queue load per refill, stays at 20.
#ifndef MOX_FETCH_THRESHOLD_CLOSEST
#define MOX_FETCH_THRESHOLD_CLOSEST 24
#endif
#ifndef MOX_FETCH_THRESHOLD_SHADOW_WIDE
#define MOX_FETCH_THRESHOLD_SHADOW_WIDE 24
#endif
static int fetchThreshold(bool anyHit, bool wide) {
  struct T { int t[3]; };
  static const T v = [] {   // thread-safe one-time initialisation
    T r;
    const char* e = getenv("MOX_FETCH_THRESHOLD");
    const char* es = getenv("MOX_FETCH_THRESHOLD_SHADOW");   // shadow rays only (A/B runs)
    r.t[0] = e ? atoi(e) : MOX_FETCH_THRESHOLD_CLOSEST;
    r.t[1] = es ? atoi(es) : e ? atoi(e) : MOX_FETCH_THRESHOLD;
    r.t[2] = es ? atoi(es) : e ? atoi(e) : MOX_FETCH_THRESHOLD_SHADOW_WIDE;
    for (int k = 0; k < 3; ++k) r.t[k] = r.t[k] < 1 ? 1 : r.t[k] > 32 ? 32 : r.t[k];
    return r;
  }();
  return v.t[anyHit ? (wide ? 2 : 1) : 0];
}

template <bool ANYHIT, bool COUNT, bool CLASSIFY>
static void launchTraverseT(const SceneView& s, const TraceJob& job, cudaStream_t stream) {
  static std::atomic<int> bpsBinary{0}, bpsWide{0}, bpsBinaryWt{0}, bpsWideWt{0};
  if (s.watertight) {
    if (s.nodes8) k_traverse_wide_wt<ANYHIT, COUNT, CLASSIFY><<<persistentGridFor(k_traverse_wide_wt<ANYHIT, COUNT, CLASSIFY>, job.count, bpsWideWt), TRAV_TPB, 0, stream>>>(s, job);
    else k_traverse_wt<ANYHIT, COUNT, CLASSIFY><<<persistentGridFor(k_traverse_wt<ANYHIT, COUNT, CLASSIFY>, job.count, bpsBinaryWt), TRAV_TPB, 0, stream>>>(s, job);
  } else if (s.nodes8) k_traverse_wide<ANYHIT, COUNT, CLASSIFY><<<persistentGridFor(k_traverse_wide<ANYHIT, COUNT, CLASSIFY>, job.count, bpsWide), TRAV_TPB, 0, stream>>>(s, job);
  else k_traverse<ANYHIT, COUNT, CLASSIFY><<<persistentGridFor(k_traverse<ANYHIT, COUNT, CLASSIFY>, job.count, bpsBinary), TRAV_TPB, 0, stream>>>(s, job);
}

// What every persistent traversal launch needs besides its rays: the refill threshold, the origin divisor and a zeroed
// fetch cursor.
static TraceJob preparedJob(TraceJob job, bool anyHit, bool wide, cudaStream_t stream) {
  job.fetchThreshold = fetchThreshold(anyHit, wide);
  job.originMagic = job.originMod ? (uint32_t)(0x100000000ull / job.originMod) + 1u : 0u;
  cudaMemsetAsync(job.cursor, 0, 4, stream);
  return job;
}

void launchTraverse(const SceneView& s, const TraceJob& jobIn, bool anyHit, bool count, cudaStream_t stream, bool classify) {
  if (!jobIn.count) return;
  const TraceJob job = preparedJob(jobIn, anyHit, s.nodes8 != nullptr, stream);
  if (anyHit && count) launchTraverseT<true, true, false>(s, job, stream);
  else if (anyHit) launchTraverseT<true, false, false>(s, job, stream);
  else if (classify && count) launchTraverseT<false, true, true>(s, job, stream);
  else if (classify) launchTraverseT<false, false, true>(s, job, stream);
  else if (count) launchTraverseT<false, true, false>(s, job, stream);
  else launchTraverseT<false, false, false>(s, job, stream);
}

// The closest-hit rays of a bounce: path rays in, render-form hit records out.
static TraceJob extendJob(const LaunchCtx& c, const uint32_t* queue, uint32_t count, const uint32_t* countPtr) {
  TraceJob job;
  job.rayO = c.pb.rayO; job.rayD = c.pb.rayD; job.queue = queue; job.count = count; job.countPtr = countPtr;
  job.cursor = c.pb.counters + C_CURSOR; job.hits2 = c.pb.hit; job.counters = c.pb.counters;
  return job;
}

void launchExtend(const LaunchCtx& c, const uint32_t* queue, uint32_t count, const uint32_t* countPtr, uint32_t depth) {
  if (count) launchTraverse(c.scene, extendJob(c, queue, count, countPtr), false, c.countTraversal, c.stream, true);
}
void launchTerminal(const LaunchCtx& c, const uint32_t* queue, uint32_t count, const uint32_t* countPtr, const TerminalLights& tl) {
  if (!count) return;
  const TraceJob job = preparedJob(extendJob(c, queue, count, countPtr), false, true, c.stream);
  static std::atomic<int> bps{0}, bpsCount{0}, bpsWt{0}, bpsWtCount{0};
  const SceneView& s = c.scene;
  if (s.watertight) {
    if (c.countTraversal) k_traverse_wide_wt_terminal<true><<<persistentGridFor(k_traverse_wide_wt_terminal<true>, count, bpsWtCount), TRAV_TPB, 0, c.stream>>>(s, job, tl);
    else k_traverse_wide_wt_terminal<false><<<persistentGridFor(k_traverse_wide_wt_terminal<false>, count, bpsWt), TRAV_TPB, 0, c.stream>>>(s, job, tl);
  } else if (c.countTraversal) k_traverse_wide_terminal<true><<<persistentGridFor(k_traverse_wide_terminal<true>, count, bpsCount), TRAV_TPB, 0, c.stream>>>(s, job, tl);
  else k_traverse_wide_terminal<false><<<persistentGridFor(k_traverse_wide_terminal<false>, count, bps), TRAV_TPB, 0, c.stream>>>(s, job, tl);
}
void launchClassify(const LaunchCtx& c, const uint32_t* queue, uint32_t count, const uint32_t* countPtr, uint32_t depth) {
  if (count) k_classify<<<grid(count), TPB, 0, c.stream>>>(c, queue, count, countPtr, depth);
}
void launchShade(const LaunchCtx& c, int kind, uint32_t count, uint32_t depth) {
  if (!count) return;
  const bool ref = c.rp.rngMode == 0;
  switch (kind) {
    case Q_LAMBERT:
      if (ref) k_shade_diffuse<false, 0><<<grid(count), TPB, 0, c.stream>>>(c, count, depth);
      else k_shade_diffuse<false, 1><<<grid(count), TPB, 0, c.stream>>>(c, count, depth);
      break;
    case Q_METAL:
      if (ref) k_shade_diffuse<true, 0><<<grid(count), TPB, 0, c.stream>>>(c, count, depth);
      else k_shade_diffuse<true, 1><<<grid(count), TPB, 0, c.stream>>>(c, count, depth);
      break;
    case Q_DIELECTRIC:
      if (ref) k_shade_dielectric<0><<<grid(count), TPB, 0, c.stream>>>(c, count, depth);
      else k_shade_dielectric<1><<<grid(count), TPB, 0, c.stream>>>(c, count, depth);
      break;
    case Q_DISNEY: {
      const unsigned g = (count + DISNEY_TPB - 1) / DISNEY_TPB;
      if (ref) {
        if (c.brdfFast) k_shade_disney<0, true><<<g, DISNEY_TPB, 0, c.stream>>>(c, count, depth);
        else k_shade_disney<0, false><<<g, DISNEY_TPB, 0, c.stream>>>(c, count, depth);
      } else {
        if (c.brdfFast) k_shade_disney<1, true><<<g, DISNEY_TPB, 0, c.stream>>>(c, count, depth);
        else k_shade_disney<1, false><<<g, DISNEY_TPB, 0, c.stream>>>(c, count, depth);
      }
      break;
    }
  }
}
void launchShadow(const LaunchCtx& c, uint32_t disneyCount, cudaStream_t stream) {
  if (!disneyCount || c.scene.nLights == 0) return;
  size_t slots = (size_t)disneyCount * c.scene.nLights;
  TraceJob job;
  // dense queue of the slots that need a ray; its length lives in device memory (no host sync)
  job.rayO = c.pb.shO; job.rayD = c.pb.shD; job.queue = c.pb.shQueue; job.count = (uint32_t)slots;
  job.countPtr = c.bc + C_SHQ; job.originMod = disneyCount;
  job.cursor = c.pb.counters + C_CURSOR_SHADOW; job.shC = c.pb.shC; job.counters = c.pb.counters;
  launchTraverse(c.scene, job, true, c.countTraversal, stream);
}
void launchApply(const LaunchCtx& c, uint32_t disneyCount, cudaStream_t stream) {
  if (disneyCount && c.scene.nLights) k_apply<<<grid(disneyCount), TPB, 0, stream>>>(c, disneyCount);
}
void launchAccumulate(const LaunchCtx& c, uint32_t nSamples) {
  if (c.nOwned) k_accumulate<false><<<grid(c.nOwned), TPB, 0, c.stream>>>(c, nSamples, PixelStats());
}
void launchAccumulateAdaptive(const LaunchCtx& c, uint32_t nSamples, const PixelStats& ps) {
  if (c.nOwned) k_accumulate<true><<<grid(c.nOwned), TPB, 0, c.stream>>>(c, nSamples, ps);
}
void launchAov(const LaunchCtx& c, uint32_t nSamples, const AovBuffers& aov) {
  if (c.nOwned) k_aov<<<grid(c.nOwned), TPB, 0, c.stream>>>(c, nSamples, aov);
}
size_t adaptiveSelectTiles(uint32_t count) { return ((size_t)count + SEL_TILE - 1) / SEL_TILE; }
void launchAdaptiveSelect(const PixelStats& ps, const AdaptiveRule& rule, const uint32_t* listIn, uint32_t count, uint32_t remaining,
                          uint32_t* listOut, uint32_t* tileSums, uint32_t* survivors, cudaStream_t stream) {
  if (!count) return;
  const unsigned tiles = (unsigned)adaptiveSelectTiles(count);
  k_adaptive_select<<<tiles, TPB, 0, stream>>>(ps, rule, listIn, count, remaining, tileSums);
  k_adaptive_compact<<<tiles, TPB, 0, stream>>>(ps, rule, listIn, count, tileSums, listOut, survivors);
}
void launchSplitRays(const float4* rays, float4* o, float4* d, size_t n, cudaStream_t stream) {
  if (n) k_split_rays<<<grid(n), TPB, 0, stream>>>(rays, o, d, n);
}
void launchBuildShadeRecords(const TriIdx* tris, const float* verts, const float* normals, const float* uvs, uint32_t n, float4* out,
                             cudaStream_t stream) {
  if (n) k_build_shade_records<<<(n + 255) / 256, 256, 0, stream>>>(tris, verts, normals, uvs, n, out);
}
void launchFillOnes(float4* p, size_t n, cudaStream_t stream) {
  if (n) k_fill_ones<<<grid(n), TPB, 0, stream>>>(p, n);
}
void launchCopyRgb(const float4* src, float* dst, size_t n, cudaStream_t stream) {
  if (n) k_copy_rgb<<<grid(n), TPB, 0, stream>>>(src, dst, n);
}
void launchPackOwned(const float* accu, const uint32_t* ownedPix, uint32_t nOwned, float* dst, cudaStream_t stream) {
  if (nOwned) k_pack_owned<<<grid(nOwned), TPB, 0, stream>>>(accu, ownedPix, nOwned, dst);
}
void launchPushOwned(const float* accu, const uint32_t* ownedPix, uint32_t nOwned, float* dstFull, cudaStream_t stream) {
  if (nOwned) k_push_owned<<<grid((size_t)nOwned * 3), TPB, 0, stream>>>(accu, ownedPix, nOwned, dstFull);
}
void launchUnpackOwned(float* accu, const uint32_t* ownedPix, uint32_t nOwned, const float* src, cudaStream_t stream) {
  if (nOwned) k_unpack_owned<<<grid(nOwned), TPB, 0, stream>>>(accu, ownedPix, nOwned, src);
}
