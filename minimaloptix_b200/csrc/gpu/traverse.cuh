// traverse.cuh — software ray traversal (what OptiX's rtTrace did inside the closed runtime;
// call sites Camera.cu:37, Material.cu:41,64,108,165,192,213) and the leaf primitive tests
// (Geometry.cu:18-55 sphere, :70-91 quad, :121-134 mesh via the SDK's intersect_triangle).
//
// Closest hit obeys the (t, primitive id) lexicographic rule; primitive tests use the exact
// operation sequence of the oracle (no FMA), so on identical rays the winning id, t, beta and
// gamma are bit-identical.  Box slabs are conservative ((lo - o) * 1/d, far side widened by
// 1e-5 relative) and may use any rounding.
#pragma once
#include "gpu_types.h"
#include "traverse_job.h"
#include "vec.cuh"

struct Hit { float t; int prim; float beta, gamma; };

// SDK intersect_triangle (branch-free variant) on a packed record.
MOX_D bool triTest(const float3& o, const float3& d, float tmin, const float3& p0, const float3& e0, const float3& e1,
                   float& t, float& beta, float& gamma) {
  const float3 n = cross(e1, e0);
  const float3 e2 = (1.0f / dot(n, d)) * (p0 - o);
  const float3 i = cross(d, e2);
  beta = dot(i, e1);
  gamma = dot(i, e0);
  t = dot(n, e2);
  return (t > tmin) & (beta >= 0.0f) & (gamma >= 0.0f) & (beta + gamma <= 1);
}

// ---- watertight ray-triangle test (Woop, Benthin, Wald 2013), opt-in with MOX_ACCEL_WATERTIGHT.
// The SDK test above works on edges rounded from the vertices and divides by a rounded n.d: a ray aimed at an edge
// or a vertex shared by two triangles can miss both.  This one shears and scales the three vertices — the raw
// coordinates, identical bits for every triangle sharing them — into ray space, where each scaled edge function
// U, V, W is evaluated from the same two sheared vertices whichever triangle asks, so two triangles sharing an
// edge can never both reject a ray crossing it; exact zeros are re-evaluated in double (products of floats are exact
// there, so the sign is).  No backface culling, like the SDK test.  beta / gamma weigh p1 / p2 as above.
// oracle/oracle.cpp::watertightTriangle is the same operation sequence (no FMA on either side).
struct WtRay { int kx, ky, kz; float Sx, Sy, Sz; };
MOX_D float pick3(const float3& v, int k) { return k == 0 ? v.x : (k == 1 ? v.y : v.z); }
MOX_D WtRay wtPrep(const float3& d) {
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
MOX_D bool triTestWt(const WtRay& w, const float3& o, float tmin, const float3& p0, const float3& p1, const float3& p2,
                     float& t, float& beta, float& gamma) {
  const float3 A = p0 - o, B = p1 - o, C = p2 - o;
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
  return t > tmin;
}

// First root in (tmin, bound) — near root, else far root (Geometry.cu:18-55).  `incl`: also accept t == bound.
MOX_D bool sphereTest(const float4& cr, const float3& o, const float3& d, float tmin, float bound, bool incl, float& t) {
  float3 oc = o - mk3(cr);
  float b = dot(d, oc);
  float c = dot(oc, oc) - cr.w * cr.w;
  float disc = b * b - c;
  if (disc < 0) return false;
  float root = sqrtf(disc);
  t = -b - root;
  if (t > tmin && (t < bound || (incl && t == bound))) return true;
  t = -b + root;
  return t > tmin && (t < bound || (incl && t == bound));
}

MOX_D bool quadTest(const Analytic& q, const float3& o, const float3& d, float tmin, float& t, float& a1, float& a2) {
  float3 n = mk3(q.a);
  float dt = dot(d, n);
  t = (q.a.w - dot(n, o)) / dt;
  if (!(t > tmin)) return false;
  float3 p = o + d * t;
  float3 vi = p - mk3(q.d);
  a1 = dot(mk3(q.b), vi);
  if (!(a1 >= 0 && a1 <= 1)) return false;
  a2 = dot(mk3(q.c), vi);
  return a2 >= 0 && a2 <= 1;
}

#ifndef MOX_VOTE_LEAF_WEIGHT
#define MOX_VOTE_LEAF_WEIGHT 2  // weight of the primitive phase in the vote (binary BVH of the bench scene: 1 -> 1035, 2 -> 1057, 3 -> 1056 Mrays/s; the wide kernel uses 4)
#endif

struct RayPre { float3 o, d, idir; float tmin; };

// 1/d feeds the box slabs only, which are conservative by more than its error (far side x 1.00001, near/far
// addends moved by 2^-21 of the origin term): the hardware reciprocal (1 ulp) instead of the IEEE sequence and its
// slow-path branch, three times per ray.  Primitive tests never see it.
MOX_D float slabRcp(float x) {
  float r;
  asm("rcp.approx.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
// A component of magnitude at most 1e-30 counts as zero: the ray then stays in that axis' slab for every t when
// lo <= o <= hi and never otherwise (oracle.cpp::slab).  What 1/d becomes for it depends on the slab test that reads it.
//  * boxEntry (binary BVH, WIDE = false): +-inf.  A plane term is then +-inf, or NaN (0 * inf) for an origin on the
//    plane, which boxEntry drops from its near or its far side: the axis culls exactly by the rule above.
//  * the wide node step (WIDE = true): +1e30 whatever the sign of the zero, so that the axis keeps culling with finite
//    terms and its far planes are the high ones.  A far term is 0 only for a plane through the origin, and the node
//    step's 2^-21 slack of the origin term (planeTerms) lifts every far plane above the node's own origin plane to a
//    huge t; what is left is a child flat at the node's origin plane with the ray running in that plane.  Every
//    primitive of such a child lies in the ray's plane, and no primitive test accepts a ray lying in its plane (the
//    product of the ray with the plane normal is exactly 0).  With the sign kept (-1e30 for -0) the far planes of
//    such a ray would be the low ones, and every child starting at the node's origin plane would be culled.
// (A clamp of +-1e30 with the sign kept culled both kinds of hit: (hi - o) * 1e30 = 0 put the far plane at t = 0.)
template <bool WIDE>
MOX_D RayPre prepRay(const float3& o, const float3& d, float tmin) {
  RayPre r;
  r.o = o; r.d = d; r.tmin = tmin;
  const float tiny = 1e-30f;
  const float rx = slabRcp(d.x), ry = slabRcp(d.y), rz = slabRcp(d.z);   // (unconditionally: selects, no branches)
  if (WIDE) {
    r.idir.x = fabsf(d.x) > tiny ? rx : 1e30f;
    r.idir.y = fabsf(d.y) > tiny ? ry : 1e30f;
    r.idir.z = fabsf(d.z) > tiny ? rz : 1e30f;
  } else {
    const float inf = __int_as_float(0x7f800000);
    r.idir.x = fabsf(d.x) > tiny ? rx : copysignf(inf, d.x);
    r.idir.y = fabsf(d.y) > tiny ? ry : copysignf(inf, d.y);
    r.idir.z = fabsf(d.z) > tiny ? rz : copysignf(inf, d.z);
  }
  return r;
}

// Shadow rays of one hit share their origin: ray id = light * hits + hit, origin = rayO[id % hits].  The quotient is
// at most the number of lights, so one multiply-high by floor(2^32 / hits) + 1 gives it or one more.
MOX_D uint32_t originIndex(const TraceJob& job, uint32_t id) {
  if (job.originMod <= 1u) return job.originMod ? 0u : id;   // (the magic of 1 does not fit 32 bits)
  const uint32_t q = __umulhi(id, job.originMagic);
  const uint32_t r = id - q * job.originMod;
  return (int32_t)r < 0 ? r + job.originMod : r;
}

// Entry distance of the slab test, or +inf when the box is missed within [tmin, tcur].  Near and far planes are
// picked by the sign of 1/d, so that a NaN term (zero component, origin on the plane) is dropped from the near side
// or from the far side as it belongs; fminf / fmaxf of the two terms of an axis would turn (-inf, NaN) into an
// empty slab.
MOX_D float boxEntry(const RayPre& r, float lox, float hix, float loy, float hiy, float loz, float hiz, float tcur) {
  const bool nx = r.idir.x < 0.f, ny = r.idir.y < 0.f, nz = r.idir.z < 0.f;
  float x0 = ((nx ? hix : lox) - r.o.x) * r.idir.x, x1 = ((nx ? lox : hix) - r.o.x) * r.idir.x;
  float y0 = ((ny ? hiy : loy) - r.o.y) * r.idir.y, y1 = ((ny ? loy : hiy) - r.o.y) * r.idir.y;
  float z0 = ((nz ? hiz : loz) - r.o.z) * r.idir.z, z1 = ((nz ? loz : hiz) - r.o.z) * r.idir.z;
  float tn = fmaxf(fmaxf(x0, y0), fmaxf(z0, r.tmin));
  float tf = fminf(fminf(x1, y1), fminf(z1, tcur)) * 1.00001f;
  return tn <= tf ? tn : __int_as_float(0x7f800000);
}

#define MOX_STACK MOX_TRAVERSAL_STACK
// Ray / hit records are touched once per launch: stream them (evict-first) so they do not push
// the BVH and the triangles out of L2.
#define MOX_LD_STREAM(p) __ldcs(p)
#define MOX_ST_STREAM(p, v) __stcs((p), (v))
#define MOX_DONE ((int)0x80000000)   // sentinel "no more nodes" (same bit pattern as an empty child)
#define MOX_FETCH_THRESHOLD 20       // refill a warp's idle lanes when fewer than this many are traversing

// Persistent-thread traversal over the binary BVH with warp-level phase voting.
//   * warps fetch rays from a global cursor: 32 at start, then whenever fewer than
//     job.fetchThreshold lanes are still busy the idle lanes are refilled (Aila & Laine 2009);
//   * every iteration the warp votes: if the lanes at an inner node outnumber MOX_VOTE_LEAF_WEIGHT x the
//     lanes inside a leaf it runs ONE inner-node step (two child slabs, near child first), otherwise ONE
//     primitive test for the lanes inside a leaf.  The branch is warp-uniform — a plain while-while loop
//     measured 10 of 32 threads per instruction;
//   * closest hit obeys the (t, id) lexicographic rule; any hit: Disney prims only, NORMAL
//     blocks, GLASS tints (SURVEY.md §8 a-11, Material.cu:225-232);
//   * per-lane traversal stack in local memory (far children only).
template <bool ANYHIT, bool COUNT, bool CLASSIFY = false, bool WT = false>
__device__ __forceinline__ void traverseWarpPersistent(const SceneView& s, const TraceJob& job) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const unsigned ltMask = (1u << lane) - 1u;
  const float INF = __int_as_float(0x7f800000);
  const uint32_t jobCount = job.countPtr ? __ldg(job.countPtr) : job.count;
  int stack[MOX_STACK];
  int sp = 0, cur = MOX_DONE;
  uint32_t lk = 0, lend = 0;  // primitive cursor inside the current leaf
  bool active = false, exhausted = false;
  uint32_t rayId = 0;
  RayPre r;
  r.o = r.d = r.idir = mk3(0.f); r.tmin = 0.f;
  float tBest = 0.f, bBeta = 0.f, bGamma = 0.f;
  int bPrim = -1;
  uint32_t bCls = 0;
  float3 atten = mk3(1.f);
  uint32_t nv = 0, np = 0;
  WtRay wr;
  wr.kx = wr.ky = wr.kz = 0; wr.Sx = wr.Sy = wr.Sz = 0.f;

#define MOX_SET_CUR(c)                                             \
  do {                                                             \
    cur = (c);                                                     \
    if (cur < 0 && cur != MOX_DONE) {                              \
      uint32_t leaf_ = (uint32_t)~cur;                             \
      lk = leaf_ >> 3; lend = lk + (leaf_ & 7u) + 1u;              \
    }                                                              \
  } while (0)

  while (true) {
    // ---------------- refill idle lanes
    if (!exhausted) {
      unsigned idle = __ballot_sync(FULL, !active);
      if (idle) {
        const int leader = __ffs(idle) - 1;
        uint32_t base = 0;
        if (lane == leader) base = atomicAdd(job.cursor, (uint32_t)__popc(idle));
        base = __shfl_sync(FULL, base, leader);
        if (!active) {
          uint32_t i = base + __popc(idle & ltMask);
          if (i < jobCount) {
            rayId = job.queue ? MOX_LD_STREAM(job.queue + i) : i;
            const uint32_t oId = originIndex(job, rayId);
            float4 ro = MOX_LD_STREAM(job.rayO + oId), rd = MOX_LD_STREAM(job.rayD + rayId);
            if (!(ANYHIT && rd.w < 0.f)) {
              r = prepRay<false>(mk3(ro), mk3(rd), ro.w);
              if (WT) wr = wtPrep(r.d);
              tBest = rd.w; bPrim = -1; bBeta = 0.f; bGamma = 0.f;
              atten = mk3(1.f);
              sp = 0; cur = 0;  // root
              active = true;
              if (COUNT) { nv = 0; np = 0; }
            }
          }
        }
        if (base + __popc(idle) >= jobCount) exhausted = true;
      }
    }
    if (!__any_sync(FULL, active)) {
      if (exhausted) break;
      continue;
    }
    // ---------------- traverse until too few lanes are busy
    while (true) {
      const bool isInner = cur >= 0;
      const bool isLeaf = !isInner && cur != MOX_DONE;
      const unsigned im = __ballot_sync(FULL, isInner), lm = __ballot_sync(FULL, isLeaf);
      const unsigned busy = im | lm;
      if (busy == 0u || (!exhausted && __popc(busy) < job.fetchThreshold)) break;
      if (__popc(im) >= MOX_VOTE_LEAF_WEIGHT * __popc(lm)) {
        if (isInner) {  // one inner-node step
          const BvhNode2* nd = s.nodes + cur;
          float4 a = __ldg(&nd->c0xy), b = __ldg(&nd->c1xy), z = __ldg(&nd->cz);
          int4 ref = __ldg(&nd->ref);
          if (COUNT) nv++;
          float t0 = boxEntry(r, a.x, a.y, a.z, a.w, z.x, z.y, tBest);
          float t1 = boxEntry(r, b.x, b.y, b.z, b.w, z.z, z.w, tBest);
          bool h0 = t0 < INF, h1 = t1 < INF;
          int next;
          if (h0 && h1) {
            bool swp = t1 < t0;
            stack[sp++] = swp ? ref.x : ref.y;
            next = swp ? ref.y : ref.x;
          } else if (h0 || h1) {
            next = h0 ? ref.x : ref.y;
          } else {
            next = sp ? stack[--sp] : MOX_DONE;
          }
          MOX_SET_CUR(next);
        }
      } else {
        if (isLeaf) {  // one primitive test
          const float4* rec = s.packed + (size_t)lk * MOX_PACKED_F4;
          float4 r0 = __ldg(rec);
          if (COUNT) np++;
          uint32_t idbits = __float_as_uint(r0.w);
          uint32_t type = idbits >> 30;
          int id = (int)(idbits & 0x3fffffffu);
          float t = 0.f, be = 0.f, ga = 0.f;
          bool hit;
          if (type == PT_TRI) {
            float4 r1 = __ldg(rec + 1), r2 = __ldg(rec + 2);
            hit = (WT ? triTestWt(wr, r.o, r.tmin, mk3(r0), mk3(r1), mk3(r2), t, be, ga) : triTest(r.o, r.d, r.tmin, mk3(r0), mk3(r1), mk3(r2), t, be, ga)) &&
                  (t < tBest || (!ANYHIT && t == tBest && id < bPrim));
          } else {
            const Analytic* an = s.analytic + __float_as_int(r0.x);
            if (type == PT_SPHERE) {
              hit = sphereTest(__ldg(&an->a), r.o, r.d, r.tmin, tBest, !ANYHIT && id < bPrim, t);
            } else {
              Analytic q;
              q.a = __ldg(&an->a); q.b = __ldg(&an->b); q.c = __ldg(&an->c); q.d = __ldg(&an->d);
              hit = quadTest(q, r.o, r.d, r.tmin, t, be, ga) && (t < tBest || (!ANYHIT && t == tBest && id < bPrim));
            }
          }
          bool blocked = false;
          if (hit) {
            if (ANYHIT) {
              // geometry first, material only on a hit: non-Disney prims do not occlude shadow rays
              const GpuMaterial* m = s.mats + (__ldg(&s.prims[id].typeMat) >> 2);
              if (__ldg(&m->kind) == MOX_MAT_DISNEY) {
                if (__ldg((const int*)&m->dis.brdfType) == GLASS) atten *= mk3(__ldg(&m->dis.color.x), __ldg(&m->dis.color.y), __ldg(&m->dis.color.z));
                else { blocked = true; atten = mk3(0.f); }
              }
            } else {
              tBest = t; bPrim = id; bBeta = be; bGamma = ga;
              if (CLASSIFY) bCls = __float_as_uint(__ldg(&rec[1].w)) >> MOX_CLASS_SHIFT;   // shade class of the winner (k_pack)
            }
          }
          ++lk;
          if (blocked) cur = MOX_DONE;
          else if (lk == lend) { int next = sp ? stack[--sp] : MOX_DONE; MOX_SET_CUR(next); }
        }
      }
      if (active && cur == MOX_DONE) {  // ray finished
        if (ANYHIT) {
          // same three cases as the wide kernel, so both report bit-identical results even when the
          // precomputed contribution is not finite: blocked -> 0 (the reference skips the term,
          // Material.cu:192), unoccluded -> untouched, tinted -> multiply
          if (atten.x == 0.f && atten.y == 0.f && atten.z == 0.f) {
            job.shC[rayId] = make_float4(0.f, 0.f, 0.f, 0.f);
          } else if (atten.x != 1.f || atten.y != 1.f || atten.z != 1.f) {
            float4 c = job.shC[rayId];
            job.shC[rayId] = make_float4(c.x * atten.x, c.y * atten.y, c.z * atten.z, c.w);
          }
        } else if (CLASSIFY) {
          MOX_ST_STREAM(job.hits2 + rayId, make_float2(tBest, __int_as_float(bPrim < 0 ? MOX_HIT_MISS : (int)((uint32_t)bPrim | (bCls << MOX_HIT_ID_BITS)))));
        } else {
          MOX_ST_STREAM(job.hits + rayId, make_float4(tBest, __int_as_float(bPrim), bBeta, bGamma));
        }
        if (COUNT) {
          atomicAdd((unsigned long long*)(job.counters + (ANYHIT ? C_NODEVIS_SH_LO : C_NODEVIS_LO)), (unsigned long long)nv);
          atomicAdd((unsigned long long*)(job.counters + (ANYHIT ? C_PRIMTEST_SH_LO : C_PRIMTEST_LO)), (unsigned long long)np);
          if (ANYHIT) {   // rays that touched their contribution record
            if (atten.x == 0.f && atten.y == 0.f && atten.z == 0.f) atomicAdd(job.counters + C_SH_BLOCKED, 1u);
            else if (atten.x != 1.f || atten.y != 1.f || atten.z != 1.f) atomicAdd(job.counters + C_SH_TINTED, 1u);
          }
        }
        active = false;
      }
    }
  }
#undef MOX_SET_CUR
}
