// traverse_wide.cuh — persistent-thread traversal of the compressed 8-wide BVH (BvhNode8,
// gpu_types.h).  Same contract as traverseWarpPersistent (traverse.cuh): identical primitive tests,
// (t, id) lexicographic closest hit, order-independent shadow transmittance; only the hierarchy
// walked differs, so results are bit-identical to the binary traversal.
//
// Per lane: a node group G = (childBase, hit bits 31..24 | primitive bits that exist 23..8 | imask 7..0) and a
// primitive group T = (primBase, 16 hit bits), plus a stack of postponed node groups (Ylitie et al. 2017).  One node
// step pops the front-most child of G (highest bit of slot ^ octant order), pushes the rest of G, fetches the 80-byte
// node and tests its 8 quantised child boxes: one FMA per plane on a grid local to the node, near/far planes picked
// per ray sign for four children at a time, one more FMA + IMAD per child for its hit bits (fixed positions per slot,
// gpu_types.h).  Warp phase voting as in the binary kernel — a node step or a primitive step (up to two primitives of
// the lane) per iteration — but weighted by cost (MOX_VOTE_TRI_WEIGHT): the cheaper primitive phase runs as soon as a
// third as many lanes want it.
#pragma once
#include "traverse.cuh"

#define MOX_WIDE_STACK MOX_TRAVERSAL_STACK

// Quantised plane byte -> float, two ways, mixed per plane so that neither pipe is the bottleneck:
//  * I2F.U8 on the conversion pipe (15.4 results/clk/SM measured, scripts/microbench/pipe_rates.cu, against 124
//    FFMA): with all 48 conversions of a node step on it that pipe was ~70 % busy and 15-19 % of the stall samples
//    were mio_throttle;
//  * one PRMT on the ALU pipe: m = 1 + b * 2^-15 — byte b dropped into mantissa bits 8..15 of 1.0f — with the
//    affine map folded back into the plane FMA:   b * ia + on  ==  m * (2^15 ia) + (on - 2^15 ia).
//    The subtraction of 2^15 ia from the addend is rounded towards the outside of the box, so boxes only ever grow.
// MOX_BYTE_MIX: bit 0..2 = near plane x, y, z, bit 3..5 = far plane x, y, z; a set bit converts that plane's eight
// bytes with PRMT (0x33 measured best, DESIGN.md section 4).
// A child's hit bits come from the sign of one FMA: tf * 1.00001 - tn < 0 is a miss, and the sign bit times the
// child's constant is subtracted from an all-hit mask by one IMAD (FFMA + SHF + IMAD; only the shift is on the ALU
// pipe, which also runs the 32 FMNMX, the PRMTs and the near/far selects of a node step).
#ifndef MOX_BYTE_MIX
#define MOX_BYTE_MIX 0x33
#endif
// `one` is 1.0f's bit pattern held in a register (see the node step of traverseWidePersistent): with the constant as an immediate
// ptxas needs the byte selector in a register and re-materialises four selectors per node.
template <bool PRMT>
MOX_D float byteToFloat(uint32_t w, int i, uint32_t one) {
  if (!PRMT) return (float)((w >> (8 * i)) & 0xffu);
  uint32_t r;
  if (i == 0) asm("prmt.b32 %0, %1, %2, 0x7604;" : "=r"(r) : "r"(w), "r"(one));
  else if (i == 1) asm("prmt.b32 %0, %1, %2, 0x7614;" : "=r"(r) : "r"(w), "r"(one));
  else if (i == 2) asm("prmt.b32 %0, %1, %2, 0x7624;" : "=r"(r) : "r"(w), "r"(one));
  else asm("prmt.b32 %0, %1, %2, 0x7634;" : "=r"(r) : "r"(w), "r"(one));
  return __uint_as_float(r);
}
// Scale and addends of one axis for the plane FMAs  t = float(byte) * scale + addend  (near: rounded down, far:
// rounded up): every axis gets its own rounding bound, 2^-21 of the local origin term, folded into the addends so a
// plane costs one conversion and one FMA.
template <bool NEAR_PRMT, bool FAR_PRMT>
MOX_D void planeTerms(float ia, float oa, float& sn, float& an, float& sf, float& af) {
  const float k = ia * 32768.f;
  // (I2F form: |oa| * 2^-21 is exact, so one FMA rounds the same sum once)
  const float an0 = fmaf(-4.76837158203125e-07f, fabsf(oa), oa), af0 = fmaf(4.76837158203125e-07f, fabsf(oa), oa);
  // PRMT form: the only new rounding is the subtraction of 2^15 ia from the addend — rounded towards the outside of the
  // box (FADD.RM / FADD.RP) it needs no bound of its own
  if (NEAR_PRMT) { sn = k; an = __fsub_rd(an0, k); } else { sn = ia; an = an0; }
  if (FAR_PRMT) { sf = k; af = __fsub_ru(af0, k); } else { sf = ia; af = af0; }
}
// index of the highest set bit (x != 0): FLO directly (written as 31 - __clz(x), ptxas keeps both subtractions)
MOX_D uint32_t highestBit(uint32_t x) {
  uint32_t r;
  asm("bfind.u32 %0, %1;" : "=r"(r) : "r"(x));
  return r;
}

// (a & m) | (b & ~m) as one LOP3 (written as two ANDs and an OR, ptxas spends two)
MOX_D uint32_t bitSelect(uint32_t a, uint32_t b, uint32_t m) {
  uint32_t r;
  asm("lop3.b32 %0, %1, %2, %3, 0xE4;" : "=r"(r) : "r"(a), "r"(b), "r"(m));
  return r;
}

// CLASSIFY (closest hit of the render path): the hit record is (t, primitive id | shade class << 28) — the class
// comes from the winning primitive's packed record — and beta / gamma are not carried (two registers less per
// lane); the shade kernels recompute them from the same operands.  The raw query keeps the four-word record.
// WT: the packed triangle records hold the raw vertices and the watertight test runs (MOX_ACCEL_WATERTIGHT).
// TERMINAL (with CLASSIFY): the bounce past rayMaxDepth.  k_classify ends every such path and k_accumulate adds one
// term chosen by the record's .y alone: miss -> bgColor, a light -> its emission, anything else -> absorbColor.  So
// the refill finds the (t, id) minimum over the light list tl with the primitive step's tests and acceptance rule;
// then an any-hit traversal bounded by that light (tBest = tL, tie id idL) ends at the first accepted hit, which
// lies ahead of every light, so the closest hit is no light either.  Every primitive blocks.  The record is
//   (t of the written primitive, id | class << 28) of that blocker, else of the light, else (tmax, MOX_HIT_MISS);
// with no light hit and bgColor == absorbColor the ray ends at the refill with the miss record.  Nothing reads .x
// of a terminal record.
template <bool ANYHIT, bool COUNT, bool CLASSIFY = false, bool WT = false, bool TERMINAL = false>
__device__ __forceinline__ void traverseWidePersistent(const SceneView& s, const TraceJob& job, const TerminalLights& tl = TerminalLights()) {
  static_assert(!TERMINAL || (CLASSIFY && !ANYHIT), "the terminal query writes the render path's hit record");
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const unsigned ltMask = (1u << lane) - 1u;
  const uint32_t jobCount = job.countPtr ? __ldg(job.countPtr) : job.count;
  // Per-lane state.  A lane is busy exactly while it has a primitive group or a node group pending (a ray with
  // neither pops its stack or finishes in the same iteration), so there is no separate "active" flag.  CLASSIFY keeps
  // the winner's shade class in bits 28..30 of bPrim (the form the hit record has anyway).  A shadow ray's
  // transmittance lives in the last two entries of the lane's stack array (local memory, no L1 footprint until
  // touched): it is needed only when a ray meets tinting glass.  (Shared memory for it cost L1: the carve-out is
  // permanent; 2.5 KB per CTA lowered the shadow kernel's L1 hit rate by a point.)
  uint2 stack[MOX_WIDE_STACK];
  int sp = 0;
  uint32_t gBase = 0, gBits = 0;  // node group
  uint32_t tBase = 0, tBits = 0;  // primitive group
  bool exhausted = false;
  uint32_t rayId = 0, octinv = 0;
  float3 o = mk3(0.f), d = mk3(0.f), idir = mk3(0.f);
  float tmin = 0.f, tBest = 0.f, bBeta = 0.f, bGamma = 0.f;
  int bPrim = -1;
  bool tinted = false;               // ANYHIT: the top of the stack array holds a product of glass colours for this ray
  uint32_t shadowEnd = 0;            // ANYHIT && COUNT: 1 blocked, 2 tinted
  uint32_t nv = 0, np = 0;
#define MOX_LANE_BUSY() (tBits != 0u || (gBits & 0xff000000u) != 0u)
  WtRay wr;
  wr.kx = wr.ky = wr.kz = 0; wr.Sx = wr.Sy = wr.Sz = 0.f;

  // Shadow rays (CHUNKED): ray ids are claimed from the global cursor 32 at a time and kept one per lane (poolId); a
  // refill hands them out by shuffle.  The claim — one atomic, then one coalesced queue load whose result nobody
  // touches yet — is issued when a pool runs dry, so what a refill waits for is one memory level (the ray itself)
  // instead of three (cursor, queue entry, ray); the whole warp sits in that wait, busy lanes included.  Measured:
  // shadow 90.6 -> 90.0 ms per step; the closest-hit kernel lost with it (69.3 -> 70.1 ms) and keeps one atomic
  // per refill.  The terminal query claims in chunks too: most of its rays end at the refill, and a warp that keeps a
  // few lanes in an any-hit traversal refills its idle ones a few at a time, one atomic on the cursor each.  (Not its
  // counting form: that one would spill at 56 registers, and the counts do not depend on how rays are claimed.)
  constexpr bool CHUNKED = ANYHIT || (TERMINAL && !COUNT);
  uint32_t poolId = 0, poolPos = 0, poolCount = 0;   // poolPos / poolCount are warp-uniform
  bool moreChunks = true;
  while (true) {
    // ---------------- refill idle lanes
    if (!exhausted) {
      const bool idleLane = !MOX_LANE_BUSY();
      unsigned idle = __ballot_sync(FULL, idleLane);
      if (idle) {
        bool take;
        uint32_t base = 0;
        if (CHUNKED) {
          if (poolPos >= poolCount && moreChunks) {   // first visit, or the last refill emptied the pool
            if (lane == 0) base = atomicAdd(job.cursor, 32u);
            base = __shfl_sync(FULL, base, 0);
            poolCount = base < jobCount ? min(32u, jobCount - base) : 0u;
            poolPos = 0;
            if ((uint32_t)lane < poolCount) poolId = job.queue ? MOX_LD_STREAM(job.queue + base + lane) : base + lane;
            if (base + 32u >= jobCount) moreChunks = false;
          }
          const uint32_t slot = poolPos + (uint32_t)__popc(idle & ltMask);
          const uint32_t got = __shfl_sync(FULL, poolId, slot & 31u);
          take = idleLane && slot < poolCount;
          poolPos = min(poolPos + (uint32_t)__popc(idle), poolCount);
          if (take) rayId = got;
        } else {
          const int leader = __ffs(idle) - 1;
          if (lane == leader) base = atomicAdd(job.cursor, (uint32_t)__popc(idle));
          base = __shfl_sync(FULL, base, leader);
          const uint32_t i = base + __popc(idle & ltMask);
          take = idleLane && i < jobCount;
          if (take) rayId = job.queue ? MOX_LD_STREAM(job.queue + i) : i;
        }
        if (take) {
          const uint32_t oId = originIndex(job, rayId);
          float4 ro = MOX_LD_STREAM(job.rayO + oId), rd = MOX_LD_STREAM(job.rayD + rayId);
          if (!(ANYHIT && rd.w < 0.f)) {
            RayPre r = prepRay<true>(mk3(ro), mk3(rd), ro.w);
            o = r.o; d = r.d; idir = r.idir; tmin = r.tmin;
            if (WT) wr = wtPrep(d);
            octinv = 7u ^ ((idir.x < 0.f ? 4u : 0u) | (idir.y < 0.f ? 2u : 0u) | (idir.z < 0.f ? 1u : 0u));   // (a zero component counts as positive, prepRay)
            tBest = rd.w; bPrim = -1;
            if (!CLASSIFY) { bBeta = 0.f; bGamma = 0.f; }
            tinted = false;
            sp = 0;
            gBase = 0; gBits = 0x80000000u;  // root: one pending child, imask 0 -> node index 0
            tBase = 0; tBits = 0;
            if (COUNT) { nv = 0; np = 0; shadowEnd = 0; }
            if (TERMINAL) {
              // closest light: same tests, same operands (the packed sphere record is analytic[].a) and same rule as
              // the primitive step, so the minimum is the one the closest-hit traversal would find among the lights
              for (int k = 0; k < tl.n; ++k) {
                const uint4 e = __ldg(tl.list + k);
                const bool tie = bPrim >= 0 && (e.x & MOX_HIT_ID_MASK) < ((uint32_t)bPrim & MOX_HIT_ID_MASK);
                const Analytic* an = s.analytic + e.z;
                float t = 0.f, a1, a2;
                bool hit = false;
                if (e.y == PT_SPHERE) hit = sphereTest(__ldg(&an->a), o, d, tmin, tBest, tie, t);
                else if (e.y == PT_QUAD) {
                  Analytic q;
                  q.a = __ldg(&an->a); q.b = __ldg(&an->b); q.c = __ldg(&an->c); q.d = __ldg(&an->d);
                  hit = quadTest(q, o, d, tmin, t, a1, a2) && (t < tBest || (t == tBest && tie));
                }
                if (hit) { tBest = t; bPrim = (int)e.x; }
              }
              if (bPrim < 0 && tl.missIsAbsorb) {   // miss and non-light end alike: nothing to traverse
                MOX_ST_STREAM(job.hits2 + rayId, make_float2(tBest, __int_as_float(MOX_HIT_MISS)));
                gBits = 0u;
              }
            }
          }
        }
        if (CHUNKED) {
          if (poolPos >= poolCount) {
            if (moreChunks) {
              // claim the next 32 now: the queue load is in flight while the warp goes back to traversing
              uint32_t nb = 0;
              if (lane == 0) nb = atomicAdd(job.cursor, 32u);
              nb = __shfl_sync(FULL, nb, 0);
              poolCount = nb < jobCount ? min(32u, jobCount - nb) : 0u;
              poolPos = 0;
              if ((uint32_t)lane < poolCount) poolId = job.queue ? MOX_LD_STREAM(job.queue + nb + lane) : nb + lane;
              if (nb + 32u >= jobCount) moreChunks = false;
            }
            if (poolPos >= poolCount && !moreChunks) exhausted = true;
          }
        } else if (base + __popc(idle) >= jobCount) exhausted = true;
      }
    }
    if (!__any_sync(FULL, MOX_LANE_BUSY())) {
      if (exhausted) break;
      continue;
    }
    // ---------------- traverse until too few lanes are busy
    while (true) {
      const bool isTri = tBits != 0u;
      const bool isNode = !isTri && (gBits & 0xff000000u) != 0u;
#ifndef MOX_VOTE_TRI_WEIGHT
#define MOX_VOTE_TRI_WEIGHT 3  // a primitive step costs less than half a node step: vote by cost, not by head count (round 1: 1: 1115, 2: 1191, 3: 1206, 4: 1214, 6: 1207, 32: 1069 Mrays/s; with the cheaper node step of round 2 and two primitives per step: 2: 1693-1696, 3: 1691-1692, 4: 1671)
#endif
      // one ballot + one warp reduction (REDUX) of the weighted vote instead of two ballots + two POPCs — POPC shares the
      // slow conversion pipe with the 48 I2F of a node step (ncu: 15-19 % of the stall samples are mio_throttle)
      const unsigned bm = __ballot_sync(FULL, isNode | isTri);
      const int score = __reduce_add_sync(FULL, isNode ? 1 : (isTri ? -MOX_VOTE_TRI_WEIGHT : 0));
      if (bm == 0u || (!exhausted && __popc(bm) < job.fetchThreshold)) break;
      if (score >= 0) {
        if (isNode) {
          // ---- pop the front-most pending child of G
          const uint32_t bit = highestBit(gBits & 0xff000000u);
          const uint32_t imaskG = gBits & 0xffu;
          gBits &= ~(1u << bit);
          const uint32_t slot = (bit - 24u) ^ octinv;
          const uint32_t nodeIdx = gBase + __popc(imaskG & ((1u << slot) - 1u));
          if (gBits & 0xff000000u) stack[sp++] = make_uint2(gBase, gBits);
          // ---- fetch and test the node
          const BvhNode8* nd = s.nodes8 + nodeIdx;
          const float4 n0 = __ldg(&nd->n0), n1 = __ldg(&nd->n1), n2 = __ldg(&nd->n2), n3 = __ldg(&nd->n3), n4 = __ldg(&nd->n4);
          if (COUNT) nv++;
          const uint32_t ew = __float_as_uint(n0.w);
          const float iax = __uint_as_float((ew & 0xffu) << 23) * idir.x;
          const float iay = __uint_as_float(((ew >> 8) & 0xffu) << 23) * idir.y;
          const float iaz = __uint_as_float(((ew >> 16) & 0xffu) << 23) * idir.z;
          const float oax = (n0.x - o.x) * idir.x, oay = (n0.y - o.y) * idir.y, oaz = (n0.z - o.z) * idir.z;
          // 1.0f's bit pattern for byteToFloat from one FMA per node step (0 * finite + 1; neither nvcc nor ptxas may
          // fold it) instead of a constant load and an ALU instruction to rebuild the value ptxas does not keep in a
          // register across the loop
          const uint32_t one = __float_as_uint(fmaf(0.f, idir.x, 1.0f));
          // conservative plane terms (planeTerms above); the far side is additionally widened by 1e-5 relative
          constexpr unsigned MIX = MOX_BYTE_MIX;
          float snx, onx, sfx, ofx, sny, ony, sfy, ofy, snz, onz, sfz, ofz;
          planeTerms<(MIX & 1u) != 0, (MIX & 8u) != 0>(iax, oax, snx, onx, sfx, ofx);
          planeTerms<(MIX & 2u) != 0, (MIX & 16u) != 0>(iay, oay, sny, ony, sfy, ofy);
          planeTerms<(MIX & 4u) != 0, (MIX & 32u) != 0>(iaz, oaz, snz, onz, sfz, ofz);
          uint32_t hitmask = 0xff00ffffu;
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            const uint32_t qlx = __float_as_uint(half ? n2.y : n2.x), qly = __float_as_uint(half ? n2.w : n2.z);
            const uint32_t qlz = __float_as_uint(half ? n3.y : n3.x), qhx = __float_as_uint(half ? n3.w : n3.z);
            const uint32_t qhy = __float_as_uint(half ? n4.y : n4.x), qhz = __float_as_uint(half ? n4.w : n4.z);
            const uint32_t nx = idir.x < 0.f ? qhx : qlx, fx = idir.x < 0.f ? qlx : qhx;
            const uint32_t ny = idir.y < 0.f ? qhy : qly, fy = idir.y < 0.f ? qly : qhy;
            const uint32_t nz = idir.z < 0.f ? qhz : qlz, fz = idir.z < 0.f ? qlz : qhz;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float tnx = fmaf(byteToFloat<(MIX & 1u) != 0>(nx, i, one), snx, onx), tfx = fmaf(byteToFloat<(MIX & 8u) != 0>(fx, i, one), sfx, ofx);
              const float tny = fmaf(byteToFloat<(MIX & 2u) != 0>(ny, i, one), sny, ony), tfy = fmaf(byteToFloat<(MIX & 16u) != 0>(fy, i, one), sfy, ofy);
              const float tnz = fmaf(byteToFloat<(MIX & 4u) != 0>(nz, i, one), snz, onz), tfz = fmaf(byteToFloat<(MIX & 32u) != 0>(fz, i, one), sfz, ofz);
              const float tn = fmaxf(fmaxf(tnx, tny), fmaxf(tnz, tmin));
              // hit <=> tf * 1.00001 - tn >= 0, read off the sign bit of one FMA (the FMA pipe has room, the ALU pipe
              // that runs FSETP / SEL does not): every miss clears the child's constant from an all-hit mask
              const float dd = fmaf(fminf(fminf(tfx, tfy), fminf(tfz, tBest)), 1.00001f, -tn);
              const uint32_t K = (1u << (24 + 4 * half + i)) | (3u << (2 * (4 * half + i)));
              asm("mad.lo.u32 %0, %1, %2, %0;" : "+r"(hitmask) : "r"(__float_as_uint(dd) >> 31), "r"(0u - K));
            }
          }
          gBase = __float_as_uint(n1.x);
          tBase = __float_as_uint(n1.y);
          // keep what exists (inner children: imask, primitives: V), then bring the inner byte into front-to-back
          // order: bit 24 + s moves to 24 + (s ^ octinv) — three conditional swaps (nibbles, pairs, neighbours) written
          // as shifts by 0 or 4 / 2 / 1, so there is no branch and no select: (x << 0 & m) | (x >> 0 & ~m) = x
          hitmask &= __float_as_uint(n1.z);
          tBits = hitmask & 0x0000ffffu;
          {
            uint32_t x = hitmask;
            // the octant mask is made of the signs of 1/d (see the refill), the predicates the near/far selects of this
            // node step hold anyway: three predicated instructions per swap
            if (!(idir.x < 0.f)) x = bitSelect(x << 4, x >> 4, 0xf0000000u);
            if (!(idir.y < 0.f)) x = bitSelect(x << 2, x >> 2, 0xcc000000u);
            if (!(idir.z < 0.f)) x = bitSelect(x << 1, x >> 1, 0xaa000000u);
            gBits = (x & 0xff000000u) | __float_as_uint(n1.w);   // n1.w = V << 8 | imask
          }
        }
      } else {
#ifndef MOX_PRIMS_PER_STEP
#define MOX_PRIMS_PER_STEP 2
#endif
        // ---- up to MOX_PRIMS_PER_STEP primitives of the current group.  Leaf children hold up to two primitives and a
        // ray often hits the boxes of several, so a lane that is in the primitive phase usually has more than one bit
        // pending: testing two per step halves the vote / loop overhead per primitive.
        // Measured (Mrays/s): 1 per step 1 656, 2 per step 1 691 (vote weight 3) / 1 696 (weight 2).
        auto recordOf = [&](uint32_t k) -> const float4* {
          // offset from the node's first primitive = rank of bit k among the primitive bits that exist (V sits in
          // bits 8..23 of the node-group word for as long as primitives of that node are pending)
          return s.packed8 + (size_t)(tBase + __popc((gBits >> 8) & ~(0xffffffffu << k))) * MOX_PACKED_F4;
        };
        // one primitive test
        auto testPrimitive = [&](const float4 r0, const float4 r1, const float4 r2) {
          if (COUNT) np++;
          const uint32_t idbits = __float_as_uint(r0.w);
          const uint32_t type = (idbits >> 30) | __float_as_uint(r2.w) | (__float_as_uint(r1.w) >> 8);
          const int id = (int)(idbits & 0x3fffffffu);
          float t = 0.f, be = 0.f, ga = 0.f;
          bool hit;
          // (t, id) rule: an equal t wins only against a hit with a higher id (CLASSIFY: the id is the low 28 bits)
#define MOX_TIE_WINS() (!ANYHIT && (CLASSIFY ? (bPrim >= 0 && id < (int)((uint32_t)bPrim & MOX_HIT_ID_MASK)) : id < bPrim))
          if (type == PT_TRI) {
            hit = (WT ? triTestWt(wr, o, tmin, mk3(r0), mk3(r1), mk3(r2), t, be, ga) : triTest(o, d, tmin, mk3(r0), mk3(r1), mk3(r2), t, be, ga)) &&
                  (t < tBest || (t == tBest && MOX_TIE_WINS()));
          } else if (type == PT_SPHERE) {
            hit = sphereTest(make_float4(r1.x, r1.y, r1.z, r2.x), o, d, tmin, tBest, MOX_TIE_WINS(), t);
          } else {
            const Analytic* an = s.analytic + __float_as_int(r0.x);
            Analytic q;
            q.a = __ldg(&an->a); q.b = __ldg(&an->b); q.c = __ldg(&an->c); q.d = __ldg(&an->d);
            hit = quadTest(q, o, d, tmin, t, be, ga) && (t < tBest || (t == tBest && MOX_TIE_WINS()));
          }
#undef MOX_TIE_WINS
          if (hit) {
            if (ANYHIT) {
              // shadow class from the record itself (k_pack): only tinting glass still needs its material
              const uint32_t cls = __float_as_uint(r1.w) & 3u;
              if (cls == MOX_SHADOW_BLOCKS) {
                // blocked: zero the contribution without reading it, drop all pending work (the lane is idle from here)
                MOX_ST_STREAM(job.shC + rayId, make_float4(0.f, 0.f, 0.f, 0.f));
                tinted = false;
                tBits = 0u; gBits = 0u; sp = 0;
                if (COUNT) shadowEnd = 1u;
              } else if (cls == MOX_SHADOW_TINTS) {
                const GpuMaterial* m = s.mats + (__ldg(&s.prims[id].typeMat) >> 2);
                const float3 col = mk3(__ldg(&m->dis.color.x), __ldg(&m->dis.color.y), __ldg(&m->dis.color.z));
                float3 a = col;   // = (1, 1, 1) * col
                if (tinted) {
                  const uint2 p0 = stack[MOX_WIDE_STACK - 2], p1 = stack[MOX_WIDE_STACK - 1];
                  a = mk3(__uint_as_float(p0.x) * col.x, __uint_as_float(p0.y) * col.y, __uint_as_float(p1.x) * col.z);
                }
                stack[MOX_WIDE_STACK - 2] = make_uint2(__float_as_uint(a.x), __float_as_uint(a.y));
                stack[MOX_WIDE_STACK - 1] = make_uint2(__float_as_uint(a.z), 0u);
                tinted = true;
              }
            } else {
              tBest = t;
              if (CLASSIFY) bPrim = (int)((uint32_t)id | ((__float_as_uint(r1.w) >> MOX_CLASS_SHIFT) << MOX_HIT_ID_BITS));
              else { bPrim = id; bBeta = be; bGamma = ga; }
              if (TERMINAL) { tBits = 0u; gBits = 0u; sp = 0; }   // the first hit ahead of the closest light decides
            }
          }
        };
#pragma unroll
        for (int rep = 0; rep < MOX_PRIMS_PER_STEP; ++rep)
        if (rep == 0 ? isTri : tBits != 0u) {
          const uint32_t k = highestBit(tBits);
          const float4* rec = recordOf(k);
          tBits &= ~(1u << k);
          // All three words are fetched before the type is known: the tag is folded from words 0 and 2 and the
          // (zero) high bits of word 1, so the loads stay together ahead of the branch — waiting for word 0
          // first would put a second memory latency into every triangle test.
          const float4 r0 = __ldg(rec), r1 = __ldg(rec + 1), r2 = __ldg(rec + 2);
          testPrimitive(r0, r1, r2);
        }
      }
      // ---- out of work in the current groups: resume a postponed node group, or finish the ray.  Only a lane that
      // was busy when this iteration started can have run dry in it.
      if ((isTri || isNode) && !MOX_LANE_BUSY()) {
        if (sp > 0) {
          const uint2 g = stack[--sp];
          gBase = g.x; gBits = g.y;
        } else {
          if (ANYHIT) {
            // unoccluded: the contribution stays as the shade kernel wrote it; blocked: already zeroed at the hit;
            // only a ray tinted by glass needs the read-modify-write (the load stalls the whole warp)
            if (tinted) {
              const uint2 p0 = stack[MOX_WIDE_STACK - 2], p1 = stack[MOX_WIDE_STACK - 1];
              float4 c = MOX_LD_STREAM(job.shC + rayId);
              MOX_ST_STREAM(job.shC + rayId, make_float4(c.x * __uint_as_float(p0.x), c.y * __uint_as_float(p0.y), c.z * __uint_as_float(p1.x), c.w));
              tinted = false;
              if (COUNT) shadowEnd = 2u;
            }
          } else if (CLASSIFY) {
            MOX_ST_STREAM(job.hits2 + rayId, make_float2(tBest, __int_as_float(bPrim)));   // -1 = MOX_HIT_MISS
          } else {
            MOX_ST_STREAM(job.hits + rayId, make_float4(tBest, __int_as_float(bPrim), bBeta, bGamma));
          }
          if (COUNT) {
            atomicAdd((unsigned long long*)(job.counters + (ANYHIT ? C_NODEVIS_SH_LO : C_NODEVIS_LO)), (unsigned long long)nv);
            atomicAdd((unsigned long long*)(job.counters + (ANYHIT ? C_PRIMTEST_SH_LO : C_PRIMTEST_LO)), (unsigned long long)np);
            if (ANYHIT && shadowEnd) atomicAdd(job.counters + (shadowEnd == 1u ? C_SH_BLOCKED : C_SH_TINTED), 1u);
          }
        }
      }
    }
  }
#undef MOX_LANE_BUSY
}
