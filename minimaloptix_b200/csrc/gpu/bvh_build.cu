// bvh_build.cu — GPU LBVH build.  This is the work OptiX's closed "Trbvh" builder did for the
// reference (MinimalOptiX.cpp:378,494,534); nothing here has a counterpart in the reference
// source.  Pipeline (all on the context's stream):
//   k_prim_bounds   primitive AABBs as the reference's bbox programs define them
//                   (Geometry.cu:57-63 sphere — with the corrected orientation, :93-110 quad,
//                   :162-175 mesh; zero-area / infinite primitives are excluded) + centroid bounds
//   k_morton        30-bit Morton code of the centroid (10 bits / axis); invalid prims sort last
//   onesweep        LSD radix sort, 8-bit digits, 4 passes, one upfront histogram, decoupled
//                   look-back between tiles (Adinets & Merrill 2022)
//   k_karras        binary radix tree over the sorted codes (Karras 2012), index tie-break
//   k_refit         bottom-up AABB refit with per-node arrival counters
//   k_emit2         Aila–Laine 64-byte nodes, subtrees of <= MOX_LEAF_MAX prims folded into leaves
//   k_pack          leaf-ordered 48-byte primitive records
#include "build.h"
#include "traverse_job.h"
#include "vec.cuh"

namespace {

constexpr float kInf = __builtin_huge_valf();

// ------------------------------------------------------------------ bounds
__device__ __forceinline__ uint32_t orderedBits(float f) {
  uint32_t u = __float_as_uint(f);
  return u ^ ((u >> 31) ? 0xffffffffu : 0x80000000u);
}
__host__ __device__ __forceinline__ float fromOrderedBits(uint32_t u) {
  u ^= (u >> 31) ? 0x80000000u : 0xffffffffu;
#ifdef __CUDA_ARCH__
  return __uint_as_float(u);
#else
  float f; memcpy(&f, &u, 4); return f;
#endif
}

// Box of primitive i and whether it takes part in the BVH (zero-area / infinite primitives do not; their box is
// empty).  The build and the refit both store what this returns, so their boxes have the same bits.
__device__ __forceinline__ bool primBounds(int i, const PrimDesc* __restrict__ prims, const TriIdx* __restrict__ tris,
                                           const float* __restrict__ verts, const Analytic* __restrict__ analytic, float3& lo,
                                           float3& hi) {
  bool valid;
  PrimDesc pd = prims[i];
  uint32_t type = pd.typeMat & 3u;
  if (type == PT_TRI) {
    TriIdx t = tris[pd.geom];
    float3 v0 = mk3(verts[3 * t.v[0]], verts[3 * t.v[0] + 1], verts[3 * t.v[0] + 2]);
    float3 v1 = mk3(verts[3 * t.v[1]], verts[3 * t.v[1] + 1], verts[3 * t.v[1] + 2]);
    float3 v2 = mk3(verts[3 * t.v[2]], verts[3 * t.v[2] + 1], verts[3 * t.v[2] + 2]);
    float area = length(cross(v1 - v0, v2 - v0));
    valid = area > 0.0f && !isinf(area);
    lo = fmin3(fmin3(v0, v1), v2);
    hi = fmax3(fmax3(v0, v1), v2);
  } else if (type == PT_SPHERE) {
    float4 cr = analytic[pd.geom].a;
    lo = mk3(cr) + (-cr.w);
    hi = mk3(cr) + cr.w;
    valid = cr.w == cr.w && !isinf(cr.w);
    if (cr.w < 0) { float3 t = lo; lo = hi; hi = t; }
  } else {
    Analytic q = analytic[pd.geom];
    float3 v1 = mk3(q.b), v2 = mk3(q.c), a = mk3(q.d);
    float3 tv1 = v1 / dot(v1, v1);
    float3 tv2 = v2 / dot(v2, v2);
    float3 p01 = a + tv1, p10 = a + tv2, p11 = a + tv1 + tv2;
    float area = length(cross(tv1, tv2));
    valid = area > 0.0f && !isinf(area);
    lo = fmin3(fmin3(a, p01), fmin3(p10, p11));
    hi = fmax3(fmax3(a, p01), fmax3(p10, p11));
  }
  if (!valid) { lo = mk3(kInf); hi = mk3(-kInf); }
  return valid;
}

__global__ void k_prim_bounds(int n, const PrimDesc* __restrict__ prims, const TriIdx* __restrict__ tris,
                              const float* __restrict__ verts, const Analytic* __restrict__ analytic,
                              float4* __restrict__ boxLo, float4* __restrict__ boxHi, uint32_t* __restrict__ cbounds,
                              uint32_t* __restrict__ invalidCount) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  float3 lo = mk3(kInf), hi = mk3(-kInf);
  bool valid = false;
  if (i < n) {
    valid = primBounds(i, prims, tris, verts, analytic, lo, hi);
    boxLo[i] = make_float4(lo.x, lo.y, lo.z, valid ? 1.f : 0.f);
    boxHi[i] = make_float4(hi.x, hi.y, hi.z, 0.f);
  }
  float3 c = valid ? (lo + hi) * 0.5f : mk3(kInf);
  float3 cmin = c, cmax = valid ? c : mk3(-kInf);
  unsigned inval = (i < n && !valid) ? 1u : 0u;
  for (int o = 16; o > 0; o >>= 1) {
    cmin.x = fminf(cmin.x, __shfl_xor_sync(0xffffffffu, cmin.x, o));
    cmin.y = fminf(cmin.y, __shfl_xor_sync(0xffffffffu, cmin.y, o));
    cmin.z = fminf(cmin.z, __shfl_xor_sync(0xffffffffu, cmin.z, o));
    cmax.x = fmaxf(cmax.x, __shfl_xor_sync(0xffffffffu, cmax.x, o));
    cmax.y = fmaxf(cmax.y, __shfl_xor_sync(0xffffffffu, cmax.y, o));
    cmax.z = fmaxf(cmax.z, __shfl_xor_sync(0xffffffffu, cmax.z, o));
    inval += __shfl_xor_sync(0xffffffffu, inval, o);
  }
  if ((threadIdx.x & 31) == 0) {
    if (cmin.x <= cmax.x) {
      atomicMin(&cbounds[0], orderedBits(cmin.x)); atomicMin(&cbounds[1], orderedBits(cmin.y)); atomicMin(&cbounds[2], orderedBits(cmin.z));
      atomicMax(&cbounds[3], orderedBits(cmax.x)); atomicMax(&cbounds[4], orderedBits(cmax.y)); atomicMax(&cbounds[5], orderedBits(cmax.z));
    }
    if (inval) atomicAdd(invalidCount, inval);
  }
}

// Refit: the boxes of the current primitive data over the stored ones.  The topology of the last build holds only
// while every primitive keeps its validity; a change raises *changed.
__global__ void k_refit_bounds(int n, const PrimDesc* __restrict__ prims, const TriIdx* __restrict__ tris,
                               const float* __restrict__ verts, const Analytic* __restrict__ analytic,
                               float4* __restrict__ boxLo, float4* __restrict__ boxHi, uint32_t* __restrict__ changed) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float3 lo, hi;
  const bool valid = primBounds(i, prims, tris, verts, analytic, lo, hi);
  if (valid != (boxLo[i].w != 0.f)) *changed = 1u;
  boxLo[i] = make_float4(lo.x, lo.y, lo.z, valid ? 1.f : 0.f);
  boxHi[i] = make_float4(hi.x, hi.y, hi.z, 0.f);
}

__device__ __forceinline__ uint32_t expandBits10(uint32_t v) {
  v = (v * 0x00010001u) & 0xFF0000FFu;
  v = (v * 0x00000101u) & 0x0F00F00Fu;
  v = (v * 0x00000011u) & 0xC30C30C3u;
  v = (v * 0x00000005u) & 0x49249249u;
  return v;
}

__global__ void k_morton(int n, const float4* __restrict__ boxLo, const float4* __restrict__ boxHi,
                         const uint32_t* __restrict__ cbounds, uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float3 bmin = mk3(fromOrderedBits(cbounds[0]), fromOrderedBits(cbounds[1]), fromOrderedBits(cbounds[2]));
  float3 bmax = mk3(fromOrderedBits(cbounds[3]), fromOrderedBits(cbounds[4]), fromOrderedBits(cbounds[5]));
  float4 lo = boxLo[i], hi = boxHi[i];
  uint32_t key;
  if (lo.w == 0.f) {
    key = 0x40000000u;  // invalid: after every valid 30-bit code
  } else {
    float3 c = (mk3(lo) + mk3(hi)) * 0.5f;
    float3 e = bmax - bmin;
    float sx = e.x > 0 ? 1024.f / e.x : 0.f, sy = e.y > 0 ? 1024.f / e.y : 0.f, sz = e.z > 0 ? 1024.f / e.z : 0.f;
    uint32_t x = (uint32_t)fminf(fmaxf((c.x - bmin.x) * sx, 0.f), 1023.f);
    uint32_t y = (uint32_t)fminf(fmaxf((c.y - bmin.y) * sy, 0.f), 1023.f);
    uint32_t z = (uint32_t)fminf(fmaxf((c.z - bmin.z) * sz, 0.f), 1023.f);
    key = (expandBits10(x) << 2) | (expandBits10(y) << 1) | expandBits10(z);
  }
  keys[i] = key;
  vals[i] = (uint32_t)i;
}

// ------------------------------------------------------------------ onesweep radix sort
constexpr int SORT_THREADS = 256;
constexpr int SORT_WARPS = SORT_THREADS / 32;
constexpr int SORT_ITEMS = 16;
constexpr int SORT_TILE = SORT_THREADS * SORT_ITEMS;
constexpr uint32_t FLAG_AGG = 1u << 30, FLAG_PREFIX = 2u << 30, FLAG_MASK = 3u << 30, VALUE_MASK = ~FLAG_MASK;

__global__ void k_sort_hist(const uint32_t* __restrict__ keys, int n, uint32_t* __restrict__ hist /*[4][256]*/) {
  __shared__ uint32_t sh[4 * 256];
  for (int i = threadIdx.x; i < 1024; i += blockDim.x) sh[i] = 0;
  __syncthreads();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    uint32_t k = keys[i];
    atomicAdd(&sh[k & 255u], 1u);
    atomicAdd(&sh[256 + ((k >> 8) & 255u)], 1u);
    atomicAdd(&sh[512 + ((k >> 16) & 255u)], 1u);
    atomicAdd(&sh[768 + (k >> 24)], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 1024; i += blockDim.x)
    if (sh[i]) atomicAdd(&hist[i], sh[i]);
}

// One block of 256 threads: exclusive scan of each of the 4 digit histograms, in place.
__global__ void k_sort_scan_hist(uint32_t* __restrict__ hist) {
  __shared__ uint32_t sh[256];
  for (int p = 0; p < 4; ++p) {
    uint32_t v = hist[p * 256 + threadIdx.x];
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int o = 1; o < 256; o <<= 1) {
      uint32_t t = threadIdx.x >= o ? sh[threadIdx.x - o] : 0u;
      __syncthreads();
      sh[threadIdx.x] += t;
      __syncthreads();
    }
    hist[p * 256 + threadIdx.x] = sh[threadIdx.x] - v;
    __syncthreads();
  }
}

__global__ void __launch_bounds__(SORT_THREADS)
k_sort_pass(const uint32_t* __restrict__ keysIn, const uint32_t* __restrict__ valsIn, uint32_t* __restrict__ keysOut,
            uint32_t* __restrict__ valsOut, int n, int shift, const uint32_t* __restrict__ digitBase,
            uint32_t* __restrict__ tileCounter, volatile uint32_t* __restrict__ status, uint32_t* __restrict__ errorFlag) {
  __shared__ uint32_t warpHist[SORT_WARPS][256];
  __shared__ uint32_t globalOffset[256];
  __shared__ uint32_t sTile;
  if (threadIdx.x == 0) sTile = atomicAdd(tileCounter, 1u);
  for (int i = threadIdx.x; i < SORT_WARPS * 256; i += SORT_THREADS) (&warpHist[0][0])[i] = 0;
  __syncthreads();
  const uint32_t tile = sTile;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t ltMask = (1u << lane) - 1u;
  const int base = tile * SORT_TILE + warp * (SORT_ITEMS * 32);

  uint32_t key[SORT_ITEMS], val[SORT_ITEMS];
  uint16_t rank[SORT_ITEMS];
#pragma unroll
  for (int r = 0; r < SORT_ITEMS; ++r) {
    int idx = base + r * 32 + lane;
    bool ok = idx < n;
    key[r] = ok ? keysIn[idx] : 0xffffffffu;
    val[r] = ok ? valsIn[idx] : 0u;
    uint32_t digit = ok ? ((key[r] >> shift) & 255u) : 0xffffu;
    uint32_t peers = __match_any_sync(0xffffffffu, digit);
    int leader = __ffs(peers) - 1;
    uint32_t prev = 0;
    if (ok && lane == leader) {
      prev = warpHist[warp][digit];
      warpHist[warp][digit] = prev + __popc(peers);
    }
    prev = __shfl_sync(0xffffffffu, prev, leader);
    rank[r] = (uint16_t)(prev + __popc(peers & ltMask));
    __syncwarp();
  }
  __syncthreads();
  {  // thread d owns digit d: exclusive prefix over warps, publish, look back
    const int d = threadIdx.x;
    uint32_t running = 0;
#pragma unroll
    for (int w = 0; w < SORT_WARPS; ++w) {
      uint32_t t = warpHist[w][d];
      warpHist[w][d] = running;
      running += t;
    }
    volatile uint32_t* myStatus = status + (size_t)tile * 256 + d;
    uint32_t excl = 0;
    if (tile == 0) {
      *myStatus = FLAG_PREFIX | running;
    } else {
      *myStatus = FLAG_AGG | running;
      int t = (int)tile - 1;
      uint32_t spins = 0;
      while (true) {
        uint32_t s = status[(size_t)t * 256 + d];
        uint32_t f = s & FLAG_MASK;
        if (f == 0) {
          if (++spins > (1u << 28)) { atomicExch(errorFlag, 1u); break; }  // never hang the GPU
          continue;
        }
        excl += s & VALUE_MASK;
        if (f == FLAG_PREFIX) break;
        --t;
      }
      *myStatus = FLAG_PREFIX | (excl + running);
    }
    globalOffset[d] = digitBase[d] + excl;
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < SORT_ITEMS; ++r) {
    int idx = base + r * 32 + lane;
    if (idx < n) {
      uint32_t digit = (key[r] >> shift) & 255u;
      uint32_t pos = globalOffset[digit] + warpHist[warp][digit] + rank[r];
      keysOut[pos] = key[r];
      valsOut[pos] = val[r];
    }
  }
}

// ------------------------------------------------------------------ Karras 2012 hierarchy
__device__ __forceinline__ int deltaKey(const uint32_t* __restrict__ keys, int n, int i, int j) {
  if (j < 0 || j >= n) return -1;
  uint32_t ki = keys[i], kj = keys[j];
  if (ki == kj) return 32 + __clz((uint32_t)i ^ (uint32_t)j);
  return __clz(ki ^ kj);
}

// Internal node i covers sorted leaves [first, last]; child refs: >= 0 internal, < 0 leaf ~idx.
__global__ void k_karras(int n, const uint32_t* __restrict__ keys, int2* __restrict__ children, int2* __restrict__ range,
                         int* __restrict__ parentInternal, int* __restrict__ parentLeaf) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n - 1) return;
  int d = (deltaKey(keys, n, i, i + 1) - deltaKey(keys, n, i, i - 1)) >= 0 ? 1 : -1;
  int dmin = deltaKey(keys, n, i, i - d);
  int lmax = 2;
  while (deltaKey(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
  int l = 0;
  for (int t = lmax >> 1; t >= 1; t >>= 1)
    if (deltaKey(keys, n, i, i + (l + t) * d) > dmin) l += t;
  int j = i + l * d;
  int dnode = deltaKey(keys, n, i, j);
  int s = 0;
  int t = l;
  do {
    t = (t + 1) >> 1;
    if (deltaKey(keys, n, i, i + (s + t) * d) > dnode) s += t;
  } while (t > 1);
  int gamma = i + s * d + min(d, 0);
  int first = min(i, j), last = max(i, j);
  int left = (first == gamma) ? ~gamma : gamma;
  int right = (last == gamma + 1) ? ~(gamma + 1) : gamma + 1;
  children[i] = make_int2(left, right);
  range[i] = make_int2(first, last);
  if (left >= 0) parentInternal[left] = i; else parentLeaf[~left] = i;
  if (right >= 0) parentInternal[right] = i; else parentLeaf[~right] = i;
  if (i == 0) parentInternal[0] = -1;
}

__global__ void k_refit(int n, const uint32_t* __restrict__ sortedIds, const float4* __restrict__ boxLo,
                        const float4* __restrict__ boxHi, const int2* __restrict__ children,
                        const int* __restrict__ parentInternal, const int* __restrict__ parentLeaf,
                        float4* __restrict__ nodeLo, float4* __restrict__ nodeHi, uint32_t* __restrict__ arrivals) {
  int leaf = blockIdx.x * blockDim.x + threadIdx.x;
  if (leaf >= n) return;
  int cur = parentLeaf[leaf];
  while (cur >= 0) {
    if (atomicAdd(&arrivals[cur], 1u) == 0u) return;  // the sibling subtree is not finished yet
    int2 ch = children[cur];
    float4 lo0, hi0, lo1, hi1;
    if (ch.x < 0) { uint32_t id = sortedIds[~ch.x]; lo0 = boxLo[id]; hi0 = boxHi[id]; }
    else { lo0 = __ldcg(&nodeLo[ch.x]); hi0 = __ldcg(&nodeHi[ch.x]); }
    if (ch.y < 0) { uint32_t id = sortedIds[~ch.y]; lo1 = boxLo[id]; hi1 = boxHi[id]; }
    else { lo1 = __ldcg(&nodeLo[ch.y]); hi1 = __ldcg(&nodeHi[ch.y]); }
    __stcg(&nodeLo[cur], make_float4(fminf(lo0.x, lo1.x), fminf(lo0.y, lo1.y), fminf(lo0.z, lo1.z), 0.f));
    __stcg(&nodeHi[cur], make_float4(fmaxf(hi0.x, hi1.x), fmaxf(hi0.y, hi1.y), fmaxf(hi0.z, hi1.z), 0.f));
    __threadfence();
    cur = parentInternal[cur];
  }
}

__global__ void k_emit2(int n, const uint32_t* __restrict__ sortedIds, const float4* __restrict__ boxLo,
                        const float4* __restrict__ boxHi, const int2* __restrict__ children, const int2* __restrict__ range,
                        const float4* __restrict__ nodeLo, const float4* __restrict__ nodeHi, BvhNode2* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n - 1) return;
  int2 ch = children[i];
  float4 lo[2], hi[2];
  int ref[2];
  int c[2] = {ch.x, ch.y};
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    if (c[k] < 0) {
      uint32_t id = sortedIds[~c[k]];
      lo[k] = boxLo[id]; hi[k] = boxHi[id];
      ref[k] = ~(((~c[k]) << 3) | 0);
    } else {
      lo[k] = nodeLo[c[k]]; hi[k] = nodeHi[c[k]];
      int2 r = range[c[k]];
      int cnt = r.y - r.x + 1;
      ref[k] = cnt <= MOX_LEAF_MAX ? ~((r.x << 3) | (cnt - 1)) : c[k];
    }
  }
  BvhNode2 nd;
  nd.c0xy = make_float4(lo[0].x, hi[0].x, lo[0].y, hi[0].y);
  nd.c1xy = make_float4(lo[1].x, hi[1].x, lo[1].y, hi[1].y);
  nd.cz = make_float4(lo[0].z, hi[0].z, lo[1].z, hi[1].z);
  nd.ref = make_int4(ref[0], ref[1], 0, 0);
  out[i] = nd;
}

__global__ void k_pack(int n, const uint32_t* __restrict__ sortedIds, const PrimDesc* __restrict__ prims,
                       const TriIdx* __restrict__ tris, const float* __restrict__ verts, const Analytic* __restrict__ analytic,
                       const GpuMaterial* __restrict__ mats, float4* __restrict__ packed, bool rawVerts) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t id = sortedIds[i];
  PrimDesc pd = prims[id];
  uint32_t type = pd.typeMat & 3u;
  uint32_t idbits = id | (type << 30);
  uint32_t shadowClass = MOX_SHADOW_INVISIBLE;
  if (mats) {
    const GpuMaterial* m = mats + (pd.typeMat >> 2);
    uint32_t cls = MOX_CLASS_LAMBERT;
    if (m->kind == MOX_MAT_DISNEY) {
      shadowClass = m->dis.brdfType == GLASS ? MOX_SHADOW_TINTS : MOX_SHADOW_BLOCKS;
      cls = m->dis.brdfType == GLASS ? MOX_CLASS_DIELECTRIC : MOX_CLASS_DISNEY;
    } else if (m->kind == MOX_MAT_METAL) cls = MOX_CLASS_METAL;
    else if (m->kind == MOX_MAT_GLASS) cls = MOX_CLASS_DIELECTRIC;
    else if (m->kind == MOX_MAT_LIGHT) cls = MOX_CLASS_LIGHT;
    shadowClass |= cls << MOX_CLASS_SHIFT;   // stays below 256: the traversal folds (word >> 8) into the type tag
  }
  // word 1 .w = shadow class | shade class << 2, word 2 .w = the type tag again: the traversal derives the type from all three
  // words, which keeps their loads together ahead of the type branch
  const float sc = __uint_as_float(shadowClass), ty = __uint_as_float(type);
  float4* rec = packed + (size_t)i * MOX_PACKED_F4;
  if (type == PT_TRI) {
    TriIdx t = tris[pd.geom];
    float3 p0 = mk3(verts[3 * t.v[0]], verts[3 * t.v[0] + 1], verts[3 * t.v[0] + 2]);
    float3 p1 = mk3(verts[3 * t.v[1]], verts[3 * t.v[1] + 1], verts[3 * t.v[1] + 2]);
    float3 p2 = mk3(verts[3 * t.v[2]], verts[3 * t.v[2] + 1], verts[3 * t.v[2] + 2]);
    // watertight traversal: the vertices as they are (a shared vertex must have the same bits in every triangle)
    float3 e0 = rawVerts ? p1 : p1 - p0, e1 = rawVerts ? p2 : p0 - p2;
    rec[0] = make_float4(p0.x, p0.y, p0.z, __uint_as_float(idbits));
    rec[1] = make_float4(e0.x, e0.y, e0.z, sc);
    rec[2] = make_float4(e1.x, e1.y, e1.z, ty);
  } else if (type == PT_SPHERE) {  // centre and radius inline: a sphere test needs no second fetch
    const float4 cr = analytic[pd.geom].a;
    rec[0] = make_float4(__int_as_float((int)pd.geom), 0.f, 0.f, __uint_as_float(idbits));
    rec[1] = make_float4(cr.x, cr.y, cr.z, sc);
    rec[2] = make_float4(cr.w, 0.f, 0.f, ty);
  } else {
    rec[0] = make_float4(__int_as_float((int)pd.geom), 0.f, 0.f, __uint_as_float(idbits));
    rec[1] = make_float4(0.f, 0.f, 0.f, sc);
    rec[2] = make_float4(0.f, 0.f, 0.f, ty);
  }
}

// Light list of the terminal query: a primitive k_prim_bounds left out of the BVH (validity in boxLo .w) must not be
// found by the list either.
__global__ void k_terminal_lights(int n, const float4* __restrict__ boxLo, uint4* __restrict__ list) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && boxLo[list[i].x & MOX_HIT_ID_MASK].w == 0.f) list[i].y = MOX_TERMINAL_EXCLUDED;
}

inline int divUp(size_t a, size_t b) { return (int)((a + b - 1) / b); }

// Grid of the grid-stride histogram kernel: eight 256-thread blocks per SM of the current device.
inline int histGridCap() {
  static const int cap = [] {   // thread-safe one-time initialisation (a multi-GPU handle builds from several host threads)
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return (sms > 0 ? sms : 148) * 8;
  }();
  return cap;
}

}  // namespace

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { err = std::string(#x) + ": " + cudaGetErrorString(e_); return false; } } while (0)

bool buildBvh(const BuildInput& in, BuildOutput& out, cudaStream_t stream, std::string& err) {
  const int n = in.nPrims;
  {  // keep the caller's reusable buffers, reset everything else
    BuildOutput fresh;
    fresh.nodes = out.nodes; fresh.packed = out.packed; fresh.nodesCap = out.nodesCap; fresh.packedCap = out.packedCap;
    fresh.nodes8 = out.nodes8; fresh.packed8 = out.packed8; fresh.nodes8Cap = out.nodes8Cap; fresh.packed8Cap = out.packed8Cap;
    out = fresh;
  }
  DeviceArena& arena = *in.arena;
  if (!arena.pinned && cudaMallocHost(&arena.pinned, 64) != cudaSuccess) { err = "cudaMallocHost failed"; return false; }
  // persistent outputs: reuse the previous build's buffers when they are large enough
  auto ensureOut = [&](size_t nodesNeeded, size_t packedNeeded) -> bool {
    if (out.nodesCap < nodesNeeded || !out.nodes) {
      cudaFree(out.nodes); out.nodes = nullptr; out.nodesCap = 0;
      if (cudaMalloc(&out.nodes, nodesNeeded * sizeof(BvhNode2)) != cudaSuccess) return false;
      out.nodesCap = nodesNeeded;
    }
    if (out.packedCap < packedNeeded || !out.packed) {
      cudaFree(out.packed); out.packed = nullptr; out.packedCap = 0;
      if (cudaMalloc(&out.packed, packedNeeded * 48) != cudaSuccess) return false;
      out.packedCap = packedNeeded;
    }
    return true;
  };
  if (n == 0) {  // empty scene: a root with two empty children
    BvhNode2 root;
    root.c0xy = root.c1xy = root.cz = make_float4(MOX_FAR, MOX_FAR, MOX_FAR, MOX_FAR);  // empty children: a point box no ray reaches
    root.ref = make_int4(MOX_EMPTY_CHILD, MOX_EMPTY_CHILD, 0, 0);
    if (!ensureOut(1, 1)) { err = "out of device memory"; return false; }
    CK(cudaMemcpyAsync(out.nodes, &root, sizeof root, cudaMemcpyHostToDevice, stream));
    CK(cudaStreamSynchronize(stream));
    out.nNodes = 1;
    out.refit.path = RefitState::TRIVIAL;
    if (in.evStart) CK(cudaEventRecord(in.evStart, stream));
    if (in.evStop) CK(cudaEventRecord(in.evStop, stream));
    return true;
  }

  uint32_t *keysA = nullptr, *keysB = nullptr, *valsA = nullptr, *valsB = nullptr, *small = nullptr, *status = nullptr;
  float4 *boxLo = nullptr, *boxHi = nullptr;
  int2 *children = nullptr, *range = nullptr;
  int *parentInternal = nullptr, *parentLeaf = nullptr;
  float4 *nodeLo = nullptr, *nodeHi = nullptr;
  uint32_t* arrivals = nullptr;
  const int nTiles = divUp(n, SORT_TILE);
  const int nInnerMax = std::max(n - 1, 1);
  // small: [0..5] centroid bounds, [6] invalid count, [7] error flag, [8..11] tile counters, [16..16+1024) histograms
  const size_t smallWords = 16 + 1024;
  PlocScratch ploc;
  auto freeScratch = [&]() { out.scratchLo = out.scratchHi = nullptr; };  // the arena keeps the memory for the next build
  auto bail = [&](const std::string& what) { freeScratch(); err = what; return false; };
#define CKB(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return bail(std::string(#x) + ": " + cudaGetErrorString(e_)); } while (0)
  // All memory is in place before the first kernel so that the timed build is kernels only.
  const size_t nn = (size_t)n, ni = (size_t)nInnerMax;
  size_t scratchBytes = nn * (2 * 16 + 4 * 4 + 4) + smallWords * 4 + (size_t)4 * nTiles * 256 * 4 + ni * (8 + 8 + 4 + 16 + 16 + 4) + 20 * 256;
  if (in.usePloc && n >= 2) scratchBytes += plocScratchBytes(n);
  const bool wantWide = in.usePloc && in.useWide && n >= 2;
  if (wantWide) scratchBytes += wideScratchBytes(n);
  if (!arena.reserve(scratchBytes)) return bail("out of device memory (build scratch)");
  boxLo = arena.take<float4>(nn); boxHi = arena.take<float4>(nn);
  keysA = arena.take<uint32_t>(nn); keysB = arena.take<uint32_t>(nn);
  valsA = arena.take<uint32_t>(nn); valsB = arena.take<uint32_t>(nn);
  small = arena.take<uint32_t>(smallWords);
  status = arena.take<uint32_t>((size_t)4 * nTiles * 256);
  children = arena.take<int2>(ni); range = arena.take<int2>(ni);
  parentInternal = arena.take<int>(ni); parentLeaf = arena.take<int>(nn);
  nodeLo = arena.take<float4>(ni); nodeHi = arena.take<float4>(ni);
  arrivals = arena.take<uint32_t>(ni);
  if (!arrivals) return bail("build arena too small");
  if (!ensureOut(ni, nn)) return bail("out of device memory (BVH)");
  if (wantWide) {
    if (out.nodes8Cap < nn || !out.nodes8) {
      cudaFree(out.nodes8); out.nodes8 = nullptr; out.nodes8Cap = 0;
      if (cudaMalloc(&out.nodes8, nn * sizeof(BvhNode8)) != cudaSuccess) return bail("out of device memory (wide BVH)");
      out.nodes8Cap = nn;
    }
    if (out.packed8Cap < nn || !out.packed8) {
      cudaFree(out.packed8); out.packed8 = nullptr; out.packed8Cap = 0;
      if (cudaMalloc(&out.packed8, nn * 48) != cudaSuccess) return bail("out of device memory (wide BVH)");
      out.packed8Cap = nn;
    }
  }
  out.scratchLo = boxLo; out.scratchHi = boxHi;
  if (in.usePloc && n >= 2) {
    std::string perr;
    if (!plocAlloc(ploc, n, arena, perr)) return bail(perr);
  }
  if (in.evStart) CKB(cudaEventRecord(in.evStart, stream));

  uint32_t init[16] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  CKB(cudaMemsetAsync(small, 0, smallWords * 4, stream));
  CKB(cudaMemcpyAsync(small, init, sizeof init, cudaMemcpyHostToDevice, stream));
  CKB(cudaMemsetAsync(status, 0, (size_t)4 * nTiles * 256 * 4, stream));
  CKB(cudaMemsetAsync(arrivals, 0, (size_t)nInnerMax * 4, stream));

  const int B = 256;
  k_prim_bounds<<<divUp(n, B), B, 0, stream>>>(n, in.prims, in.tris, in.verts, in.analytic, boxLo, boxHi, small, small + 6);
  k_morton<<<divUp(n, B), B, 0, stream>>>(n, boxLo, boxHi, small, keysA, valsA);
  k_sort_hist<<<std::min(divUp(n, B * 8), histGridCap()), B, 0, stream>>>(keysA, n, small + 16);
  k_sort_scan_hist<<<1, 256, 0, stream>>>(small + 16);
  uint32_t *kin = keysA, *vin = valsA, *kout = keysB, *vout = valsB;
  for (int p = 0; p < 4; ++p) {
    k_sort_pass<<<nTiles, SORT_THREADS, 0, stream>>>(kin, vin, kout, vout, n, 8 * p, small + 16 + 256 * p, small + 8 + p,
                                                     status + (size_t)p * nTiles * 256, small + 7);
    std::swap(kin, kout); std::swap(vin, vout);
  }
  // after 4 passes the sorted data is back in keysA / valsA (kin, vin)
  uint32_t hostSmall[8];
  CKB(cudaMemcpyAsync(hostSmall, small, sizeof hostSmall, cudaMemcpyDeviceToHost, stream));
  CKB(cudaStreamSynchronize(stream));
  if (hostSmall[7]) return bail("radix sort look-back timed out");
  const int nValid = n - (int)hostSmall[6];
  out.nValid = nValid;
  out.nInvalid = (int)hostSmall[6];
  RefitState& rs = out.refit;
  rs.nPrims = n; rs.nValid = nValid;
  rs.primLo = boxLo; rs.primHi = boxHi; rs.sortedIds = vin; rs.flag = small + 12;
  rs.ploc = ploc;
  rs.children = children; rs.range = range; rs.parentInternal = parentInternal; rs.parentLeaf = parentLeaf;
  rs.nodeLo = nodeLo; rs.nodeHi = nodeHi; rs.arrivals = arrivals;

  if (nValid > 0 && (nValid <= 1 || !in.usePloc))
    k_pack<<<divUp(nValid, B), B, 0, stream>>>(nValid, vin, in.prims, in.tris, in.verts, in.analytic, in.mats, out.packed, in.watertight);
  if (nValid <= 1) {
    BvhNode2 root;
    root.c0xy = root.c1xy = root.cz = make_float4(MOX_FAR, MOX_FAR, MOX_FAR, MOX_FAR);
    root.ref = make_int4(MOX_EMPTY_CHILD, MOX_EMPTY_CHILD, 0, 0);
    if (nValid == 1) {
      uint32_t firstId = 0;
      float4 lo, hi;
      CKB(cudaMemcpy(&firstId, vin, 4, cudaMemcpyDeviceToHost));
      CKB(cudaMemcpy(&lo, boxLo + firstId, 16, cudaMemcpyDeviceToHost));
      CKB(cudaMemcpy(&hi, boxHi + firstId, 16, cudaMemcpyDeviceToHost));
      root.c0xy = make_float4(lo.x, hi.x, lo.y, hi.y);
      root.cz = make_float4(lo.z, hi.z, MOX_FAR, MOX_FAR);
      root.ref.x = ~((0 << 3) | 0);
      out.sceneLo[0] = lo.x; out.sceneLo[1] = lo.y; out.sceneLo[2] = lo.z;
      out.sceneHi[0] = hi.x; out.sceneHi[1] = hi.y; out.sceneHi[2] = hi.z;
    }
    CKB(cudaMemcpyAsync(out.nodes, &root, sizeof root, cudaMemcpyHostToDevice, stream));
    out.nNodes = 1;
    if (in.evStop) CKB(cudaEventRecord(in.evStop, stream));
    CKB(cudaStreamSynchronize(stream));
    freeScratch();
    rs.path = RefitState::TRIVIAL;
    return true;
  }

  const int nInner = nValid - 1;
  out.nNodes = nInner;
  if (in.usePloc) {
    std::string perr;
    const PlocResult pr = plocBuild(ploc, nValid, vin, boxLo, boxHi, in.plocRadius > 0 ? in.plocRadius : (nValid > 2000000 ? 16 : 32),
                                    out.nodes, out.sceneLo, out.sceneHi, &out.maxDepth, stream, perr);
    if (pr == PlocResult::ERROR) return bail(perr);
    if (pr == PlocResult::OK && out.maxDepth <= MOX_TRAVERSAL_STACK - 2) {
    k_pack<<<divUp(nValid, B), B, 0, stream>>>(nValid, ploc.orderedIds, in.prims, in.tris, in.verts, in.analytic, in.mats, out.packed, in.watertight);
    if (wantWide) {
      uint32_t* ordered8 = nullptr;
      const uint32_t rootId = (uint32_t)(nValid + nValid - 2);  // the last node PLOC created
      if (!wideCollapse(ploc, nValid, rootId, arena, out.nodes8, &ordered8, &rs.wideSrc, &out.nNodes8, &out.wideLevels, stream, perr))
        return bail(perr);
      k_pack<<<divUp(nValid, B), B, 0, stream>>>(nValid, ordered8, in.prims, in.tris, in.verts, in.analytic, in.mats, out.packed8, in.watertight);
      rs.wide = true; rs.orderedIds8 = ordered8; rs.nNodes8 = out.nNodes8;
    }
    if (in.evStop) CKB(cudaEventRecord(in.evStop, stream));
    CKB(cudaStreamSynchronize(stream));
    CKB(cudaGetLastError());
    out.usedPloc = true;
    freeScratch();
    rs.path = RefitState::PLOC;
    return true;
    }
    // PLOC did not converge (many coincident primitives), or its tree is too deep for the traversal stack: fall through
    // to the radix tree (depth <= 62)
    k_pack<<<divUp(nValid, B), B, 0, stream>>>(nValid, vin, in.prims, in.tris, in.verts, in.analytic, in.mats, out.packed, in.watertight);
  }
  k_karras<<<divUp(nInner, B), B, 0, stream>>>(nValid, kin, children, range, parentInternal, parentLeaf);
  k_refit<<<divUp(nValid, B), B, 0, stream>>>(nValid, vin, boxLo, boxHi, children, parentInternal, parentLeaf, nodeLo, nodeHi, arrivals);
  k_emit2<<<divUp(nInner, B), B, 0, stream>>>(nValid, vin, boxLo, boxHi, children, range, nodeLo, nodeHi, out.nodes);
  if (in.evStop) CKB(cudaEventRecord(in.evStop, stream));
  // scene bounds = root box
  float4 rlo, rhi;
  CKB(cudaMemcpyAsync(&rlo, nodeLo, 16, cudaMemcpyDeviceToHost, stream));
  CKB(cudaMemcpyAsync(&rhi, nodeHi, 16, cudaMemcpyDeviceToHost, stream));
  CKB(cudaStreamSynchronize(stream));
  CKB(cudaGetLastError());
  out.sceneLo[0] = rlo.x; out.sceneLo[1] = rlo.y; out.sceneLo[2] = rlo.z;
  out.sceneHi[0] = rhi.x; out.sceneHi[1] = rhi.y; out.sceneHi[2] = rhi.z;
  freeScratch();
  rs.path = RefitState::KARRAS;
  return true;
#undef CKB
}

bool refitBvh(const BuildInput& in, BuildOutput& out, cudaStream_t stream, std::string& err, bool* validityChanged) {
  const RefitState& rs = out.refit;
  if (rs.path != RefitState::PLOC && rs.path != RefitState::KARRAS) { err = "no hierarchy to refit"; return false; }
  if (rs.nPrims != in.nPrims) { err = "primitive count differs from the build's"; return false; }
  const int n = rs.nPrims, nValid = rs.nValid, nInner = nValid - 1;
  const int B = 256;
  uint32_t* host = (uint32_t*)in.arena->pinned;
  if (in.evStart) CK(cudaEventRecord(in.evStart, stream));
  CK(cudaMemsetAsync(rs.flag, 0, 4, stream));
  k_refit_bounds<<<divUp(n, B), B, 0, stream>>>(n, in.prims, in.tris, in.verts, in.analytic, rs.primLo, rs.primHi, rs.flag);
  if (rs.path == RefitState::PLOC) {
    if (!plocRefit(rs.ploc, nValid, rs.sortedIds, rs.primLo, rs.primHi, rs.arrivals, out.nodes, stream, err)) return false;
    k_pack<<<divUp(nValid, B), B, 0, stream>>>(nValid, rs.ploc.orderedIds, in.prims, in.tris, in.verts, in.analytic, in.mats, out.packed, in.watertight);
    if (rs.wide) {
      wideRefit(rs.wideSrc, rs.nNodes8, rs.ploc.nodeLo, rs.ploc.nodeHi, out.nodes8, stream);
      k_pack<<<divUp(nValid, B), B, 0, stream>>>(nValid, rs.orderedIds8, in.prims, in.tris, in.verts, in.analytic, in.mats, out.packed8, in.watertight);
    }
  } else {
    CK(cudaMemsetAsync(rs.arrivals, 0, (size_t)nInner * 4, stream));
    k_refit<<<divUp(nValid, B), B, 0, stream>>>(nValid, rs.sortedIds, rs.primLo, rs.primHi, rs.children, rs.parentInternal, rs.parentLeaf,
                                                 rs.nodeLo, rs.nodeHi, rs.arrivals);
    k_emit2<<<divUp(nInner, B), B, 0, stream>>>(nValid, rs.sortedIds, rs.primLo, rs.primHi, rs.children, rs.range, rs.nodeLo, rs.nodeHi, out.nodes);
    k_pack<<<divUp(nValid, B), B, 0, stream>>>(nValid, rs.sortedIds, in.prims, in.tris, in.verts, in.analytic, in.mats, out.packed, in.watertight);
  }
  if (in.evStop) CK(cudaEventRecord(in.evStop, stream));
  CK(cudaMemcpyAsync(host, rs.flag, 4, cudaMemcpyDeviceToHost, stream));
  CK(cudaStreamSynchronize(stream));
  CK(cudaGetLastError());
  *validityChanged = host[0] != 0u;
  return true;
}

void excludeUnbuiltLights(uint4* list, int n, const RefitState& rs, cudaStream_t stream) {
  if (n > 0) k_terminal_lights<<<1, MOX_TERMINAL_LIGHTS_MAX, 0, stream>>>(n, rs.primLo, list);
}

// Stand-alone sort entry used by the tests (keys/vals are device pointers, sorted in place).
bool radixSortPairs(uint32_t* keys, uint32_t* vals, int n, cudaStream_t stream, std::string& err) {
  if (n <= 0) return true;
  uint32_t *keysB = nullptr, *valsB = nullptr, *small = nullptr, *status = nullptr;
  const int nTiles = divUp(n, SORT_TILE);
  CK(cudaMalloc(&keysB, (size_t)n * 4)); CK(cudaMalloc(&valsB, (size_t)n * 4));
  CK(cudaMalloc(&small, (16 + 1024) * 4)); CK(cudaMalloc(&status, (size_t)4 * nTiles * 256 * 4));
  CK(cudaMemsetAsync(small, 0, (16 + 1024) * 4, stream));
  CK(cudaMemsetAsync(status, 0, (size_t)4 * nTiles * 256 * 4, stream));
  k_sort_hist<<<std::min(divUp(n, 256 * 8), histGridCap()), 256, 0, stream>>>(keys, n, small + 16);
  k_sort_scan_hist<<<1, 256, 0, stream>>>(small + 16);
  uint32_t *kin = keys, *vin = vals, *kout = keysB, *vout = valsB;
  for (int p = 0; p < 4; ++p) {
    k_sort_pass<<<nTiles, SORT_THREADS, 0, stream>>>(kin, vin, kout, vout, n, 8 * p, small + 16 + 256 * p, small + 8 + p,
                                                     status + (size_t)p * nTiles * 256, small + 7);
    std::swap(kin, kout); std::swap(vin, vout);
  }
  uint32_t flag = 0;
  CK(cudaMemcpyAsync(&flag, small + 7, 4, cudaMemcpyDeviceToHost, stream));
  CK(cudaStreamSynchronize(stream));
  CK(cudaGetLastError());
  cudaFree(keysB); cudaFree(valsB); cudaFree(small); cudaFree(status);
  if (flag) { err = "radix sort look-back timed out"; return false; }
  return true;
}
