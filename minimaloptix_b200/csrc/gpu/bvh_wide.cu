// bvh_wide.cu — collapse of the binary PLOC tree into a compressed 8-wide BVH
// (Ylitie, Karras, Laine 2017).  One thread per wide node, level by level:
//   * the <= 8 children of a wide node are the binary subtrees chosen by the SAH-optimal collapse programme
//     (k_collapse_dp below); without it (MOX_WIDE_GREEDY, > 4 M primitives): start from the two children of a
//     binary node and keep opening the child with the largest surface area until there are 8 children or
//     nothing left to open; binary subtrees of <= MOX_WIDE_LEAF_MAX primitives become leaf children;
//   * children are placed in the 8 slots by the octant of their centroid relative to the node
//     centre (nearest free slot when taken), which is what lets traversal order them by
//     slot ^ ray-octant;
//   * child boxes are quantised to 8 bits per plane on a per-node power-of-two grid, rounded
//     outwards and verified, so the wide BVH never culls what the binary one would keep;
//   * inner children get consecutive node indices, the primitives of the leaf children a
//     consecutive block of the wide-leaf-ordered primitive array (both via atomic counters).
#include <cstdlib>
#include "build.h"
#include "vec.cuh"

namespace {

struct WorkItem { uint32_t binNode; uint32_t wideIndex; };

__device__ __forceinline__ float halfArea(const float4& lo, const float4& hi) {
  float dx = hi.x - lo.x, dy = hi.y - lo.y, dz = hi.z - lo.z;
  return dx * dy + dy * dz + dz * dx;
}

// biased exponent e such that 255 * 2^(e-127) >= extent (and >= a tiny positive grid for flat boxes)
__device__ __forceinline__ uint32_t gridExponent(float extent) {
  float v = fmaxf(extent, 1e-30f) * (1.0f / 255.0f);
  int k;
  frexpf(v, &k);  // v = m * 2^k, m in [0.5, 1)  ->  2^k > v
  int e = k + 127;
  e = max(1, min(e, 254));
  // guard against rounding in the division above
  while (e < 254 && 255.0f * __uint_as_float((uint32_t)e << 23) < extent) ++e;
  return (uint32_t)e;
}

// Grid of a wide node whose box is [blo, bhi]: biased exponents and the scales 2^(e-127) per axis.
struct WideGrid { uint32_t ex, ey, ez; float sx, sy, sz; };
__device__ __forceinline__ WideGrid wideGrid(const float4& blo, const float4& bhi) {
  WideGrid g;
  g.ex = gridExponent(bhi.x - blo.x); g.ey = gridExponent(bhi.y - blo.y); g.ez = gridExponent(bhi.z - blo.z);
  g.sx = __uint_as_float(g.ex << 23); g.sy = __uint_as_float(g.ey << 23); g.sz = __uint_as_float(g.ez << 23);
  return g;
}

// 8-bit planes of the child box [lo, hi] in slot s of a node with origin blo: outward rounding, then verified against
// the float planes the traversal will reconstruct.  The collapse and the refit both quantise here.
__device__ __forceinline__ void quantiseChild(const float4& lo, const float4& hi, const float4& blo, const WideGrid& g, int s,
                                              uint32_t* qlx, uint32_t* qly, uint32_t* qlz, uint32_t* qhx, uint32_t* qhy, uint32_t* qhz) {
  int ql, qh;
  ql = (int)floorf((lo.x - blo.x) / g.sx); ql = max(0, min(255, ql)); while (ql > 0 && blo.x + ql * g.sx > lo.x) --ql;
  qh = (int)ceilf((hi.x - blo.x) / g.sx); qh = max(0, min(255, qh)); while (qh < 255 && blo.x + qh * g.sx < hi.x) ++qh;
  qlx[s] = ql; qhx[s] = qh;
  ql = (int)floorf((lo.y - blo.y) / g.sy); ql = max(0, min(255, ql)); while (ql > 0 && blo.y + ql * g.sy > lo.y) --ql;
  qh = (int)ceilf((hi.y - blo.y) / g.sy); qh = max(0, min(255, qh)); while (qh < 255 && blo.y + qh * g.sy < hi.y) ++qh;
  qly[s] = ql; qhy[s] = qh;
  ql = (int)floorf((lo.z - blo.z) / g.sz); ql = max(0, min(255, ql)); while (ql > 0 && blo.z + ql * g.sz > lo.z) --ql;
  qh = (int)ceilf((hi.z - blo.z) / g.sz); qh = max(0, min(255, qh)); while (qh < 255 && blo.z + qh * g.sz < hi.z) ++qh;
  qlz[s] = ql; qhz[s] = qh;
}

__device__ __forceinline__ uint32_t pack4(const uint32_t* v) { return v[0] | (v[1] << 8) | (v[2] << 16) | (v[3] << 24); }

// n0 .xyz / .w and the planes n2 .. n4 of a node (n1 is the caller's)
__device__ __forceinline__ void wideBoxWords(BvhNode8& nd, const float4& blo, const WideGrid& g, uint32_t imask, const uint32_t* qlx,
                                             const uint32_t* qly, const uint32_t* qlz, const uint32_t* qhx, const uint32_t* qhy,
                                             const uint32_t* qhz) {
  nd.n0 = make_float4(blo.x, blo.y, blo.z, __uint_as_float(g.ex | (g.ey << 8) | (g.ez << 16) | (imask << 24)));
  nd.n2 = make_float4(__uint_as_float(pack4(qlx)), __uint_as_float(pack4(qlx + 4)), __uint_as_float(pack4(qly)), __uint_as_float(pack4(qly + 4)));
  nd.n3 = make_float4(__uint_as_float(pack4(qlz)), __uint_as_float(pack4(qlz + 4)), __uint_as_float(pack4(qhx)), __uint_as_float(pack4(qhx + 4)));
  nd.n4 = make_float4(__uint_as_float(pack4(qhy)), __uint_as_float(pack4(qhy + 4)), __uint_as_float(pack4(qhz)), __uint_as_float(pack4(qhz + 4)));
}

// ---- optimal collapse (Ylitie et al. 2017, section 3.1) -----------------------------------------------------
// C(n, i): cheapest way to represent the subtree of binary node n as a forest of at most i wide-BVH children,
//   C(n, 1) = min(C_leaf(n), C_distribute(n, 8) + A_n c_node),   C_leaf(n) = A_n P_n c_prim if P_n <= leaf max
//   C(n, i) = min(C_distribute(n, i), C(n, i - 1)),               C_distribute(n, j) = min_k C(left, k) + C(right, j - k)
// with surface areas A, c_prim / c_node = 0.43 (instructions of a primitive step / a node step of the traversal).
// Computed bottom-up (per-node arrival counters, as the refit of the radix tree); the decisions are packed per
// inner binary node: bit 0 = wide node, bits 1 + 3 (j - 2) .. = best k of C_distribute(n, j) for j = 2..8,
// bit 22 + (i - 2) = "C(n, i) is C(n, i - 1)" for i = 2..7.  scripts/collapse_study.py is the numpy model of this
// (4.5 - 5.4 % lower SAH cost than the greedy largest-area-first collapse on the bench scene).
#ifndef MOX_COLLAPSE_PRIM_COST
#define MOX_COLLAPSE_PRIM_COST 0.43f  // flat around it: 0.25 -> 1302, 0.43 -> 1307, 0.7 -> 1310 Mrays/s on the bench scene
#endif
constexpr float kCostNode = 1.0f, kCostPrim = MOX_COLLAPSE_PRIM_COST;

__global__ void k_collapse_dp(int nLeaves, uint32_t root, const uint2* __restrict__ children, const uint32_t* __restrict__ parent,
                              const float4* __restrict__ nodeLo, const float4* __restrict__ nodeHi, const uint32_t* __restrict__ size,
                              float4* __restrict__ cost /* 2 per inner node: C(n, 1..7), - */, uint32_t* __restrict__ decision,
                              uint32_t* __restrict__ arrivals) {
  int leaf = blockIdx.x * blockDim.x + threadIdx.x;
  if (leaf >= nLeaves) return;
  uint32_t node = parent[leaf];
  while (true) {
    const uint32_t in = node - (uint32_t)nLeaves;
    if (atomicAdd(&arrivals[in], 1u) == 0u) return;  // the sibling subtree is not finished yet
    const uint2 ch = children[in];
    float cl[8], cr[8];  // index 1..7
    if (ch.x < (uint32_t)nLeaves) { float a = kCostPrim * halfArea(nodeLo[ch.x], nodeHi[ch.x]); for (int i = 1; i < 8; ++i) cl[i] = a; }
    else {
      float4 a = __ldcg(&cost[2 * (size_t)(ch.x - nLeaves)]), b = __ldcg(&cost[2 * (size_t)(ch.x - nLeaves) + 1]);
      cl[1] = a.x; cl[2] = a.y; cl[3] = a.z; cl[4] = a.w; cl[5] = b.x; cl[6] = b.y; cl[7] = b.z;
    }
    if (ch.y < (uint32_t)nLeaves) { float a = kCostPrim * halfArea(nodeLo[ch.y], nodeHi[ch.y]); for (int i = 1; i < 8; ++i) cr[i] = a; }
    else {
      float4 a = __ldcg(&cost[2 * (size_t)(ch.y - nLeaves)]), b = __ldcg(&cost[2 * (size_t)(ch.y - nLeaves) + 1]);
      cr[1] = a.x; cr[2] = a.y; cr[3] = a.z; cr[4] = a.w; cr[5] = b.x; cr[6] = b.y; cr[7] = b.z;
    }
    const float area = halfArea(nodeLo[node], nodeHi[node]);
    float dist[9];
    uint32_t dec = 0;
#pragma unroll
    for (int j = 2; j <= 8; ++j) {
      float best = __int_as_float(0x7f800000);
      int bestK = 1;
#pragma unroll
      for (int k = 1; k < j; ++k) {
        if (k > 7 || j - k > 7) continue;
        float c = cl[k] + cr[j - k];
        if (c < best) { best = c; bestK = k; }
      }
      dist[j] = best;
      dec |= (uint32_t)bestK << (1 + 3 * (j - 2));
    }
    const uint32_t sz = size[node];
    const float cLeaf = sz <= MOX_WIDE_LEAF_MAX ? area * (float)sz * kCostPrim : __int_as_float(0x7f800000);
    const float cInt = dist[8] + area * kCostNode;
    float c[8];
    c[1] = fminf(cLeaf, cInt);
    if (cInt < cLeaf) dec |= 1u;
#pragma unroll
    for (int i = 2; i <= 7; ++i) {
      if (dist[i] < c[i - 1]) c[i] = dist[i];
      else { c[i] = c[i - 1]; dec |= 1u << (22 + (i - 2)); }
    }
    __stcg(&cost[2 * (size_t)in], make_float4(c[1], c[2], c[3], c[4]));
    __stcg(&cost[2 * (size_t)in + 1], make_float4(c[5], c[6], c[7], 0.f));
    decision[in] = dec;
    __threadfence();
    if (node == root) return;
    node = parent[node];
  }
}

__global__ void __launch_bounds__(128)
k_collapse_level(int nItems, const WorkItem* __restrict__ items, int nLeaves, const uint2* __restrict__ children,
                 const float4* __restrict__ nodeLo, const float4* __restrict__ nodeHi, const uint32_t* __restrict__ size,
                 const uint32_t* __restrict__ parent, const uint32_t* __restrict__ leafPos, const uint32_t* __restrict__ firstPos, uint32_t root,
                 const uint32_t* __restrict__ orderedIds, BvhNode8* __restrict__ out, uint32_t* __restrict__ orderedIds8,
                 WorkItem* __restrict__ nextItems, uint32_t* __restrict__ counters /* [0] nodes, [1] prims */,
                 const uint32_t* __restrict__ levelCount /* items of this level; [1]: of the next, filled here */,
                 const uint32_t* __restrict__ decision /* null: greedy collapse */, uint32_t* __restrict__ wideSrc) {
  int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= nItems || w >= (int)__ldg(levelCount)) return;   // nItems: the host's upper bound (grid size)
  const WorkItem it = items[w];
  uint32_t ch[8];
  int n = 0;
  if (decision) {
    // ---- the children the dynamic programme chose: hand the 8 slots down the binary tree along its decisions
    uint32_t stNode[16];
    int stBudget[16], sp = 0;
    {
      const uint2 c = children[it.binNode - nLeaves];
      const int k = (int)((decision[it.binNode - nLeaves] >> (1 + 3 * 6)) & 7u);  // best k of C_distribute(n, 8)
      stNode[sp] = c.y; stBudget[sp++] = 8 - k;
      stNode[sp] = c.x; stBudget[sp++] = k;
    }
    while (sp > 0) {
      const uint32_t m = stNode[--sp];
      int i = stBudget[sp];
      if (m < (uint32_t)nLeaves) { ch[n++] = m; continue; }
      const uint32_t d = decision[m - nLeaves];
      while (i > 1 && (d >> (22 + (i - 2)) & 1u)) --i;   // C(m, i) inherited from C(m, i - 1)
      if (i <= 1) { ch[n++] = m; continue; }              // one root: a leaf child or an inner wide node
      const uint2 c = children[m - nLeaves];
      const int k = (int)((d >> (1 + 3 * (i - 2))) & 7u);
      stNode[sp] = c.y; stBudget[sp++] = i - k;
      stNode[sp] = c.x; stBudget[sp++] = k;
    }
  } else {
  // ---- gather up to 8 children by repeatedly opening the largest openable one
    {
      uint2 c = children[it.binNode - nLeaves];
      ch[n++] = c.x; ch[n++] = c.y;
    }
    while (n < 8) {
      int best = -1;
      float bestA = -1.f;
      for (int i = 0; i < n; ++i) {
        if (ch[i] < (uint32_t)nLeaves || size[ch[i]] <= MOX_WIDE_LEAF_MAX) continue;  // a leaf child stays closed
        float a = halfArea(nodeLo[ch[i]], nodeHi[ch[i]]);
        if (a > bestA) { bestA = a; best = i; }
      }
      if (best < 0) break;
      uint2 c = children[ch[best] - nLeaves];
      ch[best] = c.x;
      ch[n++] = c.y;
    }
    // free slots left: also open small leaf subtrees (largest first), so the bottom nodes give every
    // primitive its own 8-bit box instead of leaving slots empty
    while (n < 8) {
      int best = -1;
      float bestA = -1.f;
      for (int i = 0; i < n; ++i) {
        if (ch[i] < (uint32_t)nLeaves) continue;  // a single primitive
        float a = halfArea(nodeLo[ch[i]], nodeHi[ch[i]]);
        if (a > bestA) { bestA = a; best = i; }
      }
      if (best < 0) break;
      uint2 c = children[ch[best] - nLeaves];
      ch[best] = c.x;
      ch[n++] = c.y;
    }
  }
  // ---- node box and grid
  const float4 blo = nodeLo[it.binNode], bhi = nodeHi[it.binNode];
  const WideGrid g = wideGrid(blo, bhi);
  const float cx = 0.5f * (blo.x + bhi.x), cy = 0.5f * (blo.y + bhi.y), cz = 0.5f * (blo.z + bhi.z);
  // ---- slots by centroid octant, nearest free slot (Hamming distance) when taken
  int slotOf[8];
  uint32_t used = 0;
  for (int i = 0; i < n; ++i) {
    float4 lo = nodeLo[ch[i]], hi = nodeHi[ch[i]];
    int want = ((0.5f * (lo.x + hi.x) > cx) ? 4 : 0) | ((0.5f * (lo.y + hi.y) > cy) ? 2 : 0) | ((0.5f * (lo.z + hi.z) > cz) ? 1 : 0);
    int bestS = -1, bestD = 99;
    for (int s = 0; s < 8; ++s) {
      if (used & (1u << s)) continue;
      int d = __popc((uint32_t)(s ^ want));
      if (d < bestD) { bestD = d; bestS = s; }
    }
    slotOf[i] = bestS;
    used |= 1u << bestS;
  }
  // ---- classify, count, allocate
  uint32_t imask = 0, nInner = 0, nPrims = 0;
  int childAt[8];
  for (int s = 0; s < 8; ++s) childAt[s] = -1;
  for (int i = 0; i < n; ++i) {
    childAt[slotOf[i]] = i;
    bool inner = ch[i] >= (uint32_t)nLeaves && size[ch[i]] > MOX_WIDE_LEAF_MAX;
    if (inner) { imask |= 1u << slotOf[i]; nInner++; }
    else nPrims += ch[i] < (uint32_t)nLeaves ? 1u : size[ch[i]];
  }
  const uint32_t childBase = nInner ? atomicAdd(&counters[0], nInner) : 0u;
  const uint32_t primBase = nPrims ? atomicAdd(&counters[1], nPrims) : 0u;
  const uint32_t nextBase = nInner ? atomicAdd(const_cast<uint32_t*>(levelCount) + 1, nInner) : 0u;
  // ---- emit
  uint32_t qlx[8], qly[8], qlz[8], qhx[8], qhy[8], qhz[8];
  uint32_t innerRank = 0, primOff = 0;
  uint32_t validPrims = 0;   // bits 2s, 2s + 1 = the primitives of the leaf child in slot s
  uint32_t* srcOut = wideSrc + 9 * (size_t)it.wideIndex;   // for the refit: this node's binary node and each slot's
  srcOut[0] = it.binNode;
  for (int s = 0; s < 8; ++s) {
    int i = childAt[s];
    if (i < 0) {  // empty slot: inverted box, never hit
      qlx[s] = qly[s] = qlz[s] = 255; qhx[s] = qhy[s] = qhz[s] = 0;
      srcOut[1 + s] = ~0u;
      continue;
    }
    const uint32_t c = ch[i];
    srcOut[1 + s] = c;
    quantiseChild(nodeLo[c], nodeHi[c], blo, g, s, qlx, qly, qlz, qhx, qhy, qhz);
    if (imask & (1u << s)) {
      nextItems[nextBase + innerRank] = WorkItem{c, childBase + innerRank};
      innerRank++;
    } else {
      uint32_t cnt = c < (uint32_t)nLeaves ? 1u : size[c];
      // first primitive of the subtree in binary leaf order
      uint32_t first;
      if (c < (uint32_t)nLeaves) first = leafPos[c];
      else first = firstPos[c - nLeaves];   // leaf-order position of the subtree's first primitive (k_ploc_leaf_order)
      for (uint32_t k = 0; k < cnt; ++k) orderedIds8[primBase + primOff + k] = orderedIds[first + k];
      validPrims |= ((1u << cnt) - 1u) << (2 * s);
      primOff += cnt;
    }
  }
  BvhNode8 nd;
  wideBoxWords(nd, blo, g, imask, qlx, qly, qlz, qhx, qhy, qhz);
  nd.n1 = make_float4(__uint_as_float(childBase), __uint_as_float(primBase), __uint_as_float((imask << 24) | validPrims),
                      __uint_as_float((validPrims << 8) | imask));
  out[it.wideIndex] = nd;
}

// Refit of the wide nodes after the binary boxes were refitted: one thread per node, no level order needed.  The box
// comes from the node's binary node, the slot planes from the binary node in each slot; n1 (bases, valid bits) and the
// inner mask stay.
__global__ void __launch_bounds__(128)
k_wide_refit(int nNodes, const uint32_t* __restrict__ wideSrc, const float4* __restrict__ nodeLo, const float4* __restrict__ nodeHi,
             BvhNode8* __restrict__ nodes) {
  int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= nNodes) return;
  const uint32_t* src = wideSrc + 9 * (size_t)w;
  const float4 blo = nodeLo[src[0]], bhi = nodeHi[src[0]];
  const WideGrid g = wideGrid(blo, bhi);
  uint32_t qlx[8], qly[8], qlz[8], qhx[8], qhy[8], qhz[8];
  for (int s = 0; s < 8; ++s) {
    const uint32_t c = src[1 + s];
    if (c == ~0u) { qlx[s] = qly[s] = qlz[s] = 255; qhx[s] = qhy[s] = qhz[s] = 0; continue; }
    quantiseChild(nodeLo[c], nodeHi[c], blo, g, s, qlx, qly, qlz, qhx, qhy, qhz);
  }
  BvhNode8 nd = nodes[w];
  wideBoxWords(nd, blo, g, __float_as_uint(nd.n0.w) >> 24, qlx, qly, qlz, qhx, qhy, qhz);
  nodes[w] = nd;
}

inline int divUp(size_t a, size_t b) { return (int)((a + b - 1) / b); }

}  // namespace

#define WCK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { err = std::string(#x) + ": " + cudaGetErrorString(e_); return false; } } while (0)

size_t wideScratchBytes(int n) {
  // two work queues of at most n/2 items (8 B each), 4 counters, 258 level counts, the wide-leaf order; slack for alignment
  // + the collapse programme: 2 float4 of costs, one decision word and one arrival counter per inner binary node
  // + the refit's slot map: 36 bytes per wide node (at most n)
  return (size_t)std::max(n, 2) * (8 + 8 + 4 + 32 + 4 + 4 + 36) + 10 * 256 + 1024 + 2048;   // + the per-level item counts
}

// Collapse the PLOC tree held in `s` (n >= 2 leaves) into outNodes (capacity >= n wide nodes) and
// fill orderedIds8 (n entries).  *nNodesOut receives the number of wide nodes.
bool wideCollapse(const PlocScratch& s, int n, uint32_t root, DeviceArena& arena, BvhNode8* outNodes, uint32_t** orderedIds8Out,
                  uint32_t** wideSrcOut, int* nNodesOut, int* levelsOut, cudaStream_t stream, std::string& err) {
  WorkItem* q[2] = {arena.take<WorkItem>((size_t)n), arena.take<WorkItem>((size_t)n)};
  uint32_t* counters = arena.take<uint32_t>(4);
  uint32_t* orderedIds8 = arena.take<uint32_t>((size_t)n);
  uint32_t* wideSrc = arena.take<uint32_t>(9 * (size_t)n);
  if (!orderedIds8 || !q[0] || !q[1] || !counters || !wideSrc) { err = "wide-BVH scratch does not fit the build arena"; return false; }
  // optimal collapse up to 4 M primitives (above, the greedy collapse keeps the build inside its time budget)
  const uint32_t* decision = nullptr;
  const char* env = getenv("MOX_WIDE_GREEDY");
  if (n <= 4000000 && !(env && atoi(env))) {
    float4* cost = arena.take<float4>(2 * (size_t)n);
    uint32_t* dec = arena.take<uint32_t>((size_t)n);
    uint32_t* arrivals = arena.take<uint32_t>((size_t)n);
    if (!cost || !dec || !arrivals) { err = "wide-BVH scratch does not fit the build arena"; return false; }
    WCK(cudaMemsetAsync(arrivals, 0, (size_t)n * 4, stream));
    k_collapse_dp<<<divUp(n, 128), 128, 0, stream>>>(n, root, s.children, s.parent, s.nodeLo, s.nodeHi, s.size, cost, dec, arrivals);
    decision = dec;
  }
  // Level by level, the item count of each level kept on the device (levelCount[l], filled by level l-1): the host
  // enqueues kLevelBatch levels back to back with grids sized for the most a level can hold (8x the level before,
  // never more than n/2 inner nodes) and reads the counts back once per batch.
  constexpr int kMaxLevels = 256, kLevelBatch = 4;
  uint32_t* levelCount = arena.take<uint32_t>(kMaxLevels + 2);
  if (!levelCount) { err = "wide-BVH scratch does not fit the build arena"; return false; }
  WCK(cudaMemsetAsync(levelCount, 0, (kMaxLevels + 2) * 4, stream));
  uint32_t* host = (uint32_t*)arena.pinned;   // 64 pinned bytes: [0..3] counters, [4..8] counts of a batch of levels
  host[0] = 1u; host[1] = 0u; host[2] = 0u; host[3] = 0u;   // node 0 is the root
  host[4] = 1u;
  WorkItem* rootItem = (WorkItem*)(host + 8);
  *rootItem = WorkItem{root, 0u};
  WCK(cudaMemcpyAsync(counters, host, 16, cudaMemcpyHostToDevice, stream));
  WCK(cudaMemcpyAsync(levelCount, host + 4, 4, cudaMemcpyHostToDevice, stream));
  WCK(cudaMemcpyAsync(q[0], rootItem, sizeof(WorkItem), cudaMemcpyHostToDevice, stream));
  int cur = 0, levels = 0;
  size_t bound = 1;   // upper bound of the items of level `levels`
  for (bool more = true; more;) {
    if (levels + kLevelBatch >= kMaxLevels) { err = "wide collapse did not terminate"; return false; }
    for (int b = 0; b < kLevelBatch; ++b, ++levels) {
      k_collapse_level<<<divUp(bound, 128), 128, 0, stream>>>((int)bound, q[cur], n, s.children, s.nodeLo, s.nodeHi, s.size, s.parent, s.leafPos, s.firstPos,
                                                             root, s.orderedIds, outNodes, orderedIds8, q[cur ^ 1], counters, levelCount + levels, decision,
                                                             wideSrc);
      cur ^= 1;
      bound = std::min<size_t>(bound * 8, (size_t)std::max(n / 2, 1));
    }
    WCK(cudaMemcpyAsync(host, counters, 16, cudaMemcpyDeviceToHost, stream));
    WCK(cudaMemcpyAsync(host + 4, levelCount + levels - kLevelBatch + 1, kLevelBatch * 4, cudaMemcpyDeviceToHost, stream));
    WCK(cudaStreamSynchronize(stream));
    *nNodesOut = (int)host[0];
    if ((int)host[1] > n) { err = "wide collapse emitted too many primitives"; return false; }
    // the first empty level ends the tree (the levels enqueued after it did nothing)
    for (int b = 0; b < kLevelBatch; ++b)
      if (host[4 + b] == 0u) { more = false; levels = levels - kLevelBatch + 1 + b; break; }
    if (more) bound = std::min<size_t>(bound, (size_t)host[4 + kLevelBatch - 1] );
  }
  if ((int)host[1] != n) { err = "wide collapse lost primitives (" + std::to_string(host[1]) + " of " + std::to_string(n) + ")"; return false; }
  WCK(cudaGetLastError());
  *orderedIds8Out = orderedIds8;
  *wideSrcOut = wideSrc;
  *levelsOut = levels;
  return true;
}

void wideRefit(const uint32_t* wideSrc, int nNodes, const float4* nodeLo, const float4* nodeHi, BvhNode8* nodes, cudaStream_t stream) {
  k_wide_refit<<<divUp((size_t)nNodes, 128), 128, 0, stream>>>(nNodes, wideSrc, nodeLo, nodeHi, nodes);
}
