// ploc.cu — higher-quality hierarchy over the Morton-sorted primitives: parallel locally-ordered
// clustering (Meister & Bittner 2018).  Starting from one cluster per primitive in Morton order,
// every iteration (1) finds each cluster's nearest neighbour — smallest merged surface area —
// within a window of +-radius, (2) merges mutual nearest-neighbour pairs into a new inner node,
// (3) compacts the cluster array, keeping its order.  The result is a binary tree whose SAH cost
// is well below the Karras radix tree's (which only looks at Morton prefixes); it then goes
// through the same emit / leaf-fold / pack stages.  Plays the role OptiX's closed "Trbvh"
// builder had for the reference (MinimalOptiX.cpp:378,494,534).
//
// Node ids: [0, N) leaves (leaf i = i-th primitive in Morton order), [N, 2N-1) inner nodes in
// creation order (the root is created last).  Ids are assigned by a prefix scan, not by atomics,
// so the build is deterministic.
#include "build.h"
#include "vec.cuh"

namespace {

constexpr int PL_THREADS = 256;
constexpr int PL_ITEMS = 4;
constexpr int PL_TILE = PL_THREADS * PL_ITEMS;
constexpr int PL_MAX_RADIUS = 128;
constexpr int PL_TAIL = 1024;      // at most this many clusters: the single-block kernel finishes the tree
constexpr int PL_MAX_ITERS = 250;  // state slots (a 10 M-primitive build takes ~40 iterations)
constexpr int PL_BATCH = 8;        // iterations enqueued between two host read-backs

// Loop state of the clustering, one slot per iteration, in device memory: iteration `it` reads slot it and its merge
// kernel (the block of the last tile) writes slot it+1, so the host can enqueue PL_BATCH iterations back to back —
// grids sized for the last count it knows (counts only shrink; surplus blocks return at once) — and read one slot back per batch instead of
// one count per iteration.  An iteration whose slot says count <= PL_TAIL does nothing.
}  // namespace
struct PlocState { int count; uint32_t nodeBase; uint32_t iters; uint32_t pad; };
namespace {

__device__ __forceinline__ float mergedArea(const float4& alo, const float4& ahi, const float4& blo, const float4& bhi) {
  float dx = fmaxf(ahi.x, bhi.x) - fminf(alo.x, blo.x);
  float dy = fmaxf(ahi.y, bhi.y) - fminf(alo.y, blo.y);
  float dz = fmaxf(ahi.z, bhi.z) - fminf(alo.z, blo.z);
  return dx * dy + dy * dz + dz * dx;
}

// leaf clusters: id = i, box = box of the i-th sorted primitive
__global__ void k_ploc_init(int n, const uint32_t* __restrict__ sortedIds, const float4* __restrict__ primLo,
                            const float4* __restrict__ primHi, uint32_t* __restrict__ cid, float4* __restrict__ cLo,
                            float4* __restrict__ cHi, float4* __restrict__ nodeLo, float4* __restrict__ nodeHi,
                            uint32_t* __restrict__ size) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t id = sortedIds[i];
  float4 lo = primLo[id], hi = primHi[id];
  cid[i] = (uint32_t)i;
  cLo[i] = lo; cHi[i] = hi;
  nodeLo[i] = lo; nodeHi[i] = hi;
  size[i] = 1u;
}

// nearest neighbour of cluster i among [i - radius, i + radius]; ties -> smaller index.
__global__ void __launch_bounds__(PL_THREADS) k_ploc_nn(const PlocState* __restrict__ st, int radius, const float4* __restrict__ cLo,
                                                        const float4* __restrict__ cHi, uint32_t* __restrict__ nn) {
  __shared__ float4 sLo[PL_THREADS + 2 * PL_MAX_RADIUS], sHi[PL_THREADS + 2 * PL_MAX_RADIUS];
  const int n = st->count;
  if (n <= PL_TAIL || blockIdx.x * PL_THREADS >= n) return;
  const int base = blockIdx.x * PL_THREADS - radius;
  for (int k = threadIdx.x; k < PL_THREADS + 2 * radius; k += PL_THREADS) {
    int j = base + k;
    if (j >= 0 && j < n) { sLo[k] = cLo[j]; sHi[k] = cHi[j]; }
  }
  __syncthreads();
  const int i = blockIdx.x * PL_THREADS + threadIdx.x;
  if (i >= n) return;
  const int me = threadIdx.x + radius;
  const float4 lo = sLo[me], hi = sHi[me];
  float best = __int_as_float(0x7f800000);
  int bestJ = -1;
  for (int o = -radius; o <= radius; ++o) {
    int j = i + o;
    if (o == 0 || j < 0 || j >= n) continue;
    float a = mergedArea(lo, hi, sLo[me + o], sHi[me + o]);
    if (a < best) { best = a; bestJ = j; }  // ascending j: the first minimum has the smallest index
  }
  nn[i] = (uint32_t)bestJ;
}

// flags of cluster i: low word = survives compaction (1/0), high word = creates a node (1/0)
__device__ __forceinline__ unsigned long long plocFlags(int i, int n, const uint32_t* __restrict__ nn) {
  if (i >= n) return 0ull;
  int j = (int)nn[i];
  bool mutual = j >= 0 && (int)nn[j] == i;
  bool merged = mutual && i < j, removed = mutual && i > j;
  return (removed ? 0ull : 1ull) | (merged ? (1ull << 32) : 0ull);
}

__device__ __forceinline__ unsigned long long blockReduce(unsigned long long v, unsigned long long* sh) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  unsigned long long t = 0;
  for (int w = 0; w < PL_THREADS / 32; ++w) t += sh[w];
  __syncthreads();
  return t;
}

__global__ void __launch_bounds__(PL_THREADS) k_ploc_tile_sums(const PlocState* __restrict__ st, const uint32_t* __restrict__ nn,
                                                               unsigned long long* __restrict__ tileSums) {
  __shared__ unsigned long long sh[PL_THREADS / 32];
  const int n = st->count;
  if (n <= PL_TAIL || blockIdx.x * PL_TILE >= n) return;
  unsigned long long v = 0;
  int base = blockIdx.x * PL_TILE + threadIdx.x * PL_ITEMS;
#pragma unroll
  for (int k = 0; k < PL_ITEMS; ++k) v += plocFlags(base + k, n, nn);
  unsigned long long t = blockReduce(v, sh);
  if (threadIdx.x == 0) tileSums[blockIdx.x] = t;
}

// merge mutual pairs and compact: new cluster arrays, new inner nodes.  Every block sums the tile totals in front of
// it itself (at most 10 K values of 8 bytes, L2-resident) — no scan kernel between the two — and the block of the
// last tile, which then knows the grand totals, advances the loop state: st[0] is this iteration's slot, st[1] the
// next one's.
__global__ void __launch_bounds__(PL_THREADS)
k_ploc_merge(PlocState* __restrict__ st, int nLeaves, const uint32_t* __restrict__ nn, const unsigned long long* __restrict__ tileSums,
             const uint32_t* __restrict__ cidIn, const float4* __restrict__ cLoIn, const float4* __restrict__ cHiIn,
             uint32_t* __restrict__ cidOut, float4* __restrict__ cLoOut, float4* __restrict__ cHiOut,
             float4* __restrict__ nodeLo, float4* __restrict__ nodeHi, uint2* __restrict__ children, uint32_t* __restrict__ parent,
             uint32_t* __restrict__ size) {
  __shared__ unsigned long long sh[PL_THREADS / 32];
  __shared__ unsigned long long warpOff[PL_THREADS / 32];
  const int n = st->count;
  if (n <= PL_TAIL) { if (blockIdx.x == 0 && threadIdx.x == 0) st[1] = st[0]; return; }   // nothing left to do here
  if (blockIdx.x * PL_TILE >= n) return;
  const uint32_t nodeBase = st->nodeBase;
  unsigned long long tileOffset;
  {
    unsigned long long part = 0;
    for (int t = threadIdx.x; t < (int)blockIdx.x; t += PL_THREADS) part += tileSums[t];
    tileOffset = blockReduce(part, sh);
  }
  const int base = blockIdx.x * PL_TILE + threadIdx.x * PL_ITEMS;
  unsigned long long f[PL_ITEMS], v = 0;
#pragma unroll
  for (int k = 0; k < PL_ITEMS; ++k) { f[k] = plocFlags(base + k, n, nn); v += f[k]; }
  // exclusive scan of v over the block
  unsigned long long incl = v;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int o = 1; o < 32; o <<= 1) {
    unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) sh[warp] = incl;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long run = 0;
    for (int w = 0; w < PL_THREADS / 32; ++w) { warpOff[w] = run; run += sh[w]; }
    if ((int)blockIdx.x == (n + PL_TILE - 1) / PL_TILE - 1) {   // last tile: totals of the iteration
      const unsigned long long total = tileOffset + run;
      PlocState nx;
      nx.count = (int)(total & 0xffffffffull);
      nx.nodeBase = nodeBase + (uint32_t)(total >> 32);
      nx.iters = st->iters + 1u;
      nx.pad = 0u;
      st[1] = nx;
    }
  }
  __syncthreads();
  unsigned long long off = tileOffset + warpOff[warp] + incl - v;
#pragma unroll
  for (int k = 0; k < PL_ITEMS; ++k) {
    int i = base + k;
    if (i < n && (f[k] & 1ull)) {
      uint32_t pos = (uint32_t)(off & 0xffffffffull);
      if (f[k] >> 32) {
        uint32_t j = nn[i];
        uint32_t node = nodeBase + (uint32_t)(off >> 32);  // id among inner nodes
        uint32_t a = cidIn[i], b = cidIn[j];
        float4 alo = cLoIn[i], ahi = cHiIn[i], blo = cLoIn[j], bhi = cHiIn[j];
        float4 lo = make_float4(fminf(alo.x, blo.x), fminf(alo.y, blo.y), fminf(alo.z, blo.z), 0.f);
        float4 hi = make_float4(fmaxf(ahi.x, bhi.x), fmaxf(ahi.y, bhi.y), fmaxf(ahi.z, bhi.z), 0.f);
        uint32_t id = (uint32_t)nLeaves + node;
        children[node] = make_uint2(a, b);
        parent[a] = id; parent[b] = id;
        size[id] = size[a] + size[b];
        nodeLo[id] = lo; nodeHi[id] = hi;
        cidOut[pos] = id; cLoOut[pos] = lo; cHiOut[pos] = hi;
      } else {
        cidOut[pos] = cidIn[i]; cLoOut[pos] = cLoIn[i]; cHiOut[pos] = cHiIn[i];
      }
    }
    off += f[k];
  }
}

// All remaining iterations once at most PL_TAIL clusters are left: one block, clusters in shared
// memory, no host round trips.  Same merge rule and the same scan-based node numbering as the
// multi-kernel iterations above.
__global__ void __launch_bounds__(PL_TAIL)
k_ploc_tail(int n, int nLeaves, int radius, uint32_t nodeBase, const uint32_t* __restrict__ cidIn, const float4* __restrict__ cLoIn,
            const float4* __restrict__ cHiIn, float4* __restrict__ nodeLo, float4* __restrict__ nodeHi, uint2* __restrict__ children,
            uint32_t* __restrict__ parent, uint32_t* __restrict__ size, uint32_t* __restrict__ nodesCreated) {
  __shared__ float4 sLo[PL_TAIL], sHi[PL_TAIL];
  __shared__ uint32_t sId[PL_TAIL];
  __shared__ int sNn[PL_TAIL];
  __shared__ uint32_t sWarp[32][2];
  const int i = threadIdx.x, lane = i & 31, warp = i >> 5;
  if (i < n) { sId[i] = cidIn[i]; sLo[i] = cLoIn[i]; sHi[i] = cHiIn[i]; }
  __syncthreads();
  while (n > 1) {
    float4 lo = make_float4(0, 0, 0, 0), hi = lo;
    int best = -1;
    if (i < n) {
      lo = sLo[i]; hi = sHi[i];
      float bestA = __int_as_float(0x7f800000);
      for (int o = -radius; o <= radius; ++o) {
        int j = i + o;
        if (o == 0 || j < 0 || j >= n) continue;
        float a = mergedArea(lo, hi, sLo[j], sHi[j]);
        if (a < bestA) { bestA = a; best = j; }
      }
      sNn[i] = best;
    }
    __syncthreads();
    bool mutual = i < n && best >= 0 && sNn[best] == i;
    bool merged = mutual && i < best, removed = mutual && i > best;
    uint32_t valid = (i < n && !removed) ? 1u : 0u, mrg = merged ? 1u : 0u;
    uint32_t myId = i < n ? sId[i] : 0u, otherId = merged ? sId[best] : 0u;
    float4 olo = lo, ohi = hi;
    if (merged) { olo = sLo[best]; ohi = sHi[best]; }
    // block-wide exclusive scans of `valid` and `mrg`
    uint32_t iv = valid, im = mrg;
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t tv = __shfl_up_sync(0xffffffffu, iv, o), tm = __shfl_up_sync(0xffffffffu, im, o);
      if (lane >= o) { iv += tv; im += tm; }
    }
    if (lane == 31) { sWarp[warp][0] = iv; sWarp[warp][1] = im; }
    __syncthreads();
    uint32_t offV = 0, offM = 0, totV = 0, totM = 0;
    for (int w = 0; w < PL_TAIL / 32; ++w) {
      if (w < warp) { offV += sWarp[w][0]; offM += sWarp[w][1]; }
      totV += sWarp[w][0]; totM += sWarp[w][1];
    }
    uint32_t pos = offV + iv - valid, mpos = offM + im - mrg;
    __syncthreads();  // everyone has read its inputs from shared memory
    if (valid) {
      if (merged) {
        uint32_t node = nodeBase + mpos, id = (uint32_t)nLeaves + node;
        float4 nlo = make_float4(fminf(lo.x, olo.x), fminf(lo.y, olo.y), fminf(lo.z, olo.z), 0.f);
        float4 nhi = make_float4(fmaxf(hi.x, ohi.x), fmaxf(hi.y, ohi.y), fmaxf(hi.z, ohi.z), 0.f);
        children[node] = make_uint2(myId, otherId);
        parent[myId] = id; parent[otherId] = id;
        size[id] = size[myId] + size[otherId];
        nodeLo[id] = nlo; nodeHi[id] = nhi;
        sId[pos] = id; sLo[pos] = nlo; sHi[pos] = nhi;
      } else {
        sId[pos] = myId; sLo[pos] = lo; sHi[pos] = hi;
      }
    }
    nodeBase += totM;
    n = (int)totV;
    __syncthreads();
  }
  if (i == 0) *nodesCreated = nodeBase;
}

// Position of the leftmost leaf of `node` in depth-first (leaf) order: walking up, every time we
// are a right child the left sibling's whole subtree precedes us.
__device__ __forceinline__ uint32_t leftmostPos(uint32_t node, uint32_t root, int nLeaves, const uint32_t* __restrict__ parent,
                                                const uint2* __restrict__ children, const uint32_t* __restrict__ size,
                                                uint32_t* depthOut = nullptr) {
  uint32_t pos = 0, depth = 0;
  while (node != root) {
    uint32_t p = parent[node];
    uint2 ch = children[p - nLeaves];
    if (ch.y == node) pos += size[ch.x];
    node = p;
    ++depth;
  }
  if (depthOut) *depthOut = depth;
  return pos;
}

__global__ void k_ploc_leaf_order(int nLeaves, uint32_t root, const uint32_t* __restrict__ parent, const uint2* __restrict__ children,
                                  const uint32_t* __restrict__ size, const uint32_t* __restrict__ sortedIds,
                                  uint32_t* __restrict__ leafPos, uint32_t* __restrict__ orderedIds, uint32_t* __restrict__ firstPos,
                                  uint32_t* __restrict__ maxDepth) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t depth = 0;
  if (i < nLeaves) {
    uint32_t pos = leftmostPos((uint32_t)i, root, nLeaves, parent, children, size, &depth);
    leafPos[i] = pos;
    orderedIds[pos] = sortedIds[i];
    // this leaf is the leftmost one of every ancestor it reaches through left links only: each inner node gets the
    // position of its first primitive from exactly one leaf, and nobody walks to the root for it again
    for (uint32_t node = (uint32_t)i; node != root;) {
      const uint32_t p = parent[node];
      if (children[p - nLeaves].x != node) break;
      firstPos[p - nLeaves] = pos;
      node = p;
    }
  }
  for (int o = 16; o > 0; o >>= 1) depth = max(depth, __shfl_xor_sync(0xffffffffu, depth, o));
  if ((threadIdx.x & 31) == 0 && depth) atomicMax(maxDepth, depth);
}

// Aila–Laine nodes; inner node k (creation order) is written at nInner-1-k so the root is node 0
// and the top of the tree is contiguous.  Subtrees of <= MOX_LEAF_MAX prims fold into one leaf.
__global__ void k_ploc_emit(int nLeaves, int nInner, uint32_t root, const uint32_t* __restrict__ parent,
                            const uint2* __restrict__ children, const uint32_t* __restrict__ size,
                            const uint32_t* __restrict__ leafPos, const uint32_t* __restrict__ firstPos, const float4* __restrict__ nodeLo,
                            const float4* __restrict__ nodeHi, BvhNode2* __restrict__ out) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nInner) return;
  uint2 ch = children[k];
  uint32_t c[2] = {ch.x, ch.y};
  int ref[2];
  float4 lo[2], hi[2];
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    lo[s] = nodeLo[c[s]]; hi[s] = nodeHi[c[s]];
    if (c[s] < (uint32_t)nLeaves) {
      ref[s] = ~((int)(leafPos[c[s]] << 3) | 0);
    } else {
      uint32_t cnt = size[c[s]];
      if (cnt <= MOX_LEAF_MAX) {
        uint32_t first = firstPos[c[s] - nLeaves];
        ref[s] = ~((int)(first << 3) | (int)(cnt - 1));
      } else {
        ref[s] = nInner - 1 - (int)(c[s] - nLeaves);
      }
    }
  }
  BvhNode2 nd;
  nd.c0xy = make_float4(lo[0].x, hi[0].x, lo[0].y, hi[0].y);
  nd.c1xy = make_float4(lo[1].x, hi[1].x, lo[1].y, hi[1].y);
  nd.cz = make_float4(lo[0].z, hi[0].z, lo[1].z, hi[1].z);
  nd.ref = make_int4(ref[0], ref[1], 0, 0);
  out[nInner - 1 - k] = nd;
}

// Refit of a finished tree: leaf i takes the box of sorted primitive i (as k_ploc_init), inner nodes are formed again
// bottom-up; the second child to arrive at a node (per-node arrival counters, as k_refit) writes it.  The union takes
// the same operands in the same order as k_ploc_merge / k_ploc_tail (children.x first), so unchanged boxes give the
// same bits, signed zeros included.
__global__ void k_ploc_refit(int nLeaves, uint32_t root, const uint32_t* __restrict__ sortedIds, const float4* __restrict__ primLo,
                             const float4* __restrict__ primHi, const uint2* __restrict__ children, const uint32_t* __restrict__ parent,
                             float4* __restrict__ nodeLo, float4* __restrict__ nodeHi, uint32_t* __restrict__ arrivals) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nLeaves) return;
  const uint32_t id = sortedIds[i];
  __stcg(&nodeLo[i], primLo[id]);
  __stcg(&nodeHi[i], primHi[id]);
  __threadfence();
  for (uint32_t node = (uint32_t)i; node != root;) {
    const uint32_t p = parent[node];
    if (atomicAdd(&arrivals[p - nLeaves], 1u) == 0u) return;  // the sibling subtree is not finished yet
    const uint2 ch = children[p - nLeaves];
    const float4 alo = __ldcg(&nodeLo[ch.x]), ahi = __ldcg(&nodeHi[ch.x]), blo = __ldcg(&nodeLo[ch.y]), bhi = __ldcg(&nodeHi[ch.y]);
    __stcg(&nodeLo[p], make_float4(fminf(alo.x, blo.x), fminf(alo.y, blo.y), fminf(alo.z, blo.z), 0.f));
    __stcg(&nodeHi[p], make_float4(fmaxf(ahi.x, bhi.x), fmaxf(ahi.y, bhi.y), fmaxf(ahi.z, bhi.z), 0.f));
    __threadfence();
    node = p;
  }
}

inline int divUp(size_t a, size_t b) { return (int)((a + b - 1) / b); }

}  // namespace

// On a CUDA error: describe it in err and return `failed`.
#define PCK(x, failed) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { err = std::string(#x) + ": " + cudaGetErrorString(e_); return failed; } } while (0)

size_t plocScratchBytes(int n) {
  const size_t nn = (size_t)std::max(n, 2);
  // 2 cid + nn + parent(2) + size(2) + leafPos + orderedIds + firstPos = 10 words, 4 cluster boxes + 2x2 node boxes = 8 float4,
  // children 8 B, tile sums; plus alignment slack for 16 slices
  return nn * (10 * 4 + 8 * 16 + 8) + (size_t)(divUp(nn, PL_TILE) + 2) * 8 + (size_t)(PL_MAX_ITERS + 1) * sizeof(PlocState) + 17 * 256;
}

bool plocAlloc(PlocScratch& s, int n, DeviceArena& a, std::string& err) {
  const size_t nn = (size_t)std::max(n, 2);
  s.cid[0] = a.take<uint32_t>(nn); s.cid[1] = a.take<uint32_t>(nn);
  s.cLo[0] = a.take<float4>(nn); s.cLo[1] = a.take<float4>(nn);
  s.cHi[0] = a.take<float4>(nn); s.cHi[1] = a.take<float4>(nn);
  s.nn = a.take<uint32_t>(nn);
  s.nodeLo = a.take<float4>(2 * nn); s.nodeHi = a.take<float4>(2 * nn);
  s.children = a.take<uint2>(nn);
  s.parent = a.take<uint32_t>(2 * nn); s.size = a.take<uint32_t>(2 * nn);
  s.leafPos = a.take<uint32_t>(nn); s.orderedIds = a.take<uint32_t>(nn); s.firstPos = a.take<uint32_t>(nn);
  s.tileSums = a.take<unsigned long long>((size_t)divUp(nn, PL_TILE) + 2);
  s.state = a.take<PlocState>(PL_MAX_ITERS + 1);
  s.hostTotal = a.pinned;
  if (!s.tileSums || !s.state || !s.firstPos || !s.hostTotal) { err = "PLOC scratch does not fit the build arena"; return false; }
  return true;
}

// n >= 2 valid primitives in Morton order (sortedIds); primLo/primHi indexed by primitive id.
// Writes n-1 nodes to outNodes (root = node 0) and the leaf-ordered ids to s.orderedIds.
PlocResult plocBuild(PlocScratch& s, int n, const uint32_t* sortedIds, const float4* primLo, const float4* primHi, int radius,
                     BvhNode2* outNodes, float rootLo[3], float rootHi[3], int* maxDepthOut, cudaStream_t stream, std::string& err) {
  radius = std::max(1, std::min(radius, PL_MAX_RADIUS));
  const int B = 256;
  k_ploc_init<<<divUp(n, B), B, 0, stream>>>(n, sortedIds, primLo, primHi, s.cid[0], s.cLo[0], s.cHi[0], s.nodeLo, s.nodeHi, s.size);
  int cur = 0, count = n;
  uint32_t nodeBase = 0;
  unsigned long long* dTotal = s.tileSums + divUp((size_t)std::max(n, 2), PL_TILE);
  PlocState* st = s.state;
  PlocState* hostState = (PlocState*)s.hostTotal;   // 16 bytes of pinned memory
  {
    PlocState s0{n, 0u, 0u, 0u};
    *hostState = s0;
    PCK(cudaMemcpyAsync(st, hostState, sizeof s0, cudaMemcpyHostToDevice, stream), PlocResult::ERROR);
  }
  int it = 0;
  while (count > PL_TAIL) {
    // Out of state slots.  Many primitives with the same box get here: equal merged areas tie towards the smaller
    // index, so each iteration merges a single pair of them.
    if (it + PL_BATCH >= PL_MAX_ITERS) return PlocResult::NOT_CONVERGED;
    // PL_BATCH iterations on the device's own counts; grids cover `count`, the last value the host has seen
    const int nTiles = divUp(count, PL_TILE);
    for (int b = 0; b < PL_BATCH; ++b, ++it) {
      const int c = it & 1;
      k_ploc_nn<<<divUp(count, PL_THREADS), PL_THREADS, 0, stream>>>(st + it, radius, s.cLo[c], s.cHi[c], s.nn);
      k_ploc_tile_sums<<<nTiles, PL_THREADS, 0, stream>>>(st + it, s.nn, s.tileSums);
      k_ploc_merge<<<nTiles, PL_THREADS, 0, stream>>>(st + it, n, s.nn, s.tileSums, s.cid[c], s.cLo[c], s.cHi[c],
                                                       s.cid[c ^ 1], s.cLo[c ^ 1], s.cHi[c ^ 1], s.nodeLo, s.nodeHi, s.children,
                                                       s.parent, s.size);
    }
    PCK(cudaMemcpyAsync(hostState, st + it, sizeof(PlocState), cudaMemcpyDeviceToHost, stream), PlocResult::ERROR);
    PCK(cudaStreamSynchronize(stream), PlocResult::ERROR);
    const PlocState got = *hostState;
    if (got.count >= count || got.count < 1 || (int)got.nodeBase != n - got.count) { err = "PLOC made no progress"; return PlocResult::ERROR; }
    count = got.count;
    nodeBase = got.nodeBase;
    cur = (int)(got.iters & 1u);   // iterations that ran (the no-op ones at the end of a batch do not swap buffers)
  }
  if (count > 1) {
    uint32_t* dCreated = (uint32_t*)(dTotal + 1) + 1;
    k_ploc_tail<<<1, PL_TAIL, 0, stream>>>(count, n, radius, nodeBase, s.cid[cur], s.cLo[cur], s.cHi[cur], s.nodeLo, s.nodeHi, s.children,
                                           s.parent, s.size, dCreated);
    uint32_t created = 0;
    PCK(cudaMemcpyAsync(&created, dCreated, 4, cudaMemcpyDeviceToHost, stream), PlocResult::ERROR);
    PCK(cudaStreamSynchronize(stream), PlocResult::ERROR);
    nodeBase = created;
  }
  const int nInner = n - 1;
  if ((int)nodeBase != nInner) { err = "PLOC node count mismatch"; return PlocResult::ERROR; }
  const uint32_t root = (uint32_t)(n + nInner - 1);
  uint32_t* dDepth = (uint32_t*)(dTotal + 1);
  PCK(cudaMemsetAsync(dDepth, 0, 4, stream), PlocResult::ERROR);
  k_ploc_leaf_order<<<divUp(n, B), B, 0, stream>>>(n, root, s.parent, s.children, s.size, sortedIds, s.leafPos, s.orderedIds, s.firstPos, dDepth);
  k_ploc_emit<<<divUp(nInner, B), B, 0, stream>>>(n, nInner, root, s.parent, s.children, s.size, s.leafPos, s.firstPos, s.nodeLo, s.nodeHi, outNodes);
  float4 lo, hi;
  PCK(cudaMemcpyAsync(&lo, s.nodeLo + root, 16, cudaMemcpyDeviceToHost, stream), PlocResult::ERROR);
  PCK(cudaMemcpyAsync(&hi, s.nodeHi + root, 16, cudaMemcpyDeviceToHost, stream), PlocResult::ERROR);
  uint32_t depth = 0;
  PCK(cudaMemcpyAsync(&depth, dDepth, 4, cudaMemcpyDeviceToHost, stream), PlocResult::ERROR);
  PCK(cudaStreamSynchronize(stream), PlocResult::ERROR);
  PCK(cudaGetLastError(), PlocResult::ERROR);
  *maxDepthOut = (int)depth;
  rootLo[0] = lo.x; rootLo[1] = lo.y; rootLo[2] = lo.z;
  rootHi[0] = hi.x; rootHi[1] = hi.y; rootHi[2] = hi.z;
  return PlocResult::OK;
}

bool plocRefit(const PlocScratch& s, int n, const uint32_t* sortedIds, const float4* primLo, const float4* primHi, uint32_t* arrivals,
               BvhNode2* outNodes, cudaStream_t stream, std::string& err) {
  const int B = 256, nInner = n - 1;
  const uint32_t root = (uint32_t)(n + nInner - 1);
  PCK(cudaMemsetAsync(arrivals, 0, (size_t)nInner * 4, stream), false);
  k_ploc_refit<<<divUp(n, B), B, 0, stream>>>(n, root, sortedIds, primLo, primHi, s.children, s.parent, s.nodeLo, s.nodeHi, arrivals);
  k_ploc_emit<<<divUp(nInner, B), B, 0, stream>>>(n, nInner, root, s.parent, s.children, s.size, s.leafPos, s.firstPos, s.nodeLo, s.nodeHi, outNodes);
  return true;
}
