// build.h — interface between the C ABI layer and the BVH builder.
#pragma once
#include <cstring>
#include <string>
#include <algorithm>
#include "gpu_types.h"

// Grow-only device scratch shared by successive builds (per-frame rebuilds of an animated scene
// must not pay ~25 cudaMalloc/cudaFree pairs).  take() hands out 256-byte aligned slices.
struct DeviceArena {
  char* base = nullptr;
  size_t cap = 0, off = 0;
  unsigned long long* pinned = nullptr;  // 64 bytes of pinned host memory for small read-backs
  bool reserve(size_t bytes) {
    off = 0;
    if (bytes <= cap) return true;
    if (base) cudaFree(base);
    base = nullptr; cap = 0;
    if (cudaMalloc(&base, bytes) != cudaSuccess) return false;
    cap = bytes;
    return true;
  }
  template <class T> T* take(size_t count) {
    size_t bytes = (count * sizeof(T) + 255) & ~(size_t)255;
    if (off + bytes > cap) return nullptr;
    T* p = (T*)(base + off);
    off += bytes;
    return p;
  }
  void release() { if (base) cudaFree(base); if (pinned) cudaFreeHost(pinned); base = nullptr; pinned = nullptr; cap = off = 0; }
};

struct BuildInput {
  int nPrims = 0;
  const PrimDesc* prims = nullptr;     // device
  const TriIdx* tris = nullptr;        // device
  const float* verts = nullptr;        // device
  const Analytic* analytic = nullptr;  // device
  const GpuMaterial* mats = nullptr;   // device: the packed records carry each primitive's shadow-ray class
  cudaEvent_t evStart = nullptr, evStop = nullptr;  // recorded around the build kernels when set
  DeviceArena* arena = nullptr;  // required
  bool usePloc = true;   // false: Karras radix tree (fastest build, lower quality)
  int plocRadius = 0;    // 0 = automatic: 32 up to 2 M primitives, 16 above.  Bench scene (1 M): 8 -> 1152, 16 -> 1234, 32 -> 1247,
                         // 48 -> 1213, 64 -> 1219, 100 -> 1248 Mrays/s, build 3.5 -> 3.8 ms (16 -> 32); 10 M soup: 16 -> 13.2 ms and
                         // 652..856 Mrays/s, 32 -> 15.2 ms and 628..832
  bool useWide = true;   // collapse the PLOC tree into the compressed 8-wide BVH
  bool watertight = false;  // packed triangle records hold the raw vertices (p0, p1, p2) for the watertight test
};

// Scratch of the PLOC hierarchy builder (ploc.cu), allocated before the timed build.
struct PlocState;
struct PlocScratch {
  uint32_t* cid[2] = {nullptr, nullptr};
  float4 *cLo[2] = {nullptr, nullptr}, *cHi[2] = {nullptr, nullptr};
  uint32_t* nn = nullptr;
  float4 *nodeLo = nullptr, *nodeHi = nullptr;
  uint2* children = nullptr;
  uint32_t *parent = nullptr, *size = nullptr, *leafPos = nullptr, *orderedIds = nullptr;
  uint32_t* firstPos = nullptr;   // per inner node (id - nLeaves): leaf-order position of its leftmost leaf
  unsigned long long* tileSums = nullptr;
  PlocState* state = nullptr;               // loop state, one slot per iteration (ploc.cu)
  unsigned long long* hostTotal = nullptr;  // pinned
};
size_t plocScratchBytes(int n);
bool plocAlloc(PlocScratch& s, int n, DeviceArena& arena, std::string& err);
// NOT_CONVERGED: the clustering ran out of iterations before one cluster was left (many primitives with the same box
// merge one pair per iteration); the caller builds another hierarchy.  ERROR: a CUDA error or an inconsistent state,
// described in err.
enum class PlocResult { OK, NOT_CONVERGED, ERROR };
PlocResult plocBuild(PlocScratch& s, int n, const uint32_t* sortedIds, const float4* primLo, const float4* primHi, int radius,
                     BvhNode2* outNodes, float rootLo[3], float rootHi[3], int* maxDepthOut, cudaStream_t stream, std::string& err);

// What an in-place refit (refitBvh) needs from the last full build.  Every pointer is a slice of the build's
// DeviceArena.  Nothing takes from the arena between two full builds, so the slices stay valid until the next
// buildBvh, which overwrites them.  A refit keeps the topology (Morton order, tree, leaf orders, wide-node slots) and
// recomputes the boxes only.
struct RefitState {
  enum Path { NONE = 0, TRIVIAL, PLOC, KARRAS };
  Path path = NONE;          // TRIVIAL: at most one valid primitive, no hierarchy to refit (the caller rebuilds)
  bool wide = false;         // the compressed 8-wide BVH was built from the PLOC tree
  int nPrims = 0, nValid = 0, nNodes8 = 0;
  float4 *primLo = nullptr, *primHi = nullptr;  // per primitive id, validity in primLo .w (1 / 0)
  uint32_t* sortedIds = nullptr;                // primitive ids in Morton order, the valid ones first
  uint32_t* flag = nullptr;                     // device word, set by the refit when a primitive's validity changed
  PlocScratch ploc;                             // PLOC: children, parent, size, leafPos, firstPos, orderedIds, node boxes
  int2 *children = nullptr, *range = nullptr;   // Karras radix tree ...
  int *parentInternal = nullptr, *parentLeaf = nullptr;
  float4 *nodeLo = nullptr, *nodeHi = nullptr;
  uint32_t* arrivals = nullptr;                 // nValid - 1 counters (both binary refits)
  uint32_t* orderedIds8 = nullptr;              // wide: primitives in wide-leaf order
  uint32_t* wideSrc = nullptr;                  // wide: per node its binary node and the binary node of each slot (~0u: empty)
};

struct BuildOutput {
  // device, owned by the caller.  On entry they may hold buffers of nodesCap / packedCap records from a
  // previous build, which are reused when large enough.
  BvhNode2* nodes = nullptr;
  int nNodes = 0;
  float4* packed = nullptr;   // 3 float4 per valid primitive in leaf order
  size_t nodesCap = 0, packedCap = 0;
  BvhNode8* nodes8 = nullptr;  // compressed wide BVH (only when built from PLOC); same reuse rule
  float4* packed8 = nullptr;   // primitives in wide-leaf order
  size_t nodes8Cap = 0, packed8Cap = 0;
  int nNodes8 = 0, wideLevels = 0;
  int nValid = 0, nInvalid = 0;
  int iterations = 0;
  bool usedPloc = false;  // false: Karras radix tree (requested, or PLOC fallback because of depth)
  int maxDepth = 0;   // deepest leaf (PLOC); the traversal stack holds MOX_STACK entries
  float sceneLo[3] = {0, 0, 0}, sceneHi[3] = {0, 0, 0};
  float4 *scratchLo = nullptr, *scratchHi = nullptr;  // builder-internal
  RefitState refit;   // what the build left for refitBvh
};

bool buildBvh(const BuildInput& in, BuildOutput& out, cudaStream_t stream, std::string& err);
// Refit of the structure out.refit describes (path PLOC or KARRAS), in place, from the current primitive data of
// `in`: new primitive boxes, binary nodes, wide nodes and packed records, with the last build's topology.  Unchanged
// geometry gives byte-identical nodes and records.  in.evStart / in.evStop are recorded around the kernels.
// *validityChanged: a primitive became valid or invalid since the build; the result is then unusable.
bool refitBvh(const BuildInput& in, BuildOutput& out, cudaStream_t stream, std::string& err, bool* validityChanged);
bool radixSortPairs(uint32_t* keys, uint32_t* vals, int n, cudaStream_t stream, std::string& err);
// Marks the entries of the terminal query's light list (n <= MOX_TERMINAL_LIGHTS_MAX, traverse_job.h) whose primitive
// the last full build left out (rs.primLo .w == 0).  A refit keeps every primitive's validity, so the list stays.
void excludeUnbuiltLights(uint4* list, int n, const RefitState& rs, cudaStream_t stream);

// Refit of a PLOC tree built by plocBuild over n leaves: new leaf and inner boxes in s.nodeLo / s.nodeHi, then the
// binary nodes again.  arrivals: n - 1 words of scratch.
bool plocRefit(const PlocScratch& s, int n, const uint32_t* sortedIds, const float4* primLo, const float4* primHi, uint32_t* arrivals,
               BvhNode2* outNodes, cudaStream_t stream, std::string& err);

// Collapse of the PLOC tree into the compressed wide BVH (bvh_wide.cu).  *wideSrcOut: 9 words per wide node (its
// binary node, then the binary node in each slot or ~0u), what wideRefit needs.
size_t wideScratchBytes(int n);
bool wideCollapse(const PlocScratch& s, int n, uint32_t root, DeviceArena& arena, BvhNode8* outNodes, uint32_t** orderedIds8Out,
                  uint32_t** wideSrcOut, int* nNodesOut, int* levelsOut, cudaStream_t stream, std::string& err);
// New boxes for the nNodes wide nodes from the refitted binary boxes; slots, masks and bases stay.
void wideRefit(const uint32_t* wideSrc, int nNodes, const float4* nodeLo, const float4* nodeHi, BvhNode8* nodes, cudaStream_t stream);
