// capi.cu — implementation of the C ABI in include/mox.h: context, scene staging and upload,
// acceleration build, the spp loop, accumulation read-back, multi-GPU pack/unpack, raw ray
// queries.  Host-side counterpart of what MinimalOptiX::setupContext / setupScene /
// renderScene do through optixpp (MinimalOptiX.cpp:130-152, 154-538, 540-560).
//
// There is no CPU path in this library: every compute entry point needs a usable sm_100 GPU.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "build.h"
#include "denoise.h"
#include "group.h"
#include "mox.h"
#include "mox_debug.h"
#include "rng.cuh"
#include "wavefront.h"

namespace {
std::string g_createError;

enum Stage { ST_GENERATE = 0, ST_EXTEND, ST_SHADE, ST_SHADOW, ST_ACCUMULATE, ST_COUNT };

// Event pairs around the kernels of each stage; summed after the batch's final synchronize.
struct StageTimer {
  std::vector<cudaEvent_t> pool;
  struct Span { int stage; size_t e0, e1; uint32_t depth; };
  std::vector<Span> spans;
  size_t used = 0;
  size_t grab(cudaStream_t s) {
    if (used == pool.size()) { cudaEvent_t e; cudaEventCreate(&e); pool.push_back(e); }
    cudaEventRecord(pool[used], s);
    return used++;
  }
  void begin(int stage, cudaStream_t s, uint32_t depth = 0) { spans.push_back({stage, grab(s), 0, depth}); }
  void end(cudaStream_t s) { spans.back().e1 = grab(s); }
  // Adds the spans into the per-stage times, and the two traversal launches into the per-depth times.
  void collect(mox_stats& st) {
    double* ms[ST_COUNT] = {&st.ms_generate, &st.ms_extend, &st.ms_shade, &st.ms_shadow, &st.ms_accumulate};
    for (auto& sp : spans) {
      float t = 0;
      if (cudaEventElapsedTime(&t, pool[sp.e0], pool[sp.e1]) != cudaSuccess) continue;
      *ms[sp.stage] += t;
      if (sp.depth) {
        double* byDepth = sp.stage == ST_SHADOW ? st.ms_shadow_depth : st.ms_extend_depth;
        byDepth[sp.depth < MOX_STATS_DEPTHS ? sp.depth : MOX_STATS_DEPTHS - 1] += t;
      }
    }
    spans.clear(); used = 0;
  }
  ~StageTimer() { for (auto e : pool) cudaEventDestroy(e); }
};

// Device (cudaMalloc) or pinned host (cudaMallocHost) memory: move-only, freed by its owner.  An empty one makes no
// CUDA call, so the shell of a multi-GPU handle, which never binds a device, frees nothing.
template <class T, bool HOST>
struct OwnedMem {
  T* p = nullptr;
  size_t bytes = 0;
  OwnedMem() = default;
  OwnedMem(OwnedMem&& o) noexcept : p(std::exchange(o.p, nullptr)), bytes(std::exchange(o.bytes, 0)) {}
  OwnedMem& operator=(OwnedMem&& o) noexcept {
    if (this != &o) { release(); p = std::exchange(o.p, nullptr); bytes = std::exchange(o.bytes, 0); }
    return *this;
  }
  ~OwnedMem() { release(); }
  void release() {
    if (p) { if (HOST) cudaFreeHost((void*)p); else cudaFree((void*)p); }
    p = nullptr; bytes = 0;
  }
  // Replaces the contents by n uninitialised bytes; empty on failure.
  cudaError_t alloc(size_t n) {
    release();
    void* q = nullptr;
    const cudaError_t e = HOST ? cudaMallocHost(&q, n) : cudaMalloc(&q, n);
    if (e == cudaSuccess) { p = (T*)q; bytes = n; }
    return e;
  }
};
using DevBuf = OwnedMem<void, false>;
template <class T> using DevArray = OwnedMem<T, false>;
template <class T> using PinnedBuf = OwnedMem<T, true>;

// A gather buffer: allocated here, opened from another process's export over CUDA IPC, or borrowed from another
// context of this process, which frees it.
struct GatherBuf {
  enum Kind { own, ipc, borrowed };
  float* p = nullptr;
  Kind kind = own;
  GatherBuf() = default;
  GatherBuf(const GatherBuf&) = delete;
  GatherBuf& operator=(const GatherBuf&) = delete;
  ~GatherBuf() { release(); }
  void release() {
    if (p && kind == ipc) cudaIpcCloseMemHandle(p);
    else if (p && kind == own) cudaFree(p);
    p = nullptr; kind = own;
  }
};

constexpr size_t kCounterWords = C_WORDS + BOUNCE_RING * C_BOUNCE_WORDS;

// The layout of the wavefront state in one device block at `base` (null: sizes only): rays, hit, throughput,
// radiance, RNG state, two queue buffers, four material queues and the second Disney queue; per light a direction,
// a contribution and a queue entry, and one shadow origin per path when there are lights; the counters and the
// launch seeds.  Every array starts 256-byte aligned, and one of 2 MiB or more on a 2 MiB boundary, where cudaMalloc
// puts it: packed at 256 bytes, the path arrays measured 0.15 % slower.  Returns the block's size.
size_t pathLayout(size_t paths, size_t nLights, size_t nSeeds, char* base, PathBuffers& pb) {
  pb = PathBuffers();
  size_t off = 0;
  auto take = [&](auto*& a, size_t bytes) {
    const size_t align = bytes >= (2u << 20) ? (2u << 20) : 256;
    off = (off + align - 1) & ~(align - 1);
    a = base ? (std::remove_reference_t<decltype(a)>)(base + off) : nullptr;
    off += bytes;
  };
  const size_t slots = paths * nLights;
  take(pb.rayO, paths * 16); take(pb.rayD, paths * 16); take(pb.hit, paths * 8); take(pb.thr, paths * 16);
  take(pb.rad, paths * 16); take(pb.state, paths * 4);
  for (auto& q : pb.qBuf) take(q, paths * 4);
  for (auto& q : pb.qMat) take(q, paths * 4);
  take(pb.qDisneyAlt, paths * 4);
  if (slots) { take(pb.shO, paths * 16); take(pb.shD, slots * 16); take(pb.shC, slots * 16); take(pb.shQueue, slots * 4); }
  take(pb.counters, kCounterWords * 4);
  take(pb.seeds, nSeeds * 4);
  pb.capacity = paths; pb.shadowSlots = slots; pb.seedCap = nSeeds;
  return off;
}

inline uint64_t counter64(const uint32_t* words, int lo) { return ((uint64_t)words[lo + 1] << 32) | words[lo]; }
}  // namespace

struct mox_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::string err;

  RenderParams rp{};
  bool haveGlobals = false, haveCamera = false;
  uint32_t rank = 0, world = 1, tile = 32;

  // host staging of the scene (copied at add_* time)
  std::vector<PrimDesc> prims;
  std::vector<TriIdx> tris;
  std::vector<float> verts, normals, uvs;
  std::vector<Analytic> analytic;
  std::vector<GpuMaterial> mats;
  std::vector<LightParams> lights;
  std::vector<float4> lightN;   // normalize(light.normal) per light, computed once with the device's operation sequence (vec.cuh)
  struct HostTexture { int w, h; std::vector<float> texels; };
  std::vector<HostTexture> textures;
  std::vector<cudaArray_t> texArrays;
  std::vector<cudaTextureObject_t> texObjects;
  bool texturesDirty = false;
  uint32_t nSpheres = 0, nQuads = 0;
  // One record per mox_add_mesh: its primitives, and its vertices / normals in verts / normals (in vertices, not floats).
  struct MeshRec { uint32_t firstPrim, nFaces; size_t vBase, nV, nBase, nN; };
  std::vector<MeshRec> meshes;
  // Float ranges of verts / normals changed by mox_update_mesh since the last upload: [lo, hi), empty when lo >= hi.
  size_t vDirtyLo = SIZE_MAX, vDirtyHi = 0, nDirtyLo = SIZE_MAX, nDirtyHi = 0;

  // device scene
  DevBuf dPrims, dTris, dVerts, dNormals, dUvs, dAnalytic, dMats, dLights, dLightN, dShadeRec;
  bool shadeRecBuilt = false;
  DevBuf dQueryO, dQueryD, dQueryCounters;  // raw ray queries
  DevBuf dQueryRays, dQueryOut, dQueryC;    // ... and their host-buffer forms: grow-only staging, no allocation per call
  DevBuf dTexObjs;
  BuildOutput accel;   // its four node and record arrays belong to the context (freed in ~mox_ctx)
  bool wideBuilt = false, useWide = true;
  DeviceArena buildArena;
  bool built = false, lightsDirty = true;
  uint32_t accelFlags = 0;
  // The last full build succeeded and no primitive was added or removed since: MOX_ACCEL_REFIT may reuse its topology
  // (accel.refit).
  bool refitOk = false;
  // Light primitives of the terminal query (traverse_job.h), from the last full build; nTerminalLights < 0: the scene
  // has a triangle-mesh light or more than MOX_TERMINAL_LIGHTS_MAX lights, and the terminal bounce runs closest hit.
  DevBuf dTerminalLights;
  int nTerminalLights = -1;

  // image
  DevArray<float> dAccu;
  uint32_t accuW = 0, accuH = 0;
  DevArray<uint32_t> dOwned;
  uint32_t nOwned = 0;
  bool ownedDirty = true;
  std::vector<DevBuf> otherOwned;  // cached owned lists of other ranks (unpack)
  std::vector<uint64_t> ownedCount; // cached |owned pixels| per rank of the current partition

  // Wavefront buffers, streams and events of renderBatch.  The shadow rays of a bounce run on their own stream
  // (overlapShadow), so two persistent traversal launches are in flight while the host waits for a bounce's material
  // counts.  Splitting a batch into sub-batches on further streams measured no faster (1347 vs 1350 Mrays/s at full
  // frame, slower on an eighth of it) and was removed (DESIGN.md section 4; the code is in the git history).
  PathBuffers pb;      // views into pathBlock (pathLayout)
  DevBuf pathBlock;
  cudaStream_t shadowStream = nullptr;  // shadow traversal + k_apply of bounce b, overlapping extend + classify of bounce b+1
  cudaEvent_t evShaded = nullptr, evApplied = nullptr;
  cudaEvent_t evReady = nullptr;   // the counters of the bounce in flight have landed in hostCnt
  PinnedBuf<uint32_t> hostCnt;     // kCounterWords
  StageTimer timer;
  PinnedBuf<float> pinned;   // mox_map_accum's image

  // Gather / asynchronous read-back: two full-size device buffers (targets of the tile pushes, possibly of other
  // GPUs), two pinned host images, a copy stream.
  GatherBuf dGather[2];
  PinnedBuf<float> hostGather[2];
  size_t gatherBytes = 0;
  cudaStream_t copyStream = nullptr;
  cudaEvent_t evPushed = nullptr, evCopied[2] = {nullptr, nullptr};
  int readCur = 0;            // buffer the next mox_read_accum_begin uses
  int readPending = -1;       // buffer of the begin that has not been ended yet

  mox_group* group = nullptr; // set on the shell handle mox_create_multi returns

  // The counters and timings of mox_get_stats; the scene-derived fields are filled in there.  st.launches is also
  // mox_render's seed counter.
  mox_stats st{};
  size_t maxBatchPaths = 32u << 20;  // paths per wavefront (264 B each with 4 lights, pathLayout); measured 4 Mi -> 947, 32 Mi -> 980 Mrays/s at 4K
  bool overlapShadow = true;     // shadow rays of bounce b on a second stream, concurrent with the extend launch of bounce b+1 (MOX_OVERLAP_SHADOW=0: serial)
  bool brdfFast = true;          // approximate reciprocal / square root inside BRDF values (MOX_BRDF_IEEE=1: IEEE, the oracle's operations)
  bool terminalQuery = true;     // the bounce past rayMaxDepth uses the light list and an any-hit query (MOX_TERMINAL_CLOSEST=1: closest hit)

  // Adaptive sampling (mox_render_adaptive), allocated at its first call: per pixel the luminance sums, the sample
  // count and the launches sat out (pixelStats, 24 bytes per pixel in one block), and the two active-pixel lists with
  // the select kernels' tile sums and survivor word.
  DevBuf adaptiveStats, adaptiveLists;
  PixelStats pixelStats;
  PinnedBuf<uint32_t> hostSurvivors;

  // First-hit AOVs (mox_set_aovs): the sums in one block (aovLayout), allocated while aovOn and the image size is
  // known.  Grow-only scratch of mox_denoise: the filter's buffers and its output; on device 0 of a multi-GPU handle
  // also the frame the devices gather their inputs into (denoiseFrame: colour, skipped launches, AOV sums).
  bool aovOn = false;
  bool aovRecorded = false;   // a camera sample added its record since the sums were last zeroed
  DevBuf aovBlock;
  AovBuffers aov;
  DevBuf denoiseScratch, denoiseOut, denoiseFrame;

  // Frees what the context holds; the device buffers go with their owners.  mox_destroy binds the device and waits
  // for the streams first.
  ~mox_ctx() {
    freeTextures();
    for (void* a : {(void*)accel.nodes, (void*)accel.packed, (void*)accel.nodes8, (void*)accel.packed8})
      if (a) cudaFree(a);
    buildArena.release();
    for (cudaEvent_t e : {ev0, ev1, evShaded, evApplied, evReady, evPushed, evCopied[0], evCopied[1]})
      if (e) cudaEventDestroy(e);
    for (cudaStream_t s : {stream, shadowStream, copyStream})
      if (s) cudaStreamDestroy(s);
  }
  void freeTextures() {
    for (auto t : texObjects) cudaDestroyTextureObject(t);
    for (auto a : texArrays) cudaFreeArray(a);
    texObjects.clear(); texArrays.clear();
  }
};

namespace {

int fail(mox_ctx* c, int code, const std::string& msg) {
  if (c) c->err = msg; else g_createError = msg;
  return code;
}

#define CUCK(c, x)                                                                                    \
  do {                                                                                                \
    cudaError_t e_ = (x);                                                                             \
    if (e_ != cudaSuccess) return fail((c), e_ == cudaErrorMemoryAllocation ? MOX_ERR_OOM : MOX_ERR_CUDA, \
                                       std::string(#x) + ": " + cudaGetErrorString(e_));             \
  } while (0)

int bind(mox_ctx* c) {
  CUCK(c, cudaSetDevice(c->device));
  return MOX_OK;
}

// Grow-only: keeps b when it holds `bytes` already.
template <class T, bool HOST>
int ensure(mox_ctx* c, OwnedMem<T, HOST>& b, size_t bytes) {
  if (b.bytes >= bytes && b.p) return MOX_OK;
  CUCK(c, b.alloc(std::max<size_t>(bytes, 16)));
  return MOX_OK;
}

template <class T>
int upload(mox_ctx* c, DevBuf& b, const std::vector<T>& v) {
  int rc = ensure(c, b, v.size() * sizeof(T));
  if (rc) return rc;
  if (!v.empty()) CUCK(c, cudaMemcpyAsync(b.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, c->stream));
  return MOX_OK;
}

int addMaterial(mox_ctx* c, int kind, const void* params) {
  GpuMaterial m;
  memset(&m, 0, sizeof m);
  m.kind = kind;
  switch (kind) {
    case MOX_MAT_LAMBERTIAN: memcpy(&m.lam, params, sizeof(LambertianParams)); break;
    case MOX_MAT_METAL: memcpy(&m.met, params, sizeof(MetalParams)); break;
    case MOX_MAT_GLASS: memcpy(&m.gls, params, sizeof(GlassParams)); break;
    case MOX_MAT_DISNEY: memcpy(&m.dis, params, sizeof(DisneyParams)); break;
    case MOX_MAT_LIGHT: memcpy(&m.lgt, params, sizeof(LightParams)); break;
    default: return -1;
  }
  c->mats.push_back(m);
  return (int)c->mats.size() - 1;
}

void ownedList(uint32_t W, uint32_t H, uint32_t tile, uint32_t world, uint32_t rank, std::vector<uint32_t>& out) {
  out.clear();
  uint32_t tx = (W + tile - 1) / tile, ty = (H + tile - 1) / tile;
  for (uint32_t j = 0; j < ty; ++j)
    for (uint32_t i = 0; i < tx; ++i) {
      if ((i + j) % world != rank) continue;
      for (uint32_t y = j * tile; y < std::min(H, (j + 1) * tile); ++y)
        for (uint32_t x = i * tile; x < std::min(W, (i + 1) * tile); ++x) out.push_back(y * W + x);
    }
}

int refreshOwned(mox_ctx* c) {
  if (!c->ownedDirty) return MOX_OK;
  std::vector<uint32_t> l;
  ownedList(c->rp.W, c->rp.H, c->tile, c->world, c->rank, l);
  int rc = ensure(c, c->dOwned, l.size() * 4);
  if (rc) return rc;
  // Stream-ordered upload: a plain cudaMemcpy from pageable memory may return before the DMA has landed, and
  // the context stream is non-blocking, so a kernel launched next could still read stale bytes.
  if (!l.empty()) { CUCK(c, cudaMemcpyAsync(c->dOwned.p, l.data(), l.size() * 4, cudaMemcpyHostToDevice, c->stream)); CUCK(c, cudaStreamSynchronize(c->stream)); }
  c->nOwned = (uint32_t)l.size();
  c->otherOwned.clear();
  c->ownedCount.clear();
  c->ownedDirty = false;
  return MOX_OK;
}

// c->pathBlock already holds `paths` paths, nLights shadow slots per path and nSeeds launch seeds.
bool pathsFit(const mox_ctx* c, size_t paths, size_t nLights, size_t nSeeds) {
  const PathBuffers& pb = c->pb;
  return c->pathBlock.p && pb.capacity >= paths && pb.shadowSlots >= paths * nLights && pb.seedCap >= nSeeds;
}

// The wavefront state of `paths` paths, nLights shadow slots per path and nSeeds launch seeds in c->pathBlock.
int ensurePaths(mox_ctx* c, size_t paths, size_t nLights, size_t nSeeds) {
  if (pathsFit(c, paths, nLights, nSeeds)) return MOX_OK;
  PathBuffers& pb = c->pb;
  cudaStreamSynchronize(c->stream);
  // grow geometrically so that a slowly growing sample count does not reallocate on every call
  if (pb.capacity && paths > pb.capacity) paths = std::max(paths, pb.capacity + pb.capacity / 2);
  nSeeds = std::max(nSeeds, pb.seedCap);
  c->pathBlock.release();
  pb = PathBuffers();
  const size_t bytes = pathLayout(paths, nLights, nSeeds, nullptr, pb);
  CUCK(c, c->pathBlock.alloc(bytes));
  pathLayout(paths, nLights, nSeeds, (char*)c->pathBlock.p, pb);
  CUCK(c, cudaMemsetAsync(pb.counters, 0, kCounterWords * 4, c->stream));
  return MOX_OK;
}

SceneView sceneView(const mox_ctx* c) {
  SceneView s;
  s.nodes = c->accel.nodes;
  s.packed = c->accel.packed;
  s.nodes8 = (c->wideBuilt && c->useWide) ? c->accel.nodes8 : nullptr;
  s.packed8 = c->accel.packed8;
  s.analytic = (const Analytic*)c->dAnalytic.p;
  s.prims = (const PrimDesc*)c->dPrims.p;
  s.mats = (const GpuMaterial*)c->dMats.p;
  s.verts = (const float*)c->dVerts.p;
  s.normals = (const float*)c->dNormals.p;
  s.uvs = (const float*)c->dUvs.p;
  s.tris = (const TriIdx*)c->dTris.p;
  s.shadeRec = c->shadeRecBuilt ? (const float4*)c->dShadeRec.p : nullptr;
  s.lights = (const LightParams*)c->dLights.p;
  s.lightN = (const float4*)c->dLightN.p;
  s.textures = (const cudaTextureObject_t*)c->dTexObjs.p;
  s.nLights = (int)c->lights.size();
  s.nPrims = (int)c->prims.size();
  s.nNodes8 = (uint32_t)c->accel.nNodes8;
  s.watertight = (c->accelFlags & MOX_ACCEL_WATERTIGHT) ? 1 : 0;
  return s;
}

// createTextureSampler: REPEAT wrap, LINEAR filter, normalized coordinates, float4 texels
// (MinimalOptiX.cpp:449-474) -> CUDA texture objects; the hardware filter is used as in OptiX.
int syncTextures(mox_ctx* c) {
  if (!c->texturesDirty) return MOX_OK;
  cudaStreamSynchronize(c->stream);
  c->freeTextures();
  for (auto& t : c->textures) {
    cudaChannelFormatDesc fmt = cudaCreateChannelDesc<float4>();
    cudaArray_t arr = nullptr;
    CUCK(c, cudaMallocArray(&arr, &fmt, t.w, t.h));
    c->texArrays.push_back(arr);
    CUCK(c, cudaMemcpy2DToArrayAsync(arr, 0, 0, t.texels.data(), (size_t)t.w * 16, (size_t)t.w * 16, t.h, cudaMemcpyHostToDevice, c->stream));
    cudaResourceDesc res;
    memset(&res, 0, sizeof res);
    res.resType = cudaResourceTypeArray;
    res.res.array.array = arr;
    cudaTextureDesc td;
    memset(&td, 0, sizeof td);
    td.addressMode[0] = td.addressMode[1] = td.addressMode[2] = cudaAddressModeWrap;
    td.filterMode = cudaFilterModeLinear;
    td.readMode = cudaReadModeElementType;
    td.normalizedCoords = 1;
    cudaTextureObject_t obj = 0;
    CUCK(c, cudaCreateTextureObject(&obj, &res, &td, nullptr));
    c->texObjects.push_back(obj);
  }
  int rc = upload(c, c->dTexObjs, c->texObjects);
  if (rc) return rc;
  c->texturesDirty = false;
  return MOX_OK;
}

int syncLights(mox_ctx* c) {
  if (!c->lightsDirty) return MOX_OK;
  int rc = upload(c, c->dLights, c->lights);
  if (rc) return rc;
  // normalize(lp->normal) is the same for every hit (Material.cu:183): IEEE multiply / add / sqrt / divide in the
  // order of vec.cuh's normalize give the same bits on the host as in the shade kernel
  c->lightN.resize(c->lights.size());
  for (size_t i = 0; i < c->lights.size(); ++i) {
    const float3 n = normalize(mk3(c->lights[i].normal.x, c->lights[i].normal.y, c->lights[i].normal.z));
    c->lightN[i] = make_float4(n.x, n.y, n.z, 0.f);
  }
  if ((rc = upload(c, c->dLightN, c->lightN))) return rc;
  c->lightsDirty = false;
  return MOX_OK;
}

// The counter block of bounce `depth` in the device counters (pb.counters) or in their host copy (hostCnt): after the
// C_WORDS batch words, a ring of BOUNCE_RING blocks.
inline uint32_t* bounceBlock(uint32_t* counters, uint32_t depth) { return counters + C_WORDS + (depth % BOUNCE_RING) * C_BOUNCE_WORDS; }

// Exact number of rays bounce `depth` traced (`bound` camera rays at depth 1), and of shadow rays the bounce before it
// queued, from the counters in hostCnt.
void countBounceRays(mox_ctx* c, uint32_t depth, uint32_t bound) {
  mox_stats& st = c->st;
  const uint32_t dIdx = std::min<uint32_t>(depth, MOX_STATS_DEPTHS - 1);
  if (depth == 1) { st.rays_primary += bound; st.rays_depth[1] += bound; }
  else {
    const uint32_t* prev = bounceBlock(c->hostCnt.p, depth - 1);
    st.rays_bounce += prev[C_NEXT];
    st.rays_shadow_traced += prev[C_SHQ];
    st.rays_depth[dIdx] += prev[C_NEXT];
    st.shadow_traced_depth[std::min<uint32_t>(depth - 1, MOX_STATS_DEPTHS - 1)] += prev[C_SHQ];
  }
}

// Events, pinned counters and wavefront buffers for a batch of S samples of `count` pixels.  renderSeeds calls it
// before its timed region, so the first launch of a context does not time its own allocations.
int prepareBatch(mox_ctx* c, uint32_t S, uint32_t count) {
  if (!c->evReady) CUCK(c, cudaEventCreateWithFlags(&c->evReady, cudaEventDisableTiming));
  if (c->overlapShadow && !c->shadowStream) {
    CUCK(c, cudaStreamCreateWithFlags(&c->shadowStream, cudaStreamNonBlocking));
    CUCK(c, cudaEventCreateWithFlags(&c->evShaded, cudaEventDisableTiming));
    CUCK(c, cudaEventCreateWithFlags(&c->evApplied, cudaEventDisableTiming));
  }
  int rc = ensure(c, c->hostCnt, kCounterWords * 4);
  return rc ? rc : ensurePaths(c, (size_t)S * count, c->lights.size(), S);
}

// One wavefront batch: the S samples seeds[0, S) of each pixel of list[0, count); with `stats`, the accumulation also
// adds every sample's luminance to them.  Generate, then bounce by bounce until no path is left: extend, classify,
// wait for the material counts, shade, shadow.  Then accumulate and collect the counters.
int renderBatch(mox_ctx* c, const int32_t* seeds, uint32_t S, const uint32_t* list, uint32_t count, const PixelStats* stats) {
  const size_t P = (size_t)S * count;
  if (P == 0) return MOX_OK;
  if (P > 0xfffffff0ull) return fail(c, MOX_ERR_INVALID, "batch too large");
  int rc;
  // all allocations first: a failure (MOX_ERR_OOM -> the caller retries with a smaller batch) must not leave work
  // in flight
  if ((rc = prepareBatch(c, S, count))) return rc;
  PathBuffers& pb = c->pb;
  StageTimer& tm = c->timer;
  mox_stats& st = c->st;
  CUCK(c, cudaMemcpyAsync(pb.seeds, seeds, S * 4, cudaMemcpyHostToDevice, c->stream));
  LaunchCtx lc;
  lc.scene = sceneView(c);
  lc.rp = c->rp;
  lc.pb = pb;
  lc.ownedPix = list;
  lc.nOwned = count;
  lc.accu = c->dAccu.p;
  lc.countTraversal = (c->accelFlags & MOX_ACCEL_COUNTERS) != 0;
  lc.brdfFast = c->brdfFast;
  lc.stream = c->stream;
  lc.pb.qCur = pb.qBuf[0]; lc.pb.qNext = pb.qBuf[1];
  lc.bc = bounceBlock(pb.counters, 1);
  CUCK(c, cudaMemsetAsync(pb.counters, 0, kCounterWords * 4, c->stream));
  tm.begin(ST_GENERATE, c->stream);
  launchGenerate(lc, S);
  tm.end(c->stream);
  st.kernel_launches++;
  // k_apply of a bounce may still run on the shadow stream (evApplied): the next kernel of the context stream that
  // touches the radiance or the shadow-ray buffers waits for it
  bool applyPending = false;
  auto waitApplied = [&]() -> int {
    if (applyPending) { CUCK(c, cudaStreamWaitEvent(c->stream, c->evApplied, 0)); applyPending = false; }
    return MOX_OK;
  };
  uint32_t bound = (uint32_t)P;   // rays this bounce traces at most: every shaded path spawns at most one
  bool ranTerminal = false;       // the last bounce ran the terminal query: its ray counts come with the final counter copy
  uint32_t depth;
  for (depth = 1;; ++depth) {
    lc.bc = bounceBlock(pb.counters, depth);
    lc.pb.qMat[Q_DISNEY] = (depth & 1u) ? pb.qMat[Q_DISNEY] : pb.qDisneyAlt;   // k_apply of bounce depth-1 may still read the other one
    // bounce 1 traces exactly `bound` camera rays; later bounces read the number of spawned rays from the previous
    // bounce's counter block, `bound` (what was shaded) only sizes the grids
    const uint32_t* countPtr = depth == 1 ? nullptr : bounceBlock(pb.counters, depth - 1) + C_NEXT;
    // k_classify's test: every path of this bounce ends in it, whatever it hits (|payload colour| = sqrt(3))
    const bool terminal = depth > c->rp.maxDepth || length(mk3(1.f)) < c->rp.minIntensity;
    // the AOVs need the camera rays' closest hits, which the terminal query does not record
    const bool aovHere = depth == 1 && c->aovBlock.p;
    if (terminal && c->terminalQuery && c->nTerminalLights >= 0 && lc.scene.nodes8 && !aovHere) {
      TerminalLights tl;
      tl.list = (const uint4*)c->dTerminalLights.p;
      tl.n = c->nTerminalLights;
      tl.missIsAbsorb = memcmp(&c->rp.bg, &c->rp.absorb, sizeof c->rp.bg) == 0;
      tm.begin(ST_EXTEND, c->stream, depth);
      launchTerminal(lc, depth == 1 ? nullptr : lc.pb.qCur, bound, countPtr, tl);
      tm.end(c->stream);
      st.extend_launches++; st.kernel_launches++;
      // k_classify would queue nothing: no counts to wait for, the accumulation follows at once
      ranTerminal = true;
      break;
    }
    tm.begin(ST_EXTEND, c->stream, depth);
    // camera rays are queued in path order (k_generate: qCur[p] = p): the traversal kernel skips the indirection
    launchExtend(lc, depth == 1 ? nullptr : lc.pb.qCur, bound, countPtr, depth);
    tm.end(c->stream);
    tm.begin(ST_SHADE, c->stream);
    launchClassify(lc, lc.pb.qCur, bound, countPtr, depth);
    tm.end(c->stream);
    st.extend_launches++; st.kernel_launches += 2;
    if (aovHere) { launchAov(lc, S, c->aov); st.kernel_launches++; c->aovRecorded = true; }
    CUCK(c, cudaMemcpyAsync(c->hostCnt.p, pb.counters, kCounterWords * 4, cudaMemcpyDeviceToHost, c->stream));
    CUCK(c, cudaEventRecord(c->evReady, c->stream));
    // the material counts size the shade launches: the host waits for them
    CUCK(c, cudaEventSynchronize(c->evReady));
    countBounceRays(c, depth, bound);
    const uint32_t* hostBounce = bounceBlock(c->hostCnt.p, depth);
    uint32_t binned[Q_COUNT], any = 0;
    for (int k = 0; k < Q_COUNT; ++k) { binned[k] = hostBounce[C_MAT0 + k]; any += binned[k]; }
    if (!any) break;
    // the shade kernels touch the radiance and rewrite the shadow-ray buffers: the previous bounce's k_apply first
    if ((rc = waitApplied())) return rc;
    tm.begin(ST_SHADE, c->stream);
    for (int k = 0; k < Q_COUNT; ++k) { launchShade(lc, k, binned[k], depth); if (binned[k]) st.kernel_launches++; }
    tm.end(c->stream);
    if (binned[Q_DISNEY] && lc.scene.nLights) {
      // Shadow rays and the NEE sum depend only on this bounce's shade kernels; the next extend launch does not
      // depend on them.  On a second stream the two persistent traversal launches overlap: each one's last CTAs
      // drain while the other's first CTAs already run.
      cudaStream_t ss = c->stream;
      if (c->overlapShadow && c->shadowStream) {
        ss = c->shadowStream;
        CUCK(c, cudaEventRecord(c->evShaded, c->stream));
        CUCK(c, cudaStreamWaitEvent(ss, c->evShaded, 0));
      }
      tm.begin(ST_SHADOW, ss, depth);
      launchShadow(lc, binned[Q_DISNEY], ss);
      tm.end(ss);
      tm.begin(ST_SHADE, ss);
      launchApply(lc, binned[Q_DISNEY], ss);
      tm.end(ss);
      if (ss != c->stream) { CUCK(c, cudaEventRecord(c->evApplied, ss)); applyPending = true; }
      st.kernel_launches += 2;
    }
    // the block bounce depth+1 will use was last written BOUNCE_RING bounces ago
    CUCK(c, cudaMemsetAsync(bounceBlock(pb.counters, depth + 1), 0, C_BOUNCE_WORDS * 4, c->stream));
    std::swap(lc.pb.qCur, lc.pb.qNext);
    bound = any;
  }
  if ((rc = waitApplied())) return rc;
  tm.begin(ST_ACCUMULATE, c->stream);
  if (stats) launchAccumulateAdaptive(lc, S, *stats);
  else launchAccumulate(lc, S);
  tm.end(c->stream);
  st.kernel_launches++;
  // the final counter read-back
  CUCK(c, cudaMemcpyAsync(c->hostCnt.p, pb.counters, kCounterWords * 4, cudaMemcpyDeviceToHost, c->stream));
  CUCK(c, cudaEventRecord(c->evReady, c->stream));
  CUCK(c, cudaEventSynchronize(c->evReady));
  const uint32_t* host = c->hostCnt.p;
  if (ranTerminal) countBounceRays(c, depth, bound);
  tm.collect(st);
  st.nonfinite_samples += host[C_NONFINITE];
  st.rays_shadow_blocked += host[C_SH_BLOCKED]; st.rays_shadow_tinted += host[C_SH_TINTED];
  st.rays_shadow += host[C_SHADOW];
  st.node_visits += counter64(host, C_NODEVIS_LO);
  st.prim_tests += counter64(host, C_PRIMTEST_LO);
  st.node_visits_shadow += counter64(host, C_NODEVIS_SH_LO);
  st.prim_tests_shadow += counter64(host, C_PRIMTEST_SH_LO);
  CUCK(c, cudaGetLastError());
  st.launches += S;
  return MOX_OK;
}

// Paths per batch: the configured cap, lowered so that the wavefront state fits into 60 % of the free device
// memory (what the current block holds counts as free) for this scene's light count (36 bytes per path and light).
size_t batchCap(mox_ctx* c, size_t wanted /* samples per pixel of this call */, uint32_t count /* pixels */) {
  size_t cap = c->maxBatchPaths;
  // The buffers of an earlier call already hold such a batch: nothing will be allocated, so there is nothing to
  // budget.  (cudaMemGetInfo is a slow driver call — it was the 20-70 ms hiccup in front of some steps.)
  if (count) {
    const size_t S = std::min(std::max<size_t>(1, cap / count), wanted);   // samples per batch at the full cap
    if (pathsFit(c, S * count, c->lights.size(), S)) return cap;
  }
  size_t freeB = 0, totalB = 0;
  if (cudaMemGetInfo(&freeB, &totalB) == cudaSuccess) {
    // bytes per path: at 2^20 paths every array is a multiple of 2 MiB, and the counters add less than a byte
    PathBuffers probe;
    const size_t perPath = pathLayout(1u << 20, c->lights.size(), 0, nullptr, probe) >> 20;
    size_t budget = (size_t)((freeB + c->pathBlock.bytes) * 0.6);
    cap = std::min(cap, std::max<size_t>(budget / perPath, 65536));
  }
  return cap;
}

int ensureAovs(mox_ctx* c);

// The preconditions of a render, then the device, the owned-pixel list, the lights, the AOV sums and the textures.
int beginRender(mox_ctx* c) {
  if (!c->built) return fail(c, MOX_ERR_STATE, "launch before mox_build_accel");
  if (!c->haveGlobals) return fail(c, MOX_ERR_STATE, "launch before mox_set_globals");
  if (!c->haveCamera) return fail(c, MOX_ERR_STATE, "launch before mox_set_camera");
  int rc = bind(c);
  if (rc) return rc;
  if ((rc = refreshOwned(c))) return rc;
  if ((rc = syncLights(c))) return rc;
  if ((rc = ensureAovs(c))) return rc;
  return syncTextures(c);
}

// One sample per seed for each pixel of list[0, count), in batches; with `stats`, the accumulation also adds every
// sample's luminance to them.  beginRender first.
int renderSeeds(mox_ctx* c, const std::vector<int32_t>& seeds, const uint32_t* list, uint32_t count, const PixelStats* stats = nullptr) {
  if (count == 0) { c->st.launches += seeds.size(); return MOX_OK; }
  size_t perBatch = std::max<size_t>(1, batchCap(c, seeds.size(), count) / count);
  int rc = prepareBatch(c, (uint32_t)std::min(perBatch, seeds.size()), count);
  if (rc && rc != MOX_ERR_OOM) return rc;   // out of memory: the loop below retries with smaller batches
  CUCK(c, cudaEventRecord(c->ev0, c->stream));
  for (size_t i = 0; i < seeds.size();) {
    const size_t n = std::min(perBatch, seeds.size() - i);
    rc = renderBatch(c, seeds.data() + i, (uint32_t)n, list, count, stats);
    if (rc == MOX_ERR_OOM && perBatch > 1) {
      // the allocation failed after all (fragmentation, another context on the device): free the wavefront
      // state, halve the batch and render this chunk again (nothing of it was enqueued)
      cudaGetLastError();
      c->pathBlock.release();
      c->pb = PathBuffers();
      perBatch = std::max<size_t>(1, perBatch / 2);
      continue;
    }
    if (rc) return rc;
    i += n;
  }
  CUCK(c, cudaEventRecord(c->ev1, c->stream));
  CUCK(c, cudaEventSynchronize(c->ev1));
  float ms = 0;
  CUCK(c, cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  c->st.ms_render += ms;
  return MOX_OK;
}

void freeGather(mox_ctx* c) {
  for (int w = 0; w < 2; ++w) { c->dGather[w].release(); c->hostGather[w].release(); }
  c->gatherBytes = 0; c->readPending = -1;
}

// The two gather buffers of this context (allocated on first use, re-allocated when the image size changes).
int ensureGather(mox_ctx* c, bool hostSide) {
  if (!c->dAccu.p) return fail(c, MOX_ERR_STATE, "no accumulation buffer (mox_set_globals first)");
  const size_t bytes = (size_t)c->accuW * c->accuH * 12;
  if (c->gatherBytes != bytes) {
    cudaStreamSynchronize(c->stream);
    if (c->copyStream) cudaStreamSynchronize(c->copyStream);
    bool peer = c->dGather[0].kind != GatherBuf::own || c->dGather[1].kind != GatherBuf::own;
    if (peer && c->gatherBytes) return fail(c, MOX_ERR_STATE, "image size changed after mox_gather_import");
    if (!peer) freeGather(c);
    c->gatherBytes = bytes;
  }
  if (!c->copyStream) CUCK(c, cudaStreamCreateWithFlags(&c->copyStream, cudaStreamNonBlocking));
  if (!c->evPushed) CUCK(c, cudaEventCreateWithFlags(&c->evPushed, cudaEventDisableTiming));
  for (int w = 0; w < 2; ++w) {
    if (!c->evCopied[w]) CUCK(c, cudaEventCreateWithFlags(&c->evCopied[w], cudaEventDisableTiming));
    GatherBuf& g = c->dGather[w];
    if (!g.p) { CUCK(c, cudaMalloc(&g.p, bytes)); CUCK(c, cudaMemsetAsync(g.p, 0, bytes, c->stream)); }
    if (hostSide && !c->hostGather[w].p) CUCK(c, c->hostGather[w].alloc(bytes));
  }
  return MOX_OK;
}

// What the builder reads of the context's device scene; the flags set the rest.
BuildInput buildInput(mox_ctx* c, uint32_t flags) {
  BuildInput in;
  in.arena = &c->buildArena;
  in.nPrims = (int)c->prims.size();
  in.prims = (const PrimDesc*)c->dPrims.p;
  in.tris = (const TriIdx*)c->dTris.p;
  in.verts = (const float*)c->dVerts.p;
  in.analytic = (const Analytic*)c->dAnalytic.p;
  in.mats = (const GpuMaterial*)c->dMats.p;
  in.evStart = c->ev0; in.evStop = c->ev1;
  in.watertight = (flags & MOX_ACCEL_WATERTIGHT) != 0;
  return in;
}

void buildShadeRecords(mox_ctx* c) {
  launchBuildShadeRecords((const TriIdx*)c->dTris.p, (const float*)c->dVerts.p, (const float*)c->dNormals.p, (const float*)c->dUvs.p,
                          (uint32_t)c->tris.size(), (float4*)c->dShadeRec.p, c->stream);
}

// The light primitives of the terminal query in id order, with their hit-record bits (k_pack gives a light material
// shade class MOX_CLASS_LIGHT).  False when a mesh has a light material or there are more than
// MOX_TERMINAL_LIGHTS_MAX of them.  Which ones the build kept is marked on the device (excludeUnbuiltLights).
bool terminalLightList(const mox_ctx* c, std::vector<uint4>& out) {
  out.clear();
  auto isLight = [&](uint32_t id) { return c->mats[c->prims[id].typeMat >> 2].kind == MOX_MAT_LIGHT; };
  for (const auto& m : c->meshes)
    if (m.nFaces && isLight(m.firstPrim)) return false;
  // the spheres and quads lie between the id ranges of the meshes (recorded in id order)
  uint32_t id = 0;
  auto scan = [&](uint32_t end) {
    for (; id < end; ++id) {
      if (!isLight(id)) continue;
      const uint32_t type = c->prims[id].typeMat & 3u;
      if (type == PT_TRI || out.size() == MOX_TERMINAL_LIGHTS_MAX) return false;
      out.push_back(make_uint4(id | (MOX_CLASS_LIGHT << MOX_HIT_ID_BITS), type, c->prims[id].geom, 0u));
    }
    return true;
  };
  for (const auto& m : c->meshes) {
    if (!scan(m.firstPrim)) return false;
    id = m.firstPrim + m.nFaces;
  }
  return scan((uint32_t)c->prims.size());
}

// ---- adaptive sampling (mox_render_adaptive)

// The per-pixel statistics (zeroed when allocated) and the active-pixel lists for the current image and partition.
int ensureAdaptive(mox_ctx* c) {
  const size_t nPix = (size_t)c->accuW * c->accuH;
  if (!c->adaptiveStats.p) {
    CUCK(c, c->adaptiveStats.alloc(nPix * 24));
    char* b = (char*)c->adaptiveStats.p;
    PixelStats& ps = c->pixelStats;
    ps.s1 = (double*)b;
    ps.s2 = (double*)(b + 8 * nPix);
    ps.n = (uint32_t*)(b + 16 * nPix);
    ps.skipped = ps.n + nPix;
    CUCK(c, cudaMemsetAsync(b, 0, nPix * 24, c->stream));
  }
  const size_t words = 2 * (size_t)c->nOwned + adaptiveSelectTiles(c->nOwned) + 1;
  int rc = ensure(c, c->adaptiveLists, words * 4);
  return rc ? rc : ensure(c, c->hostSurvivors, 4);
}

// Forget every adaptive sample: the accumulation buffer was cleared or replaced.
int resetAdaptive(mox_ctx* c) {
  if (c->adaptiveStats.p) CUCK(c, cudaMemsetAsync(c->adaptiveStats.p, 0, c->adaptiveStats.bytes, c->stream));
  return MOX_OK;
}

// Keeps the pixels of in[0, count) that have not converged under `rule`, in order, in `out`; the others sit out the
// call's `remaining` launches.  Sets `active` to the number kept.
int selectActive(mox_ctx* c, const AdaptiveRule& rule, const uint32_t* in, uint32_t count, uint32_t remaining, uint32_t* out,
                 uint32_t& active) {
  uint32_t* tileSums = (uint32_t*)c->adaptiveLists.p + 2 * (size_t)c->nOwned;
  uint32_t* survivors = tileSums + adaptiveSelectTiles(c->nOwned);
  if (count) {
    launchAdaptiveSelect(c->pixelStats, rule, in, count, remaining, out, tileSums, survivors, c->stream);
    c->st.kernel_launches += 2;
  } else CUCK(c, cudaMemsetAsync(survivors, 0, 4, c->stream));
  CUCK(c, cudaMemcpyAsync(c->hostSurvivors.p, survivors, 4, cudaMemcpyDeviceToHost, c->stream));
  CUCK(c, cudaStreamSynchronize(c->stream));
  CUCK(c, cudaGetLastError());
  active = *c->hostSurvivors.p;
  return MOX_OK;
}

// Launches st.launches .. st.launches + spp - 1 of mox_render's seed schedule for the pixels that have not converged,
// in rounds of round_spp launches with a convergence check after each.  beginRender and ensureAdaptive first.
int renderAdaptive(mox_ctx* c, uint32_t spp, uint32_t seed, const mox_adaptive& p, uint64_t& traced) {
  const AdaptiveRule rule{std::max<uint32_t>(p.min_spp, 2u), (double)p.rel_error, (double)p.abs_error};
  uint32_t* lists[2] = {(uint32_t*)c->adaptiveLists.p, (uint32_t*)c->adaptiveLists.p + c->nOwned};
  const uint64_t first = c->st.launches;
  uint32_t active = 0, cur = 0, done = 0;
  int rc = selectActive(c, rule, c->dOwned.p, c->nOwned, spp, lists[0], active);
  while (!rc && done < spp && active) {
    const uint32_t r = std::min(p.round_spp, spp - done);
    std::vector<int32_t> seeds(r);
    for (uint32_t i = 0; i < r; ++i) seeds[i] = (int32_t)tea16((uint32_t)(first + done + i), seed);
    if ((rc = renderSeeds(c, seeds, lists[cur], active, &c->pixelStats))) break;
    traced += (uint64_t)r * active;
    done += r;
    if (done == spp) break;   // a pixel that converges now sits out no launch
    rc = selectActive(c, rule, lists[cur], active, spp - done, lists[cur ^ 1], active);
    cur ^= 1;
  }
  if (rc) return rc;
  c->st.launches = first + spp;   // the launches no pixel needed still advance the seed schedule
  return MOX_OK;
}

// ---- first-hit AOVs and the denoiser (mox_set_aovs, mox_read_aovs, mox_denoise)

constexpr size_t kAovBytesPerPixel = 36;

// The AOV arrays of nPix pixels in one block at `base`: albedo xyz, normal xyz, depth, sample count, hit count.
AovBuffers aovLayout(void* base, size_t nPix) {
  AovBuffers a;
  float* f = (float*)base;
  a.albedo = f; a.normal = f + 3 * nPix; a.depth = f + 6 * nPix;
  a.n = (uint32_t*)(f + 7 * nPix); a.hits = a.n + nPix;
  return a;
}

// Allocates and zeroes the sums while AOVs are on and the image size is known.
int ensureAovs(mox_ctx* c) {
  if (!c->aovOn || c->aovBlock.p || !c->dAccu.p) return MOX_OK;
  const size_t nPix = (size_t)c->accuW * c->accuH;
  CUCK(c, c->aovBlock.alloc(nPix * kAovBytesPerPixel));
  c->aov = aovLayout(c->aovBlock.p, nPix);
  CUCK(c, cudaMemsetAsync(c->aovBlock.p, 0, nPix * kAovBytesPerPixel, c->stream));
  c->aovRecorded = false;
  return MOX_OK;
}

// Forget every AOV record: the accumulation buffer was cleared or replaced.
int resetAovs(mox_ctx* c) {
  if (c->aovBlock.p) CUCK(c, cudaMemsetAsync(c->aovBlock.p, 0, c->aovBlock.bytes, c->stream));
  c->aovRecorded = false;
  return MOX_OK;
}

// The AOV means of this context (full frame; pixels of other ranks read 0) into the destinations that are not null.
int readAovMeans(mox_ctx* c, float* albedo, float* normal, float* depth) {
  if (!c->aovOn) return fail(c, MOX_ERR_STATE, "AOVs are off (mox_set_aovs)");
  if (!c->aovBlock.p) return fail(c, MOX_ERR_STATE, "no accumulation buffer (mox_set_globals first)");
  int rc = bind(c);
  if (rc) return rc;
  const size_t nPix = (size_t)c->accuW * c->accuH;
  std::vector<float> h(nPix * (kAovBytesPerPixel / 4));
  CUCK(c, cudaMemcpyAsync(h.data(), c->aovBlock.p, nPix * kAovBytesPerPixel, cudaMemcpyDeviceToHost, c->stream));
  CUCK(c, cudaStreamSynchronize(c->stream));
  const AovBuffers s = aovLayout(h.data(), nPix);
  for (size_t p = 0; p < nPix; ++p) {
    const float n = (float)s.n[p];
    for (int k = 0; k < 3; ++k) {
      if (albedo) albedo[3 * p + k] = s.n[p] ? s.albedo[3 * p + k] / n : 0.f;
      if (normal) normal[3 * p + k] = s.n[p] ? s.normal[3 * p + k] / n : 0.f;
    }
    if (depth) depth[p] = s.hits[p] ? s.depth[p] / (float)s.hits[p] : 0.f;
  }
  return MOX_OK;
}

// params (null: the defaults) checked and converted.
int denoiseParams(mox_ctx* c, const mox_denoise_params* in, DenoiseParams& p) {
  mox_denoise_params d{MOX_DENOISE_DEFAULT_ITERATIONS, MOX_DENOISE_DEFAULT_SIGMA_COLOR, MOX_DENOISE_DEFAULT_SIGMA_NORMAL,
                       MOX_DENOISE_DEFAULT_SIGMA_DEPTH};
  if (in) d = *in;
  if (d.iterations < 1 || d.iterations > 10) return fail(c, MOX_ERR_INVALID, "mox_denoise_params.iterations must be 1..10");
  for (float s : {d.sigma_color, d.sigma_normal, d.sigma_depth})
    if (!std::isfinite(s) || !(s > 0.f)) return fail(c, MOX_ERR_INVALID, "mox_denoise_params sigmas must be finite and > 0");
  p = DenoiseParams{d.iterations, d.sigma_color, d.sigma_normal, d.sigma_depth};
  return MOX_OK;
}

// The launches pixel p sat out in adaptive renders (null: none).
const uint32_t* skippedLaunches(const mox_ctx* c) { return c->adaptiveStats.p ? c->pixelStats.skipped : nullptr; }

// Filters the frame `in` on c's device (bound) into dst (host, W*H*3 floats).
int runDenoise(mox_ctx* c, const DenoiseInput& in, const DenoiseParams& p, float* dst, float* out_ms) {
  const size_t nPix = (size_t)in.W * in.H;
  int rc = ensure(c, c->denoiseScratch, denoiseScratchBytes(in.W, in.H));
  if (rc || (rc = ensure(c, c->denoiseOut, nPix * 12))) return rc;
  CUCK(c, cudaEventRecord(c->ev0, c->stream));
  launchDenoise(in, p, c->denoiseScratch.p, (float*)c->denoiseOut.p, c->stream);
  CUCK(c, cudaEventRecord(c->ev1, c->stream));
  CUCK(c, cudaMemcpyAsync(dst, c->denoiseOut.p, nPix * 12, cudaMemcpyDeviceToHost, c->stream));
  CUCK(c, cudaStreamSynchronize(c->stream));
  CUCK(c, cudaGetLastError());
  float ms = 0;
  CUCK(c, cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  if (out_ms) *out_ms = ms;
  return MOX_OK;
}

// mox_denoise on a multi-GPU handle: every device stores the inputs of the pixels it owns into device 0's frame (peer
// stores), then device 0 filters the whole frame.  Errors are reported on the shell c.
int denoiseGroup(mox_ctx* c, const DenoiseParams& p, float* dst, float* out_ms) {
  mox_group* g = c->group;
  mox_ctx* k0 = groupChild(g, 0);
  for (int i = 0; i < groupCount(g); ++i)
    if (!groupChild(g, i)->aovOn || !groupChild(g, i)->aovBlock.p) return fail(c, MOX_ERR_STATE, "AOVs are off (mox_set_aovs)");
  bool recorded = false;
  for (int i = 0; i < groupCount(g); ++i) recorded = recorded || groupChild(g, i)->aovRecorded;
  if (!recorded) return fail(c, MOX_ERR_STATE, "mox_denoise before any sample was rendered with AOVs on");
  auto err0 = [&](int rc) { c->err = mox_last_error(k0); return rc; };
  int rc = bind(k0);
  if (rc) return err0(rc);
  const size_t nPix = (size_t)k0->accuW * k0->accuH;
  if ((rc = ensure(k0, k0->denoiseFrame, nPix * (12 + 4 + kAovBytesPerPixel)))) return err0(rc);
  float* frameAccu = (float*)k0->denoiseFrame.p;
  uint32_t* frameSkipped = (uint32_t*)(frameAccu + 3 * nPix);
  const AovBuffers frameAov = aovLayout(frameSkipped + nPix, nPix);
  if (cudaStreamSynchronize(k0->stream) != cudaSuccess) return fail(c, MOX_ERR_CUDA, "device 0 stream");
  rc = groupParallel(g, [&](mox_ctx* k, int) -> int {
    int r = bind(k);
    if (r || (r = refreshOwned(k))) return r;
    launchPushDenoiseInput(k->dOwned.p, k->nOwned, k->dAccu.p, skippedLaunches(k), k->aov, frameAccu, frameSkipped, frameAov, k->stream);
    CUCK(k, cudaStreamSynchronize(k->stream));   // the pixels have landed before device 0 reads them
    CUCK(k, cudaGetLastError());
    return MOX_OK;
  });
  if (rc) { c->err = groupError(g); return rc; }
  if ((rc = bind(k0))) return err0(rc);
  const DenoiseInput in{frameAccu, frameSkipped, (uint32_t)k0->st.launches, frameAov, k0->accuW, k0->accuH};
  if ((rc = runDenoise(k0, in, p, dst, out_ms))) return err0(rc);
  return MOX_OK;
}

constexpr int kRebuild = 1;   // refitAccel: nothing to refit, run the full build

// MOX_ACCEL_REFIT (flags without it): refit the structure of the last full build in place.  Uploads only what
// mox_update_mesh / mox_update_sphere can have changed.  Returns kRebuild when that build had at most one valid
// primitive: there is no hierarchy to keep, and a full build is as cheap.
int refitAccel(mox_ctx* c, uint32_t flags, float* out_ms) {
  if (!c->refitOk)
    return fail(c, MOX_ERR_STATE, "MOX_ACCEL_REFIT needs a successful full build with no mox_add_* / mox_clear_scene after it");
  if (const char* env = getenv("MOX_WATERTIGHT")) { if (atoi(env)) flags |= MOX_ACCEL_WATERTIGHT; }
  if (flags != c->accelFlags) return fail(c, MOX_ERR_INVALID, "MOX_ACCEL_REFIT: the other flags differ from those of the last full build");
  if (c->accel.refit.path == RefitState::TRIVIAL) return kRebuild;
  // A failed refit must not leave a context that still claims to be built, nor one that offers a refit again.
  c->built = false;
  c->refitOk = false;
  cudaStreamSynchronize(c->stream);
  if (c->vDirtyLo < c->vDirtyHi)
    CUCK(c, cudaMemcpyAsync((float*)c->dVerts.p + c->vDirtyLo, c->verts.data() + c->vDirtyLo, (c->vDirtyHi - c->vDirtyLo) * 4,
                            cudaMemcpyHostToDevice, c->stream));
  if (c->nDirtyLo < c->nDirtyHi)
    CUCK(c, cudaMemcpyAsync((float*)c->dNormals.p + c->nDirtyLo, c->normals.data() + c->nDirtyLo, (c->nDirtyHi - c->nDirtyLo) * 4,
                            cudaMemcpyHostToDevice, c->stream));
  c->vDirtyLo = c->nDirtyLo = SIZE_MAX; c->vDirtyHi = c->nDirtyHi = 0;
  int rc = upload(c, c->dAnalytic, c->analytic);
  if (rc) return rc;
  if (c->shadeRecBuilt) buildShadeRecords(c);   // ahead of the timed kernels, as in the full build
  BuildInput in = buildInput(c, flags);
  std::string err;
  bool changed = false;
  if (!refitBvh(in, c->accel, c->stream, err, &changed)) return fail(c, MOX_ERR_CUDA, "build_accel (refit): " + err);
  if (changed)
    return fail(c, MOX_ERR_STATE, "MOX_ACCEL_REFIT: a primitive became degenerate, or valid again, since the last full build; "
                                  "build without MOX_ACCEL_REFIT");
  float ms = 0;
  CUCK(c, cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  c->st.ms_build = ms;
  c->built = true;
  c->refitOk = true;
  if (out_ms) *out_ms = ms;
  return MOX_OK;
}

}  // namespace

// A multi-GPU handle (mox_create_multi) is a shell: every call is forwarded to its per-device contexts.
#define GROUP_EACH(c, expr)                                                                      \
  do {                                                                                           \
    if ((c)->group) {                                                                            \
      int rc_ = groupEach((c)->group, [&](mox_ctx* k, int) { return (expr); });                  \
      if (rc_) (c)->err = groupError((c)->group);                                                \
      return rc_;                                                                                \
    }                                                                                            \
  } while (0)
#define GROUP_PAR(c, expr)                                                                       \
  do {                                                                                           \
    if ((c)->group) {                                                                            \
      int rc_ = groupParallel((c)->group, [&](mox_ctx* k, int) { return (expr); });              \
      if (rc_) (c)->err = groupError((c)->group);                                                \
      return rc_;                                                                                \
    }                                                                                            \
  } while (0)
#define GROUP_REFUSE(c, what) \
  do { if ((c)->group) return fail((c), MOX_ERR_INVALID, what " is managed by the multi-GPU handle itself"); } while (0)
#define GROUP_FIRST(c, expr)                                                                     \
  do {                                                                                           \
    if ((c)->group) {                                                                            \
      mox_ctx* k = groupChild((c)->group, 0);                                                    \
      int rc_ = (expr);                                                                          \
      if (rc_) (c)->err = mox_last_error(k);                                                     \
      return rc_;                                                                                \
    }                                                                                            \
  } while (0)

extern "C" {

int mox_abi_version(void) { return MOX_ABI_VERSION; }

int mox_create_multi(mox_ctx** out, const int* device_ids, int n_devices) {
  if (!out) return fail(nullptr, MOX_ERR_INVALID, "null out pointer");
  *out = nullptr;
  std::string err;
  mox_group* g = nullptr;
  int rc = groupCreate(&g, device_ids, n_devices, err);
  if (rc) return fail(nullptr, rc, err);
  mox_ctx* shell = new mox_ctx();
  shell->group = g;
  *out = shell;
  return MOX_OK;
}

int mox_device_count(const mox_ctx* c) { return c ? (c->group ? groupCount(c->group) : 1) : 0; }

const char* mox_last_error(const mox_ctx* c) { return c ? c->err.c_str() : g_createError.c_str(); }

int mox_create(mox_ctx** out, int device_id) {
  if (!out) return fail(nullptr, MOX_ERR_INVALID, "null out pointer");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return fail(nullptr, MOX_ERR_CUDA, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count 0") +
                                           " (this library has no CPU fallback)");
  if (device_id < 0 || device_id >= n) return fail(nullptr, MOX_ERR_INVALID, "device_id out of range");
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device_id)) != cudaSuccess) return fail(nullptr, MOX_ERR_CUDA, cudaGetErrorString(e));
  if (prop.major != 10)
    return fail(nullptr, MOX_ERR_CUDA, std::string("device ") + prop.name + " is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                                           "; libmox.so contains sm_100a code only");
  mox_ctx* c = new mox_ctx();
  c->device = device_id;
  if ((e = cudaSetDevice(device_id)) != cudaSuccess || (e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaEventCreate(&c->ev0)) != cudaSuccess || (e = cudaEventCreate(&c->ev1)) != cudaSuccess) {
    std::string msg = cudaGetErrorString(e);
    delete c;
    return fail(nullptr, MOX_ERR_CUDA, msg);
  }
  if (const char* env = getenv("MOX_MAX_BATCH_PATHS")) { long long v = atoll(env); if (v > 0) c->maxBatchPaths = (size_t)v; }
  if (const char* env = getenv("MOX_OVERLAP_SHADOW")) c->overlapShadow = atoi(env) != 0;
  if (const char* env = getenv("MOX_BRDF_IEEE")) c->brdfFast = atoi(env) == 0;
  if (const char* env = getenv("MOX_TERMINAL_CLOSEST")) c->terminalQuery = atoi(env) == 0;
  memset(&c->rp, 0, sizeof c->rp);
  c->rp.maxDepth = 256; c->rp.eps = 0.001f; c->rp.minIntensity = 0.001f;
  c->rp.bad = make_float3(1.f, 1.f, 1.f);
  *out = c;
  return MOX_OK;
}

void mox_destroy(mox_ctx* c) {
  if (!c) return;
  if (c->group) { groupDestroy(c->group); delete c; return; }
  cudaSetDevice(c->device);
  for (cudaStream_t s : {c->stream, c->shadowStream, c->copyStream})
    if (s) cudaStreamSynchronize(s);
  delete c;
}

int mox_set_globals(mox_ctx* c, uint32_t width, uint32_t height, uint32_t rayMaxDepth, float rayEpsilonT, float rayMinIntensity,
                    const float absorbColor[3], const float badColor[3], const float bgColor[3]) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_EACH(c, mox_set_globals(k, width, height, rayMaxDepth, rayEpsilonT, rayMinIntensity, absorbColor, badColor, bgColor));
  if (!width || !height || !absorbColor || !badColor || !bgColor) return fail(c, MOX_ERR_INVALID, "bad globals");
  if ((uint64_t)width * height > 0x7fffffffull / 3) return fail(c, MOX_ERR_INVALID, "image too large");
  int rc = bind(c);
  if (rc) return rc;
  if (width != c->accuW || height != c->accuH || !c->dAccu.p) {
    cudaStreamSynchronize(c->stream);
    CUCK(c, c->dAccu.alloc((size_t)width * height * 12));
    CUCK(c, cudaMemsetAsync(c->dAccu.p, 0, (size_t)width * height * 12, c->stream));
    c->accuW = width; c->accuH = height;
    c->st.launches = 0;
    c->ownedDirty = true;
    c->adaptiveStats.release();   // allocated again, zeroed, at the next mox_render_adaptive
    c->adaptiveLists.release();
    c->pixelStats = PixelStats();
    c->aovBlock.release();       // allocated again, zeroed, for the new size (ensureAovs below)
    c->aov = AovBuffers();
  }
  c->rp.W = width; c->rp.H = height; c->rp.maxDepth = rayMaxDepth; c->rp.eps = rayEpsilonT; c->rp.minIntensity = rayMinIntensity;
  c->rp.absorb = make_float3(absorbColor[0], absorbColor[1], absorbColor[2]);
  c->rp.bad = make_float3(badColor[0], badColor[1], badColor[2]);
  c->rp.bg = make_float3(bgColor[0], bgColor[1], bgColor[2]);
  c->haveGlobals = true;
  return ensureAovs(c);
}

int mox_set_camera(mox_ctx* c, const CamParams* cam) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_EACH(c, mox_set_camera(k, cam));
  if (!cam) return fail(c, MOX_ERR_INVALID, "null camera");
  c->rp.cam = *cam;
  c->haveCamera = true;
  return MOX_OK;
}

int mox_set_rng_mode(mox_ctx* c, int mode) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_EACH(c, mox_set_rng_mode(k, mode));
  if (mode != MOX_RNG_REF && mode != MOX_RNG_PHILOX) return fail(c, MOX_ERR_INVALID, "bad rng mode");
  c->rp.rngMode = mode;
  return MOX_OK;
}

int mox_set_partition(mox_ctx* c, uint32_t rank, uint32_t world, uint32_t tile) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_REFUSE(c, "the tile partition");
  if (!world || rank >= world || !tile) return fail(c, MOX_ERR_INVALID, "bad partition");
  c->rank = rank; c->world = world; c->tile = tile;
  c->ownedDirty = true;
  return MOX_OK;
}

int mox_add_texture_rgba32f(mox_ctx* c, const float* texels, int w, int h, int* out_id) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_EACH(c, mox_add_texture_rgba32f(k, texels, w, h, out_id));
  if (!texels || w <= 0 || h <= 0 || w > 32768 || h > 32768) return fail(c, MOX_ERR_INVALID, "bad texture");
  mox_ctx::HostTexture t;
  t.w = w; t.h = h;
  t.texels.assign(texels, texels + (size_t)w * h * 4);
  c->textures.push_back(std::move(t));
  c->texturesDirty = true;
  if (out_id) *out_id = (int)c->textures.size();
  return MOX_OK;
}

int mox_add_sphere(mox_ctx* c, const SphereParams* s, int kind, const void* params, uint32_t* out_id) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_EACH(c, mox_add_sphere(k, s, kind, params, out_id));
  if (!s || !params) return fail(c, MOX_ERR_INVALID, "null argument");
  int m = addMaterial(c, kind, params);
  if (m < 0) return fail(c, MOX_ERR_INVALID, "bad material kind");
  Analytic a;
  memset(&a, 0, sizeof a);
  a.a = make_float4(s->center.x, s->center.y, s->center.z, s->radius);
  c->analytic.push_back(a);
  c->prims.push_back({PT_SPHERE | ((uint32_t)m << 2), (uint32_t)c->analytic.size() - 1});
  c->nSpheres++;
  if (out_id) *out_id = (uint32_t)c->prims.size() - 1;
  c->built = false; c->refitOk = false;
  return MOX_OK;
}

int mox_add_quad(mox_ctx* c, const QuadParams* q, int kind, const void* params, uint32_t* out_id) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_EACH(c, mox_add_quad(k, q, kind, params, out_id));
  if (!q || !params) return fail(c, MOX_ERR_INVALID, "null argument");
  int m = addMaterial(c, kind, params);
  if (m < 0) return fail(c, MOX_ERR_INVALID, "bad material kind");
  Analytic a;
  a.a = make_float4(q->plane.x, q->plane.y, q->plane.z, q->plane.w);
  a.b = make_float4(q->v1.x, q->v1.y, q->v1.z, 0.f);
  a.c = make_float4(q->v2.x, q->v2.y, q->v2.z, 0.f);
  a.d = make_float4(q->anchor.x, q->anchor.y, q->anchor.z, 0.f);
  c->analytic.push_back(a);
  c->prims.push_back({PT_QUAD | ((uint32_t)m << 2), (uint32_t)c->analytic.size() - 1});
  c->nQuads++;
  if (out_id) *out_id = (uint32_t)c->prims.size() - 1;
  c->built = false; c->refitOk = false;
  return MOX_OK;
}

int mox_add_mesh(mox_ctx* c, const float* v, size_t nv, const float* n, size_t nn, const float* uv, size_t nt, const int32_t* vIdx,
                 const int32_t* nIdx, const int32_t* tIdx, size_t nFaces, int kind, const void* params, uint32_t* out_first) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_EACH(c, mox_add_mesh(k, v, nv, n, nn, uv, nt, vIdx, nIdx, tIdx, nFaces, kind, params, out_first));
  if (!params || (nFaces && (!v || !vIdx))) return fail(c, MOX_ERR_INVALID, "null argument");
  if (c->prims.size() + nFaces >= (1u << MOX_HIT_ID_BITS)) return fail(c, MOX_ERR_INVALID, "too many primitives");
  int m = addMaterial(c, kind, params);
  if (m < 0) return fail(c, MOX_ERR_INVALID, "bad material kind");
  bool hasN = nn > 0 && n && nIdx, hasT = nt > 0 && uv && tIdx;
  for (size_t f = 0; f < nFaces * 3; ++f) {
    if (vIdx[f] < 0 || (size_t)vIdx[f] >= nv) { c->mats.pop_back(); return fail(c, MOX_ERR_INVALID, "vertex index out of range"); }
    if (hasN && (nIdx[f] < 0 || (size_t)nIdx[f] >= nn)) hasN = false;
    if (hasT && (tIdx[f] < 0 || (size_t)tIdx[f] >= nt)) hasT = false;
  }
  int vb = (int)(c->verts.size() / 3), nb = (int)(c->normals.size() / 3), tb = (int)(c->uvs.size() / 2);
  c->verts.insert(c->verts.end(), v, v + nv * 3);
  if (hasN) c->normals.insert(c->normals.end(), n, n + nn * 3);
  if (hasT) c->uvs.insert(c->uvs.end(), uv, uv + nt * 2);
  if (out_first) *out_first = (uint32_t)c->prims.size();
  c->meshes.push_back({(uint32_t)c->prims.size(), (uint32_t)nFaces, (size_t)vb, nv, (size_t)nb, hasN ? nn : 0});
  c->tris.reserve(c->tris.size() + nFaces);
  c->prims.reserve(c->prims.size() + nFaces);
  for (size_t f = 0; f < nFaces; ++f) {
    TriIdx t;
    for (int k = 0; k < 3; ++k) {
      t.v[k] = vb + vIdx[3 * f + k];
      t.n[k] = hasN ? nb + nIdx[3 * f + k] : -1;
      t.t[k] = hasT ? tb + tIdx[3 * f + k] : -1;
    }
    c->tris.push_back(t);
    c->prims.push_back({PT_TRI | ((uint32_t)m << 2), (uint32_t)c->tris.size() - 1});
  }
  c->built = false; c->refitOk = false;
  return MOX_OK;
}

int mox_set_lights(mox_ctx* c, const LightParams* l, size_t n) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_EACH(c, mox_set_lights(k, l, n));
  if (n && !l) return fail(c, MOX_ERR_INVALID, "null lights");
  c->lights.assign(l, l + n);
  c->lightsDirty = true;
  return MOX_OK;
}

int mox_clear_scene(mox_ctx* c) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_EACH(c, mox_clear_scene(k));
  c->prims.clear(); c->tris.clear(); c->verts.clear(); c->normals.clear(); c->uvs.clear(); c->analytic.clear();
  c->mats.clear(); c->lights.clear(); c->meshes.clear();
  c->textures.clear(); c->texturesDirty = true;
  c->nSpheres = c->nQuads = 0;
  c->built = false; c->refitOk = false; c->lightsDirty = true;
  return MOX_OK;
}

int mox_build_accel(mox_ctx* c, uint32_t flags, float* out_ms) {
  if (!c) return MOX_ERR_INVALID;
  if (c->group) {
    std::vector<float> ms(groupCount(c->group), 0.f);
    int rc_ = groupParallel(c->group, [&](mox_ctx* k, int i) { return mox_build_accel(k, flags, &ms[i]); });
    if (rc_) { c->err = groupError(c->group); return rc_; }
    if (out_ms) *out_ms = *std::max_element(ms.begin(), ms.end());
    return MOX_OK;
  }
  int rc = bind(c);
  if (rc) return rc;
  if (flags & MOX_ACCEL_REFIT) {
    flags &= ~MOX_ACCEL_REFIT;
    if ((rc = refitAccel(c, flags, out_ms)) != kRebuild) return rc;
  }
  // A failed rebuild must not leave a context that still claims to be built.
  c->built = false;
  c->refitOk = false;
  c->wideBuilt = false;
  c->nTerminalLights = -1;
  cudaStreamSynchronize(c->stream);
  if ((rc = upload(c, c->dPrims, c->prims))) return rc;
  if ((rc = upload(c, c->dTris, c->tris))) return rc;
  if ((rc = upload(c, c->dVerts, c->verts))) return rc;
  if ((rc = upload(c, c->dNormals, c->normals))) return rc;
  if ((rc = upload(c, c->dUvs, c->uvs))) return rc;
  if ((rc = upload(c, c->dAnalytic, c->analytic))) return rc;
  if ((rc = upload(c, c->dMats, c->mats))) return rc;
  c->vDirtyLo = c->nDirtyLo = SIZE_MAX; c->vDirtyHi = c->nDirtyHi = 0;
  c->shadeRecBuilt = false;
  {
    bool want = !c->tris.empty();
    if (const char* env = getenv("MOX_SHADE_RECORDS")) want = want && atoi(env) != 0;
    if (want) {
      if ((rc = ensure(c, c->dShadeRec, c->tris.size() * MOX_SHADE_REC_F4 * sizeof(float4)))) return rc;
      buildShadeRecords(c);
      c->shadeRecBuilt = true;
    }
  }
  if ((rc = syncLights(c))) return rc;
  if ((rc = syncTextures(c))) return rc;
  for (auto& m : c->mats) {
    if (m.kind == MOX_MAT_DISNEY && (m.dis.albedoID < 0 || m.dis.albedoID > (int)c->textures.size()))
      return fail(c, MOX_ERR_INVALID, "DisneyParams.albedoID refers to a texture that was not added");
  }
  if (const char* env = getenv("MOX_WATERTIGHT")) { if (atoi(env)) flags |= MOX_ACCEL_WATERTIGHT; }
  BuildInput in = buildInput(c, flags);
  in.usePloc = (flags & MOX_ACCEL_LBVH) == 0;
  if (const char* env = getenv("MOX_PLOC_RADIUS")) in.plocRadius = atoi(env);
  if (const char* env = getenv("MOX_FORCE_LBVH")) { if (atoi(env)) in.usePloc = false; }
  c->useWide = (flags & MOX_ACCEL_BINARY) == 0;
  if (const char* env = getenv("MOX_FORCE_BINARY")) { if (atoi(env)) c->useWide = false; }
  in.useWide = c->useWide;
  std::string err;
  if (!buildBvh(in, c->accel, c->stream, err)) return fail(c, MOX_ERR_CUDA, "build_accel: " + err);
  c->wideBuilt = c->accel.nNodes8 > 0;
  CUCK(c, cudaEventSynchronize(c->ev1));
  float ms = 0;
  CUCK(c, cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  c->st.ms_build = ms;
  c->accelFlags = flags;
  c->built = true;
  c->refitOk = true;
  {
    std::vector<uint4> tl;
    if (terminalLightList(c, tl)) {
      if ((rc = upload(c, c->dTerminalLights, tl))) return rc;
      excludeUnbuiltLights((uint4*)c->dTerminalLights.p, (int)tl.size(), c->accel.refit, c->stream);
      CUCK(c, cudaGetLastError());
      c->nTerminalLights = (int)tl.size();
    }
  }
  if (out_ms) *out_ms = ms;
  return MOX_OK;
}

int mox_launch(mox_ctx* c, int32_t randSeed) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_PAR(c, mox_launch(k, randSeed));
  int rc = beginRender(c);
  return rc ? rc : renderSeeds(c, std::vector<int32_t>{randSeed}, c->dOwned.p, c->nOwned);
}

int mox_render(mox_ctx* c, uint32_t spp, uint32_t seed) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_PAR(c, mox_render(k, spp, seed));
  int rc = beginRender(c);
  if (rc) return rc;
  std::vector<int32_t> seeds(spp);
  for (uint32_t i = 0; i < spp; ++i) seeds[i] = (int32_t)tea16((uint32_t)(c->st.launches + i), seed);
  return renderSeeds(c, seeds, c->dOwned.p, c->nOwned);
}

int mox_render_adaptive(mox_ctx* c, uint32_t spp, uint32_t seed, const mox_adaptive* params, uint64_t* out_samples) {
  if (!c) return MOX_ERR_INVALID;
  if (out_samples) *out_samples = 0;
  if (!params) return fail(c, MOX_ERR_INVALID, "null adaptive parameters");
  if (!params->round_spp) return fail(c, MOX_ERR_INVALID, "mox_adaptive.round_spp must be at least 1");
  if (!std::isfinite(params->rel_error) || !std::isfinite(params->abs_error) || params->rel_error < 0.f || params->abs_error < 0.f)
    return fail(c, MOX_ERR_INVALID, "mox_adaptive thresholds must be finite and non-negative");
  if (c->group) {
    std::vector<uint64_t> n(groupCount(c->group), 0);
    int rc_ = groupParallel(c->group, [&](mox_ctx* k, int i) { return mox_render_adaptive(k, spp, seed, params, &n[i]); });
    if (rc_) { c->err = groupError(c->group); return rc_; }
    if (out_samples) for (uint64_t v : n) *out_samples += v;
    return MOX_OK;
  }
  int rc = beginRender(c);
  if (rc) return rc;
  if ((rc = ensureAdaptive(c))) return rc;
  uint64_t traced = 0;
  rc = renderAdaptive(c, spp, seed, *params, traced);
  if (out_samples) *out_samples = traced;
  return rc;
}

int mox_read_sample_counts(mox_ctx* c, uint32_t* dst) {
  if (!c) return MOX_ERR_INVALID;
  if (!dst) return fail(c, MOX_ERR_INVALID, "null destination");
  if (c->group) {   // every pixel is owned by one device, the others hold 0 for it
    const mox_ctx* k0 = groupChild(c->group, 0);
    const size_t n = (size_t)k0->accuW * k0->accuH;
    std::vector<uint32_t> part(n);
    std::fill(dst, dst + n, 0u);
    for (int i = 0; i < groupCount(c->group); ++i) {
      mox_ctx* k = groupChild(c->group, i);
      if (int rc_ = mox_read_sample_counts(k, part.data())) { c->err = mox_last_error(k); return rc_; }
      for (size_t p = 0; p < n; ++p) dst[p] += part[p];
    }
    return MOX_OK;
  }
  if (!c->dAccu.p) return fail(c, MOX_ERR_STATE, "no accumulation buffer (mox_set_globals first)");
  int rc = bind(c);
  if (rc) return rc;
  if ((rc = refreshOwned(c))) return rc;
  const size_t n = (size_t)c->accuW * c->accuH;
  std::vector<uint32_t> skipped(n, 0u);
  if (c->adaptiveStats.p) {
    CUCK(c, cudaMemcpyAsync(skipped.data(), c->pixelStats.skipped, n * 4, cudaMemcpyDeviceToHost, c->stream));
    CUCK(c, cudaStreamSynchronize(c->stream));
  }
  std::fill(dst, dst + n, 0u);
  std::vector<uint32_t> owned;
  ownedList(c->accuW, c->accuH, c->tile, c->world, c->rank, owned);
  for (uint32_t p : owned) dst[p] = (uint32_t)(c->st.launches - skipped[p]);
  return MOX_OK;
}

int mox_map_accum(mox_ctx* c, const float** out) {
  if (!c) return MOX_ERR_INVALID;
  if (c->group) {
    int rc_ = mox_read_accum_begin(c);
    return rc_ ? rc_ : mox_read_accum_end(c, out);
  }
  if (!out || !c->dAccu.p) return fail(c, MOX_ERR_INVALID, "no accumulation buffer");
  int rc = bind(c);
  if (rc) return rc;
  size_t bytes = (size_t)c->accuW * c->accuH * 12;
  if ((rc = ensure(c, c->pinned, bytes))) return rc;
  CUCK(c, cudaMemcpyAsync(c->pinned.p, c->dAccu.p, bytes, cudaMemcpyDeviceToHost, c->stream));
  CUCK(c, cudaStreamSynchronize(c->stream));
  *out = c->pinned.p;
  return MOX_OK;
}

int mox_read_accum(mox_ctx* c, float* dst) {
  if (!c) return MOX_ERR_INVALID;
  if (!dst) return fail(c, MOX_ERR_INVALID, "null destination");
  const float* p = nullptr;
  int rc = mox_map_accum(c, &p);
  if (rc) return rc;
  const mox_ctx* k = c->group ? groupChild(c->group, 0) : c;
  memcpy(dst, p, (size_t)k->accuW * k->accuH * 12);
  return MOX_OK;
}

int mox_unmap_accum(mox_ctx* c) { return c ? MOX_OK : MOX_ERR_INVALID; }

// ---- asynchronous read-back and the peer-memory tile gather (see include/mox.h)
float* ctxGatherBuffer(mox_ctx* c, int which) {
  if (bind(c) || ensureGather(c, true)) return nullptr;
  if (c->dGather[which].kind != GatherBuf::own) { c->err = "gather buffer is imported"; return nullptr; }
  cudaStreamSynchronize(c->stream);   // the zero-fill of a fresh buffer
  return c->dGather[which].p;
}

int ctxBorrowGatherTarget(mox_ctx* c, int which, float* ptr) {
  if (c->dGather[which].p == ptr) return MOX_OK;
  if (bind(c)) return MOX_ERR_CUDA;
  GatherBuf& g = c->dGather[which];
  if (g.p) cudaStreamSynchronize(c->stream);
  g.release();
  g.p = ptr; g.kind = GatherBuf::borrowed;
  c->gatherBytes = (size_t)c->accuW * c->accuH * 12;
  return MOX_OK;
}

int mox_gather_export(mox_ctx* c, int which, void* handle_out) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_REFUSE(c, "the tile gather");
  if (!handle_out || which < 0 || which > 1) return fail(c, MOX_ERR_INVALID, "bad gather_export arguments");
  int rc = bind(c);
  if (rc) return rc;
  if ((rc = ensureGather(c, true))) return rc;
  if (c->dGather[which].kind != GatherBuf::own) return fail(c, MOX_ERR_STATE, "this rank imported its gather buffer");
  CUCK(c, cudaStreamSynchronize(c->stream));
  static_assert(sizeof(cudaIpcMemHandle_t) == MOX_IPC_HANDLE_BYTES, "IPC handle size");
  CUCK(c, cudaIpcGetMemHandle((cudaIpcMemHandle_t*)handle_out, c->dGather[which].p));
  return MOX_OK;
}

int mox_gather_import(mox_ctx* c, int which, const void* handle) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_REFUSE(c, "the tile gather");
  if (!handle || which < 0 || which > 1) return fail(c, MOX_ERR_INVALID, "bad gather_import arguments");
  if (!c->dAccu.p) return fail(c, MOX_ERR_STATE, "mox_gather_import before mox_set_globals");
  int rc = bind(c);
  if (rc) return rc;
  GatherBuf& g = c->dGather[which];
  if (g.p) cudaStreamSynchronize(c->stream);
  g.release();
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof h);
  void* p = nullptr;
  CUCK(c, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
  g.p = (float*)p; g.kind = GatherBuf::ipc;
  c->gatherBytes = (size_t)c->accuW * c->accuH * 12;
  return MOX_OK;
}

int mox_gather_push(mox_ctx* c, int which) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_REFUSE(c, "the tile gather");
  if (which < 0 || which > 1 || !c->dAccu.p) return fail(c, MOX_ERR_INVALID, "bad gather_push");
  int rc = bind(c);
  if (rc) return rc;
  if ((rc = refreshOwned(c))) return rc;
  if (!c->dGather[which].p && (rc = ensureGather(c, false))) return rc;   // the root (or a single rank) pushes into its own buffer
  launchPushOwned(c->dAccu.p, c->dOwned.p, c->nOwned, c->dGather[which].p, c->stream);
  CUCK(c, cudaStreamSynchronize(c->stream));   // the pixels have landed before a barrier tells the root to read them
  return MOX_OK;
}

int mox_read_gathered_begin(mox_ctx* c, int which) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_REFUSE(c, "the tile gather");
  if (which < 0 || which > 1) return fail(c, MOX_ERR_INVALID, "bad buffer index");
  int rc = bind(c);
  if (rc) return rc;
  if ((rc = ensureGather(c, true))) return rc;
  if (c->dGather[which].kind != GatherBuf::own) return fail(c, MOX_ERR_STATE, "only the rank that owns the gather buffer reads it");
  // pushes of this rank are ordered by its stream, pushes of the others by the caller's barrier
  CUCK(c, cudaEventRecord(c->evPushed, c->stream));
  CUCK(c, cudaStreamWaitEvent(c->copyStream, c->evPushed, 0));
  CUCK(c, cudaMemcpyAsync(c->hostGather[which].p, c->dGather[which].p, c->gatherBytes, cudaMemcpyDeviceToHost, c->copyStream));
  CUCK(c, cudaEventRecord(c->evCopied[which], c->copyStream));
  return MOX_OK;
}

int mox_read_gathered_end(mox_ctx* c, int which, const float** out) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_REFUSE(c, "the tile gather");
  if (which < 0 || which > 1 || !out || !c->hostGather[which].p) return fail(c, MOX_ERR_INVALID, "bad read_gathered_end");
  CUCK(c, cudaEventSynchronize(c->evCopied[which]));
  *out = c->hostGather[which].p;
  return MOX_OK;
}

int mox_read_accum_begin(mox_ctx* c) {
  if (!c) return MOX_ERR_INVALID;
  if (c->group) {
    int rc_ = groupReadBegin(c->group);
    if (rc_) c->err = groupError(c->group);
    return rc_;
  }
  int rc = bind(c);
  if (rc) return rc;
  if ((rc = ensureGather(c, true))) return rc;
  const int which = c->readCur;
  if (c->dGather[which].kind != GatherBuf::own) return fail(c, MOX_ERR_STATE, "this rank's gather buffers are imported: use mox_gather_push");
  // snapshot on the render stream (the next launch may start right away), copy on the copy stream; the snapshot
  // must not overwrite an image the copy stream is still sending
  CUCK(c, cudaStreamWaitEvent(c->stream, c->evCopied[which], 0));
  CUCK(c, cudaMemcpyAsync(c->dGather[which].p, c->dAccu.p, c->gatherBytes, cudaMemcpyDeviceToDevice, c->stream));
  if ((rc = mox_read_gathered_begin(c, which))) return rc;
  c->readPending = which;
  c->readCur ^= 1;
  return MOX_OK;
}

int mox_read_accum_end(mox_ctx* c, const float** out) {
  if (!c) return MOX_ERR_INVALID;
  if (c->group) {
    int rc_ = groupReadEnd(c->group, out);
    if (rc_) c->err = groupError(c->group);
    return rc_;
  }
  if (c->readPending < 0) return fail(c, MOX_ERR_STATE, "mox_read_accum_end without mox_read_accum_begin");
  int rc = mox_read_gathered_end(c, c->readPending, out);
  c->readPending = -1;
  return rc;
}

int mox_clear_accum(mox_ctx* c) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_EACH(c, mox_clear_accum(k));
  int rc = bind(c);
  if (rc) return rc;
  if (c->dAccu.p) CUCK(c, cudaMemsetAsync(c->dAccu.p, 0, (size_t)c->accuW * c->accuH * 12, c->stream));
  if ((rc = resetAdaptive(c)) || (rc = resetAovs(c))) return rc;
  CUCK(c, cudaStreamSynchronize(c->stream));
  const double msBuild = c->st.ms_build;   // describes the acceleration structure, not the image
  c->st = mox_stats{};
  c->st.ms_build = msBuild;
  return MOX_OK;
}

int mox_set_accum(mox_ctx* c, const float* src, uint64_t launches) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_EACH(c, mox_set_accum(k, src, launches));   // every device keeps the pixels it owns
  if (!src || !c->dAccu.p) return fail(c, MOX_ERR_INVALID, "no accumulation buffer");
  int rc = bind(c);
  if (rc) return rc;
  CUCK(c, cudaMemcpyAsync(c->dAccu.p, src, (size_t)c->accuW * c->accuH * 12, cudaMemcpyHostToDevice, c->stream));
  if ((rc = resetAdaptive(c)) || (rc = resetAovs(c))) return rc;   // the loaded buffer counts as a uniform render of `launches` samples
  CUCK(c, cudaStreamSynchronize(c->stream));
  c->st.launches = launches;
  return MOX_OK;
}

int mox_set_aovs(mox_ctx* c, int enable) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_EACH(c, mox_set_aovs(k, enable));
  int rc = bind(c);
  if (rc) return rc;
  if (enable) {   // already on: the sums are kept
    c->aovOn = true;
    if ((rc = ensureAovs(c))) return rc;
    CUCK(c, cudaStreamSynchronize(c->stream));
    return MOX_OK;
  }
  c->aovOn = false;
  CUCK(c, cudaStreamSynchronize(c->stream));
  c->aovBlock.release();
  c->aov = AovBuffers();
  return MOX_OK;
}

int mox_read_aovs(mox_ctx* c, float* albedo, float* normal, float* depth) {
  if (!c) return MOX_ERR_INVALID;
  if (c->group) {   // every pixel is owned by one device, the others hold 0 for it
    const mox_ctx* k0 = groupChild(c->group, 0);
    const size_t n = (size_t)k0->accuW * k0->accuH;
    std::vector<float> a(albedo ? 3 * n : 0), nr(normal ? 3 * n : 0), z(depth ? n : 0);
    if (albedo) std::fill(albedo, albedo + 3 * n, 0.f);
    if (normal) std::fill(normal, normal + 3 * n, 0.f);
    if (depth) std::fill(depth, depth + n, 0.f);
    for (int i = 0; i < groupCount(c->group); ++i) {
      mox_ctx* k = groupChild(c->group, i);
      if (int rc_ = readAovMeans(k, albedo ? a.data() : nullptr, normal ? nr.data() : nullptr, depth ? z.data() : nullptr)) {
        c->err = mox_last_error(k);
        return rc_;
      }
      for (size_t p = 0; p < a.size(); ++p) albedo[p] += a[p];
      for (size_t p = 0; p < nr.size(); ++p) normal[p] += nr[p];
      for (size_t p = 0; p < z.size(); ++p) depth[p] += z[p];
    }
    return MOX_OK;
  }
  return readAovMeans(c, albedo, normal, depth);
}

int mox_denoise(mox_ctx* c, const mox_denoise_params* params, float* dst, float* out_ms) {
  if (!c) return MOX_ERR_INVALID;
  if (out_ms) *out_ms = 0.f;
  DenoiseParams p;
  int rc = denoiseParams(c, params, p);
  if (rc) return rc;
  if (!dst) return fail(c, MOX_ERR_INVALID, "null destination");
  if (c->group) return denoiseGroup(c, p, dst, out_ms);
  if (c->world > 1) return fail(c, MOX_ERR_STATE, "mox_denoise needs the whole frame: this context renders one rank of a partition");
  if (!c->aovOn || !c->aovBlock.p) return fail(c, MOX_ERR_STATE, "AOVs are off (mox_set_aovs)");
  if (!c->aovRecorded) return fail(c, MOX_ERR_STATE, "mox_denoise before any sample was rendered with AOVs on");
  if ((rc = bind(c))) return rc;
  const DenoiseInput in{c->dAccu.p, skippedLaunches(c), (uint32_t)c->st.launches, c->aov, c->accuW, c->accuH};
  return runDenoise(c, in, p, dst, out_ms);
}

int mox_update_sphere(mox_ctx* c, uint32_t prim_id, const SphereParams* s) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_EACH(c, mox_update_sphere(k, prim_id, s));
  if (!s || prim_id >= c->prims.size() || (c->prims[prim_id].typeMat & 3u) != PT_SPHERE) return fail(c, MOX_ERR_INVALID, "not a sphere primitive");
  c->analytic[c->prims[prim_id].geom].a = make_float4(s->center.x, s->center.y, s->center.z, s->radius);
  c->built = false;
  return MOX_OK;
}

int mox_update_mesh(mox_ctx* c, uint32_t first_prim_id, const float* v, size_t nv, const float* n, size_t nn) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_EACH(c, mox_update_mesh(k, first_prim_id, v, nv, n, nn));
  auto it = std::lower_bound(c->meshes.begin(), c->meshes.end(), first_prim_id,
                             [](const mox_ctx::MeshRec& m, uint32_t id) { return m.firstPrim < id; });
  while (it != c->meshes.end() && it + 1 != c->meshes.end() && (it + 1)->firstPrim == first_prim_id && it->nFaces == 0) ++it;  // skip empty meshes
  if (it == c->meshes.end() || it->firstPrim != first_prim_id) return fail(c, MOX_ERR_INVALID, "not the first primitive id of a mesh");
  const mox_ctx::MeshRec& m = *it;
  if (nv != m.nV || (nv && !v)) return fail(c, MOX_ERR_INVALID, "vertex count differs from the one the mesh was added with");
  if (n && (m.nN == 0 || nn != m.nN)) return fail(c, MOX_ERR_INVALID, "normal count differs from the one the mesh was added with");
  std::copy(v, v + 3 * nv, c->verts.begin() + 3 * m.vBase);
  c->vDirtyLo = std::min(c->vDirtyLo, 3 * m.vBase); c->vDirtyHi = std::max(c->vDirtyHi, 3 * (m.vBase + nv));
  if (n) {
    std::copy(n, n + 3 * nn, c->normals.begin() + 3 * m.nBase);
    c->nDirtyLo = std::min(c->nDirtyLo, 3 * m.nBase); c->nDirtyHi = std::max(c->nDirtyHi, 3 * (m.nBase + nn));
  }
  c->built = false;
  return MOX_OK;
}

int mox_owned_pixels(mox_ctx* c, uint32_t rank, uint64_t* out_n) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_REFUSE(c, "the tile partition");
  if (!out_n || rank >= c->world || !c->haveGlobals) return fail(c, MOX_ERR_INVALID, "bad owned_pixels query");
  // closed form: no need to enumerate the pixels
  uint32_t W = c->rp.W, H = c->rp.H, T = c->tile, tx = (W + T - 1) / T, ty = (H + T - 1) / T;
  uint64_t n = 0;
  for (uint32_t j = 0; j < ty; ++j)
    for (uint32_t i = 0; i < tx; ++i)
      if ((i + j) % c->world == rank) n += (uint64_t)(std::min(W, (i + 1) * T) - i * T) * (std::min(H, (j + 1) * T) - j * T);
  *out_n = n;
  return MOX_OK;
}

int mox_pack_owned(mox_ctx* c, void* dev_dst) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_REFUSE(c, "the tile gather");
  if (!dev_dst || !c->dAccu.p) return fail(c, MOX_ERR_INVALID, "bad pack_owned");
  int rc = bind(c);
  if (rc) return rc;
  if ((rc = refreshOwned(c))) return rc;
  launchPackOwned(c->dAccu.p, c->dOwned.p, c->nOwned, (float*)dev_dst, c->stream);
  CUCK(c, cudaStreamSynchronize(c->stream));
  return MOX_OK;
}

int mox_unpack_owned(mox_ctx* c, uint32_t rank, const void* dev_src) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_REFUSE(c, "the tile gather");
  if (!dev_src || !c->dAccu.p || rank >= c->world) return fail(c, MOX_ERR_INVALID, "bad unpack_owned");
  int rc = bind(c);
  if (rc) return rc;
  if ((rc = refreshOwned(c))) return rc;
  if (c->otherOwned.size() != c->world) { c->otherOwned.resize(c->world); c->ownedCount.assign(c->world, 0); }
  DevBuf& b = c->otherOwned[rank];
  if (!b.p) {  // first gather of this partition: build and upload rank's pixel list once
    std::vector<uint32_t> l;
    ownedList(c->rp.W, c->rp.H, c->tile, c->world, rank, l);
    if ((rc = ensure(c, b, l.size() * 4))) return rc;
    if (!l.empty()) { CUCK(c, cudaMemcpyAsync(b.p, l.data(), l.size() * 4, cudaMemcpyHostToDevice, c->stream)); CUCK(c, cudaStreamSynchronize(c->stream)); }
    c->ownedCount[rank] = l.size();
  }
  launchUnpackOwned(c->dAccu.p, (const uint32_t*)b.p, (uint32_t)c->ownedCount[rank], (const float*)dev_src, c->stream);
  CUCK(c, cudaStreamSynchronize(c->stream));
  return MOX_OK;
}

int mox_get_stats(mox_ctx* c, mox_stats* s) {
  if (!c) return MOX_ERR_INVALID;
  if (c->group) {
    if (!s) return fail(c, MOX_ERR_INVALID, "null stats");
    int rc_ = groupStats(c->group, s);
    if (rc_) c->err = groupError(c->group);
    return rc_;
  }
  if (!s) return fail(c, MOX_ERR_INVALID, "null stats");
  *s = c->st;
  s->n_prims = (uint32_t)c->prims.size(); s->n_triangles = (uint32_t)c->tris.size();
  s->n_spheres = c->nSpheres; s->n_quads = c->nQuads;
  const bool wide = c->wideBuilt && c->useWide;
  s->n_nodes = (uint32_t)(wide ? c->accel.nNodes8 : c->accel.nNodes); s->node_bytes = wide ? sizeof(BvhNode8) : sizeof(BvhNode2); s->prim_bytes = 16 * MOX_PACKED_F4;
  s->n_lights = (uint32_t)c->lights.size();
  return MOX_OK;
}

int mox_get_device_stats(mox_ctx* c, int index, mox_stats* s) {
  if (!c) return MOX_ERR_INVALID;
  if (index < 0 || index >= mox_device_count(c)) return fail(c, MOX_ERR_INVALID, "device index out of range");
  return mox_get_stats(c->group ? groupChild(c->group, index) : c, s);
}

int mox_trace_closest_device(mox_ctx* c, const void* dev_rays, size_t n, void* dev_hits, float* out_ms) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_FIRST(c, mox_trace_closest_device(k, dev_rays, n, dev_hits, out_ms));
  if (n && (!dev_rays || !dev_hits)) return fail(c, MOX_ERR_INVALID, "null argument");
  if (n > 0xfffffff0ull) return fail(c, MOX_ERR_INVALID, "too many rays");
  if (!c->built) return fail(c, MOX_ERR_STATE, "trace before mox_build_accel");
  if (out_ms) *out_ms = 0.f;
  if (!n) return MOX_OK;
  int rc = bind(c);
  if (rc) return rc;
  bool count = (c->accelFlags & MOX_ACCEL_COUNTERS) != 0;
  if ((rc = ensure(c, c->dQueryO, n * 16))) return rc;
  if ((rc = ensure(c, c->dQueryD, n * 16))) return rc;
  if ((rc = ensure(c, c->dQueryCounters, C_WORDS * 4))) return rc;
  uint32_t* counters = (uint32_t*)c->dQueryCounters.p;
  CUCK(c, cudaMemsetAsync(counters, 0, C_WORDS * 4, c->stream));
  launchSplitRays((const float4*)dev_rays, (float4*)c->dQueryO.p, (float4*)c->dQueryD.p, n, c->stream);
  TraceJob job;
  job.rayO = (const float4*)c->dQueryO.p; job.rayD = (const float4*)c->dQueryD.p; job.count = (uint32_t)n;
  job.cursor = counters + C_CURSOR; job.hits = (float4*)dev_hits; job.counters = counters;
  CUCK(c, cudaMemsetAsync(job.cursor, 0, 4, c->stream));
  CUCK(c, cudaEventRecord(c->ev0, c->stream));
  launchTraverse(sceneView(c), job, false, count, c->stream);
  CUCK(c, cudaEventRecord(c->ev1, c->stream));
  CUCK(c, cudaEventSynchronize(c->ev1));
  CUCK(c, cudaGetLastError());
  float ms = 0;
  CUCK(c, cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  if (out_ms) *out_ms = ms;
  if (count) {
    uint32_t host[C_WORDS];
    CUCK(c, cudaMemcpyAsync(host, counters, sizeof host, cudaMemcpyDeviceToHost, c->stream));
    CUCK(c, cudaStreamSynchronize(c->stream));
    c->st.node_visits += counter64(host, C_NODEVIS_LO);
    c->st.prim_tests += counter64(host, C_PRIMTEST_LO);
  }
  return MOX_OK;
}

int mox_trace_closest(mox_ctx* c, const float* rays, size_t n, void* hits) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_FIRST(c, mox_trace_closest(k, rays, n, hits));
  if (n && (!rays || !hits)) return fail(c, MOX_ERR_INVALID, "null argument");
  if (!c->built) return fail(c, MOX_ERR_STATE, "trace before mox_build_accel");
  if (!n) return MOX_OK;
  int rc = bind(c);
  if (rc) return rc;
  if ((rc = ensure(c, c->dQueryRays, n * 32)) || (rc = ensure(c, c->dQueryOut, n * 16))) return rc;
  void *dRays = c->dQueryRays.p, *dHits = c->dQueryOut.p;
  // stream-ordered: the traversal kernel runs on the (non-blocking) context stream
  CUCK(c, cudaMemcpyAsync(dRays, rays, n * 32, cudaMemcpyHostToDevice, c->stream));
  if ((rc = mox_trace_closest_device(c, dRays, n, dHits, nullptr))) return rc;
  CUCK(c, cudaMemcpyAsync(hits, dHits, n * 16, cudaMemcpyDeviceToHost, c->stream));
  CUCK(c, cudaStreamSynchronize(c->stream));
  return MOX_OK;
}

int mox_trace_shadow(mox_ctx* c, const float* rays, size_t n, float* out_rgb) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_FIRST(c, mox_trace_shadow(k, rays, n, out_rgb));
  if (n && (!rays || !out_rgb)) return fail(c, MOX_ERR_INVALID, "null argument");
  if (n > 0xfffffff0ull) return fail(c, MOX_ERR_INVALID, "too many rays");
  if (!c->built) return fail(c, MOX_ERR_STATE, "trace before mox_build_accel");
  if (!n) return MOX_OK;
  int rc = bind(c);
  if (rc) return rc;
  if ((rc = ensure(c, c->dQueryRays, n * 32)) || (rc = ensure(c, c->dQueryOut, n * 16)) || (rc = ensure(c, c->dQueryC, n * 16)) ||
      (rc = ensure(c, c->dQueryO, n * 16)) || (rc = ensure(c, c->dQueryD, n * 16)) || (rc = ensure(c, c->dQueryCounters, C_WORDS * 4)))
    return rc;
  void *dRays = c->dQueryRays.p, *dOut = c->dQueryOut.p, *dC = c->dQueryC.p;
  uint32_t* counters = (uint32_t*)c->dQueryCounters.p;
  CUCK(c, cudaMemcpyAsync(dRays, rays, n * 32, cudaMemcpyHostToDevice, c->stream));   // stream-ordered, see mox_trace_closest
  CUCK(c, cudaMemsetAsync(counters, 0, C_WORDS * 4, c->stream));
  launchSplitRays((const float4*)dRays, (float4*)c->dQueryO.p, (float4*)c->dQueryD.p, n, c->stream);
  launchFillOnes((float4*)dC, n, c->stream);
  TraceJob job;
  job.rayO = (const float4*)c->dQueryO.p; job.rayD = (const float4*)c->dQueryD.p; job.count = (uint32_t)n;
  job.cursor = counters + C_CURSOR; job.shC = (float4*)dC; job.counters = counters;
  launchTraverse(sceneView(c), job, true, false, c->stream);
  launchCopyRgb((const float4*)dC, (float*)dOut, n, c->stream);
  cudaError_t e = cudaStreamSynchronize(c->stream);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(out_rgb, dOut, n * 12, cudaMemcpyDeviceToHost, c->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  if (e != cudaSuccess) return fail(c, MOX_ERR_CUDA, cudaGetErrorString(e));
  return MOX_OK;
}

}  // extern "C"

// ---- debug / test hooks (not part of the drop-in surface; declared in include/mox_debug.h)
extern "C" int mox_debug_radix_sort(mox_ctx* c, uint32_t* keys, uint32_t* vals, size_t n) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_FIRST(c, mox_debug_radix_sort(k, keys, vals, n));
  if (n && (!keys || !vals)) return fail(c, MOX_ERR_INVALID, "null argument");
  if (!n) return MOX_OK;
  int rc = bind(c);
  if (rc) return rc;
  DevArray<uint32_t> dk, dv;
  CUCK(c, dk.alloc(n * 4));
  CUCK(c, dv.alloc(n * 4));
  CUCK(c, cudaMemcpyAsync(dk.p, keys, n * 4, cudaMemcpyHostToDevice, c->stream));
  CUCK(c, cudaMemcpyAsync(dv.p, vals, n * 4, cudaMemcpyHostToDevice, c->stream));
  std::string err;
  if (!radixSortPairs(dk.p, dv.p, (int)n, c->stream, err)) return fail(c, MOX_ERR_CUDA, err);
  CUCK(c, cudaMemcpyAsync(keys, dk.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
  CUCK(c, cudaMemcpyAsync(vals, dv.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
  CUCK(c, cudaStreamSynchronize(c->stream));
  return MOX_OK;
}

extern "C" int mox_debug_read_accel(mox_ctx* c, int which, void* dst, size_t cap, size_t* out_bytes) {
  if (!c) return MOX_ERR_INVALID;
  GROUP_FIRST(c, mox_debug_read_accel(k, which, dst, cap, out_bytes));
  if (!c->built) return fail(c, MOX_ERR_STATE, "debug_read_accel before mox_build_accel");
  const bool wide = c->wideBuilt && c->useWide;
  const BuildOutput& a = c->accel;
  const void* src = nullptr;
  size_t bytes = 0;
  switch (which) {
    case MOX_DEBUG_ACCEL_NODES: src = a.nodes; bytes = (size_t)a.nNodes * sizeof(BvhNode2); break;
    case MOX_DEBUG_ACCEL_NODES8: src = a.nodes8; bytes = wide ? (size_t)a.nNodes8 * sizeof(BvhNode8) : 0; break;
    case MOX_DEBUG_ACCEL_PACKED: src = a.packed; bytes = (size_t)a.nValid * 16 * MOX_PACKED_F4; break;
    case MOX_DEBUG_ACCEL_PACKED8: src = a.packed8; bytes = wide ? (size_t)a.nValid * 16 * MOX_PACKED_F4 : 0; break;
    default: return fail(c, MOX_ERR_INVALID, "unknown acceleration array");
  }
  if (out_bytes) *out_bytes = bytes;
  if (!dst || !bytes) return MOX_OK;
  if (cap < bytes) return fail(c, MOX_ERR_INVALID, "destination too small");
  int rc = bind(c);
  if (rc) return rc;
  CUCK(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
  CUCK(c, cudaStreamSynchronize(c->stream));
  return MOX_OK;
}
