// wavefront.h — device buffers and launchers of the wavefront integrator.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include "gpu_types.h"
#include "traverse_job.h"

// Material queues built by the extend kernel.
enum ShadeQueue { Q_LAMBERT = 0, Q_METAL = 1, Q_DIELECTRIC = 2, Q_DISNEY = 3, Q_COUNT = 4 };

struct PathBuffers {
  size_t capacity = 0;      // paths
  size_t shadowSlots = 0;   // capacity * nLights
  float4 *rayO = nullptr, *rayD = nullptr, *thr = nullptr, *rad = nullptr;
  float2* hit = nullptr;    // (t, primitive id | shade class << 28 | MOX_HIT_MISS | MOX_HIT_DEAD)
  int* state = nullptr;
  uint32_t *qCur = nullptr, *qNext = nullptr;
  uint32_t* qBuf[2] = {nullptr, nullptr};   // queue storage; qCur / qNext point into it
  uint32_t* qMat[Q_COUNT] = {nullptr, nullptr, nullptr, nullptr};
  uint32_t* qDisneyAlt = nullptr;   // second Disney queue: bounce b's k_apply may still read its queue while bounce b+1 is classified
  float4 *shO = nullptr, *shD = nullptr, *shC = nullptr;  // shadow rays: origin per Disney path, (dir, tmax) and contribution per slot
  uint32_t* shQueue = nullptr;                            // slots that need a shadow ray
  uint32_t* counters = nullptr;   // C_WORDS per-batch words (0..7 unused) followed by BOUNCE_RING blocks of C_BOUNCE_WORDS
  int32_t* seeds = nullptr;       // launch seed per sample of the batch
  size_t seedCap = 0;
};

struct LaunchCtx {
  SceneView scene;
  RenderParams rp;
  PathBuffers pb;
  uint32_t* bc;              // this bounce's counter block (C_NEXT, C_MAT0.., C_SHQ)
  const uint32_t* ownedPix;  // device: the pixels this context renders
  uint32_t nOwned;
  float* accu;               // device W*H*3
  bool countTraversal;
  bool brdfFast;             // hardware reciprocal / square-root approximations inside BRDF values (shading.cuh::bdiv)
  cudaStream_t stream;
};

void launchGenerate(const LaunchCtx& c, uint32_t nSamples);
// countPtr (may be null): exact ray count in device memory; `count` is then an upper bound used to size the grid.
void launchExtend(const LaunchCtx& c, const uint32_t* queue, uint32_t count, const uint32_t* countPtr, uint32_t depth);
// The bounce past rayMaxDepth on the wide BVH: the same hit records k_accumulate needs, from the light list tl and an
// any-hit query instead of a closest-hit traversal.  k_classify is not needed after it (it would end every path).
void launchTerminal(const LaunchCtx& c, const uint32_t* queue, uint32_t count, const uint32_t* countPtr, const TerminalLights& tl);
void launchClassify(const LaunchCtx& c, const uint32_t* queue, uint32_t count, const uint32_t* countPtr, uint32_t depth);
void launchShade(const LaunchCtx& c, int kind, uint32_t count, uint32_t depth);
// The shadow traversal and k_apply may run on their own stream, overlapping the next bounce's extend launch.
void launchShadow(const LaunchCtx& c, uint32_t disneyCount, cudaStream_t stream);
void launchApply(const LaunchCtx& c, uint32_t disneyCount, cudaStream_t stream);
void launchAccumulate(const LaunchCtx& c, uint32_t nSamples);

// Adaptive sampling (mox_render_adaptive).  Per pixel, over the samples it received from adaptive renders since the
// last reset: the sum of the luminances y and of y^2 in float64, their number, and the launches the pixel sat out.
struct PixelStats {
  double *s1 = nullptr, *s2 = nullptr;
  uint32_t *n = nullptr, *skipped = nullptr;
};
// The stopping rule: converged when n >= minSpp (at least 2) and sqrt(s^2 / n) < max(rel * mean, abs).
struct AdaptiveRule {
  uint32_t minSpp;
  double rel, abs;
};
// k_accumulate, which also adds each sample's luminance to ps (same image, bit for bit).
void launchAccumulateAdaptive(const LaunchCtx& c, uint32_t nSamples, const PixelStats& ps);
// Words of tile sums launchAdaptiveSelect needs for `count` pixels.
size_t adaptiveSelectTiles(uint32_t count);
// Drops the converged pixels of listIn[0, count), adding `remaining` to their skipped launches, and writes the others
// to listOut in their order; their number goes to *survivors.  tileSums: adaptiveSelectTiles(count) words.  Launches
// nothing for count == 0 (*survivors is then not written).
void launchAdaptiveSelect(const PixelStats& ps, const AdaptiveRule& rule, const uint32_t* listIn, uint32_t count, uint32_t remaining,
                          uint32_t* listOut, uint32_t* tileSums, uint32_t* survivors, cudaStream_t stream);
// First-hit AOV sums (mox_set_aovs), full-frame arrays indexed by pixel: albedo and normal xyz (3 floats per pixel),
// depth, the AOV sample count and the hit count.  36 bytes per pixel.
struct AovBuffers {
  float *albedo = nullptr, *normal = nullptr, *depth = nullptr;
  uint32_t *n = nullptr, *hits = nullptr;
};
// k_aov: adds the record of every camera sample of the batch (depth 1, after k_classify, before any shade kernel) to
// aov, per pixel in launch order.
void launchAov(const LaunchCtx& c, uint32_t nSamples, const AovBuffers& aov);
// Persistent traversal over one batch of rays (closest hit or shadow transmittance).
void launchTraverse(const SceneView& s, const TraceJob& job, bool anyHit, bool count, cudaStream_t stream, bool classify = false);
void launchSplitRays(const float4* rays, float4* o, float4* d, size_t n, cudaStream_t stream);
void launchBuildShadeRecords(const TriIdx* tris, const float* verts, const float* normals, const float* uvs, uint32_t n, float4* out,
                             cudaStream_t stream);
void launchFillOnes(float4* p, size_t n, cudaStream_t stream);
void launchCopyRgb(const float4* src, float* dst, size_t n, cudaStream_t stream);
void launchPackOwned(const float* accu, const uint32_t* ownedPix, uint32_t nOwned, float* dst, cudaStream_t stream);
void launchUnpackOwned(float* accu, const uint32_t* ownedPix, uint32_t nOwned, const float* src, cudaStream_t stream);
// dst[pix] = accu[pix] for the owned pixels; dst may live on another GPU (peer stores over NVLink).
void launchPushOwned(const float* accu, const uint32_t* ownedPix, uint32_t nOwned, float* dstFull, cudaStream_t stream);
