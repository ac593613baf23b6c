/* mox.h — the C ABI of the B200-native render path.
 *
 * This is the drop-in boundary: everything MinimalOptiX does through the OptiX 5.1
 * host API (optixpp Context / Geometry / Material / GeometryInstance / Group /
 * Acceleration / Buffer / launch and the named rtVariables) is reachable through
 * the entry points below, with plain pointers and sizes only.  Each entry point
 * cites the reference call(s) it replaces (paths relative to
 * /root/reference/MinimalOptiX/).
 *
 * Conventions
 *  - every function returns MOX_OK (0) or a negative mox_status; the text of the
 *    last failure is available from mox_last_error().  No C++ exception crosses
 *    the ABI.  (The reference lets optix::Exception / std::logic_error kill the
 *    process, MinimalOptiX.cpp:388,512.)
 *  - all host inputs are copied before the call returns (the reference memcpy()s
 *    into map()ped buffers and setUserData() copies, MinimalOptiX.cpp:398,528).
 *  - a context is not thread-safe; different contexts may be used concurrently.
 *  - mox_launch / mox_render / mox_trace_* are synchronous on return.
 *  - primitive ids are global and dense in insertion order over all mox_add_*
 *    calls (mesh faces in face order).
 *  - there is NO CPU fallback: every compute entry point fails with
 *    MOX_ERR_CUDA when no sm_100-class device is usable.
 */
#ifndef MOX_H
#define MOX_H

#include <stddef.h>
#include <stdint.h>
#include "mox_structs.h"

#ifdef __cplusplus
extern "C" {
#endif

#define MOX_ABI_VERSION 3

typedef struct mox_ctx mox_ctx; /* opaque */

typedef enum mox_status {
  MOX_OK = 0,
  MOX_ERR_INVALID = -1,   /* bad argument / call order */
  MOX_ERR_CUDA = -2,      /* CUDA runtime failure or no usable device */
  MOX_ERR_OOM = -3,       /* device or host allocation failed */
  MOX_ERR_STATE = -4      /* e.g. launch before mox_build_accel */
} mox_status;

/* Which closest-hit program a primitive runs (Material.cu:28,49,72,118,238). */
typedef enum mox_material_kind {
  MOX_MAT_LAMBERTIAN = 0, /* params: LambertianParams */
  MOX_MAT_METAL = 1,      /* params: MetalParams      */
  MOX_MAT_GLASS = 2,      /* params: GlassParams      */
  MOX_MAT_DISNEY = 3,     /* params: DisneyParams     */
  MOX_MAT_LIGHT = 4       /* params: LightParams (only .emission is read) */
} mox_material_kind;

/* Per-path random numbers.  REF reproduces the reference stream exactly
 * (tea<16> seeding + 24-bit LCG, utils_device.h:8-34); PHILOX is Philox4x32-10
 * keyed by (pixel, launch seed) with the draw index as counter. */
typedef enum mox_rng_mode { MOX_RNG_REF = 0, MOX_RNG_PHILOX = 1 } mox_rng_mode;

/* mox_build_accel flags */
#define MOX_ACCEL_DEFAULT 0u
#define MOX_ACCEL_LBVH 1u        /* Karras radix tree instead of PLOC: fastest build, slower rays */
#define MOX_ACCEL_COUNTERS 2u    /* traversal kernels count node visits / prim tests */
#define MOX_ACCEL_BINARY 4u      /* traverse the binary BVH, do not build the compressed 8-wide one */
#define MOX_ACCEL_WATERTIGHT 8u  /* watertight ray-triangle test (Woop, Benthin, Wald 2013) on the raw vertices instead of the
                                    SDK's intersect_triangle (Geometry.cu:133): no ray slips between two triangles that share
                                    an edge or a vertex.  t / beta / gamma then differ from the reference's in the last bits and
                                    the winner can differ on epsilon ties; the oracle has the same switch (also: env
                                    MOX_WATERTIGHT=1 at mox_build_accel, mox_cli --watertight) */
#define MOX_ACCEL_REFIT 16u      /* refit the structure of the last full build in place: same topology, boxes and packed
                                    records from the current vertex, normal and sphere data (what OptiX's Trbvh builder
                                    does for an acceleration marked dirty with the "refit" property).  Needs a successful
                                    full build with no mox_add_* / mox_clear_scene after it (else MOX_ERR_STATE), the other
                                    flag bits equal to that build's, env switches applied (else MOX_ERR_INVALID), and every
                                    primitive still valid or still invalid (zero-area / infinite primitives are not in the
                                    BVH; else MOX_ERR_STATE and the context is not built: build again without this flag).
                                    Unchanged geometry gives node and primitive arrays byte-identical to the full build's.
                                    Tree quality falls as the geometry moves away from the built pose: rebuild now and then */

typedef struct mox_stats {
  uint64_t rays_primary;      /* camera rays traced (closest hit)                 */
  uint64_t rays_bounce;       /* scattered rays traced (closest hit)              */
  uint64_t rays_shadow;       /* NEE shadow rays traced (any hit)                 */
  uint64_t nonfinite_samples; /* samples that were NaN/Inf before the clamp       */
  uint64_t launches;          /* launches since the last clear                    */
  uint64_t node_visits;       /* only with MOX_ACCEL_COUNTERS                     */
  uint64_t prim_tests;        /* only with MOX_ACCEL_COUNTERS                     */
  double ms_render;           /* device time in launch/render since last clear    */
  double ms_build;            /* device time of the last mox_build_accel          */
  uint32_t n_prims, n_triangles, n_spheres, n_quads;
  uint32_t n_nodes;           /* nodes of the acceleration structure traversed    */
  uint32_t node_bytes;        /* bytes per node record                            */
  uint32_t prim_bytes;        /* bytes per packed triangle record                 */
  uint32_t n_lights;
  /* per-stage device time (CUDA events on the launching stream) and launch counts since the last clear */
  double ms_generate, ms_extend, ms_shade, ms_shadow, ms_accumulate;
  uint64_t extend_launches;   /* closest-hit traversal kernel launches                   */
  uint64_t kernel_launches;   /* all kernels this library launched for launch/render     */
  uint64_t node_visits_shadow; /* shadow-ray traversal, only with MOX_ACCEL_COUNTERS      */
  uint64_t prim_tests_shadow;
  uint64_t rays_shadow_traced; /* shadow rays with a non-zero contribution (the ones traversed) */
  /* traversed shadow rays that touched their 16-byte contribution record: blocked (one store) or tinted by
   * Disney GLASS (load + store); the others finish without a write.  Only with MOX_ACCEL_COUNTERS. */
  uint64_t rays_shadow_blocked, rays_shadow_tinted;
  /* per path depth d = 1 (camera rays) .. MOX_STATS_DEPTHS-1 (deeper bounces are added to the last entry; entry 0
   * is unused): closest-hit rays traced, shadow rays traversed, and the device time of the two traversal launches */
#define MOX_STATS_DEPTHS 8
  uint64_t rays_depth[MOX_STATS_DEPTHS], shadow_traced_depth[MOX_STATS_DEPTHS];
  double ms_extend_depth[MOX_STATS_DEPTHS], ms_shadow_depth[MOX_STATS_DEPTHS];
} mox_stats;

/* ---- context ------------------------------------------------------------- */

/* Context::create + setRayTypeCount(2)/setEntryPointCount(1)
 * (MinimalOptiX.cpp:130-134).  device_id is the CUDA ordinal of the ONE GPU this
 * context renders on; multi-GPU runs use one context per GPU (one process per
 * GPU) with mox_set_partition. */
int mox_create(mox_ctx** out, int device_id);
void mox_destroy(mox_ctx*);
const char* mox_last_error(const mox_ctx*); /* ctx may be NULL: last create error */
int mox_abi_version(void);

/* The context-level rtVariables rayMaxDepth, rayEpsilonT, rayMinIntensity,
 * absorbColor, badColor (MinimalOptiX.cpp:136-151), the miss program's bgColor
 * (:163-165) and the launch size / accuBuffer dimensions (:144-147, :546).
 * (Re)allocates and zeroes the accumulation buffer when the size changes. */
int mox_set_globals(mox_ctx*, uint32_t width, uint32_t height, uint32_t rayMaxDepth,
                    float rayEpsilonT, float rayMinIntensity, const float absorbColor[3],
                    const float badColor[3], const float bgColor[3]);

/* rayGenProgram["camParams"]->setUserData (MinimalOptiX.cpp:255). */
int mox_set_camera(mox_ctx*, const CamParams*);

int mox_set_rng_mode(mox_ctx*, int mode /* mox_rng_mode */);

/* Tile split for multi-GPU: the image is cut into tile x tile pixel squares and
 * this context renders those with (tx + ty) % world == rank.  Seeds depend only
 * on the global pixel index, so the union over ranks equals the 1-rank image
 * bit for bit.  Default: rank 0 of world 1 (whole image), tile 32. */
int mox_set_partition(mox_ctx*, uint32_t rank, uint32_t world, uint32_t tile);

/* ---- scene --------------------------------------------------------------- */

/* createTextureSampler + float4 buffer, REPEAT / LINEAR / normalized
 * (MinimalOptiX.cpp:445-474).  texels: w*h RGBA float, row 0 = bottom.
 * Ids start at 1; 0 == RT_TEXTURE_ID_NULL. */
int mox_add_texture_rgba32f(mox_ctx*, const float* texels, int w, int h, int* out_id);

/* createGeometry(sphere|quad) + createMaterial + createGeometryInstance
 * (MinimalOptiX.cpp:174-240, 495-518).  *out_prim_id (may be NULL) receives the
 * global primitive id. */
int mox_add_sphere(mox_ctx*, const SphereParams*, int material_kind, const void* material_params,
                   uint32_t* out_prim_id);
int mox_add_quad(mox_ctx*, const QuadParams*, int material_kind, const void* material_params,
                 uint32_t* out_prim_id);

/* One OBJ shape: vertexBuffer / normalBuffer / texcoordBuffer and the three int3
 * index buffers (MinimalOptiX.cpp:392-441).  n_normals / n_texcoords may be 0
 * (then nIdx / tIdx may be NULL).  *out_first_prim_id: id of face 0. */
int mox_add_mesh(mox_ctx*, const float* vertices, size_t n_vertices, const float* normals,
                 size_t n_normals, const float* texcoords, size_t n_texcoords,
                 const int32_t* vIdx, const int32_t* nIdx, const int32_t* tIdx, size_t n_faces,
                 int material_kind, const void* material_params, uint32_t* out_first_prim_id);

/* videoParams.spheres[i]["sphereParams"]->setUserData (MinimalOptiX.cpp:762-764): move / resize a
 * sphere added earlier.  The acceleration structure must be rebuilt (mox_build_accel) before the
 * next launch. */
int mox_update_sphere(mox_ctx*, uint32_t prim_id, const SphereParams*);

/* vertexBuffer / normalBuffer->map(), write, unmap() and acceleration->markDirty() for one OBJ shape
 * (MinimalOptiX.cpp:398-411,441): new vertices (and, when normals is not NULL, normals) for the mesh whose face 0 is
 * first_prim_id (the id mox_add_mesh returned).  n_vertices must equal the count the mesh was added with; normals
 * need a mesh added with normals and their count.  Faces, indices and texcoords do not change.  The acceleration
 * structure must be rebuilt or refitted (mox_build_accel, MOX_ACCEL_REFIT) before the next launch or trace. */
int mox_update_mesh(mox_ctx*, uint32_t first_prim_id, const float* vertices, size_t n_vertices, const float* normals,
                    size_t n_normals);

/* context["lights"] buffer used by the Disney NEE loop (MinimalOptiX.cpp:523-531,
 * Material.cu:116,172). */
int mox_set_lights(mox_ctx*, const LightParams*, size_t n);

/* Drop all geometry, materials, lights and the acceleration structure. */
int mox_clear_scene(mox_ctx*);

/* The moment OptiX builds Trbvh (context->validate() + first launch,
 * MinimalOptiX.cpp:378,494,534,542): uploads the scene and builds the BVH on
 * the GPU.  *out_build_ms (may be NULL): device time of the build kernels (with
 * MOX_ACCEL_REFIT: of the refit kernels). */
int mox_build_accel(mox_ctx*, uint32_t flags, float* out_build_ms);

/* ---- render -------------------------------------------------------------- */

/* context["randSeed"]->setInt(seed); context->launch(0, W, H)
 * (MinimalOptiX.cpp:545-546): adds one sample per (owned) pixel to the
 * accumulation buffer. */
int mox_launch(mox_ctx*, int32_t randSeed);

/* The spp loop of renderScene (MinimalOptiX.cpp:544-554) with a FIXED seed
 * schedule instead of std::random_device: launch k (counted from the last
 * clear) uses randSeed = (int32) tea<16>(k, seed).  Samples may be batched into
 * one wavefront; the result is bit-identical to spp calls of mox_launch. */
int mox_render(mox_ctx*, uint32_t spp, uint32_t seed);

/* Adaptive sampling: mox_render's launches for the pixels whose estimated error is still above a threshold.
 *
 * The call covers launches st.launches .. st.launches + spp - 1 of mox_render's seed schedule, and advances
 * mox_stats.launches by spp even when every pixel has stopped.  A pixel's estimate uses only the samples it received
 * from mox_render_adaptive since the last mox_clear_accum / mox_set_accum / size change; n is their number.  Each
 * sample adds y = 0.2126 r + 0.7152 g + 0.0722 b (float32, in that order) of the colour the accumulation buffer
 * receives (the clamped sample, or badColor for a non-finite one); S1 = sum y and S2 = sum y^2 are float64, in launch
 * order.  With m = S1 / n, s^2 = max(0, (S2 - S1 m) / (n - 1)) and err = sqrt(s^2 / n), a pixel has converged when
 * n >= max(min_spp, 2) and err < max(rel_error * m, abs_error) (strict: thresholds of 0 never stop a pixel).
 *
 * At the start of the call every owned pixel is checked; the active ones are rendered in rounds of round_spp
 * launches (the last may be shorter) and checked after each round.  A pixel that has converged gets no further
 * sample in this call; when none is left, the remaining launches run no kernel.  So a pixel that took k samples holds
 * exactly what k launches of mox_render would have left in it.  *out_samples (may be NULL): pixel-samples traced.
 * The first call allocates 24 bytes per pixel of statistics.  MOX_ERR_INVALID: null params, round_spp == 0, or a
 * negative or non-finite threshold; MOX_ERR_STATE: as mox_render.  On a multi-GPU handle every device runs the
 * rounds on its own tiles and finishes when they have converged. */
typedef struct mox_adaptive {
  uint32_t round_spp; /* launches between two convergence checks, >= 1 */
  uint32_t min_spp;   /* adaptive samples a pixel needs before it may stop */
  float rel_error;    /* stop when err < max(rel_error * mean, abs_error); both finite, >= 0 */
  float abs_error;
} mox_adaptive;
int mox_render_adaptive(mox_ctx*, uint32_t spp, uint32_t seed, const mox_adaptive* params, uint64_t* out_samples);
/* Samples per pixel (W*H, row 0 = bottom): mox_stats.launches minus the launches the pixel sat out in
 * mox_render_adaptive; 0 for pixels of other ranks.  Divide the accumulation buffer by it to get the image. */
int mox_read_sample_counts(mox_ctx*, uint32_t* dst);

/* accuBuffer map()/unmap() (MinimalOptiX.cpp:44,60): W*H*3 floats, row 0 =
 * bottom of the image, un-normalised sums.  Pixels of other ranks are 0. */
int mox_read_accum(mox_ctx*, float* dst_rgb);
/* The map()/unmap() form itself: *out points at a pinned host copy of the accumulation buffer
 * (W*H*3 floats, valid until the next mox_map_accum / mox_read_accum / mox_destroy); no second
 * host copy is made.  mox_unmap_accum is a no-op kept for symmetry with the reference. */
int mox_map_accum(mox_ctx*, const float** out);
int mox_unmap_accum(mox_ctx*);
int mox_clear_accum(mox_ctx*);
/* Resume: load a previously read accumulation buffer (W*H*3 floats) and continue the seed schedule
 * of mox_render at launch index `launches` (the reference has snapshots but no reload,
 * MinimalOptiX.cpp:543-558; this is the "dump/resume" row of SURVEY.md §8 f-2). */
int mox_set_accum(mox_ctx*, const float* src_rgb, uint64_t launches);

/* ---- first-hit AOVs and the denoiser --------------------------------------- */

/* AOVs ("arbitrary output variables"): per-pixel buffers besides the colour.  mox_set_aovs(ctx, 1) allocates and
 * zeroes 36 bytes per pixel of sums on the device; from then on every camera sample that mox_launch, mox_render or
 * mox_render_adaptive traces adds one record, taken at the closest hit of its depth-1 ray:
 *   albedo  Lambertian, metal, glass: albedo; Disney: the base colour (texture or color, not linearised); light:
 *           emission clamped to [0, 1]; miss: bgColor clamped to [0, 1]
 *   normal  the shading normal turned towards the viewer, faceforward(Ns, -d, Ng); 0 for a miss
 *   depth   the ray's t, counted for hits only
 * The AOVs keep their own sample and hit counts per pixel, so they may be switched on after some samples.  The sums
 * are reset by mox_clear_accum, mox_set_accum and a size change in mox_set_globals; mox_set_aovs(ctx, 0) frees them.
 * The image itself does not change: with AOVs on or off the accumulation buffer, the sample counts and the ray counts
 * are bit-identical.  On a multi-GPU handle the switch is replicated to every device. */
int mox_set_aovs(mox_ctx*, int enable);
/* The per-pixel means, W*H*k floats with row 0 = bottom (k = 3, 3, 1); any pointer may be NULL.  Each mean is one
 * float32 division of the sum by its count: albedo and normal by the AOV sample count, depth by the hit count.  A pixel
 * without a sample, and the depth of a pixel without a hit, read 0.  These are exactly the guides mox_denoise uses.
 * On a multi-GPU handle: the sum over the devices (each pixel is non-zero on its owner only).  MOX_ERR_STATE: AOVs off. */
int mox_read_aovs(mox_ctx*, float* albedo_rgb, float* normal_xyz, float* depth);

/* Edge-avoiding a-trous wavelet filter (Dammertz, Hanika, Keller 2010) of the mean colour, guided by the AOVs.
 *
 * c_p = accum_p / n_p is the mean colour (n_p from mox_read_sample_counts, so adaptive renders work; 0 where n_p = 0),
 * a, N, z are the AOV means of mox_read_aovs.  All arithmetic is float32, evaluated in the order written, without
 * fused multiply-adds:
 *   e0_p      = c_p / (a_p + 0.001)                                          per channel (demodulation)
 *   for i = 0 .. K-1, with step s = 2^i and sigma_i = sigma_color * 2^-i:
 *   e(i+1)_p  = sum_q h(dx) h(dy) w_pq e(i)_q / sum_q h(dx) h(dy) w_pq,  q = p + s (dx, dy)
 *               dy = -2..2 in the outer loop, dx = -2..2 in the inner one; taps outside the image are skipped
 *               (not clamped); h = (1/16, 1/4, 3/8, 1/4, 1/16); each sum adds h(dx) h(dy) w_pq (and its product
 *               with e(i)_q) in tap order
 *   w_pq      = exp(-(|e(i)_p - e(i)_q|^2 / sigma_i^2 + max(0, 1 - N_p . N_q) / sigma_normal
 *                     + |z_p - z_q| / (sigma_depth * max(z_p, z_q) + 1e-30)))
 *               with |v|^2 = (x*x + y*y) + z*z, N_p . N_q = (x*x' + y*y') + z*z', sigma_i^2 = sigma_i * sigma_i; the
 *               centre tap has w = 1; two misses (z = 0) compare as equal depth
 *   out_p     = e(K)_p * (a_p + 0.001)                                       (remodulation)
 *
 * dst_rgb: W*H*3 floats, row 0 = bottom.  params == NULL selects the defaults MOX_DENOISE_DEFAULT_*.  *out_ms (may be
 * NULL): device time of the denoise kernels (CUDA events).  Two calls on the same state give bit-identical results.
 * MOX_ERR_INVALID: iterations outside 1..10, or a sigma that is not finite and > 0.  MOX_ERR_STATE: AOVs off, no
 * camera sample rendered with AOVs on since the last reset (a buffer loaded by mox_set_accum alone has no guides), or a
 * context with mox_set_partition world > 1 (the filter needs the whole frame; a mox_create_multi handle gathers it into
 * device 0 and filters there). */
typedef struct mox_denoise_params {
  uint32_t iterations;   /* 1 .. 10 */
  float sigma_color;     /* colour (irradiance) edge stop of iteration 0; halved every iteration */
  float sigma_normal;    /* normal edge stop */
  float sigma_depth;     /* depth edge stop, relative to the larger depth */
} mox_denoise_params;
#define MOX_DENOISE_DEFAULT_ITERATIONS 5
#define MOX_DENOISE_DEFAULT_SIGMA_COLOR 1.0f
#define MOX_DENOISE_DEFAULT_SIGMA_NORMAL 0.5f
#define MOX_DENOISE_DEFAULT_SIGMA_DEPTH 0.05f
int mox_denoise(mox_ctx*, const mox_denoise_params* params, float* dst_rgb, float* out_ms);

/* Multi-GPU gather plumbing (device pointers on this context's GPU).
 * mox_owned_pixels: number of pixels rank `rank` of the current partition owns.
 * mox_pack_owned: copy this rank's owned pixels (tile order) to dev_dst
 *   (3 floats per pixel).
 * mox_unpack_owned: scatter a packed buffer produced by `rank` into this
 *   context's full accumulation buffer (overwrites those pixels). */
int mox_owned_pixels(mox_ctx*, uint32_t rank, uint64_t* out_n);
int mox_pack_owned(mox_ctx*, void* dev_dst);
int mox_unpack_owned(mox_ctx*, uint32_t rank, const void* dev_src);

int mox_get_stats(mox_ctx*, mox_stats*);

/* ---- multi-GPU inside the library ------------------------------------------ */

/* One handle that renders on several GPUs of this process (the reference has a single
 * optix::Context on one device, MinimalOptiX.cpp:131; OptiX itself would take
 * context->setDevices()).  The scene calls are replicated to every device, the image is
 * tile-split (rank i of n, mox_set_partition), build and launch run one host thread per
 * device, and a read-back gathers the tiles over NVLink: every device writes the pixels it
 * owns DIRECTLY into device 0's gather buffer (peer stores, no staging, no collective).
 * Every other entry point of this header works on the returned handle unchanged;
 * mox_set_partition / mox_owned_pixels / mox_pack_owned / mox_unpack_owned are refused.
 * n_devices == 1 is allowed. */
int mox_create_multi(mox_ctx** out, const int* device_ids, int n_devices);
int mox_device_count(const mox_ctx*);   /* 1 for a plain context */
/* mox_get_stats of device `index` (0 .. mox_device_count-1) of a multi-GPU handle alone — mox_get_stats on the handle
 * sums the counts and takes the slowest device's times; per-device render times show the balance of the tile split. */
int mox_get_device_stats(mox_ctx*, int index, mox_stats* out);

/* Asynchronous accuBuffer->map(): _begin snapshots the accumulation buffer (for a multi-GPU
 * handle: gathers the tiles) and starts the device->host copy on a copy stream; rendering
 * may continue.  _end waits for that copy; *out (W*H*3 floats, row 0 = bottom) stays valid
 * until the second next _begin (two buffers alternate).  mox_read_accum / mox_map_accum are
 * _begin + _end. */
int mox_read_accum_begin(mox_ctx*);
int mox_read_accum_end(mox_ctx*, const float** out);

/* Cross-process tile exchange over peer memory (one process per GPU, e.g. under torchrun):
 * rank 0 exports its two gather buffers as CUDA IPC handles (64 bytes each), the other
 * ranks import them once; per frame every rank — rank 0 included — pushes the pixels it
 * owns into buffer `which` with direct NVLink stores (synchronous on return), the caller
 * runs a barrier, and rank 0 reads the frame with mox_read_gathered_begin/_end. */
#define MOX_IPC_HANDLE_BYTES 64
int mox_gather_export(mox_ctx*, int which, void* handle_out);
int mox_gather_import(mox_ctx*, int which, const void* handle);
int mox_gather_push(mox_ctx*, int which);
int mox_read_gathered_begin(mox_ctx*, int which);
int mox_read_gathered_end(mox_ctx*, int which, const float** out);

/* ---- raw ray queries (BASELINE config 5, primitive-id parity) -------------- */

/* Closest hit for n rays.  rays: n x 8 floats (ox oy oz tmin dx dy dz tmax).
 * hits: n x 4 x 32 bit: (float t, int32 prim id or -1, float beta, float gamma).
 * Host-pointer and device-pointer variants; the device variant is what the
 * resident benchmark times (*out_ms, may be NULL, is the kernel time). */
int mox_trace_closest(mox_ctx*, const float* rays, size_t n, void* hits);
int mox_trace_closest_device(mox_ctx*, const void* dev_rays, size_t n, void* dev_hits,
                             float* out_ms);
/* Shadow-ray transmittance (row a-11): out: n x 3 floats. */
int mox_trace_shadow(mox_ctx*, const float* rays, size_t n, float* out_rgb);

#ifdef __cplusplus
}
#endif
#endif /* MOX_H */
