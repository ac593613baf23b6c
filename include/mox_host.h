/* mox_host.h — C ABI of the host side (libmox_host.so): scene description loader, parameter
 * builders, scene builders, image output.  This is the headless replacement of the parts of
 * MinimalOptiX::{setupScene, renderScene, updateContent, saveCurrentFrame} that are not GPU
 * work (MinimalOptiX.cpp:43-84, 154-560).  It binds a render backend through the function
 * table of include/mox.h (see moxh_api_load) and never links one.
 */
#ifndef MOX_HOST_H
#define MOX_HOST_H
#include <stddef.h>
#include <stdint.h>
#include "mox.h"
#ifdef __cplusplus
extern "C" {
#endif

typedef struct moxh_scene moxh_scene; /* opaque flattened scene */
typedef struct moxh_api moxh_api;     /* opaque bound backend (function table) */

const char* moxh_last_error(void);

/* dlopen(lib_path) and bind <prefix>create, <prefix>add_mesh, ... (prefix "mox_"). */
int moxh_api_load(const char* lib_path, const char* prefix, moxh_api** out);
void moxh_api_free(moxh_api*);

/* Parameter builders with the reference's semantics (utils_host.cpp:67-116). */
void moxh_set_quad_params(const float anchor[3], const float v1[3], const float v2[3], QuadParams* out);
void moxh_set_cam_params(const float lookFrom[3], const float lookAt[3], const float up[3], float vFoV,
                         float aspect, float aperture, float focus, CamParams* out);
void moxh_init_disney_params(DisneyParams* out);
int32_t moxh_launch_seed(uint32_t launch_index, uint32_t user_seed);

/* Scene builders.  kind: "spheres_lens" | "spheres_pinhole" | "random_spheres" | "interior" |
 * "soup".  param: interior/soup = triangle count; random_spheres = sphere count (0 -> 256).
 * seed: generator seed (0 -> the documented default of that scene). */
int moxh_scene_builtin(const char* kind, uint64_t param, uint64_t seed, moxh_scene** out);
/* setupScene(name): loads <scene_dir>/<name>.scene and the OBJ files it names. */
int moxh_scene_load(const char* scene_dir, const char* name, moxh_scene** out);
void moxh_scene_free(moxh_scene*);

typedef struct moxh_scene_info {
  uint64_t n_triangles, n_vertices;
  uint32_t n_items, n_meshes, n_spheres, n_quads, n_lights, n_warnings;
  uint32_t default_width, default_height;
  float aabb_min[3], aabb_max[3];
  float bg[3];
  float look_from[3], look_at[3], up[3];
  float vfov, aperture, focus;
} moxh_scene_info;
int moxh_scene_get_info(const moxh_scene*, moxh_scene_info* out);
const char* moxh_scene_warning(const moxh_scene*, uint32_t i);
int moxh_scene_cam_params(const moxh_scene*, uint32_t width, uint32_t height, CamParams* out);
/* Copy of light i of the NEE buffer / disney params of mesh item i (loader parity tests). */
int moxh_scene_light(const moxh_scene*, uint32_t i, LightParams* out);
int moxh_scene_mesh_info(const moxh_scene*, uint32_t mesh, uint64_t* n_faces, uint64_t* n_vertices,
                         uint64_t* n_normals, uint64_t* n_texcoords, DisneyParams* disney_or_null,
                         char* name_buf, size_t name_len);
/* FNV-1a 64 over the raw bytes of vertices / normals / texcoords / indices of a mesh. */
int moxh_scene_mesh_hash(const moxh_scene*, uint32_t mesh, uint64_t out4[4]);
/* Raw pointers into mesh storage (valid until moxh_scene_free). */
int moxh_scene_mesh_data(const moxh_scene*, uint32_t mesh, const float** v, const int32_t** vi);

/* Push the scene through the bound backend: set_globals / set_camera / add_* in primitive-id
 * order / set_lights.  ctx is the backend's context. */
int moxh_scene_upload(const moxh_scene*, const moxh_api*, void* ctx, uint32_t width, uint32_t height,
                      uint32_t max_depth);

/* Bouncing-sphere animation (MinimalOptiX::animate, MinimalOptiX.cpp:562-590): advance the sphere
 * items by `time` seconds, then push the new SphereParams through <prefix>update_sphere.  The caller
 * rebuilds the acceleration structure (mox_build_accel) before the next launch. */
int moxh_scene_animate(moxh_scene*, float time);
int moxh_scene_apply_spheres(const moxh_scene*, const moxh_api*, void* ctx);

/* updateContent (MinimalOptiX.cpp:43-66): out[H-1-i][j] = quantise(clamp(accu[i][j] / n, 0, 1)),
 * quantise(v) = round(v * 65535) >> 8 (QColor::setRedF -> RGB888).  out: W*H*3 bytes, row 0 = top. */
void moxh_accum_to_rgb8(const float* accum, uint32_t width, uint32_t height, float n_accum, uint8_t* out);
/* The same with a sample count per pixel (mox_read_sample_counts: W*H, row 0 = bottom) in place of n_accum, for
 * images of mox_render_adaptive.  A count of 0 gives black. */
void moxh_accum_to_rgb8_counts(const float* accum, uint32_t width, uint32_t height, const uint32_t* counts, uint8_t* out);
/* saveCurrentFrame: PNG (RGB8, stored deflate) or binary PPM by extension. */
int moxh_write_image(const char* path, const uint8_t* rgb, uint32_t width, uint32_t height);
/* Raw float accumulator dump / load (resume + parity artefact): magic "MOXA", W, H, launches. */
int moxh_write_accum(const char* path, const float* accum, uint32_t width, uint32_t height, uint64_t launches);
int moxh_read_accum(const char* path, float* accum, uint32_t width, uint32_t height, uint64_t* launches);

/* Texture image decoding as the loader does it (PNG 8-bit non-interlaced, binary PPM/PGM, PFM):
 * RGBA float texels, row 0 = bottom, alpha 1 (QImage::pixelColor -> redF(), MinimalOptiX.cpp:459-470).
 * *texels is malloc()ed; release with moxh_free. */
int moxh_read_image(const char* path, int* w, int* h, float** texels);
void moxh_free(void*);
uint32_t moxh_scene_texture_count(const moxh_scene*);

/* The OBJ reader on its own (loader parity tests). */
int moxh_obj_parse_double(const char* text, double* out);

#ifdef __cplusplus
}
#endif
#endif
