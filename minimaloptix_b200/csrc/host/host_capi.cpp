// host_capi.cpp — extern "C" surface of libmox_host.so (include/mox_host.h).
#include <cstdlib>
#include <cstring>
#include <string>

#include "api_table.h"
#include "image_io.h"
#include "mox_host.h"
#include "obj_loader.h"
#include "scene_desc.h"
#include "utils_host.h"

using namespace moxh;

struct moxh_scene { SceneDesc d; };
struct moxh_api { MoxApi t; };

static thread_local std::string g_err;
static int fail(const std::string& e) { g_err = e; return -1; }
static float3 a3(const float* p) { return mk3(p[0], p[1], p[2]); }

static uint64_t fnv1a(const void* data, size_t n) {
  const uint8_t* p = (const uint8_t*)data;
  uint64_t h = 1469598103934665603ull;
  for (size_t i = 0; i < n; ++i) { h ^= p[i]; h *= 1099511628211ull; }
  return h;
}

extern "C" {

const char* moxh_last_error(void) { return g_err.c_str(); }

int moxh_api_load(const char* lib, const char* prefix, moxh_api** out) {
  if (!lib || !prefix || !out) return fail("bad argument");
  moxh_api* a = new moxh_api();
  std::string err;
  if (!loadMoxApi(lib, prefix, a->t, err)) { delete a; return fail(err); }
  *out = a;
  return 0;
}
void moxh_api_free(moxh_api* a) { delete a; }

void moxh_set_quad_params(const float anchor[3], const float v1[3], const float v2[3], QuadParams* out) {
  memset(out, 0, sizeof *out);
  setQuadParams(a3(anchor), a3(v1), a3(v2), *out);
}
void moxh_set_cam_params(const float from[3], const float at[3], const float up[3], float vFoV, float aspect,
                         float aperture, float focus, CamParams* out) {
  setCamParams(a3(from), a3(at), a3(up), vFoV, aspect, aperture, focus, *out);
}
void moxh_init_disney_params(DisneyParams* out) { initDisneyParams(*out); }
int32_t moxh_launch_seed(uint32_t i, uint32_t s) { return launchSeed(i, s); }

int moxh_scene_builtin(const char* kind, uint64_t param, uint64_t seed, moxh_scene** out) {
  if (!kind || !out) return fail("bad argument");
  moxh_scene* s = new moxh_scene();
  std::string k = kind;
  bool ok = false;
  if (k == "spheres_lens") ok = buildSpheres(s->d, false, 0, 0);
  else if (k == "spheres_pinhole") ok = buildSpheres(s->d, true, 0, 0);
  else if (k == "random_spheres") ok = buildRandomSpheres(s->d, param ? (int)param : 256, seed ? (uint32_t)seed : 42u);
  else if (k == "interior") ok = buildInterior(s->d, param ? param : 1000000ull, seed ? (uint32_t)seed : 0xD1A1A6u);
  else if (k == "soup") ok = buildSoup(s->d, param ? param : 10000000ull, seed ? seed : 10000000ull);
  else { delete s; return fail("unknown builtin scene " + k); }
  if (!ok) { delete s; return fail("scene build failed"); }
  *out = s;
  return 0;
}

int moxh_scene_load(const char* dir, const char* name, moxh_scene** out) {
  if (!dir || !name || !out) return fail("bad argument");
  moxh_scene* s = new moxh_scene();
  std::string err;
  if (!loadSceneFile(s->d, dir, name, err)) { delete s; return fail(err); }
  *out = s;
  return 0;
}
void moxh_scene_free(moxh_scene* s) { delete s; }

int moxh_scene_get_info(const moxh_scene* s, moxh_scene_info* o) {
  if (!s || !o) return fail("bad argument");
  memset(o, 0, sizeof *o);
  const SceneDesc& d = s->d;
  o->n_triangles = d.nTriangles; o->n_vertices = d.nVertices;
  o->n_items = (uint32_t)d.items.size(); o->n_meshes = (uint32_t)d.meshes.size();
  for (auto& it : d.items) { if (it.type == Item::SPHERE_ITEM) o->n_spheres++; else if (it.type == Item::QUAD_ITEM) o->n_quads++; }
  o->n_lights = (uint32_t)d.lights.size(); o->n_warnings = (uint32_t)d.warnings.size();
  o->default_width = d.defaultWidth; o->default_height = d.defaultHeight;
  memcpy(o->aabb_min, &d.aabb.lo, 12); memcpy(o->aabb_max, &d.aabb.hi, 12);
  memcpy(o->bg, d.bg, 12);
  memcpy(o->look_from, &d.camera.lookFrom, 12); memcpy(o->look_at, &d.camera.lookAt, 12); memcpy(o->up, &d.camera.up, 12);
  o->vfov = d.camera.vFoV; o->aperture = d.camera.aperture; o->focus = d.camera.focus;
  return 0;
}
const char* moxh_scene_warning(const moxh_scene* s, uint32_t i) {
  return s && i < s->d.warnings.size() ? s->d.warnings[i].c_str() : "";
}
int moxh_scene_cam_params(const moxh_scene* s, uint32_t w, uint32_t h, CamParams* out) {
  if (!s || !out || !w || !h) return fail("bad argument");
  *out = s->d.camParams(w, h);
  return 0;
}
int moxh_scene_light(const moxh_scene* s, uint32_t i, LightParams* out) {
  if (!s || !out || i >= s->d.lights.size()) return fail("bad argument");
  *out = s->d.lights[i];
  return 0;
}
int moxh_scene_mesh_info(const moxh_scene* s, uint32_t mesh, uint64_t* nf, uint64_t* nv, uint64_t* nn, uint64_t* nt,
                         DisneyParams* dp, char* name, size_t nameLen) {
  if (!s || mesh >= s->d.meshes.size()) return fail("bad argument");
  const MeshDesc& m = s->d.meshes[mesh];
  if (nf) *nf = m.faces();
  if (nv) *nv = m.v.size() / 3;
  if (nn) *nn = m.n.size() / 3;
  if (nt) *nt = m.uv.size() / 2;
  if (dp) for (auto& it : s->d.items) if (it.type == Item::MESH_ITEM && it.mesh == (int)mesh && it.mat.kind == MOX_MAT_DISNEY) *dp = it.mat.dis;
  if (name && nameLen) { strncpy(name, m.name.c_str(), nameLen - 1); name[nameLen - 1] = 0; }
  return 0;
}
int moxh_scene_mesh_hash(const moxh_scene* s, uint32_t mesh, uint64_t out4[4]) {
  if (!s || !out4 || mesh >= s->d.meshes.size()) return fail("bad argument");
  const MeshDesc& m = s->d.meshes[mesh];
  out4[0] = fnv1a(m.v.data(), m.v.size() * 4);
  out4[1] = fnv1a(m.n.data(), m.n.size() * 4);
  out4[2] = fnv1a(m.uv.data(), m.uv.size() * 4);
  std::vector<int32_t> idx;
  idx.reserve(m.vi.size() * 3);
  for (size_t i = 0; i < m.vi.size(); ++i) { idx.push_back(m.vi[i]); idx.push_back(m.ni.empty() ? -1 : m.ni[i]); idx.push_back(m.ti.empty() ? -1 : m.ti[i]); }
  out4[3] = fnv1a(idx.data(), idx.size() * 4);
  return 0;
}
int moxh_scene_mesh_data(const moxh_scene* s, uint32_t mesh, const float** v, const int32_t** vi) {
  if (!s || mesh >= s->d.meshes.size()) return fail("bad argument");
  if (v) *v = s->d.meshes[mesh].v.data();
  if (vi) *vi = s->d.meshes[mesh].vi.data();
  return 0;
}

int moxh_scene_upload(const moxh_scene* s, const moxh_api* api, void* ctx, uint32_t w, uint32_t h, uint32_t maxDepth) {
  if (!s || !api || !ctx) return fail("bad argument");
  std::string err;
  if (!uploadScene(s->d, api->t, (mox_ctx*)ctx, w, h, maxDepth, err)) return fail(err);
  return 0;
}

int moxh_scene_animate(moxh_scene* s, float time) {
  if (!s) return fail("bad argument");
  animateSpheres(s->d, time);
  return 0;
}
int moxh_scene_apply_spheres(const moxh_scene* s, const moxh_api* api, void* ctx) {
  if (!s || !api || !ctx) return fail("bad argument");
  std::string err;
  return applySpheres(s->d, api->t, (mox_ctx*)ctx, err) ? 0 : fail(err);
}

void moxh_accum_to_rgb8(const float* accum, uint32_t w, uint32_t h, float n, uint8_t* out) { accumToRgb8(accum, w, h, n, out); }
void moxh_accum_to_rgb8_counts(const float* accum, uint32_t w, uint32_t h, const uint32_t* counts, uint8_t* out) {
  accumToRgb8Counts(accum, w, h, counts, out);
}
int moxh_write_image(const char* path, const uint8_t* rgb, uint32_t w, uint32_t h) {
  std::string err;
  return writeImage(path, rgb, w, h, err) ? 0 : fail(err);
}
int moxh_write_accum(const char* path, const float* accum, uint32_t w, uint32_t h, uint64_t launches) {
  std::string err;
  return writeAccum(path, accum, w, h, launches, err) ? 0 : fail(err);
}
int moxh_read_accum(const char* path, float* accum, uint32_t w, uint32_t h, uint64_t* launches) {
  std::string err;
  return readAccum(path, accum, w, h, launches, err) ? 0 : fail(err);
}
int moxh_read_image(const char* path, int* w, int* h, float** texels) {
  if (!path || !w || !h || !texels) return fail("bad argument");
  std::vector<float> t;
  std::string err;
  if (!readImageRgba(path, *w, *h, t, err)) return fail(err);
  *texels = (float*)malloc(t.size() * sizeof(float));
  if (!*texels) return fail("out of memory");
  memcpy(*texels, t.data(), t.size() * sizeof(float));
  return 0;
}
void moxh_free(void* p) { free(p); }
uint32_t moxh_scene_texture_count(const moxh_scene* s) { return s ? (uint32_t)s->d.textures.size() : 0; }

int moxh_obj_parse_double(const char* text, double* out) {
  return tinyobj::tryParseDouble(text, text + strlen(text), out) ? 1 : 0;
}

}  // extern "C"
