// oracle/refit.cpp — TEST INFRASTRUCTURE.  The oracle's side of mox_update_mesh and MOX_ACCEL_REFIT (include/mox.h).
//
// liboracle.so is built from this file: it compiles oracle.cpp unchanged and wraps the entry points whose contract
// the refit extends.  The wrapped functions keep their behaviour; the wrappers only track what a refit must find
// again — per mesh its first primitive and vertex / normal ranges, the flags and per-primitive validity of the last
// full build.  The oracle's refit is a rebuild: its results do not depend on the shape of its tree.
//
// oracle.cpp is written as a main file; included here, GCC would flag its orc_ctx fields of anonymous-namespace types,
// which are fine in a single translation unit.
#pragma GCC diagnostic ignored "-Wsubobject-linkage"
#define orc_destroy orc_destroy_base
#define orc_add_sphere orc_add_sphere_base
#define orc_add_quad orc_add_quad_base
#define orc_add_mesh orc_add_mesh_base
#define orc_clear_scene orc_clear_scene_base
#define orc_build_accel orc_build_accel_base
#include "oracle.cpp"
#undef orc_destroy
#undef orc_add_sphere
#undef orc_add_quad
#undef orc_add_mesh
#undef orc_clear_scene
#undef orc_build_accel

#include <map>
#include <mutex>

namespace {

struct MeshRec { uint32_t firstPrim, nFaces; size_t vBase, nV, nBase, nN; };  // in vertices, not floats
struct RefitInfo {
  std::vector<MeshRec> meshes;
  bool refitOk = false;          // a full build succeeded and no primitive was added or removed since
  uint32_t builtFlags = 0;       // flags of that build
  std::vector<char> builtValid;  // primBox(...).valid per primitive at that build
};

std::mutex g_refitMutex;
std::map<const orc_ctx*, RefitInfo> g_refit;   // node-based: an entry stays put while others come and go

RefitInfo& refitInfo(const orc_ctx* c) {
  std::lock_guard<std::mutex> lock(g_refitMutex);
  return g_refit[c];
}

}  // namespace

extern "C" {

int orc_update_mesh(orc_ctx*, uint32_t first_prim_id, const float* vertices, size_t n_vertices, const float* normals,
                    size_t n_normals);

void orc_destroy(orc_ctx* c) {
  {
    std::lock_guard<std::mutex> lock(g_refitMutex);
    g_refit.erase(c);
  }
  orc_destroy_base(c);
}

int orc_add_sphere(orc_ctx* c, const SphereParams* s, int kind, const void* params, uint32_t* out_id) {
  if (c) refitInfo(c).refitOk = false;
  return orc_add_sphere_base(c, s, kind, params, out_id);
}

int orc_add_quad(orc_ctx* c, const QuadParams* q, int kind, const void* params, uint32_t* out_id) {
  if (c) refitInfo(c).refitOk = false;
  return orc_add_quad_base(c, q, kind, params, out_id);
}

int orc_add_mesh(orc_ctx* c, const float* v, size_t nv, const float* n, size_t nn, const float* uv, size_t nt,
                 const int32_t* vIdx, const int32_t* nIdx, const int32_t* tIdx, size_t nFaces, int kind,
                 const void* params, uint32_t* out_first) {
  if (!c) return orc_add_mesh_base(c, v, nv, n, nn, uv, nt, vIdx, nIdx, tIdx, nFaces, kind, params, out_first);
  const size_t vb = c->verts.size(), nb = c->normals.size();
  const uint32_t first = (uint32_t)c->prims.size();
  const int rc = orc_add_mesh_base(c, v, nv, n, nn, uv, nt, vIdx, nIdx, tIdx, nFaces, kind, params, out_first);
  RefitInfo& r = refitInfo(c);
  r.refitOk = false;
  if (rc == MOX_OK) r.meshes.push_back({first, (uint32_t)nFaces, vb, c->verts.size() - vb, nb, c->normals.size() - nb});
  return rc;
}

int orc_clear_scene(orc_ctx* c) {
  const int rc = orc_clear_scene_base(c);
  if (c) {
    RefitInfo& r = refitInfo(c);
    r.meshes.clear();
    r.refitOk = false;
  }
  return rc;
}

int orc_build_accel(orc_ctx* c, uint32_t flags, float* out_ms) {
  if (!c) return MOX_ERR_INVALID;
  RefitInfo& r = refitInfo(c);
  const bool refit = (flags & MOX_ACCEL_REFIT) != 0;
  flags &= ~MOX_ACCEL_REFIT;
  std::vector<char> valid(c->prims.size());
  for (size_t i = 0; i < c->prims.size(); ++i) valid[i] = primBox(*c, c->prims[i]).valid ? 1 : 0;
  if (refit) {   // the preconditions of MOX_ACCEL_REFIT in mox.h
    if (!r.refitOk) { c->err = "MOX_ACCEL_REFIT needs a successful full build with no add / clear after it"; return MOX_ERR_STATE; }
    if (flags != r.builtFlags) { c->err = "MOX_ACCEL_REFIT: the other flags differ from those of the last full build"; return MOX_ERR_INVALID; }
    if (valid != r.builtValid) {
      c->built = false;
      r.refitOk = false;
      c->err = "MOX_ACCEL_REFIT: a primitive's validity changed since the last full build; build without MOX_ACCEL_REFIT";
      return MOX_ERR_STATE;
    }
  }
  r.refitOk = false;
  const int rc = orc_build_accel_base(c, flags, out_ms);
  if (rc == MOX_OK) {
    r.refitOk = true;
    r.builtFlags = flags;
    r.builtValid.swap(valid);
  }
  return rc;
}

int orc_update_mesh(orc_ctx* c, uint32_t first, const float* v, size_t nv, const float* n, size_t nn) {
  if (!c) return MOX_ERR_INVALID;
  const RefitInfo& r = refitInfo(c);
  auto it = std::lower_bound(r.meshes.begin(), r.meshes.end(), first, [](const MeshRec& m, uint32_t id) { return m.firstPrim < id; });
  while (it != r.meshes.end() && it + 1 != r.meshes.end() && (it + 1)->firstPrim == first && it->nFaces == 0) ++it;  // skip empty meshes
  if (it == r.meshes.end() || it->firstPrim != first) { c->err = "not the first primitive id of a mesh"; return MOX_ERR_INVALID; }
  if (nv != it->nV || (nv && !v)) { c->err = "vertex count differs from the one the mesh was added with"; return MOX_ERR_INVALID; }
  if (n && (it->nN == 0 || nn != it->nN)) { c->err = "normal count differs from the one the mesh was added with"; return MOX_ERR_INVALID; }
  for (size_t i = 0; i < nv; ++i) c->verts[it->vBase + i] = {v[3 * i], v[3 * i + 1], v[3 * i + 2]};
  if (n) for (size_t i = 0; i < nn; ++i) c->normals[it->nBase + i] = {n[3 * i], n[3 * i + 1], n[3 * i + 2]};
  c->built = false;
  return MOX_OK;
}

}  // extern "C"
