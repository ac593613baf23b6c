// api_table.h — the render-backend function table.  The host side never links a backend; it
// binds the C ABI of include/mox.h at run time (dlopen + dlsym with a symbol prefix), the
// same way a MinimalOptiX maintainer would bind it (INTEGRATION.md).
#pragma once
#include <string>
#include "mox.h"

struct MoxApi {
  void* lib = nullptr;
  int (*create)(mox_ctx**, int) = nullptr;
  void (*destroy)(mox_ctx*) = nullptr;
  const char* (*last_error)(const mox_ctx*) = nullptr;
  int (*set_globals)(mox_ctx*, uint32_t, uint32_t, uint32_t, float, float, const float*, const float*, const float*) = nullptr;
  int (*set_camera)(mox_ctx*, const CamParams*) = nullptr;
  int (*set_rng_mode)(mox_ctx*, int) = nullptr;
  int (*set_partition)(mox_ctx*, uint32_t, uint32_t, uint32_t) = nullptr;
  int (*add_texture_rgba32f)(mox_ctx*, const float*, int, int, int*) = nullptr;
  int (*add_sphere)(mox_ctx*, const SphereParams*, int, const void*, uint32_t*) = nullptr;
  int (*add_quad)(mox_ctx*, const QuadParams*, int, const void*, uint32_t*) = nullptr;
  int (*add_mesh)(mox_ctx*, const float*, size_t, const float*, size_t, const float*, size_t, const int32_t*,
                  const int32_t*, const int32_t*, size_t, int, const void*, uint32_t*) = nullptr;
  int (*set_lights)(mox_ctx*, const LightParams*, size_t) = nullptr;
  int (*clear_scene)(mox_ctx*) = nullptr;
  int (*build_accel)(mox_ctx*, uint32_t, float*) = nullptr;
  int (*launch)(mox_ctx*, int32_t) = nullptr;
  int (*render)(mox_ctx*, uint32_t, uint32_t) = nullptr;
  int (*read_accum)(mox_ctx*, float*) = nullptr;
  int (*clear_accum)(mox_ctx*) = nullptr;
  int (*get_stats)(mox_ctx*, mox_stats*) = nullptr;
  int (*set_accum)(mox_ctx*, const float*, uint64_t) = nullptr;
  int (*update_sphere)(mox_ctx*, uint32_t, const SphereParams*) = nullptr;
  // Optional (not every backend has several devices): null when the library does not export them.
  int (*create_multi)(mox_ctx**, const int*, int) = nullptr;
  int (*read_accum_begin)(mox_ctx*) = nullptr;
  int (*read_accum_end)(mox_ctx*, const float**) = nullptr;
  int (*device_count)(const mox_ctx*) = nullptr;
  int (*get_device_stats)(mox_ctx*, int, mox_stats*) = nullptr;
  int (*render_adaptive)(mox_ctx*, uint32_t, uint32_t, const mox_adaptive*, uint64_t*) = nullptr;
  int (*read_sample_counts)(mox_ctx*, uint32_t*) = nullptr;
  int (*set_aovs)(mox_ctx*, int) = nullptr;
  int (*read_aovs)(mox_ctx*, float*, float*, float*) = nullptr;
  int (*denoise)(mox_ctx*, const mox_denoise_params*, float*, float*) = nullptr;
};

// prefix is "mox_" for the product library.  Returns false and fills err on failure.
bool loadMoxApi(const char* libPath, const char* prefix, MoxApi& api, std::string& err);
