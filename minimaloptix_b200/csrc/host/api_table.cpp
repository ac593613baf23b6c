#include "api_table.h"
#include <dlfcn.h>

bool loadMoxApi(const char* libPath, const char* prefix, MoxApi& api, std::string& err) {
  void* lib = dlopen(libPath, RTLD_NOW | RTLD_LOCAL);
  if (!lib) { err = std::string("dlopen failed: ") + dlerror(); return false; }
  api.lib = lib;
  bool ok = true;
  auto bind = [&](const char* name, void** slot) {
    std::string sym = std::string(prefix) + name;
    *slot = dlsym(lib, sym.c_str());
    if (!*slot) { err += "missing symbol " + sym + "; "; ok = false; }
  };
#define BIND(n) bind(#n, (void**)&api.n)
  BIND(create); BIND(destroy); BIND(last_error); BIND(set_globals); BIND(set_camera); BIND(set_rng_mode);
  BIND(set_partition); BIND(add_texture_rgba32f); BIND(add_sphere); BIND(add_quad); BIND(add_mesh);
  BIND(set_lights); BIND(clear_scene); BIND(build_accel); BIND(launch); BIND(render); BIND(read_accum);
  BIND(clear_accum); BIND(get_stats); BIND(set_accum); BIND(update_sphere);
#undef BIND
  api.create_multi = (int (*)(mox_ctx**, const int*, int))dlsym(lib, (std::string(prefix) + "create_multi").c_str());
  api.read_accum_begin = (int (*)(mox_ctx*))dlsym(lib, (std::string(prefix) + "read_accum_begin").c_str());
  api.read_accum_end = (int (*)(mox_ctx*, const float**))dlsym(lib, (std::string(prefix) + "read_accum_end").c_str());
  api.device_count = (int (*)(const mox_ctx*))dlsym(lib, (std::string(prefix) + "device_count").c_str());
  api.get_device_stats = (int (*)(mox_ctx*, int, mox_stats*))dlsym(lib, (std::string(prefix) + "get_device_stats").c_str());
  api.render_adaptive = (int (*)(mox_ctx*, uint32_t, uint32_t, const mox_adaptive*, uint64_t*))dlsym(lib, (std::string(prefix) + "render_adaptive").c_str());
  api.read_sample_counts = (int (*)(mox_ctx*, uint32_t*))dlsym(lib, (std::string(prefix) + "read_sample_counts").c_str());
  api.set_aovs = (int (*)(mox_ctx*, int))dlsym(lib, (std::string(prefix) + "set_aovs").c_str());
  api.read_aovs = (int (*)(mox_ctx*, float*, float*, float*))dlsym(lib, (std::string(prefix) + "read_aovs").c_str());
  api.denoise = (int (*)(mox_ctx*, const mox_denoise_params*, float*, float*))dlsym(lib, (std::string(prefix) + "denoise").c_str());
  return ok;
}
