// cli_main.cpp — headless driver: the replacement of the Qt application
// (MinimalOptiX::MinimalOptiX / renderScene / imageDemo, MinimalOptiX.cpp:9-33, 86-111,
// 540-560).  Loads libmox.so (the GPU library; there is no other backend for the product),
// uploads a scene, renders spp samples with the power-of-two snapshot schedule of
// renderScene(autoSave=true) and writes PNGs plus a JSON stats line.
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "api_table.h"
#include "mox_host.h"
#include "scene_desc.h"

static void usage() {
  fprintf(stderr,
          "usage: mox_cli --scene NAME [--scene-dir DIR] [--width W --height H] [--spp N] [--max-depth D]\n"
          "               [--seed S] [--rng ref|philox] [--out PREFIX] [--snapshots] [--dump-accum] [--resume FILE.moxa] [--device K | --gpus N]\n"
          "               [--param P] [--lib PATH] [--watertight] [--adaptive REL[,ABS] [--adaptive-min N] [--adaptive-round N]]\n"
          "               [--denoise [ITER]]\n"
          "  NAME: spheres_lens spheres_pinhole random_spheres interior soup, or a folder under DIR\n"
          "        holding NAME.scene (coffee, cornell, ...).  Defaults are the reference's constants\n"
          "        (1920x1080, 32 spp, depth 256; MinimalOptiX.h:82-89); a .scene file's properties{width,height}\n"
          "        replace 1920x1080.  --gpus N renders on devices 0..N-1 of this process (tile-split, scene\n"
          "        replicated, tiles gathered over NVLink into device 0).  --watertight: MOX_ACCEL_WATERTIGHT (include/mox.h).\n"
          "  --adaptive REL[,ABS]: render with mox_render_adaptive up to --spp: a pixel stops once the standard error of its\n"
          "        luminance is below max(REL * mean, ABS) (ABS default 0); the image is divided by each pixel's sample count.\n"
          "        --adaptive-min N: samples before a pixel may stop (default 16); --adaptive-round N: launches between two\n"
          "        checks (default 8).  Not combined with --snapshots, --resume or --dump-accum.\n"
          "  --denoise [ITER]: accumulate first-hit albedo, normal and depth (mox_set_aovs) and filter the final image with\n"
          "        mox_denoise (ITER a-trous iterations, default 5): writes PREFIX_denoised.png, PREFIX_albedo.png and\n"
          "        PREFIX_normal.png (0.5 + 0.5 N) and adds ms_denoise to the JSON line.\n");
}

int main(int argc, char** argv) {
  std::string scene = "spheres_lens", dir = "scenes", out = "out", lib, rng = "ref", resume;
  uint32_t W = 0, H = 0, spp = 32, depth = 256, seed = 0xC0FFEE;
  uint64_t param = 0;
  int device = 0, gpus = 0;
  bool snapshots = false, dumpAccum = false, watertight = false, adaptive = false, denoise = false;
  mox_denoise_params dn{MOX_DENOISE_DEFAULT_ITERATIONS, MOX_DENOISE_DEFAULT_SIGMA_COLOR, MOX_DENOISE_DEFAULT_SIGMA_NORMAL,
                        MOX_DENOISE_DEFAULT_SIGMA_DEPTH};
  mox_adaptive ad{8u, 16u, 0.f, 0.f};   // round_spp, min_spp, rel_error, abs_error
  for (int i = 1; i < argc; ++i) {
    std::string a = argv[i];
    auto val = [&]() -> const char* { if (i + 1 >= argc) { usage(); exit(2); } return argv[++i]; };
    if (a == "--scene") scene = val();
    else if (a == "--scene-dir") dir = val();
    else if (a == "--width") W = (uint32_t)atoi(val());
    else if (a == "--height") H = (uint32_t)atoi(val());
    else if (a == "--spp") spp = (uint32_t)atoi(val());
    else if (a == "--max-depth") depth = (uint32_t)atoi(val());
    else if (a == "--seed") seed = (uint32_t)strtoul(val(), nullptr, 0);
    else if (a == "--rng") rng = val();
    else if (a == "--out") out = val();
    else if (a == "--snapshots") snapshots = true;
    else if (a == "--dump-accum") dumpAccum = true;
    else if (a == "--watertight") watertight = true;
    else if (a == "--resume") resume = val();
    else if (a == "--device") device = atoi(val());
    else if (a == "--gpus") gpus = atoi(val());
    else if (a == "--param") param = strtoull(val(), nullptr, 0);
    else if (a == "--lib") lib = val();
    else if (a == "--adaptive") {
      const char* v = val();
      char* end = nullptr;
      adaptive = true;
      ad.rel_error = strtof(v, &end);
      if (*end == ',') ad.abs_error = strtof(end + 1, &end);
      if (*end) { fprintf(stderr, "--adaptive wants REL or REL,ABS, got %s\n", v); return 2; }
    }
    else if (a == "--denoise") {
      denoise = true;
      if (i + 1 < argc && argv[i + 1][0] >= '0' && argv[i + 1][0] <= '9') dn.iterations = (uint32_t)atoi(argv[++i]);
    }
    else if (a == "--adaptive-min") ad.min_spp = (uint32_t)atoi(val());
    else if (a == "--adaptive-round") ad.round_spp = (uint32_t)atoi(val());
    else { usage(); return 2; }
  }
  if (adaptive && (snapshots || !resume.empty() || dumpAccum)) {
    fprintf(stderr, "--adaptive renders a different number of samples per pixel; it cannot be combined with --snapshots, --resume "
                    "or --dump-accum, which assume the same count everywhere\n");
    return 2;
  }
  if (lib.empty()) {
    std::string self = argv[0];
    size_t p = self.rfind('/');
    lib = (p == std::string::npos ? std::string(".") : self.substr(0, p)) + "/libmox.so";
  }
  MoxApi api;
  std::string err;
  if (!loadMoxApi(lib.c_str(), "mox_", api, err)) { fprintf(stderr, "cannot load %s: %s\n", lib.c_str(), err.c_str()); return 1; }
  moxh::SceneDesc sc;
  bool ok;
  if (scene == "spheres_lens" || scene == "spheres_pinhole") ok = moxh::buildSpheres(sc, scene == "spheres_pinhole", 0, 0);
  else if (scene == "random_spheres") ok = moxh::buildRandomSpheres(sc, param ? (int)param : 256, 42u);
  else if (scene == "interior") ok = moxh::buildInterior(sc, param ? param : 1000000ull, 0xD1A1A6u);
  else if (scene == "soup") ok = moxh::buildSoup(sc, param ? param : 10000000ull, 10000000ull);
  else ok = moxh::loadSceneFile(sc, dir + "/" + scene, scene, err);
  if (!ok) { fprintf(stderr, "scene: %s\n", err.c_str()); return 1; }
  for (auto& w : sc.warnings) fprintf(stderr, "warning: %s\n", w.c_str());
  if (!W) W = sc.defaultWidth;
  if (!H) H = sc.defaultHeight;

  mox_ctx* ctx = nullptr;
  if (gpus > 0) {
    if (!api.create_multi) { fprintf(stderr, "%s has no mox_create_multi\n", lib.c_str()); return 1; }
    std::vector<int> ids(gpus);
    for (int i = 0; i < gpus; ++i) ids[i] = i;
    if (api.create_multi(&ctx, ids.data(), gpus)) { fprintf(stderr, "mox_create_multi: %s\n", api.last_error(nullptr)); return 1; }
  } else if (api.create(&ctx, device)) { fprintf(stderr, "mox_create: %s\n", api.last_error(nullptr)); return 1; }
  if (adaptive && !(api.render_adaptive && api.read_sample_counts)) { fprintf(stderr, "%s has no mox_render_adaptive\n", lib.c_str()); return 1; }
  if (denoise && !(api.set_aovs && api.read_aovs && api.denoise && api.read_sample_counts)) {
    fprintf(stderr, "%s has no mox_denoise\n", lib.c_str());
    return 1;
  }
  api.set_rng_mode(ctx, rng == "philox" ? MOX_RNG_PHILOX : MOX_RNG_REF);
  if (!moxh::uploadScene(sc, api, ctx, W, H, depth, err)) { fprintf(stderr, "upload: %s\n", err.c_str()); return 1; }
  float buildMs = 0;
  if (api.build_accel(ctx, watertight ? MOX_ACCEL_WATERTIGHT : MOX_ACCEL_DEFAULT, &buildMs)) { fprintf(stderr, "build_accel: %s\n", api.last_error(ctx)); return 1; }

  std::vector<float> accum((size_t)W * H * 3);
  std::vector<uint8_t> rgb((size_t)W * H * 3);
  std::vector<uint32_t> counts(adaptive ? (size_t)W * H : 0);
  // a snapshot = updateContent (MinimalOptiX.cpp:556-560): map the accumulation buffer (on several GPUs: gather the
  // tiles into device 0 over NVLink), quantise, write the image
  double readSec = 0, writeSec = 0;
  uint32_t nSnapshots = 0;
  auto save = [&](const std::string& name, uint32_t n) {
    auto a0 = std::chrono::steady_clock::now();
    api.read_accum(ctx, accum.data());
    auto a1 = std::chrono::steady_clock::now();
    if (adaptive) {
      api.read_sample_counts(ctx, counts.data());
      moxh_accum_to_rgb8_counts(accum.data(), W, H, counts.data(), rgb.data());
    } else moxh_accum_to_rgb8(accum.data(), W, H, (float)n, rgb.data());
    if (moxh_write_image((name + ".png").c_str(), rgb.data(), W, H)) fprintf(stderr, "write: %s\n", moxh_last_error());
    readSec += std::chrono::duration<double>(a1 - a0).count();
    writeSec += std::chrono::duration<double>(std::chrono::steady_clock::now() - a1).count();
    nSnapshots++;
  };
  if (denoise && api.set_aovs(ctx, 1)) { fprintf(stderr, "set_aovs: %s\n", api.last_error(ctx)); return 1; }
  uint32_t done = 0, checkpoint = 1;
  if (!resume.empty()) {  // continue a previous run: same seed schedule, samples [launches, spp)
    uint64_t launches = 0;
    if (moxh_read_accum(resume.c_str(), accum.data(), W, H, &launches)) { fprintf(stderr, "resume: %s\n", moxh_last_error()); return 1; }
    if (api.set_accum(ctx, accum.data(), launches)) { fprintf(stderr, "set_accum: %s\n", api.last_error(ctx)); return 1; }
    done = (uint32_t)std::min<uint64_t>(launches, spp);
    while (checkpoint <= done) checkpoint *= 2;
  }
  uint64_t samples = (uint64_t)W * H * (spp - done);
  auto t0 = std::chrono::steady_clock::now();
  if (adaptive) {
    if (api.render_adaptive(ctx, spp, seed, &ad, &samples)) { fprintf(stderr, "render_adaptive: %s\n", api.last_error(ctx)); return 1; }
    done = spp;
  }
  while (done < spp) {  // renderScene: snapshots at 1, 2, 4, ... (MinimalOptiX.cpp:543-553)
    uint32_t n = snapshots ? std::min(spp, checkpoint) - done : spp - done;
    if (api.render(ctx, n, seed)) { fprintf(stderr, "render: %s\n", api.last_error(ctx)); return 1; }
    done += n;
    if (snapshots && done == checkpoint) { save(out + "_" + std::to_string(done), done); checkpoint *= 2; }
  }
  double sec = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  save(out, spp);
  if (dumpAccum) moxh_write_accum((out + ".moxa").c_str(), accum.data(), W, H, spp);
  // the denoised image and its guides, each written through the same quantisation as the image (n = 1)
  float denoiseMs = 0;
  if (denoise) {
    std::vector<float> img((size_t)W * H * 3), nrm((size_t)W * H * 3);
    if (api.denoise(ctx, &dn, img.data(), &denoiseMs)) { fprintf(stderr, "denoise: %s\n", api.last_error(ctx)); return 1; }
    auto write = [&](const char* suffix, const float* v) {
      moxh_accum_to_rgb8(v, W, H, 1.f, rgb.data());
      if (moxh_write_image((out + suffix).c_str(), rgb.data(), W, H)) fprintf(stderr, "write: %s\n", moxh_last_error());
    };
    write("_denoised.png", img.data());
    if (api.read_aovs(ctx, img.data(), nrm.data(), nullptr)) { fprintf(stderr, "read_aovs: %s\n", api.last_error(ctx)); return 1; }
    write("_albedo.png", img.data());
    for (float& v : nrm) v = 0.5f + 0.5f * v;
    write("_normal.png", nrm.data());
  }
  mox_stats st;
  api.get_stats(ctx, &st);
  // share of the pixels that received every launch (1 for a uniform render)
  double activeEnd = 1.0;
  if (adaptive) {
    uint64_t full = 0;
    for (uint32_t n : counts) full += n == spp;
    activeEnd = (double)full / ((double)W * H);
  }
  double rays = (double)(st.rays_primary + st.rays_bounce);
  printf("{\"scene\": \"%s\", \"width\": %u, \"height\": %u, \"spp\": %u, \"max_depth\": %u, \"seed\": %u, \"rng\": \"%s\", "
         "\"triangles\": %u, \"prims\": %u, \"bvh_build_ms\": %.3f, \"render_ms\": %.3f, \"wall_s\": %.3f, "
         "\"rays_primary\": %llu, \"rays_bounce\": %llu, \"rays_shadow\": %llu, \"mrays_per_s\": %.2f, \"mshadow_per_s\": %.2f, "
         "\"spp_per_s\": %.3f, \"nonfinite\": %llu, \"gpus\": %d, \"ms_extend\": %.2f, \"ms_shade\": %.2f, \"ms_shadow\": %.2f, "
         "\"kernel_launches\": %llu, \"snapshots\": %u, \"gather_and_readback_s\": %.4f, \"quantise_and_png_s\": %.3f, "
         "\"samples\": %llu, \"active_fraction_end\": %.4f, \"render_ms_per_gpu\": [",
         scene.c_str(), W, H, spp, depth, seed, rng.c_str(), st.n_triangles, st.n_prims, buildMs, st.ms_render, sec,
         (unsigned long long)st.rays_primary, (unsigned long long)st.rays_bounce, (unsigned long long)st.rays_shadow,
         rays / (st.ms_render * 1e3), (double)st.rays_shadow / (st.ms_render * 1e3), spp / (st.ms_render * 1e-3),
         (unsigned long long)st.nonfinite_samples, gpus > 0 ? gpus : 1, st.ms_extend, st.ms_shade, st.ms_shadow,
         (unsigned long long)st.kernel_launches, nSnapshots, readSec, writeSec, (unsigned long long)samples, activeEnd);
  const int nDev = api.device_count ? api.device_count(ctx) : 1;
  for (int i = 0; i < nDev; ++i) {
    mox_stats ds = st;
    if (api.get_device_stats) api.get_device_stats(ctx, i, &ds);
    printf("%s%.2f", i ? ", " : "", ds.ms_render);
  }
  printf("]");
  if (denoise) printf(", \"ms_denoise\": %.3f, \"denoise_iterations\": %u", denoiseMs, dn.iterations);
  printf("}\n");
  api.destroy(ctx);
  return 0;
}

