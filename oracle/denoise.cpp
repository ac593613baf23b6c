// oracle/denoise.cpp — TEST INFRASTRUCTURE.  The oracle's side of mox_set_aovs, mox_read_aovs and mox_denoise
// (include/mox.h).
//
// liboracle.so is built from this file: it compiles adaptive.cpp (and with it refit.cpp and oracle.cpp) unchanged and
// wraps the entry points that render.  A camera sample's AOV record comes from the same camera ray and closest hit as
// its colour (cameraSample), so the image does not change.  The denoiser is a scalar restatement of the formula in
// mox.h; the build has no FMA contraction, so every product and sum is rounded on its own.
//
// The AOV state is keyed by context.  A reset of the accumulation buffer (orc_create, orc_clear_accum, orc_set_accum,
// a size change) erases the context's adaptive record (adaptive.cpp's resetAdaptive); every entry point of this file
// leaves such a record behind and reads its absence as a reset.  The state of a destroyed context (no refit record,
// refit.cpp) is dropped at the next call of this file's entry points; a context created at the address of a destroyed one
// before that call inherits its switch, so the tests keep the contexts they switch on alive.
#define orc_launch orc_launch_base
#define orc_render orc_render_base
#define orc_render_adaptive orc_render_adaptive_base
#include "adaptive.cpp"
#undef orc_launch
#undef orc_render
#undef orc_render_adaptive

namespace {

// Per pixel: albedo and normal sums, depth sum, AOV samples, hits.
struct AovInfo {
  bool on = false;
  std::vector<float> albedo, normal, depth;
  std::vector<uint32_t> n, hits;
};

std::mutex g_aovMutex;
std::map<const orc_ctx*, AovInfo> g_aov;

// The context's AOV state, with its sums zeroed when the accumulation buffer was reset since the last call and sized
// for the image.  Drops the state of destroyed contexts.
AovInfo& aovInfo(const orc_ctx* c) {
  std::lock_guard<std::mutex> lock(g_aovMutex);
  {
    std::lock_guard<std::mutex> lr(g_refitMutex);
    for (auto it = g_aov.begin(); it != g_aov.end();) it = g_refit.count(it->first) ? std::next(it) : g_aov.erase(it);
    g_refit[c];   // a live context has a refit record
  }
  AovInfo& a = g_aov[c];
  bool reset;
  {
    std::lock_guard<std::mutex> la(g_adaptiveMutex);
    reset = !g_adaptive.count(c);
    g_adaptive[c];   // an empty record: adaptive.cpp sizes it at its first use
  }
  const size_t nPix = (size_t)c->W * c->H;
  if (reset || a.n.size() != nPix) {
    a.albedo.assign(3 * nPix, 0.f); a.normal.assign(3 * nPix, 0.f); a.depth.assign(nPix, 0.f);
    a.n.assign(nPix, 0u); a.hits.assign(nPix, 0u);
  }
  return a;
}

// Camera.cu:21-36 for pixel (x, y) of launch `launchSeed`: the ray cameraSample traces.
Ray cameraRay(const orc_ctx& c, uint32_t x, uint32_t y, int32_t launchSeed) {
  Rng rng = rngForPixel(c.rngMode, y * c.W + x, (uint32_t)launchSeed);
  const CamParams& cp = c.cam;
  float3 randInLens = cp.lensRadius * randInUnitDisk(rng);
  float3 offset = f3(cp.u) * randInLens.x + f3(cp.v) * randInLens.y;
  float r1 = rnd(rng);
  float r2 = rnd(rng);
  float sx = ((float)x + r1 - 0.5f) / (float)c.W;
  float sy = ((float)y + r2 - 0.5f) / (float)c.H;
  Ray ray;
  ray.origin = f3(cp.origin) + offset;
  ray.direction = normalize(f3(cp.scrLowerLeftCorner) + sx * f3(cp.horizontal) + sy * f3(cp.vertical) - f3(cp.origin) - offset);
  ray.tmin = c.eps;
  ray.tmax = RT_DEFAULT_MAX;
  return ray;
}

float3 clamp01(const float3& v) { return clamp(v, make_float3(0.f), make_float3(1.f)); }

// Adds the records of launch seeds[0, k_p) to every owned pixel p, in launch order; k_p = taken[p] (null: all).
void addRecords(const orc_ctx* c, AovInfo& a, const std::vector<int32_t>& seeds, const uint32_t* taken) {
  std::vector<uint32_t> owned;
  ownedList(*c, c->rank, owned);
  for (uint32_t px : owned) {
    const uint32_t x = px % c->W, y = px / c->W;
    const size_t k = taken ? taken[px] : seeds.size();
    for (size_t i = 0; i < k; ++i) {
      const Ray ray = cameraRay(*c, x, y, seeds[i]);
      HitAttr h;
      float3 alb, nrm = make_float3(0.f);
      if (!closestHit(*c, ray, h)) alb = clamp01(c->bg);
      else {
        const Material& m = c->mats[c->prims[h.prim].mat];
        switch (m.kind) {
          case MOX_MAT_LAMBERTIAN: alb = f3(m.lam.albedo); break;
          case MOX_MAT_METAL: alb = f3(m.met.albedo); break;
          case MOX_MAT_GLASS: alb = f3(m.gls.albedo); break;
          case MOX_MAT_DISNEY:
            alb = m.dis.albedoID == MOX_TEXTURE_ID_NULL ? f3(m.dis.color) : sampleTexture(*c, m.dis.albedoID, h.texcoord.x, h.texcoord.y);
            break;
          default: alb = clamp01(f3(m.lgt.emission));
        }
        nrm = faceforward(h.shadingNormal, -ray.direction, h.geoNormal);
        a.depth[px] += h.t;
        a.hits[px]++;
      }
      a.albedo[3 * px] += alb.x; a.albedo[3 * px + 1] += alb.y; a.albedo[3 * px + 2] += alb.z;
      a.normal[3 * px] += nrm.x; a.normal[3 * px + 1] += nrm.y; a.normal[3 * px + 2] += nrm.z;
    }
    a.n[px] += (uint32_t)k;
  }
}

// The filter of mox.h on W x H pixels: colour c, albedo a, normal N, depth z in; out (3 floats per pixel) out.
void atrous(uint32_t W, uint32_t H, const std::vector<float>& c, const std::vector<float>& a, const std::vector<float>& N,
            const std::vector<float>& z, const mox_denoise_params& p, float* out) {
  const size_t nPix = (size_t)W * H;
  std::vector<float> e(3 * nPix), next(3 * nPix), m(3 * nPix);
  for (size_t i = 0; i < 3 * nPix; ++i) { m[i] = a[i] + 0.001f; e[i] = c[i] / m[i]; }
  const float h[5] = {1.f / 16.f, 1.f / 4.f, 3.f / 8.f, 1.f / 4.f, 1.f / 16.f};
  for (uint32_t it = 0; it < p.iterations; ++it) {
    const int step = 1 << it;
    const float sigma = p.sigma_color * std::ldexp(1.f, -(int)it);
    const float sig2 = sigma * sigma;
    for (int y = 0; y < (int)H; ++y)
      for (int x = 0; x < (int)W; ++x) {
        const size_t pp = (size_t)y * W + x;
        const float* ep = &e[3 * pp];
        const float* np = &N[3 * pp];
        float sx = 0.f, sy = 0.f, sz = 0.f, sw = 0.f;
        for (int dy = -2; dy <= 2; ++dy)
          for (int dx = -2; dx <= 2; ++dx) {
            const int qx = x + step * dx, qy = y + step * dy;
            if (qx < 0 || qx >= (int)W || qy < 0 || qy >= (int)H) continue;
            const size_t q = (size_t)qy * W + qx;
            const float* eq = &e[3 * q];
            float w = 1.f;
            if (dx != 0 || dy != 0) {
              const float* nq = &N[3 * q];
              const float ex = ep[0] - eq[0], ey = ep[1] - eq[1], ez = ep[2] - eq[2];
              const float tc = (ex * ex + ey * ey + ez * ez) / sig2;
              const float tn = std::max(0.f, 1.f - (np[0] * nq[0] + np[1] * nq[1] + np[2] * nq[2])) / p.sigma_normal;
              const float tz = std::fabs(z[pp] - z[q]) / (p.sigma_depth * std::max(z[pp], z[q]) + 1e-30f);
              w = std::exp(-(tc + tn + tz));
            }
            const float k = h[dx + 2] * h[dy + 2] * w;
            sx += k * eq[0]; sy += k * eq[1]; sz += k * eq[2];
            sw += k;
          }
        next[3 * pp] = sx / sw; next[3 * pp + 1] = sy / sw; next[3 * pp + 2] = sz / sw;
      }
    e.swap(next);
  }
  for (size_t i = 0; i < 3 * nPix; ++i) out[i] = e[i] * m[i];
}

}  // namespace

extern "C" {

int orc_set_aovs(orc_ctx* c, int enable) {
  if (!c) return MOX_ERR_INVALID;
  AovInfo& a = aovInfo(c);
  if (enable) a.on = true;
  else a = AovInfo();
  return MOX_OK;
}

int orc_launch(orc_ctx* c, int32_t seed) {
  if (!c) return MOX_ERR_INVALID;
  AovInfo& a = aovInfo(c);
  const int rc = orc_launch_base(c, seed);
  if (rc == MOX_OK && a.on) addRecords(c, a, {seed}, nullptr);
  return rc;
}

int orc_render(orc_ctx* c, uint32_t spp, uint32_t seed) {
  if (!c) return MOX_ERR_INVALID;
  std::vector<int32_t> seeds(spp);
  for (uint32_t i = 0; i < spp; ++i) seeds[i] = (int32_t)tea<16>((uint32_t)(c->launches + i), seed);
  AovInfo& a = aovInfo(c);
  const int rc = orc_render_base(c, spp, seed);
  if (rc == MOX_OK && a.on) addRecords(c, a, seeds, nullptr);
  return rc;
}

// Pixels only ever stop during an adaptive call, so a pixel that took k samples in it took the call's first k launches.
int orc_render_adaptive(orc_ctx* c, uint32_t spp, uint32_t seed, const mox_adaptive* p, uint64_t* out_samples) {
  if (!c) return MOX_ERR_INVALID;
  AovInfo& a = aovInfo(c);   // first: orc_read_sample_counts leaves an adaptive record behind
  const size_t nPix = (size_t)c->W * c->H;
  std::vector<uint32_t> before(nPix), after(nPix);
  orc_read_sample_counts(c, before.data());
  const uint64_t first = c->launches;
  const int rc = orc_render_adaptive_base(c, spp, seed, p, out_samples);
  if (rc != MOX_OK || !a.on) return rc;
  orc_read_sample_counts(c, after.data());
  for (size_t i = 0; i < nPix; ++i) after[i] -= before[i];
  std::vector<int32_t> seeds(spp);
  for (uint32_t i = 0; i < spp; ++i) seeds[i] = (int32_t)tea<16>((uint32_t)(first + i), seed);
  addRecords(c, a, seeds, after.data());
  return rc;
}

int orc_read_aovs(orc_ctx* c, float* albedo, float* normal, float* depth) {
  if (!c) return MOX_ERR_INVALID;
  const AovInfo& a = aovInfo(c);
  if (!a.on) { c->err = "AOVs are off (orc_set_aovs)"; return MOX_ERR_STATE; }
  for (size_t p = 0; p < a.n.size(); ++p) {
    const float n = (float)a.n[p];
    for (int k = 0; k < 3; ++k) {
      if (albedo) albedo[3 * p + k] = a.n[p] ? a.albedo[3 * p + k] / n : 0.f;
      if (normal) normal[3 * p + k] = a.n[p] ? a.normal[3 * p + k] / n : 0.f;
    }
    if (depth) depth[p] = a.hits[p] ? a.depth[p] / (float)a.hits[p] : 0.f;
  }
  return MOX_OK;
}

int orc_denoise(orc_ctx* c, const mox_denoise_params* params, float* dst, float* out_ms) {
  if (!c) return MOX_ERR_INVALID;
  if (out_ms) *out_ms = 0.f;
  mox_denoise_params p{MOX_DENOISE_DEFAULT_ITERATIONS, MOX_DENOISE_DEFAULT_SIGMA_COLOR, MOX_DENOISE_DEFAULT_SIGMA_NORMAL,
                       MOX_DENOISE_DEFAULT_SIGMA_DEPTH};
  if (params) p = *params;
  if (p.iterations < 1 || p.iterations > 10) { c->err = "iterations must be 1..10"; return MOX_ERR_INVALID; }
  for (float s : {p.sigma_color, p.sigma_normal, p.sigma_depth})
    if (!std::isfinite(s) || !(s > 0.f)) { c->err = "sigmas must be finite and > 0"; return MOX_ERR_INVALID; }
  if (!dst) return MOX_ERR_INVALID;
  if (c->world > 1) { c->err = "denoise needs the whole frame"; return MOX_ERR_STATE; }
  const AovInfo& a = aovInfo(c);
  if (!a.on) { c->err = "AOVs are off (orc_set_aovs)"; return MOX_ERR_STATE; }
  if (std::none_of(a.n.begin(), a.n.end(), [](uint32_t n) { return n != 0; })) {
    c->err = "denoise before any sample was rendered with AOVs on";
    return MOX_ERR_STATE;
  }
  const auto t0 = std::chrono::steady_clock::now();
  const size_t nPix = (size_t)c->W * c->H;
  std::vector<uint32_t> counts(nPix);
  orc_read_sample_counts(c, counts.data());
  std::vector<float> col(3 * nPix), alb(3 * nPix), nrm(3 * nPix), z(nPix);
  for (size_t i = 0; i < 3 * nPix; ++i) col[i] = counts[i / 3] ? c->accu[i] / (float)counts[i / 3] : 0.f;
  orc_read_aovs(c, alb.data(), nrm.data(), z.data());
  atrous(c->W, c->H, col, alb, nrm, z, p, dst);
  if (out_ms) *out_ms = (float)std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return MOX_OK;
}

}  // extern "C"
