// oracle/adaptive.cpp — TEST INFRASTRUCTURE.  The oracle's side of mox_render_adaptive and mox_read_sample_counts
// (include/mox.h).
//
// liboracle.so is built from this file: it compiles refit.cpp (and with it oracle.cpp) unchanged and wraps the entry
// points that reset the adaptive state.  Samples are per-pixel independent, so each launch renders the whole image
// into a zeroed buffer, which gives every pixel's sample colour exactly, and only the active pixels add it to the
// accumulation buffer and to their luminance sums.
#define orc_create orc_create_base
#define orc_set_globals orc_set_globals_base
#define orc_clear_accum orc_clear_accum_base
#define orc_set_accum orc_set_accum_base
#include "refit.cpp"
#undef orc_create
#undef orc_set_globals
#undef orc_clear_accum
#undef orc_set_accum

#include <cmath>

namespace {

// Per pixel: S1 = sum y, S2 = sum y^2 (float64), n adaptive samples, launches sat out.
struct AdaptiveInfo {
  std::vector<double> s1, s2;
  std::vector<uint32_t> n, skipped;
};

std::mutex g_adaptiveMutex;
// Keyed by context.  orc_destroy is refit.cpp's wrapper, which erases the context's refit record (g_refit, which
// every built context has); the entries of contexts without one are dropped at the next call of this file's entry
// points, so the state of a destroyed context lives on only until then.
std::map<const orc_ctx*, AdaptiveInfo> g_adaptive;

// Drops the entries of destroyed contexts.  Call with g_adaptiveMutex held.
void dropDestroyed() {
  std::lock_guard<std::mutex> lock(g_refitMutex);
  for (auto it = g_adaptive.begin(); it != g_adaptive.end();)
    it = g_refit.count(it->first) ? std::next(it) : g_adaptive.erase(it);
}

AdaptiveInfo& adaptiveInfo(const orc_ctx* c) {
  std::lock_guard<std::mutex> lock(g_adaptiveMutex);
  dropDestroyed();
  return g_adaptive[c];
}

void resetAdaptive(const orc_ctx* c) {
  std::lock_guard<std::mutex> lock(g_adaptiveMutex);
  dropDestroyed();
  g_adaptive.erase(c);
}

// y = 0.2126 r + 0.7152 g + 0.0722 b, each product and sum rounded to float32 (the build has no FMA contraction).
float luminance(float r, float g, float b) { return 0.2126f * r + 0.7152f * g + 0.0722f * b; }

bool converged(const AdaptiveInfo& a, size_t p, uint32_t minSpp, double rel, double abs) {
  const uint32_t n = a.n[p];
  if (n < minSpp) return false;
  const double dn = (double)n, m = a.s1[p] / dn;
  const double var = std::max(0.0, (a.s2[p] - a.s1[p] * m) / (dn - 1.0));
  return std::sqrt(var / dn) < std::max(rel * m, abs);
}

}  // namespace

extern "C" {

int orc_create(orc_ctx** out, int device) {
  const int rc = orc_create_base(out, device);
  if (rc == MOX_OK) resetAdaptive(*out);
  return rc;
}

int orc_set_globals(orc_ctx* c, uint32_t w, uint32_t h, uint32_t maxDepth, float eps, float minI, const float absorb[3],
                    const float bad[3], const float bg[3]) {
  const bool resize = c && (w != c->W || h != c->H);
  const int rc = orc_set_globals_base(c, w, h, maxDepth, eps, minI, absorb, bad, bg);
  if (rc == MOX_OK && resize) resetAdaptive(c);
  return rc;
}

int orc_clear_accum(orc_ctx* c) {
  const int rc = orc_clear_accum_base(c);
  if (rc == MOX_OK) resetAdaptive(c);
  return rc;
}

int orc_set_accum(orc_ctx* c, const float* src, uint64_t launches) {
  const int rc = orc_set_accum_base(c, src, launches);
  if (rc == MOX_OK) resetAdaptive(c);
  return rc;
}

int orc_render_adaptive(orc_ctx* c, uint32_t spp, uint32_t seed, const mox_adaptive* p, uint64_t* out_samples) {
  if (!c) return MOX_ERR_INVALID;
  if (out_samples) *out_samples = 0;
  if (!p || !p->round_spp || !std::isfinite(p->rel_error) || !std::isfinite(p->abs_error) || p->rel_error < 0.f || p->abs_error < 0.f) {
    c->err = "bad adaptive parameters";
    return MOX_ERR_INVALID;
  }
  if (!c->built) { c->err = "launch before build_accel"; return MOX_ERR_STATE; }
  if (c->W == 0 || c->H == 0) { c->err = "launch before set_globals"; return MOX_ERR_STATE; }
  const size_t nPix = (size_t)c->W * c->H;
  AdaptiveInfo& a = adaptiveInfo(c);
  if (a.n.size() != nPix) { a.s1.assign(nPix, 0.0); a.s2.assign(nPix, 0.0); a.n.assign(nPix, 0u); a.skipped.assign(nPix, 0u); }
  const uint32_t minSpp = std::max<uint32_t>(p->min_spp, 2u);
  const double rel = p->rel_error, abs = p->abs_error;
  // drops the converged pixels of `active`; they sit out the call's remaining launches
  auto select = [&](std::vector<uint32_t>& active, uint32_t remaining) {
    size_t k = 0;
    for (uint32_t px : active) {
      if (converged(a, px, minSpp, rel, abs)) a.skipped[px] += remaining;
      else active[k++] = px;
    }
    active.resize(k);
  };
  std::vector<uint32_t> active;
  ownedList(*c, c->rank, active);
  select(active, spp);
  const uint64_t first = c->launches;
  uint32_t done = 0;
  std::vector<float> kept;
  while (done < spp && !active.empty()) {
    const uint32_t r = std::min(p->round_spp, spp - done);
    for (uint32_t i = 0; i < r; ++i) {
      kept.swap(c->accu);
      c->accu.assign(kept.size(), 0.f);
      const int rc = launchSeeds(c, {(int32_t)tea<16>((uint32_t)(first + done + i), seed)});
      if (rc) { c->accu.swap(kept); return rc; }
      for (uint32_t px : active) {
        const float* s = &c->accu[3 * (size_t)px];
        float* d = &kept[3 * (size_t)px];
        d[0] += s[0]; d[1] += s[1]; d[2] += s[2];
        const double y = luminance(s[0], s[1], s[2]);
        a.s1[px] += y;
        a.s2[px] += y * y;
        a.n[px]++;
      }
      c->accu.swap(kept);
    }
    if (out_samples) *out_samples += (uint64_t)r * active.size();
    done += r;
    if (done < spp) select(active, spp - done);
  }
  c->launches = first + spp;
  return MOX_OK;
}

int orc_read_sample_counts(orc_ctx* c, uint32_t* dst) {
  if (!c || !dst) return MOX_ERR_INVALID;
  const size_t nPix = (size_t)c->W * c->H;
  const AdaptiveInfo& a = adaptiveInfo(c);
  std::fill(dst, dst + nPix, 0u);
  std::vector<uint32_t> owned;
  ownedList(*c, c->rank, owned);
  for (uint32_t px : owned) dst[px] = (uint32_t)(c->launches - (a.skipped.size() == nPix ? a.skipped[px] : 0u));
  return MOX_OK;
}

}  // extern "C"
