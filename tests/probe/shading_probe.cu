// shading_probe.cu — TEST INFRASTRUCTURE: the device shading math of shading.cuh, one thread per case, behind a C ABI
// that tests/test_shading_math.py loads with ctypes.  Built by `make probe` with the flags of libmox.so, so the
// functions under test are compiled exactly as the render kernels compile them; never linked into the product.
//
// Every entry point takes host arrays (vectors as n x 3 floats), copies them to the device, runs one thread per
// case, copies the results back and returns the CUDA error code (0 = success).
#include <vector>
#include "shading.cuh"

namespace {

// rnd() returns the next of the case's draws; `used` counts the calls.
struct FeedRng {
  const float* draws;
  int n, used;
  __device__ float rnd() { float r = used < n ? draws[used] : 0.f; ++used; return r; }
};

MOX_D float3 ld3(const float* p, int i) { return mk3(p[3 * i], p[3 * i + 1], p[3 * i + 2]); }
MOX_D void st3(float* p, int i, const float3& v) { p[3 * i] = v.x; p[3 * i + 1] = v.y; p[3 * i + 2] = v.z; }

// What k_shade_disney does for one light sample (H = bnormalize<F>(L + V)) or for the sampled direction (H given).
template <bool F>
__global__ void k_disney_hit_eval(int n, const DisneyParams* mp, const float* baseColor, const float* N, const float* V,
                                  const float* L, const float* Hin, float* outPdf, float* outDr, float* outEval, float* outH) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  DisneyHit<F> dh(mp[i], ld3(baseColor, i), ld3(N, i));
  float3 v = ld3(V, i), l = ld3(L, i);
  dh.setView(v);
  float3 h = Hin ? ld3(Hin, i) : bnormalize<F>(l + v);
  float dr;
  outPdf[i] = dh.pdf(l, h, dr);
  outDr[i] = dr;
  st3(outEval, i, dh.eval(l, h, dr));
  st3(outH, i, h);
}

__global__ void k_disney_sample(int n, const DisneyParams* mp, const float* N, const float* V, const float* draws,
                                float* outL, float* outH, int* outUsed) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  FeedRng r{draws + 4 * i, 4, 0};
  float3 L, H;
  disneySample(r, mp[i], ld3(N, i), L, ld3(V, i), H);
  st3(outL, i, L);
  st3(outH, i, H);
  outUsed[i] = r.used;
}

// k_shade_dielectric up to the coin flip.
__global__ void k_refract_fresnel(int n, const float* D, const float* Ns, const float* ior, float* outR, int* outTir,
                                  float* outReflectProb) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float3 d = ld3(D, i), normal = ld3(Ns, i);
  float cosI = -dot(d, normal);
  float refIdx;
  if (cosI > 0.f) { refIdx = ior[i]; }
  else { refIdx = 1.f / ior[i]; cosI = -cosI; normal = -normal; }
  float3 refracted;
  bool tir = !refract3(refracted, d, normal, refIdx);
  float cosT = -dot(normal, refracted);
  st3(outR, i, refracted);
  outTir[i] = tir ? 1 : 0;
  outReflectProb[i] = tir ? 1.f : fresnelDielectric(cosI, cosT, refIdx);
}

__global__ void k_libm(int n, const float* x, float* outPow22, float* outLog) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  outPow22[i] = powf(x[i], 2.2f);
  outLog[i] = logf(x[i]);
}

// Device buffers of one call: inputs copied up on creation, outputs copied back by fetch(); freed on scope exit.
struct Buffers {
  std::vector<void*> ptrs;
  cudaError_t err = cudaSuccess;
  template <class T> T* up(const T* host, size_t count) {
    if (!host) return nullptr;
    T* d = alloc<T>(count);
    if (d && err == cudaSuccess) err = cudaMemcpy(d, host, count * sizeof(T), cudaMemcpyHostToDevice);
    return d;
  }
  template <class T> T* alloc(size_t count) {
    void* d = nullptr;
    if (err == cudaSuccess) err = cudaMalloc(&d, count * sizeof(T));
    if (d) ptrs.push_back(d);
    return (T*)d;
  }
  template <class T> void fetch(T* host, const T* dev, size_t count) {
    if (err == cudaSuccess) err = cudaMemcpy(host, dev, count * sizeof(T), cudaMemcpyDeviceToHost);
  }
  cudaError_t launched() {
    if (err == cudaSuccess) err = cudaGetLastError();
    return err;
  }
  ~Buffers() { for (void* p : ptrs) cudaFree(p); }
};

constexpr int kThreads = 128;
int blocks(int n) { return (n + kThreads - 1) / kThreads; }

}  // namespace

extern "C" {

// fast != 0: DisneyHit<true> (the default render mode); 0: DisneyHit<false> (MOX_BRDF_IEEE=1).
// H == nullptr: H = bnormalize<F>(L + V) as in the light loop; out_H receives the H that was used.
int probe_disney_hit_eval(int fast, int n, const DisneyParams* params, const float* baseColor, const float* N,
                          const float* V, const float* L, const float* H, float* out_pdf, float* out_dr, float* out_eval,
                          float* out_H) {
  if (n <= 0) return 0;
  Buffers b;
  const DisneyParams* dp = b.up(params, n);
  const float *dc = b.up(baseColor, 3 * n), *dn = b.up(N, 3 * n), *dv = b.up(V, 3 * n), *dl = b.up(L, 3 * n);
  const float* dh = b.up(H, 3 * n);
  float *pdf = b.alloc<float>(n), *dr = b.alloc<float>(n), *ev = b.alloc<float>(3 * n), *ho = b.alloc<float>(3 * n);
  if (b.err) return b.err;
  if (fast) k_disney_hit_eval<true><<<blocks(n), kThreads>>>(n, dp, dc, dn, dv, dl, dh, pdf, dr, ev, ho);
  else k_disney_hit_eval<false><<<blocks(n), kThreads>>>(n, dp, dc, dn, dv, dl, dh, pdf, dr, ev, ho);
  if (b.launched()) return b.err;
  b.fetch(out_pdf, pdf, n);
  b.fetch(out_dr, dr, n);
  b.fetch(out_eval, ev, 3 * n);
  b.fetch(out_H, ho, 3 * n);
  return b.err;
}

// draws: 4 per case; out_draws_used: how many disneySample consumed.
int probe_disney_sample(int n, const DisneyParams* params, const float* N, const float* V, const float* draws,
                        float* out_L, float* out_H, int* out_draws_used) {
  if (n <= 0) return 0;
  Buffers b;
  const DisneyParams* dp = b.up(params, n);
  const float *dn = b.up(N, 3 * n), *dv = b.up(V, 3 * n), *dd = b.up(draws, 4 * n);
  float *lo = b.alloc<float>(3 * n), *ho = b.alloc<float>(3 * n);
  int* used = b.alloc<int>(n);
  if (b.err) return b.err;
  k_disney_sample<<<blocks(n), kThreads>>>(n, dp, dn, dv, dd, lo, ho, used);
  if (b.launched()) return b.err;
  b.fetch(out_L, lo, 3 * n);
  b.fetch(out_H, ho, 3 * n);
  b.fetch(out_draws_used, used, n);
  return b.err;
}

int probe_refract_fresnel(int n, const float* d, const float* Ns, const float* ior, float* out_refracted, int* out_tir,
                          float* out_reflect_prob) {
  if (n <= 0) return 0;
  Buffers b;
  const float *dd = b.up(d, 3 * n), *dn = b.up(Ns, 3 * n), *di = b.up(ior, n);
  float *r = b.alloc<float>(3 * n), *p = b.alloc<float>(n);
  int* t = b.alloc<int>(n);
  if (b.err) return b.err;
  k_refract_fresnel<<<blocks(n), kThreads>>>(n, dd, dn, di, r, t, p);
  if (b.launched()) return b.err;
  b.fetch(out_refracted, r, 3 * n);
  b.fetch(out_tir, t, n);
  b.fetch(out_reflect_prob, p, n);
  return b.err;
}

// CUDA's powf(x, 2.2f) and logf(x): the libm calls of the IEEE BRDF mode (srgb2lin, GTR1's log(a^2)).
int probe_libm(int n, const float* x, float* out_pow22, float* out_log) {
  if (n <= 0) return 0;
  Buffers b;
  const float* dx = b.up(x, n);
  float *p = b.alloc<float>(n), *l = b.alloc<float>(n);
  if (b.err) return b.err;
  k_libm<<<blocks(n), kThreads>>>(n, dx, p, l);
  if (b.launched()) return b.err;
  b.fetch(out_pow22, p, n);
  b.fetch(out_log, l, n);
  return b.err;
}

}  // extern "C"
