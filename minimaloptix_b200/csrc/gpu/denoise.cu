// denoise.cu — mox_denoise: the edge-avoiding a-trous wavelet filter of Dammertz, Hanika and Keller (2010) on the
// mean colour, guided by the first-hit AOVs.  The formula, and the order of its float32 operations, are in
// include/mox.h; the library is built with -fmad=false, so every product and sum is rounded on its own, and the
// divisions are IEEE divisions.
//
//   k_denoise_prep   per pixel: mean colour, AOV means, the demodulated irradiance e0 and the guide records
//   k_atrous         one launch per iteration, 2D blocks, ping-pong irradiance buffers; the last one remodulates
#include "denoise.h"

#include <algorithm>

#include "vec.cuh"

namespace {

constexpr int BX = 16, BY = 16;

struct Scratch {
  float4 *irr[2], *guide, *mod;   // irradiance (e.xyz), guide (N.xyz, z), albedo factor (a + 0.001)
};

Scratch scratchViews(void* base, size_t nPix) {
  float4* p = (float4*)base;
  return {{p, p + nPix}, p + 2 * nPix, p + 3 * nPix};
}

__global__ void __launch_bounds__(256) k_denoise_prep(DenoiseInput in, Scratch sc) {
  const size_t nPix = (size_t)in.W * in.H;
  const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nPix) return;
  const uint32_t n = in.launches - (in.skipped ? in.skipped[p] : 0u);
  const float fn = (float)n;
  const float3 c = n ? mk3(in.accu[3 * p] / fn, in.accu[3 * p + 1] / fn, in.accu[3 * p + 2] / fn) : mk3(0.f);
  const uint32_t na = in.aov.n[p], nh = in.aov.hits[p];
  const float fa = (float)na;
  float3 a = mk3(0.f), N = mk3(0.f);
  if (na) {
    a = mk3(in.aov.albedo[3 * p] / fa, in.aov.albedo[3 * p + 1] / fa, in.aov.albedo[3 * p + 2] / fa);
    N = mk3(in.aov.normal[3 * p] / fa, in.aov.normal[3 * p + 1] / fa, in.aov.normal[3 * p + 2] / fa);
  }
  const float z = nh ? in.aov.depth[p] / (float)nh : 0.f;
  const float3 m = mk3(a.x + 0.001f, a.y + 0.001f, a.z + 0.001f);
  sc.irr[0][p] = make_float4(c.x / m.x, c.y / m.y, c.z / m.z, 0.f);
  sc.guide[p] = make_float4(N.x, N.y, N.z, z);
  sc.mod[p] = make_float4(m.x, m.y, m.z, 0.f);
}

// The B3-spline taps h = (1/16, 1/4, 3/8, 1/4, 1/16) at offset d = -2..2.
__device__ __forceinline__ float hTap(int d) { return d == 0 ? 3.f / 8.f : (d == 1 || d == -1) ? 1.f / 4.f : 1.f / 16.f; }

// One a-trous iteration with step `step` at pixel (x, y).  sig2 = sigma_i * sigma_i.  LAST: out_p = e_p * (a_p + 0.001)
// into dst (3 floats per pixel); otherwise e_p into out.
template <bool LAST>
__device__ __forceinline__ void atrousPixel(const float4* __restrict__ in, const float4* __restrict__ guide, const float4* __restrict__ mod,
                                            float4* __restrict__ out, float* __restrict__ dst, int W, int H, int x, int y, int step,
                                            float sig2, float sigmaNormal, float sigmaDepth) {
  const size_t p = (size_t)y * W + x;
  const float4 ep = __ldg(&in[p]), gp = __ldg(&guide[p]);
  float sx = 0.f, sy = 0.f, sz = 0.f, sw = 0.f;
#pragma unroll
  for (int dy = -2; dy <= 2; ++dy) {
    const int qy = y + step * dy;
#pragma unroll
    for (int dx = -2; dx <= 2; ++dx) {
      const int qx = x + step * dx;
      if (qx < 0 || qx >= W || qy < 0 || qy >= H) continue;
      float4 eq = ep;
      float w = 1.f;
      if (dx != 0 || dy != 0) {
        const size_t q = (size_t)qy * W + qx;
        eq = __ldg(&in[q]);
        const float4 gq = __ldg(&guide[q]);
        const float ex = ep.x - eq.x, ey = ep.y - eq.y, ez = ep.z - eq.z;
        const float tc = (ex * ex + ey * ey + ez * ez) / sig2;
        const float tn = fmaxf(0.f, 1.f - (gp.x * gq.x + gp.y * gq.y + gp.z * gq.z)) / sigmaNormal;
        const float tz = fabsf(gp.w - gq.w) / (sigmaDepth * fmaxf(gp.w, gq.w) + 1e-30f);
        w = expf(-(tc + tn + tz));
      }
      const float k = hTap(dx) * hTap(dy) * w;
      sx += k * eq.x; sy += k * eq.y; sz += k * eq.z;
      sw += k;
    }
  }
  const float ox = sx / sw, oy = sy / sw, oz = sz / sw;
  if (LAST) {
    const float4 m = __ldg(&mod[p]);
    dst[3 * p] = ox * m.x; dst[3 * p + 1] = oy * m.y; dst[3 * p + 2] = oz * m.z;
  } else {
    out[p] = make_float4(ox, oy, oz, 0.f);
  }
}

// 16 x 16 pixel blocks; rows y0 + blockIdx.y * 16 .. (an image taller than 65535 blocks takes several launches).
template <bool LAST>
__global__ void __launch_bounds__(BX* BY) k_atrous(const float4* __restrict__ in, const float4* __restrict__ guide, const float4* __restrict__ mod,
                                                   float4* __restrict__ out, float* __restrict__ dst, int W, int H, int y0, int step,
                                                   float sig2, float sigmaNormal, float sigmaDepth) {
  const int x = blockIdx.x * BX + threadIdx.x, y = y0 + blockIdx.y * BY + threadIdx.y;
  if (x >= W || y >= H) return;
  atrousPixel<LAST>(in, guide, mod, out, dst, W, H, x, y, step, sig2, sigmaNormal, sigmaDepth);
}

__global__ void k_push_denoise_input(const uint32_t* __restrict__ ownedPix, uint32_t n, const float* __restrict__ accu,
                                     const uint32_t* __restrict__ skipped, AovBuffers aov, float* __restrict__ dstAccu,
                                     uint32_t* __restrict__ dstSkipped, AovBuffers dstAov) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const size_t p = ownedPix[j];
  for (int k = 0; k < 3; ++k) {
    dstAccu[3 * p + k] = accu[3 * p + k];
    dstAov.albedo[3 * p + k] = aov.albedo[3 * p + k];
    dstAov.normal[3 * p + k] = aov.normal[3 * p + k];
  }
  dstSkipped[p] = skipped ? skipped[p] : 0u;
  dstAov.depth[p] = aov.depth[p];
  dstAov.n[p] = aov.n[p];
  dstAov.hits[p] = aov.hits[p];
}

}  // namespace

size_t denoiseScratchBytes(uint32_t W, uint32_t H) { return (size_t)W * H * 4 * sizeof(float4); }

void launchDenoise(const DenoiseInput& in, const DenoiseParams& p, void* scratch, float* dst, cudaStream_t stream) {
  const size_t nPix = (size_t)in.W * in.H;
  const Scratch sc = scratchViews(scratch, nPix);
  k_denoise_prep<<<(unsigned)((nPix + 255) / 256), 256, 0, stream>>>(in, sc);
  const uint32_t maxRows = 65535u * BY;   // the grid's y dimension is limited to 65535 blocks
  for (uint32_t i = 0; i < p.iterations; ++i) {
    const float sigma = p.sigmaColor * ldexpf(1.f, -(int)i);   // exact: a power-of-two scale
    const float4* src = sc.irr[i & 1];
    for (uint32_t y0 = 0; y0 < in.H; y0 += maxRows) {
      const uint32_t rows = std::min(in.H - y0, maxRows);
      const dim3 block(BX, BY), grid((in.W + BX - 1) / BX, (rows + BY - 1) / BY);
      if (i + 1 == p.iterations)
        k_atrous<true><<<grid, block, 0, stream>>>(src, sc.guide, sc.mod, nullptr, dst, (int)in.W, (int)in.H, (int)y0, 1 << i,
                                                   sigma * sigma, p.sigmaNormal, p.sigmaDepth);
      else
        k_atrous<false><<<grid, block, 0, stream>>>(src, sc.guide, sc.mod, sc.irr[(i + 1) & 1], nullptr, (int)in.W, (int)in.H, (int)y0,
                                                    1 << i, sigma * sigma, p.sigmaNormal, p.sigmaDepth);
    }
  }
}

void launchPushDenoiseInput(const uint32_t* ownedPix, uint32_t n, const float* accu, const uint32_t* skipped, const AovBuffers& aov,
                            float* dstAccu, uint32_t* dstSkipped, const AovBuffers& dstAov, cudaStream_t stream) {
  if (n) k_push_denoise_input<<<(n + 255) / 256, 256, 0, stream>>>(ownedPix, n, accu, skipped, aov, dstAccu, dstSkipped, dstAov);
}
