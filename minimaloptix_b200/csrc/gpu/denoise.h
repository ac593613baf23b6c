// denoise.h — the edge-avoiding a-trous wavelet filter of mox_denoise (the formula is in include/mox.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "wavefront.h"

struct DenoiseParams {
  uint32_t iterations;
  float sigmaColor, sigmaNormal, sigmaDepth;
};

// What the filter reads, full-frame W x H: the accumulation buffer, the launches each pixel sat out in adaptive renders
// (null: none), the launch count (a pixel's samples are launches - skipped) and the AOV sums.
struct DenoiseInput {
  const float* accu;
  const uint32_t* skipped;
  uint32_t launches;
  AovBuffers aov;
  uint32_t W, H;
};

// Bytes of scratch launchDenoise needs: two irradiance buffers, the guides and the albedo factor, a float4 each.
size_t denoiseScratchBytes(uint32_t W, uint32_t H);
// Enqueues the prep kernel and one kernel per iteration on `stream`; dst: W*H*3 floats on the device.
void launchDenoise(const DenoiseInput& in, const DenoiseParams& p, void* scratch, float* dst, cudaStream_t stream);
// Copies this context's share of the filter's inputs (colour, skipped launches, AOV sums) of the pixels ownedPix[0, n)
// into the full-frame arrays of `dst`, which may live on another GPU (peer stores).
void launchPushDenoiseInput(const uint32_t* ownedPix, uint32_t n, const float* accu, const uint32_t* skipped, const AovBuffers& aov,
                            float* dstAccu, uint32_t* dstSkipped, const AovBuffers& dstAov, cudaStream_t stream);
