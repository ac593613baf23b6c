// traverse_job.h — launch descriptor of the persistent traversal kernel.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#ifndef MOX_TRAV_TPB
#define MOX_TRAV_TPB 128   // threads per CTA of the persistent traversal kernels (64 x 18 CTAs per SM and 256 x 4 measured: see DESIGN.md)
#endif

// One batch of rays for the persistent traversal kernel.
//   rayO[id] = (origin, tmin)   rayD[id] = (direction, tmax); tmax < 0 marks an unused slot
//   queue    : optional indirection, ray id = queue[i] for i < count
//   cursor   : global fetch cursor, zeroed before the launch
//   hits     : closest hit, raw query form: hits[id] = (t, prim id as int bits or -1, beta, gamma)
//   hits2    : closest hit, render form (CLASSIFY kernels): hits2[id] = (t, prim id | class << 28, or -1)
//   shC      : any hit: shC[id].xyz *= transmittance
struct TraceJob {
  const float4* rayO;
  const float4* rayD;
  const uint32_t* queue;
  uint32_t count;
  const uint32_t* countPtr;  // when set, the ray count is read from device memory instead
  uint32_t originMod;        // when non-zero, the origin of ray id is rayO[id % originMod]
  uint32_t originMagic;      // floor(2^32 / originMod) + 1: id / originMod = umulhi(id, magic) or one less (set by launchTraverse)
  uint32_t* cursor;
  float4* hits;
  float2* hits2;
  float4* shC;
  uint32_t* counters;
  int fetchThreshold;   // refill idle lanes when fewer than this many lanes are traversing
};

// Light primitives of the terminal query (the bounce past rayMaxDepth, traverse_wide.cuh), one uint4 each:
//   x = primitive id | MOX_CLASS_LIGHT << 28 (the hit record's form), y = primitive type (PT_QUAD or PT_SPHERE; any
//   other value marks a primitive the build left out, which is skipped), z = index into analytic[].
#define MOX_TERMINAL_LIGHTS_MAX 32
#define MOX_TERMINAL_EXCLUDED 3u
struct TerminalLights {
  const uint4* list = nullptr;
  int n = 0;
  int missIsAbsorb = 0;   // bgColor and absorbColor are bit-equal: a ray that hits no light needs no traversal
};

