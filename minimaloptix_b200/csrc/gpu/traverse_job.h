// traverse_job.h — launch descriptor of the persistent traversal kernel.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#ifndef MOX_TRAV_TPB
#define MOX_TRAV_TPB 128   // threads per CTA of the persistent traversal kernels (64 x 18 CTAs per SM and 256 x 4 measured: see DESIGN.md)
#endif

// Device counters (uint32 words).  Words 0..7 exist once per bounce in a small ring (LaunchCtx::bc points at the
// current bounce's block), so the host never has to zero them between two kernels of the same bounce loop:
//   C_NEXT  rays spawned by this bounce's shade kernels (= the next extend launch's ray count, read on the device)
//   C_MAT0+k paths binned into material queue k by this bounce's classify kernel
//   C_SHQ   shadow rays queued by this bounce's Disney kernel
// Words 8.. are per batch.  A *_LO word and the word after it hold one 64-bit count (low word first).
enum CounterSlot { C_NEXT = 0, C_MAT0 = 1 /* ..4 */, C_SHQ = 5 /* shadow queue length */, C_BOUNCE_WORDS = 8,
                   C_NONFINITE = 8, C_SHADOW = 9, C_NODEVIS_LO = 10, C_NODEVIS_HI = 11,
                   C_PRIMTEST_LO = 12, C_PRIMTEST_HI = 13, C_CURSOR = 14, C_CURSOR_SHADOW = 15 /* the shadow launch may overlap the next extend launch */,
                   C_NODEVIS_SH_LO = 16, C_PRIMTEST_SH_LO = 18, C_SH_BLOCKED = 20, C_SH_TINTED = 21, C_WORDS = 24 };
constexpr int BOUNCE_RING = 4;   // per-bounce counter blocks kept alive at once

// One batch of rays for the persistent traversal kernel.
//   rayO[id] = (origin, tmin)   rayD[id] = (direction, tmax); tmax < 0 marks an unused slot
//   queue    : optional indirection, ray id = queue[i] for i < count
//   cursor   : global fetch cursor, zeroed before the launch
//   hits     : closest hit, raw query form: hits[id] = (t, prim id as int bits or -1, beta, gamma)
//   hits2    : closest hit, render form (CLASSIFY kernels): hits2[id] = (t, prim id | class << 28, or -1)
//   shC      : any hit: shC[id].xyz *= transmittance
struct TraceJob {
  const float4* rayO = nullptr;
  const float4* rayD = nullptr;
  const uint32_t* queue = nullptr;
  uint32_t count = 0;
  const uint32_t* countPtr = nullptr;  // when set, the ray count is read from device memory instead
  uint32_t originMod = 0;              // when non-zero, the origin of ray id is rayO[id % originMod]
  uint32_t originMagic = 0;            // floor(2^32 / originMod) + 1: id / originMod = umulhi(id, magic) or one less (set by launchTraverse)
  uint32_t* cursor = nullptr;
  float4* hits = nullptr;
  float2* hits2 = nullptr;
  float4* shC = nullptr;
  uint32_t* counters = nullptr;        // CounterSlot words
  int fetchThreshold = 0;              // refill idle lanes when fewer than this many lanes are traversing (set by launchTraverse)
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

