// gpu_types.h — HBM data layout of a built scene (all arrays 16-byte aligned; see DESIGN.md).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "mox.h"

enum PrimType : uint32_t { PT_TRI = 0, PT_SPHERE = 1, PT_QUAD = 2 };

// 80-byte material record: kind + the reference's parameter struct verbatim.
struct __align__(16) GpuMaterial {
  int kind;  // mox_material_kind
  int pad;
  union {
    LambertianParams lam;
    MetalParams met;
    GlassParams gls;
    DisneyParams dis;
    LightParams lgt;
  };
};
static_assert(sizeof(GpuMaterial) == 80, "GpuMaterial");

// Per primitive id: type (2 bits) | material index (30 bits); index into tris / analytic.
struct PrimDesc { uint32_t typeMat; uint32_t geom; };

// Global (mesh-base-added) indices of a triangle; n[0] < 0: no normals; t[0] < 0: no texcoords.
struct TriIdx { int v[3]; int n[3]; int t[3]; };

// Sphere: a = (center, radius).  Quad: a = plane, b = v1, c = v2, d = anchor (QuadParams).
struct __align__(16) Analytic { float4 a, b, c, d; };

// Binary BVH node in the Aila–Laine layout: both child boxes in the parent, 64 bytes.
//   c0xy = (c0.lo.x, c0.hi.x, c0.lo.y, c0.hi.y)   c1xy likewise
//   cz   = (c0.lo.z, c0.hi.z, c1.lo.z, c1.hi.z)
//   ref  = (child0, child1, -, -): >= 0 inner node index; < 0 leaf: ~((first << 3) | (count - 1))
//          over the leaf-ordered packed primitive array; 0x80000000 = empty child (its box is the
//          point (MOX_FAR, MOX_FAR, MOX_FAR), which no ray reaches, so the hot loop never tests for it).
struct __align__(16) BvhNode2 { float4 c0xy, c1xy, cz; int4 ref; };
static_assert(sizeof(BvhNode2) == 64, "BvhNode2");
#define MOX_EMPTY_CHILD ((int)0x80000000)
#define MOX_FAR 3.0e38f   // box coordinates of an empty child: every slab test misses it
#ifndef MOX_LEAF_MAX
#define MOX_LEAF_MAX 2  // measured on the 1M-triangle bench: 2 -> 946, 1 -> 940, 3 -> 935, 4 -> 909, 8 -> 837 Mrays/s
#endif
// Per-lane traversal stack entries (far children only): a tree of depth d needs at most d.
// The Karras radix tree is at most 62 deep (30 key bits + 32 index tie-break bits); PLOC trees
// are usually ~2 log2(n) deep but can degenerate on scenes with very uneven primitive sizes
// (measured: 103 levels on the coffee scene), so the builder checks the depth and falls back to
// the radix tree when a PLOC tree would not fit.
#define MOX_TRAVERSAL_STACK 128

// Compressed 8-wide node (after Ylitie, Karras, Laine 2017), 80 bytes = 5 x float4, 16-byte aligned:
//   n0 = (p.x, p.y, p.z, ex | ey << 8 | ez << 16 | imask << 24)   p: box minimum; e*: biased exponents of the
//        per-axis grid scale 2^(e-127); imask bit s: the child in slot s is an inner node
//   n1 = (childBase, primBase, valid, group)
//        inner children are stored contiguously from childBase in slot order; the primitives of all leaf
//        children are contiguous from primBase in the wide-leaf-ordered packed array, in slot order.
//        Hit bits have FIXED positions per slot s: bit 24 + s = "the inner child in slot s is hit", bits 2s and
//        2s + 1 = "primitive 0 / 1 of the leaf child in slot s is hit" (a leaf child holds <= 2 primitives), so the
//        traversal ORs one compile-time constant per hit child and masks the result once:
//        valid = imask << 24 | V,  V = the primitive bits that exist (16 bits);  group = V << 8 | imask (the low
//        24 bits of the lane's node-group word).  The rank of primitive bit k among V's set bits is its offset
//        from primBase.
//   n2 = (qlo.x[0..3], qlo.x[4..7], qlo.y[0..3], qlo.y[4..7])      child boxes, 8 bit per plane:
//   n3 = (qlo.z[0..3], qlo.z[4..7], qhi.x[0..3], qhi.x[4..7])      lo = p + qlo * scale (rounded down),
//   n4 = (qhi.y[0..3], qhi.y[4..7], qhi.z[0..3], qhi.z[4..7])      hi = p + qhi * scale (rounded up)
// Slots are assigned by octant of the child centroid so that (slot ^ octant-mask of the ray) orders
// the children front to back without computing distances.
struct __align__(16) BvhNode8 { float4 n0, n1, n2, n3, n4; };
static_assert(sizeof(BvhNode8) == 80, "BvhNode8");
#ifndef MOX_WIDE_LEAF_MAX
#define MOX_WIDE_LEAF_MAX 2  // measured: 2 -> 1037, 1 -> 1036, 3 -> 1013 Mrays/s (binary BVH: 1029)
#endif
static_assert(MOX_WIDE_LEAF_MAX <= 2, "the fixed-slot node layout has two primitive bits per slot: a wide leaf holds at most two primitives");

// Leaf-ordered packed primitive, 3 x float4 = 48 bytes per slot.
//   triangle: (p0, idbits) (e0 = p1 - p0, -) (e1 = p0 - p2, -); with MOX_ACCEL_WATERTIGHT the raw vertices (p0) (p1) (p2)
//   analytic: (index into Analytic[] as int bits, -, -, idbits)
// idbits = prim id | type << 30.
#define MOX_PACKED_F4 3

// How a primitive answers a shadow ray (the order-independent any-hit rule, Material.cu:225-232): stored in
// word 1 .w of its packed record so an occluded shadow ray needs no material lookup.
#define MOX_SHADOW_INVISIBLE 0u  // no any-hit program (lambertian, metal, glass, light)
#define MOX_SHADOW_BLOCKS 1u     // Disney NORMAL
#define MOX_SHADOW_TINTS 2u      // Disney GLASS: attenuation *= color
// Which closest-hit program the primitive runs, bits 2..4 of the same word: the traversal kernel writes it into
// the hit record, so classifying a hit needs no prims -> mats -> brdfType chain (three dependent loads).
#define MOX_CLASS_LAMBERT 0u
#define MOX_CLASS_METAL 1u
#define MOX_CLASS_DIELECTRIC 2u  // glass, and Disney with brdfType GLASS
#define MOX_CLASS_DISNEY 3u      // Disney NORMAL
#define MOX_CLASS_LIGHT 4u
#define MOX_CLASS_SHIFT 2
// Hit record of the render path: (t, bits) with bits = primitive id | class << 28; -1 = miss; -2 = the path was
// shaded and did not spawn a ray (nothing more to add).  Primitive ids are therefore limited to 2^28.
#define MOX_HIT_ID_BITS 28
#define MOX_HIT_ID_MASK 0x0fffffffu
#define MOX_HIT_MISS (-1)
#define MOX_HIT_DEAD (-2)

// Per-triangle shading record, 128 bytes, indexed like `tris`:
//   r0 = p0.xyz | flags (bit 0: has normals, bit 1: has uvs)     r1 = p1.xyz | uv0.x     r2 = p2.xyz | uv0.y
//   r3 = n0.xyz | uv1.x     r4 = n1.xyz | uv1.y     r5 = n2.xyz | uv2.x     r6 = uv2.y, -, -, -     r7 unused
#define MOX_SHADE_REC_F4 8

struct SceneView {
  const BvhNode2* nodes;
  const float4* packed;
  const BvhNode8* nodes8;   // compressed wide BVH (null: traverse the binary BVH)
  const float4* packed8;    // primitives in wide-leaf order
  const Analytic* analytic;
  const PrimDesc* prims;
  const GpuMaterial* mats;
  const float* verts;    // xyz
  const float* normals;  // xyz
  const float* uvs;      // uv
  const TriIdx* tris;
  const float4* shadeRec;   // MOX_SHADE_REC_F4 float4 per triangle: what a hit needs for shading, pre-gathered (null: gather through tris)
  const LightParams* lights;
  const float4* lightN;     // normalize(lights[i].normal), precomputed at upload
  const cudaTextureObject_t* textures;  // id - 1 -> float4 texture, bilinear, REPEAT, normalized coords
  int nLights;
  int nPrims;
  uint32_t nNodes8;         // nodes of the wide BVH
  int watertight;           // packed / packed8 triangle records hold raw vertices; the traversal runs the watertight test
};

struct RenderParams {
  uint32_t W, H, maxDepth;
  float eps, minIntensity;
  float3 absorb, bad, bg;
  CamParams cam;
  int rngMode;
};
