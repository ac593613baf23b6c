/* mox_debug.h — test hooks exported by libmox.so next to the drop-in ABI of mox.h.  They have no
 * counterpart in the reference; tests/ uses them to check GPU building blocks in isolation. */
#ifndef MOX_DEBUG_H
#define MOX_DEBUG_H
#include "mox.h"
#ifdef __cplusplus
extern "C" {
#endif
/* Stable LSD radix sort of (key, value) pairs with the builder's onesweep kernels.
 * Host pointers; sorted in place. */
int mox_debug_radix_sort(mox_ctx*, uint32_t* keys, uint32_t* vals, size_t n);
/* Copy one array of the built acceleration structure to host memory dst (cap bytes); *out_bytes (may be NULL)
 * receives its size, which is 0 for the wide arrays when no wide BVH is in use.  dst may be NULL to ask for the size. */
#define MOX_DEBUG_ACCEL_NODES 0    /* binary nodes, 64 bytes each */
#define MOX_DEBUG_ACCEL_NODES8 1   /* compressed 8-wide nodes, 80 bytes each */
#define MOX_DEBUG_ACCEL_PACKED 2   /* primitive records in binary leaf order, 48 bytes each */
#define MOX_DEBUG_ACCEL_PACKED8 3  /* primitive records in wide leaf order */
int mox_debug_read_accel(mox_ctx*, int which, void* dst, size_t cap, size_t* out_bytes);
#ifdef __cplusplus
}
#endif
#endif
