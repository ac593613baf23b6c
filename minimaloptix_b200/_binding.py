"""ctypes binding of the render C ABI (include/mox.h).

The same binding code serves any library that exports that ABI under a symbol prefix: the
product library libmox.so (prefix ``mox_``) and, for tests only, the CPU oracle (prefix
``orc_``).  Nothing in this package loads the oracle.
"""
import ctypes as C
import os

import numpy as np

from . import structs as S

_MAT_STRUCT = {S.MAT_LAMBERTIAN: S.LambertianParams, S.MAT_METAL: S.MetalParams, S.MAT_GLASS: S.GlassParams,
               S.MAT_DISNEY: S.DisneyParams, S.MAT_LIGHT: S.LightParams}

_u32, _u64, _i32, _f32 = C.c_uint32, C.c_uint64, C.c_int32, C.c_float
_vp, _fp = C.c_void_p, C.POINTER(C.c_float)

# name -> (restype, argtypes) for everything include/mox.h declares.
SIGNATURES = {
    "create": (C.c_int, [C.POINTER(_vp), C.c_int]),
    "destroy": (None, [_vp]),
    "last_error": (C.c_char_p, [_vp]),
    "abi_version": (C.c_int, []),
    "set_globals": (C.c_int, [_vp, _u32, _u32, _u32, _f32, _f32, _fp, _fp, _fp]),
    "set_camera": (C.c_int, [_vp, C.POINTER(S.CamParams)]),
    "set_rng_mode": (C.c_int, [_vp, C.c_int]),
    "set_partition": (C.c_int, [_vp, _u32, _u32, _u32]),
    "add_texture_rgba32f": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    "add_sphere": (C.c_int, [_vp, C.POINTER(S.SphereParams), C.c_int, _vp, C.POINTER(_u32)]),
    "add_quad": (C.c_int, [_vp, C.POINTER(S.QuadParams), C.c_int, _vp, C.POINTER(_u32)]),
    "add_mesh": (C.c_int, [_vp, _vp, C.c_size_t, _vp, C.c_size_t, _vp, C.c_size_t, _vp, _vp, _vp, C.c_size_t,
                           C.c_int, _vp, C.POINTER(_u32)]),
    "set_lights": (C.c_int, [_vp, _vp, C.c_size_t]),
    "clear_scene": (C.c_int, [_vp]),
    "build_accel": (C.c_int, [_vp, _u32, C.POINTER(_f32)]),
    "launch": (C.c_int, [_vp, _i32]),
    "render": (C.c_int, [_vp, _u32, _u32]),
    "render_adaptive": (C.c_int, [_vp, _u32, _u32, C.POINTER(S.Adaptive), C.POINTER(_u64)]),
    "read_sample_counts": (C.c_int, [_vp, _vp]),
    "read_accum": (C.c_int, [_vp, _vp]),
    "map_accum": (C.c_int, [_vp, C.POINTER(_fp)]),
    "unmap_accum": (C.c_int, [_vp]),
    "clear_accum": (C.c_int, [_vp]),
    "set_accum": (C.c_int, [_vp, _vp, _u64]),
    "update_sphere": (C.c_int, [_vp, _u32, C.POINTER(S.SphereParams)]),
    "update_mesh": (C.c_int, [_vp, _u32, _vp, C.c_size_t, _vp, C.c_size_t]),
    "owned_pixels": (C.c_int, [_vp, _u32, C.POINTER(_u64)]),
    "pack_owned": (C.c_int, [_vp, _vp]),
    "unpack_owned": (C.c_int, [_vp, _u32, _vp]),
    "get_stats": (C.c_int, [_vp, C.POINTER(S.Stats)]),
    "device_count": (C.c_int, [_vp]),
    "get_device_stats": (C.c_int, [_vp, C.c_int, C.POINTER(S.Stats)]),
    "read_accum_begin": (C.c_int, [_vp]),
    "read_accum_end": (C.c_int, [_vp, C.POINTER(_fp)]),
    "trace_closest": (C.c_int, [_vp, _vp, C.c_size_t, _vp]),
    "trace_shadow": (C.c_int, [_vp, _vp, C.c_size_t, _vp]),
    "set_aovs": (C.c_int, [_vp, C.c_int]),
    "read_aovs": (C.c_int, [_vp, _vp, _vp, _vp]),
    "denoise": (C.c_int, [_vp, C.POINTER(S.DenoiseParams), _vp, C.POINTER(_f32)]),
}
# Only the GPU library has the device-pointer query.
GPU_ONLY = {"create_multi": (C.c_int, [C.POINTER(_vp), C.POINTER(C.c_int), C.c_int]),
            "gather_export": (C.c_int, [_vp, C.c_int, _vp]),
            "gather_import": (C.c_int, [_vp, C.c_int, _vp]),
            "gather_push": (C.c_int, [_vp, C.c_int]),
            "read_gathered_begin": (C.c_int, [_vp, C.c_int]),
            "read_gathered_end": (C.c_int, [_vp, C.c_int, C.POINTER(_fp)]),
            "trace_closest_device": (C.c_int, [_vp, _vp, C.c_size_t, _vp, C.POINTER(_f32)]),
            "debug_radix_sort": (C.c_int, [_vp, _vp, _vp, C.c_size_t]),
            "debug_read_accel": (C.c_int, [_vp, C.c_int, _vp, C.c_size_t, C.POINTER(C.c_size_t)])}
# Arrays of a built acceleration structure, in the order of include/mox_debug.h's MOX_DEBUG_ACCEL_*.
ACCEL_ARRAYS = ("nodes", "nodes8", "packed", "packed8")


class MoxError(RuntimeError):
    pass


class Backend:
    """A loaded library exporting the mox C ABI under ``prefix``."""

    def __init__(self, lib_path, prefix, extra=None):
        if not os.path.exists(lib_path):
            raise MoxError(f"{lib_path} not found — run `make` (or __graft_entry__.build()) first")
        self.path, self.prefix = lib_path, prefix
        self.lib = C.CDLL(lib_path)
        sigs = dict(SIGNATURES)
        sigs.update(extra or {})
        for name, (res, args) in sigs.items():
            fn = getattr(self.lib, prefix + name)  # AttributeError if the symbol is missing
            fn.restype, fn.argtypes = res, args
            setattr(self, name, fn)

    def context(self, device=0):
        return Context(self, device)

    def multi_context(self, devices):
        """One handle rendering on several GPUs of this process (mox_create_multi)."""
        return Context(self, list(devices))


def _f32c(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _i32c(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _ptr(a):
    return None if a is None else a.ctypes.data_as(_vp)


class Context:
    """One render context (the reference's optix::Context for this path)."""

    def __init__(self, backend, device=0):
        self.b = backend
        self.h = _vp()
        if isinstance(device, (list, tuple)):
            ids = (C.c_int * len(device))(*device)
            rc = backend.create_multi(C.byref(self.h), ids, len(device))
        else:
            rc = backend.create(C.byref(self.h), device)
        if rc != 0:
            raise MoxError(f"{backend.prefix}create failed ({rc}): {backend.last_error(None).decode()}")
        self.width = self.height = 0

    def _ck(self, rc, what):
        if rc != 0:
            raise MoxError(f"{self.b.prefix}{what} failed ({rc}): {self.b.last_error(self.h).decode()}")

    def close(self):
        if self.h:
            self.b.destroy(self.h)
            self.h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- globals / camera
    def set_globals(self, width, height, max_depth=256, eps=1e-3, min_intensity=1e-3, absorb=(0, 0, 0),
                    bad=(1, 1, 1), bg=(0, 0, 0)):
        a, bd, g = (C.c_float * 3)(*absorb), (C.c_float * 3)(*bad), (C.c_float * 3)(*bg)
        self._ck(self.b.set_globals(self.h, width, height, max_depth, eps, min_intensity, a, bd, g), "set_globals")
        self.width, self.height = width, height

    def set_camera(self, cam):
        self._ck(self.b.set_camera(self.h, C.byref(cam)), "set_camera")

    def set_rng_mode(self, mode):
        self._ck(self.b.set_rng_mode(self.h, mode), "set_rng_mode")

    def set_partition(self, rank, world, tile=32):
        self._ck(self.b.set_partition(self.h, rank, world, tile), "set_partition")

    # -- scene
    def _mat(self, kind, params):
        want = _MAT_STRUCT[kind]
        if not isinstance(params, want):
            raise TypeError(f"material kind {kind} needs {want.__name__}")
        return C.cast(C.byref(params), _vp)

    def add_sphere(self, sphere, kind, params):
        pid = _u32()
        self._ck(self.b.add_sphere(self.h, C.byref(sphere), kind, self._mat(kind, params), C.byref(pid)), "add_sphere")
        return pid.value

    def add_quad(self, quad, kind, params):
        pid = _u32()
        self._ck(self.b.add_quad(self.h, C.byref(quad), kind, self._mat(kind, params), C.byref(pid)), "add_quad")
        return pid.value

    def add_mesh(self, vertices, v_idx, kind, params, normals=None, n_idx=None, texcoords=None, t_idx=None):
        v = _f32c(vertices).reshape(-1, 3)
        vi = _i32c(v_idx).reshape(-1, 3)
        n = None if normals is None else _f32c(normals).reshape(-1, 3)
        ni = None if n_idx is None else _i32c(n_idx).reshape(-1, 3)
        t = None if texcoords is None else _f32c(texcoords).reshape(-1, 2)
        ti = None if t_idx is None else _i32c(t_idx).reshape(-1, 3)
        pid = _u32()
        self._ck(self.b.add_mesh(self.h, _ptr(v), len(v), _ptr(n), 0 if n is None else len(n), _ptr(t),
                                 0 if t is None else len(t), _ptr(vi), _ptr(ni), _ptr(ti), len(vi), kind,
                                 self._mat(kind, params), C.byref(pid)), "add_mesh")
        return pid.value

    def add_texture(self, texels_rgba):
        t = _f32c(texels_rgba)
        h, w = t.shape[0], t.shape[1]
        tid = C.c_int()
        self._ck(self.b.add_texture_rgba32f(self.h, _ptr(t), w, h, C.byref(tid)), "add_texture_rgba32f")
        return tid.value

    def set_lights(self, lights):
        arr = (S.LightParams * max(1, len(lights)))(*lights)
        self._ck(self.b.set_lights(self.h, C.cast(arr, _vp), len(lights)), "set_lights")

    def clear_scene(self):
        self._ck(self.b.clear_scene(self.h), "clear_scene")

    def build_accel(self, flags=0):
        ms = _f32()
        self._ck(self.b.build_accel(self.h, flags, C.byref(ms)), "build_accel")
        return ms.value

    # -- render
    def launch(self, seed):
        self._ck(self.b.launch(self.h, int(np.int32(np.uint32(seed & 0xFFFFFFFF)))), "launch")

    def render(self, spp, seed):
        self._ck(self.b.render(self.h, spp, seed & 0xFFFFFFFF), "render")

    def render_adaptive(self, spp, seed, rel_error, abs_error=0.0, min_spp=16, round_spp=8):
        """mox_render_adaptive: up to spp more samples per pixel, until its estimated error is below the threshold.
        Returns the number of pixel-samples traced."""
        p = S.Adaptive(round_spp, min_spp, rel_error, abs_error)
        n = _u64()
        self._ck(self.b.render_adaptive(self.h, spp, seed & 0xFFFFFFFF, C.byref(p), C.byref(n)), "render_adaptive")
        return n.value

    def read_sample_counts(self):
        """Samples per pixel, (H, W) uint32, row 0 = bottom: divide the accumulation buffer by it."""
        out = np.empty((self.height, self.width), dtype=np.uint32)
        self._ck(self.b.read_sample_counts(self.h, _ptr(out)), "read_sample_counts")
        return out

    def set_aovs(self, on):
        """mox_set_aovs: accumulate every camera sample's first-hit albedo, normal and depth (on) or free them (off)."""
        self._ck(self.b.set_aovs(self.h, 1 if on else 0), "set_aovs")

    def read_aovs(self):
        """The AOV means, row 0 = bottom: (albedo (H, W, 3), normal (H, W, 3), depth (H, W))."""
        a = np.empty((self.height, self.width, 3), dtype=np.float32)
        n = np.empty((self.height, self.width, 3), dtype=np.float32)
        z = np.empty((self.height, self.width), dtype=np.float32)
        self._ck(self.b.read_aovs(self.h, _ptr(a), _ptr(n), _ptr(z)), "read_aovs")
        return a, n, z

    def denoise(self, iterations=S.DENOISE_DEFAULTS["iterations"], sigma_color=S.DENOISE_DEFAULTS["sigma_color"],
                sigma_normal=S.DENOISE_DEFAULTS["sigma_normal"], sigma_depth=S.DENOISE_DEFAULTS["sigma_depth"]):
        """mox_denoise: the edge-avoiding a-trous filter of the mean colour, guided by the AOVs.
        Returns (image (H, W, 3), ms of the filter kernels)."""
        p = S.DenoiseParams(iterations, sigma_color, sigma_normal, sigma_depth)
        out = np.empty((self.height, self.width, 3), dtype=np.float32)
        ms = _f32()
        self._ck(self.b.denoise(self.h, C.byref(p), _ptr(out), C.byref(ms)), "denoise")
        return out, ms.value

    def read_accum(self):
        out = np.empty((self.height, self.width, 3), dtype=np.float32)
        self._ck(self.b.read_accum(self.h, _ptr(out)), "read_accum")
        return out

    def map_accum(self):
        """Zero-copy view (H, W, 3) of the pinned host copy; valid until the next map/read."""
        p = _fp()
        self._ck(self.b.map_accum(self.h, C.byref(p)), "map_accum")
        return np.ctypeslib.as_array(p, shape=(self.height, self.width, 3))

    def read_accum_begin(self):
        """Start the asynchronous read-back (snapshot / multi-GPU gather + device->host copy)."""
        self._ck(self.b.read_accum_begin(self.h), "read_accum_begin")

    def read_accum_end(self):
        """Wait for the read-back started last; zero-copy (H, W, 3) view of the pinned host image."""
        p = _fp()
        self._ck(self.b.read_accum_end(self.h, C.byref(p)), "read_accum_end")
        return np.ctypeslib.as_array(p, shape=(self.height, self.width, 3))

    def device_count(self):
        return self.b.device_count(self.h)

    def device_stats(self, index):
        st = S.Stats()
        self._ck(self.b.get_device_stats(self.h, index, C.byref(st)), "get_device_stats")
        return st.asdict()

    # -- peer-memory tile gather across processes (one process per GPU)
    def gather_export(self, which):
        buf = C.create_string_buffer(64)
        self._ck(self.b.gather_export(self.h, which, C.cast(buf, _vp)), "gather_export")
        return buf.raw

    def gather_import(self, which, handle):
        buf = C.create_string_buffer(handle, 64)
        self._ck(self.b.gather_import(self.h, which, C.cast(buf, _vp)), "gather_import")

    def gather_push(self, which):
        self._ck(self.b.gather_push(self.h, which), "gather_push")

    def read_gathered_begin(self, which):
        self._ck(self.b.read_gathered_begin(self.h, which), "read_gathered_begin")

    def read_gathered_end(self, which):
        p = _fp()
        self._ck(self.b.read_gathered_end(self.h, which, C.byref(p)), "read_gathered_end")
        return np.ctypeslib.as_array(p, shape=(self.height, self.width, 3))

    def set_accum(self, accum, launches):
        a = _f32c(accum)
        self._ck(self.b.set_accum(self.h, _ptr(a), launches), "set_accum")

    def update_sphere(self, prim_id, sphere):
        self._ck(self.b.update_sphere(self.h, prim_id, C.byref(sphere)), "update_sphere")

    def update_mesh(self, first_prim_id, vertices, normals=None):
        """New vertices (and normals) of the mesh whose first primitive id add_mesh returned; build or refit next."""
        v = _f32c(vertices).reshape(-1, 3)
        n = None if normals is None else _f32c(normals).reshape(-1, 3)
        self._ck(self.b.update_mesh(self.h, first_prim_id, _ptr(v), len(v), _ptr(n), 0 if n is None else len(n)), "update_mesh")

    def clear_accum(self):
        self._ck(self.b.clear_accum(self.h), "clear_accum")

    def owned_pixels(self, rank):
        n = _u64()
        self._ck(self.b.owned_pixels(self.h, rank, C.byref(n)), "owned_pixels")
        return n.value

    def pack_owned(self, ptr):
        self._ck(self.b.pack_owned(self.h, _vp(ptr)), "pack_owned")

    def unpack_owned(self, rank, ptr):
        self._ck(self.b.unpack_owned(self.h, rank, _vp(ptr)), "unpack_owned")

    def stats(self):
        s = S.Stats()
        self._ck(self.b.get_stats(self.h, C.byref(s)), "get_stats")
        return s.asdict()

    # -- raw queries
    def trace_closest(self, rays):
        r = _f32c(rays).reshape(-1, 8)
        hits = np.empty((len(r), 4), dtype=np.float32)
        self._ck(self.b.trace_closest(self.h, _ptr(r), len(r), _ptr(hits)), "trace_closest")
        return hits[:, 0].copy(), hits[:, 1].copy().view(np.int32), hits[:, 2].copy(), hits[:, 3].copy()

    def trace_closest_device(self, rays_ptr, n, hits_ptr):
        ms = _f32()
        self._ck(self.b.trace_closest_device(self.h, _vp(rays_ptr), n, _vp(hits_ptr), C.byref(ms)), "trace_closest_device")
        return ms.value

    def debug_radix_sort(self, keys, vals):
        k = np.ascontiguousarray(keys, dtype=np.uint32).copy()
        v = np.ascontiguousarray(vals, dtype=np.uint32).copy()
        self._ck(self.b.debug_radix_sort(self.h, _ptr(k), _ptr(v), len(k)), "debug_radix_sort")
        return k, v

    def debug_read_accel(self, which):
        """Bytes of one array of the built acceleration structure (a name of ACCEL_ARRAYS) as uint8."""
        k = ACCEL_ARRAYS.index(which)
        size = C.c_size_t()
        self._ck(self.b.debug_read_accel(self.h, k, None, 0, C.byref(size)), "debug_read_accel")
        out = np.empty(size.value, dtype=np.uint8)
        self._ck(self.b.debug_read_accel(self.h, k, _ptr(out), len(out), C.byref(size)), "debug_read_accel")
        return out

    def trace_shadow(self, rays):
        r = _f32c(rays).reshape(-1, 8)
        out = np.empty((len(r), 3), dtype=np.float32)
        self._ck(self.b.trace_shadow(self.h, _ptr(r), len(r), _ptr(out)), "trace_shadow")
        return out
