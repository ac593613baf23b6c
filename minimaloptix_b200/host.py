"""ctypes binding of libmox_host.so (include/mox_host.h): scene loader, builders, image IO."""
import ctypes as C
import os

import numpy as np

from . import structs as S
from ._binding import MoxError

_HERE = os.path.dirname(os.path.abspath(__file__))
HOST_LIB = os.path.join(_HERE, "libmox_host.so")

_vp, _u32, _u64, _f3 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_float * 3


class SceneInfo(C.Structure):
    _fields_ = [("n_triangles", _u64), ("n_vertices", _u64), ("n_items", _u32), ("n_meshes", _u32),
                ("n_spheres", _u32), ("n_quads", _u32), ("n_lights", _u32), ("n_warnings", _u32),
                ("default_width", _u32), ("default_height", _u32), ("aabb_min", _f3), ("aabb_max", _f3),
                ("bg", _f3), ("look_from", _f3), ("look_at", _f3), ("up", _f3), ("vfov", C.c_float),
                ("aperture", C.c_float), ("focus", C.c_float)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(HOST_LIB):
            raise MoxError(f"{HOST_LIB} not found — run `make host`")
        L = C.CDLL(HOST_LIB)
        L.moxh_last_error.restype = C.c_char_p
        L.moxh_api_load.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(_vp)]
        L.moxh_api_free.argtypes = [_vp]
        L.moxh_set_quad_params.argtypes = [_f3, _f3, _f3, C.POINTER(S.QuadParams)]
        L.moxh_set_cam_params.argtypes = [_f3, _f3, _f3, C.c_float, C.c_float, C.c_float, C.c_float, C.POINTER(S.CamParams)]
        L.moxh_init_disney_params.argtypes = [C.POINTER(S.DisneyParams)]
        L.moxh_launch_seed.argtypes = [_u32, _u32]
        L.moxh_launch_seed.restype = C.c_int32
        L.moxh_scene_builtin.argtypes = [C.c_char_p, _u64, _u64, C.POINTER(_vp)]
        L.moxh_scene_load.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(_vp)]
        L.moxh_scene_free.argtypes = [_vp]
        L.moxh_scene_get_info.argtypes = [_vp, C.POINTER(SceneInfo)]
        L.moxh_scene_warning.argtypes = [_vp, _u32]
        L.moxh_scene_warning.restype = C.c_char_p
        L.moxh_scene_cam_params.argtypes = [_vp, _u32, _u32, C.POINTER(S.CamParams)]
        L.moxh_scene_light.argtypes = [_vp, _u32, C.POINTER(S.LightParams)]
        L.moxh_scene_mesh_info.argtypes = [_vp, _u32, C.POINTER(_u64), C.POINTER(_u64), C.POINTER(_u64), C.POINTER(_u64),
                                           C.POINTER(S.DisneyParams), C.c_char_p, C.c_size_t]
        L.moxh_scene_mesh_hash.argtypes = [_vp, _u32, C.POINTER(_u64 * 4)]
        L.moxh_scene_mesh_data.argtypes = [_vp, _u32, C.POINTER(C.POINTER(C.c_float)), C.POINTER(C.POINTER(C.c_int32))]
        L.moxh_scene_upload.argtypes = [_vp, _vp, _vp, _u32, _u32, _u32]
        L.moxh_scene_animate.argtypes = [_vp, C.c_float]
        L.moxh_scene_apply_spheres.argtypes = [_vp, _vp, _vp]
        L.moxh_accum_to_rgb8.argtypes = [_vp, _u32, _u32, C.c_float, _vp]
        L.moxh_accum_to_rgb8_counts.argtypes = [_vp, _u32, _u32, _vp, _vp]
        L.moxh_write_image.argtypes = [C.c_char_p, _vp, _u32, _u32]
        L.moxh_write_accum.argtypes = [C.c_char_p, _vp, _u32, _u32, _u64]
        L.moxh_read_accum.argtypes = [C.c_char_p, _vp, _u32, _u32, C.POINTER(_u64)]
        L.moxh_obj_parse_double.argtypes = [C.c_char_p, C.POINTER(C.c_double)]
        L.moxh_read_image.argtypes = [C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.POINTER(C.c_float))]
        L.moxh_free.argtypes = [_vp]
        L.moxh_scene_texture_count.argtypes = [_vp]
        L.moxh_scene_texture_count.restype = _u32
        _lib = L
    return _lib


def _err():
    return lib().moxh_last_error().decode()


def set_quad_params(anchor, v1, v2):
    q = S.QuadParams()
    lib().moxh_set_quad_params(_f3(*anchor), _f3(*v1), _f3(*v2), C.byref(q))
    return q


def set_cam_params(look_from, look_at, up, vfov, aspect, aperture, focus):
    c = S.CamParams()
    lib().moxh_set_cam_params(_f3(*look_from), _f3(*look_at), _f3(*up), vfov, aspect, aperture, focus, C.byref(c))
    return c


def init_disney_params():
    d = S.DisneyParams()
    lib().moxh_init_disney_params(C.byref(d))
    return d


def launch_seed(i, seed):
    return lib().moxh_launch_seed(i, seed & 0xFFFFFFFF)


def parse_double(text):
    d = C.c_double()
    ok = lib().moxh_obj_parse_double(text.encode(), C.byref(d))
    return d.value if ok else None


class ApiTable:
    """A backend bound through the host library's own dlopen/dlsym table."""

    def __init__(self, lib_path, prefix):
        self.h = _vp()
        if lib().moxh_api_load(lib_path.encode(), prefix.encode(), C.byref(self.h)) != 0:
            raise MoxError("moxh_api_load: " + _err())

    def __del__(self):
        if getattr(self, "h", None):
            lib().moxh_api_free(self.h)
            self.h = None


class Scene:
    """Flattened host scene (moxh_scene)."""

    def __init__(self, handle):
        self.h = handle

    @classmethod
    def builtin(cls, kind, param=0, seed=0):
        h = _vp()
        if lib().moxh_scene_builtin(kind.encode(), param, seed, C.byref(h)) != 0:
            raise MoxError("moxh_scene_builtin: " + _err())
        return cls(h)

    @classmethod
    def load(cls, scene_dir, name):
        h = _vp()
        if lib().moxh_scene_load(scene_dir.encode(), name.encode(), C.byref(h)) != 0:
            raise MoxError("moxh_scene_load: " + _err())
        return cls(h)

    def __del__(self):
        if getattr(self, "h", None):
            try:
                lib().moxh_scene_free(self.h)
            except TypeError:   # interpreter shutdown: the module globals are already gone
                pass
            self.h = None

    def info(self):
        i = SceneInfo()
        lib().moxh_scene_get_info(self.h, C.byref(i))
        return i

    def warnings(self):
        return [lib().moxh_scene_warning(self.h, k).decode() for k in range(self.info().n_warnings)]

    def cam_params(self, width, height):
        c = S.CamParams()
        lib().moxh_scene_cam_params(self.h, width, height, C.byref(c))
        return c

    def light(self, i):
        l = S.LightParams()
        if lib().moxh_scene_light(self.h, i, C.byref(l)) != 0:
            raise MoxError(_err())
        return l

    def mesh_info(self, m):
        nf, nv, nn, nt = _u64(), _u64(), _u64(), _u64()
        d = S.DisneyParams()
        name = C.create_string_buffer(256)
        if lib().moxh_scene_mesh_info(self.h, m, C.byref(nf), C.byref(nv), C.byref(nn), C.byref(nt), C.byref(d), name, 256) != 0:
            raise MoxError(_err())
        return dict(faces=nf.value, vertices=nv.value, normals=nn.value, texcoords=nt.value, disney=d, name=name.value.decode())

    def mesh_hash(self, m):
        out = (_u64 * 4)()
        lib().moxh_scene_mesh_hash(self.h, m, C.byref(out))
        return tuple(out)

    def mesh_arrays(self, m):
        info = self.mesh_info(m)
        v, vi = C.POINTER(C.c_float)(), C.POINTER(C.c_int32)()
        lib().moxh_scene_mesh_data(self.h, m, C.byref(v), C.byref(vi))
        verts = np.ctypeslib.as_array(v, shape=(info["vertices"], 3)).copy()
        idx = np.ctypeslib.as_array(vi, shape=(info["faces"], 3)).copy()
        return verts, idx

    def animate(self, time):
        if lib().moxh_scene_animate(self.h, time) != 0:
            raise MoxError(_err())

    def apply_spheres(self, api_table, ctx):
        if lib().moxh_scene_apply_spheres(self.h, api_table.h, ctx.h) != 0:
            raise MoxError("moxh_scene_apply_spheres: " + _err())

    def texture_count(self):
        return lib().moxh_scene_texture_count(self.h)

    def upload(self, api_table, ctx, width, height, max_depth):
        if lib().moxh_scene_upload(self.h, api_table.h, ctx.h, width, height, max_depth) != 0:
            raise MoxError("moxh_scene_upload: " + _err())
        ctx.width, ctx.height = width, height


def read_image(path):
    """Decode a texture image the way the loader does: (H, W, 4) float32, row 0 = bottom, alpha 1."""
    w, h, p = C.c_int(), C.c_int(), C.POINTER(C.c_float)()
    if lib().moxh_read_image(path.encode(), C.byref(w), C.byref(h), C.byref(p)) != 0:
        raise MoxError("moxh_read_image: " + _err())
    try:
        return np.ctypeslib.as_array(p, shape=(h.value, w.value, 4)).copy()
    finally:
        lib().moxh_free(p)


def accum_to_rgb8(accum, n_accum):
    a = np.ascontiguousarray(accum, dtype=np.float32)
    h, w = a.shape[:2]
    out = np.empty((h, w, 3), dtype=np.uint8)
    lib().moxh_accum_to_rgb8(a.ctypes.data_as(_vp), w, h, float(n_accum), out.ctypes.data_as(_vp))
    return out


def accum_to_rgb8_counts(accum, counts):
    """accum_to_rgb8 with a sample count per pixel ((H, W), as read_sample_counts returns it); 0 gives black."""
    a = np.ascontiguousarray(accum, dtype=np.float32)
    n = np.ascontiguousarray(counts, dtype=np.uint32)
    h, w = a.shape[:2]
    if n.shape != (h, w):
        raise ValueError(f"counts of shape {n.shape} for a {h}x{w} image")
    out = np.empty((h, w, 3), dtype=np.uint8)
    lib().moxh_accum_to_rgb8_counts(a.ctypes.data_as(_vp), w, h, n.ctypes.data_as(_vp), out.ctypes.data_as(_vp))
    return out


def write_image(path, rgb8):
    r = np.ascontiguousarray(rgb8, dtype=np.uint8)
    if lib().moxh_write_image(path.encode(), r.ctypes.data_as(_vp), r.shape[1], r.shape[0]) != 0:
        raise MoxError(_err())


def write_accum(path, accum, launches):
    a = np.ascontiguousarray(accum, dtype=np.float32)
    if lib().moxh_write_accum(path.encode(), a.ctypes.data_as(_vp), a.shape[1], a.shape[0], launches) != 0:
        raise MoxError(_err())


def read_accum(path, width, height):
    a = np.empty((height, width, 3), dtype=np.float32)
    n = _u64()
    if lib().moxh_read_accum(path.encode(), a.ctypes.data_as(_vp), width, height, C.byref(n)) != 0:
        raise MoxError(_err())
    return a, n.value
