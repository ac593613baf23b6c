"""ctypes mirrors of include/mox_structs.h (reference: MinimalOptiX/Structures.h:5-80)."""
import ctypes as C


class float3(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("z", C.c_float)]

    def __init__(self, x=0.0, y=0.0, z=0.0):
        super().__init__(x, y, z)

    def tuple(self):
        return (self.x, self.y, self.z)


class float4(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("z", C.c_float), ("w", C.c_float)]
    _pack_ = 16


class Payload(C.Structure):
    _fields_ = [("color", float3), ("depth", C.c_int), ("randSeed", C.c_int), ("attenuation", float3)]


class CamParams(C.Structure):
    _fields_ = [("origin", float3), ("horizontal", float3), ("vertical", float3), ("scrLowerLeftCorner", float3),
                ("u", float3), ("v", float3), ("lensRadius", C.c_float)]


class SphereParams(C.Structure):
    _fields_ = [("radius", C.c_float), ("center", float3), ("velocity", float3)]


class QuadParams(C.Structure):
    # 16-byte aligned, 64 bytes: plane@0 v1@16 v2@28 anchor@40 + 12 bytes tail padding
    _fields_ = [("plane", float4), ("v1", float3), ("v2", float3), ("anchor", float3), ("_pad", C.c_float * 3)]


class LambertianParams(C.Structure):
    _fields_ = [("albedo", float3)]


class MetalParams(C.Structure):
    _fields_ = [("albedo", float3), ("fuzz", C.c_float)]


class GlassParams(C.Structure):
    _fields_ = [("albedo", float3), ("refIdx", C.c_float)]


NORMAL, GLASS = 0, 1
SPHERE, QUAD = 0, 1


class DisneyParams(C.Structure):
    _fields_ = [("albedoID", C.c_int), ("color", float3), ("emission", float3), ("metallic", C.c_float),
                ("subsurface", C.c_float), ("specular", C.c_float), ("roughness", C.c_float),
                ("specularTint", C.c_float), ("anisotropic", C.c_float), ("sheen", C.c_float),
                ("sheenTint", C.c_float), ("clearcoat", C.c_float), ("clearcoatGloss", C.c_float),
                ("brdfType", C.c_int)]


class LightParams(C.Structure):
    _fields_ = [("position", float3), ("normal", float3), ("emission", float3), ("u", float3), ("v", float3),
                ("area", C.c_float), ("radius", C.c_float), ("shape", C.c_int)]


class Stats(C.Structure):
    _fields_ = [("rays_primary", C.c_uint64), ("rays_bounce", C.c_uint64), ("rays_shadow", C.c_uint64),
                ("nonfinite_samples", C.c_uint64), ("launches", C.c_uint64), ("node_visits", C.c_uint64),
                ("prim_tests", C.c_uint64), ("ms_render", C.c_double), ("ms_build", C.c_double),
                ("n_prims", C.c_uint32), ("n_triangles", C.c_uint32), ("n_spheres", C.c_uint32),
                ("n_quads", C.c_uint32), ("n_nodes", C.c_uint32), ("node_bytes", C.c_uint32),
                ("prim_bytes", C.c_uint32), ("n_lights", C.c_uint32),
                ("ms_generate", C.c_double), ("ms_extend", C.c_double), ("ms_shade", C.c_double),
                ("ms_shadow", C.c_double), ("ms_accumulate", C.c_double), ("extend_launches", C.c_uint64),
                ("kernel_launches", C.c_uint64), ("node_visits_shadow", C.c_uint64), ("prim_tests_shadow", C.c_uint64), ("rays_shadow_traced", C.c_uint64),
                ("rays_shadow_blocked", C.c_uint64), ("rays_shadow_tinted", C.c_uint64),
                ("rays_depth", C.c_uint64 * 8), ("shadow_traced_depth", C.c_uint64 * 8),
                ("ms_extend_depth", C.c_double * 8), ("ms_shadow_depth", C.c_double * 8)]

    def asdict(self):
        return {k: (list(getattr(self, k)) if hasattr(getattr(self, k), "__len__") else getattr(self, k)) for k, _ in self._fields_}


class Adaptive(C.Structure):
    """mox_adaptive: the rounds and thresholds of mox_render_adaptive."""
    _fields_ = [("round_spp", C.c_uint32), ("min_spp", C.c_uint32), ("rel_error", C.c_float), ("abs_error", C.c_float)]


class DenoiseParams(C.Structure):
    """mox_denoise_params: the iterations and edge stops of mox_denoise."""
    _fields_ = [("iterations", C.c_uint32), ("sigma_color", C.c_float), ("sigma_normal", C.c_float), ("sigma_depth", C.c_float)]


# mox.h MOX_DENOISE_DEFAULT_*
DENOISE_DEFAULTS = {"iterations": 5, "sigma_color": 1.0, "sigma_normal": 0.5, "sigma_depth": 0.05}

MAT_LAMBERTIAN, MAT_METAL, MAT_GLASS, MAT_DISNEY, MAT_LIGHT = range(5)
RNG_REF, RNG_PHILOX = 0, 1
ACCEL_DEFAULT, ACCEL_LBVH, ACCEL_COUNTERS, ACCEL_BINARY, ACCEL_WATERTIGHT = 0, 1, 2, 4, 8
ACCEL_REFIT = 16   # refit the last full build in place (mox.h MOX_ACCEL_REFIT)

SIZES = {Payload: 32, CamParams: 76, SphereParams: 28, QuadParams: 64, LambertianParams: 12, MetalParams: 16,
         GlassParams: 16, DisneyParams: 72, LightParams: 72, Adaptive: 16}
for _t, _s in SIZES.items():
    assert C.sizeof(_t) == _s, (_t.__name__, C.sizeof(_t), _s)
