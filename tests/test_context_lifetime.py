"""What a render context keeps between calls: its statistics record, and the device and pinned memory it frees
when it is closed."""
import numpy as np
import pytest

from conftest import random_rays
from minimaloptix_b200 import structs as S

pytestmark = pytest.mark.gpu

# stats fields that describe the scene and its acceleration structure, not the rendering since the last clear
SCENE_FIELDS = ("n_prims", "n_triangles", "n_spheres", "n_quads", "n_nodes", "node_bytes", "prim_bytes", "n_lights", "ms_build")
INTERIOR_BOX = ([0.05, 0.05, 0.05], [9.95, 3.95, 7.95])


def _render(ctx, host, api_tables, w, h, spp, seed, flags=S.ACCEL_COUNTERS):
    sc = host.Scene.builtin("interior", 20000)
    sc.upload(api_tables.gpu, ctx, w, h, 5)
    ctx.build_accel(flags)
    ctx.render(spp, seed)


def test_clear_accum_resets_counters_and_timings(host, api_tables, gpu_backend):
    g = gpu_backend.context(0)
    _render(g, host, api_tables, 160, 120, 3, 11)
    g.trace_closest(random_rays(2000, *INTERIOR_BOX, 5))
    before = g.stats()
    for k in ("rays_primary", "rays_bounce", "rays_shadow", "launches", "node_visits", "prim_tests", "node_visits_shadow",
              "kernel_launches", "extend_launches", "ms_render", "ms_extend", "ms_build", "n_nodes", "n_prims"):
        assert before[k] > 0, k
    g.clear_accum()
    after = g.stats()
    assert not g.read_accum().any()
    for k, v in after.items():
        if k in SCENE_FIELDS:
            assert v == before[k], k
        else:
            assert v == ([0] * len(v) if isinstance(v, list) else 0), k
    g.render(1, 11)   # the seed counter restarted with the statistics
    assert g.stats()["launches"] == 1


def test_multi_handle_stats_equal_plain_context(host, api_tables, gpu_backend):
    stats = []
    for ctx in (gpu_backend.context(0), gpu_backend.multi_context([0])):
        _render(ctx, host, api_tables, 200, 120, 3, 17)
        ctx.read_accum()
        stats.append(ctx.stats())
        ctx.close()
    plain, multi = stats
    assert plain["rays_primary"] > 0 and plain["node_visits"] > 0
    for k, v in plain.items():
        if not k.startswith("ms_"):
            assert multi[k] == v, k


def test_closed_contexts_return_their_memory(host, api_tables, gpu_backend):
    """About 1 GB of path state per context (1280x720 pixels, 4 samples each), plus the read-back images and the
    raw-query buffers: closing the context frees all of it."""
    import torch
    rays = random_rays(100000, *INTERIOR_BOX, 9)
    free = []
    for i in range(8):
        g = gpu_backend.context(0)
        _render(g, host, api_tables, 1280, 720, 4, 100 + i, flags=S.ACCEL_DEFAULT)
        g.read_accum_begin()
        assert g.read_accum_end().any()
        g.trace_closest(rays)
        g.trace_shadow(rays)
        g.close()
        free.append(torch.cuda.mem_get_info(0)[0])
    assert free[0] - free[-1] <= 64 << 20, [f >> 20 for f in free]
