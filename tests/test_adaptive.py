"""Adaptive sampling on the GPU (mox_render_adaptive, mox_read_sample_counts).

Every sample is keyed by its pixel and launch only, so a pixel that took n samples in an adaptive render must hold,
bit for bit, what a uniform render of the same seed schedule holds after n launches."""
import ctypes as C

import numpy as np
import pytest

import adaptive_model as M
from minimaloptix_b200 import structs as S

pytestmark = pytest.mark.gpu

ERR_INVALID, ERR_STATE = -1, -4
COUNTS = ("rays_primary", "rays_bounce", "rays_shadow", "rays_shadow_traced", "nonfinite_samples", "rays_depth",
          "shadow_traced_depth")


def cornell(host):
    return M.load_cornell(host), 64, 64


def interior(host):
    return host.Scene.builtin("interior", 30000), 160, 120


def spheres(host):
    return host.Scene.builtin("random_spheres"), 128, 72


SCENES = {"cornell": cornell, "interior": interior, "random_spheres": spheres}


def make(gpu_backend, api_tables, scene, w, h, mode=S.RNG_REF, device=0):
    g = gpu_backend.context(device)
    scene.upload(api_tables.gpu, g, w, h, 5)
    g.set_rng_mode(mode)
    g.build_accel()
    return g


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def uniform_snapshots(g, spp, step, seed):
    """Accumulation buffers of a uniform render after step, 2 step, ... launches."""
    out = []
    for _ in range(spp // step):
        g.render(step, seed)
        out.append(g.read_accum())
    return out


def mixed_adaptive(make_ctx, spp, seed, round_spp, min_spp):
    """An adaptive render in which some pixels stop early and some take every launch: (context, rel threshold)."""
    for rel in (0.3, 0.15, 0.08, 0.04, 0.02, 0.01):
        g = make_ctx()
        g.render_adaptive(spp, seed, rel, abs_error=1e-3, min_spp=min_spp, round_spp=round_spp)
        n = g.read_sample_counts()
        if (n < spp).any() and (n == spp).any():
            return g, rel
        g.close()
    pytest.fail("no threshold gives a mix of stopped and running pixels")


PREFIX_CASES = [("cornell", S.RNG_REF), ("cornell", S.RNG_PHILOX), ("interior", S.RNG_REF), ("random_spheres", S.RNG_REF)]


@pytest.mark.parametrize("name,mode", PREFIX_CASES, ids=[f"{n}-{'ref' if m == S.RNG_REF else 'philox'}" for n, m in PREFIX_CASES])
def test_prefix_property(host, api_tables, gpu_backend, name, mode):
    scene, w, h = SCENES[name](host)
    seed = 0xA11CE
    g, rel = mixed_adaptive(lambda: make(gpu_backend, api_tables, scene, w, h, mode), 32, seed, 4, 8)
    counts = g.read_sample_counts()
    acc = g.read_accum()
    snaps = uniform_snapshots(make(gpu_backend, api_tables, scene, w, h, mode), 32, 4, seed)
    assert (counts % 4 == 0).all() and counts.min() >= 8 and counts.max() == 32
    assert (counts < 32).any()
    for k, snap in enumerate(snaps):
        sel = counts == 4 * (k + 1)
        assert np.array_equal(bits(acc[sel]), bits(snap[sel])), (name, rel, 4 * (k + 1))
    assert g.stats()["launches"] == 32


def test_zero_thresholds_equal_a_uniform_render(host, api_tables, gpu_backend):
    scene, w, h = interior(host)
    a = make(gpu_backend, api_tables, scene, w, h)
    traced = a.render_adaptive(12, 99, 0.0, 0.0, min_spp=2, round_spp=5)
    b = make(gpu_backend, api_tables, scene, w, h)
    b.render(12, 99)
    assert traced == w * h * 12
    assert np.array_equal(bits(a.read_accum()), bits(b.read_accum()))
    assert (a.read_sample_counts() == 12).all()
    sa, sb = a.stats(), b.stats()
    for k in COUNTS:
        assert sa[k] == sb[k], k


@pytest.mark.parametrize("mode", [S.RNG_REF, S.RNG_PHILOX], ids=["ref", "philox"])
def test_stopping_rule_matches_numpy(host, api_tables, gpu_backend, mode):
    scene, w, h = cornell(host)
    seed, spp = 0x5EED, 24
    samples = M.sample_images(make(gpu_backend, api_tables, scene, w, h, mode), spp, seed)
    for rel, abs_ in ((0.2, 0.0), (0.05, 2e-3)):
        want, near = M.predict(samples, 4, 6, rel, abs_)
        g = make(gpu_backend, api_tables, scene, w, h, mode)
        traced = g.render_adaptive(spp, seed, rel, abs_, min_spp=6, round_spp=4)
        got = g.read_sample_counts()
        bad = (got != want) & ~near
        assert not bad.any(), (rel, np.argwhere(bad)[:10])
        assert traced == int(got.sum())


def test_deterministic_and_independent_of_batching(host, api_tables, gpu_backend, monkeypatch):
    scene, w, h = interior(host)
    runs = []
    for cap in (None, None, str(w * h // 3)):
        if cap:
            monkeypatch.setenv("MOX_MAX_BATCH_PATHS", cap)   # several batches per round
        g = make(gpu_backend, api_tables, scene, w, h)
        n = g.render_adaptive(24, 7, 0.05, 1e-3, min_spp=8, round_spp=8)
        runs.append((bits(g.read_accum()), g.read_sample_counts(), n, g.stats()["kernel_launches"]))
    assert runs[2][3] > runs[0][3]
    for r in runs[1:]:
        assert np.array_equal(r[0], runs[0][0]) and np.array_equal(r[1], runs[0][1]) and r[2] == runs[0][2]
    assert (runs[0][1] < 24).any()


def test_two_ranks_unite_to_one(host, api_tables, gpu_backend):
    scene, w, h = cornell(host)
    args = (32, 3, 0.05, 1e-3, 8, 4)
    one = make(gpu_backend, api_tables, scene, w, h)
    n1 = one.render_adaptive(*args)
    acc, counts, n = 0, 0, 0
    for rank in range(2):
        g = make(gpu_backend, api_tables, scene, w, h)
        g.set_partition(rank, 2, 16)
        n += g.render_adaptive(*args)
        acc = acc + g.read_accum()
        counts = counts + g.read_sample_counts()
    assert n == n1
    assert np.array_equal(bits(acc.astype(np.float32)), bits(one.read_accum()))
    assert np.array_equal(counts, one.read_sample_counts())


def test_one_device_multi_handle_equals_plain(host, api_tables, gpu_backend):
    scene, w, h = cornell(host)
    plain = make(gpu_backend, api_tables, scene, w, h)
    multi = make(gpu_backend, api_tables, scene, w, h, device=[0])
    args = (16, 5, 0.05, 1e-3, 4, 4)
    assert plain.render_adaptive(*args) == multi.render_adaptive(*args)
    assert np.array_equal(bits(plain.read_accum()), bits(multi.read_accum()))
    assert np.array_equal(plain.read_sample_counts(), multi.read_sample_counts())


def test_state(host, api_tables, gpu_backend):
    scene, w, h = cornell(host)
    g, rel = mixed_adaptive(lambda: make(gpu_backend, api_tables, scene, w, h), 16, 11, 4, 4)
    first, acc1 = g.read_sample_counts(), g.read_accum()
    stopped = first < 16
    # a second call with the same thresholds renders no pixel the first one stopped
    g.render_adaptive(8, 11, rel, 1e-3, min_spp=4, round_spp=4)
    second, acc2 = g.read_sample_counts(), g.read_accum()
    assert np.array_equal(second[stopped], first[stopped])
    assert np.array_equal(bits(acc2[stopped]), bits(acc1[stopped]))
    assert g.stats()["launches"] == 24
    # a uniform render adds its launches to every count
    g.render(3, 11)
    assert np.array_equal(g.read_sample_counts(), second + 3)
    g.clear_accum()
    assert not g.read_sample_counts().any()
    g.render_adaptive(8, 11, 0.05, 1e-3, min_spp=4, round_spp=4)
    g.set_accum(np.zeros((h, w, 3), np.float32), 5)
    assert (g.read_sample_counts() == 5).all()
    g.render_adaptive(8, 11, 0.05, 1e-3, min_spp=4, round_spp=4)
    g.set_globals(w // 2, h // 2, 5)
    assert not g.read_sample_counts().any()
    # after the resize the statistics start again: thresholds 0 give every pixel every launch
    g.render_adaptive(4, 11, 0.0, 0.0, min_spp=2, round_spp=2)
    assert (g.read_sample_counts() == 4).all()


def test_errors(host, api_tables, gpu_backend):
    scene, w, h = cornell(host)
    g = make(gpu_backend, api_tables, scene, w, h)
    n = C.c_uint64()

    def rc(p):
        return g.b.render_adaptive(g.h, 4, 1, None if p is None else C.byref(p), C.byref(n))
    assert rc(None) == ERR_INVALID
    assert rc(S.Adaptive(0, 4, 0.1, 0.0)) == ERR_INVALID
    for rel, abs_ in ((-0.1, 0.0), (0.1, -1e-3), (float("nan"), 0.0), (0.1, float("inf"))):
        assert rc(S.Adaptive(4, 4, rel, abs_)) == ERR_INVALID
    assert g.b.read_sample_counts(g.h, None) == ERR_INVALID
    assert rc(S.Adaptive(4, 4, 0.1, 0.0)) == 0
    fresh = gpu_backend.context(0)   # no globals, camera or acceleration structure
    assert fresh.b.render_adaptive(fresh.h, 4, 1, C.byref(S.Adaptive(4, 4, 0.1, 0.0)), None) == ERR_STATE
    unbuilt = gpu_backend.context(0)
    scene.upload(api_tables.gpu, unbuilt, w, h, 5)
    assert unbuilt.b.render_adaptive(unbuilt.h, 4, 1, C.byref(S.Adaptive(4, 4, 0.1, 0.0)), None) == ERR_STATE


def test_matches_the_oracle(host, api_tables, orc, gpu_backend):
    scene, w, h = cornell(host)
    o = orc.context()
    scene.upload(api_tables.oracle, o, w, h, 5)
    o.build_accel()
    g, rel = mixed_adaptive(lambda: make(gpu_backend, api_tables, scene, w, h), 16, 0xC0FFEE, 4, 4)
    o.render_adaptive(16, 0xC0FFEE, rel, 1e-3, min_spp=4, round_spp=4)
    cg, co = g.read_sample_counts(), o.read_sample_counts()
    agree = cg == co
    assert agree.mean() >= 0.995, agree.mean()
    # the cornell tolerance of test_gpu_parity.py::test_render_matches_oracle_ref_rng, on the pixels whose counts agree
    a = (g.read_accum()[agree] / cg[agree][:, None])[:, None, :]
    b = (o.read_accum()[agree] / co[agree][:, None])[:, None, :]
    rmse = float(np.sqrt(np.mean((np.clip(a, 0, 1) - np.clip(b, 0, 1)) ** 2)))
    qa, qb = host.accum_to_rgb8(a, 1).astype(np.int32), host.accum_to_rgb8(b, 1).astype(np.int32)
    within = float(np.mean(np.all(np.abs(qa - qb) <= 1, axis=2)))
    assert rmse <= 1e-5, rmse
    assert within >= 0.9999, within
