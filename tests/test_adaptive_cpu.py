"""Adaptive sampling without a GPU: the oracle's orc_render_adaptive against the numpy restatement of the stopping rule,
the per-pixel display conversion, and the ctypes mirror of mox_adaptive."""
import ctypes as C

import numpy as np
import pytest

import adaptive_model as M
from minimaloptix_b200 import structs as S

W, H, SPP, SEED = 16, 12, 16, 0xADA


@pytest.fixture(scope="module")
def cornell_samples(host, api_tables, orc):
    sc = M.load_cornell(host)
    o = orc.context()
    sc.upload(api_tables.oracle, o, W, H, 5)
    o.build_accel()
    return sc, M.sample_images(o, SPP, SEED)


def mixed_threshold(samples, round_spp, min_spp):
    """A relative threshold under which some pixels stop early and some take every sample."""
    for rel in (0.5, 0.3, 0.2, 0.1, 0.05, 0.02):
        counts, _ = M.predict(samples, round_spp, min_spp, rel)
        if (counts < len(samples)).any() and (counts == len(samples)).any():
            return rel
    pytest.fail("no threshold gives a mix of stopped and running pixels")


def test_oracle_follows_the_stopping_rule(host, api_tables, orc, cornell_samples):
    sc, samples = cornell_samples
    rel = mixed_threshold(samples, 4, 4)
    want, near = M.predict(samples, 4, 4, rel)
    o = orc.context()
    sc.upload(api_tables.oracle, o, W, H, 5)
    o.build_accel()
    traced = o.render_adaptive(SPP, SEED, rel, min_spp=4, round_spp=4)
    counts = o.read_sample_counts()
    ok = (counts == want) | near
    assert ok.all(), np.argwhere(~ok)[:10]
    assert traced == int(counts.sum())
    assert o.stats()["launches"] == SPP
    # every pixel holds the sum of its first `count` samples, bit for bit
    sums = M.prefix_sums(samples)
    acc = o.read_accum()
    agree = counts == want
    picked = sums[counts.astype(np.int64) - 1, np.arange(H)[:, None], np.arange(W)[None, :]]
    assert np.array_equal(acc[agree].view(np.uint32), picked[agree].view(np.uint32))


def test_oracle_uniform_render_adds_to_every_count(host, api_tables, orc, cornell_samples):
    sc, samples = cornell_samples
    o = orc.context()
    sc.upload(api_tables.oracle, o, W, H, 5)
    o.build_accel()
    o.render_adaptive(8, SEED, 0.5, abs_error=0.01, min_spp=2, round_spp=2)
    before = o.read_sample_counts()
    o.render(3, SEED)
    assert np.array_equal(o.read_sample_counts(), before + 3)
    o.clear_accum()
    assert not o.read_sample_counts().any()


def test_rgb8_with_uniform_counts_equals_rgb8(host):
    rng = np.random.default_rng(7)
    for n in (1, 3, 32):
        accum = (rng.random((9, 13, 3)) * n * 1.2).astype(np.float32)
        counts = np.full((9, 13), n, np.uint32)
        assert np.array_equal(host.accum_to_rgb8_counts(accum, counts), host.accum_to_rgb8(accum, n))


def test_rgb8_with_zero_count_is_black(host):
    accum = np.full((4, 5, 3), 2.5, np.float32)
    counts = np.full((4, 5), 4, np.uint32)
    counts[1, 2] = counts[3, 0] = 0
    out = host.accum_to_rgb8_counts(accum, counts)
    # output row 0 is the top of the image, accumulator row 0 its bottom
    assert not out[4 - 1 - 1, 2].any() and not out[4 - 1 - 3, 0].any()
    assert (out.reshape(-1, 3).any(axis=1)).sum() == 18


def test_adaptive_struct_matches_header():
    assert C.sizeof(S.Adaptive) == 16
    assert [f[0] for f in S.Adaptive._fields_] == ["round_spp", "min_spp", "rel_error", "abs_error"]
