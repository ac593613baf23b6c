"""The stopping rule of mox_render_adaptive (include/mox.h) restated in numpy, for the adaptive-sampling tests.

Given the exact colour of every sample of every pixel, it predicts how many samples each pixel takes in one call that
starts from a fresh state (after a clear): luminance y = 0.2126 r + 0.7152 g + 0.0722 b in float32, S1 and S2 summed
in float64 in launch order, the rule checked after every round but the last."""
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def luminance(rgb):
    rgb = np.asarray(rgb, dtype=np.float32)
    return (np.float32(0.2126) * rgb[..., 0] + np.float32(0.7152) * rgb[..., 1]) + np.float32(0.0722) * rgb[..., 2]


def sample_images(ctx, spp, seed):
    """Sample k (k < spp) of mox_render's schedule for every pixel, exactly: the context's buffer is cleared, set to
    zeros at launch k, and rendered once.  Leaves the context cleared."""
    zeros = np.zeros((ctx.height, ctx.width, 3), np.float32)
    out = []
    for k in range(spp):
        ctx.clear_accum()
        ctx.set_accum(zeros, k)
        ctx.render(1, seed)
        out.append(ctx.read_accum())
    ctx.clear_accum()
    return np.stack(out)


def predict(samples, round_spp, min_spp, rel, abs_=0.0):
    """(counts, near): the predicted sample count of every pixel, and a mask of the pixels whose error came within a
    relative 1e-6 of their threshold at a check, where float64 rounding may decide differently."""
    spp = len(samples)
    y = luminance(samples).astype(np.float64)
    s1 = np.zeros(y.shape[1:])
    s2 = np.zeros(y.shape[1:])
    n = np.zeros(y.shape[1:], np.int64)
    active = np.ones(y.shape[1:], bool)
    near = np.zeros(y.shape[1:], bool)
    rel, abs_ = float(np.float32(rel)), float(np.float32(abs_))
    min_spp = max(min_spp, 2)
    done = 0
    while done < spp and active.any():
        r = min(round_spp, spp - done)
        for k in range(done, done + r):
            s1 = np.where(active, s1 + y[k], s1)
            s2 = np.where(active, s2 + y[k] * y[k], s2)
            n = n + active
        done += r
        if done == spp:
            break
        with np.errstate(divide="ignore", invalid="ignore"):
            dn = n.astype(np.float64)
            m = s1 / dn
            var = np.maximum(0.0, (s2 - s1 * m) / (dn - 1.0))
            err = np.sqrt(var / dn)
            thr = np.maximum(rel * m, abs_)
        check = active & (n >= min_spp)
        near |= check & (np.abs(err - thr) <= 1e-6 * np.abs(thr))
        active &= ~(check & (err < thr))
    return n.astype(np.uint32), near


def prefix_sums(samples):
    """Accumulation buffers after 1, 2, ... samples, added in launch order in float32 as the renderer adds them."""
    out = np.empty_like(samples)
    acc = np.zeros(samples.shape[1:], np.float32)
    for k in range(len(samples)):
        acc = acc + samples[k]
        out[k] = acc
    return out


def load_cornell(host):
    return host.Scene.load(os.path.join(ROOT, "scenes", "cornell"), "cornell")
