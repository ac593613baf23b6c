#!/usr/bin/env python3
"""Refit against full build for animated scenes (mox_update_mesh / mox_update_sphere + MOX_ACCEL_REFIT).

Two workloads:
  interior  the ~1 M-triangle interior of bench.py at 3840x2160: every frame moves each blob and torus by a drift
            along its own direction plus a small sinusoidal displacement (no triangle degenerates)
  spheres   the 292-primitive random-spheres animation (Scene.animate(0.002) + apply_spheres) at 1920x1080

Per workload: the device time (CUDA events around the kernels, what mox_build_accel reports) and the wall time
(update calls and uploads included, the call returns synchronised) of a refit and of a full build, medians over
the frames; and the Mrays/s (primary + bounce) of an 8-spp step after K = 1, 10 and 60 frames of refits against a
context fully built at the same pose, which is what the refitted tree has lost in quality.  One JSON line per
workload, with the GPU's name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import minimaloptix_b200 as mox  # noqa: E402
from minimaloptix_b200 import host  # noqa: E402
from minimaloptix_b200 import structs as S  # noqa: E402

ROOM_MESHES = 11   # buildInterior adds the room, the table top and its legs first; blobs and tori follow
CHECKPOINTS = (1, 10, 60)
SPP, MAX_DEPTH, SEED = 8, 5, 0xD1A1A6


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, timeout=60)
    name, power = [x.strip() for x in out.stdout.strip().split(",")]
    return {"gpu": name, "power_limit": power}


def mrays(ctx, reps):
    """Median Mrays/s (primary + bounce) of `reps` 8-spp steps."""
    vals = []
    for r in range(reps):
        ctx.clear_accum()
        ctx.render(SPP, SEED + r)
        st = ctx.stats()
        vals.append((st["rays_primary"] + st["rays_bounce"]) / (st["ms_render"] * 1e3))
    return float(np.median(vals))


class Interior:
    name = "interior"

    def __init__(self, tris, width, height):
        self.sc = host.Scene.builtin("interior", tris)
        self.width, self.height = width, height
        first, self.movers = 0, []
        rng = np.random.default_rng(1)
        for m in range(self.sc.info().n_meshes):
            info = self.sc.mesh_info(m)
            if m >= ROOM_MESHES:
                a = rng.uniform(0, 2 * np.pi)
                self.movers.append((first, self.sc.mesh_arrays(m)[0], np.array([np.cos(a), 0, np.sin(a)], np.float32)))
            first += info["faces"]
        self.n_tris = self.sc.info().n_triangles

    def setup(self, ctx, api):
        self.sc.upload(api, ctx, self.width, self.height, MAX_DEPTH)

    def pose(self, frame):
        t = np.float32(0.05 * frame)
        return [(first, (v + d * (0.2 * t) + 0.004 * np.sin(7.0 * v[:, [1, 2, 0]] + t)).astype(np.float32))
                for first, v, d in self.movers]

    def apply(self, ctx, api, pose):
        for first, v in pose:
            ctx.update_mesh(first, v)


class Spheres:
    name = "spheres"

    def __init__(self, width, height):
        self.sc = host.Scene.builtin("random_spheres")
        self.width, self.height = width, height
        self.n_tris = 0
        self.frame = 0

    def setup(self, ctx, api):
        self.sc.upload(api, ctx, self.width, self.height, MAX_DEPTH)

    def pose(self, frame):
        while self.frame < frame:   # Scene.animate steps the scene's own sphere state
            self.sc.animate(0.002)
            self.frame += 1
        return None

    def apply(self, ctx, api, pose):
        self.sc.apply_spheres(api, ctx)


def run(work, reps):
    api = host.ApiTable(mox.GPU_LIB, "mox_")
    ctx, fresh = mox.gpu().context(0), mox.gpu().context(0)
    for c in (ctx, fresh):
        work.setup(c, api)
        c.build_accel()            # loads the build kernels, sizes the arena
        c.render(1, 1)             # loads the render kernels, allocates the wavefront state
    ctx.build_accel()
    ctx.build_accel(S.ACCEL_REFIT)   # loads the refit kernels
    refit_dev, refit_wall, build_dev, build_wall, quality = [], [], [], [], []
    for frame in range(1, max(CHECKPOINTS) + 1):
        pose = work.pose(frame)
        t0 = time.perf_counter()
        work.apply(ctx, api, pose)
        refit_dev.append(ctx.build_accel(S.ACCEL_REFIT))
        refit_wall.append((time.perf_counter() - t0) * 1e3)
        t0 = time.perf_counter()
        work.apply(fresh, api, pose)
        build_dev.append(fresh.build_accel())
        build_wall.append((time.perf_counter() - t0) * 1e3)
        if frame in CHECKPOINTS:
            r, b = mrays(ctx, reps), mrays(fresh, reps)
            quality.append({"frames_of_refits": frame, "mrays_refit": r, "mrays_full_build": b, "ratio": r / b})
    med = lambda x: float(np.median(x))
    return {"workload": work.name, "triangles": int(work.n_tris), "width": work.width, "height": work.height, "spp_per_step": SPP,
            "frames": max(CHECKPOINTS), "refit_ms_device": med(refit_dev), "refit_ms_wall": med(refit_wall),
            "build_ms_device": med(build_dev), "build_ms_wall": med(build_wall),
            "device_speedup": med(build_dev) / med(refit_dev), "quality": quality}


def main():
    p = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    p.add_argument("--tris", type=int, default=1_000_000)
    p.add_argument("--reps", type=int, default=3, help="8-spp steps per Mrays/s figure (median)")
    p.add_argument("--workload", choices=["interior", "spheres", "both"], default="both")
    p.add_argument("--out", help="also append the JSON lines to this file")
    args = p.parse_args()
    info = gpu_info()
    works = []
    if args.workload in ("interior", "both"):
        works.append(Interior(args.tris, 3840, 2160))
    if args.workload in ("spheres", "both"):
        works.append(Spheres(1920, 1080))
    for w in works:
        line = json.dumps(dict(run(w, args.reps), **info))
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
