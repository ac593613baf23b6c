"""Adaptive sampling against a uniform render of the same number of pixel-samples (mox_render_adaptive).

For each scene:
  - the reference is a uniform render of --ref-spp samples (seed REF_SEED); its two halves give a per-pixel noise
    estimate, and the 10 % of pixels where the halves differ most are the "noisiest pixels";
  - the uniform render takes --spp samples per pixel (seed EVAL_SEED);
  - the adaptive render may take up to --max-spp; its relative threshold is found by bisection, on renders with
    CAL_SEED, so that it traces about as many pixel-samples as the uniform render (abs_error = ABS_FRACTION * rel);
  - both are compared with the reference: RMSE of the normalised image overall and on the noisiest pixels, device
    time (mox_stats.ms_render) and wall time of the call, Mrays/s, pixel-samples.  The adaptive render is also run
    one round per call, which leaves the same image and counts, to give each round's active fraction and Mrays/s.
One JSON line per scene and method, plus one line naming the card and its power limit, go to stdout and to --out.

  python scripts/adaptive_bench.py --out profiles/adaptive_b200.jsonl
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import minimaloptix_b200 as mox  # noqa: E402
from minimaloptix_b200 import host  # noqa: E402

REF_SEED, CAL_SEED, EVAL_SEED = 0x5EF, 0xCA1, 0xE7A1
ABS_FRACTION = 0.05
MAX_DEPTH = 5
SCENES = {"cornell": (512, 512), "interior": (1920, 1080)}


def card():
    """Name and power limit of GPU 0, read with nvidia-smi's query (no setting is changed)."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"card": name, "power_limit": power, "sm_clock_max": clock}
    except Exception as e:   # report, do not guess
        return {"card": "unknown", "power_limit": "unknown", "error": str(e)}


def load(name, tris):
    if name == "cornell":
        return host.Scene.load(os.path.join(ROOT, "scenes", "cornell"), "cornell")
    return host.Scene.builtin("interior", tris)


def context(api, scene, w, h):
    g = mox.gpu().context(0)
    scene.upload(api, g, w, h, MAX_DEPTH)
    g.build_accel()
    return g


def rays(st):
    return st["rays_primary"] + st["rays_bounce"]


def metrics(img, ref, noisy):
    err = (np.clip(img, 0, 1) - np.clip(ref, 0, 1)) ** 2
    return float(np.sqrt(err.mean())), float(np.sqrt(err[noisy].mean()))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--scenes", default="cornell,interior")
    ap.add_argument("--tris", type=int, default=1_000_000)
    ap.add_argument("--ref-spp", type=int, default=1024)
    ap.add_argument("--spp", type=int, default=64, help="samples per pixel of the uniform render")
    ap.add_argument("--max-spp", type=int, default=256, help="samples a pixel may take in the adaptive render")
    ap.add_argument("--min-spp", type=int, default=16)
    ap.add_argument("--round-spp", type=int, default=8)
    ap.add_argument("--bisect", type=int, default=10, help="bisection steps for the threshold")
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    api = host.ApiTable(mox.GPU_LIB, "mox_")
    lines = [dict(kind="card", **card())]
    print(json.dumps(lines[-1]), flush=True)
    for name in args.scenes.split(","):
        w, h = SCENES[name]
        scene = load(name, args.tris)
        g = context(api, scene, w, h)
        half = args.ref_spp // 2
        g.render(half, REF_SEED)
        a = g.read_accum()
        g.render(args.ref_spp - half, REF_SEED)
        full = g.read_accum()
        ref = full / args.ref_spp
        lum = lambda x: 0.2126 * x[..., 0] + 0.7152 * x[..., 1] + 0.0722 * x[..., 2]
        noise = np.abs(lum(a / half) - lum((full - a) / (args.ref_spp - half)))
        noisy = noise >= np.quantile(noise, 0.9)
        g.close()
        budget = args.spp * w * h
        base = dict(scene=name, width=w, height=h, ref_spp=args.ref_spp, max_depth=MAX_DEPTH,
                    triangles=args.tris if name == "interior" else None)

        # uniform render of --spp samples
        g = context(api, scene, w, h)
        t0 = time.perf_counter()
        g.render(args.spp, EVAL_SEED)
        wall = (time.perf_counter() - t0) * 1e3
        st = g.stats()
        rm, rn = metrics(g.read_accum() / args.spp, ref, noisy)
        lines.append(dict(base, kind="uniform", spp=args.spp, samples=budget, rmse=rm, rmse_noisiest10=rn, ms_render=st["ms_render"],
                          wall_ms=wall, mrays_per_s=rays(st) / (st["ms_render"] * 1e3)))
        print(json.dumps(lines[-1]), flush=True)
        g.close()

        # threshold by bisection (log scale) on the calibration seed: samples fall as rel grows
        lo, hi, best = 1e-4, 1.0, None
        for _ in range(args.bisect):
            rel = float(np.sqrt(lo * hi))
            g = context(api, scene, w, h)
            n = g.render_adaptive(args.max_spp, CAL_SEED, rel, ABS_FRACTION * rel, args.min_spp, args.round_spp)
            g.close()
            if best is None or abs(n - budget) < abs(best[1] - budget):
                best = (rel, n)
            if n > budget:
                lo = rel
            else:
                hi = rel
        rel = best[0]

        # adaptive render, one call
        g = context(api, scene, w, h)
        t0 = time.perf_counter()
        n = g.render_adaptive(args.max_spp, EVAL_SEED, rel, ABS_FRACTION * rel, args.min_spp, args.round_spp)
        wall = (time.perf_counter() - t0) * 1e3
        st = g.stats()
        counts = g.read_sample_counts()
        img = g.read_accum() / np.maximum(counts, 1)[..., None]
        acc_one = g.read_accum()
        g.close()
        rm, rn = metrics(img, ref, noisy)

        # the same render one round per call: each round's active fraction and ray rate
        g = context(api, scene, w, h)
        rounds, prev = [], g.stats()
        for done in range(0, args.max_spp, args.round_spp):
            r = min(args.round_spp, args.max_spp - done)   # the single call's last round may be shorter
            k = g.render_adaptive(r, EVAL_SEED, rel, ABS_FRACTION * rel, args.min_spp, args.round_spp)
            s = g.stats()
            dms = s["ms_render"] - prev["ms_render"]
            rounds.append(dict(active_fraction=k / (r * w * h), ms_render=dms,
                               mrays_per_s=(rays(s) - rays(prev)) / (dms * 1e3) if dms > 0 else None))
            prev = s
        same = bool(np.array_equal(g.read_sample_counts(), counts)) and bool(np.array_equal(g.read_accum().view(np.uint32), acc_one.view(np.uint32)))
        g.close()
        lines.append(dict(base, kind="adaptive", max_spp=args.max_spp, min_spp=args.min_spp, round_spp=args.round_spp, rel_error=rel,
                          abs_error=ABS_FRACTION * rel, calibration_samples=best[1], samples=n, samples_vs_uniform=n / budget,
                          rmse=rm, rmse_noisiest10=rn, ms_render=st["ms_render"], wall_ms=wall,
                          mrays_per_s=rays(st) / (st["ms_render"] * 1e3), spp_min=int(counts.min()), spp_max=int(counts.max()),
                          rounds=rounds, round_by_round_identical=same))
        print(json.dumps(lines[-1]), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            for l in lines:
                f.write(json.dumps(l) + "\n")


if __name__ == "__main__":
    main()
