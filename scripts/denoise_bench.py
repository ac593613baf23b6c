"""First-hit AOVs and mox_denoise on the GPU: what the AOVs cost a render, what the filter costs, what it gains.

For each scene (the interior at 3840 x 2160, Cornell at 512 x 512, depth 5):
  - the ms of an 8-spp mox_render step with AOVs off and on, two contexts stepped alternately (--steps each after
    --warmup), from mox_stats.ms_render; the difference is k_aov;
  - the ms of mox_denoise with the default parameters (its CUDA-event time), the median of --calls calls after warm-up;
  - the RMSE against a render of --ref-spp samples, of the noisy mean and of the denoised image, at 16 and 64 spp.
One JSON line per scene, plus one line naming the card and its power limit first, go to stdout and to --out.

  python scripts/denoise_bench.py --out profiles/denoise_b200.jsonl
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import minimaloptix_b200 as mox  # noqa: E402
from minimaloptix_b200 import host  # noqa: E402

MAX_DEPTH = 5
SCENES = {"interior": (3840, 2160), "cornell": (512, 512)}
REF_SEED, EVAL_SEED, STEP_SEED = 0x5EF, 0xE7A1, 0x57E9


def card():
    """Name and power limit of GPU 0, read with nvidia-smi's query (no setting is changed)."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"card": name, "power_limit": power, "sm_clock_max": clock}
    except Exception as e:   # report, do not guess
        return {"card": "unknown", "power_limit": "unknown", "error": str(e)}


def load(name):
    if name == "cornell":
        return host.Scene.load(os.path.join(ROOT, "scenes", "cornell"), "cornell")
    return host.Scene.builtin("interior", 1000000, 0xD1A1A6)   # the interior of mox_cli and bench.py


def context(api, scene, w, h, aovs):
    g = mox.gpu().context(0)
    scene.upload(api, g, w, h, MAX_DEPTH)
    g.build_accel()
    if aovs:
        g.set_aovs(True)
    return g


def rmse(a, b):
    return float(np.sqrt(np.mean((np.clip(a, 0, 1) - np.clip(b, 0, 1)) ** 2)))


def step_ms(g, seed):
    before = g.stats()["ms_render"]
    g.render(8, seed)
    return g.stats()["ms_render"] - before


def run(name, args, api):
    w, h = SCENES[name]
    scene = load(name)
    row = {"scene": name, "width": w, "height": h, "max_depth": MAX_DEPTH}
    off, on = context(api, scene, w, h, False), context(api, scene, w, h, True)
    t_off, t_on = [], []
    for k in range(args.warmup + args.steps):
        a, b = step_ms(off, STEP_SEED), step_ms(on, STEP_SEED)
        if k >= args.warmup:
            t_off.append(a)
            t_on.append(b)
    row["step_8spp_ms_aov_off"] = t_off
    row["step_8spp_ms_aov_on"] = t_on
    row["aov_overhead_pct_median"] = 100.0 * (np.median(t_on) / np.median(t_off) - 1.0)
    assert np.array_equal(off.read_accum(), on.read_accum()), "AOVs changed the image"
    for _ in range(3):
        on.denoise()
    ms = [on.denoise()[1] for _ in range(args.calls)]
    row["denoise_ms_median"] = float(np.median(ms))
    row["denoise_ms_min_max"] = [float(min(ms)), float(max(ms))]
    off.close()
    on.close()
    ref = context(api, scene, w, h, False)
    ref.render(args.ref_spp, REF_SEED)
    truth = ref.read_accum() / args.ref_spp
    ref.close()
    for spp in (16, 64):
        g = context(api, scene, w, h, True)
        g.render(spp, EVAL_SEED)
        den, _ = g.denoise()
        noisy = g.read_accum() / spp
        row[f"rmse_{spp}spp_noisy"] = rmse(noisy, truth)
        row[f"rmse_{spp}spp_denoised"] = rmse(den, truth)
        g.close()
    row["ref_spp"] = args.ref_spp
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--ref-spp", type=int, default=1024)
    args = ap.parse_args()
    api = host.ApiTable(mox.GPU_LIB, "mox_")
    lines = [dict(card(), defaults=mox.structs.DENOISE_DEFAULTS)]
    print(json.dumps(lines[0]), flush=True)
    for name in SCENES:
        lines.append(run(name, args, api))
        print(json.dumps(lines[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
