#!/usr/bin/env python3
"""bench.py — headline benchmark of the render hot path (BASELINE.json: Mrays/s primary+bounce).

  python bench.py --gpus N --steps K --warmup W            # our CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # the CPU oracle (the reference has no
                                                           # CPU path and cannot run here)

Workload (config.workload): BASELINE configs[3] — the synthetic ~1 M-triangle interior with Disney
materials and 4 quad lights at 3840x2160, max depth 5, rng=ref, fixed seed schedule — the
configuration the 1 Grays/s target is quoted on.  It fits one GPU, so N=1 runs exactly this; for
N>1 the image is tile-split across ranks with the scene replicated (STRONG scaling: total work is
fixed) and the accumulation buffer is gathered once at the end over NCCL.
A step = SPP_PER_STEP (8) iterations of the reference's spp loop (MinimalOptiX.cpp:544-546), i.e.
mox_render(ctx, 8, seed): +8 samples for every pixel, rendered in wavefronts of at most 32 Mi paths.

  value   Mrays/s over the K timed steps, scene + BVH resident in HBM, device time = CUDA events on
          the launching stream (mox_stats.ms_render) + the gather, max over ranks.
  e2e     same metric through the C ABI with host buffers: per step set_camera (host struct),
          launch(seed), gather to rank 0, read_accum into a host array (device->host of the whole
          accumulation buffer inside the timed region).

  --dump-outputs DIR  after the timed steps, rank 0 writes what they computed, so that two builds can
          be compared output for output (the inputs are the same from run to run):
            accum.npy        float32 (N, 3): the gathered accumulation buffer (warm-up + timed steps, 8 spp
                             each) at N pixels: all of them when width*height <= 2^21, else a seeded
                             sample of 2^21 pixels
            accum_pixel.npy  float64 (N,): the row-major pixel index (y * width + x) of each row
            ray_counts.npy   float64 [primary + bounce rays, shadow rays] of the K timed steps, all ranks
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WIDTH, HEIGHT, MAX_DEPTH, SEED = 3840, 2160, 5, 0xD1A1A6
# One step = mox_render(8 spp): eight iterations of the spp loop of renderScene.  The library renders them in
# wavefronts of at most 32 Mi paths: two of 4 spp on one GPU, one of 8 spp per GPU on eight (each GPU then owns an
# eighth of the pixels) — the persistent traversal launches keep their length when the frame is split.
SPP_PER_STEP = 8
TRIS = 1_000_000
WORKLOAD = f"interior ~1M-triangle Disney scene (BASELINE configs[3]), 3840x2160, {SPP_PER_STEP} spp per step, max depth 5, rng=ref"
DUMP_PIXELS = 1 << 21   # 2^21 pixels: 24 MiB of float32 RGB + 16 MiB of float64 indices, under 64 MB in all


def positive(text):
    v = int(text)
    if v < 1:
        raise argparse.ArgumentTypeError("must be at least 1")
    return v


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the accumulation buffer (warm-up + timed steps; a seeded sample of "
                         "2^21 pixels when larger) and the ray counts of the timed steps to DIR/*.npy (see the module docstring)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--width", type=int, default=WIDTH)
    ap.add_argument("--height", type=int, default=HEIGHT)
    ap.add_argument("--tris", type=int, default=TRIS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--emulate-world", type=int, default=0,
                    help="experiment: render only rank 0's tile set of an N-rank partition on this one GPU (what each GPU of an N-GPU run does)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


def dump_arrays(img, rays, shadow):
    """The arrays of --dump-outputs from the gathered (H, W, 3) accumulation buffer and the timed steps' ray counts."""
    import numpy as np
    flat = img.reshape(-1, 3)
    n = len(flat)
    pix = np.arange(n) if n <= DUMP_PIXELS else np.sort(np.random.default_rng(SEED).choice(n, DUMP_PIXELS, replace=False))
    return {"accum": flat[pix].astype(np.float32), "accum_pixel": pix.astype(np.float64),
            "ray_counts": np.array([rays, shadow], dtype=np.float64)}


def write_dump(directory, arrays):
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


class ClockSampler:
    """SM clock and throttle reasons during the timed region (B200_PROFILING.md recipe: clocks.sm, clocks.max.sm and
    the clocks_event_reasons of `nvidia-smi --query-gpu ... -lms 200`).  Read through NVML in a thread of this process
    — the same counters nvidia-smi prints — because an nvidia-smi child polling at 200 ms stalled this process's CUDA
    calls by 40-60 ms per poll (measured: steps of 151-173 ms wall next to 107.6 ms ones, device time unchanged);
    nvidia-smi is the fallback when the NVML binding is missing."""

    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.proc = None
        self.marks = []
        self.how = None
        self.poll_ms = []
        self._stop = threading.Event()

    def mark(self):
        self.marks.append(len(self.samples))

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES renumbers CUDA ordinals; NVML does not
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else self.index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.how = "NVML (nvmlDeviceGetClockInfo / nvmlDeviceGetCurrentClocksEventReasons) every 200 ms"
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        q = ("index,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.how = "nvidia-smi -lms 200"
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _poll_nvml(self):
        n = self.nvml
        while not self._stop.is_set():
            t0 = time.perf_counter()
            try:
                self.samples.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
                try:
                    bits = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except AttributeError:
                    bits = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                for name, bit in self.REASONS.items():
                    if bits & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self.poll_ms.append((time.perf_counter() - t0) * 1e3)
            self._stop.wait(0.2)

    def _read(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                self.samples.append(float(f[1]))
                self.max_mhz = float(f[2])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    self.reasons.add(n)

    def stop(self):
        self._stop.set()
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        timed = self.samples[self.marks[0]:self.marks[1]] if len(self.marks) >= 2 else []
        timed = timed or self.samples   # a timed region shorter than one sampling period: all samples under load
        return {"sm_mhz": statistics.median(timed) if timed else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples), "samples_in_timed_region": len(timed),
                "how": self.how, "poll_ms_max": round(max(self.poll_ms), 2) if self.poll_ms else None,
                "note": "sampled from before the warm-up to the end of the e2e run; sm_mhz = median inside the timed region"}


def cpu_sample(args, steps, threads=0):
    """The oracle on the host cores on a bounded sample of the same workload: same scene, camera,
    depth and seed schedule at 1/16 of the pixels (W/4 x H/4), `steps` spp."""
    import oracle
    from minimaloptix_b200 import host
    w, h = max(args.width // 4, 16), max(args.height // 4, 16)
    sc = host.Scene.builtin("interior", args.tris)
    ctx = oracle.context(threads=threads)
    sc.upload(host.ApiTable(oracle.ORACLE_LIB, "orc_"), ctx, w, h, MAX_DEPTH)
    ctx.build_accel()
    per_step = []
    rays_total = 0
    for k in range(steps):
        before = ctx.stats()
        t0 = time.perf_counter()
        ctx.render(1, SEED)
        dt = time.perf_counter() - t0
        after = ctx.stats()
        rays = (after["rays_primary"] + after["rays_bounce"]) - (before["rays_primary"] + before["rays_bounce"])
        per_step.append((rays, dt))
        rays_total += rays
    cores = threads if threads > 0 else (os.cpu_count() or 1)
    return per_step, {"cores": cores, "kind": "port", "triangles": int(sc.info().n_triangles),
                      "sample": f"{w}x{h} (1/16 of the pixels), {steps} spp, same scene/camera/depth/seed schedule, oracle BVH (binned SAH)"}


def run_reference(args):
    """--impl reference: the reference's algorithm on the CPU (oracle port; the reference itself is
    OptiX-only and cannot be built here).  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    per_step, info = cpu_sample(args, args.warmup + args.steps)
    timed = per_step[args.warmup:]
    rays = sum(r for r, _ in timed)
    sec = sum(t for _, t in timed)
    value = rays / sec / 1e6
    line = {"impl": "reference", "metric": "Mrays/s (primary+bounce)", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sec / max(len(timed), 1), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "triangles": info["triangles"], "sample": info["sample"]},
            "cpu_baseline": dict(info, value=value, unit="Mrays/s"),
            "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import minimaloptix_b200 as mox
    from minimaloptix_b200 import host
    from minimaloptix_b200.parallel import TileGather

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (no CPU fallback); use --impl reference for the CPU arm")
    dev = torch.device("cuda", local)

    W, H = args.width, args.height
    sc = host.Scene.builtin("interior", args.tris)
    info = sc.info()
    api = host.ApiTable(mox.GPU_LIB, "mox_")
    ctx = mox.gpu().context(local)
    sc.upload(api, ctx, W, H, MAX_DEPTH)
    TILE = int(os.environ.get("MOX_BENCH_TILE", "32"))  # edge of the interleaved tiles (pixels)
    ctx.set_partition(rank, world, TILE)
    if args.emulate_world > 1 and world == 1:
        ctx.set_partition(0, args.emulate_world, TILE)
    ctx.build_accel()              # warm-up build: loads the build kernels (lazy module loading), sizes the arena
    build_ms = ctx.build_accel()   # the build that is reported (CUDA events around the build kernels)
    cam = sc.cam_params(W, H)

    tiles = TileGather(ctx, rank, world, dev)
    gather = tiles.gather  # final exchange: every rank's owned pixels to rank 0 (NCCL gather)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    step_no = [0]

    def step():
        ctx.render(SPP_PER_STEP, SEED)  # continues the fixed seed schedule seed_k = tea<16>(k, SEED)
        step_no[0] += 1

    def rays_of(st):
        return st["rays_primary"] + st["rays_bounce"]

    # ---- resident run: W warm-up steps, K timed steps + the gather
    # the clock sampler starts before the warm-up: launching nvidia-smi takes driver locks for ~0.1 s, which must
    # not fall into a timed region (it did: wall 123.7 ms/step against 111.3 on the device)
    sampler = ClockSampler(local)
    if rank == 0 and os.environ.get("MOX_BENCH_NO_SAMPLER") != "1":   # (the switch exists to measure the sampler's own cost)
        sampler.start()
    for _ in range(args.warmup):
        step()
    gather()  # warm-up of the exchange too (communicator / peer-mapping set-up happens on the first call)
    if rank == 0:
        for _ in range(2):   # ... and of the read-back path: both pinned host images and gather buffers get allocated here
            tiles.read()
    barrier()
    s0 = ctx.stats()
    if rank == 0:
        sampler.mark()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.perf_counter()
    step_wall = []
    for _ in range(args.steps):
        t_ = time.perf_counter()
        step()
        step_wall.append(round((time.perf_counter() - t_) * 1e3, 2))
    g0.record()
    gather()
    g1.record()
    barrier()
    wall = time.perf_counter() - wall0
    if rank == 0:
        sampler.mark()
    s1 = ctx.stats()
    dev_ms = (s1["ms_render"] - s0["ms_render"]) + g0.elapsed_time(g1)
    rays = rays_of(s1) - rays_of(s0)
    shadow = s1["rays_shadow"] - s0["rays_shadow"]
    t = torch.tensor([dev_ms, wall * 1e3], dtype=torch.float64, device=dev)
    cnt = torch.tensor([rays, shadow, s1["kernel_launches"] - s0["kernel_launches"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    render_per_rank = [s1["ms_render"] - s0["ms_render"]]
    if world > 1:
        rr = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(rr, torch.tensor([render_per_rank[0]], dtype=torch.float64, device=dev))
        render_per_rank = [round(x.item(), 2) for x in rr]
    dev_ms, wall_ms = t.tolist()
    rays_all, shadow_all, launches_all = cnt.tolist()
    value = rays_all / (dev_ms * 1e3)

    dump = None
    if args.dump_outputs and rank == 0:   # read now: the e2e run below clears the accumulation buffer
        dump = dump_arrays(tiles.read(), rays_all, shadow_all)

    # dominant kernel: closest-hit traversal (k_extend), timed live with CUDA events on its stream
    ext_ms = s1["ms_extend"] - s0["ms_extend"]
    ext_launches = s1["extend_launches"] - s0["extend_launches"]
    stage_ms = {k: s1[k] - s0[k] for k in ("ms_generate", "ms_extend", "ms_shade", "ms_shadow", "ms_accumulate")}

    # ---- e2e run: through the C ABI with HOST buffers.  Every step: camera struct from host memory, render, gather
    # to rank 0, device->host copy of the whole frame into pinned memory.  The read-back is the asynchronous form of
    # accuBuffer->map() (mox_read_accum_begin/_end, two buffers): the copy of frame k runs on a copy stream while
    # frame k+1 renders, and frame k is touched on the host one step later — every copy is inside the timed region.
    ctx.clear_accum()
    step_no[0] = 0
    barrier()
    e0 = ctx.stats()
    t0 = time.perf_counter()
    d2h = 0
    checksum = 0.0
    pending = False
    e2e_step_wall = []
    for _ in range(args.steps):
        t_ = time.perf_counter()
        ctx.set_camera(cam)
        step()
        gather()
        if rank == 0:
            if pending:
                img = tiles.read_end()
                d2h = img.nbytes
                checksum += float(img[::64, ::64].sum())  # touch the mapped result
            tiles.read_begin()
            pending = True
        e2e_step_wall.append(round((time.perf_counter() - t_) * 1e3, 2))
    if rank == 0 and pending:
        img = tiles.read_end()
        d2h = img.nbytes
        checksum += float(img[::64, ::64].sum())
    barrier()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    e1 = ctx.stats()
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    ce = torch.tensor([rays_of(e1) - rays_of(e0)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
        dist.all_reduce(ce, op=dist.ReduceOp.SUM)
    e2e_value = ce.item() / te.item() / 1e6

    # ---- serial pass (rank 0, untimed for `value`): the same steps on a context whose launches do not overlap
    # (MOX_OVERLAP_SHADOW=0, one slice), so a CUDA-event span on the launching stream is one kernel alone on the
    # GPU.  The timed region above runs the shadow launch of bounce b next to the extend launch of bounce b+1;
    # there the spans of the two overlap and do not add up to the step.
    roofline = roofline_shadow = roofline_build = per_depth = None
    serial = None
    if rank == 0:
        saved = {k: os.environ.get(k) for k in ("MOX_OVERLAP_SHADOW", "MOX_SLICES")}
        os.environ["MOX_OVERLAP_SHADOW"], os.environ["MOX_SLICES"] = "0", "1"
        sctx = mox.gpu().context(local)
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        sc.upload(api, sctx, W, H, MAX_DEPTH)
        sctx.set_partition(rank, world, TILE)
        if args.emulate_world > 1 and world == 1:
            sctx.set_partition(0, args.emulate_world, TILE)
        sctx.build_accel()
        sctx.render(SPP_PER_STEP, SEED)
        q0 = sctx.stats()
        n_serial = max(1, min(args.steps, 4))
        for _ in range(n_serial):
            sctx.render(SPP_PER_STEP, SEED)
        q1 = sctx.stats()
        dd = lambda k: [b - a for a, b in zip(q0[k], q1[k])]
        serial = {"steps": n_serial, "ms_per_step": (q1["ms_render"] - q0["ms_render"]) / n_serial,
                  "stage_ms_per_step": {k: (q1[k] - q0[k]) / n_serial for k in ("ms_generate", "ms_extend", "ms_shade", "ms_shadow", "ms_accumulate")}}
        rays_d, sh_d, ms_e, ms_s = dd("rays_depth"), dd("shadow_traced_depth"), dd("ms_extend_depth"), dd("ms_shadow_depth")
        per_depth = [{"depth": d, "rays": int(rays_d[d]), "ms_extend": ms_e[d], "extend_mrays_per_s": rays_d[d] / (ms_e[d] * 1e3) if ms_e[d] > 0 else None,
                      "shadow_rays_traversed": int(sh_d[d]), "ms_shadow": ms_s[d], "shadow_mrays_per_s": sh_d[d] / (ms_s[d] * 1e3) if ms_s[d] > 0 else None}
                     for d in range(1, 8) if rays_d[d]]
        b_rays, b_ms = sum(rays_d[2:]), sum(ms_e[2:])
        serial["bounce_only_extend_mrays_per_s"] = b_rays / (b_ms * 1e3) if b_ms > 0 else None   # traversal kernel alone, depth >= 2
        serial["primary_extend_mrays_per_s"] = rays_d[1] / (ms_e[1] * 1e3) if ms_e[1] > 0 else None

        # ---- counting pass for the algorithmic bytes of the traversal kernels (untimed)
        cctx = mox.gpu().context(local)
        sc.upload(api, cctx, W, H, MAX_DEPTH)
        cctx.set_partition(rank, world, TILE)
        cctx.build_accel(mox.structs.ACCEL_COUNTERS)
        cctx.render(1, SEED)
        cs = cctx.stats()
        peaks, traffic = {}, {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json, HBM copy)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"

        def roof(kernel, key, rays_counted, nodes, prims, fixed_bytes, fixed_note, rays_timed, ms, launches, ms_overlapped):
            n_node, n_prim = nodes / max(rays_counted, 1), prims / max(rays_counted, 1)
            b_ray = fixed_bytes + n_node * cs["node_bytes"] + n_prim * cs["prim_bytes"]
            achieved = rays_timed * b_ray / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
            t = traffic.get(key, {})
            return {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": t.get("dram_bytes_per_launch"),
                    "l2_bytes_per_launch": t.get("lts_bytes_per_launch"), "l2_gbs_under_ncu": t.get("lts_gbs_under_ncu"),
                    "traffic_note": traffic.get("_source") if t else None,
                    "bytes_per_ray": b_ray, "fixed_bytes_per_ray": fixed_bytes, "fixed_bytes_note": fixed_note,
                    "nodes_per_ray": n_node, "prims_per_ray": n_prim, "node_bytes": cs["node_bytes"],
                    "prim_bytes": cs["prim_bytes"], "rays_per_s": rays_timed / (ms * 1e-3) if ms > 0 else 0.0,
                    "launches": launches, "avg_launch_ms": ms / max(launches, 1), "rays_per_launch": rays_timed / max(launches, 1),
                    "timing": "CUDA events on the launching stream, %d steps of the serial pass (kernel alone on the GPU)" % n_serial,
                    "avg_launch_ms_in_timed_region": ms_overlapped,
                    "share_of_step": ms / max(q1["ms_render"] - q0["ms_render"], 1e-9),
                    "note": "BVH + triangles are L2-resident (126 MB L2): the algorithmic bytes are served by L1/L2, DRAM traffic is far "
                            "smaller; ncu shows the kernel latency/issue-bound (profiles/README.md)"}

        launches_s = q1["extend_launches"] - q0["extend_launches"]
        # extend ray: 32 B ray + 16 B hit (SURVEY 8d).  Shadow ray: 32 B ray + 4 B queue entry, + 16 B for a blocked ray
        # (one store of its contribution) and 32 B for a tinted one (load + store), by their counted shares.
        traced = max(cs["rays_shadow_traced"], 1)
        f_blk, f_tnt = cs["rays_shadow_blocked"] / traced, cs["rays_shadow_tinted"] / traced
        roofline = roof("k_traverse_wide<closest> (extend rays)", "k_traverse_closest", rays_of(cs), cs["node_visits"], cs["prim_tests"], 48,
                        "32 ray + 16 hit", rays_of(q1) - rays_of(q0), q1["ms_extend"] - q0["ms_extend"], launches_s,
                        ext_ms / max(ext_launches, 1))
        roofline_shadow = roof("k_traverse_wide<anyhit> (shadow rays)", "k_traverse_shadow", cs["rays_shadow_traced"], cs["node_visits_shadow"],
                               cs["prim_tests_shadow"], 36 + 16 * f_blk + 32 * f_tnt,
                               "32 ray + 4 queue + 16 x %.3f blocked + 32 x %.3f tinted" % (f_blk, f_tnt),
                               q1["rays_shadow_traced"] - q0["rays_shadow_traced"], q1["ms_shadow"] - q0["ms_shadow"], launches_s,
                               (s1["ms_shadow"] - s0["ms_shadow"]) / max(ext_launches, 1))
        b_bytes = 450.0 * info.n_triangles
        roofline_build = {"bound": "hbm", "kernel": "mox_build_accel (Morton + onesweep sort + PLOC + SAH-optimal collapse + pack)",
                          "achieved": b_bytes / (build_ms * 1e-3) / 1e9 if build_ms > 0 else 0.0, "peak": peak, "unit": "GB/s",
                          "frac": b_bytes / (build_ms * 1e-3) / 1e9 / peak if build_ms > 0 else 0.0, "bytes_per_triangle": 450,
                          "triangles": int(info.n_triangles), "ms": build_ms, "traffic": None}
        del cctx, sctx

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        per_step, cinfo = cpu_sample(args, 3)
        crays = sum(r for r, _ in per_step[1:])
        csec = sum(s for _, s in per_step[1:])
        cpu_baseline = dict(cinfo, value=crays / csec / 1e6, unit="Mrays/s")

    if rank == 0:
        line = {"metric": "Mrays/s (primary+bounce)", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": WORKLOAD, "triangles": int(info.n_triangles), "width": W, "height": H, "max_depth": MAX_DEPTH,
                           "rng": "ref", "parallelism": f"tile-split x{world}, scene replicated, one gather per read-back",
                           "l2": "per-step path state (>0.7 GB) + scene exceed the 126 MB L2; no explicit flush"},
                "spp_per_s": args.steps * SPP_PER_STEP / (dev_ms * 1e-3), "mshadow_per_s": shadow_all / (dev_ms * 1e3), "bvh_build_ms": build_ms,
                "wall_ms_per_step": wall_ms / args.steps, "step_wall_ms": step_wall, "e2e_step_wall_ms": e2e_step_wall, "stage_ms": stage_ms,
                "e2e": {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": 76 + 4, "d2h_bytes_per_step": int(d2h)},
                "gather_bytes": tiles.bytes_on_the_wire(), "gather_transport": tiles.transport(), "gather_ms": g0.elapsed_time(g1), "render_ms_rank0": s1["ms_render"] - s0["ms_render"], "render_ms_per_rank": render_per_rank, "tile": TILE, "gpu_launches": int(launches_all), "clocks": clocks, "roofline": roofline_shadow if (roofline_shadow and roofline and roofline_shadow["share_of_step"] > roofline["share_of_step"]) else roofline,
                "roofline_closest": roofline, "roofline_shadow": roofline_shadow, "roofline_build": roofline_build,
                "serial_pass": serial, "per_depth": per_depth, "cpu_baseline": cpu_baseline}
        if dump is not None:
            write_dump(args.dump_outputs, dump)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
