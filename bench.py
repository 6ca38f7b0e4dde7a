#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (see DESIGN.md "Measurement").

  python bench.py --gpus N --steps K --warmup W [--workload cfg4|cfg3|cfg2|small] [--impl reference]

Default workload (round 2): cfg4 = BASELINE configs[3], the 10 M-triangle soup with four BSDF families and 16
area lights at 1920x1080 x 1024 spp -- configs[2]'s scene (the one the north-star target is quoted on) under
configs[3]'s lights -- at every N, so that the N=1 line and the scaling lines describe the same job.

One "step" = one complete pass of the hot path over the workload: every 16x16
tile of the film rendered with all its samples per pixel (SamplerIntegrator::
Render), film tiles sharded over the ranks (tile i -> rank i mod N) and the raw
film sums reduced to rank 0 (one NCCL reduce) when N > 1.
Metric: Mrays/s = (Scene::Intersect + Scene::IntersectP calls of all ranks) / time,
the reference's own ray counters (core/scene.cpp:40-52).
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as graft  # noqa: E402

WORKLOADS = {
    # name: (n_tris, materials, xres, yres, spp, max_depth, n_lights, description)
    "cfg2": (1000000, ("matte",), 1024, 1024, 256, 5, None,
             "synthetic 1M random triangles (soup v1), single diffuse BSDF, 256spp, 1024x1024"),
    "cfg3": (10000000, ("matte", "glass", "metal", "plastic"), 1920, 1080, 1024, 5, None,
             "synthetic 10M triangles, 4 BSDF types, 1024spp, 1920x1080"),
    "cfg4": (10000000, ("matte", "glass", "metal", "plastic"), 1920, 1080, 1024, 5, 16,
             "synthetic 10M triangles + 16 area lights (MIS), 1024spp, 1920x1080, tile-sharded"),
    # BASELINE configs[4] without its SampledSpectrum half and at a reduced film / sample count (the full
    # 3840x2160 x 4096 spp job is sized for 8 GPUs): 50 M instanced triangles = 1000 instances of one 50k-triangle object
    "cfg5rgb": (100000, ("matte", "glass", "metal", "plastic"), 1920, 1080, 64, 16, None,
                "synthetic 50M triangles instanced (1000 x 50k, RGB spectrum), maxdepth 16, 64spp, 1920x1080"),
    # the same with the reference's SampledSpectrum build (60 bins): both halves of BASELINE configs[4]'s feature set
    "cfg5": (100000, ("matte", "glass", "metal", "plastic"), 1920, 1080, 64, 16, None,
             "synthetic 50M triangles instanced (1000 x 50k), SampledSpectrum (60 bins), maxdepth 16, 64spp, 1920x1080"),
    # the instanced scene as SURVEY 8(d) words it: 50 ObjectInstances of one 1 M-triangle soup under distinct transforms
    # (= 50 M instanced triangles) around a 100 k-triangle top-level soup
    "cfg5s": (100000, ("matte", "glass", "metal", "plastic"), 1920, 1080, 64, 16, None,
              "synthetic 50M triangles instanced (50 x 1M, RGB spectrum), maxdepth 16, 64spp, 1920x1080"),
    # cfg2's scene inside a thin homogeneous medium, VolPathIntegrator (SURVEY 8(f) row 4)
    "cfg2fog": (1000000, ("matte",), 1024, 1024, 256, 5, None,
                "synthetic 1M triangles in a homogeneous medium (sigma_t ~0.3, g 0.4), volpath, maxdepth 5, 256spp, 1024x1024"),
    "small": (100000, ("matte", "glass", "metal", "plastic"), 256, 256, 16, 5, None,
              "smoke-sized: 100k triangles, 4 BSDF types, 16spp, 256x256"),
}


def workload_scene_kwargs(name):
    """Extra SceneArrays arguments of a workload (object instancing for cfg5rgb)."""
    if name == "cfg5s":
        inst = []
        for k in range(50):  # 5 x 5 x 2 lattice, every third instance mirrored / stretched
            c = (-0.8 + 0.4 * (k % 5), -0.8 + 0.4 * ((k // 5) % 5), -0.4 + 0.8 * (k // 25))
            sc = (1.0, 1.0, 1.0) if k % 3 == 0 else ((1.2, 0.8, 1.0) if k % 3 == 1 else (1.0, 1.0, -1.1))
            inst.append(dict(object=0, center=c, scale=sc))
        return dict(objects=(dict(n_tris=1000000, seed=77, material="plastic", size=0.25),), instances=tuple(inst))
    if name not in ("cfg5rgb", "cfg5"):
        return {}
    inst = []
    for k in range(1000):  # 10 x 10 x 10 lattice through the soup's volume, every third one mirrored / stretched
        c = (-0.9 + 0.2 * (k % 10), -0.9 + 0.2 * ((k // 10) % 10), -0.9 + 0.2 * (k // 100))
        sc = (1.0, 1.0, 1.0) if k % 3 == 0 else ((1.2, 0.8, 1.0) if k % 3 == 1 else (1.0, 1.0, -1.1))
        inst.append(dict(object=0, center=c, scale=sc))
    return dict(objects=(dict(n_tris=50000, seed=77, material="plastic", size=0.09),), instances=tuple(inst))


SPECTRAL_WORKLOADS = ("cfg5",)
# workload -> keyword arguments for RenderSetup / write_pbrt: VolPathIntegrator and its medium
VOLUMETRIC_WORKLOADS = {"cfg2fog": dict(integrator="volpath", medium=dict(sigma_a=(0.05, 0.08, 0.12), sigma_s=(0.3, 0.25, 0.2), g=0.4))}


def spectral_tables():
    """The 60-bin spectra of the harness's materials and lights as the SampledSpectrum reference holds them (fixtures)."""
    return json.load(open(os.path.join(ROOT, "tests", "golden", "spectral_tables.json")))


def rank_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons of one GPU during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 7:
                    self.samples.append(f)
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[3 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.samples[0][1]),
                "power_w_max": max(float(s[2]) for s in self.samples), "samples": len(self.samples),
                "reasons": reasons}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dirname, arrays):
    """Writes each array as dirname/<name>.npy, so that two builds can be compared output for output on the same
    seeded workload.  Every workload's film (at most 1920x1080) fits the limit whole, so nothing is sampled."""
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError("outputs of %d bytes exceed the %d-byte dump limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(dirname, name + ".npy"), a)


def write_reference_scene(scenes, arr, wl, spp, tmp):
    n_tris, mats, xres, yres, _, depth, n_lights, _ = wl
    return scenes.write_pbrt(tmp, "bench", arr, xres, yres, spp, max_depth=depth, strategy="uniform", **getattr(arr, "bench_integrator", {}))


def parse_pbrt_output(out):
    def num(pat):
        m = re.search(pat, out)
        return float(m.group(1)) if m else 0.0
    secs = [float(x) for x in re.findall(r"\((\d+\.\d+)s\)", out)]
    return {"render_s": secs[-1] if secs else None,
            "camera": num(r"Camera rays traced\s+(\d+)"),
            "regular": num(r"Regular ray intersection tests\s+(\d+)"),
            "shadow": num(r"Shadow ray intersection tests\s+(\d+)")}


def reference_step(ob, scenes, abi, arr, wl, setup_small, sample_spp, tmp, pbrt_path, spectral=False):
    """One bounded sample of the workload on the host cores: the unmodified
    reference when oracle/_ref exists (kind 'reference'), else the oracle port."""
    cores = os.cpu_count() or 1
    if pbrt_path is not None:
        t0 = time.time()
        out = ob.run_pbrt_ref(pbrt_path, threads=cores, spectral=spectral)
        wall = time.time() - t0
        st = parse_pbrt_output(out)
        secs = st["render_s"] or wall
        return {"kind": "reference", "cores": cores, "rays": st["regular"] + st["shadow"], "samples": st["camera"],
                "seconds": secs}
    o = ob.Oracle(abi, arr)
    t0 = time.time()
    _, st = o.render(setup_small, threads=cores)
    secs = time.time() - t0
    o.close()
    return {"kind": "port", "cores": cores, "rays": st["regular_rays"] + st["shadow_rays"],
            "samples": st["camera_rays"], "seconds": secs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="cfg4", choices=sorted(WORKLOADS))
    ap.add_argument("--e2e-steps", type=int, default=None, help="timed steps of the end-to-end leg (default: min(steps, 5))")
    ap.add_argument("--no-parity", action="store_true", help="skip the full-size comparison with the reference's image")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-sample-spp", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--pixel-filter", default=None,
                    help="a key of tests/golden/filter_tables.json (gaussian, mitchell, sinc ...); default: box filter")
    ap.add_argument("--bvh", default="host", choices=["host", "gpu"],
                    help="acceleration structure builder: host SAH (default) or the on-device builder")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the film of the last timed step as DIR/image_rgb.npy and DIR/film_raw.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank, local_rank, world = rank_env()
    wl = WORKLOADS[args.workload]
    n_tris, mats, xres, yres, spp, depth, n_lights, desc = wl

    if args.impl == "reference":
        abi, scenes = graft.load_harness()  # descriptor helpers only: the reference arm maps none of the repo's CUDA code
    else:
        pkg = graft.load_package()
        from pbrt_v3_distributed_b200 import abi, scenes
    config = {"workload": "%s: %s, maxdepth %d, Sobol, box filter, lightsamplestrategy uniform" %
              (args.workload, desc, depth),
              "n_triangles": n_tris, "resolution": [xres, yres], "spp": spp,
              "scene": "soup v1 (s=0.5*N^-1/3, seed 1234) + %s" %
                       ("%d emissive triangles at y=+3" % n_lights if n_lights else "5 inward emissive quads (10 lights), L=40"),
              "parallelism": "tiles i mod %d over %d GPU(s), one film reduce" % (world, world) if world > 1 else "1 GPU",
              "l2_policy": "inputs larger than L2 (BVH+triangles %s MB, path state > 0.5 GB); no flush needed",
              "excluded_from_timing": "scene_create (host BVH build + first upload), like the reference arm's parse + BVH build"}

    # ------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        ob = graft.load_oracle()
        arr = scenes.SceneArrays(n_tris, materials=mats, soup_version=1, n_lights=n_lights, **workload_scene_kwargs(args.workload))
        spectral = args.workload in SPECTRAL_WORKLOADS
        if spectral:
            arr.attach_spectral(spectral_tables())  # the oracle port reads the tables; the reference binary has its own
        arr.bench_integrator = VOLUMETRIC_WORKLOADS.get(args.workload, {})
        tmp = tempfile.mkdtemp(prefix="b200pt_ref_")
        have_ref = os.path.exists(ob.PBRT_REF_SPECTRAL) if spectral else ob.have_reference()
        pbrt_path = write_reference_scene(scenes, arr, wl, args.cpu_sample_spp, tmp) if have_ref else None
        setup_small = None
        if not have_ref:
            # no reference binary on this box: the oracle port renders the sample; its camera descriptor comes from the
            # library's host helper (no kernel of the repo runs in this arm either way)
            graft.load_package()
            from pbrt_v3_distributed_b200 import scenes as scenes_full
            setup_small = scenes_full.RenderSetup(xres, yres, args.cpu_sample_spp, max_depth=depth, **arr.bench_integrator)
        # A step is one launch of the reference on the bounded sample (scene load + BVH build + render; only the render
        # is timed, like scene_create is excluded on the GPU arm).  The whole arm must end within a few minutes whatever
        # --steps / --warmup ask for: the wall time of the first launch decides how many launches fit the budget
        # (B200PT_REF_BUDGET_S, default 420 s); the rate does not depend on their number.
        budget_s = float(os.environ.get("B200PT_REF_BUDGET_S", "420"))
        rays = secs = samples = 0.0
        last = None
        total, warm = args.warmup + args.steps, args.warmup
        i = 0
        t_arm = time.time()
        wall_first = None
        while i < total:
            last = reference_step(ob, scenes, abi, arr, wl, setup_small, args.cpu_sample_spp, tmp, pbrt_path, spectral)
            if wall_first is None:
                wall_first = time.time() - t_arm
                fit = max(2 if args.warmup > 0 else 1, int(budget_s // max(wall_first, 1e-3)))
                if fit < total:
                    total = fit
                    warm = min(args.warmup, max(total - max(1, min(args.steps, total // 2 + 1)), 0))
                    if args.warmup > 0:
                        warm = max(warm, 1)
            if i >= warm:
                rays += last["rays"]
                secs += last["seconds"]
                samples += last["samples"]
            i += 1
        timed = total - warm
        value = rays / secs / 1e6
        sample = "%dx%d film, %d spp of %d, all tiles, per step; %d timed + %d warm-up launches (%.0f s wall each, budget %.0f s)" % (
            xres, yres, args.cpu_sample_spp, spp, timed, warm, wall_first, budget_s)
        config["l2_policy"] = "n/a (CPU)"
        print(json.dumps({
            "impl": "reference", "metric": "Mrays/s (primary+secondary)", "value": value, "unit": "Mrays/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * secs / max(timed, 1), "steps_run": timed, "warmup_run": warm,
            "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32 x 60 spectral bins" if args.workload in SPECTRAL_WORKLOADS else "f32", "data": "synthetic", "config": config,
            "msamples_per_s": samples / secs / 1e6,
            "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": last["cores"], "kind": last["kind"],
                             "sample": sample},
            "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return 0

    # ------------------------------------------------------------------ B200 arm
    import torch
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device; this benchmark has no CPU fallback"}))
        return 2
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    arr = scenes.SceneArrays(n_tris, materials=mats, soup_version=1, n_lights=n_lights, **workload_scene_kwargs(args.workload))
    if args.workload in SPECTRAL_WORKLOADS:
        arr.attach_spectral(spectral_tables())
    arr.bench_integrator = VOLUMETRIC_WORKLOADS.get(args.workload, {})
    setup = scenes.RenderSetup(xres, yres, spp, max_depth=depth, pixel_filter=args.pixel_filter, **arr.bench_integrator)
    if args.pixel_filter:
        config["pixel_filter"] = args.pixel_filter
    ctx = pkg.Context(local_rank)
    if args.bvh == "gpu":
        ctx.set_option("gpu_bvh_build", 1)
    t0 = time.time()
    scene = pkg.Scene(ctx, arr.desc(), keepalive=arr)
    build_s = time.time() - t0
    info = scene.info()
    config["l2_policy"] = config["l2_policy"] % ("%.0f" % ((info["node_bytes"] + info["tri_bytes"]) / 1e6))
    config["bvh"] = {"nodes": info["n_nodes"], "node_bytes": info["node_bytes"], "tri_bytes": info["tri_bytes"],
                     "host_build_s": round(build_s, 2),
                     "builder": "device (Morton order -> radix tree -> 7-wide collapse)" if args.bvh == "gpu" else "host SAH",
                     "layout": "7-wide, 64-byte nodes + 4-byte triangle base per node, 48-byte triangles"}
    render = pkg.Render(scene, setup)
    comm = None
    if world > 1:
        # the library's own communicator for the film merge (b200pt_comm_create: NCCL id through a file); torch.distributed
        # stays the launcher's plumbing (rendezvous of this file name, barriers, the max / sum of the timing scalars)
        token = [os.path.join(tempfile.gettempdir(), "b200pt_nccl_%d_%d.id" % (os.getpid(), int(time.time() * 1e3)))]
        dist.broadcast_object_list(token, src=0)
        comm = pkg.Comm(ctx, rank, world, token[0])
    my_tiles = scenes.rank_tiles(render.n_tiles, rank, world)
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local_rank))
    film_ptr, film_n = render.film_device_buffer()

    class _Film:
        __cuda_array_interface__ = {"shape": (film_n,), "typestr": "<f4", "data": (film_ptr, False), "version": 2}
    film_t = torch.as_tensor(_Film(), device=torch.device("cuda", local_rank))
    host_rgb = torch.empty((render.height, render.width, 3), dtype=torch.float32).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(e2e, marks=None):
        h2d = 0
        if e2e:
            h2d = scene.upload()                      # pinned host -> device: BVH nodes + triangle records
        render.clear()
        if marks is not None and world > 1:
            m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(stream):
                m0.record()
        render.render_tiles(my_tiles)
        if marks is not None and world > 1:
            with torch.cuda.stream(stream):
                m1.record()
            marks.append((m0, m1))
        if world > 1:
            render.film_reduce(comm, 0)               # one ncclReduce of the raw film sums, behind the C ABI
        if e2e and rank == 0:
            pkg._check(pkg.lib.b200pt_film_read_rgb(render.h, host_rgb.data_ptr()))
        return h2d

    # instrumented pass (untimed): BVH nodes fetched / triangles tested per ray -> algorithmic bytes
    render.set_option("instrument", 1)
    step(False)
    ctx.synchronize()
    st_i = render.stats()
    render.set_option("instrument", 0)
    render.reset_stats()

    def timed(e2e, steps, warmup):
        for _ in range(warmup):
            step(e2e)
        barrier()
        render.reset_stats()
        render.set_option("profile", 1)
        sampler = ClockSampler(local_rank)
        sampler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            ev0.record()
        h2d = 0
        marks = []
        for _ in range(steps):
            h2d = step(e2e, marks)
        with torch.cuda.stream(stream):
            ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        busy_ms = sum(a.elapsed_time(b) for a, b in marks) if marks else ms
        clocks = sampler.summary()
        st = render.stats()
        render.set_option("profile", 0)
        t = torch.tensor([ms, float(st["regular_rays"] + st["shadow_rays"]), float(st["camera_rays"])],
                         dtype=torch.float64, device="cuda")
        rank_ms = [ms]
        if world > 1:
            # every rank's device time for rendering its own tiles in the same K steps (before the film reduce, which makes
            # the fast ranks wait): the load balance of the static tile split shows as the spread of these
            every = [torch.zeros(1, dtype=torch.float64, device="cuda") for _ in range(world)]
            dist.all_gather(every, torch.tensor([busy_ms], dtype=torch.float64, device="cuda"))
            rank_ms = [float(x[0]) for x in every]
            mx = t.clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            ms = float(mx[0])
        timed.rank_ms = rank_ms
        return ms, float(t[1]), float(t[2]), st, clocks, h2d

    ms, rays, samples, st, clocks, _ = timed(False, args.steps, args.warmup)
    rank_ms = list(timed.rank_ms)
    if args.dump_outputs and rank == 0:
        # read before the end-to-end leg renders into the same film; on rank 0 it holds every rank's reduced sums
        dump_outputs(args.dump_outputs, {"image_rgb": render.read_rgb(), "film_raw": render.read_raw()})
    e2e_steps = args.e2e_steps if args.e2e_steps else min(args.steps, 5)
    ms_e, rays_e, samples_e, st_e, _, h2d = timed(True, e2e_steps, 1)
    # one more end-to-end step with events between its three parts (reported, not part of any timed figure)
    breakdown = None
    if world == 1:
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        with torch.cuda.stream(stream):
            evs[0].record()
        scene.upload()
        with torch.cuda.stream(stream):
            evs[1].record()
        render.clear()
        render.render_tiles(my_tiles)
        with torch.cuda.stream(stream):
            evs[2].record()
        pkg._check(pkg.lib.b200pt_film_read_rgb(render.h, host_rgb.data_ptr()))
        with torch.cuda.stream(stream):
            evs[3].record()
        torch.cuda.synchronize()
        breakdown = {"upload_ms": evs[0].elapsed_time(evs[1]), "render_ms": evs[1].elapsed_time(evs[2]),
                     "readback_ms": evs[2].elapsed_time(evs[3])}

    out = None
    if rank == 0:
        peaks, peak_kind = measured_peaks()
        value = rays / (ms * 1e-3) / 1e6
        # roofline of the dominant kernel: closest-hit traversal (k_trace<false,...>)
        n_reg = st_i["regular_rays"]
        bytes_per_closest_ray = 32 + 4 + (st_i["nodes_visited"] * 64.0 + st_i["tris_tested"] * 48.0) / max(n_reg, 1)
        closest_bytes = bytes_per_closest_ray * st["regular_rays"]
        achieved = closest_bytes / (st["closest_ms"] * 1e-3) / 1e9 if st["closest_ms"] > 0 else 0.0
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get(args.workload)
        cpu = None
        parity = None
        if not args.no_cpu_baseline:
            ob = graft.load_oracle()
            tmp = tempfile.mkdtemp(prefix="b200pt_cpu_")
            setup_small = scenes.RenderSetup(xres, yres, args.cpu_sample_spp, max_depth=depth, **arr.bench_integrator)
            spectral = args.workload in SPECTRAL_WORKLOADS
            have_ref = os.path.exists(ob.PBRT_REF_SPECTRAL) if spectral else ob.have_reference()
            pbrt_path = write_reference_scene(scenes, arr, wl, args.cpu_sample_spp, tmp) if have_ref else None
            c = reference_step(ob, scenes, abi, arr, wl, setup_small, args.cpu_sample_spp, tmp, pbrt_path, spectral)
            if pbrt_path is not None and not args.no_parity and world == 1:
                # full-size parity (SURVEY 8d protocol): the image the reference just rendered (same scene, same film,
                # cpu_sample_spp samples per pixel) against the GPU render of the same job
                ref_img = scenes.read_pfm(os.path.join(tmp, "bench.pfm"))
                r2 = pkg.Render(scene, setup_small)
                r2.clear()
                r2.render_tiles()
                got = r2.read_rgb()
                st2 = r2.stats()
                r2.close()
                a, b = got.astype(np.float64), ref_img.astype(np.float64)
                eps = 1e-3 * float(b.mean())
                rel = np.abs(a - b) / np.maximum(np.abs(b), eps)
                parity = {"against": "oracle/_ref/pbrt_ref PFM of the same scene, %dx%d, %d spp" % (xres, yres, args.cpu_sample_spp),
                          "max_rel": float(rel.max()), "p99_9_rel": float(np.percentile(rel, 99.9)),
                          "components_over_1e-4": int((rel > 1e-4).sum()),
                          "components_bits_differ": int((got.view(np.uint32) != ref_img.view(np.uint32)).sum()),
                          "components": int(got.size),
                          "ray_counters_equal": bool(st2["regular_rays"] + st2["shadow_rays"] == c["rays"] and st2["camera_rays"] == c["samples"]),
                          "rays_gpu_reference": [int(st2["regular_rays"] + st2["shadow_rays"]), int(c["rays"])],
                          "samples_gpu_reference": [int(st2["camera_rays"]), int(c["samples"])],
                          "stack_overflows": int(st2.get("stack_overflows", 0))}
            cpu = {"value": c["rays"] / c["seconds"] / 1e6, "unit": "Mrays/s", "cores": c["cores"], "kind": c["kind"],
                   "sample": "%dx%d film, %d spp of %d, all tiles (%.1f s render)" %
                             (xres, yres, args.cpu_sample_spp, spp, c["seconds"]),
                   "msamples_per_s": c["samples"] / c["seconds"] / 1e6}
        out = {
            "metric": "Mrays/s (primary+secondary)", "value": value, "unit": "Mrays/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32 x 60 spectral bins" if args.workload in SPECTRAL_WORKLOADS else "f32", "data": "synthetic", "config": config,
            "msamples_per_s": samples / (ms * 1e-3) / 1e6,
            "rays_per_sample": rays / max(samples, 1),
            "ray_mix_per_step": {"camera": int(st["camera_rays"] // args.steps), "regular": int(st["regular_rays"] // args.steps),
                                 "shadow": int(st["shadow_rays"] // args.steps)},
            # frac = ALGORITHMIC bytes (nodes fetched + triangles tested + ray in / hit out) / time / HBM peak.  Those bytes
            # are mostly served by L2 (the BVH's hot part is cache resident), so frac is NOT DRAM utilisation: dram_frac is,
            # from the ncu capture of the same kernel and workload under profiles/ (traffic.source).
            "roofline": {"bound": "hbm (north_star's roofline; ncu: the kernel is issue / L2->SM bound, see dram_frac and profiles/README.md)",
                         "kernel": "k_trace<closest-hit> (7-wide BVH traversal)",
                         "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": achieved / peaks["hbm_gbs"], "peak_kind": peak_kind, "traffic": traffic,
                         "dram_frac": (traffic or {}).get("dram_frac"),
                         "algorithmic_bytes_per_ray": bytes_per_closest_ray,
                         "nodes_per_ray": st_i["nodes_visited"] / max(n_reg, 1),
                         "tris_per_ray": st_i["tris_tested"] / max(n_reg, 1),
                         "avg_launch_ms": st["closest_ms"] / max(st["closest_launches"], 1),
                         "launches": st["closest_launches"],
                         "share_of_step": st["closest_ms"] / ms if ms > 0 else None},
            "kernel_ms_per_step": {"closest_hit": st["closest_ms"] / args.steps, "any_hit": st["any_ms"] / args.steps,
                                   "shade_raygen_film": st["shade_ms"] / args.steps},
            "cpu_baseline": cpu,
            "parity": parity,
            "e2e": {"value": rays_e / (ms_e * 1e-3) / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(host_rgb.numel() * 4), "ms_per_step": ms_e / e2e_steps, "steps": e2e_steps,
                    "excludes": "scene_create", "breakdown_ms": breakdown},
            "stack_overflows": int(st.get("stack_overflows", 0)),
            "per_rank_render_ms_per_step": [x / args.steps for x in rank_ms],
            "gpu_launches": int(st["launches"]),
            "clocks": clocks,
        }
        print(json.dumps(out))
    if comm is not None:
        comm.close()
    render.close()
    scene.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
