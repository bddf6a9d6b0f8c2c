#!/usr/bin/env python
"""Headline benchmark: frames/sec (+ HBM GB/s of the dominant kernel) of the clustered deferred
lighting + HDR post chain on a 3840x2160 synthetic G-buffer with 4096 lights (BASELINE.json).

  python bench.py --gpus N --steps K --warmup W            # our CUDA path (torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's algorithm on the host cores
                                                           # (CPU oracle; the reference has no CPU path
                                                           #  and no Vulkan device exists here)
Prints ONE JSON line on rank 0.  A "step" is one frame.  --dump-outputs DIR writes the output frame of
the last timed step as .npy files, so that two builds can be compared on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import atexit
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

WORKLOADS = {
    # name: (width, height, lights, post_aa, description)
    "c1": (256, 256, 16, "none", "256x256 G-buffer, 16 point lights + directional, tonemap only (no bloom, fixed exposure): the reference's smallest case"),
    "c3": (3840, 2160, 4096, "none", "3840x2160 G-buffer, 4096 clustered point lights + directional, bloom + luminance + tonemap"),
    "c2": (1920, 1080, 1024, "none", "1920x1080 G-buffer, 1024 clustered lights, full bloom/tonemap chain"),
    "c5": (3840, 2160, 4096, "taa+fxaa", "3840x2160 TAA(q2) + FXAA post-AA with history buffer"),
}
NO_BLOOM = {"c1"}  # BASELINE config 1: DYNAMIC_EXPOSURE=0, bloom disabled
LIGHTING_BYTES_PER_PIXEL = 22  # SURVEY.md §8d: 4 albedo + 4 normal + 2 pbr + 4 depth + 4 emissive read, 4 HDR write


def algorithmic_bytes(w, h, aa, bloom=True):
    """Compulsory HBM traffic per frame, unfused pass-by-pass accounting of SURVEY.md §8d."""
    px = w * h
    if not bloom:
        return px * LIGHTING_BYTES_PER_PIXEL, px * 8, px * (LIGHTING_BYTES_PER_PIXEL + 8)
    sz = [(math.ceil(w * s), math.ceil(h * s)) for s in (0.5, 0.25, 0.125, 0.0625, 0.03125)]
    t, d0, d1, d2, d3 = [a * b for a, b in sz]
    lighting = px * LIGHTING_BYTES_PER_PIXEL
    chain = (px * 4 + t * 8) + (t * 8 + d0 * 8) + (d0 * 8 + d1 * 8) + (d1 * 8 + d2 * 8) + (d2 * 8 + d3 * 8 + d3 * 8) \
        + d3 * 8 // 4 + (d3 * 8 + d2 * 8) + (d2 * 8 + d1 * 8) + (d1 * 8 + d0 * 8) + (px * 4 + d0 * 8 + px * 4)
    total = lighting + chain
    if aa == "taa+fxaa":
        total += px * 32 + px * 8
    return lighting, chain, total


DUMP_PIXELS = 1 << 21  # a larger frame is dumped as this many pixels, a seeded sample: 48 MB with their indices


def dump_outputs(out_dir, frame):
    """Writes the RGBA8 output frame (rows, width) uint32 as out_dir/frame_rgba8.npy: float32 (rows, width, 4)
    of the 0..255 channel values, or, above DUMP_PIXELS pixels, float32 (DUMP_PIXELS, 4) for a fixed seeded
    sample of them plus out_dir/frame_rgba8_index.npy, their row-major pixel indices as float64."""
    os.makedirs(out_dir, exist_ok=True)
    rgba = np.ascontiguousarray(frame).view(np.uint8).reshape(frame.shape[0], frame.shape[1], 4).astype(np.float32)
    if frame.size > DUMP_PIXELS:
        idx = np.sort(np.random.default_rng(0).choice(frame.size, DUMP_PIXELS, replace=False))
        rgba = rgba.reshape(-1, 4)[idx]
        np.save(os.path.join(out_dir, "frame_rgba8_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "frame_rgba8.npy"), rgba)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.stop)  # never outlives the benchmark, even when it fails
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        sm, mx, reasons = [], 0.0, set()
        for t, line in self.samples:
            if t < t0 - 0.05 or t > t1 + 0.05:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0]))
                mx = max(mx, float(f[1]))
            except Exception:
                continue
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def ncu_traffic():
    """dram bytes per launch of the lighting kernel from the committed ncu capture, if any."""
    p = os.path.join(ROOT, "profiles", "lighting_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("dram_bytes_per_launch")
        except Exception:
            return None
    return None


# ------------------------------------------------------------------------------------------------
def _native_oracle():
    """The oracle rebuilt for THIS machine's cores (-O3 -march=native, BASELINE.md section 4) in a
    temporary directory (the source tree may be read-only): the in-tree liboracle.so is a portable -O2
    build because it may be built on another machine.  Same sources, same -ffp-contract=off arithmetic contract."""
    import shutil
    import subprocess
    import tempfile
    from oracle import pyoracle as oracle

    src_dir = os.path.dirname(os.path.abspath(oracle.__file__))
    in_tree = oracle._LIB_PATH
    out_dir = tempfile.mkdtemp(prefix="granite_b200_oracle_")
    out = os.path.join(out_dir, "liboracle.so")
    srcs = [os.path.join(src_dir, f) for f in ("oracle_host.c", "oracle_cluster.c", "oracle_lighting.c", "oracle_post.c", "oracle_smaa.c")]
    try:
        subprocess.run(["gcc", "-O3", "-march=native", "-std=c11", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-shared", "-o", out,
                        *srcs, "-lm"], check=True, capture_output=True)
        oracle._LIB_PATH = out
        oracle._lib = None
        oracle.lib()  # loaded now, so the temporary file can go
        return "-O3 -march=native"
    except Exception:
        oracle._LIB_PATH, oracle._lib = in_tree, None
        oracle.build(ref=False)
        return "-O2 (native rebuild failed)"
    finally:
        shutil.rmtree(out_dir, ignore_errors=True)


def oracle_frame_time(w, h, n_lights, aa, steps, warmup, budget_s=150.0, bloom=True):
    """Times the CPU oracle (the reference's algorithm restated in C, OpenMP over rows) on a bounded
    sample of the frame: the cluster build and the pyramid tail in full, the per-pixel passes on a
    band of rows, scaled to the whole frame.  ONE code path for the `cpu_baseline` key and the
    `--impl reference` arm: native build, threads bound to cores, `warmup` untimed steps, then the
    MEDIAN of `steps` timed steps."""
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    from granite_b200 import synth
    from oracle import pyoracle as oracle

    build_flags = _native_oracle()
    steps = max(int(steps), 1)
    warmup = max(int(warmup), 1)
    cores = os.cpu_count() or 1
    scene = synth.make_scene(w, h)
    cam = oracle.camera_setup(scene.projection, scene.view)
    lights = synth.make_lights(n_lights, aspect=w / h)
    prep = oracle.prepare_lights(cam, lights, res=synth.CLUSTER_RES)
    sz = oracle.pyramid_sizes(w, h)

    def frame(rows):
        """One frame with the per-pixel passes restricted to full-res rows [0, rows)."""
        t0 = time.perf_counter()
        clus = oracle.cluster_build(cam, prep)
        t1 = time.perf_counter()
        hdr = oracle.deferred_lighting(scene, cam, prep, clus, rows=(0, rows))
        t2 = time.perf_counter()
        hs = hdr[:rows]
        if not bloom:
            zero = np.zeros((-(-rows // 4), -(-w // 4), 4), np.uint16)
            oracle.tonemap(hs, zero, None, 1.0)
            t3 = time.perf_counter()
            return (t3 - t1), (t1 - t0), 0.0
        psz = oracle.pyramid_sizes(w, rows)
        t = oracle.bloom_threshold(hs, np.zeros(3, np.float32), psz[0])
        d0 = oracle.bloom_downsample(t, psz[1])
        t3 = time.perf_counter()
        # pyramid tail at FULL frame size (it is tiny): d1..d3, luminance, u2, u1
        full_d0 = np.zeros((sz[1][1], sz[1][0], 4), np.uint16)
        d1 = oracle.bloom_downsample(full_d0, sz[2])
        d2 = oracle.bloom_downsample(d1, sz[3])
        d3 = oracle.bloom_downsample(d2, sz[4], d2[: sz[4][1], : sz[4][0]].copy(), 0.1)
        lum = oracle.luminance(d3, np.zeros(3, np.float32), 0.01)
        u2 = oracle.bloom_upsample(d3, sz[3])
        u1 = oracle.bloom_upsample(u2, sz[2])
        t4 = time.perf_counter()
        u0 = oracle.bloom_upsample(u1[: psz[2][1]], psz[1])
        ldr = oracle.tonemap(hs, u0, lum, 1.0)
        extra = 0.0
        if aa == "taa+fxaa":
            ta = time.perf_counter()
            mv = np.zeros((rows, w, 2), np.uint16)
            hist = np.zeros((rows, w, 4), np.uint16)
            oracle.taa_resolve(hs, scene.depth[:rows], mv, hist, np.eye(4, dtype=np.float32), 2)
            oracle.fxaa(ldr, True)
            extra = time.perf_counter() - ta
        t5 = time.perf_counter()
        band = (t2 - t1) + (t3 - t2) + (t5 - t4)  # scales with rows
        fixed = (t1 - t0) + (t4 - t3)             # cluster build + pyramid tail
        return band, fixed, extra

    # calibrate on one 64-row band, then pick the largest band that fits the budget
    band, fixed, _ = frame(min(64, h))
    est_full = band * (h / float(min(64, h))) + fixed
    frac = min(1.0, budget_s / max(est_full * (steps + warmup), 1e-9))
    rows = int(max(64, min(h, (int(h * frac) // 64) * 64)))
    for _ in range(warmup):
        frame(rows)
    times = []
    for _ in range(steps):
        b, f, _ = frame(rows)
        times.append(b * (h / rows) + f)
    sec = float(np.median(times))
    return sec, cores, (f"median of {steps} steps after {warmup} warm-up, oracle built {build_flags}, OMP_PROC_BIND={os.environ.get('OMP_PROC_BIND')}; "
                        f"per step: cluster build + pyramid tail in full, per-pixel passes on rows [0,{rows}) of {h} scaled x{h / rows:.2f}")


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the output frame of the last timed step to DIR/*.npy (all ranks' rows, written by rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    w, h, n_lights, aa, desc = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    bloom = args.workload not in NO_BLOOM
    lighting_b, chain_b, total_b = algorithmic_bytes(w, h, aa, bloom)
    config = {"workload": f"{args.workload}: {desc}", "width": w, "height": h, "lights": n_lights, "cluster_grid": "128x64x4096",
              "sharding": f"{world} row bands (8-row units): balanced by measured lighting time for the resident region, equal rows for the end-to-end region" if world > 1 else "none",
              "l2": (f"per-frame inputs ({w * h * LIGHTING_BYTES_PER_PIXEL / 1e6:.0f} MB of G-buffer + HDR) exceed the 126 MB L2; no explicit flush"
                     if w * h * LIGHTING_BYTES_PER_PIXEL > 126e6 else
                     f"per-frame inputs ({w * h * LIGHTING_BYTES_PER_PIXEL / 1e6:.1f} MB) fit in the 126 MB L2 and are not flushed: not a headline configuration"),
              "algorithmic_mb_per_frame": round(total_b / 1e6, 2)}

    if args.impl == "reference":
        if rank != 0:
            return 0
        # the row sample inside oracle_frame_time fits the run into its budget down to a band of 64 rows per step;
        # beyond that the run time grows with --steps
        steps = args.steps
        sec, cores, sample = oracle_frame_time(w, h, n_lights, aa, steps, 1, bloom=bloom)
        fps = 1.0 / sec
        line = {"impl": "reference", "metric": "frames/sec", "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": steps,
                "warmup": 1, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak" if world == 1 else "strong",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
                "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "note": "the reference has no CPU path for these passes and cannot run here (no Vulkan device); this is its algorithm restated in C (oracle/), all host threads"}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist

    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback for the product path)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from granite_b200 import synth, viewer

    scene = synth.make_scene(w, h)
    lights = synth.make_lights(n_lights, aspect=w / h)
    post = {"none": viewer.AA_NONE, "taa+fxaa": viewer.AA_TAA_HIGH_PLUS_FXAA}[aa]
    stream = torch.cuda.current_stream()

    def make_viewer(timestamps, pipelined_io=False, use_bands=None):
        v = viewer.Viewer(w, h, post_aa=post, hdr_bloom=bloom, dynamic_exposure=bloom, cuda_device=local_rank, timestamps=timestamps,
                          stream=stream.cuda_stream, pipelined_io=pipelined_io)
        v.set_camera(scene.projection, scene.view)
        v.set_directional(scene.dir_color, scene.dir_direction)
        v.set_lights(lights)
        if world > 1:
            if aa != "none":
                raise SystemExit("row-sharded TAA is not supported")
            uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
            if rank == 0:
                uid.copy_(torch.frombuffer(bytearray(viewer.nccl_unique_id()), dtype=torch.uint8))
            dist.broadcast(uid, 0)
            v.init_collectives(bytes(uid.cpu().numpy().tobytes()), rank, world)
            v.set_row_shards(use_bands if use_bands is not None else bands, rank)
        v.bake()
        return v

    # Row bands: lighting cost follows the lights (in this scene 3 % of the rows hold over half of the
    # light evaluations), so bands are cut for equal estimated work, in units of 8 rows.  The estimate
    # is the lighting kernel's own cluster walk without shading (grb_lighting_row_cost), run once on
    # an unsharded frame before the ranks split it.
    if world > 1:
        cal = viewer.Viewer(w, h, post_aa=viewer.AA_NONE, cuda_device=local_rank, stream=stream.cuda_stream)
        cal.set_camera(scene.projection, scene.view)
        cal.set_directional(scene.dir_color, scene.dir_direction)
        cal.set_lights(lights)
        cal.bake()
        full = [np.ascontiguousarray(a) for a in (scene.albedo, scene.normal, scene.pbr, scene.depth, scene.emissive)]
        cal.render_frame(viewer.Viewer.host_gbuffer(*full))
        cost4 = torch.from_numpy(cal.measure_row_cost().astype(np.int64)).cuda()
        cal.close()
        del full
        dist.broadcast(cost4, 0)
        cost4 = cost4.cpu().numpy()
        bands = viewer.band_partition_measured(h, w, world, cost4, align=8)
        # ... then a few steps of feedback: each rank times the band-dependent passes of its own
        # band (lighting + the per-row post work), the cuts move towards equal time.  Per-band times
        # of this pass are not additive (a narrow band of light-dense rows leaves SMs idle), which a
        # work estimate alone cannot see.
        cal_gb = viewer.Viewer.host_gbuffer(*[np.ascontiguousarray(a) for a in (scene.albedo, scene.normal, scene.pbr, scene.depth, scene.emissive)])
        prior = np.repeat(cost4.astype(np.float64) / 4.0, 4)[:h] + 9.4 * w
        history = []
        for _ in range(6):
            vt = make_viewer(True, use_bands=bands)
            vt.render_frame(cal_gb)
            for _ in range(4):
                vt.render_frame(None)
            vt.sync()
            vt.collect_timings()
            for _ in range(30):
                vt.render_frame(None)
            vt.sync()
            tm = {k: ms / max(c, 1) for k, (ms, c) in vt.collect_timings().items()}
            vt.close()
            mine = torch.tensor([tm.get("lighting", 0.0) + 2.5 * tm.get("tonemap", 0.0)], dtype=torch.float64, device="cuda")
            allt = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(allt, mine)
            times = [float(x.item()) for x in allt]
            history.append((max(times), list(bands)))
            bands = viewer.rebalance_bands(bands, times, h, align=8, damping=0.7, prior_per_row=prior)
        bands = min(history, key=lambda e: e[0])[1]
        e2e_bands = viewer.band_partition(h, world, align=8)  # uploads dominate end to end: equal rows
    else:
        bands = [(0, h)]
        e2e_bands = bands
    if world > 1:
        config["resident_bands"] = [list(b) for b in bands]
    v = make_viewer(False)
    own = bands[rank]
    plan = viewer.shard_plan(w, h, bands if world > 1 else [], rank, aa == "taa+fxaa")
    in_rows = plan["lighting"]

    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int32 if a.dtype == np.uint32 else (np.int16 if a.dtype == np.uint16 else a.dtype))).pin_memory()
    mv = None
    if aa == "taa+fxaa":
        rng = np.random.default_rng(5)
        mvf = np.zeros((h, w, 2), np.float16)
        m = rng.random((h, w)) < 0.1
        mvf[m] = (rng.uniform(-2, 2, size=(int(m.sum()), 2)) / np.array([w, h])).astype(np.float16)
        mv = pin(np.ascontiguousarray(mvf).view(np.uint32)[..., 0])
    host = [pin(scene.albedo), pin(scene.normal), pin(scene.pbr), pin(scene.depth), pin(scene.emissive)]
    gb = viewer.Viewer.host_gbuffer(*host, mv)
    out = torch.zeros((h, w), dtype=torch.int32).pin_memory()
    # bytes the whole job copies per step in the end-to-end region (all ranks)
    e2e_plans = [viewer.shard_plan(w, h, e2e_bands if world > 1 else [], r, aa == "taa+fxaa") for r in range(world)]
    h2d = sum((pl["lighting"][1] - pl["lighting"][0]) for pl in e2e_plans) * w * (LIGHTING_BYTES_PER_PIXEL - 4 + (4 if mv is not None else 0))
    d2h = sum((pl["own"][1] - pl["own"][0]) for pl in e2e_plans) * w * 4

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)

    # warm-up: uploads the G-buffer, builds the history images, adapts the luminance.  It runs after the
    # sampler's start-up pause, so that the single timed window follows a busy device, not an idle one.
    for _ in range(args.warmup):
        v.render_frame(gb)
        v.read_output(out)

    # ---- timed region 1: device-resident inputs (value) ----
    # ONE window of EXACTLY K steps between two events (barrier + synchronize on both sides, max over
    # ranks).  A frame of c3 lasts about half a millisecond on a B200, so a window long enough to be
    # a steady state wants K of a few hundred (the default, 200, times about 0.1 s).
    PREROLL = 4

    def resident_window():
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # Frames overlap on the device (cluster build and pyramid tail of one frame run beside the lighting of the
        # next), so K frames started from an idle device are not K steady-state frames: a few untimed frames fill the
        # pipeline first, the start event follows the last of them on the main stream, and the end event follows
        # the K-th timed frame after ALL streams have drained (so the window is K periods plus the drain).
        for _ in range(PREROLL):
            v.render_frame(None)
        e0.record(stream)
        h0 = time.perf_counter()
        for _ in range(args.steps):
            v.render_frame(None)
        host = (time.perf_counter() - h0) * 1e3  # CPU time to prepare + record the frames (no waiting)
        v.join_streams()  # the end event must cover the side streams (cluster build, post chain) too
        e1.record(stream)
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)), host

    t_begin = time.time()
    ms_resident, host_ms = resident_window()
    frame_stats = {"windows": 1, "steps_per_window": args.steps, "preroll_frames": PREROLL}
    if args.dump_outputs:
        y0, y1 = v.read_output(out)  # the frame of the last timed step, as a caller of the viewer receives it
        frame = out.numpy()
        if world > 1:  # each rank holds its band of rows: rank 0 assembles the whole frame
            parts = [torch.zeros((h, w), dtype=torch.int32, device="cuda") for _ in range(world)]
            spans = [torch.zeros(2, dtype=torch.int64, device="cuda") for _ in range(world)]
            dist.all_gather(parts, out.cuda())
            dist.all_gather(spans, torch.tensor([y0, y1], dtype=torch.int64, device="cuda"))
            frame = np.zeros((h, w), np.int32)
            covered = np.zeros(h, bool)
            for part, span in zip(parts, spans):
                a, b = (int(x) for x in span.tolist())
                frame[a:b] = part[a:b].cpu().numpy()
                covered[a:b] = True
            assert covered.all(), "the ranks' output bands do not cover the frame"
            y0, y1 = 0, h
        if rank == 0:
            dump_outputs(args.dump_outputs, frame[y0:y1])

    # ---- timed region 2: end to end through the host API.  Every step copies its G-buffer rows from
    # pinned host memory to the device and its result rows back; frames are pipelined two deep (the
    # upload of step i+1 and the readback of step i-1 overlap the compute of step i), so the wall
    # clock below is the sustained frame rate of the public API, PCIe included. ----
    v.close()
    v = make_viewer(False, pipelined_io=True, use_bands=e2e_bands)
    outs = [out, torch.zeros((h, w), dtype=torch.int32).pin_memory()]
    for i in range(max(args.warmup // 2, 3)):
        v.render_frame(gb)
        v.read_output_async(outs[i & 1])
    v.wait_outputs(0)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    f0.record(stream)
    for i in range(args.steps):
        v.render_frame(gb)
        v.read_output_async(outs[i & 1])
        v.wait_outputs(1)  # at most one readback in flight: step i-1's result is on the host now
    v.wait_outputs(0)
    v.join_streams()
    f1.record(stream)
    barrier()
    w1 = time.perf_counter()
    t_end = time.time()
    ms_e2e = max_over_ranks(max(f0.elapsed_time(f1), (w1 - w0) * 1e3))
    if rank == 0:
        sampler.stop()
    clocks = sampler.summary(t_begin, t_end) if rank == 0 else None
    v.close()

    # ---- per-pass GPU time (CUDA events around each pass), outside the timed regions ----
    vt = make_viewer(True)
    for _ in range(3):
        vt.render_frame(gb)
    vt.sync()
    vt.collect_timings()
    n_t = min(args.steps, 50)
    for _ in range(n_t):
        vt.render_frame(None)
    vt.sync()
    timings = {k: ms / max(c, 1) for k, (ms, c) in vt.collect_timings().items()}
    # bloom-compute: the fused threshold + d0 kernel (which also stores the band to the peers when row-sharded) and one
    # cooperative launch for d1, d2, d3, luminance, u2, u1, u0 (which also waits for the peers' bands)
    n_launch = {"clustering-bindless": 4, "lighting": 1, "bloom-compute": 2, "tonemap": 1, "bloom-disabled": 0, "taa-resolve": 1, "fxaa": 1,
                "gbuffer": 0, "mv": 0}
    launches_per_frame = sum(n_launch.get(p, 0) for p in vt.pass_names())
    vt.close()

    peak, peak_kind = measured_peak()
    light_ms = timings.get("lighting")
    light_rows = (in_rows[1] - in_rows[0])
    achieved = (light_rows * w * LIGHTING_BYTES_PER_PIXEL) / (light_ms * 1e-3) / 1e9 if light_ms else None
    fps = args.steps / (ms_resident * 1e-3)
    line = {
        "metric": "frames/sec", "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_resident / args.steps, "higher_is_better": True, "scaling": "strong" if world > 1 else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config, "clocks": clocks,
        "e2e": {"value": args.steps / (ms_e2e * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches_per_frame * args.steps,
        "hbm_gbs_whole_frame": total_b / (ms_resident / args.steps * 1e-3) / 1e9 / 1.0,
        "roofline": {"kernel": "deferred_lighting_persistent_kernel (pass 'lighting')", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": (achieved / peak) if achieved else None, "traffic": ncu_traffic(), "peak_source": f"of {peak_kind}",
                     "bytes_per_pixel": LIGHTING_BYTES_PER_PIXEL, "note": "ALU-bound at this light density: see DESIGN.md"},
        "pass_ms": {k: round(val, 4) for k, val in timings.items()},
        "host_record_ms_per_step": round(host_ms / args.steps, 4),
        "ms_per_step_windows": frame_stats,
    }
    # ---- the other single-GPU configurations of BASELINE.json (c2: 1080p / 1024 lights, c5: 4K TAA +
    # FXAA with history): device-resident frames/s over one window of >= 0.25 s plus per-pass times,
    # so that every configuration has a driver-run number.  Not part of `value`.
    if rank == 0 and world == 1 and args.workload == "c3":
        line["other_configs"] = {}
        for name in ("c2", "c5"):
            try:
                ow, oh, on, oaa, odesc = WORKLOADS[name]
                osc = scene if (ow, oh) == (w, h) else synth.make_scene(ow, oh)
                oli = lights if on == n_lights and (ow, oh) == (w, h) else synth.make_lights(on, aspect=ow / oh)
                ov = viewer.Viewer(ow, oh, post_aa={"none": viewer.AA_NONE, "taa+fxaa": viewer.AA_TAA_HIGH_PLUS_FXAA}[oaa], cuda_device=local_rank,
                                   timestamps=True, stream=stream.cuda_stream)
                ov.set_camera(osc.projection, osc.view)
                ov.set_directional(osc.dir_color, osc.dir_direction)
                ov.set_lights(oli)
                ov.bake()
                arrays = [np.ascontiguousarray(a) for a in (osc.albedo, osc.normal, osc.pbr, osc.depth, osc.emissive)]
                if oaa == "taa+fxaa":
                    # SURVEY.md section 8d: zero motion vectors on 90 % of the pixels, <= 2 px on the rest
                    orng = np.random.default_rng(5)
                    omv = np.zeros((oh, ow, 2), np.float16)
                    om = orng.random((oh, ow)) < 0.1
                    omv[om] = (orng.uniform(-2, 2, size=(int(om.sum()), 2)) / np.array([ow, oh])).astype(np.float16)
                    arrays.append(np.ascontiguousarray(omv).view(np.uint32)[..., 0])
                ogb = viewer.Viewer.host_gbuffer(*arrays)
                ov.render_frame(ogb)
                for _ in range(5):
                    ov.render_frame(None)
                ov.sync()
                ov.collect_timings()
                frames, total_ms = 0, 0.0
                while total_ms < 250.0 and frames < 4000:
                    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    torch.cuda.synchronize()
                    a0.record(stream)
                    for _ in range(50):
                        ov.render_frame(None)
                    ov.join_streams()
                    a1.record(stream)
                    torch.cuda.synchronize()
                    total_ms += a0.elapsed_time(a1)
                    frames += 50
                tm = {k: round(ms / max(c, 1), 4) for k, (ms, c) in ov.collect_timings().items()}
                ov.close()
                _, _, ob = algorithmic_bytes(ow, oh, oaa)
                ofps = frames / (total_ms * 1e-3)
                line["other_configs"][name] = {"workload": odesc, "value": ofps, "unit": "frames/s", "frames_timed": frames, "pass_ms": tm,
                                               "algorithmic_mb_per_frame": round(ob / 1e6, 2),
                                               "hbm_gbs_whole_frame": ob * ofps / 1e9, "roofline_frac_whole_frame": ob * ofps / 1e9 / peak}
            except Exception as exc:  # informational: never let it cost the headline run
                line["other_configs"][name] = {"error": str(exc)[:200]}
    line["roofline_whole_frame"] = {"bound": "hbm", "achieved": total_b * fps / 1e9, "peak": peak, "unit": "GB/s", "frac": total_b * fps / 1e9 / peak}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sec, cores, sample = oracle_frame_time(w, h, n_lights, aa, steps=3, warmup=1, budget_s=25.0, bloom=bloom)
        line["cpu_baseline"] = {"value": 1.0 / sec, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
