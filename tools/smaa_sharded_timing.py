#!/usr/bin/env python3
"""SMAA in row-sharded frames: resident frames/s, the per-pass times of smaa-edge, smaa-weights and smaa-blend and the
SMAA edge bytes each rank stores to its peers per frame, for both exchange paths of the edges (peer-memory stores from
the edge kernel, NCCL broadcasts), at 3840x2160 with 4096 lights and SMAA Ultra.

    torchrun --nproc-per-node N tools/smaa_sharded_timing.py [--out profiles/smaa_sharded_timing.jsonl] [--frames-ms 500]

Run it once per rank count (1, 2, 4, 8).  Rank 0 prints one JSON line per exchange path (and appends it to --out),
with the card's name and power limit read in the same run.  Frames/s: the G-buffer stays resident (uploaded once),
CUDA events around batches of 25 frames on the viewer's stream until every rank has timed >= --frames-ms; the slowest
rank's time counts.  Pass times: a second viewer with per-pass timestamps (max over ranks of the per-rank mean)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

W, H, N_LIGHTS = 3840, 2160, 4096


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                       capture_output=True, text=True)
    name, _, power = q.stdout.strip().partition(",")
    return {"name": name.strip() or torch.cuda.get_device_name(), "power_limit": power.strip() or "unknown"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--frames-ms", type=float, default=500.0)
    args = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from granite_b200 import synth, viewer

    scene = synth.make_scene(W, H)
    lights = synth.make_lights(N_LIGHTS, aspect=W / H)
    arrays = [np.ascontiguousarray(a) for a in (scene.albedo, scene.normal, scene.pbr, scene.depth, scene.emissive)]
    gb = viewer.Viewer.host_gbuffer(*arrays)
    luts = np.load(os.path.join(ROOT, "tests", "golden", "refsmaa_160x96.npz"))
    bands = viewer.band_partition(H, world, align=8)
    stream = torch.cuda.Stream()

    def make(timestamps):
        v = viewer.Viewer(W, H, post_aa=viewer.AA_SMAA_ULTRA, cuda_device=local, timestamps=timestamps, stream=stream.cuda_stream)
        v.set_camera(scene.projection, scene.view)
        v.set_directional(scene.dir_color, scene.dir_direction)
        v.set_lights(lights)
        v.set_smaa_lookup_textures(luts["area"], luts["search"])
        if world > 1:
            uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
            if rank == 0:
                uid.copy_(torch.frombuffer(bytearray(viewer.nccl_unique_id()), dtype=torch.uint8))
            dist.broadcast(uid, 0)
            v.init_collectives(uid.cpu().numpy().tobytes(), rank, world)
            v.set_row_shards(bands, rank)
        v.bake()
        v.render_frame(gb)
        for _ in range(5):
            v.render_frame(None)
        v.sync()
        return v

    def max_over_ranks(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    info = card()
    for exchange in (("peer", "nccl") if world > 1 else ("none",)):
        os.environ["GRB_SHARD_EXCHANGE"] = exchange  # read when the viewer's exchange buffers are created
        v = make(False)
        frames, total_ms = 0, 0.0
        while True:
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            dist.barrier()
            a0.record(stream)
            for _ in range(25):
                v.render_frame(None)
            v.join_streams()
            a1.record(stream)
            torch.cuda.synchronize()
            total_ms += a0.elapsed_time(a1)
            frames += 25
            if max_over_ranks(-total_ms) > -args.frames_ms:  # the fastest rank is not done yet: every rank continues
                continue
            break
        ms = max_over_ranks(total_ms)
        v.close()
        vt = make(True)
        vt.collect_timings()
        for _ in range(30):
            vt.render_frame(None)
        vt.sync()
        tm = {k: ms_ / max(c, 1) for k, (ms_, c) in vt.collect_timings().items()}
        vt.close()
        pass_ms = {p: max_over_ranks(next((t for k, t in tm.items() if k.endswith(p)), float("nan"))) for p in ("smaa-edge", "smaa-weights", "smaa-blend")}
        # edge rows (R8G8: 2 bytes a texel) the busiest rank stores into other ranks' slots: own_q and r's window
        plans = [viewer.shard_plan(W, H, bands, r, smaa=3) for r in range(world)]
        to_peers = [sum(max(0, min(plans[q]["own"][1], plans[r]["smaa_edges"][1]) - max(plans[q]["own"][0], plans[r]["smaa_edges"][0]))
                        for r in range(world) if r != q) * W * 2 for q in range(world)]
        line = {
            "size": [W, H], "lights": N_LIGHTS, "post_aa": "SMAA_ULTRA", "ranks": world, "exchange": exchange,
            "bands": [list(b) for b in bands], "frames_timed": frames, "frames_per_s": frames / (ms * 1e-3),
            "smaa_edge_ms": pass_ms["smaa-edge"], "smaa_weights_ms": pass_ms["smaa-weights"], "smaa_blend_ms": pass_ms["smaa-blend"],
            "edge_bytes_to_peers_per_rank": max(to_peers) if exchange != "none" else 0,
            "card": info["name"], "power_limit": info["power_limit"], "torch": torch.__version__,
        }
        if rank == 0:
            print(json.dumps(line), flush=True)
            if args.out:
                with open(args.out, "a") as f:
                    f.write(json.dumps(line) + "\n")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
