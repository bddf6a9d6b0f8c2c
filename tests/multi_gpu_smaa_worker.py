"""torchrun worker for tests/test_multi_gpu_smaa.py: renders the same SMAA frames (moving camera) row-sharded over all
ranks and, on rank 0, unsharded; every assembled sharded frame and the average luminance must equal the single-GPU
viewer's bit for bit.  The exchange path of the SMAA edges follows GRB_SHARD_EXCHANGE."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FRAMES = 6


def main():
    w, h, n_lights, post_aa = int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4])
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from granite_b200 import synth, viewer

    scene = synth.make_scene(w, h)
    lights = synth.make_lights(n_lights, spot_fraction=0.25, aspect=w / h)
    keep = [np.ascontiguousarray(a) for a in (scene.albedo, scene.normal, scene.pbr, scene.depth, scene.emissive)]
    luts = np.load(os.path.join(ROOT, "tests", "golden", "refsmaa_160x96.npz"))
    gb = viewer.Viewer.host_gbuffer(*keep)
    # the camera pans and dollies every frame
    views = [synth.look_at_view((0.15 * i, 0.1 * i, 8.0 - 0.2 * i), (0.1 * i, 0.0, 0.0)) for i in range(FRAMES)]

    def make(sharded):
        v = viewer.Viewer(w, h, post_aa=post_aa, cuda_device=local)
        v.set_camera(scene.projection, views[0])
        v.set_directional(scene.dir_color, scene.dir_direction)
        v.set_lights(lights)
        v.set_smaa_lookup_textures(luts["area"], luts["search"])
        if sharded:
            uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
            if rank == 0:
                uid.copy_(torch.frombuffer(bytearray(viewer.nccl_unique_id()), dtype=torch.uint8))
            dist.broadcast(uid, 0)
            v.init_collectives(uid.cpu().numpy().tobytes(), rank, world)
            v.set_row_shards(viewer.band_partition(h, world), rank)
        v.bake()
        return v

    def frame(v, i):
        v.set_camera(scene.projection, views[i])
        v.render_frame(gb)

    vs = make(True)
    frames = []
    for i in range(FRAMES):
        frame(vs, i)
        out = np.zeros((h, w), np.uint32)
        vs.read_output(out)
        full = torch.from_numpy(out.view(np.int32)).cuda()
        dist.all_reduce(full, op=dist.ReduceOp.SUM)  # bands are disjoint, zeros elsewhere
        frames.append(full.cpu().numpy().view(np.uint32))
    lum_sharded = vs.download_buffer("average-luminance", np.float32, 3).copy()
    vs.close()
    ok = True
    if rank == 0:
        v1 = make(False)
        for i in range(FRAMES):
            frame(v1, i)
            ref = np.zeros((h, w), np.uint32)
            v1.read_output(ref)
            same = np.array_equal(ref, frames[i])
            print(f"frame {i}: sharded over {world} ranks == single GPU: {same} ({int((ref != frames[i]).sum())} pixels differ)", flush=True)
            ok &= same
        # the frames must actually change: a moving camera
        ok &= not np.array_equal(frames[1], frames[FRAMES - 1])
        lum1 = v1.download_buffer("average-luminance", np.float32, 3)
        same = np.array_equal(lum1.view(np.uint32), lum_sharded.view(np.uint32))
        print(f"average luminance identical: {same}", flush=True)
        ok &= same
        v1.close()
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.broadcast(flag, 0)
    dist.destroy_process_group()
    sys.exit(0 if int(flag.item()) == 1 else 1)


if __name__ == "__main__":
    main()
