"""TAA in row-sharded frames on CPU: the row plan with a TAA resolve (grbh_shard_plan_ex), a `gloo` run of the
history exchange over several frames with the oracle standing in for the kernels, and the argument checks of
grb_taa_resolve_to_peers (no CUDA call is reached).

A pixel reads last frame's history at its reprojected position, which can be anywhere in the frame, so every rank
holds the whole history: each rank resolves only plan["taa"] from inputs that are zero outside plan["lighting"], and
the next frame's history is assembled from every rank's `own` band.  The camera moves every frame and some pixels
carry motion vectors of 40+ rows, so history reads cross band borders."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

W, H = 320, 256  # 4 bands of 64 rows
FRAMES = 5
QUALITY = 2  # TAA_HIGH: the widest footprint (Catmull-Rom history, 3x3 neighbourhood)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _frame_inputs(frame):
    """HDR-main, depth, motion vectors and the clip -> previous-UV reprojection of one frame (moving camera)."""
    from tests import common

    rng = np.random.default_rng(1000 + frame)
    hdr = common.random_hdr(rng, W, H, scale=2.0)
    depth = rng.uniform(0.0005, 0.03, size=(H, W)).astype(np.float32)
    depth[rng.random((H, W)) < 0.1] = 0.0
    mv = np.zeros((H, W, 2), np.float16)
    small = rng.random((H, W)) < 0.1
    mv[small] = (rng.uniform(-2.0, 2.0, size=(int(small.sum()), 2)) / np.array([W, H])).astype(np.float16)
    # fast movers: 40 - 90 rows up or down, reading history one or two bands away
    fast = rng.random((H, W)) < 0.05
    rows = rng.uniform(40.0, 90.0, size=int(fast.sum())) * rng.choice([-1.0, 1.0], size=int(fast.sum()))
    mv[fast, 0] = (rng.uniform(-8.0, 8.0, size=int(fast.sum())) / W).astype(np.float16)
    mv[fast, 1] = (rows / H).astype(np.float16)
    # the camera pans 7 columns and 11 rows per frame (pixels with a zero MV reproject through this matrix)
    reproj = np.array([[0.5, 0, 0, 0], [0, 0.5, 0, 0], [0.3, -0.2, 1, 0],
                       [0.5 + (0.4 + 7.0 * frame) / W, 0.5 - (0.3 + 11.0 * frame) / H, 0, 1]], np.float32)
    return hdr, depth, mv.view(np.uint16), reproj


def _post_chain(oracle, resolved, plan, fxaa, gather_fn, reduce_fn, world_plans):
    """The post chain of tests/test_sharding_gloo.py on a rank's band of the resolved image."""
    lum0 = np.array([0.2, 2 ** 0.2, 2 ** -0.2], np.float32)
    sz = oracle.pyramid_sizes(W, H)

    def keep(img, rows):
        out = np.zeros_like(img)
        out[rows[0]:rows[1]] = img[rows[0]:rows[1]]
        return out

    t = keep(oracle.bloom_threshold(resolved, lum0, sz[0]), plan["threshold"])
    d0 = keep(oracle.bloom_downsample(t, sz[1]), plan["downsample0"])
    d0 = gather_fn(d0, [p["downsample0"] for p in world_plans])
    d1 = oracle.bloom_downsample(d0, sz[2])
    d2 = oracle.bloom_downsample(d1, sz[3])
    d3 = oracle.bloom_downsample(d2, sz[4])
    _, grid = oracle.luminance(d3, lum0, 0.0115, want_grid=True)
    reduce_fn(keep(grid, plan["lum_grid"]))
    lum = oracle.luminance(d3, lum0, float(np.float32(1.0 - 0.5 ** (1 / 60))))
    u2 = oracle.bloom_upsample(d3, sz[3])
    u1 = oracle.bloom_upsample(u2, sz[2])
    u0 = keep(oracle.bloom_upsample(u1, sz[1]), plan["upsample0"])
    ldr = keep(oracle.tonemap(resolved, u0, lum, 1.0, rows=plan["tonemap"]), plan["tonemap"])
    return oracle.fxaa(ldr, True, rows=plan["fxaa"]) if fxaa else ldr


def _reference_frames(oracle, fxaa):
    """Unsharded: TAA resolve + post chain of every frame, history fed back."""
    lum0 = np.array([0.2, 2 ** 0.2, 2 ** -0.2], np.float32)
    history, frames, resolved_frames = None, [], []
    for f in range(FRAMES):
        hdr, depth, mv, reproj = _frame_inputs(f)
        resolved, history = oracle.taa_resolve(hdr, depth, mv, history, reproj, QUALITY)
        ldr = oracle.hdr_chain(resolved, lum0, None).ldr
        frames.append(oracle.fxaa(ldr, True) if fxaa else ldr)
        resolved_frames.append(resolved)
    return frames, resolved_frames


def _sharded_frames(oracle, rank, world, fxaa, gather_fn, reduce_fn):
    """One rank's frames.  Everything outside the planned rows is left ZERO on purpose."""
    from granite_b200 import viewer

    bands = viewer.band_partition(H, world)
    world_plans = [viewer.shard_plan(W, H, bands, r, fxaa, taa=True) for r in range(world)]
    plan = world_plans[rank]
    lo, hi = plan["lighting"]
    history, outs, resolved_rows = None, [], []
    for f in range(FRAMES):
        hdr, depth, mv, reproj = _frame_inputs(f)
        for a in (hdr, depth, mv):
            a[:lo] = 0
            a[hi:] = 0
        resolved, band_history = oracle.taa_resolve(hdr, depth, mv, history, reproj, QUALITY, rows=plan["taa"])
        resolved[:plan["taa"][0]] = 0
        resolved[plan["taa"][1]:] = 0
        # the history exchange: every rank contributes its own band; rows it resolved beyond it are not sent
        mine = np.zeros_like(band_history)
        mine[plan["own"][0]:plan["own"][1]] = band_history[plan["own"][0]:plan["own"][1]]
        history = gather_fn(mine, [p["own"] for p in world_plans])
        outs.append(_post_chain(oracle, resolved, plan, fxaa, gather_fn, reduce_fn, world_plans))
        resolved_rows.append(resolved[plan["taa"][0]:plan["taa"][1]].copy())
    return plan, outs, resolved_rows


def _worker(rank, world, port, fxaa, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from oracle import pyoracle as oracle

        def gather(img, rows_per_rank):
            t = torch.from_numpy(np.ascontiguousarray(img).view(np.uint8).copy())  # gloo has no 16-bit integer types
            for r, (a, b) in enumerate(rows_per_rank):  # one broadcast per band, like the NCCL group
                part = t[a:b].contiguous()
                dist.broadcast(part, r)
                t[a:b] = part
            return t.numpy().view(np.uint16).reshape(img.shape)

        def reduce(grid):
            t = torch.from_numpy(grid.copy())
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            return t.numpy()

        plan, outs, resolved_rows = _sharded_frames(oracle, rank, world, fxaa, gather, reduce)
        a, b = plan["own"]
        q.put((rank, plan["own"], [o[a:b].copy() for o in outs], plan["taa"], resolved_rows))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,fxaa", [(2, False), (4, False), (4, True)])
def test_gloo_taa_frames_equal_single_rank(oracle, world, fxaa):
    expect, expect_resolved = _reference_frames(oracle, fxaa)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, fxaa, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    covered = 0
    for rank, (a, b), frames, (ta, tb), resolved in sorted(got, key=lambda g: g[0]):
        for f, rows in enumerate(frames):
            assert np.array_equal(rows, expect[f][a:b]), f"frame {f}: rank {rank} rows [{a},{b}) differ from the unsharded frame"
            # every resolved row a rank computes (not only those its band's output happens to depend on) is exact
            assert np.array_equal(resolved[f], expect_resolved[f][ta:tb]), f"frame {f}: rank {rank} resolved rows [{ta},{tb}) differ"
        covered += b - a
    assert covered == H


def test_inputs_cross_band_borders():
    """The fixture does what the docstring claims: history reads land 40+ rows (more than a band's halo) away."""
    _, _, mv, _ = _frame_inputs(1)
    dy = np.abs(mv.view(np.float16)[..., 1].astype(np.float32)) * H
    assert (dy >= 40.0).sum() > 100


def test_taa_plan_invariants():
    from granite_b200 import viewer

    for w, h, world in [(3840, 2160, 2), (3840, 2160, 4), (3840, 2160, 8), (1920, 1080, 8), (384, 384, 6), (W, H, 4)]:
        bands = viewer.band_partition(h, world)
        for fxaa in (False, True):
            old = [viewer.shard_plan(w, h, bands, r, fxaa) for r in range(world)]
            new = [viewer.shard_plan(w, h, bands, r, fxaa, taa=True) for r in range(world)]
            assert old[0]["own"][0] == 0 and old[-1]["own"][1] == h
            assert all(a["own"][1] == b["own"][0] for a, b in zip(new, new[1:])), "own bands tile the frame"
            for o, n in zip(old, new):
                # the resolved rows are the old lighting rows (what the threshold and the tonemap read) ...
                assert n["taa"][0] <= o["lighting"][0] and o["lighting"][1] <= n["taa"][1]
                assert n["taa"] == o["lighting"]
                # ... and lighting covers them +- 1 row, clamped
                assert n["lighting"] == (max(n["taa"][0] - 1, 0), min(n["taa"][1] + 1, h))
                assert n["own"][0] >= n["taa"][0] and n["own"][1] <= n["taa"][1]
                # every other stage is unchanged
                assert {k: v for k, v in n.items() if k not in ("taa", "lighting")} == {k: v for k, v in o.items() if k != "lighting"}
        # unsharded: everything is the whole frame
        whole = viewer.shard_plan(w, h, [], 0, True, taa=True)
        assert whole["taa"] == whole["lighting"] == (0, h)


def test_plan_without_taa_is_unchanged():
    """shard_plan(..., taa=False) is the eight-field plan of grbh_shard_plan."""
    from granite_b200 import viewer

    bands = viewer.band_partition(2160, 4)
    p = viewer.shard_plan(3840, 2160, bands, 1, True)
    assert set(p) == set(viewer.PLAN_FIELDS) and p == viewer.shard_plan(3840, 2160, bands, 1, True, taa=False)


# ----------------------------------------------------------------------------- argument checks (no CUDA call reached)
OK, ERR_ARG, ERR_FORMAT = 0, -1, -2


@pytest.fixture(scope="module")
def lib():
    from granite_b200 import build, capi

    build.build_all()
    L = C.CDLL(capi.LIB_PATH)
    L.grb_last_error_string.restype = C.c_char_p
    IMG = C.POINTER(capi.GrbImage)
    P, I = C.c_void_p, C.c_int32
    L.grb_taa_resolve_to_peers.argtypes = [IMG, IMG, IMG, IMG, P, I, IMG, IMG, P, P, I, I, C.c_uint32, P, capi.GrbRows, capi.GrbRows, P]
    return L


def _msg(lib):
    return (lib.grb_last_error_string() or b"").decode()


def test_taa_resolve_to_peers_argument_checks(lib):
    from granite_b200 import capi

    w, h = 16, 12
    keep = []

    def img(fmt, ww=w, hh=h):
        a = np.zeros((hh, ww * capi.TEXEL_BYTES[fmt]), np.uint8)
        keep.append(a)
        return capi.GrbImage(a.ctypes.data, ww, hh, ww * capi.TEXEL_BYTES[fmt], fmt)

    hdr, depth, mv = img(capi.FORMAT_B10G11R11_UFLOAT), img(capi.FORMAT_D32_SFLOAT), img(capi.FORMAT_R16G16_SFLOAT)
    hist, oc = img(capi.FORMAT_R16G16B16A16_SFLOAT), img(capi.FORMAT_B10G11R11_UFLOAT)
    layout = capi.GrbImage(None, w, h, w * 8, capi.FORMAT_R16G16B16A16_SFLOAT)
    slots = [img(capi.FORMAT_R16G16B16A16_SFLOAT) for _ in range(2)]
    flags = np.zeros((2, 16), np.uint32)
    counter = np.zeros(1, np.uint32)
    reproj = (C.c_float * 16)()
    images = (C.c_void_p * 8)(*[s.data for s in slots])
    flag_ptrs = (C.c_void_p * 8)(*[flags[r].ctypes.data for r in range(2)])
    cnt = counter.ctypes.data_as(C.c_void_p)
    R = capi.GrbRows

    def call(hdr_=hdr, history=hist, quality=2, out_layout=layout, imgs=images, fl=flag_ptrs, count=2, index=0, scratch=cnt,
             rows=R(0, 8), own=R(0, 6), oc_=oc):
        return lib.grb_taa_resolve_to_peers(C.byref(hdr_), C.byref(depth), C.byref(mv), C.byref(history) if history is not None else None,
                                            reproj, quality, C.byref(oc_), C.byref(out_layout) if out_layout is not None else None,
                                            imgs, fl, count, index, 1, scratch, rows, own, None)

    assert call(count=0) == ERR_ARG and "peer_count" in _msg(lib)
    assert call(count=9) == ERR_ARG
    assert call(index=2) == ERR_ARG and "flag_index" in _msg(lib)
    assert call(index=-1) == ERR_ARG
    assert call(imgs=None) == ERR_ARG
    assert call(fl=None) == ERR_ARG
    assert call(scratch=None) == ERR_ARG
    assert call(out_layout=None) == ERR_ARG
    assert call(imgs=(C.c_void_p * 8)(slots[0].data, None)) == ERR_ARG and "null peer pointer" in _msg(lib)
    assert call(fl=(C.c_void_p * 8)(flag_ptrs[0], None)) == ERR_ARG and "null peer pointer" in _msg(lib)
    # formats and sizes follow grb_taa_resolve
    assert call(hdr_=img(capi.FORMAT_R8G8B8A8_UNORM)) == ERR_FORMAT and "grb_taa_resolve_to_peers" in _msg(lib)
    assert call(out_layout=capi.GrbImage(None, w + 1, h, (w + 1) * 8, capi.FORMAT_R16G16B16A16_SFLOAT)) == ERR_FORMAT
    assert call(oc_=img(capi.FORMAT_B10G11R11_UFLOAT, w, h + 1)) == ERR_FORMAT
    assert call(quality=3) == ERR_ARG and "quality" in _msg(lib)
    # the history read must not be a slot this call writes
    assert call(history=slots[1]) == ERR_ARG and "history" in _msg(lib)
    # own_rows inside rows, both non-empty
    assert call(rows=R(2, 8), own=R(0, 6)) == ERR_ARG and "own_rows" in _msg(lib)
    assert call(rows=R(0, 8), own=R(4, 10)) == ERR_ARG
    assert call(rows=R(5, 5), own=R(5, 5)) == ERR_ARG
    assert call(rows=R(0, 8), own=R(3, 3)) == ERR_ARG
    assert not flags.any() and not counter.any(), "a refused call must not touch the flags"
