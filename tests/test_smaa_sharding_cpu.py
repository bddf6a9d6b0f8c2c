"""SMAA in row-sharded frames on CPU: the row plan with SMAA (grbh_shard_plan_smaa), the fp32 rounding its reaches
rest on, the argument checks of grb_smaa_edge_detection_to_peers (no CUDA call is reached), and a `gloo` run of the
edge exchange with the oracle standing in for the kernels.

Each rank detects the edges of its own band only, from a colour image that is valid on plan["tonemap"] and garbage
elsewhere.  Rank q sends edge row y to rank r exactly when y is in own_q and in r's window plan["smaa_edges"]; the
receiving edge image is 255 (an edge everywhere) outside the rows received.  Then every rank computes
plan["smaa_weights"] and blends its own band.  The input has full-height vertical edges, a staircase of 90-row
vertical segments and long diagonals, all crossing band borders, so the searches run their full length."""
import ctypes as C
import os
import socket
import subprocess

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
W, H = 192, 256
MAX_SEARCH_STEPS = (4, 8, 16, 32)
# bands of 64 rows (band_partition) and uneven 8-row-aligned bands, some narrower than the Ultra reach
UNEVEN = {2: [(0, 96), (96, 256)], 3: [(0, 48), (48, 200), (200, 256)], 4: [(0, 40), (40, 136), (136, 184), (184, 256)]}


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _luts():
    f = np.load(os.path.join(GOLDEN, "refsmaa_160x96.npz"))
    return np.ascontiguousarray(f["area"]), np.ascontiguousarray(f["search"])


def _image():
    """smaa_test_image plus edges longer than 2 * 32 rows that cross every band border."""
    from tests.test_oracle_ref_smaa import smaa_test_image

    img = smaa_test_image(W, H, 11).view(np.uint8).reshape(H, W, 4).copy()
    yy, xx = np.mgrid[0:H, 0:W]
    img[(xx >= 8) & (xx < 20), :3] = (240, 240, 240)                      # full-height vertical edges
    stair = 30 + 3 * (yy // 90)                                              # vertical segments of 90 rows + jogs
    img[(xx >= stair) & (xx < stair + 10), :3] = (20, 20, 230)
    img[(np.abs(xx - 0.5 * yy - 60) < 2.0), :3] = (250, 40, 40)             # steep diagonal (2 rows per column)
    img[(np.abs(xx - yy + 20) < 1.5) & (xx > 100), :3] = (10, 10, 10)        # 45-degree diagonal
    return np.ascontiguousarray(img).view(np.uint32).reshape(H, W)


def _emu_library(tmp_dir):
    """The SMAA kernels' source compiled for the CPU (the blend with a UNORM target, which the oracle lacks)."""
    out = os.path.join(tmp_dir, "libemu_smaa.so")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    cmd = ["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-w", "-x", "c++", f"-I{cuda}/include",
           os.path.join(ROOT, "tests", "cpp", "emulate_smaa.cpp"), "-o", out]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return out


def _blend(oracle, emu, color, weights, srgb, rows):
    if srgb:
        return oracle.smaa_blend(color, weights, rows=rows)
    h, w = color.shape
    out = np.zeros((h, w), np.uint32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    emu.emu_smaa_blend(p(np.ascontiguousarray(color)), p(np.ascontiguousarray(weights)), w, h, 0, p(out), rows[0], rows[1])
    return out


def _reference(oracle, emu, img, q, srgb):
    area, search = _luts()
    e = oracle.smaa_edge(img, q)
    wg = oracle.smaa_weights(e, area, search, q)
    return e, wg, _blend(oracle, emu, img, wg, srgb, (0, H))


def _rank_frame(oracle, emu, img, q, srgb, plan, slot):
    """Weights and blend of one rank from its received edge slot (255 outside the rows received)."""
    area, search = _luts()
    rng = np.random.default_rng(q)
    wg = oracle.smaa_weights(slot, area, search, q, rows=plan["smaa_weights"])
    a, b = plan["smaa_weights"]
    wg[:a] = rng.integers(0, 2 ** 32, size=(a, W), dtype=np.uint32)           # garbage outside the computed rows
    wg[b:] = rng.integers(0, 2 ** 32, size=(H - b, W), dtype=np.uint32)
    return wg, _blend(oracle, emu, img, wg, srgb, plan["own"])


def _garbage_outside(img, rows, seed):
    out = np.random.default_rng(seed).integers(0, 2 ** 32, size=img.shape, dtype=np.uint32)
    out[rows[0]:rows[1]] = img[rows[0]:rows[1]]
    return out


def _worker(rank, world, bands, port, emu_path, q_out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from granite_b200 import viewer
        from oracle import pyoracle as oracle

        emu = C.CDLL(emu_path)
        img = _image()
        results = []
        for q in range(4):
            plans = [viewer.shard_plan(W, H, bands, r, smaa=q) for r in range(world)]
            plan = plans[rank]
            color = _garbage_outside(img, plan["tonemap"], 100 + rank)
            edges = oracle.smaa_edge(color, q, rows=plan["own"])
            slot = np.full((H, W, 2), 255, np.uint8)
            # the exchange: rank q stores row y into rank r exactly when y is in own_q and in r's window
            reqs, incoming = [], []
            for src in range(world):
                for dst in range(world):
                    a = max(plans[src]["own"][0], plans[dst]["smaa_edges"][0])
                    b = min(plans[src]["own"][1], plans[dst]["smaa_edges"][1])
                    if a >= b:
                        continue
                    if src == rank and dst == rank:
                        slot[a:b] = edges[a:b]
                    elif src == rank:
                        reqs.append(dist.isend(torch.from_numpy(np.ascontiguousarray(edges[a:b])), dst, tag=src))
                    elif dst == rank:
                        buf = torch.zeros((b - a, W, 2), dtype=torch.uint8)
                        reqs.append(dist.irecv(buf, src, tag=src))
                        incoming.append((a, b, buf))
            for r in reqs:
                r.wait()
            for a, b, buf in incoming:
                slot[a:b] = buf.numpy()
            for srgb in (True, False):
                wg, out = _rank_frame(oracle, emu, color, q, srgb, plan, slot)
                a, b = plan["own"]
                wa, wb = plan["smaa_weights"]
                ea, eb = plan["smaa_edges"]
                results.append((q, srgb, (a, b), out[a:b].copy(), (wa, wb), wg[wa:wb].copy(), (ea, eb), slot[ea:eb].copy()))
        q_out.put((rank, results))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,layout", [(2, "64"), (3, "uneven"), (4, "64"), (4, "uneven"), (2, "uneven")])
def test_gloo_smaa_bands_equal_unsharded(oracle, tmp_path, world, layout):
    from granite_b200 import viewer

    emu_path = _emu_library(str(tmp_path))
    emu = C.CDLL(emu_path)
    bands = viewer.band_partition(H, world) if layout == "64" else UNEVEN[world]
    img = _image()
    ref = {(q, s): _reference(oracle, emu, img, q, s) for q in range(4) for s in (True, False)}
    ctx = mp.get_context("spawn")
    q_out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, bands, port, emu_path, q_out)) for r in range(world)]
    for p in procs:
        p.start()
    got = [q_out.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, results in got:
        for q, srgb, (a, b), out, (wa, wb), wg, (ea, eb), slot in results:
            e_ref, w_ref, o_ref = ref[(q, srgb)]
            what = f"rank {rank}, quality {q}, {'sRGB' if srgb else 'UNORM'}"
            assert np.array_equal(slot, e_ref[ea:eb]), f"{what}: edge window [{ea},{eb}) differs from the unsharded edges"
            assert np.array_equal(wg, w_ref[wa:wb]), f"{what}: weights [{wa},{wb}) differ"
            assert np.array_equal(out, o_ref[a:b]), f"{what}: blended rows [{a},{b}) differ"


def test_input_runs_full_length_searches(oracle):
    """The fixture does what the docstring claims: at Ultra, vertical edges run longer than a search (2 * 32 rows)."""
    e = oracle.smaa_edge(_image(), 3)
    left = e[..., 0] > 0
    run = np.zeros(W, np.int64)
    best = np.zeros(W, np.int64)
    for y in range(H):
        run = np.where(left[y], run + 1, 0)
        best = np.maximum(best, run)
    assert (best > 2 * 32 + 4).sum() >= 2


def _reads_library(tmp_dir):
    """The weights kernel's source compiled for the CPU with every texel load recorded (tests/cpp/emulate_smaa_reads.cpp)."""
    out = os.path.join(tmp_dir, "libemu_smaa_reads.so")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    cmd = ["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-w", "-x", "c++", f"-I{cuda}/include",
           os.path.join(ROOT, "tests", "cpp", "emulate_smaa_reads.cpp"), "-o", out]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return C.CDLL(out)


def _long_vertical_edges(h, w, seed, p):
    """Every texel a vertical edge, crossing edges with probability p: the vertical searches run their full length and
    end on every pattern of the last sample."""
    e = np.zeros((h, w, 2), np.uint8)
    e[..., 0] = 255
    e[..., 1] = np.where(np.random.default_rng(seed).random((h, w)) < p, 255, 0)
    return e


def test_edge_window_is_the_read_reach(oracle, tmp_path):
    """The rows of the edge image the weights pass of row y reads (every texel load of the kernel source recorded) lie
    in [y - R_up, y + R_down), and the reaches are attained: R_down = 2S + 4 at every quality, R_up = 2S + 2 at Ultra
    (at the lower presets the inputs here reach 2S + 1 above).  So the window can be neither a row smaller nor needs
    to be larger, on these inputs and heights that are not powers of two (where fp32 coordinates round)."""
    from granite_b200 import viewer

    lib = _reads_library(str(tmp_path))
    area, search = _luts()
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    for q in range(4):
        s = MAX_SEARCH_STEPS[q]
        plan = viewer.shard_plan(W, 2160, [(0, 1080), (1080, 2160)], 0, smaa=q)
        assert plan["smaa_edges"][1] - plan["smaa_weights"][1] == 2 * s + 4  # R_down of the plan
        r_up, r_down = 2 * s + 2, 2 * s + 4
        most_up = most_down = 0
        inputs = [(h, _long_vertical_edges(h, 64, h + q, pr)) for h in (777, 1080, 2160) for pr in (1 / 40, 1 / 20)]
        inputs.append((H, np.ascontiguousarray(oracle.smaa_edge(_image(), q))))
        for h, e in inputs:
            w = e.shape[1]
            y0, y1 = 80, h - 80
            lo = np.zeros((h, w), np.int32)
            hi = np.zeros((h, w), np.int32)
            lib.emu_smaa_weight_reads(p(e), w, h, p(area), p(search), q, y0, y1, p(lo), p(hi))
            y = np.arange(y0, y1)[:, None]
            up, down = int((y - lo[y0:y1]).max()), int((hi[y0:y1] - y).max())  # window of row y: [y - R_up, y + 1 + R_down)
            assert up <= r_up and down <= r_down, (q, h, up, down)
            most_up, most_down = max(most_up, up), max(most_down, down)
        assert most_down == r_down, (q, most_down)
        assert most_up == (r_up if q == 3 else r_up - 1), (q, most_up)


def test_band_start_where_the_blend_reads_the_row_above(oracle, tmp_path):
    """At h = 2160 the blend of rows 704 and 1080 reads weights row y - 1 (test_row_taps_can_weight_the_next_row).
    Bands starting there, weights garbage outside plan["smaa_weights"], colour garbage outside plan["tonemap"], edges
    255 outside the rows received: every band equals the unsharded SMAA bit for bit, sRGB and UNORM, and leaving the
    row above the band out of the weights changes some pixel."""
    from granite_b200 import viewer

    emu = C.CDLL(_emu_library(str(tmp_path)))
    h, w = 2160, 512
    bands = [(0, 704), (704, 1080), (1080, 2160)]
    img = np.random.default_rng(3).integers(0, 2 ** 32, size=(h, w), dtype=np.uint32)  # noise: weights everywhere
    area, search = _luts()
    for q in range(4):
        e_ref = oracle.smaa_edge(img, q)
        w_ref = oracle.smaa_weights(e_ref, area, search, q)
        ref = {srgb: _blend(oracle, emu, img, w_ref, srgb, (0, h)) for srgb in (True, False)}
        plans = [viewer.shard_plan(w, h, bands, r, smaa=q) for r in range(3)]
        colors = [_garbage_outside(img, pl["tonemap"], 7 + r) for r, pl in enumerate(plans)]
        edges = [oracle.smaa_edge(c, q, rows=pl["own"]) for c, pl in zip(colors, plans)]
        changed = 0
        for r, pl in enumerate(plans):
            slot = np.full((h, w, 2), 255, np.uint8)
            for src, other in enumerate(plans):
                a, b = max(other["own"][0], pl["smaa_edges"][0]), min(other["own"][1], pl["smaa_edges"][1])
                if a < b:
                    slot[a:b] = edges[src][a:b]
            wa, wb = pl["smaa_weights"]
            assert r == 0 or wa == pl["own"][0] - 1
            wg = oracle.smaa_weights(slot, area, search, q, rows=(wa, wb))
            rng = np.random.default_rng(r)
            wg[:wa] = rng.integers(0, 2 ** 32, size=(wa, w), dtype=np.uint32)
            wg[wb:] = rng.integers(0, 2 ** 32, size=(h - wb, w), dtype=np.uint32)
            a, b = pl["own"]
            for srgb in (True, False):
                out = _blend(oracle, emu, colors[r], wg, srgb, (a, b))
                assert np.array_equal(out[a:b], ref[srgb][a:b]), (q, r, srgb)
            if r:
                short = wg.copy()
                short[a - 1] = rng.integers(0, 2 ** 32, size=w, dtype=np.uint32)
                changed += int((_blend(oracle, emu, colors[r], short, True, (a, a + 1))[a] != ref[True][a]).sum())
        assert changed > 0, q


# ----------------------------------------------------------------------------- the plan
def _fields(p):
    return {k: v for k, v in p.items() if k not in ("smaa_weights", "smaa_edges")}


def _uneven_bands(h, world, seed):
    rng = np.random.default_rng(seed)
    while True:
        cuts = sorted(rng.choice(np.arange(1, h // 8), size=world - 1, replace=False) * 8)
        bands = list(zip([0] + cuts, cuts + [h]))
        if all(b > a for a, b in bands):
            return [(int(a), int(b)) for a, b in bands]


def test_smaa_plan_invariants():
    from granite_b200 import viewer

    cases = []
    for h in (2160, 1080, 768):
        for world in range(1, 9):
            cases.append((h, viewer.band_partition(h, world)))
            if world > 1:
                cases.append((h, _uneven_bands(h, world, h + world)))
    cases.append((256, UNEVEN[4]))
    narrow = 0
    for h, bands in cases:
        world = len(bands)
        for q in range(4):
            s = MAX_SEARCH_STEPS[q]
            plans = [viewer.shard_plan(3840, h, bands, r, smaa=q) for r in range(world)]
            for r, p in enumerate(plans):
                (a, b), (wa, wb), (ea, eb), (ta, tb) = p["own"], p["smaa_weights"], p["smaa_edges"], p["tonemap"]
                if world == 1:
                    assert (wa, wb) == (ea, eb) == (0, h)
                    continue
                narrow += (b - a) < 2 * s + 4
                assert (wa, wb) == (max(a - 1, 0), min(b + 2, h))
                assert (ea, eb) == (max(wa - (2 * s + 2), 0), min(wb + 2 * s + 4, h))
                assert ea <= wa and wb <= eb, "smaa_weights inside smaa_edges"
                assert ta <= max(a - 2, 0) and tb >= min(b + 1, h), "tonemap covers own widened by (2, 1)"
                assert (ta, tb) == (max(a - 3, 0), min(b + 2, h))
                # every row of the window is stored by exactly one rank (own bands tile the frame)
                count = np.zeros(h, np.int64)
                for o in plans:
                    lo, hi = max(o["own"][0], ea), min(o["own"][1], eb)
                    if lo < hi:
                        count[lo:hi] += 1
                assert (count[ea:eb] == 1).all() and not count[:ea].any() and not count[eb:].any()
    assert narrow > 0, "some bands are narrower than the Ultra reach"


def test_plan_without_smaa_is_unchanged():
    """smaa=None is today's plan; smaa=-1 adds the two fields (= own) and changes nothing else."""
    from granite_b200 import viewer

    for bands in (viewer.band_partition(2160, 4), UNEVEN[3]):
        h = bands[-1][1]
        for r in range(len(bands)):
            for fxaa in (False, True):
                for taa in (False, True):
                    old = viewer.shard_plan(3840, h, bands, r, fxaa, taa=taa)
                    off = viewer.shard_plan(3840, h, bands, r, fxaa, taa=taa, smaa=-1)
                    assert _fields(off) == old
                    assert off["smaa_weights"] == off["smaa_edges"] == old["own"]
    p = viewer.shard_plan(3840, 2160, viewer.band_partition(2160, 4), 1, True)
    assert set(p) == set(viewer.PLAN_FIELDS)


# ----------------------------------------------------------------------------- the fp32 rounding the reaches rest on
def _fmaf(a, b, c):
    """fmaf for the operands below: the product and the sum are exact in float64, then one rounding to float32."""
    return np.float32(np.float64(a) * np.float64(b) + np.float64(c))


def test_row_taps_can_weight_the_next_row():
    """A tap that is not at the fragment's own coordinate is a bilinear fetch at the row coordinate
    fp32 ((y+0.5)/h + k/h) * h - 0.5, also when k = 0 and only the column is shifted (the blend's `ax` tap, the edge
    pass's Lleft / Lright / Lleftleft).  For some rows it lands a hair above or below the texel centre, so the row
    beyond gets a nonzero weight: a tap at row offset k reads rows k-1 .. k+1.  The edge pass taps k = -2 .. +1 (the
    tonemap covers own - 3 .. own + 2), the blend taps weights at k = 0 and +1 (the weights cover own - 1 .. own + 2)."""
    reach = {k: [0, 0] for k in (-2, -1, 0, 1)}
    for h in (1080, 2160, 777, 1440):
        my = np.float32(1.0) / np.float32(h)
        y = np.arange(h)
        v = (y.astype(np.float32) + np.float32(0.5)) * my
        for k in reach:
            t = (v + np.float32(k) * my).astype(np.float32)  # fmaf(my, k, v): my * k is exact
            fy = t * np.float32(h) - np.float32(0.5)
            fl = np.floor(fy)
            reach[k][0] = min(reach[k][0], int((fl - y).min()) - k)
            reach[k][1] = max(reach[k][1], int((fl + (fy > fl) - y).max()) - k)
    assert all(r == [-1, 1] for r in reach.values()), reach
    # the rows of a 2160-row frame whose blend reads weights row y - 1 include band starts 704 and 1080
    my = np.float32(1.0) / np.float32(2160)
    fy = ((np.array([704, 1080, 1024], np.float32) + np.float32(0.5)) * my).astype(np.float32) * np.float32(2160) - np.float32(0.5)
    assert list(np.floor(fy).astype(int)) == [703, 1079, 1024]


def test_vertical_search_can_take_one_more_step():
    """The vertical search samples while its fmaf-accumulated coordinate is short of the end: S steps in exact
    arithmetic, S + 1 for some rows of any height.  The plan's reaches (2S + 2 up, 2S + 4 down) count S + 1."""
    for s in MAX_SEARCH_STEPS:
        most = 0
        for h in (1080, 2160, 777):
            my = np.float32(1.0) / np.float32(h)
            for y in range(0, h, 7):
                v = np.float32(np.float32(y + 0.5) * my)
                o1w = _fmaf(my, 1.25, v)
                end = _fmaf(my, 2.0 * s, o1w)
                tv, k = o1w, 0
                while tv < end and k < 2 * s:
                    k += 1
                    tv = _fmaf(2.0, my, tv)
                most = max(most, k)
        assert most == s + 1, (s, most)


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
    L.grb_smaa_edge_detection_to_peers.argtypes = [IMG, I, IMG, P, C.POINTER(capi.GrbRows), P, I, I, C.c_uint32, P, capi.GrbRows, P]
    return L


def _msg(lib):
    return (lib.grb_last_error_string() or b"").decode()


def test_smaa_edge_detection_to_peers_argument_checks(lib):
    from granite_b200 import capi

    w, h = 16, 12
    keep = []

    def img(fmt, ww=w, hh=h):
        a = np.zeros((hh, ww * capi.TEXEL_BYTES[fmt]), np.uint8)
        keep.append(a)
        return capi.GrbImage(a.ctypes.data, ww, hh, ww * capi.TEXEL_BYTES[fmt], fmt)

    color = img(capi.FORMAT_R8G8B8A8_UNORM)
    layout = capi.GrbImage(None, w, h, w * 2, capi.FORMAT_R8G8_UNORM)
    slots = [img(capi.FORMAT_R8G8_UNORM) for _ in range(2)]
    flags = np.zeros((2, 16), np.uint32)
    counter = np.zeros(1, np.uint32)
    images = (C.c_void_p * 8)(*[s.data for s in slots])
    flag_ptrs = (C.c_void_p * 8)(*[flags[r].ctypes.data for r in range(2)])
    cnt = counter.ctypes.data_as(C.c_void_p)
    R = capi.GrbRows

    def prs(*rows):
        return (R * 8)(*[R(a, b) for a, b in rows])

    def call(color_=color, quality=3, out_layout=layout, imgs=images, peer_rows=None, fl=flag_ptrs, count=2, index=0, scratch=cnt, rows=R(0, 6)):
        pr = peer_rows if peer_rows is not None else prs((0, 6), (2, 6))
        return lib.grb_smaa_edge_detection_to_peers(C.byref(color_), quality, C.byref(out_layout) if out_layout is not None else None, imgs, pr, fl,
                                                    count, index, 1, scratch, rows, None)

    assert call(count=0) == ERR_ARG and "peer_count" in _msg(lib)
    assert call(count=9) == ERR_ARG
    assert call(index=2) == ERR_ARG and "flag_index" in _msg(lib)
    assert call(index=-1) == ERR_ARG
    assert call(imgs=None) == ERR_ARG
    assert call(fl=None) == ERR_ARG
    assert call(scratch=None) == ERR_ARG
    assert call(out_layout=None) == ERR_ARG
    assert lib.grb_smaa_edge_detection_to_peers(C.byref(color), 3, C.byref(layout), images, None, flag_ptrs, 2, 0, 1, cnt, R(0, 6), None) == ERR_ARG
    assert call(imgs=(C.c_void_p * 8)(slots[0].data, None)) == ERR_ARG and "null peer pointer" in _msg(lib)
    assert call(fl=(C.c_void_p * 8)(flag_ptrs[0], None)) == ERR_ARG and "null peer pointer" in _msg(lib)
    # formats and sizes: colour R8G8B8A8, every slot R8G8_UNORM of the colour's size
    assert call(color_=img(capi.FORMAT_B10G11R11_UFLOAT)) == ERR_FORMAT and "grb_smaa_edge_detection_to_peers" in _msg(lib)
    assert call(out_layout=capi.GrbImage(None, w + 1, h, (w + 1) * 2, capi.FORMAT_R8G8_UNORM)) == ERR_FORMAT
    assert call(out_layout=capi.GrbImage(None, w, h, w * 4, capi.FORMAT_R8G8B8A8_UNORM)) == ERR_FORMAT
    assert call(quality=4) == ERR_FORMAT and "quality" in _msg(lib)
    assert call(quality=-1) == ERR_FORMAT
    # rows: a non-empty range of the image
    assert call(rows=R(5, 5), peer_rows=prs((5, 5), (5, 5))) == ERR_ARG and "rows" in _msg(lib)
    assert call(rows=R(-1, 6), peer_rows=prs((-1, 6), (2, 6))) == ERR_ARG
    assert call(rows=R(6, h + 1), peer_rows=prs((6, h + 1), (6, 8))) == ERR_ARG
    # peer_rows[flag_index] equals rows; every peer_rows[r] lies inside rows
    assert call(peer_rows=prs((0, 5), (2, 6))) == ERR_ARG and "peer_rows[flag_index]" in _msg(lib)
    assert call(index=1, peer_rows=prs((0, 6), (2, 6))) == ERR_ARG
    assert call(peer_rows=prs((0, 6), (2, 7))) == ERR_ARG and "inside rows" in _msg(lib)
    assert call(peer_rows=prs((0, 6), (4, 3))) == ERR_ARG
    assert not flags.any() and not counter.any(), "a refused call must not touch the flags"
