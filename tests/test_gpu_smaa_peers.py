"""grb_smaa_edge_detection_to_peers on one GPU: 2 - 4 "peer" edge slots and flag arrays, all on the one device, and one
call per band.  Each rank's colour is valid on its plan["tonemap"] rows only, and its slot starts as 255 (an edge
everywhere).  Every slot must equal the unsharded edges on the rank's whole plan["smaa_edges"] window (and be untouched
outside it), the weights a rank computes from its slot and the rows it blends must equal one unsharded SMAA bit for bit,
and grb_peer_wait must return on every flag array."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from tests.test_oracle_ref_smaa import smaa_test_image

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _bands(h, world, layout):
    from granite_b200 import viewer

    if layout == "64":
        return viewer.band_partition(h, world)
    # uneven 8-row-aligned bands with narrow ones (24 and 40 rows: narrower than the Ultra reach)
    mid = (h // 16) * 8
    cuts = {2: [0, 24, h], 3: [0, 24, mid, h], 4: [0, mid, mid + 40, mid + 80, h]}[world]
    return list(zip(cuts[:-1], cuts[1:]))


def _peer_call(cuda, color_t, quality, slots, peer_rows, flags, counter, flag_index, epoch, rows):
    from granite_b200 import capi

    ci = capi.image(color_t, capi.FORMAT_R8G8B8A8_UNORM)
    layout = capi.image(slots[0], capi.FORMAT_R8G8_UNORM)
    layout.data = None
    images = (C.c_void_p * 8)(*[s.data_ptr() for s in slots])
    flag_ptrs = (C.c_void_p * 8)(*[f.data_ptr() for f in flags])
    pr = (capi.GrbRows * 8)(*[capi.GrbRows(a, b) for a, b in peer_rows])
    cuda.check(cuda.lib().grb_smaa_edge_detection_to_peers(C.byref(ci), int(quality), C.byref(layout), images, pr, flag_ptrs, len(slots), flag_index,
                                                           epoch, C.c_void_p(counter.data_ptr()), capi.rows(rows), capi.stream_ptr()),
               "grb_smaa_edge_detection_to_peers")


@pytest.mark.parametrize("w,h", [(1920, 1080), (3840, 2160), (1001, 777)])
@pytest.mark.parametrize("world,layout", [(2, "64"), (2, "uneven"), (3, "uneven"), (4, "64"), (4, "uneven")])
@pytest.mark.parametrize("quality", [0, 1, 2, 3])
def test_smaa_edges_to_peers_equal_unsharded(cuda, quality, world, layout, w, h):
    from granite_b200 import harness, viewer

    f = np.load(os.path.join(GOLDEN, "refsmaa_160x96.npz"))
    area = harness.to_dev(np.ascontiguousarray(f["area"]))
    search = harness.to_dev(np.ascontiguousarray(f["search"]).reshape(16, 64))
    img = smaa_test_image(w, h, w + h + quality)
    # noise on the right half: weights on almost every pixel, so the blend's taps that round to the row above a band
    # start (rows 704 and 1080 of 2160) see them
    img[:, w // 2:] = np.random.default_rng(quality).integers(0, 2 ** 32, size=(h, w - w // 2), dtype=np.uint32)
    color = harness.to_dev(img)

    ref_e = torch.zeros((h, w, 2), dtype=torch.uint8, device="cuda")
    ref_w = torch.zeros((h, w), dtype=torch.int32, device="cuda")
    harness.smaa_edge_detection(color, quality, ref_e)
    harness.smaa_blend_weights(ref_e, area, search, quality, ref_w)
    ref_out = {}
    for srgb in (True, False):
        ref_out[srgb] = torch.zeros((h, w), dtype=torch.int32, device="cuda")
        harness.smaa_neighborhood_blend(color, ref_w, ref_out[srgb], target_srgb=srgb)

    bands = _bands(h, world, layout)
    plans = [viewer.shard_plan(w, h, bands, r, smaa=quality) for r in range(world)]
    slots = [torch.full((h, w, 2), 255, dtype=torch.uint8, device="cuda") for _ in range(world)]
    flags = [torch.zeros(16, dtype=torch.int32, device="cuda") for _ in range(world)]
    counter = torch.zeros(1, dtype=torch.int32, device="cuda")
    epoch = 7
    gen = torch.Generator(device="cuda").manual_seed(quality)
    colors = []
    for q in range(world):
        own = plans[q]["own"]
        ta, tb = plans[q]["tonemap"]
        c = torch.randint(-2 ** 31, 2 ** 31 - 1, (h, w), dtype=torch.int32, device="cuda", generator=gen)  # garbage off the tonemap rows
        c[ta:tb] = color[ta:tb]
        colors.append(c)
        peer_rows = []
        for r in range(world):
            a, b = max(own[0], plans[r]["smaa_edges"][0]), min(own[1], plans[r]["smaa_edges"][1])
            peer_rows.append((a, b) if a < b else (own[0], own[0]))
        _peer_call(cuda, c, quality, slots, peer_rows, flags, counter, q, epoch, own)
    L = cuda.lib()
    L.grb_peer_wait.argtypes = [C.c_void_p, C.c_int32, C.c_uint32, C.c_void_p]
    for fl in flags:
        cuda.check(L.grb_peer_wait(C.c_void_p(fl.data_ptr()), world, epoch, cuda.stream_ptr()), "grb_peer_wait")
    torch.cuda.synchronize()
    for r, fl in enumerate(flags):
        got = fl.cpu().numpy()
        assert (got[:world] == epoch).all() and not got[world:].any(), f"flag array of rank {r}: {got}"
    assert int(counter.item()) == 0, "the last CTA resets the scratch counter"

    want_e = ref_e.cpu().numpy()
    for r in range(world):
        p = plans[r]
        ea, eb = p["smaa_edges"]
        s = slots[r].cpu().numpy()
        assert np.array_equal(s[ea:eb], want_e[ea:eb]), f"rank {r}: edge window [{ea},{eb}) differs from the unsharded edges"
        assert (s[:ea] == 255).all() and (s[eb:] == 255).all(), f"rank {r}: rows outside the window were written"
        wg = torch.randint(-2 ** 31, 2 ** 31 - 1, (h, w), dtype=torch.int32, device="cuda", generator=gen)  # garbage off the computed rows
        harness.smaa_blend_weights(slots[r], area, search, quality, wg, rows=p["smaa_weights"])
        wa, wb = p["smaa_weights"]
        assert torch.equal(wg[wa:wb], ref_w[wa:wb]), f"rank {r}: weights [{wa},{wb}) differ"
        a, b = p["own"]
        for srgb in (True, False):
            out = torch.zeros((h, w), dtype=torch.int32, device="cuda")
            harness.smaa_neighborhood_blend(colors[r], wg, out, target_srgb=srgb, rows=(a, b))
            assert torch.equal(out[a:b], ref_out[srgb][a:b]), f"rank {r}: blended rows [{a},{b}) differ ({'sRGB' if srgb else 'UNORM'})"
