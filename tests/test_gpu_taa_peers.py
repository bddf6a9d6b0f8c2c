"""grb_taa_resolve_to_peers on one GPU: 2 - 4 "peer" history slots and flag arrays, all on the one device, and one
call per band.  Every slot must equal the out_history of one unsharded grb_taa_resolve bit for bit, each band's
out_color rows must equal the unsharded ones, and every flag must reach the epoch (grb_peer_wait returns)."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _peer_call(capi, harness, hdr_t, depth_t, mv_t, hist_t, reproj, quality, oc_t, slots, flags, counter, flag_index, epoch, rows, own):
    L = capi.lib()
    hi = harness._hdr_img(hdr_t)
    oc = capi.image(oc_t, capi.FORMAT_B10G11R11_UFLOAT)
    layout = harness._img16(slots[0])
    di = C.byref(capi.image(depth_t, capi.FORMAT_D32_SFLOAT)) if depth_t is not None else None
    mi = C.byref(capi.image(mv_t, capi.FORMAT_R16G16_SFLOAT)) if mv_t is not None else None
    hs = C.byref(harness._img16(hist_t)) if hist_t is not None else None
    rp = (C.c_float * 16)(*np.asarray(reproj, np.float32).reshape(-1).tolist()) if reproj is not None else None
    images = (C.c_void_p * 8)(*[s.data_ptr() for s in slots])
    flag_ptrs = (C.c_void_p * 8)(*[f.data_ptr() for f in flags])
    capi.check(L.grb_taa_resolve_to_peers(C.byref(hi), di, mi, hs, rp, int(quality), C.byref(oc), C.byref(layout), images, flag_ptrs,
                                          len(slots), flag_index, epoch, C.c_void_p(counter.data_ptr()), capi.rows(rows), capi.rows(own),
                                          capi.stream_ptr()),
               "grb_taa_resolve_to_peers")


@pytest.mark.parametrize("hdr16", [False, True], ids=["b10g11r11", "rgba16f"])
@pytest.mark.parametrize("quality,history", [(0, False), (0, True), (1, True), (2, True)])
@pytest.mark.parametrize("world", [2, 3, 4])
def test_taa_resolve_to_peers_equals_unsharded(cuda, world, quality, history, hdr16):
    from granite_b200 import harness, viewer
    from tests import common
    from tests.test_gpu_parity import _taa_inputs

    w, h = 640, 384
    rng = np.random.default_rng(17 * world + 5 * quality + int(history) + 2 * int(hdr16))
    hdr, depth, mv, hist, reproj = _taa_inputs(rng, w, h)
    # motion vectors of 40+ rows: history reads from other bands
    fast = rng.random((h, w)) < 0.03
    mv16 = mv.reshape(h, w, 2).view(np.float16).copy()
    mv16[fast, 1] = (rng.uniform(40.0, 90.0, size=int(fast.sum())) * rng.choice([-1.0, 1.0], size=int(fast.sum())) / h).astype(np.float16)
    mv = mv16.view(np.uint16)
    if hdr16:
        hdr = common.random_hdr_f16(rng, w, h, scale=2.0)
    hdr_t = harness.to_dev(hdr)
    depth_t = harness.to_dev(depth) if history else None
    mv_t = harness.to_dev(mv.reshape(h, w, 2)).view(torch.int32).reshape(h, w) if history else None
    hist_t = harness.to_dev(hist) if history else None
    rp = reproj if history else None

    ref_c = torch.zeros((h, w), dtype=torch.int32, device="cuda")
    ref_h = harness.new_rgba16f(w, h)
    harness.taa_resolve(hdr_t, depth_t, mv_t, hist_t, rp, quality, ref_c, ref_h)

    bands = viewer.band_partition(h, world)
    slots = [harness.new_rgba16f(w, h) for _ in range(world)]
    flags = [torch.zeros(16, dtype=torch.int32, device="cuda") for _ in range(world)]
    counter = torch.zeros(1, dtype=torch.int32, device="cuda")
    epoch = 5
    colors = []
    for r in range(world):
        plan = viewer.shard_plan(w, h, bands, r, True, taa=True)
        oc = torch.zeros((h, w), dtype=torch.int32, device="cuda")
        _peer_call(cuda, harness, hdr_t, depth_t, mv_t, hist_t, rp, quality, oc, slots, flags, counter, r, epoch, plan["taa"], plan["own"])
        colors.append((plan["taa"], oc))
    L = cuda.lib()
    L.grb_peer_wait.argtypes = [C.c_void_p, C.c_int32, C.c_uint32, C.c_void_p]
    for f in flags:
        cuda.check(L.grb_peer_wait(C.c_void_p(f.data_ptr()), world, epoch, cuda.stream_ptr()), "grb_peer_wait")
    torch.cuda.synchronize()

    want_h = harness.to_host(ref_h, np.uint16)
    for r, s in enumerate(slots):
        assert np.array_equal(harness.to_host(s, np.uint16), want_h), f"history slot of rank {r} differs from the unsharded out_history"
    want_c = harness.to_host(ref_c, np.uint32)
    for (a, b), oc in colors:
        got = harness.to_host(oc, np.uint32)
        assert np.array_equal(got[a:b], want_c[a:b]), f"out_color rows [{a},{b}) differ"
        assert not got[:a].any() and not got[b:].any(), "nothing outside the resolved rows is written"
    for r, f in enumerate(flags):
        got = f.cpu().numpy()
        assert (got[:world] == epoch).all() and not got[world:].any(), f"flag array of rank {r}: {got}"
    assert int(counter.item()) == 0, "the last CTA resets the scratch counter"
    # a second frame on the same flags and counter (epoch + 1) publishes again
    plan = viewer.shard_plan(w, h, bands, 0, True, taa=True)
    oc = torch.zeros((h, w), dtype=torch.int32, device="cuda")
    _peer_call(cuda, harness, hdr_t, depth_t, mv_t, hist_t, rp, quality, oc, slots, flags, counter, 0, epoch + 1, plan["taa"], plan["own"])
    torch.cuda.synchronize()
    assert all(int(f[0].item()) == epoch + 1 for f in flags)
