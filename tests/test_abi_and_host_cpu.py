"""CPU-only checks of the product's boundary and host logic (no compute calls, no GPU):
the C-ABI libraries load and export every symbol the headers declare, struct layouts match the
reference's, the C++ RenderGraph surface behaves (tests/cpp), and host light preparation is
byte-identical to the oracle's restatement of lights.cpp / clusterer.cpp."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built():
    from granite_b200 import build

    return build.build_all()


def _declared(header):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(grbh?_[a-z0-9_]+)\s*\(", text)))


def test_kernel_library_exports_every_declared_symbol(built):
    from granite_b200 import capi

    lib = capi.lib()
    names = _declared("granite_b200.h")
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), f"libgranite_b200.so does not export {n}"
    assert set(names) == set(capi.ENTRY_POINTS), "capi.ENTRY_POINTS out of sync with include/granite_b200.h"
    assert lib.grb_abi_version() == 1
    # nm: no undefined reference into the oracle, no exported symbol outside the grb_ prefix besides C++ internals
    out = subprocess.run(["nm", "-D", "--defined-only", capi.LIB_PATH], capture_output=True, text=True).stdout
    assert "orc_" not in out


def test_host_library_exports_every_declared_symbol(built):
    from granite_b200 import viewer

    lib = viewer.lib()
    for n in _declared("granite_b200_host.h"):
        if n.startswith("grbh_"):
            assert hasattr(lib, n), f"libgranite_b200_host.so does not export {n}"
    out = subprocess.run(["nm", "-D", viewer.HOST_LIB_PATH], capture_output=True, text=True).stdout
    assert "orc_" not in out, "the product must not link the oracle"


def test_struct_layouts():
    from granite_b200 import capi

    assert C.sizeof(capi.GrbPositionalLight) == 48          # light_info.hpp:44 static_assert
    assert capi.GrbPositionalLight.position.offset == 16 and capi.GrbPositionalLight.inv_radius.offset == 44
    assert C.sizeof(capi.GrbImage) == 24
    assert C.sizeof(capi.GrbRows) == 8
    assert C.sizeof(capi.GrbCamera) == 3 * 64 + 2 * 12 + 8
    assert capi.FORMAT_B10G11R11_UFLOAT == 122 and capi.FORMAT_R16G16B16A16_SFLOAT == 97 and capi.FORMAT_R8G8B8A8_SRGB == 43  # VkFormat values


def test_missing_extension_fails_loudly(monkeypatch):
    from granite_b200 import capi

    monkeypatch.setattr(capi, "_lib", None)
    monkeypatch.setattr(capi, "LIB_PATH", "/nonexistent/libgranite_b200.so")
    with pytest.raises(capi.GrbError):
        capi.lib()


def test_product_sources_never_touch_the_oracle():
    bad = []
    for base in ("granite_b200", "include"):
        for root, _, files in os.walk(os.path.join(ROOT, base)):
            if "build" in root.split(os.sep):
                continue
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".cpp", ".hpp", ".h")):
                    text = open(os.path.join(root, f), errors="ignore").read()
                    if re.search(r"(import|from)\s+oracle|pyoracle|liboracle|orc_[a-z]", text):
                        bad.append(os.path.join(root, f))
    assert not bad, f"product files reference the oracle: {bad}"


def _smaa_lut_dir(tmp_path):
    """The reference's SMAA lookup textures: its own asset directory where it exists, else the same texels (recorded
    from those files in tests/golden/refsmaa_160x96.npz) in .gtx containers written to tmp_path."""
    from oracle import pyoracle

    if os.path.isdir(pyoracle.SMAA_LUT_DIR):
        return pyoracle.SMAA_LUT_DIR
    f = np.load(os.path.join(ROOT, "tests", "golden", "refsmaa_160x96.npz"))
    for name, fmt in (("area", 16), ("search", 9)):  # VK_FORMAT_R8G8_UNORM, VK_FORMAT_R8_UNORM
        texels = np.ascontiguousarray(f[name])
        h, w, _ = texels.shape
        # 64-byte header (memory_mapped_texture.cpp:29-46): magic, 2-D type, format, size, depth, layers, levels, flags, payload
        header = b"GRANITE TEXFMT1\0" + np.array([1, fmt, w, h, 1, 1, 1, 0], np.uint32).tobytes() + np.uint64(texels.size).tobytes() + bytes(8)
        (tmp_path / f"{name}.gtx").write_bytes(header + texels.tobytes())
    return str(tmp_path)


def test_render_graph_cpp(built, tmp_path):
    exe = str(tmp_path / "test_render_graph")
    luts = tmp_path / "smaa"
    luts.mkdir()
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    libdir = os.path.join(ROOT, "granite_b200")
    cmd = ["g++", "-O1", "-std=c++17", f"-I{cuda}/include", os.path.join(ROOT, "tests", "cpp", "test_render_graph.cpp"), "-o", exe,
           f"-L{libdir}", "-lgranite_b200_host", "-lgranite_b200", f"-Wl,-rpath,{libdir}", f"-Wl,-rpath,{cuda}/lib64"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe, _smaa_lut_dir(luts)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


def _host_viewer(w=1920, h=1080):
    from granite_b200 import synth, viewer

    v = viewer.Viewer(w, h, cuda_device=-1)  # host-only: no device is created
    v.set_camera(synth.perspective_inf(np.pi / 4, w / h, 1 / 16), synth.look_at_view((0, 0, 8), (0, 0, 0)))
    return v


def test_host_float_to_half_matches_oracle(built, oracle):
    from granite_b200 import viewer

    L, H = oracle.lib(), viewer.lib()
    rng = np.random.default_rng(11)
    bits = np.concatenate([rng.integers(0, 2 ** 32, size=40000, dtype=np.uint64).astype(np.uint32),
                           np.arange(0x38000000 - 50, 0x38000000 + 20000, dtype=np.uint32),
                           np.arange(0x33000000 - 50, 0x33000000 + 50, dtype=np.uint32),
                           np.arange(0x477FE000 - 100, 0x477FE000 + 100, dtype=np.uint32),
                           np.array([0, 0x80000000, 0x7F800000, 0xFF800000, 0x7FC00000, 0x7F800001], np.uint32)])
    for f in bits.view(np.float32):
        assert H.grbh_float_to_half(C.c_float(f)) == L.orc_float_to_half(C.c_float(f)), hex(np.float32(f).view(np.uint32))


def test_host_camera_block(built, oracle):
    from granite_b200 import synth

    v = _host_viewer()
    cam, proj, inv_proj = v.camera()
    ref = oracle.camera_setup(synth.perspective_inf(np.pi / 4, 16 / 9, 1 / 16), synth.look_at_view((0, 0, 8), (0, 0, 0)))
    assert np.array_equal(np.array(list(cam.view_projection), np.float32), np.array(list(ref.view_projection), np.float32))
    # the host layer's general inverse is not the reference's cofactor expansion: equal to an ulp
    assert np.allclose(np.array(list(cam.inv_view_projection)), np.array(list(ref.inv_view_projection)), rtol=3e-7, atol=1e-7)
    assert list(cam.camera_position) == [0.0, 0.0, 8.0] and list(cam.camera_front) == [0.0, 0.0, -1.0]
    assert cam.z_near == ref.z_near and cam.z_far == pytest.approx(ref.z_far, rel=1e-6)


@pytest.mark.parametrize("n,spots", [(0, 0.0), (16, 0.0), (300, 0.25), (4096, 0.25)])
def test_host_light_prep_is_byte_identical_to_oracle(built, oracle, n, spots):
    from granite_b200 import synth
    from tests import common

    v = _host_viewer()
    lights = synth.make_lights(n, spot_fraction=spots)
    # hand the lights over in a shuffled order: the clusterer must restore front-to-back order
    perm = np.random.default_rng(1).permutation(n)
    shuffled = synth.Lights(lights.color[perm], lights.position[perm], lights.is_point[perm], lights.rot[perm],
                            lights.inner_cone[perm], lights.outer_cone[perm])
    v.set_lights(shuffled)
    k, recs, model, tmask, zr = v.light_prep()
    assert k == n
    cam = common.oracle_camera_from_viewer(oracle, v)
    prep = oracle.prepare_lights(cam, lights)
    assert recs.tobytes() == prep.records[:n].tobytes()
    assert np.array_equal(model.view(np.uint32), prep.model[:n].view(np.uint32))
    assert np.array_equal(tmask, prep.type_mask[: len(tmask)])
    assert np.array_equal(zr, prep.z_ranges)
    p = prep.params
    # ClustererParametersBindless: z_scale = 1 / min(0.5, z_far / res_z) = 2, 128x64 tiles
    assert p.z_scale == 2.0 and p.z_max_index == 4095 and list(p.resolution_xy) == [128, 64] and p.num_lights_32 == (n + 31) // 32


def test_hdr10_output_rejects_fxaa(built):
    """FXAA reads the tonemapped 8-bit image; the HDR10 path (scene_viewer_application.cpp:1233-1288) has none."""
    from granite_b200 import viewer

    with pytest.raises(RuntimeError, match="FXAA"):
        viewer.Viewer(640, 360, cuda_device=-1, post_aa=viewer.AA_FXAA, hdr10_output=True)
    v = viewer.Viewer(640, 360, cuda_device=-1, post_aa=viewer.AA_TAA_HIGH, hdr10_output=True)  # host-only: accepted, nothing baked
    v.close()


def test_gtx_reader_reads_the_reference_lookup_textures(built, oracle, tmp_path):
    """The host library's .gtx reader (host/post/smaa.cpp) against the Python reader the oracle tests use, on the
    reference's lookup textures, whose texels the SMAA fixture holds."""
    from granite_b200 import capi, viewer

    d = _smaa_lut_dir(tmp_path)
    area, search = oracle.load_gtx(os.path.join(d, "area.gtx")), oracle.load_gtx(os.path.join(d, "search.gtx"))
    f = np.load(os.path.join(ROOT, "tests", "golden", "refsmaa_160x96.npz"))
    assert np.array_equal(area, f["area"]) and np.array_equal(search, f["search"])
    fmt, a = viewer.load_gtx(os.path.join(d, "area.gtx"))
    assert fmt == capi.FORMAT_R8G8_UNORM and np.array_equal(a, area)
    fmt, s = viewer.load_gtx(os.path.join(d, "search.gtx"))
    assert fmt == capi.FORMAT_R8_UNORM and np.array_equal(s, search)
    with pytest.raises(RuntimeError):
        viewer.load_gtx("/nonexistent.gtx")


def test_band_partition():
    from granite_b200 import viewer

    assert viewer.band_partition(2160, 1) == [(0, 2160)]
    assert viewer.band_partition(2160, 2) == [(0, 1088), (1088, 2160)]
    assert viewer.band_partition(2160, 4) == [(0, 512), (512, 1024), (1024, 1536), (1536, 2160)]
    b8 = viewer.band_partition(2160, 8)
    assert b8[0] == (0, 256) and b8[-1] == (1792, 2160) and all(a[1] == b[0] for a, b in zip(b8, b8[1:]))
    with pytest.raises(ValueError):
        viewer.band_partition(256, 8)


def test_measured_and_feedback_band_partitions():
    """band_partition_measured / rebalance_bands: valid tilings in 8-row units, one unit per rank at
    least, and the feedback step converges on a synthetic cost peaked like the bench scene's
    (a few dozen very expensive rows)."""
    from granite_b200 import viewer

    h, w = 2160, 3840
    rows = np.arange(h)
    per_row = 1.0 + 60.0 * np.exp(-(((rows - 1130) / 25.0) ** 2))

    def check(bands, world):
        assert len(bands) == world and bands[0][0] == 0 and bands[-1][1] == h
        assert all(a[1] == b[0] for a, b in zip(bands, bands[1:]))
        assert all((b[1] - b[0]) >= 8 and b[0] % 8 == 0 for b in bands)

    cost4 = (per_row.reshape(-1, 4).sum(axis=1) * 1e4).astype(np.uint32)
    for world in (2, 4, 8):
        bands = viewer.band_partition_measured(h, w, world, cost4, align=8, post_warp_inst_per_pixel=0.0)
        check(bands, world)
        work = [per_row[a:b].sum() for a, b in bands]
        assert max(work) < 1.6 * per_row.sum() / world  # equal work up to the 8-row granularity at the peak
        # the thin bands sit on the expensive rows
        assert min(b[1] - b[0] for b in bands) < h // world

        # feedback from "measured times" that are NOT the work: a band never beats a latency floor
        def times(bs):
            return [max(per_row[a:b].sum(), 0.12 * per_row.sum()) if per_row[a:b].max() > 30 else per_row[a:b].sum() for a, b in bs]

        cur = viewer.band_partition(h, world, align=8)
        first = max(times(cur))
        best = first
        for _ in range(8):
            cur = viewer.rebalance_bands(cur, times(cur), h, align=8, prior_per_row=per_row)
            check(cur, world)
            best = min(best, max(times(cur)))
        assert best <= first
    assert viewer.rebalance_bands([(0, h)], [1.0], h) == [(0, h)]
