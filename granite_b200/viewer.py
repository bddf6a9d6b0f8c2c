"""ctypes binding of libgranite_b200_host.so (include/granite_b200_host.h): the application-side
harness over the C++ host layer (RenderGraph, LightClusterer, pass builders).  This is the
repo's public end-to-end API: host G-buffer in -> frame on the GPU(s) -> tonemapped image out.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import capi

_HERE = os.path.dirname(os.path.abspath(__file__))
HOST_LIB_PATH = os.path.join(_HERE, "libgranite_b200_host.so")

AA_NONE, AA_FXAA, AA_TAA_LOW, AA_TAA_MEDIUM, AA_TAA_HIGH, AA_TAA_HIGH_PLUS_FXAA = 0, 1, 8, 9, 10, 100
AA_SMAA_LOW, AA_SMAA_MEDIUM, AA_SMAA_HIGH, AA_SMAA_ULTRA = 3, 4, 5, 6


class GrbhViewerConfig(C.Structure):
    _fields_ = [("cuda_device", C.c_int32), ("width", C.c_int32), ("height", C.c_int32), ("post_aa", C.c_int32),
                ("hdr_bloom", C.c_int32), ("dynamic_exposure", C.c_int32), ("cluster_res", C.c_int32 * 3),
                ("timestamps", C.c_int32), ("cuda_stream", C.c_void_p), ("pipelined_io", C.c_int32),
                ("hdr10_output", C.c_int32), ("hdr10_max_content_light_level", C.c_float),
                ("clustered_lights_shadows", C.c_int32), ("clustered_lights_shadow_resolution", C.c_int32),
                ("resolution_scale", C.c_float), ("resolution_scale_sharpen", C.c_int32), ("render_target_fp16", C.c_int32), ("volumetric_decals", C.c_int32)]


class GrbhLights(C.Structure):
    _fields_ = [("count", C.c_int32), ("color", C.c_void_p), ("position", C.c_void_p), ("is_point", C.c_void_p),
                ("rotation", C.c_void_p), ("inner_cone", C.c_void_p), ("outer_cone", C.c_void_p), ("cutoff_range", C.c_float)]


class GrbhHostGBuffer(C.Structure):
    _fields_ = [("albedo", C.c_void_p), ("normal", C.c_void_p), ("pbr", C.c_void_p), ("depth", C.c_void_p),
                ("emissive", C.c_void_p), ("mv", C.c_void_p)]


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        capi.lib()  # libgranite_b200.so first (the host library links against it)
        if not os.path.exists(HOST_LIB_PATH):
            raise capi.GrbError(f"{HOST_LIB_PATH} is missing: run `python -m granite_b200.build`")
        _lib = C.CDLL(HOST_LIB_PATH)
        _lib.grbh_last_error.restype = C.c_char_p
        _lib.grbh_float_to_half.restype = C.c_uint16
        _lib.grbh_float_to_half.argtypes = [C.c_float]
        _lib.grbh_viewer_destroy.restype = None
        _lib.grbh_viewer_destroy.argtypes = [C.c_void_p]
        _lib.grbh_viewer_render_frame.argtypes = [C.c_void_p, C.POINTER(GrbhHostGBuffer), C.c_double]
        _lib.grbh_viewer_set_exposure.argtypes = [C.c_void_p, C.c_float]
    return _lib


def _check(rc, what):
    if rc < 0:
        raise capi.GrbError(f"{what}: {lib().grbh_last_error().decode()}")
    return rc


def _vp(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def band_partition(height: int, world: int, align: int = 64):
    """Contiguous row bands aligned to `align` full-res rows (= 2 rows of the 1/32 bloom level,
    SURVEY.md §8e), remainder on the last rank."""
    n_units = (height + align - 1) // align
    per = n_units // world
    if per == 0:
        raise ValueError("frame too small for this many ranks")
    bands = []
    y = 0
    for r in range(world):
        y1 = height if r == world - 1 else (y + per * align)
        bands.append((y, y1))
        y = y1
    return bands


def band_partition_weighted(height: int, world: int, band_cost, align: int = 64):
    """Contiguous `align`-row bands with roughly equal COST per rank (band_cost[i] = estimated work of
    rows [i*align, (i+1)*align)).  Lighting cost follows the lights, not the pixel count, so equal-height
    bands leave ranks idle; this balances the per-rank sum greedily along the prefix sums."""
    cost = np.asarray(band_cost, np.float64)
    n_units = (height + align - 1) // align
    assert len(cost) == n_units
    if world == 1:
        return [(0, height)]
    if n_units < world:
        raise ValueError("frame too small for this many ranks")
    prefix = np.concatenate([[0.0], np.cumsum(cost)])
    total = prefix[-1]
    cuts = [0]
    for r in range(1, world):
        target = total * r / world
        k = int(np.searchsorted(prefix, target))
        if k > 0 and abs(prefix[k - 1] - target) < abs(prefix[min(k, n_units)] - target):
            k -= 1
        k = max(k, cuts[-1] + 1)               # at least one unit per rank
        k = min(k, n_units - (world - r))       # leave one unit for each remaining rank
        cuts.append(k)
    cuts.append(n_units)
    return [(cuts[i] * align, min(cuts[i + 1] * align, height)) for i in range(world)]


def estimate_band_cost(projection, view, light_positions, light_colors, width, height, depth=None, near=1.0 / 16.0,
                       align: int = 64, tiles_x: int = 128, base_lights: float = 4.0):
    """Host-side cost model for band_partition_weighted.  Per (64-row band, screen tile): pixels x
    (base + number of lights whose projected bounding square AND view-depth range overlap the tile).
    Light radius = sqrt(max colour / 0.1) (lights.cpp:63-70); tile depth range from the reverse-Z
    depth image when given (view depth = near / depth), else unbounded.  Only relative weights matter."""
    P = np.asarray(projection, np.float64).reshape(4, 4).T  # column-major storage -> math matrix
    V = np.asarray(view, np.float64).reshape(4, 4).T
    pos = np.asarray(light_positions, np.float64)
    n_units = (height + align - 1) // align
    if len(pos) == 0:
        return np.full(n_units, float(width * align))
    radius = np.sqrt(np.asarray(light_colors, np.float64).max(axis=1) / 0.1)
    pv = (V @ np.concatenate([pos, np.ones((len(pos), 1))], axis=1).T).T
    z = np.maximum(-pv[:, 2], 1e-3)
    cy = (P[1, 1] * pv[:, 1] / z * 0.5 + 0.5) * height
    cx = (P[0, 0] * pv[:, 0] / z * 0.5 + 0.5) * width
    inside = z <= radius * 1.05
    ry = np.where(inside, height, radius / z * abs(P[1, 1]) * height * 0.5)
    rx = np.where(inside, width, radius / z * abs(P[0, 0]) * width * 0.5)
    ly0, ly1, lx0, lx1 = cy - ry, cy + ry, cx - rx, cx + rx
    lz0, lz1 = z - radius, z + radius

    tile_w = width / tiles_x
    tx0 = np.arange(tiles_x) * tile_w
    by0 = np.arange(n_units) * align
    by1 = np.minimum(by0 + align, height)
    if depth is not None:
        d = np.asarray(depth, np.float32)
        zmin = np.full((n_units, tiles_x), np.inf)
        zmax = np.full((n_units, tiles_x), -np.inf)
        lit = np.zeros((n_units, tiles_x))
        step = max(int(tile_w), 1)
        for u in range(n_units):
            rows = d[by0[u]:by1[u]]
            cols = (rows.shape[1] // step) * step
            blk = rows[:, :cols].reshape(rows.shape[0], -1, step)[:, :tiles_x]
            with np.errstate(divide="ignore"):
                vz = np.where(blk > 0, near / np.maximum(blk, 1e-30), np.nan)
            has = np.isfinite(vz).any(axis=(0, 2))
            k = vz.shape[1]
            zmin[u, :k] = np.where(has, np.nanmin(np.where(np.isfinite(vz), vz, np.inf), axis=(0, 2)), np.inf)
            zmax[u, :k] = np.where(has, np.nanmax(np.where(np.isfinite(vz), vz, -np.inf), axis=(0, 2)), -np.inf)
            lit[u, :k] = np.isfinite(vz).mean(axis=(0, 2))
    else:
        zmin = np.zeros((n_units, tiles_x))
        zmax = np.full((n_units, tiles_x), np.inf)
        lit = np.ones((n_units, tiles_x))
    cost = np.zeros(n_units)
    for u in range(n_units):
        row_ok = (ly1 > by0[u]) & (ly0 < by1[u])                                   # (L,)
        xo = (lx1[None, :] > tx0[:, None]) & (lx0[None, :] < tx0[:, None] + tile_w)   # (T, L)
        zo = (lz1[None, :] > zmin[u][:, None]) & (lz0[None, :] < zmax[u][:, None])    # (T, L)
        n_l = (xo & zo & row_ok[None, :]).sum(axis=1)                              # lights per tile
        cost[u] = float(((base_lights + n_l) * lit[u]).sum() * tile_w * (by1[u] - by0[u])) + 0.5 * width * (by1[u] - by0[u])
    return cost


def band_partition_measured(height: int, width: int, world: int, cost_per_4_rows, align: int = 8, post_warp_inst_per_pixel: float = 9.4):
    """Row bands of equal estimated GPU work from Viewer.measure_row_cost() (warp instructions of the
    lighting pass per 4-row group).  The band-proportional part of the post chain (threshold,
    first down/upsample, tonemap: ~300 thread instructions = 9.4 warp instructions per pixel, from
    profiles/round1c_frame_launches.md) is added per row so that light-free bands are not free."""
    assert align % 4 == 0
    c = np.asarray(cost_per_4_rows, np.float64)
    groups = (height + 3) // 4
    assert len(c) == groups
    c = c + post_warp_inst_per_pixel * width * 4.0
    per = align // 4
    n_units = (height + align - 1) // align
    c = np.concatenate([c, np.zeros(n_units * per - groups)]).reshape(n_units, per).sum(axis=1)
    return band_partition_weighted(height, world, c, align=align)


def rebalance_bands(bands, band_times, height: int, align: int = 8, damping: float = 0.7, prior_per_row=None):
    """One step of feedback load balancing for row bands: `band_times[r]` is what rank r needed for
    the band-dependent part of its last frames (e.g. the lighting pass, GPU-timed).  The time is
    taken as uniformly spread over the band's rows -- or along `prior_per_row` (e.g. the measured
    work estimate) within the band -- and the cuts are moved towards equal time, damped, in units
    of `align` rows, keeping at least one unit per rank.  Iterate a few times: the per-band times of
    this pass are not additive over rows (a band that leaves SMs idle is slower than its share)."""
    world = len(bands)
    t = np.asarray(band_times, np.float64)
    assert len(t) == world and world >= 1
    n_units = (height + align - 1) // align
    density = np.zeros(n_units)
    for (y0, y1), tr in zip(bands, t):
        u0, u1 = y0 // align, (y1 + align - 1) // align
        if prior_per_row is not None:
            w = np.add.reduceat(np.asarray(prior_per_row, np.float64)[y0:y1], np.arange(0, y1 - y0, align)) + 1e-9
        else:
            w = np.ones(u1 - u0)
        density[u0:u1] = tr * w / w.sum()
    target = band_partition_weighted(height, world, density, align=align)
    out = []
    prev = 0
    for r in range(world):
        if r == world - 1:
            y1 = height
        else:
            want = bands[r][1] + damping * (target[r][1] - bands[r][1])
            y1 = int(round(want / align)) * align
            y1 = max(y1, prev + align)
            y1 = min(y1, height - (world - 1 - r) * align)
        out.append((prev, y1))
        prev = y1
    return out


PLAN_FIELDS = ("own", "fxaa", "tonemap", "upsample0", "downsample0", "threshold", "lighting", "lum_grid")


def shard_plan(width, height, bands, rank, fxaa=False, taa=False, smaa=None) -> dict:
    """Rows of every stage one rank computes (host math of granite_b200/host/shard_plan.cpp).  taa=True: a TAA
    resolve precedes the post chain; the dict then also has "taa" (rows of the resolved image) and "lighting"
    covers taa +- 1 row.  smaa=0..3 (Low .. Ultra): SMAA follows the tonemap; the dict then also has "smaa_weights"
    (rows of the weights a rank computes) and "smaa_edges" (rows of the edges its weights pass reads), and
    "tonemap" covers own - 3 .. own + 2."""
    arr = (capi.GrbRows * max(len(bands), 1))(*[capi.GrbRows(a, b) for a, b in bands])
    if smaa is not None:
        out = (capi.GrbRows * 11)()
        _check(lib().grbh_shard_plan_smaa(width, height, arr, len(bands), rank, int(fxaa), int(taa), int(smaa), out), "grbh_shard_plan_smaa")
        names = PLAN_FIELDS + ("taa", "smaa_weights", "smaa_edges")
        return {k: (out[i].y0, out[i].y1) for i, k in enumerate(names) if k != "taa" or taa}
    if taa:
        out = (capi.GrbRows * 9)()
        _check(lib().grbh_shard_plan_ex(width, height, arr, len(bands), rank, int(fxaa), 1, out), "grbh_shard_plan_ex")
        return {k: (out[i].y0, out[i].y1) for i, k in enumerate(PLAN_FIELDS + ("taa",))}
    out = (capi.GrbRows * 8)()
    _check(lib().grbh_shard_plan(width, height, arr, len(bands), rank, int(fxaa), out), "grbh_shard_plan")
    return {k: (out[i].y0, out[i].y1) for i, k in enumerate(PLAN_FIELDS)}


class Viewer:
    def __init__(self, width, height, post_aa=AA_NONE, hdr_bloom=True, dynamic_exposure=True, cuda_device=0,
                 cluster_res=(128, 64, 4096), timestamps=False, stream=None, pipelined_io=False, hdr10_output=False, hdr10_max_cll=1000.0,
                 light_shadows=False, shadow_resolution=512, resolution_scale=0.0, resolution_scale_sharpen=True,
                 render_target_fp16=False, volumetric_decals=False):
        cfg = GrbhViewerConfig()
        cfg.cuda_device = cuda_device
        cfg.width, cfg.height = width, height
        cfg.post_aa = post_aa
        cfg.hdr_bloom = int(hdr_bloom)
        cfg.dynamic_exposure = int(dynamic_exposure)
        cfg.cluster_res = (C.c_int32 * 3)(*cluster_res)
        cfg.timestamps = int(timestamps)  # 1: aggregate per-pass times, 2: keep the raw timeline
        cfg.cuda_stream = stream
        cfg.pipelined_io = int(pipelined_io)
        cfg.hdr10_output = int(hdr10_output)
        cfg.hdr10_max_content_light_level = float(hdr10_max_cll)
        cfg.clustered_lights_shadows = int(light_shadows)
        cfg.clustered_lights_shadow_resolution = int(shadow_resolution)
        cfg.resolution_scale = float(resolution_scale)  # < 1: width x height is the display size, FSR 1 upscales to it
        cfg.resolution_scale_sharpen = int(resolution_scale_sharpen)
        cfg.volumetric_decals = int(volumetric_decals)
        cfg.render_target_fp16 = int(render_target_fp16)  # emissive / HDR-main as RGBA16F: host_gbuffer's emissive is (H, W, 4) uint16
        self.width, self.height = width, height
        self._h = C.c_void_p()
        _check(lib().grbh_viewer_create(C.byref(cfg), C.byref(self._h)), "grbh_viewer_create")
        self._keep = []

    def set_smaa_lookup_textures(self, area_rg8, search_r8):
        """area: (560, 160, 2) uint8, search: (16, 64[, 1]) uint8 -- the payloads of the reference's area.gtx / search.gtx."""
        a, s_ = np.ascontiguousarray(area_rg8, np.uint8), np.ascontiguousarray(search_r8, np.uint8)
        assert a.size == 160 * 560 * 2 and s_.size == 64 * 16
        _check(lib().grbh_viewer_set_smaa_lookup_textures(self._h, a.ctypes.data_as(C.c_void_p), s_.ctypes.data_as(C.c_void_p)),
               "grbh_viewer_set_smaa_lookup_textures")

    def set_decals(self, world_rows):
        """(n, 12) float32: world transforms (mat_affine rows) of the scene's volumetric decals (unit cubes in decal space)."""
        w = np.ascontiguousarray(world_rows, np.float32).reshape(-1, 12)
        self._keep.append(w)
        _check(lib().grbh_viewer_set_decals(self._h, w.ctypes.data_as(C.c_void_p), len(w)), "grbh_viewer_set_decals")

    def decal_prep(self, capacity=4096):
        """Host prep of the decal binning: ((n, 16) f32 mvps, (n, 2) u32 Z-slice ranges) of the visible decals, front to back."""
        m, z = np.zeros((capacity, 16), np.float32), np.zeros((capacity, 2), np.uint32)
        n = _check(lib().grbh_viewer_get_decal_prep(self._h, m.ctypes.data_as(C.c_void_p), z.ctypes.data_as(C.c_void_p), capacity), "grbh_viewer_get_decal_prep")
        return m[:n].copy(), z[:n].copy()

    def render_size(self):
        """(width, height) of the G-buffer the viewer expects (smaller than the display size when resolution_scale < 1)."""
        w, h = C.c_int32(), C.c_int32()
        _check(lib().grbh_viewer_get_render_size(self._h, C.byref(w), C.byref(h)), "grbh_viewer_get_render_size")
        return w.value, h.value

    def set_light_shadow_maps(self, device_pointers):
        """One device pointer (int, 0 = no shadow) per light of the last set_lights call, in that order."""
        arr = (C.c_void_p * len(device_pointers))(*[C.c_void_p(int(p) or None) for p in device_pointers])
        _check(lib().grbh_viewer_set_light_shadow_maps(self._h, arr, len(device_pointers)), "grbh_viewer_set_light_shadow_maps")

    def shadow_transforms(self, capacity=4096):
        """(n, 16) float32: ClustererBindlessTransforms::shadow of the visible lights in cluster order (host prep only)."""
        out = np.zeros((capacity, 16), np.float32)
        n = lib().grbh_viewer_get_shadow_transforms(self._h, out.ctypes.data_as(C.c_void_p), capacity)
        if n < 0:
            raise capi.GrbError("grbh_viewer_get_shadow_transforms: " + (lib().grbh_last_error() or b"").decode())
        return out[:n].copy()

    def close(self):
        if self._h:
            lib().grbh_viewer_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_camera(self, projection, view):
        p = np.ascontiguousarray(projection, np.float32)
        v = np.ascontiguousarray(view, np.float32)
        _check(lib().grbh_viewer_set_camera(self._h, _vp(p), _vp(v)), "grbh_viewer_set_camera")

    def set_directional(self, color, direction):
        c = np.ascontiguousarray(color, np.float32)
        d = np.ascontiguousarray(direction, np.float32)
        _check(lib().grbh_viewer_set_directional(self._h, _vp(c), _vp(d)), "grbh_viewer_set_directional")

    def set_exposure(self, e):
        _check(lib().grbh_viewer_set_exposure(self._h, C.c_float(e)), "grbh_viewer_set_exposure")

    def set_lights(self, lights, cutoff=1e10):
        n = len(lights.color)
        arrs = dict(color=np.ascontiguousarray(lights.color, np.float32), position=np.ascontiguousarray(lights.position, np.float32),
                    is_point=np.ascontiguousarray(lights.is_point, np.uint8), rotation=np.ascontiguousarray(lights.rot, np.float32),
                    inner=np.ascontiguousarray(lights.inner_cone, np.float32), outer=np.ascontiguousarray(lights.outer_cone, np.float32))
        l = GrbhLights(n, _vp(arrs["color"]), _vp(arrs["position"]), _vp(arrs["is_point"]), _vp(arrs["rotation"]),
                       _vp(arrs["inner"]), _vp(arrs["outer"]), cutoff)
        _check(lib().grbh_viewer_set_lights(self._h, C.byref(l)), "grbh_viewer_set_lights")

    def init_collectives(self, unique_id: bytes, rank: int, world: int):
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        _check(lib().grbh_viewer_init_collectives(self._h, buf, rank, world), "grbh_viewer_init_collectives")

    def set_row_shards(self, bands, rank):
        arr = (capi.GrbRows * len(bands))(*[capi.GrbRows(a, b) for a, b in bands])
        _check(lib().grbh_viewer_set_row_shards(self._h, arr, len(bands), rank), "grbh_viewer_set_row_shards")

    def bake(self):
        _check(lib().grbh_viewer_bake(self._h), "grbh_viewer_bake")

    @staticmethod
    def host_gbuffer(albedo, normal, pbr, depth, emissive, mv=None) -> GrbhHostGBuffer:
        """Arguments: objects with a data pointer (numpy arrays or pinned torch tensors)."""
        def ptr(x):
            if x is None:
                return None
            return x.data_ptr() if hasattr(x, "data_ptr") else x.ctypes.data
        return GrbhHostGBuffer(ptr(albedo), ptr(normal), ptr(pbr), ptr(depth), ptr(emissive), ptr(mv))

    def render_frame(self, host_gbuffer: GrbhHostGBuffer | None, frame_time=1.0 / 60.0):
        arg = C.byref(host_gbuffer) if host_gbuffer is not None else None
        _check(lib().grbh_viewer_render_frame(self._h, arg, C.c_double(frame_time)), "grbh_viewer_render_frame")

    def read_output(self, dst):
        """dst: full-frame uint32 buffer (numpy array or pinned torch tensor). Returns the (y0, y1) band written."""
        r = capi.GrbRows()
        p = dst.data_ptr() if hasattr(dst, "data_ptr") else dst.ctypes.data
        _check(lib().grbh_viewer_read_output(self._h, C.c_void_p(p), C.byref(r)), "grbh_viewer_read_output")
        return r.y0, r.y1

    def read_output_async(self, dst):
        """Enqueue the device->host copy of this frame's rows; pair with wait_outputs()."""
        r = capi.GrbRows()
        ptr = dst.data_ptr() if hasattr(dst, "data_ptr") else dst.ctypes.data
        _check(lib().grbh_viewer_read_output_async(self._h, C.c_void_p(ptr), C.byref(r)), "grbh_viewer_read_output_async")
        return r.y0, r.y1

    def wait_outputs(self, max_pending=0):
        _check(lib().grbh_viewer_wait_outputs(self._h, int(max_pending)), "grbh_viewer_wait_outputs")

    def join_streams(self):
        _check(lib().grbh_viewer_join_streams(self._h), "grbh_viewer_join_streams")

    def sync(self):
        _check(lib().grbh_viewer_sync(self._h), "grbh_viewer_sync")

    def image(self, name) -> capi.GrbImage:
        img = capi.GrbImage()
        _check(lib().grbh_viewer_get_image(self._h, name.encode(), C.byref(img)), f"grbh_viewer_get_image({name})")
        return img

    def download_image(self, name) -> np.ndarray:
        """Device image -> numpy (H, W[, C]) of the format's natural integer type."""
        import torch

        img = self.image(name)
        bpp = capi.TEXEL_BYTES[img.format]
        self.sync()
        out = np.empty((img.height, img.width * bpp), np.uint8)
        t = torch.empty((img.height, img.row_pitch), dtype=torch.uint8, device="cuda")
        rt = C.CDLL("libcudart.so.12")
        rt.cudaMemcpy(C.c_void_p(t.data_ptr()), C.c_void_p(img.data), C.c_size_t(img.height * img.row_pitch), 3)
        out[:] = t.cpu().numpy()[:, : img.width * bpp]
        if bpp == 8:
            return out.view(np.uint16).reshape(img.height, img.width, 4)
        if bpp == 2:
            return out.view(np.uint16).reshape(img.height, img.width)
        if img.format == capi.FORMAT_D32_SFLOAT:
            return out.view(np.float32).reshape(img.height, img.width)
        return out.view(np.uint32).reshape(img.height, img.width)

    def buffer(self, name):
        ptr = C.c_void_p()
        size = C.c_uint64()
        _check(lib().grbh_viewer_get_buffer(self._h, name.encode(), C.byref(ptr), C.byref(size)), f"grbh_viewer_get_buffer({name})")
        return ptr.value, size.value

    def download_buffer(self, name, dtype=np.float32, count=None) -> np.ndarray:
        ptr, size = self.buffer(name)
        self.sync()
        n = size if count is None else count * np.dtype(dtype).itemsize
        out = np.empty(n, np.uint8)
        rt = C.CDLL("libcudart.so.12")
        rt.cudaMemcpy(_vp(out), C.c_void_p(ptr), C.c_size_t(n), 2)
        return out.view(dtype)

    def cluster(self):
        p = capi.GrbClusterParameters()
        b = capi.GrbClusterBuffers()
        _check(lib().grbh_viewer_get_cluster(self._h, C.byref(p), C.byref(b)), "grbh_viewer_get_cluster")
        return p, b

    def light_prep(self, capacity=4096):
        recs = np.zeros(capacity, capi.LIGHT_DTYPE)
        model = np.zeros((capacity, 12), np.float32)
        tmask = np.zeros(capacity // 32 + 1, np.uint32)
        zr = np.zeros((capacity + 1, 2), np.uint32)
        n = _check(lib().grbh_viewer_get_light_prep(self._h, _vp(recs), _vp(model), _vp(tmask), _vp(zr), capacity), "grbh_viewer_get_light_prep")
        return n, recs[:n], model[:n], tmask[: (n + 31) // 32], zr[: max(n, 1)]

    def camera(self):
        cam = capi.GrbCamera()
        proj = np.zeros(16, np.float32)
        inv_proj = np.zeros(16, np.float32)
        _check(lib().grbh_viewer_get_camera(self._h, C.byref(cam), _vp(proj), _vp(inv_proj)), "grbh_viewer_get_camera")
        return cam, proj.reshape(4, 4), inv_proj.reshape(4, 4)

    def taa_reprojection(self) -> np.ndarray:
        """clip(now) -> UV(previous frame) of the last rendered frame (4x4, column-major rows as stored)."""
        out = np.zeros(16, np.float32)
        _check(lib().grbh_viewer_get_taa_reprojection(self._h, _vp(out)), "grbh_viewer_get_taa_reprojection")
        return out.reshape(4, 4)

    def measure_row_cost(self) -> np.ndarray:
        """Estimated lighting work (warp instructions) per group of 4 rows of the frame rendered last;
        unsharded viewers only (grbh_viewer_measure_row_cost)."""
        groups = (self.height + 3) // 4
        out = np.zeros(groups, np.uint32)
        _check(lib().grbh_viewer_measure_row_cost(self._h, _vp(out), groups), "grbh_viewer_measure_row_cost")
        return out

    def pass_names(self):
        buf = C.create_string_buffer(4096)
        _check(lib().grbh_viewer_get_pass_names(self._h, buf, 4096), "grbh_viewer_get_pass_names")
        return [n for n in buf.value.decode().split("\n") if n]

    def collect_timings(self):
        names = C.create_string_buffer(4096)
        ms = (C.c_float * 64)()
        cnt = (C.c_int32 * 64)()
        n = _check(lib().grbh_viewer_collect_timings(self._h, names, 4096, ms, cnt, 64), "grbh_viewer_collect_timings")
        nm = [x for x in names.value.decode().split("\n") if x]
        return {nm[i]: (ms[i], cnt[i]) for i in range(min(n, len(nm)))}

    def collect_timeline(self, capacity=4096):
        """[(pass name, begin ms, end ms)] relative to the first recorded pass (viewer created with timestamps=2)."""
        names = C.create_string_buffer(64 * capacity)
        b = (C.c_float * capacity)()
        e = (C.c_float * capacity)()
        n = _check(lib().grbh_viewer_collect_timeline(self._h, names, 64 * capacity, b, e, capacity), "grbh_viewer_collect_timeline")
        nm = [x for x in names.value.decode().split("\n") if x]
        return [(nm[i], b[i], e[i]) for i in range(min(n, len(nm), capacity))]


def load_gtx(path):
    """Granite's texture container (the reference's textures/smaa/*.gtx) -> (VkFormat, numpy (H, W, C) uint8) through the host library's reader."""
    fmt, w, h = C.c_int32(), C.c_int32(), C.c_int32()
    _check(lib().grbh_load_gtx(path.encode(), C.byref(fmt), C.byref(w), C.byref(h), None, C.c_int64(0)), "grbh_load_gtx")
    ch = {capi.FORMAT_R8_UNORM: 1, capi.FORMAT_R8G8_UNORM: 2, capi.FORMAT_R8G8B8A8_UNORM: 4, capi.FORMAT_R8G8B8A8_SRGB: 4}[fmt.value]
    out = np.zeros((h.value, w.value, ch), np.uint8)
    _check(lib().grbh_load_gtx(path.encode(), C.byref(fmt), C.byref(w), C.byref(h), out.ctypes.data_as(C.c_void_p), C.c_int64(out.nbytes)), "grbh_load_gtx")
    return fmt.value, out


def rec709_to_display_primaries(primaries_xy8) -> np.ndarray:
    """The "pq10" pass's primary_conversion (host/post/hdr.cpp, renderer/post/hdr.cpp:580-593) as a column-major 4x4."""
    p = (C.c_float * 8)(*np.asarray(primaries_xy8, np.float32).reshape(-1).tolist())
    out = (C.c_float * 16)()
    _check(lib().grbh_rec709_to_display_primaries(p, out), "grbh_rec709_to_display_primaries")
    return np.array(out, np.float32)


def nccl_unique_id() -> bytes:
    buf = (C.c_uint8 * 128)()
    _check(lib().grbh_nccl_unique_id(buf), "grbh_nccl_unique_id")
    return bytes(buf)
