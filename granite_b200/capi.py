"""ctypes binding of libgranite_b200.so (the C ABI declared in include/granite_b200.h).

PyTorch is used here only as the owner of device memory and streams; every compute call goes
through the extern "C" entry points.  There is no CPU fallback: if the shared library is
missing this module raises at import of `lib()`.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgranite_b200.so")

# GrbFormat (== VkFormat values)
FORMAT_R8_UNORM = 9
FORMAT_R8G8_UNORM = 16
FORMAT_R8G8B8A8_UNORM = 37
FORMAT_R8G8B8A8_SRGB = 43
FORMAT_A2B10G10R10_UNORM = 64
FORMAT_R16G16_SFLOAT = 83
FORMAT_R16G16B16A16_SFLOAT = 97
FORMAT_B10G11R11_UFLOAT = 122
FORMAT_D32_SFLOAT = 126

TEXEL_BYTES = {FORMAT_R8_UNORM: 1, FORMAT_R8G8_UNORM: 2, FORMAT_R8G8B8A8_UNORM: 4, FORMAT_R8G8B8A8_SRGB: 4,
               FORMAT_A2B10G10R10_UNORM: 4, FORMAT_R16G16_SFLOAT: 4, FORMAT_R16G16B16A16_SFLOAT: 8,
               FORMAT_B10G11R11_UFLOAT: 4, FORMAT_D32_SFLOAT: 4}


class GrbImage(C.Structure):
    _fields_ = [("data", C.c_void_p), ("width", C.c_int32), ("height", C.c_int32),
                ("row_pitch", C.c_int32), ("format", C.c_int32)]


class GrbRows(C.Structure):
    _fields_ = [("y0", C.c_int32), ("y1", C.c_int32)]


class GrbBloomTailOptions(C.Structure):
    _fields_ = [("u0", C.c_void_p), ("u0_rows", GrbRows), ("peer_flags", C.c_void_p), ("peer_count", C.c_int32), ("peer_epoch", C.c_uint32),
                ("max_ctas", C.c_int32)]


class GrbPositionalLight(C.Structure):
    _fields_ = [("color", C.c_float * 3), ("spot_scale_bias", C.c_uint16 * 2),
                ("position", C.c_float * 3), ("offset_radius", C.c_uint16 * 2),
                ("direction", C.c_float * 3), ("inv_radius", C.c_float)]


LIGHT_DTYPE = np.dtype([("color", "<f4", 3), ("spot_scale_bias", "<u2", 2), ("position", "<f4", 3),
                        ("offset_radius", "<u2", 2), ("direction", "<f4", 3), ("inv_radius", "<f4")])
assert C.sizeof(GrbPositionalLight) == 48 and LIGHT_DTYPE.itemsize == 48


class GrbClusterParameters(C.Structure):
    _fields_ = [("transform", C.c_float * 16), ("clip_scale", C.c_float * 4),
                ("camera_base", C.c_float * 3), ("camera_front", C.c_float * 3),
                ("xy_scale", C.c_float * 2), ("resolution_xy", C.c_int32 * 2),
                ("inv_resolution_xy", C.c_float * 2), ("num_lights", C.c_int32),
                ("num_lights_32", C.c_int32), ("z_max_index", C.c_int32), ("z_scale", C.c_float)]


class GrbCamera(C.Structure):
    _fields_ = [("view", C.c_float * 16), ("view_projection", C.c_float * 16),
                ("inv_view_projection", C.c_float * 16), ("camera_position", C.c_float * 3),
                ("camera_front", C.c_float * 3), ("z_near", C.c_float), ("z_far", C.c_float)]


class GrbClusterBuffers(C.Structure):
    _fields_ = [("lights", C.c_void_p), ("model", C.c_void_p), ("type_mask", C.c_void_p),
                ("z_ranges", C.c_void_p), ("transformed_spots", C.c_void_p), ("cull_setup", C.c_void_p),
                ("bitmask", C.c_void_p), ("cluster_range", C.c_void_p), ("resolution_z", C.c_int32)]


class GrbGBuffer(C.Structure):
    _fields_ = [("albedo", GrbImage), ("normal", GrbImage), ("pbr", GrbImage), ("depth", GrbImage),
                ("directional_color", C.c_float * 3), ("directional_direction", C.c_float * 3), ("emissive", GrbImage)]


class GrbFogParameters(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("depth", C.c_int32), ("dither_offset", C.c_int32),
                ("slice_z_log2_scale", C.c_float), ("density_mod", C.c_float), ("in_scatter_strength", C.c_float)]


class GrbLightShadows(C.Structure):
    _fields_ = [("transforms", C.c_void_p), ("maps", C.c_void_p), ("resolution", C.c_int32), ("pcf_wide", C.c_int32)]


ENTRY_POINTS = [
    "grb_abi_version", "grb_init", "grb_last_error_string",
    "grb_cluster_spot_transform", "grb_cluster_cull_setup", "grb_cluster_binning", "grb_cluster_binning_rows", "grb_cluster_z_range",
    "grb_cluster_build", "grb_cluster_decal_binning", "grb_fog_light_density", "grb_fog_accumulate", "grb_deferred_lighting", "grb_deferred_lighting_blocks", "grb_deferred_lighting_scheduled", "grb_deferred_lighting_shadowed", "grb_lighting_schedule_bytes", "grb_debug_cluster_indices", "grb_lighting_row_cost",
    "grb_bloom_threshold", "grb_bloom_threshold_downsample", "grb_bloom_threshold_downsample_to_peers", "grb_bloom_downsample", "grb_bloom_downsample_to_peers", "grb_peer_wait", "grb_bloom_upsample", "grb_bloom_upsample_exact",
    "grb_luminance", "grb_luminance_grid", "grb_luminance_finalize", "grb_bloom_tail", "grb_bloom_tail_ex", "grb_tonemap",
    "grb_pq10_encode", "grb_smaa_edge_detection", "grb_smaa_blend_weights", "grb_smaa_neighborhood_blend", "grb_smaa_edge_detection_to_peers", "grb_fsr_easu_constants", "grb_fsr_upscale", "grb_fsr_sharpen", "grb_fxaa", "grb_taa_resolve", "grb_taa_resolve_to_peers",
]

_lib = None


class GrbError(RuntimeError):
    pass


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GrbError(f"{LIB_PATH} is missing: run `python -m granite_b200.build` "
                           "(there is no CPU fallback for this path)")
        _lib = C.CDLL(LIB_PATH)
        _lib.grb_last_error_string.restype = C.c_char_p
        P = C.c_void_p
        I = C.c_int32
        F = C.c_float
        IMG = C.POINTER(GrbImage)
        sig = {
            "grb_cluster_spot_transform": [C.POINTER(GrbCamera), C.POINTER(GrbClusterParameters), C.POINTER(GrbClusterBuffers), P],
            "grb_cluster_cull_setup": [C.POINTER(GrbCamera), C.POINTER(GrbClusterParameters), C.POINTER(GrbClusterBuffers), P],
            "grb_cluster_binning": [C.POINTER(GrbClusterParameters), C.POINTER(GrbClusterBuffers), P],
            "grb_cluster_binning_rows": [C.POINTER(GrbClusterParameters), C.POINTER(GrbClusterBuffers), I, I, P],
            "grb_cluster_z_range": [C.POINTER(GrbClusterBuffers), I, P],
            "grb_cluster_build": [C.POINTER(GrbCamera), C.POINTER(GrbClusterParameters), C.POINTER(GrbClusterBuffers), P],
            "grb_deferred_lighting": [C.POINTER(GrbGBuffer), C.POINTER(GrbCamera), C.POINTER(GrbClusterParameters),
                                      C.POINTER(GrbClusterBuffers), IMG, GrbRows, P],
            "grb_deferred_lighting_blocks": [C.POINTER(GrbGBuffer), C.POINTER(GrbCamera), C.POINTER(GrbClusterParameters),
                                             C.POINTER(GrbClusterBuffers), IMG, GrbRows, P],
            "grb_deferred_lighting_scheduled": [C.POINTER(GrbGBuffer), C.POINTER(GrbCamera), C.POINTER(GrbClusterParameters),
                                                C.POINTER(GrbClusterBuffers), IMG, GrbRows, P, P],
            "grb_debug_cluster_indices": [IMG, C.POINTER(GrbCamera), C.POINTER(GrbClusterParameters), P, P, GrbRows, P],
            "grb_lighting_row_cost": [IMG, C.POINTER(GrbCamera), C.POINTER(GrbClusterParameters), C.POINTER(GrbClusterBuffers), GrbRows, P, P],
            "grb_bloom_threshold": [IMG, P, IMG, GrbRows, P],
            "grb_bloom_threshold_downsample": [IMG, P, IMG, IMG, GrbRows, P],
            "grb_bloom_downsample": [IMG, IMG, F, IMG, GrbRows, P],
            "grb_bloom_upsample": [IMG, IMG, GrbRows, P],
            "grb_bloom_upsample_exact": [IMG, IMG, GrbRows, P],
            "grb_luminance": [IMG, P, F, F, F, P],
            "grb_luminance_grid": [IMG, P, GrbRows, P],
            "grb_luminance_finalize": [P, I, I, P, F, F, F, P],
            "grb_bloom_tail": [IMG, IMG, IMG, IMG, IMG, F, P, F, F, F, IMG, IMG, P],
            "grb_bloom_tail_ex": [IMG, IMG, IMG, IMG, IMG, F, P, F, F, F, IMG, IMG, P, P],
            "grb_tonemap": [IMG, IMG, P, F, IMG, GrbRows, P],
            "grb_pq10_encode": [IMG, IMG, P, F, F, F, IMG, GrbRows, P],
            "grb_smaa_edge_detection": [IMG, I, IMG, GrbRows, P],
            "grb_smaa_blend_weights": [IMG, IMG, IMG, I, IMG, GrbRows, P],
            "grb_smaa_neighborhood_blend": [IMG, IMG, IMG, GrbRows, P],
            "grb_smaa_edge_detection_to_peers": [IMG, I, IMG, P, C.POINTER(GrbRows), P, I, I, C.c_uint32, P, GrbRows, P],
            "grb_fxaa": [IMG, IMG, GrbRows, P],
            "grb_taa_resolve": [IMG, IMG, IMG, IMG, P, I, IMG, IMG, GrbRows, P],
            "grb_taa_resolve_to_peers": [IMG, IMG, IMG, IMG, P, I, IMG, IMG, P, P, I, I, C.c_uint32, P, GrbRows, GrbRows, P],
        }
        for name, args in sig.items():
            fn = getattr(_lib, name)
            fn.argtypes = args
            fn.restype = I
        _lib.grb_lighting_schedule_bytes.argtypes = [I]
        _lib.grb_lighting_schedule_bytes.restype = C.c_uint64
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().grb_last_error_string()
        raise GrbError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")


_initialised_devices: set[int] = set()


def init() -> None:
    """grb_init() on the current CUDA device (once per device)."""
    import torch

    dev = torch.cuda.current_device()
    if dev not in _initialised_devices:
        check(lib().grb_init(), "grb_init")
        _initialised_devices.add(dev)


def image(t, fmt: int) -> GrbImage:
    """Wrap a contiguous CUDA tensor laid out (H, W[, C]) as a GrbImage of format `fmt`."""
    assert t.is_cuda and t.is_contiguous()
    h, w = int(t.shape[0]), int(t.shape[1])
    bpp = TEXEL_BYTES[fmt]
    row = t.stride(0) * t.element_size()
    assert row == w * bpp, (row, w, bpp)
    return GrbImage(t.data_ptr(), w, h, row, fmt)


def rows(r=None) -> GrbRows:
    return GrbRows(0, 0) if r is None else GrbRows(int(r[0]), int(r[1]))


def stream_ptr():
    import torch

    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
