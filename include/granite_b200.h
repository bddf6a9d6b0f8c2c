/*
 * granite_b200.h -- C ABI of the B200-native executor for Granite's clustered deferred
 * lighting + HDR post chain (libgranite_b200.so).
 *
 * This is the drop-in boundary: every entry point replaces one shader dispatch / draw that
 * the reference's pass builders record into a Vulkan::CommandBuffer.  The reference has no
 * FFI for this path (the "binding" is set_program + push_constants + dispatch on GLSL), so
 * each declaration cites the builder code (file:line, relative to the Granite tree at
 * 7c59ad8089) whose push-constant block and bindings it mirrors.  INTEGRATION.md shows the
 * build_render_pass lambdas a maintainer would write against these.
 *
 * Conventions
 *   - plain C types only; all pointers are DEVICE pointers owned by the caller (the render
 *     graph owns every image/buffer, renderer/render_graph.hpp:988-992); nothing here
 *     allocates, frees or synchronises the device;
 *   - `stream` is a cudaStream_t passed as void*; the caller has made the right device
 *     current (the reference records on whatever queue the graph picked);
 *   - every function returns 0 (GRB_OK) or a negative GrbResult; the CUDA error text of the
 *     last failure on the calling thread is available from grb_last_error_string();
 *   - re-entrant and thread-safe for distinct streams (callbacks run on arbitrary worker
 *     threads, renderer/render_graph.cpp:2384-2397);
 *   - matrices are column-major float[16] exactly as muglm::mat4 lays them out;
 *   - images are row-major, `row_pitch` in BYTES (multiple of the texel size);
 *   - `rows` selects the OUTPUT rows [y0, y1) a call produces -- the screen-row shard of a
 *     multi-GPU frame; {0, 0} means the whole image.
 */
#ifndef GRANITE_B200_H_
#define GRANITE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GRB_ABI_VERSION 1

typedef enum GrbResult
{
	GRB_OK = 0,
	GRB_ERR_INVALID_ARGUMENT = -1,
	GRB_ERR_UNSUPPORTED_FORMAT = -2,
	GRB_ERR_CUDA = -3,
	GRB_ERR_NOT_INITIALIZED = -4
} GrbResult;

/* VkFormat values the path uses, kept numerically identical to Vulkan's so the graph layer
 * can pass AttachmentInfo::format straight through (renderer/render_graph.hpp:154-167). */
typedef enum GrbFormat
{
	GRB_FORMAT_UNDEFINED = 0,
	GRB_FORMAT_R8_UNORM = 9,
	GRB_FORMAT_R8G8_UNORM = 16,
	GRB_FORMAT_R8G8B8A8_UNORM = 37,
	GRB_FORMAT_R8G8B8A8_SRGB = 43,
	GRB_FORMAT_A2B10G10R10_UNORM_PACK32 = 64,
	GRB_FORMAT_R16G16_SFLOAT = 83,
	GRB_FORMAT_R16G16B16A16_SFLOAT = 97,
	GRB_FORMAT_B10G11R11_UFLOAT_PACK32 = 122,
	GRB_FORMAT_D32_SFLOAT = 126
} GrbFormat;

typedef struct GrbImage
{
	void *data;
	int32_t width;
	int32_t height;
	int32_t row_pitch; /* bytes */
	int32_t format;    /* GrbFormat */
} GrbImage;

typedef struct GrbRows
{
	int32_t y0, y1;
} GrbRows;

/* renderer/lights/light_info.hpp:35-44 PositionalFragmentInfo == GLSL PositionalLightInfo
 * (assets/shaders/lights/clusterer_data.h:10-18). 48 bytes. */
typedef struct GrbPositionalLight
{
	float color[3];
	uint16_t spot_scale_bias[2]; /* fp16 x2 */
	float position[3];
	uint16_t offset_radius[2];   /* fp16 x2 */
	float direction[3];
	float inv_radius;
} GrbPositionalLight;

/* math/render_parameters.hpp:90-108 ClustererParametersBindless (fields the path reads). */
typedef struct GrbClusterParameters
{
	float transform[16];
	float clip_scale[4];
	float camera_base[3];
	float camera_front[3];
	float xy_scale[2];
	int32_t resolution_xy[2];
	float inv_resolution_xy[2];
	int32_t num_lights;
	int32_t num_lights_32;
	int32_t z_max_index;
	float z_scale;
} GrbClusterParameters;

/* Camera block: the RenderParameters fields (math/render_parameters.hpp:37-59) that
 * clusterer.cpp:1469-1509 and renderer.cpp:1073-1121 push to the shaders. */
typedef struct GrbCamera
{
	float view[16];
	float view_projection[16];
	float inv_view_projection[16];
	float camera_position[3];
	float camera_front[3];
	float z_near;
	float z_far;
} GrbCamera;

/* The light-cluster structure ("cluster-bitmask", "cluster-range", "cluster-transforms",
 * "cluster-cull-setup", "cluster-transformed-spot": renderer/lights/clusterer.cpp:1575-1613).
 * `lights`, `model`, `type_mask` are the three members of ClustererBindlessTransforms the
 * path reads (math/render_parameters.hpp:155-162), passed as separate device arrays. */
typedef struct GrbClusterBuffers
{
	const GrbPositionalLight *lights; /* num_lights */
	const float *model;               /* num_lights x 12: mat_affine rows */
	const uint32_t *type_mask;        /* num_lights_32 words, bit = 1 => point light */
	const uint32_t *z_ranges;         /* max(num_lights,1) x uvec2, host-computed (clusterer.cpp:1322-1346) */
	float *transformed_spots;         /* num_lights x 6 vec4 */
	float *cull_setup;                /* num_lights x 32 vec4 */
	uint32_t *bitmask;                /* res_x * res_y * num_lights_32 */
	uint32_t *cluster_range;          /* res_z x uvec2 */
	int32_t resolution_z;
} GrbClusterBuffers;

/* ---- library ---- */
int32_t grb_abi_version(void);
/* Uploads the constant tables (sRGB decode LUT) to the CURRENT device. Call once per device
 * before any other entry point; idempotent and thread-safe. */
int32_t grb_init(void);
const char *grb_last_error_string(void);

/* ---- clusterer: replaces LightClusterer::build_cluster_bindless_gpu
 * (renderer/lights/clusterer.cpp:1463-1573) ---- */
/* K1 clusterer_bindless_spot_transform.comp; push block clusterer.cpp:1477-1493. */
int32_t grb_cluster_spot_transform(const GrbCamera *cam, const GrbClusterParameters *params,
                                   const GrbClusterBuffers *buf, void *stream);
/* K2 clusterer_bindless_setup.comp; push block clusterer.cpp:1502-1509. */
int32_t grb_cluster_cull_setup(const GrbCamera *cam, const GrbClusterParameters *params,
                               const GrbClusterBuffers *buf, void *stream);
/* K3 clusterer_bindless_binning.comp (SUBGROUPS=1, 32-wide: clusterer.cpp:1519-1561). */
int32_t grb_cluster_binning(const GrbClusterParameters *params, const GrbClusterBuffers *buf, void *stream);
/* The same for tile rows [tile_y0, tile_y1) only (widened to whole blocks of 4 tile rows; an empty range = all rows):
 * a rank of a row-sharded frame bins the tile rows its own pixel rows fall into, the other rows of the bitmask are
 * left as they are. */
int32_t grb_cluster_binning_rows(const GrbClusterParameters *params, const GrbClusterBuffers *buffers, int32_t tile_y0,
                                 int32_t tile_y1, void *stream);
/* K4 clusterer_bindless_z_range[_opt].comp; push block clusterer.cpp:1291-1300. */
int32_t grb_cluster_z_range(const GrbClusterBuffers *buf, int32_t num_ranges, void *stream);
/* All four in the order build_cluster_bindless_gpu records them. */
int32_t grb_cluster_build(const GrbCamera *cam, const GrbClusterParameters *params,
                          const GrbClusterBuffers *buf, void *stream);

/* Volumetric-decal binning over the clusterer's tile grid: LightClusterer::update_bindless_mask_buffer_decal_gpu
 * (clusterer.cpp:1391-1461) + clusterer_bindless_binning_decal.comp.  mvps: num_decals x mat4 (column-major, device) =
 * view_projection * decal world transform (clusterer.cpp:1406-1410); boxes: scratch, num_decals x 4 floats (the decals'
 * screen-space bounding boxes); bitmask: resolution_x * resolution_y * ((num_decals + 31) / 32) words,
 * [(tile_y * resolution_x + tile_x) * num_decals_32 + decal / 32].  The decals' Z-slice ranges go through
 * grb_cluster_z_range like the lights' (clusterer.cpp:1371-1389).  num_decals == 0: nothing is launched. */
int32_t grb_cluster_decal_binning(const GrbClusterParameters *params, const float *mvps, int32_t num_decals, float *boxes, uint32_t *bitmask,
                                  void *stream);

/* Volumetric fog, accumulation pass: VolumetricFog::build_fog (renderer/lights/volumetric_fog.cpp:236-254) + fog_accumulate.comp.
 * light_density / fog: device pointers to R16G16B16A16_SFLOAT volumes of width x height x depth texels (x fastest, then y, then
 * slices), distinct and 8-byte aligned; light_density = (in-scattered light rgb, optical depth) per froxel, as the reference's
 * "volumetric-fog-inscatter" image holds it (grb_fog_light_density below, or the caller's own); fog = (light accumulated front to
 * back, transmittance). */
/* Volumetric fog, light-density pass: VolumetricFog::build_light_density (volumetric_fog.cpp:142-228) + fog_light_density.comp in
 * its base variant: constant medium (no FOG_REGIONS), no TEMPORAL_REPROJECTION (the first frame of the reference), no
 * FLOOR_LIGHTING, unshadowed directional and clustered positional lights.  projection16 / inv_projection16: the camera's
 * (z_transform and xy_scale come from them, :161-168); slice_extents: depth floats (compute_slice_extents, :115-126);
 * dither_lut: N layers of 128 x 128 R8G8B8A8_UNORM texels (build_dither_lut, :356-395), layer fog->dither_offset is read;
 * light_density: depth x height x width R16G16B16A16_SFLOAT, 8-byte aligned = (in-scattered light, fog albedo). */
typedef struct GrbFogParameters
{
	int32_t width, height, depth; /* VolumetricFog::set_resolution */
	int32_t dither_offset;
	float slice_z_log2_scale;     /* 1 / log2(1 + z_range) (:87-91) */
	float density_mod;            /* set_fog_density */
	float in_scatter_strength;    /* inscatter_mod */
} GrbFogParameters;
int32_t grb_fog_light_density(const GrbFogParameters *fog, const GrbCamera *cam, const float *projection16, const float *inv_projection16,
                              const GrbClusterParameters *params, const GrbClusterBuffers *buf, const float *directional_color3,
                              const float *directional_direction3, const float *slice_extents, const void *dither_lut, void *light_density,
                              void *stream);
int32_t grb_fog_accumulate(const void *light_density, int32_t width, int32_t height, int32_t depth, void *fog, void *stream);

/* ---- deferred lighting: replaces DeferredLightRenderer::render_light
 * (renderer/renderer.cpp:1004-1156): directional.frag + clustering.frag, both additively
 * blended into HDR-main, sky (depth == 0) skipped. ---- */
typedef struct GrbGBuffer
{
	GrbImage albedo;   /* R8G8B8A8_SRGB       (scene_viewer_application.cpp:880-900) */
	GrbImage normal;   /* A2B10G10R10_UNORM */
	GrbImage pbr;      /* R8G8_UNORM */
	GrbImage depth;    /* D32_SFLOAT, reverse-Z, 0 = far */
	float directional_color[3];     /* DirectionalLightPush, renderer.cpp:1073-1103 */
	float directional_direction[3];
	/* Initial contents of the blend destination ("emissive", B10G11R11_UFLOAT).  data == NULL:
	 * `hdr` itself holds them (HDR-main aliases emissive in the reference) and is updated in place. */
	GrbImage emissive;
} GrbGBuffer;

/* hdr: B10G11R11_UFLOAT; read-modify-write when gbuffer->emissive.data is NULL ("HDR-main"
 * aliases "emissive", scene_viewer_application.cpp:956-963), write-only otherwise.
 * "renderTargetFp16" (scene_viewer_application.cpp:880-884): hdr (and emissive) may be R16G16B16A16_SFLOAT instead -- each of
 * the two additive blends then rounds to fp16 (RNE) and alpha passes through; the pass runs on the generic one-pixel kernel.
 * grb_bloom_threshold, grb_tonemap and grb_taa_resolve accept an R16G16B16A16_SFLOAT hdr likewise (TAA's own output stays
 * B10G11R11, temporal.cpp:209-212); the fused / tile forms (grb_bloom_threshold_downsample*) take B10G11R11 only and
 * return GRB_ERR_UNSUPPORTED_FORMAT, on which the caller issues the unfused pair. */
int32_t grb_deferred_lighting(const GrbGBuffer *gbuffer, const GrbCamera *cam,
                              const GrbClusterParameters *params, const GrbClusterBuffers *buf,
                              const GrbImage *hdr, GrbRows rows, void *stream);
/* Same pass as a plain grid of short-lived CTAs (no persistent CTAs, no schedule): the form for callers whose
 * other streams must get SMs while lighting runs, e.g. every rank of a row-sharded frame (granite_b200/csrc/
 * grb_lighting.cu).  Within the same parity bar; not bit-identical to the persistent form. */
int32_t grb_deferred_lighting_blocks(const GrbGBuffer *gbuffer, const GrbCamera *cam, const GrbClusterParameters *params,
                                     const GrbClusterBuffers *buf, const GrbImage *hdr, GrbRows rows, void *stream);
/* Same pass with a caller-owned SCHEDULE buffer: grb_lighting_schedule_bytes(image height) bytes of
 * device memory, zero-initialised once and then left alone, used by one stream at a time.  Each
 * launch measures what every row of pixel blocks cost and leaves them sorted by falling cost; the
 * next launch hands the rows out in that order (longest first), so the pass no longer ends with a
 * few warps holding the expensive blocks.  Results are identical with or without it.  A null
 * schedule is allowed (raster order). */
uint64_t grb_lighting_schedule_bytes(int32_t height);
int32_t grb_deferred_lighting_scheduled(const GrbGBuffer *gbuffer, const GrbCamera *cam, const GrbClusterParameters *params,
                                        const GrbClusterBuffers *buffers, const GrbImage *hdr_inout, GrbRows rows, void *schedule,
                                        void *stream);

/* ---- shadowed positional lights: clustering.frag with POSITIONAL_LIGHTS_SHADOW and the PCF sampler
 * (renderer.cpp:369,1126; assets/shaders/lights/point.h:45-74, spot.h:51-77, pcf.h:98-99).  The shadow maps are
 * INPUTS, as the G-buffer is: what LightClusterer::render_shadow (clusterer.cpp:206-330) rasterised, one D16_UNORM
 * image per light (clusterer.cpp:397-407), bound bindlessly by update_bindless_descriptors (clusterer.cpp:1209-1252).
 * Sampling follows StockSampler::LinearShadow (vulkan/device.cpp:1086-1088: GREATER_OR_EQUAL, linear, clamp to edge)
 * as the Vulkan specification defines comparison filtering, cube maps with edge handling across faces. ---- */
typedef struct GrbLightShadows
{
	/* num_lights x 16 floats, device: ClustererBindlessTransforms::shadow[index], column-major.  Spot light: bias *
	 * projection * view (clusterer.cpp:467-474); point light: column 0 = (proj[2].zw, proj[3].zw) (clusterer.cpp:518-521). */
	const float *transforms;
	/* num_lights device pointers, device array: resolution^2 D16 texels for a spot light, 6 x resolution^2 (layers
	 * +X -X +Y -Y +Z -Z) for a point light; a null entry = the light casts no shadow (its falloff stays 1). */
	const void *const *maps;
	int32_t resolution; /* LightClusterer::set_shadow_resolution (clusterer.cpp:78-81), 512 by default */
	int32_t pcf_wide;   /* != 0: SHADOW_MAP_PCF_KERNEL_WIDE (config "PCFKernelWide", renderer.cpp:380-381): spot lights filter with the
	                     * 6 x 6 kernel of pcf.h:7-80 instead of the sampler's 2 x 2; point lights keep the cube sampler */
} GrbLightShadows;
/* The lighting pass with shadowed positional lights; every other argument as grb_deferred_lighting. */
int32_t grb_deferred_lighting_shadowed(const GrbGBuffer *gbuffer, const GrbCamera *cam, const GrbClusterParameters *params,
                                       const GrbClusterBuffers *buf, const GrbLightShadows *shadows, const GrbImage *hdr, GrbRows rows,
                                       void *stream);

/* Diagnostic: the (tile index, Z slice) the lighting kernel addresses for every pixel, -1 for sky
 * (clusterer_bindless.h:39-47).  Same device function as grb_deferred_lighting uses; exists so
 * the "bit-exact cluster indices" contract can be checked directly. */
int32_t grb_debug_cluster_indices(const GrbImage *depth, const GrbCamera *cam, const GrbClusterParameters *params,
                                  int32_t *out_tile, int32_t *out_z, GrbRows rows, void *stream);

/* Work estimate of grb_deferred_lighting per group of 4 pixel rows (rows.y0 + 4 i ...), in warp
 * instructions: the same cluster walk (clusterer_bindless.h:39-81) without shading.  The
 * reference has no equivalent -- it never splits a frame; here the figure weighs the screen-row
 * bands of a multi-GPU run (SURVEY.md section 8e).  cost_per_4_rows: device array of
 * ceil(rows / 4) uint32, overwritten. */
int32_t grb_lighting_row_cost(const GrbImage *depth, const GrbCamera *cam, const GrbClusterParameters *params,
                              const GrbClusterBuffers *buf, GrbRows rows, uint32_t *cost_per_4_rows, void *stream);

/* ---- HDR post chain: replaces the "bloom-compute" and "tonemap" passes
 * (renderer/post/hdr.cpp:308-400) ---- */
/* K7 bloom_threshold.comp; hdr.cpp:115-144. luminance: device float[3] {avg_log, avg_lin,
 * avg_inv_lin} or NULL for DYNAMIC_EXPOSURE=0. */
int32_t grb_bloom_threshold(const GrbImage *hdr, const float *luminance, const GrbImage *out,
                            GrbRows rows, void *stream);
/* K8 bloom_downsample.comp; hdr.cpp:146-187. history (NULL => FEEDBACK=0) is last frame's
 * image of the same size; lerp = 1 - 0.001^frame_time. */
int32_t grb_bloom_downsample(const GrbImage *in, const GrbImage *history, float lerp,
                             const GrbImage *out, GrbRows rows, void *stream);
/* K7 + the first K8 dispatch in one pass: d0 = downsample(threshold(hdr)) with the 1/2-resolution
 * threshold image kept in shared memory (TMA-loaded HDR tiles; granite_b200/csrc/grb_post_tiles.cu).
 * threshold_out may be NULL; when given, its rows 2*rows.y0 .. 2*rows.y1 are written too (within 1 fp16
 * ulp of grb_bloom_threshold: FMA, one reciprocal, hardware log2).  Needs exact 2:1 size steps hdr -> threshold -> d0 and 16-byte aligned rows;
 * otherwise returns GRB_ERR_UNSUPPORTED_FORMAT and the caller issues the two calls above.
 * Replaces hdr.cpp:355-356 (bloom_threshold_build_compute + bloom_downsample_build_compute). */
int32_t grb_bloom_threshold_downsample(const GrbImage *hdr, const float *luminance, const GrbImage *threshold_out,
                                       const GrbImage *d0, GrbRows rows, void *stream);
/* K8 fused with the exchange a row-sharded frame needs after it (SURVEY.md section 8e): the band
 * rows [rows.y0, rows.y1) of the 1/4-resolution level are stored into that image on EVERY rank --
 * peer_images[r] is the base address, valid on this device, of rank r's image (cudaIpc-mapped
 * peer memory over NVLink / NVSwitch; one entry is this rank's own image), all with out_layout's
 * size and pitch -- and then flags[flag_index] = epoch is release-stored into every rank's flag
 * array.  scratch_counter: one zero-initialised uint32 in local device memory.  No reference
 * equivalent (the reference never splits a frame). */
#define GRB_MAX_PEERS 8
int32_t grb_bloom_downsample_to_peers(const GrbImage *in, const GrbImage *out_layout, void *const *peer_images,
                                      uint32_t *const *peer_flags, int32_t peer_count, int32_t flag_index, uint32_t epoch,
                                      uint32_t *scratch_counter, GrbRows rows, void *stream);
/* grb_bloom_threshold_downsample with the same exchange fused in (threshold tile in shared memory, d0
 * band stored to every rank, flags raised).  Same eligibility rule; GRB_ERR_UNSUPPORTED_FORMAT otherwise. */
int32_t grb_bloom_threshold_downsample_to_peers(const GrbImage *hdr, const float *luminance, const GrbImage *d0_layout,
                                                void *const *peer_images, uint32_t *const *peer_flags, int32_t peer_count,
                                                int32_t flag_index, uint32_t epoch, uint32_t *scratch_counter, GrbRows rows,
                                                void *stream);
/* Stream-ordered wait until local_flags[0..count) have all reached `epoch` (acquire, system scope). */
int32_t grb_peer_wait(const uint32_t *local_flags, int32_t count, uint32_t epoch, void *stream);
/* K9 bloom_upsample.comp; hdr.cpp:189-216. */
int32_t grb_bloom_upsample(const GrbImage *in, const GrbImage *out, GrbRows rows, void *stream);
/* Same, never through the tile kernel: the shader's arithmetic statement for statement at every size (bit-exact to the
 * oracle; the tile kernel is within 1 fp16 ulp). */
int32_t grb_bloom_upsample_exact(const GrbImage *in, const GrbImage *out, GrbRows rows, void *stream);
/* K10 luminance.comp; hdr.cpp:68-98 (size = d3 / 2, lerp = 1 - 0.5^frame_time, clamp [-3,2]).
 * Single-device form: reads d3, updates luminance[3] in place. */
int32_t grb_luminance(const GrbImage *d3, float *luminance, float lerp, float min_loglum,
                      float max_loglum, void *stream);
/* Sharded form of K10 for row-sharded frames: step 1 samples the (w/2 x h/2) grid rows
 * [rows.y0, rows.y1) into `grid` (float, size_x*size_y, other rows untouched -- zero them
 * once so an all-reduce(sum) across ranks assembles the grid exactly); step 2 reduces a
 * complete grid in the shader's association order and updates luminance[3]. */
int32_t grb_luminance_grid(const GrbImage *d3, float *grid, GrbRows rows, void *stream);
int32_t grb_luminance_finalize(const float *grid, int32_t size_x, int32_t size_y, float *luminance,
                               float lerp, float min_loglum, float max_loglum, void *stream);
/* Everything of "bloom-compute" below 1/4 resolution in ONE cooperative launch with grid barriers between
 * the levels: d1, d2, d3 (history / lerp_d3 as in grb_bloom_downsample), the luminance update (luminance may
 * be NULL), u2, u1 (hdr.cpp:357-376).  Bit-identical to the six separate calls on their generic kernels.
 * GRB_ERR_UNSUPPORTED_FORMAT when the device cannot launch cooperatively: issue the six calls instead. */
int32_t grb_bloom_tail(const GrbImage *d0, const GrbImage *d1, const GrbImage *d2, const GrbImage *d3,
                       const GrbImage *history, float lerp_d3, float *luminance, float lerp_luminance,
                       float min_loglum, float max_loglum, const GrbImage *u2, const GrbImage *u1, void *stream);

/* The same launch with optional extras.  u0 / u0_rows: also compute those rows of u0 from u1 (the last upsample of
 * hdr.cpp:376) after u1.  peer_flags / peer_count / peer_epoch: row-sharded frames whose d0 was assembled by
 * grb_bloom_*_to_peers -- the kernel itself waits (bounded) until every rank's flag reached peer_epoch, replacing
 * grb_peer_wait.  max_ctas > 0 caps the launch so that it can run beside a kernel that fills the other SMs. */
typedef struct GrbBloomTailOptions
{
	const GrbImage *u0;
	GrbRows u0_rows;
	const uint32_t *peer_flags;
	int32_t peer_count;
	uint32_t peer_epoch;
	int32_t max_ctas;
} GrbBloomTailOptions;
int32_t grb_bloom_tail_ex(const GrbImage *d0, const GrbImage *d1, const GrbImage *d2, const GrbImage *d3,
                          const GrbImage *history, float lerp_d3, float *luminance, float lerp_luminance,
                          float min_loglum, float max_loglum, const GrbImage *u2, const GrbImage *u1,
                          const GrbBloomTailOptions *options, void *stream);
/* K11 tonemap.frag; hdr.cpp:283-306. out: R8G8B8A8_SRGB (or _UNORM: stores linear). */
int32_t grb_tonemap(const GrbImage *hdr, const GrbImage *bloom, const float *luminance,
                    float dynamic_exposure, const GrbImage *out, GrbRows rows, void *stream);

/* ---- post AA ---- */
/* HDR10 output encoding: pq10_encode.frag, the "pq10" pass of setup_hdr10_pq_encoding (renderer/post/hdr.cpp:595-658).
 * hdr: linear scene colour (B10G11R11); ui: R8G8B8A8_UNORM layer, alpha = share of the scene that shows through;
 * primary_conversion16: column-major mat4 (upper 3x3 used) Rec.709 -> display primaries (hdr.cpp:580-593);
 * out: A2B10G10R10_UNORM_PACK32 holding ST.2084 (PQ) code values, alpha = 1. */
int32_t grb_pq10_encode(const GrbImage *hdr, const GrbImage *ui, const float *primary_conversion16, float hdr_pre_exposure,
                        float ui_pre_exposure, float max_light_level, const GrbImage *out, GrbRows rows, void *stream);
/* SMAA 1x (renderer/post/smaa.cpp:32-209; assets/shaders/post/SMAA.hlsl through smaa_edge_detection / smaa_blend_weight /
 * smaa_neighbor_blend .vert + .frag).  quality = SMAA_QUALITY 0..3 = presets Low / Medium / High / Ultra (SMAA.hlsl:304-324).
 * color: the tonemapped 8-bit image, read as UNORM whatever its format says (smaa.cpp:124 set_unorm_texture);
 * edges: R8G8_UNORM; weights: R8G8B8A8_UNORM; area (160x560 R8G8_UNORM) and search (64x16 R8_UNORM) are the payloads
 * of the reference's textures/smaa/{area,search}.gtx (SMAA's precomputed lookup tables), supplied by the caller;
 * out: R8G8B8A8_SRGB (the blended colour is decoded to linear and encoded on store, SMAA_TARGET_SRGB) or _UNORM.
 * The reference's depth mask between the first two passes (smaa.cpp:101-118) keeps every pixel (both passes emit depth
 * 0 = the clear value), so there is nothing to emulate: pixels without an edge get zero weights from the second call. */
int32_t grb_smaa_edge_detection(const GrbImage *color, int32_t quality, const GrbImage *edges, GrbRows rows, void *stream);
int32_t grb_smaa_blend_weights(const GrbImage *edges, const GrbImage *area, const GrbImage *search, int32_t quality,
                               const GrbImage *weights, GrbRows rows, void *stream);
int32_t grb_smaa_neighborhood_blend(const GrbImage *color, const GrbImage *weights, const GrbImage *out, GrbRows rows, void *stream);
/* grb_smaa_edge_detection for one rank of a row-sharded frame, with the edge exchange fused in.  The edges of `rows` (this
 * rank's band) are computed once; each texel of row y is stored into the edge slot of every rank r with y in
 * peer_rows[r] -- peer_images[r], valid on this device, all with edges_layout's size and pitch (its data pointer is not
 * written) -- and then peer_flags[r][flag_index] = epoch is release-stored on EVERY rank, also on ranks that received
 * no rows, as in grb_bloom_downsample_to_peers.  peer_rows[flag_index] (this rank's own slot) must equal rows; every
 * peer_rows[r] must lie inside rows (empty: y0 == y1).  Launches nothing on a bad argument.  No reference equivalent. */
int32_t grb_smaa_edge_detection_to_peers(const GrbImage *color, int32_t quality, const GrbImage *edges_layout, void *const *peer_images,
                                         const GrbRows *peer_rows, uint32_t *const *peer_flags, int32_t peer_count, int32_t flag_index,
                                         uint32_t epoch, uint32_t *scratch_counter, GrbRows rows, void *stream);

/* FidelityFX FSR 1 after the post chain (renderer/post/aa.cpp:75-174 setup_after_post_chain_upscaling;
 * assets/shaders/post/ffx-fsr/{upscale,sharpen}.frag over ffx_fsr1.h, 32-bit paths).
 * grb_fsr_upscale = the "<output>-scale" pass (FsrEasuF): color is the low-resolution 8-bit image, read as UNORM whatever its
 * format says (aa.cpp:90 set_unorm_texture); out has the display resolution -- R8G8B8A8_UNORM when a sharpen pass follows
 * (TARGET_SRGB = 0), R8G8B8A8_SRGB when it is the last pass (TARGET_SRGB = 1: decode_srgb, the store encodes).  The EASU
 * constants are FsrEasuCon of the two sizes (aa.cpp:33-61; grb_fsr_easu_constants returns them, 16 floats).
 * grb_fsr_sharpen = the "<output>-sharpen" pass (FsrRcasF): color and out of one size; with an SRGB out the input is read
 * through an sRGB view (aa.cpp:141-144) and the result encoded on store.  sharpness_stops as FsrRcasCon takes it
 * (aa.cpp:63-73; the reference passes 0.5): the lobe is scaled by 2^-stops. */
int32_t grb_fsr_easu_constants(int32_t in_width, int32_t in_height, int32_t out_width, int32_t out_height, float *con16);
int32_t grb_fsr_upscale(const GrbImage *color, const GrbImage *out, GrbRows rows, void *stream);
int32_t grb_fsr_sharpen(const GrbImage *color, const GrbImage *out, float sharpness_stops, GrbRows rows, void *stream);

/* K12 fxaa.frag; renderer/post/fxaa.cpp:41-55. in: 8-bit image viewed as UNORM; if out's
 * format is *_SRGB the shader's FXAA_TARGET_SRGB path applies. */
int32_t grb_fxaa(const GrbImage *in, const GrbImage *out, GrbRows rows, void *stream);
/* K13 taa_resolve.frag; renderer/post/temporal.cpp:226-265. history NULL on the first
 * frame (REPROJECTION_HISTORY=0). quality 0..2 = TAAQuality. mv: R16G16_SFLOAT.
 * out_color: B10G11R11_UFLOAT; out_history: R16G16B16A16_SFLOAT. */
int32_t grb_taa_resolve(const GrbImage *hdr, const GrbImage *depth, const GrbImage *mv,
                        const GrbImage *history, const float *reproj16, int32_t quality,
                        const GrbImage *out_color, const GrbImage *out_history, GrbRows rows, void *stream);
/* grb_taa_resolve for one rank of a row-sharded frame, with the history exchange fused in (the exact kernel; the
 * GRB_TAA_TILES form has no peer variant).  out_color gets the rows [rows.y0, rows.y1); the history texels of
 * own_rows (inside rows: this rank's band) are stored into the history slot of EVERY rank -- peer_images[r], valid on
 * this device, one of them this rank's own, all with out_history_layout's size and pitch (its data pointer is not
 * written) -- and then peer_flags[r][flag_index] = epoch is release-stored on every rank, as in
 * grb_bloom_downsample_to_peers.  `history` (last frame's full history) must not be one of the slots written.
 * A raised flag also means the producing rank has finished reading its `history`.  No reference equivalent. */
int32_t grb_taa_resolve_to_peers(const GrbImage *hdr, const GrbImage *depth, const GrbImage *mv,
                                 const GrbImage *history, const float *reproj16, int32_t quality,
                                 const GrbImage *out_color, const GrbImage *out_history_layout,
                                 void *const *peer_images, uint32_t *const *peer_flags, int32_t peer_count,
                                 int32_t flag_index, uint32_t epoch, uint32_t *scratch_counter, GrbRows rows,
                                 GrbRows own_rows, void *stream);

#ifdef __cplusplus
}
#endif
#endif
