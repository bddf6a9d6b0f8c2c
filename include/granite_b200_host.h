/*
 * granite_b200_host.h -- C entry points of libgranite_b200_host.so: the application-side
 * harness that drives the C++ host layer (granite_b200/host/: RenderGraph, LightClusterer,
 * DeferredLightRenderer, setup_hdr_postprocess_compute, setup_taa_resolve,
 * setup_fxaa_postprocess) the way SceneViewerApplication does in the reference
 * (application/scene_viewer_application.cpp:876-991 add_main_pass_deferred, :1167-1318
 * bake_render_graph, :1540-1611 render_frame).  The G-buffer, which the reference rasterises,
 * is an INPUT here: it is uploaded from host memory by a "gbuffer" pass at the head of the graph.
 *
 * This is what bench.py's end-to-end measurement and the graph-level tests call.  All
 * functions return 0 on success, negative on failure (grbh_last_error()).
 */
#ifndef GRANITE_B200_HOST_H_
#define GRANITE_B200_HOST_H_

#include <stdint.h>

#include "granite_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct GrbhViewer GrbhViewer;

typedef enum GrbhPostAA
{
	GRBH_AA_NONE = 0,
	GRBH_AA_FXAA = 1,
	/* SMAA 1x after the tonemap, presets Low .. Ultra; needs grbh_viewer_set_smaa_lookup_textures before the first frame */
	GRBH_AA_SMAA_LOW = 3,
	GRBH_AA_SMAA_MEDIUM = 4,
	GRBH_AA_SMAA_HIGH = 5,
	GRBH_AA_SMAA_ULTRA = 6,
	GRBH_AA_TAA_LOW = 8,
	GRBH_AA_TAA_MEDIUM = 9,
	GRBH_AA_TAA_HIGH = 10,
	/* BASELINE config 5: TAA (pre-tonemap) and FXAA (post-tonemap) chained explicitly */
	GRBH_AA_TAA_HIGH_PLUS_FXAA = 100
} GrbhPostAA;

typedef struct GrbhViewerConfig
{
	int32_t cuda_device;
	int32_t width, height;
	int32_t post_aa;            /* GrbhPostAA */
	int32_t hdr_bloom;          /* 1: full bloom chain; 0: tonemap only (BASELINE config 1) */
	int32_t dynamic_exposure;   /* HDROptions::dynamic_exposure */
	int32_t cluster_res[3];     /* LightClusterer::set_resolution; viewer default 128,64,4096 */
	int32_t timestamps;         /* RenderGraph::enable_timestamps */
	void *cuda_stream;          /* NULL: the device creates its own stream */
	int32_t pipelined_io;       /* 1: the G-buffer upload runs on a side stream into images that alternate
	                             * per frame, so frame N+1's host->device copy overlaps frame N's compute
	                             * (every frame must then bring its G-buffer: render_frame(NULL) is an error) */
	int32_t hdr10_output;       /* 1: HDR10 swapchain (scene_viewer_application.cpp:1233-1288): no bloom / tonemap; the lit
	                             * (and TAA-resolved) scene goes through a "ui" pass (cleared to 0,0,0,1: no widgets) and the
	                             * "pq10" pass into an A2B10G10R10 image of ST.2084 codes, BT.2020 primaries, D65 */
	float hdr10_max_content_light_level; /* VkHdrMetadataEXT::maxContentLightLevel in nits; <= 0: 1000 */
	int32_t clustered_lights_shadows;           /* config "clusteredLightsShadows" (scene_viewer_application.cpp:214-215): the lighting
	                                             * pass samples the per-light shadow maps of grbh_viewer_set_light_shadow_maps */
	int32_t clustered_lights_shadow_resolution; /* "clusteredLightsShadowsResolution" (:216-217); <= 0: 512 */
	float resolution_scale;          /* "resolutionScale" (scene_viewer_application.cpp:247-248): 0 or 1 = off.  < 1: width x height
	                                  * is the DISPLAY size; the G-buffer the caller supplies (and every pass up to the post-chain
	                                  * output) has ceil(scale * size) texels (:758-761, 888-889), and FSR 1 upscales the result
	                                  * to the display size (:1263-1268).  Not with row sharding or HDR10 output. */
	int32_t resolution_scale_sharpen; /* "resolutionScaleSharpen" (:249-250): the RCAS pass after the upscale */
	int32_t render_target_fp16;       /* "renderTargetFp16" (:235-236, 880-884): emissive / HDR-main are R16G16B16A16_SFLOAT (8 bytes per
	                                   * texel -- GrbhHostGBuffer::emissive then points at RGBA16F texels); lighting, bloom threshold,
	                                   * tonemap and TAA read / write that format (TAA's own output stays B10G11R11).  Not with HDR10. */
	int32_t volumetric_decals;        /* LightClusterer::set_enable_volumetric_decals (clusterer.cpp:153-156): the decals of
	                                   * grbh_viewer_set_decals are binned into "cluster-bitmask-decal" / "cluster-range-decal" */
} GrbhViewerConfig;

/* Raw light list as the application owns it (before the clusterer sorts/packs it). */
typedef struct GrbhLights
{
	int32_t count;
	const float *color;       /* count x 3 */
	const float *position;    /* count x 3 */
	const uint8_t *is_point;  /* count */
	const float *rotation;    /* count x 9, column-major node rotation (spots) */
	const float *inner_cone;  /* count */
	const float *outer_cone;  /* count */
	float cutoff_range;       /* PositionalLight::set_maximum_range */
} GrbhLights;

/* Host-memory G-buffer of the full frame (pinned memory makes the uploads asynchronous).
 * Only the rows this rank needs (its band + halo) are copied.  mv may be NULL without TAA. */
typedef struct GrbhHostGBuffer
{
	const uint32_t *albedo;
	const uint32_t *normal;
	const uint16_t *pbr;
	const float *depth;
	const uint32_t *emissive;
	const uint32_t *mv; /* R16G16_SFLOAT */
} GrbhHostGBuffer;

const char *grbh_last_error(void);

int32_t grbh_viewer_create(const GrbhViewerConfig *config, GrbhViewer **out);
void grbh_viewer_destroy(GrbhViewer *viewer);

/* RenderContext::set_camera(projection, view) (renderer/render_context.cpp:54-87). */
int32_t grbh_viewer_set_camera(GrbhViewer *viewer, const float *projection16, const float *view16);
int32_t grbh_viewer_set_directional(GrbhViewer *viewer, const float *color3, const float *direction3);
int32_t grbh_viewer_set_lights(GrbhViewer *viewer, const GrbhLights *lights);
int32_t grbh_viewer_set_exposure(GrbhViewer *viewer, float exposure);
/* Shadow maps of the lights of the last grbh_viewer_set_lights call, in THAT order: `count` device pointers (host array),
 * each D16_UNORM of resolution^2 texels (spot) or 6 x resolution^2 (point, faces +X -X +Y -Y +Z -Z); null = no shadow.
 * The caller renders and owns them (the reference's LightClusterer::render_shadow is rasterisation, outside the path). */
int32_t grbh_viewer_set_light_shadow_maps(GrbhViewer *viewer, const void *const *device_maps, int32_t count);
/* ClustererBindlessTransforms::shadow[i] of the visible lights in cluster order, as the clusterer uploads them (host
 * preparation only, no GPU work): capacity x 16 floats.  Returns the light count. */
int32_t grbh_viewer_get_shadow_transforms(GrbhViewer *viewer, float *out16_per_light, int32_t capacity);

/* The two lookup textures SMAA samples (the payloads of the reference's assets/textures/smaa/area.gtx: 160x560 R8G8_UNORM,
 * and search.gtx: 64x16 R8_UNORM), uploaded once to the viewer's device.  grbh_load_gtx reads such a container from a
 * file: returns the VkFormat and fills width / height; texels (capacity bytes) receives the level-0 payload. */
int32_t grbh_viewer_set_smaa_lookup_textures(GrbhViewer *viewer, const uint8_t *area_rg8, const uint8_t *search_r8);
int32_t grbh_load_gtx(const char *path, int32_t *format, int32_t *width, int32_t *height, uint8_t *texels, int64_t capacity);

/* Rec.709 -> display primaries, the matrix setup_hdr10_pq_encoding pushes (renderer/post/hdr.cpp:580-593, 651).
 * primaries_xy8: red, green, blue, white chromaticities (VkHdrMetadataEXT order); out16: column-major mat4. */
int32_t grbh_rec709_to_display_primaries(const float *primaries_xy8, float *out16);

/* Row sharding (multi-GPU): bands[r] = backbuffer rows of rank r.  Must precede bake. */
int32_t grbh_nccl_unique_id(uint8_t out128[128]);
int32_t grbh_viewer_init_collectives(GrbhViewer *viewer, const uint8_t id128[128], int32_t rank, int32_t world_size);
int32_t grbh_viewer_set_row_shards(GrbhViewer *viewer, const GrbRows *bands, int32_t count, int32_t rank);

/* Work estimate of the lighting pass per group of 4 backbuffer rows for the frame last rendered by
 * an UNSHARDED viewer (its depth image and light cluster are resident): grb_lighting_row_cost() on
 * the viewer's resources, copied to the host.  out: ceil(height / 4) values.  Feed the sums per
 * band unit to a weighted partition to get bands of equal lighting work (granite_b200/viewer.py). */
int32_t grbh_viewer_measure_row_cost(GrbhViewer *viewer, uint32_t *out, int32_t capacity);

/* The row plan of one rank of a row-sharded frame (granite_b200/host/shard_plan.hpp): out8 =
 * {own, fxaa, tonemap, upsample0, downsample0, threshold, lighting, lum_grid}.  Pure host math. */
int32_t grbh_shard_plan(int32_t width, int32_t height, const GrbRows *bands, int32_t count, int32_t rank, int32_t fxaa, GrbRows *out8);
/* The same with a TAA resolve between lighting and the post chain (taa != 0): out9 = the eight rows above followed by
 * taa, the rows of the resolved image (what the threshold and the tonemap read); lighting is then taa +- 1 row. */
int32_t grbh_shard_plan_ex(int32_t width, int32_t height, const GrbRows *bands, int32_t count, int32_t rank, int32_t fxaa, int32_t taa,
                           GrbRows *out9);
/* The same with SMAA after the tonemap (smaa_quality 0..3 = Low .. Ultra; < 0: no SMAA, then out11 = out9 of
 * grbh_shard_plan_ex with smaa_weights = smaa_edges = own): out11 = the nine rows above followed by smaa_weights (the
 * rows of "smaa-weights" a rank computes: what its blend reads, own - 1 .. own + 2) and smaa_edges (the rows of "smaa-edge" its weights
 * pass reads: the window its neighbours store into its edge slot).  With SMAA the tonemap covers own - 3 .. own + 2. */
int32_t grbh_shard_plan_smaa(int32_t width, int32_t height, const GrbRows *bands, int32_t count, int32_t rank, int32_t fxaa, int32_t taa,
                             int32_t smaa_quality, GrbRows *out11);

/* bake_render_graph: declares the passes, bakes, allocates attachments. */
int32_t grbh_viewer_bake(GrbhViewer *viewer);

/* One frame: (optionally) upload the host G-buffer rows, refresh the clusterer, record every
 * pass on the stream.  Asynchronous; ordering with later calls is stream order. */
int32_t grbh_viewer_render_frame(GrbhViewer *viewer, const GrbhHostGBuffer *host_gbuffer, double frame_time);
/* Copies this rank's rows of the final image (R8G8B8A8) to host memory laid out as the full
 * frame (row pitch = width*4) and waits for it. rows_out receives the band. */
int32_t grbh_viewer_read_output(GrbhViewer *viewer, uint32_t *dst_full_frame, GrbRows *rows_out);
/* Asynchronous form: enqueues the device->host copy of this frame's rows behind the frame and
 * returns; grbh_viewer_wait_outputs(viewer, k) blocks until at most k such copies are pending
 * (k = 0: all done).  With pipelined_io this keeps PCIe busy in both directions while the GPU
 * computes the next frame. */
int32_t grbh_viewer_read_output_async(GrbhViewer *viewer, uint32_t *dst_full_frame, GrbRows *rows_out);
int32_t grbh_viewer_wait_outputs(GrbhViewer *viewer, int32_t max_pending);
int32_t grbh_viewer_sync(GrbhViewer *viewer);
/* Makes the viewer's main stream (config.cuda_stream) wait for everything recorded so far on its
 * side streams (async cluster build, async post chain), so an event recorded on the main stream
 * afterwards covers the whole frame. */
int32_t grbh_viewer_join_streams(GrbhViewer *viewer);

/* Introspection for tests: device views of graph resources by name (valid until next bake). */
int32_t grbh_viewer_get_image(GrbhViewer *viewer, const char *resource_name, GrbImage *out);
int32_t grbh_viewer_get_buffer(GrbhViewer *viewer, const char *resource_name, void **device_ptr, uint64_t *size);
int32_t grbh_viewer_get_cluster(GrbhViewer *viewer, GrbClusterParameters *params, GrbClusterBuffers *buffers);
/* Copies the sorted/packed host-side light data of the last refresh (for host-prep parity tests). */
int32_t grbh_viewer_get_light_prep(GrbhViewer *viewer, GrbPositionalLight *records, float *model_rows, uint32_t *type_mask, uint32_t *z_ranges,
                                   int32_t capacity);
int32_t grbh_viewer_get_camera(GrbhViewer *viewer, GrbCamera *out, float *projection16, float *inv_projection16);
/* clip(now) -> UV(previous frame) as the taa-resolve pass of the last rendered frame used it
 * (renderer/post/temporal.cpp:239-243: unjittered history matrices). */
int32_t grbh_viewer_get_taa_reprojection(GrbhViewer *viewer, float *out16);
/* Names of the baked passes, '\n' separated. Returns the length needed. */
/* The scene's volumetric decals: `count` world transforms, 12 floats each (mat_affine rows) of unit cubes in decal space. */
int32_t grbh_viewer_set_decals(GrbhViewer *viewer, const float *world_rows12, int32_t count);
/* Host preparation of the decal binning (no GPU work): the visible decals front to back -- view_projection * world
 * (capacity x 16 floats) and their Z-slice ranges (capacity x 2 words).  Returns the count. */
int32_t grbh_viewer_get_decal_prep(GrbhViewer *viewer, float *mvps16, uint32_t *z_ranges2, int32_t capacity);
/* Size of the G-buffer the viewer expects (= width x height unless resolution_scale < 1). */
int32_t grbh_viewer_get_render_size(GrbhViewer *viewer, int32_t *width, int32_t *height);
int32_t grbh_viewer_get_pass_names(GrbhViewer *viewer, char *buffer, int32_t capacity);
/* Per-pass GPU time of the frames since the last call (needs config.timestamps):
 * writes up to `capacity` (name, total ms, count) triples. Returns the number of passes. */
int32_t grbh_viewer_collect_timings(GrbhViewer *viewer, char *names, int32_t names_capacity, float *total_ms, int32_t *counts, int32_t capacity);
/* GPU timeline of the passes recorded since the last call (config.timestamps == 2: intervals are
 * kept, not aggregated): (name, begin ms, end ms) relative to the first interval. Returns the count. */
int32_t grbh_viewer_collect_timeline(GrbhViewer *viewer, char *names, int32_t names_capacity, float *begin_ms, float *end_ms, int32_t capacity);
uint16_t grbh_float_to_half(float v);

#ifdef __cplusplus
}
#endif
#endif
