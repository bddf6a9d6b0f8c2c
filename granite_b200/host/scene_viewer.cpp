// scene_viewer.cpp -- application-side harness + its C API (include/granite_b200_host.h).
// Mirrors the parts of SceneViewerApplication that assemble and drive the hot path:
// add_main_pass_deferred (application/scene_viewer_application.cpp:876-991), bake_render_graph
// (:1167-1318), render_frame (:1540-1611).  The G-buffer (and motion vectors) the reference
// rasterises are uploaded from host memory by the "gbuffer" pass at the head of the graph.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/granite_b200_host.h"
#include "clusterer.hpp"
#include "nccl_collectives.hpp"
#include "post/aa.hpp"
#include "post/fxaa.hpp"
#include "post/smaa.hpp"
#include "post/hdr.hpp"
#include "renderer.hpp"

using namespace Granite;

namespace
{
thread_local std::string t_error;

int32_t fail(const std::string &msg)
{
	t_error = msg;
	return -1;
}

struct FixedExposure : HDRDynamicExposureInterface
{
	float exposure = 1.0f;
	float get_exposure() const override { return exposure; }
};
} // namespace

struct GrbhViewer
{
	GrbhViewerConfig config;
	std::unique_ptr<Vulkan::Device> device;
	RenderGraph graph;
	RenderContext context;
	LightingParameters lighting;
	LightClusterer cluster;
	TemporalJitter jitter;
	FixedExposure exposure;
	TaskComposer composer;
	std::unique_ptr<NcclCollectives> collectives;
	std::vector<GrbRows> bands;
	unsigned rank = 0;

	std::vector<std::unique_ptr<PositionalLight>> light_storage;
	PositionalLightList scene_lights;
	std::vector<mat_affine> scene_decals;

	mat4 projection = mat4(1.0f), view = mat4(1.0f);
	bool baked = false;
	std::string output_name;
	bool ui_layer_cleared = false;
	const GrbhHostGBuffer *pending_upload = nullptr;
	unsigned profiled_frames = 0;
	std::map<std::string, std::pair<double, int>> timings;
	std::vector<cudaEvent_t> pending_outputs; // one per async readback still in flight (oldest first)
	std::vector<cudaEvent_t> free_output_events;

	RenderTextureResource *res_emissive = nullptr, *res_albedo = nullptr, *res_normal = nullptr, *res_pbr = nullptr, *res_depth = nullptr,
	                      *res_mv = nullptr;

	bool uses_taa() const
	{
		return config.post_aa == GRBH_AA_TAA_LOW || config.post_aa == GRBH_AA_TAA_MEDIUM || config.post_aa == GRBH_AA_TAA_HIGH ||
		       config.post_aa == GRBH_AA_TAA_HIGH_PLUS_FXAA;
	}
	// "resolutionScale": the scene is rendered at ceil(scale * display size) (render_graph.cpp's relative-size rule)
	bool upscales() const { return config.resolution_scale > 0.0f && config.resolution_scale < 1.0f; }
	float scene_scale() const { return upscales() ? config.resolution_scale : 1.0f; }
	int render_width() const { return upscales() ? std::max(int(std::ceil(config.resolution_scale * float(config.width))), 1) : config.width; }
	int render_height() const { return upscales() ? std::max(int(std::ceil(config.resolution_scale * float(config.height))), 1) : config.height; }
	bool uses_fxaa() const { return config.post_aa == GRBH_AA_FXAA || config.post_aa == GRBH_AA_TAA_HIGH_PLUS_FXAA; }
	bool uses_smaa() const { return config.post_aa >= GRBH_AA_SMAA_LOW && config.post_aa <= GRBH_AA_SMAA_ULTRA; }
	int smaa_quality() const { return uses_smaa() ? config.post_aa - GRBH_AA_SMAA_LOW : -1; }

	// rows of the full-resolution inputs this rank must hold: its band + the halo the bloom
	// threshold (and FXAA or SMAA through the tonemap, and the TAA resolve) reaches into
	GrbRows input_rows() const
	{
		return compute_shard_plan((unsigned)render_width(), (unsigned)render_height(), bands, rank, uses_fxaa(), uses_taa(), smaa_quality()).lighting;
	}

	void upload_rows(Vulkan::CommandBuffer &cmd, RenderTextureResource *res, const void *host, unsigned texel)
	{
		if (!res || !host)
			return;
		auto &view_ = graph.get_physical_texture_resource(*res);
		GrbRows r = input_rows();
		size_t pitch = (size_t)render_width() * texel;
		auto *dst = static_cast<uint8_t *>(view_.get_image().get_device_pointer()) + (size_t)r.y0 * pitch;
		auto *src = static_cast<const uint8_t *>(host) + (size_t)r.y0 * pitch;
		Vulkan::cuda_ok(cudaMemcpyAsync(dst, src, pitch * (size_t)(r.y1 - r.y0), cudaMemcpyHostToDevice, reinterpret_cast<cudaStream_t>(cmd.get_stream())),
		                "G-buffer upload");
	}

	void bake_render_graph();
	void render_frame(const GrbhHostGBuffer *host, double frame_time);
};

void GrbhViewer::bake_render_graph()
{
	auto physical_buffers = graph.consume_physical_buffers();
	graph.reset();
	graph.set_device(device.get());
	graph.enable_timestamps(config.timestamps != 0);

	ResourceDimensions dim;
	dim.width = (unsigned)config.width;
	dim.height = (unsigned)config.height;
	dim.format = VK_FORMAT_R8G8B8A8_SRGB; // headless swapchain format (application_headless.cpp:207)
	graph.set_backbuffer_dimensions(dim);
	if (!bands.empty())
		graph.set_row_shards(bands, rank, collectives.get(), uses_fxaa(), uses_taa(), smaa_quality());

	// scene.add_render_passes(graph) -> LightClusterer::add_render_passes
	cluster.set_resolution((unsigned)config.cluster_res[0], (unsigned)config.cluster_res[1], (unsigned)config.cluster_res[2]);
	cluster.set_scene_lights(&scene_lights);
	cluster.set_base_render_context(&context);
	cluster.set_async_compute(getenv("GRB_NO_ASYNC_CLUSTER") == nullptr);
	cluster.set_enable_volumetric_decals(config.volumetric_decals != 0);
	cluster.set_scene_decals(&scene_decals);
	cluster.set_enable_shadows(config.clustered_lights_shadows != 0);
	cluster.set_shadow_resolution(config.clustered_lights_shadow_resolution > 0 ? (unsigned)config.clustered_lights_shadow_resolution : 512u);
	if (bands.size() > 1)
	{
		const GrbRows lit = input_rows();
		cluster.set_lit_pixel_rows(lit.y0, lit.y1, render_height());
	}
	else
		cluster.set_lit_pixel_rows(0, 0, 0);
	cluster.add_render_passes(graph);
	lighting.cluster = &cluster;
	context.set_lighting_parameters(&lighting);

	// Post chain on its own stream (the reference's async-compute post, scene_viewer_application.cpp:
	// 1238-1247) unless disabled; its input image then alternates between two copies per frame.
	const bool async_post = getenv("GRB_NO_ASYNC_POST") == nullptr;
	RenderGraph::set_async_post(async_post);

	// ---- add_main_pass_deferred ----
	AttachmentInfo emissive, albedo, normal, pbr, depth;
	emissive.format = config.render_target_fp16 ? VK_FORMAT_R16G16B16A16_SFLOAT : VK_FORMAT_B10G11R11_UFLOAT_PACK32; // scene_viewer_application.cpp:882-884
	albedo.format = VK_FORMAT_R8G8B8A8_SRGB;
	normal.format = VK_FORMAT_A2B10G10R10_UNORM_PACK32;
	pbr.format = VK_FORMAT_R8G8_UNORM;
	depth.format = VK_FORMAT_D32_SFLOAT;

	// pipelined I/O: uploads on the async-compute stream into ping-pong images, so the copy of the
	// next frame's inputs overlaps this frame's lighting
	// scene_viewer_application.cpp:758-761, 888-889: the scene attachments scale with "resolutionScale"; everything
	// downstream is sized relative to them
	for (auto *info : { &emissive, &albedo, &normal, &pbr, &depth })
		info->size_x = info->size_y = scene_scale();
	const bool pipelined = config.pipelined_io != 0;
	if (pipelined)
		for (auto *info : { &emissive, &albedo, &normal, &pbr, &depth })
			info->flags |= ATTACHMENT_INFO_PINGPONG_BIT;
	auto &gbuffer = graph.add_pass("gbuffer", pipelined ? RENDER_GRAPH_QUEUE_ASYNC_COMPUTE_BIT : RENDER_GRAPH_QUEUE_GRAPHICS_BIT);
	res_emissive = &gbuffer.add_color_output("emissive", emissive);
	res_albedo = &gbuffer.add_color_output("albedo", albedo);
	res_normal = &gbuffer.add_color_output("normal", normal);
	res_pbr = &gbuffer.add_color_output("pbr", pbr);
	res_depth = &gbuffer.set_depth_stencil_output("depth-transient", depth);
	gbuffer.set_build_render_pass([this](Vulkan::CommandBuffer &cmd) {
		if (!pending_upload)
			return; // inputs already resident from an earlier frame
		upload_rows(cmd, res_emissive, pending_upload->emissive, config.render_target_fp16 ? 8 : 4);
		upload_rows(cmd, res_albedo, pending_upload->albedo, 4);
		upload_rows(cmd, res_normal, pending_upload->normal, 4);
		upload_rows(cmd, res_pbr, pending_upload->pbr, 2);
		upload_rows(cmd, res_depth, pending_upload->depth, 4);
	});

	auto &lighting_pass = graph.add_pass("lighting", RENDER_GRAPH_QUEUE_GRAPHICS_BIT);
	// The reference lets HDR-main alias emissive (add_color_output(..., "emissive")) and blends in
	// place.  Here HDR-main is its own image and emissive a read-only input: same bytes moved,
	// and the uploaded G-buffer stays intact, so a resident G-buffer can be lit again next frame.
	AttachmentInfo hdr_info = emissive;
	if (async_post)
		hdr_info.flags |= ATTACHMENT_INFO_PINGPONG_BIT;
	auto &hdr_main = lighting_pass.add_color_output("HDR-main", hdr_info);
	auto &in_emissive = lighting_pass.add_attachment_input("emissive");
	auto &in_albedo = lighting_pass.add_attachment_input("albedo");
	auto &in_normal = lighting_pass.add_attachment_input("normal");
	auto &in_pbr = lighting_pass.add_attachment_input("pbr");
	auto &in_depth = lighting_pass.add_attachment_input("depth-transient");
	lighting_pass.set_depth_stencil_input("depth-transient");
	// work schedule of the lighting kernel: row costs of this frame order the next frame's rows
	BufferInfo schedule_info;
	schedule_info.size = (size_t)grb_lighting_schedule_bytes(render_height());
	schedule_info.usage = VK_BUFFER_USAGE_STORAGE_BUFFER_BIT;
	auto &schedule = lighting_pass.add_storage_output("lighting-schedule", schedule_info);
	auto light_iface = std::make_shared<DeferredLightingPass>(context, &cluster);
	light_iface->set_resources(graph, in_albedo, in_normal, in_pbr, in_depth, hdr_main, &in_emissive);
	light_iface->set_schedule(schedule);
	light_iface->set_shard_halo(uses_fxaa() ? 12u : 8u);
	lighting_pass.set_render_pass_interface(light_iface);

	std::string light_output = "HDR-main";

	// ---- AA before the post chain (TAA) ----
	PostAAType before = PostAAType::None;
	switch (config.post_aa)
	{
	case GRBH_AA_TAA_LOW: before = PostAAType::TAA_Low; break;
	case GRBH_AA_TAA_MEDIUM: before = PostAAType::TAA_Medium; break;
	case GRBH_AA_TAA_HIGH:
	case GRBH_AA_TAA_HIGH_PLUS_FXAA: before = PostAAType::TAA_High; break;
	default: break;
	}
	res_mv = nullptr;
	if (uses_taa())
	{
		// add_mv_pass: the motion-vector image is an input of this path
		AttachmentInfo mv;
		mv.format = VK_FORMAT_R16G16_SFLOAT;
		mv.size_x = mv.size_y = scene_scale();
		if (pipelined)
			mv.flags |= ATTACHMENT_INFO_PINGPONG_BIT;
		auto &mv_pass = graph.add_pass("mv", pipelined ? RENDER_GRAPH_QUEUE_ASYNC_COMPUTE_BIT : RENDER_GRAPH_QUEUE_GRAPHICS_BIT);
		res_mv = &mv_pass.add_color_output("mv-main", mv);
		mv_pass.set_build_render_pass([this](Vulkan::CommandBuffer &cmd) {
			if (pending_upload)
				upload_rows(cmd, res_mv, pending_upload->mv, 4);
		});
	}
	bool resolved = setup_before_post_chain_antialiasing(before, graph, jitter, scene_scale(), light_output, "depth-transient", "mv-main", "HDR-resolved");
	if (resolved && async_post)
		graph.get_texture_resource("HDR-resolved").get_attachment_info().flags |= ATTACHMENT_INFO_PINGPONG_BIT;

	// ---- HDR10 swapchain: no bloom / tonemap, the scene goes to the PQ encoder (scene_viewer_application.cpp:1233-1288) ----
	std::string chain_input = resolved ? "HDR-resolved" : light_output;
	std::string ui_source;
	if (config.hdr10_output)
	{
		// "ui": the application's widgets over a layer cleared to (0, 0, 0, 1) (scene_viewer_application.cpp:1296-1302).
		// Widget rendering is the application's; this viewer draws none, so the layer is its clear colour.
		AttachmentInfo ui_info;
		ui_info.format = VK_FORMAT_R8G8B8A8_UNORM;
		ui_info.size_class = SizeClass::InputRelative;
		ui_info.size_relative_name = chain_input;
		auto &ui = graph.add_pass("ui", RENDER_GRAPH_QUEUE_GRAPHICS_BIT);
		auto &ui_layer = ui.add_color_output("ui-temporary", ui_info);
		ui.add_texture_input(chain_input);
		ui.set_get_clear_color([](unsigned, VkClearColorValue *value) {
			if (value)
			{
				value->float32[0] = value->float32[1] = value->float32[2] = 0.0f;
				value->float32[3] = 1.0f;
			}
			return true;
		});
		ui_layer_cleared = false;
		ui.set_build_render_pass([this, &ui_layer](Vulkan::CommandBuffer &cmd) {
			if (ui_layer_cleared)
				return; // nothing draws into the layer afterwards
			auto &view_ = graph.get_physical_texture_resource(ui_layer);
			const std::vector<uint32_t> clear((size_t)config.width * (size_t)config.height, 0xff000000u);
			Vulkan::cuda_ok(cudaMemcpyAsync(view_.get_image().get_device_pointer(), clear.data(), clear.size() * 4, cudaMemcpyHostToDevice,
			                                reinterpret_cast<cudaStream_t>(cmd.get_stream())),
			                "ui layer clear");
			Vulkan::cuda_ok(cudaStreamSynchronize(reinterpret_cast<cudaStream_t>(cmd.get_stream())), "ui layer clear");
			ui_layer_cleared = true;
		});

		HDR10PQEncodingConfig hdr10_config = {};
		hdr10_config.hdr_pre_exposure = 500.0f; // scene_viewer_application.cpp:1284-1285
		hdr10_config.ui_pre_exposure = 400.0f;
		VkHdrMetadataEXT md = {};
		md.displayPrimaryRed = { 0.708f, 0.292f }; // BT.2020, D65
		md.displayPrimaryGreen = { 0.170f, 0.797f };
		md.displayPrimaryBlue = { 0.131f, 0.046f };
		md.whitePoint = { 0.3127f, 0.3290f };
		md.maxContentLightLevel = config.hdr10_max_content_light_level > 0.0f ? config.hdr10_max_content_light_level : 1000.0f;
		setup_hdr10_pq_encoding(graph, "ui-output", chain_input, "ui-temporary", hdr10_config, md);
		ui_source = "ui-output";
	}
	else
	{
		// ---- HDR chain ----
		HDROptions opts;
		opts.dynamic_exposure = config.dynamic_exposure != 0;
		if (config.hdr_bloom)
			setup_hdr_postprocess_compute(graph, context.get_frame_parameters(), chain_input, "tonemapped", opts, &exposure);
		else
		{
			// BASELINE config 1: a single tonemap pass.  tonemap.frag always samples uBloom; with
			// bloom off that image is the zero-initialised one nothing ever writes.
			AttachmentInfo quarter;
			quarter.format = VK_FORMAT_R16G16B16A16_SFLOAT;
			quarter.size_class = SizeClass::InputRelative;
			quarter.size_relative_name = chain_input;
			quarter.size_x = 0.25f;
			quarter.size_y = 0.25f;
			auto &off = graph.add_pass("bloom-disabled", RENDER_GRAPH_QUEUE_COMPUTE_BIT);
			off.add_storage_texture_output("upsample-0", quarter);
			off.add_texture_input(chain_input);
			off.set_build_render_pass([](Vulkan::CommandBuffer &) {});
			AttachmentInfo tonemap_info;
			tonemap_info.size_class = SizeClass::InputRelative;
			tonemap_info.size_relative_name = chain_input;
			auto &tonemap = graph.add_pass("tonemap", RenderGraph::get_default_post_graphics_queue());
			auto &out = tonemap.add_color_output("tonemapped", tonemap_info);
			auto &hdr_res = tonemap.add_texture_input(chain_input);
			auto &bloom_res = tonemap.add_texture_input("upsample-0");
			tonemap.set_build_render_pass([this, &out, &hdr_res, &bloom_res](Vulkan::CommandBuffer &cmd) {
				GrbImage hdr = graph.get_physical_texture_resource(hdr_res).as_grb();
				GrbImage bloom = graph.get_physical_texture_resource(bloom_res).as_grb();
				auto &ov = graph.get_physical_texture_resource(out);
				GrbImage o = ov.as_grb();
				cmd.check(grb_tonemap(&hdr, &bloom, nullptr, exposure.get_exposure(), &o, graph.is_sharded() ? graph.get_shard_plan().tonemap : GrbRows{ 0, 0 },
				                      cmd.get_stream_handle()),
				          "grb_tonemap");
			});
		}
		ui_source = "tonemapped";

		// ---- AA after the post chain (FXAA) ----
		if (uses_fxaa())
		{
			setup_fxaa_postprocess(graph, ui_source, "post-aa-output");
			ui_source = "post-aa-output";
		}
		else if (uses_smaa())
		{
			const PostAAType type = config.post_aa == GRBH_AA_SMAA_LOW ? PostAAType::SMAA_Low :
			                        (config.post_aa == GRBH_AA_SMAA_MEDIUM ? PostAAType::SMAA_Medium :
			                                                                 (config.post_aa == GRBH_AA_SMAA_HIGH ? PostAAType::SMAA_High : PostAAType::SMAA_Ultra));
			if (setup_after_post_chain_antialiasing(type, graph, jitter, scene_scale(), ui_source, "depth-transient", "post-aa-output"))
				ui_source = "post-aa-output";
		}
	}
	// scene_viewer_application.cpp:1263-1268: FSR 1 from the scaled-down image to the swapchain size
	if (upscales() && setup_after_post_chain_upscaling(graph, ui_source, "post-scale-output", config.resolution_scale_sharpen != 0))
		ui_source = "post-scale-output";
	output_name = ui_source;
	graph.set_backbuffer_source(ui_source);
	graph.bake();
	// keep feed-back buffers (average luminance) across re-bakes
	graph.install_physical_buffers(std::move(physical_buffers));
	baked = true;
}

void GrbhViewer::render_frame(const GrbhHostGBuffer *host, double frame_time)
{
	FrameParameters frame = context.get_frame_parameters();
	frame.frame_time = frame_time;
	frame.elapsed_time += frame_time;
	context.set_frame_parameters(frame);

	{
		Vulkan::ScopedHostTimer timer("frame.setup_attachments");
		graph.setup_attachments(*device, nullptr);
		cluster.setup_render_pass_resources(graph);
	}

	// update_scene: jitter.step, context.set_camera, LightClusterer::refresh
	{
		Vulkan::ScopedHostTimer timer("frame.camera + cluster refresh");
		// scene_viewer_application.cpp:1431-1432: the frame is rendered (and clustered, and lit) with the
		// jittered projection; the reprojection keeps the unjittered history (temporal.cpp:239-243)
		jitter.step(projection, view);
		context.set_camera(jitter.get_jittered_projection(), view);
		cluster.refresh(context);
	}

	pending_upload = host;
	{
		Vulkan::ScopedHostTimer timer("frame.enqueue_render_passes");
		graph.enqueue_render_passes(*device, composer);
	}
	pending_upload = nullptr;
	profiled_frames++;

	if (config.timestamps == 1)
		for (auto &iv : device->collect_time_intervals())
		{
			auto &slot = timings[iv.first];
			slot.first += iv.second;
			slot.second++;
		}
}

// ----------------------------------------------------------------------------- C API
#define GRBH_TRY try {
#define GRBH_CATCH                                  \
	}                                               \
	catch (const std::exception &e)                 \
	{                                               \
		return fail(e.what());                      \
	}                                               \
	catch (...)                                     \
	{                                               \
		return fail("unknown C++ exception");       \
	}

extern "C" const char *grbh_last_error(void)
{
	return t_error.c_str();
}

extern "C" uint16_t grbh_float_to_half(float v)
{
	return muglm::floatToHalf(v);
}

extern "C" int32_t grbh_viewer_create(const GrbhViewerConfig *config, GrbhViewer **out)
{
	if (!config || !out || config->width <= 0 || config->height <= 0)
		return fail("grbh_viewer_create: bad config");
	if (config->hdr10_output && (config->post_aa == GRBH_AA_FXAA || config->post_aa == GRBH_AA_TAA_HIGH_PLUS_FXAA))
		return fail("grbh_viewer_create: FXAA reads the tonemapped 8-bit image; an HDR10 output has none (use TAA)");
	if (config->hdr10_output && config->post_aa >= GRBH_AA_SMAA_LOW && config->post_aa <= GRBH_AA_SMAA_ULTRA)
		return fail("grbh_viewer_create: SMAA reads the tonemapped 8-bit image; an HDR10 output has none (use TAA)");
	if (config->resolution_scale > 0.0f && config->resolution_scale < 1.0f && config->hdr10_output)
		return fail("grbh_viewer_create: FSR 1 upscaling reads the tonemapped 8-bit image; an HDR10 output has none");
	if (config->render_target_fp16 && config->hdr10_output)
		return fail("grbh_viewer_create: the HDR10 / PQ encoder reads a B10G11R11 scene image; render_target_fp16 is not supported with it");
	if (!(config->resolution_scale >= 0.0f && config->resolution_scale <= 1.0f))
		return fail("grbh_viewer_create: resolution_scale must be within [0, 1] (0 or 1 = off)");
	GRBH_TRY
	auto v = std::make_unique<GrbhViewer>();
	v->config = *config;
	if (v->config.cluster_res[0] == 0)
	{
		v->config.cluster_res[0] = 128; // scene_viewer_application.cpp:407
		v->config.cluster_res[1] = 64;
		v->config.cluster_res[2] = 4096;
	}
	// cuda_device < 0: host-only viewer (camera / light preparation without touching a GPU)
	if (config->cuda_device >= 0)
		v->device = std::make_unique<Vulkan::Device>(config->cuda_device, static_cast<Vulkan::Stream>(config->cuda_stream));
	v->lighting.directional.color = vec3(6.0f, 5.5f, 4.5f); // scene_viewer_application.cpp:380
	v->lighting.directional.direction = normalize(vec3(0.3f, 0.8f, 0.5f));
	*out = v.release();
	return 0;
	GRBH_CATCH
}

extern "C" void grbh_viewer_destroy(GrbhViewer *viewer)
{
	if (!viewer)
		return;
	if (viewer->device)
		viewer->device->wait_idle();
	Vulkan::HostProfile::report(viewer->profiled_frames);
	for (auto e : viewer->pending_outputs)
		cudaEventDestroy(e);
	for (auto e : viewer->free_output_events)
		cudaEventDestroy(e);
	viewer->graph.reset();
	if (viewer->device)
		Granite::release_smaa_lookup_textures(*viewer->device); // device images: must go before the device does
	delete viewer;
}

extern "C" int32_t grbh_viewer_set_camera(GrbhViewer *v, const float *projection16, const float *view16)
{
	if (!v || !projection16 || !view16)
		return fail("grbh_viewer_set_camera: null");
	std::memcpy(v->projection.data(), projection16, 64);
	std::memcpy(v->view.data(), view16, 64);
	v->context.set_camera(v->projection, v->view);
	return 0;
}

extern "C" int32_t grbh_viewer_set_directional(GrbhViewer *v, const float *color3, const float *direction3)
{
	if (!v || !color3 || !direction3)
		return fail("grbh_viewer_set_directional: null");
	v->lighting.directional.color = vec3(color3[0], color3[1], color3[2]);
	v->lighting.directional.direction = vec3(direction3[0], direction3[1], direction3[2]);
	return 0;
}

extern "C" int32_t grbh_viewer_set_exposure(GrbhViewer *v, float exposure)
{
	if (!v)
		return fail("null viewer");
	v->exposure.exposure = exposure;
	return 0;
}

extern "C" int32_t grbh_viewer_set_lights(GrbhViewer *v, const GrbhLights *l)
{
	if (!v || !l || l->count < 0)
		return fail("grbh_viewer_set_lights: bad arguments");
	GRBH_TRY
	v->light_storage.clear();
	v->scene_lights.clear();
	for (int i = 0; i < l->count; i++)
	{
		vec3 color(l->color[3 * i], l->color[3 * i + 1], l->color[3 * i + 2]);
		vec3 pos(l->position[3 * i], l->position[3 * i + 1], l->position[3 * i + 2]);
		PositionalLightInfo info;
		if (l->is_point[i])
		{
			auto p = std::make_unique<PointLight>();
			p->set_maximum_range(l->cutoff_range);
			p->set_color(color);
			info.transform = mat_affine(vec4(1, 0, 0, pos.x), vec4(0, 1, 0, pos.y), vec4(0, 0, 1, pos.z));
			info.light = p.get();
			v->light_storage.push_back(std::move(p));
		}
		else
		{
			auto s = std::make_unique<SpotLight>();
			s->set_maximum_range(l->cutoff_range);
			s->set_color(color);
			s->set_spot_parameters(l->inner_cone[i], l->outer_cone[i]);
			const float *r = l->rotation + 9 * i; // column-major 3x3
			info.transform = mat_affine(vec4(r[0], r[3], r[6], pos.x), vec4(r[1], r[4], r[7], pos.y), vec4(r[2], r[5], r[8], pos.z));
			info.light = s.get();
			v->light_storage.push_back(std::move(s));
		}
		v->scene_lights.push_back(info);
	}
	return 0;
	GRBH_CATCH
}

extern "C" int32_t grbh_viewer_set_light_shadow_maps(GrbhViewer *v, const void *const *device_maps, int32_t count)
{
	if (!v || count < 0 || (count > 0 && !device_maps))
		return fail("grbh_viewer_set_light_shadow_maps: bad arguments");
	if ((size_t)count != v->scene_lights.size())
		return fail("grbh_viewer_set_light_shadow_maps: one entry per light of the last grbh_viewer_set_lights call");
	if (!v->config.clustered_lights_shadows)
		return fail("grbh_viewer_set_light_shadow_maps: the viewer was created without clustered_lights_shadows");
	for (int i = 0; i < count; i++)
		v->scene_lights[(size_t)i].light->set_shadow_map(device_maps[i]);
	return 0;
}

extern "C" int32_t grbh_viewer_get_shadow_transforms(GrbhViewer *v, float *out16_per_light, int32_t capacity)
{
	if (!v)
		return fail("null viewer");
	// host prep only (no GPU work), like grbh_viewer_get_light_prep
	v->cluster.set_scene_lights(&v->scene_lights);
	v->cluster.set_enable_shadows(true);
	v->cluster.refresh(v->context);
	v->cluster.set_enable_shadows(v->config.clustered_lights_shadows != 0);
	const auto &t = v->cluster.get_shadow_transforms();
	if ((int64_t)t.size() > capacity)
		return fail("grbh_viewer_get_shadow_transforms: capacity too small");
	if (out16_per_light && !t.empty())
		std::memcpy(out16_per_light, t.data(), 64 * t.size());
	return (int32_t)t.size();
}

extern "C" int32_t grbh_viewer_set_smaa_lookup_textures(GrbhViewer *v, const uint8_t *area_rg8, const uint8_t *search_r8)
{
	if (!v || !area_rg8 || !search_r8)
		return fail("grbh_viewer_set_smaa_lookup_textures: bad arguments");
	if (!v->device)
		return fail("grbh_viewer_set_smaa_lookup_textures: host-only viewer (no CUDA device)");
	GRBH_TRY
	if (!Granite::set_smaa_lookup_textures(*v->device, area_rg8, search_r8))
		return fail("grbh_viewer_set_smaa_lookup_textures: upload failed");
	return 0;
	GRBH_CATCH
}

extern "C" int32_t grbh_load_gtx(const char *path, int32_t *format, int32_t *width, int32_t *height, uint8_t *texels, int64_t capacity)
{
	if (!path || !format || !width || !height)
		return fail("grbh_load_gtx: bad arguments");
	GRBH_TRY
	Granite::GtxImage img;
	std::string error;
	if (!Granite::load_gtx(path, img, error))
		return fail(error.c_str());
	*format = (int32_t)img.format;
	*width = (int32_t)img.width;
	*height = (int32_t)img.height;
	if (texels)
	{
		if (capacity < (int64_t)img.texels.size())
			return fail("grbh_load_gtx: texel buffer too small");
		std::memcpy(texels, img.texels.data(), img.texels.size());
	}
	return 0;
	GRBH_CATCH
}

extern "C" int32_t grbh_rec709_to_display_primaries(const float *primaries_xy8, float *out16)
{
	if (!primaries_xy8 || !out16)
		return fail("grbh_rec709_to_display_primaries: bad arguments");
	VkHdrMetadataEXT md = {};
	md.displayPrimaryRed = { primaries_xy8[0], primaries_xy8[1] };
	md.displayPrimaryGreen = { primaries_xy8[2], primaries_xy8[3] };
	md.displayPrimaryBlue = { primaries_xy8[4], primaries_xy8[5] };
	md.whitePoint = { primaries_xy8[6], primaries_xy8[7] };
	const muglm::mat4 m = Granite::compute_rec709_to_display_primaries(md);
	std::memcpy(out16, m.data(), 64);
	return GRB_OK;
}

extern "C" int32_t grbh_nccl_unique_id(uint8_t out128[128])
{
	std::string err;
	if (!NcclCollectives::get_unique_id(out128, err))
		return fail(err);
	return 0;
}

extern "C" int32_t grbh_viewer_init_collectives(GrbhViewer *v, const uint8_t id128[128], int32_t rank, int32_t world_size)
{
	if (!v || !id128 || rank < 0 || world_size <= 0 || rank >= world_size)
		return fail("grbh_viewer_init_collectives: bad arguments");
	if (!v->device)
		return fail("grbh_viewer_init_collectives: host-only viewer (cuda_device < 0) has no device to communicate from");
	GRBH_TRY
	cudaSetDevice(v->device->get_device_index());
	auto c = std::make_unique<NcclCollectives>();
	std::string err;
	if (!c->init(id128, (unsigned)rank, (unsigned)world_size, err))
		return fail(err);
	v->collectives = std::move(c);
	return 0;
	GRBH_CATCH
}

extern "C" int32_t grbh_viewer_set_row_shards(GrbhViewer *v, const GrbRows *bands, int32_t count, int32_t rank)
{
	if (!v || count < 0 || (count && !bands) || (count && (rank < 0 || rank >= count)))
		return fail("grbh_viewer_set_row_shards: bad arguments");
	if (count > 1 && v->upscales())
		return fail("grbh_viewer_set_row_shards: FSR 1 upscaling (resolution_scale < 1) is not row-sharded");
	GRBH_TRY
	v->bands.assign(bands, bands + count);
	v->rank = (unsigned)rank;
	v->baked = false;
	return 0;
	GRBH_CATCH
}

extern "C" int32_t grbh_shard_plan(int32_t width, int32_t height, const GrbRows *bands, int32_t count, int32_t rank, int32_t fxaa, GrbRows *out9)
{
	if (width <= 0 || height <= 0 || count < 0 || (count && !bands) || !out9 || (count && (rank < 0 || rank >= count)))
		return fail("grbh_shard_plan: bad arguments");
	GRBH_TRY
	std::vector<GrbRows> b(bands, bands + count);
	ShardPlan p = compute_shard_plan((unsigned)width, (unsigned)height, b, (unsigned)rank, fxaa != 0);
	const GrbRows all[8] = { p.own, p.fxaa, p.tonemap, p.upsample0, p.downsample0, p.threshold, p.lighting, p.lum_grid };
	for (int i = 0; i < 8; i++)
		out9[i] = all[i];
	return 0;
	GRBH_CATCH
}

extern "C" int32_t grbh_shard_plan_ex(int32_t width, int32_t height, const GrbRows *bands, int32_t count, int32_t rank, int32_t fxaa, int32_t taa, GrbRows *out9)
{
	if (width <= 0 || height <= 0 || count < 0 || (count && !bands) || !out9 || (count && (rank < 0 || rank >= count)))
		return fail("grbh_shard_plan_ex: bad arguments");
	GRBH_TRY
	std::vector<GrbRows> b(bands, bands + count);
	ShardPlan p = compute_shard_plan((unsigned)width, (unsigned)height, b, (unsigned)rank, fxaa != 0, taa != 0);
	const GrbRows all[9] = { p.own, p.fxaa, p.tonemap, p.upsample0, p.downsample0, p.threshold, p.lighting, p.lum_grid, p.taa };
	for (int i = 0; i < 9; i++)
		out9[i] = all[i];
	return 0;
	GRBH_CATCH
}

extern "C" int32_t grbh_shard_plan_smaa(int32_t width, int32_t height, const GrbRows *bands, int32_t count, int32_t rank, int32_t fxaa, int32_t taa,
                                        int32_t smaa_quality, GrbRows *out11)
{
	if (width <= 0 || height <= 0 || count < 0 || (count && !bands) || !out11 || (count && (rank < 0 || rank >= count)) || smaa_quality > 3)
		return fail("grbh_shard_plan_smaa: bad arguments");
	GRBH_TRY
	std::vector<GrbRows> b(bands, bands + count);
	ShardPlan p = compute_shard_plan((unsigned)width, (unsigned)height, b, (unsigned)rank, fxaa != 0, taa != 0, smaa_quality < 0 ? -1 : smaa_quality);
	const GrbRows all[11] = { p.own, p.fxaa, p.tonemap, p.upsample0, p.downsample0, p.threshold, p.lighting, p.lum_grid, p.taa, p.smaa_weights, p.smaa_edges };
	for (int i = 0; i < 11; i++)
		out11[i] = all[i];
	return 0;
	GRBH_CATCH
}

extern "C" int32_t grbh_viewer_bake(GrbhViewer *v)
{
	if (!v)
		return fail("null viewer");
	if (!v->device)
		return fail("grbh_viewer_bake: host-only viewer (cuda_device < 0) cannot bake");
	GRBH_TRY
	cudaSetDevice(v->device->get_device_index());
	// attachments are set up by the first render_frame (calling setup_attachments here as well
	// would swap the history images once too often and fake a previous frame)
	v->bake_render_graph();
	return 0;
	GRBH_CATCH
}

extern "C" int32_t grbh_viewer_render_frame(GrbhViewer *v, const GrbhHostGBuffer *host, double frame_time)
{
	if (!v || !v->baked)
		return fail("grbh_viewer_render_frame: viewer not baked");
	if (v->config.pipelined_io && !host)
		return fail("grbh_viewer_render_frame: pipelined_io viewers need the host G-buffer every frame");
	GRBH_TRY
	cudaSetDevice(v->device->get_device_index());
	v->render_frame(host, frame_time);
	return 0;
	GRBH_CATCH
}

extern "C" int32_t grbh_viewer_read_output(GrbhViewer *v, uint32_t *dst, GrbRows *rows_out)
{
	if (!v || !v->baked || !dst)
		return fail("grbh_viewer_read_output: bad arguments");
	GRBH_TRY
	auto &view_ = v->graph.get_physical_texture_resource(v->graph.get_texture_resource(v->output_name));
	GrbRows r = v->bands.size() > 1 ? v->bands[v->rank] : GrbRows{ 0, v->config.height };
	size_t pitch = (size_t)v->config.width * 4;
	// read back on the stream of the pass that produced the image
	auto stream = reinterpret_cast<cudaStream_t>(v->graph.get_writer_stream(v->graph.get_texture_resource(v->output_name)));
	auto *src = static_cast<const uint8_t *>(view_.get_image().get_device_pointer()) + (size_t)r.y0 * pitch;
	if (!Vulkan::cuda_ok(cudaMemcpyAsync(reinterpret_cast<uint8_t *>(dst) + (size_t)r.y0 * pitch, src, pitch * (size_t)(r.y1 - r.y0),
	                                     cudaMemcpyDeviceToHost, stream),
	                     "output readback"))
		return fail("cudaMemcpyAsync failed");
	if (!Vulkan::cuda_ok(cudaStreamSynchronize(stream), "cudaStreamSynchronize"))
		return fail("cudaStreamSynchronize failed");
	if (rows_out)
		*rows_out = r;
	return 0;
	GRBH_CATCH
}

extern "C" int32_t grbh_viewer_read_output_async(GrbhViewer *v, uint32_t *dst, GrbRows *rows_out)
{
	if (!v || !v->baked || !dst)
		return fail("grbh_viewer_read_output_async: bad arguments");
	GRBH_TRY
	auto &view_ = v->graph.get_physical_texture_resource(v->graph.get_texture_resource(v->output_name));
	GrbRows r = v->bands.size() > 1 ? v->bands[v->rank] : GrbRows{ 0, v->config.height };
	size_t pitch = (size_t)v->config.width * 4;
	auto stream = reinterpret_cast<cudaStream_t>(v->graph.get_writer_stream(v->graph.get_texture_resource(v->output_name)));
	auto *src = static_cast<const uint8_t *>(view_.get_image().get_device_pointer()) + (size_t)r.y0 * pitch;
	if (!Vulkan::cuda_ok(cudaMemcpyAsync(reinterpret_cast<uint8_t *>(dst) + (size_t)r.y0 * pitch, src, pitch * (size_t)(r.y1 - r.y0),
	                                     cudaMemcpyDeviceToHost, stream),
	                     "output readback"))
		return fail("cudaMemcpyAsync failed");
	cudaEvent_t e;
	if (!v->free_output_events.empty())
	{
		e = v->free_output_events.back();
		v->free_output_events.pop_back();
	}
	else
		cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
	cudaEventRecord(e, stream);
	v->pending_outputs.push_back(e);
	if (rows_out)
		*rows_out = r;
	return 0;
	GRBH_CATCH
}

extern "C" int32_t grbh_viewer_wait_outputs(GrbhViewer *v, int32_t max_pending)
{
	if (!v || max_pending < 0)
		return fail("grbh_viewer_wait_outputs: bad arguments");
	GRBH_TRY
	while ((int32_t)v->pending_outputs.size() > max_pending)
	{
		cudaEvent_t e = v->pending_outputs.front();
		if (!Vulkan::cuda_ok(cudaEventSynchronize(e), "cudaEventSynchronize"))
			return fail("cudaEventSynchronize failed");
		v->pending_outputs.erase(v->pending_outputs.begin());
		v->free_output_events.push_back(e);
	}
	return 0;
	GRBH_CATCH
}

extern "C" int32_t grbh_viewer_collect_timeline(GrbhViewer *v, char *names, int32_t names_capacity, float *begin_ms, float *end_ms, int32_t capacity)
{
	if (!v || !v->device)
		return fail("null viewer");
	GRBH_TRY
	auto tl = v->device->collect_timeline();
	std::string all;
	int i = 0;
	for (auto &e : tl)
	{
		if (i < capacity)
		{
			if (begin_ms)
				begin_ms[i] = e.begin_ms;
			if (end_ms)
				end_ms[i] = e.end_ms;
		}
		all += e.tag + "\n";
		i++;
	}
	if (names && names_capacity > 0)
		std::snprintf(names, (size_t)names_capacity, "%s", all.c_str());
	return i;
	GRBH_CATCH
}

extern "C" int32_t grbh_viewer_join_streams(GrbhViewer *v)
{
	if (!v || !v->device)
		return fail("null viewer");
	v->device->join_side_streams();
	return 0;
}

extern "C" int32_t grbh_viewer_sync(GrbhViewer *v)
{
	if (!v)
		return fail("null viewer");
	if (!v->device)
		return fail("grbh_viewer_sync: host-only viewer (no CUDA device)");
	GRBH_TRY
	v->device->wait_idle();
	cudaError_t err = cudaGetLastError();
	if (err != cudaSuccess)
		return fail(cudaGetErrorString(err));
	return 0;
	GRBH_CATCH
}

extern "C" int32_t grbh_viewer_get_taa_reprojection(GrbhViewer *v, float *out16)
{
	if (!v || !out16)
		return fail("grbh_viewer_get_taa_reprojection: bad arguments");
	GRBH_TRY
	// the matrix the taa-resolve pass pushed for the LAST rendered frame (temporal.cpp:239-243)
	mat4 reproj = translate(vec3(0.5f, 0.5f, 0.0f)) * scale(vec3(0.5f, 0.5f, 1.0f)) * v->jitter.get_history_view_proj(1) *
	              v->jitter.get_history_inv_view_proj(0);
	std::memcpy(out16, reproj.data(), 16 * sizeof(float));
	return 0;
	GRBH_CATCH
}

extern "C" int32_t grbh_viewer_get_image(GrbhViewer *v, const char *name, GrbImage *out)
{
	if (!v || !name || !out || !v->baked)
		return fail("grbh_viewer_get_image: bad arguments");
	GRBH_TRY
	if (!v->graph.has_texture_resource(name))
		return fail(std::string("no such resource: ") + name);
	auto &res = v->graph.get_texture_resource(name);
	*out = v->graph.get_physical_texture_resource(res).as_grb();
	return 0;
	GRBH_CATCH
}

extern "C" int32_t grbh_viewer_get_buffer(GrbhViewer *v, const char *name, void **ptr, uint64_t *size)
{
	if (!v || !name || !ptr || !v->baked)
		return fail("grbh_viewer_get_buffer: bad arguments");
	GRBH_TRY
	if (!v->graph.has_texture_resource(name))
		return fail(std::string("no such resource: ") + name);
	auto &buf = v->graph.get_physical_buffer_resource(v->graph.get_buffer_resource(name));
	*ptr = buf.get_device_pointer();
	if (size)
		*size = buf.get_create_info().size;
	return 0;
	GRBH_CATCH
}

extern "C" int32_t grbh_viewer_get_cluster(GrbhViewer *v, GrbClusterParameters *params, GrbClusterBuffers *buffers)
{
	if (!v || !v->baked)
		return fail("grbh_viewer_get_cluster: viewer not baked");
	if (params)
		*params = v->cluster.get_cluster_parameters_bindless();
	if (buffers)
		*buffers = v->cluster.get_cluster_buffers();
	return 0;
}

extern "C" int32_t grbh_viewer_get_light_prep(GrbhViewer *v, GrbPositionalLight *records, float *model_rows, uint32_t *type_mask, uint32_t *z_ranges,
                                              int32_t capacity)
{
	if (!v)
		return fail("null viewer");
	// host prep only (no GPU work): usable on a machine without a device
	v->cluster.set_scene_lights(&v->scene_lights);
	if (v->config.cluster_res[0])
		v->cluster.set_resolution((unsigned)v->config.cluster_res[0], (unsigned)v->config.cluster_res[1], (unsigned)v->config.cluster_res[2]);
	v->cluster.refresh(v->context);
	int n = (int)v->cluster.get_active_light_count();
	if (n > capacity)
		return fail("grbh_viewer_get_light_prep: capacity too small");
	if (records)
		std::memcpy(records, v->cluster.get_light_records().data(), sizeof(GrbPositionalLight) * n);
	if (model_rows)
		std::memcpy(model_rows, v->cluster.get_model_transforms().data(), 48 * (size_t)n);
	if (type_mask)
		std::memcpy(type_mask, v->cluster.get_type_mask().data(), sizeof(uint32_t) * ((n + 31) / 32));
	if (z_ranges)
		std::memcpy(z_ranges, v->cluster.get_z_ranges().data(), sizeof(uint32_t) * 2 * v->cluster.get_z_ranges().size());
	return n;
}

extern "C" int32_t grbh_viewer_set_decals(GrbhViewer *v, const float *world_rows12, int32_t count)
{
	if (!v || count < 0 || (count > 0 && !world_rows12))
		return fail("grbh_viewer_set_decals: bad arguments");
	GRBH_TRY
	v->scene_decals.clear();
	for (int i = 0; i < count; i++)
	{
		const float *r = world_rows12 + 12 * (size_t)i;
		v->scene_decals.push_back(mat_affine(vec4(r[0], r[1], r[2], r[3]), vec4(r[4], r[5], r[6], r[7]), vec4(r[8], r[9], r[10], r[11])));
	}
	return 0;
	GRBH_CATCH
}

extern "C" int32_t grbh_viewer_get_decal_prep(GrbhViewer *v, float *mvps16, uint32_t *z_ranges2, int32_t capacity)
{
	if (!v)
		return fail("null viewer");
	GRBH_TRY
	if (v->config.cluster_res[0])
		v->cluster.set_resolution((unsigned)v->config.cluster_res[0], (unsigned)v->config.cluster_res[1], (unsigned)v->config.cluster_res[2]);
	v->cluster.set_scene_lights(&v->scene_lights);
	v->cluster.set_scene_decals(&v->scene_decals);
	v->cluster.set_enable_volumetric_decals(true);
	v->cluster.refresh(v->context);
	v->cluster.set_enable_volumetric_decals(v->config.volumetric_decals != 0);
	const int n = (int)v->cluster.get_active_decal_count();
	if (n > capacity)
		return fail("grbh_viewer_get_decal_prep: capacity too small");
	if (mvps16 && n)
		std::memcpy(mvps16, v->cluster.get_decal_mvps().data(), 64 * (size_t)n);
	if (z_ranges2 && n)
		std::memcpy(z_ranges2, v->cluster.get_decal_z_ranges().data(), 8 * (size_t)n);
	return n;
	GRBH_CATCH
}

extern "C" int32_t grbh_viewer_get_render_size(GrbhViewer *v, int32_t *width, int32_t *height)
{
	if (!v || !width || !height)
		return fail("grbh_viewer_get_render_size: null");
	*width = v->render_width();
	*height = v->render_height();
	return 0;
}

extern "C" int32_t grbh_viewer_get_camera(GrbhViewer *v, GrbCamera *out, float *projection16, float *inv_projection16)
{
	if (!v || !out)
		return fail("grbh_viewer_get_camera: null");
	const auto &rp = v->context.get_render_parameters();
	std::memcpy(out->view, rp.view.data(), 64);
	std::memcpy(out->view_projection, rp.view_projection.data(), 64);
	std::memcpy(out->inv_view_projection, rp.inv_view_projection.data(), 64);
	for (int i = 0; i < 3; i++)
	{
		out->camera_position[i] = rp.camera_position[i];
		out->camera_front[i] = rp.camera_front[i];
	}
	out->z_near = rp.z_near;
	out->z_far = rp.z_far;
	if (projection16)
		std::memcpy(projection16, rp.projection.data(), 64);
	if (inv_projection16)
		std::memcpy(inv_projection16, rp.inv_projection.data(), 64);
	return 0;
}

extern "C" int32_t grbh_viewer_measure_row_cost(GrbhViewer *v, uint32_t *out, int32_t capacity)
{
	if (!v || !v->baked || !v->device || !out)
		return fail("grbh_viewer_measure_row_cost: needs a baked device viewer");
	if (v->graph.is_sharded())
		return fail("grbh_viewer_measure_row_cost: the viewer must hold the whole frame (not row-sharded)");
	GRBH_TRY
	const int groups = (v->render_height() + 3) / 4;
	if (capacity < groups)
		return fail("grbh_viewer_measure_row_cost: capacity too small");
	v->device->wait_idle();
	GrbImage depth = v->graph.get_physical_texture_resource(*v->res_depth).as_grb();
	GrbCamera cam;
	if (grbh_viewer_get_camera(v, &cam, nullptr, nullptr) != 0)
		return -1;
	GrbClusterParameters params = v->cluster.get_cluster_parameters_bindless();
	GrbClusterBuffers buffers = v->cluster.get_cluster_buffers();
	uint32_t *dev = nullptr;
	if (!Vulkan::cuda_ok(cudaMalloc(&dev, sizeof(uint32_t) * groups), "cudaMalloc"))
		return fail("cudaMalloc failed");
	int32_t rc = grb_lighting_row_cost(&depth, &cam, &params, &buffers, GrbRows{ 0, 0 }, dev, v->device->get_stream());
	bool ok = rc == GRB_OK && Vulkan::cuda_ok(cudaStreamSynchronize(reinterpret_cast<cudaStream_t>(v->device->get_stream())), "cudaStreamSynchronize") &&
	          Vulkan::cuda_ok(cudaMemcpy(out, dev, sizeof(uint32_t) * groups, cudaMemcpyDeviceToHost), "cudaMemcpy");
	cudaFree(dev);
	if (!ok)
		return fail(rc != GRB_OK ? grb_last_error_string() : "grbh_viewer_measure_row_cost: copy failed");
	return groups;
	GRBH_CATCH
}

extern "C" int32_t grbh_viewer_get_pass_names(GrbhViewer *v, char *buffer, int32_t capacity)
{
	if (!v || !v->baked)
		return fail("viewer not baked");
	GRBH_TRY
	std::string all;
	for (auto &n : v->graph.get_baked_pass_names())
		all += n + "\n";
	if (buffer && capacity > 0)
		std::snprintf(buffer, (size_t)capacity, "%s", all.c_str());
	return (int32_t)all.size() + 1;
	GRBH_CATCH
}

extern "C" int32_t grbh_viewer_collect_timings(GrbhViewer *v, char *names, int32_t names_capacity, float *total_ms, int32_t *counts, int32_t capacity)
{
	if (!v)
		return fail("null viewer");
	std::string all;
	int i = 0;
	for (auto &kv : v->timings)
	{
		if (i < capacity)
		{
			if (total_ms)
				total_ms[i] = (float)kv.second.first;
			if (counts)
				counts[i] = kv.second.second;
		}
		all += kv.first + "\n";
		i++;
	}
	if (names && names_capacity > 0)
		std::snprintf(names, (size_t)names_capacity, "%s", all.c_str());
	v->timings.clear();
	return i;
}
