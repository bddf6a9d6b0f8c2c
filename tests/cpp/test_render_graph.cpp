// CPU-only checks of the RenderGraph declaration surface / bake logic (no device is touched:
// bake() only needs one when a pass interface wants setup(device)).
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../granite_b200/host/post/aa.hpp"
#include "../../granite_b200/host/post/fxaa.hpp"
#include "../../granite_b200/host/post/hdr.hpp"
#include "../../granite_b200/host/post/smaa.hpp"
#include "../../granite_b200/host/render_graph.hpp"

using namespace Granite;

#define CHECK(cond)                                                         \
	do                                                                      \
	{                                                                       \
		if (!(cond))                                                        \
		{                                                                   \
			std::fprintf(stderr, "FAIL %s:%d: %s\n", __FILE__, __LINE__, #cond); \
			std::exit(1);                                                   \
		}                                                                   \
	} while (0)

template <typename F>
static bool throws_logic_error(F &&f)
{
	try
	{
		f();
	}
	catch (const std::logic_error &)
	{
		return true;
	}
	return false;
}

static std::string join(const std::vector<std::string> &v)
{
	std::string s;
	for (auto &x : v)
		s += x + ",";
	return s;
}

int main(int argc, char **argv)
{
	ResourceDimensions dim;
	dim.width = 3840;
	dim.height = 2160;
	dim.format = VK_FORMAT_R8G8B8A8_SRGB;

	// --- add_pass is idempotent by name; declarators build the dependency DAG ---
	{
		RenderGraph graph;
		graph.set_backbuffer_dimensions(dim);
		auto &a = graph.add_pass("a", RENDER_GRAPH_QUEUE_GRAPHICS_BIT);
		CHECK(&a == &graph.add_pass("a", RENDER_GRAPH_QUEUE_COMPUTE_BIT));
		CHECK(graph.find_pass("a") == &a && graph.find_pass("zzz") == nullptr);
		AttachmentInfo hdr;
		hdr.format = VK_FORMAT_B10G11R11_UFLOAT_PACK32;
		a.add_color_output("HDR-main", hdr);
		// a pass that does not contribute to the backbuffer is culled
		auto &unused = graph.add_pass("unused", RENDER_GRAPH_QUEUE_COMPUTE_BIT);
		BufferInfo bi;
		bi.size = 64;
		unused.add_storage_output("junk", bi);
		FrameParameters frame;
		HDROptions opts;
		setup_hdr_postprocess_compute(graph, frame, "HDR-main", "tonemapped", opts);
		setup_fxaa_postprocess(graph, "tonemapped", "post-aa-output");
		graph.set_backbuffer_source("post-aa-output");
		graph.bake();
		CHECK(join(graph.get_baked_pass_names()) == "a,bloom-compute,tonemap,fxaa,");

		// ceil(parent * scale) sizing (render_graph.cpp:3160-3171), incl. the non-2:1 step 135 -> 68
		auto size_of = [&](const char *name) {
			auto d = graph.get_resource_dimensions(graph.get_texture_resource(name));
			return std::make_pair(d.width, d.height);
		};
		CHECK(size_of("threshold") == std::make_pair(1920u, 1080u));
		CHECK(size_of("downsample-0") == std::make_pair(960u, 540u));
		CHECK(size_of("downsample-2") == std::make_pair(240u, 135u));
		CHECK(size_of("downsample-3") == std::make_pair(120u, 68u));
		CHECK(size_of("tonemapped") == std::make_pair(3840u, 2160u));
		// undefined formats inherit the backbuffer's
		CHECK(graph.get_resource_dimensions(graph.get_texture_resource("tonemapped")).format == VK_FORMAT_R8G8B8A8_SRGB);
		// FXAA flags its input for a UNORM alias view
		CHECK(graph.get_texture_resource("tonemapped").get_attachment_info().flags & ATTACHMENT_INFO_UNORM_SRGB_ALIAS_BIT);
		// physical indices: outputs distinct, culled resources unassigned
		CHECK(graph.get_texture_resource("threshold").get_physical_index() != graph.get_texture_resource("downsample-0").get_physical_index());
		CHECK(graph.get_buffer_resource("junk").get_physical_index() == RenderResource::Unused);
	}

	// --- 1080p pyramid: 1920x1080 -> 960x540, 480x270, 240x135, 120x68, 60x34 ---
	{
		RenderGraph graph;
		ResourceDimensions d2 = dim;
		d2.width = 1920;
		d2.height = 1080;
		graph.set_backbuffer_dimensions(d2);
		AttachmentInfo hdr;
		hdr.format = VK_FORMAT_B10G11R11_UFLOAT_PACK32;
		graph.add_pass("a", RENDER_GRAPH_QUEUE_GRAPHICS_BIT).add_color_output("HDR-main", hdr);
		FrameParameters frame;
		setup_hdr_postprocess(graph, frame, "HDR-main", "tonemapped", HDROptions{});
		graph.set_backbuffer_source("tonemapped");
		graph.bake();
		auto d3 = graph.get_resource_dimensions(graph.get_texture_resource("downsample-3"));
		CHECK(d3.width == 60 && d3.height == 34);
	}

	// --- read-modify-write aliasing shares the physical image ---
	{
		RenderGraph graph;
		graph.set_backbuffer_dimensions(dim);
		AttachmentInfo info;
		info.format = VK_FORMAT_B10G11R11_UFLOAT_PACK32;
		graph.add_pass("gbuffer", RENDER_GRAPH_QUEUE_GRAPHICS_BIT).add_color_output("emissive", info);
		graph.add_pass("lighting", RENDER_GRAPH_QUEUE_GRAPHICS_BIT).add_color_output("HDR-main", info, "emissive");
		graph.set_backbuffer_source("HDR-main");
		graph.bake();
		CHECK(graph.get_texture_resource("emissive").get_physical_index() == graph.get_texture_resource("HDR-main").get_physical_index());
		CHECK(join(graph.get_baked_pass_names()) == "gbuffer,lighting,");
	}

	// --- misuse throws std::logic_error like the reference ---
	{
		RenderGraph graph;
		graph.set_backbuffer_dimensions(dim);
		AttachmentInfo info;
		graph.add_pass("a", RENDER_GRAPH_QUEUE_GRAPHICS_BIT).add_color_output("out", info);
		graph.set_backbuffer_source("nope");
		CHECK(throws_logic_error([&] { graph.bake(); }));
		graph.set_backbuffer_source("out");
		graph.find_pass("a")->add_texture_input("never-written");
		CHECK(throws_logic_error([&] { graph.bake(); }));
	}
	{
		RenderGraph graph; // cycle a -> b -> a
		graph.set_backbuffer_dimensions(dim);
		AttachmentInfo info;
		auto &a = graph.add_pass("a", RENDER_GRAPH_QUEUE_GRAPHICS_BIT);
		auto &b = graph.add_pass("b", RENDER_GRAPH_QUEUE_GRAPHICS_BIT);
		a.add_color_output("x", info);
		a.add_texture_input("y");
		b.add_color_output("y", info);
		b.add_texture_input("x");
		graph.set_backbuffer_source("x");
		CHECK(throws_logic_error([&] { graph.bake(); }));
	}
	{
		RenderGraph graph; // executing before bake
		Vulkan::Device *none = nullptr;
		TaskComposer composer;
		CHECK(throws_logic_error([&] { graph.enqueue_render_passes(*none, composer); }));
		CHECK(throws_logic_error([&] { graph.set_row_shards({ GrbRows{ 0, 100 }, GrbRows{ 120, 200 } }, 0, nullptr); }));
	}

	// --- row shards scale per resource and tile every level exactly ---
	{
		struct NoCollectives : RenderGraphCollectives
		{
			unsigned get_rank() const override { return 0; }
			unsigned get_world_size() const override { return 8; }
			bool all_gather_rows(Vulkan::CommandBuffer &, Vulkan::ImageView &, const std::vector<GrbRows> &) override { return true; }
			bool all_reduce_sum(Vulkan::CommandBuffer &, float *, size_t) override { return true; }
		} coll;
		RenderGraph graph;
		graph.set_backbuffer_dimensions(dim);
		std::vector<GrbRows> bands;
		for (int r = 0; r < 8; r++)
			bands.push_back(GrbRows{ r * 256, r == 7 ? 2160 : (r + 1) * 256 });
		graph.set_row_shards(bands, 3, &coll);
		CHECK(graph.is_sharded() && graph.get_shard_count() == 8 && graph.get_shard_rank() == 3);
		for (unsigned hgt : { 2160u, 1080u, 540u })
		{
			int expect = 0;
			for (unsigned r = 0; r < 8; r++)
			{
				GrbRows rows = graph.shard_rows_for_rank(r, hgt);
				CHECK(rows.y0 == expect);
				expect = rows.y1;
			}
			CHECK(expect == (int)hgt);
		}
		GrbRows halo = graph.shard_rows_for(2160, 8);
		CHECK(halo.y0 == 3 * 256 - 8 && halo.y1 == 4 * 256 + 8);
		GrbRows edge = graph.shard_rows_for_rank(0, 2160, 8);
		CHECK(edge.y0 == 0 && edge.y1 == 264);
	}

	// --- PostAAType dispatch ---
	{
		CHECK(post_aa_type_is_supported(PostAAType::TAA_High) && post_aa_type_is_supported(PostAAType::SMAA_Ultra));
		CHECK(!post_aa_type_is_supported(PostAAType::SMAA_Ultra_T2X) && !post_aa_type_is_supported(PostAAType::FXAA_2Phase));
		RenderGraph graph;
		graph.set_backbuffer_dimensions(dim);
		TemporalJitter jitter;
		CHECK(throws_logic_error([&] { setup_after_post_chain_antialiasing(PostAAType::SMAA_Ultra_T2X, graph, jitter, 1.0f, "a", "d", "o"); }));
		CHECK(throws_logic_error([&] { setup_after_post_chain_antialiasing(PostAAType::FXAA_2Phase, graph, jitter, 1.0f, "a", "d", "o"); }));
		CHECK(!setup_before_post_chain_antialiasing(PostAAType::FXAA, graph, jitter, 1.0f, "a", "d", "mv", "o"));
		CHECK(setup_before_post_chain_antialiasing(PostAAType::TAA_High, graph, jitter, 1.0f, "HDR-main", "depth", "mv", "HDR-resolved"));
		CHECK(graph.find_pass("taa-resolve") != nullptr);
		// 16-phase table: phases cycle, matrices are pure sub-pixel translations
		mat4 p = perspective(0.785398f, 16.0f / 9.0f, 0.0625f, InfiniteFarPlane), v(1.0f);
		for (int i = 0; i < 40; i++)
		{
			jitter.step(p, v);
			CHECK(jitter.get_jitter_phase() < 16);
			const mat4 &j = jitter.get_jitter_matrix();
			CHECK(j[0][0] == 1.0f && j[1][1] == 1.0f && std::fabs(j[3][0]) <= 1.0f / 3840.0f + 1e-9f && std::fabs(j[3][1]) <= 1.0f / 2160.0f + 1e-9f);
		}
	}
	// --- proxies order passes that share no memory; raster-stage buffer inputs are read dependencies ---
	{
		RenderGraph graph;
		graph.set_backbuffer_dimensions(dim);
		AttachmentInfo info;
		info.format = VK_FORMAT_B10G11R11_UFLOAT_PACK32;
		BufferInfo bi;
		bi.size = 256;
		auto &final_pass = graph.add_pass("final", RENDER_GRAPH_QUEUE_GRAPHICS_BIT); // declared first: order must come from the DAG
		auto &prep = graph.add_pass("prep", RENDER_GRAPH_QUEUE_ASYNC_COMPUTE_BIT);
		auto &geometry = graph.add_pass("geometry", RENDER_GRAPH_QUEUE_COMPUTE_BIT);
		graph.add_pass("a", RENDER_GRAPH_QUEUE_GRAPHICS_BIT).add_color_output("HDR-main", info);
		prep.add_proxy_output("prep-done", VK_PIPELINE_STAGE_2_COMPUTE_SHADER_BIT, VK_ACCESS_2_SHADER_STORAGE_WRITE_BIT);
		geometry.add_storage_output("vertices", bi);
		geometry.add_storage_output("indices", bi);
		geometry.add_storage_output("draws", bi);
		final_pass.add_color_output("out", info);
		final_pass.add_texture_input("HDR-main");
		final_pass.add_proxy_input("prep-done", VK_PIPELINE_STAGE_FRAGMENT_SHADER_BIT, VK_ACCESS_2_SHADER_SAMPLED_READ_BIT);
		final_pass.add_vertex_buffer_input("vertices");
		final_pass.add_index_buffer_input("indices");
		final_pass.add_indirect_buffer_input("draws");
		CHECK(throws_logic_error([&] { final_pass.add_proxy_input("x", 0, 0); }));
		graph.set_backbuffer_source("out");
		graph.bake();
		auto names = graph.get_baked_pass_names();
		CHECK(names.size() == 4 && names.back() == "final");
		auto has = [&](const char *n) { return std::find(names.begin(), names.end(), std::string(n)) != names.end(); };
		CHECK(has("prep") && has("geometry") && has("a"));
		CHECK(graph.get_buffer_resource("prep-done").is_proxy() && !graph.get_buffer_resource("vertices").is_proxy());
	}

	// --- external locks: a no-op until an interface is registered under the name (render_graph.cpp:390-411) ---
	{
		struct ShadowAtlas : RenderPassExternalLockInterface
		{
			const char *get_ident() const override { return "shadow-atlas"; }
		} atlas;
		RenderGraph graph;
		graph.set_backbuffer_dimensions(dim);
		AttachmentInfo info;
		auto &lighting = graph.add_pass("lighting", RENDER_GRAPH_QUEUE_GRAPHICS_BIT);
		lighting.add_color_output("HDR-main", info);
		lighting.add_external_lock("bindless-shadowmaps", VK_PIPELINE_STAGE_FRAGMENT_SHADER_BIT, VK_ACCESS_2_SHADER_SAMPLED_READ_BIT);
		CHECK(lighting.get_lock_interfaces().empty() && graph.find_external_lock_interface("bindless-shadowmaps") == nullptr);
		graph.add_external_lock_interface("bindless-shadowmaps", &atlas);
		lighting.add_external_lock("bindless-shadowmaps", VK_PIPELINE_STAGE_FRAGMENT_SHADER_BIT, VK_ACCESS_2_SHADER_SAMPLED_READ_BIT);
		lighting.add_external_lock("bindless-shadowmaps", VK_PIPELINE_STAGE_2_COMPUTE_SHADER_BIT, VK_ACCESS_2_SHADER_SAMPLED_READ_BIT);
		CHECK(lighting.get_lock_interfaces().size() == 1 && lighting.get_lock_interfaces()[0].iface == &atlas);
		CHECK(lighting.get_lock_interfaces()[0].stages == (VK_PIPELINE_STAGE_FRAGMENT_SHADER_BIT | VK_PIPELINE_STAGE_2_COMPUTE_SHADER_BIT));
		CHECK(atlas.has_foreign_access() && atlas.external_acquire_event() == nullptr); // nothing produced yet: nothing to wait for
		graph.reset();
		CHECK(graph.find_external_lock_interface("bindless-shadowmaps") == nullptr);
	}

	// --- HDR10 output: lit scene + UI layer -> "pq10" (renderer/post/hdr.cpp:595-658) ---
	{
		RenderGraph graph;
		graph.set_backbuffer_dimensions(dim);
		AttachmentInfo hdr;
		hdr.format = VK_FORMAT_B10G11R11_UFLOAT_PACK32;
		graph.add_pass("lighting", RENDER_GRAPH_QUEUE_GRAPHICS_BIT).add_color_output("HDR-main", hdr);
		AttachmentInfo ui;
		ui.format = VK_FORMAT_R8G8B8A8_UNORM;
		auto &ui_pass = graph.add_pass("ui", RENDER_GRAPH_QUEUE_GRAPHICS_BIT);
		ui_pass.add_color_output("ui-temporary", ui);
		ui_pass.add_texture_input("HDR-main");
		VkHdrMetadataEXT rec709 = {};
		rec709.displayPrimaryRed = { 0.640f, 0.330f };
		rec709.displayPrimaryGreen = { 0.3f, 0.6f };
		rec709.displayPrimaryBlue = { 0.150f, 0.060f };
		rec709.whitePoint = { 0.3127f, 0.3290f };
		rec709.maxContentLightLevel = 1000.0f;
		setup_hdr10_pq_encoding(graph, "ui-output", "HDR-main", "ui-temporary", HDR10PQEncodingConfig{ 500.0f, 400.0f }, rec709);
		graph.set_backbuffer_source("ui-output");
		graph.bake();
		CHECK(join(graph.get_baked_pass_names()) == "lighting,ui,pq10,");
		auto out = graph.get_resource_dimensions(graph.get_texture_resource("ui-output"));
		CHECK(out.format == VK_FORMAT_A2B10G10R10_UNORM_PACK32 && out.width == 3840 && out.height == 2160);
		// Rec.709 -> Rec.709 is the identity; BT.2020 rows sum to 1 (white stays white)
		mat4 ident = compute_rec709_to_display_primaries(rec709);
		for (int c = 0; c < 4; c++)
			for (int r = 0; r < 4; r++)
				CHECK(std::fabs(ident[c][r] - (c == r ? 1.0f : 0.0f)) < 2e-7f);
		VkHdrMetadataEXT bt2020 = rec709;
		bt2020.displayPrimaryRed = { 0.708f, 0.292f };
		bt2020.displayPrimaryGreen = { 0.170f, 0.797f };
		bt2020.displayPrimaryBlue = { 0.131f, 0.046f };
		mat4 m = compute_rec709_to_display_primaries(bt2020);
		for (int r = 0; r < 3; r++)
			CHECK(std::fabs(m[0][r] + m[1][r] + m[2][r] - 1.0f) < 1e-6f);
		CHECK(m[0][0] > 0.62f && m[0][0] < 0.63f); // 0.6274: the familiar BT.709 -> BT.2020 coefficient
	}

	// --- SMAA: three passes behind the tonemap (renderer/post/smaa.cpp:32-209), formats and sizes of the intermediates ---
	{
		RenderGraph graph;
		graph.set_backbuffer_dimensions(dim);
		AttachmentInfo hdr;
		hdr.format = VK_FORMAT_B10G11R11_UFLOAT_PACK32;
		graph.add_pass("lighting", RENDER_GRAPH_QUEUE_GRAPHICS_BIT).add_color_output("HDR-main", hdr);
		FrameParameters frame;
		setup_hdr_postprocess(graph, frame, "HDR-main", "tonemapped", HDROptions{});
		TemporalJitter jitter;
		CHECK(setup_after_post_chain_antialiasing(PostAAType::SMAA_High, graph, jitter, 1.0f, "tonemapped", "depth", "post-aa-output"));
		graph.set_backbuffer_source("post-aa-output");
		graph.bake();
		CHECK(join(graph.get_baked_pass_names()) == "lighting,bloom-compute,tonemap,smaa-edge,smaa-weights,smaa-blend,");
		auto e = graph.get_resource_dimensions(graph.get_texture_resource("smaa-edge"));
		auto w = graph.get_resource_dimensions(graph.get_texture_resource("smaa-weights"));
		auto o = graph.get_resource_dimensions(graph.get_texture_resource("post-aa-output"));
		CHECK(e.format == VK_FORMAT_R8G8_UNORM && e.width == 3840 && e.height == 2160);
		CHECK(w.format == VK_FORMAT_R8G8B8A8_UNORM && w.width == 3840);
		CHECK(o.format == VK_FORMAT_R8G8B8A8_SRGB); // undefined format: the backbuffer's
		CHECK(graph.get_texture_resource("tonemapped").get_attachment_info().flags & ATTACHMENT_INFO_UNORM_SRGB_ALIAS_BIT);
		CHECK(jitter.get_jitter_type() == TemporalJitter::Type::None);
	}
	// --- FSR 1 behind a scaled-down scene (renderer/post/aa.cpp:75-174): "resolutionScale" 0.75 of a 4K swapchain ---
	{
		RenderGraph graph;
		graph.set_backbuffer_dimensions(dim);
		AttachmentInfo hdr;
		hdr.format = VK_FORMAT_B10G11R11_UFLOAT_PACK32;
		hdr.size_x = hdr.size_y = 0.75f;
		graph.add_pass("lighting", RENDER_GRAPH_QUEUE_GRAPHICS_BIT).add_color_output("HDR-main", hdr);
		FrameParameters frame;
		setup_hdr_postprocess(graph, frame, "HDR-main", "tonemapped", HDROptions{});
		CHECK(setup_after_post_chain_upscaling(graph, "tonemapped", "post-scale-output", true));
		graph.set_backbuffer_source("post-scale-output");
		graph.bake();
		CHECK(join(graph.get_baked_pass_names()) == "lighting,bloom-compute,tonemap,post-scale-output-scale,post-scale-output-sharpen,");
		auto t = graph.get_resource_dimensions(graph.get_texture_resource("tonemapped"));
		auto u = graph.get_resource_dimensions(graph.get_texture_resource("post-scale-output-scale"));
		auto o = graph.get_resource_dimensions(graph.get_texture_resource("post-scale-output"));
		CHECK(t.width == 2880 && t.height == 1620);
		CHECK(u.format == VK_FORMAT_R8G8B8A8_UNORM && u.width == 3840 && u.height == 2160);
		CHECK(o.format == VK_FORMAT_R8G8B8A8_SRGB && o.width == 3840 && o.height == 2160);
		CHECK(graph.get_texture_resource("tonemapped").get_attachment_info().flags & ATTACHMENT_INFO_UNORM_SRGB_ALIAS_BIT);
	}
	{
		// without the sharpen pass the upscale writes `output` itself, as R8G8B8A8_UNORM (aa.cpp:80-84)
		RenderGraph graph;
		graph.set_backbuffer_dimensions(dim);
		AttachmentInfo hdr;
		hdr.format = VK_FORMAT_B10G11R11_UFLOAT_PACK32;
		hdr.size_x = hdr.size_y = 0.5f;
		graph.add_pass("lighting", RENDER_GRAPH_QUEUE_GRAPHICS_BIT).add_color_output("HDR-main", hdr);
		FrameParameters frame;
		setup_hdr_postprocess(graph, frame, "HDR-main", "tonemapped", HDROptions{});
		CHECK(setup_after_post_chain_upscaling(graph, "tonemapped", "post-scale-output", false));
		graph.set_backbuffer_source("post-scale-output");
		graph.bake();
		CHECK(join(graph.get_baked_pass_names()) == "lighting,bloom-compute,tonemap,post-scale-output-scale,");
		auto o = graph.get_resource_dimensions(graph.get_texture_resource("post-scale-output"));
		CHECK(o.format == VK_FORMAT_R8G8B8A8_UNORM && o.width == 3840 && o.height == 2160);
	}

	// --- the .gtx container the lookup textures come in (vulkan/texture/memory_mapped_texture.cpp:29-46) ---
	{
		std::vector<uint8_t> file(64 + 4 * 3 * 2, 0);
		std::memcpy(file.data(), "GRANITE TEXFMT1", 16);
		const uint32_t header[8] = { 1u, (uint32_t)VK_FORMAT_R8G8_UNORM, 4u, 3u, 1u, 1u, 1u, 0u };
		std::memcpy(file.data() + 16, header, sizeof(header));
		const uint64_t payload = 4 * 3 * 2;
		std::memcpy(file.data() + 48, &payload, 8);
		for (size_t i = 64; i < file.size(); i++)
			file[i] = (uint8_t)(i - 64);
		GtxImage img;
		std::string err;
		CHECK(parse_gtx(file.data(), file.size(), img, err));
		CHECK(img.format == VK_FORMAT_R8G8_UNORM && img.width == 4 && img.height == 3 && img.texels.size() == 24 && img.texels[23] == 23);
		CHECK(!parse_gtx(file.data(), 63, img, err) && !parse_gtx(file.data(), file.size() - 1, img, err));
		file[0] = 'X';
		CHECK(!parse_gtx(file.data(), file.size(), img, err));
		// the reference's SMAA lookup textures, from the directory given as the first argument
		if (argc > 1)
		{
			const std::string dir = argv[1];
			GtxImage area, search;
			CHECK(load_gtx(dir + "/area.gtx", area, err) && load_gtx(dir + "/search.gtx", search, err));
			CHECK(area.format == VK_FORMAT_R8G8_UNORM && area.width == 160 && area.height == 560 && area.texels.size() == 160u * 560u * 2u);
			CHECK(search.format == VK_FORMAT_R8_UNORM && search.width == 64 && search.height == 16 && search.texels.size() == 1024u);
		}
	}

	// --- queues map to streams: main, cluster build, tonemap / AA, bloom ---
	{
		CHECK(RenderGraph::queue_stream_index(RENDER_GRAPH_QUEUE_GRAPHICS_BIT) == 0 && RenderGraph::queue_stream_index(RENDER_GRAPH_QUEUE_COMPUTE_BIT) == 0);
		CHECK(RenderGraph::queue_stream_index(RENDER_GRAPH_QUEUE_ASYNC_COMPUTE_BIT) == 1);
		CHECK(RenderGraph::queue_stream_index(RENDER_GRAPH_QUEUE_ASYNC_GRAPHICS_BIT) == 2);
		CHECK(RenderGraph::queue_stream_index(RENDER_GRAPH_QUEUE_ASYNC_POST_COMPUTE_BIT) == 3);
		RenderGraph::set_async_post(true);
		CHECK(RenderGraph::get_default_compute_queue() != RenderGraph::get_default_post_graphics_queue());
		RenderGraph::set_async_post(false);
		CHECK(RenderGraph::get_default_compute_queue() == RENDER_GRAPH_QUEUE_COMPUTE_BIT);
	}
	std::printf("render graph checks passed\n");
	return 0;
}
