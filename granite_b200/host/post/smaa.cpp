// smaa.cpp -- "smaa-edge" / "smaa-weights" / "smaa-blend" pass builders (renderer/post/smaa.cpp:32-209), the lookup
// textures they sample and the .gtx reader for them.
#include "smaa.hpp"

#include <cuda_runtime.h>

#include <cstdio>
#include <algorithm>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <stdexcept>

namespace Granite
{
namespace
{
struct Lookup
{
	Vulkan::ImageHandle area, search;
};
std::mutex g_lookup_lock;
std::map<Vulkan::Device *, Lookup> g_lookup;

constexpr unsigned kAreaW = 160, kAreaH = 560, kSearchW = 64, kSearchH = 16;
} // namespace

bool set_smaa_lookup_textures(Vulkan::Device &device, const uint8_t *area_rg8, const uint8_t *search_r8)
{
	if (!area_rg8 || !search_r8)
		return false;
	Lookup l;
	Vulkan::ImageCreateInfo info;
	info.width = kAreaW;
	info.height = kAreaH;
	info.format = VK_FORMAT_R8G8_UNORM;
	l.area = device.create_image(info);
	info.width = kSearchW;
	info.height = kSearchH;
	info.format = VK_FORMAT_R8_UNORM;
	l.search = device.create_image(info);
	// once per device, before the first frame: plain synchronous copies
	if (!Vulkan::cuda_ok(cudaMemcpy(l.area->get_device_pointer(), area_rg8, (size_t)kAreaW * kAreaH * 2, cudaMemcpyHostToDevice), "SMAA area texture upload") ||
	    !Vulkan::cuda_ok(cudaMemcpy(l.search->get_device_pointer(), search_r8, (size_t)kSearchW * kSearchH, cudaMemcpyHostToDevice), "SMAA search texture upload"))
		return false;
	std::lock_guard<std::mutex> hold(g_lookup_lock);
	g_lookup[&device] = std::move(l);
	return true;
}

bool get_smaa_lookup_textures(Vulkan::Device &device, GrbImage *area, GrbImage *search)
{
	std::lock_guard<std::mutex> hold(g_lookup_lock);
	auto itr = g_lookup.find(&device);
	if (itr == g_lookup.end())
		return false;
	*area = Vulkan::ImageView(itr->second.area).as_grb();
	*search = Vulkan::ImageView(itr->second.search).as_grb();
	return true;
}

void release_smaa_lookup_textures(Vulkan::Device &device)
{
	std::lock_guard<std::mutex> hold(g_lookup_lock);
	g_lookup.erase(&device);
}

bool parse_gtx(const uint8_t *bytes, size_t size, GtxImage &out, std::string &error)
{
	static const char magic[16] = "GRANITE TEXFMT1";
	if (!bytes || size < 64 || std::memcmp(bytes, magic, 16) != 0)
	{
		error = "not a GRANITE TEXFMT1 container";
		return false;
	}
	uint32_t h[8];
	uint64_t payload = 0;
	std::memcpy(h, bytes + 16, sizeof(h));
	std::memcpy(&payload, bytes + 48, 8);
	const uint32_t type = h[0], format = h[1], width = h[2], height = h[3], depth = h[4], layers = h[5], levels = h[6];
	if (type != 1 /* VK_IMAGE_TYPE_2D */ || depth != 1 || layers != 1 || levels != 1 || width == 0 || height == 0)
	{
		error = "only single-level, single-layer 2-D images are read";
		return false;
	}
	const unsigned texel = format_texel_size((VkFormat)format);
	if (!texel)
	{
		error = "texel format not handled by this executor";
		return false;
	}
	const size_t need = (size_t)width * height * texel;
	if (payload < need || size < 64 + need)
	{
		error = "payload shorter than width x height texels";
		return false;
	}
	out.format = (VkFormat)format;
	out.width = width;
	out.height = height;
	out.texels.assign(bytes + 64, bytes + 64 + need);
	return true;
}

bool load_gtx(const std::string &path, GtxImage &out, std::string &error)
{
	std::FILE *f = std::fopen(path.c_str(), "rb");
	if (!f)
	{
		error = "cannot open " + path;
		return false;
	}
	std::vector<uint8_t> bytes;
	uint8_t chunk[65536];
	size_t n;
	while ((n = std::fread(chunk, 1, sizeof(chunk), f)) > 0)
		bytes.insert(bytes.end(), chunk, chunk + n);
	std::fclose(f);
	if (!parse_gtx(bytes.data(), bytes.size(), out, error))
	{
		error = path + ": " + error;
		return false;
	}
	return true;
}

bool load_smaa_lookup_textures(Vulkan::Device &device, const std::string &directory, std::string &error)
{
	GtxImage area, search;
	if (!load_gtx(directory + "/area.gtx", area, error) || !load_gtx(directory + "/search.gtx", search, error))
		return false;
	if (area.format != VK_FORMAT_R8G8_UNORM || area.width != kAreaW || area.height != kAreaH || search.format != VK_FORMAT_R8_UNORM || search.width != kSearchW ||
	    search.height != kSearchH)
	{
		error = "area.gtx must be 160x560 R8G8_UNORM and search.gtx 64x16 R8_UNORM";
		return false;
	}
	if (!set_smaa_lookup_textures(device, area.texels.data(), search.texels.data()))
	{
		error = "upload of the SMAA lookup textures failed";
		return false;
	}
	return true;
}

void setup_smaa_postprocess(RenderGraph &graph, TemporalJitter &jitter, float, const std::string &input, const std::string &, const std::string &output,
                            SMAAPreset preset)
{
	if (preset == SMAAPreset::Ultra_T2X)
		throw std::logic_error("SMAA T2X (two jittered frames + smaa-t2x-resolve) is not built by this executor.");
	const int quality = preset == SMAAPreset::Low ? 0 : (preset == SMAAPreset::Medium ? 1 : (preset == SMAAPreset::High ? 2 : 3));
	jitter.init(TemporalJitter::Type::None, vec2(1.0f)); // smaa.cpp:66-67

	// the input is sampled through a UNORM view of its sRGB storage (smaa.cpp:70, 124, 178)
	graph.get_texture_resource(input).get_attachment_info().flags |= ATTACHMENT_INFO_UNORM_SRGB_ALIAS_BIT;

	AttachmentInfo edge_info;
	edge_info.size_class = SizeClass::InputRelative;
	edge_info.size_relative_name = input;
	edge_info.format = VK_FORMAT_R8G8_UNORM;
	AttachmentInfo weight_info = edge_info;
	weight_info.format = VK_FORMAT_R8G8B8A8_UNORM;
	AttachmentInfo final_info;
	final_info.size_class = SizeClass::InputRelative;
	final_info.size_relative_name = input;

	auto &smaa_edge = graph.add_pass("smaa-edge", RenderGraph::get_default_post_graphics_queue());
	auto &smaa_weight = graph.add_pass("smaa-weights", RenderGraph::get_default_post_graphics_queue());
	auto &smaa_blend = graph.add_pass("smaa-blend", RenderGraph::get_default_post_graphics_queue());

	// The reference also attaches a D16 "smaa-mask" to the first two passes (smaa.cpp:101-118, 148-149): both draw at
	// depth 0, which is the clear value, so the EQUAL test of the second pass keeps every pixel -- nothing to carry over.
	auto &edge_out = smaa_edge.add_color_output("smaa-edge", edge_info);
	auto &edge_input = smaa_edge.add_texture_input(input);
	auto &weight_out = smaa_weight.add_color_output("smaa-weights", weight_info);
	auto &weight_input = smaa_weight.add_texture_input("smaa-edge");
	auto &blend_out = smaa_blend.add_color_output(output, final_info);
	auto &blend_input = smaa_blend.add_texture_input(input);
	auto &blend_weights = smaa_blend.add_texture_input("smaa-weights");

	// Row-sharded frames (graph.get_shard_plan(): smaa_weights, smaa_edges): the weights pass of a rank walks edges up to
	// 2 * max_search_steps + 4 rows beyond its band, so the edges are exchanged rather than recomputed.  Each rank
	// detects the edges of its own band only; on the peer path "smaa-edge" stores every edge row into the slot of each
	// rank whose window (plan.smaa_edges) holds it and raises a flag on every rank, and "smaa-weights" waits for every
	// rank's flag of this frame, then reads this rank's slot.  Two slots suffice: the three passes share one stream (the
	// post-graphics queue), so a rank's frame N+1 edge pass runs after its frame N weights pass, which waited for every
	// rank's frame-N flag; each of those was raised after that rank's frame N-1 weights pass, the last reader of slot
	// (N+1) mod 2.  On the NCCL path "smaa-edge" writes the band into the graph's image and all-gathers the bands.
	// `edges_slot` carries this frame's slot from the edge pass to the weights pass (both record on this thread, in order).
	auto edges_slot = std::make_shared<RenderGraphCollectives::PeerSlot>();
	auto sharded = [&graph] { return graph.is_sharded() && graph.get_shard_count() > 1; };
	smaa_edge.set_build_render_pass([&graph, &edge_out, &edge_input, quality, edges_slot, sharded](Vulkan::CommandBuffer &cmd) {
		GrbImage color = graph.get_physical_texture_resource(edge_input).as_grb_unorm();
		GrbImage edges = graph.get_physical_texture_resource(edge_out).as_grb();
		*edges_slot = RenderGraphCollectives::PeerSlot{};
		if (!sharded())
		{
			cmd.check(grb_smaa_edge_detection(&color, quality, &edges, GrbRows{ 0, 0 }, cmd.get_stream_handle()), "grb_smaa_edge_detection");
			return;
		}
		const ShardPlan plan = graph.get_shard_plan();
		auto *collectives = graph.get_collectives();
		const unsigned self = collectives->get_rank(), count = graph.get_shard_count();
		RenderGraphCollectives::PeerSlot slot;
		if (collectives->smaa_edges_begin_frame((size_t)edges.row_pitch * (size_t)edges.height, slot))
		{
			// rank r receives the rows of this band its window holds (own ∩ smaa_edges of r; empty: y0 == y1)
			GrbRows peer_rows[GRB_MAX_PEERS] = {};
			for (unsigned r = 0; r < count; r++)
			{
				const GrbRows window = graph.get_shard_plan(r).smaa_edges;
				const int y0 = std::max(plan.own.y0, window.y0), y1 = std::min(plan.own.y1, window.y1);
				peer_rows[r] = y0 < y1 ? GrbRows{ y0, y1 } : GrbRows{ plan.own.y0, plan.own.y0 };
			}
			GrbImage layout = edges;
			layout.data = nullptr;
			cmd.check(grb_smaa_edge_detection_to_peers(&color, quality, &layout, slot.images, peer_rows, slot.flags, (int32_t)slot.count, (int32_t)self,
			                                           slot.epoch, slot.counter, plan.own, cmd.get_stream_handle()),
			          "grb_smaa_edge_detection_to_peers");
			*edges_slot = slot;
			return;
		}
		// NCCL path: this band into the graph's image, then every rank broadcasts its band
		cmd.check(grb_smaa_edge_detection(&color, quality, &edges, plan.own, cmd.get_stream_handle()), "grb_smaa_edge_detection");
		std::vector<GrbRows> bands;
		for (unsigned r = 0; r < count; r++)
			bands.push_back(graph.get_shard_plan(r).own);
		collectives->all_gather_rows(cmd, graph.get_physical_texture_resource(edge_out), bands);
	});
	smaa_weight.set_build_render_pass([&graph, &weight_out, &weight_input, quality, edges_slot, sharded](Vulkan::CommandBuffer &cmd) {
		GrbImage edges = graph.get_physical_texture_resource(weight_input).as_grb();
		GrbImage weights = graph.get_physical_texture_resource(weight_out).as_grb();
		GrbImage area, search;
		if (!get_smaa_lookup_textures(cmd.get_device(), &area, &search))
		{
			Vulkan::log_error("smaa-weights: no lookup textures on this device (set_smaa_lookup_textures / load_smaa_lookup_textures).\n");
			return;
		}
		GrbRows rows = GrbRows{ 0, 0 };
		if (sharded())
		{
			rows = graph.get_shard_plan().smaa_weights;
			if (edges_slot->count)
			{
				// peer path: every rank's edges of this frame have arrived in this rank's slot
				const unsigned self = graph.get_collectives()->get_rank();
				cmd.check(grb_peer_wait(edges_slot->flags[self], (int32_t)edges_slot->count, edges_slot->epoch, cmd.get_stream_handle()),
				          "grb_peer_wait(smaa edges)");
				edges.data = edges_slot->images[self];
			}
		}
		cmd.check(grb_smaa_blend_weights(&edges, &area, &search, quality, &weights, rows, cmd.get_stream_handle()), "grb_smaa_blend_weights");
	});
	smaa_blend.set_build_render_pass([&graph, &blend_out, &blend_input, &blend_weights, sharded](Vulkan::CommandBuffer &cmd) {
		GrbImage color = graph.get_physical_texture_resource(blend_input).as_grb_unorm();
		GrbImage weights = graph.get_physical_texture_resource(blend_weights).as_grb();
		GrbImage out = graph.get_physical_texture_resource(blend_out).as_grb(); // SMAA_TARGET_SRGB follows the output format (smaa.cpp:193-194)
		const GrbRows rows = sharded() ? graph.get_shard_plan().own : GrbRows{ 0, 0 };
		cmd.check(grb_smaa_neighborhood_blend(&color, &weights, &out, rows, cmd.get_stream_handle()), "grb_smaa_neighborhood_blend");
	});
}
} // namespace Granite
