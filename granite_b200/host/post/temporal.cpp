// temporal.cpp -- sub-pixel jitter sequences and the "taa-resolve" pass builder
// (renderer/post/temporal.cpp:40-266).  The jitter tables are data (sample positions in 1/8
// pixel units) and are reproduced as such; everything else is written against this executor.
#include "temporal.hpp"

#include <cstring>

namespace Granite
{
TemporalJitter::TemporalJitter()
{
	init(Type::None, vec2(0.0f));
}

void TemporalJitter::init_banks()
{
	saved_jittered_view_proj.assign(jitter_count, mat4(1.0f));
	saved_jittered_inv_view_proj.assign(jitter_count, mat4(1.0f));
	saved_view_proj.assign(jitter_count, mat4(1.0f));
	saved_inv_view_proj.assign(jitter_count, mat4(1.0f));
}

void TemporalJitter::init_custom(const vec2 *phases, unsigned phase_count, vec2 res)
{
	jitter_table.clear();
	for (unsigned i = 0; i < phase_count; i++)
		jitter_table.push_back(translate(vec3(phases[i].x / res.x, phases[i].y / res.y, 0.0f) * 2.0f));
	jitter_count = phase_count;
	type = Type::Custom;
	phase = 0;
	init_banks();
}

namespace
{
// sample offsets in 1/8 pixel (temporal.cpp:89-124)
const int kTaa8[8][2] = { { -7, 1 }, { -5, -5 }, { -1, -3 }, { 3, -7 }, { -5, -1 }, { 7, 7 }, { 1, 3 }, { -3, 5 } };
const int kTaa16[16][2] = { { -8, 0 }, { -6, -4 }, { -3, -2 }, { -2, -6 }, { 1, -1 }, { 2, -5 }, { 6, -7 }, { 5, -3 },
	                        { 4, 1 },  { 7, 4 },   { 3, 5 },   { 0, 7 },   { -1, 3 }, { -4, 6 }, { -7, 8 }, { -5, 2 } };
} // namespace

void TemporalJitter::init(Type type_, vec2 res)
{
	type = type_;
	phase = 0;
	jitter_table.clear();
	auto eighth = [&](const int (*tab)[2], unsigned n) {
		for (unsigned i = 0; i < n; i++)
			jitter_table.push_back(translate(vec3(float(tab[i][0]) / res.x, float(tab[i][1]) / res.y, 0.0f) * 0.125f));
	};
	switch (type)
	{
	case Type::FXAA_2Phase:
		jitter_table.push_back(translate(vec3(0.5f / res.x, 0.0f, 0.0f) * 2.0f));
		jitter_table.push_back(translate(vec3(0.0f, 0.5f / res.y, 0.0f) * 2.0f));
		break;
	case Type::SMAA_T2X:
		jitter_table.push_back(translate(vec3(-0.25f / res.x, -0.25f / res.y, 0.0f) * 2.0f));
		jitter_table.push_back(translate(vec3(+0.25f / res.x, +0.25f / res.y, 0.0f) * 2.0f));
		break;
	case Type::TAA_8Phase:
		eighth(kTaa8, 8);
		break;
	case Type::TAA_16Phase:
		eighth(kTaa16, 16);
		break;
	default:
		jitter_table.push_back(mat4(1.0f));
		break;
	}
	jitter_count = (unsigned)jitter_table.size();
	init_banks();
}

void TemporalJitter::step(const mat4 &proj, const mat4 &view)
{
	phase++;
	if (phase >= jitter_count)
		phase = 0;
	saved_view_proj[phase] = proj * view;
	saved_jittered_projection = get_jitter_matrix() * proj;
	saved_jittered_view_proj[phase] = get_jitter_matrix() * saved_view_proj[phase];
	saved_inv_view_proj[phase] = inverse(saved_view_proj[phase]);
	saved_jittered_inv_view_proj[phase] = inverse(saved_jittered_view_proj[phase]);
}

unsigned TemporalJitter::get_offset_phase(int frames) const
{
	if (phase >= unsigned(frames))
		return phase - frames;
	return jitter_count - frames;
}

const mat4 &TemporalJitter::get_jitter_matrix() const { return jitter_table[phase]; }
const mat4 &TemporalJitter::get_history_view_proj(int frames) const { return saved_view_proj[get_offset_phase(frames)]; }
const mat4 &TemporalJitter::get_history_inv_view_proj(int frames) const { return saved_inv_view_proj[get_offset_phase(frames)]; }
const mat4 &TemporalJitter::get_history_jittered_view_proj(int frames) const { return saved_jittered_view_proj[get_offset_phase(frames)]; }
const mat4 &TemporalJitter::get_history_jittered_inv_view_proj(int frames) const { return saved_jittered_inv_view_proj[get_offset_phase(frames)]; }

void setup_taa_resolve(RenderGraph &graph, TemporalJitter &jitter, float scaling_factor, const std::string &input, const std::string &input_depth,
                       const std::string &input_mv, const std::string &output, TAAQuality quality)
{
	jitter.init(TemporalJitter::Type::TAA_16Phase,
	            vec2(graph.get_backbuffer_dimensions().width * scaling_factor, graph.get_backbuffer_dimensions().height * scaling_factor));

	AttachmentInfo taa_output;
	taa_output.size_class = SizeClass::InputRelative;
	taa_output.size_relative_name = input;
	taa_output.format = VK_FORMAT_B10G11R11_UFLOAT_PACK32;
	AttachmentInfo taa_history = taa_output;
	taa_history.format = VK_FORMAT_R16G16B16A16_SFLOAT;

	auto &resolve = graph.add_pass("taa-resolve", RENDER_GRAPH_QUEUE_GRAPHICS_BIT);
	auto &out_color = resolve.add_color_output(output, taa_output);
	auto &out_history = resolve.add_color_output(output + "-history", taa_history);
	auto &input_res = resolve.add_texture_input(input);
	auto &input_res_mv = resolve.add_texture_input(input_mv);
	auto &input_depth_res = resolve.add_texture_input(input_depth);
	auto &history = resolve.add_history_input(output + "-history");

	resolve.set_build_render_pass([&graph, &jitter, &out_color, &out_history, &input_res, &input_res_mv, &input_depth_res, &history,
	                               q = int(quality)](Vulkan::CommandBuffer &cmd) {
		GrbImage image = graph.get_physical_texture_resource(input_res).as_grb();
		GrbImage image_mv = graph.get_physical_texture_resource(input_res_mv).as_grb();
		GrbImage depth = graph.get_physical_texture_resource(input_depth_res).as_grb();
		auto *prev = graph.get_physical_history_texture_resource(history);
		GrbImage prev_img;
		if (prev)
			prev_img = prev->as_grb();
		GrbImage oc = graph.get_physical_texture_resource(out_color).as_grb();
		GrbImage oh = graph.get_physical_texture_resource(out_history).as_grb();

		// temporal.cpp:239-243: clip(now) -> UV(previous frame)
		mat4 reproj = translate(vec3(0.5f, 0.5f, 0.0f)) * scale(vec3(0.5f, 0.5f, 1.0f)) * jitter.get_history_view_proj(1) *
		              jitter.get_history_inv_view_proj(0);
		if (graph.is_sharded() && graph.get_shard_count() > 1)
		{
			// Row-sharded frames: a pixel reads last frame's history at its reprojected position, which can be anywhere
			// in the frame, so every rank holds the whole history.  This rank resolves plan.taa (what the threshold and
			// the tonemap read) and contributes the history of its own band.
			const ShardPlan plan = graph.get_shard_plan();
			auto *collectives = graph.get_collectives();
			const unsigned self = collectives->get_rank();
			RenderGraphCollectives::PeerSlot slot;
			void *previous = nullptr;
			if (collectives->taa_history_begin_frame((size_t)oh.row_pitch * (size_t)oh.height, slot, previous))
			{
				// Peer path: the resolve stores its band into this frame's slot on every rank, the previous frame's slot
				// is the history.  Two slots suffice: before its frame N+1 resolve a rank waits until every rank's
				// frame-N flag has arrived (it needs that wait anyway to read the history), and a rank raises that flag
				// at the end of its frame-N resolve, after reading slot (N-1) mod 2.  So by the time a rank stores into
				// slot (N+1) mod 2 on a peer, that peer has finished reading it.  The wait is kept on the first frame
				// after a re-bake too (no history is read then, but the slot is still reused).
				if (previous)
					cmd.check(grb_peer_wait(slot.flags[self], (int32_t)slot.count, slot.epoch - 1u, cmd.get_stream_handle()), "grb_peer_wait(taa history)");
				GrbImage full_history = oh;
				full_history.data = previous;
				cmd.check(grb_taa_resolve_to_peers(&image, &depth, &image_mv, prev && previous ? &full_history : nullptr, reproj.data(), q, &oc, &oh,
				                                   slot.images, slot.flags, (int32_t)slot.count, (int32_t)self, slot.epoch, slot.counter, plan.taa,
				                                   plan.own, cmd.get_stream_handle()),
				          "grb_taa_resolve_to_peers");
				return;
			}
			// NCCL path: resolve into the graph's history image, then every rank broadcasts its band of it
			cmd.check(grb_taa_resolve(&image, &depth, &image_mv, prev ? &prev_img : nullptr, reproj.data(), q, &oc, &oh, plan.taa, cmd.get_stream_handle()),
			          "grb_taa_resolve");
			std::vector<GrbRows> bands;
			for (unsigned rank = 0; rank < graph.get_shard_count(); rank++)
				bands.push_back(graph.get_shard_plan(rank).own);
			collectives->all_gather_rows(cmd, graph.get_physical_texture_resource(out_history), bands);
			return;
		}
		cmd.check(grb_taa_resolve(&image, &depth, &image_mv, prev ? &prev_img : nullptr, reproj.data(), q, &oc, &oh, GrbRows{ 0, 0 },
		                          cmd.get_stream_handle()),
		          "grb_taa_resolve");
	});
}
} // namespace Granite
