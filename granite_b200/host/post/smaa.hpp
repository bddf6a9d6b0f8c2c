// smaa.hpp -- SMAA pass builder, same entry point as renderer/post/smaa.hpp:33-41.
#pragma once

#include <cstdint>
#include <string>
#include <vector>

#include "../render_graph.hpp"
#include "temporal.hpp"

namespace Granite
{
enum class SMAAPreset
{
	Low,
	Medium,
	High,
	Ultra,
	Ultra_T2X
};

// Three passes on the post-graphics queue -- "smaa-edge" (R8G8_UNORM), "smaa-weights" (R8G8B8A8_UNORM), "smaa-blend" --
// reading `input` (the tonemapped image, viewed as UNORM) and writing `output` (renderer/post/smaa.cpp:32-209).
// Ultra_T2X (two jittered frames + "smaa-t2x-resolve") is not built: std::logic_error.  In row-sharded graphs each rank
// detects the edges of its band, the edge rows another rank's searches reach are exchanged (peer stores from the edge
// kernel, or NCCL broadcasts), and each rank computes the weights of ShardPlan::smaa_weights and blends its band.
void setup_smaa_postprocess(RenderGraph &graph, TemporalJitter &jitter, float scaling_factor, const std::string &input, const std::string &input_depth,
                            const std::string &output, SMAAPreset preset);

// The two lookup textures SMAA samples: the reference loads builtin://textures/smaa/{area,search}.gtx through its asset
// manager (smaa.cpp:137-142); here the application hands their texels over once per device.
// area: 160 x 560 R8G8_UNORM, search: 64 x 16 R8_UNORM, tightly packed rows.
bool set_smaa_lookup_textures(Vulkan::Device &device, const uint8_t *area_rg8, const uint8_t *search_r8);
bool get_smaa_lookup_textures(Vulkan::Device &device, GrbImage *area, GrbImage *search);
void release_smaa_lookup_textures(Vulkan::Device &device);

// Reader of Granite's memory-mapped texture container (vulkan/texture/memory_mapped_texture.cpp:29-46): a 64-byte
// header -- 16-byte magic "GRANITE TEXFMT1", VkImageType, VkFormat, width, height, depth, layers, levels, flags, 64-bit
// payload size, 64 reserved bits -- followed by the texels of level 0 (only single-level 2-D images are accepted).
struct GtxImage
{
	VkFormat format = VK_FORMAT_UNDEFINED;
	unsigned width = 0, height = 0;
	std::vector<uint8_t> texels;
};
bool parse_gtx(const uint8_t *bytes, size_t size, GtxImage &out, std::string &error);
bool load_gtx(const std::string &path, GtxImage &out, std::string &error);
// Both lookup textures from a directory holding area.gtx and search.gtx (the reference's assets/textures/smaa).
bool load_smaa_lookup_textures(Vulkan::Device &device, const std::string &directory, std::string &error);
} // namespace Granite
