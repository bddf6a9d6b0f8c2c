// nccl_collectives.hpp -- RenderGraphCollectives over NCCL (NVLink 5 / NVSwitch), one rank per
// process/GPU.  libnccl is resolved at run time (dlopen of libnccl.so.2 -- the copy PyTorch
// already loaded when the host process is a torchrun rank), so the host library itself has no
// link-time NCCL dependency.  The unique id is created on rank 0 and distributed by the caller
// (bench.py / tests use torch.distributed for that plumbing).
#pragma once

#include <string>
#include <vector>

#include "render_graph.hpp"

namespace Granite
{
constexpr unsigned NcclUniqueIdBytes = 128;

class NcclCollectives : public RenderGraphCollectives
{
public:
	NcclCollectives() = default;
	~NcclCollectives() override;
	static bool get_unique_id(unsigned char out[NcclUniqueIdBytes], std::string &error);
	bool init(const unsigned char id[NcclUniqueIdBytes], unsigned rank, unsigned world_size, std::string &error);
	unsigned get_rank() const override { return rank; }
	unsigned get_world_size() const override { return world; }
	bool all_gather_rows(Vulkan::CommandBuffer &cmd, Vulkan::ImageView &image, const std::vector<GrbRows> &rows) override;
	bool all_reduce_sum(Vulkan::CommandBuffer &cmd, float *data, size_t count) override;
	// Peer-memory exchange: two image slots + a flag array per rank, cudaIpc-mapped into every
	// other rank (handles are exchanged with one ncclAllGather).  GRB_SHARD_EXCHANGE=nccl disables it.
	bool peer_exchange_begin_frame(size_t image_bytes, PeerSlot &slot) override;
	// The TAA history channel: a second set of the same buffers.
	bool taa_history_begin_frame(size_t image_bytes, PeerSlot &slot, void *&previous) override;
	// The SMAA edge channel: a third set.
	bool smaa_edges_begin_frame(size_t image_bytes, PeerSlot &slot) override;

private:
	bool collective_failed(const char *what);
	void *comm = nullptr;
	unsigned rank = 0, world = 1;

	struct PeerState
	{
		bool tried = false, ok = false;
		size_t image_bytes = 0;
		void *local_images[2] = {};
		uint32_t *local_flags = nullptr; // [world] flags followed by the scratch counter
		void *images[2][8] = {};
		uint32_t *flags[8] = {};
		std::vector<void *> opened;
		uint32_t epoch = 0;
		unsigned frames = 0; // frames begun since the buffers were (re-)created
	} peer, taa_history, smaa_edges;
	bool begin_frame(PeerState &peer, size_t image_bytes, PeerSlot &slot);
	bool setup_peer_exchange(PeerState &peer, size_t image_bytes);
	void release_peer_exchange(PeerState &peer);
};
} // namespace Granite
