#include "nccl_collectives.hpp"

#include <cuda_runtime.h>
#include <dlfcn.h>

#include <cstdlib>

#include <cstring>
#include <mutex>

namespace Granite
{
namespace
{
// Minimal NCCL ABI (stable across 2.x): opaque comm, 128-byte unique id, enums as ints.
struct NcclUniqueId
{
	char internal[NcclUniqueIdBytes];
};
using ncclComm_t = void *;
constexpr int ncclSuccess = 0;
constexpr int ncclInt8 = 0;   // ncclChar
constexpr int ncclFloat32 = 7; // ncclFloat
constexpr int ncclSum = 0;

struct NcclApi
{
	void *handle = nullptr;
	int (*GetUniqueId)(NcclUniqueId *) = nullptr;
	int (*CommInitRank)(ncclComm_t *, int, NcclUniqueId, int) = nullptr;
	int (*CommDestroy)(ncclComm_t) = nullptr;
	int (*CommAbort)(ncclComm_t) = nullptr; // optional
	int (*AllReduce)(const void *, void *, size_t, int, int, ncclComm_t, void *) = nullptr;
	int (*Broadcast)(const void *, void *, size_t, int, int, ncclComm_t, void *) = nullptr;
	int (*AllGather)(const void *, void *, size_t, int, ncclComm_t, void *) = nullptr;
	int (*GroupStart)() = nullptr;
	int (*GroupEnd)() = nullptr;
	const char *(*GetErrorString)(int) = nullptr;
	std::string error;
};

NcclApi &api()
{
	static NcclApi a;
	static std::once_flag once;
	std::call_once(once, [] {
		const char *names[] = { "libnccl.so.2", "libnccl.so" };
		for (auto *n : names)
		{
			a.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
			if (a.handle)
				break;
		}
		if (!a.handle)
		{
			a.error = "libnccl.so.2 not found (import torch first, or add NCCL to LD_LIBRARY_PATH)";
			return;
		}
#define GRB_SYM(field, name)                                              \
	a.field = reinterpret_cast<decltype(a.field)>(dlsym(a.handle, name)); \
	if (!a.field)                                                         \
		a.error = std::string("missing NCCL symbol ") + name;
		GRB_SYM(GetUniqueId, "ncclGetUniqueId")
		GRB_SYM(CommInitRank, "ncclCommInitRank")
		GRB_SYM(CommDestroy, "ncclCommDestroy")
		GRB_SYM(AllReduce, "ncclAllReduce")
		GRB_SYM(Broadcast, "ncclBroadcast")
		GRB_SYM(AllGather, "ncclAllGather")
		GRB_SYM(GroupStart, "ncclGroupStart")
		GRB_SYM(GroupEnd, "ncclGroupEnd")
		GRB_SYM(GetErrorString, "ncclGetErrorString")
#undef GRB_SYM
		a.CommAbort = reinterpret_cast<decltype(a.CommAbort)>(dlsym(a.handle, "ncclCommAbort"));
	});
	return a;
}

bool nccl_ok(int rc, const char *what)
{
	if (rc == ncclSuccess)
		return true;
	Vulkan::log_error("%s: %s\n", what, api().GetErrorString ? api().GetErrorString(rc) : "NCCL error");
	return false;
}
} // namespace

NcclCollectives::~NcclCollectives()
{
	release_peer_exchange(peer);
	release_peer_exchange(taa_history);
	release_peer_exchange(smaa_edges);
	if (comm && api().CommDestroy)
		api().CommDestroy(comm);
}

// A collective that failed leaves the communicator in an undefined state and its peers possibly blocked inside
// the same collective: abort it (ncclCommAbort frees the resources without waiting for outstanding operations) so
// that every later call on this rank fails fast -- the sharded passes then report errors frame by frame, the
// reference's LOGE-and-continue convention -- instead of queueing more work behind a dead collective.
bool NcclCollectives::collective_failed(const char *what)
{
	Vulkan::log_error("%s failed: aborting the communicator of rank %u; row-sharded passes will report errors from here on.\n", what, rank);
	if (comm)
	{
		if (api().CommAbort)
			api().CommAbort(comm);
		comm = nullptr;
	}
	return false;
}

bool NcclCollectives::get_unique_id(unsigned char out[NcclUniqueIdBytes], std::string &error)
{
	auto &a = api();
	if (!a.error.empty())
	{
		error = a.error;
		return false;
	}
	NcclUniqueId id;
	if (a.GetUniqueId(&id) != ncclSuccess)
	{
		error = "ncclGetUniqueId failed";
		return false;
	}
	std::memcpy(out, id.internal, NcclUniqueIdBytes);
	return true;
}

bool NcclCollectives::init(const unsigned char id_bytes[NcclUniqueIdBytes], unsigned rank_, unsigned world_size, std::string &error)
{
	auto &a = api();
	if (!a.error.empty())
	{
		error = a.error;
		return false;
	}
	NcclUniqueId id;
	std::memcpy(id.internal, id_bytes, NcclUniqueIdBytes);
	int rc = a.CommInitRank(&comm, (int)world_size, id, (int)rank_);
	if (rc != ncclSuccess)
	{
		error = std::string("ncclCommInitRank: ") + a.GetErrorString(rc);
		comm = nullptr;
		return false;
	}
	rank = rank_;
	world = world_size;
	return true;
}

bool NcclCollectives::all_gather_rows(Vulkan::CommandBuffer &cmd, Vulkan::ImageView &image, const std::vector<GrbRows> &rows)
{
	if (!comm || rows.size() != world)
		return false;
	// Bands differ in height, so this is a grouped set of broadcasts (one root per band), which
	// NCCL fuses into a single launch over NVLink.
	auto &a = api();
	auto *base = static_cast<unsigned char *>(image.get_image().get_device_pointer());
	const size_t pitch = image.get_image().get_row_pitch();
	bool ok = nccl_ok(a.GroupStart(), "ncclGroupStart");
	for (unsigned r = 0; r < world && ok; r++)
	{
		size_t bytes = (size_t)(rows[r].y1 - rows[r].y0) * pitch;
		void *p = base + (size_t)rows[r].y0 * pitch;
		ok = nccl_ok(a.Broadcast(p, p, bytes, ncclInt8, (int)r, comm, cmd.get_stream_handle()), "ncclBroadcast");
	}
	ok = nccl_ok(a.GroupEnd(), "ncclGroupEnd") && ok;
	return ok ? true : collective_failed("all_gather_rows");
}

bool NcclCollectives::all_reduce_sum(Vulkan::CommandBuffer &cmd, float *data, size_t count)
{
	if (!comm)
		return false;
	if (nccl_ok(api().AllReduce(data, data, count, ncclFloat32, ncclSum, comm, cmd.get_stream_handle()), "ncclAllReduce"))
		return true;
	return collective_failed("all_reduce_sum");
}

// ----------------------------------------------------------------------------- peer exchange
void NcclCollectives::release_peer_exchange(PeerState &peer)
{
	for (void *p : peer.opened)
		cudaIpcCloseMemHandle(p);
	peer.opened.clear();
	for (auto &img : peer.local_images)
	{
		if (img)
			cudaFree(img);
		img = nullptr;
	}
	if (peer.local_flags)
		cudaFree(peer.local_flags);
	peer.local_flags = nullptr;
	peer.ok = false;
}

bool NcclCollectives::setup_peer_exchange(PeerState &peer, size_t image_bytes)
{
	// Collective: every rank calls this with the same size at the same point of its first sharded frame.
	struct Handles
	{
		cudaIpcMemHandle_t image[2];
		cudaIpcMemHandle_t flags;
		int ok;
	};
	auto &a = api();
	Handles mine = {};
	mine.ok = 1;
	const char *mode = std::getenv("GRB_SHARD_EXCHANGE");
	if (!comm || world > 8 || (mode && std::string(mode) == "nccl"))
		mine.ok = 0;
	if (mine.ok)
	{
		for (auto &img : peer.local_images)
			mine.ok = mine.ok && cudaMalloc(&img, image_bytes) == cudaSuccess && cudaMemset(img, 0, image_bytes) == cudaSuccess;
		void *f = nullptr;
		mine.ok = mine.ok && cudaMalloc(&f, sizeof(uint32_t) * 16) == cudaSuccess && cudaMemset(f, 0, sizeof(uint32_t) * 16) == cudaSuccess;
		peer.local_flags = static_cast<uint32_t *>(f);
		for (int k = 0; k < 2 && mine.ok; k++)
			mine.ok = cudaIpcGetMemHandle(&mine.image[k], peer.local_images[k]) == cudaSuccess;
		mine.ok = mine.ok && cudaIpcGetMemHandle(&mine.flags, peer.local_flags) == cudaSuccess;
		if (!mine.ok)
			cudaGetLastError();
	}

	// exchange the handles (and whether every rank could create them) through the communicator
	Handles *dev = nullptr;
	std::vector<Handles> all(world);
	bool ok = cudaMalloc(&dev, sizeof(Handles) * (world + 1)) == cudaSuccess;
	cudaStream_t s = nullptr;
	ok = ok && cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) == cudaSuccess;
	ok = ok && cudaMemcpyAsync(dev + world, &mine, sizeof(Handles), cudaMemcpyHostToDevice, s) == cudaSuccess;
	ok = ok && nccl_ok(a.AllGather(dev + world, dev, sizeof(Handles), ncclInt8, comm, s), "ncclAllGather(ipc handles)");
	ok = ok && cudaMemcpyAsync(all.data(), dev, sizeof(Handles) * world, cudaMemcpyDeviceToHost, s) == cudaSuccess;
	ok = ok && cudaStreamSynchronize(s) == cudaSuccess;
	if (s)
		cudaStreamDestroy(s);
	if (dev)
		cudaFree(dev);
	for (unsigned r = 0; r < world && ok; r++)
		ok = all[r].ok != 0;
	for (unsigned r = 0; r < world && ok; r++)
	{
		if (r == rank)
		{
			peer.images[0][r] = peer.local_images[0];
			peer.images[1][r] = peer.local_images[1];
			peer.flags[r] = peer.local_flags;
			continue;
		}
		void *p[3] = {};
		ok = cudaIpcOpenMemHandle(&p[0], all[r].image[0], cudaIpcMemLazyEnablePeerAccess) == cudaSuccess &&
		     cudaIpcOpenMemHandle(&p[1], all[r].image[1], cudaIpcMemLazyEnablePeerAccess) == cudaSuccess &&
		     cudaIpcOpenMemHandle(&p[2], all[r].flags, cudaIpcMemLazyEnablePeerAccess) == cudaSuccess;
		for (void *q : p)
			if (q)
				peer.opened.push_back(q);
		peer.images[0][r] = p[0];
		peer.images[1][r] = p[1];
		peer.flags[r] = static_cast<uint32_t *>(p[2]);
	}
	if (!ok)
	{
		cudaGetLastError();
		if (!(mode && std::string(mode) == "nccl"))
			Vulkan::log_info("peer-memory exchange unavailable on rank %u (no IPC / peer access); using NCCL broadcasts.\n", rank);
		release_peer_exchange(peer);
		return false;
	}
	peer.image_bytes = image_bytes;
	peer.frames = 0;
	return true;
}

bool NcclCollectives::begin_frame(PeerState &peer, size_t image_bytes, PeerSlot &slot)
{
	if (!peer.tried || (peer.ok && peer.image_bytes != image_bytes))
	{
		// (a re-bake at another size re-creates the buffers; all ranks re-bake together)
		if (peer.tried)
			release_peer_exchange(peer);
		peer.tried = true;
		peer.ok = setup_peer_exchange(peer, image_bytes);
	}
	if (!peer.ok)
		return false;
	peer.frames++;
	peer.epoch++;
	const unsigned k = peer.epoch & 1u;
	slot.count = world;
	slot.epoch = peer.epoch;
	slot.counter = peer.local_flags + 8;
	for (unsigned r = 0; r < world; r++)
	{
		slot.images[r] = peer.images[k][r];
		slot.flags[r] = peer.flags[r];
	}
	return true;
}

bool NcclCollectives::peer_exchange_begin_frame(size_t image_bytes, PeerSlot &slot)
{
	return begin_frame(peer, image_bytes, slot);
}

bool NcclCollectives::taa_history_begin_frame(size_t image_bytes, PeerSlot &slot, void *&previous)
{
	previous = nullptr;
	if (!begin_frame(taa_history, image_bytes, slot))
		return false;
	if (taa_history.frames > 1)
		previous = taa_history.local_images[(taa_history.epoch - 1) & 1u];
	return true;
}

bool NcclCollectives::smaa_edges_begin_frame(size_t image_bytes, PeerSlot &slot)
{
	return begin_frame(smaa_edges, image_bytes, slot);
}
} // namespace Granite
