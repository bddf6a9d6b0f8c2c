// render_graph.hpp -- Granite's RenderGraph declaration / callback surface
// (renderer/render_graph.hpp:48-73, 154-186, 488-516, 685-716, 793-866) over a CUDA executor.
//
// What is kept: the names, signatures and semantics a pass builder sees -- add_pass (idempotent
// by name), the resource declarators, AttachmentInfo/BufferInfo/SizeClass, set_build_render_pass,
// RenderPassInterface with its virtuals, bake(), setup_attachments(), enqueue_render_passes(),
// get_physical_{texture,buffer,history_texture}_resource, persistent-buffer consume/install,
// history images that swap every frame and are null on the first one, std::logic_error on
// graph misuse.
//
// What is new: everything below that surface.  There are no barriers, layouts, queues or
// semaphores to plan -- a baked graph is a topologically ordered list of passes recorded on one
// CUDA stream per device (stream order IS the dependency), physical images are plain device
// allocations (no aliasing: 180 GB of HBM3e makes the reference's transient aliasing pointless),
// and per-pass GPU timestamps are CUDA events.
#pragma once

#include <array>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "cuda_backend.hpp"
#include "shard_plan.hpp"

namespace Granite
{
class RenderGraph;
class RenderPass;

// Stand-in for threading/task_composer.hpp: callbacks that receive it run inline on the
// recording thread.
class TaskComposer
{
};

// Exchange steps of a row-sharded frame.  The reference has no counterpart (single GPU); the
// implementation shipped with the host library runs them with NCCL on the graph's stream.
class RenderGraphCollectives
{
public:
	virtual ~RenderGraphCollectives() = default;
	virtual unsigned get_rank() const = 0;
	virtual unsigned get_world_size() const = 0;
	// Every rank contributes rows [rows[r].y0, rows[r].y1) of an image all ranks hold at full size.
	virtual bool all_gather_rows(Vulkan::CommandBuffer &cmd, Vulkan::ImageView &image, const std::vector<GrbRows> &rows) = 0;
	virtual bool all_reduce_sum(Vulkan::CommandBuffer &cmd, float *data, size_t count) = 0;

	// Peer-memory exchange: a double-buffered image every rank holds in full, of which each rank
	// PRODUCES some rows per frame by storing them into all ranks' copies from its own kernel
	// (NVLink / NVSwitch peer stores) and then raising a per-rank flag.  begin_frame() returns
	// this frame's slot: the copy's address on every rank as seen from this device, every rank's
	// flag array, and the epoch to publish / wait for.  false = not available (single process
	// without peer access, IPC refused...): callers then use all_gather_rows().
	struct PeerSlot
	{
		void *images[8] = {};     // [rank] base address of this frame's slot on that rank
		uint32_t *flags[8] = {};  // [rank] that rank's flag array (one uint32 per producing rank)
		uint32_t *counter = nullptr; // local scratch for the producing kernel
		uint32_t epoch = 0;
		unsigned count = 0;
	};
	virtual bool peer_exchange_begin_frame(size_t image_bytes, PeerSlot &slot)
	{
		(void)image_bytes;
		(void)slot;
		return false;
	}
	// The same kind of exchange for the TAA history, as a channel of its own (its own double-buffered image, flag
	// arrays and scratch counter: the resolve runs on another stream than the bloom exchange).  Besides this frame's
	// slot it returns `previous`, this rank's copy of the previous frame's slot: the full history the resolve reads
	// (nullptr on the channel's first frame).  false = not available: callers then use all_gather_rows().
	virtual bool taa_history_begin_frame(size_t image_bytes, PeerSlot &slot, void *&previous)
	{
		(void)image_bytes;
		(void)slot;
		previous = nullptr;
		return false;
	}
	// A third channel of the same kind for the SMAA edges: each rank stores the edge rows of its band that another
	// rank's weights pass reads into that rank's slot (slot.images[get_rank()] is this rank's own copy, which its
	// weights pass reads).  false = not available: callers then use all_gather_rows().
	virtual bool smaa_edges_begin_frame(size_t image_bytes, PeerSlot &slot)
	{
		(void)image_bytes;
		(void)slot;
		return false;
	}
};

class RenderPassInterface
{
public:
	virtual ~RenderPassInterface() = default;
	// This information must remain fixed.
	virtual bool render_pass_is_conditional() const { return false; }
	virtual bool render_pass_is_separate_layered() const { return false; }
	// Can change per frame.
	virtual bool need_render_pass() const { return true; }
	virtual bool get_clear_depth_stencil(VkClearDepthStencilValue *value) const;
	virtual bool get_clear_color(unsigned attachment, VkClearColorValue *value) const;
	// Called once before bake().
	virtual void setup_dependencies(RenderPass &self, RenderGraph &graph);
	// Called once after bake().
	virtual void setup(Vulkan::Device &device);
	// Called every frame, before build_render_pass.
	virtual void enqueue_prepare_render_pass(RenderGraph &graph, TaskComposer &composer);
	virtual void build_render_pass(Vulkan::CommandBuffer &cmd);
	virtual void build_render_pass_separate_layer(Vulkan::CommandBuffer &cmd, unsigned layer);
};
using RenderPassInterfaceHandle = std::shared_ptr<RenderPassInterface>;

enum SizeClass
{
	Absolute,
	SwapchainRelative,
	InputRelative
};

enum RenderGraphQueueFlagBits
{
	RENDER_GRAPH_QUEUE_GRAPHICS_BIT = 1 << 0,
	RENDER_GRAPH_QUEUE_COMPUTE_BIT = 1 << 1,
	RENDER_GRAPH_QUEUE_ASYNC_COMPUTE_BIT = 1 << 2,
	// A second asynchronous queue for the post chain, so the (HBM-bound) post passes of frame N
	// run beside the (ALU-bound) lighting of frame N+1.
	RENDER_GRAPH_QUEUE_ASYNC_GRAPHICS_BIT = 1 << 3,
	// Not in the reference: a third asynchronous queue, so that the bloom pyramid of frame N (whose tail
	// runs beside the lighting of frame N+1) does not hold back the tonemap of frame N-1 or vice versa.
	RENDER_GRAPH_QUEUE_ASYNC_POST_COMPUTE_BIT = 1 << 4
};
using RenderGraphQueueFlags = uint32_t;

// A resource managed OUTSIDE the graph (the reference's clustered shadow atlas, its scene transform buffer:
// render_graph.hpp:76-126), which passes of the graph read.  The reference hands Vulkan semaphores back and forth;
// here they are CUDA events: the owner records one behind its writes (release_internal), consumer passes declared
// with RenderPass::add_external_lock(name, ...) make their stream wait for it and hand back the event recorded
// behind their own work, and the owner's next acquire_internal waits for those before it writes again.
class RenderPassExternalLockInterface
{
public:
	virtual ~RenderPassExternalLockInterface() = default;
	virtual const char *get_ident() const { return "external-lock"; }

	// consumer side (called by the graph while it records a pass)
	Vulkan::Event external_acquire_event();
	void external_release_event(Vulkan::Event event);
	// External accesses are read-only; the reference records which queues touch the resource, the stream order
	// plus the two calls above make that unnecessary here.  Kept so that builder code compiles unchanged.
	void mark_access_in_queue(RenderGraphQueueFlagBits, VkPipelineStageFlags2, VkAccessFlags2) { foreign_access = true; }
	bool has_foreign_access() const { return foreign_access; }

protected:
	// owner side (the derived class calls these around its own work on `stream`)
	void acquire_internal(Vulkan::Device &device, Vulkan::Stream stream);
	void release_internal(Vulkan::Device &device, Vulkan::Stream stream);

private:
	std::mutex lock;
	Vulkan::Event produced = nullptr;            // recorded by release_internal
	std::vector<Vulkan::Event> consumed;         // handed back by consumer passes since the last acquire_internal
	bool foreign_access = false;
};


enum AttachmentInfoFlagBits
{
	ATTACHMENT_INFO_PERSISTENT_BIT = 1 << 0,
	ATTACHMENT_INFO_UNORM_SRGB_ALIAS_BIT = 1 << 1,
	ATTACHMENT_INFO_SUPPORTS_PREROTATE_BIT = 1 << 2,
	ATTACHMENT_INFO_MIPGEN_BIT = 1 << 3,
	// Two physical images used on alternate frames: removes the write-after-read dependency
	// between frame N's consumers and frame N+1's producer when they run on different streams.
	ATTACHMENT_INFO_PINGPONG_BIT = 1 << 8
};
using AttachmentInfoFlags = uint32_t;

struct AttachmentInfo
{
	SizeClass size_class = SizeClass::SwapchainRelative;
	float size_x = 1.0f;
	float size_y = 1.0f;
	float size_z = 0.0f;
	VkFormat format = VK_FORMAT_UNDEFINED;
	std::string size_relative_name;
	unsigned samples = 1;
	unsigned levels = 1;
	unsigned layers = 1;
	VkImageUsageFlags aux_usage = 0;
	AttachmentInfoFlags flags = ATTACHMENT_INFO_PERSISTENT_BIT;
};

struct BufferInfo
{
	VkDeviceSize size = 0;
	VkBufferUsageFlags usage = 0;
	AttachmentInfoFlags flags = ATTACHMENT_INFO_PERSISTENT_BIT;
	bool operator==(const BufferInfo &other) const { return size == other.size && usage == other.usage && flags == other.flags; }
	bool operator!=(const BufferInfo &other) const { return !(*this == other); }
};

struct ResourceDimensions
{
	VkFormat format = VK_FORMAT_UNDEFINED;
	BufferInfo buffer_info;
	unsigned width = 0;
	unsigned height = 0;
	unsigned depth = 1;
	unsigned layers = 1;
	unsigned levels = 1;
	unsigned samples = 1;
	AttachmentInfoFlags flags = ATTACHMENT_INFO_PERSISTENT_BIT;
	RenderGraphQueueFlags queues = 0;
	std::string name;
};

class RenderResource
{
public:
	enum class Type
	{
		Buffer,
		Texture
	};
	enum { Unused = ~0u };

	RenderResource(Type type_, unsigned index_) : resource_type(type_), index(index_) {}
	virtual ~RenderResource() = default;
	Type get_type() const { return resource_type; }
	void written_in_pass(unsigned pass) { written_in_passes.insert(pass); }
	void read_in_pass(unsigned pass) { read_in_passes.insert(pass); }
	const std::unordered_set<unsigned> &get_read_passes() const { return read_in_passes; }
	const std::unordered_set<unsigned> &get_write_passes() const { return written_in_passes; }
	unsigned get_index() const { return index; }
	void set_physical_index(unsigned index_) { physical_index = index_; }
	unsigned get_physical_index() const { return physical_index; }
	void set_name(const std::string &name_) { name = name_; }
	const std::string &get_name() const { return name; }

private:
	Type resource_type;
	unsigned index;
	unsigned physical_index = Unused;
	std::unordered_set<unsigned> written_in_passes;
	std::unordered_set<unsigned> read_in_passes;
	std::string name;
};

class RenderBufferResource : public RenderResource
{
public:
	explicit RenderBufferResource(unsigned index_) : RenderResource(RenderResource::Type::Buffer, index_) {}
	void set_buffer_info(const BufferInfo &info_) { info = info_; }
	const BufferInfo &get_buffer_info() const { return info; }
	// a proxy has no memory (size 0): it exists for the ordering its writer / readers imply
	void set_proxy(bool enable) { proxy = enable; }
	bool is_proxy() const { return proxy; }

private:
	BufferInfo info;
	bool proxy = false;
};

class RenderTextureResource : public RenderResource
{
public:
	explicit RenderTextureResource(unsigned index_) : RenderResource(RenderResource::Type::Texture, index_) {}
	void set_attachment_info(const AttachmentInfo &info_) { info = info_; }
	const AttachmentInfo &get_attachment_info() const { return info; }
	AttachmentInfo &get_attachment_info() { return info; }

private:
	AttachmentInfo info;
};

class RenderPass
{
public:
	RenderPass(RenderGraph &graph_, unsigned index_, RenderGraphQueueFlagBits queue_) : graph(graph_), index(index_), queue(queue_) {}

	RenderGraphQueueFlagBits get_queue() const { return queue; }
	RenderGraph &get_graph() { return graph; }
	unsigned get_index() const { return index; }

	RenderTextureResource &set_depth_stencil_input(const std::string &name);
	RenderTextureResource &set_depth_stencil_output(const std::string &name, const AttachmentInfo &info);
	RenderTextureResource &add_color_output(const std::string &name, const AttachmentInfo &info, const std::string &input = "");
	RenderTextureResource &add_attachment_input(const std::string &name);
	RenderTextureResource &add_history_input(const std::string &name);
	RenderTextureResource &add_texture_input(const std::string &name, VkPipelineStageFlags2 stages = 0);
	RenderBufferResource &add_uniform_input(const std::string &name, VkPipelineStageFlags2 stages = 0);
	RenderBufferResource &add_storage_read_only_input(const std::string &name, VkPipelineStageFlags2 stages = 0);
	RenderBufferResource &add_storage_output(const std::string &name, const BufferInfo &info, const std::string &input = "");
	RenderBufferResource &add_transfer_output(const std::string &name, const BufferInfo &info);
	RenderTextureResource &add_storage_texture_output(const std::string &name, const AttachmentInfo &info, const std::string &input = "");
	void add_fake_resource_write_alias(const std::string &from, const std::string &to);
	// Buffers a raster pass reads through fixed-function stages (render_graph.hpp:509-511): plain read dependencies here.
	RenderBufferResource &add_vertex_buffer_input(const std::string &name) { return add_uniform_input(name); }
	RenderBufferResource &add_index_buffer_input(const std::string &name) { return add_uniform_input(name); }
	RenderBufferResource &add_indirect_buffer_input(const std::string &name) { return add_uniform_input(name); }
	// Proxy resources (render_graph.hpp:513-514, render_graph.cpp:305-343): no memory, only ordering -- the writer of
	// a proxy runs before its readers, across streams too.
	void add_proxy_output(const std::string &name, VkPipelineStageFlags2 stages, VkAccessFlags2 access, const std::string &input = "");
	void add_proxy_input(const std::string &name, VkPipelineStageFlags2 stages, VkAccessFlags2 access);
	// render_graph.cpp:390-411: no-op unless RenderGraph::add_external_lock_interface registered `name`.
	void add_external_lock(const std::string &name, VkPipelineStageFlags2 stages, VkAccessFlags2 access);
	struct AccessedExternalLockInterface
	{
		RenderPassExternalLockInterface *iface;
		VkPipelineStageFlags2 stages;
	};
	const std::vector<AccessedExternalLockInterface> &get_lock_interfaces() const { return lock_interfaces; }

	const std::vector<RenderTextureResource *> &get_color_outputs() const { return color_outputs; }
	const std::vector<RenderTextureResource *> &get_color_inputs() const { return color_inputs; }
	const std::vector<RenderTextureResource *> &get_storage_texture_outputs() const { return storage_texture_outputs; }
	const std::vector<RenderTextureResource *> &get_attachment_inputs() const { return attachments_inputs; }
	const std::vector<RenderTextureResource *> &get_history_inputs() const { return history_inputs; }
	// Not in the reference: this pass starts only after the latest RenderGraph::signal_mark(name) (any frame).
	void add_wait_mark(const std::string &name) { wait_marks.push_back(name); }
	const std::vector<std::string> &get_wait_marks() const { return wait_marks; }
	const std::vector<RenderTextureResource *> &get_texture_inputs() const { return texture_inputs; }
	const std::vector<RenderBufferResource *> &get_storage_outputs() const { return storage_outputs; }
	const std::vector<RenderBufferResource *> &get_transfer_outputs() const { return transfer_outputs; }
	const std::vector<RenderBufferResource *> &get_buffer_inputs() const { return buffer_inputs; }
	RenderTextureResource *get_depth_stencil_input() const { return depth_stencil_input; }
	RenderTextureResource *get_depth_stencil_output() const { return depth_stencil_output; }

	bool need_render_pass() const { return render_pass_handle ? render_pass_handle->need_render_pass() : true; }
	bool get_clear_color(unsigned attachment, VkClearColorValue *value = nullptr) const;
	bool get_clear_depth_stencil(VkClearDepthStencilValue *value = nullptr) const;

	void prepare_render_pass(TaskComposer &composer)
	{
		if (render_pass_handle)
			render_pass_handle->enqueue_prepare_render_pass(graph, composer);
	}

	void setup(Vulkan::Device &device)
	{
		if (render_pass_handle)
			render_pass_handle->setup(device);
	}

	void setup_dependencies()
	{
		if (render_pass_handle)
			render_pass_handle->setup_dependencies(*this, graph);
	}

	// Dispatch rule of renderer/render_graph.hpp:685-696.
	void build_render_pass(Vulkan::CommandBuffer &cmd, unsigned layer)
	{
		if (render_pass_handle)
		{
			if (render_pass_handle->render_pass_is_separate_layered())
				render_pass_handle->build_render_pass_separate_layer(cmd, layer);
			else
				render_pass_handle->build_render_pass(cmd);
		}
		else if (build_render_pass_cb)
			build_render_pass_cb(cmd);
	}

	void set_render_pass_interface(RenderPassInterfaceHandle handle) { render_pass_handle = std::move(handle); }
	void set_build_render_pass(std::function<void(Vulkan::CommandBuffer &)> func) { build_render_pass_cb = std::move(func); }
	void set_get_clear_depth_stencil(std::function<bool(VkClearDepthStencilValue *)> func) { get_clear_depth_stencil_cb = std::move(func); }
	void set_get_clear_color(std::function<bool(unsigned, VkClearColorValue *)> func) { get_clear_color_cb = std::move(func); }
	void set_name(const std::string &name) { pass_name = name; }
	const std::string &get_name() const { return pass_name; }

	// dependency bookkeeping used by bake()
	const std::vector<RenderResource *> &get_all_reads() const { return reads; }
	const std::vector<RenderResource *> &get_all_writes() const { return writes; }
	const std::vector<std::pair<RenderResource *, RenderResource *>> &get_write_aliases() const { return rmw_aliases; }

private:
	RenderGraph &graph;
	unsigned index;
	RenderGraphQueueFlagBits queue;
	RenderPassInterfaceHandle render_pass_handle;
	std::vector<std::string> wait_marks;
	std::function<void(Vulkan::CommandBuffer &)> build_render_pass_cb;
	std::function<bool(VkClearDepthStencilValue *)> get_clear_depth_stencil_cb;
	std::function<bool(unsigned, VkClearColorValue *)> get_clear_color_cb;
	std::string pass_name;

	std::vector<RenderTextureResource *> color_outputs, color_inputs, storage_texture_outputs, attachments_inputs, history_inputs, texture_inputs;
	std::vector<RenderBufferResource *> storage_outputs, transfer_outputs, buffer_inputs;
	RenderTextureResource *depth_stencil_input = nullptr;
	RenderTextureResource *depth_stencil_output = nullptr;
	std::vector<RenderResource *> reads, writes;
	std::vector<std::pair<RenderResource *, RenderResource *>> rmw_aliases; // (output, input it modifies in place)
	std::vector<std::pair<RenderResource *, RenderResource *>> fake_aliases;
	std::vector<AccessedExternalLockInterface> lock_interfaces;
	friend class RenderGraph;
};

class RenderGraph
{
public:
	RenderGraph() = default;
	~RenderGraph() = default;
	RenderGraph(const RenderGraph &) = delete;
	void operator=(const RenderGraph &) = delete;

	void set_device(Vulkan::Device *device_) { device = device_; }
	Vulkan::Device &get_device();

	RenderPass &add_pass(const std::string &name, RenderGraphQueueFlagBits queue);
	RenderPass *find_pass(const std::string &name);
	void set_backbuffer_source(const std::string &name);
	void set_backbuffer_dimensions(const ResourceDimensions &dim) { swapchain_dimensions = dim; }
	const ResourceDimensions &get_backbuffer_dimensions() const { return swapchain_dimensions; }

	ResourceDimensions get_resource_dimensions(const RenderBufferResource &resource) const;
	ResourceDimensions get_resource_dimensions(const RenderTextureResource &resource) const;

	void enable_timestamps(bool enable) { timestamps = enable; }
	// Misconfiguration throws std::logic_error, as in the reference (render_graph.cpp:568-619, 3003).
	void bake();
	void reset();
	void log();
	// Allocates / reuses physical images and buffers, swaps history <-> current
	// (render_graph.cpp:2686-2765).  `swapchain` may be null: the backbuffer source is then a
	// graph-owned image of the backbuffer dimensions.
	void setup_attachments(Vulkan::Device &device, Vulkan::ImageView *swapchain);
	// Records every baked pass, in order, on the device's stream.
	void enqueue_render_passes(Vulkan::Device &device, TaskComposer &composer);

	RenderTextureResource &get_texture_resource(const std::string &name);
	RenderBufferResource &get_buffer_resource(const std::string &name);
	bool has_texture_resource(const std::string &name) const { return resource_to_index.count(name) != 0; }

	Vulkan::ImageView &get_physical_texture_resource(unsigned index);
	Vulkan::ImageView *get_physical_history_texture_resource(unsigned index);
	Vulkan::Buffer &get_physical_buffer_resource(unsigned index);
	Vulkan::ImageView &get_physical_texture_resource(const RenderTextureResource &resource) { return get_physical_texture_resource(resource.get_physical_index()); }
	Vulkan::ImageView *maybe_get_physical_texture_resource(RenderTextureResource *resource);
	Vulkan::ImageView *get_physical_history_texture_resource(const RenderTextureResource &resource) { return get_physical_history_texture_resource(resource.get_physical_index()); }
	Vulkan::Buffer &get_physical_buffer_resource(const RenderBufferResource &resource) { return get_physical_buffer_resource(resource.get_physical_index()); }
	Vulkan::Buffer *maybe_get_physical_buffer_resource(RenderBufferResource *resource);

	// For keeping feed-back resources alive during rebaking (scene_viewer_application.cpp:1169,1315).
	std::vector<Vulkan::BufferHandle> consume_physical_buffers() const;
	void install_physical_buffers(std::vector<Vulkan::BufferHandle> buffers);

	// Like the reference these default to the main queue ("Don't use async compute by default",
	// render_graph.hpp:889-893); set_async_post(true) moves the post chain to its own stream.
	static RenderGraphQueueFlagBits get_default_post_graphics_queue() { return async_post ? RENDER_GRAPH_QUEUE_ASYNC_GRAPHICS_BIT : RENDER_GRAPH_QUEUE_GRAPHICS_BIT; }
	static RenderGraphQueueFlagBits get_default_compute_queue() { return async_post ? RENDER_GRAPH_QUEUE_ASYNC_POST_COMPUTE_BIT : RENDER_GRAPH_QUEUE_COMPUTE_BIT; }
	static void set_async_post(bool enable) { async_post = enable; }
	// Stream index a queue flag records on: 0 main, 1 async compute, 2 async graphics (tonemap, AA), 3 async post compute (bloom).
	static unsigned queue_stream_index(RenderGraphQueueFlagBits queue)
	{
		return queue == RENDER_GRAPH_QUEUE_ASYNC_COMPUTE_BIT ? 1u :
		       (queue == RENDER_GRAPH_QUEUE_ASYNC_GRAPHICS_BIT ? 2u : (queue == RENDER_GRAPH_QUEUE_ASYNC_POST_COMPUTE_BIT ? 3u : 0u));
	}
	// Ordering marks between passes that share no resource: signal_mark records an event at the current point of the
	// pass being built (cmd's stream); wait_mark makes cmd's stream wait for the latest signal of that name (no-op
	// before the first signal).  Used to phase the frame: the next lighting pass starts after this frame's
	// full-machine bloom kernel, see host/post/hdr.cpp.
	// render_graph.hpp:790-791 / render_graph.cpp:3771-3783
	void add_external_lock_interface(const std::string &name, RenderPassExternalLockInterface *iface) { external_lock_interfaces[name] = iface; }
	RenderPassExternalLockInterface *find_external_lock_interface(const std::string &name) const
	{
		auto itr = external_lock_interfaces.find(name);
		return itr != external_lock_interfaces.end() ? itr->second : nullptr;
	}
	void signal_mark(const std::string &name, Vulkan::CommandBuffer &cmd);
	void wait_mark(const std::string &name, Vulkan::CommandBuffer &cmd);
	// Stream of the pass that writes `resource` (for host readbacks of a graph output).
	Vulkan::Stream get_writer_stream(const RenderResource &resource);

	// Execution order decided by bake(): names of the passes that will run.
	std::vector<std::string> get_baked_pass_names() const;
	// Row-sharded frames (multi-GPU, one graph per device/process): `bands[r]` = backbuffer rows
	// [y0, y1) owned by rank r; they must tile the frame.  Builders scale the local band per
	// resource with shard_rows_for(); an unsharded graph returns {0,0} (= all rows).
	// smaa_quality: SMAA (0..3) after the tonemap, -1 = none (ShardPlan::smaa_weights / smaa_edges).
	void set_row_shards(const std::vector<GrbRows> &bands, unsigned rank, RenderGraphCollectives *collectives, bool fxaa_downstream = false,
	                    bool taa_upstream = false, int smaa_quality = -1);
	// Rows of every stage for `rank` (this rank by default); whole images when unsharded.
	ShardPlan get_shard_plan() const { return get_shard_plan(shard_rank); }
	ShardPlan get_shard_plan(unsigned rank) const
	{
		return compute_shard_plan(swapchain_dimensions.width, swapchain_dimensions.height, shard_bands, rank, shard_fxaa, shard_taa, shard_smaa);
	}
	GrbRows shard_rows_for(unsigned resource_height, unsigned halo_rows = 0) const;
	GrbRows shard_rows_for_rank(unsigned rank, unsigned resource_height, unsigned halo_rows = 0) const;
	bool is_sharded() const { return !shard_bands.empty(); }
	unsigned get_shard_rank() const { return shard_rank; }
	unsigned get_shard_count() const { return (unsigned)shard_bands.size(); }
	RenderGraphCollectives *get_collectives() const { return collectives; }

private:
	Vulkan::Device *device = nullptr;
	std::vector<std::unique_ptr<RenderPass>> passes;
	std::vector<std::unique_ptr<RenderResource>> resources;
	std::unordered_map<std::string, unsigned> pass_to_index;
	std::unordered_map<std::string, unsigned> resource_to_index;
	std::string backbuffer_source;
	ResourceDimensions swapchain_dimensions;
	bool timestamps = false;

	std::vector<unsigned> pass_stack; // baked order
	std::vector<ResourceDimensions> physical_dimensions;
	std::vector<bool> physical_has_history;
	std::vector<std::unique_ptr<Vulkan::ImageView>> physical_attachments;
	std::vector<std::unique_ptr<Vulkan::ImageView>> physical_history_attachments; // previous frame (may be null)
	std::vector<std::unique_ptr<Vulkan::ImageView>> physical_history_spare;       // image to become "current" next frame
	std::vector<Vulkan::BufferHandle> physical_buffers;
	unsigned backbuffer_physical = RenderResource::Unused;
	bool baked = false;
	// cross-stream ordering per physical resource: the last writer, and the last access (read or
	// write) recorded on each of the three queue streams.  A reader waits for the writer; a writer
	// waits for the last access on every other stream (RAW, WAW and WAR, also when two passes on
	// different streams read the resource before the next write).
	struct LastAccess
	{
		Vulkan::Event write_event = nullptr;
		Vulkan::Stream write_stream = nullptr;
		Vulkan::Event stream_event[4] = { nullptr, nullptr, nullptr, nullptr };
		Vulkan::Stream stream_of[4] = { nullptr, nullptr, nullptr, nullptr };
	};
	std::unordered_map<const void *, LastAccess> last_access; // keyed by the physical image / buffer
	struct Mark
	{
		std::array<Vulkan::Event, 4> events = { nullptr, nullptr, nullptr, nullptr };
		unsigned next = 0;
		Vulkan::Event latest = nullptr;
		Vulkan::Stream stream = nullptr;
	};
	std::unordered_map<std::string, Mark> marks;
	std::unordered_map<std::string, RenderPassExternalLockInterface *> external_lock_interfaces;
	// one "pass done" event per pass per frame slot: a later frame re-recording the same event
	// would turn "wait for frame N-2's reader" into "wait for frame N's", serialising the streams
	enum { EventRing = 4 };
	std::vector<std::array<Vulkan::Event, EventRing>> pass_done_events;
	uint64_t frame_counter = 0;
	std::vector<std::unique_ptr<Vulkan::ImageView>> physical_pingpong_spare;
	std::vector<Vulkan::BufferHandle> physical_buffer_spare;
	static bool async_post;
	const void *physical_key(const RenderResource &res, bool history);
	std::vector<GrbRows> shard_bands;
	unsigned shard_rank = 0;
	bool shard_fxaa = false;
	bool shard_taa = false;
	int shard_smaa = -1;
	RenderGraphCollectives *collectives = nullptr;

	RenderTextureResource &get_or_create_texture(const std::string &name);
	RenderBufferResource &get_or_create_buffer(const std::string &name);
	RenderBufferResource &get_proxy_resource(const std::string &name);
	void traverse_dependencies(unsigned pass_index, std::vector<uint8_t> &state);
	void build_physical_resources();
	friend class RenderPass;
};
} // namespace Granite
