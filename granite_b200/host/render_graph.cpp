#include "render_graph.hpp"

#include <algorithm>
#include <cmath>
#include <stdexcept>

namespace Granite
{
bool RenderGraph::async_post = false;

// ---------------------------------------------------------------- RenderPassInterface defaults
bool RenderPassInterface::get_clear_depth_stencil(VkClearDepthStencilValue *value) const
{
	if (value)
		*value = { 1.0f, 0u };
	return true;
}

bool RenderPassInterface::get_clear_color(unsigned, VkClearColorValue *value) const
{
	if (value)
		*value = {};
	return true;
}

void RenderPassInterface::setup_dependencies(RenderPass &, RenderGraph &) {}
void RenderPassInterface::setup(Vulkan::Device &) {}
void RenderPassInterface::enqueue_prepare_render_pass(RenderGraph &, TaskComposer &) {}
void RenderPassInterface::build_render_pass(Vulkan::CommandBuffer &) {}
void RenderPassInterface::build_render_pass_separate_layer(Vulkan::CommandBuffer &, unsigned) {}

// ---------------------------------------------------------------- RenderPass declarators
bool RenderPass::get_clear_color(unsigned attachment, VkClearColorValue *value) const
{
	if (render_pass_handle)
		return render_pass_handle->get_clear_color(attachment, value);
	if (get_clear_color_cb)
		return get_clear_color_cb(attachment, value);
	return false;
}

bool RenderPass::get_clear_depth_stencil(VkClearDepthStencilValue *value) const
{
	if (render_pass_handle)
		return render_pass_handle->get_clear_depth_stencil(value);
	if (get_clear_depth_stencil_cb)
		return get_clear_depth_stencil_cb(value);
	return false;
}

RenderTextureResource &RenderPass::set_depth_stencil_input(const std::string &name)
{
	auto &res = graph.get_or_create_texture(name);
	res.read_in_pass(index);
	depth_stencil_input = &res;
	reads.push_back(&res);
	return res;
}

RenderTextureResource &RenderPass::set_depth_stencil_output(const std::string &name, const AttachmentInfo &info)
{
	auto &res = graph.get_or_create_texture(name);
	res.written_in_pass(index);
	res.set_attachment_info(info);
	depth_stencil_output = &res;
	writes.push_back(&res);
	return res;
}

RenderTextureResource &RenderPass::add_color_output(const std::string &name, const AttachmentInfo &info, const std::string &input)
{
	auto &res = graph.get_or_create_texture(name);
	res.written_in_pass(index);
	res.set_attachment_info(info);
	color_outputs.push_back(&res);
	writes.push_back(&res);
	if (!input.empty())
	{
		auto &input_res = graph.get_or_create_texture(input);
		input_res.read_in_pass(index);
		color_inputs.push_back(&input_res);
		reads.push_back(&input_res);
		rmw_aliases.emplace_back(&res, &input_res);
	}
	else
		color_inputs.push_back(nullptr);
	return res;
}

RenderTextureResource &RenderPass::add_attachment_input(const std::string &name)
{
	auto &res = graph.get_or_create_texture(name);
	res.read_in_pass(index);
	attachments_inputs.push_back(&res);
	reads.push_back(&res);
	return res;
}

RenderTextureResource &RenderPass::add_history_input(const std::string &name)
{
	auto &res = graph.get_or_create_texture(name);
	// History inputs are not used in any particular pass, but next frame.
	history_inputs.push_back(&res);
	return res;
}

RenderTextureResource &RenderPass::add_texture_input(const std::string &name, VkPipelineStageFlags2)
{
	auto &res = graph.get_or_create_texture(name);
	res.read_in_pass(index);
	texture_inputs.push_back(&res);
	reads.push_back(&res);
	return res;
}

RenderBufferResource &RenderPass::add_uniform_input(const std::string &name, VkPipelineStageFlags2)
{
	auto &res = graph.get_or_create_buffer(name);
	res.read_in_pass(index);
	buffer_inputs.push_back(&res);
	reads.push_back(&res);
	return res;
}

RenderBufferResource &RenderPass::add_storage_read_only_input(const std::string &name, VkPipelineStageFlags2 stages)
{
	return add_uniform_input(name, stages);
}

void RenderPass::add_proxy_output(const std::string &name, VkPipelineStageFlags2 stages, VkAccessFlags2, const std::string &input)
{
	if (stages == 0)
		throw std::logic_error("add_proxy_output: stages must not be 0.");
	auto &res = graph.get_proxy_resource(name);
	res.written_in_pass(index);
	writes.push_back(&res);
	if (!input.empty())
	{
		auto &input_res = graph.get_proxy_resource(input);
		input_res.read_in_pass(index);
		reads.push_back(&input_res);
	}
}

void RenderPass::add_proxy_input(const std::string &name, VkPipelineStageFlags2 stages, VkAccessFlags2)
{
	if (stages == 0)
		throw std::logic_error("add_proxy_input: stages must not be 0.");
	auto &res = graph.get_proxy_resource(name);
	res.read_in_pass(index);
	reads.push_back(&res);
}

void RenderPass::add_external_lock(const std::string &name, VkPipelineStageFlags2 stages, VkAccessFlags2 access)
{
	auto *iface = graph.find_external_lock_interface(name);
	if (!iface)
		return;
	iface->mark_access_in_queue(queue, stages, access);
	for (auto &l : lock_interfaces)
		if (l.iface == iface)
		{
			l.stages |= stages;
			return;
		}
	lock_interfaces.push_back({ iface, stages });
}

Vulkan::Event RenderPassExternalLockInterface::external_acquire_event()
{
	std::lock_guard<std::mutex> hold(lock);
	return produced;
}

void RenderPassExternalLockInterface::external_release_event(Vulkan::Event event)
{
	if (!event)
		return;
	std::lock_guard<std::mutex> hold(lock);
	for (auto e : consumed)
		if (e == event)
			return;
	consumed.push_back(event);
}

void RenderPassExternalLockInterface::acquire_internal(Vulkan::Device &device, Vulkan::Stream stream)
{
	std::lock_guard<std::mutex> hold(lock);
	for (auto e : consumed)
		device.stream_wait_event(stream, e);
	consumed.clear();
}

void RenderPassExternalLockInterface::release_internal(Vulkan::Device &device, Vulkan::Stream stream)
{
	std::lock_guard<std::mutex> hold(lock);
	if (!produced)
		produced = device.request_event();
	device.record_event_on(produced, stream);
}

RenderBufferResource &RenderPass::add_storage_output(const std::string &name, const BufferInfo &info, const std::string &input)
{
	auto &res = graph.get_or_create_buffer(name);
	res.set_buffer_info(info);
	res.written_in_pass(index);
	storage_outputs.push_back(&res);
	writes.push_back(&res);
	if (!input.empty())
	{
		auto &input_res = graph.get_or_create_buffer(input);
		input_res.read_in_pass(index);
		reads.push_back(&input_res);
		rmw_aliases.emplace_back(&res, &input_res);
	}
	return res;
}

RenderBufferResource &RenderPass::add_transfer_output(const std::string &name, const BufferInfo &info)
{
	auto &res = graph.get_or_create_buffer(name);
	res.set_buffer_info(info);
	res.written_in_pass(index);
	transfer_outputs.push_back(&res);
	writes.push_back(&res);
	return res;
}

RenderTextureResource &RenderPass::add_storage_texture_output(const std::string &name, const AttachmentInfo &info, const std::string &input)
{
	auto &res = graph.get_or_create_texture(name);
	res.written_in_pass(index);
	res.set_attachment_info(info);
	storage_texture_outputs.push_back(&res);
	writes.push_back(&res);
	if (!input.empty())
	{
		auto &input_res = graph.get_or_create_texture(input);
		input_res.read_in_pass(index);
		reads.push_back(&input_res);
		rmw_aliases.emplace_back(&res, &input_res);
	}
	return res;
}

void RenderPass::add_fake_resource_write_alias(const std::string &from, const std::string &to)
{
	auto &from_res = graph.get_or_create_texture(from);
	auto &to_res = graph.get_or_create_texture(to);
	to_res.set_attachment_info(from_res.get_attachment_info());
	to_res.written_in_pass(index);
	from_res.read_in_pass(index);
	reads.push_back(&from_res);
	writes.push_back(&to_res);
	rmw_aliases.emplace_back(&to_res, &from_res);
}

// ---------------------------------------------------------------- RenderGraph
Vulkan::Device &RenderGraph::get_device()
{
	if (!device)
		throw std::logic_error("RenderGraph: no device set.");
	return *device;
}

RenderTextureResource &RenderGraph::get_or_create_texture(const std::string &name)
{
	auto itr = resource_to_index.find(name);
	if (itr != resource_to_index.end())
	{
		if (resources[itr->second]->get_type() != RenderResource::Type::Texture)
			throw std::logic_error("Resource '" + name + "' is not a texture.");
		return static_cast<RenderTextureResource &>(*resources[itr->second]);
	}
	unsigned index = (unsigned)resources.size();
	resources.emplace_back(new RenderTextureResource(index));
	resources.back()->set_name(name);
	resource_to_index[name] = index;
	return static_cast<RenderTextureResource &>(*resources.back());
}

RenderBufferResource &RenderGraph::get_or_create_buffer(const std::string &name)
{
	auto itr = resource_to_index.find(name);
	if (itr != resource_to_index.end())
	{
		if (resources[itr->second]->get_type() != RenderResource::Type::Buffer)
			throw std::logic_error("Resource '" + name + "' is not a buffer.");
		return static_cast<RenderBufferResource &>(*resources[itr->second]);
	}
	unsigned index = (unsigned)resources.size();
	resources.emplace_back(new RenderBufferResource(index));
	resources.back()->set_name(name);
	resource_to_index[name] = index;
	return static_cast<RenderBufferResource &>(*resources.back());
}

RenderTextureResource &RenderGraph::get_texture_resource(const std::string &name) { return get_or_create_texture(name); }
RenderBufferResource &RenderGraph::get_buffer_resource(const std::string &name) { return get_or_create_buffer(name); }

RenderBufferResource &RenderGraph::get_proxy_resource(const std::string &name)
{
	auto &res = get_or_create_buffer(name);
	res.set_proxy(true);
	return res;
}

RenderPass &RenderGraph::add_pass(const std::string &name, RenderGraphQueueFlagBits queue)
{
	auto itr = pass_to_index.find(name);
	if (itr != pass_to_index.end())
		return *passes[itr->second];
	unsigned index = (unsigned)passes.size();
	passes.emplace_back(new RenderPass(*this, index, queue));
	passes.back()->set_name(name);
	pass_to_index[name] = index;
	return *passes.back();
}

RenderPass *RenderGraph::find_pass(const std::string &name)
{
	auto itr = pass_to_index.find(name);
	return itr != pass_to_index.end() ? passes[itr->second].get() : nullptr;
}

void RenderGraph::set_backbuffer_source(const std::string &name) { backbuffer_source = name; }

void RenderGraph::reset()
{
	passes.clear();
	resources.clear();
	pass_to_index.clear();
	resource_to_index.clear();
	pass_stack.clear();
	physical_dimensions.clear();
	physical_has_history.clear();
	physical_attachments.clear();
	physical_history_attachments.clear();
	physical_history_spare.clear();
	physical_buffers.clear();
	last_access.clear();
	marks.clear();
	external_lock_interfaces.clear();
	pass_done_events.clear();
	physical_pingpong_spare.clear();
	physical_buffer_spare.clear();
	backbuffer_physical = RenderResource::Unused;
	baked = false;
}

void RenderGraph::traverse_dependencies(unsigned pass_index, std::vector<uint8_t> &state)
{
	// state: 0 = unvisited, 1 = on the stack, 2 = done
	if (state[pass_index] == 2)
		return;
	if (state[pass_index] == 1)
		throw std::logic_error("Cycle detected in render graph at pass '" + passes[pass_index]->get_name() + "'.");
	state[pass_index] = 1;
	auto &pass = *passes[pass_index];
	for (auto *res : pass.get_all_reads())
	{
		if (res->get_write_passes().empty())
			throw std::logic_error("No pass exists which writes to resource '" + res->get_name() + "'.");
		// deterministic order: ascending pass index
		std::vector<unsigned> writers(res->get_write_passes().begin(), res->get_write_passes().end());
		std::sort(writers.begin(), writers.end());
		for (unsigned w : writers)
			if (w != pass_index)
				traverse_dependencies(w, state);
	}
	state[pass_index] = 2;
	pass_stack.push_back(pass_index);
}

void RenderGraph::bake()
{
	for (auto &pass : passes)
		pass->setup_dependencies();

	auto itr = resource_to_index.find(backbuffer_source);
	if (itr == resource_to_index.end())
		throw std::logic_error("Backbuffer source does not exist.");
	auto &bb = *resources[itr->second];
	if (bb.get_write_passes().empty())
		throw std::logic_error("No pass exists which writes to resource.");

	for (auto &pass : passes)
	{
		for (auto &alias : pass->get_write_aliases())
		{
			if (alias.first->get_type() != alias.second->get_type())
				throw std::logic_error("Read-modify-write alias between a texture and a buffer.");
		}
		if (pass->get_color_inputs().size() != pass->get_color_outputs().size())
			throw std::logic_error("Size of color inputs must match color outputs.");
	}

	pass_stack.clear();
	std::vector<uint8_t> state(passes.size(), 0);
	std::vector<unsigned> writers(bb.get_write_passes().begin(), bb.get_write_passes().end());
	std::sort(writers.begin(), writers.end());
	for (unsigned w : writers)
		traverse_dependencies(w, state);

	build_physical_resources();
	baked = true;

	if (device)
		for (unsigned p : pass_stack)
			passes[p]->setup(*device);
}

ResourceDimensions RenderGraph::get_resource_dimensions(const RenderBufferResource &resource) const
{
	ResourceDimensions dim;
	dim.buffer_info = resource.get_buffer_info();
	dim.flags = resource.get_buffer_info().flags;
	dim.name = resource.get_name();
	return dim;
}

ResourceDimensions RenderGraph::get_resource_dimensions(const RenderTextureResource &resource) const
{
	ResourceDimensions dim;
	auto &info = resource.get_attachment_info();
	dim.format = info.format;
	dim.flags = info.flags;
	dim.name = resource.get_name();
	// renderer/render_graph.cpp:3160-3171: every relative size is ceil(parent * scale)
	switch (info.size_class)
	{
	case SizeClass::SwapchainRelative:
		dim.width = std::max(unsigned(std::ceil(info.size_x * swapchain_dimensions.width)), 1u);
		dim.height = std::max(unsigned(std::ceil(info.size_y * swapchain_dimensions.height)), 1u);
		break;
	case SizeClass::Absolute:
		dim.width = std::max(unsigned(info.size_x), 1u);
		dim.height = std::max(unsigned(info.size_y), 1u);
		break;
	case SizeClass::InputRelative:
	{
		auto itr = resource_to_index.find(info.size_relative_name);
		if (itr == resource_to_index.end())
			throw std::logic_error("Resource does not exist.");
		auto &input = static_cast<const RenderTextureResource &>(*resources[itr->second]);
		auto input_dim = get_resource_dimensions(input);
		dim.width = std::max(unsigned(std::ceil(input_dim.width * info.size_x)), 1u);
		dim.height = std::max(unsigned(std::ceil(input_dim.height * info.size_y)), 1u);
		break;
	}
	}
	if (dim.format == VK_FORMAT_UNDEFINED)
		dim.format = swapchain_dimensions.format;
	return dim;
}

void RenderGraph::build_physical_resources()
{
	physical_dimensions.clear();
	physical_has_history.clear();
	for (auto &res : resources)
		res->set_physical_index(RenderResource::Unused);

	auto assign = [&](RenderResource *res) {
		if (res->get_physical_index() != RenderResource::Unused)
			return;
		unsigned phys = (unsigned)physical_dimensions.size();
		if (res->get_type() == RenderResource::Type::Texture)
			physical_dimensions.push_back(get_resource_dimensions(static_cast<RenderTextureResource &>(*res)));
		else
			physical_dimensions.push_back(get_resource_dimensions(static_cast<RenderBufferResource &>(*res)));
		physical_has_history.push_back(false);
		res->set_physical_index(phys);
	};

	for (unsigned p : pass_stack)
	{
		auto &pass = *passes[p];
		for (auto *res : pass.get_all_reads())
			assign(res);
		// in-place outputs share the physical resource of the input they modify
		for (auto &alias : pass.get_write_aliases())
		{
			assign(alias.second);
			if (alias.first->get_physical_index() == RenderResource::Unused)
				alias.first->set_physical_index(alias.second->get_physical_index());
			else if (alias.first->get_physical_index() != alias.second->get_physical_index())
				throw std::logic_error("Cannot alias resources. Index already claimed.");
		}
		for (auto *res : pass.get_all_writes())
			assign(res);
	}
	for (unsigned p : pass_stack)
		for (auto *res : passes[p]->get_history_inputs())
		{
			if (res->get_physical_index() == RenderResource::Unused)
				throw std::logic_error("History input is used, but it was never written to.");
			physical_has_history[res->get_physical_index()] = true;
		}

	backbuffer_physical = resources[resource_to_index[backbuffer_source]]->get_physical_index();
	physical_attachments.clear();
	physical_attachments.resize(physical_dimensions.size());
	physical_history_attachments.clear();
	physical_history_attachments.resize(physical_dimensions.size());
	physical_buffers.resize(physical_dimensions.size());
}

void RenderGraph::setup_attachments(Vulkan::Device &dev, Vulkan::ImageView *swapchain)
{
	if (!baked)
		throw std::logic_error("setup_attachments() before bake().");
	device = &dev;
	for (unsigned i = 0; i < physical_dimensions.size(); i++)
	{
		auto &dim = physical_dimensions[i];
		if (dim.buffer_info.size != 0)
		{
			// ping-pong buffers alternate between two allocations (fully rewritten every frame)
			if (dim.flags & ATTACHMENT_INFO_PINGPONG_BIT)
			{
				if (physical_buffer_spare.size() != physical_dimensions.size())
					physical_buffer_spare.resize(physical_dimensions.size());
				std::swap(physical_buffer_spare[i], physical_buffers[i]);
			}
			// persistent across frames (and re-bakes via install_physical_buffers)
			if (!physical_buffers[i] || physical_buffers[i]->get_create_info().size != dim.buffer_info.size)
			{
				Vulkan::BufferCreateInfo info;
				info.size = (size_t)dim.buffer_info.size;
				physical_buffers[i] = dev.create_buffer(info);
			}
			continue;
		}
		if (dim.width == 0)
			continue;
		if (i == backbuffer_physical && swapchain)
		{
			if (swapchain->get_view_width() != dim.width || swapchain->get_view_height() != dim.height)
				throw std::logic_error("Swapchain image does not match the backbuffer dimensions.");
			physical_attachments[i].reset(new Vulkan::ImageView(swapchain->get_image_handle()));
			continue;
		}
		// history <-> current swap, renderer/render_graph.cpp:2706-2710
		if (physical_has_history[i])
			std::swap(physical_history_attachments[i], physical_attachments[i]);
		else if (dim.flags & ATTACHMENT_INFO_PINGPONG_BIT)
		{
			if (physical_pingpong_spare.size() != physical_dimensions.size())
				physical_pingpong_spare.resize(physical_dimensions.size());
			std::swap(physical_pingpong_spare[i], physical_attachments[i]);
		}
		auto &att = physical_attachments[i];
		if (!att || att->get_view_width() != dim.width || att->get_view_height() != dim.height || att->get_format() != dim.format)
		{
			Vulkan::ImageCreateInfo info;
			info.width = dim.width;
			info.height = dim.height;
			info.format = dim.format;
			att.reset(new Vulkan::ImageView(dev.create_image(info)));
		}
	}
}

const void *RenderGraph::physical_key(const RenderResource &res, bool history)
{
	unsigned phys = res.get_physical_index();
	if (phys == RenderResource::Unused)
		return nullptr;
	if (res.get_type() == RenderResource::Type::Buffer)
	{
		if (static_cast<const RenderBufferResource &>(res).is_proxy())
			return &res; // no memory behind it: the resource object itself is the key the ordering hangs on
		return physical_buffers[phys] ? physical_buffers[phys].get() : nullptr;
	}
	auto &view = history ? physical_history_attachments[phys] : physical_attachments[phys];
	return view ? static_cast<const void *>(&view->get_image()) : nullptr;
}

Vulkan::Stream RenderGraph::get_writer_stream(const RenderResource &resource)
{
	unsigned idx = 0;
	for (unsigned p : pass_stack)
		if (resource.get_write_passes().count(p))
			idx = queue_stream_index(passes[p]->get_queue());
	return get_device().get_queue_stream(idx);
}

void RenderGraph::enqueue_render_passes(Vulkan::Device &dev, TaskComposer &composer)
{
	if (!baked)
		throw std::logic_error("enqueue_render_passes() before bake().");
	// Each pass records on the stream of its queue (main, async compute, async graphics).
	// Ordering ACROSS streams is derived from the declared resources: before a pass is recorded,
	// its stream waits for the last pass that touched any of its physical images / buffers on
	// another stream: readers wait for the last writer, writers for the last access on every other
	// stream (RAW, WAR and WAW, also across frames because physical resources persist; ping-pong
	// images alternate so consecutive frames do not meet on them).  Within a stream, stream order is
	// the dependency.
	if (pass_done_events.size() != passes.size())
		pass_done_events.assign(passes.size(), std::array<Vulkan::Event, EventRing>{});
	const unsigned slot = unsigned(frame_counter++ % EventRing);
	unsigned errors = 0;
	for (unsigned p : pass_stack)
	{
		auto &pass = *passes[p];
		pass.prepare_render_pass(composer);
		if (!pass.need_render_pass())
			continue;
		Vulkan::Stream stream = dev.get_queue_stream(queue_stream_index(pass.get_queue()));
		Vulkan::CommandBuffer cmd(dev, stream);

		const unsigned stream_index = queue_stream_index(pass.get_queue());
		auto wait_for = [&](const void *key, bool writes) {
			if (!key)
				return;
			auto itr = last_access.find(key);
			if (itr == last_access.end())
				return;
			auto &la = itr->second;
			if (la.write_event && la.write_stream != stream)
				dev.stream_wait_event(stream, la.write_event);
			if (writes)
				for (unsigned i = 0; i < 4; i++)
					if (la.stream_event[i] && la.stream_of[i] != stream && la.stream_event[i] != la.write_event)
						dev.stream_wait_event(stream, la.stream_event[i]);
		};
		auto mark = [&](const void *key, bool writes) {
			if (!key)
				return;
			auto &la = last_access[key];
			la.stream_event[stream_index % 4] = pass_done_events[p][slot];
			la.stream_of[stream_index % 4] = stream;
			if (writes)
			{
				la.write_event = pass_done_events[p][slot];
				la.write_stream = stream;
			}
		};
		{
			Vulkan::ScopedHostTimer timer("graph.cross-stream waits");
			for (auto *r : pass.get_all_reads())
				wait_for(physical_key(*r, false), false);
			for (auto *w : pass.get_all_writes())
				wait_for(physical_key(*w, false), true);
			for (auto *h : pass.get_history_inputs())
				wait_for(physical_key(*h, true), false);
			for (auto &name : pass.get_wait_marks())
				wait_mark(name, cmd);
			for (auto &l : pass.get_lock_interfaces())
				if (Vulkan::Event e = l.iface->external_acquire_event())
					dev.stream_wait_event(stream, e);
		}

		Vulkan::Event begin = nullptr, end = nullptr;
		if (timestamps)
		{
			begin = dev.request_event();
			end = dev.request_event();
			dev.record_event_on(begin, stream);
		}
		cmd.begin_region(pass.get_name().c_str());
		{
			Vulkan::ScopedHostTimer timer(pass.get_name().c_str());
			pass.build_render_pass(cmd, 0);
		}
		cmd.end_region();
		if (timestamps)
		{
			dev.record_event_on(end, stream);
			dev.register_time_interval(pass.get_name(), begin, end);
		}
		Vulkan::ScopedHostTimer timer("graph.pass-done event + marks");
		if (!pass_done_events[p][slot])
			pass_done_events[p][slot] = dev.request_event();
		dev.record_event_on(pass_done_events[p][slot], stream);
		for (auto &l : pass.get_lock_interfaces())
			l.iface->external_release_event(pass_done_events[p][slot]);
		for (auto *r : pass.get_all_reads())
			mark(physical_key(*r, false), false);
		for (auto *w : pass.get_all_writes())
			mark(physical_key(*w, false), true);
		for (auto *h : pass.get_history_inputs())
			mark(physical_key(*h, true), false);
		errors += cmd.get_error_count();
	}
	if (errors)
		Vulkan::log_error("%u pass callback(s) reported errors this frame.\n", errors);
}

void RenderGraph::signal_mark(const std::string &name, Vulkan::CommandBuffer &cmd)
{
	auto &m = marks[name];
	// a small ring: re-recording the event a waiter of an earlier frame still refers to would move its wait forward
	auto &e = m.events[m.next];
	m.next = (m.next + 1) % m.events.size();
	if (!e)
		e = cmd.get_device().request_event();
	cmd.get_device().record_event_on(e, cmd.get_stream());
	m.latest = e;
	m.stream = cmd.get_stream();
}

void RenderGraph::wait_mark(const std::string &name, Vulkan::CommandBuffer &cmd)
{
	auto itr = marks.find(name);
	if (itr != marks.end() && itr->second.latest && itr->second.stream != cmd.get_stream())
		cmd.get_device().stream_wait_event(cmd.get_stream(), itr->second.latest);
}

Vulkan::ImageView &RenderGraph::get_physical_texture_resource(unsigned index)
{
	if (index == RenderResource::Unused || index >= physical_attachments.size() || !physical_attachments[index])
		throw std::logic_error("Physical texture resource is not available (pass culled, or setup_attachments not called).");
	return *physical_attachments[index];
}

Vulkan::ImageView *RenderGraph::get_physical_history_texture_resource(unsigned index)
{
	if (index == RenderResource::Unused || index >= physical_history_attachments.size())
		throw std::logic_error("Invalid physical index.");
	return physical_history_attachments[index].get();
}

Vulkan::Buffer &RenderGraph::get_physical_buffer_resource(unsigned index)
{
	if (index == RenderResource::Unused || index >= physical_buffers.size() || !physical_buffers[index])
		throw std::logic_error("Physical buffer resource is not available.");
	return *physical_buffers[index];
}

Vulkan::ImageView *RenderGraph::maybe_get_physical_texture_resource(RenderTextureResource *resource)
{
	if (resource && resource->get_physical_index() != RenderResource::Unused && physical_attachments[resource->get_physical_index()])
		return physical_attachments[resource->get_physical_index()].get();
	return nullptr;
}

Vulkan::Buffer *RenderGraph::maybe_get_physical_buffer_resource(RenderBufferResource *resource)
{
	if (resource && resource->get_physical_index() != RenderResource::Unused && physical_buffers[resource->get_physical_index()])
		return physical_buffers[resource->get_physical_index()].get();
	return nullptr;
}

std::vector<Vulkan::BufferHandle> RenderGraph::consume_physical_buffers() const { return physical_buffers; }

void RenderGraph::install_physical_buffers(std::vector<Vulkan::BufferHandle> buffers)
{
	// keep a feed-back buffer only where the new bake has a buffer of the same size at that slot
	for (size_t i = 0; i < buffers.size() && i < physical_buffers.size(); i++)
		if (buffers[i] && physical_dimensions[i].buffer_info.size == buffers[i]->get_create_info().size)
			physical_buffers[i] = std::move(buffers[i]);
}

std::vector<std::string> RenderGraph::get_baked_pass_names() const
{
	std::vector<std::string> names;
	for (unsigned p : pass_stack)
		names.push_back(passes[p]->get_name());
	return names;
}

void RenderGraph::log()
{
	for (unsigned p : pass_stack)
	{
		auto &pass = *passes[p];
		Vulkan::log_info("Pass: %s\n", pass.get_name().c_str());
		for (auto *r : pass.get_all_reads())
			Vulkan::log_info("  reads  %s (phys %u)\n", r->get_name().c_str(), r->get_physical_index());
		for (auto *w : pass.get_all_writes())
			Vulkan::log_info("  writes %s (phys %u)\n", w->get_name().c_str(), w->get_physical_index());
	}
}

void RenderGraph::set_row_shards(const std::vector<GrbRows> &bands, unsigned rank, RenderGraphCollectives *collectives_, bool fxaa_downstream,
                                 bool taa_upstream, int smaa_quality)
{
	shard_fxaa = fxaa_downstream;
	shard_taa = taa_upstream;
	shard_smaa = smaa_quality;
	if (!bands.empty())
	{
		if (rank >= bands.size())
			throw std::logic_error("set_row_shards: rank out of range.");
		int expect = 0;
		for (auto &b : bands)
		{
			if (b.y0 != expect || b.y1 <= b.y0)
				throw std::logic_error("set_row_shards: bands must tile the frame in order.");
			expect = b.y1;
		}
		if (bands.size() > 1 && !collectives_)
			throw std::logic_error("set_row_shards: more than one band needs a collectives implementation.");
	}
	shard_bands = bands;
	shard_rank = rank;
	collectives = collectives_;
}

GrbRows RenderGraph::shard_rows_for_rank(unsigned rank, unsigned resource_height, unsigned halo_rows) const
{
	GrbRows r = { 0, 0 };
	if (!is_sharded())
		return r;
	const unsigned H = swapchain_dimensions.height;
	const auto &band = shard_bands[rank];
	// rows of a (possibly smaller) resource that cover the band's backbuffer rows
	uint64_t lo = (uint64_t)band.y0 * resource_height / H;
	uint64_t hi = ((uint64_t)band.y1 * resource_height + H - 1) / H;
	r.y0 = std::max((int)lo - (int)halo_rows, 0);
	r.y1 = std::min((int)hi + (int)halo_rows, (int)resource_height);
	if (r.y1 <= r.y0)
		r.y1 = r.y0 + 1; // never the {0,0} "all rows" value for a shard
	return r;
}

GrbRows RenderGraph::shard_rows_for(unsigned resource_height, unsigned halo_rows) const
{
	return shard_rows_for_rank(shard_rank, resource_height, halo_rows);
}
} // namespace Granite
