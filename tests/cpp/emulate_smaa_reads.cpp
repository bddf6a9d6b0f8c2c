// emulate_smaa_reads.cpp -- the SMAA weights kernel of granite_b200/csrc/grb_smaa.cu compiled for the CPU
// (cuda_host_emul.h) with every texel load recorded: for each pixel, the lowest and highest row of the edge image it
// reads.  tests/test_smaa_sharding_cpu.py checks the edge window of the row-sharded plan against these rows.
#include "cuda_host_emul.h"

#include <cstddef>
#include <vector>

namespace
{
thread_local const uint8_t *g_edges = nullptr; // the edge image whose reads are recorded
thread_local size_t g_edges_bytes = 0, g_edges_pitch = 0;
thread_local int g_lo = 0, g_hi = 0;

template <typename T>
inline T recording_ldg(const T *p)
{
	const uint8_t *q = reinterpret_cast<const uint8_t *>(p);
	if (q >= g_edges && q < g_edges + g_edges_bytes)
	{
		const int row = (int)((size_t)(q - g_edges) / g_edges_pitch);
		g_lo = row < g_lo ? row : g_lo;
		g_hi = row > g_hi ? row : g_hi;
	}
	return *p;
}
} // namespace

#define __ldg recording_ldg
#define GRB_HOST_EMULATION 1
#include "../../granite_b200/csrc/grb_smaa.cu"

// lo[y * w + x] / hi[...]: the rows of `edges` the weights pass of pixel (x, y) reads, for the rows [y0, y1)
extern "C" void emu_smaa_weight_reads(const uint8_t *edges, int w, int h, const uint8_t *area, const uint8_t *search, int quality, int y0, int y1, int *lo,
                                      int *hi)
{
	GrbImage e = {}, a = {}, s = {}, o = {};
	e.data = const_cast<uint8_t *>(edges);
	e.width = w;
	e.height = h;
	e.row_pitch = w * 2;
	e.format = GRB_FORMAT_R8G8_UNORM;
	a.data = const_cast<uint8_t *>(area);
	a.width = 160;
	a.height = 560;
	a.row_pitch = 320;
	a.format = GRB_FORMAT_R8G8_UNORM;
	s.data = const_cast<uint8_t *>(search);
	s.width = 64;
	s.height = 16;
	s.row_pitch = 64;
	s.format = GRB_FORMAT_R8_UNORM;
	std::vector<uint32_t> weights((size_t)w * h);
	o.data = weights.data();
	o.width = w;
	o.height = h;
	o.row_pitch = w * 4;
	o.format = GRB_FORMAT_R8G8B8A8_UNORM;
	g_edges = edges;
	g_edges_bytes = (size_t)w * h * 2;
	g_edges_pitch = (size_t)w * 2;
	const unsigned gx = (unsigned)((w + 31) / 32), gy = (unsigned)((y1 - y0 + 7) / 8);
	for (unsigned by = 0; by < gy; by++)
		for (unsigned bx = 0; bx < gx; bx++)
			for (unsigned ty = 0; ty < 8; ty++)
				for (unsigned tx = 0; tx < 32; tx++)
				{
					emu_blockIdx.x = bx;
					emu_blockIdx.y = by;
					emu_threadIdx.x = tx;
					emu_threadIdx.y = ty;
					const int x = (int)(bx * 32 + tx), y = y0 + (int)(by * 8 + ty);
					g_lo = h;
					g_hi = -1;
					grb::smaa_weights_kernel(grb::tex_of<2>(&e), grb::tex_of<2>(&a), grb::tex_of<1>(&s), grb::view_of<uint32_t>(&o), grb::preset_of(quality), y0, y1);
					if (x < w && y < y1)
					{
						lo[(size_t)y * w + x] = g_lo;
						hi[(size_t)y * w + x] = g_hi;
					}
				}
	g_edges = nullptr;
}
