#include "shard_plan.hpp"

#include <algorithm>
#include <cmath>

namespace Granite
{
namespace
{
unsigned ceil_scale(unsigned v, float s) { return (unsigned)std::max(1.0f, std::ceil(v * s)); }

GrbRows clamp_rows(int y0, int y1, unsigned h)
{
	GrbRows r;
	r.y0 = std::max(y0, 0);
	r.y1 = std::min(y1, (int)h);
	if (r.y1 <= r.y0)
		r.y1 = r.y0 + 1;
	return r;
}

GrbRows scale_band(GrbRows band, unsigned from_h, unsigned to_h)
{
	GrbRows r;
	r.y0 = (int)(((uint64_t)band.y0 * to_h) / from_h);
	r.y1 = (int)(((uint64_t)band.y1 * to_h + from_h - 1) / from_h);
	return r;
}
} // namespace

void smaa_edge_reach(int quality, int &up, int &down)
{
	static const int max_search_steps[4] = { 4, 8, 16, 32 }; // SMAA.hlsl:304-324, grb_smaa.cu preset_of()
	const int s = max_search_steps[quality < 0 ? 0 : (quality > 3 ? 3 : quality)];
	up = 2 * s + 2;
	down = 2 * s + 4;
}

ShardPlan compute_shard_plan(unsigned, unsigned height, const std::vector<GrbRows> &bands, unsigned rank, bool fxaa, bool taa, int smaa_quality)
{
	ShardPlan p = {};
	const unsigned h_half = ceil_scale(height, 0.5f), h_quarter = ceil_scale(height, 0.25f);
	const unsigned h_d3 = ceil_scale(height, 0.03125f), h_grid = h_d3 / 2;
	if (bands.size() <= 1)
	{
		GrbRows all = { 0, (int)height };
		p.own = p.fxaa = p.tonemap = p.lighting = p.taa = p.smaa_weights = p.smaa_edges = all;
		p.upsample0 = p.downsample0 = GrbRows{ 0, (int)h_quarter };
		p.threshold = GrbRows{ 0, (int)h_half };
		p.lum_grid = GrbRows{ 0, (int)h_grid };
		return p;
	}
	p.own = bands[rank];
	p.fxaa = p.own;
	p.tonemap = fxaa ? clamp_rows(p.own.y0 - 6, p.own.y1 + 6, height) : p.own;
	p.smaa_weights = p.smaa_edges = p.own;
	if (smaa_quality >= 0)
	{
		int up = 0, down = 0;
		smaa_edge_reach(smaa_quality, up, down);
		p.tonemap = clamp_rows(p.own.y0 - 3, p.own.y1 + 2, height);
		p.smaa_weights = clamp_rows(p.own.y0 - 1, p.own.y1 + 2, height);
		p.smaa_edges = clamp_rows(p.smaa_weights.y0 - up, p.smaa_weights.y1 + down, height);
	}
	p.upsample0 = clamp_rows(p.tonemap.y0 / 4 - 1, (p.tonemap.y1 + 3) / 4 + 1, h_quarter);
	p.downsample0 = scale_band(p.own, height, h_quarter);
	p.threshold = clamp_rows(2 * p.downsample0.y0 - 2, 2 * p.downsample0.y1 + 2, h_half);
	GrbRows hdr_for_threshold = clamp_rows(2 * p.threshold.y0 - 1, 2 * p.threshold.y1 + 1, height);
	p.taa = clamp_rows(std::min(p.tonemap.y0, hdr_for_threshold.y0), std::max(p.tonemap.y1, hdr_for_threshold.y1), height);
	p.lighting = taa ? clamp_rows(p.taa.y0 - 1, p.taa.y1 + 1, height) : p.taa;
	// luminance grid rows: row g belongs to the rank whose band holds the first backbuffer row it maps to
	auto begin_of = [&](unsigned r) { return (int)(((uint64_t)bands[r].y0 * h_grid + height - 1) / height); };
	p.lum_grid.y0 = begin_of(rank);
	p.lum_grid.y1 = rank + 1 < bands.size() ? begin_of(rank + 1) : (int)h_grid;
	return p;
}
} // namespace Granite
