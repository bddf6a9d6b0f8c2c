// shard_plan.hpp -- which rows of which image one rank of a row-sharded frame computes.
//
// Derived backwards from the rows a rank OWNS (its band of the backbuffer): every stage computes
// exactly the rows its consumers on this rank read, so nothing is missing at band edges and the
// sharded frame is bit-identical to the unsharded one.  Stencil reaches used:
//   FXAA      : +-1 px diagonal taps, direction taps <= 8 px * 0.5 + bilinear  -> 6 rows of tonemapped
//   tonemap   : bloom tap = bilinear of upsample-0 at (y+0.5)/4                 -> u0 rows y/4 -+ 1
//   d0 (1/4)  : 9-tap tent, +-1.75 texels of threshold around 2y+1 + bilinear   -> t rows 2y-2 .. 2y+3
//   threshold : bilinear of HDR at 2y+1                                         -> HDR rows 2y .. 2y+1 (+-1)
//   TAA       : current colour, depth and MV at +-1 row (the history is exchanged in full) -> HDR-main rows +-1
// Bands are aligned to 64 full-res rows, so the 1/4-res d0 bands tile that level exactly.
#pragma once

#include <vector>

#include "../../include/granite_b200.h"

namespace Granite
{
struct ShardPlan
{
	GrbRows own;        // backbuffer rows this rank owns (and reads back)
	GrbRows fxaa;       // rows of the FXAA output
	GrbRows tonemap;    // rows of "tonemapped"
	GrbRows upsample0;  // rows of "upsample-0" (1/4)
	GrbRows downsample0; // rows of "downsample-0" (1/4): this rank's contribution to the all-gather
	GrbRows threshold;  // rows of "threshold" (1/2)
	GrbRows lighting;   // rows of "HDR-main" (= rows of the G-buffer that must be resident)
	GrbRows lum_grid;   // rows of the (d3/2) luminance grid this rank samples
	GrbRows taa;        // rows of "HDR-resolved" (what the threshold and the tonemap read); = lighting without TAA
};

// taa: a TAA resolve sits between lighting and the post chain; lighting then covers taa +-1 row.
ShardPlan compute_shard_plan(unsigned width, unsigned height, const std::vector<GrbRows> &bands, unsigned rank, bool fxaa, bool taa = false);
} // namespace Granite
