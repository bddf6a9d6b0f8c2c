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
//   SMAA blend (grb_smaa.cu:500, 501, 525): weights at row 0 one texel right (ax) and at row +1 (ay), colour at rows
//               -1 .. +1 (a blend offset of up to one texel) -> weights rows y-1 .. y+2, tonemapped rows y-2 .. y+2
//               (see "rounding" below)
//   SMAA edges (grb_smaa.cu:167-178): luma at rows -2 (Ltoptop), -1 (Ltop), 0 one or two texels left / right, +1
//               (Lbottom)                                                                -> tonemapped rows y-3 .. y+2
//   SMAA weights (smaa_weights_kernel, S = max_search_steps = 4, 8, 16, 32 for Low .. Ultra):
//               vertical search up (search_axis, grb_smaa.cu:333-355): samples at y-0.25-2k for k = 0 .. K-1, rows
//               y-2k-1, y-2k; then e1 (:465) and the corner taps (:389, :391) at the search end + (3.25 - 2.008*len)
//               >= 1.25 rows (len <= 254/255, the search texture's largest value) -> edge rows up to 2K above y.  Down: samples at y+1.25+2k, rows y+1+2k, y+2+2k; e2 (:471)
//               and the corner taps (:390, :392) at offset +1 from the search end - >= 1.25 rows -> edge rows down to
//               y+2K+2.  K <= S+1:
//               the end test compares fmaf-accumulated coordinates, and for about half the rows of any height the
//               S-th step still lands inside.  Diagonal searches (:215-313; Ultra 16 steps) and the horizontal path
//               (:441-455) reach at most 18 rows.  So an edge window of R_up = 2S+2 rows above the first
//               weights row and R_down = 2S+4 rows past the end of the last (Low 10/12, Medium 18/20, High 34/36,
//               Ultra 66/68).  The kernel source compiled for the CPU with every texel load recorded reads exactly
//               these rows at Ultra and R_down at every preset (tests/test_smaa_sharding_cpu.py).  The edges are
//               exchanged, not recomputed: smaa_edges rows come from their owners.
// Rounding: a tap that is not at the fragment's own coordinate is a bilinear fetch at a row coordinate computed in fp32
// ((y+0.5)/h + k/h, then *h - 0.5), also when k = 0 and only the column is shifted.  For some rows of any height it
// lands a hair off the texel centre, above or below, and the row beyond gets a small nonzero weight: a tap at row
// offset k reads rows k-1 .. k+1 (tests/test_smaa_sharding_cpu.py checks k = -2 .. +1 over several heights).  The
// SMAA rows above include those rows, so a sharded frame stays bit-identical.
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
	GrbRows smaa_weights; // rows of "smaa-weights" (what the blend of `own` reads: own -1 .. +2); = own without SMAA
	GrbRows smaa_edges;   // rows of "smaa-edge" the weights pass reads (own's edges are computed here, the rest received
	                      // from their owners); = own without SMAA
};

// Rows the SMAA weights pass reads above its first row (up) and past its last row (down) for quality 0..3.
void smaa_edge_reach(int quality, int &up, int &down);

// taa: a TAA resolve sits between lighting and the post chain; lighting then covers taa +-1 row.
// smaa_quality: SMAA (0..3 = Low .. Ultra) after the tonemap, < 0 = none; the tonemap then covers own -3 .. +2 rows.
ShardPlan compute_shard_plan(unsigned width, unsigned height, const std::vector<GrbRows> &bands, unsigned rank, bool fxaa, bool taa = false,
                             int smaa_quality = -1);
} // namespace Granite
