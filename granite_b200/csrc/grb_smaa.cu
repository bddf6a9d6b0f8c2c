// grb_smaa.cu -- SMAA 1x (renderer/post/smaa.cpp:32-209): luma edge detection, blending-weight calculation
// (orthogonal and diagonal searches through the area / search lookup textures, corner detection), neighbourhood
// blending; presets Low .. Ultra = SMAA_QUALITY 0..3 (SMAA.hlsl:304-324).
//
// The arithmetic follows assets/shaders/post/SMAA.hlsl as the reference compiles it (SMAA_GLSL_4: mad() is a fused
// multiply-add) statement for statement, with the sampler decisions of DESIGN.md section 2: LinearClamp = bilinear with
// exact fp32 weights, a sample at the fragment's own coordinate is a texel fetch, the vertex stage's offsets are
// evaluated per fragment.  Compiled with -fmad=false: the only fused operations are the fmaf() calls that stand for
// the shader's mad().
//
// One thread per pixel.  The edge and blend passes are streaming; the weight pass returns at once for the pixels
// without an edge (the vast majority) and walks the searches for the rest.
#include <cstdint>
#include <type_traits>

#include "grb_common.cuh"

namespace grb
{
namespace
{
struct SmaaPreset
{
	float threshold;
	float max_search_steps;
	float max_search_steps_diag; // 0: SMAA_DISABLE_DIAG_DETECTION
	int corner_detection;        // 0: SMAA_DISABLE_CORNER_DETECTION (rounding 25 % when on)
};

SmaaPreset preset_of(int quality)
{
	static const SmaaPreset p[4] = {
		{ 0.15f, 4.0f, 0.0f, 0 },
		{ 0.1f, 8.0f, 0.0f, 0 },
		{ 0.1f, 16.0f, 8.0f, 1 },
		{ 0.05f, 32.0f, 16.0f, 1 },
	};
	return p[quality < 0 ? 0 : (quality > 3 ? 3 : quality)];
}

// An 8-bit UNORM texture with C channels per texel (1: search, 2: edges / area, 4: colour / weights).
template <int C>
struct Tex8
{
	const uint8_t *p;
	int w, h;
	size_t pitch; // bytes per row
};

template <int C>
GRB_DEV float4 texel8(const Tex8<C> &t, int x, int y)
{
	x = iclamp(x, 0, t.w - 1);
	y = iclamp(y, 0, t.h - 1);
	const uint8_t *q = t.p + (size_t)y * t.pitch + (size_t)x * C;
	float4 r = make_float4(0.0f, 0.0f, 0.0f, 1.0f);
	if (C == 1)
		r.x = fdiv((float)__ldg(q), 255.0f);
	else if (C == 2)
	{
		const uchar2 v = __ldg(reinterpret_cast<const uchar2 *>(q));
		r.x = fdiv((float)v.x, 255.0f);
		r.y = fdiv((float)v.y, 255.0f);
	}
	else
	{
		const uchar4 v = __ldg(reinterpret_cast<const uchar4 *>(q));
		r.x = fdiv((float)v.x, 255.0f);
		r.y = fdiv((float)v.y, 255.0f);
		r.z = fdiv((float)v.z, 255.0f);
		r.w = fdiv((float)v.w, 255.0f);
	}
	return r;
}

struct Frag
{
	float u, v;
	int x, y;
};

// textureLod / texture / textureLodOffset.  `f` non-null: a texture of the render target's size, fetched when the
// coordinate is the fragment's own.
template <int C>
GRB_DEV float4 sample8(const Tex8<C> &t, float u, float v, int ox, int oy, const Frag *f)
{
	if (f && u == f->u && v == f->v)
		return texel8(t, f->x + ox, f->y + oy);
	const float fx = fsub(fmul(u, (float)t.w), 0.5f), fy = fsub(fmul(v, (float)t.h), 0.5f);
	float flx = floorf(fx), fly = floorf(fy);
	const float a = fsub(fx, flx), b = fsub(fy, fly);
	flx = fclamp(flx, -2.0f, (float)t.w + 1.0f);
	fly = fclamp(fly, -2.0f, (float)t.h + 1.0f);
	if (!(flx == flx)) flx = 0.0f;
	if (!(fly == fly)) fly = 0.0f;
	const int x0 = (int)flx, y0 = (int)fly;
	const float4 t00 = texel8(t, x0 + ox, y0 + oy), t10 = texel8(t, x0 + 1 + ox, y0 + oy);
	const float4 t01 = texel8(t, x0 + ox, y0 + 1 + oy), t11 = texel8(t, x0 + 1 + ox, y0 + 1 + oy);
	return bilin_mix4(t00, t10, t01, t11, a, b);
}

GRB_DEV float step_f(float edge, float x) { return x < edge ? 0.0f : 1.0f; }
GRB_DEV uint32_t unorm8(float c)
{
	c = c > 0.0f ? (c < 1.0f ? c : 1.0f) : 0.0f;
	return (uint32_t)floorf(fadd(fmul(c, 255.0f), 0.5f));
}

// ------------------------------------------------------------------------------------------------ edges
// The edge exchange of a row-sharded frame (the peer form of the edge pass): each edge texel of the rows [y0, y1) goes
// to the edge slot of every rank r whose rows[r] hold its row instead of `edges`, then the last CTA raises
// flags[flag_index] = epoch on every rank (as bloom_downsample_peers_kernel in grb_post.cu).  NoSmaaPeerStore: the
// plain pass.  SmaaPeerStore and its two members exist only in the device build; the host emulation of this file
// (tests/cpp/emulate_smaa.cpp) never instantiates the peer form.
struct NoSmaaPeerStore
{
};
#ifndef GRB_HOST_EMULATION
struct SmaaPeerStore
{
	uchar2 *data[GRB_MAX_PEERS];
	uint32_t *flags[GRB_MAX_PEERS];
	int row0[GRB_MAX_PEERS], row1[GRB_MAX_PEERS];
	int count, pitch_texels, flag_index;
	uint32_t epoch;
	unsigned *ctas_done;

	// A warp is 32 consecutive texels of one row: each store below is 64 contiguous bytes, and the row test is
	// uniform across the warp.
	GRB_DEV void store(int x, int y, uchar2 v) const
	{
		const size_t at = (size_t)y * pitch_texels + x;
		for (int r = 0; r < count; r++)
			if (y >= row0[r] && y < row1[r])
				data[r][at] = v;
	}
	// every CTA has stored its texels before it arrives; the last one raises the flag on every rank, also on ranks that
	// received no rows
	GRB_DEV void publish() const { publish_to_peers(flags, count, flag_index, epoch, ctas_done); }
};
#endif

// SMAALumaEdgeDetectionPS (SMAA.hlsl:689-746) + SMAAEdgeDetectionVS (:645-650)
template <typename PeerStore = NoSmaaPeerStore>
__global__ void __launch_bounds__(256) smaa_edge_kernel(Tex8<4> col, View<uchar2> edges, SmaaPreset P, int y0, int y1, PeerStore peers = PeerStore{})
{
	constexpr bool kPeers = !std::is_same<PeerStore, NoSmaaPeerStore>::value;
	int x = blockIdx.x * 32 + threadIdx.x, y = y0 + blockIdx.y * 8 + threadIdx.y;
	const bool inside = x < col.w && y < y1;
	if (!inside)
	{
		if (!kPeers)
			return;
		// every thread of the peer form reaches the CTA barrier of publish(): off the band it computes a clamped pixel
		// and stores nothing
		x = min(x, col.w - 1);
		y = min(y, y1 - 1);
	}
	const float mx = fdiv(1.0f, (float)col.w), my = fdiv(1.0f, (float)col.h);
	const Frag f = { fmul((float)x + 0.5f, mx), fmul((float)y + 0.5f, my), x, y };
	uchar2 out = make_uchar2(0, 0);
	auto luma = [&](float u, float v) {
		const float4 c = sample8(col, u, v, 0, 0, &f);
		return fadd(fadd(fmul(c.x, 0.2126f), fmul(c.y, 0.7152f)), fmul(c.z, 0.0722f));
	};
	const float L = luma(f.u, f.v);
	const float Lleft = luma(fmaf(mx, -1.0f, f.u), fmaf(my, 0.0f, f.v));
	const float Ltop = luma(fmaf(mx, 0.0f, f.u), fmaf(my, -1.0f, f.v));
	const float dx = fabsf(fsub(L, Lleft)), dy = fabsf(fsub(L, Ltop));
	float ex = step_f(P.threshold, dx), ey = step_f(P.threshold, dy);
	if (fadd(ex, ey) != 0.0f) // otherwise the shader discards: the attachment keeps its clear colour, 0
	{
		const float Lright = luma(fmaf(mx, 1.0f, f.u), fmaf(my, 0.0f, f.v));
		const float Lbottom = luma(fmaf(mx, 0.0f, f.u), fmaf(my, 1.0f, f.v));
		float dz = fabsf(fsub(L, Lright)), dw = fabsf(fsub(L, Lbottom));
		float maxx = fmax_(dx, dz), maxy = fmax_(dy, dw);
		const float Lleftleft = luma(fmaf(mx, -2.0f, f.u), fmaf(my, 0.0f, f.v));
		const float Ltoptop = luma(fmaf(mx, 0.0f, f.u), fmaf(my, -2.0f, f.v));
		dz = fabsf(fsub(Lleft, Lleftleft));
		dw = fabsf(fsub(Ltop, Ltoptop));
		maxx = fmax_(maxx, dz);
		maxy = fmax_(maxy, dw);
		const float final_delta = fmax_(maxx, maxy);
		ex = fmul(ex, step_f(final_delta, fmul(dx, 2.0f)));
		ey = fmul(ey, step_f(final_delta, fmul(dy, 2.0f)));
		out = make_uchar2((unsigned char)unorm8(ex), (unsigned char)unorm8(ey));
	}
	if constexpr (!kPeers)
		edges.at(x, y) = out;
	else
	{
		if (inside)
			peers.store(x, y, out);
		peers.publish();
	}
}

// ------------------------------------------------------------------------------------------------ weights
struct WCtx
{
	Tex8<2> edges, area;
	Tex8<1> search;
	float mx, my, mz, mw;
	SmaaPreset P;
	const Frag *f;
};

GRB_DEV float2 decode_diag2(float2 e)
{
	e.x = fmul(e.x, fabsf(fsub(fmul(5.0f, e.x), 3.75f)));
	return make_float2(roundf(e.x), roundf(e.y));
}

// SMAASearchDiag1 / 2 (SMAA.hlsl:862-895)
GRB_DEV float2 search_diag(const WCtx &c, float tu, float tv, float dirx, float diry, float2 &e, bool second)
{
	float cx = tu, cy = tv, cz = -1.0f, cw = 1.0f;
	if (second)
		cx = fadd(cx, fmul(0.25f, c.mx));
	while (cz < fsub(c.P.max_search_steps_diag, 1.0f) && cw > 0.9f)
	{
		cx = fmaf(c.mx, dirx, cx);
		cy = fmaf(c.my, diry, cy);
		cz = fmaf(1.0f, 1.0f, cz);
		const float4 s = sample8(c.edges, cx, cy, 0, 0, c.f);
		e = make_float2(s.x, s.y);
		if (second)
			e = decode_diag2(e);
		cw = fadd(fmul(e.x, 0.5f), fmul(e.y, 0.5f));
	}
	return make_float2(cz, cw);
}

// SMAAAreaDiag (SMAA.hlsl:900-914)
GRB_DEV float2 area_diag(const WCtx &c, float distx, float disty, float ex, float ey, float offset)
{
	float tx = fmaf(20.0f, ex, distx), ty = fmaf(20.0f, ey, disty);
	tx = fmaf(0.0062500000931322574615478515625f, tx, 0.00312500004656612873077392578125f);
	ty = fmaf(0.001785714295692741870880126953125f, ty, 0.0008928571478463709354400634765625f);
	tx = fadd(tx, 0.5f);
	ty = fadd(ty, fmul(0.14285714924335479736328125f, offset));
	const float4 s = sample8(c.area, tx, ty, 0, 0, nullptr);
	return make_float2(s.x, s.y);
}

// SMAACalculateDiagWeights (SMAA.hlsl:919-985)
GRB_DEV float2 diag_weights(const WCtx &c, float e_in_x)
{
	const float tu = c.f->u, tv = c.f->v;
	float2 weights = make_float2(0.0f, 0.0f), end = make_float2(0.0f, 0.0f);
	float d_x, d_y, d_z, d_w;
	if (e_in_x > 0.0f)
	{
		const float2 r = search_diag(c, tu, tv, -1.0f, 1.0f, end, false);
		d_x = r.x;
		d_z = r.y;
		d_x = fadd(d_x, end.y > 0.9f ? 1.0f : 0.0f);
	}
	else
		d_x = d_z = 0.0f;
	{
		const float2 r = search_diag(c, tu, tv, 1.0f, -1.0f, end, false);
		d_y = r.x;
		d_w = r.y;
	}
	if (fadd(d_x, d_y) > 2.0f)
	{
		const float c0x = fmaf(fadd(-d_x, 0.25f), c.mx, tu), c0y = fmaf(d_x, c.my, tv);
		const float c1x = fmaf(d_y, c.mx, tu), c1y = fmaf(fsub(-d_y, 0.25f), c.my, tv);
		const float4 a = sample8(c.edges, c0x, c0y, -1, 0, c.f), b = sample8(c.edges, c1x, c1y, 1, 0, c.f);
		const float qx = fmul(a.x, fabsf(fsub(fmul(a.x, 5.0f), 3.75f))), qz = fmul(b.x, fabsf(fsub(fmul(b.x, 5.0f), 3.75f)));
		const float rx = roundf(qx), ry = roundf(a.y), rz = roundf(qz), rw = roundf(b.y);
		float ccx = fmaf(2.0f, ry, rx), ccy = fmaf(2.0f, rw, rz);
		if (step_f(0.9f, d_z) != 0.0f)
			ccx = 0.0f;
		if (step_f(0.9f, d_w) != 0.0f)
			ccy = 0.0f;
		const float2 ar = area_diag(c, d_x, d_y, ccx, ccy, 0.0f);
		weights.x = fadd(weights.x, ar.x);
		weights.y = fadd(weights.y, ar.y);
	}
	{
		const float2 r = search_diag(c, tu, tv, -1.0f, -1.0f, end, true);
		d_x = r.x;
		d_z = r.y;
	}
	if (sample8(c.edges, tu, tv, 1, 0, c.f).x > 0.0f)
	{
		const float2 r = search_diag(c, tu, tv, 1.0f, 1.0f, end, true);
		d_y = r.x;
		d_w = r.y;
		d_y = fadd(d_y, end.y > 0.9f ? 1.0f : 0.0f);
	}
	else
		d_y = d_w = 0.0f;
	if (fadd(d_x, d_y) > 2.0f)
	{
		const float c0x = fmaf(-d_x, c.mx, tu), c0y = fmaf(-d_x, c.my, tv);
		const float c1x = fmaf(d_y, c.mx, tu), c1y = fmaf(d_y, c.my, tv);
		const float c_x = sample8(c.edges, c0x, c0y, -1, 0, c.f).y;
		const float c_y = sample8(c.edges, c0x, c0y, 0, -1, c.f).x;
		const float4 s = sample8(c.edges, c1x, c1y, 1, 0, c.f);
		const float c_z = s.y, c_w = s.x;
		float ccx = fmaf(2.0f, c_x, c_y), ccy = fmaf(2.0f, c_z, c_w);
		if (step_f(0.9f, d_z) != 0.0f)
			ccx = 0.0f;
		if (step_f(0.9f, d_w) != 0.0f)
			ccy = 0.0f;
		const float2 ar = area_diag(c, d_x, d_y, ccx, ccy, 0.0f);
		weights.x = fadd(weights.x, ar.y);
		weights.y = fadd(weights.y, ar.x);
	}
	return weights;
}

// SMAASearchLength (SMAA.hlsl:997-1014)
GRB_DEV float search_length(const WCtx &c, float ex, float ey, float offset)
{
	float sx = 33.0f, sy = -33.0f;
	float bx = fmul(66.0f, offset), by = fmul(33.0f, 1.0f);
	sx = fadd(sx, -1.0f);
	sy = fadd(sy, 1.0f);
	bx = fadd(bx, 0.5f);
	by = fadd(by, -0.5f);
	sx = fmul(sx, 0.015625f);
	sy = fmul(sy, 0.0625f);
	bx = fmul(bx, 0.015625f);
	by = fmul(by, 0.0625f);
	return sample8(c.search, fmaf(sx, ex, bx), fmaf(sy, ey, by), 0, 0, nullptr).x;
}

// SMAASearchXLeft / XRight / YUp / YDown (SMAA.hlsl:1019-1086).  axis 0: x, 1: y; sign -1: towards smaller.
GRB_DEV float search_axis(const WCtx &c, float tu, float tv, float end, int axis, float sign)
{
	float ex = axis ? 1.0f : 0.0f, ey = axis ? 0.0f : 1.0f;
	for (;;)
	{
		const float pos = axis ? tv : tu;
		const bool inside = sign < 0.0f ? pos > end : pos < end;
		const float along = axis ? ex : ey, cross = axis ? ey : ex;
		if (!(inside && along > 0.828100025653839111328125f && cross == 0.0f))
			break;
		const float4 s = sample8(c.edges, tu, tv, 0, 0, c.f);
		ex = s.x;
		ey = s.y;
		if (axis)
			tv = fmaf(fmul(sign, 2.0f), c.my, tv); // the other component is mad(+-0, rt, t) = t
		else
			tu = fmaf(fmul(sign, 2.0f), c.mx, tu);
	}
	const float len = axis ? search_length(c, ey, ex, sign < 0.0f ? 0.0f : 0.5f) : search_length(c, ex, ey, sign < 0.0f ? 0.0f : 0.5f);
	const float offset = fmaf(-2.007874011993408203125f, len, 3.25f);
	if (axis)
		return fmaf(sign < 0.0f ? c.my : -c.my, offset, tv);
	return fmaf(sign < 0.0f ? c.mx : -c.mx, offset, tu);
}

// SMAAArea (SMAA.hlsl:1091-1103)
GRB_DEV float2 area_ortho(const WCtx &c, float dx, float dy, float e1, float e2, float offset)
{
	float tx = fmaf(16.0f, roundf(fmul(e1, 4.0f)), dx), ty = fmaf(16.0f, roundf(fmul(e2, 4.0f)), dy);
	tx = fmaf(0.0062500000931322574615478515625f, tx, 0.00312500004656612873077392578125f);
	ty = fmaf(0.001785714295692741870880126953125f, ty, 0.0008928571478463709354400634765625f);
	ty = fmaf(0.14285714924335479736328125f, offset, ty);
	const float4 s = sample8(c.area, tx, ty, 0, 0, nullptr);
	return make_float2(s.x, s.y);
}

// SMAADetectHorizontal / VerticalCornerPattern (SMAA.hlsl:1108-1140)
GRB_DEV void corner_pattern(const WCtx &c, float &w0, float &w1, float ax, float ay, float bx, float by, float dx, float dy, bool vertical)
{
	if (!c.P.corner_detection)
		return;
	const float lx = step_f(dx, dy), ly = step_f(dy, dx);
	float rx = fmul(lx, 0.75f), ry = fmul(ly, 0.75f);
	const float sum = fadd(lx, ly);
	rx = fdiv(rx, sum);
	ry = fdiv(ry, sum);
	float fx = 1.0f, fy = 1.0f;
	if (!vertical)
	{
		fx = fsub(fx, fmul(rx, sample8(c.edges, ax, ay, 0, 1, c.f).x));
		fx = fsub(fx, fmul(ry, sample8(c.edges, bx, by, 1, 1, c.f).x));
		fy = fsub(fy, fmul(rx, sample8(c.edges, ax, ay, 0, -2, c.f).x));
		fy = fsub(fy, fmul(ry, sample8(c.edges, bx, by, 1, -2, c.f).x));
	}
	else
	{
		fx = fsub(fx, fmul(rx, sample8(c.edges, ax, ay, 1, 0, c.f).y));
		fx = fsub(fx, fmul(ry, sample8(c.edges, bx, by, 1, 1, c.f).y));
		fy = fsub(fy, fmul(rx, sample8(c.edges, ax, ay, -2, 0, c.f).y));
		fy = fsub(fy, fmul(ry, sample8(c.edges, bx, by, -2, 1, c.f).y));
	}
	w0 = fmul(w0, fclamp(fx, 0.0f, 1.0f));
	w1 = fmul(w1, fclamp(fy, 0.0f, 1.0f));
}

// SMAABlendingWeightCalculationPS (SMAA.hlsl:1145-1247) + SMAABlendingWeightCalculationVS (:655-668), subsampleIndices = 0
__global__ void __launch_bounds__(256) smaa_weights_kernel(Tex8<2> edges, Tex8<2> area, Tex8<1> search, View<uint32_t> weights, SmaaPreset P, int y0, int y1)
{
	const int x = blockIdx.x * 32 + threadIdx.x, y = y0 + blockIdx.y * 8 + threadIdx.y;
	if (x >= edges.w || y >= y1)
		return;
	WCtx c;
	c.edges = edges;
	c.area = area;
	c.search = search;
	c.mx = fdiv(1.0f, (float)edges.w);
	c.my = fdiv(1.0f, (float)edges.h);
	c.mz = (float)edges.w;
	c.mw = (float)edges.h;
	c.P = P;
	const Frag f = { fmul((float)x + 0.5f, c.mx), fmul((float)y + 0.5f, c.my), x, y };
	c.f = &f;
	const float4 e4 = texel8(edges, x, y);
	float ex = e4.x, ey = e4.y;
	if (!(ex > 0.0f) && !(ey > 0.0f))
	{
		weights.at(x, y) = 0u;
		return;
	}
	const float pixx = fmul(f.u, c.mz), pixy = fmul(f.v, c.mw);
	const float o0x = fmaf(c.mx, -0.25f, f.u), o0y = fmaf(c.my, -0.125f, f.v), o0z = fmaf(c.mx, 1.25f, f.u), o0w = fmaf(c.my, -0.125f, f.v);
	const float o1x = fmaf(c.mx, -0.125f, f.u), o1y = fmaf(c.my, -0.25f, f.v), o1z = fmaf(c.mx, -0.125f, f.u), o1w = fmaf(c.my, 1.25f, f.v);
	const float o2x = fmaf(c.mx, fmul(-2.0f, P.max_search_steps), o0x), o2y = fmaf(c.mx, fmul(2.0f, P.max_search_steps), o0z);
	const float o2z = fmaf(c.my, fmul(-2.0f, P.max_search_steps), o1y), o2w = fmaf(c.my, fmul(2.0f, P.max_search_steps), o1w);

	float wx = 0.0f, wy = 0.0f, wz = 0.0f, ww = 0.0f;
	if (ey > 0.0f)
	{
		bool ortho = true;
		if (P.max_search_steps_diag > 0.0f)
		{
			const float2 dw = diag_weights(c, ex);
			wx = dw.x;
			wy = dw.y;
			ortho = wx == -wy;
		}
		if (ortho)
		{
			const float cx = search_axis(c, o0x, o0y, o2x, 0, -1.0f);
			float cy = o1y;
			float d_x = cx;
			const float e1 = sample8(edges, cx, cy, 0, 0, &f).x;
			const float cz = search_axis(c, o0z, o0w, o2y, 0, 1.0f);
			float d_y = cz;
			d_x = fabsf(roundf(fmaf(c.mz, d_x, -pixx)));
			d_y = fabsf(roundf(fmaf(c.mz, d_y, -pixx)));
			const float sx = sqrtf(d_x), sy = sqrtf(d_y);
			const float e2 = sample8(edges, cz, cy, 1, 0, &f).x;
			const float2 a = area_ortho(c, sx, sy, e1, e2, 0.0f);
			wx = a.x;
			wy = a.y;
			cy = f.v;
			corner_pattern(c, wx, wy, cx, cy, cz, cy, d_x, d_y, false);
		}
		else
			ex = 0.0f;
	}
	if (ex > 0.0f)
	{
		const float cy = search_axis(c, o1x, o1y, o2z, 1, -1.0f);
		float cx = o0x;
		float d_x = cy;
		const float e1 = sample8(edges, cx, cy, 0, 0, &f).y;
		const float cz = search_axis(c, o1z, o1w, o2w, 1, 1.0f);
		float d_y = cz;
		d_x = fabsf(roundf(fmaf(c.mw, d_x, -pixy)));
		d_y = fabsf(roundf(fmaf(c.mw, d_y, -pixy)));
		const float sx = sqrtf(d_x), sy = sqrtf(d_y);
		const float e2 = sample8(edges, cx, cz, 0, 1, &f).y;
		const float2 a = area_ortho(c, sx, sy, e1, e2, 0.0f);
		wz = a.x;
		ww = a.y;
		cx = f.u;
		corner_pattern(c, wz, ww, cx, cy, cx, cz, d_x, d_y, true);
	}
	weights.at(x, y) = unorm8(wx) | (unorm8(wy) << 8) | (unorm8(wz) << 16) | (unorm8(ww) << 24);
}

// ------------------------------------------------------------------------------------------------ blend
// inc/srgb.h:4-10 with the literals glslang folds
GRB_DEV float smaa_decode_srgb(float c)
{
	const float small_side = fdiv(c, 12.9200000762939453125f);
	const float pow_side = powf(fdiv(fadd(c, 0.054999999701976776123046875f), 1.05499994754791259765625f), 2.400000095367431640625f);
	return fclamp(c <= 0.0404482372105121612548828125f ? small_side : pow_side, 0.0f, 1.0f);
}

// SMAANeighborhoodBlendingPS (SMAA.hlsl:1252-1307) + SMAANeighborhoodBlendingVS (:673-676)
template <bool SrgbTarget>
__global__ void __launch_bounds__(256) smaa_blend_kernel(Tex8<4> col, Tex8<4> bl, View<uint32_t> out, int y0, int y1)
{
	const int x = blockIdx.x * 32 + threadIdx.x, y = y0 + blockIdx.y * 8 + threadIdx.y;
	if (x >= col.w || y >= y1)
		return;
	const float mx = fdiv(1.0f, (float)col.w), my = fdiv(1.0f, (float)col.h);
	const Frag f = { fmul((float)x + 0.5f, mx), fmul((float)y + 0.5f, my), x, y };
	const float ox = fmaf(mx, 1.0f, f.u), oy = fmaf(my, 0.0f, f.v), oz = fmaf(mx, 0.0f, f.u), ow = fmaf(my, 1.0f, f.v);
	const float ax = sample8(bl, ox, oy, 0, 0, &f).w;
	const float ay = sample8(bl, oz, ow, 0, 0, &f).y;
	const float4 here = texel8(bl, x, y);
	const float aw = here.x, az = here.z;
	float4 color;
	if (fadd(fadd(ax, ay), fadd(az, aw)) < 9.9999997473787516355514526367188e-06f)
		color = texel8(col, x, y);
	else
	{
		const bool hz = fmax_(ax, az) > fmax_(ay, aw);
		float box = 0.0f, boy = ay, boz = 0.0f, bow = aw;
		float bwx = ay, bwy = aw;
		if (hz)
		{
			box = ax;
			boy = 0.0f;
			boz = az;
			bow = 0.0f;
			bwx = ax;
			bwy = az;
		}
		const float sum = fadd(bwx, bwy);
		bwx = fdiv(bwx, sum);
		bwy = fdiv(bwy, sum);
		const float cx = fmaf(box, mx, f.u), cy = fmaf(boy, my, f.v), cz = fmaf(boz, -mx, f.u), cw = fmaf(bow, -my, f.v);
		const float4 c0 = sample8(col, cx, cy, 0, 0, &f), c1 = sample8(col, cz, cw, 0, 0, &f);
		color = make_float4(fmul(c0.x, bwx), fmul(c0.y, bwx), fmul(c0.z, bwx), fmul(c0.w, bwx));
		color.x = fadd(color.x, fmul(c1.x, bwy));
		color.y = fadd(color.y, fmul(c1.y, bwy));
		color.z = fadd(color.z, fmul(c1.z, bwy));
		color.w = fadd(color.w, fmul(c1.w, bwy));
	}
	uint32_t px;
	if (SrgbTarget) // the shader decodes to linear (SMAA_TARGET_SRGB), the sRGB attachment encodes on store
		px = linear_to_srgb8(smaa_decode_srgb(color.x)) | (linear_to_srgb8(smaa_decode_srgb(color.y)) << 8) | (linear_to_srgb8(smaa_decode_srgb(color.z)) << 16);
	else
		px = unorm8(color.x) | (unorm8(color.y) << 8) | (unorm8(color.z) << 16);
	out.at(x, y) = px | (unorm8(color.w) << 24);
}

template <int C>
Tex8<C> tex_of(const GrbImage *im)
{
	Tex8<C> t;
	t.p = static_cast<const uint8_t *>(im->data);
	t.w = im->width;
	t.h = im->height;
	t.pitch = (size_t)im->row_pitch;
	return t;
}

bool rgba8(const GrbImage *im) { return image_ok(im, GRB_FORMAT_R8G8B8A8_UNORM, 4) || image_ok(im, GRB_FORMAT_R8G8B8A8_SRGB, 4); }
bool same_size(const GrbImage *a, const GrbImage *b) { return a->width == b->width && a->height == b->height; }
dim3 smaa_grid(int w, int rows) { return dim3((unsigned)((w + 31) / 32), (unsigned)((rows + 7) / 8), 1); }
} // namespace
} // namespace grb

#ifndef GRB_HOST_EMULATION // tests/cpp/emulate_smaa.cpp compiles the kernels above for the CPU and supplies its own loops
using namespace grb;

extern "C" int32_t grb_smaa_edge_detection(const GrbImage *color, int32_t quality, const GrbImage *edges, GrbRows rows, void *stream)
{
	if (!color || !rgba8(color) || !image_ok(edges, GRB_FORMAT_R8G8_UNORM, 2) || !same_size(color, edges) || quality < 0 || quality > 3)
	{
		set_last_error("grb_smaa_edge_detection: color R8G8B8A8 (read as UNORM), edges R8G8_UNORM of the same size, quality 0..3");
		return GRB_ERR_UNSUPPORTED_FORMAT;
	}
	rows = full_rows(rows, edges->height);
	if (rows.y1 <= rows.y0)
		return GRB_OK;
	smaa_edge_kernel<<<smaa_grid(edges->width, rows.y1 - rows.y0), dim3(32, 8), 0, as_stream(stream)>>>(tex_of<4>(color), view_of<uchar2>(edges), preset_of(quality),
	                                                                                                    rows.y0, rows.y1);
	return check_launch("grb_smaa_edge_detection");
}

extern "C" int32_t grb_smaa_edge_detection_to_peers(const GrbImage *color, int32_t quality, const GrbImage *edges_layout, void *const *peer_images,
                                                    const GrbRows *peer_rows, uint32_t *const *peer_flags, int32_t peer_count, int32_t flag_index,
                                                    uint32_t epoch, uint32_t *scratch_counter, GrbRows rows, void *stream)
{
	if (!color || !edges_layout || !peer_images || !peer_rows || !peer_flags || !scratch_counter || peer_count < 1 || peer_count > GRB_MAX_PEERS ||
	    flag_index < 0 || flag_index >= peer_count)
	{
		set_last_error("grb_smaa_edge_detection_to_peers: bad arguments (edges_layout, peer_images, peer_rows, peer_flags, scratch_counter; "
		               "peer_count 1..GRB_MAX_PEERS, 0 <= flag_index < peer_count)");
		return GRB_ERR_INVALID_ARGUMENT;
	}
	// the layout describes every rank's edge slot; its data pointer is not written (only the peer images are)
	GrbImage layout = *edges_layout;
	if (!layout.data)
		layout.data = peer_images[0];
	if (!rgba8(color) || !image_ok(&layout, GRB_FORMAT_R8G8_UNORM, 2) || !same_size(color, &layout) || quality < 0 || quality > 3)
	{
		set_last_error("grb_smaa_edge_detection_to_peers: color R8G8B8A8 (read as UNORM), edges_layout R8G8_UNORM of the same size, quality 0..3");
		return GRB_ERR_UNSUPPORTED_FORMAT;
	}
	if (rows.y0 < 0 || rows.y1 <= rows.y0 || rows.y1 > color->height)
	{
		set_last_error("grb_smaa_edge_detection_to_peers: rows must be a non-empty range of the image (this rank's band)");
		return GRB_ERR_INVALID_ARGUMENT;
	}
	if (peer_rows[flag_index].y0 != rows.y0 || peer_rows[flag_index].y1 != rows.y1)
	{
		set_last_error("grb_smaa_edge_detection_to_peers: peer_rows[flag_index] must equal rows (this rank's slot receives its whole band)");
		return GRB_ERR_INVALID_ARGUMENT;
	}
	SmaaPeerStore peers{};
	peers.count = peer_count;
	for (int r = 0; r < peer_count; r++)
	{
		if (!peer_images[r] || !peer_flags[r])
		{
			set_last_error("grb_smaa_edge_detection_to_peers: null peer pointer");
			return GRB_ERR_INVALID_ARGUMENT;
		}
		if (peer_rows[r].y0 > peer_rows[r].y1 || peer_rows[r].y0 < rows.y0 || peer_rows[r].y1 > rows.y1)
		{
			set_last_error("grb_smaa_edge_detection_to_peers: every peer_rows[r] must lie inside rows (y0 <= y1; empty: y0 == y1)");
			return GRB_ERR_INVALID_ARGUMENT;
		}
		peers.data[r] = static_cast<uchar2 *>(peer_images[r]);
		peers.flags[r] = peer_flags[r];
		peers.row0[r] = peer_rows[r].y0;
		peers.row1[r] = peer_rows[r].y1;
	}
	peers.pitch_texels = layout.row_pitch / 2;
	peers.flag_index = flag_index;
	peers.epoch = epoch;
	peers.ctas_done = scratch_counter;
	smaa_edge_kernel<SmaaPeerStore><<<smaa_grid(color->width, rows.y1 - rows.y0), dim3(32, 8), 0, as_stream(stream)>>>(tex_of<4>(color), View<uchar2>{}, preset_of(quality),
	                                                                                                                 rows.y0, rows.y1, peers);
	return check_launch("grb_smaa_edge_detection_to_peers");
}

extern "C" int32_t grb_smaa_blend_weights(const GrbImage *edges, const GrbImage *area, const GrbImage *search, int32_t quality, const GrbImage *weights,
                                          GrbRows rows, void *stream)
{
	if (!image_ok(edges, GRB_FORMAT_R8G8_UNORM, 2) || !image_ok(area, GRB_FORMAT_R8G8_UNORM, 2) || !image_ok(search, GRB_FORMAT_R8_UNORM, 1) ||
	    !image_ok(weights, GRB_FORMAT_R8G8B8A8_UNORM, 4) || !same_size(edges, weights) || area->width != 160 || area->height != 560 || search->width != 64 ||
	    search->height != 16 || quality < 0 || quality > 3)
	{
		set_last_error("grb_smaa_blend_weights: edges R8G8_UNORM, area 160x560 R8G8_UNORM, search 64x16 R8_UNORM, weights R8G8B8A8_UNORM of the edges' size, quality 0..3");
		return GRB_ERR_UNSUPPORTED_FORMAT;
	}
	rows = full_rows(rows, weights->height);
	if (rows.y1 <= rows.y0)
		return GRB_OK;
	smaa_weights_kernel<<<smaa_grid(weights->width, rows.y1 - rows.y0), dim3(32, 8), 0, as_stream(stream)>>>(tex_of<2>(edges), tex_of<2>(area), tex_of<1>(search),
	                                                                                                         view_of<uint32_t>(weights), preset_of(quality), rows.y0,
	                                                                                                         rows.y1);
	return check_launch("grb_smaa_blend_weights");
}

extern "C" int32_t grb_smaa_neighborhood_blend(const GrbImage *color, const GrbImage *weights, const GrbImage *out, GrbRows rows, void *stream)
{
	if (!color || !out || !rgba8(color) || !image_ok(weights, GRB_FORMAT_R8G8B8A8_UNORM, 4) || !rgba8(out) || !same_size(color, weights) || !same_size(color, out) ||
	    color->data == out->data)
	{
		set_last_error("grb_smaa_neighborhood_blend: color R8G8B8A8 (read as UNORM), weights R8G8B8A8_UNORM, out R8G8B8A8 (SRGB: decode + encode), one size, out != color");
		return GRB_ERR_UNSUPPORTED_FORMAT;
	}
	rows = full_rows(rows, out->height);
	if (rows.y1 <= rows.y0)
		return GRB_OK;
	const dim3 grid = smaa_grid(out->width, rows.y1 - rows.y0), block(32, 8);
	if (out->format == GRB_FORMAT_R8G8B8A8_SRGB)
		smaa_blend_kernel<true><<<grid, block, 0, as_stream(stream)>>>(tex_of<4>(color), tex_of<4>(weights), view_of<uint32_t>(out), rows.y0, rows.y1);
	else
		smaa_blend_kernel<false><<<grid, block, 0, as_stream(stream)>>>(tex_of<4>(color), tex_of<4>(weights), view_of<uint32_t>(out), rows.y0, rows.y1);
	return check_launch("grb_smaa_neighborhood_blend");
}
#endif // GRB_HOST_EMULATION
