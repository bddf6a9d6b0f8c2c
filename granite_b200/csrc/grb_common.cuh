// grb_common.cuh -- device-side helpers shared by the sm_100a kernels of libgranite_b200.
//
// Storage-format conversions and the LinearClamp sampler, written so that every operation is
// a single IEEE fp32 op in a fixed order (the *_rn intrinsics are never contracted into FMAs,
// whatever -fmad says).  That is what lets the post chain and the cluster indices be compared
// bit-for-bit with the CPU oracle.
#pragma once

#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/granite_b200.h"

namespace grb
{
// ---------------------------------------------------------------------------------------
// error plumbing (host)
// ---------------------------------------------------------------------------------------
void set_last_error(const char *msg);
int32_t check_launch(const char *what);
// mapped host word of the current device for device-side failures (null before grb_init)
uint32_t *device_error_word();
constexpr uint32_t GRB_DEVICE_ERROR_PEER_TIMEOUT = 1u; // word = code << 24 | rank << 16 | (epoch & 0xffff)

static inline cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }

static inline bool image_ok(const GrbImage *im, int32_t format, int texel_bytes)
{
	return im && im->data && im->width > 0 && im->height > 0 && im->format == format &&
	       im->row_pitch >= im->width * texel_bytes && (im->row_pitch % texel_bytes) == 0;
}

static inline GrbRows full_rows(GrbRows r, int height)
{
	if (r.y0 == 0 && r.y1 == 0)
		r.y1 = height;
	if (r.y0 < 0) r.y0 = 0;
	if (r.y1 > height) r.y1 = height;
	return r;
}

// Image view handed to kernels (pitch in texels).
template <typename T>
struct View
{
	T *p;
	int w, h, pitch;
	__device__ __forceinline__ T &at(int x, int y) const { return p[(size_t)y * pitch + x]; }
};

template <typename T>
static inline View<T> view_of(const GrbImage *im)
{
	View<T> v;
	v.p = static_cast<T *>(im->data);
	v.w = im->width;
	v.h = im->height;
	v.pitch = im->row_pitch / (int)sizeof(T);
	return v;
}

// ---------------------------------------------------------------------------------------
// exact fp32 arithmetic helpers
// ---------------------------------------------------------------------------------------
#define GRB_DEV __device__ __forceinline__

GRB_DEV float fmul(float a, float b) { return __fmul_rn(a, b); }
GRB_DEV float fadd(float a, float b) { return __fadd_rn(a, b); }
GRB_DEV float fsub(float a, float b) { return __fsub_rn(a, b); }
GRB_DEV float fdiv(float a, float b) { return __fdiv_rn(a, b); }
GRB_DEV float fmin_(float a, float b) { return a < b ? a : b; }
GRB_DEV float fmax_(float a, float b) { return a > b ? a : b; }
GRB_DEV float fclamp(float x, float lo, float hi) { return fmin_(fmax_(x, lo), hi); }
// GLSL mix(a, b, t) = a*(1-t) + b*t
GRB_DEV float fmix(float a, float b, float t) { return fadd(fmul(a, fsub(1.0f, t)), fmul(b, t)); }
GRB_DEV int iclamp(int x, int lo, int hi) { return min(max(x, lo), hi); }

// ---------------------------------------------------------------------------------------
// storage formats
// ---------------------------------------------------------------------------------------
// Unsigned small floats of B10G11R11_UFLOAT_PACK32 (5-bit exponent, MBITS mantissa):
// negative -> 0, NaN -> NaN, +inf -> inf, finite values truncate toward zero and saturate
// at the largest finite value.
template <int MBITS>
GRB_DEV uint32_t f32_to_ufloat(float f)
{
	uint32_t x = __float_as_uint(f);
	const uint32_t max_finite = (30u << MBITS) | ((1u << MBITS) - 1u);
	if ((x & 0x7fffffffu) > 0x7f800000u)
		return (31u << MBITS) | 1u;
	if (x & 0x80000000u)
		return 0u;
	if (x == 0x7f800000u)
		return 31u << MBITS;
	int e = (int)(x >> 23) - 127;
	uint32_t m = (x & 0x7fffffu) | 0x800000u;
	if (e > 15)
		return max_finite;
	if (e >= -14)
		return ((uint32_t)(e + 15) << MBITS) | ((m >> (23 - MBITS)) & ((1u << MBITS) - 1u));
	int shift = (23 - MBITS) + (-14 - e);
	return shift > 24 ? 0u : (m >> shift);
}

template <int MBITS>
GRB_DEV float ufloat_to_f32(uint32_t v)
{
	uint32_t e = v >> MBITS;
	uint32_t m = v & ((1u << MBITS) - 1u);
	if (e == 0u)
		return (float)m * (MBITS == 6 ? 9.5367431640625e-7f : 1.9073486328125e-6f); // exact: m < 64, power-of-two scale
	if (e == 31u)
		return __uint_as_float(0x7f800000u | (m << (23 - MBITS)));
	return __uint_as_float(((e + 112u) << 23) | (m << (23 - MBITS)));
}

// The 11/10-bit unsigned floats are binary16 with the sign and the low 4/5 mantissa bits cut off
// (same 5-bit exponent, bias 15, same denormal rule), so the hardware fp16 converters do all of
// the work: decode = shift the code into a half and widen (exact, denormals/inf/NaN included);
// encode = clamp negatives, convert round-toward-zero (never rounds up to inf) and drop the low
// bits (truncation composes).  Bit-identical to f32_to_ufloat / ufloat_to_f32 above, which stay
// as the readable definition.
GRB_DEV uint32_t pack_r11g11b10(float r, float g, float b)
{
	// fmaxf(NaN, 0) is 0 in CUDA; keep NaN a NaN like the reference conversion
	uint32_t hr = __half_as_ushort(__float2half_rz(r != r ? r : fmaxf(r, 0.0f)));
	uint32_t hg = __half_as_ushort(__float2half_rz(g != g ? g : fmaxf(g, 0.0f)));
	uint32_t hb = __half_as_ushort(__float2half_rz(b != b ? b : fmaxf(b, 0.0f)));
	return ((hr & 0x7fffu) >> 4) | (((hg & 0x7fffu) >> 4) << 11) | (((hb & 0x7fffu) >> 5) << 22);
}

GRB_DEV float3 unpack_r11g11b10(uint32_t p)
{
	return make_float3(__half2float(__ushort_as_half((unsigned short)((p & 0x7ffu) << 4))),
	                   __half2float(__ushort_as_half((unsigned short)(((p >> 11) & 0x7ffu) << 4))),
	                   __half2float(__ushort_as_half((unsigned short)((p >> 22) << 5))));
}

GRB_DEV float h2f(uint16_t h) { return __half2float(__ushort_as_half(h)); }
GRB_DEV uint16_t f2h(float f) { return __half_as_ushort(__float2half_rn(f)); }

// RGBA16F texel <-> float4 (8-byte accesses)
GRB_DEV float4 unpack_rgba16f(uint2 t)
{
	return make_float4(h2f((uint16_t)(t.x & 0xffffu)), h2f((uint16_t)(t.x >> 16)), h2f((uint16_t)(t.y & 0xffffu)), h2f((uint16_t)(t.y >> 16)));
}

GRB_DEV uint2 pack_rgba16f(float4 v)
{
	uint2 t;
	t.x = (uint32_t)f2h(v.x) | ((uint32_t)f2h(v.y) << 16);
	t.y = (uint32_t)f2h(v.z) | ((uint32_t)f2h(v.w) << 16);
	return t;
}

// Store to an R8G8B8A8_SRGB attachment: clamp, exact OETF, round half up.
GRB_DEV uint32_t linear_to_srgb8(float c)
{
	if (!(c > 0.0f)) c = 0.0f;
	if (c > 1.0f) c = 1.0f;
	float s = c <= 0.0031308f ? fmul(c, 12.92f) : fsub(fmul(1.055f, powf(c, 1.0f / 2.4f)), 0.055f);
	int q = (int)floorf(fadd(fmul(s, 255.0f), 0.5f));
	return (uint32_t)iclamp(q, 0, 255);
}

GRB_DEV uint32_t float_to_unorm8(float c)
{
	if (!(c > 0.0f)) c = 0.0f;
	if (c > 1.0f) c = 1.0f;
	return (uint32_t)floorf(fadd(fmul(c, 255.0f), 0.5f));
}

// Raw MUFU ops.  rsqrtf() / __fdividef() / __log2f() / __exp2f() without -ftz wrap the MUFU in a
// denormal rescue (compare, select and rescale on the way in and out) that costs more issue slots
// than the operation itself.  Used only where the contract is "within 1 ULP of the stored
// format" and a denormal argument can only mean a value the surrounding clamps absorb.
__device__ __forceinline__ float rsqrt_fast(float x)
{
	float y;
	asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
	return y;
}
__device__ __forceinline__ float rcp_fast(float x)
{
	float y;
	asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
	return y;
}
__device__ __forceinline__ float lg2_fast(float x)
{
	float y;
	asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
	return y;
}
__device__ __forceinline__ float ex2_fast(float x)
{
	float y;
	asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
	return y;
}

// ---------------------------------------------------------------------------------------
// StockSampler::LinearClamp (vulkan/device.cpp:1077-1170): bilinear, clamp-to-edge, texel
// centres at +0.5, exact fp32 weights.  (u, v) are the normalised coordinates the shader
// would have produced.
// ---------------------------------------------------------------------------------------
struct Bilin
{
	int x0, x1, y0, y1;
	float a, b;
};

GRB_DEV Bilin bilin_setup(float u, float v, int w, int h)
{
	Bilin s;
	float fx = fsub(fmul(u, (float)w), 0.5f);
	float fy = fsub(fmul(v, (float)h), 0.5f);
	float flx = floorf(fx), fly = floorf(fy);
	s.a = fsub(fx, flx);
	s.b = fsub(fy, fly);
	flx = fclamp(flx, -2.0f, (float)w + 1.0f);
	fly = fclamp(fly, -2.0f, (float)h + 1.0f);
	if (!(flx == flx)) flx = 0.0f;
	if (!(fly == fly)) fly = 0.0f;
	int x0 = (int)flx, y0 = (int)fly;
	s.x0 = iclamp(x0, 0, w - 1);
	s.x1 = iclamp(x0 + 1, 0, w - 1);
	s.y0 = iclamp(y0, 0, h - 1);
	s.y1 = iclamp(y0 + 1, 0, h - 1);
	return s;
}

GRB_DEV float bilin_mix(float t00, float t10, float t01, float t11, float a, float b)
{
	float ia = fsub(1.0f, a), ib = fsub(1.0f, b);
	float top = fadd(fmul(t00, ia), fmul(t10, a));
	float bot = fadd(fmul(t01, ia), fmul(t11, a));
	return fadd(fmul(top, ib), fmul(bot, b));
}

GRB_DEV float4 bilin_mix4(float4 t00, float4 t10, float4 t01, float4 t11, float a, float b)
{
	return make_float4(bilin_mix(t00.x, t10.x, t01.x, t11.x, a, b), bilin_mix(t00.y, t10.y, t01.y, t11.y, a, b),
	                   bilin_mix(t00.z, t10.z, t01.z, t11.z, a, b), bilin_mix(t00.w, t10.w, t01.w, t11.w, a, b));
}

GRB_DEV float4 sample_rgba16f(const View<const uint2> &im, float u, float v)
{
	Bilin s = bilin_setup(u, v, im.w, im.h);
	float4 t00 = unpack_rgba16f(__ldg(&im.at(s.x0, s.y0)));
	float4 t10 = unpack_rgba16f(__ldg(&im.at(s.x1, s.y0)));
	float4 t01 = unpack_rgba16f(__ldg(&im.at(s.x0, s.y1)));
	float4 t11 = unpack_rgba16f(__ldg(&im.at(s.x1, s.y1)));
	return bilin_mix4(t00, t10, t01, t11, s.a, s.b);
}

// Bilinear weight within 2^-9 of 0 or 1 -> exactly 0 or 1: the TAA history taps only (oracle_math.h
// snap_weight; a sampler's fixed-point position has 8 fractional bits).
GRB_DEV float snap_weight(float f) { return f <= 0.001953125f ? 0.0f : (f >= 1.0f - 0.001953125f ? 1.0f : f); }

GRB_DEV float4 sample_rgba16f_snap(const View<const uint2> &im, float u, float v)
{
	Bilin s = bilin_setup(u, v, im.w, im.h);
	s.a = snap_weight(s.a);
	s.b = snap_weight(s.b);
	float4 t00 = unpack_rgba16f(__ldg(&im.at(s.x0, s.y0)));
	float4 t10 = unpack_rgba16f(__ldg(&im.at(s.x1, s.y0)));
	float4 t01 = unpack_rgba16f(__ldg(&im.at(s.x0, s.y1)));
	float4 t11 = unpack_rgba16f(__ldg(&im.at(s.x1, s.y1)));
	return bilin_mix4(t00, t10, t01, t11, s.a, s.b);
}

GRB_DEV float3 fetch_hdr_clamped(const View<const uint32_t> &im, int x, int y)
{
	return unpack_r11g11b10(__ldg(&im.at(iclamp(x, 0, im.w - 1), iclamp(y, 0, im.h - 1))));
}

// The HDR image in its other storage format, R16G16B16A16_SFLOAT ("renderTargetFp16", scene_viewer_application.cpp:
// 880-884): the kernels that read HDR-main are templated on the texel type and decode through these overloads.
GRB_DEV float3 hdr_texel(const View<const uint32_t> &im, int x, int y) { return unpack_r11g11b10(__ldg(&im.at(x, y))); }
GRB_DEV float3 hdr_texel(const View<const uint2> &im, int x, int y)
{
	const float4 t = unpack_rgba16f(__ldg(&im.at(x, y)));
	return make_float3(t.x, t.y, t.z);
}
GRB_DEV float3 fetch_hdr_clamped(const View<const uint2> &im, int x, int y)
{
	return hdr_texel(im, iclamp(x, 0, im.w - 1), iclamp(y, 0, im.h - 1));
}

#ifndef GRB_HOST_EMULATION
// ---- the producing side of the peer exchanges of a row-sharded frame (bloom d0, TAA history, SMAA edges)
GRB_DEV void store_release_system(uint32_t *p, uint32_t v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }

// Called by every thread of every CTA after its peer stores: each thread's stores are ordered before its CTA's
// arrival, and the last CTA to arrive resets the counter and release-stores flags[r][flag_index] = epoch on every rank r
// (threadFenceReduction pattern at system scope).  The consumer side is grb_peer_wait.
GRB_DEV void publish_to_peers(uint32_t *const *flags, int count, int flag_index, uint32_t epoch, unsigned *ctas_done)
{
	__threadfence_system();
	__syncthreads();
	if (threadIdx.x == 0 && threadIdx.y == 0)
	{
		const unsigned total = gridDim.x * gridDim.y;
		if (atomicAdd(ctas_done, 1u) == total - 1u)
		{
			*ctas_done = 0u;
			__threadfence_system();
			for (int r = 0; r < count; r++)
				store_release_system(flags[r] + flag_index, epoch);
		}
	}
}
#endif

} // namespace grb
