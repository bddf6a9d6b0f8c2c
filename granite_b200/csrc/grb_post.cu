// grb_post.cu -- HDR post chain (bloom threshold / pyramid / luminance / tonemap) and post-AA
// (FXAA, TAA resolve) as sm_100a kernels.  Compiled with -fmad=false: every multiply/add is a
// separate IEEE op in source order, so results are comparable bit-for-bit with the CPU oracle
// except where a transcendental (log2f, exp2f, powf) is involved.
//
// What each kernel replaces in the reference is cited at its entry point.  None of these is a
// translation of the GLSL: a pass here is one CUDA grid over OUTPUT texels (optionally only the
// rows of one screen-row shard), reading packed texels straight from HBM/L2 with 4/8-byte
// coalesced accesses; the small pyramid levels live entirely in the 126 MB L2.
#include "grb_common.cuh"

#include <cooperative_groups.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <type_traits>

namespace grb
{
namespace
{
constexpr int kBlockX = 32;
constexpr int kBlockY = 8;

inline dim3 grid_for(int w, int rows) { return dim3((w + kBlockX - 1) / kBlockX, (rows + kBlockY - 1) / kBlockY, 1); }

// ------------------------------------------------------------------------------- K7
// bloom_threshold: out(x,y) = f(bilinear HDR at the output texel centre).
template <bool DynamicExposure, typename HdrTexel = uint32_t>
__global__ void __launch_bounds__(kBlockX *kBlockY) bloom_threshold_kernel(View<const HdrTexel> hdr, const float *__restrict__ lum,
                                                                          View<uint2> out, int y0, int y1, float inv_w, float inv_h)
{
	int x = blockIdx.x * kBlockX + threadIdx.x;
	int y = y0 + blockIdx.y * kBlockY + threadIdx.y;
	if (x >= out.w || y >= y1)
		return;
	float u = ((float)x + 0.5f) * inv_w;
	float v = ((float)y + 0.5f) * inv_h;
	Bilin s = bilin_setup(u, v, hdr.w, hdr.h);
	float3 t00 = hdr_texel(hdr, s.x0, s.y0);
	float3 t10 = hdr_texel(hdr, s.x1, s.y0);
	float3 t01 = hdr_texel(hdr, s.x0, s.y1);
	float3 t11 = hdr_texel(hdr, s.x1, s.y1);
	float3 c = make_float3(bilin_mix(t00.x, t10.x, t01.x, t11.x, s.a, s.b), bilin_mix(t00.y, t10.y, t01.y, t11.y, s.a, s.b),
	                       bilin_mix(t00.z, t10.z, t01.z, t11.z, s.a, s.b));
	float luminance = fmax_(fmax_(c.x, c.y), c.z) + 0.0001f;
	float loglum = log2f(luminance);
	c.x = c.x / luminance;
	c.y = c.y / luminance;
	c.z = c.z / luminance;
	if (DynamicExposure)
		luminance -= 8.0f * __ldg(&lum[1]);
	else
		luminance -= 8.0f;
	out.at(x, y) = pack_rgba16f(make_float4(fmax_(c.x * luminance, 0.0f), fmax_(c.y * luminance, 0.0f), fmax_(c.z * luminance, 0.0f), loglum));
}

// ------------------------------------------------------------------------------- K8 / K9
// 9-tap tent over a LinearClamp source; tap order and weights are the contract (fp32 sums are
// order-sensitive): centre 1/4, then (-,+) (0,+) (+,+) (-,0) (+,0) (-,-) (0,-) (+,-).
__device__ __forceinline__ float4 tent9(const View<const uint2> &src, float u, float v, float off, float inv_in_w, float inv_in_h)
{
	const float du = off * inv_in_w, dv = off * inv_in_h;
	const float um = u + (-du), up = u + du;
	const float vm = v + (-dv), vp = v + dv;
	float4 s = sample_rgba16f(src, u, v);
	float4 acc = make_float4(0.25f * s.x, 0.25f * s.y, 0.25f * s.z, 0.25f * s.w);
#define GRB_TAP(W, U, V)                     \
	s = sample_rgba16f(src, (U), (V));       \
	acc.x += (W)*s.x;                        \
	acc.y += (W)*s.y;                        \
	acc.z += (W)*s.z;                        \
	acc.w += (W)*s.w;
	GRB_TAP(0.0625f, um, vp)
	GRB_TAP(0.125f, u, vp)
	GRB_TAP(0.0625f, up, vp)
	GRB_TAP(0.125f, um, v)
	GRB_TAP(0.125f, up, v)
	GRB_TAP(0.0625f, um, vm)
	GRB_TAP(0.125f, u, vm)
	GRB_TAP(0.0625f, up, vm)
#undef GRB_TAP
	return acc;
}

template <bool Feedback>
__global__ void __launch_bounds__(kBlockX *kBlockY) bloom_downsample_kernel(View<const uint2> src, View<const uint2> history, float lerp,
                                                                           View<uint2> out, int y0, int y1, float inv_w, float inv_h,
                                                                           float inv_in_w, float inv_in_h)
{
	int x = blockIdx.x * kBlockX + threadIdx.x;
	int y = y0 + blockIdx.y * kBlockY + threadIdx.y;
	if (x >= out.w || y >= y1)
		return;
	float u = ((float)x + 0.5f) * inv_w;
	float v = ((float)y + 0.5f) * inv_h;
	float4 value = tent9(src, u, v, 1.75f, inv_in_w, inv_in_h);
	if (Feedback)
	{
		float4 hs = unpack_rgba16f(__ldg(&history.at(x, y)));
		value = make_float4(fmix(hs.x, value.x, lerp), fmix(hs.y, value.y, lerp), fmix(hs.z, value.z, lerp), fmix(hs.w, value.w, 1.0f));
	}
	out.at(x, y) = pack_rgba16f(value);
}

__global__ void __launch_bounds__(kBlockX *kBlockY) bloom_upsample_kernel(View<const uint2> src, View<uint2> out, int y0, int y1, float inv_w,
                                                                         float inv_h, float inv_in_w, float inv_in_h)
{
	int x = blockIdx.x * kBlockX + threadIdx.x;
	int y = y0 + blockIdx.y * kBlockY + threadIdx.y;
	if (x >= out.w || y >= y1)
		return;
	float u = ((float)x + 0.5f) * inv_w;
	float v = ((float)y + 0.5f) * inv_h;
	out.at(x, y) = pack_rgba16f(tent9(src, u, v, 0.875f, inv_in_w, inv_in_h));
}


// ------------------------------------------------------------------------------- K8 + all-gather
// Row-sharded frames: the first downsample (1/2 -> 1/4 resolution) of a rank's band is needed in
// full by every rank for the pyramid tail.  Instead of producing the band locally and handing it
// to a collective afterwards, the kernel stores each texel straight into the 1/4-resolution image
// of every rank (its own and the peers' over NVLink / NVSwitch, plain 8-byte stores to mapped
// peer memory) and then publishes "band of frame <epoch> landed" in every rank's flag array.
// The consumer side is peer_wait_kernel below.  Texel values are those of
// bloom_downsample_kernel<false>.
struct PeerTargets
{
	uint2 *data[GRB_MAX_PEERS];
	uint32_t *flags[GRB_MAX_PEERS];
	int count;
};

__device__ __forceinline__ uint32_t load_acquire_system(const uint32_t *p)
{
	uint32_t v;
	asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
	return v;
}

__global__ void __launch_bounds__(kBlockX *kBlockY) bloom_downsample_peers_kernel(View<const uint2> src, PeerTargets targets, int out_w, int out_pitch_texels,
                                                                                 int y0, int y1, float inv_w, float inv_h, float inv_in_w, float inv_in_h,
                                                                                 int flag_index, uint32_t epoch, unsigned *ctas_done)
{
	const int x = blockIdx.x * kBlockX + threadIdx.x;
	const int y = y0 + blockIdx.y * kBlockY + threadIdx.y;
	if (x < out_w && y < y1)
	{
		const float u = ((float)x + 0.5f) * inv_w;
		const float v = ((float)y + 0.5f) * inv_h;
		const uint2 texel = pack_rgba16f(tent9(src, u, v, 1.75f, inv_in_w, inv_in_h));
		const size_t at = (size_t)y * out_pitch_texels + x;
		for (int r = 0; r < targets.count; r++)
			targets.data[r][at] = texel;
	}
	// publish: the last CTA to arrive raises this rank's flag on every peer
	publish_to_peers(targets.flags, targets.count, flag_index, epoch, ctas_done);
}

// One thread per producing rank spins until that rank's band of frame `epoch` has landed here.
__global__ void peer_wait_kernel(const uint32_t *flags, int count, uint32_t epoch, uint32_t *error_word, unsigned max_spins)
{
	if ((int)threadIdx.x < count)
	{
		// bounded (~4 s): a rank that died must not hang the GPUs of the others
		for (unsigned spins = 0; (int32_t)(load_acquire_system(flags + threadIdx.x) - epoch) < 0; spins++)
		{
			if (spins > max_spins)
			{
				printf("granite_b200: timed out waiting for rank %d's band of frame %u\n", (int)threadIdx.x, epoch);
				if (error_word) // picked up by the next grb_* call on this device (check_launch)
				{
					*reinterpret_cast<volatile uint32_t *>(error_word) = (GRB_DEVICE_ERROR_PEER_TIMEOUT << 24) | ((uint32_t)threadIdx.x << 16) | (epoch & 0xffffu);
					__threadfence_system();
				}
				break;
			}
			__nanosleep(128);
		}
	}
}

// ------------------------------------------------------------------------------- K10
// Average log-luminance.  The reference sums with one 8x8 workgroup: each invocation adds its
// strided samples in (y-iter, x-iter) order, then a shared-memory tree 32,16,8,4,2 and a final
// s[0]+s[1].  fp32 addition is not associative, so the same association is kept here: the
// strided partials are per-thread, and the tree is five xor-free shuffle-down steps over two
// warps' worth of values held in shared memory.
__device__ __forceinline__ float luminance_sample(const View<const uint2> &d3, int sx, int sy, float inv_sx, float inv_sy)
{
	return sample_rgba16f(d3, ((float)sx + 0.5f) * inv_sx, ((float)sy + 0.5f) * inv_sy).w;
}

__device__ __forceinline__ void luminance_tail(float *s, int tid, int size_x, int size_y, float inv_sx, float inv_sy, float *lum, float lerp,
                                              float lo, float hi)
{
	// s[0..63] holds the 64 strided partials (index = ly * 8 + lx).
	__syncthreads();
	if (tid < 32)
	{
		float a = s[tid] + s[tid + 32];                     // STEP(32)
		a = a + __shfl_down_sync(0xffffffffu, a, 16);       // STEP(16): lanes 0..15 valid
		a = a + __shfl_down_sync(0xffffffffu, a, 8);        // STEP(8)
		a = a + __shfl_down_sync(0xffffffffu, a, 4);        // STEP(4)
		a = a + __shfl_down_sync(0xffffffffu, a, 2);        // STEP(2): lanes 0,1 valid
		float b = __shfl_down_sync(0xffffffffu, a, 1);
		if (tid == 0)
		{
			float loglum = a + b;
			loglum *= inv_sx * inv_sy;
			loglum = fclamp(loglum, lo, hi);
			float new_log = fmix(lum[0], loglum, lerp);
			lum[0] = new_log;
			lum[1] = exp2f(new_log);
			lum[2] = exp2f(-new_log);
		}
	}
	(void)size_x;
	(void)size_y;
}

__global__ void __launch_bounds__(64) luminance_kernel(View<const uint2> d3, float *lum, float lerp, float lo, float hi)
{
	__shared__ float s[64];
	const int size_x = d3.w / 2, size_y = d3.h / 2;
	const int iter_y = (size_y + 7) >> 3, iter_x = (size_x + 7) >> 3;
	const float inv_sx = 1.0f / (float)size_x, inv_sy = 1.0f / (float)size_y;
	const int lx = threadIdx.x & 7, ly = threadIdx.x >> 3;
	float total = 0.0f;
	for (int y = 0; y < iter_y; y++)
		for (int x = 0; x < iter_x; x++)
		{
			int sx = x * 8 + lx, sy = y * 8 + ly;
			if (sx < size_x && sy < size_y)
				total += luminance_sample(d3, sx, sy, inv_sx, inv_sy);
		}
	s[threadIdx.x] = total;
	luminance_tail(s, threadIdx.x, size_x, size_y, inv_sx, inv_sy, lum, lerp, lo, hi);
}

// Same function, restructured for latency: the reference's single 64-thread group is a serial
// chain of ~32 dependent texture fetches per thread.  Here 256 threads first sample the whole
// (w/2 x h/2) grid into shared memory (independent loads, one barrier), then 64 of them add their
// strided samples in the reference's (y-iter, x-iter) order and run the same tree -- identical
// association, so identical bits.
constexpr int kLumFastThreads = 256;
constexpr int kLumFastMaxSamples = 8192; // 32 KiB of shared memory

__global__ void __launch_bounds__(kLumFastThreads) luminance_fast_kernel(View<const uint2> d3, float *lum, float lerp, float lo, float hi)
{
	__shared__ float grid[kLumFastMaxSamples];
	__shared__ float s[64];
	const int size_x = d3.w / 2, size_y = d3.h / 2;
	const float inv_sx = 1.0f / (float)size_x, inv_sy = 1.0f / (float)size_y;
	for (int i = threadIdx.x; i < size_x * size_y; i += kLumFastThreads)
	{
		int sy = i / size_x, sx = i - sy * size_x;
		grid[i] = luminance_sample(d3, sx, sy, inv_sx, inv_sy);
	}
	__syncthreads();
	if (threadIdx.x < 64)
	{
		const int iter_y = (size_y + 7) >> 3, iter_x = (size_x + 7) >> 3;
		const int lx = threadIdx.x & 7, ly = threadIdx.x >> 3;
		float total = 0.0f;
		for (int y = 0; y < iter_y; y++)
			for (int x = 0; x < iter_x; x++)
			{
				int sx = x * 8 + lx, sy = y * 8 + ly;
				if (sx < size_x && sy < size_y)
					total += grid[sy * size_x + sx];
			}
		s[threadIdx.x] = total;
	}
	luminance_tail(s, threadIdx.x, size_x, size_y, inv_sx, inv_sy, lum, lerp, lo, hi);
}

// Sharded form, step 1: every thread samples one grid texel of the rows this rank owns.
__global__ void __launch_bounds__(kBlockX *kBlockY) luminance_grid_kernel(View<const uint2> d3, float *grid, int y0, int y1)
{
	const int size_x = d3.w / 2, size_y = d3.h / 2;
	int x = blockIdx.x * kBlockX + threadIdx.x;
	int y = y0 + blockIdx.y * kBlockY + threadIdx.y;
	if (x >= size_x || y >= y1 || y >= size_y)
		return;
	grid[y * size_x + x] = luminance_sample(d3, x, y, 1.0f / (float)size_x, 1.0f / (float)size_y);
}

// step 2: identical association order to luminance_kernel, reading the assembled grid.
__global__ void __launch_bounds__(64) luminance_finalize_kernel(const float *__restrict__ grid, int size_x, int size_y, float *lum, float lerp,
                                                               float lo, float hi)
{
	__shared__ float s[64];
	const int iter_y = (size_y + 7) >> 3, iter_x = (size_x + 7) >> 3;
	const int lx = threadIdx.x & 7, ly = threadIdx.x >> 3;
	float total = 0.0f;
	for (int y = 0; y < iter_y; y++)
		for (int x = 0; x < iter_x; x++)
		{
			int sx = x * 8 + lx, sy = y * 8 + ly;
			if (sx < size_x && sy < size_y)
				total += grid[sy * size_x + sx];
		}
	s[threadIdx.x] = total;
	luminance_tail(s, threadIdx.x, size_x, size_y, 1.0f / (float)size_x, 1.0f / (float)size_y, lum, lerp, lo, hi);
}

// ------------------------------------------------------------------------------- K11
__device__ __forceinline__ float uncharted2(float x)
{
	// glslang folds C*B, D*E, D*F and E/F in double precision from the literals and rounds once:
	// D*F = (float)0.06 = 0x3d75c28f (0.2f * 0.3f would be 0x3d75c290), E/F = (float)(0.02 / 0.30).
	const float A = 0.15f, B = 0.50f, CB = (float)(0.10 * 0.50), DE = (float)(0.20 * 0.02), DF = (float)(0.20 * 0.30), EF = (float)(0.02 / 0.30);
	return ((x * (A * x + CB) + DE) / (x * (A * x + B) + DF)) - EF;
}

template <bool DynamicExposure, bool SrgbTarget, typename HdrTexel = uint32_t>
__global__ void __launch_bounds__(kBlockX *kBlockY) tonemap_kernel(View<const HdrTexel> hdr, View<const uint2> bloom, const float *__restrict__ lum,
                                                                  float exposure, View<uint32_t> out, int y0, int y1, float inv_w, float inv_h)
{
	int x = blockIdx.x * kBlockX + threadIdx.x;
	int y = y0 + blockIdx.y * kBlockY + threadIdx.y;
	if (x >= out.w || y >= y1)
		return;
	float3 c = hdr_texel(hdr, x, y);
	float u = ((float)x + 0.5f) * inv_w;
	float v = ((float)y + 0.5f) * inv_h;
	float4 b = sample_rgba16f(bloom, u, v);
	const float white_scale = 1.0f / uncharted2(11.2f);
	const float k = DynamicExposure ? (__ldg(&lum[2]) * exposure) : exposure;
	float r = uncharted2((c.x + b.x) * k) * white_scale;
	float g = uncharted2((c.y + b.y) * k) * white_scale;
	float bl = uncharted2((c.z + b.z) * k) * white_scale;
	uint32_t px;
	if (SrgbTarget)
		px = linear_to_srgb8(r) | (linear_to_srgb8(g) << 8) | (linear_to_srgb8(bl) << 16) | 0xff000000u;
	else
		px = float_to_unorm8(r) | (float_to_unorm8(g) << 8) | (float_to_unorm8(bl) << 16) | 0xff000000u;
	out.at(x, y) = px;
}

// Vectorised tonemap: one thread produces 4 horizontally adjacent pixels (16-byte HDR load,
// 16-byte store) and shares the bloom taps between them -- at an exact 1/4-resolution bloom image
// the four pixels' bilinear footprints cover only 3 columns x 2 rows.  Weights are computed per
// pixel with the same exact fp32 expressions as the generic kernel; the tone curve and the sRGB
// OETF use the fast reciprocal / lg2 / ex2 units (error ~1e-4 LSB, the bar is 1 LSB), because
// with the accurate powf this streaming pass was issue-bound at 8 % of the HBM roofline.
// (uncharted2(x)) * white_scale with the constant term folded into one FMA
__device__ __forceinline__ float uncharted2_fast_scaled(float x, float white_scale)
{
	const float A = 0.15f, B = 0.50f, CB = (float)(0.10 * 0.50), DE = (float)(0.20 * 0.02), DF = (float)(0.20 * 0.30), EF = (float)(0.02 / 0.30);
	const float q = fmaf(x, fmaf(A, x, CB), DE) * rcp_fast(fmaf(x, fmaf(A, x, B), DF));
	return fmaf(q, white_scale, -EF * white_scale);
}

__device__ __forceinline__ uint32_t srgb8_fast(float c)
{
	c = __saturatef(c); // also NaN -> 0
	float s = c <= 0.0031308f ? c * (12.92f * 255.0f) : fmaf(ex2_fast(lg2_fast(c) * (1.0f / 2.4f)), 1.055f * 255.0f, -0.055f * 255.0f);
	return (uint32_t)min(__float2int_rd(s + 0.5f), 255);
}

__device__ __forceinline__ uint32_t unorm8_fast(float c)
{
	return (uint32_t)__float2int_rd(fmaf(__saturatef(c), 255.0f, 0.5f));
}

template <bool DynamicExposure, bool SrgbTarget>
__global__ void __launch_bounds__(kBlockX *kBlockY) tonemap4_kernel(View<const uint32_t> hdr, View<const uint2> bloom, const float *__restrict__ lum,
                                                                   float exposure, View<uint32_t> out, int y0, int y1, float inv_w, float inv_h)
{
	const int x4 = (blockIdx.x * kBlockX + threadIdx.x) * 4;
	const int y = y0 + blockIdx.y * kBlockY + threadIdx.y;
	if (x4 >= out.w || y >= y1)
		return;
	const uint4 h4 = __ldg(reinterpret_cast<const uint4 *>(&hdr.at(x4, y)));
	const uint32_t hp[4] = { h4.x, h4.y, h4.z, h4.w };

	// bloom rows (shared by the 4 pixels)
	const float v = ((float)y + 0.5f) * inv_h;
	const float fy = fsub(fmul(v, (float)bloom.h), 0.5f);
	const float fly = floorf(fy);
	const float wb = fsub(fy, fly);
	const int by = (int)fly;
	const int r0 = iclamp(by, 0, bloom.h - 1), r1 = iclamp(by + 1, 0, bloom.h - 1);
	// bloom columns k-1, k, k+1 with k = x4 / 4
	const int k = x4 >> 2;
	const int c0 = iclamp(k - 1, 0, bloom.w - 1), c1 = iclamp(k, 0, bloom.w - 1), c2 = iclamp(k + 1, 0, bloom.w - 1);
	float3 top[3], bot[3];
	{
		const int cols[3] = { c0, c1, c2 };
#pragma unroll
		for (int i = 0; i < 3; i++)
		{
			float4 a = unpack_rgba16f(__ldg(&bloom.at(cols[i], r0)));
			float4 b = unpack_rgba16f(__ldg(&bloom.at(cols[i], r1)));
			top[i] = make_float3(a.x, a.y, a.z);
			bot[i] = make_float3(b.x, b.y, b.z);
		}
	}
	const float white_scale = 1.0f / uncharted2(11.2f);
	const float kexp = DynamicExposure ? (__ldg(&lum[2]) * exposure) : exposure;
	uint32_t px[4];
#pragma unroll
	for (int j = 0; j < 4; j++)
	{
		// horizontal weight with the generic sampler's exact arithmetic; its floor is k-1 for
		// j < 2 and k for j >= 2 (ideal fractions .625 .875 .125 .375, never near an integer)
		const float u = ((float)(x4 + j) + 0.5f) * inv_w;
		const float fx = fsub(fmul(u, (float)bloom.w), 0.5f);
		const float wa = fsub(fx, floorf(fx));
		const int i0 = j < 2 ? 0 : 1;
		const float3 t00 = top[i0], t10 = top[i0 + 1], t01 = bot[i0], t11 = bot[i0 + 1];
		const float bx = bilin_mix(t00.x, t10.x, t01.x, t11.x, wa, wb);
		const float bgr = bilin_mix(t00.y, t10.y, t01.y, t11.y, wa, wb);
		const float bb = bilin_mix(t00.z, t10.z, t01.z, t11.z, wa, wb);
		const float3 c = unpack_r11g11b10(hp[j]);
		const float r = uncharted2_fast_scaled(fmul(fadd(c.x, bx), kexp), white_scale);
		const float g = uncharted2_fast_scaled(fmul(fadd(c.y, bgr), kexp), white_scale);
		const float b = uncharted2_fast_scaled(fmul(fadd(c.z, bb), kexp), white_scale);
		px[j] = SrgbTarget ? (srgb8_fast(r) | (srgb8_fast(g) << 8) | (srgb8_fast(b) << 16) | 0xff000000u)
		                   : (unorm8_fast(r) | (unorm8_fast(g) << 8) | (unorm8_fast(b) << 16) | 0xff000000u);
	}
	*reinterpret_cast<uint4 *>(&out.at(x4, y)) = make_uint4(px[0], px[1], px[2], px[3]);
}

// ------------------------------------------------------------------------------- K12
__device__ __forceinline__ float3 fxaa_unpack(const float *lut, uint32_t p)
{
	return make_float3(lut[p & 0xffu], lut[(p >> 8) & 0xffu], lut[(p >> 16) & 0xffu]);
}

__device__ __forceinline__ float3 fxaa_fetch(const float *lut, const View<const uint32_t> &im, int x, int y)
{
	return fxaa_unpack(lut, __ldg(&im.at(iclamp(x, 0, im.w - 1), iclamp(y, 0, im.h - 1))));
}

__device__ __forceinline__ float3 fxaa_sample(const float *lut, const View<const uint32_t> &im, float u, float v)
{
	Bilin s = bilin_setup(u, v, im.w, im.h);
	float3 t00 = fxaa_unpack(lut, __ldg(&im.at(s.x0, s.y0))), t10 = fxaa_unpack(lut, __ldg(&im.at(s.x1, s.y0)));
	float3 t01 = fxaa_unpack(lut, __ldg(&im.at(s.x0, s.y1))), t11 = fxaa_unpack(lut, __ldg(&im.at(s.x1, s.y1)));
	return make_float3(bilin_mix(t00.x, t10.x, t01.x, t11.x, s.a, s.b), bilin_mix(t00.y, t10.y, t01.y, t11.y, s.a, s.b),
	                   bilin_mix(t00.z, t10.z, t01.z, t11.z, s.a, s.b));
}

__device__ __forceinline__ float luma_of(float3 c) { return c.x * 0.299f + c.y * 0.587f + c.z * 0.114f; }

__device__ __forceinline__ float decode_srgb1(float c)
{
	float small_side = c / 12.92f;
	float pow_side = powf((c + 0.055f) / 1.055f, 2.4f);
	return fclamp(c <= 0.0404482362771082f ? small_side : pow_side, 0.0f, 1.0f);
}

// UNORM8 -> float is an IEEE division by 255 per channel in the contract; 63 of them per pixel
// made this pass ALU-bound.  The 256 possible quotients are computed once per CTA (same IEEE
// division) into shared memory, so the values are bit-identical and the pass is a table lookup.
template <bool SrgbTarget>
__global__ void __launch_bounds__(kBlockX *kBlockY) fxaa_kernel(View<const uint32_t> in, View<uint32_t> out, int y0, int y1, float inv_w, float inv_h)
{
	__shared__ float s_unorm[256];
	{
		int t = threadIdx.y * kBlockX + threadIdx.x;
		s_unorm[t] = (float)t / 255.0f;
	}
	__syncthreads();
	int x = blockIdx.x * kBlockX + threadIdx.x;
	int y = y0 + blockIdx.y * kBlockY + threadIdx.y;
	if (x >= out.w || y >= y1)
		return;
#define fetch_unorm8(IM, X, Y) fxaa_fetch(s_unorm, IM, X, Y)
#define sample_unorm8(IM, U, V) fxaa_sample(s_unorm, IM, U, V)
	const float FXAA_REDUCE_MIN = 1.0f / 128.0f, FXAA_REDUCE_MUL = 1.0f / 8.0f, FXAA_SPAN_MAX = 8.0f;
	float u = ((float)x + 0.5f) * inv_w, v = ((float)y + 0.5f) * inv_h;
	float lumaNW = luma_of(fetch_unorm8(in, x - 1, y - 1));
	float lumaNE = luma_of(fetch_unorm8(in, x + 1, y - 1));
	float lumaSW = luma_of(fetch_unorm8(in, x - 1, y + 1));
	float lumaSE = luma_of(fetch_unorm8(in, x + 1, y + 1));
	float lumaM = luma_of(fetch_unorm8(in, x, y));
	float lumaMin = fmin_(lumaM, fmin_(fmin_(lumaNW, lumaNE), fmin_(lumaSW, lumaSE)));
	float lumaMax = fmax_(lumaM, fmax_(fmax_(lumaNW, lumaNE), fmax_(lumaSW, lumaSE)));
	float dx = -((lumaNW + lumaNE) - (lumaSW + lumaSE));
	float dy = ((lumaNW + lumaSW) - (lumaNE + lumaSE));
	float dirReduce = fmax_((lumaNW + lumaNE + lumaSW + lumaSE) * (0.25f * FXAA_REDUCE_MUL), FXAA_REDUCE_MIN);
	float rcpDirMin = 1.0f / (fmin_(fabsf(dx), fabsf(dy)) + dirReduce);
	dx = fclamp(dx * rcpDirMin, -FXAA_SPAN_MAX, FXAA_SPAN_MAX) * inv_w;
	dy = fclamp(dy * rcpDirMin, -FXAA_SPAN_MAX, FXAA_SPAN_MAX) * inv_h;
	const float k0 = (float)(1.0 / 3.0 - 0.5), k1 = (float)(2.0 / 3.0 - 0.5); // folded by glslang in double, then rounded
	float3 a0 = sample_unorm8(in, u + dx * k0, v + dy * k0);
	float3 a1 = sample_unorm8(in, u + dx * k1, v + dy * k1);
	float3 rgbA = make_float3(0.5f * (a0.x + a1.x), 0.5f * (a0.y + a1.y), 0.5f * (a0.z + a1.z));
	float3 b0 = sample_unorm8(in, u + dx * -0.5f, v + dy * -0.5f);
	float3 b1 = sample_unorm8(in, u + dx * 0.5f, v + dy * 0.5f);
	float3 rgbB = make_float3(rgbA.x * 0.5f + 0.25f * (b0.x + b1.x), rgbA.y * 0.5f + 0.25f * (b0.y + b1.y), rgbA.z * 0.5f + 0.25f * (b0.z + b1.z));
	float lumaB = luma_of(rgbB);
	float3 c = ((lumaB < lumaMin) || (lumaB > lumaMax)) ? rgbA : rgbB;
	uint32_t px;
	if (SrgbTarget)
		px = linear_to_srgb8(decode_srgb1(c.x)) | (linear_to_srgb8(decode_srgb1(c.y)) << 8) | (linear_to_srgb8(decode_srgb1(c.z)) << 16);
	else
		px = float_to_unorm8(c.x) | (float_to_unorm8(c.y) << 8) | (float_to_unorm8(c.z) << 16);
	out.at(x, y) = px | 0xff000000u;
#undef fetch_unorm8
#undef sample_unorm8
}

// ------------------------------------------------------------------------------- K13
__device__ __forceinline__ float3 hdr_to_taa(float3 c)
{
	c = make_float3(c.x * 8.0f, c.y * 8.0f, c.z * 8.0f);
	float r = 1.0f / (fmax_(c.x, fmax_(c.y, c.z)) + 1.0f);
	c = make_float3(c.x * r, c.y * r, c.z * r);
	return make_float3(0.25f * c.x + 0.5f * c.y + 0.25f * c.z, 0.5f * c.y - 0.25f * c.x - 0.25f * c.z, 0.5f * c.x - 0.5f * c.z);
}

__device__ __forceinline__ float3 taa_to_hdr(float3 c)
{
	float tmp = c.x - c.y;
	float3 rgb = make_float3(fclamp(tmp + c.z, 0.0f, 0.999f), fclamp(c.x + c.y, 0.0f, 0.999f), fclamp(tmp - c.z, 0.0f, 0.999f));
	float r = 1.0f / (1.0f - fmax_(rgb.x, fmax_(rgb.y, rgb.z)));
	return make_float3((1.0f / 8.0f) * rgb.x * r, (1.0f / 8.0f) * rgb.y * r, (1.0f / 8.0f) * rgb.z * r);
}

__device__ __forceinline__ float3 min3(float3 a, float3 b) { return make_float3(fmin_(a.x, b.x), fmin_(a.y, b.y), fmin_(a.z, b.z)); }
__device__ __forceinline__ float3 max3(float3 a, float3 b) { return make_float3(fmax_(a.x, b.x), fmax_(a.y, b.y), fmax_(a.z, b.z)); }

template <bool Aabb>
__device__ __forceinline__ float3 clamp_box(float3 color, float3 lo, float3 hi)
{
	if (!Aabb)
		return make_float3(fclamp(color.x, lo.x, hi.x), fclamp(color.y, lo.y, hi.y), fclamp(color.z, lo.z, hi.z));
	float3 center = make_float3(0.5f * (lo.x + hi.x), 0.5f * (lo.y + hi.y), 0.5f * (lo.z + hi.z));
	float3 radius = make_float3(fmax_(0.5f * (hi.x - lo.x), 0.0001f), fmax_(0.5f * (hi.y - lo.y), 0.0001f), fmax_(0.5f * (hi.z - lo.z), 0.0001f));
	float3 v = make_float3(color.x - center.x, color.y - center.y, color.z - center.z);
	float3 units = make_float3(v.x / radius.x, v.y / radius.y, v.z / radius.z);
	float max_unit = fmax_(fmax_(fabsf(units.x), fabsf(units.y)), fabsf(units.z));
	if (max_unit > 1.0f)
		return make_float3(center.x + v.x / max_unit, center.y + v.y / max_unit, center.z + v.z / max_unit);
	return color;
}

template <typename HdrTexel>
struct TaaInputsT
{
	View<const HdrTexel> hdr;
	View<const float> depth;
	View<const uint32_t> mv; // RG16F packed
	View<const uint2> history;
};
using TaaInputs = TaaInputsT<uint32_t>;

__device__ __forceinline__ float3 sample_rgb16f(const View<const uint2> &im, float u, float v)
{
	float4 s = sample_rgba16f(im, u, v);
	return make_float3(s.x, s.y, s.z);
}

__device__ __forceinline__ float3 sample_catmull_rom(const View<const uint2> &tex, float u, float v, float4 rt)
{
	float spx = u * rt.z, spy = v * rt.w;
	float t1x = floorf(spx - 0.5f) + 0.5f, t1y = floorf(spy - 0.5f) + 0.5f;
	float fx = spx - t1x, fy = spy - t1y;
#define GRB_W0(f) ((f) * (-0.5f + (f) * (1.0f - 0.5f * (f))))
#define GRB_W1(f) (1.0f + (f) * (f) * (-2.5f + 1.5f * (f)))
#define GRB_W2(f) ((f) * (0.5f + (f) * (2.0f - 1.5f * (f))))
#define GRB_W3(f) ((f) * (f) * (-0.5f + 0.5f * (f)))
	float w0x = GRB_W0(fx), w1x = GRB_W1(fx), w2x = GRB_W2(fx), w3x = GRB_W3(fx);
	float w0y = GRB_W0(fy), w1y = GRB_W1(fy), w2y = GRB_W2(fy), w3y = GRB_W3(fy);
#undef GRB_W0
#undef GRB_W1
#undef GRB_W2
#undef GRB_W3
	float w12x = w1x + w2x, w12y = w1y + w2y;
	float o12x = w2x / (w1x + w2x), o12y = w2y / (w1y + w2y);
	float t0x = (t1x - 1.0f) * rt.x, t0y = (t1y - 1.0f) * rt.y;
	float t3x = (t1x + 2.0f) * rt.x, t3y = (t1y + 2.0f) * rt.y;
	float t12x = (t1x + o12x) * rt.x, t12y = (t1y + o12y) * rt.y;
	float3 result = make_float3(0.0f, 0.0f, 0.0f);
#define GRB_ACC(UU, VV, WA, WB)                      \
	{                                                \
		float4 s4 = sample_rgba16f_snap(tex, (UU), (VV)); float3 s = make_float3(s4.x, s4.y, s4.z); \
		result.x += s.x * (WA) * (WB);               \
		result.y += s.y * (WA) * (WB);               \
		result.z += s.z * (WA) * (WB);               \
	}
	GRB_ACC(t0x, t0y, w0x, w0y)
	GRB_ACC(t12x, t0y, w12x, w0y)
	GRB_ACC(t3x, t0y, w3x, w0y)
	GRB_ACC(t0x, t12y, w0x, w12y)
	GRB_ACC(t12x, t12y, w12x, w12y)
	GRB_ACC(t3x, t12y, w3x, w12y)
	GRB_ACC(t0x, t3y, w0x, w3y)
	GRB_ACC(t12x, t3y, w12x, w3y)
	GRB_ACC(t3x, t3y, w3x, w3y)
#undef GRB_ACC
	return result;
}

struct Mat4
{
	float m[16];
};

// The history exchange of a row-sharded frame (the peer form of the resolve): the history texels of the rows
// [own_y0, own_y1) go to the history slot of every rank instead of out_history, then the last CTA raises
// flags[flag_index] = epoch on every rank (as bloom_downsample_peers_kernel).  NoTaaPeerStore: the plain resolve.
struct NoTaaPeerStore
{
};
struct TaaPeerStore
{
	PeerTargets targets;
	int pitch_texels, own_y0, own_y1, flag_index;
	uint32_t epoch;
	unsigned *ctas_done;
};

template <int Quality, bool History, typename HdrTexel = uint32_t, typename PeerStore = NoTaaPeerStore>
__global__ void __launch_bounds__(kBlockX *kBlockY) taa_kernel(TaaInputsT<HdrTexel> in, Mat4 reproj, View<uint32_t> out_color, View<uint2> out_history, int y0,
                                                              int y1, float4 rt, PeerStore peers)
{
	constexpr bool kPeers = std::is_same<PeerStore, TaaPeerStore>::value;
	int x = blockIdx.x * kBlockX + threadIdx.x;
	int y = y0 + blockIdx.y * kBlockY + threadIdx.y;
	const bool inside = x < out_color.w && y < y1;
	if (!inside)
	{
		if (!kPeers)
			return;
		// every thread of the peer form reaches the CTA barrier of the epilogue: off the image it resolves a clamped
		// pixel and stores nothing
		x = min(x, out_color.w - 1);
		y = min(y, y1 - 1);
	}
	const int w = in.hdr.w, h = in.hdr.h;
#define GRB_CUR(DX, DY) hdr_to_taa(fetch_hdr_clamped(in.hdr, x + (DX), y + (DY)))
	float3 current = GRB_CUR(0, 0);
	float3 out_c = current;
	if (History)
	{
		float u = ((float)x + 0.5f) * rt.x, v = ((float)y + 0.5f) * rt.y;
		// sample_nearest_velocity: the closest (largest reverse-Z) depth in the footprint picks the MV
		float d;
		uint32_t mvp;
#define GRB_TRY(PX, PY)                                                 \
	{                                                                   \
		int qx = iclamp((PX), 0, w - 1), qy = iclamp((PY), 0, h - 1);   \
		float dd = __ldg(&in.depth.at(qx, qy));                         \
		if (dd > d)                                                     \
		{                                                               \
			d = dd;                                                     \
			mvp = __ldg(&in.mv.at(qx, qy));                             \
		}                                                               \
	}
		if (Quality == 2)
		{
			int qx = iclamp(x + 1, 0, w - 1), qy = iclamp(y + 1, 0, h - 1);
			d = __ldg(&in.depth.at(qx, qy));
			mvp = __ldg(&in.mv.at(qx, qy));
			GRB_TRY(x - 1, y) GRB_TRY(x, y) GRB_TRY(x, y - 1) GRB_TRY(x - 1, y - 1)
			GRB_TRY(x + 1, y) GRB_TRY(x + 1, y - 1)
			GRB_TRY(x - 1, y + 1) GRB_TRY(x, y + 1)
		}
		else
		{
			int qx = iclamp(x - 1, 0, w - 1);
			d = __ldg(&in.depth.at(qx, y));
			mvp = __ldg(&in.mv.at(qx, y));
			GRB_TRY(x, y) GRB_TRY(x, y - 1) GRB_TRY(x, y + 1) GRB_TRY(x + 1, y)
		}
#undef GRB_TRY
		float mvx = h2f((uint16_t)(mvp & 0xffffu)), mvy = h2f((uint16_t)(mvp >> 16));
		float old_u, old_v;
		if (mvx == 0.0f && mvy == 0.0f)
		{
			float cx = 2.0f * u - 1.0f, cy = 2.0f * v - 1.0f;
			const float *m = reproj.m;
			float px = m[0] * cx + m[4] * cy + m[8] * d + m[12] * 1.0f;
			float py = m[1] * cx + m[5] * cy + m[9] * d + m[13] * 1.0f;
			float pw = m[3] * cx + m[7] * cy + m[11] * d + m[15] * 1.0f;
			old_u = px / pw;
			old_v = py / pw;
			mvx = u - old_u;
			mvy = v - old_v;
		}
		else
		{
			old_u = u - mvx;
			old_v = v - mvy;
		}
		float3 hist = Quality == 2 ? sample_catmull_rom(in.history, old_u, old_v, rt) : sample_rgb16f(in.history, old_u, old_v);
		float mv_len = sqrtf(mvx * mvx + mvy * mvy);
		float mv_fast = fmin_(mv_len * 50.0f, 1.0f);
		float gamma = fmix(1.5f, 0.5f, mv_fast);
		hist = make_float3(fclamp(hist.x, 0.0f, 1.0f), fclamp(hist.y, -1.0f, 1.0f), fclamp(hist.z, -1.0f, 1.0f));
		float lerp_factor = (1.0f + 2.0f * mv_fast) / 16.0f;

		float3 c11 = current;
		float3 c01 = GRB_CUR(-1, 0), c21 = GRB_CUR(+1, 0), c10 = GRB_CUR(0, -1), c12 = GRB_CUR(0, +1);
		float3 lo = c11, hi = c11;
		if (Quality == 0 || Quality == 1)
		{
			lo = min3(lo, c01); lo = min3(lo, c21); lo = min3(lo, c10); lo = min3(lo, c12);
			hi = max3(hi, c01); hi = max3(hi, c21); hi = max3(hi, c10); hi = max3(hi, c12);
		}
		if (Quality >= 1)
		{
			float3 corner_lo = lo, corner_hi = hi;
			float3 c00 = GRB_CUR(-1, -1), c22 = GRB_CUR(+1, +1), c02 = GRB_CUR(-1, +1), c20 = GRB_CUR(+1, -1);
			if (Quality == 1)
			{
				lo = min3(lo, c00); lo = min3(lo, c22); lo = min3(lo, c02); lo = min3(lo, c20);
				hi = max3(hi, c00); hi = max3(hi, c22); hi = max3(hi, c02); hi = max3(hi, c20);
				lo = make_float3(0.5f * (corner_lo.x + lo.x), 0.5f * (corner_lo.y + lo.y), 0.5f * (corner_lo.z + lo.z));
				hi = make_float3(0.5f * (corner_hi.x + hi.x), 0.5f * (corner_hi.y + hi.y), 0.5f * (corner_hi.z + hi.z));
			}
			else
			{
#define GRB_M1(C) ((c00.C + 2.0f * c01.C + c02.C + 2.0f * c10.C + 4.0f * c11.C + 2.0f * c12.C + c20.C + 2.0f * c21.C + c22.C) / 16.0f)
#define GRB_M2(C)                                                                                                                            \
	(c00.C * c00.C + 2.0f * c01.C * c01.C + c02.C * c02.C + 2.0f * c10.C * c10.C + 4.0f * c11.C * c11.C + 2.0f * c12.C * c12.C + c20.C * c20.C + \
	 2.0f * c21.C * c21.C + c22.C * c22.C)
				float3 m1 = make_float3(GRB_M1(x), GRB_M1(y), GRB_M1(z));
				float3 m2 = make_float3(GRB_M2(x), GRB_M2(y), GRB_M2(z));
#undef GRB_M1
#undef GRB_M2
				float3 sigma = make_float3(sqrtf(fmax_(m2.x / 16.0f - m1.x * m1.x, 0.0f)), sqrtf(fmax_(m2.y / 16.0f - m1.y * m1.y, 0.0f)),
				                           sqrtf(fmax_(m2.z / 16.0f - m1.z * m1.z, 0.0f)));
				lo = make_float3(m1.x - gamma * sigma.x, m1.y - gamma * sigma.y, m1.z - gamma * sigma.z);
				hi = make_float3(m1.x + gamma * sigma.x, m1.y + gamma * sigma.y, m1.z + gamma * sigma.z);
			}
		}
		hist = clamp_box<Quality != 0>(hist, lo, hi);
		out_c = make_float3(fmix(hist.x, current.x, lerp_factor), fmix(hist.y, current.y, lerp_factor), fmix(hist.z, current.z, lerp_factor));
	}
#undef GRB_CUR
	float3 color = taa_to_hdr(out_c);
	if constexpr (!kPeers)
	{
		out_color.at(x, y) = pack_r11g11b10(color.x, color.y, color.z);
		out_history.at(x, y) = pack_rgba16f(make_float4(out_c.x, out_c.y, out_c.z, 1.0f));
	}
	else
	{
		if (inside)
		{
			out_color.at(x, y) = pack_r11g11b10(color.x, color.y, color.z);
			if (y >= peers.own_y0 && y < peers.own_y1)
			{
				const uint2 texel = pack_rgba16f(make_float4(out_c.x, out_c.y, out_c.z, 1.0f));
				const size_t at = (size_t)y * peers.pitch_texels + x;
				for (int r = 0; r < peers.targets.count; r++)
					peers.targets.data[r][at] = texel;
			}
		}
		// publish, as bloom_downsample_peers_kernel: every CTA has read its history texels and stored its band texels
		// before it arrives, so a raised flag also says "this rank is done reading last frame's slot"
		publish_to_peers(peers.targets.flags, peers.targets.count, peers.flag_index, peers.epoch, peers.ctas_done);
	}
}

// ------------------------------------------------------------------------------- pyramid tail
// d1, d2, d3 (+FEEDBACK), luminance, u2, u1 -- everything of "bloom-compute" below 1/4 resolution
// (hdr.cpp:357-376) -- as ONE cooperative launch with a grid barrier between levels.  At 4K these six
// dispatches touch 1.4 MB and 0.3 M texels altogether; as separate kernels each costs a launch and an
// almost empty GPU (7 - 9 us apiece, 46 us in a row), which is what a frame's latency and a row-sharded
// frame's replicated part consist of.  The arithmetic is the bit-exact form of this file (tent9 /
// luminance_tail), so every level equals the oracle bit for bit; sources are read with ld.global.cg
// (L2): they were written by other SMs earlier in the same launch.
__device__ __forceinline__ float4 sample_rgba16f_cg(const View<const uint2> &im, float u, float v)
{
	Bilin s = bilin_setup(u, v, im.w, im.h);
	float4 t00 = unpack_rgba16f(__ldcg(&im.at(s.x0, s.y0)));
	float4 t10 = unpack_rgba16f(__ldcg(&im.at(s.x1, s.y0)));
	float4 t01 = unpack_rgba16f(__ldcg(&im.at(s.x0, s.y1)));
	float4 t11 = unpack_rgba16f(__ldcg(&im.at(s.x1, s.y1)));
	return bilin_mix4(t00, t10, t01, t11, s.a, s.b);
}

__device__ __forceinline__ float4 tent9_cg(const View<const uint2> &src, float u, float v, float off, float inv_in_w, float inv_in_h)
{
	const float du = off * inv_in_w, dv = off * inv_in_h;
	const float um = u + (-du), up = u + du;
	const float vm = v + (-dv), vp = v + dv;
	float4 s = sample_rgba16f_cg(src, u, v);
	float4 acc = make_float4(0.25f * s.x, 0.25f * s.y, 0.25f * s.z, 0.25f * s.w);
#define GRB_TAP(W, U, V)                     \
	s = sample_rgba16f_cg(src, (U), (V));    \
	acc.x += (W)*s.x;                        \
	acc.y += (W)*s.y;                        \
	acc.z += (W)*s.z;                        \
	acc.w += (W)*s.w;
	GRB_TAP(0.0625f, um, vp)
	GRB_TAP(0.125f, u, vp)
	GRB_TAP(0.0625f, up, vp)
	GRB_TAP(0.125f, um, v)
	GRB_TAP(0.125f, up, v)
	GRB_TAP(0.0625f, um, vm)
	GRB_TAP(0.125f, u, vm)
	GRB_TAP(0.0625f, up, vm)
#undef GRB_TAP
	return acc;
}

struct TailArgs
{
	View<const uint2> d0;
	View<uint2> d1, d2, d3, u2, u1;
	View<const uint2> history; // p == nullptr: FEEDBACK = 0
	float lerp_d3;
	float *lum; // nullptr: no dynamic exposure
	float lerp_lum, lo, hi;
	// optional extras (grb_bloom_tail_ex)
	View<uint2> u0; // p == nullptr: u0 is a separate dispatch
	int u0_y0, u0_y1;
	const uint32_t *wait_flags; // row-sharded frames: every rank's "d0 band of frame wait_epoch landed" flag
	int wait_count;
	uint32_t wait_epoch;
	uint32_t *error_word;
	unsigned max_spins;
};

constexpr int kTailThreads = 1024; // few, fat CTAs: the launch shares the machine with the next frame's lighting pass, one CTA per SM it touches

__device__ __forceinline__ void tail_level(const View<const uint2> &src, const View<uint2> &dst, float off, const View<const uint2> *history, float lerp,
                                          unsigned first_cta, unsigned num_ctas, int y0 = 0, int y1 = -1)
{
	const float inv_w = 1.0f / (float)dst.w, inv_h = 1.0f / (float)dst.h, inv_in_w = 1.0f / (float)src.w, inv_in_h = 1.0f / (float)src.h;
	if (y1 < 0)
		y1 = dst.h;
	const int total = dst.w * (y1 - y0);
	for (int i = (int)((blockIdx.x - first_cta) * kTailThreads + threadIdx.x); i < total; i += (int)(num_ctas * kTailThreads))
	{
		const int yr = i / dst.w, x = i - yr * dst.w, y = y0 + yr;
		const float u = ((float)x + 0.5f) * inv_w, v = ((float)y + 0.5f) * inv_h;
		float4 value = tent9_cg(src, u, v, off, inv_in_w, inv_in_h);
		if (history)
		{
			const float4 hs = unpack_rgba16f(__ldg(&history->at(x, y))); // last frame's image: read-only here
			value = make_float4(fmix(hs.x, value.x, lerp), fmix(hs.y, value.y, lerp), fmix(hs.z, value.z, lerp), fmix(hs.w, value.w, 1.0f));
		}
		dst.at(x, y) = pack_rgba16f(value);
	}
}

__global__ void __launch_bounds__(kTailThreads) bloom_tail_kernel(const TailArgs a)
{
	namespace cg = cooperative_groups;
	cg::grid_group grid = cg::this_grid();
	__shared__ float s_grid[kLumFastMaxSamples];
	__shared__ float s_part[64];
	auto as_src = [](const View<uint2> &v) { return View<const uint2>{ v.p, v.w, v.h, v.pitch }; };
	if (a.wait_flags)
	{
		// Row-sharded frames: d0 is assembled from every rank's band (stores over NVLink peer memory, then a
		// release-store of the frame's epoch into this rank's flag array).  Waiting HERE instead of in a kernel
		// of its own lets the CTAs of this launch take their SM slots before the next frame's lighting pass
		// fills the machine; they are few (max_ctas) and spin with nanosleep.  Bounded (~4 s): a rank that
		// died must not hang the GPUs of the others.
		if ((int)threadIdx.x < a.wait_count)
			for (unsigned spins = 0; (int32_t)(load_acquire_system(a.wait_flags + threadIdx.x) - a.wait_epoch) < 0; spins++)
			{
				if (spins > a.max_spins)
				{
					if (blockIdx.x == 0)
						printf("granite_b200: timed out waiting for rank %d's band of frame %u\n", (int)threadIdx.x, a.wait_epoch);
					if (a.error_word) // picked up by the next grb_* call on this device (check_launch)
					{
						*reinterpret_cast<volatile uint32_t *>(a.error_word) = (GRB_DEVICE_ERROR_PEER_TIMEOUT << 24) | ((uint32_t)threadIdx.x << 16) | (a.wait_epoch & 0xffffu);
						__threadfence_system();
					}
					break;
				}
				__nanosleep(128);
			}
		__syncthreads();
	}
	tail_level(a.d0, a.d1, 1.75f, nullptr, 0.0f, 0u, gridDim.x);
	grid.sync();
	tail_level(as_src(a.d1), a.d2, 1.75f, nullptr, 0.0f, 0u, gridDim.x);
	grid.sync();
	tail_level(as_src(a.d2), a.d3, 1.75f, a.history.p ? &a.history : nullptr, a.lerp_d3, 0u, gridDim.x);
	grid.sync();
	// the luminance reduction (one CTA, luminance.comp's association order) runs beside the first upsample
	const bool lum_cta = a.lum != nullptr && blockIdx.x == 0 && gridDim.x > 1;
	if (a.lum != nullptr && (lum_cta || gridDim.x == 1))
	{
		const View<const uint2> d3 = as_src(a.d3);
		const int size_x = d3.w / 2, size_y = d3.h / 2;
		const float inv_sx = 1.0f / (float)size_x, inv_sy = 1.0f / (float)size_y;
		for (int i = threadIdx.x; i < size_x * size_y; i += kTailThreads)
		{
			const int sy = i / size_x, sx = i - sy * size_x;
			s_grid[i] = sample_rgba16f_cg(d3, ((float)sx + 0.5f) * inv_sx, ((float)sy + 0.5f) * inv_sy).w;
		}
		__syncthreads();
		if (threadIdx.x < 64)
		{
			const int iter_y = (size_y + 7) >> 3, iter_x = (size_x + 7) >> 3;
			const int lx = threadIdx.x & 7, ly = threadIdx.x >> 3;
			float total = 0.0f;
			for (int y = 0; y < iter_y; y++)
				for (int x = 0; x < iter_x; x++)
				{
					const int sx = x * 8 + lx, sy = y * 8 + ly;
					if (sx < size_x && sy < size_y)
						total += s_grid[sy * size_x + sx];
				}
			s_part[threadIdx.x] = total;
		}
		luminance_tail(s_part, threadIdx.x, size_x, size_y, inv_sx, inv_sy, a.lum, a.lerp_lum, a.lo, a.hi);
	}
	if (!lum_cta)
		tail_level(as_src(a.d3), a.u2, 0.875f, nullptr, 0.0f, a.lum != nullptr && gridDim.x > 1 ? 1u : 0u, a.lum != nullptr && gridDim.x > 1 ? gridDim.x - 1u : gridDim.x);
	grid.sync();
	tail_level(as_src(a.u2), a.u1, 0.875f, nullptr, 0.0f, 0u, gridDim.x);
	if (a.u0.p)
	{
		grid.sync();
		tail_level(as_src(a.u1), a.u0, 0.875f, nullptr, 0.0f, 0u, gridDim.x, a.u0_y0, a.u0_y1);
	}
}
} // namespace
} // namespace grb

namespace grb
{
// grb_post_tiles.cu: TMA + shared-memory tile form of the 2:1 pyramid steps; false = not eligible
bool launch_tent_tiled(bool up, const GrbImage *in, const GrbImage *history, float lerp, const GrbImage *out, GrbRows rows, cudaStream_t stream, int32_t *rc);
// grb_post_fast.cu: issue-optimised forms of the full-resolution passes (1 unit of the stored format)
bool launch_tonemap_fast(const GrbImage *hdr, const GrbImage *bloom, const float *luminance, float exposure, const GrbImage *out, GrbRows rows, cudaStream_t stream,
                         int32_t *rc);
bool launch_fxaa_fast(const GrbImage *in, const GrbImage *out, GrbRows rows, cudaStream_t stream, int32_t *rc);
bool launch_taa_fast(const GrbImage *hdr, const GrbImage *depth, const GrbImage *mv, const GrbImage *history, const float *reproj16, const GrbImage *out_color,
                     const GrbImage *out_history, GrbRows rows, cudaStream_t stream, int32_t *rc);
} // namespace grb

using namespace grb;

extern "C" int32_t grb_bloom_threshold(const GrbImage *hdr, const float *luminance, const GrbImage *out, GrbRows rows, void *stream)
{
	const bool hdr16 = image_ok(hdr, GRB_FORMAT_R16G16B16A16_SFLOAT, 8); // "renderTargetFp16"
	if ((!hdr16 && !image_ok(hdr, GRB_FORMAT_B10G11R11_UFLOAT_PACK32, 4)) || !image_ok(out, GRB_FORMAT_R16G16B16A16_SFLOAT, 8))
	{
		set_last_error("grb_bloom_threshold: hdr must be B10G11R11_UFLOAT or R16G16B16A16_SFLOAT and out R16G16B16A16_SFLOAT");
		return GRB_ERR_UNSUPPORTED_FORMAT;
	}
	rows = full_rows(rows, out->height);
	if (rows.y1 <= rows.y0)
		return GRB_OK;
	auto o = view_of<uint2>(out);
	dim3 grid = grid_for(out->width, rows.y1 - rows.y0), block(kBlockX, kBlockY);
	float inv_w = 1.0f / (float)out->width, inv_h = 1.0f / (float)out->height; // hdr.cpp:140-141
	if (hdr16)
	{
		if (luminance)
			bloom_threshold_kernel<true, uint2><<<grid, block, 0, as_stream(stream)>>>(view_of<const uint2>(hdr), luminance, o, rows.y0, rows.y1, inv_w, inv_h);
		else
			bloom_threshold_kernel<false, uint2><<<grid, block, 0, as_stream(stream)>>>(view_of<const uint2>(hdr), nullptr, o, rows.y0, rows.y1, inv_w, inv_h);
		return check_launch("grb_bloom_threshold");
	}
	if (luminance)
		bloom_threshold_kernel<true><<<grid, block, 0, as_stream(stream)>>>(view_of<const uint32_t>(hdr), luminance, o, rows.y0, rows.y1, inv_w, inv_h);
	else
		bloom_threshold_kernel<false><<<grid, block, 0, as_stream(stream)>>>(view_of<const uint32_t>(hdr), nullptr, o, rows.y0, rows.y1, inv_w, inv_h);
	return check_launch("grb_bloom_threshold");
}

extern "C" int32_t grb_bloom_downsample(const GrbImage *in, const GrbImage *history, float lerp, const GrbImage *out, GrbRows rows, void *stream)
{
	if (!image_ok(in, GRB_FORMAT_R16G16B16A16_SFLOAT, 8) || !image_ok(out, GRB_FORMAT_R16G16B16A16_SFLOAT, 8) ||
	    (history && (!image_ok(history, GRB_FORMAT_R16G16B16A16_SFLOAT, 8) || history->width != out->width || history->height != out->height)))
	{
		set_last_error("grb_bloom_downsample: images must be R16G16B16A16_SFLOAT and history must match out");
		return GRB_ERR_UNSUPPORTED_FORMAT;
	}
	if (history && history->data == out->data)
	{
		set_last_error("grb_bloom_downsample: history must not alias the output");
		return GRB_ERR_INVALID_ARGUMENT;
	}
	rows = full_rows(rows, out->height);
	if (rows.y1 <= rows.y0)
		return GRB_OK;
	{
		int32_t rc = GRB_OK;
		if (launch_tent_tiled(false, in, history, lerp, out, rows, as_stream(stream), &rc))
			return rc;
	}
	dim3 grid = grid_for(out->width, rows.y1 - rows.y0), block(kBlockX, kBlockY);
	float inv_w = 1.0f / (float)out->width, inv_h = 1.0f / (float)out->height;   // hdr.cpp:178-179
	float inv_in_w = 1.0f / (float)in->width, inv_in_h = 1.0f / (float)in->height; // hdr.cpp:180-181
	if (history)
		bloom_downsample_kernel<true><<<grid, block, 0, as_stream(stream)>>>(view_of<const uint2>(in), view_of<const uint2>(history), lerp,
		                                                                      view_of<uint2>(out), rows.y0, rows.y1, inv_w, inv_h, inv_in_w, inv_in_h);
	else
		bloom_downsample_kernel<false><<<grid, block, 0, as_stream(stream)>>>(view_of<const uint2>(in), View<const uint2>{}, lerp, view_of<uint2>(out),
		                                                                       rows.y0, rows.y1, inv_w, inv_h, inv_in_w, inv_in_h);
	return check_launch("grb_bloom_downsample");
}

extern "C" int32_t grb_bloom_downsample_to_peers(const GrbImage *in, const GrbImage *out_layout, void *const *peer_images, uint32_t *const *peer_flags,
                                                 int32_t peer_count, int32_t flag_index, uint32_t epoch, uint32_t *scratch_counter, GrbRows rows,
                                                 void *stream)
{
	if (!image_ok(in, GRB_FORMAT_R16G16B16A16_SFLOAT, 8) || !out_layout || out_layout->format != GRB_FORMAT_R16G16B16A16_SFLOAT || !peer_images ||
	    !peer_flags || !scratch_counter || peer_count < 1 || peer_count > GRB_MAX_PEERS || flag_index < 0 || (out_layout->row_pitch % 8) != 0)
	{
		set_last_error("grb_bloom_downsample_to_peers: bad arguments");
		return GRB_ERR_INVALID_ARGUMENT;
	}
	rows = full_rows(rows, out_layout->height);
	PeerTargets targets{};
	targets.count = peer_count;
	for (int r = 0; r < peer_count; r++)
	{
		if (!peer_images[r] || !peer_flags[r])
		{
			set_last_error("grb_bloom_downsample_to_peers: null peer pointer");
			return GRB_ERR_INVALID_ARGUMENT;
		}
		targets.data[r] = static_cast<uint2 *>(peer_images[r]);
		targets.flags[r] = peer_flags[r];
	}
	// an empty band still has to raise the flags: one CTA with nothing to store
	const int row_count = rows.y1 > rows.y0 ? rows.y1 - rows.y0 : 0;
	dim3 grid = grid_for(out_layout->width, row_count > 0 ? row_count : 1), block(kBlockX, kBlockY);
	if (row_count == 0)
		grid = dim3(1, 1, 1);
	bloom_downsample_peers_kernel<<<grid, block, 0, as_stream(stream)>>>(
	    view_of<const uint2>(in), targets, row_count > 0 ? out_layout->width : 0, out_layout->row_pitch / 8, rows.y0, rows.y0 + row_count,
	    1.0f / (float)out_layout->width, 1.0f / (float)out_layout->height, 1.0f / (float)in->width, 1.0f / (float)in->height, flag_index, epoch,
	    scratch_counter);
	return check_launch("grb_bloom_downsample_to_peers");
}

extern "C" int32_t grb_peer_wait(const uint32_t *local_flags, int32_t count, uint32_t epoch, void *stream)
{
	if (!local_flags || count < 1 || count > GRB_MAX_PEERS)
	{
		set_last_error("grb_peer_wait: bad arguments");
		return GRB_ERR_INVALID_ARGUMENT;
	}
	// ~4 s by default; GRB_PEER_WAIT_SPINS shortens the bound (tests of the timeout path)
	unsigned max_spins = 1u << 25;
	if (const char *e = getenv("GRB_PEER_WAIT_SPINS"))
		max_spins = (unsigned)strtoul(e, nullptr, 10);
	peer_wait_kernel<<<1, 32, 0, as_stream(stream)>>>(local_flags, count, epoch, device_error_word(), max_spins);
	return check_launch("grb_peer_wait");
}

static int32_t bloom_upsample_impl(const GrbImage *in, const GrbImage *out, GrbRows rows, void *stream, bool allow_tiles)
{
	if (!image_ok(in, GRB_FORMAT_R16G16B16A16_SFLOAT, 8) || !image_ok(out, GRB_FORMAT_R16G16B16A16_SFLOAT, 8))
	{
		set_last_error("grb_bloom_upsample: images must be R16G16B16A16_SFLOAT");
		return GRB_ERR_UNSUPPORTED_FORMAT;
	}
	rows = full_rows(rows, out->height);
	if (rows.y1 <= rows.y0)
		return GRB_OK;
	if (allow_tiles)
	{
		int32_t rc = GRB_OK;
		if (launch_tent_tiled(true, in, nullptr, 0.0f, out, rows, as_stream(stream), &rc))
			return rc;
	}
	dim3 grid = grid_for(out->width, rows.y1 - rows.y0), block(kBlockX, kBlockY);
	bloom_upsample_kernel<<<grid, block, 0, as_stream(stream)>>>(view_of<const uint2>(in), view_of<uint2>(out), rows.y0, rows.y1,
	                                                              1.0f / (float)out->width, 1.0f / (float)out->height, 1.0f / (float)in->width,
	                                                              1.0f / (float)in->height);
	return check_launch("grb_bloom_upsample");
}

extern "C" int32_t grb_bloom_upsample(const GrbImage *in, const GrbImage *out, GrbRows rows, void *stream)
{
	return bloom_upsample_impl(in, out, rows, stream, true);
}

// The shader's arithmetic, statement for statement, at every size (the form the fused tail uses for u0): what a
// frame falls back to when the cooperative launch is not available, so that its texels do not depend on that.
extern "C" int32_t grb_bloom_upsample_exact(const GrbImage *in, const GrbImage *out, GrbRows rows, void *stream)
{
	return bloom_upsample_impl(in, out, rows, stream, false);
}

extern "C" int32_t grb_luminance(const GrbImage *d3, float *luminance, float lerp, float min_loglum, float max_loglum, void *stream)
{
	if (!image_ok(d3, GRB_FORMAT_R16G16B16A16_SFLOAT, 8) || !luminance || d3->width < 2 || d3->height < 2)
	{
		set_last_error("grb_luminance: d3 must be R16G16B16A16_SFLOAT (>= 2x2) and luminance non-null");
		return GRB_ERR_INVALID_ARGUMENT;
	}
	if ((d3->width / 2) * (d3->height / 2) <= kLumFastMaxSamples)
		luminance_fast_kernel<<<1, kLumFastThreads, 0, as_stream(stream)>>>(view_of<const uint2>(d3), luminance, lerp, min_loglum, max_loglum);
	else
		luminance_kernel<<<1, 64, 0, as_stream(stream)>>>(view_of<const uint2>(d3), luminance, lerp, min_loglum, max_loglum);
	return check_launch("grb_luminance");
}

extern "C" int32_t grb_luminance_grid(const GrbImage *d3, float *grid, GrbRows rows, void *stream)
{
	if (!image_ok(d3, GRB_FORMAT_R16G16B16A16_SFLOAT, 8) || !grid || d3->width < 2 || d3->height < 2)
	{
		set_last_error("grb_luminance_grid: d3 must be R16G16B16A16_SFLOAT (>= 2x2) and grid non-null");
		return GRB_ERR_INVALID_ARGUMENT;
	}
	rows = full_rows(rows, d3->height / 2);
	if (rows.y1 <= rows.y0)
		return GRB_OK;
	dim3 grid_dim = grid_for(d3->width / 2, rows.y1 - rows.y0), block(kBlockX, kBlockY);
	luminance_grid_kernel<<<grid_dim, block, 0, as_stream(stream)>>>(view_of<const uint2>(d3), grid, rows.y0, rows.y1);
	return check_launch("grb_luminance_grid");
}

extern "C" int32_t grb_luminance_finalize(const float *grid, int32_t size_x, int32_t size_y, float *luminance, float lerp, float min_loglum,
                                          float max_loglum, void *stream)
{
	if (!grid || !luminance || size_x <= 0 || size_y <= 0)
	{
		set_last_error("grb_luminance_finalize: null grid/luminance or empty size");
		return GRB_ERR_INVALID_ARGUMENT;
	}
	luminance_finalize_kernel<<<1, 64, 0, as_stream(stream)>>>(grid, size_x, size_y, luminance, lerp, min_loglum, max_loglum);
	return check_launch("grb_luminance_finalize");
}

extern "C" int32_t grb_tonemap(const GrbImage *hdr, const GrbImage *bloom, const float *luminance, float dynamic_exposure, const GrbImage *out,
                               GrbRows rows, void *stream)
{
	bool srgb = out && out->format == GRB_FORMAT_R8G8B8A8_SRGB;
	const bool hdr16 = image_ok(hdr, GRB_FORMAT_R16G16B16A16_SFLOAT, 8); // "renderTargetFp16"
	if ((!hdr16 && !image_ok(hdr, GRB_FORMAT_B10G11R11_UFLOAT_PACK32, 4)) || !image_ok(bloom, GRB_FORMAT_R16G16B16A16_SFLOAT, 8) ||
	    !(image_ok(out, GRB_FORMAT_R8G8B8A8_SRGB, 4) || image_ok(out, GRB_FORMAT_R8G8B8A8_UNORM, 4)) || out->width != hdr->width ||
	    out->height != hdr->height)
	{
		set_last_error("grb_tonemap: hdr B10G11R11_UFLOAT or R16G16B16A16_SFLOAT, bloom R16G16B16A16_SFLOAT, out R8G8B8A8_{SRGB,UNORM} of hdr's size");
		return GRB_ERR_UNSUPPORTED_FORMAT;
	}
	rows = full_rows(rows, out->height);
	if (rows.y1 <= rows.y0)
		return GRB_OK;
	dim3 grid = grid_for(out->width, rows.y1 - rows.y0), block(kBlockX, kBlockY);
	float inv_w = 1.0f / (float)out->width, inv_h = 1.0f / (float)out->height;
	auto b = view_of<const uint2>(bloom);
	auto o = view_of<uint32_t>(out);
	cudaStream_t s = as_stream(stream);
	if (hdr16)
	{
		// the generic one-pixel kernel with the fp16 texel decode (the tile and 4-pixel forms read B10G11R11 only)
		auto h16 = view_of<const uint2>(hdr);
		if (luminance && srgb)
			tonemap_kernel<true, true, uint2><<<grid, block, 0, s>>>(h16, b, luminance, dynamic_exposure, o, rows.y0, rows.y1, inv_w, inv_h);
		else if (luminance)
			tonemap_kernel<true, false, uint2><<<grid, block, 0, s>>>(h16, b, luminance, dynamic_exposure, o, rows.y0, rows.y1, inv_w, inv_h);
		else if (srgb)
			tonemap_kernel<false, true, uint2><<<grid, block, 0, s>>>(h16, b, nullptr, dynamic_exposure, o, rows.y0, rows.y1, inv_w, inv_h);
		else
			tonemap_kernel<false, false, uint2><<<grid, block, 0, s>>>(h16, b, nullptr, dynamic_exposure, o, rows.y0, rows.y1, inv_w, inv_h);
		return check_launch("grb_tonemap");
	}
	auto h = view_of<const uint32_t>(hdr);
	{
		int32_t rc = GRB_OK;
		if (launch_tonemap_fast(hdr, bloom, luminance, dynamic_exposure, out, rows, s, &rc))
			return rc;
	}
	// 4-pixel path: rows 16-byte aligned and the bloom image at exactly 1/4 width
	const bool vec4 = (out->width % 4) == 0 && bloom->width * 4 == out->width && (hdr->row_pitch % 16) == 0 && (out->row_pitch % 16) == 0 &&
	                  (reinterpret_cast<uintptr_t>(hdr->data) % 16) == 0 && (reinterpret_cast<uintptr_t>(out->data) % 16) == 0;
	if (vec4)
	{
		dim3 grid4((out->width / 4 + kBlockX - 1) / kBlockX, (rows.y1 - rows.y0 + kBlockY - 1) / kBlockY, 1);
		if (luminance && srgb)
			tonemap4_kernel<true, true><<<grid4, block, 0, s>>>(h, b, luminance, dynamic_exposure, o, rows.y0, rows.y1, inv_w, inv_h);
		else if (luminance)
			tonemap4_kernel<true, false><<<grid4, block, 0, s>>>(h, b, luminance, dynamic_exposure, o, rows.y0, rows.y1, inv_w, inv_h);
		else if (srgb)
			tonemap4_kernel<false, true><<<grid4, block, 0, s>>>(h, b, nullptr, dynamic_exposure, o, rows.y0, rows.y1, inv_w, inv_h);
		else
			tonemap4_kernel<false, false><<<grid4, block, 0, s>>>(h, b, nullptr, dynamic_exposure, o, rows.y0, rows.y1, inv_w, inv_h);
		return check_launch("grb_tonemap");
	}
	if (luminance && srgb)
		tonemap_kernel<true, true><<<grid, block, 0, s>>>(h, b, luminance, dynamic_exposure, o, rows.y0, rows.y1, inv_w, inv_h);
	else if (luminance)
		tonemap_kernel<true, false><<<grid, block, 0, s>>>(h, b, luminance, dynamic_exposure, o, rows.y0, rows.y1, inv_w, inv_h);
	else if (srgb)
		tonemap_kernel<false, true><<<grid, block, 0, s>>>(h, b, nullptr, dynamic_exposure, o, rows.y0, rows.y1, inv_w, inv_h);
	else
		tonemap_kernel<false, false><<<grid, block, 0, s>>>(h, b, nullptr, dynamic_exposure, o, rows.y0, rows.y1, inv_w, inv_h);
	return check_launch("grb_tonemap");
}

extern "C" int32_t grb_fxaa(const GrbImage *in, const GrbImage *out, GrbRows rows, void *stream)
{
	auto is8 = [](const GrbImage *im) { return image_ok(im, GRB_FORMAT_R8G8B8A8_SRGB, 4) || image_ok(im, GRB_FORMAT_R8G8B8A8_UNORM, 4); };
	if (!is8(in) || !is8(out) || in->width != out->width || in->height != out->height || in->data == out->data)
	{
		set_last_error("grb_fxaa: in/out must be distinct R8G8B8A8 images of equal size");
		return GRB_ERR_UNSUPPORTED_FORMAT;
	}
	rows = full_rows(rows, out->height);
	if (rows.y1 <= rows.y0)
		return GRB_OK;
	{
		int32_t rc = GRB_OK;
		if (launch_fxaa_fast(in, out, rows, as_stream(stream), &rc))
			return rc;
	}
	dim3 grid = grid_for(out->width, rows.y1 - rows.y0), block(kBlockX, kBlockY);
	float inv_w = 1.0f / (float)in->width, inv_h = 1.0f / (float)in->height; // fxaa.cpp:45-46
	if (out->format == GRB_FORMAT_R8G8B8A8_SRGB)
		fxaa_kernel<true><<<grid, block, 0, as_stream(stream)>>>(view_of<const uint32_t>(in), view_of<uint32_t>(out), rows.y0, rows.y1, inv_w, inv_h);
	else
		fxaa_kernel<false><<<grid, block, 0, as_stream(stream)>>>(view_of<const uint32_t>(in), view_of<uint32_t>(out), rows.y0, rows.y1, inv_w, inv_h);
	return check_launch("grb_fxaa");
}

// Argument checks shared by grb_taa_resolve and grb_taa_resolve_to_peers (`what` names the entry point).  The
// history image the call writes is out_history (its layout only, for the peer form); with history it must not be the
// image the call reads.
static int32_t taa_arguments_ok(const char *what, const GrbImage *hdr, const GrbImage *depth, const GrbImage *mv, const GrbImage *history,
                                const float *reproj16, int32_t quality, const GrbImage *out_color, const GrbImage *out_history, bool *hdr16_out)
{
	char msg[256];
	const bool hdr16 = image_ok(hdr, GRB_FORMAT_R16G16B16A16_SFLOAT, 8); // "renderTargetFp16": the resolve's own output stays B10G11R11 (temporal.cpp:209-212)
	if ((!hdr16 && !image_ok(hdr, GRB_FORMAT_B10G11R11_UFLOAT_PACK32, 4)) || !image_ok(out_color, GRB_FORMAT_B10G11R11_UFLOAT_PACK32, 4) ||
	    !image_ok(out_history, GRB_FORMAT_R16G16B16A16_SFLOAT, 8) || out_color->width != hdr->width || out_color->height != hdr->height ||
	    out_history->width != hdr->width || out_history->height != hdr->height)
	{
		snprintf(msg, sizeof(msg), "%s: hdr B10G11R11_UFLOAT or R16G16B16A16_SFLOAT, out_color B10G11R11_UFLOAT, out_history R16G16B16A16_SFLOAT, equal sizes", what);
		set_last_error(msg);
		return GRB_ERR_UNSUPPORTED_FORMAT;
	}
	if (history && (!image_ok(history, GRB_FORMAT_R16G16B16A16_SFLOAT, 8) || !image_ok(depth, GRB_FORMAT_D32_SFLOAT, 4) ||
	                !image_ok(mv, GRB_FORMAT_R16G16_SFLOAT, 4) || !reproj16 || history->width != hdr->width || history->height != hdr->height ||
	                depth->width != hdr->width || depth->height != hdr->height || mv->width != hdr->width || mv->height != hdr->height ||
	                history->data == out_history->data))
	{
		snprintf(msg, sizeof(msg), "%s: with history, depth (D32_SFLOAT), mv (R16G16_SFLOAT), reproj and a distinct history image are required", what);
		set_last_error(msg);
		return GRB_ERR_INVALID_ARGUMENT;
	}
	if (quality < 0 || quality > 2)
	{
		snprintf(msg, sizeof(msg), "%s: quality must be 0..2", what);
		set_last_error(msg);
		return GRB_ERR_INVALID_ARGUMENT;
	}
	*hdr16_out = hdr16;
	return GRB_OK;
}

// The exact resolve (taa_kernel) over `rows`, for both HDR texel types, all qualities, with and without history;
// PeerStore selects the plain form (out_history) or the peer form (TaaPeerStore).
template <typename PeerStore>
static void launch_taa_exact(bool hdr16, const GrbImage *hdr, const GrbImage *depth, const GrbImage *mv, const GrbImage *history, const float *reproj16,
                             int32_t quality, const GrbImage *out_color, View<uint2> oh, GrbRows rows, cudaStream_t s, const PeerStore &peers)
{
	TaaInputs in{};
	in.hdr = view_of<const uint32_t>(hdr);
	Mat4 m{};
	if (history)
	{
		in.depth = view_of<const float>(depth);
		in.mv = view_of<const uint32_t>(mv);
		in.history = view_of<const uint2>(history);
		for (int i = 0; i < 16; i++)
			m.m[i] = reproj16[i];
	}
	auto oc = view_of<uint32_t>(out_color);
	float4 rt = make_float4(1.0f / (float)hdr->width, 1.0f / (float)hdr->height, (float)hdr->width, (float)hdr->height); // temporal.cpp:245-248
	dim3 grid = grid_for(hdr->width, rows.y1 - rows.y0), block(kBlockX, kBlockY);
	if (hdr16)
	{
		TaaInputsT<uint2> in16{};
		in16.hdr = view_of<const uint2>(hdr);
		in16.depth = in.depth;
		in16.mv = in.mv;
		in16.history = in.history;
#define GRB_LAUNCH16(Q, H) taa_kernel<Q, H, uint2, PeerStore><<<grid, block, 0, s>>>(in16, m, oc, oh, rows.y0, rows.y1, rt, peers)
		if (!history)
			GRB_LAUNCH16(0, false);
		else if (quality == 0)
			GRB_LAUNCH16(0, true);
		else if (quality == 1)
			GRB_LAUNCH16(1, true);
		else
			GRB_LAUNCH16(2, true);
#undef GRB_LAUNCH16
		return;
	}
#define GRB_LAUNCH(Q, H) taa_kernel<Q, H, uint32_t, PeerStore><<<grid, block, 0, s>>>(in, m, oc, oh, rows.y0, rows.y1, rt, peers)
	if (!history)
		GRB_LAUNCH(0, false);
	else if (quality == 0)
		GRB_LAUNCH(0, true);
	else if (quality == 1)
		GRB_LAUNCH(1, true);
	else
		GRB_LAUNCH(2, true);
#undef GRB_LAUNCH
}

extern "C" int32_t grb_taa_resolve(const GrbImage *hdr, const GrbImage *depth, const GrbImage *mv, const GrbImage *history, const float *reproj16,
                                   int32_t quality, const GrbImage *out_color, const GrbImage *out_history, GrbRows rows, void *stream)
{
	bool hdr16 = false;
	if (int32_t rc = taa_arguments_ok("grb_taa_resolve", hdr, depth, mv, history, reproj16, quality, out_color, out_history, &hdr16))
		return rc;
	rows = full_rows(rows, hdr->height);
	if (rows.y1 <= rows.y0)
		return GRB_OK;
	if (history && quality == 2 && !hdr16)
	{
		int32_t rc = GRB_OK;
		if (launch_taa_fast(hdr, depth, mv, history, reproj16, out_color, out_history, rows, as_stream(stream), &rc))
			return rc;
	}
	launch_taa_exact(hdr16, hdr, depth, mv, history, reproj16, quality, out_color, view_of<uint2>(out_history), rows, as_stream(stream), NoTaaPeerStore{});
	return check_launch("grb_taa_resolve");
}

extern "C" int32_t grb_taa_resolve_to_peers(const GrbImage *hdr, const GrbImage *depth, const GrbImage *mv, const GrbImage *history, const float *reproj16,
                                            int32_t quality, const GrbImage *out_color, const GrbImage *out_history_layout, void *const *peer_images,
                                            uint32_t *const *peer_flags, int32_t peer_count, int32_t flag_index, uint32_t epoch,
                                            uint32_t *scratch_counter, GrbRows rows, GrbRows own_rows, void *stream)
{
	if (!hdr || !out_history_layout || !peer_images || !peer_flags || !scratch_counter || peer_count < 1 || peer_count > GRB_MAX_PEERS ||
	    flag_index < 0 || flag_index >= peer_count)
	{
		set_last_error("grb_taa_resolve_to_peers: bad arguments (out_history_layout, peer_images, peer_flags, scratch_counter; peer_count 1..GRB_MAX_PEERS, "
		               "0 <= flag_index < peer_count)");
		return GRB_ERR_INVALID_ARGUMENT;
	}
	for (int r = 0; r < peer_count; r++)
		if (!peer_images[r] || !peer_flags[r])
		{
			set_last_error("grb_taa_resolve_to_peers: null peer pointer");
			return GRB_ERR_INVALID_ARGUMENT;
		}
	// the layout describes every rank's history slot; its data pointer is not written (only the peer images are)
	GrbImage layout = *out_history_layout;
	if (!layout.data)
		layout.data = peer_images[0];
	bool hdr16 = false;
	if (int32_t rc = taa_arguments_ok("grb_taa_resolve_to_peers", hdr, depth, mv, history, reproj16, quality, out_color, &layout, &hdr16))
		return rc;
	TaaPeerStore peers{};
	peers.targets.count = peer_count;
	for (int r = 0; r < peer_count; r++)
	{
		if (history && history->data == peer_images[r])
		{
			set_last_error("grb_taa_resolve_to_peers: the history image read must not be a history slot this call writes");
			return GRB_ERR_INVALID_ARGUMENT;
		}
		peers.targets.data[r] = static_cast<uint2 *>(peer_images[r]);
		peers.targets.flags[r] = peer_flags[r];
	}
	rows = full_rows(rows, hdr->height);
	own_rows = full_rows(own_rows, hdr->height);
	if (rows.y1 <= rows.y0 || own_rows.y1 <= own_rows.y0 || own_rows.y0 < rows.y0 || own_rows.y1 > rows.y1)
	{
		set_last_error("grb_taa_resolve_to_peers: rows and own_rows must be non-empty, own_rows inside rows");
		return GRB_ERR_INVALID_ARGUMENT;
	}
	peers.pitch_texels = layout.row_pitch / 8;
	peers.own_y0 = own_rows.y0;
	peers.own_y1 = own_rows.y1;
	peers.flag_index = flag_index;
	peers.epoch = epoch;
	peers.ctas_done = scratch_counter;
	launch_taa_exact(hdr16, hdr, depth, mv, history, reproj16, quality, out_color, View<uint2>{}, rows, as_stream(stream), peers);
	return check_launch("grb_taa_resolve_to_peers");
}

// d1 .. d3 (+ temporal feedback), the average-luminance update, u2 and u1 in one cooperative launch
// (hdr.cpp:357-376: three bloom_downsample dispatches, luminance, two bloom_upsample dispatches).
// `history` (last frame's d3) and `luminance` may be NULL.  Returns GRB_ERR_UNSUPPORTED_FORMAT when the
// device cannot launch cooperatively or the luminance grid exceeds the kernel's shared memory; the
// caller then issues the six calls.
extern "C" int32_t grb_bloom_tail_ex(const GrbImage *d0, const GrbImage *d1, const GrbImage *d2, const GrbImage *d3, const GrbImage *history, float lerp_d3,
                                     float *luminance, float lerp_luminance, float min_loglum, float max_loglum, const GrbImage *u2, const GrbImage *u1,
                                     const GrbBloomTailOptions *opt, void *stream);

extern "C" int32_t grb_bloom_tail(const GrbImage *d0, const GrbImage *d1, const GrbImage *d2, const GrbImage *d3, const GrbImage *history, float lerp_d3,
                                  float *luminance, float lerp_luminance, float min_loglum, float max_loglum, const GrbImage *u2, const GrbImage *u1,
                                  void *stream)
{
	return grb_bloom_tail_ex(d0, d1, d2, d3, history, lerp_d3, luminance, lerp_luminance, min_loglum, max_loglum, u2, u1, nullptr, stream);
}

// The same launch with extras (all optional): u0 rows computed after u1 (the seventh dispatch of the pyramid), a wait
// for the peer-stored d0 bands of a row-sharded frame at the start of the kernel (instead of grb_peer_wait), and a
// cap on the number of CTAs so that the launch can sit beside another kernel that wants the rest of the machine.
extern "C" int32_t grb_bloom_tail_ex(const GrbImage *d0, const GrbImage *d1, const GrbImage *d2, const GrbImage *d3, const GrbImage *history, float lerp_d3,
                                     float *luminance, float lerp_luminance, float min_loglum, float max_loglum, const GrbImage *u2, const GrbImage *u1,
                                     const GrbBloomTailOptions *opt, void *stream)
{
	if (opt && opt->u0 &&
	    (!image_ok(opt->u0, GRB_FORMAT_R16G16B16A16_SFLOAT, 8) || opt->u0->width != d0->width || opt->u0->height != d0->height || opt->u0->data == d0->data))
	{
		set_last_error("grb_bloom_tail_ex: u0 must be R16G16B16A16_SFLOAT of d0's size and not alias it");
		return GRB_ERR_INVALID_ARGUMENT;
	}
	if (opt && opt->peer_flags && (opt->peer_count <= 0 || opt->peer_count > GRB_MAX_PEERS))
	{
		set_last_error("grb_bloom_tail_ex: peer_count out of range");
		return GRB_ERR_INVALID_ARGUMENT;
	}
	const GrbImage *all[6] = { d0, d1, d2, d3, u2, u1 };
	for (const GrbImage *im : all)
		if (!image_ok(im, GRB_FORMAT_R16G16B16A16_SFLOAT, 8))
		{
			set_last_error("grb_bloom_tail: every level must be R16G16B16A16_SFLOAT");
			return GRB_ERR_UNSUPPORTED_FORMAT;
		}
	if (history && (!image_ok(history, GRB_FORMAT_R16G16B16A16_SFLOAT, 8) || history->width != d3->width || history->height != d3->height || history->data == d3->data))
	{
		set_last_error("grb_bloom_tail: history must match d3 and not alias it");
		return GRB_ERR_INVALID_ARGUMENT;
	}
	if (u2->width != d2->width || u2->height != d2->height || u1->width != d1->width || u1->height != d1->height)
	{
		set_last_error("grb_bloom_tail: u2 / u1 must have the sizes of d2 / d1");
		return GRB_ERR_INVALID_ARGUMENT;
	}
	static const bool disabled = getenv("GRB_BLOOM_NO_FUSED_TAIL") != nullptr;
	int device = 0, coop = 0, sms = 0;
	if (disabled || cudaGetDevice(&device) != cudaSuccess || cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device) != cudaSuccess || !coop ||
	    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess ||
	    (luminance && (d3->width < 2 || d3->height < 2 || (d3->width / 2) * (d3->height / 2) > kLumFastMaxSamples)))
	{
		set_last_error("grb_bloom_tail: cooperative launch unavailable (or luminance grid too large); issue the separate calls");
		return GRB_ERR_UNSUPPORTED_FORMAT;
	}
	TailArgs a;
	a.d0 = view_of<const uint2>(d0);
	a.d1 = view_of<uint2>(d1);
	a.d2 = view_of<uint2>(d2);
	a.d3 = view_of<uint2>(d3);
	a.u2 = view_of<uint2>(u2);
	a.u1 = view_of<uint2>(u1);
	a.history = history ? view_of<const uint2>(history) : View<const uint2>{};
	a.lerp_d3 = lerp_d3;
	a.lum = luminance;
	a.lerp_lum = lerp_luminance;
	a.lo = min_loglum;
	a.hi = max_loglum;
	a.u0 = View<uint2>{};
	a.u0_y0 = a.u0_y1 = 0;
	a.wait_flags = nullptr;
	a.wait_count = 0;
	a.wait_epoch = 0u;
	a.error_word = nullptr;
	a.max_spins = 1u << 25;
	int max_ctas = 0;
	if (opt)
	{
		if (opt->u0)
		{
			const GrbRows r = full_rows(opt->u0_rows, opt->u0->height);
			if (r.y1 > r.y0)
			{
				a.u0 = view_of<uint2>(opt->u0);
				a.u0_y0 = r.y0;
				a.u0_y1 = r.y1;
			}
		}
		if (opt->peer_flags)
		{
			a.wait_flags = opt->peer_flags;
			a.wait_count = opt->peer_count;
			a.wait_epoch = opt->peer_epoch;
			a.error_word = device_error_word();
			if (const char *e = getenv("GRB_PEER_WAIT_SPINS"))
				a.max_spins = (unsigned)strtoul(e, nullptr, 10);
		}
		max_ctas = opt->max_ctas;
	}
	// every CTA must be co-resident (grid barrier): ask the occupancy calculator; the largest level
	// (d1 / u1) decides how many CTAs are useful
	int per_sm = 0;
	if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bloom_tail_kernel, kTailThreads, 0) != cudaSuccess || per_sm < 1)
	{
		cudaGetLastError();
		set_last_error("grb_bloom_tail: occupancy query failed");
		return GRB_ERR_UNSUPPORTED_FORMAT;
	}
	const int texels = d1->width * d1->height;
	int ctas = std::min(sms * std::min(per_sm, 2), std::max(1, (texels + kTailThreads - 1) / kTailThreads));
	if (max_ctas > 0)
		ctas = std::min(ctas, max_ctas);
	void *params[] = { &a };
	cudaError_t err = cudaLaunchCooperativeKernel(reinterpret_cast<const void *>(bloom_tail_kernel), dim3(ctas), dim3(kTailThreads), params, 0, as_stream(stream));
	if (err != cudaSuccess)
	{
		set_last_error(cudaGetErrorString(err));
		return GRB_ERR_CUDA;
	}
	return check_launch("grb_bloom_tail");
}
