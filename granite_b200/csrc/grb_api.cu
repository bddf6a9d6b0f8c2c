// grb_api.cu -- library-level entry points of libgranite_b200: ABI version, per-device
// initialisation of constant tables, and the thread-local error string behind the C ABI's
// "int return code + grb_last_error_string()" convention (SURVEY.md §8b error conventions:
// no exceptions and no aborts cross the C boundary).
#include "grb_common.cuh"

#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>

namespace grb
{
static thread_local char t_last_error[512] = "";

void set_last_error(const char *msg)
{
	std::snprintf(t_last_error, sizeof(t_last_error), "%s", msg ? msg : "");
}

// Device-side failures that no CUDA error code reports (a bounded spin that ran out) are written by
// the kernel into a word of mapped pinned host memory, one per device, allocated by grb_init.  Every
// entry point ends in check_launch, which reads the word without synchronising: the call after the
// failing kernel has run returns GRB_ERR_CUDA with the decoded reason.
struct DeviceErrorWord
{
	volatile uint32_t *host = nullptr;
	uint32_t *device = nullptr;
};
static DeviceErrorWord g_error_words[64];
static std::mutex g_error_lock;

uint32_t *device_error_word()
{
	int device = -1;
	if (cudaGetDevice(&device) != cudaSuccess || device < 0 || device >= 64)
		return nullptr;
	return g_error_words[device].device;
}

static int32_t poll_device_error(const char *what)
{
	int device = -1;
	if (cudaGetDevice(&device) != cudaSuccess || device < 0 || device >= 64)
		return GRB_OK;
	volatile uint32_t *w = g_error_words[device].host;
	if (!w || *w == 0u)
		return GRB_OK;
	const uint32_t code = *w;
	*w = 0u; // reported once
	if ((code >> 24) == GRB_DEVICE_ERROR_PEER_TIMEOUT)
		std::snprintf(t_last_error, sizeof(t_last_error), "%s: an earlier wait for the peers' bands (grb_peer_wait / grb_bloom_tail_ex) timed out waiting for rank %u's band (frame epoch %u, low 16 bits); the "
		              "frame that followed used stale data", what, (code >> 16) & 0xffu, code & 0xffffu);
	else
		std::snprintf(t_last_error, sizeof(t_last_error), "%s: device-side error word 0x%08x", what, code);
	return GRB_ERR_CUDA;
}

int32_t check_launch(const char *what)
{
	cudaError_t err = cudaGetLastError();
	if (err != cudaSuccess)
	{
		std::snprintf(t_last_error, sizeof(t_last_error), "%s: %s", what, cudaGetErrorString(err));
		return GRB_ERR_CUDA;
	}
	return poll_device_error(what);
}

int32_t upload_srgb_lut(const float *lut256); // grb_lighting.cu
} // namespace grb

extern "C" int32_t grb_abi_version(void)
{
	return GRB_ABI_VERSION;
}

extern "C" const char *grb_last_error_string(void)
{
	return grb::t_last_error;
}

extern "C" int32_t grb_init(void)
{
	int device = -1;
	cudaError_t err = cudaGetDevice(&device);
	if (err != cudaSuccess)
	{
		grb::set_last_error(cudaGetErrorString(err));
		return GRB_ERR_CUDA;
	}
	cudaDeviceProp prop;
	err = cudaGetDeviceProperties(&prop, device);
	if (err != cudaSuccess)
	{
		grb::set_last_error(cudaGetErrorString(err));
		return GRB_ERR_CUDA;
	}
	if (prop.major != 10)
	{
		char msg[256];
		std::snprintf(msg, sizeof(msg), "grb_init: libgranite_b200 is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
		grb::set_last_error(msg);
		return GRB_ERR_NOT_INITIALIZED;
	}
	// R8G8B8A8_SRGB texel fetch: exact EOTF evaluated in double, rounded once to fp32.
	float lut[256];
	for (int v = 0; v < 256; v++)
	{
		double c = (double)v / 255.0;
		double l = c <= 0.04045 ? c / 12.92 : std::pow((c + 0.055) / 1.055, 2.4);
		lut[v] = (float)l;
	}
	static std::mutex lock;
	std::lock_guard<std::mutex> hold(lock);
	if (device < 64 && !grb::g_error_words[device].host)
	{
		void *host = nullptr, *dev = nullptr;
		if (cudaHostAlloc(&host, sizeof(uint32_t), cudaHostAllocMapped) == cudaSuccess && cudaHostGetDevicePointer(&dev, host, 0) == cudaSuccess)
		{
			*static_cast<uint32_t *>(host) = 0u;
			grb::g_error_words[device].host = static_cast<volatile uint32_t *>(host);
			grb::g_error_words[device].device = static_cast<uint32_t *>(dev);
		}
		else
			cudaGetLastError(); // the error word is optional: without it a timeout is only printed
	}
	return grb::upload_srgb_lut(lut);
}
