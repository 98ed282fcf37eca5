// TEST INFRASTRUCTURE ONLY (tests/test_emu_resources.py).  capi.cu compiled under the SIMT emulator (cuda_emu.h) with its CUDA
// allocation and event calls routed through counters of the live device allocations, pinned allocations and events, which
// fastf_emu_live_counts reads.  Linked with sharded.cu into a variant of the emulator library; the product never sees it.
#include "cuda_emu.h"
#include <atomic>

static std::atomic<long> emu_live_dev{0}, emu_live_pin{0}, emu_live_events{0};
extern "C" __attribute__((visibility("default"))) void fastf_emu_live_counts(long *dev, long *pin, long *events)
{
    *dev = emu_live_dev;
    *pin = emu_live_pin;
    *events = emu_live_events;
}
static cudaError_t counted_cudaMalloc(void **p, size_t n) { const cudaError_t e = cudaMalloc(p, n); if (e == cudaSuccess) emu_live_dev++; return e; }
static cudaError_t counted_cudaFree(void *p) { if (p) emu_live_dev--; return cudaFree(p); }
static cudaError_t counted_cudaMallocHost(void **p, size_t n) { const cudaError_t e = cudaMallocHost(p, n); if (e == cudaSuccess) emu_live_pin++; return e; }
static cudaError_t counted_cudaFreeHost(void *p) { if (p) emu_live_pin--; return cudaFreeHost(p); }
static cudaError_t counted_cudaEventCreate(cudaEvent_t *e) { const cudaError_t r = cudaEventCreate(e); if (r == cudaSuccess) emu_live_events++; return r; }
static cudaError_t counted_cudaEventCreateWithFlags(cudaEvent_t *e, unsigned f) { const cudaError_t r = cudaEventCreateWithFlags(e, f); if (r == cudaSuccess) emu_live_events++; return r; }
static cudaError_t counted_cudaEventDestroy(cudaEvent_t e) { if (e) emu_live_events--; return cudaEventDestroy(e); }
#define cudaMalloc counted_cudaMalloc
#define cudaFree counted_cudaFree
#define cudaMallocHost counted_cudaMallocHost
#define cudaFreeHost counted_cudaFreeHost
#define cudaEventCreate counted_cudaEventCreate
#define cudaEventCreateWithFlags counted_cudaEventCreateWithFlags
#define cudaEventDestroy counted_cudaEventDestroy

#include "../../fastf_b200/csrc/capi.cu"
