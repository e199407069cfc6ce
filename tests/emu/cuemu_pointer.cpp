// tests/emu/cuemu_pointer.cpp -- TEST INFRASTRUCTURE: the device-block registry behind tests/emu/cuemu_pointer.h.
#define CUEMU_POINTER_IMPL 1
#include "cuemu_pointer.h"

#include <map>
#include <mutex>

namespace {
std::mutex g_mu;
std::map<uintptr_t, std::pair<uintptr_t, int>> g_blocks;       // start -> (end, device)
}  // namespace

cudaError_t cuemu_tracked_malloc(void** p, size_t n) {
    cudaError_t e = cudaMallocBytes(p, n);
    if (e != cudaSuccess) return e;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lk(g_mu);
    g_blocks[(uintptr_t)*p] = {(uintptr_t)*p + std::max<size_t>(n, 1), dev};
    return cudaSuccess;
}

cudaError_t cuemu_tracked_free(void* p) {
    {
        std::lock_guard<std::mutex> lk(g_mu);
        g_blocks.erase((uintptr_t)p);
    }
    return cudaFree(p);
}

cudaError_t cudaPointerGetAttributes(cudaPointerAttributes* a, const void* p) {
    std::memset(a, 0, sizeof(*a));
    a->type = cudaMemoryTypeUnregistered;
    a->device = -2;
    a->hostPointer = const_cast<void*>(p);
    std::lock_guard<std::mutex> lk(g_mu);
    auto it = g_blocks.upper_bound((uintptr_t)p);
    if (it != g_blocks.begin() && (uintptr_t)p < std::prev(it)->second.first) {
        a->type = cudaMemoryTypeDevice;
        a->device = std::prev(it)->second.second;
        a->devicePointer = const_cast<void*>(p);
        a->hostPointer = nullptr;
    }
    return cudaSuccess;
}

extern "C" void* cuemu_device_alloc(size_t bytes, int device) {
    int keep = 0;
    cudaGetDevice(&keep);
    if (device >= 0) cudaSetDevice(device);
    void* p = nullptr;
    cudaError_t e = cuemu_tracked_malloc(&p, bytes);
    cudaSetDevice(keep);
    return e == cudaSuccess ? p : nullptr;
}

extern "C" void cuemu_device_free(void* p) { cuemu_tracked_free(p); }
