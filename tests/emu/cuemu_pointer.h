// tests/emu/cuemu_pointer.h -- TEST INFRASTRUCTURE, not product code.
//
// cudaPointerGetAttributes for the CPU emulation of tests/emu, so that pa_field_upload_device / pa_field_download_device
// (which reject host memory and memory of another device) run on the CPU tier too.  The variant library of build_emu_ptr.py
// compiles the kernel sources with this header force-included (-include): their device allocations (cudaMalloc / cudaFree)
// are routed through cuemu_pointer.cpp, which records every block.  cudaPointerGetAttributes then reports those blocks -- and
// the test-only blocks of cuemu_device_alloc -- as device memory of the device that was current when they were made, and
// every other address (numpy arrays, the emulator's "pinned" host buffers) as unregistered host memory.
// cuemu.cpp itself is compiled without this header and keeps the plain allocator underneath.
#ifndef PA_TESTS_EMU_CUEMU_POINTER_H
#define PA_TESTS_EMU_CUEMU_POINTER_H

#ifndef CUEMU_POINTER_IMPL
#define cudaMallocBytes cuemu_tracked_malloc
#define cudaFree cuemu_tracked_free
#endif
#include "cuda_runtime.h"

#define PA_EMU_POINTER_ATTRIBUTES 1

enum cudaMemoryType { cudaMemoryTypeUnregistered = 0, cudaMemoryTypeHost = 1, cudaMemoryTypeDevice = 2, cudaMemoryTypeManaged = 3 };
struct cudaPointerAttributes { cudaMemoryType type; int device; void* devicePointer; void* hostPointer; };
cudaError_t cudaPointerGetAttributes(cudaPointerAttributes* a, const void* p);

cudaError_t cuemu_tracked_malloc(void** p, size_t n);
cudaError_t cuemu_tracked_free(void* p);

// test-only "device" blocks for tests that hand the library device arrays; device < 0 = the current device
extern "C" void* cuemu_device_alloc(size_t bytes, int device);
extern "C" void cuemu_device_free(void* p);

#endif
