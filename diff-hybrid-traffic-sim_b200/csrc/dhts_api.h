// Internal: pulls in the public C ABI, defines the export attribute and the launch helpers every entry point shares.
#pragma once
#include <cuda_runtime.h>
#include "../../include/dhts.h"
#define DHTS_EXPORT extern "C" __attribute__((visibility("default")))

namespace dhts {

// SMs of the current device, read once per process.
static inline int sm_count() {
    static int n = 0;
    if (!n) {
        int dev = 0; cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

// Lets `kernel` take `smem` bytes of dynamic shared memory: above the default 48 KB the attribute has to be set, above
// the 227 KB a CTA can have the shape is not supported.
template <typename K> static int set_smem(K kernel, size_t smem) {
    if (smem > 227 * 1024) return DHTS_ERR_UNSUPPORTED;
    if (smem > 48 * 1024 && cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
        cudaGetLastError();
        return DHTS_ERR_CUDA;
    }
    return DHTS_OK;
}

// set_smem, then the grid of a persistent kernel: as many CTAs as are resident on all SMs at once, at most `work`.
template <typename K> static int persistent_grid(K kernel, int threads, size_t smem, long long work, int* grid) {
    const int rc = set_smem(kernel, smem);
    if (rc) return rc;
    int occ = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, smem);
    if (occ < 1) occ = 1;
    const long long g = (long long)sm_count() * occ;
    *grid = (int)(g < work ? g : work);
    return DHTS_OK;
}

// Status of the launches just enqueued.
static inline int launch_status() { return cudaGetLastError() == cudaSuccess ? DHTS_OK : DHTS_ERR_CUDA; }

}  // namespace dhts
