// Host-only helpers of the stateless entry points (no handle, include/hdgnn.h).  Every argument check of an entry point comes
// before its first CUDA call, and a refusal records a message naming the entry point and the argument.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <initializer_list>
#include <string>

#include "bits.cuh"

namespace hdgnn {

extern thread_local std::string g_error;   // hdgnn_last_error(NULL): the thread's last failed call without a handle (hdgnn.cu)

struct Ptr { const char* name; const void* p; unsigned align; bool required = true; };   // NULL passes unless required
struct Device { int sms, optin, per_sm; };   // SM count, opt-in shared memory per block, shared memory per SM (bytes)

struct Call {
    const char* fn;
    int fail(int code, const std::string& why) const { g_error = std::string(fn) + ": " + why; return code; }
    int invalid(const std::string& why) const { return fail(HDGNN_E_INVALID, why); }
    int cuda(cudaError_t e) const { return e == cudaSuccess ? HDGNN_OK : fail(HDGNN_E_CUDA, cudaGetErrorString(e)); }
    int launched() const { return cuda(cudaGetLastError()); }
    // a batch of B >= 1 grids of n x n, 2 <= n <= HDGNN_MAX_N
    int sizes(const char* B_name, int B, const char* n_name, int n) const {
        if (B < 1) return invalid(std::string(B_name) + " < 1");
        return n < 2 || n > HDGNN_MAX_N ? invalid(std::string(n_name) + " outside [2, HDGNN_MAX_N]") : HDGNN_OK;
    }
    int pointers(std::initializer_list<Ptr> ptrs) const {
        for (const Ptr& a : ptrs) {
            if (!a.p && a.required) return invalid(std::string(a.name) + " is null");
            if ((uintptr_t)a.p % a.align) return invalid(std::string(a.name) + " is not " + std::to_string(a.align) + "-byte aligned");
        }
        return HDGNN_OK;
    }
    int device(Device* d) const {   // the current device, which the call launches on
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&d->sms, cudaDevAttrMultiProcessorCount, dev);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&d->optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&d->per_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
        return cuda(e);
    }
    // The opt-in is one attribute per function for the whole process, so it is raised to the device maximum: a concurrent
    // caller with a smaller launch never lowers it under another's.  Not a stream operation: allowed while a graph is captured.
    template <typename K>
    int raise_smem(K* kernel, const Device& d) const {
        return cuda(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, d.optin));
    }
};

// Commits per CTA of a warp-per-commit kernel: one until the batch covers the SMs, then up to warps_max as smem_max allows.
inline int commits_per_cta(int B, int sms, size_t per_commit, size_t smem_max, int warps_max) {
    return std::max(1, std::min({B / sms, (int)(smem_max / per_commit), warps_max}));
}

// The arguments the four legacy entry points share (k_conv.cu, k_conv_bwd.cu).  The adjacency is checked before any launch
// because a tile size that does not match the bulk copy leaves a CTA waiting on its mbarrier.
inline int legacy_check(const Call& c, int B, int n, int pitch, const void* adj, int flags) {
    if (int rc = c.sizes("B", B, "N", n)) return rc;
    if (int rc = c.pointers({{"adj", adj, 16}})) return rc;
    if (flags & HDGNN_P_LABEL_BITS)
        return pitch == 4 * bit_words(n) ? HDGNN_OK : c.invalid("adj_pitch of a label bitmap must be 4 * hdgnn_bit_words(N)");
    return pitch >= n && !(pitch & 15) ? HDGNN_OK : c.invalid("adj_pitch of a byte grid must be a multiple of 16 and >= N");
}

}  // namespace hdgnn
