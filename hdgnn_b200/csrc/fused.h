// Launchers of the fused-path kernels; each kernel family is compiled in its own translation unit
// (k_ent.cu, k_mid.cu) so the template instantiations build in parallel.
#pragma once
#include <cuda_runtime.h>
#include "ent2.cuh"
#include "mid2.cuh"

namespace hdgnn {

// kernel handle for cudaFuncSetAttribute / occupancy queries (nullptr if not instantiated)
const void* ent2_fn_rt(int cwt, bool bwd);
const void* mid2_fn_rt(int cwt, bool train, bool gt, bool cl = false);
int mid2_max_clusters(int cwt, bool train, size_t smem);
// which table placements are compiled for a hunk-grid width: shared memory for cwt <= 5, global memory for cwt >= 5
bool mid2_gt_supported(int cwt, bool gt);
// pdl: launch with programmatic stream serialization (the kernel calls pdl_wait() before it reads its
// predecessor's outputs, so its prologue overlaps the predecessor's tail)
void launch_ent2(int cwt, bool bwd, int grid, size_t smem, cudaStream_t st, const Ent2Args& a, bool pdl);
void launch_mid2(int cwt, bool train, bool gt, bool cl, int grid, size_t smem, cudaStream_t st, const Mid2Args& a, bool pdl);

// cluster: CTAs per thread-block cluster (1 = none; the grid must be a multiple)
template <typename Kern, typename Args>
inline cudaError_t launch_ex(Kern kern, int grid, int block, size_t smem, cudaStream_t st, bool pdl, const Args& a, int cluster = 1) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[2];
    int n = 0;
    if (pdl) {
        attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[n].val.programmaticStreamSerializationAllowed = 1;
        ++n;
    }
    if (cluster > 1) {
        attr[n].id = cudaLaunchAttributeClusterDimension;
        attr[n].val.clusterDim.x = cluster; attr[n].val.clusterDim.y = 1; attr[n].val.clusterDim.z = 1;
        ++n;
    }
    cfg.attrs = attr; cfg.numAttrs = n;
    return cudaLaunchKernelEx(&cfg, kern, a);
}

#define HDGNN_CWT_SWITCH(cwt, ...)                                                                  \
    switch (cwt) {                                                                                  \
        case 1: { constexpr int CWT = 1; __VA_ARGS__; } break; case 2: { constexpr int CWT = 2; __VA_ARGS__; } break; \
        case 3: { constexpr int CWT = 3; __VA_ARGS__; } break; case 4: { constexpr int CWT = 4; __VA_ARGS__; } break; \
        case 5: { constexpr int CWT = 5; __VA_ARGS__; } break; case 6: { constexpr int CWT = 6; __VA_ARGS__; } break; \
        case 7: { constexpr int CWT = 7; __VA_ARGS__; } break; case 8: { constexpr int CWT = 8; __VA_ARGS__; } break; \
        default: break;                                                                             \
    }

}  // namespace hdgnn
