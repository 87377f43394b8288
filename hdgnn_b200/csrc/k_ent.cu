// Translation unit of the entity-grid sweeps (ent2.cuh).
#include "fused.h"

namespace hdgnn {

const void* ent2_fn_rt(int cwt, bool bwd) {
    const void* fn = nullptr;
    HDGNN_CWT_SWITCH(cwt, fn = bwd ? (const void*)ent_bwd2_kernel<CWT> : (const void*)ent_fwd2_kernel<CWT>);
    return fn;
}

void launch_ent2(int cwt, bool bwd, int grid, size_t smem, cudaStream_t st, const Ent2Args& a, bool pdl) {
    if (bwd) { HDGNN_CWT_SWITCH(cwt, launch_ex(ent_bwd2_kernel<CWT>, grid, KG * 32, smem, st, pdl, a)); }
    else { HDGNN_CWT_SWITCH(cwt, launch_ex(ent_fwd2_kernel<CWT>, grid, KG * 32, smem, st, pdl, a)); }
}

}  // namespace hdgnn
