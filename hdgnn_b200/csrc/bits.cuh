// bits: label bitmaps.  The dense one-hot label tensors of the reference (E_edge / C_edge,
// utils2.py:82,105) carry one bit per ordered pair; the kernels consume them as
//     bits[(b*N + i) * WP + sg]  bit l  =  (lab[b][i][sg*32 + l] != 0)  for  sg*32 + l != i,  < N
// (diagonal and padding bits zero), WP = words per row rounded up to 4 (16-byte rows).
#pragma once
#include "../../include/hdgnn.h"
#include "common.cuh"

namespace hdgnn {

// words per bitmap row: 16-byte rows; grids wider than 8 segments are swept in passes of 8 segments
__host__ __device__ __forceinline__ int bit_words(int n) { const int cw = (n + 31) / 32; return cw <= 8 ? round_up(cw, 4) : round_up(cw, 8); }

// Adjacency argument of the legacy operator (k_conv.cu, k_conv_bwd.cu), checked before any launch because a tile size
// that does not match the bulk copy leaves a CTA waiting on its mbarrier: a byte grid's row pitch is >= n and a multiple
// of 16, a label bitmap's (HDGNN_P_LABEL_BITS) exactly 4 * bit_words(n) bytes; the base is 16-byte aligned.
inline bool legacy_adj_ok(int n, int pitch, const void* adj, int flags) {
    if ((uintptr_t)adj & 15) return false;
    if (flags & HDGNN_P_LABEL_BITS) return pitch == 4 * bit_words(n);
    return pitch >= n && !(pitch & 15);
}

struct PackArgs {
    const uint8_t* adj; int Ne, pe, WPe; uint32_t* ebits;     // (B,Ne,pe) -> (B,Ne,WPe)
    const uint8_t* Y;   int Nc, pc, WPc; uint32_t* ybits;     // (B,Nc,pc) -> (B,Nc,WPc)
    int B;
};

}  // namespace hdgnn
