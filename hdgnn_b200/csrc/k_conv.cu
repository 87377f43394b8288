// Legacy operator of the reference's model.py (SURVEY K15 / row a16): symmetric adjacency normalisation
// fused with propagation, and the Chebyshev "map_conv" regulariser built on it.
//
//   normalize_adj   model.py:360-367   A_hat = D^-1/2 A^T D^-1/2,  D = rowsum(A) + 1e-3  (no self loop; the
//                                      transpose comes from tf.transpose(matmul(adj, D)) @ D)
//   chebyshev       model.py:335-391   T_0 = I, T_1 = (2 / 1.5)(I - A_hat) - I          (k = 2: the recurrence loop is empty)
//   map_conv        model.py:394-403   mean_b (x^T (softmax(theta)_0 T_0 + softmax(theta)_1 T_1) x)^2,  Ds = 1
//
// hdgnn_normalize_propagate is the general form  out = act(A_hat (H W) + b)  with switches for the north-star's
// A + I variant and for the un-transposed normalisation; default flags = the reference's formula.
//
// One CTA per commit.  The whole per-commit adjacency tile (N x pitch bytes) is staged in shared memory by ONE
// 1-D TMA bulk copy; the degree scan runs while the tile is resident and packs the rows into bitmaps, the
// bitmap is transposed with ballots when the reference's A^T form is asked for, and the propagation walks the
// set bits (lanes = output channels).  HBM traffic = the adjacency bytes once + H in + out.
//
// Every kernel takes the adjacency in either format (template parameter BITS): byte grids, or with
// HDGNN_P_LABEL_BITS the label bitmaps of HDGNN_F_LABEL_BITS (bits.cuh; pitch = 4 * bit_words(N) bytes).  Only the
// stage that turns the staged tile into edge bits and degrees differs; diagonal and padding bits are masked there,
// as the byte stage ignores the diagonal byte and the padding columns.
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

#include "../../include/hdgnn.h"
#include "bits.cuh"

namespace hdgnn {

constexpr int CONV_T = 256;
constexpr int CONV_MAXD = 32;       // d_in, d_out <= 32

struct ConvArgs {
    int B, N, pitch, d_in, d_out, flags;
    float eps, lam_max;
    const uint8_t* adj; const float* H; const float* W; const float* bias;
    float* out; float* dinv_out;
    const float* x; const float* theta; float* per_commit;       // map_conv
};

__host__ __device__ inline int conv_words(int N) { return (N + 31) / 32; }
__host__ __device__ inline size_t conv_smem_bytes(int N, int pitch, int d_out) {
    const int WP = conv_words(N), NP = WP * 32;
    size_t off = 16 + (size_t)round_up(N * pitch, 128);     // mbarrier, staged tile
    off += (size_t)2 * NP * WP * 4;                          // row bitmap, column bitmap (padded to 32 rows)
    off += (size_t)N * 4;                                    // dinv
    off += (size_t)N * (d_out > 0 ? d_out : 1) * 4;          // Hs (or x scaled)
    off += (size_t)(CONV_MAXD * CONV_MAXD + CONV_MAXD + 64) * 4;
    return off + 16;
}

__device__ __forceinline__ uint32_t nz4(uint32_t v) {
    const uint32_t t = (((v & 0x7f7f7f7fu) + 0x7f7f7f7fu) | v) & 0x80808080u;
    return ((t >> 7) | (t >> 14) | (t >> 21) | (t >> 28)) & 0xfu;
}

// Stages the tile, builds rbits[j][w] (bit i of word i>>5 = A[j][i] != 0, diagonal cleared), the degrees and
// dinv[j] = (deg_j + [self loop] + eps)^-1/2, and (if `transpose`) cbits[i][w] = rbits^T.  Returns pointers.
struct ConvSmem { uint8_t* tile; uint32_t* rbits; uint32_t* cbits; float* dinv; float* Hs; float* Ws; float* red; uint64_t* bar; };

__device__ __forceinline__ ConvSmem conv_carve(unsigned char* smem, int N, int pitch, int d_out) {
    const int WP = conv_words(N), NP = WP * 32;
    ConvSmem s;
    s.bar = reinterpret_cast<uint64_t*>(smem);
    s.tile = smem + 16;
    s.rbits = reinterpret_cast<uint32_t*>(smem + 16 + round_up(N * pitch, 128));
    s.cbits = s.rbits + (size_t)NP * WP;
    s.dinv = reinterpret_cast<float*>(s.cbits + (size_t)NP * WP);
    s.Hs = s.dinv + N;
    s.Ws = s.Hs + (size_t)N * (d_out > 0 ? d_out : 1);
    s.red = s.Ws + CONV_MAXD * CONV_MAXD + CONV_MAXD;
    return s;
}

// Word sg of row j of the edge bitmap (bit l = column 32 sg + l) from a label-bitmap tile (row stride bit_words(N)
// words): the diagonal and the columns >= N cleared, 0 for the padding rows j >= N.
__device__ __forceinline__ uint32_t bits_row_word(const uint8_t* tile, int j, int N, int pitch, int sg) {
    if (j >= N) return 0u;
    uint32_t w = reinterpret_cast<const uint32_t*>(tile + (size_t)j * pitch)[sg];
    const int c0 = sg * 32;
    if (c0 + 32 > N) w &= (c0 >= N) ? 0u : (0xffffffffu >> (c0 + 32 - N));
    if ((j >> 5) == sg) w &= ~(1u << (j & 31));
    return w;
}

template <bool BITS>
__device__ __forceinline__ void conv_degree_scan(const ConvSmem& s, int N, int pitch, bool self_loop, float eps, bool transpose) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, WP = conv_words(N), NP = WP * 32;
    // rows: 32 lanes x 16 bytes cover 512 columns (a bitmap row: lane = word); one row per warp iteration
    for (int j = warp; j < NP; j += CONV_T / 32) {
        uint32_t w = 0u;
        if constexpr (BITS) {
            if (lane < WP) {
                w = bits_row_word(s.tile, j, N, pitch, lane);
                s.rbits[(size_t)j * WP + lane] = w;
            }
        } else {
            uint32_t m = 0u;
            if (j < N && lane * 16 < pitch) {
                const uint4 v = *reinterpret_cast<const uint4*>(s.tile + (size_t)j * pitch + lane * 16);
                m = nz4(v.x) | (nz4(v.y) << 4) | (nz4(v.z) << 8) | (nz4(v.w) << 12);
            }
            const uint32_t hi = __shfl_down_sync(0xffffffffu, m, 1);
            const int sg = lane >> 1;
            if ((lane & 1) == 0 && sg < WP) {
                w = m | (hi << 16);
                const int c0 = sg * 32;
                if (c0 + 32 > N) w &= (c0 >= N) ? 0u : (0xffffffffu >> (c0 + 32 - N));
                if ((j >> 5) == sg) w &= ~(1u << (j & 31));
                s.rbits[(size_t)j * WP + sg] = w;
            }
        }
        const int deg = __reduce_add_sync(0xffffffffu, __popc(w));
        if (lane == 0 && j < N) s.dinv[j] = 1.f / sqrtf((float)deg + (self_loop ? 1.f : 0.f) + eps);
    }
    __syncthreads();
    if (transpose) {
        // 32 x 32 bit-block transposes: lane l holds row (jw*32 + l)'s word iw; ballot over bit c gives column c
        for (int blk = warp; blk < WP * WP; blk += CONV_T / 32) {
            const int jw = blk / WP, iw = blk - jw * WP;
            const uint32_t word = s.rbits[(size_t)(jw * 32 + lane) * WP + iw];
            uint32_t mine = 0u;
#pragma unroll
            for (int c = 0; c < 32; ++c) {
                const uint32_t col = __ballot_sync(0xffffffffu, (word >> c) & 1u);
                if (lane == c) mine = col;
            }
            s.cbits[(size_t)(iw * 32 + lane) * WP + jw] = mine;
        }
        __syncthreads();
    }
}

template <bool BITS>
__global__ void __launch_bounds__(CONV_T) propagate_kernel(const ConvArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int N = a.N, pitch = a.pitch, b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int d_in = a.d_in, d_out = a.d_out, WP = conv_words(N);
    const ConvSmem s = conv_carve(smem, N, pitch, d_out);
    if (tid == 0) {
        mbar_init(s.bar, 1);
        fence_mbar_init();
        mbar_arrive_expect_tx(s.bar, (uint32_t)N * pitch);
        bulk_g2s(s.tile, a.adj + (size_t)b * N * pitch, (uint32_t)N * pitch, s.bar);
    }
    // H W while the tile is in flight
    if (a.W) for (int i = tid; i < d_in * d_out; i += CONV_T) s.Ws[i] = a.W[i];
    __syncthreads();
    const float* Hb = a.H + (size_t)b * N * d_in;
    for (int idx = tid; idx < N * d_out; idx += CONV_T) {
        const int j = idx / d_out, c = idx - j * d_out;
        float acc = 0.f;
        if (a.W) { for (int k = 0; k < d_in; ++k) acc = fmaf(Hb[(size_t)j * d_in + k], s.Ws[k * d_out + c], acc); }
        else acc = Hb[(size_t)j * d_in + c];
        s.Hs[idx] = acc;
    }
    mbar_wait(s.bar, 0);
    __syncthreads();
    const bool self_loop = a.flags & HDGNN_P_SELF_LOOP, transpose = !(a.flags & HDGNN_P_NO_TRANSPOSE);
    conv_degree_scan<BITS>(s, N, pitch, self_loop, a.eps, transpose);
    for (int idx = tid; idx < N * d_out; idx += CONV_T) s.Hs[idx] *= s.dinv[idx / d_out];
    if (a.dinv_out) for (int j = tid; j < N; j += CONV_T) a.dinv_out[(size_t)b * N + j] = s.dinv[j];
    __syncthreads();
    // out_i = act(dinv_i * sum_{j in nbr(i)} Hs_j + b): lanes = channels, one output row per warp iteration
    const uint32_t* nb = transpose ? s.cbits : s.rbits;
    for (int i = warp; i < N; i += CONV_T / 32) {
        float acc = (self_loop && lane < d_out) ? s.Hs[(size_t)i * d_out + lane] : 0.f;
        for (int w = 0; w < WP; ++w) {
            uint32_t bits = nb[(size_t)i * WP + w];
            while (bits) {
                const int j = w * 32 + __ffs(bits) - 1;
                bits &= bits - 1;
                if (lane < d_out) acc += s.Hs[(size_t)j * d_out + lane];
            }
        }
        if (lane < d_out) {
            float v = fmaf(s.dinv[i], acc, a.bias ? a.bias[lane] : 0.f);
            if (a.flags & HDGNN_P_RELU) v = fmaxf(v, 0.f);
            a.out[((size_t)b * N + i) * d_out + lane] = v;
        }
    }
}

// ---- tcgen05 variant of the propagation ---------------------------------------------------------------------
// The per-commit product  (A or A^T, N x N, entries 0/1)  x  (D^-1/2 H W, N x d_out)  is a dense contraction:
// the adjacency is exact in bf16 and the scaled features are split into three bf16 terms (hi + mid + lo carries
// 24 mantissa bits), so one tcgen05.mma chain with fp32 accumulation in TMEM reproduces the fp32 result whatever
// the edge density.  Operands are written to shared memory by the CTA itself in the canonical no-swizzle K-major
// layout ([K/8][rows][8] bf16: 8 x 16-byte core matrices, LBO = rows * 16 B, SBO = 128 B); one thread issues
// the MMAs (M = 128 per tile, N = 4 d_out rounded to 16, K = 16 per instruction), tcgen05.commit signals an
// mbarrier and the eight warps read their 32 TMEM lanes back with tcgen05.ld for the epilogue.
constexpr int TC_T = 512;

__host__ __device__ inline int tc_np(int d_out) { return round_up(4 * d_out, 16); }
__host__ __device__ inline int tc_mp(int N) { return N <= 128 ? 128 : 256; }
__host__ __device__ inline size_t tc_smem_bytes(int N, int pitch, int d_in, int d_out) {
    const int WP = conv_words(N), NP32 = WP * 32, KP = round_up(N, 16);
    const size_t tile = (size_t)round_up(N * pitch, 128), sa = (size_t)tc_mp(N) * KP * 2;
    size_t off = 32 + (tile > sa ? tile : sa);                 // mbarrier + tmem slot | staged tile, later the A operand
    off += (size_t)tc_np(d_out) * KP * 2;                      // B operand
    off += (size_t)NP32 * WP * 4;                              // row bitmap
    off += (size_t)round_up(N, 4) * 4 + (size_t)round_up(N * d_out, 4) * 4;     // dinv, Hs
    off += (size_t)(CONV_MAXD * CONV_MAXD + CONV_MAXD) * 4;    // W
    off += (size_t)round_up(N * d_in, 4) * 4;                  // H tile (TMA)
    return off + 128;
}

__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    // cute/arch/mma_sm100_desc.hpp UMMA::SmemDescriptor: start >> 4 [0,14), LBO >> 4 [16,30), SBO >> 4 [32,46), version 1 [46,48)
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) | ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) |
           ((uint64_t)1 << 46);
}
// UMMA::InstrDescriptor: D = F32 [4,6), A = B = BF16 [7,10) [10,13), K-major, N >> 3 [17,23), M >> 4 [24,29)
__device__ __forceinline__ uint32_t umma_idesc(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

template <bool BITS>
__global__ void __launch_bounds__(TC_T, 1) propagate_tc_kernel(const ConvArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int N = a.N, pitch = a.pitch, b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int d_in = a.d_in, d_out = a.d_out, WP = conv_words(N), NP32 = WP * 32, KP = round_up(N, 16);
    const int MP = tc_mp(N), NPc = tc_np(d_out), MT = MP / 128;
    uint64_t* bar_tma = reinterpret_cast<uint64_t*>(smem);
    uint64_t* bar_mma = bar_tma + 1;
    uint32_t* tslot = reinterpret_cast<uint32_t*>(bar_tma + 2);
    uint8_t* tile = smem + 32;
    __nv_bfloat16* sA = reinterpret_cast<__nv_bfloat16*>(smem + 32);                    // aliases the staged tile
    const size_t tile_b = (size_t)round_up(N * pitch, 128), sa_b = (size_t)MP * KP * 2;
    __nv_bfloat16* sB = reinterpret_cast<__nv_bfloat16*>(smem + 32 + (tile_b > sa_b ? tile_b : sa_b));
    uint32_t* rbits = reinterpret_cast<uint32_t*>(sB + (size_t)NPc * KP);
    float* dinv = reinterpret_cast<float*>(rbits + (size_t)NP32 * WP);
    float* Hs = dinv + round_up(N, 4);
    float* Ws = Hs + (size_t)round_up(N * d_out, 4);
    float* Hin = Ws + CONV_MAXD * CONV_MAXD + CONV_MAXD;        // 16-byte aligned: every block above is a multiple of 4 floats
    int tcols = 32;
    while (tcols < MT * NPc) tcols <<= 1;
    if (tid == 0) {
        mbar_init(bar_tma, 1); mbar_init(bar_mma, 1);
        fence_mbar_init();
        const uint32_t hbytes = (uint32_t)N * d_in * 4;
        const bool htma = (hbytes & 15u) == 0 && ((((size_t)b * N * d_in * 4) & 15) == 0) && (((uintptr_t)a.H & 15) == 0);
        mbar_arrive_expect_tx(bar_tma, (uint32_t)N * pitch + (htma ? hbytes : 0u));
        bulk_g2s(tile, a.adj + (size_t)b * N * pitch, (uint32_t)N * pitch, bar_tma);
        if (htma) bulk_g2s(Hin, a.H + (size_t)b * N * d_in, hbytes, bar_tma);
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tslot)), "r"(tcols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (a.W) for (int i = tid; i < d_in * d_out; i += TC_T) Ws[i] = a.W[i];
    {
        const uint32_t hbytes = (uint32_t)N * d_in * 4;
        const bool htma = (hbytes & 15u) == 0 && ((((size_t)b * N * d_in * 4) & 15) == 0) && (((uintptr_t)a.H & 15) == 0);
        if (!htma) {            // odd shapes: plain coalesced copy of the feature tile
            const float* Hb = a.H + (size_t)b * N * d_in;
            for (int i = tid; i < N * d_in; i += TC_T) Hin[i] = Hb[i];
        }
    }
    mbar_wait(bar_tma, 0);
    __syncthreads();
    for (int idx = tid; idx < N * d_out; idx += TC_T) {         // H W from shared memory
        const int j = idx / d_out, c = idx - j * d_out;
        float acc = 0.f;
        if (a.W) { for (int k = 0; k < d_in; ++k) acc = fmaf(Hin[j * d_in + k], Ws[k * d_out + c], acc); }
        else acc = Hin[j * d_in + c];
        Hs[idx] = acc;
    }
    const bool self_loop = a.flags & HDGNN_P_SELF_LOOP, transpose = !(a.flags & HDGNN_P_NO_TRANSPOSE);
    // degree scan + row bitmap while the tile is resident (same as conv_degree_scan, no transpose needed)
    for (int j = warp; j < NP32; j += TC_T / 32) {
        uint32_t w = 0u;
        if constexpr (BITS) {
            if (lane < WP) {
                w = bits_row_word(tile, j, N, pitch, lane);
                rbits[(size_t)j * WP + lane] = w;
            }
        } else {
            uint32_t m = 0u;
            if (j < N && lane * 16 < pitch) {
                const uint4 v = *reinterpret_cast<const uint4*>(tile + (size_t)j * pitch + lane * 16);
                m = nz4(v.x) | (nz4(v.y) << 4) | (nz4(v.z) << 8) | (nz4(v.w) << 12);
            }
            const uint32_t hi = __shfl_down_sync(0xffffffffu, m, 1);
            const int sg = lane >> 1;
            if ((lane & 1) == 0 && sg < WP) {
                w = m | (hi << 16);
                const int c0 = sg * 32;
                if (c0 + 32 > N) w &= (c0 >= N) ? 0u : (0xffffffffu >> (c0 + 32 - N));
                if ((j >> 5) == sg) w &= ~(1u << (j & 31));
                rbits[(size_t)j * WP + sg] = w;
            }
        }
        const int deg = __reduce_add_sync(0xffffffffu, __popc(w));
        if (lane == 0 && j < N) dinv[j] = 1.f / sqrtf((float)deg + (self_loop ? 1.f : 0.f) + a.eps);
    }
    __syncthreads();                    // the staged tile is dead from here on: sA overwrites it
    if (a.dinv_out) for (int j = tid; j < N; j += TC_T) a.dinv_out[(size_t)b * N + j] = dinv[j];
    // A operand: A_mma[m = i][k = j] = adj[j][i] (reference form) or adj[i][j]; + I with the self loop; zero padding
    const uint32_t one = 0x3F80u;       // bf16 1.0
    for (int t = tid; t < MP * (KP >> 3); t += TC_T) {
        const int kk = t / MP, m = t - kk * MP;
        uint32_t bits8 = 0u;
        if (m < N) {
            if (transpose) {
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int j = kk * 8 + u;
                    bits8 |= ((rbits[(size_t)j * WP + (m >> 5)] >> (m & 31)) & 1u) << u;     // rows j >= N are zero (padded bitmap)
                }
            } else {
                bits8 = (rbits[(size_t)m * WP + (kk >> 2)] >> ((kk & 3) * 8)) & 0xffu;
            }
            if (self_loop && (m >> 3) == kk) bits8 |= 1u << (m & 7);
        }
        uint4 v;
        v.x = ((bits8 & 1u) ? one : 0u) | ((bits8 & 2u) ? one << 16 : 0u);
        v.y = ((bits8 & 4u) ? one : 0u) | ((bits8 & 8u) ? one << 16 : 0u);
        v.z = ((bits8 & 16u) ? one : 0u) | ((bits8 & 32u) ? one << 16 : 0u);
        v.w = ((bits8 & 64u) ? one : 0u) | ((bits8 & 128u) ? one << 16 : 0u);
        *reinterpret_cast<uint4*>(sA + ((size_t)kk * MP + m) * 8) = v;
    }
    // B operand: B_mma[n = 4 c + s][k = j] = s-th bf16 term of dinv_j * Hs[j][c] (s = 0, 1, 2), zero elsewhere
    for (int t = tid; t < (NPc >> 2) * (KP >> 3); t += TC_T) {
        const int kk = t / (NPc >> 2), c = t - kk * (NPc >> 2);
        __nv_bfloat16 o0[8], o1[8], o2[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int j = kk * 8 + u;
            const float v = (c < d_out && j < N) ? Hs[(size_t)j * d_out + c] * dinv[j] : 0.f;
            o0[u] = __float2bfloat16_rn(v);
            const float r1 = v - __bfloat162float(o0[u]);
            o1[u] = __float2bfloat16_rn(r1);
            o2[u] = __float2bfloat16_rn(r1 - __bfloat162float(o1[u]));
        }
        uint4* dst = reinterpret_cast<uint4*>(sB + ((size_t)kk * NPc + 4 * c) * 8);
        dst[0] = *reinterpret_cast<const uint4*>(o0); dst[1] = *reinterpret_cast<const uint4*>(o1);
        dst[2] = *reinterpret_cast<const uint4*>(o2); dst[3] = make_uint4(0u, 0u, 0u, 0u);
    }
    fence_proxy_async();                // generic-proxy smem writes -> visible to the tensor core (async proxy)
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tslot;
    if (tid == 0) {
        const uint32_t idesc = umma_idesc(128, NPc);
        for (int mt = 0; mt < MT; ++mt) {
            for (int ks = 0; ks < (KP >> 4); ++ks) {
                const uint64_t da = umma_desc(smem_u32(sA) + (uint32_t)(ks * 2 * MP + mt * 128) * 16, (uint32_t)MP * 16, 128);
                const uint64_t db = umma_desc(smem_u32(sB) + (uint32_t)(ks * 2 * NPc) * 16, (uint32_t)NPc * 16, 128);
                const uint32_t accum = ks > 0;
                asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                             ::"r"(tmem + (uint32_t)(mt * NPc)), "l"(da), "l"(db), "r"(idesc), "r"(accum) : "memory");
            }
        }
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar_mma)) : "memory");
    }
    mbar_wait(bar_mma, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    // epilogue: warp w owns TMEM lanes 32 (w % 4) .. + 31 of M tile w / 4
    if (warp / 4 < MT) {
        const int mt = warp >> 2, i = mt * 128 + (warp & 3) * 32 + lane;
        const float di = i < N ? dinv[i] : 0.f;
        for (int c0 = 0; c0 < d_out; c0 += 4) {
            uint32_t r[16];
            const uint32_t taddr = tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(mt * NPc + 4 * c0);
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                         : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                           "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                         : "r"(taddr) : "memory");
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            if (i < N) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int c = c0 + q;
                    if (c < d_out) {
                        const float acc = (__uint_as_float(r[4 * q]) + __uint_as_float(r[4 * q + 1])) + __uint_as_float(r[4 * q + 2]);
                        float v = fmaf(di, acc, a.bias ? a.bias[c] : 0.f);
                        if (a.flags & HDGNN_P_RELU) v = fmaxf(v, 0.f);
                        a.out[((size_t)b * N + i) * d_out + c] = v;
                    }
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(tcols) : "memory");
}

// ---- persistent tcgen05 variant: the adjacency is the wide operand ------------------------------------------------
// out^T (4 d_out x N) = Z^T (4 d_out x N_j) . Adj (N_j x N_i): the feature terms are the (small) A operand, the adjacency
// tile is the B operand with n = output node.  Every 8 consecutive bytes of adjacency row r become ONE 16-byte bf16
// chunk stored at chunk index c8 * KP + r -- and that single image serves both forms of the normalisation, because the
// canonical no-swizzle layouts only differ in which of LBO / SBO strides over which index:
//   reference form  out_i = sum_j adj[j][i] z_j : k = r, n = 8 c8 + u  -> MN-major B (SBO = KP * 16 B, LBO = 128 B)
//   un-transposed   out_i = sum_j adj[i][j] z_j : n = r, k = 8 c8 + u  -> K-major  B (LBO = KP * 16 B, SBO = 128 B)
// so there is no bit transpose at all; the row degrees fall out of the same pass over the bytes.  From a label bitmap the
// 8-column edge mask of a chunk is simply byte c8 of the row's bitmap.  A CTA is persistent over commits: as soon as a
// tile has been converted the TMA for the CTA's next commit is issued into the same buffer and lands while the operands
// are finished, the MMA chain runs and the epilogue drains TMEM.
constexpr int TC2_T = 512;
// four bytes -> four bits (bit i = byte i != 0): bytes to 0/1, then one multiply gathers them into the top nibble
__device__ __forceinline__ uint32_t nzn(uint32_t v) {
    const uint32_t t = ((((v & 0x7f7f7f7fu) + 0x7f7f7f7fu) | v) >> 7) & 0x01010101u;
    return (t * 0x01020408u) >> 24;
}
__host__ __device__ inline size_t tc2_adj_bytes(int KP) {
    const size_t adj = (size_t)(KP / 8) * (KP + 1) * 16, stage = (size_t)3 * KP * 32 * 4;
    return adj > stage ? adj : stage;
}
__host__ __device__ inline size_t tc2_smem_bytes(int N, int pitch, int d_in) {
    const int KP = round_up(N, 16), K8 = KP / 8, KS = KP + 1;   // KS: chunk stride per c8 (odd: conflict-free 16-byte stores)
    size_t off = 256;                                           // two mbarriers + TMEM slot, nibble table
    off += (size_t)round_up(N * pitch, 128);                    // staged tile (TMA destination)
    off += tc2_adj_bytes(KP);                                   // adjacency chunks [c8][r] | epilogue staging [3][KP][32] f32
    off += (size_t)K8 * 128 * 16;                               // feature chunks   [k8][m], m = 4 c + term
    off += (size_t)round_up(N * d_in, 4) * 4;                   // H tile (TMA destination)
    off += (size_t)round_up(N, 4) * 4;                          // dinv
    off += (size_t)(CONV_MAXD * CONV_MAXD + CONV_MAXD) * 4;     // W, bias
    off += (size_t)KP * 32;                                     // edge-mask bytes
    return off + 128;
}

template <bool BITS>
__global__ void __launch_bounds__(TC2_T, 1) propagate_tc2_kernel(const ConvArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int N = a.N, pitch = a.pitch, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int d_in = a.d_in, d_out = a.d_out, KP = round_up(N, 16), K8 = KP / 8, KS = KP + 1;
    uint64_t* bar_tma = reinterpret_cast<uint64_t*>(smem);
    uint64_t* bar_mma = bar_tma + 1;
    uint32_t* tslot = reinterpret_cast<uint32_t*>(bar_tma + 2);
    uint8_t* tile = smem + 256;
    uint4* sAdj = reinterpret_cast<uint4*>(tile + round_up(N * pitch, 128));
    uint4* sZ = reinterpret_cast<uint4*>(reinterpret_cast<unsigned char*>(sAdj) + tc2_adj_bytes(KP));
    float* Hin = reinterpret_cast<float*>(sZ + (size_t)K8 * 128);
    float* dinv = Hin + round_up(N * d_in, 4);
    float* Ws = dinv + round_up(N, 4);
    float* bs = Ws + CONV_MAXD * CONV_MAXD;
    uint2* lut = reinterpret_cast<uint2*>(smem + 32);           // [16] nibble -> four bf16 {0, 1}
    uint8_t* mask8 = reinterpret_cast<uint8_t*>(bs + CONV_MAXD);    // [KP][32] edge masks of a row, one byte per 8 columns
    const bool self_loop = a.flags & HDGNN_P_SELF_LOOP, transpose = !(a.flags & HDGNN_P_NO_TRANSPOSE);
    const uint32_t tbytes = (uint32_t)N * pitch, hbytes = (uint32_t)N * d_in * 4;
    const bool htma = (hbytes & 15u) == 0 && (((uintptr_t)a.H & 15) == 0);
    constexpr int TCOLS = 256;
    if (tid == 0) {
        mbar_init(bar_tma, 1); mbar_init(bar_mma, 1);
        fence_mbar_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tslot)), "r"(TCOLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (a.W) for (int i = tid; i < d_in * d_out; i += TC2_T) Ws[i] = a.W[i];
    if (tid < CONV_MAXD) bs[tid] = (a.bias && tid < d_out) ? a.bias[tid] : 0.f;
    if (tid < 16) {
        const uint32_t o1 = 0x3F80u;    // bf16 1.0
        lut[tid] = make_uint2(((tid & 1) ? o1 : 0u) | ((tid & 2) ? o1 << 16 : 0u), ((tid & 4) ? o1 : 0u) | ((tid & 8) ? o1 << 16 : 0u));
    }
    for (int i = tid; i < K8 * 128; i += TC2_T) sZ[i] = make_uint4(0u, 0u, 0u, 0u);     // rows 32 s + c with c >= d_out and rows >= 96 stay zero
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tslot;
    int b = blockIdx.x;
    if (tid == 0 && b < a.B) {
        mbar_arrive_expect_tx(bar_tma, tbytes + (htma ? hbytes : 0u));
        bulk_g2s(tile, a.adj + (size_t)b * tbytes, tbytes, bar_tma);
        if (htma) bulk_g2s(Hin, a.H + (size_t)b * N * d_in, hbytes, bar_tma);
    }
    // per-lane constants of the conversion: valid-column mask of the lane's 8 columns
    const uint32_t colmask = lane * 8 + 8 <= N ? 0xffu : (lane * 8 >= N ? 0u : (0xffu >> (lane * 8 + 8 - N)));
    uint32_t ph = 0;
    for (; b < a.B; b += gridDim.x, ph ^= 1u) {
        mbar_wait(bar_tma, ph);
        // tile -> bf16 chunks + row degrees: a warp takes four rows at a time (all loads first), a lane per 8 columns
        // (8 bytes of a byte row, or byte `lane` of a bitmap row)
        for (int r0 = warp; r0 < KP; r0 += 4 * (TC2_T / 32)) {
            uint32_t lo[4], hi[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int r = r0 + q * (TC2_T / 32);
                lo[q] = 0u; hi[q] = 0u;
                if constexpr (BITS) {
                    if (lane < K8 && r < N) lo[q] = tile[(size_t)r * pitch + lane];
                } else {
                    if (lane < K8 && r < N && lane * 8 < pitch) {
                        const uint2 v = *reinterpret_cast<const uint2*>(tile + (size_t)r * pitch + lane * 8);
                        lo[q] = v.x; hi[q] = v.y;
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int r = r0 + q * (TC2_T / 32);
                uint32_t m = (BITS ? lo[q] : (nzn(lo[q]) | (nzn(hi[q]) << 4))) & colmask;    // bit u = column 8 lane + u is an edge
                const bool dg = (r >> 3) == lane;
                if (dg) m &= ~(1u << (r & 7));                                            // the diagonal is not an edge
                if (r < KP) mask8[r * 32 + lane] = (uint8_t)m;                            // edge masks of the row, for the degree
                if (dg && self_loop && r < N) m |= 1u << (r & 7);                         // A + I
                if (lane < K8 && r < KP) {
                    const uint2 a0 = lut[m & 15u], a1 = lut[m >> 4];
                    sAdj[(size_t)lane * KS + r] = make_uint4(a0.x, a0.y, a1.x, a1.y);
                }
            }
        }
        __syncthreads();
        for (int j = tid; j < N; j += TC2_T) {              // degree = popcount of the row's 32 mask bytes (no warp reductions: REDUX is slow)
            const uint4 m0 = *reinterpret_cast<const uint4*>(mask8 + j * 32), m1 = *reinterpret_cast<const uint4*>(mask8 + j * 32 + 16);
            const int deg = __popc(m0.x) + __popc(m0.y) + __popc(m0.z) + __popc(m0.w) + __popc(m1.x) + __popc(m1.y) + __popc(m1.z) + __popc(m1.w);
            dinv[j] = 1.f / sqrtf((float)deg + (self_loop ? 1.f : 0.f) + a.eps);
        }
        fence_proxy_async();            // the generic reads of the tile are ordered before the next bulk copy into it
        __syncthreads();
        const int nb = b + gridDim.x;
        if (tid == 0 && nb < a.B) {     // prefetch: the tile buffer is free, the H buffer after the operand build below
            mbar_arrive_expect_tx(bar_tma, tbytes + (htma ? hbytes : 0u));
            bulk_g2s(tile, a.adj + (size_t)nb * tbytes, tbytes, bar_tma);
        }
        if (a.dinv_out) for (int j = tid; j < N; j += TC2_T) a.dinv_out[(size_t)b * N + j] = dinv[j];
        // feature operand: row m = 32 s + c holds the s-th bf16 term of dinv_j (H W)[j][c]; two threads per 16-byte chunk
        const float* Hb = htma ? Hin : a.H + (size_t)b * N * d_in;
        for (int t = tid; t < K8 * d_out * 2; t += TC2_T) {
            const int half = t & 1, t2 = t >> 1, kk = t2 / d_out, c = t2 - kk * d_out;
            float v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int j = kk * 8 + half * 4 + u;
                v[u] = 0.f;
                if (j < N) {
                    float acc = 0.f;
                    if (a.W) { for (int k = 0; k < d_in; ++k) acc = fmaf(Hb[(size_t)j * d_in + k], Ws[k * d_out + c], acc); }
                    else acc = Hb[(size_t)j * d_in + c];
                    v[u] = acc * dinv[j];
                }
            }
            // hi / mid / lo bf16 terms, two values per conversion (cvt.rn.bf16x2.f32)
            __nv_bfloat162 o0[2], o1[2], o2[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                o0[h] = __floats2bfloat162_rn(v[2 * h], v[2 * h + 1]);
                const float ra = v[2 * h] - __low2float(o0[h]), rb = v[2 * h + 1] - __high2float(o0[h]);
                o1[h] = __floats2bfloat162_rn(ra, rb);
                o2[h] = __floats2bfloat162_rn(ra - __low2float(o1[h]), rb - __high2float(o1[h]));
            }
            uint2* dst = reinterpret_cast<uint2*>(sZ + (size_t)kk * 128 + c) + half;
            dst[0] = *reinterpret_cast<const uint2*>(o0); dst[2 * 32] = *reinterpret_cast<const uint2*>(o1);
            dst[2 * 64] = *reinterpret_cast<const uint2*>(o2);
        }
        fence_proxy_async();            // generic-proxy smem writes -> visible to the tensor core (async proxy)
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (tid == 0) {
            if (nb < a.B && htma) bulk_g2s(Hin, a.H + (size_t)nb * N * d_in, hbytes, bar_tma);
            const uint32_t idesc = umma_idesc(128, KP) | (transpose ? (1u << 16) : 0u);       // bit 16: B is MN-major
            const uint32_t za = smem_u32(sZ), ba = smem_u32(sAdj);
            for (int ks = 0; ks < (KP >> 4); ++ks) {
                const uint64_t da = umma_desc(za + (uint32_t)ks * 2u * 128u * 16u, 128u * 16u, 128u);
                const uint64_t db = transpose ? umma_desc(ba + (uint32_t)ks * 256u, 128u, (uint32_t)KS * 16u)
                                              : umma_desc(ba + (uint32_t)ks * 2u * (uint32_t)KS * 16u, (uint32_t)KS * 16u, 128u);
                const uint32_t accum = ks > 0;
                asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                             ::"r"(tmem), "l"(da), "l"(db), "r"(idesc), "r"(accum) : "memory");
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar_mma)) : "memory");
        }
        mbar_wait(bar_mma, ph);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // epilogue: quadrant q of TMEM (lanes 32 q .. + 31) holds term q of channel c = lane for every output node.
        // Warp w drains quadrant w & 3 for the column slice w >> 2 into shared memory (the adjacency operand is dead),
        // then all threads add the three terms, scale and store the (N, d_out) tile fully coalesced.
        float* stage = reinterpret_cast<float*>(sAdj);                  // [3][KP][32]
        {
            const int q = warp & 3, sl = warp >> 2;
            if (q < 3) {
                // all loads of the warp's column slice in flight, one wait
                uint32_t r[4][16];
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    const int n0 = sl * 16 + g * 16 * (TC2_T / 128);
                    if (n0 < KP) {
                        const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)n0;
                        asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                                     : "=r"(r[g][0]), "=r"(r[g][1]), "=r"(r[g][2]), "=r"(r[g][3]), "=r"(r[g][4]), "=r"(r[g][5]), "=r"(r[g][6]),
                                       "=r"(r[g][7]), "=r"(r[g][8]), "=r"(r[g][9]), "=r"(r[g][10]), "=r"(r[g][11]), "=r"(r[g][12]),
                                       "=r"(r[g][13]), "=r"(r[g][14]), "=r"(r[g][15])
                                     : "r"(taddr) : "memory");
                    }
                }
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    const int n0 = sl * 16 + g * 16 * (TC2_T / 128);
                    if (n0 < KP) {
#pragma unroll
                        for (int u = 0; u < 16; ++u) stage[((size_t)q * KP + n0 + u) * 32 + lane] = __uint_as_float(r[g][u]);
                    }
                }
            }
        }
        __syncthreads();
        for (int i = warp; i < N; i += TC2_T / 32) {            // lanes = channels: 3 conflict-free loads, one contiguous store per row
            if (lane < d_out) {
                const float acc = (stage[(size_t)i * 32 + lane] + stage[((size_t)KP + i) * 32 + lane]) + stage[((size_t)2 * KP + i) * 32 + lane];
                float o = fmaf(dinv[i], acc, bs[lane]);
                if (a.flags & HDGNN_P_RELU) o = fmaxf(o, 0.f);
                a.out[((size_t)b * N + i) * d_out + lane] = o;
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();                // TMEM, dinv and both operand buffers are free for the next commit
    }
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TCOLS) : "memory");
}

// per commit: q_b = x^T (t0 x + t1 ((2/lam)(x - A_hat x) - x)),  t = softmax(theta)
template <bool BITS>
__global__ void __launch_bounds__(CONV_T) map_conv_kernel(const ConvArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int N = a.N, pitch = a.pitch, b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int WP = conv_words(N);
    const ConvSmem s = conv_carve(smem, N, pitch, 1);
    if (tid == 0) {
        mbar_init(s.bar, 1);
        fence_mbar_init();
        mbar_arrive_expect_tx(s.bar, (uint32_t)N * pitch);
        bulk_g2s(s.tile, a.adj + (size_t)b * N * pitch, (uint32_t)N * pitch, s.bar);
    }
    __syncthreads();
    mbar_wait(s.bar, 0);
    const bool self_loop = a.flags & HDGNN_P_SELF_LOOP, transpose = !(a.flags & HDGNN_P_NO_TRANSPOSE);
    conv_degree_scan<BITS>(s, N, pitch, self_loop, a.eps, false);
    const float* xb = a.x + (size_t)b * N;
    for (int j = tid; j < N; j += CONV_T) s.Hs[j] = xb[j] * s.dinv[j];
    __syncthreads();
    // (A_hat x)_i = dinv_i sum_j A[j][i] xs_j (reference form) or dinv_i sum_j A[i][j] xs_j
    float part = 0.f;
    const float th0 = a.theta[0], th1 = a.theta[1], mx = fmaxf(th0, th1);
    const float e0 = expf(th0 - mx), e1 = expf(th1 - mx), t0 = e0 / (e0 + e1), t1 = e1 / (e0 + e1);
    if (transpose) {
        // thread per column i: walk the rows, one broadcast word per row
        for (int i = tid; i < N; i += CONV_T) {
            const int w = i >> 5, sh = i & 31;
            float acc = self_loop ? s.Hs[i] : 0.f;
            for (int j = 0; j < N; ++j) acc += ((s.rbits[(size_t)j * WP + w] >> sh) & 1u) ? s.Hs[j] : 0.f;
            const float xi = xb[i], ax = s.dinv[i] * acc;
            part += xi * fmaf(t1, (2.f / a.lam_max) * (xi - ax) - xi, t0 * xi);
        }
    } else {
        for (int i = tid; i < N; i += CONV_T) {
            float acc = self_loop ? s.Hs[i] : 0.f;
            for (int w = 0; w < WP; ++w) {
                uint32_t bits = s.rbits[(size_t)i * WP + w];
                while (bits) { acc += s.Hs[w * 32 + __ffs(bits) - 1]; bits &= bits - 1; }
            }
            const float xi = xb[i], ax = s.dinv[i] * acc;
            part += xi * fmaf(t1, (2.f / a.lam_max) * (xi - ax) - xi, t0 * xi);
        }
    }
    const float q = block_sum(part, s.red);
    if (tid == 0) a.per_commit[b] = q * q;
    (void)lane; (void)warp;
}

// ---- map_conv for the reference's (transposed) form, straight on the staged tile ---------------------------------------
// (A_hat x)_i = dinv_i sum_j A[j][i] dinv_j x_j is a weighted COLUMN sum of the tile: no bitmap, no transpose.
// Pass 1: row degrees, one thread per row (16-byte loads; at pitch 208 the rows of 8 lanes fall on distinct banks).
// Pass 2: 4 columns per thread and row (one 4-byte word of a byte row, one nibble of a bitmap word), the rows split
// over the thread groups.  A bitmap tile keeps the byte tile's partition (WR = label_pitch(N) / 4 column groups), so
// both formats add the same terms in the same order.  The quadratic form is reduced in a fixed order.  The tile (one
// buffer, 1-D TMA bulk copy) is 42 KB at N = 200 as bytes, so five CTAs share an SM and cover each other's copy
// latency; a CTA walks commits b, b + grid, ...
constexpr int MC2_T = 256;
// WR: 4-column groups of pass 2 per row, pitch / 4 for a byte tile, label_pitch(N) / 4 for a bitmap tile
__host__ __device__ inline size_t mc2_smem_bytes(int N, int pitch, int WR) {
    const int G = MC2_T / WR > 0 ? MC2_T / WR : 1;
    return 64 + (size_t)round_up(N * pitch, 128) + (size_t)(2 * round_up(N, 4) + G * WR * 4 + 64) * 4 + 64;
}
__device__ __forceinline__ int nzcount4(uint32_t v) {      // number of non-zero bytes
    return __popc((((v & 0x7f7f7f7fu) + 0x7f7f7f7fu) | v) & 0x80808080u);
}

template <bool BITS>
__global__ void __launch_bounds__(MC2_T) map_conv2_kernel(const ConvArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int N = a.N, pitch = a.pitch, tid = threadIdx.x;
    const int WR = BITS ? round_up(N, 16) >> 2 : pitch >> 2;   // 4-column groups per row (words per byte tile row)
    const int G = MC2_T / WR > 0 ? MC2_T / WR : 1;          // row groups of pass 2 (4 at N = 200)
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
    const uint32_t tbytes = (uint32_t)N * pitch;
    uint8_t* tile = smem + 64;
    float* xs = reinterpret_cast<float*>(tile + round_up(N * pitch, 128));       // x_j dinv_j
    float* dinv = xs + round_up(N, 4);
    float* part = dinv + round_up(N, 4);                    // [G][WR * 4] column partials
    float* red = part + (size_t)G * WR * 4;
    const bool self_loop = a.flags & HDGNN_P_SELF_LOOP;
    const float th0 = a.theta[0], th1 = a.theta[1], mx = fmaxf(th0, th1);
    const float e0 = expf(th0 - mx), e1 = expf(th1 - mx), t0 = e0 / (e0 + e1), t1 = e1 / (e0 + e1);
    if (tid == 0) { mbar_init(bar, 1); fence_mbar_init(); }
    __syncthreads();
    uint32_t ph = 0u;
    for (int b = blockIdx.x; b < a.B; b += gridDim.x, ph ^= 1u) {
        if (tid == 0) {
            mbar_arrive_expect_tx(bar, tbytes);
            bulk_g2s(tile, a.adj + (size_t)b * tbytes, tbytes, bar);
        }
        const float* xb = a.x + (size_t)b * N;
        const float xmine = tid < N ? xb[tid] : 0.f;        // in flight with the tile (N <= MC2_T; else re-read below)
        mbar_wait(bar, ph);
        // pass 1: row degrees, thread per row
        for (int j = tid; j < N; j += MC2_T) {
            int c = 0;
            if constexpr (BITS) {
                for (int w = 0; w < conv_words(N); ++w) c += __popc(bits_row_word(tile, j, N, pitch, w));
                // the diagonal is not an edge: cleared in the tile, so pass 2 needs no correction
                reinterpret_cast<uint32_t*>(tile + (size_t)j * pitch)[j >> 5] &= ~(1u << (j & 31));
            } else {
                const uint4* row = reinterpret_cast<const uint4*>(tile + (size_t)j * pitch);
                for (int q = 0; q * 16 < N; ++q) {
                    const uint4 v = row[q];
                    uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const int c0 = q * 16 + k * 4;
                        if (c0 + 4 > N) w[k] = c0 >= N ? 0u : (w[k] & (0xffffffffu >> (8 * (c0 + 4 - N))));     // columns >= N
                        c += nzcount4(w[k]);
                    }
                }
                c -= tile[(size_t)j * pitch + j] != 0;      // the diagonal is not an edge
            }
            const float d = 1.f / sqrtf((float)c + (self_loop ? 1.f : 0.f) + a.eps);
            dinv[j] = d; xs[j] = (j == tid ? xmine : xb[j]) * d;
        }
        __syncthreads();
        // pass 2: weighted column sums; thread = (row group g, column group w), 4 columns per thread
        {
            const int g = tid / WR, w = tid - g * WR;
            if (g < G) {
                const int r0 = (g * N) / G, r1 = ((g + 1) * N) / G;
                float c0 = 0.f, c1 = 0.f, c2 = 0.f, c3 = 0.f;
                // byte tile: word w of the row, a byte per column; bitmap tile: nibble w & 7 of word w >> 3, a bit per column
                const uint32_t* col = reinterpret_cast<const uint32_t*>(tile) + (BITS ? w >> 3 : w);
                const int rs = BITS ? pitch >> 2 : WR;
                const uint32_t m0 = BITS ? 1u << (4 * (w & 7)) : 0x000000ffu;
                const uint32_t m1 = BITS ? m0 << 1 : 0x0000ff00u, m2 = BITS ? m0 << 2 : 0x00ff0000u, m3 = BITS ? m0 << 3 : 0xff000000u;
#pragma unroll 8
                for (int j = r0; j < r1; ++j) {
                    const uint32_t v = col[(size_t)j * rs];
                    const float xj = xs[j];
                    c0 += (v & m0) ? xj : 0.f; c1 += (v & m1) ? xj : 0.f;
                    c2 += (v & m2) ? xj : 0.f; c3 += (v & m3) ? xj : 0.f;
                }
                // the diagonal entry is not an edge: take it out again (row i of column i lies in exactly one group)
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int i = 4 * w + u;
                    if (!BITS && i < N && i >= r0 && i < r1 && tile[(size_t)i * pitch + i]) {
                        const float xi = xs[i];
                        if (u == 0) c0 -= xi; else if (u == 1) c1 -= xi; else if (u == 2) c2 -= xi; else c3 -= xi;
                    }
                }
                *reinterpret_cast<float4*>(part + ((size_t)g * WR + w) * 4) = make_float4(c0, c1, c2, c3);
            }
        }
        fence_proxy_async();                                // generic reads of the tile are ordered before the next bulk copy into it
        __syncthreads();
        float pq = 0.f;
        for (int i = tid; i < N; i += MC2_T) {
            float acc = self_loop ? xs[i] : 0.f;
            for (int g = 0; g < G; ++g) acc += part[(size_t)g * WR * 4 + i];
            const float xi = i == tid ? xmine : xb[i], ax = dinv[i] * acc;
            pq += xi * fmaf(t1, (2.f / a.lam_max) * (xi - ax) - xi, t0 * xi);
        }
        const float q = block_sum(pq, red);                 // two barriers inside: xs / dinv / part are free afterwards
        if (tid == 0) a.per_commit[b] = q * q;
    }
}

__global__ void mean_kernel(const float* v, int n, float* out) {
    __shared__ float scratch[32];
    float acc = 0.f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) acc += v[i];
    const float t = block_sum(acc, scratch);
    if (threadIdx.x == 0) *out = t / (float)n;
}

}  // namespace hdgnn

using namespace hdgnn;

static int conv_check(int B, int N, int pitch, const void* adj, int flags) {
    if (B < 1 || N < 2 || N > HDGNN_MAX_N || !adj || !legacy_adj_ok(N, pitch, adj, flags)) return HDGNN_E_INVALID;
    return HDGNN_OK;
}

extern "C" int hdgnn_normalize_propagate(int B, int N, const uint8_t* adj, int pitch, const float* H, int d_in, const float* W,
                                         const float* bias, int d_out, float eps, int flags, float* out, float* dinv_out,
                                         void* stream) {
    int rc = conv_check(B, N, pitch, adj, flags);
    if (rc) return rc;
    if (!H || !out || d_in < 1 || d_in > CONV_MAXD || d_out < 1 || d_out > CONV_MAXD) return HDGNN_E_INVALID;
    if (!W && d_in != d_out) return HDGNN_E_INVALID;
    int dev = 0, optin = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess)
        return HDGNN_E_CUDA;
    const bool bits = flags & HDGNN_P_LABEL_BITS;
    ConvArgs a{};
    a.B = B; a.N = N; a.pitch = pitch; a.d_in = d_in; a.d_out = d_out; a.flags = flags; a.eps = eps;
    a.adj = adj; a.H = H; a.W = W; a.bias = bias; a.out = out; a.dinv_out = dinv_out;
    // tensor-core paths (tcgen05), N <= 256: the persistent kernel with the adjacency as the wide operand when its
    // buffers fit one SM, else the one-CTA-per-commit kernel; else the set-bit walk on the CUDA cores.  Every size is
    // that of the tile as staged (N * pitch bytes): a bitmap tile is 1/8 of a byte tile, so the persistent kernel takes
    // bitmaps up to N = 240 at d_in = 20 where byte grids fall back to the one-CTA-per-commit kernel above N = 208.
    const size_t smem_tc2 = tc2_smem_bytes(N, pitch, d_in);
    if (!(flags & (HDGNN_P_NO_TENSOR | HDGNN_P_TENSOR_V1)) && N <= 256 && smem_tc2 <= (size_t)optin) {
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        const auto k = bits ? propagate_tc2_kernel<true> : propagate_tc2_kernel<false>;
        if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, optin) != cudaSuccess) return HDGNN_E_CUDA;
        k<<<B < sms ? B : sms, TC2_T, smem_tc2, (cudaStream_t)stream>>>(a);
        return cudaGetLastError() == cudaSuccess ? HDGNN_OK : HDGNN_E_CUDA;
    }
    const size_t smem_tc = tc_smem_bytes(N, pitch, d_in, d_out);
    if (!(flags & HDGNN_P_NO_TENSOR) && N <= 256 && smem_tc <= (size_t)optin) {
        const auto k = bits ? propagate_tc_kernel<true> : propagate_tc_kernel<false>;
        if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, optin) != cudaSuccess) return HDGNN_E_CUDA;
        k<<<B, TC_T, smem_tc, (cudaStream_t)stream>>>(a);
        return cudaGetLastError() == cudaSuccess ? HDGNN_OK : HDGNN_E_CUDA;
    }
    const size_t smem = conv_smem_bytes(N, pitch, d_out);
    if (smem > (size_t)optin) return HDGNN_E_UNSUPPORTED;       // the per-commit tile must fit one SM
    const auto k = bits ? propagate_kernel<true> : propagate_kernel<false>;
    if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, optin) != cudaSuccess) return HDGNN_E_CUDA;
    k<<<B, CONV_T, smem, (cudaStream_t)stream>>>(a);
    return cudaGetLastError() == cudaSuccess ? HDGNN_OK : HDGNN_E_CUDA;
}

extern "C" int hdgnn_map_conv(int B, int N, const uint8_t* adj, int pitch, const float* x, const float* theta, float lam_max,
                              float eps, int flags, float* per_commit, float* loss, void* stream) {
    int rc = conv_check(B, N, pitch, adj, flags);
    if (rc) return rc;
    if (!x || !theta || !per_commit || lam_max <= 0.f) return HDGNN_E_INVALID;
    const bool bits = flags & HDGNN_P_LABEL_BITS;
    const size_t smem = conv_smem_bytes(N, pitch, 1);
    int dev = 0, optin = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess)
        return HDGNN_E_CUDA;
    // the reference's (transposed) form: persistent kernel on the staged tile, several tiles in flight per SM
    const size_t smem2 = mc2_smem_bytes(N, pitch, bits ? round_up(N, 16) / 4 : pitch / 4);
    if (!(flags & (HDGNN_P_NO_TRANSPOSE | HDGNN_P_TENSOR_V1)) && smem2 <= (size_t)optin) {
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        const auto k2 = bits ? map_conv2_kernel<true> : map_conv2_kernel<false>;
        if (cudaFuncSetAttribute(k2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2) != cudaSuccess) return HDGNN_E_CUDA;
        ConvArgs a2{};
        a2.B = B; a2.N = N; a2.pitch = pitch; a2.flags = flags; a2.eps = eps; a2.lam_max = lam_max;
        a2.adj = adj; a2.x = x; a2.theta = theta; a2.per_commit = per_commit;
        int per_sm = (int)((size_t)(228 * 1024) / (smem2 + 1024));       // resident CTAs an SM's shared memory allows
        per_sm = per_sm < 1 ? 1 : (per_sm > 8 ? 8 : per_sm);
        const int grid = B < sms * per_sm ? B : sms * per_sm;
        if (!x || !theta || !per_commit || lam_max <= 0.f) return HDGNN_E_INVALID;
        k2<<<grid, MC2_T, smem2, (cudaStream_t)stream>>>(a2);
        if (loss) mean_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(per_commit, B, loss);
        return cudaGetLastError() == cudaSuccess ? HDGNN_OK : HDGNN_E_CUDA;
    }
    if (smem > (size_t)optin) return HDGNN_E_UNSUPPORTED;
    const auto k = bits ? map_conv_kernel<true> : map_conv_kernel<false>;
    if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, optin) != cudaSuccess) return HDGNN_E_CUDA;
    ConvArgs a{};
    a.B = B; a.N = N; a.pitch = pitch; a.flags = flags; a.eps = eps; a.lam_max = lam_max;
    a.adj = adj; a.x = x; a.theta = theta; a.per_commit = per_commit;
    k<<<B, CONV_T, smem, (cudaStream_t)stream>>>(a);
    if (loss) mean_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(per_commit, B, loss);
    return cudaGetLastError() == cudaSuccess ? HDGNN_OK : HDGNN_E_CUDA;
}
