// pairsum: the O(N^2 * 20) kernel of the hot path.
//
// For one commit and an N x N grid of ordered pairs (i != j) it evaluates the first layer of a
// per-pair MLP in the separable form
//        pre_ij[k] = P_i[k] + Q_j[k] + l_ij * D[k]          l_ij in {0,1} from the label bitmap
// and reduces over the grid.  Because the second layer of every pair MLP in the reference is
// linear and immediately row/column-summed by a one-hot matmul (model_2.py:172-188 entity
// effects, model_2.py:263-275 hunk "edge translation", model_4.py:226-240 entity-edge effects)
// only the row sums RS_i = sum_{j!=i} relu(pre_ij) and column sums CS_j = sum_{i!=j} relu(pre_ij)
// are ever needed; the 20x20 layer is applied to the sums by the node kernels.
//
//   FWD:  h = relu(pre)                    -> RS (B,N,20), CS partial (B,S,N,20)
//   BWD:  v = (GR_i + GC_j) * [pre > 0]    -> RSd, CSd partial, LS = sum_{l_ij = 1} v  (B,S,20)
//
// Mapping: grid (S row tiles, B commits); one warp per hidden channel k (20 warps); lane owns
// columns j = seg*32 + lane, seg < CW (column sums live in registers for the whole tile); rows
// are swept four at a time, their sums reduced across lanes by a fixed-order shuffle butterfly.
// The label tile (RT bitmap rows of WP words, contiguous) is staged by one 1-D TMA bulk copy and
// re-packed once per CTA into float4 {l(i..i+3, j)} so the inner loop issues one LDS.128 per four
// pairs.  The diagonal pair (i,i) is carried through with l = 0 and subtracted once at the
// end.  No atomics: every sum has a fixed order.
#pragma once
#include "common.cuh"

namespace hdgnn {

struct PairSumArgs {
    const uint32_t* bits; // (B, N, WP) label bitmap (bits.cuh)
    int WP;
    int N, RT, S;         // grid size, rows per CTA (multiple of 4, >= 20), row tiles
    const float* params;
    // RANK1: P_i = x_i*par[o_u+k] + par[o_b+k] + par[o_l+k];  Q_j = x_j*par[o_v+k]
    // TABLE: P_i = Ptab[b,i,k] (bias and label-0 row already folded in);  Q_j = Qtab[b,j,k]
    // both:  D = par[o_l+20+k] - par[o_l+k]
    const float* x;
    int o_u, o_v, o_b, o_l;
    const float* Ptab;
    const float* Qtab;
    const float* GR;      // BWD: (B,N,20) upstream gradient of the row sums
    const float* GC;      // BWD: (B,N,20) upstream gradient of the column sums
    float* RS;            // (B,N,20)
    float* CSp;           // (B,S,N,20)
    float* LSp;           // BWD: (B,S,20)
};

__host__ __device__ inline size_t pairsum_smem_bytes(int CW, int RT, int row_bytes, bool bwd) {
    size_t off = round_up(RT * row_bytes, 128);
    size_t labf = (size_t)(RT / 4) * (CW * 32) * 16;
    size_t cst = (size_t)(CW * 32) * HD * 4;
    off += labf > cst ? labf : cst;
    off += (size_t)RT * HD * 4 * (bwd ? 4 : 3);
    return off + 16;
}

template <int CW, bool BWD, bool RANK1>
__global__ void __launch_bounds__(32 * HD) pairsum_kernel(const PairSumArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int NP = CW * 32;
    const int N = a.N, RT = a.RT, WP = a.WP;
    const int b = blockIdx.y, s = blockIdx.x;
    const int r0 = s * RT;
    const int nrows = min(RT, N - r0);
    const int tid = threadIdx.x, lane = tid & 31, k = tid >> 5;

    uint32_t* stage = reinterpret_cast<uint32_t*>(smem);
    size_t off = round_up(RT * WP * 4, 128);
    float4* labf = reinterpret_cast<float4*>(smem + off);
    float* CSt = reinterpret_cast<float*>(smem + off);          // reused after the sweep
    {
        size_t l1 = (size_t)(RT / 4) * NP * 16, l2 = (size_t)NP * HD * 4;
        off += l1 > l2 ? l1 : l2;
    }
    float* Pt = reinterpret_cast<float*>(smem + off);  off += (size_t)RT * HD * 4;
    float* GRt = reinterpret_cast<float*>(smem + off); if (BWD) off += (size_t)RT * HD * 4;
    float* RSt = reinterpret_cast<float*>(smem + off); off += (size_t)RT * HD * 4;
    float* dg = reinterpret_cast<float*>(smem + off);  off += (size_t)RT * HD * 4;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + off);

    if (tid == 0) { mbar_init(bar, 1); fence_mbar_init(); }
    __syncthreads();
    if (tid == 0) {
        const uint32_t bytes = (uint32_t)nrows * WP * 4;
        mbar_arrive_expect_tx(bar, bytes);
        bulk_g2s(stage, a.bits + ((size_t)b * N + r0) * WP, bytes, bar);
    }

    const float* par = a.params;
    const float D = par[a.o_l + HD + k] - par[a.o_l + k];
    // row tables for this tile
    for (int idx = tid; idx < RT * HD; idx += blockDim.x) {
        const int r = idx / HD, kk = idx - r * HD, i = r0 + r;
        float p = NEG_BIG, g = 0.f;
        if (r < nrows) {
            if (RANK1) p = __fmul_rn(a.x[(size_t)b * N + i], par[a.o_u + kk]) + (par[a.o_b + kk] + par[a.o_l + kk]);
            else p = a.Ptab[((size_t)b * N + i) * HD + kk];
            if (BWD) g = a.GR[((size_t)b * N + i) * HD + kk];
        }
        Pt[idx] = p;
        if (BWD) GRt[idx] = g;
    }
    // column values held in registers
    float Q[CW], GCr[CW], col[CW];
    const float vk = RANK1 ? par[a.o_v + k] : 0.f;
#pragma unroll
    for (int seg = 0; seg < CW; ++seg) {
        const int j = seg * 32 + lane;
        Q[seg] = NEG_BIG; GCr[seg] = 0.f; col[seg] = 0.f;
        if (j < N) {
            Q[seg] = RANK1 ? __fmul_rn(a.x[(size_t)b * N + j], vk) : a.Qtab[((size_t)b * N + j) * HD + k];
            if (BWD) GCr[seg] = a.GC[((size_t)b * N + j) * HD + k];
        }
    }
    // labels: bits -> float4 {rows 4rq..4rq+3} per column; diagonal and padding -> 0
    mbar_wait(bar, 0);
    for (int idx = tid; idx < (RT / 4) * NP; idx += blockDim.x) {
        const int rq = idx / NP, c = idx - rq * NP;
        float v[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int row = 4 * rq + r;
            v[r] = (row < nrows && c < N && c != r0 + row && ((stage[row * WP + (c >> 5)] >> (c & 31)) & 1u)) ? 1.f : 0.f;
        }
        labf[idx] = make_float4(v[0], v[1], v[2], v[3]);
    }
    __syncthreads();

    float lacc = 0.f;
    for (int rq = 0; rq < RT / 4; ++rq) {
        float P[4], G[4], row[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            P[r] = Pt[(4 * rq + r) * HD + k];
            G[r] = BWD ? GRt[(4 * rq + r) * HD + k] : 0.f;
            row[r] = 0.f;
        }
#pragma unroll
        for (int seg = 0; seg < CW; ++seg) {
            const float4 l4 = labf[rq * NP + seg * 32 + lane];
            const float l[4] = {l4.x, l4.y, l4.z, l4.w};
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const float t = fmaf(l[r], D, P[r]) + Q[seg];
                if (!BWD) {
                    const float h = fmaxf(t, 0.f);
                    row[r] += h;
                    col[seg] += h;
                } else {
                    const float v = t > 0.f ? (G[r] + GCr[seg]) : 0.f;
                    row[r] += v;
                    col[seg] += v;
                    lacc = fmaf(l[r], v, lacc);
                }
            }
        }
        const float tot = warp_rowsum4(row[0], row[1], row[2], row[3], lane);
        if ((lane & 7) == 0) RSt[(4 * rq + ((lane >> 4) & 1) * 2 + ((lane >> 3) & 1)) * HD + k] = tot;
    }
    // diagonal terms (l_ii = 0), computed with the same operation order as the sweep
    for (int r = lane; r < RT; r += 32) {
        float d = 0.f;
        if (r < nrows) {
            const int i = r0 + r;
            const float qi = RANK1 ? __fmul_rn(a.x[(size_t)b * N + i], vk) : a.Qtab[((size_t)b * N + i) * HD + k];
            const float t = fmaf(0.f, D, Pt[r * HD + k]) + qi;
            if (!BWD) d = fmaxf(t, 0.f);
            else d = t > 0.f ? (GRt[r * HD + k] + a.GC[((size_t)b * N + i) * HD + k]) : 0.f;
        }
        dg[r * HD + k] = d;
    }
    if (BWD) {
        const float ls = warp_sum(lacc);
        if (lane == 0) a.LSp[((size_t)b * a.S + s) * HD + k] = ls;
    }
    __syncthreads();   // sweep done: label tile is dead, RSt/dg complete
#pragma unroll
    for (int seg = 0; seg < CW; ++seg) {
        const int j = seg * 32 + lane;
        if (j < N) CSt[j * HD + k] = col[seg];
    }
    for (int idx = tid; idx < nrows * HD; idx += blockDim.x)
        a.RS[((size_t)b * N + r0) * HD + idx] = RSt[idx] - dg[idx];
    __syncthreads();
    float* cs = a.CSp + ((size_t)b * a.S + s) * N * HD;
    for (int idx = tid; idx < N * HD; idx += blockDim.x) {
        const int j = idx / HD, r = j - r0;
        float v = CSt[idx];
        if (r >= 0 && r < nrows) v -= dg[r * HD + (idx - j * HD)];
        cs[idx] = v;
    }
}

}  // namespace hdgnn
