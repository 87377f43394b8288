// Entity-grid kernels: the two big sweeps of a training step (model_2.py:161-188 forward and its
// backward).
//
//   ent_fwd2:  RS_i = sum_{j != i} relu(pre_ij)                       (complete rows)
//              CS_j = sum_{i in chunk, i != j} relu(pre_ij)           (per-chunk partial, slot layout below)
//   ent_bwd2:  v_ij = [pre_ij > 0] (GR_i + GC_j); the chunk's contribution to the first-layer weight
//              gradients is reduced inside the CTA:
//                  gpart[cta] = { db[k] = sum_i RSd_i[k],  dU[k] = sum_i x_i RSd_i[k],
//                                 dV[k] = sum_j x_j CSd_j[k],  LS[k] = sum_{l_ij = 1} v_ij[k] }
//              so nothing of size N x 20 leaves the SM.
//
// pre_ij[k] = x_i U[k] + x_j V[k] + b[k] + W_l[l_ij][k]  (rank-1 form of the 4 -> 20 layer,
// model_2.py:144,167-170).
//
// Work decomposition: the B*N grid rows of the batch form ONE global row list that is cut into
// gridDim.x equal chunks of R rows, so every CTA does the same amount of work whatever B and N are
// (grid = 2 CTAs per SM, one wave).  A chunk may straddle commits; each (commit, chunk)
// intersection is a "sub-tile" with its own column tables.  The chunk that holds row b*N is slot 0
// of commit b, the next chunk slot 1, ...: CSp is (B, SL, N, 20), and a consumer sums the slots
// first_slot .. last_slot of its commit (ent2_slots).  The label bitmap rows of a sub-tile are
// contiguous in HBM and staged by one 1-D TMA bulk copy.
#pragma once
#include "bits.cuh"
#include "sweep2.cuh"

namespace hdgnn {

struct Ent2Args {
    const uint32_t* bits; int WP;      // (B,N,WP) label bitmap
    int N, B, R, SL;                   // R = global rows per CTA, SL = column-partial slots per commit
    const float* params; const float* x;   // x (B,N)
    int o_u, o_v, o_b, o_l;
    const float* GR; const float* GC;  // bwd: (B,N,20) d/dRS, d/dCS
    float* RS; float* CSp;             // fwd: (B,N,20), (B,SL,N,20)
    float* gpart;                      // bwd: (gridDim.x, 80)
    int head;                          // fwd: first kernel of the step (bitmaps given): the weights come from the previous
                                       // step's optimizer kernel, so they too are read after pdl_wait()
};

// number of chunks that intersect commit b = slots to sum
__host__ __device__ __forceinline__ int ent2_slots(int b, int N, int R) {
    return (int)((((long long)(b + 1) * N - 1) / R) - (((long long)b * N) / R)) + 1;
}
__host__ __device__ __forceinline__ int ent2_max_slots(int N, int R) { return (N + R - 1) / R + 1; }

__host__ __device__ inline size_t ent2_smem_bytes(int CWT, int N, int R, int WP, bool bwd) {
    const int RC = R < N ? R : N;
    size_t off = (size_t)round_up(RC * WP * 4, 128);                      // bitmap rows
    off += (size_t)RC * PROW * 4;                                           // P01
    off += (size_t)RC * HD * 4 * (bwd ? 3 : 2);                             // rowacc, diag (, GRt)
    // unused column-combine scratch of the multi-row-group layouts: dropping it would change ent2_occupancy, hence the chunking
    // and the summation order of the dense path
    off += (size_t)CWT * 32 * HD * 4;
    off += (size_t)(5 * HD + HD + 3 * 8 * HD + 4 * HD + 2 * HD) * 4;       // weights, lsw, red, acc80, dvw+pad
    return off + 16;
}

// one row group of KG warps (rg = 0); launch bounds: 20 resident warps per SM
template <int CWT>
__global__ void __launch_bounds__(KG * 32, 4) ent_fwd2_kernel(const Ent2Args a) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int N = a.N, WP = a.WP, RC = a.R < N ? a.R : N;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, kg = warp % KG, rg = warp / KG;
    constexpr int NT = KG * 32;
    uint32_t* sbits = reinterpret_cast<uint32_t*>(smem);
    float* P01 = reinterpret_cast<float*>(smem + round_up(RC * WP * 4, 128));
    float* rowacc = P01 + (size_t)RC * PROW;
    float* diag = rowacc + (size_t)RC * HD;
    float* scratch = diag + (size_t)RC * HD;      // unused (ent2_smem_bytes)
    float* wts = scratch + (size_t)CWT * 32 * HD;   // U V bsum D
    uint64_t* bar = reinterpret_cast<uint64_t*>(wts + 5 * HD + HD + 3 * 8 * HD + 4 * HD + 2 * HD);

    if (tid == 0) { mbar_init(bar, 1); fence_mbar_init(); }
    if (a.head) pdl_wait();
    if (tid < HD) {
        const float* par = a.params;
        wts[tid] = par[a.o_u + tid]; wts[HD + tid] = par[a.o_v + tid];
        wts[2 * HD + tid] = par[a.o_b + tid] + par[a.o_l + tid];
        wts[3 * HD + tid] = par[a.o_l + HD + tid] - par[a.o_l + tid];
    }
    __syncthreads();
    pdl_wait();                     // the label bitmap comes from pack_bits
    pdl_launch_dependents();
    const int k0 = kg * 4;
    const float V0 = wts[HD + k0], V1 = wts[HD + k0 + 1], V2 = wts[HD + k0 + 2], V3 = wts[HD + k0 + 3];
    const int cw = (N + 31) >> 5, npass = (cw + CWT - 1) / CWT;
    const long long rows_total = (long long)a.B * N;
    long long g0 = (long long)blockIdx.x * a.R;
    const long long g1 = g0 + a.R < rows_total ? g0 + a.R : rows_total;
    uint32_t phase = 0;
    while (g0 < g1) {
        const int b = (int)(g0 / N), r0 = (int)(g0 - (long long)b * N);
        const int nr = (int)((g1 - g0) < (long long)(N - r0) ? (g1 - g0) : (long long)(N - r0));
        const int slot = (int)(blockIdx.x - ((long long)b * N) / a.R);
        const float* xb = a.x + (size_t)b * N;
        if (tid == 0) {
            const uint32_t bytes = (uint32_t)nr * WP * 4;
            mbar_arrive_expect_tx(bar, bytes);
            bulk_g2s(sbits, a.bits + ((size_t)b * N + r0) * WP, bytes, bar);
        }
        for (int base = tid; base < nr * HD; base += 4 * NT) {      // four elements per thread per trip: their loads overlap
            float xv[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) { const int idx = base + u * NT; xv[u] = idx < nr * HD ? xb[r0 + idx / HD] : 0.f; }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int idx = base + u * NT;
                if (idx < nr * HD) {
                    const int r = idx / HD, k = idx - r * HD;
                    const float xi = xv[u];
                    const float p0 = fmaf(xi, wts[k], wts[2 * HD + k]);
                    float* dst = P01 + (size_t)r * PROW + (k >> 2) * 8 + (k & 3);
                    dst[0] = p0; dst[4] = p0 + wts[3 * HD + k];
                    diag[idx] = fmaxf(fmaf(xi, wts[HD + k], p0), 0.f);
                }
            }
        }
        mbar_wait(bar, phase);
        phase ^= 1u;
        __syncthreads();
        float* csp = a.CSp + ((size_t)b * a.SL + slot) * N * HD;
        for (int pass = 0; pass < npass; ++pass) {
            u64 Q[CWT][2], col[CWT][2];
#pragma unroll
            for (int sg = 0; sg < CWT; ++sg) {
                const int j = (pass * CWT + sg) * 32 + lane;
                const bool ok = j < N;
                const float xj = ok ? xb[j] : 0.f;
                Q[sg][0] = ok ? pk2(xj * V0, xj * V1) : pk2(NEG_BIG, NEG_BIG);
                Q[sg][1] = ok ? pk2(xj * V2, xj * V3) : pk2(NEG_BIG, NEG_BIG);
                col[sg][0] = 0ull; col[sg][1] = 0ull;
            }
            if (pass == 0) sweep2_fwd<CWT, false>(P01, sbits, WP, nr, rg, 1, kg, Q, col, rowacc, lane);
            else sweep2_fwd<CWT, true>(P01, sbits + pass * CWT, WP, nr, rg, 1, kg, Q, col, rowacc, lane);
            if (rg == 0) {
#pragma unroll
                for (int sg = 0; sg < CWT; ++sg) {
                    const int j = (pass * CWT + sg) * 32 + lane;
                    if (j < N) {
                        float c0, c1, c2, c3;
                        upk2(col[sg][0], c0, c1); upk2(col[sg][1], c2, c3);
                        const int r = j - r0;
                        if (r >= 0 && r < nr) {
                            const float4 d = *reinterpret_cast<const float4*>(diag + (size_t)r * HD + k0);
                            c0 -= d.x; c1 -= d.y; c2 -= d.z; c3 -= d.w;
                        }
                        *reinterpret_cast<float4*>(csp + (size_t)j * HD + k0) = make_float4(c0, c1, c2, c3);
                    }
                }
            }
        }
        __syncthreads();
        for (int idx = tid; idx < nr * HD; idx += NT)
            a.RS[((size_t)b * N + r0) * HD + idx] = rowacc[idx] - diag[idx];
        __syncthreads();
        g0 += nr;
    }
}

template <int CWT>
__global__ void __launch_bounds__(KG * 32, 3) ent_bwd2_kernel(const Ent2Args a) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int N = a.N, WP = a.WP, RC = a.R < N ? a.R : N;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, kg = warp % KG, rg = warp / KG;
    constexpr int NT = KG * 32;
    uint32_t* sbits = reinterpret_cast<uint32_t*>(smem);
    float* P01 = reinterpret_cast<float*>(smem + round_up(RC * WP * 4, 128));
    float* rowacc = P01 + (size_t)RC * PROW;
    float* dgv = rowacc + (size_t)RC * HD;
    float* GRt = dgv + (size_t)RC * HD;
    float* scratch = GRt + (size_t)RC * HD;       // unused (ent2_smem_bytes)
    float* wts = scratch + (size_t)CWT * 32 * HD;   // U V bsum D (W unused slot)
    float* lsw = wts + 5 * HD;                  // [20]
    float* red = lsw + HD;                      // [3][8][20]
    float* acc80 = red + 3 * 8 * HD;            // [4][20] db dU dV LS over the CTA's sub-tiles
    float* dvw = acc80 + 4 * HD;                // [20] dV of the current sub-tile
    uint64_t* bar = reinterpret_cast<uint64_t*>(dvw + 2 * HD);

    if (tid == 0) { mbar_init(bar, 1); fence_mbar_init(); }
    if (tid < HD) {
        const float* par = a.params;
        wts[tid] = par[a.o_u + tid]; wts[HD + tid] = par[a.o_v + tid];
        wts[2 * HD + tid] = par[a.o_b + tid] + par[a.o_l + tid];
        wts[3 * HD + tid] = par[a.o_l + HD + tid] - par[a.o_l + tid];
    }
    if (tid < 4 * HD) acc80[tid] = 0.f;
    __syncthreads();
    pdl_wait();                     // GE comes from mid2
    pdl_launch_dependents();
    const int k0 = kg * 4;
    const float V0 = wts[HD + k0], V1 = wts[HD + k0 + 1], V2 = wts[HD + k0 + 2], V3 = wts[HD + k0 + 3];
    const int cw = (N + 31) >> 5, npass = (cw + CWT - 1) / CWT;
    const int ch = reduce4_channel(lane);
    const long long rows_total = (long long)a.B * N;
    long long g0 = (long long)blockIdx.x * a.R;
    const long long g1 = g0 + a.R < rows_total ? g0 + a.R : rows_total;
    uint32_t phase = 0;
    while (g0 < g1) {
        const int b = (int)(g0 / N), r0 = (int)(g0 - (long long)b * N);
        const int nr = (int)((g1 - g0) < (long long)(N - r0) ? (g1 - g0) : (long long)(N - r0));
        const float* xb = a.x + (size_t)b * N;
        const float* grb = a.GR + (size_t)b * N * HD;
        const float* gcb = a.GC + (size_t)b * N * HD;
        if (tid == 0) {
            const uint32_t bytes = (uint32_t)nr * WP * 4;
            mbar_arrive_expect_tx(bar, bytes);
            bulk_g2s(sbits, a.bits + ((size_t)b * N + r0) * WP, bytes, bar);
        }
        for (int base = tid; base < nr * HD; base += 4 * NT) {      // four elements per thread per trip: their loads overlap
            float xv[4], gv[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int idx = base + u * NT;
                const bool ok = idx < nr * HD;
                xv[u] = ok ? xb[r0 + idx / HD] : 0.f;
                gv[u] = ok ? grb[(size_t)r0 * HD + idx] : 0.f;          // GR = GC = d/dS of row r0 + idx / HD, channel idx % HD
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int idx = base + u * NT;
                if (idx < nr * HD) {
                    const int r = idx / HD, k = idx - r * HD;
                    const float xi = xv[u];
                    const float p0 = fmaf(xi, wts[k], wts[2 * HD + k]);
                    float* dst = P01 + (size_t)r * PROW + (k >> 2) * 8 + (k & 3);
                    dst[0] = p0; dst[4] = p0 + wts[3 * HD + k];
                    const float g = gv[u];
                    GRt[idx] = g;
                    dgv[idx] = fmaf(xi, wts[HD + k], p0) > 0.f ? g + (gcb == grb ? g : gcb[(size_t)(r0 + r) * HD + k]) : 0.f;
                }
            }
        }
        if (tid < HD) dvw[tid] = 0.f;
        mbar_wait(bar, phase);
        phase ^= 1u;
        __syncthreads();
        u64 lacc[2] = {0ull, 0ull};
        for (int pass = 0; pass < npass; ++pass) {
            u64 Q[CWT][2], GC[CWT][2], col[CWT][2];
#pragma unroll
            for (int sg = 0; sg < CWT; ++sg) {
                const int j = (pass * CWT + sg) * 32 + lane;
                const bool ok = j < N;
                const float xj = ok ? xb[j] : 0.f;
                Q[sg][0] = ok ? pk2(xj * V0, xj * V1) : pk2(NEG_BIG, NEG_BIG);
                Q[sg][1] = ok ? pk2(xj * V2, xj * V3) : pk2(NEG_BIG, NEG_BIG);
                ulonglong2 g = make_ulonglong2(0ull, 0ull);
                if (ok) g = *reinterpret_cast<const ulonglong2*>(gcb + (size_t)j * HD + k0);
                GC[sg][0] = g.x; GC[sg][1] = g.y;
                col[sg][0] = 0ull; col[sg][1] = 0ull;
            }
            if (pass == 0) sweep2_bwd<CWT, false>(P01, GRt, sbits, WP, nr, rg, 1, kg, Q, GC, col, lacc, rowacc, lane);
            else sweep2_bwd<CWT, true>(P01, GRt, sbits + pass * CWT, WP, nr, rg, 1, kg, Q, GC, col, lacc, rowacc, lane);
            if (rg == 0) {       // dV partial of this pass: sum_j x_j (col_j - diag_j)
                u64 dv0 = 0ull, dv1 = 0ull;
#pragma unroll
                for (int sg = 0; sg < CWT; ++sg) {
                    const int j = (pass * CWT + sg) * 32 + lane;
                    if (j < N) {
                        float c0, c1, c2, c3;
                        upk2(col[sg][0], c0, c1); upk2(col[sg][1], c2, c3);
                        const int r = j - r0;
                        if (r >= 0 && r < nr) {
                            const float4 d = *reinterpret_cast<const float4*>(dgv + (size_t)r * HD + k0);
                            c0 -= d.x; c1 -= d.y; c2 -= d.z; c3 -= d.w;
                        }
                        const float xj = xb[j];
                        const u64 x2 = pk2(xj, xj);
                        dv0 = fma2(x2, pk2(c0, c1), dv0); dv1 = fma2(x2, pk2(c2, c3), dv1);
                    }
                }
                const float t = reduce4(dv0, dv1, lane);
                if ((lane & 7) == 0) dvw[k0 + ch] += t;
            }
        }
        {   // label-1 sums: warp totals
            const float t = reduce4(lacc[0], lacc[1], lane);
            if ((lane & 7) == 0) lsw[rg * HD + k0 + ch] = t;
        }
        __syncthreads();
        // db, dU over the sub-tile's rows: 8 interleaved partials per channel, fixed order
        if (tid < 8 * HD) {
            const int p = tid / HD, k = tid - p * HD;
            float sb = 0.f, su = 0.f;
            for (int r = p; r < nr; r += 8) {
                const float rs = rowacc[r * HD + k] - dgv[r * HD + k];
                sb += rs;
                su = fmaf(xb[r0 + r], rs, su);
            }
            red[(0 * 8 + p) * HD + k] = sb; red[(1 * 8 + p) * HD + k] = su;
        }
        __syncthreads();
        if (tid < HD) {
            const int k = tid;
            float sb = 0.f, su = 0.f, ls = 0.f;
            for (int p = 0; p < 8; ++p) { sb += red[(0 * 8 + p) * HD + k]; su += red[(1 * 8 + p) * HD + k]; }
            ls += lsw[k];
            acc80[k] += sb; acc80[HD + k] += su; acc80[2 * HD + k] += dvw[k]; acc80[3 * HD + k] += ls;
        }
        __syncthreads();
        g0 += nr;
    }
    if (tid < 4 * HD) a.gpart[(size_t)blockIdx.x * 4 * HD + tid] = acc80[tid];
}

}  // namespace hdgnn
