// Node-level kernels: everything that is O(N * 20 * 20) per commit -- the linear second layers
// applied to the row/column sums, the entity-state MLP (model_2.py:190-205), the entity->hunk
// pooling (model_2.py:146-150 with the index semantics of utils2.py:111-137), the tables
// P/Q for the next pair sweep, and the hand-written backward of all of it including the
// per-commit weight-gradient partials.  One CTA per commit; nodes are processed in chunks of
// NCH so shared memory does not grow with N.  All reductions run in a fixed order.
#pragma once
#include "common.cuh"

namespace hdgnn {

constexpr int NCH = 128;          // nodes per shared-memory chunk
constexpr int NODE_THREADS = 512;

// ============================================================================================
// forward: entity-state MLP + pooling + hunk-stage tables
// ============================================================================================
struct PoolFwdArgs {
    int Ne, Nc, Se;
    int ent;                // entity-node branch present (variants 2, 4)
    const float* x;         // (B,Ne)
    const float* RS1;       // (B,Ne,20)
    const float* CS1p;      // (B,Se,Ne,20)
    const float* params;
    ParamOff po;
    const uint32_t* bits; int WP;   // (B,Ne,WP) entity label bitmap (bits.cuh)
    const float* soft;      // (B,Ne,Ne,2) soft edges (variant 4) or nullptr
    const int* hmap;        // (B,Ne)
    const int* L;           // (B)
    float* S1;              // (B,Ne,20)  RS1 + CS1 (complete)
    float* X2;              // (B,Ne)     updated node state x'
    float* NB;              // (B,Nc,4)
    float* PH;              // (B,Nc,20)
    float* QH;              // (B,Nc,20)
};

__host__ __device__ inline size_t pool_fwd_smem_bytes(int Ne, int Nc) {
    size_t f = 400 + 20 + 420 + 20 + 20 + 4 + 200 + 20;      // weights
    f += 3 * NCH * HD;                                       // sS, sE, sZ
    f += Ne + Ne + 8 * Ne + 4 * Nc;                          // x2s, hm, SP, TP, nbs
    return f * 4 + 16;
}

__global__ void __launch_bounds__(NODE_THREADS) pool_fwd_kernel(const PoolFwdArgs a) {
    extern __shared__ __align__(16) float sm[];
    const int Ne = a.Ne, Nc = a.Nc, b = blockIdx.x, tid = threadIdx.x;
    float* W5 = sm;            float* b5 = W5 + 400;   float* U1 = b5 + 20;   float* c1 = U1 + 420;
    float* u2 = c1 + 20;       float* c2 = u2 + 20;    float* V1 = c2 + 4;    float* d1 = V1 + 200;
    float* sS = d1 + 20;       float* sE = sS + NCH * HD;  float* sZ = sE + NCH * HD;
    float* x2s = sZ + NCH * HD;
    int* hm = reinterpret_cast<int*>(x2s + Ne);
    float* SP = reinterpret_cast<float*>(hm + Ne);
    float* TP = SP + 4 * Ne;
    float* nbs = TP + 4 * Ne;
    const float* par = a.params;
    const ParamOff& po = a.po;
    if (a.ent) {
        copy_to_smem(W5, par + po.ent_w5, 400); copy_to_smem(b5, par + po.ent_b5, 20);
        copy_to_smem(U1, par + po.nod_w1, 420); copy_to_smem(c1, par + po.nod_b1, 20);
        copy_to_smem(u2, par + po.nod_w2, 20);  copy_to_smem(c2, par + po.nod_b2, 1);
    }
    copy_to_smem(V1, par + po.hnk_w1, 200); copy_to_smem(d1, par + po.hnk_b1, 20);
    const int Lb = min(max(a.L[b], 0), Ne);      // 0 <= L <= Ne is the ABI's contract; clamped so a bad value cannot index out of the tile
    for (int i = tid; i < Ne; i += blockDim.x) {
        const int h = a.hmap[(size_t)b * Ne + i];
        hm[i] = (h >= 0 && h < Nc) ? h : -1;
        if (!a.ent) x2s[i] = a.x[(size_t)b * Ne + i];
    }
    __syncthreads();
    if (a.ent) {
        const float nb5 = 2.f * (float)(Ne - 1);
        for (int c0 = 0; c0 < Ne; c0 += NCH) {
            const int nn = min(NCH, Ne - c0);
            for (int idx = tid; idx < nn * HD; idx += blockDim.x) {
                const size_t g = ((size_t)b * Ne + c0) * HD + idx;
                float v = a.RS1[g];
                for (int s = 0; s < a.Se; ++s) v += a.CS1p[((size_t)b * a.Se + s) * Ne * HD + (size_t)c0 * HD + idx];
                sS[idx] = v;
                a.S1[g] = v;
            }
            __syncthreads();
            for (int idx = tid; idx < nn * HD; idx += blockDim.x) {
                const int n = idx / HD, m = idx - n * HD;
                float acc = nb5 * b5[m];
#pragma unroll
                for (int q = 0; q < HD; ++q) acc = fmaf(sS[n * HD + q], W5[q * HD + m], acc);
                sE[idx] = acc;
            }
            __syncthreads();
            for (int idx = tid; idx < nn * HD; idx += blockDim.x) {
                const int n = idx / HD, k = idx - n * HD;
                float acc = fmaf(a.x[(size_t)b * Ne + c0 + n], U1[k], c1[k]);
#pragma unroll
                for (int m = 0; m < HD; ++m) acc = fmaf(sE[n * HD + m], U1[(1 + m) * HD + k], acc);
                sZ[idx] = fmaxf(acc, 0.f);
            }
            __syncthreads();
            for (int n = tid; n < nn; n += blockDim.x) {
                float acc = c2[0];
#pragma unroll
                for (int k = 0; k < HD; ++k) acc = fmaf(sZ[n * HD + k], u2[k], acc);
                const float v = fmaxf(acc, 0.f);
                x2s[c0 + n] = v;
                a.X2[(size_t)b * Ne + c0 + n] = v;
            }
            __syncthreads();
        }
    }
    // ---- pooling: row sums SP_i' and column sums TP_j' of B2[q] over the L x L local grid,
    //      where q indexes the Ne-grid enumeration (quirk Q3, utils2.py:123-137) -------------
    const int nm1 = Ne - 1;
    const float inv = 1.f / (float)nm1;
    for (int task = tid; task < 2 * Lb; task += blockDim.x) {
        const bool colpass = task >= Lb;
        const int me = colpass ? task - Lb : task;
        float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
        for (int o = 0; o < Lb; ++o) {
            if (o == me) continue;
            const int li = colpass ? o : me, lj = colpass ? me : o;
            const int q = li * (Lb - 1) + lj - (lj > li);
            int gi, gj;
            if (Lb == Ne) { gi = li; gj = lj; }
            else unflat_pair(q, nm1, inv, gi, gj);
            float v2, v3;
            if (a.soft) {
                const float2 s2 = reinterpret_cast<const float2*>(a.soft)[((size_t)b * Ne + gi) * Ne + gj];
                v2 = s2.x; v3 = s2.y;
            } else {
                v3 = (a.bits[((size_t)b * Ne + gi) * a.WP + (gj >> 5)] >> (gj & 31)) & 1u ? 1.f : 0.f;
                v2 = 1.f - v3;
            }
            acc0 += x2s[gi]; acc1 += x2s[gj]; acc2 += v2; acc3 += v3;
        }
        float* dst = (colpass ? TP : SP) + 4 * me;
        dst[0] = acc0; dst[1] = acc1; dst[2] = acc2; dst[3] = acc3;
    }
    __syncthreads();
    // ---- segmented reduce by hunk id, ascending entity line order (deterministic) ----------
    for (int idx = tid; idx < Nc * 4; idx += blockDim.x) {
        const int c = idx >> 2, ch = idx & 3;
        float acc = 0.f;
        for (int i = 0; i < Lb; ++i)
            if (hm[i] == c) acc += SP[4 * i + ch] + TP[4 * i + ch];
        nbs[idx] = acc;
        a.NB[(size_t)b * Nc * 4 + idx] = acc;
    }
    __syncthreads();
    // ---- tables of the hunk pair layer (model_2.py:257-260): rows 0-3 source, 4-7 target,
    //      8/9 label one-hot; bias and the label-0 row are folded into PH ----------------------
    for (int idx = tid; idx < Nc * HD; idx += blockDim.x) {
        const int c = idx / HD, k = idx - c * HD;
        float p = d1[k] + V1[8 * HD + k], q = 0.f;
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
            p = fmaf(nbs[4 * c + ch], V1[ch * HD + k], p);
            q = fmaf(nbs[4 * c + ch], V1[(4 + ch) * HD + k], q);
        }
        a.PH[(size_t)b * Nc * HD + idx] = p;
        a.QH[(size_t)b * Nc * HD + idx] = q;
    }
}

// ============================================================================================
// forward: linear second layer on the sums + tables of the head  (model_2.py:263-275, 311-315)
// ============================================================================================
struct HeadFwdArgs {
    int N, S;
    const float* RS;        // (B,N,20)
    const float* CSp;       // (B,S,N,20)
    const float* params;
    HeadOff ho;
    float* CSf;             // (B,N,20) complete column sums
    float* PR;              // (B,N,20)
    float* PC;              // (B,N,20)
};

__host__ __device__ inline size_t head_fwd_smem_bytes() { return (size_t)(400 + 20 + 440 + 20 + 4 * NCH * HD) * 4 + 16; }

__global__ void __launch_bounds__(NODE_THREADS) head_fwd_kernel(const HeadFwdArgs a) {
    extern __shared__ __align__(16) float sm[];
    const int N = a.N, b = blockIdx.x, tid = threadIdx.x;
    float* W2 = sm; float* b2 = W2 + 400; float* G1 = b2 + 20; float* g1b = G1 + 440;
    float* sR = g1b + 20; float* sC = sR + NCH * HD; float* rr = sC + NCH * HD; float* cc = rr + NCH * HD;
    const float* par = a.params;
    copy_to_smem(W2, par + a.ho.w2p, 400); copy_to_smem(b2, par + a.ho.b2p, 20);
    copy_to_smem(G1, par + a.ho.w1h, 440); copy_to_smem(g1b, par + a.ho.b1h, 20);
    __syncthreads();
    const float nm1 = (float)(N - 1);
    for (int c0 = 0; c0 < N; c0 += NCH) {
        const int nn = min(NCH, N - c0);
        for (int idx = tid; idx < nn * HD; idx += blockDim.x) {
            const size_t g = ((size_t)b * N + c0) * HD + idx;
            sR[idx] = a.RS[g];
            float v = 0.f;
            for (int s = 0; s < a.S; ++s) v += a.CSp[((size_t)b * a.S + s) * N * HD + (size_t)c0 * HD + idx];
            sC[idx] = v;
            a.CSf[g] = v;
        }
        __syncthreads();
        for (int idx = tid; idx < nn * HD; idx += blockDim.x) {
            const int n = idx / HD, m = idx - n * HD;
            float r = nm1 * b2[m], c = r;
#pragma unroll
            for (int q = 0; q < HD; ++q) {
                r = fmaf(sR[n * HD + q], W2[q * HD + m], r);
                c = fmaf(sC[n * HD + q], W2[q * HD + m], c);
            }
            rr[idx] = r; cc[idx] = c;
        }
        __syncthreads();
        for (int idx = tid; idx < nn * HD; idx += blockDim.x) {
            const int n = idx / HD, k = idx - n * HD;
            float p = g1b[k] + G1[k], q = 0.f;
#pragma unroll
            for (int m = 0; m < HD; ++m) {
                p = fmaf(rr[n * HD + m], G1[(2 + m) * HD + k], p);
                q = fmaf(cc[n * HD + m], G1[(2 + m) * HD + k], q);
            }
            const size_t g = ((size_t)b * N + c0) * HD + idx;
            a.PR[g] = p; a.PC[g] = q;
        }
        __syncthreads();
    }
}

// mean CE: fixed-order sum of the per-tile partials (model_2.py:115-118)
__global__ void loss_reduce_kernel(const float* cep, int n, float denom, float* loss) {
    __shared__ float scratch[32];
    float acc = 0.f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) acc += cep[i];
    const float t = block_sum(acc, scratch);
    if (threadIdx.x == 0) *loss = t / denom;
}

// ============================================================================================
// backward of head_fwd + the head's weights
// ============================================================================================
struct HeadBwdArgs {
    int N, S;
    const float* RSm;  const float* CSmp;  const float* LSmp;  const float* HSp;  const float* dsump;
    const float* RS;   const float* CSf;   // forward sums of the pair layer
    const float* params;
    HeadOff ho;
    float* gpart;      // (B, total) per-commit gradient partials
    int total;
    float* GR;         // (B,N,20) d/dRS
    float* GC;         // (B,N,20) d/dCS
};

__host__ __device__ inline size_t head_bwd_smem_bytes() { return (size_t)(400 + 20 + 400 + 20 + 64 + 8 * NCH * HD) * 4 + 16; }

__global__ void __launch_bounds__(NODE_THREADS) head_bwd_kernel(const HeadBwdArgs a) {
    extern __shared__ __align__(16) float sm[];
    const int N = a.N, S = a.S, b = blockIdx.x, tid = threadIdx.x;
    float* W2 = sm; float* b2 = W2 + 400; float* G1e = b2 + 20; float* gam = G1e + 400; float* red = gam + 20;
    float* sRS4 = red + 64; float* sCS4 = sRS4 + NCH * HD; float* sR3 = sCS4 + NCH * HD; float* sC3 = sR3 + NCH * HD;
    float* rr = sC3 + NCH * HD; float* cc = rr + NCH * HD; float* dr = cc + NCH * HD; float* dc = dr + NCH * HD;
    const float* par = a.params;
    copy_to_smem(W2, par + a.ho.w2p, 400); copy_to_smem(b2, par + a.ho.b2p, 20);
    copy_to_smem(G1e, par + a.ho.w1h + 2 * HD, 400);
    if (tid < HD) gam[tid] = par[a.ho.w2h + 2 * tid + 1] - par[a.ho.w2h + 2 * tid];
    __syncthreads();
    const float nm1 = (float)(N - 1);
    float accA = 0.f, accB = 0.f;       // tid<400: dG1e[m][k], dW2p[a][m];  400..419: db1h[k];  420..439: db2p[m]
    for (int c0 = 0; c0 < N; c0 += NCH) {
        const int nn = min(NCH, N - c0);
        for (int idx = tid; idx < nn * HD; idx += blockDim.x) {
            const int k = idx % HD;
            const size_t g = ((size_t)b * N + c0) * HD + idx;
            sRS4[idx] = gam[k] * a.RSm[g];
            float v = 0.f;
            for (int s = 0; s < S; ++s) v += a.CSmp[((size_t)b * S + s) * N * HD + (size_t)c0 * HD + idx];
            sCS4[idx] = gam[k] * v;
            sR3[idx] = a.RS[g];
            sC3[idx] = a.CSf[g];
        }
        __syncthreads();
        for (int idx = tid; idx < nn * HD; idx += blockDim.x) {
            const int n = idx / HD, m = idx - n * HD;
            float r = nm1 * b2[m], c = r, d1 = 0.f, d2 = 0.f;
#pragma unroll
            for (int q = 0; q < HD; ++q) {
                r = fmaf(sR3[n * HD + q], W2[q * HD + m], r);
                c = fmaf(sC3[n * HD + q], W2[q * HD + m], c);
                d1 = fmaf(G1e[m * HD + q], sRS4[n * HD + q], d1);
                d2 = fmaf(G1e[m * HD + q], sCS4[n * HD + q], d2);
            }
            rr[idx] = r; cc[idx] = c; dr[idx] = d1; dc[idx] = d2;
        }
        __syncthreads();
        if (tid < 400) {
            const int p = tid / HD, q = tid - p * HD;
            for (int n = 0; n < nn; ++n) {
                accA = fmaf(rr[n * HD + p], sRS4[n * HD + q], accA);
                accA = fmaf(cc[n * HD + p], sCS4[n * HD + q], accA);
                accB = fmaf(sR3[n * HD + p], dr[n * HD + q], accB);
                accB = fmaf(sC3[n * HD + p], dc[n * HD + q], accB);
            }
        } else if (tid < 420) {
            const int k = tid - 400;
            for (int n = 0; n < nn; ++n) accA += sRS4[n * HD + k];
        } else if (tid < 440) {
            const int m = tid - 420;
            for (int n = 0; n < nn; ++n) accA += dr[n * HD + m] + dc[n * HD + m];
        }
        for (int idx = tid; idx < nn * HD; idx += blockDim.x) {
            const int n = idx / HD, q = idx - n * HD;
            float gr = 0.f, gc = 0.f;
#pragma unroll
            for (int m = 0; m < HD; ++m) {
                gr = fmaf(W2[q * HD + m], dr[n * HD + m], gr);
                gc = fmaf(W2[q * HD + m], dc[n * HD + m], gc);
            }
            const size_t g = ((size_t)b * N + c0) * HD + idx;
            a.GR[g] = gr; a.GC[g] = gc;
        }
        __syncthreads();
    }
    float* gp = a.gpart + (size_t)b * a.total;
    if (tid < 400) {
        gp[a.ho.w1h + 2 * HD + tid] = accA;
        gp[a.ho.w2p + tid] = accB;
    } else if (tid < 420) {
        const int k = tid - 400;
        float ls = 0.f, hs = 0.f;
        for (int s = 0; s < S; ++s) { ls += a.LSmp[((size_t)b * S + s) * HD + k]; hs += a.HSp[((size_t)b * S + s) * HD + k]; }
        ls *= gam[k];
        gp[a.ho.b1h + k] = accA;
        gp[a.ho.w1h + HD + k] = ls;
        gp[a.ho.w1h + k] = accA - ls;
        gp[a.ho.w2h + 2 * k + 1] = hs;
        gp[a.ho.w2h + 2 * k] = -hs;
    } else if (tid < 440) {
        gp[a.ho.b2p + (tid - 420)] = nm1 * accA;
    } else if (tid == 440) {
        float ds = 0.f;
        for (int s = 0; s < S; ++s) ds += a.dsump[(size_t)b * S + s];
        gp[a.ho.b2h + 1] = ds;
        gp[a.ho.b2h] = -ds;
    }
}

// ============================================================================================
// backward: hunk pair-layer weights, pooling, entity-state MLP
// ============================================================================================
struct PoolBwdArgs {
    int Ne, Nc, Sc;
    int ent;
    const float* RS3D; const float* CS3Dp; const float* LS3p;   // pairsum-bwd outputs on the hunk grid
    const float* NB;
    const float* x; const float* S1; const float* X2;
    const float* params;
    ParamOff po;
    const int* hmap; const int* L;
    float* gpart; int total;
    float* DNB;        // (B,Nc,4)
    float* GE;         // (B,Ne,20)  d/dRS1 = d/dCS1
    float* DX2;        // (B,Ne)     debug
    float* dsoft;      // (B,Ne,Ne,2) d/d(soft edge) for variant 4, or nullptr
};

__host__ __device__ inline size_t pool_bwd_smem_bytes(int Ne, int Nc) {
    size_t f = 400 + 20 + 420 + 20 + 20 + 4 + 200 + 20;
    f += 5 * NCH * HD;                 // chunk arrays
    f += NCH;                          // sdu
    f += 4 * Nc + 4 * Nc;              // nbs, dnbs
    f += 4 * Ne + Ne + Ne;             // dl, dx2, hm
    return f * 4 + 16;
}

__global__ void __launch_bounds__(NODE_THREADS) pool_bwd_kernel(const PoolBwdArgs a) {
    extern __shared__ __align__(16) float sm[];
    const int Ne = a.Ne, Nc = a.Nc, Sc = a.Sc, b = blockIdx.x, tid = threadIdx.x;
    float* W5 = sm;            float* b5 = W5 + 400;   float* U1 = b5 + 20;   float* c1 = U1 + 420;
    float* u2 = c1 + 20;       float* c2 = u2 + 20;    float* V1 = c2 + 4;    float* d1 = V1 + 200;
    float* A0 = d1 + 20;       float* A1 = A0 + NCH * HD; float* A2 = A1 + NCH * HD;
    float* A3 = A2 + NCH * HD; float* A4 = A3 + NCH * HD; float* sdu = A4 + NCH * HD;
    float* nbs = sdu + NCH;    float* dnbs = nbs + 4 * Nc;
    float* dl = dnbs + 4 * Nc; float* dx2 = dl + 4 * Ne;
    int* hm = reinterpret_cast<int*>(dx2 + Ne);
    const float* par = a.params;
    const ParamOff& po = a.po;
    if (a.ent) {
        copy_to_smem(W5, par + po.ent_w5, 400); copy_to_smem(b5, par + po.ent_b5, 20);
        copy_to_smem(U1, par + po.nod_w1, 420); copy_to_smem(c1, par + po.nod_b1, 20);
        copy_to_smem(u2, par + po.nod_w2, 20);  copy_to_smem(c2, par + po.nod_b2, 1);
    }
    copy_to_smem(V1, par + po.hnk_w1, 200);
    copy_to_smem(nbs, a.NB + (size_t)b * Nc * 4, Nc * 4);
    const int Lb = min(max(a.L[b], 0), Ne);      // 0 <= L <= Ne is the ABI's contract; clamped so a bad value cannot index out of the tile
    for (int i = tid; i < Ne; i += blockDim.x) {
        const int h = a.hmap[(size_t)b * Ne + i];
        hm[i] = (h >= 0 && h < Nc) ? h : -1;
    }
    __syncthreads();
    float* gp = a.gpart + (size_t)b * a.total;

    // ---- part 1: hunk pair layer first-layer weights + d/dnb --------------------------------
    {
        float acc = 0.f;      // tid<160: dV1[row<8][k]; 160..179: db[k]
        float* sRd = A0; float* sCd = A1;
        for (int c0 = 0; c0 < Nc; c0 += NCH) {
            const int nn = min(NCH, Nc - c0);
            for (int idx = tid; idx < nn * HD; idx += blockDim.x) {
                const size_t g = ((size_t)b * Nc + c0) * HD + idx;
                sRd[idx] = a.RS3D[g];
                float v = 0.f;
                for (int s = 0; s < Sc; ++s) v += a.CS3Dp[((size_t)b * Sc + s) * Nc * HD + (size_t)c0 * HD + idx];
                sCd[idx] = v;
            }
            __syncthreads();
            if (tid < 160) {
                const int row = tid / HD, k = tid - row * HD;
                const float* src = row < 4 ? sRd : sCd;
                const int ch = row & 3;
                for (int n = 0; n < nn; ++n) acc = fmaf(nbs[4 * (c0 + n) + ch], src[n * HD + k], acc);
            } else if (tid < 180) {
                const int k = tid - 160;
                for (int n = 0; n < nn; ++n) acc += sRd[n * HD + k];
            }
            for (int idx = tid; idx < nn * 4; idx += blockDim.x) {
                const int n = idx >> 2, ch = idx & 3;
                float v = 0.f;
#pragma unroll
                for (int k = 0; k < HD; ++k) {
                    v = fmaf(V1[ch * HD + k], sRd[n * HD + k], v);
                    v = fmaf(V1[(4 + ch) * HD + k], sCd[n * HD + k], v);
                }
                dnbs[4 * (c0 + n) + ch] = v;
                a.DNB[((size_t)b * Nc + c0) * 4 + idx] = v;
            }
            __syncthreads();
        }
        if (tid < 160) gp[po.hnk_w1 + tid] = acc;
        else if (tid < 180) {
            const int k = tid - 160;
            float ls = 0.f;
            for (int s = 0; s < Sc; ++s) ls += a.LS3p[((size_t)b * Sc + s) * HD + k];
            gp[po.hnk_b1 + k] = acc;
            gp[po.hnk_w1 + 9 * HD + k] = ls;
            gp[po.hnk_w1 + 8 * HD + k] = acc - ls;
        }
    }
    if (!a.ent && !a.dsoft) return;

    // ---- part 2: pooling backward.  dB2[q] = dnb[hunk(i')] + dnb[hunk(j')] for q < L(L-1) ------
    for (int idx = tid; idx < Ne * 4; idx += blockDim.x) {
        const int i = idx >> 2, ch = idx & 3;
        dl[idx] = (i < Lb && hm[i] >= 0) ? dnbs[4 * hm[i] + ch] : 0.f;
    }
    __syncthreads();
    {
        const int lm1 = Lb - 1, nm1 = Ne - 1, qmax = Lb * lm1;
        const float invl = 1.f / (float)lm1;
        for (int task = tid; task < 2 * Ne; task += blockDim.x) {
            const bool colpass = task >= Ne;
            const int me = colpass ? task - Ne : task;
            float acc = 0.f;
            for (int o = 0; o < Ne; ++o) {
                if (o == me) continue;
                const int gi = colpass ? o : me, gj = colpass ? me : o;
                const int q = gi * nm1 + gj - (gj > gi);
                float w0 = 0.f, w1 = 0.f, w2 = 0.f, w3 = 0.f;
                if (q < qmax) {
                    int li, lj;
                    if (Lb == Ne) { li = gi; lj = gj; }
                    else unflat_pair(q, lm1, invl, li, lj);
                    w0 = dl[4 * li + 0] + dl[4 * lj + 0];
                    w1 = dl[4 * li + 1] + dl[4 * lj + 1];
                    if (a.dsoft && !colpass) { w2 = dl[4 * li + 2] + dl[4 * lj + 2]; w3 = dl[4 * li + 3] + dl[4 * lj + 3]; }
                }
                acc += colpass ? w1 : w0;
                if (a.dsoft && !colpass)
                    reinterpret_cast<float2*>(a.dsoft)[((size_t)b * Ne + gi) * Ne + gj] = make_float2(w2, w3);
            }
            if (colpass) A0[me] = acc; else dx2[me] = acc;       // A0 used as scratch (Ne <= NCH*HD)
        }
        __syncthreads();
        for (int n = tid; n < Ne; n += blockDim.x) {
            dx2[n] += A0[n];
            if (a.DX2) a.DX2[(size_t)b * Ne + n] = dx2[n];
        }
        __syncthreads();
    }
    if (!a.ent) return;

    // ---- part 3: entity-state MLP backward (model_2.py:190-205) and W5/b5 (model_2.py:172-175) -
    {
        float* sS = A0; float* sE = A1; float* sZp = A2; float* sDz = A3; float* sDE = A4;
        const float nb5 = 2.f * (float)(Ne - 1);
        float acc0 = 0.f, acc1 = 0.f;   // entry e = tid and tid + 512, e < 881
        for (int c0 = 0; c0 < Ne; c0 += NCH) {
            const int nn = min(NCH, Ne - c0);
            for (int idx = tid; idx < nn * HD; idx += blockDim.x) sS[idx] = a.S1[((size_t)b * Ne + c0) * HD + idx];
            __syncthreads();
            for (int idx = tid; idx < nn * HD; idx += blockDim.x) {
                const int n = idx / HD, m = idx - n * HD;
                float acc = nb5 * b5[m];
#pragma unroll
                for (int q = 0; q < HD; ++q) acc = fmaf(sS[n * HD + q], W5[q * HD + m], acc);
                sE[idx] = acc;
            }
            __syncthreads();
            for (int idx = tid; idx < nn * HD; idx += blockDim.x) {
                const int n = idx / HD, k = idx - n * HD;
                float acc = fmaf(a.x[(size_t)b * Ne + c0 + n], U1[k], c1[k]);
#pragma unroll
                for (int m = 0; m < HD; ++m) acc = fmaf(sE[n * HD + m], U1[(1 + m) * HD + k], acc);
                sZp[idx] = acc;
            }
            __syncthreads();
            for (int n = tid; n < nn; n += blockDim.x)
                sdu[n] = a.X2[(size_t)b * Ne + c0 + n] > 0.f ? dx2[c0 + n] : 0.f;
            __syncthreads();
            for (int idx = tid; idx < nn * HD; idx += blockDim.x) {
                const int n = idx / HD, k = idx - n * HD;
                sDz[idx] = sZp[idx] > 0.f ? sdu[n] * u2[k] : 0.f;
            }
            __syncthreads();
            for (int idx = tid; idx < nn * HD; idx += blockDim.x) {
                const int n = idx / HD, m = idx - n * HD;
                float acc = 0.f;
#pragma unroll
                for (int k = 0; k < HD; ++k) acc = fmaf(U1[(1 + m) * HD + k], sDz[n * HD + k], acc);
                sDE[idx] = acc;
            }
            __syncthreads();
#pragma unroll
            for (int rep = 0; rep < 2; ++rep) {
                const int e = tid + rep * NODE_THREADS;
                float acc = 0.f;
                if (e < 400) {                       // dU1[1+m][k]
                    const int m = e / HD, k = e - m * HD;
                    for (int n = 0; n < nn; ++n) acc = fmaf(sE[n * HD + m], sDz[n * HD + k], acc);
                } else if (e < 420) {                // dU1[0][k]
                    const int k = e - 400;
                    for (int n = 0; n < nn; ++n) acc = fmaf(a.x[(size_t)b * Ne + c0 + n], sDz[n * HD + k], acc);
                } else if (e < 440) {                // dc1[k]
                    const int k = e - 420;
                    for (int n = 0; n < nn; ++n) acc += sDz[n * HD + k];
                } else if (e < 460) {                // du2[k]
                    const int k = e - 440;
                    for (int n = 0; n < nn; ++n) acc = fmaf(sdu[n], fmaxf(sZp[n * HD + k], 0.f), acc);
                } else if (e == 460) {               // dc2
                    for (int n = 0; n < nn; ++n) acc += sdu[n];
                } else if (e < 861) {                // dW5[a][m]
                    const int q = (e - 461) / HD, m = (e - 461) - q * HD;
                    for (int n = 0; n < nn; ++n) acc = fmaf(sS[n * HD + q], sDE[n * HD + m], acc);
                } else if (e < 881) {                // db5[m]
                    const int m = e - 861;
                    for (int n = 0; n < nn; ++n) acc += sDE[n * HD + m];
                    acc *= nb5;
                }
                if (rep == 0) acc0 += acc; else acc1 += acc;
            }
            for (int idx = tid; idx < nn * HD; idx += blockDim.x) {
                const int n = idx / HD, q = idx - n * HD;
                float acc = 0.f;
#pragma unroll
                for (int m = 0; m < HD; ++m) acc = fmaf(W5[q * HD + m], sDE[n * HD + m], acc);
                a.GE[((size_t)b * Ne + c0) * HD + idx] = acc;
            }
            __syncthreads();
        }
#pragma unroll
        for (int rep = 0; rep < 2; ++rep) {
            const int e = tid + rep * NODE_THREADS;
            const float v = rep == 0 ? acc0 : acc1;
            if (e < 400) gp[po.nod_w1 + HD + e] = v;
            else if (e < 420) gp[po.nod_w1 + (e - 400)] = v;
            else if (e < 440) gp[po.nod_b1 + (e - 420)] = v;
            else if (e < 460) gp[po.nod_w2 + (e - 440)] = v;
            else if (e == 460) gp[po.nod_b2] = v;
            else if (e < 861) gp[po.ent_w5 + (e - 461)] = v;
            else if (e < 881) gp[po.ent_b5 + (e - 861)] = v;
        }
    }
}

// ============================================================================================
// backward: first-layer weights of a RANK1 pair layer  (entity effects model_2.py:167-170;
// entity-edge model_4.py:219-225 with the tied node row)
// ============================================================================================
struct Rank1GradArgs {
    int N, S;
    const float* x; const float* RSd; const float* CSdp; const float* LSp;
    int o_u, o_v, o_b, o_l;   // o_u == o_v  => tied (gradients added)
    float* gpart; int total;
};

__global__ void __launch_bounds__(256) rank1_grad_kernel(const Rank1GradArgs a) {
    __shared__ float part[3][8][HD];
    const int N = a.N, S = a.S, b = blockIdx.x, tid = threadIdx.x;
    if (tid < 8 * HD) {
        const int p = tid / HD, k = tid - p * HD;
        float sb = 0.f, su = 0.f, sv = 0.f;
        for (int n = p; n < N; n += 8) {
            const float xv = a.x[(size_t)b * N + n];
            const float r = a.RSd[((size_t)b * N + n) * HD + k];
            float c = 0.f;
            for (int s = 0; s < S; ++s) c += a.CSdp[((size_t)b * S + s) * N * HD + (size_t)n * HD + k];
            sb += r;
            su = fmaf(xv, r, su);
            sv = fmaf(xv, c, sv);
        }
        part[0][p][k] = sb; part[1][p][k] = su; part[2][p][k] = sv;
    }
    __syncthreads();
    if (tid < HD) {
        const int k = tid;
        float sb = 0.f, su = 0.f, sv = 0.f, ls = 0.f;
        for (int p = 0; p < 8; ++p) { sb += part[0][p][k]; su += part[1][p][k]; sv += part[2][p][k]; }
        for (int s = 0; s < S; ++s) ls += a.LSp[((size_t)b * S + s) * HD + k];
        float* gp = a.gpart + (size_t)b * a.total;
        gp[a.o_b + k] = sb;
        gp[a.o_l + HD + k] = ls;
        gp[a.o_l + k] = sb - ls;
        if (a.o_u == a.o_v) gp[a.o_u + k] = su + sv;
        else { gp[a.o_u + k] = su; gp[a.o_v + k] = sv; }
    }
}

// ============================================================================================
// gradient reduction over commits, regularisers, TF1 Adam
// ============================================================================================
__global__ void grad_reduce_kernel(const float* gpart, int B, int total, float* grads) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= total) return;
    float acc = 0.f;
    int b = 0;
    for (; b + 7 < B; b += 8) {          // eight loads in flight, fixed summation order
        float g[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) g[u] = gpart[(size_t)(b + u) * total + p];
#pragma unroll
        for (int u = 0; u < 8; ++u) acc += g[u];
    }
    for (; b < B; ++b) acc += gpart[(size_t)b * total + p];
    grads[p] = acc;
}

// regularisers: model_2.py:121-130 (0.001 * l2_loss over ALL variables) and 326-336
// (0.1 * 0.01 * (|theta1| + |theta2|)); Adam: tf.train.AdamOptimizer(3e-4), model_2.py:337.
__global__ void __launch_bounds__(1024) adam_kernel(float* p, const float* g, float* m, float* v, int n,
                                                    int o_t1, int o_t2, int* step, float lr, float b1,
                                                    float b2, float eps, float* reg_losses) {
    __shared__ float scratch[32];
    __shared__ float tn[3];
    const int tid = threadIdx.x;
    const int t = *step + 1;
    if (tid < 2) {
        const int o = tid == 0 ? o_t1 : o_t2;
        tn[tid] = sqrtf(p[o] * p[o] + p[o + 1] * p[o + 1]);
    }
    if (tid == 32) {       // 1 - b^t = -expm1(t log b): full float precision without the fp64 pipe
        const float omb2 = -expm1f((float)t * logf(b2)), omb1 = -expm1f((float)t * logf(b1));
        tn[2] = lr * sqrtf(omb2) / omb1;
    }
    float sq = 0.f;
    for (int i = tid; i < n; i += blockDim.x) sq = fmaf(p[i], p[i], sq);
    const float l2 = block_sum(sq, scratch);
    __syncthreads();
    if (tid == 0 && reg_losses) {
        reg_losses[0] = 0.01f * (tn[0] + tn[1]);
        reg_losses[1] = 0.001f * 0.5f * l2;
    }
    const float lr_t = tn[2];
    for (int i = tid; i < n; i += blockDim.x) {
        float gi = g[i] + 0.001f * p[i];
        if (i >= o_t1 && i < o_t1 + 2) gi += 0.001f * p[i] / tn[0];
        if (i >= o_t2 && i < o_t2 + 2) gi += 0.001f * p[i] / tn[1];
        const float mi = b1 * m[i] + (1.f - b1) * gi;
        const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
        m[i] = mi; v[i] = vi;
        p[i] -= lr_t * mi / (sqrtf(vi) + eps);
    }
    __syncthreads();
    if (tid == 0) *step = t;
}

}  // namespace hdgnn
