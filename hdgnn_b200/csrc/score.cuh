// score: the all-pairs relation head  (model_2.py:304-324 mlp_hunkedge_B2 on the hunk grid;
// model_4.py:286-304 mlp2_entityedge_B1 on the entity grid), fused with the softmax, the
// cross-entropy (model_2.py:115-118) and -- when training -- the first half of its backward.
//
//   pre_st[k]  = PR_s[k] + PC_t[k] + l_st * D[k]       (the 22->20 layer in separable form; the
//                                                      20-d "effect" r_s + c_t is never built)
//   logit_st   = W2^T relu(pre_st) + b2  (2 classes),  prob = softmax,  CE_st = -log prob[l_st]
//
// Pass 1 (thread = pair): logits / probs / CE, and delta_st = dL/dlogit1 = -dL/dlogit0 into a
//         shared-memory tile (never written to HBM).
// Pass 2 (warp = channel, same sweep as pairsum): with m = [pre>0],
//         RSm_s = sum_t delta*m, CSm_t = sum_s delta*m, LSm = sum_{l=1} delta*m,
//         HS = sum relu(pre)*delta   -- everything the node-level backward needs.
// The N^2 x 20 hidden tensor and the N^2 x 22 concat of model_2.py:279-281 are never materialised.
#pragma once
#include "common.cuh"

namespace hdgnn {

struct ScoreArgs {
    const uint32_t* bits; // (B, N, WP) label bitmap (bits.cuh)
    int WP;
    int N, RT, S;
    const float* PR;      // (B,N,20), bias + label-0 row folded in
    const float* PC;      // (B,N,20)
    const float* params;
    int o_l, o_w2, o_b2;  // head: label rows (2,20), W2 (20,2), b2 (2)
    float* logits;        // (B,2,N(N-1)) or nullptr
    float* probs;         // (B,2,N(N-1)) or nullptr
    float* soft;          // (B,N,N,2) soft labels for the entity-edge branch, or nullptr
    uint32_t* pred;       // (B,N,WP) predicted relations [p1 > p0] as a label bitmap (hdgnn_set_predictions), or nullptr
    float* cep;           // (B,S) sum of CE over the tile
    float scale;          // delta = scale * (p1 - l)            (hunk head, CE loss)
    const float* dsoft;   // (B,N,N,2) upstream d/d(a0,a1): delta = a1*a0*(da1-da0)   (edge head)
    float* RSm;           // (B,N,20)
    float* CSmp;          // (B,S,N,20)
    float* LSmp;          // (B,S,20)
    float* HSp;           // (B,S,20)
    float* dsump;         // (B,S)
};

__host__ __device__ inline size_t score_smem_bytes(int CW, int RT, int row_bytes, bool train) {
    const size_t NP = (size_t)CW * 32;
    size_t off = round_up(RT * row_bytes, 128);
    size_t labf = (size_t)(RT / 4) * NP * 16;
    size_t cst = NP * HD * 4;
    off += labf > cst ? labf : cst;
    if (train) off += labf;
    off += NP * HD * 4;                  // PCt
    off += (size_t)RT * HD * 4 * 2;      // PRt, RSt
    off += 64 * 4 + 32 * 4;              // weights, scratch
    return off + 16;
}

// PRED: the launch writes the predicted-relation bitmap (a.pred).  The flag is a template parameter so that the instantiations
// without it keep the plain lane loop and its register allocation.
template <int CW, bool TRAIN, bool PRED>
__global__ void __launch_bounds__(32 * HD, 1) score_kernel(const ScoreArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int NP = CW * 32;
    const int N = a.N, RT = a.RT, WP = a.WP;
    const int b = blockIdx.y, s = blockIdx.x;
    const int r0 = s * RT;
    const int nrows = min(RT, N - r0);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    uint32_t* stage = reinterpret_cast<uint32_t*>(smem);
    size_t off = round_up(RT * WP * 4, 128);
    float4* labf = reinterpret_cast<float4*>(smem + off);
    float* CSt = reinterpret_cast<float*>(smem + off);
    const size_t labf_bytes = (size_t)(RT / 4) * NP * 16;
    {
        size_t l2 = (size_t)NP * HD * 4;
        off += labf_bytes > l2 ? labf_bytes : l2;
    }
    float4* delt = reinterpret_cast<float4*>(smem + off); if (TRAIN) off += labf_bytes;
    float* PCt = reinterpret_cast<float*>(smem + off); off += (size_t)NP * HD * 4;     // [k][j]
    float* PRt = reinterpret_cast<float*>(smem + off); off += (size_t)RT * HD * 4;     // [r][k]
    float* RSt = reinterpret_cast<float*>(smem + off); off += (size_t)RT * HD * 4;
    float* Wsm = reinterpret_cast<float*>(smem + off); off += 64 * 4;                  // D, G0, G1, b2
    float* scratch = reinterpret_cast<float*>(smem + off); off += 32 * 4;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + off);

    if (tid == 0) { mbar_init(bar, 1); fence_mbar_init(); }
    __syncthreads();
    if (tid == 0) {
        const uint32_t bytes = (uint32_t)nrows * WP * 4;
        mbar_arrive_expect_tx(bar, bytes);
        bulk_g2s(stage, a.bits + ((size_t)b * N + r0) * WP, bytes, bar);
    }
    const float* par = a.params;
    if (tid < HD) {
        Wsm[tid] = par[a.o_l + HD + tid] - par[a.o_l + tid];
        Wsm[HD + tid] = par[a.o_w2 + 2 * tid];
        Wsm[2 * HD + tid] = par[a.o_w2 + 2 * tid + 1];
    }
    if (tid < 2) Wsm[3 * HD + tid] = par[a.o_b2 + tid];
    for (int idx = tid; idx < NP * HD; idx += blockDim.x) {
        const int j = idx / HD, kk = idx - j * HD;
        PCt[kk * NP + j] = j < N ? a.PC[((size_t)b * N + j) * HD + kk] : NEG_BIG;
    }
    for (int idx = tid; idx < RT * HD; idx += blockDim.x) {
        const int r = idx / HD;
        PRt[idx] = r < nrows ? a.PR[((size_t)b * N + r0) * HD + idx] : NEG_BIG;
    }
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
        if (TRAIN) delt[idx] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __syncthreads();

    // ------------------------------ pass 1: thread = pair ------------------------------
    float ce_acc = 0.f, d_acc = 0.f;
    {
        float Dk[HD], G0[HD], G1[HD];
#pragma unroll
        for (int kk = 0; kk < HD; ++kk) { Dk[kk] = Wsm[kk]; G0[kk] = Wsm[HD + kk]; G1[kk] = Wsm[2 * HD + kk]; }
        const float b20 = Wsm[3 * HD], b21 = Wsm[3 * HD + 1];
        const size_t npair = (size_t)N * (N - 1);
        for (int row = warp; row < nrows; row += HD) {
            const int i = r0 + row;
            float Rs[HD];
#pragma unroll
            for (int kk = 0; kk < HD; ++kk) Rs[kk] = PRt[row * HD + kk];
            const float* lrow = reinterpret_cast<const float*>(labf + (row >> 2) * NP) + (row & 3);
            float* drow = reinterpret_cast<float*>(delt + (row >> 2) * NP) + (row & 3);
            // PRED: whole 32-column segments, so that the prediction ballot is warp-uniform; columns >= N read the NEG_BIG / zero
            // padding of PCt and the label tile and store nothing
            for (int j = lane; j < (PRED ? CW * 32 : N); j += 32) {
                if (!PRED && j == i) continue;
                const float l = lrow[4 * j];
                float l0 = b20, l1 = b21;
#pragma unroll
                for (int kk = 0; kk < HD; ++kk) {
                    const float t = fmaf(l, Dk[kk], Rs[kk]) + PCt[kk * NP + j];
                    const float h = fmaxf(t, 0.f);
                    l0 = fmaf(h, G0[kk], l0);
                    l1 = fmaf(h, G1[kk], l1);
                }
                const float d = l1 - l0;
                const float e = expf(-fabsf(d));
                const float inv = 1.f / (1.f + e);
                const float pb = inv, ps = e * inv;
                const float p1 = d >= 0.f ? pb : ps, p0 = d >= 0.f ? ps : pb;
                if (PRED) {         // predicted relation: np.argmax over the two channels, a tie is class 0
                    const bool valid = j < N && j != i;
                    const uint32_t am = __ballot_sync(0xffffffffu, valid && p1 > p0);
                    if (lane == 0) a.pred[((size_t)b * N + i) * WP + (j >> 5)] = am;
                    if (!valid) continue;
                }
                const size_t q = (size_t)i * (N - 1) + j - (j > i);
                if (a.logits) {
                    a.logits[((size_t)b * 2 + 0) * npair + q] = l0;
                    a.logits[((size_t)b * 2 + 1) * npair + q] = l1;
                }
                if (a.probs) {
                    a.probs[((size_t)b * 2 + 0) * npair + q] = p0;
                    a.probs[((size_t)b * 2 + 1) * npair + q] = p1;
                }
                if (a.soft) {
                    float2* sp = reinterpret_cast<float2*>(a.soft) + ((size_t)b * N + i) * N + j;
                    *sp = make_float2(p0, p1);
                }
                const float z = l > 0.5f ? -d : d;
                ce_acc += fmaxf(z, 0.f) + log1pf(e);
                if (TRAIN) {
                    float dl;
                    if (a.dsoft) {
                        const float2 da = reinterpret_cast<const float2*>(a.dsoft)[((size_t)b * N + i) * N + j];
                        dl = p1 * p0 * (da.y - da.x);
                    } else {
                        dl = a.scale * (p1 - l);
                    }
                    drow[4 * j] = dl;
                    d_acc += dl;
                }
            }
            if (PRED && lane < WP - CW) a.pred[((size_t)b * N + i) * WP + CW + lane] = 0u;      // padding words of the row
        }
    }
    const float ce_tot = block_sum(ce_acc, scratch);
    if (tid == 0 && a.cep) a.cep[(size_t)b * a.S + s] = ce_tot;
    if (!TRAIN) return;
    const float d_tot = block_sum(d_acc, scratch);      // also orders the delta tile before pass 2
    if (tid == 0) a.dsump[(size_t)b * a.S + s] = d_tot;
    __syncthreads();

    // ------------------------------ pass 2: warp = channel ------------------------------
    const int k = warp;
    const float D = Wsm[k];
    float Q[CW], col[CW];
#pragma unroll
    for (int seg = 0; seg < CW; ++seg) { Q[seg] = PCt[k * NP + seg * 32 + lane]; col[seg] = 0.f; }
    float lacc = 0.f, hacc = 0.f;
    for (int rq = 0; rq < RT / 4; ++rq) {
        float P[4], row[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) { P[r] = PRt[(4 * rq + r) * HD + k]; row[r] = 0.f; }
#pragma unroll
        for (int seg = 0; seg < CW; ++seg) {
            const float4 l4 = labf[rq * NP + seg * 32 + lane];
            const float4 d4 = delt[rq * NP + seg * 32 + lane];
            const float l[4] = {l4.x, l4.y, l4.z, l4.w};
            const float dl[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const float t = fmaf(l[r], D, P[r]) + Q[seg];
                const float v = t > 0.f ? dl[r] : 0.f;
                row[r] += v;
                col[seg] += v;
                lacc = fmaf(l[r], v, lacc);
                hacc = fmaf(fmaxf(t, 0.f), dl[r], hacc);
            }
        }
        const float tot = warp_rowsum4(row[0], row[1], row[2], row[3], lane);
        if ((lane & 7) == 0) RSt[(4 * rq + ((lane >> 4) & 1) * 2 + ((lane >> 3) & 1)) * HD + k] = tot;
    }
    {
        const float ls = warp_sum(lacc), hs = warp_sum(hacc);
        if (lane == 0) {
            a.LSmp[((size_t)b * a.S + s) * HD + k] = ls;
            a.HSp[((size_t)b * a.S + s) * HD + k] = hs;
        }
    }
    __syncthreads();
#pragma unroll
    for (int seg = 0; seg < CW; ++seg) {
        const int j = seg * 32 + lane;
        if (j < N) CSt[j * HD + k] = col[seg];
    }
    for (int idx = tid; idx < nrows * HD; idx += blockDim.x)
        a.RSm[((size_t)b * N + r0) * HD + idx] = RSt[idx];
    __syncthreads();
    float* cs = a.CSmp + ((size_t)b * a.S + s) * N * HD;
    for (int idx = tid; idx < N * HD; idx += blockDim.x) cs[idx] = CSt[idx];
}

}  // namespace hdgnn
