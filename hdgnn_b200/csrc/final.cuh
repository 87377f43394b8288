// final: deterministic reduction of the per-commit / per-tile gradient partials into the flat
// gradient, the mean cross-entropy (model_2.py:115-118) and -- on one GPU -- the regularisers
// and TF1 Adam update (model_2.py:121-130, 326-338) in the same launch.
#pragma once
#include "common.cuh"

namespace hdgnn {

struct Rank1Map {            // where the four 20-vectors of an ent_bwd partial land in the flat gradient
    const float* gp;         // (n,80) {db, dU, dV, LS} per ent_bwd2 CTA, or null
    int n, o_u, o_v, o_b, o_l;   // o_u == o_v: tied first-layer row (model_4.py:219-222)
};

// Peer exchange over NVLink / NVSwitch (commit sharding, one process per GPU): every rank owns a MAILBOX in its own
// HBM that its peers write into directly (P2P stores through IPC-mapped pointers):
//   inbox  [2][world][stride] u64   gradient slices by step parity and sending rank; each entry = {sequence number of
//   lossin [2][world]         u64   the step : fp32 payload} written with ONE 8-byte store (single-copy atomic), so the
//                                   payload needs no separate flag and no fence (the scheme of NCCL's LL protocol)
// A CTA of reduce_adam_kernel pushes its 128-parameter slice to every rank, then every thread polls its own entry of
// the rank's OWN mailbox until the step's sequence number shows up, and the slices are summed in rank order -- every
// rank forms the bitwise identical sum, so the replicas never diverge.  Two parities suffice: a rank can only be one
// step ahead of a peer (it needs that peer's slice to finish the step).
constexpr int PEER_MAX = 8;
typedef unsigned long long peer_word;
struct PeerArgs {
    int world, rank, stride, ncta;
    peer_word* inbox[PEER_MAX];  // mailbox of rank r as mapped into this process (own entry = local pointer)
    peer_word* lossin[PEER_MAX];
    int* seq;                    // device counter: exchanges completed so far (local)
    int* error;                  // set to 1 when a wait timed out (hdgnn_peer_status reads it)
    unsigned int max_spins;      // polls of ~1 us before a wait gives up (HDGNN_PEER_TIMEOUT_MS, default 20 s)
    unsigned long long* stamps;  // debug (HDGNN_PEER_STAMPS=1): [4096][2] globaltimer ns of CTA 0 at its push and after its last pull
};

__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void peer_push(peer_word* p, float v, int seq) {
    const peer_word w = ((peer_word)(unsigned int)seq << 32) | (peer_word)__float_as_uint(v);
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(w) : "memory");
}
// Bounded wait: a lost or very late peer sets the error flag and the wait returns 0 (the step's result is then
// meaningless, but the context survives: the host sees the flag through hdgnn_peer_status and raises).
__device__ __forceinline__ float peer_pull(const peer_word* p, int seq, int* error, unsigned int max_spins) {
    peer_word w;
    unsigned int spin = 0;
    for (;;) {
        asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(w) : "l"(p) : "memory");
        if ((int)(w >> 32) == seq) break;
        if (++spin > max_spins || *reinterpret_cast<volatile int*>(error)) { *error = 1; return 0.f; }
        __nanosleep(spin < 64 ? 32 : 1000);
    }
    return __uint_as_float((unsigned int)(w & 0xffffffffu));
}

struct FinalArgs {
    int B, total;
    PeerArgs peer;           // peer.world <= 1: single GPU
    const float* gpart;      // (B,total)
    Rank1Map ent, edge;
    const float* cep; int ncep; float loss_denom; float* loss;
    float* grads;            // out: d(10 CE)/dparams for the local commits
    // optional fused optimizer step
    int apply_adam;
    float* params; float* m; float* v; int* step; int o_t1, o_t2;
    float lr, b1, b2, eps;
    float* reg_losses;       // {loss_map, loss_para} at the pre-update parameters, or null
    float* l2part;           // (gridDim.x) scratch
    unsigned int* counter;   // zero-initialised; reset by the last CTA
};

// lr_t = lr sqrt(1 - b2^t) / (1 - b1^t) (tf.train.AdamOptimizer), with 1 - b^t = -expm1(t log b) so that the
// small differences keep full float precision (fp64 pow costs ~10 us on this part's fp64 pipe)
__device__ __forceinline__ float adam_lr_t(float lr, float b1, float b2, int t) {
    const float omb2 = -expm1f((float)t * logf(b2)), omb1 = -expm1f((float)t * logf(b1));
    return lr * sqrtf(omb2) / omb1;
}

constexpr int FIN_P = 16;    // parameters per CTA: ~133 small CTAs, every thread has all its loads in flight at once (one L2 round trip)
constexpr int FIN_SL = 16;   // commit slices per parameter

__device__ __forceinline__ float rank1_extra(const Rank1Map& r, int p, int slice, int nslice) {
    if (!r.gp) return 0.f;
    // which of the four 20-vectors {db, dU, dV, LS} of a partial feed parameter p: c1 * g[i1] + c2 * g[i2]
    int i1 = -1, i2 = -1; float c2 = 1.f;
    if (p >= r.o_b && p < r.o_b + HD) { i1 = p - r.o_b; }                                                  // bias: db
    else if (p >= r.o_l && p < r.o_l + HD) { i1 = p - r.o_l; i2 = 3 * HD + i1; c2 = -1.f; }                 // label-0 row: db - LS
    else if (p >= r.o_l + HD && p < r.o_l + 2 * HD) { i1 = 3 * HD + (p - r.o_l - HD); }                     // label-1 row: LS
    else if (p >= r.o_u && p < r.o_u + HD) { i1 = HD + (p - r.o_u); if (r.o_v == r.o_u) i2 = 2 * HD + (p - r.o_u); }
    else if (r.o_v != r.o_u && p >= r.o_v && p < r.o_v + HD) { i1 = 2 * HD + (p - r.o_v); }
    if (i1 < 0) return 0.f;
    const bool two = i2 >= 0;
    if (!two) i2 = i1;
    float acc = 0.f;
    const int n = r.n;
    const size_t stride = (size_t)nslice * 4 * HD;
    constexpr int U = 16;                             // independent loads in flight; fixed summation order
    int t = slice;
    for (; t + (U - 1) * nslice < n; t += U * nslice) {
        const float* g = r.gp + (size_t)t * 4 * HD;
        float av[U], bv[U];
#pragma unroll
        for (int u = 0; u < U; ++u) { av[u] = g[u * stride + i1]; bv[u] = two ? g[u * stride + i2] : 0.f; }
#pragma unroll
        for (int u = 0; u < U; ++u) acc += two ? fmaf(c2, bv[u], av[u]) : av[u];
    }
    for (; t < n; t += nslice) {
        const float* g = r.gp + (size_t)t * 4 * HD;
        acc += two ? fmaf(c2, g[i2], g[i1]) : g[i1];
    }
    return acc;
}

__global__ void __launch_bounds__(FIN_P * FIN_SL) reduce_adam_kernel(const FinalArgs a) {
    __shared__ float part[FIN_SL][FIN_P];
    __shared__ float scratch[32];
    __shared__ float tn[3];
    __shared__ float ce_sh;
    __shared__ int last;
    const int tid = threadIdx.x, pl = tid % FIN_P, sl = tid / FIN_P;
    const int p = blockIdx.x * FIN_P + pl;
    pdl_launch_dependents();        // the next step's pack_bits may run beside this kernel (see pack.cuh)
    // optimizer state first: these loads overlap the reduction below (the kernel is a chain of global latencies)
    const bool own = a.apply_adam && sl == 0 && p < a.total;
    const float pv = own ? a.params[p] : 0.f, m_old = own ? a.m[p] : 0.f, v_old = own ? a.v[p] : 0.f;
    const int t = a.apply_adam ? *a.step + 1 : 0;       // read before any CTA can publish the new count
    float th[4] = {0.f, 0.f, 0.f, 0.f};
    if (a.apply_adam && tid < 2) {
        const int o = tid == 0 ? a.o_t1 : a.o_t2;
        th[0] = a.params[o]; th[1] = a.params[o + 1];
    }
    pdl_wait();                     // gradient partials come from mid2 / ent_bwd2
    float acc = 0.f;
    if (p < a.total) {
        for (int bb = sl; bb < a.B; bb += 16 * FIN_SL) {      // sixteen guarded loads in flight, fixed summation order
            float g[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) {
                const int idx = bb + u * FIN_SL;
                g[u] = idx < a.B ? a.gpart[(size_t)idx * a.total + p] : 0.f;
            }
#pragma unroll
            for (int u = 0; u < 16; ++u) acc += g[u];
        }
        acc += rank1_extra(a.ent, p, sl, FIN_SL);
        acc += rank1_extra(a.edge, p, sl, FIN_SL);
    }
    part[sl][pl] = acc;
    float ce_local = 0.f;
    if (blockIdx.x == 0 && a.loss) {          // mean CE: fixed-order block sum of the per-commit partials
        float c = 0.f;
        for (int i = tid; i < a.ncep; i += blockDim.x) c += a.cep[i];
        ce_local = block_sum(c, scratch) / a.loss_denom;
        if (tid == 0) *a.loss = ce_local;
    }
    __syncthreads();
    float g = 0.f;
    if (sl == 0 && p < a.total) {
#pragma unroll
        for (int s = 0; s < FIN_SL; ++s) g += part[s][pl];
    }
    if (a.peer.world > 1) {
        // ---- gradient all-reduce over peer memory, fused with the reduction above and the optimizer below ----
        const PeerArgs& pr = a.peer;
        const int W = pr.world, seq = *pr.seq + 1, par = seq & 1;
        __syncthreads();                                   // part[][] has been consumed
        if (sl == 0) part[0][pl] = g;
        if (blockIdx.x == 0 && tid == 0) ce_sh = ce_local;
        __syncthreads();
        const float mine = part[0][pl];
        const size_t slot = (size_t)par * W;
        if (pr.stamps && blockIdx.x == 0 && tid == 0) pr.stamps[2 * (seq & 4095)] = global_ns();
        if (sl < W && p < a.total) peer_push(pr.inbox[sl] + (slot + pr.rank) * pr.stride + p, mine, seq);
        if (blockIdx.x == 0 && tid < W && a.loss) peer_push(pr.lossin[tid] + slot + pr.rank, ce_sh, seq);
        __syncthreads();                                   // part[0][] has been read
        part[sl][pl] = (sl < W && p < a.total) ? peer_pull(pr.inbox[pr.rank] + (slot + sl) * pr.stride + p, seq, pr.error, pr.max_spins) : 0.f;
        __syncthreads();
        if (pr.stamps && blockIdx.x == 0 && tid == 0) pr.stamps[2 * (seq & 4095) + 1] = global_ns();
        if (sl == 0 && p < a.total) {
            g = 0.f;
            for (int r = 0; r < W; ++r) g += part[r][pl];  // rank order: identical on every rank
        }
        if (blockIdx.x == 0 && tid == 0 && a.loss) {
            float c = 0.f;
            for (int r = 0; r < W; ++r) c += peer_pull(pr.lossin[pr.rank] + slot + r, seq, pr.error, pr.max_spins);
            *a.loss = c;                                   // global mean CE
        }
        // *pr.seq is advanced by the last CTA of the optimizer tail below: by then every CTA has read it
    }
    if (sl == 0 && p < a.total) a.grads[p] = g;
    if (!a.apply_adam) return;

    // regularisers (evaluated at the pre-update parameters) + TF1 Adam
    if (tid < 2) tn[tid] = sqrtf(th[0] * th[0] + th[1] * th[1]);
    if (tid == 2) tn[2] = adam_lr_t(a.lr, a.b1, a.b2, t);
    const float sq = block_sum(pv * pv, scratch);       // also orders tn[]
    if (sl == 0 && p < a.total) {
        float gi = g + 0.001f * pv;
        if (p >= a.o_t1 && p < a.o_t1 + 2) gi += 0.001f * pv / tn[0];
        if (p >= a.o_t2 && p < a.o_t2 + 2) gi += 0.001f * pv / tn[1];
        const float lr_t = tn[2];
        const float mi = a.b1 * m_old + (1.f - a.b1) * gi;
        const float vi = a.b2 * v_old + (1.f - a.b2) * gi * gi;
        a.m[p] = mi; a.v[p] = vi;
        a.params[p] = pv - lr_t * mi / (sqrtf(vi) + a.eps);
    }
    // last CTA: step counter and the two regulariser values
    if (tid == 0) {
        a.l2part[blockIdx.x] = sq;
        __threadfence();
        const unsigned int done = atomicAdd(a.counter, 1u);
        last = (done == gridDim.x - 1);
    }
    __syncthreads();
    if (last && tid < 32) {
        // the last CTA's first warp: the per-CTA partials with all loads in flight (lane-strided, then a fixed shuffle tree)
        __threadfence();
        float l2 = 0.f;
        for (unsigned int i = tid; i < gridDim.x; i += 32) l2 += __ldcg(a.l2part + i);
        l2 = warp_sum(l2);
        if (tid == 0) {
            if (a.reg_losses) a.reg_losses[1] = 0.001f * 0.5f * l2;
            *a.step = t;
            if (a.peer.world > 1) *a.peer.seq = *a.peer.seq + 1;
            *a.counter = 0u;
        }
    }
    // loss_map = 0.01 (|theta1| + |theta2|): written by the CTA that read the thetas before updating them
    if (a.reg_losses && tid == 0 && a.o_t1 >= (int)(blockIdx.x * FIN_P) && a.o_t1 < (int)((blockIdx.x + 1) * FIN_P))
        a.reg_losses[0] = 0.01f * (tn[0] + tn[1]);
}

}  // namespace hdgnn
