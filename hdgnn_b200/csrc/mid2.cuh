// mid2: everything of a training step that is per-commit and smaller than the entity sweeps, fused
// into ONE kernel with one CTA per commit and every intermediate in shared memory:
//
//   entity-state MLP (model_2.py:181-205)  ->  entity->hunk pooling (model_2.py:146-150, index
//   semantics of utils2.py:111-137)  ->  hunk pair layer + "edge translation" (model_2.py:245-277)
//   ->  relation head + softmax + cross-entropy (model_2.py:304-324, 115-118)
//   ->  [training] the hand-written backward of all of the above down to d/d(entity effect sums).
//
// Only RS1 / CS1p (from ent_fwd2) and the two label bitmaps are read (bitmaps: one TMA bulk copy
// each); GE (for ent_bwd2), the per-commit gradient partials, probs / logits and the CE partial are
// written.  All reductions run in a fixed order.
//
// Pooling: with all L = Ne index lines present the L x L local grid IS the Ne x Ne grid and the
// per-entity sums have the closed form {(Ne-1) x_i, X - x_i, (Ne-1) - deg_i, deg_i} (row / column
// degrees from popcounts of the bitmap); with L < Ne (quirk Q3: the local counter of
// utils2.py:123-137 runs with stride L-1) the L x L grid is gathered pair by pair from shared memory.
#pragma once
#include "sweep2.cuh"
#include "ent2.cuh"
#include "entsp.cuh"

namespace hdgnn {

constexpr int M2_NRG = 4;
constexpr int M2_NW = KG * M2_NRG;        // 20 warps
constexpr int M2_T = M2_NW * 32;          // 640 threads
constexpr int M2_CH = 256;                // entity nodes per chunk of the entity-state MLP backward
constexpr int M2_NODE_F = 24 + 20 + 24;   // floats per node of that chunk: [S|x|1|0|0] dz [relu(Z) du|du|0|0|0]
// The entity block ent_w5 .. nod_b2 and the hunk block hnk_w1 .. scr_b2 are each contiguous in the
// parameter blob (TF creation order, hdgnn.cu) with every array at a multiple of 4 floats from the
// block start, so one copy per block keeps every matrix 16-byte aligned in shared memory.
constexpr int M2_MCLS = 16;               // inline entity stage: most distinct node-attribute values served by the class tables
constexpr int M2_BLK1 = 400 + 20 + 420 + 20 + 20 + 1;              // 881
constexpr int M2_BLK2 = 200 + 20 + 400 + 20 + 440 + 20 + 40 + 2;   // 1142
// variant 4's edge block edg_w11 .. eup_b2 (model_4.py:219-229, 292-297): offsets 0 20 60 80 480 500 940 960 1000
constexpr int M2_BLKE = 20 + 40 + 20 + 400 + 20 + 440 + 20 + 40 + 2;    // 1002

// debug dump layout per commit (floats): S1[Ne*20] X2[Ne] NB[Nc*4] RS3[Nc*20] CS3[Nc*20] PR[Nc*20] PC[Nc*20]
// DNB[Nc*4] DX2[Ne]
__host__ __device__ inline size_t mid2_dbg_floats(int Ne, int Nc) { return (size_t)Ne * 22 + (size_t)Nc * 88; }

// floats of the twelve hunk-stage tables of one commit (PH01 x2, QH, RS3, CS3, r, c, PR01 x2, PC, RSm, CSm), 32-byte granule
__host__ __device__ inline int mid2_tab_floats(int Nc) { return (12 * Nc * HD + 7) & ~7; }

// float offset of the pooling row table inside the scratch region: behind the column partials [nchunk][L][4], nchunk L <= min(4 Ne, M2_T)
__host__ __device__ inline int mid2_rowtab_off(int Ne) { return 4 * (4 * Ne < M2_T ? 4 * Ne : M2_T); }      // a multiple of 4: 16-byte aligned

struct Mid2Smem {
    // offsets in floats
    int blk1, blk2, gam, Dh, Dg, G1g, W5U, c1p;   // weight blocks (contiguous copies of the parameter blob), derived tables
    int x, x2, hm, SP, TP, dl, dx2, nb, dnb, ebits, ybits, scratch, red, uni, sc, total;
    int entw, xsort, ordv, sx;               // inline entity stage: U V c D, x sorted, rank -> node, suffix sums of sorted x
    int rptr, cptr, headrow, headp;          // edge prefix counts by row / by column, head partials of the edge-walk slots
    int ebt, cls, cval, csize, cmask, cmeta;  // transposed bitmap; attribute classes: class of a node, value / size / node mask of a class
    int blkE, wEe, gamE, DgE, RA, CA, cpart; // variant 4: edge-branch weight block, its first layer (U V c D), head tables, row / column sums of a1
    int gt;                                  // hunk-stage tables (12 Nc 20 floats) in global memory (Mid2Args::tabs_g) instead of the union region
    int scg;                                 // (GT kernels) the S / GE rows (Ne x 20) in global memory (Mid2Args::GE) instead of the sc region
    int stg;                                 // (GT kernels) staging region of the hunk sweeps' row tables (3 Nc 20 floats), behind the dlt table
};

// what a mid2 launch keeps where; mid2_layout turns it into offsets
struct Mid2Opts {
    bool train = false;      // the training kernel (forward + backward)
    bool dlt_smem = true;    // the per-pair dL/dlogit table of the training path in shared memory (else it lives in HBM / L2)
    bool scache = false;     // the entity effect sums S (Ne x 20) in shared memory from the forward to the backward
    bool inl = false;        // entity pair layer inside mid2 (entsp.cuh); implies scache
    bool edge = false;       // variant 4: the entity-edge branch inside mid2 as well
    bool gt = false;         // the twelve hunk-stage tables in global memory (per-commit scratch, L1/L2-resident) -- the form
                             // for hunk grids whose tables do not fit one SM beside the rest of the commit's state (Nc > 128)
    bool scg = false;        // ... and the S / GE rows in global memory as well; only with gt
};

// the options as mid2 runs with them: every layout and every kernel flag derives from these
__host__ __device__ inline Mid2Opts mid2_normalize(Mid2Opts o) {
    if (o.inl) o.scache = true;
    if (!o.gt) o.scg = false;
    return o;
}

__host__ __device__ inline Mid2Smem mid2_layout(int Ne, int Nc, Mid2Opts opt) {
    const Mid2Opts no = mid2_normalize(opt);
    const bool train = no.train, dlt_smem = no.dlt_smem, scache = no.scache, inl = no.inl, edge = no.edge, gt = no.gt;
    Mid2Smem m;
    m.gt = gt ? 1 : 0; m.scg = no.scg ? 1 : 0;
    int o = 0;
    auto take = [&](int n) { int r = o; o += (n + 7) & ~7; return r; };      // 32-byte granules
    m.blk1 = take(M2_BLK1); m.blk2 = take(M2_BLK2); m.gam = take(20); m.Dh = take(20); m.Dg = take(20); m.G1g = take(400);
    m.W5U = take(400); m.c1p = take(20);
    m.x = take(Ne); m.x2 = take(Ne); m.hm = take(Ne);
    m.entw = m.xsort = m.ordv = m.sx = m.rptr = m.cptr = m.headrow = m.headp = 0;
    m.ebt = m.cls = m.cval = m.csize = m.cmask = m.cmeta = 0;
    if (inl) {
        m.entw = take(4 * HD); m.xsort = take(Ne); m.ordv = take(Ne); m.sx = take(Ne + 1);
        m.rptr = take(Ne + 1); m.cptr = take(Ne + 1); m.headrow = take(M2_T / 10); m.headp = take(M2_T / 10 * HD);
        m.ebt = take(Ne * bit_words(Ne)); m.cls = take(Ne); m.cval = take(M2_MCLS); m.csize = take(M2_MCLS);
        m.cmask = take(M2_MCLS * bit_words(Ne)); m.cmeta = take(8);
        m.blkE = m.wEe = m.gamE = m.DgE = m.RA = m.CA = m.cpart = 0;
        if (edge) { m.blkE = take(M2_BLKE); m.wEe = take(4 * HD); m.gamE = take(HD); m.DgE = take(HD); m.RA = take(Ne); m.CA = take(Ne); m.cpart = take(M2_NW * 32); }
    }
    m.dx2 = take(Ne); m.nb = take(4 * Nc); m.dnb = take(4 * Nc);
    m.ebits = take(Ne * bit_words(Ne)); m.ybits = take(Nc * bit_words(Nc));
    const int cwc = (Nc + 31) / 32, wue = (Ne + 31) / 32;
    // scratch users: column combine of the hunk sweeps (two passes of half the segments for 5-6 segments, column passes of four
    // segments from 7 on) | pooling partials
    // [<= 4 chunks][L][4] + the row table [L] int4 | prologue counters [8][wue][8] + [wue][Nc] | backward partials [<= M2_T]
    const int comb = (M2_NRG / 2) * (cwc >= 7 ? 4 : cwc >= 5 ? (cwc + 1) / 2 : cwc) * 32 * HD;
    const int pool = mid2_rowtab_off(Ne) + 4 * Ne, prol = 64 * wue + wue * Nc;
    const int comb_e = edge ? (M2_NRG / 2) * 4 * 32 * HD : 0;      // variant 4: combine_cols<4> of the soft-edge delta sweep
    int scr = comb > pool ? comb : pool;
    scr = scr > comb_e ? scr : comb_e; scr = scr > prol ? scr : prol; scr = scr > M2_T ? scr : M2_T;
    m.scratch = take(scr);
    m.red = take(64 + M2_NW * HD + 64);
    m.uni = o;
    // union region: [hunk tables 12 Nc 20][dlt (training) | SP TP dl (pooling: dead while dlt is live)]; the
    // entity-state backward (after the pooling backward) reuses it from the start
    // (the inline entity stage keeps its transposed bitmap, Ne * bit_words(Ne) words, resp. 20 suffix tables of Ne + 1 floats
    // plus 8 partial sums per thread here: both below M2_CH * M2_NODE_F for Ne <= 512)
    const int ent_phase = M2_CH * M2_NODE_F;
    const int dlt = (train && dlt_smem) ? Nc * cwc * 32 : 0, pool3 = 3 * ((4 * Ne + 7) & ~7);
    const int tabs = gt ? 0 : mid2_tab_floats(Nc);
    // global tables: the row tables of a sweep (P01 rows, and the row gradients of the backward sweep) are staged in shared memory
    // for the duration of the sweep, behind the dlt table (SP / TP / dl are dead while the sweeps run)
    const int stage = gt ? (((train ? 3 : 2) * Nc * HD + 7) & ~7) : 0;
    m.stg = m.uni + dlt;
    const int hunk_phase = gt ? (dlt + stage > pool3 ? dlt + stage : pool3) : tabs + (dlt > pool3 ? dlt : pool3);
    m.SP = m.uni + tabs; m.TP = m.SP + ((4 * Ne + 7) & ~7); m.dl = m.TP + ((4 * Ne + 7) & ~7);
    o += ent_phase > hunk_phase ? ent_phase : hunk_phase;
    m.sc = o;
    if (scache && !m.scg) o += (Ne * HD + 7) & ~7;
    m.total = o;
    return m;
}
__host__ __device__ inline size_t mid2_smem_bytes(const Mid2Smem& m) { return (size_t)m.total * 4 + 16; }
__host__ __device__ inline size_t mid2_smem_bytes(int Ne, int Nc, const Mid2Opts& o) { return mid2_smem_bytes(mid2_layout(Ne, Nc, o)); }

// Variant 4 (layout m with Mid2Opts::edge): the forward of the entity-edge branch keeps the soft-edge head tables (Ne x 60 floats
// + a 128-row staging tile) and the edge branch's pair sums (2 Ne x 20) side by side in the union region
__host__ __device__ inline bool mid2_edge_fwd_fits(int Ne, const Mid2Smem& m) {
    return Ne * 60 + (M2_T / KG) * HD <= (m.sc - m.uni) - 2 * Ne * HD;
}
// ... its backward needs the head tables + column delta sums + a 32-row de tile; later five Ne x 20 arrays + GCe at the end; the
// general-attribute form of ent_bwd needs two sets of suffix tables beside GCe
__host__ __device__ inline bool mid2_edge_bwd_fits(int Ne, const Mid2Smem& m) {
    const int uf = m.sc - m.uni, wue = (Ne + 31) / 32;
    return Ne * 80 + 32 * wue * 32 <= uf && Ne * 120 <= uf && 40 * (Ne + 1) + 8 * M2_T + Ne * HD <= uf;
}

struct Mid2Args {
    int Ne, Nc, ent, R, SL;                  // R, SL: row-chunk decomposition of ent_fwd2 (ent2.cuh)
    const uint32_t* ebits; int WPe;          // (B,Ne,WPe)
    const uint32_t* ybits; int WPc;          // (B,Nc,WPc)
    const float* x; const int* hmap; const int* L;
    const float* params; ParamOff po;
    const float* RS1; const float* CS1p;     // (B,Ne,20), (B,SL,Ne,20)
    float* logits; float* probs;             // (B,2,Ncr) or null
    float* cep;                              // (B) sum of CE over the commit's pairs
    float scale;                             // dL/dlogit scale: 10 / (B_global * Ncr)
    float* GE;                               // (B,Ne,20) d/dS1
    float* gpart; int total;                 // (B,total)
    float* dbg;                              // debug dumps (HDGNN_F_DEBUG) or null; layout below
    long long* clk;                          // per-phase clock64 stamps (B,24) or null
    float* dlt_g;                            // (B, Nc, CW*32) dL/dlogit table in HBM when it does not fit smem, else null
    int scache;                              // keep the entity effect sums S (Ne x 20) in shared memory from the forward to the backward
    int edge;                                // variant 4: the entity-edge branch (model_4.py:92-98, 206-304) inside this kernel
    float* RSEg; float* CSEg; float* REg; float* CEg;      // (B,Ne,20) each: edge-branch pair sums and second-layer outputs, kept for the backward
    float* PREg;                             // (B,Ne,60): soft-edge head tables PRe01 (Ne x 40) then PCe (Ne x 20), kept for the backward
    float* A1F;                              // (B, Ne (Ne-1)) soft edges a1 in flat pair order, written and read for commits with L < Ne only
    unsigned long long* hits_acc;            // running count of arg-max hits (EvaluationFuncs.py:27-37) over all commits, or null
    unsigned long long* evc;                 // (B,8) per-commit evaluation counters in the layout of hdgnn_eval_counts (EvaluationFuncs.py:27-37,
                                             // 92-117), ADDED to by the relation head, or null
    const int* wait_flag; int wait_tag;      // host-fed step: the staging copies of this step are complete once *wait_flag == wait_tag
                                             // (written by the copy stream's DMA after the data); null = inputs already ordered
    Mid2Smem lay;                            // shared-memory layout (mid2_layout), computed once on the host: the offsets are kernel
                                             // arguments (constant bank) instead of per-thread arithmetic
    float* tabs_g;                           // (B, mid2_tab_floats(Nc)) hunk-stage tables when lay.gt (kernel template GT), else unused
    int B, nsplit;                           // (kernel template CL: launched as clusters of two CTAs) commits of the launch; the first
                                             // `nsplit` commits of the cost order (short index files first) are shared by the two CTAs
                                             // of a cluster -- row halves of the four hunk sweeps --, the rest take one CTA each
    int inl;                                 // entity pair layer and its backward INSIDE this kernel (entsp.cuh: sorted prefix sums +
                                             // edge walk): RS1 / CS1p / GE are not used, the step has no ent_fwd2 / ent_bwd2 launch and
                                             // this kernel follows the previous step's optimizer kernel (weights are read after pdl_wait)
};

// fixed-order block sum for M2_T threads; every thread gets the result
__device__ __forceinline__ float mid2_block_sum(float v, float* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < M2_NW; ++w) t += scratch[w];
    return t;
}

// y[m] += sum_q x[q] * W[q][m]        (W: 20 x 20 row-major in shared memory, 16-byte aligned; thread-private x, y)
__device__ __forceinline__ void gemv20(float (&y)[HD], const float (&x)[HD], const float* W) {
#pragma unroll
    for (int q = 0; q < HD; ++q) {
#pragma unroll
        for (int j = 0; j < 5; ++j) {
            const float4 w = *reinterpret_cast<const float4*>(W + q * HD + 4 * j);
            y[4 * j] = fmaf(x[q], w.x, y[4 * j]); y[4 * j + 1] = fmaf(x[q], w.y, y[4 * j + 1]);
            y[4 * j + 2] = fmaf(x[q], w.z, y[4 * j + 2]); y[4 * j + 3] = fmaf(x[q], w.w, y[4 * j + 3]);
        }
    }
}
// y[q] = sum_m W[q][m] * x[m]          (multiply by W^T)
__device__ __forceinline__ void gemv20t(float (&y)[HD], const float (&x)[HD], const float* W) {
#pragma unroll
    for (int q = 0; q < HD; ++q) {
        float acc = 0.f;
#pragma unroll
        for (int j = 0; j < 5; ++j) {
            const float4 w = *reinterpret_cast<const float4*>(W + q * HD + 4 * j);
            acc = fmaf(w.x, x[4 * j], acc); acc = fmaf(w.y, x[4 * j + 1], acc);
            acc = fmaf(w.z, x[4 * j + 2], acc); acc = fmaf(w.w, x[4 * j + 3], acc);
        }
        y[q] = acc;
    }
}
// y[k4 .. k4+3] = init + sum_q x[q] W[q][k4 ..]      (x: 20 floats in shared memory, 16-byte aligned; one quarter-row per thread)
__device__ __forceinline__ float4 gemv20_k4(const float* x, const float* W, int k4, float4 acc) {
#pragma unroll
    for (int q4 = 0; q4 < 5; ++q4) {
        const float4 xv = *reinterpret_cast<const float4*>(x + 4 * q4);
        const float xr[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float4 w = *reinterpret_cast<const float4*>(W + (4 * q4 + j) * HD + k4);
            acc.x = fmaf(xr[j], w.x, acc.x); acc.y = fmaf(xr[j], w.y, acc.y); acc.z = fmaf(xr[j], w.z, acc.z); acc.w = fmaf(xr[j], w.w, acc.w);
        }
    }
    return acc;
}
// y[k4 + j] = sum_m W[k4 + j][m] x[m]               (multiply by W^T)
__device__ __forceinline__ float4 gemv20t_k4(const float* x, const float* W, int k4) {
    float out[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int m4 = 0; m4 < 5; ++m4) {
        const float4 xv = *reinterpret_cast<const float4*>(x + 4 * m4);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float4 w = *reinterpret_cast<const float4*>(W + (k4 + j) * HD + 4 * m4);
            out[j] = fmaf(w.x, xv.x, out[j]); out[j] = fmaf(w.y, xv.y, out[j]); out[j] = fmaf(w.z, xv.z, out[j]); out[j] = fmaf(w.w, xv.w, out[j]);
        }
    }
    return make_float4(out[0], out[1], out[2], out[3]);
}
__device__ __forceinline__ void load20s(float (&v)[HD], const float* src) {      // 16-byte aligned source
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        const float4 t = reinterpret_cast<const float4*>(src)[j];
        v[4 * j] = t.x; v[4 * j + 1] = t.y; v[4 * j + 2] = t.z; v[4 * j + 3] = t.w;
    }
}
__device__ __forceinline__ void store20s(float* dst, const float (&v)[HD]) {
#pragma unroll
    for (int j = 0; j < 5; ++j) reinterpret_cast<float4*>(dst)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
}
// acc[4 i + j] += sum_{n = n0, n0 + 16, ... < nn} A[n][a0 + i] * B[n][b0 + j]     (4 x 4 register tile of A^T B)
__device__ __forceinline__ void tile_acc(float (&acc)[16], const float* A, int lda, const float* B, int ldb, int a0, int b0,
                                         int n0, int nn) {
    for (int n = n0; n < nn; n += 16) {
        const float4 av = *reinterpret_cast<const float4*>(A + (size_t)n * lda + a0);
        const float4 bv = *reinterpret_cast<const float4*>(B + (size_t)n * ldb + b0);
        const float ar[4] = {av.x, av.y, av.z, av.w}, br[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[4 * i + j] = fmaf(ar[i], br[j], acc[4 * i + j]);
    }
}
// Transpose-reduce 16 per-lane values over the 16 lanes of a half warp (xor 8, 4, 2, 1): returns the
// total of value (lane & 15).  Fixed exchange order.
__device__ __forceinline__ float reduce16(const float (&v)[16], int lane) {
    const unsigned hm16 = (lane & 16) ? 0xffff0000u : 0x0000ffffu;     // the two half warps may be in different branches
    float a[8], b4[4], c[2];
    const bool h8 = lane & 8, h4 = lane & 4, h2 = lane & 2, h1 = lane & 1;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const float keep = h8 ? v[i + 8] : v[i], send = h8 ? v[i] : v[i + 8];
        a[i] = keep + __shfl_xor_sync(hm16, send, 8);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float keep = h4 ? a[i + 4] : a[i], send = h4 ? a[i] : a[i + 4];
        b4[i] = keep + __shfl_xor_sync(hm16, send, 4);
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const float keep = h2 ? b4[i + 2] : b4[i], send = h2 ? b4[i] : b4[i + 2];
        c[i] = keep + __shfl_xor_sync(hm16, send, 2);
    }
    const float keep = h1 ? c[1] : c[0], send = h1 ? c[0] : c[1];
    return keep + __shfl_xor_sync(hm16, send, 1);
}
// sum over the 16 lanes of a half warp, every lane gets the total
__device__ __forceinline__ float half_sum(float v) {
    const unsigned hm16 = (threadIdx.x & 16) ? 0xffff0000u : 0x0000ffffu;
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(hm16, v, o);
    return v;
}
// dst[0..n] = exclusive prefix sums of src[0], src[stride], ... (dst[n] = total); executed by ONE warp, fixed order
__device__ __forceinline__ void warp_excl_scan(float* dst, const float* src, int stride, int n, int lane) {
    const int per = (n + 31) >> 5, lo = min(lane * per, n), hi = min(lo + per, n);
    float sum = 0.f;
    for (int i = lo; i < hi; ++i) sum += src[(size_t)i * stride];
    float incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const float t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    float run = incl - sum;
    for (int i = lo; i < hi; ++i) { dst[i] = run; run += src[(size_t)i * stride]; }
    if (lane == 31) dst[n] = incl;
}
// number of set bits of a bitmap row in columns [ja, jb)
__device__ __forceinline__ int range_popc(const uint32_t* row, int ja, int jb) {
    if (jb <= ja) return 0;
    const int wa = ja >> 5, wb = (jb - 1) >> 5;
    int c = 0;
    for (int w = wa; w <= wb; ++w) {
        uint32_t v = row[w];
        if (w == wa) v &= 0xffffffffu << (ja & 31);
        if (w == wb) { const int e = jb - (wb << 5); if (e < 32) v &= (1u << e) - 1u; }
        c += __popc(v);
    }
    return c;
}
// sum_{p' < p} v[p' + (p' >= g)]  from the exclusive prefix PV of v  (off-diagonal enumeration of row g)
__device__ __forceinline__ float offdiag_prefix(const float* PV, const float* v, int vstride, int g, int p) {
    return p > g ? PV[p + 1] - v[(size_t)g * vstride] : PV[p];
}
// element k of row n of a [n][KG][2][4] table (half 0)
__device__ __forceinline__ int p01_idx(int n, int k) { return n * PROW + (k >> 2) * 8 + (k & 3); }

#define M2_PHASE(i) do { if (a.clk && tid == 0) a.clk[(size_t)b * 24 + (i)] = clock64(); } while (0)

// GT: the hunk-stage tables are addressed in global memory (a.tabs_g, this commit's private slice: written and read by this CTA
// only, ordered by the block barriers) -- same code, generic loads / stores instead of shared ones
// CL: the grid is launched as clusters of two CTAs so that a batch below one wave still occupies the SMs.  A cluster either
// SHARES one commit (both CTAs run every phase redundantly on identical state, except the four hunk sweeps, of which each takes
// half the rows; row sums, column partials and the scalar sums cross through distributed shared memory and are added in rank
// order, so both CTAs -- and any other launch geometry -- hold bitwise the same values; rank 0 writes the outputs) or holds two
// independent commits (no cluster barrier is ever executed in such a cluster).
template <int CWT, bool TRAIN, bool GT, bool CL>
__global__ void __launch_bounds__(M2_T, 1) mid2_kernel(const Mid2Args a) {
    extern __shared__ __align__(128) unsigned char sm_raw[];
    float* sm = reinterpret_cast<float*>(sm_raw);
    const int Ne = a.Ne, Nc = a.Nc, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int b = blockIdx.x;
    bool split = false, wr = true;          // wr: this CTA writes the commit's global outputs
    uint32_t crank = 0;
    if constexpr (CL) {
        if (a.wait_flag) {                  // the commit assignment reads L: wait for the staged inputs first (see phase A)
            if (tid == 0) {
                unsigned int spin = 0;
                while (*reinterpret_cast<const volatile int*>(a.wait_flag) != a.wait_tag) {
                    __nanosleep(spin < 16 ? 64 : 2000);
                    if (++spin > (1u << 22)) __trap();
                }
                asm volatile("fence.acq_rel.sys;" ::: "memory");       // the data were written before the tag
            }
            __syncthreads();
        }
        // cost order: commits with a short index file (2 <= L < Ne: the O(L^2) pooling gathers) first, otherwise by index
        uint32_t* gen_w = reinterpret_cast<uint32_t*>(sm + a.lay.red);       // [8] (no static shared memory: the dynamic size is the opt-in maximum)
        int* role = reinterpret_cast<int*>(gen_w + 8);                       // [2]
        crank = cluster_ctarank();
        const int nw = (a.B + 31) >> 5;
        if (warp < nw) {
            const int i = warp * 32 + lane;
            const int Li = i < a.B ? a.L[i] : Ne;
            const uint32_t bal = __ballot_sync(0xffffffffu, i < a.B && Li < Ne && Li >= 2);
            if (lane == 0) gen_w[warp] = bal;
        }
        __syncthreads();
        if (tid == 0) {
            const int c = blockIdx.x >> 1, S = a.nsplit;
            const int idx = c < S ? c : S + 2 * (c - S) + (int)crank;
            int commit = -1;
            if (idx < a.B) {
                int G = 0;
                for (int w = 0; w < nw; ++w) G += __popc(gen_w[w]);
                const bool gen = idx < G;
                int k = gen ? idx : idx - G;                 // k-th commit of its class, in index order
                for (int w = 0; w < nw && commit < 0; ++w) {
                    const uint32_t valid = (w + 1) * 32 <= a.B ? 0xffffffffu : (1u << (a.B - w * 32)) - 1u;
                    uint32_t m = gen ? gen_w[w] : ~gen_w[w] & valid;
                    const int pc = __popc(m);
                    if (k < pc) { for (int t = 0; t < k; ++t) m &= m - 1u; commit = w * 32 + __ffs(m) - 1; }
                    k -= pc;
                }
            }
            role[0] = commit; role[1] = c < S ? 1 : 0;
        }
        __syncthreads();
        b = role[0]; split = role[1] != 0;
        if (b < 0) return;                  // odd number of unshared commits: the last cluster's second CTA has nothing to do
        wr = !split || crank == 0;
    }
    const int Nh = (Nc + 1) >> 1;           // hunk-grid rows of rank 0 of a sharing cluster
    const int hr0 = split && crank ? Nh : 0, hr1 = split && !crank ? Nh : Nc;      // this CTA's rows in the four hunk sweeps
    const int kg = warp % KG, rg = warp / KG, k0 = kg * 4;
    const int WPe = a.WPe, WPc = a.WPc;
    const Mid2Smem& L_ = a.lay;
    float* blk1 = sm + L_.blk1; float* blk2 = sm + L_.blk2;
    float* W5 = blk1; float* b5 = blk1 + 400; float* U1 = blk1 + 420; float* c1 = blk1 + 840;
    float* u2 = blk1 + 860; float* c2 = blk1 + 880;
    float* V1 = blk2; float* d1 = blk2 + 200; float* W2 = blk2 + 220; float* b2 = blk2 + 620;
    float* G1 = blk2 + 640; float* g1b = blk2 + 1080; float* G2 = blk2 + 1100; float* gb2 = blk2 + 1140;
    float* gam = sm + L_.gam; float* Dh = sm + L_.Dh; float* Dg = sm + L_.Dg; float* G1g = sm + L_.G1g;
    float* W5U = sm + L_.W5U; float* c1p = sm + L_.c1p;
    float* xs = sm + L_.x; float* x2 = sm + L_.x2; int* hm = reinterpret_cast<int*>(sm + L_.hm);
    float* SP = sm + L_.SP; float* TP = sm + L_.TP; float* dl = sm + L_.dl; float* dx2 = sm + L_.dx2;
    float* nb = sm + L_.nb; float* dnb = sm + L_.dnb;
    uint32_t* ebits = reinterpret_cast<uint32_t*>(sm + L_.ebits);
    uint32_t* ybits = reinterpret_cast<uint32_t*>(sm + L_.ybits);
    float* scratch = sm + L_.scratch; float* red = sm + L_.red;
    float* uni = sm + L_.uni;
    // S (entity effect sums, forward -> backward), later GE: its own region, or (wide GT shapes) this commit's rows of a.GE
    float* SC = (GT && L_.scg) ? a.GE + (size_t)b * Ne * HD : sm + L_.sc;
    // hunk-stage tables: union region, or (GT) this commit's slice of global memory -- there the slice also holds the neighbour
    // counts of the class-table entity stage while the hunk tables are not live
    float* tabs = GT ? a.tabs_g + (size_t)b * mid2_tab_floats(Nc) : uni;
    float* stg = sm + L_.stg;
    auto stage_rows = [&](float* dst, const float* src, int nfl) {       // nfl: multiple of 4, both 16-byte aligned
        for (int e = tid; e < (nfl >> 2); e += M2_T) reinterpret_cast<float4*>(dst)[e] = reinterpret_cast<const float4*>(src)[e];
    };
    uint64_t* bar = reinterpret_cast<uint64_t*>(sm + L_.total);
    const float* par = a.params;
    const ParamOff& po = a.po;
    const int ch = reduce4_channel(lane);
    const bool LOGITS = a.logits != nullptr;
    float* dbg = a.dbg ? a.dbg + (size_t)b * mid2_dbg_floats(Ne, Nc) : nullptr;
    // gradient partials of the commit; the second CTA of a sharing cluster computes the same values and parks them in a spare row
    float* gp = a.gpart ? a.gpart + (size_t)(wr ? b : a.B + (int)(blockIdx.x >> 1)) * a.total : nullptr;
    // exchange after a split sweep: the peer's rows of RS are copied in, the column partials CS (Nc x 20 <= M2_T float4) and a
    // small vector `sv` (n <= 64 floats, may be null) become rank 0's + rank 1's on both CTAs (`CS` is any array of ncs4 float4)
    auto xchg = [&](float* RS, float* CS, int ncs4, float* sv, int n) {
        cluster_sync_all();                                     // both partials are complete
        const uint32_t peer = crank ^ 1u;
        const int pr0 = crank ? 0 : Nh, pr1 = crank ? Nh : Nc;  // the peer's rows
        if (RS) {
            const uint32_t prs = peer_smem(RS + (size_t)pr0 * HD, peer);
            for (int e = tid; e < (pr1 - pr0) * (HD / 4); e += M2_T) reinterpret_cast<float4*>(RS + (size_t)pr0 * HD)[e] = ld_peer4(prs + 16u * e);
        }
        float4 pc = make_float4(0.f, 0.f, 0.f, 0.f);
        const bool have = CS && tid < ncs4;                      // ncs4 <= M2_T float4 of column partials
        if (have) pc = ld_peer4(peer_smem(CS, peer) + 16u * tid);
        float ps = 0.f;
        const bool hs = sv && tid >= M2_T - 64 && tid - (M2_T - 64) < n;
        if (hs) ps = ld_peer(peer_smem(sv, peer) + 4u * (tid - (M2_T - 64)));
        cluster_sync_all();                                     // both have read the other's partials
        if (have) {
            const float4 own = reinterpret_cast<float4*>(CS)[tid];
            const float4 lo = crank ? pc : own, hi = crank ? own : pc;
            reinterpret_cast<float4*>(CS)[tid] = make_float4(lo.x + hi.x, lo.y + hi.y, lo.z + hi.z, lo.w + hi.w);
        }
        if (hs) { const float own = sv[tid - (M2_T - 64)]; sv[tid - (M2_T - 64)] = crank ? ps + own : own + ps; }
        __syncthreads();
    };
    M2_PHASE(0);

    // ---------------- A. label bitmaps (TMA), weights and per-commit vectors -> shared memory ------
    if (!CL && a.wait_flag) {               // (the cluster form has waited before it assigned the commits)
        // Host-fed step: the inputs are copied on the library's copy stream.  A cross-stream event wait in front of this
        // kernel would undo its programmatic launch behind the optimizer kernel, so the copy stream's LAST DMA writes a tag
        // and the kernel polls it here (the copies were enqueued a whole step earlier: the first poll normally succeeds).
        if (tid == 0) {
            unsigned int spin = 0;
            while (*reinterpret_cast<const volatile int*>(a.wait_flag) != a.wait_tag) {
                __nanosleep(spin < 16 ? 64 : 2000);
                if (++spin > (1u << 22)) __trap();          // ~8 s without the copy: a lost DMA traps instead of hanging the GPU
            }
            asm volatile("fence.acq_rel.sys;" ::: "memory");
        }
        __syncthreads();
    }
    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
        const uint32_t be = (uint32_t)Ne * WPe * 4, bc = (uint32_t)Nc * WPc * 4;
        mbar_arrive_expect_tx(bar, be + bc);
        bulk_g2s(ebits, a.ebits + (size_t)b * Ne * WPe, be, bar);
        bulk_g2s(ybits, a.ybits + (size_t)b * Nc * WPc, bc, bar);
    }
    // per-commit inputs: in flight together with the weight loads below (Ne <= 512 < M2_T: one element per thread)
    const int Lb = min(max(a.L[b], 0), Ne);      // 0 <= L <= Ne is the ABI's contract; clamped so a bad value cannot index out of the tile
    const int h_in = tid < Ne ? a.hmap[(size_t)b * Ne + tid] : -1;
    const float x_in = tid < Ne ? a.x[(size_t)b * Ne + tid] : 0.f;
    // Weights -> shared memory and the tables derived from them.  With the entity stage inline this kernel follows the
    // previous step's optimizer kernel, so the weights are read after pdl_wait (below); otherwise its predecessor is
    // ent_fwd2, which does not write them, and the loads overlap that kernel's tail.
    float* wE = sm + L_.entw;                   // inline entity stage: U[20] V[20] c[20] D[20] (model_2.py:167-170)
    float* blkE = sm + L_.blkE; float* wEe = sm + L_.wEe; float* gamE = sm + L_.gamE; float* DgE = sm + L_.DgE;     // variant 4
    const float nb5 = 2.f * (float)(Ne - 1);
    auto load_weights = [&]() {
        {   // both weight blocks with all global loads in flight before the first store
            const float* p1 = par + (a.ent ? po.ent_w5 : po.hnk_w1);
            const float* p2 = par + po.hnk_w1;
            const int n1 = a.ent ? M2_BLK1 : 0;
            constexpr int NLD = (M2_BLK1 + M2_BLK2 + M2_T - 1) / M2_T;
            float v[NLD];
#pragma unroll
            for (int u = 0; u < NLD; ++u) {
                const int idx = tid + u * M2_T;
                v[u] = idx < n1 ? p1[idx] : (idx < n1 + M2_BLK2 ? p2[idx - n1] : 0.f);
            }
            if (a.edge) for (int i = tid; i < M2_BLKE; i += M2_T) blkE[i] = par[po.edg_w11 + i];
            float e0 = 0.f, e1 = 0.f, e2 = 0.f;
            if (a.inl && tid < HD) {
                e0 = par[po.ent_w1 + 2 * HD + tid]; e1 = par[po.ent_w1 + 3 * HD + tid]; e2 = par[po.ent_b1 + tid];
                wE[tid] = par[po.ent_w1 + tid]; wE[HD + tid] = par[po.ent_w1 + HD + tid];
                wE[2 * HD + tid] = e2 + e0; wE[3 * HD + tid] = e1 - e0;
            }
#pragma unroll
            for (int u = 0; u < NLD; ++u) {
                const int idx = tid + u * M2_T;
                if (idx < n1) blk1[idx] = v[u];
                else if (idx < n1 + M2_BLK2) blk2[idx - n1] = v[u];
            }
        }
        __syncthreads();
        if (tid < HD) {
            gam[tid] = G2[2 * tid + 1] - G2[2 * tid];
            Dh[tid] = V1[9 * HD + tid] - V1[8 * HD + tid];
            Dg[tid] = G1[HD + tid] - G1[tid];
        }
        if (a.edge && tid < HD) {
            // edge-branch first layer, tied weights (model_4.py:219-222): pre = w11 (x_i + x_j) + b1 + W12[l]
            wEe[tid] = blkE[tid]; wEe[HD + tid] = blkE[tid];
            wEe[2 * HD + tid] = blkE[60 + tid] + blkE[20 + tid]; wEe[3 * HD + tid] = blkE[40 + tid] - blkE[20 + tid];
            gamE[tid] = blkE[960 + 2 * tid + 1] - blkE[960 + 2 * tid];
            DgE[tid] = blkE[500 + HD + tid] - blkE[500 + tid];
        }
        if (TRAIN) for (int e = tid; e < 400; e += M2_T) G1g[e] = G1[2 * HD + e] * (G2[2 * (e % HD) + 1] - G2[2 * (e % HD)]);
        if (a.ent) {
            // the entity effect layer (x W5 + (Ne-1) 2 b5, model_2.py:172-175 after aggregation) and the first layer of
            // the entity-state MLP compose into one 20 x 20 map: Z = c1' + x U1[0] + S W5U
            for (int e = tid; e < 420; e += M2_T) {
                float acc = 0.f;
                if (e < 400) {
                    const int q = e / HD, k = e - q * HD;
#pragma unroll
                    for (int m = 0; m < HD; ++m) acc = fmaf(W5[q * HD + m], U1[(1 + m) * HD + k], acc);
                    W5U[e] = acc;
                } else {
                    const int k = e - 400;
#pragma unroll
                    for (int m = 0; m < HD; ++m) acc = fmaf(b5[m], U1[(1 + m) * HD + k], acc);
                    c1p[k] = fmaf(nb5, acc, c1[k]);
                }
            }
        }
        __syncthreads();
    };
    if (tid < Ne) {
        hm[tid] = (h_in >= 0 && h_in < Nc) ? h_in : -1;
        xs[tid] = x_in;
        if (!a.ent) x2[tid] = x_in;
    }
    if (!a.inl) load_weights(); else __syncthreads();
    // ---- everything that depends on the inputs only (bitmaps, hunk ids, L) is done BEFORE the dependency on ent_fwd2:
    // under programmatic dependent launch it overlaps that kernel's tail
    const int nm1 = Ne - 1;
    const bool ident = Lb == Ne;
    int* horder = reinterpret_cast<int*>(dx2);          // index lines sorted by hunk id, ascending within a hunk (dx2 is dead until K)
    int* hstart = reinterpret_cast<int*>(dnb);          // [Nc + 1] list offsets (dnb is dead until J)
    mbar_wait(bar, 0);
    {
        // (1) stable counting sort of the index lines by hunk id.  Warp w owns the lines 32 w .. 32 w + 31: match_any
        // gives every line its rank among the equal keys of the warp, the per-warp counts are laid out [warp][hunk],
        // thread c turns them into bases, one warp scans the hunk totals.
        const int WU = (Ne + 31) >> 5, NLW = (Lb + 31) >> 5;        // used bitmap words per row; warps holding index lines
        uint32_t* cparts = reinterpret_cast<uint32_t*>(scratch);    // [8 row parts][WU][8] byte counters (column degrees)
        int* wcnt = reinterpret_cast<int*>(scratch) + 8 * WU * 8;   // [NLW][Nc]
        int* hcnt = reinterpret_cast<int*>(red);                    // [Nc]
        for (int e = tid; e < NLW * Nc; e += M2_T) wcnt[e] = 0;
        __syncthreads();
        int key = -1, rank = 0;
        for (int w0 = 0; w0 < NLW; w0 += M2_NW) {                   // one round unless L > 32 * 20
            const int w = w0 + warp, i = w * 32 + lane;
            if (w < NLW) {
                key = i < Lb ? hm[i] : -1;
                const uint32_t peers = __match_any_sync(0xffffffffu, key);
                rank = __popc(peers & ((1u << lane) - 1u));
                if (key >= 0 && rank == 0) wcnt[w * Nc + key] = __popc(peers);
            }
        }
        // (2) degrees (only the closed-form pooling uses them).  Rows: one thread per row.  Columns, bit-sliced: thread
        // (row part, word, k) adds (w >> k) & 0x01010101 over its rows -- four column counters in the bytes of one
        // register -- and the eight row parts are summed per column afterwards.  No votes, no warp reductions.
        if (ident && !a.inl) {
            for (int i = tid; i < Ne; i += M2_T) {
                int c = 0;
                for (int w = 0; w < WU; ++w) c += __popc(ebits[i * WPe + w]);
                SP[4 * i + 3] = (float)c;
            }
            const int rows_per = (Ne + 7) >> 3;                     // <= 64: no byte overflow
            for (int t = tid; t < 8 * WU * 8; t += M2_T) {
                const int k = t & 7, sg = (t >> 3) % WU, rp = t / (8 * WU);
                const int r0 = rp * rows_per, r1 = min(r0 + rows_per, Ne);
                uint32_t acc = 0u;
                for (int r = r0; r < r1; ++r) acc += (ebits[r * WPe + sg] >> k) & 0x01010101u;
                cparts[t] = acc;
            }
        }
        __syncthreads();
        if (ident && !a.inl) {
            for (int j = tid; j < Ne; j += M2_T) {
                const int sg = j >> 5, bit = j & 31, k = bit & 7, sh = (bit >> 3) * 8;
                int cd = 0;
#pragma unroll
                for (int rp = 0; rp < 8; ++rp) cd += (cparts[(rp * WU + sg) * 8 + k] >> sh) & 0xffu;
                TP[4 * j + 3] = (float)cd;
            }
        }
        if (tid < Nc) {                                             // per-warp counts -> bases within the hunk, hunk total
            int run = 0;
            for (int w = 0; w < NLW; ++w) { const int c = wcnt[w * Nc + tid]; wcnt[w * Nc + tid] = run; run += c; }
            hcnt[tid] = run;
        }
        __syncthreads();
        if (warp == 0) {                                            // exclusive scan of the hunk totals (Nc <= 256: 8 per lane)
            const int per = (Nc + 31) >> 5, lo = min(lane * per, Nc), hi = min(lo + per, Nc);
            int sum = 0;
            for (int c = lo; c < hi; ++c) sum += hcnt[c];
            int incl = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
            int run = incl - sum;
            for (int c = lo; c < hi; ++c) { hstart[c] = run; run += hcnt[c]; }
            if (lane == 31) hstart[Nc] = incl;
        }
        __syncthreads();
        if (NLW <= M2_NW) {
            if (warp < NLW && key >= 0) horder[hstart[key] + wcnt[warp * Nc + key] + rank] = warp * 32 + lane;
        } else {                                                    // more index lines than one round of warps: recompute the ranks
            for (int w = warp; w < NLW; w += M2_NW) {
                const int i = w * 32 + lane, ky = i < Lb ? hm[i] : -1;
                const uint32_t peers = __match_any_sync(0xffffffffu, ky);
                if (ky >= 0) horder[hstart[ky] + wcnt[w * Nc + ky] + __popc(peers & ((1u << lane) - 1u))] = i;
            }
        }
    }
    // ---- inline entity stage, input-only half (entsp.cuh): nodes sorted by attribute, suffix sums, transposed bitmap,
    // edge prefix counts by row and by column
    float* xsort = sm + L_.xsort; int* ordv = reinterpret_cast<int*>(sm + L_.ordv); float* SXs = sm + L_.sx;
    int* rptr = reinterpret_cast<int*>(sm + L_.rptr); int* cptr = reinterpret_cast<int*>(sm + L_.cptr);
    uint32_t* ebT = reinterpret_cast<uint32_t*>(sm + L_.ebt);      // [Ne][WPe]: bit i of row j = A_ij
    // attribute classes: the distinct values of x in ascending order.  With at most m_max of them the pair layer is evaluated
    // from per-class tables and per-(node, class) neighbour counts (popcounts), see below; otherwise by search + edge walk
    int* clsv = reinterpret_cast<int*>(sm + L_.cls); float* cval = sm + L_.cval; int* csize = reinterpret_cast<int*>(sm + L_.csize);
    uint32_t* cmask = reinterpret_cast<uint32_t*>(sm + L_.cmask); int* cmeta = reinterpret_cast<int*>(sm + L_.cmeta);
    // the union region must hold: forward 2 m^2 20 table floats + 4 Ne m count floats; backward the tables + Ne m packed counts +
    // 16 partial sums per thread
    const int uni_floats = L_.sc - L_.uni;
    int m_max = M2_MCLS;
    const int uni_edge = a.edge ? 2 * Ne * HD : 0;          // variant 4: the edge branch's RS / CS sit at the end of the union region
    if (GT) {       // the count tables ([Ne][m] float4 forward, [m][Ne] packed backward) sit in the global slice
        while (m_max > 0 && (2 * m_max * m_max * HD + 16 * M2_T + 4 + uni_edge > uni_floats || 4 * Ne * m_max > mid2_tab_floats(Nc))) --m_max;
    } else {
        while (m_max > 0 && (2 * m_max * m_max * HD + 4 * Ne * m_max + uni_edge > uni_floats ||
                             2 * m_max * m_max * HD + Ne * m_max + 16 * M2_T + uni_edge > uni_floats)) --m_max;
    }
    if (a.inl) {
        const int WU = (Ne + 31) >> 5;
        {   // stable rank sort: three threads per node count over a third of the nodes each (integer atomics: exact)
            int* rk = ordv;                                  // ranks accumulate here, then the rank -> node map replaces them
            for (int i = tid; i < Ne; i += M2_T) rk[i] = 0;
            __syncthreads();
            const int third = (Ne + 2) / 3;
            for (int t = tid; t < 3 * Ne; t += M2_T) {
                const int i = t % Ne, part = t / Ne, j0 = part * third, j1 = min(j0 + third, Ne);
                const float xi = xs[i];
                int r = 0;
                for (int j = j0; j < j1; ++j) { const float xj = xs[j]; r += (xj < xi || (xj == xi && j < i)) ? 1 : 0; }
                atomicAdd(&rk[i], r);
            }
        }
        for (int blk = warp; blk < WPe * WU; blk += M2_NW) {  // 32 x 32 bit blocks (row block, column word)
            const int rb = blk / WPe, cw = blk - rb * WPe, row = rb * 32 + lane;
            const uint32_t w = warp_transpose32(row < Ne ? ebits[row * WPe + cw] : 0u, lane);
            const int col = cw * 32 + lane;
            if (col < Ne) ebT[col * WPe + rb] = w;
        }
        __syncthreads();
        int myrank = 0;
        if (tid < Ne) myrank = ordv[tid];
        for (int i = tid; i < Ne; i += M2_T) {               // out- and in-degrees
            int rc = 0, cc = 0;
            for (int w = 0; w < WU; ++w) { rc += __popc(ebits[i * WPe + w]); cc += __popc(ebT[i * WPe + w]); }
            rptr[i] = rc; cptr[i] = cc;
        }
        __syncthreads();
        if (tid < Ne) { xsort[myrank] = xs[tid]; ordv[myrank] = tid; }
        if (warp == 1) warp_excl_scan_int(rptr, Ne, lane);
        if (warp == 2) warp_excl_scan_int(cptr, Ne, lane);
        for (int e = tid; e < M2_MCLS * WPe; e += M2_T) cmask[e] = 0u;
        __syncthreads();
        if (warp == 3) {                                     // class of every rank: runs of equal values in the sorted order
            const int per = (Ne + 31) >> 5, lo = min(lane * per, Ne), hi = min(lo + per, Ne);
            int cnt = 0;
            for (int r = lo; r < hi; ++r) cnt += (r == 0 || xsort[r] != xsort[r - 1]) ? 1 : 0;
            int incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
            int c = incl - cnt - 1;                          // class of the rank before this lane's chunk
            for (int r = lo; r < hi; ++r) {
                if (r == 0 || xsort[r] != xsort[r - 1]) { ++c; if (c < M2_MCLS) { cval[c] = xsort[r]; csize[c] = r; } }
                clsv[ordv[r]] = (c & 0xffff) | (r << 16);        // class of the node | its rank in the sorted order
            }
            const int m = __shfl_sync(0xffffffffu, incl, 31);
            __syncwarp();
            if (lane < M2_MCLS && lane < m) {                // run starts -> sizes
                const int start = csize[lane], next = lane + 1 < m && lane + 1 < M2_MCLS ? csize[lane + 1] : Ne;
                __syncwarp();
                csize[lane] = next - start;
            } else { __syncwarp(); }
            if (lane == 0) { cmeta[0] = m; cmeta[1] = (m <= m_max) ? 1 : 0; }
        }
        if (warp == 0) {                                     // SXs[r] = sum of the sorted attributes from rank r on, SXs[Ne] = 0
            const int per = (Ne + 31) >> 5, lo = min(lane * per, Ne), hi = min(lo + per, Ne);
            float sum = 0.f;
            for (int r = hi - 1; r >= lo; --r) sum += xsort[r];
            float incl = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const float t = __shfl_down_sync(0xffffffffu, incl, o); if (lane + o < 32) incl += t; }
            float run = incl - sum;
            for (int r = hi - 1; r >= lo; --r) { run += xsort[r]; SXs[r] = run; }
            if (lane == 0) SXs[Ne] = 0.f;
        }
        __syncthreads();
        if (cmeta[1]) {                                      // node masks of the classes: one ballot per (32 nodes, class)
            const int m = cmeta[0];
            for (int w = warp; w < WU; w += M2_NW) {
                const int node = w * 32 + lane, c = node < Ne ? (clsv[node] & 0xffff) : -1;
                for (int bcl = 0; bcl < m; ++bcl) {
                    const uint32_t bal = __ballot_sync(0xffffffffu, c == bcl);
                    if (lane == 0) cmask[bcl * WPe + w] = bal;
                }
            }
        }
    }
    __syncthreads();
    pdl_wait();                     // RS1 / CS1p come from ent_fwd2, or (inline entity stage) the weights from the previous step's optimizer
    pdl_launch_dependents();
    M2_PHASE(1);
    if (a.inl) {
        load_weights();
        M2_PHASE(16);
        // ---------------- entity pair layer forward: S_n = sum_{j != n} relu(pre_nj) + sum_{i != n} relu(pre_in) -------------
        const bool use_cls = cmeta[1] != 0;
        // w: U V c D of the layer (80 floats); outR / outC: [Ne][20] row-sum and column-sum targets (the same array: their sum);
        // counts: build the neighbour counts (first call)
        auto ent_fwd = [&](const float* w, float* outR, float* outC, bool counts) {
        const bool sum_mode = outR == outC;
        if (use_cls) {
            // CLASS TABLES (at most m_max distinct attribute values).  relu(pre_ij[k]) depends on (class of i, class of j,
            // l_ij, k) only: H_l[a][b][k] = relu(U_k val_a + V_k val_b + c_k + l D_k).  With c1o(n,b) / c1i(n,b) = number of
            // out- / in-neighbours of n in class b (popcounts of bitmap row AND class mask) and c0 = |b| - [a == b] - c1,
            //     S_n[k] = sum_b  c0o H_0[a][b] + c1o H_1[a][b] + c0i H_0[b][a] + c1i H_1[b][a],      a = class of n:
            // no search, no edge walk, every sum in class order.
            const int m = cmeta[0];
            float* H0 = uni; float* H1 = uni + m * m * HD;
            float4* cntf = reinterpret_cast<float4*>(GT ? tabs : uni + 2 * m * m * HD);      // [Ne][m]  {c0o, c1o, c0i, c1i} as floats
            for (int e = tid; e < m * m * HD; e += M2_T) {
                const int k = e % HD, ab = e / HD, bq = ab % m, aq = ab / m;
                const float t0 = fmaf(cval[bq], w[HD + k], fmaf(cval[aq], w[k], w[2 * HD + k]));
                H0[e] = fmaxf(t0, 0.f); H1[e] = fmaxf(t0 + w[3 * HD + k], 0.f);
            }
            const int WU = (Ne + 31) >> 5;
            if (counts) for (int e = tid; e < Ne * m; e += M2_T) {
                const int n = e / m, bq = e - n * m;
                int co = 0, ci = 0;
                for (int w = 0; w < WU; ++w) {
                    const uint32_t mk = cmask[bq * WPe + w];
                    co += __popc(ebits[n * WPe + w] & mk); ci += __popc(ebT[n * WPe + w] & mk);
                }
                const int cr = clsv[n], tot = csize[bq] - ((cr & 0xffff) == bq ? 1 : 0);
                cntf[bq * Ne + (cr >> 16)] = make_float4((float)(tot - co), (float)co, (float)(tot - ci), (float)ci);      // [class][rank]
            }
            __syncthreads();
            // One owner per (node, 4 channels); the lanes of a warp take CONSECUTIVE RANKS of the sorted order, i.e. mostly one
            // class: the four table loads of an iteration are (near-)uniform across the warp and the count loads are contiguous,
            // so the loop is not bound by shared-memory bandwidth.  Every sum runs in class order.
            const int k4 = 4 * (tid / (M2_T / KG));
            for (int r = tid % (M2_T / KG); r < Ne; r += M2_T / KG) {
                const int n = ordv[r], aq = clsv[n] & 0xffff;
                float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f), t4 = make_float4(0.f, 0.f, 0.f, 0.f);
                const float* hab0 = H0 + aq * m * HD + k4; const float* hab1 = H1 + aq * m * HD + k4;
                const float* hba0 = H0 + aq * HD + k4;     const float* hba1 = H1 + aq * HD + k4;
                const float4* cf = cntf + r;
                for (int bq = 0; bq < m; ++bq) {
                    const float4 c = cf[bq * Ne];
                    const float4 a0 = *reinterpret_cast<const float4*>(hab0 + bq * HD), a1 = *reinterpret_cast<const float4*>(hab1 + bq * HD);
                    const float4 b0 = *reinterpret_cast<const float4*>(hba0 + bq * m * HD), b1 = *reinterpret_cast<const float4*>(hba1 + bq * m * HD);
                    if (sum_mode) {
                        s4.x = fmaf(c.x, a0.x, s4.x); s4.x = fmaf(c.y, a1.x, s4.x); s4.x = fmaf(c.z, b0.x, s4.x); s4.x = fmaf(c.w, b1.x, s4.x);
                        s4.y = fmaf(c.x, a0.y, s4.y); s4.y = fmaf(c.y, a1.y, s4.y); s4.y = fmaf(c.z, b0.y, s4.y); s4.y = fmaf(c.w, b1.y, s4.y);
                        s4.z = fmaf(c.x, a0.z, s4.z); s4.z = fmaf(c.y, a1.z, s4.z); s4.z = fmaf(c.z, b0.z, s4.z); s4.z = fmaf(c.w, b1.z, s4.z);
                        s4.w = fmaf(c.x, a0.w, s4.w); s4.w = fmaf(c.y, a1.w, s4.w); s4.w = fmaf(c.z, b0.w, s4.w); s4.w = fmaf(c.w, b1.w, s4.w);
                    } else {        // row sums (out-neighbours) and column sums (in-neighbours) kept apart
                        s4.x = fmaf(c.x, a0.x, s4.x); s4.x = fmaf(c.y, a1.x, s4.x); t4.x = fmaf(c.z, b0.x, t4.x); t4.x = fmaf(c.w, b1.x, t4.x);
                        s4.y = fmaf(c.x, a0.y, s4.y); s4.y = fmaf(c.y, a1.y, s4.y); t4.y = fmaf(c.z, b0.y, t4.y); t4.y = fmaf(c.w, b1.y, t4.y);
                        s4.z = fmaf(c.x, a0.z, s4.z); s4.z = fmaf(c.y, a1.z, s4.z); t4.z = fmaf(c.z, b0.z, t4.z); t4.z = fmaf(c.w, b1.z, t4.z);
                        s4.w = fmaf(c.x, a0.w, s4.w); s4.w = fmaf(c.y, a1.w, s4.w); t4.w = fmaf(c.z, b0.w, t4.w); t4.w = fmaf(c.w, b1.w, t4.w);
                    }
                }
                *reinterpret_cast<float4*>(outR + (size_t)n * HD + k4) = s4;
                if (!sum_mode) *reinterpret_cast<float4*>(outC + (size_t)n * HD + k4) = t4;
            }
            __syncthreads();
        } else {
            // GENERAL attributes: sorted prefix sums for the l = 0 part, edge walk for the l = 1 pairs (entsp.cuh)
            // dense (l = 0) part: one owner thread per (node, channel pair), two binary searches per channel
            int* headrow = reinterpret_cast<int*>(sm + L_.headrow); float* headp = sm + L_.headp;
            int P2 = 1;
            while (P2 <= Ne) P2 <<= 1;
            constexpr int NSLOT = M2_T / 10;
            const int slot = tid / 10, c0 = 2 * (tid % 10);
            const float Uc[2] = {w[c0], w[c0 + 1]}, Vc[2] = {w[HD + c0], w[HD + c0 + 1]};
            const float Cc[2] = {w[2 * HD + c0], w[2 * HD + c0 + 1]}, Dc[2] = {w[3 * HD + c0], w[3 * HD + c0 + 1]};
            const int WU = (Ne + 31) >> 5;
            for (int n = slot; n < Ne; n += NSLOT) {
                const float xn = xs[n];
                float pb[2], qb[2];
#pragma unroll
                for (int h = 0; h < 2; ++h) { pb[h] = fmaf(xn, Uc[h], Cc[h]); qb[h] = fmaf(xn, Vc[h], Cc[h]); }
                int r[4] = {0, 0, 0, 0};
                const float sw[4] = {Vc[0], Vc[1], Uc[0], Uc[1]}, sb[4] = {pb[0], pb[1], qb[0], qb[1]};
                for (int step = P2 >> 1; step > 0; step >>= 1) {        // the four searches advance together
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int probe = r[u] + step - 1;
                        const float xv = xsort[probe < Ne ? probe : Ne - 1];
                        const bool act = fmaf(xv, sw[u], sb[u]) > 0.f;
                        if (probe < Ne && act != (sw[u] >= 0.f)) r[u] += step;
                    }
                }
                float acc[2], acd[2];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    float cnt, sx;
                    entsp_active(r[h], Ne, Vc[h] >= 0.f, SXs, cnt, sx);
                    acc[h] = fmaf(cnt, pb[h], Vc[h] * sx) - fmaxf(fmaf(xn, Vc[h], pb[h]), 0.f);
                    entsp_active(r[2 + h], Ne, Uc[h] >= 0.f, SXs, cnt, sx);
                    acd[h] = fmaf(cnt, qb[h], Uc[h] * sx) - fmaxf(fmaf(xn, Uc[h], qb[h]), 0.f);
                }
                if (sum_mode) {
                    *reinterpret_cast<float2*>(outR + (size_t)n * HD + c0) = make_float2(acc[0] + acd[0], acc[1] + acd[1]);
                } else {
                    *reinterpret_cast<float2*>(outR + (size_t)n * HD + c0) = make_float2(acc[0], acc[1]);
                    *reinterpret_cast<float2*>(outC + (size_t)n * HD + c0) = make_float2(acd[0], acd[1]);
                }
            }
            __syncthreads();
            M2_PHASE(20);
            // l = 1 pairs, edge by edge: pass 0 walks the rows (edges n -> j add to S_n), pass 1 the transposed bitmap (edges
            // i -> n).  Every slot of 10 threads takes an equal share of the edges in row-major order; a slot adds the sums of
            // the rows that START inside its share directly, the partial sum of its first row goes through headp and is
            // added afterwards in slot order (fixed order, one writer per row at a time).
            for (int pass = 0; pass < 2; ++pass) {
                const uint32_t* bm = pass ? ebT : ebits;
                const int* ptr = pass ? cptr : rptr;
                float* Sall = pass ? outC : outR;
                const float Wo[2] = {pass ? Vc[0] : Uc[0], pass ? Vc[1] : Uc[1]}, Wn[2] = {pass ? Uc[0] : Vc[0], pass ? Uc[1] : Vc[1]};
                const int nnz = ptr[Ne], per = (nnz + NSLOT - 1) / NSLOT, e0 = min(slot * per, nnz), e1 = min(e0 + per, nnz);
                int hrow = -1;
                float h0 = 0.f, h1 = 0.f;
                if (e1 > e0) {
                    const EdgeCursor cur = edge_seek(bm, WPe, ptr, Ne, P2, e0);
                    int row = cur.row, w = cur.w;
                    uint32_t bits = cur.bits;
                    float xo = xs[row], b0 = fmaf(xo, Wo[0], Cc[0]), b1 = fmaf(xo, Wo[1], Cc[1]), a0 = 0.f, a1 = 0.f;
                    bool first = true;
                    for (int e = e0; e < e1; ++e) {
                        while (!bits) {
                            if (++w == WU) {
                                if (first) { hrow = row; h0 = a0; h1 = a1; first = false; }
                                else { float2* d = reinterpret_cast<float2*>(Sall + (size_t)row * HD + c0); const float2 o = *d; *d = make_float2(o.x + a0, o.y + a1); }
                                a0 = 0.f; a1 = 0.f; w = 0; ++row;
                                xo = xs[row]; b0 = fmaf(xo, Wo[0], Cc[0]); b1 = fmaf(xo, Wo[1], Cc[1]);
                            }
                            bits = bm[row * WPe + w];
                        }
                        const float xv = xs[(w << 5) + __ffs(bits) - 1];
                        bits &= bits - 1;
                        const float t0 = fmaf(xv, Wn[0], b0), t1 = fmaf(xv, Wn[1], b1);
                        a0 += fmaxf(t0 + Dc[0], 0.f) - fmaxf(t0, 0.f);
                        a1 += fmaxf(t1 + Dc[1], 0.f) - fmaxf(t1, 0.f);
                    }
                    if (first) { hrow = row; h0 = a0; h1 = a1; }
                    else { float2* d = reinterpret_cast<float2*>(Sall + (size_t)row * HD + c0); const float2 o = *d; *d = make_float2(o.x + a0, o.y + a1); }
                }
                if (c0 == 0) headrow[slot] = hrow;
                *reinterpret_cast<float2*>(headp + slot * HD + c0) = make_float2(h0, h1);
                __syncthreads();
                if (hrow >= 0 && (slot == 0 || headrow[slot - 1] != hrow)) {
                    float s0 = 0.f, s1 = 0.f;
                    for (int t = slot; t < NSLOT && headrow[t] == hrow; ++t) {
                        const float2 v = *reinterpret_cast<const float2*>(headp + t * HD + c0);
                        s0 += v.x; s1 += v.y;
                    }
                    float2* d = reinterpret_cast<float2*>(Sall + (size_t)hrow * HD + c0);
                    const float2 o = *d;
                    *d = make_float2(o.x + s0, o.y + s1);
                }
                __syncthreads();
                M2_PHASE(21 + pass);
            }
        }
        };
        ent_fwd(wE, SC, SC, true);
        if (a.edge) {
            // ---------------- variant 4: entity-edge branch forward (model_4.py:92-94, 206-304) -----------------------------
            // pair sums of relu(w11 (x_i + x_j) + b1 + W12[l_ij]) by the same machinery, rows and columns kept apart
            float* RSs = uni + uni_floats - 2 * Ne * HD; float* CSs = RSs + Ne * HD;
            ent_fwd(wEe, RSs, CSs, false);
            M2_PHASE(20);
            float* rse_g = a.RSEg + (size_t)b * Ne * HD; float* cse_g = a.CSEg + (size_t)b * Ne * HD;
            float* re_g = a.REg + (size_t)b * Ne * HD;   float* ce_g = a.CEg + (size_t)b * Ne * HD;
            if (TRAIN) for (int i = tid; i < Ne * 5; i += M2_T) {      // kept for the backward
                reinterpret_cast<float4*>(rse_g)[i] = reinterpret_cast<const float4*>(RSs)[i];
                reinterpret_cast<float4*>(cse_g)[i] = reinterpret_cast<const float4*>(CSs)[i];
            }
            // second (linear) layer on the sums and the tables of the soft-edge head (model_4.py:225-240, 292-297):
            //   r_n = (Ne-1) b2 + RSe_n W2,  PRe_n = b1h + G1[0] + r_n G1e;   c_n = (Ne-1) b2 + CSe_n W2,  PCe_n = c_n G1e
            const float* W2e = blkE + 80; const float* b2e = blkE + 480; const float* G1E = blkE + 500; const float* g1be = blkE + 940;
            float* PRe01 = uni; float* PCe = uni + Ne * PROW; float* rtmp = PCe + Ne * HD;       // rtmp [M2_T / KG][20]
            for (int it0 = 0; it0 < 2 * Ne; it0 += M2_T / KG) {
                const int t = it0 + tid / KG, k4 = 4 * (tid % KG);
                const bool live = t < 2 * Ne, cside = t >= Ne;
                const int n = cside ? t - Ne : t;
                if (live) {
                    const float fn1 = (float)(Ne - 1);
                    const float4 bb = *reinterpret_cast<const float4*>(b2e + k4);
                    const float4 r4 = gemv20_k4((cside ? CSs : RSs) + n * HD, W2e, k4, make_float4(fn1 * bb.x, fn1 * bb.y, fn1 * bb.z, fn1 * bb.w));
                    *reinterpret_cast<float4*>(rtmp + (tid / KG) * HD + k4) = r4;
                    if (TRAIN) *reinterpret_cast<float4*>((cside ? ce_g : re_g) + n * HD + k4) = r4;
                }
                __syncthreads();
                if (live) {
                    float4 init = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (!cside) {
                        const float4 g = *reinterpret_cast<const float4*>(g1be + k4), g0 = *reinterpret_cast<const float4*>(G1E + k4);
                        init = make_float4(g.x + g0.x, g.y + g0.y, g.z + g0.z, g.w + g0.w);
                    }
                    const float4 pq = gemv20_k4(rtmp + (tid / KG) * HD, G1E + 2 * HD, k4, init);
                    if (cside) {
                        *reinterpret_cast<float4*>(PCe + n * HD + k4) = pq;
                    } else {
                        const float4 d = *reinterpret_cast<const float4*>(DgE + k4);
                        float* dst = PRe01 + (size_t)n * PROW + 2 * k4;
                        *reinterpret_cast<float4*>(dst) = pq;
                        *reinterpret_cast<float4*>(dst + 4) = make_float4(pq.x + d.x, pq.y + d.y, pq.z + d.z, pq.w + d.w);
                    }
                }
                __syncthreads();
            }
            // soft edges a_ij = softmax(G2^T relu(PRe_i + PCe_j + l_ij DgE) + b2h) (model_4.py:286-304).  Pooling consumes their row
            // and column sums; with every index line present (L = Ne) these are the sums over the grid rows / columns (RA, CA), with
            // L < Ne the local L x L grid is a reshape of the FLAT pair order, so those commits keep a1 in that order (A1F).
            M2_PHASE(21);
            if (TRAIN) {
                float4* dst = reinterpret_cast<float4*>(a.PREg + (size_t)b * Ne * 60);
                for (int i = tid; i < Ne * 15; i += M2_T) dst[i] = reinterpret_cast<const float4*>(uni)[i];      // PRe01 | PCe are contiguous
            }
            float* RA = sm + L_.RA; float* CA = sm + L_.CA;
            float* a1f = (!ident && Lb >= 2) ? a.A1F + (size_t)b * Ne * nm1 : nullptr;
            float* cpart = sm + L_.cpart;                       // [M2_NW][32] column partials of one column block
            const float bdE = blkE[1001] - blkE[1000];
            u64 gam2[HD / 2];
#pragma unroll
            for (int k = 0; k < HD / 2; ++k) gam2[k] = pk2(gamE[2 * k], gamE[2 * k + 1]);
            for (int i = tid; i < Ne; i += M2_T) RA[i] = 0.f;
            __syncthreads();
            const int WUe = (Ne + 31) >> 5;
            for (int cb = 0; cb < WUe; ++cb) {
                const int j = cb * 32 + lane;
                const bool ok = j < Ne;
                u64 Q2[HD / 2];          // packed pairs: one add2 / fma2 per two channels
#pragma unroll
                for (int q4 = 0; q4 < 5; ++q4) {
                    ulonglong2 v = make_ulonglong2(pk2(NEG_BIG, NEG_BIG), pk2(NEG_BIG, NEG_BIG));
                    if (ok) v = *reinterpret_cast<const ulonglong2*>(PCe + j * HD + 4 * q4);
                    Q2[2 * q4] = v.x; Q2[2 * q4 + 1] = v.y;
                }
                float cacc = 0.f;
                for (int r = warp; r < Ne; r += M2_NW) {
                    const uint32_t bit = (ebits[r * WPe + cb] >> lane) & 1u;
                    const float* prow = PRe01 + (size_t)r * PROW + bit * 4;
                    u64 da = pk2(bdE, 0.f), db2 = 0ull;
#pragma unroll
                    for (int q4 = 0; q4 < 5; ++q4) {
                        const ulonglong2 pv = *reinterpret_cast<const ulonglong2*>(prow + q4 * 8);
                        da = fma2(relu2(add2(pv.x, Q2[2 * q4])), gam2[2 * q4], da);
                        db2 = fma2(relu2(add2(pv.y, Q2[2 * q4 + 1])), gam2[2 * q4 + 1], db2);
                    }
                    float dlo, dhi;
                    upk2(add2(da, db2), dlo, dhi);
                    const float d = dlo + dhi;
                    const float e = expf(-fabsf(d)), inv = 1.f / (1.f + e);
                    const float a1 = (ok && j != r) ? (d >= 0.f ? inv : e * inv) : 0.f;
                    cacc += a1;
                    const float rs = warp_sum(a1);
                    if (lane == 0) RA[r] += rs;                 // one owner warp per row, column blocks in order
                    if (a1f && ok && j != r) a1f[(size_t)r * nm1 + j - (j > r)] = a1;
                }
                cpart[warp * 32 + lane] = cacc;
                __syncthreads();
                if (tid < 32 && cb * 32 + tid < Ne) {
                    float t = 0.f;
#pragma unroll
                    for (int w = 0; w < M2_NW; ++w) t += cpart[w * 32 + tid];
                    CA[cb * 32 + tid] = t;
                }
                __syncthreads();
            }
            M2_PHASE(22);
        }
        M2_PHASE(17);
    }

    // ---------------- B/C. entity-state MLP forward: two threads per entity (10 hidden units each) ----------
    const int nsl = a.ent ? ent2_slots(b, Ne, a.R) : 0;
    // S_n = RS1_n + sum_slots CS1p_n  (all loads of a node in flight at once)
    auto load_S = [&](float (&S)[HD], int node) {
        load20s(S, a.RS1 + ((size_t)b * Ne + node) * HD);
        for (int sl = 0; sl < nsl; ++sl) {
            float t[HD];
            load20s(t, a.CS1p + (((size_t)b * a.SL + sl) * Ne + node) * HD);
#pragma unroll
            for (int k = 0; k < HD; ++k) S[k] += t[k];
        }
    };
    // The same sums for `count` nodes at once, written to shared memory (row stride in floats): every thread takes one
    // float4 of one node and has the loads of ALL slots in flight, so the block pays one or two global round trips
    // instead of 1 + nsl dependent ones per thread (nsl = 6-7 at glide).  Same summation order as load_S.
    auto coop_load_S = [&](float* dst, int stride, int node0, int count) {
        const float4* rs = reinterpret_cast<const float4*>(a.RS1 + ((size_t)b * Ne + node0) * HD);
        const float4* cs = reinterpret_cast<const float4*>(a.CS1p + ((size_t)b * a.SL * Ne + node0) * HD);
        const size_t slot4 = (size_t)Ne * HD / 4;
        for (int e = tid; e < count * 5; e += M2_T) {
            float4 acc = rs[e];
            for (int s0 = 0; s0 < nsl; s0 += 8) {
                float4 v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = s0 + u < nsl ? cs[(size_t)(s0 + u) * slot4 + e] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int u = 0; u < 8; ++u) { acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w; }
            }
            const int n = e / 5, j = e - n * 5;
            *reinterpret_cast<float4*>(dst + (size_t)n * stride + 4 * j) = acc;
        }
    };
    // Zh[j] = pre-activation of hidden unit 10 h + j of the entity-state MLP for effect sums S and attribute xv
    auto hidden_half = [&](float (&Zh)[10], const float (&S)[HD], float xv, int h) {
#pragma unroll
        for (int j = 0; j < 10; ++j) Zh[j] = fmaf(xv, U1[10 * h + j], c1p[10 * h + j]);
#pragma unroll
        for (int q = 0; q < HD; ++q) {
#pragma unroll
            for (int j2 = 0; j2 < 5; ++j2) {
                const float2 w = *reinterpret_cast<const float2*>(W5U + q * HD + 10 * h + 2 * j2);
                Zh[2 * j2] = fmaf(S[q], w.x, Zh[2 * j2]); Zh[2 * j2 + 1] = fmaf(S[q], w.y, Zh[2 * j2 + 1]);
            }
        }
    };
    if (a.ent) {
        // S for all nodes -> its own region (kept for the backward) or the still unused head of the union region (unless
        // that would run into SP / TP)
        const bool coopS = a.scache || (!GT && Ne <= 12 * Nc);
        float* Sall = a.scache ? SC : uni;
        if (coopS && !a.inl) { coop_load_S(Sall, HD, 0, Ne); __syncthreads(); }
        for (int base = 0; base < 2 * Ne; base += M2_T) {
            const int t = base + tid, node = t >> 1, h = t & 1;
            const bool valid = node < Ne;
            float acc = 0.f;
            if (valid) {
                float S[HD], Zh[10];
                if (coopS) load20s(S, Sall + (size_t)node * HD); else load_S(S, node);
                if (dbg && h == 0) for (int k = 0; k < HD; ++k) dbg[(size_t)node * HD + k] = S[k];
                hidden_half(Zh, S, xs[node], h);
#pragma unroll
                for (int j = 0; j < 10; ++j) acc = fmaf(fmaxf(Zh[j], 0.f), u2[10 * h + j], acc);
            }
            acc += __shfl_xor_sync(0xffffffffu, acc, 1);
            if (valid && h == 0) x2[node] = fmaxf(acc + c2[0], 0.f);
        }
        __syncthreads();
    }
    if (dbg) for (int i = tid; i < Ne; i += M2_T) dbg[(size_t)Ne * HD + i] = x2[i];
    M2_PHASE(2);

    // ---------------- D. pooling forward -------------------------------------------------------
    // B2[q] = [x2_gi, x2_gj, 1 - A, A] over the Ne-grid enumeration q; the L x L local grid selects
    // q = li (L-1) + lj - [lj > li]  (utils2.py:123-137, quirk Q3).  SP[li] = row sums, TP[lj] = column sums.
    if (ident) {
        float part = 0.f;
        for (int i = tid; i < Ne; i += M2_T) part += x2[i];
        const float X = mid2_block_sum(part, red);
        M2_PHASE(13);
        M2_PHASE(14);
        for (int i = tid; i < Ne; i += M2_T) {              // degrees: SP[.][3] / TP[.][3] (computed before the wait), or the edge
            const float xi = x2[i], fn = (float)nm1;        // prefix counts of the inline entity stage
            if (a.edge) { SP[4 * i + 3] = (sm + L_.RA)[i]; TP[4 * i + 3] = (sm + L_.CA)[i]; }       // variant 4: soft edges instead of degrees
            else if (a.inl) { SP[4 * i + 3] = (float)(rptr[i + 1] - rptr[i]); TP[4 * i + 3] = (float)(cptr[i + 1] - cptr[i]); }
            SP[4 * i] = fn * xi; SP[4 * i + 1] = X - xi; SP[4 * i + 2] = fn - SP[4 * i + 3];
            TP[4 * i] = X - xi; TP[4 * i + 1] = fn * xi; TP[4 * i + 2] = fn - TP[4 * i + 3];
        }
    } else if (Lb < 2) {
        // an index file with fewer than two lines has no local pair (utils2.py:123-137): nothing is pooled
        for (int idx = tid; idx < 4 * Ne; idx += M2_T) { SP[idx] = 0.f; TP[idx] = 0.f; }
    } else {
        // general path: SP[li] = sum of the m = L-1 consecutive entries B2[li m .. li m + m) (closed form from
        // prefix sums and bit-range popcounts); TP[lj] = sum_li B2[li m + lj - (lj > li)] gathered with
        // incrementally updated grid coordinates.
        const int n = nm1, m = Lb - 1;
        float* PX = dl;                                 // exclusive prefix of x2 (dl is free until the backward)
        if (warp == 0) warp_excl_scan(PX, x2, 1, Ne, lane);
        int nchunk = M2_T / Lb;
        nchunk = nchunk < 1 ? 1 : (nchunk > 4 ? 4 : nchunk);
        float* partC = scratch;                         // [nchunk][Lb][4]
        // per index line li: grid coordinates (row g0, offset p0) of flat index li m as {p0 - n, g0} and the two node values a local
        // row can see in channel 0 (m < n: at most one row wrap), one 16-byte broadcast load per visit
        int4* rowtab = reinterpret_cast<int4*>(scratch + mid2_rowtab_off(Ne));      // [Lb]
        for (int li = tid; li < Lb; li += M2_T) {
            const int q = li * m, g = q / n;
            rowtab[li] = make_int4(q - g * n - n, g, __float_as_int(x2[g]), __float_as_int(x2[min(g + 1, Ne - 1)]));
        }
        __syncthreads();
        // index lines of this CTA: all of them, or (a cluster shares the commit) one half -- the column sums are added below
        const int lr0 = CL && split && crank ? (Lb + 1) >> 1 : 0, lr1 = CL && split && !crank ? (Lb + 1) >> 1 : Lb;
        for (int t = tid; t < nchunk * Lb; t += M2_T) {
            const int c = t / Lb, me = t - c * Lb;
            const int lo = lr0 + (c * (lr1 - lr0)) / nchunk, hi = lr0 + ((c + 1) * (lr1 - lr0)) / nchunk;
            float q0 = 0.f, q1 = 0.f;
            int q3 = 0;
            const bool own = me >= lo && me < hi;       // the chunk holds the diagonal visit li == me
            const int cnt = (hi - lo) - (own ? 1 : 0);
            // one visit: local pair (li, me) -> flat index li m + me - (me > li) -> grid pair (gi, gj).  No loop-carried index
            // state, so the loads of several iterations overlap.  The diagonal visit is swept like the others (its indices stay
            // inside the commit's tile) and taken out again below: no per-visit select
            auto visit = [&](int li, float& xa, float& xb, int& bit) {
                const int4 e = rowtab[li];
                const int tt = e.x + me - (li < me ? 1 : 0);       // p - n
                const bool w = tt >= 0;                            // the local row has wrapped into grid row g0 + 1
                const int pp = w ? tt : tt + n;
                const int gi = e.y + (w ? 1 : 0), gj = pp + (pp >= gi ? 1 : 0);
                xa = __int_as_float(w ? e.w : e.z);
                xb = x2[gj];
                bit = (int)((ebits[gi * WPe + (gj >> 5)] >> (gj & 31)) & 1u);
            };
#pragma unroll 4
            for (int li = lo; li < hi; ++li) {
                float xa, xb; int bit;
                visit(li, xa, xb, bit);
                q0 += xa; q1 += xb; q3 += bit;
            }
            if (own) {
                float xa, xb; int bit;
                visit(me, xa, xb, bit);
                q0 -= xa; q1 -= xb; q3 -= bit;
            }
            float* pc = partC + ((size_t)c * Lb + me) * 4;
            pc[0] = q0; pc[1] = q1; pc[2] = (float)(cnt - q3); pc[3] = (float)q3;
        }
        __syncthreads();
        M2_PHASE(14);
        for (int li = tid; li < Lb; li += M2_T) {
            const int qs = li * m;
            int g = qs / n, p0 = qs - g * n, rem = m, c3 = 0;
            float a0 = 0.f, a1 = 0.f;
            while (rem > 0) {
                const int c = min(rem, n - p0), pb = p0 + c;
                a0 = fmaf((float)c, x2[g], a0);
                a1 += offdiag_prefix(PX, x2, 1, g, pb) - offdiag_prefix(PX, x2, 1, g, p0);
                c3 += range_popc(ebits + g * WPe, p0 + (p0 >= g), pb - 1 + (pb - 1 >= g) + 1);
                rem -= c; ++g; p0 = 0;
            }
            SP[4 * li] = a0; SP[4 * li + 1] = a1; SP[4 * li + 2] = (float)(m - c3); SP[4 * li + 3] = (float)c3;
        }
        for (int idx = tid; idx < 4 * Lb; idx += M2_T) {
            float t = 0.f;
            for (int c = 0; c < nchunk; ++c) t += partC[(size_t)c * Lb * 4 + idx];
            TP[idx] = t;
        }
        if (CL && split) { __syncthreads(); xchg(nullptr, TP, Lb, nullptr, 0); }
        if (a.edge) {
            // variant 4: channels 2, 3 are the soft edges.  In the flat pair order the local grid is the row-major [L][m] reshape of
            // the first L m entries: SP = its row sums, TP[lj] = sum_li a1[li m + lj - (lj > li)]
            __syncthreads();
            const float* a1f = a.A1F + (size_t)b * Ne * nm1;
            for (int li = warp; li < Lb; li += M2_NW) {
                float acc = 0.f;
                for (int sidx = lane; sidx < m; sidx += 32) acc += __ldcg(a1f + (size_t)li * m + sidx);
                acc = warp_sum(acc);
                if (lane == 0) { SP[4 * li + 3] = acc; SP[4 * li + 2] = (float)m - acc; }
            }
            for (int t0 = 0; t0 < 4 * Lb; t0 += M2_T) {           // four threads per column (interleaved rows), eight loads in flight each
                const int t = t0 + tid, lj = t >> 2, part = t & 3;
                const bool live = t < 4 * Lb;
                float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                for (int li0 = part; live && li0 < Lb; li0 += 32) {
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int li = li0 + 4 * u;
                        if (li < Lb && li != lj) acc[u] += __ldcg(a1f + (size_t)li * m + lj - (lj > li ? 1 : 0));
                    }
                }
                float tot = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
                tot += __shfl_xor_sync(0xffffffffu, tot, 1);
                tot += __shfl_xor_sync(0xffffffffu, tot, 2);
                if (live && part == 0) { TP[4 * lj + 3] = tot; TP[4 * lj + 2] = (float)m - tot; }
            }
        }
    }
    __syncthreads();
    // segmented reduce by hunk id over the sorted lists: one thread per (hunk, channel), ascending index-line order
    M2_PHASE(15);
    for (int idx = tid; idx < Nc * 4; idx += M2_T) {
        const int c = idx >> 2, chn = idx & 3;
        float acc = 0.f;
        for (int k = hstart[c]; k < hstart[c + 1]; ++k) { const int i = horder[k]; acc += SP[4 * i + chn] + TP[4 * i + chn]; }
        nb[idx] = acc;
        if (dbg) dbg[(size_t)Ne * 21 + idx] = acc;
    }
    __syncthreads();
    M2_PHASE(3);

    // ---------------- hunk-stage tables (union region) ---------------------------------------------
    const int T = Nc * HD;
    float* PH01 = tabs;             // [Nc][KG][2][4]
    float* QH = tabs + 2 * T;
    float* RS3 = tabs + 3 * T;
    float* CS3 = tabs + 4 * T;
    float* rr = tabs + 5 * T;       // r, later GC
    float* cc = tabs + 6 * T;
    float* PR01 = tabs + 7 * T;     // [Nc][KG][2][4]; later dr (first T) and GR (second T)
    float* PC = tabs + 9 * T;       // later dc
    float* RSm = tabs + 10 * T;     // later RS3d
    float* CSm = tabs + 11 * T;     // later CS3d
    constexpr int DW = CWT * 32;
    // [Nc][CWT*32] dL/dlogit-difference per pair (training); in smem it aliases SP/TP/dl, else HBM (L2-resident)
    float* dlt = a.dlt_g ? a.dlt_g + (size_t)b * Nc * DW : uni + (GT ? 0 : mid2_tab_floats(Nc));
    for (int idx = tid; idx < T; idx += M2_T) {
        const int c = idx / HD, k = idx - c * HD;
        float p = d1[k] + V1[8 * HD + k], q = 0.f;
#pragma unroll
        for (int chn = 0; chn < 4; ++chn) {
            p = fmaf(nb[4 * c + chn], V1[chn * HD + k], p);
            q = fmaf(nb[4 * c + chn], V1[(4 + chn) * HD + k], q);
        }
        const int pi = p01_idx(c, k);
        PH01[pi] = p; PH01[pi + 4] = p + Dh[k]; QH[idx] = q;
    }
    __syncthreads();

    // ---------------- E. hunk pair layer forward: row / column sums ---------------------------------
    // Grids of 7 and more column segments take the columns in passes of four segments (the accumulators of eight do not fit the
    // register file: measured spills); later passes add to the row sums of the first.  The widest instantiation (CWT = 16) also
    // serves every narrower grid above 256 hunks: passes / segments beyond Nc are skipped.
    constexpr int PWC = CWT >= 7 ? 4 : CWT;             // segments per column pass
    constexpr int NPASS = (CWT + PWC - 1) / PWC;
    {
        const float* PH01s = PH01;
        if (GT) { stage_rows(stg, PH01, 2 * T); __syncthreads(); PH01s = stg; }
#pragma unroll
        for (int pass = 0; pass < NPASS; ++pass) {
            const int sg0 = pass * PWC;
            if (sg0 * 32 >= Nc) break;
            u64 Q[PWC][2], col[PWC][2];
#pragma unroll
            for (int sg = 0; sg < PWC; ++sg) {
                const int j = (sg0 + sg) * 32 + lane;
                ulonglong2 q = make_ulonglong2(pk2(NEG_BIG, NEG_BIG), pk2(NEG_BIG, NEG_BIG));
                if (j < Nc) q = *reinterpret_cast<const ulonglong2*>(QH + j * HD + k0);
                Q[sg][0] = q.x; Q[sg][1] = q.y; col[sg][0] = 0ull; col[sg][1] = 0ull;
            }
            // rows hr0 .. hr1 (all of them unless a cluster shares the commit)
            const float* Prow = PH01s + (size_t)hr0 * PROW; const uint32_t* brow = ybits + sg0 + (size_t)hr0 * WPc; float* rsrow = RS3 + (size_t)hr0 * HD;
            if (pass == 0) sweep2_fwd<PWC, false>(Prow, brow, WPc, hr1 - hr0, rg, M2_NRG, kg, Q, col, rsrow, lane);
            else sweep2_fwd<PWC, true>(Prow, brow, WPc, hr1 - hr0, rg, M2_NRG, kg, Q, col, rsrow, lane);
            if constexpr (PWC >= 5) combine_cols_2pass<PWC>(col, scratch, rg, M2_NRG, kg, lane);
            else combine_cols<PWC>(col, scratch, rg, M2_NRG, kg, lane);
            if (rg == 0) {
#pragma unroll
                for (int sg = 0; sg < PWC; ++sg) {
                    const int j = (sg0 + sg) * 32 + lane;
                    if (j < Nc) *reinterpret_cast<ulonglong2*>(CS3 + j * HD + k0) = make_ulonglong2(col[sg][0], col[sg][1]);
                }
            }
        }
    }
    __syncthreads();
    if (CL && split) xchg(RS3, CS3, Nc * (HD / 4), nullptr, 0);
    for (int idx = tid; idx < T; idx += M2_T) {       // remove the diagonal pair (l = 0)
        const int c = idx / HD, k = idx - c * HD;
        const float d = fmaxf(PH01[p01_idx(c, k)] + QH[idx], 0.f);
        RS3[idx] -= d; CS3[idx] -= d;
        if (dbg) { dbg[(size_t)Ne * 21 + Nc * 4 + idx] = RS3[idx]; dbg[(size_t)Ne * 21 + Nc * 4 + T + idx] = CS3[idx]; }
    }
    __syncthreads();
    M2_PHASE(4);

    // ---------------- F. linear second layer on the sums + head tables (model_2.py:263-275, 311-315) --
    // five threads per (hunk, side), four output channels each: r_n = (Nc-1) b2 + RS3_n W2, then (after the block has the whole
    // r_n) PR_n = g1b + G1[0] + r_n G1e, or the c / PC side
    for (int it0 = 0; it0 < 2 * Nc; it0 += M2_T / KG) {
        const int t = it0 + tid / KG, k4 = 4 * (tid % KG);
        const bool live = t < 2 * Nc, cside = t >= Nc;
        const int n = cside ? t - Nc : t;
        if (live) {
            const float fn1 = (float)(Nc - 1);
            const float4 bb = *reinterpret_cast<const float4*>(b2 + k4);
            const float4 r4 = gemv20_k4((cside ? CS3 : RS3) + n * HD, W2, k4, make_float4(fn1 * bb.x, fn1 * bb.y, fn1 * bb.z, fn1 * bb.w));
            *reinterpret_cast<float4*>((cside ? cc : rr) + n * HD + k4) = r4;
        }
        __syncthreads();
        if (live) {
            float4 init = make_float4(0.f, 0.f, 0.f, 0.f);
            if (!cside) {
                const float4 g = *reinterpret_cast<const float4*>(g1b + k4), g0 = *reinterpret_cast<const float4*>(G1 + k4);
                init = make_float4(g.x + g0.x, g.y + g0.y, g.z + g0.z, g.w + g0.w);
            }
            const float4 pq = gemv20_k4((cside ? cc : rr) + n * HD, G1 + 2 * HD, k4, init);
            if (cside) {
                *reinterpret_cast<float4*>(PC + n * HD + k4) = pq;
            } else {
                const float4 d = *reinterpret_cast<const float4*>(Dg + k4);
                float* dst = PR01 + (size_t)n * PROW + 2 * k4;        // [n][kg][2][4]
                *reinterpret_cast<float4*>(dst) = pq;
                *reinterpret_cast<float4*>(dst + 4) = make_float4(pq.x + d.x, pq.y + d.y, pq.z + d.z, pq.w + d.w);
            }
            if (dbg) { float* dd = dbg + (size_t)Ne * 21 + Nc * 4 + (cside ? 3 : 2) * T + n * HD + k4; dd[0] = pq.x; dd[1] = pq.y; dd[2] = pq.z; dd[3] = pq.w; }
        }
    }
    __syncthreads();
    M2_PHASE(5);

    // ---------------- G1. relation head: logits, softmax, CE (lanes = columns, all 20 channels) ---------
    float ce_acc = 0.f, d_acc = 0.f, hit_acc = 0.f;
    const bool EVC = a.evc != nullptr;
    uint32_t ev_tpc = 0u, ev_fpc = 0u, ev_tpq = 0u, ev_fpq = 0u, ev_pos = 0u;      // warp-uniform partial counts
    const float* PR01s = PR01;          // row tables of the two head sweeps (G1, G2)
    if (GT) { stage_rows(stg, PR01, 2 * T); __syncthreads(); PR01s = stg; }
    {
        const size_t npair = (size_t)Nc * (Nc - 1);
        const float bd = gb2[1] - gb2[0], b20 = gb2[0];
        u64 gam2[HD / 2];        // packed pairs in registers: one add2 / fma2 per two channels
#pragma unroll
        for (int k = 0; k < HD / 2; ++k) gam2[k] = pk2(gam[2 * k], gam[2 * k + 1]);
        for (int cb = 0; cb < CWT; ++cb) {
            if (cb * 32 >= Nc) break;
            const int j = cb * 32 + lane;
            const bool ok = j < Nc;
            const uint32_t colmask = Nc - cb * 32 >= 32 ? 0xffffffffu : (1u << (Nc - cb * 32)) - 1u;      // columns of this segment below Nc
            u64 Q2[HD / 2];
#pragma unroll
            for (int q4 = 0; q4 < 5; ++q4) {
                ulonglong2 v = make_ulonglong2(pk2(NEG_BIG, NEG_BIG), pk2(NEG_BIG, NEG_BIG));
                if (ok) v = *reinterpret_cast<const ulonglong2*>(PC + j * HD + 4 * q4);
                Q2[2 * q4] = v.x; Q2[2 * q4 + 1] = v.y;
            }
            for (int r = hr0 + warp; r < hr1; r += M2_NW) {
                const bool valid = ok && j != r;
                const uint32_t yw = ybits[r * WPc + cb];
                const uint32_t bit = (yw >> lane) & 1u;
                const bool lab = bit != 0u;
                const float* prow = PR01s + (size_t)r * PROW + bit * 4;
                u64 da = pk2(bd, 0.f), db2 = 0ull;
                float l0 = b20;
#pragma unroll
                for (int q4 = 0; q4 < 5; ++q4) {
                    const ulonglong2 p = *reinterpret_cast<const ulonglong2*>(prow + q4 * 8);
                    const u64 ha = relu2(add2(p.x, Q2[2 * q4])), hb = relu2(add2(p.y, Q2[2 * q4 + 1]));
                    da = fma2(ha, gam2[2 * q4], da); db2 = fma2(hb, gam2[2 * q4 + 1], db2);
                    if (LOGITS) {
                        float h0, h1, h2, h3;
                        upk2(ha, h0, h1); upk2(hb, h2, h3);
                        l0 = fmaf(h0, G2[2 * (4 * q4)], l0); l0 = fmaf(h1, G2[2 * (4 * q4 + 1)], l0);
                        l0 = fmaf(h2, G2[2 * (4 * q4 + 2)], l0); l0 = fmaf(h3, G2[2 * (4 * q4 + 3)], l0);
                    }
                }
                float dlo, dhi;
                upk2(add2(da, db2), dlo, dhi);
                const float d = dlo + dhi;
                const float e = expf(-fabsf(d));
                const float inv = 1.f / (1.f + e);
                const float p1 = d >= 0.f ? inv : e * inv, p0 = d >= 0.f ? e * inv : inv;
                if (valid) {
                    const size_t q = (size_t)r * (Nc - 1) + j - (j > r);
                    if (a.probs) {
                        a.probs[((size_t)b * 2 + 0) * npair + q] = p0;
                        a.probs[((size_t)b * 2 + 1) * npair + q] = p1;
                    }
                    if (LOGITS) {
                        a.logits[((size_t)b * 2 + 0) * npair + q] = l0;
                        a.logits[((size_t)b * 2 + 1) * npair + q] = l0 + d;
                    }
                    const float z = lab ? -d : d;
                    ce_acc += fmaxf(z, 0.f) + __logf(1.f + e);     // e in (0, 1]: absolute error ~1e-7
                    hit_acc += ((p1 > p0) == lab) ? 1.f : 0.f;      // np.argmax over the two channels: a tie is class 0
                }
                if (EVC) {
                    // evaluation counters: two ballots per 32 pairs, then warp-uniform popcounts against the label word (its
                    // diagonal and padding bits are zero).  am: arg-max is class 1 (a tie is class 0); qp: the reference's
                    // ceil-on-channel-0 prediction (EvaluationFuncs.py:95-99)
                    const uint32_t vm = (r >> 5) == cb ? colmask & ~(1u << (r & 31)) : colmask;
                    const uint32_t am = __ballot_sync(0xffffffffu, p1 > p0) & vm, qp = __ballot_sync(0xffffffffu, p0 > 0.f) & vm;
                    ev_tpc += __popc(am & yw); ev_fpc += __popc(am & ~yw); ev_tpq += __popc(qp & ~yw); ev_fpq += __popc(qp & yw);
                    ev_pos += __popc(yw & vm);
                }
                if (TRAIN) {
                    const float dv = valid ? a.scale * (p1 - (lab ? 1.f : 0.f)) : 0.f;
                    d_acc += dv;
                    dlt[r * DW + j] = dv;
                }
            }
        }
    }
    {
        float ce_tot = mid2_block_sum(ce_acc, red);
        float hit_tot = a.hits_acc ? mid2_block_sum(hit_acc, red) : 0.f;     // per-commit counts are below 2^24: exact in float
        uint32_t* evs = reinterpret_cast<uint32_t*>(red + 64);        // [M2_NW][8] (the label-sum slots of G2: not live yet)
        unsigned long long t[5] = {0ull, 0ull, 0ull, 0ull, 0ull};
        if (EVC) {
            __syncthreads();
            if (lane == 0) { uint32_t* e = evs + warp * 8; e[0] = ev_tpc; e[1] = ev_fpc; e[2] = ev_tpq; e[3] = ev_fpq; e[4] = ev_pos; }
            __syncthreads();
            if (tid == 0)
                for (int w = 0; w < M2_NW; ++w)
                    for (int q = 0; q < 5; ++q) t[q] += evs[w * 8 + q];
        }
        if (CL && split) {
            // the two halves' scalars: rank 0 adds the peer's (integers and a two-term float sum: order-free)
            float* xs = red + 64 + M2_NW * 8;                         // [8]
            __syncthreads();
            if (tid == 0) {
                xs[0] = ce_tot; xs[1] = hit_tot;
                for (int q = 0; q < 5; ++q) xs[2 + q] = __uint_as_float((uint32_t)t[q]);
            }
            cluster_sync_all();
            if (tid == 0 && wr) {
                const uint32_t px = peer_smem(xs, crank ^ 1u);
                ce_tot += ld_peer(px); hit_tot += ld_peer(px + 4u);
                for (int q = 0; q < 5; ++q) t[q] += __float_as_uint(ld_peer(px + 4u * (2 + q)));
            }
            cluster_sync_all();
        }
        if (wr && tid == 0) {
            if (a.cep) a.cep[b] = ce_tot;
            if (a.hits_acc) atomicAdd(a.hits_acc, (unsigned long long)(hit_tot + 0.5f));      // integer atomic: order independent
            if (EVC) {
                const unsigned long long npair = (unsigned long long)Nc * (Nc - 1), pos = t[4], neg = npair - pos;
                unsigned long long* o = a.evc + (size_t)b * 8;       // this commit's slots: one writer
                o[0] += t[0] + (neg - t[1]);                          // arg-max hits = tp + tn
                o[1] += t[2]; o[2] += t[3]; o[3] += neg - t[2];       // reference form: y_true = 1 - Y, y_pred = [p0 > 0]
                o[4] += t[0]; o[5] += t[1]; o[6] += pos - t[0];       // conventional form: y_true = Y, y_pred = [p1 > p0]
                o[7] += pos;
            }
        }
        if (EVC || (CL && split)) __syncthreads();
    }
    M2_PHASE(6);
    if (!TRAIN) return;

    // ---------------- G2. delta sums: RSm_i = sum_j m_ij dlt_ij, CSm_j, LSm (label-1 pairs) ----------------
    // column passes as in E
    float* lsw = red + 64;                   // [M2_NRG][20]
    float* misc = red + 64 + M2_NW * HD;     // [0..19] LSm then LS4, [40] dsum
    {
        const float d_tot = mid2_block_sum(d_acc, red);      // leading __syncthreads orders the dlt stores
        if (tid == 0) misc[40] = d_tot;
        u64 lsm[2] = {0ull, 0ull};
        const uint32_t lmask = 1u << lane;
#pragma unroll
        for (int pass = 0; pass < NPASS; ++pass) {
            const int sg0 = pass * PWC;
            u64 Q[PWC][2], col[PWC][2];
#pragma unroll
            for (int sg = 0; sg < PWC; ++sg) {
                const int j = (sg0 + sg) * 32 + lane;
                ulonglong2 q = make_ulonglong2(pk2(NEG_BIG, NEG_BIG), pk2(NEG_BIG, NEG_BIG));
                if (j < Nc) q = *reinterpret_cast<const ulonglong2*>(PC + j * HD + k0);
                Q[sg][0] = q.x; Q[sg][1] = q.y; col[sg][0] = 0ull; col[sg][1] = 0ull;
            }
            auto delta_row = [&](int r, u64& rp0, u64& rp1) {
                uint32_t w[PWC];
                load_words<PWC>(w, ybits + (size_t)r * WPc + sg0);
                const float* prow0 = PR01s + (size_t)r * PROW + kg * 8;
                const float* prow1 = prow0 + 4;
                const float* drow = dlt + (size_t)r * DW + sg0 * 32 + lane;
                float dvs[PWC];
#pragma unroll
                for (int sg = 0; sg < PWC; ++sg) dvs[sg] = sg0 + sg < CWT ? drow[sg * 32] : 0.f;      // all loads of the row in flight (HBM/L2 when spilled)
                rp0 = 0ull; rp1 = 0ull;
#pragma unroll
                for (int sg = 0; sg < PWC; ++sg) {
                    const bool bit = (w[sg] & lmask) != 0u;
                    const ulonglong2 p = *reinterpret_cast<const ulonglong2*>(bit ? prow1 : prow0);
                    const float dv = dvs[sg];
                    const u64 d2 = pk2(dv, dv);
                    const u64 v0 = gate2(add2(p.x, Q[sg][0]), d2), v1 = gate2(add2(p.y, Q[sg][1]), d2);
                    col[sg][0] = add2(col[sg][0], v0); col[sg][1] = add2(col[sg][1], v1);
                    rp0 = add2(rp0, v0); rp1 = add2(rp1, v1);
                    const float lf = bit ? 1.f : 0.f;
                    const u64 l2 = pk2(lf, lf);
                    lsm[0] = fma2(l2, v0, lsm[0]); lsm[1] = fma2(l2, v1, lsm[1]);
                }
            };
            auto put = [&](int row, int k, float tot) { float* d = RSm + row * HD + k; if (pass == 0) *d = tot; else *d += tot; };
            int r = hr0 + rg;
            for (; r + 3 * M2_NRG < hr1; r += 4 * M2_NRG) {      // four rows per trip: two independent transpose-reduces in flight
                u64 a0, a1, c0, c1, e0, e1, g0, g1;
                delta_row(r, a0, a1);
                delta_row(r + M2_NRG, c0, c1);
                delta_row(r + 2 * M2_NRG, e0, e1);
                delta_row(r + 3 * M2_NRG, g0, g1);
                const float tot = reduce8(a0, a1, c0, c1, lane), tot2 = reduce8(e0, e1, g0, g1, lane);
                if ((lane & 3) == 0) {
                    put((lane & 16) ? r + M2_NRG : r, k0 + reduce8_channel(lane), tot);
                    put((lane & 16) ? r + 3 * M2_NRG : r + 2 * M2_NRG, k0 + reduce8_channel(lane), tot2);
                }
            }
            for (; r + M2_NRG < hr1; r += 2 * M2_NRG) {
                u64 a0, a1, c0, c1;
                delta_row(r, a0, a1);
                delta_row(r + M2_NRG, c0, c1);
                const float tot = reduce8(a0, a1, c0, c1, lane);
                if ((lane & 3) == 0) put((lane & 16) ? r + M2_NRG : r, k0 + reduce8_channel(lane), tot);
            }
            if (r < hr1) {
                u64 a0, a1;
                delta_row(r, a0, a1);
                const float tot = reduce4(a0, a1, lane);
                if ((lane & 7) == 0) put(r, k0 + ch, tot);
            }
            if constexpr (PWC >= 5) combine_cols_2pass<PWC>(col, scratch, rg, M2_NRG, kg, lane);
            else combine_cols<PWC>(col, scratch, rg, M2_NRG, kg, lane);
            if (rg == 0) {
#pragma unroll
                for (int sg = 0; sg < PWC; ++sg) {
                    const int j = (sg0 + sg) * 32 + lane;
                    if (j < Nc) *reinterpret_cast<ulonglong2*>(CSm + j * HD + k0) = make_ulonglong2(col[sg][0], col[sg][1]);
                }
            }
        }
        const float t = reduce4(lsm[0], lsm[1], lane);
        if ((lane & 7) == 0) lsw[rg * HD + k0 + ch] = t;
        __syncthreads();
        if (tid < HD) {
            float ls = 0.f;
            for (int w = 0; w < M2_NRG; ++w) ls += lsw[w * HD + tid];
            misc[tid] = ls;
        }
        __syncthreads();
        if (CL && split) xchg(RSm, CSm, Nc * (HD / 4), misc, 41);        // label sums [0, 20) and the sum of the deltas [40]
    }
    M2_PHASE(7);

    // ---------------- H. head backward (node level) ------------------------------------------------------
    // RS4 = gam * RSm and CS4 = gam * CSm are never formed: gam is applied to the outputs / folded into G1g.
    float* dr = PR01; float* dc = PC;          // written in round 2, after their last readers of round 1
    {
        const int slice = tid & 15, grp = tid >> 4;
        // round 1: scr_w1 rows 2.. (25 tiles), HS -> scr_w2, column sums of RSm -> scr_b1 and the label rows
        if (grp < 25) {
            float acc[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) acc[i] = 0.f;
            const int a0 = 4 * (grp / 5), b0 = 4 * (grp % 5);
            tile_acc(acc, rr, HD, RSm, HD, a0, b0, slice, Nc);
            tile_acc(acc, cc, HD, CSm, HD, a0, b0, slice, Nc);
            const float v = reduce16(acc, lane);
            const int m = a0 + (slice >> 2), k = b0 + (slice & 3);
            gp[po.scr_w1 + 2 * HD + m * HD + k] = v * gam[k];            // dG1e[m][k]
        } else if (grp < 30) {
            // HS[k] = sum_pairs relu(pre)[k] * delta  via  relu(pre) = m * (PR0_i + l Dg + PC_j); 4 channels per group
            const int kb = 4 * (grp - 25);
            float hs[4] = {0.f, 0.f, 0.f, 0.f}, cs[4] = {0.f, 0.f, 0.f, 0.f};
            for (int n = slice; n < Nc; n += 16) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float rs = RSm[n * HD + kb + j];
                    hs[j] = fmaf(PR01[p01_idx(n, kb + j)], rs, hs[j]);
                    hs[j] = fmaf(PC[n * HD + kb + j], CSm[n * HD + kb + j], hs[j]);
                    cs[j] += rs;
                }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) { hs[j] = half_sum(hs[j]); cs[j] = half_sum(cs[j]); }
            if (slice < 4) {
                const int k = kb + slice;
                const float h = fmaf(Dg[k], misc[k], slice == 0 ? hs[0] : slice == 1 ? hs[1] : slice == 2 ? hs[2] : hs[3]);
                const float c = (slice == 0 ? cs[0] : slice == 1 ? cs[1] : slice == 2 ? cs[2] : cs[3]) * gam[k];
                const float ls4 = misc[k] * gam[k];
                gp[po.scr_w2 + 2 * k + 1] = h; gp[po.scr_w2 + 2 * k] = -h;
                gp[po.scr_b1 + k] = c; gp[po.scr_w1 + HD + k] = ls4; gp[po.scr_w1 + k] = c - ls4;
            }
        }
        if (tid == 0) { gp[po.scr_b2 + 1] = misc[40]; gp[po.scr_b2] = -misc[40]; }
        __syncthreads();
        // round 2: dr = RS4 G1e^T = RSm G1g^T, dc = CSm G1g^T (one thread per (hunk, side))
        for (int t = tid; t < 2 * Nc; t += M2_T) {
            if (GT) asm volatile("" ::: "memory");      // global tables: keeps the (loop-invariant) weight loads inside the loop; hoisted, they spill
            const bool cside = t >= Nc;
            const int n = cside ? t - Nc : t;
            float in[HD], out[HD];
            load20s(in, (cside ? CSm : RSm) + n * HD);
            gemv20t(out, in, G1g);
            store20s((cside ? dc : dr) + n * HD, out);
        }
        __syncthreads();
        // round 3: hnk_w2 / hnk_b2 gradients (25 tiles + 5 groups of column sums) and GR = dr W2^T, GC = dc W2^T
        float* GR = PR01 + T; float* GC = rr;
        if (grp < 25) {
            float acc[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) acc[i] = 0.f;
            const int a0 = 4 * (grp / 5), b0 = 4 * (grp % 5);
            tile_acc(acc, RS3, HD, dr, HD, a0, b0, slice, Nc);
            tile_acc(acc, CS3, HD, dc, HD, a0, b0, slice, Nc);
            const float v = reduce16(acc, lane);
            gp[po.hnk_w2 + (a0 + (slice >> 2)) * HD + b0 + (slice & 3)] = v;
        } else if (grp < 30) {
            const int kb = 4 * (grp - 25);
            float cs[4] = {0.f, 0.f, 0.f, 0.f};
            for (int n = slice; n < Nc; n += 16)
#pragma unroll
                for (int j = 0; j < 4; ++j) cs[j] += dr[n * HD + kb + j] + dc[n * HD + kb + j];
#pragma unroll
            for (int j = 0; j < 4; ++j) cs[j] = half_sum(cs[j]);
            if (slice < 4)
                gp[po.hnk_b2 + kb + slice] = (float)(Nc - 1) * (slice == 0 ? cs[0] : slice == 1 ? cs[1] : slice == 2 ? cs[2] : cs[3]);
        } else {
            // threads 480..639: GR / GC rows (rr is dead: its last readers ran in round 1)
            for (int t = tid - 480; t < 2 * Nc; t += M2_T - 480) {
                if (GT) asm volatile("" ::: "memory");
                const bool cside = t >= Nc;
                const int n = cside ? t - Nc : t;
                float in[HD], out[HD];
                load20s(in, (cside ? dc : dr) + n * HD);
                gemv20t(out, in, W2);
                store20s((cside ? GC : GR) + n * HD, out);
            }
        }
        __syncthreads();
    }
    float* GR = PR01 + T; float* GC = rr;
    float* RS3d = RSm; float* CS3d = CSm;
    M2_PHASE(8);

    // ---------------- I. hunk pair layer backward sweep ------------------------------------------------------
    {
        u64 ls3[2] = {0ull, 0ull};
        const float* PH01s = PH01; const float* GRs = GR;
        if (GT) { stage_rows(stg, PH01, 2 * T); stage_rows(stg + 2 * T, GR, T); __syncthreads(); PH01s = stg; GRs = stg + 2 * T; }
#pragma unroll
        for (int pass = 0; pass < NPASS; ++pass) {          // column passes as in G2
            const int sg0 = pass * PWC;
            u64 Q[PWC][2], GCr[PWC][2], col[PWC][2];
#pragma unroll
            for (int sg = 0; sg < PWC; ++sg) {
                const int j = (sg0 + sg) * 32 + lane;
                ulonglong2 q = make_ulonglong2(pk2(NEG_BIG, NEG_BIG), pk2(NEG_BIG, NEG_BIG)), g = make_ulonglong2(0ull, 0ull);
                if (j < Nc) {
                    q = *reinterpret_cast<const ulonglong2*>(QH + j * HD + k0);
                    g = *reinterpret_cast<const ulonglong2*>(GC + j * HD + k0);
                }
                Q[sg][0] = q.x; Q[sg][1] = q.y; GCr[sg][0] = g.x; GCr[sg][1] = g.y; col[sg][0] = 0ull; col[sg][1] = 0ull;
            }
            const float* Prow = PH01s + (size_t)hr0 * PROW; const float* Grow = GRs + (size_t)hr0 * HD;
            const uint32_t* brow = ybits + sg0 + (size_t)hr0 * WPc; float* rsrow = RS3d + (size_t)hr0 * HD;
            if (pass == 0) sweep2_bwd<PWC, false>(Prow, Grow, brow, WPc, hr1 - hr0, rg, M2_NRG, kg, Q, GCr, col, ls3, rsrow, lane);
            else sweep2_bwd<PWC, true>(Prow, Grow, brow, WPc, hr1 - hr0, rg, M2_NRG, kg, Q, GCr, col, ls3, rsrow, lane);
            if constexpr (PWC >= 5) combine_cols_2pass<PWC>(col, scratch, rg, M2_NRG, kg, lane);
            else combine_cols<PWC>(col, scratch, rg, M2_NRG, kg, lane);
            if (rg == 0) {
#pragma unroll
                for (int sg = 0; sg < PWC; ++sg) {
                    const int j = (sg0 + sg) * 32 + lane;
                    if (j < Nc) *reinterpret_cast<ulonglong2*>(CS3d + j * HD + k0) = make_ulonglong2(col[sg][0], col[sg][1]);
                }
            }
        }
        const float t = reduce4(ls3[0], ls3[1], lane);
        if ((lane & 7) == 0) lsw[rg * HD + k0 + ch] = t;
    }
    __syncthreads();
    if (CL && split) {
        // label sums of this half in row-group order -> lsw[0][.], the other row groups zero, so that phase J's sum over the row
        // groups yields rank 0's + rank 1's
        float ls = 0.f;
        if (tid < HD) for (int w = 0; w < M2_NRG; ++w) ls += lsw[w * HD + tid];
        __syncthreads();
        if (tid < M2_NRG * HD) lsw[tid] = tid < HD ? ls : 0.f;
        __syncthreads();
        xchg(RS3d, CS3d, Nc * (HD / 4), lsw, HD);
    }
    for (int idx = tid; idx < T; idx += M2_T) {       // diagonal pair: l = 0
        const int c = idx / HD, k = idx - c * HD;
        const float d = (PH01[p01_idx(c, k)] + QH[idx]) > 0.f ? GR[idx] + GC[idx] : 0.f;
        RS3d[idx] -= d; CS3d[idx] -= d;
    }
    __syncthreads();
    M2_PHASE(9);

    // ---------------- J. hunk first-layer weights, d/dnb -----------------------------------------------------
    for (int e = tid; e < 8 * HD + HD; e += M2_T) {
        if (e < 8 * HD) {
            const int row = e / HD, k = e - row * HD, chn = row & 3;
            const float* src = row < 4 ? RS3d : CS3d;
            float acc = 0.f;
            for (int n = 0; n < Nc; ++n) acc = fmaf(nb[4 * n + chn], src[n * HD + k], acc);
            gp[po.hnk_w1 + e] = acc;
        } else {
            const int k = e - 8 * HD;
            float acc = 0.f, ls = 0.f;
            for (int n = 0; n < Nc; ++n) acc += RS3d[n * HD + k];
            for (int w = 0; w < M2_NRG; ++w) ls += lsw[w * HD + k];
            gp[po.hnk_b1 + k] = acc;
            gp[po.hnk_w1 + 9 * HD + k] = ls;
            gp[po.hnk_w1 + 8 * HD + k] = acc - ls;
        }
    }
    for (int idx = tid; idx < Nc * 4; idx += M2_T) {
        const int n = idx >> 2, chn = idx & 3;
        float v = 0.f;
#pragma unroll
        for (int k = 0; k < HD; ++k) {
            v = fmaf(V1[chn * HD + k], RS3d[n * HD + k], v);
            v = fmaf(V1[(4 + chn) * HD + k], CS3d[n * HD + k], v);
        }
        dnb[idx] = v;
        if (dbg) dbg[(size_t)Ne * 21 + Nc * 4 + 4 * T + idx] = v;
    }
    __syncthreads();
    if (!a.ent) return;

    // ---------------- K. pooling backward ---------------------------------------------------------------------
    // dB2[q] = dnb[hunk(li)] + dnb[hunk(lj)] for q < L(L-1);  dx2[gi] += dB2[q][0], dx2[gj] += dB2[q][1]
    for (int idx = tid; idx < Ne * 4; idx += M2_T) {
        const int i = idx >> 2, chn = idx & 3;
        dl[idx] = (i < Lb && hm[i] >= 0) ? dnb[4 * hm[i] + chn] : 0.f;
    }
    __syncthreads();
    if (a.edge) {       // variant 4: d/d(a1 - a0) per index line, u_l = dl[l][3] - dl[l][2]; a pair (li, lj) receives u_li + u_lj
        float* uE = sm + L_.RA;                             // the row sums of a1 are dead since the pooling forward
        for (int i = tid; i < Ne; i += M2_T) uE[i] = dl[4 * i + 3] - dl[4 * i + 2];
    }
    M2_PHASE(12);
    if (ident) {
        float p0 = 0.f, p1 = 0.f;
        for (int i = tid; i < Ne; i += M2_T) { p0 += dl[4 * i]; p1 += dl[4 * i + 1]; }
        const float D0 = mid2_block_sum(p0, red);
        const float D1 = mid2_block_sum(p1, red);
        const float fn = (float)nm1;
        for (int i = tid; i < Ne; i += M2_T) {
            const float a0 = dl[4 * i], a1 = dl[4 * i + 1];
            dx2[i] = (fmaf(fn, a0, D0 - a0)) + (fmaf(fn, a1, D1 - a1));
        }
    } else if (Lb < 2) {
        for (int i = tid; i < Ne; i += M2_T) dx2[i] = 0.f;
    } else {
        // general path (mirror of the forward): the row part of dx2[gi] runs over the consecutive flat indices
        // [gi n, gi n + n) below qmax = L (L-1) -> closed form from prefix sums of dl; the column part is gathered
        // with incrementally updated local coordinates.
        const int n = nm1, m = Lb - 1, qmax = Lb * m, d = n - m;
        float* PD = SP;                                 // exclusive prefix of dl[.][0] over the L index lines
        if (warp == 0) warp_excl_scan(PD, dl, 4, Lb, lane);
        int nchunk = M2_T / Ne;
        nchunk = nchunk < 1 ? 1 : (nchunk > 4 ? 4 : nchunk);
        float* partC = scratch;                         // [nchunk][Ne]
        float* dl1 = TP;                                // channel 1 of dl, planar (TP is dead after the forward)
        for (int i = tid; i < Ne; i += M2_T) dl1[i] = dl[4 * i + 1];
        __syncthreads();
        // grid rows of this CTA: all of them, or (a cluster shares the commit) one half of the rows below qmax
        const int gtot = min(Ne, (qmax + n - 1) / n);
        const int gr0 = CL && split && crank ? (gtot + 1) >> 1 : 0, gr1 = CL && split ? (crank ? gtot : (gtot + 1) >> 1) : Ne;
        for (int t = tid; t < nchunk * Ne; t += M2_T) {
            const int c = t / Ne, me = t - c * Ne;
            const int lo = gr0 + (c * (gr1 - gr0)) / nchunk, hi = gr0 + ((c + 1) * (gr1 - gr0)) / nchunk;
            float acc = 0.f;
#pragma unroll
            for (int part = 0; part < 2; ++part) {      // gi < gj (flat column gj - 1), then gi > gj (flat column gj)
                const int g0 = part == 0 ? lo : max(lo, me + 1), g1 = part == 0 ? min(hi, me) : hi;
                if (g0 >= g1) continue;
                const int q = g0 * n + me - (part == 0 ? 1 : 0);
                if (q >= qmax) continue;
                int li = q / m, sloc = q - li * m;
                const int trips = min(g1 - g0, (qmax - 1 - q) / n + 1);      // rows with flat index below qmax
                if (d < m) {                            // counted and branch-free: at most one local-row wrap per step
#pragma unroll 4
                    for (int it = 0; it < trips; ++it) {
                        const int lj = sloc + (sloc >= li);
                        acc += dl1[li] + dl1[lj];
                        sloc += d;
                        const int w = sloc >= m;
                        sloc -= w ? m : 0;
                        li += 1 + w;
                    }
                } else {
                    for (int it = 0; it < trips; ++it) {
                        const int lj = sloc + (sloc >= li);
                        acc += dl1[li] + dl1[lj];
                        sloc += d; ++li;
                        while (sloc >= m) { sloc -= m; ++li; }
                    }
                }
            }
            partC[(size_t)c * Ne + me] = acc;
        }
        __syncthreads();
        M2_PHASE(13);
        for (int gi = tid; gi < Ne; gi += M2_T) {
            const int qa = gi * n, qb = min(qa + n, qmax);
            float acc = 0.f;
            if (qa < qmax) {
                int li = qa / m, sloc = qa - li * m, rem = qb - qa;
                while (rem > 0) {
                    const int c = min(rem, m - sloc), sb = sloc + c;
                    acc = fmaf((float)c, dl[4 * li], acc);
                    acc += offdiag_prefix(PD, dl, 4, li, sb) - offdiag_prefix(PD, dl, 4, li, sloc);
                    rem -= c; ++li; sloc = 0;
                }
            }
            float t = 0.f;
            for (int c = 0; c < nchunk; ++c) t += partC[(size_t)c * Ne + gi];
            if (CL && split) { dx2[gi] = acc; partC[gi] = t; }     // the column part is this half's: completed below
            else dx2[gi] = acc + t;
        }
        if (CL && split) {
            __syncthreads();
            xchg(nullptr, partC, (Ne + 3) >> 2, nullptr, 0);
            for (int gi = tid; gi < Ne; gi += M2_T) dx2[gi] += partC[gi];
        }
    }
    __syncthreads();
    if (dbg) for (int n = tid; n < Ne; n += M2_T) dbg[(size_t)Ne * 21 + Nc * 8 + 4 * T + n] = dx2[n];
    M2_PHASE(10);

    // ---------------- L. entity-state MLP backward (model_2.py:190-205) and W5/b5 (model_2.py:172-175) ------------
    {
        // per-node rows of a chunk: Sa [S | x 1 0 0], dz, ZD [relu(Z) du | du 0 0 0]
        float* Sa = uni; float* dzs = Sa + M2_CH * 24; float* ZD = dzs + M2_CH * HD;
        float* Mx = scratch;                           // [22][20]: M = S^T dz, then sum_n x dz, sum_n dz
        const int slice = tid & 15, grp = tid >> 4;
        float accA = 0.f, accC = 0.f;                  // one reduced output per thread, summed over the chunks
        for (int c0 = 0; c0 < Ne; c0 += M2_CH) {
            const int nn = min(M2_CH, Ne - c0);
            if (a.scache) {                              // S rows of the chunk: from the forward's copy, else from HBM / L2 again
                const float* Sall = SC;
                for (int e = tid; e < nn * 5; e += M2_T) {
                    const int n = e / 5, j = e - n * 5;
                    *reinterpret_cast<float4*>(Sa + n * 24 + 4 * j) = *reinterpret_cast<const float4*>(Sall + (size_t)(c0 + n) * HD + 4 * j);
                }
            } else {
                coop_load_S(Sa, 24, c0, nn);
            }
            __syncthreads();
            // step 1: two threads per entity: recompute the hidden layer, back-propagate, write GE
            for (int base = 0; base < 2 * nn; base += M2_T) {
                const int t = base + tid, n = t >> 1, h = t & 1, node = c0 + n;
                const bool valid = n < nn;
                float dzh[10];
#pragma unroll
                for (int j = 0; j < 10; ++j) dzh[j] = 0.f;
                if (valid) {
                    float S[HD], Zh[10];
                    load20s(S, Sa + n * 24);
                    const float xv = xs[node];
                    hidden_half(Zh, S, xv, h);
                    const float du = x2[node] > 0.f ? dx2[node] : 0.f;
#pragma unroll
                    for (int j2 = 0; j2 < 5; ++j2) {
                        const int k = 10 * h + 2 * j2;
                        dzh[2 * j2] = Zh[2 * j2] > 0.f ? du * u2[k] : 0.f;
                        dzh[2 * j2 + 1] = Zh[2 * j2 + 1] > 0.f ? du * u2[k + 1] : 0.f;
                        *reinterpret_cast<float2*>(dzs + n * HD + k) = make_float2(dzh[2 * j2], dzh[2 * j2 + 1]);
                        *reinterpret_cast<float2*>(ZD + n * 24 + k) =
                            make_float2(fmaxf(Zh[2 * j2], 0.f) * du, fmaxf(Zh[2 * j2 + 1], 0.f) * du);
                    }
                    if (h == 0) {
                        *reinterpret_cast<float4*>(Sa + n * 24 + HD) = make_float4(xv, 1.f, 0.f, 0.f);
                        *reinterpret_cast<float4*>(ZD + n * 24 + HD) = make_float4(du, 0.f, 0.f, 0.f);
                    }
                }
                float dz[HD];
#pragma unroll
                for (int j = 0; j < 10; ++j) {
                    const float o = __shfl_xor_sync(0xffffffffu, dzh[j], 1);
                    dz[j] = h ? o : dzh[j]; dz[10 + j] = h ? dzh[j] : o;
                }
                if (valid) {                           // GE_n[q] = sum_k W5U[q][k] dz[k], q = 10 h .. 10 h + 9
                    // inline entity stage: GE takes the place of S in shared memory (this chunk's S rows were copied to Sa)
                    float* ge = (a.inl ? SC + (size_t)node * HD : a.GE + ((size_t)b * Ne + node) * HD) + 10 * h;
                    float* ge_dbg = (a.inl && dbg) ? a.GE + ((size_t)b * Ne + node) * HD + 10 * h : nullptr;
#pragma unroll
                    for (int j2 = 0; j2 < 5; ++j2) {
                        float g0 = 0.f, g1 = 0.f;
                        const float* w0 = W5U + (10 * h + 2 * j2) * HD;
#pragma unroll
                        for (int k4 = 0; k4 < 5; ++k4) {
                            const float4 u = *reinterpret_cast<const float4*>(w0 + 4 * k4);
                            const float4 v = *reinterpret_cast<const float4*>(w0 + HD + 4 * k4);
                            g0 = fmaf(u.x, dz[4 * k4], g0); g0 = fmaf(u.y, dz[4 * k4 + 1], g0);
                            g0 = fmaf(u.z, dz[4 * k4 + 2], g0); g0 = fmaf(u.w, dz[4 * k4 + 3], g0);
                            g1 = fmaf(v.x, dz[4 * k4], g1); g1 = fmaf(v.y, dz[4 * k4 + 1], g1);
                            g1 = fmaf(v.z, dz[4 * k4 + 2], g1); g1 = fmaf(v.w, dz[4 * k4 + 3], g1);
                        }
                        *reinterpret_cast<float2*>(ge + 2 * j2) = make_float2(g0, g1);
                        if (ge_dbg) *reinterpret_cast<float2*>(ge_dbg + 2 * j2) = make_float2(g0, g1);
                    }
                }
            }
            __syncthreads();
            // step 2: [S | x | 1]^T dz over the chunk's nodes, 4 x 4 register tiles, 16 node slices per tile
            if (grp < 30) {
                const int a0 = 4 * (grp / 5), b0 = 4 * (grp % 5);
                float acc[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) acc[i] = 0.f;
                tile_acc(acc, Sa, 24, dzs, HD, a0, b0, slice, nn);
                accA += reduce16(acc, lane);
            } else if (grp < 36) {
                const int kb = 4 * (grp - 30);                             // column sums of ZD: du2[0..19], dc2
                float cs[4] = {0.f, 0.f, 0.f, 0.f};
                for (int n = slice; n < nn; n += 16) {
                    const float4 v = *reinterpret_cast<const float4*>(ZD + n * 24 + kb);
                    cs[0] += v.x; cs[1] += v.y; cs[2] += v.z; cs[3] += v.w;
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) cs[j] = half_sum(cs[j]);
                accC += slice == 0 ? cs[0] : slice == 1 ? cs[1] : slice == 2 ? cs[2] : cs[3];
            }
            __syncthreads();
        }
        if (grp < 30) {
            const int r = 4 * (grp / 5) + (slice >> 2), k = 4 * (grp % 5) + (slice & 3);
            if (r < HD + 2) Mx[r * HD + k] = accA;
        } else if (grp < 36 && slice < 4) {
            const int k = 4 * (grp - 30) + slice;
            if (k < HD) gp[po.nod_w2 + k] = accC;
            else if (k == HD) gp[po.nod_b2] = accC;
        }
        __syncthreads();
        // dU1e = W5^T M + nb5 b5 (x) dc1 ; dW5 = M U1e^T ; db5 = nb5 U1e dc1 ; dU1[0] = sum x dz ; dc1 = sum dz
        const float* dc1v = Mx + (HD + 1) * HD;
        for (int e = tid; e < 860; e += M2_T) {
            float acc = 0.f;
            if (e < 400) {
                const int m = e / HD, k = e - m * HD;
#pragma unroll
                for (int q = 0; q < HD; ++q) acc = fmaf(W5[q * HD + m], Mx[q * HD + k], acc);
                gp[po.nod_w1 + HD + e] = fmaf(nb5 * b5[m], dc1v[k], acc);
            } else if (e < 800) {
                const int q = (e - 400) / HD, m = (e - 400) - q * HD;
#pragma unroll
                for (int k = 0; k < HD; ++k) acc = fmaf(Mx[q * HD + k], U1[(1 + m) * HD + k], acc);
                gp[po.ent_w5 + (e - 400)] = acc;
            } else if (e < 820) {
                const int m = e - 800;
#pragma unroll
                for (int k = 0; k < HD; ++k) acc = fmaf(U1[(1 + m) * HD + k], dc1v[k], acc);
                gp[po.ent_b5 + m] = nb5 * acc;
            } else if (e < 840) {
                gp[po.nod_w1 + (e - 820)] = Mx[HD * HD + (e - 820)];
            } else {
                gp[po.nod_b1 + (e - 840)] = dc1v[e - 840];
            }
        }
    }
    if (a.inl) {
        // ---------------- entity pair layer backward (entsp.cuh): first-layer weight gradients from GE ---------------------
        // v_ij[k] = [pre_ij[k] > 0] (GE_i[k] + GE_j[k]);  db = sum v, dU = sum x_i v, dV = sum x_j v, LS = sum over l_ij = 1
        __syncthreads();
        M2_PHASE(18);
        const bool use_cls = cmeta[1] != 0;
        const int mcl = cmeta[0];
        // w: U V c D of the layer; GRs / GCs: [Ne][20] d/d(row sums), d/d(column sums) (the node branch passes GE twice).
        // Leaves db, dU, dV, LS (20 each) in red[0..80).  Uses the union region from its start.
        auto ent_bwd = [&](const float* w, const float* GRs, const float* GCs) {
        const bool same = GRs == GCs;
        if (use_cls) {
            // CLASS TABLES: v_ij[k] = g_l[a][b][k] (GR_i[k] + GC_j[k]) with the 0/1 gates g_l[a][b][k] = [H_l[a][b][k] > 0].  All four
            // results are sums over pairs, so with the number of active pairs per node,
            //   Wrow_i = sum_j g_ij,  XWrow_i = sum_j x_j g_ij,  W1row_i = sum_{l_ij = 1} g_ij   (and the column forms over i),
            //   db = sum_n GR_n Wrow_n + GC_n Wcol_n,          dU = sum_n GR_n x_n Wrow_n + GC_n XWcol_n,
            //   dV = sum_n GR_n XWrow_n + GC_n x_n Wcol_n,     LS = sum_n GR_n W1row_n + GC_n W1col_n,
            // and the W's come from the same neighbour counts as the forward.
            const int m = mcl;
            float* G0 = uni; float* G1t = uni + m * m * HD;
            uint32_t* cnt = reinterpret_cast<uint32_t*>(GT ? tabs : uni + 2 * m * m * HD);      // [m][Ne]  c1o | c1i << 16
            float* part = uni + ((2 * m * m * HD + (GT ? 0 : Ne * m) + 3) & ~3);     // [M2_T][16] per-thread partial sums
            for (int e = tid; e < m * m * HD; e += M2_T) {
                const int k = e % HD, ab = e / HD, bq = ab % m, aq = ab / m;
                const float t0 = fmaf(cval[bq], w[HD + k], fmaf(cval[aq], w[k], w[2 * HD + k]));      // as in the forward: same gates
                G0[e] = t0 > 0.f ? 1.f : 0.f; G1t[e] = (t0 + w[3 * HD + k]) > 0.f ? 1.f : 0.f;
            }
            const int WU = (Ne + 31) >> 5;
            for (int e = tid; e < Ne * m; e += M2_T) {
                const int n = e / m, bq = e - n * m;
                int co = 0, ci = 0;
                for (int wq = 0; wq < WU; ++wq) {
                    const uint32_t mk = cmask[bq * WPe + wq];
                    co += __popc(ebits[n * WPe + wq] & mk); ci += __popc(ebT[n * WPe + wq] & mk);
                }
                cnt[bq * Ne + (clsv[n] >> 16)] = (uint32_t)co | ((uint32_t)ci << 16);      // [class][rank]
            }
            __syncthreads();
            const int k4 = 4 * (tid / (M2_T / KG));
            float a_db[4] = {0.f, 0.f, 0.f, 0.f}, a_dU[4] = {0.f, 0.f, 0.f, 0.f}, a_dV[4] = {0.f, 0.f, 0.f, 0.f}, a_LS[4] = {0.f, 0.f, 0.f, 0.f};
            for (int r = tid % (M2_T / KG); r < Ne; r += M2_T / KG) {      // lanes = consecutive ranks (see the forward)
                const int n = ordv[r], aq = clsv[n] & 0xffff;
                const float xn = xs[n];
                const float4 gr4 = *reinterpret_cast<const float4*>(GRs + (size_t)n * HD + k4);
                const float4 gc4 = *reinterpret_cast<const float4*>(GCs + (size_t)n * HD + k4);
                float wr[4] = {0.f, 0.f, 0.f, 0.f}, xwr[4] = {0.f, 0.f, 0.f, 0.f}, w1r[4] = {0.f, 0.f, 0.f, 0.f};
                float wc[4] = {0.f, 0.f, 0.f, 0.f}, xwc[4] = {0.f, 0.f, 0.f, 0.f}, w1c[4] = {0.f, 0.f, 0.f, 0.f};
                const float* gab0 = G0 + aq * m * HD + k4; const float* gab1 = G1t + aq * m * HD + k4;
                const float* gba0 = G0 + aq * HD + k4;     const float* gba1 = G1t + aq * HD + k4;
                for (int bq = 0; bq < m; ++bq) {
                    const uint32_t pk = cnt[bq * Ne + r];
                    const int c1o = (int)(pk & 0xffffu), c1i = (int)(pk >> 16), tot = csize[bq] - (aq == bq ? 1 : 0);
                    const float f1o = (float)c1o, f1i = (float)c1i, f0o = (float)(tot - c1o), f0i = (float)(tot - c1i), vb = cval[bq];
                    const float4 q0 = *reinterpret_cast<const float4*>(gab0 + bq * HD), q1 = *reinterpret_cast<const float4*>(gab1 + bq * HD);
                    const float4 r0 = *reinterpret_cast<const float4*>(gba0 + bq * m * HD), r1 = *reinterpret_cast<const float4*>(gba1 + bq * m * HD);
                    const float a0[4] = {q0.x, q0.y, q0.z, q0.w}, a1[4] = {q1.x, q1.y, q1.z, q1.w};
                    const float b0[4] = {r0.x, r0.y, r0.z, r0.w}, b1[4] = {r1.x, r1.y, r1.z, r1.w};
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const float l1o = f1o * a1[c], ro = fmaf(f0o, a0[c], l1o), l1i = f1i * b1[c], ci2 = fmaf(f0i, b0[c], l1i);
                        wr[c] += ro; xwr[c] = fmaf(vb, ro, xwr[c]); w1r[c] += l1o;
                        wc[c] += ci2; xwc[c] = fmaf(vb, ci2, xwc[c]); w1c[c] += l1i;
                    }
                }
                const float gr[4] = {gr4.x, gr4.y, gr4.z, gr4.w}, gc[4] = {gc4.x, gc4.y, gc4.z, gc4.w};
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    a_db[c] = fmaf(gr[c], wr[c], fmaf(gc[c], wc[c], a_db[c]));
                    a_dU[c] = fmaf(gr[c], xn * wr[c], fmaf(gc[c], xwc[c], a_dU[c]));
                    a_dV[c] = fmaf(gr[c], xwr[c], fmaf(gc[c], xn * wc[c], a_dV[c]));
                    a_LS[c] = fmaf(gr[c], w1r[c], fmaf(gc[c], w1c[c], a_LS[c]));
                }
            }
            float4* p4 = reinterpret_cast<float4*>(part + (size_t)tid * 16);
            p4[0] = make_float4(a_db[0], a_db[1], a_db[2], a_db[3]); p4[1] = make_float4(a_dU[0], a_dU[1], a_dU[2], a_dU[3]);
            p4[2] = make_float4(a_dV[0], a_dV[1], a_dV[2], a_dV[3]); p4[3] = make_float4(a_LS[0], a_LS[1], a_LS[2], a_LS[3]);
            __syncthreads();
            if (tid < 4 * HD) {                             // fixed-order sum over the 128 node slots of a channel group
                const int qn = tid / HD, k = tid - qn * HD, kgq = k >> 2, cc2 = k & 3;
                float t = 0.f;
                for (int s2 = 0; s2 < M2_T / KG; ++s2) t += part[(size_t)(kgq * (M2_T / KG) + s2) * 16 + 4 * qn + cc2];
                red[tid] = t;
            }
        } else {
            // GENERAL attributes: suffix sums of GC (for the row sums) and of GR (for the column sums) over the sorted order,
            // one warp per channel (M2_NW == HD), then searches + the edge walk
            float* SGC = uni; float* SGR = same ? uni : uni + 20 * (Ne + 1);
            float* part = uni + (same ? 20 : 40) * (Ne + 1);                         // [M2_T][8]
            for (int pass = 0; pass < (same ? 1 : 2); ++pass) {
                const float* G = pass ? GRs : GCs;
                const int k = warp;
                const int per = (Ne + 31) >> 5, lo = min(lane * per, Ne), hi = min(lo + per, Ne);
                float sum = 0.f;
                for (int r = hi - 1; r >= lo; --r) sum += G[(size_t)ordv[r] * HD + k];
                float incl = sum;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const float t = __shfl_down_sync(0xffffffffu, incl, o); if (lane + o < 32) incl += t; }
                float run = incl - sum;
                float* dst = (pass ? SGR : SGC) + (size_t)k * (Ne + 1);
                for (int r = hi - 1; r >= lo; --r) { run += G[(size_t)ordv[r] * HD + k]; dst[r] = run; }
                if (lane == 0) dst[Ne] = 0.f;
            }
            __syncthreads();
            int P2 = 1;
            while (P2 <= Ne) P2 <<= 1;
            constexpr int NSLOT = M2_T / 10;
            const int slot = tid / 10, c0 = 2 * (tid % 10);
            const float Uc[2] = {w[c0], w[c0 + 1]}, Vc[2] = {w[HD + c0], w[HD + c0 + 1]};
            const float Cc[2] = {w[2 * HD + c0], w[2 * HD + c0 + 1]}, Dc[2] = {w[3 * HD + c0], w[3 * HD + c0 + 1]};
            const int WU = (Ne + 31) >> 5;
            float db[2] = {0.f, 0.f}, dU[2] = {0.f, 0.f}, dV[2] = {0.f, 0.f}, LS[2] = {0.f, 0.f};
            for (int n = slot; n < Ne; n += NSLOT) {             // dense (l = 0) part
                const float xn = xs[n];
                const float2 gr2 = *reinterpret_cast<const float2*>(GRs + (size_t)n * HD + c0);
                const float2 gc2 = *reinterpret_cast<const float2*>(GCs + (size_t)n * HD + c0);
                const float gr[2] = {gr2.x, gr2.y}, gc[2] = {gc2.x, gc2.y};
                float pb[2], qb[2];
#pragma unroll
                for (int h = 0; h < 2; ++h) { pb[h] = fmaf(xn, Uc[h], Cc[h]); qb[h] = fmaf(xn, Vc[h], Cc[h]); }
                int r[4] = {0, 0, 0, 0};
                const float sw[4] = {Vc[0], Vc[1], Uc[0], Uc[1]}, sb[4] = {pb[0], pb[1], qb[0], qb[1]};
                for (int step = P2 >> 1; step > 0; step >>= 1) {        // same predicate as the forward: identical gates
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int probe = r[u] + step - 1;
                        const float xv = xsort[probe < Ne ? probe : Ne - 1];
                        const bool act = fmaf(xv, sw[u], sb[u]) > 0.f;
                        if (probe < Ne && act != (sw[u] >= 0.f)) r[u] += step;
                    }
                }
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    float cnt, sg;
                    entsp_active(r[h], Ne, Vc[h] >= 0.f, SGC + (size_t)(c0 + h) * (Ne + 1), cnt, sg);
                    const float rsd = fmaf(cnt, gr[h], sg) - (fmaf(xn, Vc[h], pb[h]) > 0.f ? gr[h] + gc[h] : 0.f);
                    entsp_active(r[2 + h], Ne, Uc[h] >= 0.f, SGR + (size_t)(c0 + h) * (Ne + 1), cnt, sg);
                    const float csd = fmaf(cnt, gc[h], sg) - (fmaf(xn, Uc[h], qb[h]) > 0.f ? gr[h] + gc[h] : 0.f);
                    db[h] += rsd; dU[h] = fmaf(xn, rsd, dU[h]); dV[h] = fmaf(xn, csd, dV[h]);
                }
            }
            {   // l = 1 pairs: every slot walks an equal share of the edges; all four results are sums over edges
                const int nnz = rptr[Ne], per = (nnz + NSLOT - 1) / NSLOT, e0 = min(slot * per, nnz), e1 = min(e0 + per, nnz);
                if (e1 > e0) {
                    const EdgeCursor cur = edge_seek(ebits, WPe, rptr, Ne, P2, e0);
                    int row = cur.row, wq = cur.w;
                    uint32_t bits = cur.bits;
                    float xo = xs[row], b0 = fmaf(xo, Uc[0], Cc[0]), b1 = fmaf(xo, Uc[1], Cc[1]);
                    float2 go = *reinterpret_cast<const float2*>(GRs + (size_t)row * HD + c0);
                    for (int e = e0; e < e1; ++e) {
                        while (!bits) {
                            if (++wq == WU) {
                                wq = 0; ++row;
                                xo = xs[row]; b0 = fmaf(xo, Uc[0], Cc[0]); b1 = fmaf(xo, Uc[1], Cc[1]);
                                go = *reinterpret_cast<const float2*>(GRs + (size_t)row * HD + c0);
                            }
                            bits = ebits[row * WPe + wq];
                        }
                        const int j = (wq << 5) + __ffs(bits) - 1;
                        bits &= bits - 1;
                        const float xj = xs[j];
                        const float2 gj = *reinterpret_cast<const float2*>(GCs + (size_t)j * HD + c0);
                        const float t0 = fmaf(xj, Vc[0], b0), t1 = fmaf(xj, Vc[1], b1), g0 = go.x + gj.x, g1 = go.y + gj.y;
                        const float v10 = (t0 + Dc[0]) > 0.f ? g0 : 0.f, v11 = (t1 + Dc[1]) > 0.f ? g1 : 0.f;
                        const float d0 = v10 - (t0 > 0.f ? g0 : 0.f), d1 = v11 - (t1 > 0.f ? g1 : 0.f);
                        db[0] += d0; db[1] += d1;
                        dU[0] = fmaf(xo, d0, dU[0]); dU[1] = fmaf(xo, d1, dU[1]);
                        dV[0] = fmaf(xj, d0, dV[0]); dV[1] = fmaf(xj, d1, dV[1]);
                        LS[0] += v10; LS[1] += v11;
                    }
                }
            }
            *reinterpret_cast<float4*>(part + (size_t)tid * 8) = make_float4(db[0], db[1], dU[0], dU[1]);
            *reinterpret_cast<float4*>(part + (size_t)tid * 8 + 4) = make_float4(dV[0], dV[1], LS[0], LS[1]);
            __syncthreads();
            if (tid < 4 * HD) {                                 // fixed-order sum over the 64 threads that own a channel pair
                const int qn = tid / HD, k = tid - qn * HD, kp = k >> 1, hh = k & 1;
                float t = 0.f;
                for (int s2 = 0; s2 < M2_T / 10; ++s2) t += part[(size_t)(kp + 10 * s2) * 8 + 2 * qn + hh];      // slot order
                red[tid] = t;
            }
        }
        __syncthreads();
        };
        ent_bwd(wE, SC, SC);
        M2_PHASE(19);
        if (tid < HD) {
            const float dbk = red[tid], lsk = red[3 * HD + tid];
            gp[po.ent_b1 + tid] = dbk;
            gp[po.ent_w1 + tid] = red[HD + tid];
            gp[po.ent_w1 + HD + tid] = red[2 * HD + tid];
            gp[po.ent_w1 + 2 * HD + tid] = dbk - lsk;
            gp[po.ent_w1 + 3 * HD + tid] = lsk;
        }
        if (a.edge) {
            // ---------------- variant 4: entity-edge branch backward (model_4.py:92-98, 206-304) ----------------------------------
            // de_ij = a1 a0 (u_li + u_lj) is d/d(logit difference) of the soft edge of pair (i,j); from there the chain is the relation
            // head's: delta sums over the Ne x Ne grid (rows in chunks of E_RCH: pass A recomputes the soft edge and tabulates de,
            // pass B accumulates the gated row / column / label sums four channels per warp), the head's node-level backward, and
            // the first (tied, rank-1) layer through ent_bwd.
            constexpr int E_RCH = 32;
            __syncthreads();
            const int WUe = (Ne + 31) >> 5, DWe = WUe * 32;
            const float* uE = sm + L_.RA;
            float* PRe01 = uni; float* PCe = uni + Ne * PROW;
            float* CSmE = uni + Ne * 60;                        // [Ne][20]
            float* det = CSmE + Ne * HD;                        // [E_RCH][DWe] de of the current row chunk
            float* RSmE = SC;                           // [Ne][20] (GE is dead)
            {
                const float4* src = reinterpret_cast<const float4*>(a.PREg + (size_t)b * Ne * 60);
                for (int i = tid; i < Ne * 15; i += M2_T) reinterpret_cast<float4*>(uni)[i] = __ldcg(src + i);
            }
            const float bdE = blkE[1001] - blkE[1000];
            u64 gam2[HD / 2];
#pragma unroll
            for (int k = 0; k < HD / 2; ++k) gam2[k] = pk2(gamE[2 * k], gamE[2 * k + 1]);
            const bool gen = !ident;
            const int mloc = Lb - 1, qmaxE = Lb >= 2 ? Lb * mloc : 0;
            const float inv_m = mloc > 0 ? 1.f / (float)mloc : 0.f;
            float dsum_acc = 0.f;
            u64 lsmE[2] = {0ull, 0ull};
            __syncthreads();
            for (int r0 = 0; r0 < Ne; r0 += E_RCH) {
                const int nr = min(E_RCH, Ne - r0);
                // pass A: lanes = columns, all 20 channels: the soft edge again, then de
                for (int cb = 0; cb < WUe; ++cb) {
                    const int j = cb * 32 + lane;
                    const bool ok = j < Ne;
                    u64 Q2[HD / 2];
#pragma unroll
                    for (int q4 = 0; q4 < 5; ++q4) {
                        ulonglong2 v = make_ulonglong2(pk2(NEG_BIG, NEG_BIG), pk2(NEG_BIG, NEG_BIG));
                        if (ok) v = *reinterpret_cast<const ulonglong2*>(PCe + j * HD + 4 * q4);
                        Q2[2 * q4] = v.x; Q2[2 * q4 + 1] = v.y;
                    }
                    const float uj = ok ? uE[j] : 0.f;
                    for (int rl = warp; rl < nr; rl += M2_NW) {
                        const int r = r0 + rl;
                        const uint32_t bit = (ebits[r * WPe + cb] >> lane) & 1u;
                        const float* prow = PRe01 + (size_t)r * PROW + bit * 4;
                        u64 da = pk2(bdE, 0.f), db2 = 0ull;         // the forward's arithmetic, operation for operation
#pragma unroll
                        for (int q4 = 0; q4 < 5; ++q4) {
                            const ulonglong2 pv = *reinterpret_cast<const ulonglong2*>(prow + q4 * 8);
                            da = fma2(relu2(add2(pv.x, Q2[2 * q4])), gam2[2 * q4], da);
                            db2 = fma2(relu2(add2(pv.y, Q2[2 * q4 + 1])), gam2[2 * q4 + 1], db2);
                        }
                        float dlo, dhi;
                        upk2(add2(da, db2), dlo, dhi);
                        const float d = dlo + dhi;
                        const float e = expf(-fabsf(d)), inv = 1.f / (1.f + e);
                        const float a1 = d >= 0.f ? inv : e * inv, a0 = d >= 0.f ? e * inv : inv;
                        float up = 0.f;
                        if (ok && j != r) {
                            if (!gen) {
                                up = uE[r] + uj;
                            } else {
                                const int q = r * nm1 + j - (j > r ? 1 : 0);
                                if (q < qmaxE) {                    // local coordinates of the pair (utils2.py:123-137)
                                    int li = (int)(((float)q + 0.5f) * inv_m);
                                    int sl = q - li * mloc;
                                    if (sl < 0) { --li; sl += mloc; } else if (sl >= mloc) { ++li; sl -= mloc; }
                                    up = uE[li] + uE[sl + (sl >= li ? 1 : 0)];
                                }
                            }
                        }
                        const float de = a1 * a0 * up;
                        det[rl * DWe + cb * 32 + lane] = de;
                        dsum_acc += de;
                    }
                }
                __syncthreads();
                // pass B: a warp owns four channels and a quarter of the chunk's rows; columns in passes of four segments
                for (int cp = 0; cp * 4 < WUe; ++cp) {
                    u64 Q[4][2], col[4][2];
#pragma unroll
                    for (int sg = 0; sg < 4; ++sg) {
                        const int j = (cp * 4 + sg) * 32 + lane;
                        ulonglong2 q = make_ulonglong2(pk2(NEG_BIG, NEG_BIG), pk2(NEG_BIG, NEG_BIG));
                        if (j < Ne) q = *reinterpret_cast<const ulonglong2*>(PCe + j * HD + k0);
                        Q[sg][0] = q.x; Q[sg][1] = q.y; col[sg][0] = 0ull; col[sg][1] = 0ull;
                    }
                    const uint32_t lmask = 1u << lane;
                    for (int rl = rg; rl < nr; rl += M2_NRG) {
                        const int r = r0 + rl;
                        const float* prow0 = PRe01 + (size_t)r * PROW + kg * 8;
                        const float* prow1 = prow0 + 4;
                        u64 rp0 = 0ull, rp1 = 0ull;
#pragma unroll
                        for (int sg = 0; sg < 4; ++sg) {
                            const int wi = cp * 4 + sg;
                            if (wi < WUe) {
                                const bool bit = (ebits[r * WPe + wi] & lmask) != 0u;
                                const ulonglong2 pq = *reinterpret_cast<const ulonglong2*>(bit ? prow1 : prow0);
                                const float dv = det[rl * DWe + wi * 32 + lane];
                                const u64 d2 = pk2(dv, dv);
                                const u64 v0 = gate2(add2(pq.x, Q[sg][0]), d2), v1 = gate2(add2(pq.y, Q[sg][1]), d2);
                                col[sg][0] = add2(col[sg][0], v0); col[sg][1] = add2(col[sg][1], v1);
                                rp0 = add2(rp0, v0); rp1 = add2(rp1, v1);
                                const float lf = bit ? 1.f : 0.f;
                                const u64 l2 = pk2(lf, lf);
                                lsmE[0] = fma2(l2, v0, lsmE[0]); lsmE[1] = fma2(l2, v1, lsmE[1]);
                            }
                        }
                        const float tot = reduce4(rp0, rp1, lane);
                        if ((lane & 7) == 0) {
                            float* dst = RSmE + (size_t)r * HD + k0 + ch;
                            if (cp == 0) *dst = tot; else *dst += tot;
                        }
                    }
                    combine_cols<4>(col, scratch, rg, M2_NRG, kg, lane);
                    if (rg == 0) {
#pragma unroll
                        for (int sg = 0; sg < 4; ++sg) {
                            const int j = (cp * 4 + sg) * 32 + lane;
                            if (j < Ne) {
                                float c0v, c1v, c2v, c3v;
                                upk2(col[sg][0], c0v, c1v); upk2(col[sg][1], c2v, c3v);
                                float4* dst = reinterpret_cast<float4*>(CSmE + (size_t)j * HD + k0);
                                if (r0 == 0) *dst = make_float4(c0v, c1v, c2v, c3v);
                                else { const float4 o = *dst; *dst = make_float4(o.x + c0v, o.y + c1v, o.z + c2v, o.w + c3v); }
                            }
                        }
                    }
                }
                __syncthreads();
            }
            {
                const float t = reduce4(lsmE[0], lsmE[1], lane);
                if ((lane & 7) == 0) lsw[rg * HD + k0 + ch] = t;
            }
            M2_PHASE(23);
            const float dsumE = mid2_block_sum(dsum_acc, red);
            if (tid < HD) {
                float ls = 0.f;
                for (int w = 0; w < M2_NRG; ++w) ls += lsw[w * HD + tid];
                misc[tid] = ls;
            }
            if (tid == 0) { gp[po.eup_b2 + 1] = dsumE; gp[po.eup_b2] = -dsumE; }
            __syncthreads();
            // node level (the hunk head's phase H with the edge branch's weights): HS, bias and label rows
            const int slice = tid & 15, grp = tid >> 4;
            if (grp < 5) {
                const int kb = 4 * grp;
                float hs[4] = {0.f, 0.f, 0.f, 0.f}, cs[4] = {0.f, 0.f, 0.f, 0.f};
                for (int n = slice; n < Ne; n += 16) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float rs = RSmE[n * HD + kb + j];
                        hs[j] = fmaf(PRe01[p01_idx(n, kb + j)], rs, hs[j]);
                        hs[j] = fmaf(PCe[n * HD + kb + j], CSmE[n * HD + kb + j], hs[j]);
                        cs[j] += rs;
                    }
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) { hs[j] = half_sum(hs[j]); cs[j] = half_sum(cs[j]); }
                if (slice < 4) {
                    const int k = kb + slice;
                    const float hh = fmaf(DgE[k], misc[k], slice == 0 ? hs[0] : slice == 1 ? hs[1] : slice == 2 ? hs[2] : hs[3]);
                    const float c = (slice == 0 ? cs[0] : slice == 1 ? cs[1] : slice == 2 ? cs[2] : cs[3]) * gamE[k];
                    const float ls4 = misc[k] * gamE[k];
                    gp[po.eup_w2 + 2 * k + 1] = hh; gp[po.eup_w2 + 2 * k] = -hh;
                    gp[po.eup_b1 + k] = c; gp[po.eup_w1 + HD + k] = ls4; gp[po.eup_w1 + k] = c - ls4;
                }
            }
            // G1g of the edge head (the hunk head's table is dead): G1gE[q][m] = G1E[2 + q][m] gamE[m]
            for (int e = tid; e < 400; e += M2_T) G1g[e] = blkE[500 + 2 * HD + e] * gamE[e % HD];
            __syncthreads();
            // r, c -> shared memory over the (dead) head tables; eup_w1 rows 2.. = r^T RS4 + c^T CS4
            float* reS = uni; float* ceS = uni + Ne * HD; float* drE = uni + 2 * Ne * HD; float* dcE = det;     // det is dead
            for (int i = tid; i < Ne * 5; i += M2_T) {
                reinterpret_cast<float4*>(reS)[i] = __ldcg(reinterpret_cast<const float4*>(a.REg + (size_t)b * Ne * HD) + i);
                reinterpret_cast<float4*>(ceS)[i] = __ldcg(reinterpret_cast<const float4*>(a.CEg + (size_t)b * Ne * HD) + i);
            }
            __syncthreads();
            if (grp < 25) {
                float acc[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) acc[i] = 0.f;
                const int a0 = 4 * (grp / 5), b0 = 4 * (grp % 5);
                tile_acc(acc, reS, HD, RSmE, HD, a0, b0, slice, Ne);
                tile_acc(acc, ceS, HD, CSmE, HD, a0, b0, slice, Ne);
                const float v = reduce16(acc, lane);
                const int mm = a0 + (slice >> 2), k = b0 + (slice & 3);
                gp[po.eup_w1 + 2 * HD + mm * HD + k] = v * gamE[k];
            }
            // dr = RSm G1gE^T, dc = CSm G1gE^T (one thread per (node, side))
            for (int t = tid; t < 2 * Ne; t += M2_T) {
                const bool cside = t >= Ne;
                const int n = cside ? t - Ne : t;
                float in[HD], out[HD];
                load20s(in, (cside ? CSmE : RSmE) + n * HD);
                gemv20t(out, in, G1g);
                store20s((cside ? dcE : drE) + n * HD, out);
            }
            __syncthreads();
            // edg_w2 = RSe^T dr + CSe^T dc, edg_b2 = (Ne-1) sum (dr + dc); RSe / CSe over r / c (dead)
            for (int i = tid; i < Ne * 5; i += M2_T) {
                reinterpret_cast<float4*>(reS)[i] = __ldcg(reinterpret_cast<const float4*>(a.RSEg + (size_t)b * Ne * HD) + i);
                reinterpret_cast<float4*>(ceS)[i] = __ldcg(reinterpret_cast<const float4*>(a.CSEg + (size_t)b * Ne * HD) + i);
            }
            __syncthreads();
            if (grp < 25) {
                float acc[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) acc[i] = 0.f;
                const int a0 = 4 * (grp / 5), b0 = 4 * (grp % 5);
                tile_acc(acc, reS, HD, drE, HD, a0, b0, slice, Ne);
                tile_acc(acc, ceS, HD, dcE, HD, a0, b0, slice, Ne);
                const float v = reduce16(acc, lane);
                gp[po.edg_w2 + (a0 + (slice >> 2)) * HD + b0 + (slice & 3)] = v;
            } else if (grp < 30) {
                const int kb = 4 * (grp - 25);
                float cs[4] = {0.f, 0.f, 0.f, 0.f};
                for (int n = slice; n < Ne; n += 16)
#pragma unroll
                    for (int j = 0; j < 4; ++j) cs[j] += drE[n * HD + kb + j] + dcE[n * HD + kb + j];
#pragma unroll
                for (int j = 0; j < 4; ++j) cs[j] = half_sum(cs[j]);
                if (slice < 4)
                    gp[po.edg_b2 + kb + slice] = (float)(Ne - 1) * (slice == 0 ? cs[0] : slice == 1 ? cs[1] : slice == 2 ? cs[2] : cs[3]);
            }
            __syncthreads();
            // GRe = dr W2e^T -> the S / GE region, GCe = dc W2e^T -> the end of the union region; then the tied first layer
            float* GRe = SC; float* GCe = uni + uni_floats - Ne * HD;
            for (int t = tid; t < 2 * Ne; t += M2_T) {
                const bool cside = t >= Ne;
                const int n = cside ? t - Ne : t;
                float in[HD], out[HD];
                load20s(in, (cside ? dcE : drE) + n * HD);
                gemv20t(out, in, blkE + 80);
                store20s((cside ? GCe : GRe) + n * HD, out);
            }
            __syncthreads();
            ent_bwd(wEe, GRe, GCe);
            if (tid < HD) {
                const float dbk = red[tid], lsk = red[3 * HD + tid];
                gp[po.edg_b1 + tid] = dbk;
                gp[po.edg_w11 + tid] = red[HD + tid] + red[2 * HD + tid];      // tied: the same row multiplies x_i and x_j
                gp[po.edg_w12 + tid] = dbk - lsk;
                gp[po.edg_w12 + HD + tid] = lsk;
            }
        }
    }
    M2_PHASE(11);
}

}  // namespace hdgnn
