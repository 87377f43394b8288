// k_io: the two data formats either side of the hot path (SURVEY 8(f) rows 1 and 2), both HBM-bound byte/integer work.
//
//  * compact_from_raw_kernel  -- utils2.py:29-47 and the int() indexing of utils2.py:82,105 on the device: the arrays as
//    stored in CAdjs_{step}.npy / CHunkAdjs_{step}.npy (float64 or float32, diagonal = node attribute) become the u8
//    label grid + f32 diagonal the hot path reads.  8 (or 4) bytes in, 1 byte out per element.
//  * eval_counts_kernel       -- EvaluationFuncs.py:27-37 (top_ACC), :92-117 (prec / recall / f1, with and without the
//    ceil-on-channel-0 quirk) and :119-153 (AUC) as integer counters per commit, read straight from the probs the
//    relation head wrote; the (N,2,Ncr) device->host copy and the Python double loops disappear.
//  * hunk_groups_kernel       -- the commit-level answer of an untangling: the groups of hunks that a label bitmap (the
//    predicted relations of hdgnn_set_predictions, or the labels) joins, as connected components.
//  * partition_counts_kernel  -- how well two such groupings agree, per commit and over its real hunks only: pair counts,
//    group counts and largest overlaps, from which EvaluationFuncs.partition_metrics_from_counts derives pair precision /
//    recall / F1, the (adjusted) Rand index and purity.
//  * hunk_clusters_kernel     -- hunk groups formed from the relation probabilities instead of the arg-max bitmap: average
//    linkage over each commit's real hunks, merging two groups only while their mean relation probability clears a threshold;
//    its LINK instantiation records the whole merge sequence instead (hdgnn_hunk_linkage).
//  * linkage_cut_kernel       -- hunk groups from such a record at many thresholds, or at a group count, in one pass.
//
// Everything here except hunk_clusters_kernel is integer counting => bit-exact and order independent (integer atomics).  The
// clustering is fp32, but its merge sequence fixes every rounding, so it is deterministic and reproducible on the host.
#include "../../include/hdgnn.h"
#include "bits.cuh"
#include "common.cuh"
#include "host.cuh"

namespace hdgnn {

// ---------------------------------------------------------------------------------------------------------------
// raw (N,n,n) -> grid u8 (N,n,pitch), diag f32 (N,n).  One warp per ROWS_PER_WARP consecutive rows; lanes own the columns
// lane + 32 k, so every load instruction of a warp covers 256 (f64) contiguous bytes.  All loads of a row are in
// flight before the first convert.
// int(v) of utils2.py:82,105 truncates toward zero and indexes a size-2 axis: {-2,-1,0,1} are legal (python negative
// indices), anything else raises IndexError there -> *err = 1 here.  NaN fails the range test as well.
template <typename T, int KMAX>
__global__ void __launch_bounds__(256) compact_from_raw_kernel(const T* __restrict__ raw, int rows, int n, uint8_t* __restrict__ grid,
                                                               int pitch, float* __restrict__ diag, int* __restrict__ err) {
    const int lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    int bad = 0;
    for (int row = blockIdx.x * wpb + (threadIdx.x >> 5); row < rows; row += gridDim.x * wpb) {
        const int i = row % n;                              // row index inside its commit
        const T* src = raw + (size_t)row * n;
        T v[KMAX];
#pragma unroll
        for (int k = 0; k < KMAX; ++k) {
            const int j = lane + 32 * k;
            v[k] = j < n ? __ldg(src + j) : T(0);
        }
        uint8_t* dst = grid + (size_t)row * pitch;
#pragma unroll
        for (int k = 0; k < KMAX; ++k) {
            const int j = lane + 32 * k;
            if (j >= pitch) continue;
            uint8_t o = 0;
            if (j < n) {
                if (j == i) {
                    if (diag) diag[row] = (float)v[k];      // utils2.py:31-36: x_i = A_ii (float64 -> float32, round to nearest)
                } else {
                    const T t = v[k];
                    if (!(t > T(-3) && t < T(2))) bad = 1;
                    o = (uint8_t)(((int)t) & 1);            // -1 -> channel 1, -2 -> channel 0 (python indexing from the end)
                }
            }
            dst[j] = o;
        }
    }
    if (bad && err) atomicOr(err, 1);
}

// ---------------------------------------------------------------------------------------------------------------
// counts (B,8) int64: [0] arg-max hits, [1..3] tp fp fn of the reference's quirk form (y_true = ceil(label ch 0) = 1 - Y,
// y_pred = ceil(prob ch 0) = [prob0 > 0]), [4..6] tp fp fn of the conventional form (y_true = Y, y_pred = [p1 > p0]),
// [7] number of related pairs.  auc (B,2) int64: Mann-Whitney numerators 2 #{(pos,neg): s_neg < s_pos} + #{s_neg == s_pos}
// with [0] the reference's scoring (EvaluationFuncs.py:128-143: a pair is scored with the probability of the channel
// its label does NOT have) and [1] the conventional one (score = p1).  AUC = auc / (2 npos nneg).
constexpr int EV_T = 256;
constexpr int EV_PER = 8;                   // pairs per thread
constexpr int EV_CHUNK = EV_T * EV_PER;     // pairs per CTA
constexpr int EV_TILE = 2048;               // positives staged per round

__global__ void __launch_bounds__(EV_T) eval_counts_kernel(int Nc, const float* __restrict__ probs, const uint8_t* __restrict__ Y,
                                                           int y_pitch, unsigned long long* __restrict__ counts,
                                                           unsigned long long* __restrict__ auc, int auc_first) {
    __shared__ float posq[EV_TILE], posc[EV_TILE];
    __shared__ int npos_s;
    __shared__ unsigned long long red[8];
    const int b = blockIdx.y, tid = threadIdx.x, lane = tid & 31;
    const int nm1 = Nc - 1, Ncr = Nc * nm1;
    const float inv = 1.f / (float)nm1;
    const float* p0 = probs + (size_t)b * 2 * Ncr;
    const float* p1 = p0 + Ncr;
    const uint8_t* Yb = Y + (size_t)b * Nc * y_pitch;
    if (tid < 8) red[tid] = 0ull;
    __syncthreads();

    float sneg[EV_PER];                      // this thread's pairs as negatives (score p1 in both forms); +inf = not a negative
    int c[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int k = 0; k < EV_PER; ++k) {
        const int p = blockIdx.x * EV_CHUNK + k * EV_T + tid;
        sneg[k] = __int_as_float(0x7f800000);
        if (p < Ncr) {
            int s, t;
            unflat_pair(p, nm1, inv, s, t);
            const int y = Yb[(size_t)s * y_pitch + t] != 0;
            const float a = p0[p], d = p1[p];
            const int am = d > a;                             // np.argmax: ties -> channel 0
            c[0] += am == y;
            const int qt = !y, qp = a > 0.f;                  // quirk form scores channel 0
            c[1] += qt & qp; c[2] += (!qt) & qp; c[3] += qt & (!qp);
            c[4] += y & am; c[5] += (!y) & am; c[6] += y & (!am);
            c[7] += y;
            if (!y) sneg[k] = d;
        }
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int w = __reduce_add_sync(0xffffffffu, c[q]);
        if (lane == 0 && w) atomicAdd(&red[q], (unsigned long long)w);
    }
    __syncthreads();
    if (tid < 8 && red[tid]) atomicAdd(&counts[(size_t)b * 8 + tid], red[tid]);
    if (!auc || b < auc_first) return;

    // every CTA of the commit walks ALL pairs of the commit for the positives, EV_TILE candidates at a time
    unsigned long long nq = 0ull, ncv = 0ull;
    for (int base = 0; base < Ncr; base += EV_TILE) {
        __syncthreads();
        if (tid == 0) npos_s = 0;
        __syncthreads();
        for (int p = base + tid; p < min(base + EV_TILE, Ncr); p += EV_T) {
            int s, t;
            unflat_pair(p, nm1, inv, s, t);
            if (Yb[(size_t)s * y_pitch + t] != 0) {
                const int slot = atomicAdd(&npos_s, 1);       // order is irrelevant: the counters below are integers
                posq[slot] = p0[p]; posc[slot] = p1[p];
            }
        }
        __syncthreads();
        const int np = npos_s;
        unsigned int lq = 0u, lc = 0u;                        // <= 2 * EV_TILE * EV_PER per round
        for (int i = 0; i < np; ++i) {
            const float sq = posq[i], sc = posc[i];
#pragma unroll
            for (int k = 0; k < EV_PER; ++k) {
                lq += (sneg[k] < sq ? 2u : 0u) + (sneg[k] == sq ? 1u : 0u);
                lc += (sneg[k] < sc ? 2u : 0u) + (sneg[k] == sc ? 1u : 0u);
            }
        }
        nq += lq; ncv += lc;
    }
    nq = __reduce_add_sync(0xffffffffu, (unsigned int)(nq & 0xffffffffu)) + ((unsigned long long)__reduce_add_sync(0xffffffffu, (unsigned int)(nq >> 32)) << 32);
    ncv = __reduce_add_sync(0xffffffffu, (unsigned int)(ncv & 0xffffffffu)) + ((unsigned long long)__reduce_add_sync(0xffffffffu, (unsigned int)(ncv >> 32)) << 32);
    if (lane == 0) {
        if (nq) atomicAdd(&auc[(size_t)b * 2], nq);
        if (ncv) atomicAdd(&auc[(size_t)b * 2 + 1], ncv);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Hunk groups: weakly connected components of per-commit hunk graphs given as label bitmaps (bits.cuh layout).  One warp per
// commit.  The commit's rows are staged in shared memory and symmetrised in place, S = A | A^T with the diagonal and the padding
// dropped (32 x 32 ballot transposes, one unordered block pair at a time, so every block is read before it is written).  The
// sweep then works on bitsets: lane w holds word w of the unvisited set and of the frontier; a component is seeded at the
// lowest unvisited hunk -- which is therefore its smallest index, the label -- and every hunk of it ORs its row of S in once.
// Integer work only: the result does not depend on scheduling.
constexpr int HG_WARPS_MAX = 4;
constexpr size_t HG_SMEM_MAX = 48 * 1024;   // commits per CTA are chosen to stay within the default dynamic shared memory

__global__ void __launch_bounds__(32 * HG_WARPS_MAX) hunk_groups_kernel(int B, int n, int WP, const uint32_t* __restrict__ bits,
                                                                       int32_t* __restrict__ groups, int32_t* __restrict__ ngroups) {
    extern __shared__ __align__(16) uint32_t hg_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int b = blockIdx.x * (blockDim.x >> 5) + warp;
    if (b >= B) return;
    const int CW = (n + 31) >> 5;
    uint32_t* S = hg_smem + (size_t)warp * n * WP;
    {
        const uint4* src = reinterpret_cast<const uint4*>(bits + (size_t)b * n * WP);
        uint4* dst = reinterpret_cast<uint4*>(S);
        for (int i = lane; i < n * WP / 4; i += 32) dst[i] = __ldg(src + i);
    }
    __syncwarp();
    auto colmask = [n](int w) { const int c = n - 32 * w; return c >= 32 ? 0xffffffffu : (1u << c) - 1u; };     // w < CW: c >= 1
    for (int I = 0; I < CW; ++I) {
        for (int J = I; J < CW; ++J) {
            // lane l: word J of row 32 I + l (a) and word I of row 32 J + l (c)
            const int ri = 32 * I + lane, rj = 32 * J + lane;
            uint32_t a = ri < n ? S[ri * WP + J] & colmask(J) : 0u;
            uint32_t c = rj < n ? S[rj * WP + I] & colmask(I) : 0u;
            if (I == J) { a &= ~(1u << lane); c = a; }
            uint32_t ta = 0u, tc = 0u;          // lane k: bit k of every lane's a (word I of row 32 J + k of A^T), of c likewise
#pragma unroll
            for (int k = 0; k < 32; ++k) {
                const uint32_t x = __ballot_sync(0xffffffffu, (a >> k) & 1u), y = __ballot_sync(0xffffffffu, (c >> k) & 1u);
                if (lane == k) { ta = x; tc = y; }
            }
            if (ri < n) S[ri * WP + J] = a | tc;
            if (rj < n && I != J) S[rj * WP + I] = c | ta;
        }
    }
    __syncwarp();
    uint32_t U = lane < CW ? colmask(lane) : 0u;        // unvisited hunks
    int32_t* g = groups + (size_t)b * n;
    int ncomp = 0;
    for (;;) {
        const uint32_t any = __ballot_sync(0xffffffffu, U != 0u);
        if (!any) break;
        const int sl = __ffs(any) - 1;
        const int seed = 32 * sl + __ffs(__shfl_sync(0xffffffffu, U, sl)) - 1;
        const uint32_t U0 = U;
        uint32_t F = lane == sl ? 1u << (seed & 31) : 0u;      // frontier
        U &= ~F;
        for (;;) {
            const uint32_t fa = __ballot_sync(0xffffffffu, F != 0u);
            if (!fa) break;
            const int fl = __ffs(fa) - 1;
            const int v = 32 * fl + __ffs(__shfl_sync(0xffffffffu, F, fl)) - 1;
            if (lane == fl) F &= F - 1u;
            const uint32_t nw = lane < CW ? S[v * WP + lane] & U : 0u;
            U &= ~nw;
            F |= nw;
        }
        for (uint32_t m = U0 & ~U; m; m &= m - 1u) g[32 * lane + __ffs(m) - 1] = seed;
        ++ncomp;
    }
    if (lane == 0 && ngroups) ngroups[b] = ncomp;
}

// ---------------------------------------------------------------------------------------------------------------
// Partition agreement of two hunk labellings per commit, over the real hunks s < m = nh[b].  One warp per commit.  Every label
// value l owns a bitmap row of its hunks, Gp[l] (pred) and Gt[l] (truth), built by shared-memory atomicOr (integer, order-free);
// only the words below ceil(m / 32) of a row are used, and only the rows of labels that occur are cleared.  For hunk s with
// P = Gp[pred[s]], T = Gt[truth[s]]: popc(P & T) is the contingency cell n_ij holding s, so
//   sum_s (popc(P & T) - 1) = 2 * pairs joined in both, sum_s (popc(P) - 1) = 2 * pairs joined by pred (truth likewise);
//   s is its pred group's representative when it is the lowest bit of P, so the representatives count the groups;
//   max_j n_ij of pred group i is the max of popc(P & T) over its hunks (every non-empty cell holds one of them): an atomicMax
//   per pred label, summed over the representatives, gives counter 6, the same per truth label counter 7.
// The row stride is odd so that lanes reading word w of different rows mostly hit different banks.
constexpr int PC_WARPS_MAX = 4;
constexpr size_t PC_SMEM_MAX = 200 * 1024;   // two commits per CTA at n = 512 (76 KB each)

__host__ __device__ inline int pc_stride(int n) { return ((n + 31) >> 5) | 1; }
__host__ __device__ inline size_t pc_smem_words(int n) { return (size_t)n * (2 * pc_stride(n) + 4); }

__global__ void __launch_bounds__(32 * PC_WARPS_MAX) partition_counts_kernel(int B, int n, const int32_t* __restrict__ pred,
                                                                             const int32_t* __restrict__ truth,
                                                                             const int32_t* __restrict__ nh,
                                                                             long long* __restrict__ counts) {
    extern __shared__ __align__(16) uint32_t pc_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int b = blockIdx.x * (blockDim.x >> 5) + warp;
    if (b >= B) return;
    const int ST = pc_stride(n);
    uint32_t* Gp = pc_smem + (size_t)warp * pc_smem_words(n);
    uint32_t* Gt = Gp + (size_t)n * ST;
    int* mp = reinterpret_cast<int*>(Gt + (size_t)n * ST);      // largest cell per pred label
    int* mt = mp + n;                                           // largest cell per truth label
    int* ps = mt + n;                                           // the labels of the real hunks
    int* ts = ps + n;
    long long* out = counts + (size_t)b * 8;
    const int m = nh ? __ldg(nh + b) : n;
    bool bad = m < 0 || m > n;
    if (!bad) {
        for (int s = lane; s < m; s += 32) {
            const int p = __ldg(pred + (size_t)b * n + s), t = __ldg(truth + (size_t)b * n + s);
            bad |= (unsigned)p >= (unsigned)n || (unsigned)t >= (unsigned)n;
            ps[s] = p; ts[s] = t;
        }
    }
    if (__any_sync(0xffffffffu, bad)) {
        if (lane < 8) out[lane] = -1;
        return;
    }
    const int KW = (m + 31) >> 5;                               // bitmap words in use; lane owns hunks lane + 32 k, k < KW
    for (int s = lane; s < m; s += 32) {
        const int p = ps[s], t = ts[s];
        for (int w = 0; w < KW; ++w) { Gp[p * ST + w] = 0u; Gt[t * ST + w] = 0u; }
        mp[p] = 0; mt[t] = 0;
    }
    __syncwarp();
    for (int k = 0; k < KW && lane + 32 * k < m; ++k) {
        const int s = lane + 32 * k;
        atomicOr(&Gp[ps[s] * ST + k], 1u << lane);
        atomicOr(&Gt[ts[s] * ST + k], 1u << lane);
    }
    __syncwarp();
    unsigned both = 0u, jp = 0u, jt = 0u, gp = 0u, gt = 0u, repP = 0u, repT = 0u;
    const uint32_t below = (1u << lane) - 1u;
    for (int k = 0; k < KW && lane + 32 * k < m; ++k) {
        const int s = lane + 32 * k;
        const int p = ps[s], t = ts[s];
        const uint32_t* P = Gp + p * ST;
        const uint32_t* T = Gt + t * ST;
        int a = 0, c = 0, d = 0;
        bool lowP = true, lowT = true;                           // s is the lowest hunk of its pred / truth group
        for (int w = 0; w < KW; ++w) {
            const uint32_t x = P[w], y = T[w];
            a += __popc(x); d += __popc(y); c += __popc(x & y);
            const uint32_t lim = w < k ? 0xffffffffu : w == k ? below : 0u;
            lowP &= !(x & lim); lowT &= !(y & lim);
        }
        both += c - 1; jp += a - 1; jt += d - 1;
        gp += lowP; gt += lowT;
        repP |= (uint32_t)lowP << k; repT |= (uint32_t)lowT << k;
        atomicMax(&mp[p], c);
        atomicMax(&mt[t], c);
    }
    __syncwarp();
    unsigned op = 0u, ot = 0u;
    for (uint32_t r = repP; r; r &= r - 1u) op += mp[ps[lane + 32 * (__ffs(r) - 1)]];
    for (uint32_t r = repT; r; r &= r - 1u) ot += mt[ts[lane + 32 * (__ffs(r) - 1)]];
    both = __reduce_add_sync(0xffffffffu, both); jp = __reduce_add_sync(0xffffffffu, jp); jt = __reduce_add_sync(0xffffffffu, jt);
    gp = __reduce_add_sync(0xffffffffu, gp); gt = __reduce_add_sync(0xffffffffu, gt);
    op = __reduce_add_sync(0xffffffffu, op); ot = __reduce_add_sync(0xffffffffu, ot);
    const unsigned v = lane == 0 ? (unsigned)m : lane == 1 ? both / 2 : lane == 2 ? jp / 2 : lane == 3 ? jt / 2
                     : lane == 4 ? gp : lane == 5 ? gt : lane == 6 ? op : ot;
    if (lane < 8) out[lane] = (long long)v;
}

// ---------------------------------------------------------------------------------------------------------------
// Hunk clusters: average linkage (UPGMA) of the relation probabilities per commit, over the real hunks s < m = nh[b].  One CTA
// per commit (the workspace form: persistent CTAs, one slice of `work` each, walking the commits).
//   w(s,t) = fmaxf(p1(s,t), p1(t,s)); S(A,C) = sum of w over A x C, kept for every pair of live clusters (the full symmetric
//   m x m table, row r = the cluster whose representative -- smallest hunk -- is r) and updated by Lance-Williams,
//   S(A u B, C) = S(A,C) + S(B,C): one fp32 add per entry per merge, so the merge sequence fixes every rounding;
//   mean(A,C) = __fdiv_rn(S(A,C), (float)(|A| |C|)) (|A| |C| <= 256^2: exact in fp32).
//   Beside S, the table O holds the ordered bits of every live pair's mean (0: NaN, dead or diagonal), so a rescan of a row is
//   an integer max over it: no division, no sizes.
// A pair is ranked by the 64-bit key  [ordered bits of its mean | ~(lo << 16 | hi)]  (lo < hi its representatives): the larger
// key has the larger mean, and among equal means the smaller (lo, hi).  -0 is keyed as +0, NaN gets key 0 ("no pair"; every
// real pair's key is > 0), so a NaN mean never merges.  Row r keeps key[r] = the largest key over the live partners of r.
// Argmax over the row bests = argmax over all pairs: every pair (r, t) is a candidate of row r, so max_r key[r] >= its key,
// and every key[r] is the key of a live pair; the keys are distinct (they encode the pair), so the maximum is one pair.
// One merge of the best pair (a, c), a < c, keeping a:
//   A. block arg-max over key[]; stop when it is 0 (one cluster left, or only NaN) or its mean is not > threshold;
//   B. thread per row x: S(a,x) = S(x,a) = S(a,x) + S(c,x), O(a,x) = O(x,a) = the new mean's bits, O(x,c) = 0, and the new
//      key of (x, a); a row whose best partner was a or c goes on the rescan list, every other row takes max(key[x], key(x, a))
//      -- exact, since the pairs that left (x,a), (x,c) were not its best and the one that came is compared; row a's best is
//      the block max of the new keys (x, a);
//   C. warp per listed row: full rescan of its row of O.
// Barriers: A, B and C (C only when the list is not empty).  The sizes of a and c change only at the start of the next A (each
// row's owner thread writes its own row), so every thread reads the old sizes in B.
// The tables live in shared memory when they fit beside the row arrays (n <= 169), else in a slice of `work`; the same code
// reaches both through generic pointers.
// LINK (hdgnn_hunk_linkage): the same merges without a threshold -- A stops only when the arg-max key is 0 -- and thread 0
// records each one, (a, c) and the winning key's mean, after the A barrier; the trailing parameters are used only then, so the
// threshold form keeps its code.  Rows past the last merge are filled with (-1, -1) and NaN.
constexpr int HC_T_MAX = 512;
constexpr int HC_WARPS = HC_T_MAX / 32;
constexpr int HC_WORK_SLICES = 296;                        // CTAs of the workspace form: two per SM of a B200
constexpr size_t HC_SMEM_MAX = 227 * 1024;

__host__ __device__ inline int hc_stride(int n) { return n | 1; }                      // odd: column writes spread over banks
__host__ __device__ inline size_t hc_table_words(int n) { return (size_t)n * hc_stride(n); }
// key u64[n], two u64 slot arrays, size / lab / list int32[n], two list counters and two spare words; then S and O
__host__ __device__ inline size_t hc_rows_bytes(int n) { return (size_t)n * 8 + 2 * HC_WARPS * 8 + (size_t)n * 12 + 16; }
inline bool hc_table_in_smem(int n) { return hc_rows_bytes(n) + 2 * hc_table_words(n) * 4 <= HC_SMEM_MAX; }
inline int hc_threads(int n) { return n <= 128 ? 128 : n <= 256 ? 256 : HC_T_MAX; }

// ordered bits of a mean: larger mean <=> larger bits, -0 as +0, NaN -> 0 (every other value gives >= 0x007fffff)
__device__ __forceinline__ uint32_t hc_ord(float v) {
    uint32_t u = __float_as_uint(v);
    if ((u & 0x7fffffffu) > 0x7f800000u) return 0u;       // NaN
    if ((u << 1) == 0u) u = 0u;                             // -0 -> +0
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ unsigned long long hc_key(uint32_t o, int s, int t) {
    if (!o) return 0ull;
    const uint32_t lo = (uint32_t)min(s, t), hi = (uint32_t)max(s, t);
    return ((unsigned long long)o << 32) | (uint32_t)~((lo << 16) | hi);
}
__device__ __forceinline__ float hc_key_mean(unsigned long long k) {
    const uint32_t o = (uint32_t)(k >> 32);
    return __uint_as_float((o & 0x80000000u) ? (o ^ 0x80000000u) : ~o);
}
__device__ __forceinline__ int hc_key_lo(unsigned long long k) { return (int)((~(uint32_t)k) >> 16); }
__device__ __forceinline__ int hc_key_hi(unsigned long long k) { return (int)((~(uint32_t)k) & 0xffffu); }
__device__ __forceinline__ unsigned long long hc_max(unsigned long long x, unsigned long long y) { return x > y ? x : y; }
__device__ __forceinline__ unsigned long long hc_warp_max(unsigned long long k) {
    const uint32_t h = __reduce_max_sync(0xffffffffu, (uint32_t)(k >> 32));
    const uint32_t l = __reduce_max_sync(0xffffffffu, (uint32_t)(k >> 32) == h ? (uint32_t)k : 0u);
    return ((unsigned long long)h << 32) | l;
}

// The best key of row x over its live partners (one warp): the largest bits of its row of O, the smallest column among equals.
__device__ __forceinline__ unsigned long long hc_rescan(const uint32_t* O, int ST, int m, int x, int lane) {
    const uint32_t* Ox = O + (size_t)x * ST;
    uint32_t bo = 0u;
    int bt = 0xffff;
    for (int t = lane; t < m; t += 32) {
        const uint32_t o = Ox[t];
        if (o > bo) { bo = o; bt = t; }                     // t ascends: the first of equal bits is the smallest column
    }
    const uint32_t h = __reduce_max_sync(0xffffffffu, bo);
    const int t = (int)__reduce_min_sync(0xffffffffu, bo == h ? (uint32_t)bt : 0xffffu);
    return hc_key(h, x, t);
}

template <bool LINK>
__global__ void __launch_bounds__(HC_T_MAX) hunk_clusters_kernel(int B, int n, const float* __restrict__ probs,
                                                                 const int32_t* __restrict__ nh, float threshold,
                                                                 int32_t* __restrict__ groups, int32_t* __restrict__ ngroups,
                                                                 float* work, int32_t* __restrict__ rec_pairs,
                                                                 float* __restrict__ rec_heights, int32_t* __restrict__ rec_count) {
    extern __shared__ __align__(16) unsigned char hc_smem[];
    const int T = blockDim.x, NW = T >> 5, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    unsigned long long* key = reinterpret_cast<unsigned long long*>(hc_smem);
    unsigned long long* slot = key + n;                    // per-warp maxima of phase A
    unsigned long long* slotA = slot + HC_WARPS;           // per-warp maxima of the new keys (x, a) of phase B
    int* size = reinterpret_cast<int*>(slotA + HC_WARPS);  // cluster size of a representative, 0 = not a live cluster
    int* lab = size + n;                                   // representative of every hunk's cluster
    int* list = lab + n;                                   // rows to rescan
    int* cnt = list + n;                                   // list lengths of even / odd merges
    const int ST = hc_stride(n);
    const size_t TW = hc_table_words(n);
    float* S = work ? work + (size_t)blockIdx.x * 2 * TW : reinterpret_cast<float*>(cnt + 4);
    uint32_t* O = reinterpret_cast<uint32_t*>(S + TW);
    const size_t Ncr = (size_t)n * (n - 1);
    for (int b = blockIdx.x; b < B; b += gridDim.x) {
        const int m = nh ? __ldg(nh + b) : n;
        int32_t* g = groups + (size_t)b * n;
        int32_t* rp = rec_pairs + (size_t)b * (n - 1) * 2;
        float* rh = rec_heights + (size_t)b * (n - 1);
        if (m < 0 || m > n) {
            if constexpr (LINK) {
                for (int i = tid; i < n - 1; i += T) { rp[2 * i] = -1; rp[2 * i + 1] = -1; rh[i] = __int_as_float(0x7fffffff); }
                if (tid == 0) rec_count[b] = -1;
            } else {
                for (int s = tid; s < n; s += T) g[s] = -1;
                if (tid == 0 && ngroups) ngroups[b] = -1;
            }
            continue;
        }
        // channel 1 of the real block, row s of p1 (pairs s(n-1) .. s(n-1)+n-2) read along t; the padding pairs are never read
        const float* p1 = probs + (size_t)b * 2 * Ncr + Ncr;
        for (int s = warp; s < m; s += NW) {
            const float* row = p1 + (size_t)s * (n - 1);
            for (int t = lane; t < m; t += 32)
                if (t != s) S[(size_t)s * ST + t] = __ldg(row + t - (t > s));
        }
        for (int s = tid; s < n; s += T) {
            size[s] = s < m ? 1 : 0;
            lab[s] = s;
            if (s < m) O[(size_t)s * ST + s] = 0u;
        }
        if (tid < 2) cnt[tid] = 0;
        __syncthreads();
        for (int s = warp; s < m; s += NW)                  // w = fmaxf of both directions, each unordered pair by one lane
            for (int t = s + 1 + lane; t < m; t += 32) {
                const float v = fmaxf(S[(size_t)s * ST + t], S[(size_t)t * ST + s]);
                const uint32_t o = hc_ord(v);                   // mean of two singletons = w
                S[(size_t)s * ST + t] = v;
                S[(size_t)t * ST + s] = v;
                O[(size_t)s * ST + t] = o;
                O[(size_t)t * ST + s] = o;
            }
        __syncthreads();
        for (int x = warp; x < m; x += NW) {
            const unsigned long long k = hc_rescan(O, ST, m, x, lane);
            if (lane == 0) key[x] = k;
        }
        __syncthreads();
        int merges = 0, pa = -1, pc = -1, psz = 0;         // the last merge, whose sizes the owner threads write in A
        for (;;) {
            // A: block arg-max over the row bests (thread tid owns rows tid + k T throughout)
            if (pa >= 0) {
                if (pa % T == tid) size[pa] = psz;
                if (pc % T == tid) size[pc] = 0;
            }
            unsigned long long kb = 0ull;
            for (int x = tid; x < m; x += T) kb = hc_max(kb, key[x]);
            kb = hc_warp_max(kb);
            if (lane == 0) slot[warp] = kb;
            __syncthreads();
            kb = 0ull;
            for (int w = 0; w < NW; ++w) kb = hc_max(kb, slot[w]);
            if constexpr (LINK) {
                if (kb == 0ull) break;
            } else {
                if (kb == 0ull || !(hc_key_mean(kb) > threshold)) break;
            }
            // B: Lance-Williams update of row / column a, compare-and-update or rescan listing of every other row
            const int a = hc_key_lo(kb), c = hc_key_hi(kb);
            if constexpr (LINK) {
                if (tid == 0) { rp[2 * merges] = a; rp[2 * merges + 1] = c; rh[merges] = hc_key_mean(kb); }
            }
            const int sn = size[a] + size[c];
            int* L = cnt + (merges & 1);
            if (tid == 0) cnt[(merges & 1) ^ 1] = 0;       // the other counter was last read before this merge's A barrier
            unsigned long long kA = 0ull;
            for (int x = tid; x < m; x += T) {
                if (lab[x] == c) lab[x] = a;
                if (x == c) key[x] = 0ull;
                if (x == a) O[(size_t)a * ST + c] = 0u;
                const int sx = size[x];
                if (x == a || x == c || sx == 0) continue;
                const float v = S[(size_t)a * ST + x] + S[(size_t)c * ST + x];
                const uint32_t o = hc_ord(__fdiv_rn(v, (float)(sx * sn)));
                S[(size_t)a * ST + x] = v;
                S[(size_t)x * ST + a] = v;
                O[(size_t)a * ST + x] = o;
                O[(size_t)x * ST + a] = o;
                O[(size_t)x * ST + c] = 0u;
                const unsigned long long k = hc_key(o, x, a);
                kA = hc_max(kA, k);
                const unsigned long long kx = key[x];
                const int px = kx ? (hc_key_lo(kx) == x ? hc_key_hi(kx) : hc_key_lo(kx)) : -1;
                if (px == a || px == c) list[atomicAdd(L, 1)] = x;
                else if (k > kx) key[x] = k;
            }
            kA = hc_warp_max(kA);
            if (lane == 0) slotA[warp] = kA;
            __syncthreads();
            // C: row a from the new keys, full rescans of the listed rows
            if (a % T == tid) {
                kA = 0ull;
                for (int w = 0; w < NW; ++w) kA = hc_max(kA, slotA[w]);
                key[a] = kA;
            }
            const int nl = *L;
            if (nl) {
                for (int i = warp; i < nl; i += NW) {
                    const int x = list[i];
                    const unsigned long long k = hc_rescan(O, ST, m, x, lane);
                    if (lane == 0) key[x] = k;
                }
                __syncthreads();
            }
            pa = a; pc = c; psz = sn;
            ++merges;
        }
        if constexpr (LINK) {
            for (int i = merges + tid; i < n - 1; i += T) { rp[2 * i] = -1; rp[2 * i + 1] = -1; rh[i] = __int_as_float(0x7fffffff); }
            if (tid == 0) rec_count[b] = merges;
        } else {
            for (int s = tid; s < n; s += T) g[s] = s < m ? lab[s] : s;
            if (tid == 0 && ngroups) ngroups[b] = n - merges;
        }
        __syncthreads();                                    // before the next commit reuses the arrays and the table
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Cuts of recorded merge sequences (hdgnn_hunk_linkage) at K thresholds, or at one group count per commit.  One CTA per commit.
// The record is checked once and turned into parent[c] = a and step[c] = i (the row that absorbed c; LC_LIVE: none).  The
// checks -- every row 0 <= a < c < m, no c twice, no a absorbed at an earlier row -- make each hunk's chain of absorptions run
// to ever smaller hunks at ever later rows, so the first hunk of the chain not absorbed before the cut's merge count is the
// representative (smallest hunk) of the hunk's cluster after those merges, and the walk ends within m steps.  The record may
// come from a file: a commit that fails a check gets -1 throughout, and nothing is read past its nmerges rows.
// Then one warp per cut: the threshold cut's merge count is the longest prefix of heights > t (ballot scan), and every real
// hunk follows its chain while step < count.  Integer work: exact and deterministic.
constexpr int LC_K_MAX = 64;
constexpr int LC_WARPS = 8;
constexpr int LC_LIVE = 0x7fffffff;
struct LcThresholds { float t[LC_K_MAX]; };                // by value, so a captured graph keeps the caller's thresholds

__global__ void __launch_bounds__(32 * LC_WARPS) linkage_cut_kernel(int B, int n, const int32_t* __restrict__ pairs,
                                                                    const float* __restrict__ heights,
                                                                    const int32_t* __restrict__ count,
                                                                    const int32_t* __restrict__ nh, int K, LcThresholds thr,
                                                                    const int32_t* __restrict__ target,
                                                                    int32_t* __restrict__ groups, int32_t* __restrict__ ngroups) {
    __shared__ int parent[HDGNN_MAX_N], step[HDGNN_MAX_N];
    const int b = blockIdx.x, T = blockDim.x, tid = threadIdx.x, lane = tid & 31;
    const int m = nh ? __ldg(nh + b) : n;
    const int nm = __ldg(count + b);
    const int32_t* rp = pairs + (size_t)b * (n - 1) * 2;
    const float* rh = heights + (size_t)b * (n - 1);
    int bad = m < 0 || m > n || nm < 0 || nm > max(m - 1, 0);
    if (!bad)
        for (int s = tid; s < m; s += T) step[s] = LC_LIVE;
    __syncthreads();
    if (!bad)
        for (int i = tid; i < nm; i += T) {
            const int a = __ldg(rp + 2 * i), c = __ldg(rp + 2 * i + 1);
            if (!(0 <= a && a < c && c < m)) bad = 1;
            else if (atomicCAS(&step[c], LC_LIVE, i) != LC_LIVE) bad = 1;      // c absorbed twice
            else parent[c] = a;
        }
    bad = __syncthreads_or(bad);
    if (!bad)
        for (int i = tid; i < nm; i += T)
            if (step[__ldg(rp + 2 * i)] < i) bad = 1;                          // a absorbed before row i
    bad = __syncthreads_or(bad);
    for (int k = tid >> 5; k < K; k += T >> 5) {
        int32_t* g = groups + ((size_t)k * B + b) * n;
        int c = -1;
        if (!bad) {
            if (target) {
                c = min(nm, max(0, m - max(__ldg(target + b), 1)));
            } else {
                const float t = thr.t[k];
                c = nm;
                for (int base = 0; base < nm; base += 32) {
                    const int i = base + lane;
                    const uint32_t stop = __ballot_sync(0xffffffffu, i < nm && !(__ldg(rh + i) > t));
                    if (stop) { c = base + __ffs(stop) - 1; break; }
                }
            }
        }
        for (int s = lane; s < n; s += 32) {
            int x = s;
            if (bad) x = -1;
            else if (s < m)
                while (step[x] < c) x = parent[x];
            g[s] = x;
        }
        if (lane == 0 && ngroups) ngroups[(size_t)k * B + b] = bad ? -1 : n - c;
    }
}

}  // namespace hdgnn

using namespace hdgnn;

extern "C" int hdgnn_compact_from_raw(int N, int n, const void* raw, int raw_is_f64, uint8_t* grid, int pitch, float* diag,
                                      int32_t* err, void* stream) {
    const Call c{"hdgnn_compact_from_raw"};
    if (int rc = c.sizes("N", N, "n", n)) return rc;
    if (pitch < n || (pitch & 15) || pitch > 512 + 16) return c.invalid("pitch must be a multiple of 16 in [n, 528]");
    const long long rows = (long long)N * n;
    if (rows > 0x7fffffffLL) return c.invalid("N * n above 2^31 - 1");
    if (int rc = c.pointers({{"raw", raw, raw_is_f64 ? 8u : 4u}, {"grid", grid, 1}, {"diag", diag, 4, false}, {"err", err, 4, false}})) return rc;
    Device d; if (int rc = c.device(&d)) return rc;
    const int wpb = 8;
    long long want = (rows + wpb - 1) / wpb;
    const int grid_x = (int)(want < (long long)d.sms * 8 ? want : (long long)d.sms * 8);      // 8 CTAs of 8 warps per SM, grid-stride
    cudaStream_t st = (cudaStream_t)stream;
    const int kmax = (pitch + 31) / 32;
#define LAUNCH(T, K) compact_from_raw_kernel<T, K><<<grid_x, 256, 0, st>>>((const T*)raw, (int)rows, n, grid, pitch, diag, err)
    if (raw_is_f64) {
        if (kmax <= 4) LAUNCH(double, 4); else if (kmax <= 8) LAUNCH(double, 8); else if (kmax <= 12) LAUNCH(double, 12); else LAUNCH(double, 17);
    } else {
        if (kmax <= 4) LAUNCH(float, 4); else if (kmax <= 8) LAUNCH(float, 8); else if (kmax <= 12) LAUNCH(float, 12); else LAUNCH(float, 17);
    }
#undef LAUNCH
    return c.launched();
}

extern "C" int hdgnn_eval_counts(int B, int Nc, const float* probs, const uint8_t* Y, int y_pitch, int64_t* counts, int64_t* auc,
                                 int auc_first, void* stream) {
    const Call c{"hdgnn_eval_counts"};
    if (int rc = c.sizes("B", B, "Nc", Nc)) return rc;
    if (y_pitch < Nc) return c.invalid("y_pitch < Nc");
    if (int rc = c.pointers({{"probs", probs, 4}, {"Y", Y, 1}, {"counts", counts, 8}, {"auc", auc, 8, false}})) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = c.cuda(cudaMemsetAsync(counts, 0, (size_t)B * 8 * sizeof(int64_t), st))) return rc;
    if (int rc = c.cuda(auc ? cudaMemsetAsync(auc, 0, (size_t)B * 2 * sizeof(int64_t), st) : cudaSuccess)) return rc;
    const int Ncr = Nc * (Nc - 1);
    dim3 g((Ncr + EV_CHUNK - 1) / EV_CHUNK, B);
    eval_counts_kernel<<<g, EV_T, 0, st>>>(Nc, probs, Y, y_pitch, (unsigned long long*)counts, (unsigned long long*)auc,
                                          auc_first < 0 ? 0 : auc_first);
    return c.launched();
}

extern "C" int hdgnn_hunk_groups(int B, int n, const uint32_t* bits, int32_t* groups, int32_t* ngroups, void* stream) {
    const Call c{"hdgnn_hunk_groups"};
    if (int rc = c.sizes("B", B, "n", n)) return rc;
    if (int rc = c.pointers({{"bits", bits, 16}, {"groups", groups, 4}, {"ngroups", ngroups, 4, false}})) return rc;
    Device d; if (int rc = c.device(&d)) return rc;
    const int WP = bit_words(n);
    const size_t per = (size_t)n * WP * 4;
    const int cpc = commits_per_cta(B, d.sms, per, HG_SMEM_MAX, HG_WARPS_MAX);
    hunk_groups_kernel<<<(B + cpc - 1) / cpc, 32 * cpc, cpc * per, (cudaStream_t)stream>>>(B, n, WP, bits, groups, ngroups);
    return c.launched();
}

extern "C" int hdgnn_partition_counts(int B, int n, const int32_t* pred, const int32_t* truth, const int32_t* nh, int64_t* counts,
                                      void* stream) {
    const Call c{"hdgnn_partition_counts"};
    if (int rc = c.sizes("B", B, "n", n)) return rc;
    if (int rc = c.pointers({{"pred", pred, 4}, {"truth", truth, 4}, {"nh", nh, 4, false}, {"counts", counts, 8}})) return rc;
    Device d; if (int rc = c.device(&d)) return rc;
    const size_t per = pc_smem_words(n) * 4;
    const int cpc = commits_per_cta(B, d.sms, per, PC_SMEM_MAX, PC_WARPS_MAX);
    const size_t smem = cpc * per;     // above the 48 KB default: one commit from n = 410 on, or several smaller ones
    if (int rc = smem > 48 * 1024 ? c.raise_smem(partition_counts_kernel, d) : HDGNN_OK) return rc;
    partition_counts_kernel<<<(B + cpc - 1) / cpc, 32 * cpc, smem, (cudaStream_t)stream>>>(B, n, pred, truth, nh,
                                                                                           (long long*)counts);
    return c.launched();
}

// One CTA per commit; the workspace form walks the commits with one slice (S and O) per CTA.  Called once the entry point has
// checked its arguments.
template <bool LINK>
static int hc_launch(const Call& c, int B, int n, const float* probs, const int32_t* nh, float threshold, int32_t* groups,
                     int32_t* ngroups, void* work, int32_t* merges, float* heights, int32_t* nmerges, void* stream) {
    Device d; if (int rc = c.device(&d)) return rc;
    const bool in_smem = hc_table_in_smem(n);
    const size_t smem = hc_rows_bytes(n) + (in_smem ? 2 * hc_table_words(n) * 4 : 0);
    if (int rc = smem > 48 * 1024 ? c.raise_smem(hunk_clusters_kernel<LINK>, d) : HDGNN_OK) return rc;
    const int grid = in_smem ? B : (B < HC_WORK_SLICES ? B : HC_WORK_SLICES);
    hunk_clusters_kernel<LINK><<<grid, hc_threads(n), smem, (cudaStream_t)stream>>>(B, n, probs, nh, threshold, groups, ngroups,
                                                                                   in_smem ? nullptr : (float*)work, merges,
                                                                                   heights, nmerges);
    return c.launched();
}

extern "C" size_t hdgnn_hunk_clusters_work(int B, int n) {
    if (B < 1 || n < 2 || n > HDGNN_MAX_N || hc_table_in_smem(n)) return 0;
    return (size_t)(B < HC_WORK_SLICES ? B : HC_WORK_SLICES) * 2 * hc_table_words(n) * sizeof(float);
}

extern "C" int hdgnn_hunk_clusters(int B, int n, const float* probs, const int32_t* nh, float threshold, int32_t* groups,
                                   int32_t* ngroups, void* work, void* stream) {
    const Call c{"hdgnn_hunk_clusters"};
    if (int rc = c.sizes("B", B, "n", n)) return rc;
    if (threshold != threshold) return c.invalid("threshold is NaN");
    const bool in_smem = hc_table_in_smem(n);
    if (int rc = c.pointers({{"probs", probs, 4}, {"nh", nh, 4, false}, {"groups", groups, 4}, {"ngroups", ngroups, 4, false},
                             {"work", work, 4, !in_smem}}))
        return rc;
    return hc_launch<false>(c, B, n, probs, nh, threshold, groups, ngroups, work, nullptr, nullptr, nullptr, stream);
}

extern "C" int hdgnn_hunk_linkage(int B, int n, const float* probs, const int32_t* nh, int32_t* merges, float* heights,
                                  int32_t* nmerges, void* work, void* stream) {
    const Call c{"hdgnn_hunk_linkage"};
    if (int rc = c.sizes("B", B, "n", n)) return rc;
    if (int rc = c.pointers({{"probs", probs, 4}, {"nh", nh, 4, false}, {"merges", merges, 4}, {"heights", heights, 4},
                             {"nmerges", nmerges, 4}, {"work", work, 4, !hc_table_in_smem(n)}}))
        return rc;
    return hc_launch<true>(c, B, n, probs, nh, 0.f, nullptr, nullptr, work, merges, heights, nmerges, stream);
}

extern "C" int hdgnn_linkage_cut(int B, int n, const int32_t* merges, const float* heights, const int32_t* nmerges,
                                 const int32_t* nh, int K, const float* thresholds_host, const int32_t* target, int32_t* groups,
                                 int32_t* ngroups, void* stream) {
    const Call c{"hdgnn_linkage_cut"};
    if (int rc = c.sizes("B", B, "n", n)) return rc;
    if (K < 1 || K > LC_K_MAX) return c.invalid("K outside [1, 64]");
    if (int rc = c.pointers({{"merges", merges, 4}, {"heights", heights, 4}, {"nmerges", nmerges, 4}, {"nh", nh, 4, false},
                             {"thresholds_host", thresholds_host, 4, false}, {"target", target, 4, false},
                             {"groups", groups, 4}, {"ngroups", ngroups, 4, false}}))
        return rc;
    if (!thresholds_host == !target) return c.invalid("thresholds_host and target: exactly one must be given");
    if (target && K != 1) return c.invalid("K must be 1 with target");
    LcThresholds thr{};
    for (int k = 0; thresholds_host && k < K; ++k) {
        if (thresholds_host[k] != thresholds_host[k]) return c.invalid("thresholds_host[" + std::to_string(k) + "] is NaN");
        thr.t[k] = thresholds_host[k];
    }
    linkage_cut_kernel<<<B, 32 * std::min(K, LC_WARPS), 0, (cudaStream_t)stream>>>(B, n, merges, heights, nmerges, nh, K, thr,
                                                                                    target, groups, ngroups);
    return c.launched();
}

// ---------------------------------------------------------------------------------------------------------------
// Measured fp32 CUDA-core peaks for bench.py's roofline denominators (not part of the hot path): a register-resident chain
// of independent fused multiply-adds, scalar (FFMA) or packed (fma.rn.f32x2, SASS FFMA2 -- the form the pair sweeps use).
namespace hdgnn {
template <bool PACKED>
__global__ void __launch_bounds__(256) fma_peak_kernel(int iters, float seed, float* sink) {
    constexpr int NA = 8;
    if (PACKED) {
        unsigned long long acc[NA], m, c;
        asm("mov.b64 %0, {%1, %1};" : "=l"(m) : "f"(1.0f + seed * 1e-7f));
        asm("mov.b64 %0, {%1, %1};" : "=l"(c) : "f"(seed * 1e-3f));
#pragma unroll
        for (int i = 0; i < NA; ++i) asm("mov.b64 %0, {%1, %2};" : "=l"(acc[i]) : "f"((float)(threadIdx.x + i)), "f"((float)i));
        for (int it = 0; it < iters; ++it)
#pragma unroll
            for (int i = 0; i < NA; ++i) asm volatile("fma.rn.f32x2 %0, %0, %1, %2;" : "+l"(acc[i]) : "l"(m), "l"(c));
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < NA; ++i) { float lo, hi; asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(acc[i])); s += lo + hi; }
        if (s == 12345.678f) sink[0] = s;
    } else {
        float acc[NA];
        const float m = 1.0f + seed * 1e-7f, c = seed * 1e-3f;
#pragma unroll
        for (int i = 0; i < NA; ++i) acc[i] = (float)(threadIdx.x + i);
        for (int it = 0; it < iters; ++it)
#pragma unroll
            for (int i = 0; i < NA; ++i) asm volatile("fma.rn.f32 %0, %0, %1, %2;" : "+f"(acc[i]) : "f"(m), "f"(c));
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < NA; ++i) s += acc[i];
        if (s == 12345.678f) sink[0] = s;
    }
}
}  // namespace hdgnn

extern "C" int hdgnn_measure_fp32_peak(int packed, float* tflops_out) {
    const Call c{"hdgnn_measure_fp32_peak"};
    if (int rc = c.pointers({{"tflops_out", tflops_out, 4}})) return rc;
    Device d; if (int rc = c.device(&d)) return rc;
    float* sink = nullptr;
    if (cudaMalloc(&sink, 16) != cudaSuccess) return HDGNN_E_NOMEM;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    const int iters = 20000, grid = d.sms * 8, block = 256;
    float best = 0.f;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(e0);
        if (packed) hdgnn::fma_peak_kernel<true><<<grid, block>>>(iters, 1.f, sink);
        else hdgnn::fma_peak_kernel<false><<<grid, block>>>(iters, 1.f, sink);
        cudaEventRecord(e1);
        if (cudaEventSynchronize(e1) != cudaSuccess) { cudaFree(sink); return HDGNN_E_CUDA; }
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        const double flops = (double)grid * block * iters * 8.0 * 2.0 * (packed ? 2.0 : 1.0);
        const float tf = (float)(flops / (ms * 1e-3) / 1e12);
        if (rep > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(sink);
    *tflops_out = best;
    return HDGNN_OK;
}
