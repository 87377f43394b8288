// k_conv_bwd: backward of the legacy operator of model.py (SURVEY K15, row a16).
//
// The reference trains THROUGH chebyshev_polynomials / map_conv (model.py:150-155, 405-417), but the edge tensor enters
// through tf.argmax (model.py:337), so the adjacency is a hard {0,1} grid that carries NO gradient: the backward runs
// w.r.t. the node features and the Chebyshev coefficients only.
//
//  * hdgnn_normalize_propagate_backward: out = act(A_hat (H W) + b).  With dPre = dOut * act'(out),
//        dZ = A_hat^T dPre,   dH = dZ W^T,   dW = sum_b H_b^T dZ_b,   db = sum_{b,n} dPre.
//    A_hat^T = D^-1/2 A D^-1/2 is the SAME normalise+propagate operator with the transposition flag flipped (the degrees
//    are those of A either way, model.py:362), so dZ comes from the forward's own tcgen05 kernel (k_conv.cu); the small
//    per-commit products and the fixed-order reduction over the batch are the two kernels below.
//  * hdgnn_map_conv_backward: loss = mean_b s_b^2, s_b = x^T (t0 I + t1 L~) x, t = softmax(theta), L~ = (2/lam)(I - A_hat) - I:
//        ds/dx = 2 t0 x + t1 ((4/lam - 2) x - (2/lam)(A_hat + A_hat^T) x),
//        dloss/dx_b = (2 s_b / B) ds/dx,   dloss/dt0 = sum_b (2 s_b / B) x^T x,   dloss/dt1 = sum_b (2 s_b / B) x^T L~ x,
//    then through the softmax.  One CTA per commit on the staged tile (byte grid, or label bitmap with HDGNN_P_LABEL_BITS):
//    degrees, then the row and column mat-vecs in two passes.
// All sums run in a fixed order (no float atomics).
#include "../../include/hdgnn.h"
#include "bits.cuh"
#include "host.cuh"

namespace hdgnn {

constexpr int CB_T = 256;
constexpr int CB_MAXD = 32;

__global__ void relu_mask_kernel(const float* __restrict__ dOut, const float* __restrict__ out, float* __restrict__ dPre, size_t n) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        dPre[i] = out[i] > 0.f ? dOut[i] : 0.f;
}

// per commit: dH_b = dZ_b W^T, partial[b] = { H_b^T dZ_b (d_in x d_out), sum_n dPre_b (d_out) }
__global__ void __launch_bounds__(CB_T) prop_bwd_commit_kernel(int N, int d_in, int d_out, const float* __restrict__ H, const float* __restrict__ W,
                                                               const float* __restrict__ dZ, const float* __restrict__ dPre,
                                                               float* __restrict__ dH, float* __restrict__ partial) {
    extern __shared__ float sm[];
    float* Hs = sm;                         // [N][d_in]
    float* Zs = Hs + (size_t)N * d_in;      // [N][d_out]
    float* Ws = Zs + (size_t)N * d_out;     // [d_in][d_out]
    const int b = blockIdx.x, tid = threadIdx.x;
    const float* Hb = H + (size_t)b * N * d_in;
    const float* Zb = dZ + (size_t)b * N * d_out;
    for (int i = tid; i < N * d_in; i += CB_T) Hs[i] = Hb[i];
    for (int i = tid; i < N * d_out; i += CB_T) Zs[i] = Zb[i];
    for (int i = tid; i < d_in * d_out; i += CB_T) Ws[i] = W ? W[i] : ((i / d_out) == (i % d_out) ? 1.f : 0.f);
    __syncthreads();
    if (dH) {
        float* dHb = dH + (size_t)b * N * d_in;
        for (int e = tid; e < N * d_in; e += CB_T) {
            const int n = e / d_in, i = e - n * d_in;
            float acc = 0.f;
            for (int o = 0; o < d_out; ++o) acc = fmaf(Zs[n * d_out + o], Ws[i * d_out + o], acc);
            dHb[e] = acc;
        }
    }
    float* pb = partial + (size_t)b * (d_in * d_out + d_out);
    for (int e = tid; e < d_in * d_out; e += CB_T) {
        const int i = e / d_out, o = e - i * d_out;
        float acc = 0.f;
        for (int n = 0; n < N; ++n) acc = fmaf(Hs[n * d_in + i], Zs[n * d_out + o], acc);
        pb[e] = acc;
    }
    // bias partial: column sums of dPre, coalesced (thread -> column t % d_out, row slot t / d_out), slots combined in order
    __syncthreads();
    const float* Pb = dPre + (size_t)b * N * d_out;
    const int nslot = CB_T / d_out;
    float* red = Hs;                                        // Hs is dead
    if (tid < nslot * d_out) {
        const int o = tid % d_out, sl = tid / d_out;
        float acc = 0.f;
        for (int n = sl; n < N; n += nslot) acc += Pb[(size_t)n * d_out + o];
        red[sl * d_out + o] = acc;
    }
    __syncthreads();
    for (int o = tid; o < d_out; o += CB_T) {
        float acc = 0.f;
        for (int sl = 0; sl < nslot; ++sl) acc += red[sl * d_out + o];
        pb[d_in * d_out + o] = acc;
    }
}

// stage 1: part2[c][e] = sum over the c-th of BS_CH batch chunks of partial[b][e] (batch order); stage 2 adds the chunks in order
constexpr int BS_CH = 32;
__global__ void batch_sum1_kernel(const float* __restrict__ partial, int B, int stride, float* __restrict__ part2) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x, c = blockIdx.y;
    if (e >= stride) return;
    const int per = (B + BS_CH - 1) / BS_CH, b0 = c * per, b1 = min(b0 + per, B);
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int b = b0;
    for (; b + 3 < b1; b += 4) {                            // four loads in flight, fixed combination order
        a0 += partial[(size_t)b * stride + e]; a1 += partial[(size_t)(b + 1) * stride + e];
        a2 += partial[(size_t)(b + 2) * stride + e]; a3 += partial[(size_t)(b + 3) * stride + e];
    }
    for (; b < b1; ++b) a0 += partial[(size_t)b * stride + e];
    part2[(size_t)c * stride + e] = (a0 + a1) + (a2 + a3);
}
__global__ void batch_sum2_kernel(const float* __restrict__ part2, int stride, int lo, int n, float* __restrict__ out) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    float acc = 0.f;
    for (int c = 0; c < BS_CH; ++c) acc += part2[(size_t)c * stride + lo + e];
    out[e] = acc;
}

struct McbArgs {
    int B, N, pitch, flags;
    float eps, lam_max, gscale;
    const uint8_t* adj; const float* x; const float* theta;
    float* dx; float* part;      // part (B,2): (2 s_b g / B) x^T x, (2 s_b g / B) x^T L~ x
};

template <bool BITS>
__global__ void __launch_bounds__(CB_T) map_conv_bwd_kernel(const McbArgs a) {
    extern __shared__ __align__(16) unsigned char smraw[];
    const int N = a.N, pitch = a.pitch, b = blockIdx.x, tid = threadIdx.x;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smraw);
    uint8_t* tile = smraw + 16;
    float* u = reinterpret_cast<float*>(tile + round_up(N * pitch, 16));   // dinv * x
    float* dinv = u + N;
    float* xs = dinv + N;
    float* rr = xs + N;          // (A u)_i
    float* pp = rr + N;          // (A^T u)_j
    float* red = pp + N;         // 32
    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
        const uint32_t bytes = (uint32_t)N * pitch;
        mbar_arrive_expect_tx(bar, bytes);
        bulk_g2s(tile, a.adj + (size_t)b * N * pitch, bytes, bar);
    }
    for (int i = tid; i < N; i += CB_T) xs[i] = a.x[(size_t)b * N + i];
    __syncthreads();
    mbar_wait(bar, 0);
    const bool self = (a.flags & HDGNN_P_SELF_LOOP) != 0, notr = (a.flags & HDGNN_P_NO_TRANSPOSE) != 0;
    const int NW = pitch >> 2;
    // a bitmap row: bit (j & 31) of word j >> 5; only columns < N are read below, and the diagonal is skipped
    const uint32_t* tbits = reinterpret_cast<const uint32_t*>(tile);
    for (int i = tid; i < N; i += CB_T) {                     // degrees (diagonal ignored)
        const uint32_t* row = reinterpret_cast<const uint32_t*>(tile + (size_t)i * pitch);
        int deg = 0;
        if constexpr (BITS) {
            for (int w = 0; w < (N + 31) / 32; ++w) {
                uint32_t v = row[w];
                if (32 * w + 32 > N) v &= 0xffffffffu >> (32 * w + 32 - N);
                if ((i >> 5) == w) v &= ~(1u << (i & 31));
                deg += __popc(v);
            }
        } else {
            for (int w = 0; w < NW; ++w) {
                uint32_t v = row[w];
                if ((i >> 2) == w) v &= ~(0xffu << (8 * (i & 3)));
                deg += ((v & 0xffu) != 0) + ((v & 0xff00u) != 0) + ((v & 0xff0000u) != 0) + ((v & 0xff000000u) != 0);
            }
        }
        const float di = rsqrtf((float)deg + (self ? 1.f : 0.f) + a.eps);
        dinv[i] = di; u[i] = di * xs[i];
    }
    __syncthreads();
    for (int i = tid; i < N; i += CB_T) {                     // rr_i = sum_j A_ij u_j
        const uint8_t* row = tile + (size_t)i * pitch;
        float acc = self ? u[i] : 0.f;
        if constexpr (BITS) {
            for (int j0 = 0; j0 < N; j0 += 32) {              // one word load per 32 columns, the same additions as below
                const uint32_t v = tbits[(size_t)i * NW + (j0 >> 5)];
                const int j1 = j0 + 32 < N ? j0 + 32 : N;
                for (int j = j0; j < j1; ++j) acc += (((v >> (j & 31)) & 1u) && j != i) ? u[j] : 0.f;
            }
        } else {
            for (int j = 0; j < N; ++j) acc += (row[j] != 0 && j != i) ? u[j] : 0.f;
        }
        rr[i] = acc;
    }
    for (int j = tid; j < N; j += CB_T) {                     // pp_j = sum_i A_ij u_i
        float acc = self ? u[j] : 0.f;
        if constexpr (BITS) {
            for (int i = 0; i < N; ++i) acc += (((tbits[(size_t)i * NW + (j >> 5)] >> (j & 31)) & 1u) && i != j) ? u[i] : 0.f;
        } else {
            for (int i = 0; i < N; ++i) acc += (tile[(size_t)i * pitch + j] != 0 && i != j) ? u[i] : 0.f;
        }
        pp[j] = acc;
    }
    __syncthreads();
    // A_hat x = dinv * (A^T u) (reference form) or dinv * (A u); the other one is A_hat^T x
    float pa = 0.f, pe = 0.f;
    for (int i = tid; i < N; i += CB_T) {
        const float ax = dinv[i] * (notr ? rr[i] : pp[i]);
        pa = fmaf(xs[i], xs[i], pa); pe = fmaf(xs[i], ax, pe);
    }
    const float aa = block_sum(pa, red);
    const float ee = block_sum(pe, red);
    const float th0 = a.theta[0], th1 = a.theta[1], mx = fmaxf(th0, th1);
    const float e0 = expf(th0 - mx), e1 = expf(th1 - mx), t0 = e0 / (e0 + e1), t1 = e1 / (e0 + e1);
    const float il = 2.f / a.lam_max;
    const float cc = (il - 1.f) * aa - il * ee;               // x^T L~ x
    const float s = t0 * aa + t1 * cc;
    const float gs = 2.f * s * a.gscale / (float)a.B;
    if (a.dx)
        for (int i = tid; i < N; i += CB_T) {
            const float sym = dinv[i] * (rr[i] + pp[i]);      // ((A_hat + A_hat^T) x)_i
            a.dx[(size_t)b * N + i] = gs * (2.f * t0 * xs[i] + t1 * ((2.f * il - 2.f) * xs[i] - il * sym));
        }
    if (tid == 0 && a.part) { a.part[2 * b] = gs * aa; a.part[2 * b + 1] = gs * cc; }
}

__global__ void theta_grad_kernel(const float* __restrict__ part, int B, const float* __restrict__ theta, float* __restrict__ dtheta) {
    __shared__ float scratch[32];
    float p0 = 0.f, p1 = 0.f;
    for (int b = threadIdx.x; b < B; b += blockDim.x) { p0 += part[2 * b]; p1 += part[2 * b + 1]; }
    const float d0 = block_sum(p0, scratch);
    const float d1 = block_sum(p1, scratch);
    if (threadIdx.x == 0) {
        const float mx = fmaxf(theta[0], theta[1]), e0 = expf(theta[0] - mx), e1 = expf(theta[1] - mx);
        const float t0 = e0 / (e0 + e1), t1 = e1 / (e0 + e1), dot = t0 * d0 + t1 * d1;
        dtheta[0] = t0 * (d0 - dot); dtheta[1] = t1 * (d1 - dot);
    }
}

}  // namespace hdgnn

using namespace hdgnn;

extern "C" size_t hdgnn_propagate_backward_work(int B, int N, int d_in, int d_out) {
    if (B < 1 || N < 1 || d_in < 1 || d_out < 1) return 0;
    return (size_t)2 * B * N * d_out + (size_t)(B + BS_CH) * (d_in * d_out + d_out);
}

extern "C" int hdgnn_normalize_propagate_backward(int B, int N, const uint8_t* adj, int adj_pitch, const float* H, int d_in,
                                                  const float* W, int d_out, float eps, int flags, const float* out, const float* dOut,
                                                  float* dH, float* dW, float* dbias, float* work, void* stream) {
    const Call c{"hdgnn_normalize_propagate_backward"};
    if (int rc = legacy_check(c, B, N, adj_pitch, adj, flags)) return rc;
    if (d_in < 1 || d_in > CB_MAXD || d_out < 1 || d_out > CB_MAXD || (!W && d_in != d_out))
        return c.invalid("d_in or d_out outside [1, 32], or W null with d_in != d_out");
    if (int rc = c.pointers({{"H", H, 4}, {"W", W, 4, false}, {"out", out, 4, (flags & HDGNN_P_RELU) != 0}, {"dOut", dOut, 4},
                             {"dH", dH, 4, false}, {"dW", dW, 4, false}, {"dbias", dbias, 4, false}, {"work", work, 4}}))
        return rc;
    size_t smem = ((size_t)N * (d_in + d_out) + (size_t)d_in * d_out) * sizeof(float);
    if (smem < CB_T * sizeof(float)) smem = CB_T * sizeof(float);      // the bias slots reuse the head of the tile
    Device d; if (int rc = c.device(&d)) return rc;
    if (smem > (size_t)d.optin) return c.fail(HDGNN_E_UNSUPPORTED, "the per-commit tile does not fit one SM's shared memory");
    if (int rc = c.raise_smem(prop_bwd_commit_kernel, d)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t nel = (size_t)B * N * d_out;
    float* dPre = work; float* dZ = work + nel; float* partial = work + 2 * nel;
    const float* dpre_src = dOut;
    if (flags & HDGNN_P_RELU) {
        relu_mask_kernel<<<(int)((nel + 255) / 256 > 1184 ? 1184 : (nel + 255) / 256), 256, 0, st>>>(dOut, out, dPre, nel);
        dpre_src = dPre;
    }
    // dZ = A_hat^T dPre: the forward operator with the transposition flipped, no weights, no bias, no activation
    const int keep = flags & (HDGNN_P_SELF_LOOP | HDGNN_P_NO_TENSOR | HDGNN_P_TENSOR_V1 | HDGNN_P_LABEL_BITS);
    const int flipped = keep | ((flags & HDGNN_P_NO_TRANSPOSE) ? 0 : HDGNN_P_NO_TRANSPOSE);
    int rc = hdgnn_normalize_propagate(B, N, adj, adj_pitch, dpre_src, d_out, nullptr, nullptr, d_out, eps, flipped, dZ, nullptr, stream);
    if (rc) return rc;
    prop_bwd_commit_kernel<<<B, CB_T, smem, st>>>(N, d_in, d_out, H, W, dZ, dpre_src, dH, partial);
    const int stride = d_in * d_out + d_out;
    float* part2 = partial + (size_t)B * stride;
    if ((dW && W) || dbias) batch_sum1_kernel<<<dim3((stride + 127) / 128, BS_CH), 128, 0, st>>>(partial, B, stride, part2);
    if (dW && W) batch_sum2_kernel<<<(d_in * d_out + 127) / 128, 128, 0, st>>>(part2, stride, 0, d_in * d_out, dW);
    if (dbias) batch_sum2_kernel<<<1, 128, 0, st>>>(part2, stride, d_in * d_out, d_out, dbias);
    return c.launched();
}

extern "C" int hdgnn_map_conv_backward(int B, int N, const uint8_t* adj, int adj_pitch, const float* x, const float* theta, float lam_max,
                                       float eps, int flags, float gscale, float* dx, float* dtheta, float* work, void* stream) {
    const Call c{"hdgnn_map_conv_backward"};
    if (int rc = legacy_check(c, B, N, adj_pitch, adj, flags)) return rc;
    if (!(lam_max > 0.f)) return c.invalid("lam_max must be > 0");
    if (int rc = c.pointers({{"x", x, 4}, {"theta", theta, 4}, {"dx", dx, 4, false}, {"dtheta", dtheta, 4, false},
                             {"work", work, 4, dtheta != nullptr}}))
        return rc;
    const size_t smem = 16 + (size_t)round_up(N * adj_pitch, 16) + (size_t)(5 * N + 32) * sizeof(float);
    Device d; if (int rc = c.device(&d)) return rc;
    if (smem > (size_t)d.optin) return c.fail(HDGNN_E_UNSUPPORTED, "the per-commit tile does not fit one SM's shared memory");
    const auto k = (flags & HDGNN_P_LABEL_BITS) ? map_conv_bwd_kernel<true> : map_conv_bwd_kernel<false>;
    if (int rc = c.raise_smem(k, d)) return rc;
    McbArgs a{};
    a.B = B; a.N = N; a.pitch = adj_pitch; a.flags = flags; a.eps = eps; a.lam_max = lam_max; a.gscale = gscale;
    a.adj = adj; a.x = x; a.theta = theta; a.dx = dx; a.part = dtheta ? work : nullptr;
    cudaStream_t st = (cudaStream_t)stream;
    k<<<B, CB_T, smem, st>>>(a);
    if (dtheta) theta_grad_kernel<<<1, 256, 0, st>>>(work, B, theta, dtheta);
    return c.launched();
}
