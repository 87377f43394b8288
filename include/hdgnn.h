/*
 * hdgnn.h -- C ABI of the B200-native HD-GNN hot path (libhdgnn.so).
 *
 * The reference (fanmengdan/HD-GNN) has no FFI of its own: the seam this library sits
 * behind is the body of one `sess.run([... trainer], feed_dict=...)` call
 * (model_2.py:369-383 for training, model_2.py:486-502 for inference), i.e. the forward
 * graph built in model_2.py:86-118 (and its model_1/3/4 variants), its autodiff backward
 * and the AdamOptimizer update of model_2.py:336-338.  Each entry point below names the
 * reference lines it replaces.  INTEGRATION.md shows the ctypes binding a maintainer of the
 * reference would add.
 *
 * Conventions
 *  - plain C types only; every pointer is a DEVICE pointer unless the name ends in _host;
 *  - every call is asynchronous on the caller's `stream` (a cudaStream_t passed as void*),
 *    no hidden synchronisation, CUDA-graph capturable; the *_host entry points enqueue
 *    their own copies on that stream and are asynchronous as well;
 *  - every pointer is aligned to its element type (8 bytes for int64 / double, 4 for float / int32); label bitmaps, and the
 *    adj / Y byte grids of the handle's entry points and of the legacy operator, to 16 bytes; an optional pointer may be NULL;
 *  - return value: 0 = ok, <0 = error (HDGNN_E_*); text via hdgnn_last_error(), which names the entry point and the
 *    argument of a refused stateless call;
 *  - a handle belongs to one device and one host thread at a time;
 *  - the caller owns params / grads / Adam moments (one flat fp32 blob each, laid out in
 *    the TF variable-creation order of the variant's build_model, see hdgnn_param_layout);
 *    the handle owns only scratch.
 *
 * Compact inputs (replace the nine dense feeds of model_2.py:54-82, built by
 * utils2.py:29-137):
 *   adj  uint8  (B, Ne, adj_pitch)  off-diagonal entity adjacency A_ij in {0,1}; the diagonal
 *                                   is ignored.  Row pitch in bytes, multiple of 16, >= Ne.
 *   x    float  (B, Ne)             node attribute x_i = raw A_ii            (utils2.py:35)
 *   hmap int32  (B, Ne)             hunk id of index line i; <0 or >=Nc = none (utils2.py:129-136)
 *   L    int32  (B)                 index lines read, 0 <= L <= Ne (fewer than 2: nothing is pooled)  (utils2.py:121)
 *   Y    uint8  (B, Nc, y_pitch)    off-diagonal hunk adjacency = label      (utils2.py:47,105)
 * Outputs
 *   logits, probs  float (B, 2, Ncr), Ncr = Nc(Nc-1), pair order p(s,t) = s(Nc-1)+t-[t>s]
 *                  (utils2.py:91-106); channel 0 = "no relation"             (model_2.py:321-323)
 */
#ifndef HDGNN_H_INCLUDED
#define HDGNN_H_INCLUDED

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HDGNN_OK              0
#define HDGNN_E_INVALID      -1   /* bad argument (shape, variant, pitch, null pointer) */
#define HDGNN_E_CUDA         -2   /* a CUDA runtime call failed; see hdgnn_last_error */
#define HDGNN_E_NOMEM        -3
#define HDGNN_E_UNSUPPORTED  -4   /* e.g. Ne or Nc above the compiled limit */
#define HDGNN_E_PEER         -5   /* a peer's share of the gradient exchange did not arrive in time (hdgnn_peer_status) */

#define HDGNN_MAX_N          512  /* largest Ne / Nc the kernels are instantiated for */
#define HDGNN_HIDDEN         20   /* hidden / effect width: h_size, De_e, De_er (main.py:31-32) */

typedef struct hdgnn_handle_s* hdgnn_handle_t;

typedef struct {
    int32_t Ne;             /* --Ne  main.py:38 */
    int32_t Nc;             /* --Nc  main.py:39 */
    int32_t variant;        /* 1 = model_1 (HD-GNN/ES), 2 = model_2 (HD-GNN/S, main.py:6),
                               3 = model_3 (HD-GNN/E), 4 = model_4 (HD-GNN) */
    int32_t max_batch;      /* largest B any later call will pass */
    int32_t device;         /* CUDA device ordinal */
    int32_t rows_per_cta_e; /* tuning of the multi-kernel path: entity-grid rows per CTA, 0 = default */
    int32_t rows_per_cta_c; /* tuning of the multi-kernel path: hunk-grid rows per CTA, 0 = default */
    int32_t flags;          /* HDGNN_F_* */
} hdgnn_config_t;

/* flag value 1 is reserved */
#define HDGNN_F_DEBUG   2   /* keep named copies of intermediates for hdgnn_workspace (tests) */
#define HDGNN_F_LEGACY  4   /* force the multi-kernel path (otherwise taken only by TRAINING above 256 hunks; the per-commit kernel
                               serves every variant up to Nc = 256 and the forward pass up to Nc = 512) */
#define HDGNN_F_LABEL_BITS 8 /* every entry point receives LABEL BITMAPS instead of byte grids: adj (device) / adj_host is
                               (B, Ne, hdgnn_bit_words(Ne)) uint32 and Y / Y_host (B, Nc, hdgnn_bit_words(Nc)) uint32, word w of a
                               row holding column 32 w + k at bit k (little-endian np.packbits order), diagonal and padding
                               bits ZERO; adj_pitch / y_pitch = 4 * hdgnn_bit_words(n).  1/8 of the bytes on the wire and
                               in HBM and no packing kernel; the same results as byte grids.  The *_host entry points copy the five arrays with ONE DMA when
                               they sit back to back in one pinned block in the order adj, Y, x, hmap, L, every array starting
                               at the next multiple of 16 bytes (what hdgnn_b200.model.HostBatch builds); any other placement
                               is copied array by array.  hdgnn_pack_label_bits builds the format on the device. */

#define HDGNN_F_DENSE_SWEEP 16 /* variants 2 / 3: run the entity pair layer (model_2.py:161-188) as the dense Ne x Ne sweep kernels
                               (ent_fwd2 / ent_bwd2) instead of the default sorted-prefix + edge-walk form inside the per-commit
                               kernel, whose cost grows with the number of edges: choose this for adjacency densities above ~25 % */

/* number of fp32 parameters of a variant (2127 for variant 2, 3129 for variant 4) */
int hdgnn_param_count(int variant);
/* offset (in floats) of a named block in the flat parameter blob, or -1.  Names:
 * ent_w1 ent_b1 ent_w5 ent_b5 nod_w1 nod_b1 nod_w2 nod_b2 edg_w11 edg_w12 edg_b1 edg_w2 edg_b2
 * eup_w1 eup_b1 eup_w2 eup_b2 hnk_w1 hnk_b1 hnk_w2 hnk_b2 scr_w1 scr_b1 scr_w2 scr_b2 theta1 theta2
 * (= r1_w1o r1_b1o r1_w5o r1_b5o o1_w1o o1_b1o o1_w2o o1_b2o | r1_w1r1 r1_w1r2 r1_b1r r1_w2r r1_b2r
 *    o1_w1r o1_b1r o1_w2r o1_b2r | w1 b1 r1_w2r b2 C_edge_w1 C_edge_b1 o1_w2r o1_b2r | map_theta1/2) */
int hdgnn_param_offset(int variant, const char* name);

int hdgnn_create(const hdgnn_config_t* cfg, hdgnn_handle_t* out);
int hdgnn_destroy(hdgnn_handle_t h);
/* h may be NULL: the message of the calling thread's last failed call without a handle (hdgnn_create or a stateless entry point) */
const char* hdgnn_last_error(hdgnn_handle_t h);
int hdgnn_label_pitch(int n);                         /* required row pitch for an n x n byte grid */
int hdgnn_bit_words(int n);                           /* uint32 words per row of an n x n label bitmap (16-byte rows) */

/* Forward only.  Replaces sess.run([loss_Hedge_mse, loss_map, C_edge_output2]) of
 * model_2.py:486-502 (graph of model_2.py:86-118).  `loss` receives the mean softmax
 * cross-entropy over B*Ncr pairs (model_2.py:115-118).  logits may be NULL. */
int hdgnn_forward(hdgnn_handle_t h, int B,
                  const uint8_t* adj, int adj_pitch, const float* x, const int32_t* hmap,
                  const int32_t* L, const uint8_t* Y, int y_pitch,
                  const float* params, float* logits, float* probs, float* loss, void* stream);

/* Forward + backward.  Replaces the forward and autodiff part of
 * sess.run([merged, C_edge_output2, loss_Hedge_mse, loss_map, theta, trainer]) of
 * model_2.py:369-383.  grads (param_count floats) receives d(10*CE)/dparams where CE is the
 * mean over `B_global`*Ncr pairs (pass B_global = B on one GPU; with commit sharding each
 * rank passes its local B and the global count, and the ranks' grads are summed).  The
 * regularisers of model_2.py:121-130,326-336 are replica-identical and are applied inside
 * hdgnn_adam_step.  `loss` receives sum(CE)/(B_global*Ncr) for the local commits. */
int hdgnn_forward_backward(hdgnn_handle_t h, int B, int B_global,
                           const uint8_t* adj, int adj_pitch, const float* x, const int32_t* hmap,
                           const int32_t* L, const uint8_t* Y, int y_pitch,
                           const float* params, float* logits, float* probs, float* loss,
                           float* grads, void* stream);

/* Regularisers + TF1 Adam (model_2.py:336-338; tf.train.AdamOptimizer semantics:
 * lr_t = lr*sqrt(1-b2^t)/(1-b1^t), p -= lr_t*m/(sqrt(v)+eps), m and v un-corrected).
 * Adds d/dp [0.1*0.01*(|theta1|+|theta2|) + 0.001*sum_v l2_loss(v)] to grads first.
 * `step_counter` is a device int32 holding t-1; the kernel uses t = *step_counter+1 and
 * stores it back, so the call is replayable from a CUDA graph.  reg_losses (device, 2
 * floats, may be NULL) receives {loss_map, loss_para} evaluated at the pre-update params. */
int hdgnn_adam_step(hdgnn_handle_t h, float* params, const float* grads, float* m, float* v,
                    int32_t* step_counter, float lr, float beta1, float beta2, float eps,
                    float* reg_losses, void* stream);

/* One whole training step on device-resident inputs: forward, backward, regularisers and TF1 Adam
 * (= hdgnn_forward_backward with B_global = B followed by hdgnn_adam_step, with the gradient
 * reduction and the optimizer fused into one launch).  Replaces one
 * sess.run([merged, C_edge_output2, loss_Hedge_mse, loss_map, theta, trainer]) of model_2.py:369-383
 * on ONE GPU (with commit sharding use hdgnn_forward_backward + all-reduce + hdgnn_adam_step).
 * loss3 (device, 3 floats) receives {CE, loss_map, loss_para}; probs / logits may be NULL. */
int hdgnn_train_step(hdgnn_handle_t h, int B,
                     const uint8_t* adj, int adj_pitch, const float* x, const int32_t* hmap,
                     const int32_t* L, const uint8_t* Y, int y_pitch,
                     float* params, float* m, float* v, int32_t* step_counter,
                     float lr, float beta1, float beta2, float eps,
                     float* logits, float* probs, float* loss3, void* stream);

/* One whole training step from HOST buffers (pinned recommended): H2D copies of the five
 * compact inputs, forward, backward, Adam, and {CE, loss_map, loss_para} into loss3_host (stored by the last kernel
 * when loss3_host is pinned and the step runs on the fused path, else copied D2H).  The kernels and the D2H copies are
 * enqueued on `stream`; the H2D copies go through two staging slots on a copy stream owned by the handle, so the copies
 * of one call overlap the kernels of the previous one.  A slot is refilled after an event `stream` records behind the
 * call's kernels; the kernels wait for the copies through an event, or, when the per-commit kernel is the first kernel
 * of the step (label bitmaps, HDGNN_F_LABEL_BITS, and no dense entity sweep), by polling a tag the copy stream's last
 * DMA writes, which keeps `stream` free of cross-stream waits.  Host buffers must stay unchanged until `stream` has passed the call.  Un-pitched host layouts: adj (B,Ne,Ne), Y (B,Nc,Nc).
 * probs_host may be NULL (otherwise B*2*Ncr floats are copied out; the pointer may also be a DEVICE buffer, e.g. to feed
 * hdgnn_eval_counts without a round trip through the host). */
int hdgnn_train_step_host(hdgnn_handle_t h, int B,
                          const uint8_t* adj_host, const float* x_host, const int32_t* hmap_host,
                          const int32_t* L_host, const uint8_t* Y_host,
                          float* params, float* m, float* v, int32_t* step_counter,
                          float lr, float beta1, float beta2, float eps,
                          float* probs_host, float* loss3_host, void* stream);

/* Forward + backward from HOST buffers (the commit-sharded form of hdgnn_train_step_host): H2D copies of this
 * rank's commits, then as hdgnn_forward_backward.  probs / loss / grads are DEVICE pointers (grads is the buffer
 * the caller all-reduces before hdgnn_adam_step); probs and loss may be NULL. */
int hdgnn_forward_backward_host(hdgnn_handle_t h, int B, int B_global,
                                const uint8_t* adj_host, const float* x_host, const int32_t* hmap_host,
                                const int32_t* L_host, const uint8_t* Y_host,
                                const float* params, float* probs, float* loss, float* grads, void* stream);

/* ---- commit sharding with the gradient all-reduce fused into the reduce + Adam kernel (one process per GPU) --------
 * The reference is single-device; this replaces what a data-parallel port would do with an NCCL all-reduce between
 * hdgnn_forward_backward and hdgnn_adam_step.  Every rank owns a mailbox in its HBM; the last kernel of the step pushes
 * its 16-parameter gradient slices into every peer's mailbox over NVLink (P2P stores of {sequence number : value}
 * words, no flag and no fence), polls its own mailbox for the peers' slices, sums them in rank order (bitwise identical
 * on all ranks) and applies the regularisers + TF1 Adam -- the step has the same launches as on one GPU (two with label bitmaps) and no NCCL call.
 * Set-up: (1) every rank calls hdgnn_peer_export and receives a 64-byte CUDA IPC handle; (2) the handles are gathered by
 * the caller (torch.distributed / MPI / files) into world*64 bytes ordered by rank; (3) every rank calls
 * hdgnn_peer_attach, then the ranks synchronise once (barrier) before the first step.  Fused path only (Nc <= 256),
 * world <= 8, equal shards. */
#define HDGNN_IPC_HANDLE_BYTES 64
int hdgnn_peer_export(hdgnn_handle_t h, int world, unsigned char* ipc_handle_out);
int hdgnn_peer_attach(hdgnn_handle_t h, int rank, int world, const unsigned char* ipc_handles);
/* Synchronises with the device and reports whether any exchange since hdgnn_peer_attach timed out (HDGNN_E_PEER): a wait
 * that sees no data for HDGNN_PEER_TIMEOUT_MS (environment, default 20000) gives up WITHOUT killing the context; the
 * parameters are then out of step with the peers' and training must stop.  Cheap enough for once per epoch. */
int hdgnn_peer_status(hdgnn_handle_t h);
/* As hdgnn_train_step / hdgnn_train_step_host for this rank's B commits of a global batch of B_global = B * world.
 * loss3[0] receives the GLOBAL mean cross-entropy (the ranks' shares are exchanged with the gradients). */
int hdgnn_train_step_peer(hdgnn_handle_t h, int B, int B_global,
                          const uint8_t* adj, int adj_pitch, const float* x, const int32_t* hmap,
                          const int32_t* L, const uint8_t* Y, int y_pitch,
                          float* params, float* m, float* v, int32_t* step_counter,
                          float lr, float beta1, float beta2, float eps,
                          float* logits, float* probs, float* loss3, void* stream);
int hdgnn_train_step_peer_host(hdgnn_handle_t h, int B, int B_global,
                               const uint8_t* adj_host, const float* x_host, const int32_t* hmap_host,
                               const int32_t* L_host, const uint8_t* Y_host,
                               float* params, float* m, float* v, int32_t* step_counter,
                               float lr, float beta1, float beta2, float eps,
                               float* probs_out, float* loss3_host, void* stream);

/* Inference from HOST buffers: H2D, forward, copy-out of probs (B*2*Ncr floats; host or device pointer) and D2H of CE.
 * probs_host may be NULL: the probabilities are then neither written nor copied (a caller that wants only the predicted
 * relations of hdgnn_set_predictions, the counters of hdgnn_set_eval_counters or the loss). */
int hdgnn_infer_host(hdgnn_handle_t h, int B,
                     const uint8_t* adj_host, const float* x_host, const int32_t* hmap_host,
                     const int32_t* L_host, const uint8_t* Y_host,
                     const float* params, float* probs_host, float* loss_host, void* stream);

/* ---- legacy operator of model.py (not used by the live model_1..4; SURVEY K15) ------------------------------
 * out (B,N,d_out) = act( A_hat (H W) + bias ),  A_hat = D^-1/2 A^T D^-1/2,  D = rowsum(A) + eps: the
 * normalize_adj of model.py:360-367 (eps = 1e-3, no self loop, transposed) fused with one propagation.
 * H (B,N,d_in); W (d_in,d_out) row-major or NULL (then d_in == d_out); bias (d_out) or NULL; d_in, d_out <= 32;
 * dinv_out (B,N) optionally receives D^-1/2.  flags select the variants.  Stateless (no handle).
 * The adjacency of the four legacy entry points is either
 *   - a byte grid: uint8 (B, N, adj_pitch), A_ij != 0 is an edge, adj_pitch >= N and a multiple of 16; or
 *   - with HDGNN_P_LABEL_BITS, a label bitmap in the layout of HDGNN_F_LABEL_BITS: (B, N, hdgnn_bit_words(N)) uint32,
 *     bit k of word w of row i = A_i,32w+k, adj_pitch = 4 * hdgnn_bit_words(N) exactly (what hdgnn_pack_label_bits writes).
 * Either way the diagonal (and for bitmaps the padding bits, columns >= N) is ignored.
 * The per-commit state (N * adj_pitch bytes of adjacency + two bitmaps + N * d_out floats) must fit one SM's shared
 * memory, else HDGNN_E_UNSUPPORTED: byte grids up to N ~ 380 at d_out = 20, label bitmaps up to N = HDGNN_MAX_N = 512
 * (a 32 KB tile).  With bitmaps the persistent tcgen05 kernel is the default up to N = 240 at d_in = 20 (byte grids: N = 208). */
#define HDGNN_P_SELF_LOOP     1   /* normalise and propagate A + I (the textbook GCN form) */
#define HDGNN_P_RELU          2
#define HDGNN_P_NO_TRANSPOSE  4   /* A_hat = D^-1/2 A D^-1/2 */
#define HDGNN_P_NO_TENSOR     8   /* force the CUDA-core set-bit walk (default for N <= 256: tcgen05, bf16 x 3 split, fp32 in TMEM) */
#define HDGNN_P_TENSOR_V1    16   /* force the one-CTA-per-commit tcgen05 kernel (default: the persistent kernel when its buffers fit) */
#define HDGNN_P_LABEL_BITS   32   /* adj is a label bitmap, not a byte grid (see above); same kernels, same results */
int hdgnn_normalize_propagate(int B, int N, const uint8_t* adj, int adj_pitch, const float* H, int d_in,
                              const float* W, const float* bias, int d_out, float eps, int flags,
                              float* out, float* dinv_out, void* stream);

/* map_conv of model.py:394-403 with k = 2 and Ds = 1 (chebyshev_polynomials, model.py:335-391):
 * per_commit[b] = (x_b^T (t0 I + t1 ((2/lam_max)(I - A_hat) - I)) x_b)^2,  t = softmax(theta),  and
 * *loss = mean_b per_commit[b] (loss may be NULL).  theta: device, 2 floats (raw).  The reference uses
 * lam_max = 1.5, eps = 1e-3, flags = 0. */
int hdgnn_map_conv(int B, int N, const uint8_t* adj, int adj_pitch, const float* x, const float* theta,
                   float lam_max, float eps, int flags, float* per_commit, float* loss, void* stream);

/* Backward of the legacy operator.  The reference trains through map_conv (model.py:150-155, 405-417), but the edge tensor
 * enters chebyshev_polynomials through tf.argmax (model.py:337): the adjacency is a hard {0,1} grid without gradient, so the
 * backward runs w.r.t. the node features / weights / Chebyshev coefficients only.
 *
 * hdgnn_normalize_propagate_backward: out = act(A_hat (H W) + bias).  dOut (B,N,d_out); `out` is the forward's output (read
 * only with HDGNN_P_RELU, for the mask).  dH (B,N,d_in), dW (d_in,d_out), dbias (d_out): each may be NULL.  dZ = A_hat^T dPre is
 * computed by the forward's own kernel with the transposition flipped (same tcgen05 path).  work: device scratch of
 * hdgnn_propagate_backward_work(B,N,d_in,d_out) floats.  Same flags as the forward. */
size_t hdgnn_propagate_backward_work(int B, int N, int d_in, int d_out);
int hdgnn_normalize_propagate_backward(int B, int N, const uint8_t* adj, int adj_pitch, const float* H, int d_in, const float* W,
                                       int d_out, float eps, int flags, const float* out, const float* dOut,
                                       float* dH, float* dW, float* dbias, float* work, void* stream);
/* hdgnn_map_conv_backward: gscale * d loss / d x -> dx (B,N) and gscale * d loss / d theta -> dtheta (2) for the loss of
 * hdgnn_map_conv (either output may be NULL).  work: 2*B floats (needed for dtheta). */
int hdgnn_map_conv_backward(int B, int N, const uint8_t* adj, int adj_pitch, const float* x, const float* theta, float lam_max,
                            float eps, int flags, float gscale, float* dx, float* dtheta, float* work, void* stream);

/* ---- the data formats either side of the hot path (SURVEY 8(f) rows 1 and 2); stateless, asynchronous on `stream` ----
 * Device-side loader, replaces the array half of utils2.py:29-47 (diagonal -> node attribute, diagonal zeroed) and the
 * int() label indexing of utils2.py:82,105.  raw: (N,n,n) float64 (raw_is_f64 != 0) or float32, exactly as stored in
 * CAdjs_{step}.npy / CHunkAdjs_{step}.npy.  grid: (N,n,pitch) u8 in {0,1}, zero diagonal, zero padding (pitch as
 * hdgnn_label_pitch(n)); diag: (N,n) f32 or NULL; err: device int32, OR-ed with 1 when an off-diagonal entry does
 * not truncate to -2,-1,0 or 1 (an IndexError in the reference), may be NULL. */
int hdgnn_compact_from_raw(int N, int n, const void* raw, int raw_is_f64, uint8_t* grid, int pitch, float* diag,
                           int32_t* err, void* stream);

/* Byte grids -> label bitmaps (the format of HDGNN_F_LABEL_BITS) on the device: grid (N,n,pitch) u8, 16-byte aligned, as
 * written by hdgnn_compact_from_raw, bits (N,n,hdgnn_bit_words(n)) uint32; diagonal and padding bits come out zero. */
int hdgnn_pack_label_bits(int N, int n, const uint8_t* grid, int pitch, uint32_t* bits, void* stream);

/* Weakly connected components of per-commit hunk graphs given as label bitmaps (HDGNN_F_LABEL_BITS layout, e.g. the output of
 * hdgnn_set_predictions, or the labels Y): hunks s and t are joined when bit (s,t) OR bit (t,s) is set; diagonal and padding
 * bits are ignored.  bits (B, n, hdgnn_bit_words(n)) uint32; groups (B, n) int32 receives, for every hunk, the
 * SMALLEST hunk index of its component (a canonical labelling: two partitions are equal iff the arrays are equal); ngroups (B)
 * int32 or NULL receives the number of components.  2 <= n <= HDGNN_MAX_N.  Integer-exact, deterministic.  Stateless. */
int hdgnn_hunk_groups(int B, int n, const uint32_t* bits, int32_t* groups, int32_t* ngroups, void* stream);

/* Partition agreement of two hunk groupings per commit (e.g. hdgnn_hunk_groups of the predicted relations and of the labels),
 * over the REAL hunks 0 .. m-1 of each commit, m = nh[b] (nh (B) int32, or NULL: m = n).  pred, truth (B, n) int32: any
 * labelling with values in [0, n) on the real hunks (hunks >= m are ignored, whatever they hold).  counts (B, 8) int64 is
 * WRITTEN (not added), row b =
 *   {m, pairs joined in both, pairs joined by pred, pairs joined by truth, groups of pred, groups of truth,
 *    sum over pred groups of the largest overlap with a truth group, sum over truth groups of the largest overlap with a pred group}
 * (pairs = unordered pairs {s,t}, s < t < m).  A commit with nh[b] outside [0, n] or a real hunk labelled outside [0, n) gets
 * the row all -1.  2 <= n <= HDGNN_MAX_N.  Integer-exact, deterministic,
 * stateless, asynchronous on `stream`. */
int hdgnn_partition_counts(int B, int n, const int32_t* pred, const int32_t* truth, const int32_t* nh,
                           int64_t* counts, void* stream);

/* Hunk groups by average-linkage (UPGMA) clustering of the relation probabilities, over the REAL hunks 0 .. m-1 of each commit,
 * m = nh[b] (nh (B) int32, or NULL: m = n).  probs (B, 2, n(n-1)) f32 as the relation head writes it (pair order
 * p(s,t) = s(n-1)+t-[t>s]); only channel 1 of the real pairs is read.  The similarity of hunks s != t is
 * w(s,t) = fmaxf(p1(s,t), p1(t,s)) (either direction joins, as in hdgnn_hunk_groups).  From the m singletons, the two clusters
 * with the largest mean similarity mean(A,C) = S(A,C) / (float)(|A| |C|) (S the fp32 sum of w over A x C, updated by
 * S(A u B, C) = S(A,C) + S(B,C); IEEE division) are merged while that mean is > threshold; ties go to the smaller
 * (min representative, max representative), a cluster's representative being its smallest hunk; a NaN mean never merges.
 * A confident pair between two groups therefore does not join them unless the groups' mean clears the threshold.
 * groups (B, n) int32 receives the representative of every real hunk's cluster and s for every hunk s >= m (the canonical
 * labelling of hdgnn_hunk_groups, which hdgnn_partition_counts takes); ngroups (B) int32 or NULL the number of distinct values.
 * A commit with nh[b] outside [0, n] gets groups all -1 and ngroups -1.  `work`: device scratch of
 * hdgnn_hunk_clusters_work(B, n) bytes (0 for n <= 169: the commit's tables live in shared memory; else min(B, 296)
 * pairs of tables of n (n|1) 4-byte words), may be NULL when that is 0.  2 <= n <= HDGNN_MAX_N;
 * threshold not NaN.  Deterministic (the merge sequence fixes every rounding), stateless, asynchronous on `stream`. */
size_t hdgnn_hunk_clusters_work(int B, int n);
int hdgnn_hunk_clusters(int B, int n, const float* probs, const int32_t* nh, float threshold,
                        int32_t* groups, int32_t* ngroups, void* work, void* stream);

/* The dendrogram of hdgnn_hunk_clusters: the same clustering (inputs, w, fp32 sums, tie rule, `work` of
 * hdgnn_hunk_clusters_work) without a threshold, recording every merge.  It stops only when no pair with a non-NaN mean is
 * left; a mean of +-inf merges like any other.  merges (B, n-1, 2) int32: row i = (a, c), a < c, cluster c joined cluster a,
 * which stays the representative; heights (B, n-1) f32: that pair's mean (-0 stored as +0); nmerges (B) int32: the rows
 * recorded, m - 1 unless NaN means were left over.  Rows from nmerges on hold (-1, -1) and NaN.  A commit with nh[b] outside
 * [0, n] gets nmerges -1 and every row -1 / NaN.  2 <= n <= HDGNN_MAX_N.  Deterministic, stateless, asynchronous on `stream`.
 *
 * Merge heights need not be monotone: UPGMA is in exact arithmetic, but the fp32 sums and the division can put a later height
 * one ulp above an earlier one.  So a threshold cut is defined as a PREFIX: hdgnn_hunk_clusters(t) performs the same merges
 * and stops at the first whose mean is not > t, hence hdgnn_linkage_cut(hdgnn_hunk_linkage(p), t) equals
 * hdgnn_hunk_clusters(p, t) bit for bit, groups and ngroups, for every non-NaN t. */
int hdgnn_hunk_linkage(int B, int n, const float* probs, const int32_t* nh, int32_t* merges, float* heights, int32_t* nmerges,
                       void* work, void* stream);

/* Hunk groups at K cuts of recorded merge sequences (the outputs of hdgnn_hunk_linkage, or the same arrays read back from a
 * file).  Cut k of commit b applies the commit's first c merges, m = nh[b] (nh NULL: m = n):
 *   threshold mode (thresholds_host: K host floats, 1 <= K <= 64, none NaN, taken by value; target NULL): c = the length of
 *     the longest prefix of the commit's merges whose heights are all > thresholds_host[k];
 *   group-count mode (target: device (B) int32; K = 1; thresholds_host NULL): c = min(nmerges[b], max(0, m - max(target[b], 1))),
 *     scipy's maxclust, except that a sequence stopped early by NaN means leaves more groups than asked for.
 * groups (K, B, n) int32: the representative (smallest hunk) of s's cluster after those merges for s < m, s for s >= m;
 * ngroups (K, B) int32 or NULL: n - c.  This is the labelling of hdgnn_hunk_clusters, which hdgnn_partition_counts takes.
 * A commit whose record is inconsistent -- nh[b] outside [0, n], nmerges[b] outside [0, max(m - 1, 0)], a row without
 * 0 <= a < c < m, a c that appears twice, or an a absorbed at an earlier row -- gets groups and ngroups -1 for every cut; no
 * row past nmerges[b] is read.  2 <= n <= HDGNN_MAX_N.  Integer-exact, deterministic, stateless, asynchronous on `stream`. */
int hdgnn_linkage_cut(int B, int n, const int32_t* merges, const float* heights, const int32_t* nmerges, const int32_t* nh,
                      int K, const float* thresholds_host, const int32_t* target, int32_t* groups, int32_t* ngroups,
                      void* stream);

/* Evaluation counters on the device, replaces the loops of EvaluationFuncs.py:27-37 (top_ACC), :92-117 (prec / recall /
 * f1) and :119-153 (AUC) over the probs the relation head wrote.  probs (B,2,Ncr) f32, Y (B,Nc,y_pitch) u8.
 * counts (B,8) int64: {arg-max hits, quirk tp, fp, fn (ceil of channel 0, as the reference scores), conventional tp, fp,
 * fn (relation = channel 1, p1 > p0), related pairs}.  auc (B,2) int64 or NULL: Mann-Whitney numerators
 * 2 #{s_neg < s_pos} + #{s_neg == s_pos} for {the reference's scoring, score = p1}, computed for commits >= auc_first
 * (the reference's AUC only keeps the LAST commit, quirk Q7); AUC = auc / (2 npos nneg). */
int hdgnn_eval_counts(int B, int Nc, const float* probs, const uint8_t* Y, int y_pitch, int64_t* counts, int64_t* auc,
                      int auc_first, void* stream);

/* Accuracy counter of the training loop without a second kernel: while `acc` (device, one uint64, caller-owned) is set, every
 * forward / training call ADDS the number of hunk pairs whose arg-max class equals the label (EvaluationFuncs.py:27-37, a
 * tie is class 0) for all commits of the call; the caller zeroes it when a new epoch starts.  NULL switches it off.  Fused
 * path only (HDGNN_E_UNSUPPORTED otherwise: use hdgnn_eval_counts). */
int hdgnn_set_hits_accumulator(hdgnn_handle_t h, uint64_t* acc);

/* The evaluation counters of hdgnn_eval_counts without a second kernel and without the label bytes: while `counts` (device,
 * (B,8) int64 in that function's layout, caller-owned, row b = commit b of a call) is set, the relation head of every forward
 * / training call ADDS the commit's counters (EvaluationFuncs.py:27-37 top_ACC, :92-117 prec / recall / f1 in the reference's
 * and in the conventional form) -- two warp votes per 32 hunk pairs against the label bitmap the kernel already holds.  The
 * caller zeroes the rows and re-points `counts` per batch.  NULL switches it off.  AUC (EvaluationFuncs.py:119-153) needs the
 * sorted scores: hdgnn_eval_counts.  Fused path only (HDGNN_E_UNSUPPORTED otherwise). */
int hdgnn_set_eval_counters(hdgnn_handle_t h, int64_t* counts);

/* The model's answer in the label format: while `pred` (device, (B, Nc, hdgnn_bit_words(Nc)) uint32, 16-byte aligned,
 * caller-owned; row b = commit b of a call) is set, every forward / training call WRITES (does not add) each commit's
 * predicted relations in the HDGNN_F_LABEL_BITS layout: bit (s,t) = [p1(s,t) > p0(s,t)] (np.argmax over the two channels, a
 * tie is class 0: the y_pred of top_ACC and of the conventional prec / recall form, EvaluationFuncs.py:27-37, 92-117);
 * diagonal bits, padding bits and padding words are written zero.  The relation head stores one word per 32 hunk pairs; the
 * probabilities may be switched off (probs = NULL).  NULL switches it off.  Available on the fused and on the multi-kernel
 * path.  hdgnn_hunk_groups turns the bitmap into hunk groups. */
int hdgnn_set_predictions(hdgnn_handle_t h, uint32_t* pred);

/* Debug / test introspection: device pointer and size in bytes of a named scratch buffer of the handle.  With HDGNN_F_DEBUG
 * the intermediates of the last step: S1 X2 NB RS3 CS3F PR PC DNB DX2 GE, RS1 beside the dense entity sweeps and on the
 * multi-kernel path, and on the fused path the per-commit phase clocks CLK; PEER_STAMPS with HDGNN_PEER_STAMPS set.  A name
 * the library does not know, and a buffer this handle does not have, each return HDGNN_E_INVALID. */
int hdgnn_workspace(hdgnn_handle_t h, const char* name, void** ptr, size_t* bytes);
/* copy the first `bytes` bytes of a named scratch buffer to dst (device or host pointer) on `stream` */
int hdgnn_workspace_copy(hdgnn_handle_t h, const char* name, void* dst, size_t bytes, void* stream);

/* Opt-in per-launch timing for bench.py's roofline line: while enabled, every kernel launch is
 * bracketed by CUDA events on the caller's stream (this perturbs the step; never enable it for
 * a headline timing).  enable=0/1 also clears the recorded list.  hdgnn_profile_get returns the
 * kernel's label and elapsed milliseconds of record `idx` (synchronises on its stop event). */
int hdgnn_profile(hdgnn_handle_t h, int enable);
int hdgnn_profile_count(hdgnn_handle_t h);
int hdgnn_profile_get(hdgnn_handle_t h, int idx, char* name, int name_cap, float* ms);

/* Measurement utility for the roofline denominators (synchronous, current device): sustained fp32 TFLOP/s of the CUDA cores
 * with scalar FFMA (packed = 0) or the packed fma.rn.f32x2 form the pair sweeps use (packed = 1). */
int hdgnn_measure_fp32_peak(int packed, float* tflops_out);

/* number of kernel launches the last forward / forward_backward / adam call enqueued */
int hdgnn_last_launch_count(hdgnn_handle_t h);

#ifdef __cplusplus
}
#endif
#endif /* HDGNN_H_INCLUDED */
