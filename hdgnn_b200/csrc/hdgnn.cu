// libhdgnn.so -- C ABI (include/hdgnn.h) over the sm_100a kernels.  Host side only: argument validation, scratch
// ownership, the launch sequence of one forward / forward+backward / optimizer step, staging of host buffers, the
// peer-memory set-up.  No torch types.
//
// Launch sequences of a training step.  Byte-grid inputs are first turned into label bitmaps (bits.cuh) by pack_bits
// (pack_step); no kernel after it reads a byte grid.  With HDGNN_F_LABEL_BITS the inputs are bitmaps and there is no pack_bits.
//   fused path (all four variants, Nc <= 256, forward only up to Nc = 512; mid2.cuh, entsp.cuh, final.cuh):
//       mid2 (the whole per-commit forward + backward; above 128 hunks with its hunk-stage tables in the per-commit global
//       slice TABS) -> reduce_adam (gradient reduction [+ peer all-reduce] + regularisers + TF-Adam).  With
//       HDGNN_F_DENSE_SWEEP, or when the inline entity state does not fit (Ne = 512 beside Nc <= 128):
//       ent_fwd2 -> mid2 -> ent_bwd2 -> reduce_adam (ent2.cuh).
//   multi-kernel path (HDGNN_F_LEGACY, training with Nc > 256; pairsum.cuh, score.cuh, node.cuh;
//   [E] = entity-edge branch of model_4.py:92-98):
//       fwd : pairsum(ent) -> [E: pairsum(edge) -> head_fwd(edge) -> score(edge, soft out)] -> pool_fwd
//             -> pairsum(hunk) -> head_fwd(hunk) -> score(hunk: logits/probs/CE [+ delta sums]) -> loss
//       bwd : head_bwd(hunk) -> pairsum_bwd(hunk) -> pool_bwd -> pairsum_bwd(ent) -> rank1_grad(ent)
//             -> [E: score(edge, train: recompute + delta sums) -> head_bwd(edge) -> pairsum_bwd(edge)
//                 -> rank1_grad(edge, tied)] -> grad_reduce
//       opt : adam (regularisers fused)
// Which path each mode (forward only / training) takes, and the form of the fused path -- table placement, inline or dense
// entity stage, mid2's shared-memory layout, the cluster form -- is decided once at hdgnn_create by plan_fused (FusedPlan).
//
// Entry points: each checks its arguments and makes one call -- device_step for the device-resident entries, host_step for the
// *_host entries.  host_step stages the host inputs into one of two slots on the handle's copy stream (stage_inputs), runs the
// step on the slot, releases it by an event on the caller's stream (release_slot) and copies the outputs out.  The step
// waits for its staged inputs through an event, or, when mid2 is its first kernel, by polling a tag the copy stream's last DMA
// writes (an event wait would break the programmatic launch chain reduce_adam -> mid2).
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <array>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/hdgnn.h"
#include "common.cuh"
#include "node.cuh"
#include "pairsum.cuh"
#include "score.cuh"
#include "pack.cuh"
#include "fused.h"
#include "final.cuh"
#include "host.cuh"

using namespace hdgnn;

thread_local std::string hdgnn::g_error;

namespace {

struct Block { const char* name; int rows, cols; };
const Block kEnt[] = {{"ent_w1", 4, 20}, {"ent_b1", 1, 20}, {"ent_w5", 20, 20}, {"ent_b5", 1, 20},
                      {"nod_w1", 21, 20}, {"nod_b1", 1, 20}, {"nod_w2", 20, 1}, {"nod_b2", 1, 1}};
const Block kEdge[] = {{"edg_w11", 1, 20}, {"edg_w12", 2, 20}, {"edg_b1", 1, 20}, {"edg_w2", 20, 20},
                       {"edg_b2", 1, 20}, {"eup_w1", 22, 20}, {"eup_b1", 1, 20}, {"eup_w2", 20, 2},
                       {"eup_b2", 1, 2}};
const Block kHunk[] = {{"hnk_w1", 10, 20}, {"hnk_b1", 1, 20}, {"hnk_w2", 20, 20}, {"hnk_b2", 1, 20},
                       {"scr_w1", 22, 20}, {"scr_b1", 1, 20}, {"scr_w2", 20, 2}, {"scr_b2", 1, 2},
                       {"theta1", 1, 2}, {"theta2", 1, 2}};

// TF variable-creation order of build_model: entity-node block (model_2.py:89-91), entity-edge
// block (model_4.py:92-94), hunk block (model_2.py:103-105), thetas (model_2.py:121).
std::vector<std::pair<std::string, int>> layout(int variant) {
    std::vector<std::pair<std::string, int>> out;
    int off = 0;
    auto add = [&](const Block* b, int n) {
        for (int i = 0; i < n; ++i) { out.push_back({b[i].name, off}); off += b[i].rows * b[i].cols; }
    };
    if (variant == 2 || variant == 4) add(kEnt, 8);
    if (variant == 3 || variant == 4) add(kEdge, 9);
    add(kHunk, 10);
    out.push_back({"", off});
    return out;
}

int find_off(const std::vector<std::pair<std::string, int>>& l, const char* name) {
    for (auto& p : l) if (p.first == name) return p.second;
    return -1;
}

ParamOff make_off(int variant) {
    auto l = layout(variant);
    ParamOff o;
    o.ent_w1 = find_off(l, "ent_w1"); o.ent_b1 = find_off(l, "ent_b1"); o.ent_w5 = find_off(l, "ent_w5");
    o.ent_b5 = find_off(l, "ent_b5"); o.nod_w1 = find_off(l, "nod_w1"); o.nod_b1 = find_off(l, "nod_b1");
    o.nod_w2 = find_off(l, "nod_w2"); o.nod_b2 = find_off(l, "nod_b2");
    o.edg_w11 = find_off(l, "edg_w11"); o.edg_w12 = find_off(l, "edg_w12"); o.edg_b1 = find_off(l, "edg_b1");
    o.edg_w2 = find_off(l, "edg_w2"); o.edg_b2 = find_off(l, "edg_b2"); o.eup_w1 = find_off(l, "eup_w1");
    o.eup_b1 = find_off(l, "eup_b1"); o.eup_w2 = find_off(l, "eup_w2"); o.eup_b2 = find_off(l, "eup_b2");
    o.hnk_w1 = find_off(l, "hnk_w1"); o.hnk_b1 = find_off(l, "hnk_b1"); o.hnk_w2 = find_off(l, "hnk_w2");
    o.hnk_b2 = find_off(l, "hnk_b2"); o.scr_w1 = find_off(l, "scr_w1"); o.scr_b1 = find_off(l, "scr_b1");
    o.scr_w2 = find_off(l, "scr_w2"); o.scr_b2 = find_off(l, "scr_b2");
    o.theta1 = find_off(l, "theta1"); o.theta2 = find_off(l, "theta2");
    o.total = l.back().second;
    return o;
}

struct Buf { void* p = nullptr; size_t bytes = 0; };

// The handle's scratch buffers, in the order hdgnn_create allocates them (workspace_bytes sizes them).  The buffers of the
// two staging slots of the *_host entry points are adjacent ids, base + slot.  hdgnn_peer_attach allocates PEER_SEQ and
// PEER_STAMPS.
#define HDGNN_WORKSPACE(X)                                                                                                  \
    X(RS1) X(CS1P) X(S1) X(X2) X(NB) X(PH) X(QH) X(RS3) X(CS3P) X(CS3F) X(PR) X(PC) X(CEP)                                 \
    X(RSM) X(CSMP) X(LSMP) X(HSP) X(DSUMP) X(GRH) X(GCH) X(RS3D) X(CS3DP) X(LS3P) X(DNB) X(GE) X(DX2)                      \
    X(RS1D) X(CS1DP) X(LS1P) X(GPART) X(GPE) X(FIN_L2) X(FIN_CNT) X(EBITS0) X(EBITS1) X(YBITS0) X(YBITS1)                  \
    X(DBG) X(CLK) X(DLT) X(TABS) X(RSEG) X(CSEG) X(REG) X(CEG) X(A1F) X(PREG)                                               \
    X(RSE) X(CSEP) X(CSEF) X(PRE) X(PCE) X(SOFT) X(DSOFT) X(RSME) X(CSMEP) X(LSMEP) X(HSEP) X(DSUMEP)                      \
    X(GRE) X(GCE) X(RSED) X(CSEDP) X(LSEP)                                                                                  \
    X(H_WIRE0) X(H_WIRE1) X(H_ADJ0) X(H_ADJ1) X(H_Y0) X(H_Y1) X(H_ADJ_RAW0) X(H_ADJ_RAW1) X(H_Y_RAW0) X(H_Y_RAW1)          \
    X(H_FLAG) X(H_PROBS) X(H_LOSS) X(H_GRADS) X(PEER_SEQ) X(PEER_STAMPS)

#define WS_ID(n) WS_##n,
enum WsId { HDGNN_WORKSPACE(WS_ID) WS_COUNT };
#undef WS_ID
#define WS_NAME(n) #n,
const char* const kWsName[WS_COUNT] = {HDGNN_WORKSPACE(WS_NAME)};
#undef WS_NAME

// mid2 in one mode of a handle (FusedPlan::mode[0]: forward only, mode[1]: training)
struct Mid2Mode {
    bool fused = false;        // this mode runs on the fused path, else on the multi-kernel path
    Mid2Opts opt;              // mid2's options, normalised; opt.dlt_smem = false: the dL/dlogit table is the DLT workspace
    Mid2Smem lay{}; size_t smem = 0;     // the layout they give and its dynamic shared memory
    int clusters = 0;          // co-resident clusters of two CTAs of the cluster form (mid2.cuh); 0: one CTA per commit
};

// the fused path of a handle, fixed at create by plan_fused; the fields below `mode` apply when mode[0].fused
struct FusedPlan {
    Mid2Mode mode[2];
    bool gt = false;           // mid2's hunk-stage tables in global memory (Nc > 128), workspace TABS; see also Mid2Opts::scg
    bool inl = false;          // entity pair layer inside mid2 (entsp.cuh)
    bool dense = false;        // the entity branch runs as the dense sweeps ent_fwd2 / ent_bwd2 around mid2 (ent2.cuh)
    bool mid2_first = false;   // no dense sweeps: mid2 is the step's first kernel (after pack_bits for byte grids)
    bool edge = false;         // variant 4: the entity-edge branch inside mid2 (its backward too when mode[1].fused)
    int fwd_occ = 1, bwd_occ = 1;  // resident CTAs per SM of the dense sweeps
    bool pdl = true;           // programmatic dependent launch between the fused kernels (off with HDGNN_F_DEBUG)
};

}  // namespace

constexpr int NSLOT = 2;         // staging slots of the *_host entry points

struct hdgnn_handle_s {
    hdgnn_config_t cfg;
    ParamOff po;
    HeadOff ho_hunk, ho_edge;
    int Ne, Nc, pe, pc;        // sizes and byte-grid label pitches
    int WPe = 0, WPc = 0;      // label-bitmap words per row
    int RTe, Se, CWe;          // entity grid tiling
    int RTc, Sc, CWc;          // hunk grid tiling
    bool ent, edge;            // branches that feed the loss
    bool debug = false;
    FusedPlan plan;
    int nsm = 148;
    int cwt = 0;                                               // column segments per pass of the entity sweeps (ent2.cuh)
    int bslot = 0;                                             // bitmap buffer of the current device-fed step (two alternate)
    Buf ws[WS_COUNT];                                          // p = nullptr: not allocated for this handle
    std::string err;
    int launches = 0;
    // opt-in per-launch timing (hdgnn_profile): events bracket every kernel launch
    bool prof = false;
    cudaEvent_t prof_start = nullptr;
    std::vector<std::pair<std::string, std::pair<cudaEvent_t, cudaEvent_t>>> prof_ev;
    // host-entry staging: two slots filled on a private copy stream so the H2D copies of call k+1 overlap
    // the kernels of call k (both calls only enqueue work; the copies are ordered by events or by a tag, stage_inputs)
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_copy[NSLOT] = {}, ev_done[NSLOT] = {};
    bool done_valid[NSLOT] = {};
    int slot = 0, cur = 0, cur_B = 0;      // next slot, the slot (and its batch size) filled by the last stage_inputs call
    // peer exchange (commit sharding over NVLink, final.cuh): own mailbox + the peers' mailboxes mapped through CUDA IPC
    PeerArgs peer{};
    void* peer_box = nullptr;              // own mailbox (cudaMalloc)
    void* peer_map[PEER_MAX] = {};         // IPC mappings of the other ranks' mailboxes
    size_t peer_bytes = 0;
    int peer_world = 0;
    bool peer_ready = false;
    // host-fed steps whose first kernel is mid2: that kernel polls a tag the copy stream's last DMA writes (no event wait on
    // the caller's stream, which would break the programmatic launch chain optimizer -> mid2)
    unsigned long long* hits_acc = nullptr;   // hdgnn_set_hits_accumulator
    unsigned long long* evc = nullptr;        // hdgnn_set_eval_counters
    uint32_t* pred = nullptr;                 // hdgnn_set_predictions
    uint32_t* tag_table = nullptr;         // pinned, tag_table[i] = i: immutable DMA source
    unsigned int slot_uses[NSLOT] = {};
    int cur_tag = -1;                      // tag of the staging slot filled by the last stage_inputs call, -1 = ordered by event
    // HDGNN_F_LABEL_BITS: the entry points receive label bitmaps (bits.cuh layout) instead of byte grids
    bool host_bits = false;
};

namespace {

#define CK(h, call)                                                                               \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess) {                                                                  \
            (h)->err = std::string(#call) + ": " + cudaGetErrorString(e_);                        \
            return HDGNN_E_CUDA;                                                                  \
        }                                                                                         \
    } while (0)

#define PROF_BEGIN(h, st)                                                                         \
    do {                                                                                          \
        if ((h)->prof) {                                                                          \
            cudaEventCreate(&(h)->prof_start);                                                    \
            cudaEventRecord((h)->prof_start, st);                                                 \
        }                                                                                         \
    } while (0)

#define LAUNCH_CHECK(h, what, st)                                                                 \
    do {                                                                                          \
        cudaError_t e_ = cudaGetLastError();                                                      \
        if (e_ != cudaSuccess) {                                                                  \
            (h)->err = std::string(what) + ": " + cudaGetErrorString(e_);                         \
            return HDGNN_E_CUDA;                                                                  \
        }                                                                                         \
        ++(h)->launches;                                                                          \
        if ((h)->prof) {                                                                          \
            cudaEvent_t stop_;                                                                    \
            cudaEventCreate(&stop_);                                                              \
            cudaEventRecord(stop_, st);                                                           \
            (h)->prof_ev.push_back({what, {(h)->prof_start, stop_}});                             \
        }                                                                                         \
    } while (0)

int fail(hdgnn_handle_t h, int code, const std::string& msg) {
    if (h) h->err = msg; else g_error = msg;
    return code;
}

float* F(hdgnn_handle_t h, WsId id) { return static_cast<float*>(h->ws[id].p); }

// a zeroed buffer (FIN_CNT, FIN_L2, H_FLAG and PEER_SEQ rely on starting at zero)
int alloc(hdgnn_handle_t h, WsId id, size_t bytes) {
    Buf& b = h->ws[id];
    cudaError_t e = cudaMalloc(&b.p, bytes);
    if (e != cudaSuccess) { b.p = nullptr; h->err = std::string("cudaMalloc(") + kWsName[id] + "): " + cudaGetErrorString(e); return HDGNN_E_NOMEM; }
    b.bytes = bytes;
    e = cudaMemset(b.p, 0, bytes);
    if (e != cudaSuccess) { h->err = std::string("cudaMemset(") + kWsName[id] + "): " + cudaGetErrorString(e); return HDGNN_E_CUDA; }
    return HDGNN_OK;
}

// hdgnn_workspace*: the buffer called `name`, if this handle has it
int find_ws(hdgnn_handle_t h, const char* name, const Buf** out) {
    for (int i = 0; i < WS_COUNT; ++i) {
        if (strcmp(name, kWsName[i])) continue;
        if (!h->ws[i].p) return fail(h, HDGNN_E_INVALID, std::string("workspace buffer ") + name + " is not allocated for this handle");
        *out = &h->ws[i];
        return HDGNN_OK;
    }
    return fail(h, HDGNN_E_INVALID, std::string("no workspace buffer named ") + name);
}


// ---- template dispatch over the column width CW = ceil(N / 32) ---------------------------------
#define CW_SWITCH(cw, ...)                                                                        \
    switch (cw) {                                                                                  \
        case 1: { constexpr int CW = 1; __VA_ARGS__; } break;   case 2: { constexpr int CW = 2; __VA_ARGS__; } break;   \
        case 3: { constexpr int CW = 3; __VA_ARGS__; } break;   case 4: { constexpr int CW = 4; __VA_ARGS__; } break;   \
        case 5: { constexpr int CW = 5; __VA_ARGS__; } break;   case 6: { constexpr int CW = 6; __VA_ARGS__; } break;   \
        case 7: { constexpr int CW = 7; __VA_ARGS__; } break;   case 8: { constexpr int CW = 8; __VA_ARGS__; } break;   \
        case 9: { constexpr int CW = 9; __VA_ARGS__; } break;   case 10: { constexpr int CW = 10; __VA_ARGS__; } break; \
        case 11: { constexpr int CW = 11; __VA_ARGS__; } break; case 12: { constexpr int CW = 12; __VA_ARGS__; } break; \
        case 13: { constexpr int CW = 13; __VA_ARGS__; } break; case 14: { constexpr int CW = 14; __VA_ARGS__; } break; \
        case 15: { constexpr int CW = 15; __VA_ARGS__; } break; case 16: { constexpr int CW = 16; __VA_ARGS__; } break; \
        default: break;                                                                            \
    }

template <int CW, bool BWD, bool RANK1>
cudaError_t pairsum_attr(size_t smem) {
    return cudaFuncSetAttribute(pairsum_kernel<CW, BWD, RANK1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
}
template <int CW, bool TRAIN, bool PRED>
cudaError_t score_attr(size_t smem) {
    return cudaFuncSetAttribute(score_kernel<CW, TRAIN, PRED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
}

// MaxDynamicSharedMemorySize is a per-function hard cap shared by every handle of the process, so it
// is raised to the device's opt-in maximum once (occupancy follows the size actually launched).
cudaError_t set_attrs(hdgnn_handle_t h, int optin) {
    cudaError_t e = cudaSuccess;
    auto acc = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    const cudaFuncAttribute A = cudaFuncAttributeMaxDynamicSharedMemorySize;
    CW_SWITCH(h->CWe, {
        acc(cudaFuncSetAttribute(pairsum_kernel<CW, false, true>, A, optin));
        acc(cudaFuncSetAttribute(pairsum_kernel<CW, true, true>, A, optin));
        acc(cudaFuncSetAttribute(score_kernel<CW, false, false>, A, optin));
        acc(cudaFuncSetAttribute(score_kernel<CW, true, false>, A, optin));
    });
    CW_SWITCH(h->CWc, {
        acc(cudaFuncSetAttribute(pairsum_kernel<CW, false, false>, A, optin));
        acc(cudaFuncSetAttribute(pairsum_kernel<CW, true, false>, A, optin));
        acc(cudaFuncSetAttribute(score_kernel<CW, false, false>, A, optin));
        acc(cudaFuncSetAttribute(score_kernel<CW, true, false>, A, optin));
        acc(cudaFuncSetAttribute(score_kernel<CW, false, true>, A, optin));       // the hunk head writing predictions
        acc(cudaFuncSetAttribute(score_kernel<CW, true, true>, A, optin));
    });
    acc(cudaFuncSetAttribute(pool_fwd_kernel, A, optin));
    acc(cudaFuncSetAttribute(pool_bwd_kernel, A, optin));
    acc(cudaFuncSetAttribute(head_fwd_kernel, A, optin));
    acc(cudaFuncSetAttribute(head_bwd_kernel, A, optin));
    return e;
}

// grid: which N x N grid a launch runs on
struct GridCfg { int N, RT, S, CW, WP; };
GridCfg ent_grid(hdgnn_handle_t h) { return {h->Ne, h->RTe, h->Se, h->CWe, h->WPe}; }
GridCfg hunk_grid(hdgnn_handle_t h) { return {h->Nc, h->RTc, h->Sc, h->CWc, h->WPc}; }

int launch_pairsum(hdgnn_handle_t h, const char* what, const GridCfg& g, int B, bool bwd, bool rank1, PairSumArgs a, cudaStream_t st) {
    a.N = g.N; a.RT = g.RT; a.S = g.S; a.WP = g.WP;
    const dim3 grid(g.S, B), block(32 * HD);
    PROF_BEGIN(h, st);
    CW_SWITCH(g.CW, {
        const size_t smem = pairsum_smem_bytes(CW, g.RT, 4 * g.WP, bwd);
        if (bwd) {
            if (rank1) pairsum_kernel<CW, true, true><<<grid, block, smem, st>>>(a);
            else pairsum_kernel<CW, true, false><<<grid, block, smem, st>>>(a);
        } else {
            if (rank1) pairsum_kernel<CW, false, true><<<grid, block, smem, st>>>(a);
            else pairsum_kernel<CW, false, false><<<grid, block, smem, st>>>(a);
        }
    });
    LAUNCH_CHECK(h, what, st);
    return HDGNN_OK;
}

int launch_score(hdgnn_handle_t h, const char* what, const GridCfg& g, int B, bool train, ScoreArgs a, cudaStream_t st) {
    a.N = g.N; a.RT = g.RT; a.S = g.S; a.WP = g.WP;
    const dim3 grid(g.S, B), block(32 * HD);
    PROF_BEGIN(h, st);
    CW_SWITCH(g.CW, {
        const size_t smem = score_smem_bytes(CW, g.RT, 4 * g.WP, train);
        if (a.pred) {
            if (train) score_kernel<CW, true, true><<<grid, block, smem, st>>>(a);
            else score_kernel<CW, false, true><<<grid, block, smem, st>>>(a);
        } else {
            if (train) score_kernel<CW, true, false><<<grid, block, smem, st>>>(a);
            else score_kernel<CW, false, false><<<grid, block, smem, st>>>(a);
        }
    });
    LAUNCH_CHECK(h, what, st);
    return HDGNN_OK;
}

int check_inputs(hdgnn_handle_t h, int B, const void* adj, int adj_pitch, const void* x, const void* hmap,
                 const void* L, const void* Y, int y_pitch, const void* params) {
    if (!h) return HDGNN_E_INVALID;
    if (B < 1 || B > h->cfg.max_batch) return fail(h, HDGNN_E_INVALID, "B out of range [1, max_batch]");
    if (!adj || !x || !hmap || !L || !Y || !params) return fail(h, HDGNN_E_INVALID, "null input pointer");
    if (h->host_bits) {
        if (adj_pitch != h->WPe * 4) return fail(h, HDGNN_E_INVALID, "HDGNN_F_LABEL_BITS: adj_pitch must equal 4 * hdgnn_bit_words(Ne)");
        if (y_pitch != h->WPc * 4) return fail(h, HDGNN_E_INVALID, "HDGNN_F_LABEL_BITS: y_pitch must equal 4 * hdgnn_bit_words(Nc)");
    } else {
        if (adj_pitch != h->pe) return fail(h, HDGNN_E_INVALID, "adj_pitch must equal hdgnn_label_pitch(Ne)");
        if (y_pitch != h->pc) return fail(h, HDGNN_E_INVALID, "y_pitch must equal hdgnn_label_pitch(Nc)");
    }
    if (((uintptr_t)adj & 15) || ((uintptr_t)Y & 15)) return fail(h, HDGNN_E_INVALID, "adj and Y must be 16-byte aligned");
    return HDGNN_OK;
}

// the device inputs of a step, its label grids as bitmaps (bits.cuh): given, or made by pack_step
struct Inputs {
    const uint32_t* ebits; const uint32_t* ybits;
    const float* x; const int32_t* hmap; const int32_t* L;
    const float* params;
    const int* wait_flag = nullptr; int wait_tag = 0;                    // staged inputs ordered by a DMA-written tag (mid2 polls it)
};

int forward_impl(hdgnn_handle_t h, int B, int B_global, const Inputs& in, float* logits, float* probs,
                 float* loss, bool train, cudaStream_t st) {
    const ParamOff& po = h->po;
    const GridCfg ge = ent_grid(h), gc = hunk_grid(h);
    int rc;
    if (h->ent) {
        PairSumArgs a{};
        a.bits = in.ebits; a.params = in.params; a.x = in.x;
        a.o_u = po.ent_w1; a.o_v = po.ent_w1 + HD; a.o_b = po.ent_b1; a.o_l = po.ent_w1 + 2 * HD;
        a.RS = F(h, WS_RS1); a.CSp = F(h, WS_CS1P);
        if ((rc = launch_pairsum(h, "pairsum_fwd(ent)", ge, B, false, true, a, st))) return rc;
    }
    if (h->edge) {
        PairSumArgs a{};
        a.bits = in.ebits; a.params = in.params; a.x = in.x;
        a.o_u = po.edg_w11; a.o_v = po.edg_w11; a.o_b = po.edg_b1; a.o_l = po.edg_w12;
        a.RS = F(h, WS_RSE); a.CSp = F(h, WS_CSEP);
        if ((rc = launch_pairsum(h, "pairsum_fwd(edge)", ge, B, false, true, a, st))) return rc;
        HeadFwdArgs hf{};
        hf.N = h->Ne; hf.S = h->Se; hf.RS = F(h, WS_RSE); hf.CSp = F(h, WS_CSEP); hf.params = in.params;
        hf.ho = h->ho_edge; hf.CSf = F(h, WS_CSEF); hf.PR = F(h, WS_PRE); hf.PC = F(h, WS_PCE);
        PROF_BEGIN(h, st);
        head_fwd_kernel<<<B, NODE_THREADS, head_fwd_smem_bytes(), st>>>(hf);
        LAUNCH_CHECK(h, "head_fwd_kernel(edge)", st);
        ScoreArgs s{};
        s.bits = in.ebits; s.PR = F(h, WS_PRE); s.PC = F(h, WS_PCE); s.params = in.params;
        s.o_l = po.eup_w1; s.o_w2 = po.eup_w2; s.o_b2 = po.eup_b2;
        s.soft = F(h, WS_SOFT);
        if ((rc = launch_score(h, "score_fwd(edge)", ge, B, false, s, st))) return rc;
    }
    {
        PoolFwdArgs a{};
        a.Ne = h->Ne; a.Nc = h->Nc; a.Se = h->Se; a.ent = h->ent ? 1 : 0;
        a.x = in.x; a.RS1 = F(h, WS_RS1); a.CS1p = F(h, WS_CS1P); a.params = in.params; a.po = po;
        a.bits = in.ebits; a.WP = h->WPe; a.soft = h->edge ? F(h, WS_SOFT) : nullptr;
        a.hmap = in.hmap; a.L = in.L;
        a.S1 = F(h, WS_S1); a.X2 = F(h, WS_X2); a.NB = F(h, WS_NB); a.PH = F(h, WS_PH); a.QH = F(h, WS_QH);
        PROF_BEGIN(h, st);
        pool_fwd_kernel<<<B, NODE_THREADS, pool_fwd_smem_bytes(h->Ne, h->Nc), st>>>(a);
        LAUNCH_CHECK(h, "pool_fwd_kernel", st);
    }
    {
        PairSumArgs a{};
        a.bits = in.ybits; a.params = in.params; a.o_l = po.hnk_w1 + 8 * HD;
        a.Ptab = F(h, WS_PH); a.Qtab = F(h, WS_QH);
        a.RS = F(h, WS_RS3); a.CSp = F(h, WS_CS3P);
        if ((rc = launch_pairsum(h, "pairsum_fwd(hunk)", gc, B, false, false, a, st))) return rc;
    }
    {
        HeadFwdArgs hf{};
        hf.N = h->Nc; hf.S = h->Sc; hf.RS = F(h, WS_RS3); hf.CSp = F(h, WS_CS3P); hf.params = in.params;
        hf.ho = h->ho_hunk; hf.CSf = F(h, WS_CS3F); hf.PR = F(h, WS_PR); hf.PC = F(h, WS_PC);
        PROF_BEGIN(h, st);
        head_fwd_kernel<<<B, NODE_THREADS, head_fwd_smem_bytes(), st>>>(hf);
        LAUNCH_CHECK(h, "head_fwd_kernel(hunk)", st);
    }
    {
        ScoreArgs s{};
        s.bits = in.ybits; s.PR = F(h, WS_PR); s.PC = F(h, WS_PC); s.params = in.params;
        s.o_l = po.scr_w1; s.o_w2 = po.scr_w2; s.o_b2 = po.scr_b2;
        s.logits = logits; s.probs = probs; s.cep = F(h, WS_CEP); s.pred = h->pred;
        s.scale = 10.f / ((float)B_global * (float)(h->Nc * (h->Nc - 1)));
        s.RSm = F(h, WS_RSM); s.CSmp = F(h, WS_CSMP); s.LSmp = F(h, WS_LSMP); s.HSp = F(h, WS_HSP); s.dsump = F(h, WS_DSUMP);
        if ((rc = launch_score(h, "score(hunk)", gc, B, train, s, st))) return rc;
    }
    if (loss) {
        PROF_BEGIN(h, st);
        loss_reduce_kernel<<<1, 256, 0, st>>>(F(h, WS_CEP), B * h->Sc, (float)B_global * (float)(h->Nc * (h->Nc - 1)), loss);
        LAUNCH_CHECK(h, "loss_reduce_kernel", st);
    }
    return HDGNN_OK;
}

int backward_impl(hdgnn_handle_t h, int B, const Inputs& in, float* grads, cudaStream_t st) {
    const ParamOff& po = h->po;
    const GridCfg ge = ent_grid(h), gc = hunk_grid(h);
    int rc;
    {
        HeadBwdArgs a{};
        a.N = h->Nc; a.S = h->Sc;
        a.RSm = F(h, WS_RSM); a.CSmp = F(h, WS_CSMP); a.LSmp = F(h, WS_LSMP); a.HSp = F(h, WS_HSP); a.dsump = F(h, WS_DSUMP);
        a.RS = F(h, WS_RS3); a.CSf = F(h, WS_CS3F); a.params = in.params; a.ho = h->ho_hunk;
        a.gpart = F(h, WS_GPART); a.total = po.total; a.GR = F(h, WS_GRH); a.GC = F(h, WS_GCH);
        PROF_BEGIN(h, st);
        head_bwd_kernel<<<B, NODE_THREADS, head_bwd_smem_bytes(), st>>>(a);
        LAUNCH_CHECK(h, "head_bwd_kernel(hunk)", st);
    }
    {
        PairSumArgs a{};
        a.bits = in.ybits; a.params = in.params; a.o_l = po.hnk_w1 + 8 * HD;
        a.Ptab = F(h, WS_PH); a.Qtab = F(h, WS_QH); a.GR = F(h, WS_GRH); a.GC = F(h, WS_GCH);
        a.RS = F(h, WS_RS3D); a.CSp = F(h, WS_CS3DP); a.LSp = F(h, WS_LS3P);
        if ((rc = launch_pairsum(h, "pairsum_bwd(hunk)", gc, B, true, false, a, st))) return rc;
    }
    {
        PoolBwdArgs a{};
        a.Ne = h->Ne; a.Nc = h->Nc; a.Sc = h->Sc; a.ent = h->ent ? 1 : 0;
        a.RS3D = F(h, WS_RS3D); a.CS3Dp = F(h, WS_CS3DP); a.LS3p = F(h, WS_LS3P); a.NB = F(h, WS_NB);
        a.x = in.x; a.S1 = F(h, WS_S1); a.X2 = F(h, WS_X2); a.params = in.params; a.po = po;
        a.hmap = in.hmap; a.L = in.L; a.gpart = F(h, WS_GPART); a.total = po.total;
        a.DNB = F(h, WS_DNB); a.GE = F(h, WS_GE); a.DX2 = F(h, WS_DX2);
        a.dsoft = h->edge ? F(h, WS_DSOFT) : nullptr;
        PROF_BEGIN(h, st);
        pool_bwd_kernel<<<B, NODE_THREADS, pool_bwd_smem_bytes(h->Ne, h->Nc), st>>>(a);
        LAUNCH_CHECK(h, "pool_bwd_kernel", st);
    }
    if (h->ent) {
        PairSumArgs a{};
        a.bits = in.ebits; a.params = in.params; a.x = in.x;
        a.o_u = po.ent_w1; a.o_v = po.ent_w1 + HD; a.o_b = po.ent_b1; a.o_l = po.ent_w1 + 2 * HD;
        a.GR = F(h, WS_GE); a.GC = F(h, WS_GE);
        a.RS = F(h, WS_RS1D); a.CSp = F(h, WS_CS1DP); a.LSp = F(h, WS_LS1P);
        if ((rc = launch_pairsum(h, "pairsum_bwd(ent)", ge, B, true, true, a, st))) return rc;
        Rank1GradArgs r{};
        r.N = h->Ne; r.S = h->Se; r.x = in.x; r.RSd = F(h, WS_RS1D); r.CSdp = F(h, WS_CS1DP); r.LSp = F(h, WS_LS1P);
        r.o_u = po.ent_w1; r.o_v = po.ent_w1 + HD; r.o_b = po.ent_b1; r.o_l = po.ent_w1 + 2 * HD;
        r.gpart = F(h, WS_GPART); r.total = po.total;
        PROF_BEGIN(h, st);
        rank1_grad_kernel<<<B, 256, 0, st>>>(r);
        LAUNCH_CHECK(h, "rank1_grad_kernel(ent)", st);
    }
    if (h->edge) {
        ScoreArgs s{};
        s.bits = in.ebits; s.PR = F(h, WS_PRE); s.PC = F(h, WS_PCE); s.params = in.params;
        s.o_l = po.eup_w1; s.o_w2 = po.eup_w2; s.o_b2 = po.eup_b2;
        s.dsoft = F(h, WS_DSOFT);
        s.RSm = F(h, WS_RSME); s.CSmp = F(h, WS_CSMEP); s.LSmp = F(h, WS_LSMEP); s.HSp = F(h, WS_HSEP); s.dsump = F(h, WS_DSUMEP);
        if ((rc = launch_score(h, "score_bwd(edge)", ge, B, true, s, st))) return rc;
        HeadBwdArgs a{};
        a.N = h->Ne; a.S = h->Se;
        a.RSm = F(h, WS_RSME); a.CSmp = F(h, WS_CSMEP); a.LSmp = F(h, WS_LSMEP); a.HSp = F(h, WS_HSEP); a.dsump = F(h, WS_DSUMEP);
        a.RS = F(h, WS_RSE); a.CSf = F(h, WS_CSEF); a.params = in.params; a.ho = h->ho_edge;
        a.gpart = F(h, WS_GPART); a.total = po.total; a.GR = F(h, WS_GRE); a.GC = F(h, WS_GCE);
        PROF_BEGIN(h, st);
        head_bwd_kernel<<<B, NODE_THREADS, head_bwd_smem_bytes(), st>>>(a);
        LAUNCH_CHECK(h, "head_bwd_kernel(edge)", st);
        PairSumArgs p{};
        p.bits = in.ebits; p.params = in.params; p.x = in.x;
        p.o_u = po.edg_w11; p.o_v = po.edg_w11; p.o_b = po.edg_b1; p.o_l = po.edg_w12;
        p.GR = F(h, WS_GRE); p.GC = F(h, WS_GCE);
        p.RS = F(h, WS_RSED); p.CSp = F(h, WS_CSEDP); p.LSp = F(h, WS_LSEP);
        if ((rc = launch_pairsum(h, "pairsum_bwd(edge)", ge, B, true, true, p, st))) return rc;
        Rank1GradArgs r{};
        r.N = h->Ne; r.S = h->Se; r.x = in.x; r.RSd = F(h, WS_RSED); r.CSdp = F(h, WS_CSEDP); r.LSp = F(h, WS_LSEP);
        r.o_u = po.edg_w11; r.o_v = po.edg_w11; r.o_b = po.edg_b1; r.o_l = po.edg_w12;
        r.gpart = F(h, WS_GPART); r.total = po.total;
        PROF_BEGIN(h, st);
        rank1_grad_kernel<<<B, 256, 0, st>>>(r);
        LAUNCH_CHECK(h, "rank1_grad_kernel(edge)", st);
    }
    PROF_BEGIN(h, st);
    grad_reduce_kernel<<<(po.total + 127) / 128, 128, 0, st>>>(F(h, WS_GPART), B, po.total, grads);
    LAUNCH_CHECK(h, "grad_reduce_kernel", st);
    return HDGNN_OK;
}

int adam_impl(hdgnn_handle_t h, float* params, const float* grads, float* m, float* v, int32_t* step,
              float lr, float b1, float b2, float eps, float* reg_losses, cudaStream_t st) {
    PROF_BEGIN(h, st);
    adam_kernel<<<1, 1024, 0, st>>>(params, grads, m, v, h->po.total, h->po.theta1, h->po.theta2, step, lr, b1, b2,
                                    eps, reg_losses);
    LAUNCH_CHECK(h, "adam_kernel", st);
    return HDGNN_OK;
}


// (rows, n) contiguous bytes -> (rows, pitch): cudaMemcpy2DAsync with 200-byte rows is ~30x slower
// than one contiguous DMA plus this kernel.
__global__ void repitch_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, size_t rows, int n, int pitch) {
    if ((n & 3) == 0) {
        const int nw = n >> 2, pw = pitch >> 2;
        const size_t total = rows * (size_t)pw;
        const uint32_t* s4 = reinterpret_cast<const uint32_t*>(src);
        uint32_t* d4 = reinterpret_cast<uint32_t*>(dst);
        for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
            const size_t r = i / pw; const int c = (int)(i - r * pw);
            d4[i] = c < nw ? s4[r * nw + c] : 0u;
        }
    } else {
        const size_t total = rows * (size_t)pitch;
        for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
            const size_t r = i / pitch; const int c = (int)(i - r * pitch);
            dst[i] = c < n ? src[r * n + c] : (uint8_t)0;
        }
    }
}

// ================================================================================================
// pack step (both paths); fused path: ent_fwd2 -> mid2 -> ent_bwd2 -> reduce (+ adam)
// ================================================================================================

struct AdamArgs { float* params; float* m; float* v; int32_t* step; float lr, b1, b2, eps; float* reg; bool peer = false; };

// column segments per pass of an entity sweep: the whole row when it fits 8 segments, else passes of 8
int ent2_cwt(int N) { const int cw = (N + 31) / 32; return cw <= 8 ? cw : 8; }

// Grid of an entity sweep over B commits of N entities: `occ` resident CTAs on each of `nsm` SMs, one wave, the
// B*N rows cut into equal chunks (at least 8 rows each).
void ent2_grid(int B, int N, int occ, int nsm, int* G, int* R) {
    const long long rows = (long long)B * N;
    long long g = (long long)occ * nsm;
    if (g > rows / 8) g = rows / 8 > 0 ? rows / 8 : 1;
    *R = (int)((rows + g - 1) / g);
    *G = (int)((rows + *R - 1) / *R);
}

// largest number of co-resident CTAs per SM (<= 4) whose row chunk of a full batch fits next to each other
int ent2_occupancy(const hdgnn_config_t& cfg, int nsm, bool bwd) {
    const int cwt = ent2_cwt(cfg.Ne); const void* fn = ent2_fn_rt(cwt, bwd);
    for (int occ = 4; occ > 1; --occ) {
        int G, R, got = 0;
        ent2_grid(cfg.max_batch, cfg.Ne, occ, nsm, &G, &R);
        const size_t smem = ent2_smem_bytes(cwt, cfg.Ne, R, bit_words(cfg.Ne), bwd);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&got, fn, KG * 32, smem) == cudaSuccess && got >= occ) return occ;
    }
    return 1;
}

Ent2Args ent2_args(hdgnn_handle_t h, int B, const Inputs& in) {
    Ent2Args a{};
    a.bits = in.ebits; a.WP = h->WPe; a.N = h->Ne; a.B = B;
    a.params = in.params; a.x = in.x;
    a.o_u = h->po.ent_w1; a.o_v = h->po.ent_w1 + HD; a.o_b = h->po.ent_b1; a.o_l = h->po.ent_w1 + 2 * HD;
    return a;
}

int debug_scatter(hdgnn_handle_t h, int B, cudaStream_t st) {
    const size_t Ne = h->Ne, Nc = h->Nc, T = Nc * HD, stride = mid2_dbg_floats(h->Ne, h->Nc) * 4;
    const char* src = (const char*)h->ws[WS_DBG].p;
    struct { WsId id; size_t off, n; } parts[] = {
        {WS_S1, 0, Ne * HD}, {WS_X2, Ne * HD, Ne}, {WS_NB, Ne * 21, Nc * 4}, {WS_RS3, Ne * 21 + Nc * 4, T},
        {WS_CS3F, Ne * 21 + Nc * 4 + T, T}, {WS_PR, Ne * 21 + Nc * 4 + 2 * T, T}, {WS_PC, Ne * 21 + Nc * 4 + 3 * T, T},
        {WS_DNB, Ne * 21 + Nc * 4 + 4 * T, Nc * 4}, {WS_DX2, Ne * 21 + Nc * 8 + 4 * T, Ne}};
    for (auto& p : parts)
        CK(h, cudaMemcpy2DAsync(h->ws[p.id].p, p.n * 4, src + p.off * 4, stride, p.n * 4, B, cudaMemcpyDeviceToDevice, st));
    return HDGNN_OK;
}

// Byte grids adj / Y -> the label bitmaps of the step, in.ebits / in.ybits: a staging slot's bitmap sections when the host
// entry points stage them, else the next of the two alternating EBITS / YBITS buffers (pack_bits may overlap the previous
// step's last kernel, pack.cuh).
int pack_step(hdgnn_handle_t h, int B, const uint8_t* adj, const uint8_t* Y, Inputs& in, cudaStream_t st) {
    if (!in.ebits) {
        h->bslot ^= 1;
        in.ebits = (const uint32_t*)h->ws[WS_EBITS0 + h->bslot].p;
        in.ybits = (const uint32_t*)h->ws[WS_YBITS0 + h->bslot].p;
    }
    PackArgs p{};
    p.adj = adj; p.Ne = h->Ne; p.pe = h->pe; p.WPe = h->WPe; p.ebits = const_cast<uint32_t*>(in.ebits);
    p.Y = Y; p.Nc = h->Nc; p.pc = h->pc; p.WPc = h->WPc; p.ybits = const_cast<uint32_t*>(in.ybits);
    p.B = B;
    const long long rows = (long long)B * (h->Ne + h->Nc);
    PROF_BEGIN(h, st);
    if (h->pe <= 256 && h->pc <= 256) launch_ex(pack_bits_kernel<16>, (int)((rows + 15) / 16), 256, 0, st, h->plan.pdl, p);
    else launch_ex(pack_bits_kernel<32>, (int)((rows + 7) / 8), 256, 0, st, h->plan.pdl, p);
    LAUNCH_CHECK(h, "pack_bits", st);
    return HDGNN_OK;
}

// head: no pack_bits in front of the step.  Its first kernel then follows the previous step's optimizer kernel directly and
// reads the weights it updates: ent_fwd2 defers those loads behind its pdl_wait (Ent2Args::head), mid2 is launched normally
int fused_forward(hdgnn_handle_t h, int B, int B_global, const Inputs& in, float* logits, float* probs, bool train, bool head,
                  cudaStream_t st) {
    const FusedPlan& P = h->plan; const Mid2Mode& md = P.mode[train];
    int G, R = 0, SL = 0;       // grid and row chunks of ent_fwd2, which mid2 reads back
    if (P.dense) {
        Ent2Args a = ent2_args(h, B, in);
        ent2_grid(B, h->Ne, P.fwd_occ, h->nsm, &G, &R);
        SL = ent2_max_slots(h->Ne, R);
        a.R = R; a.SL = SL; a.RS = F(h, WS_RS1); a.CSp = F(h, WS_CS1P); a.head = head ? 1 : 0;
        const size_t smem = ent2_smem_bytes(h->cwt, h->Ne, R, h->WPe, false);
        PROF_BEGIN(h, st);
        launch_ent2(h->cwt, false, G, smem, st, a, P.pdl);
        LAUNCH_CHECK(h, "ent_fwd", st);
    }
    Mid2Args m{};
    m.Ne = h->Ne; m.Nc = h->Nc; m.ent = h->ent ? 1 : 0; m.R = R; m.SL = SL;
    m.ebits = in.ebits; m.WPe = h->WPe;
    m.ybits = in.ybits; m.WPc = h->WPc;
    m.x = in.x; m.hmap = in.hmap; m.L = in.L;
    m.params = in.params; m.po = h->po; m.RS1 = F(h, WS_RS1); m.CS1p = F(h, WS_CS1P);
    m.logits = logits; m.probs = probs; m.cep = F(h, WS_CEP);
    m.scale = 10.f / ((float)B_global * (float)(h->Nc * (h->Nc - 1)));
    m.GE = F(h, WS_GE); m.gpart = F(h, WS_GPART); m.total = h->po.total;
    m.dbg = h->debug ? F(h, WS_DBG) : nullptr;
    m.clk = h->debug ? (long long*)h->ws[WS_CLK].p : nullptr;
    m.dlt_g = md.opt.dlt_smem ? nullptr : F(h, WS_DLT);
    m.scache = md.opt.scache ? 1 : 0;
    m.inl = P.inl ? 1 : 0;
    m.wait_flag = in.wait_flag; m.wait_tag = in.wait_tag;
    m.hits_acc = h->hits_acc;
    m.evc = h->evc;
    m.pred = h->pred;
    m.edge = P.edge ? 1 : 0;
    if (m.edge) { m.RSEg = F(h, WS_RSEG); m.CSEg = F(h, WS_CSEG); m.REg = F(h, WS_REG); m.CEg = F(h, WS_CEG); m.A1F = F(h, WS_A1F); m.PREg = F(h, WS_PREG); }
    m.lay = md.lay;
    m.tabs_g = P.gt ? F(h, WS_TABS) : nullptr;
    // Batches below one wave of SMs: clusters of two CTAs, the `S` costliest commits shared by both CTAs of a cluster (mid2.cuh),
    // as many as there are spare SMs and co-resident clusters
    bool cl = false;
    int grid = B;
    if (md.clusters > 0 && B < h->nsm) {
        int S = B < h->nsm - B ? B : h->nsm - B;
        if (S > 2 * md.clusters - B) S = 2 * md.clusters - B;
        if (S > 0) { cl = true; m.B = B; m.nsplit = S; grid = 2 * (S + (B - S + 1) / 2); }
    }
    PROF_BEGIN(h, st);
    // inline entity stage: this kernel reads the weights after its pdl_wait, so it may follow the previous step's optimizer
    // kernel (or pack_bits) under programmatic dependent launch; otherwise PDL only behind ent_fwd2
    launch_mid2(h->CWc, train, P.gt, cl, grid, md.smem, st, m, P.pdl && (h->ent || P.inl));
    LAUNCH_CHECK(h, train ? "mid(train)" : "mid(infer)", st);
    if (h->debug) return debug_scatter(h, B, st);
    return HDGNN_OK;
}

int fused_backward(hdgnn_handle_t h, int B, int B_global, const Inputs& in, float* loss, float* grads,
                   const AdamArgs* adam, cudaStream_t st) {
    const FusedPlan& P = h->plan;
    int G = 0, R;               // grid (reduce_adam adds its gradient partials) and row chunks of ent_bwd2
    if (P.dense) {
        Ent2Args a = ent2_args(h, B, in);
        ent2_grid(B, h->Ne, P.bwd_occ, h->nsm, &G, &R);
        a.R = R; a.SL = 0; a.GR = F(h, WS_GE); a.GC = F(h, WS_GE); a.gpart = F(h, WS_GPE);
        const size_t smem = ent2_smem_bytes(h->cwt, h->Ne, R, h->WPe, true);
        PROF_BEGIN(h, st);
        launch_ent2(h->cwt, true, G, smem, st, a, P.pdl);
        LAUNCH_CHECK(h, "ent_bwd", st);
    }
    FinalArgs f{};
    f.B = B; f.total = h->po.total; f.gpart = F(h, WS_GPART);
    if (P.dense) f.ent = {F(h, WS_GPE), G, h->po.ent_w1, h->po.ent_w1 + HD, h->po.ent_b1, h->po.ent_w1 + 2 * HD};
    f.cep = F(h, WS_CEP); f.ncep = B; f.loss_denom = (float)B_global * (float)(h->Nc * (h->Nc - 1)); f.loss = loss;
    f.grads = grads;
    f.l2part = F(h, WS_FIN_L2); f.counter = (unsigned int*)h->ws[WS_FIN_CNT].p;
    if (adam) {
        f.apply_adam = 1; f.params = adam->params; f.m = adam->m; f.v = adam->v; f.step = adam->step;
        f.o_t1 = h->po.theta1; f.o_t2 = h->po.theta2; f.lr = adam->lr; f.b1 = adam->b1; f.b2 = adam->b2; f.eps = adam->eps;
        f.reg_losses = adam->reg;
        if (adam->peer) f.peer = h->peer;
    }
    PROF_BEGIN(h, st);
    launch_ex(reduce_adam_kernel, (h->po.total + FIN_P - 1) / FIN_P, FIN_P * FIN_SL, 0, st, P.pdl, f);
    LAUNCH_CHECK(h, adam ? (adam->peer ? "reduce_allreduce_adam(peer)" : "reduce_adam") : "grad_reduce", st);
    return HDGNN_OK;
}

// Byte offsets of the five inputs of a batch of B commits, labels as bitmaps, inside one staging block (every section starts
// at the next multiple of 16 bytes).  Host buffers laid out the same way travel in ONE DMA (stage_inputs).
struct WireOff { size_t eb, yb, x, hm, L, total; };
WireOff wire_layout(const hdgnn_handle_s* h, int B) {
    WireOff w{};
    size_t o = 0;
    auto take = [&](size_t n) { const size_t r = o; o += (n + 15) & ~(size_t)15; return r; };
    w.eb = take((size_t)B * h->Ne * h->WPe * 4); w.yb = take((size_t)B * h->Nc * h->WPc * 4);
    w.x = take((size_t)B * h->Ne * 4); w.hm = take((size_t)B * h->Ne * 4); w.L = take((size_t)B * 4);
    w.total = o;
    return w;
}

int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return v && *v ? atoi(v) : dflt;
}

// The form of the fused path for a handle: first, from the shapes and the flags alone, which modes fit one SM's `optin` bytes
// of shared memory, and how; then the kernels' shared-memory opt-in and their co-residency on `nsm` SMs.  The fused path needs
// the per-commit state of mid2 in one SM's shared memory and a hunk grid of <= 8 segments (forward only: <= 16).  The twelve
// hunk-stage tables (12 Nc 20 floats) either sit in shared memory (compiled for Nc <= 160) or in a per-commit slice of global
// memory (compiled for Nc > 128: mid2_kernel<.., GT>); the placement that admits the inline entity stage wins, shared memory on
// a tie.
FusedPlan plan_fused(const hdgnn_config_t& cfg, int optin, int nsm, cudaError_t* err) {
    const int Ne = cfg.Ne, Nc = cfg.Nc, cwc = (Nc + 31) / 32;
    const bool ent = cfg.variant == 2 || cfg.variant == 4, edge = cfg.variant == 4;
    const size_t lim = (size_t)optin;
    const bool tr = Nc <= 256;      // above 256 hunks only the forward kernel exists (BASELINE config 5: the inference sweep)
    auto fits = [&](const Mid2Opts& o) { return mid2_smem_bytes(Ne, Nc, o) <= lim; };
    // mid2 with its hunk-stage tables placed as `gt` says, in the layout it must fit: training, or forward only above 256 hunks.
    // opt.scache: S also fits beside the rest for the training kernel's backward
    struct Place { bool fused = false; Mid2Opts opt; };
    auto place = [&](bool gt) {
        Place p;
        if ((cfg.flags & HDGNN_F_LEGACY) || (!tr && edge) || !mid2_gt_supported(cwc, gt)) return p;
        Mid2Opts& o = p.opt; o.train = tr; o.gt = gt;
        // per-commit state of mid2 in one SM; the per-pair dL/dlogit table may spill to HBM (L2-resident)
        o.dlt_smem = !tr || fits(o);
        p.fused = fits(o);
        Mid2Opts s = o; s.scache = true;
        o.scache = ent && p.fused && fits(s);
        if (p.fused && ent && !(cfg.flags & HDGNN_F_DENSE_SWEEP)) {
            // entity pair layer inside mid2 (sorted prefix sums + edge walk) when its extra state fits beside mid2's: with the
            // dL/dlogit table in shared memory, else in HBM, else (global tables only) with the S / GE rows in global memory as
            // well (Ne = 512 beside Nc = 256)
            Mid2Opts i = o; i.inl = i.scache = true;
            Mid2Opts d = i; d.dlt_smem = false;
            Mid2Opts g = i; g.dlt_smem = !tr; g.scg = true;
            if (fits(i)) o = i;
            else if (tr && fits(d)) o = d;
            else if (gt && fits(g)) o = g;
        }
        return p;
    };
    const Place ps = place(false), pg = place(true);
    Place pp = pg.fused && (!ps.fused || (pg.opt.inl && !ps.opt.inl)) ? pg : ps;
    bool edge_train = false;
    if (edge && pp.fused) {
        // variant 4 on the fused path: needs the inline entity stage and room for the edge branch in mid2's union region, with
        // the dL/dlogit table in HBM if need be
        Mid2Opts& o = pp.opt; o.edge = o.dlt_smem = true;
        o.dlt_smem = fits(o);
        const Mid2Smem L = mid2_layout(Ne, Nc, o);
        pp.fused = o.inl && mid2_smem_bytes(L) <= lim && mid2_edge_fwd_fits(Ne, L);
        edge_train = pp.fused && mid2_edge_bwd_fits(Ne, L);
    }
    FusedPlan P;
    P.pdl = !(cfg.flags & HDGNN_F_DEBUG);
    cudaError_t& e = *err = cudaSuccess;
    if (!pp.fused) return P;
    P.gt = pp.opt.gt; P.inl = pp.opt.inl; P.edge = edge;
    P.dense = ent && !P.inl; P.mid2_first = !P.dense;
    auto resolve = [&](Mid2Mode& md, bool fused, const Mid2Opts& o) {
        md.fused = fused; md.opt = mid2_normalize(o); md.lay = mid2_layout(Ne, Nc, md.opt); md.smem = mid2_smem_bytes(md.lay);
    };
    Mid2Opts f = pp.opt; f.train = false; f.dlt_smem = true; f.scache = false;
    Mid2Opts t = pp.opt; t.train = true;
    resolve(P.mode[0], true, f);
    resolve(P.mode[1], tr && (!edge || edge_train), t);

    const cudaFuncAttribute A = cudaFuncAttributeMaxDynamicSharedMemorySize;
    auto acc = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    if (P.mode[1].fused) acc(cudaFuncSetAttribute(mid2_fn_rt(cwc, true, P.gt), A, optin));
    acc(cudaFuncSetAttribute(mid2_fn_rt(cwc, false, P.gt), A, optin));
    // cluster form: shared-memory tables, at most 128 hunks, no global side outputs of the entity stage, not variant 4, not the
    // debug dumps
    if (!P.gt && cwc <= 4 && P.mid2_first && !P.edge && !(cfg.flags & HDGNN_F_DEBUG) && env_int("HDGNN_CLUSTER", 1) != 0) {
        acc(cudaFuncSetAttribute(mid2_fn_rt(cwc, true, false, true), A, optin));
        acc(cudaFuncSetAttribute(mid2_fn_rt(cwc, false, false, true), A, optin));
        if (e == cudaSuccess) {
            const int ct = mid2_max_clusters(cwc, true, P.mode[1].smem), cf = mid2_max_clusters(cwc, false, P.mode[0].smem);
            if (ct > 0 && cf > 0) { P.mode[1].clusters = ct; P.mode[0].clusters = cf; }
        }
    }
    // the occupancy of the sweeps also sizes CS1P, so it is taken for the inline entity stage as well (variant 4 with a fused
    // forward and multi-kernel training)
    if (ent) {
        const int cwt = ent2_cwt(Ne);
        acc(cudaFuncSetAttribute(ent2_fn_rt(cwt, false), A, optin));
        acc(cudaFuncSetAttribute(ent2_fn_rt(cwt, true), A, optin));
        if (e != cudaSuccess) return P;
        P.fwd_occ = ent2_occupancy(cfg, nsm, false); P.bwd_occ = ent2_occupancy(cfg, nsm, true);
    }
    return P;
}

int pick_rt(int N, int B, int requested) {
    if (requested > 0) return round_up(requested < 4 ? 4 : requested, 4);
    // Aim for >= 2 waves of 148 SMs x 3 resident CTAs while keeping >= 16 rows per CTA so the
    // per-CTA column staging (N x 20 floats) is amortised.
    int rt = 32;
    while (rt > 16 && (long)B * ((N + rt - 1) / rt) < 2 * 148 * 3) rt -= 4;
    if (rt > round_up(N, 4)) rt = round_up(N, 4);
    return rt;
}

// Bytes of each workspace buffer of a handle, 0 for a buffer it does not have: a function of its configuration, its plan and the
// sizes derived from them, without CUDA calls.  PEER_SEQ and PEER_STAMPS are 0 here (hdgnn_peer_attach).
std::array<size_t, WS_COUNT> workspace_bytes(const hdgnn_handle_s& h) {
    const FusedPlan& P = h.plan;
    const bool fused = P.mode[0].fused;       // the forward is fused whenever the training step is
    const int Gf_max = fused && h.ent ? P.fwd_occ * h.nsm : 0, Gb_max = fused && h.ent ? P.bwd_occ * h.nsm : 0;
    const size_t B = h.cfg.max_batch, Ne = h.Ne, Nc = h.Nc, Se = h.Se, Sc = h.Sc, f = sizeof(float);
    // (B, SL, Ne, 20) column partials of ent_fwd2: B * SL <= grid + 2 B for every batch size <= max_batch
    const size_t cs1p_f = ((size_t)Gf_max + 2 * B + 2) * Ne * HD * f, cs1p_l = B * Se * Ne * HD * f;
    const bool mixed = fused && !P.mode[1].fused;        // variant 4: fused forward, multi-kernel training
    const size_t cs1p = !fused ? cs1p_l : (mixed && cs1p_l > cs1p_f ? cs1p_l : cs1p_f);
    const bool lg = !P.mode[1].fused;     // buffers only the multi-kernel path needs (kept when debugging: dump targets)
    const bool dbgbuf = lg || h.debug;
    // the entity state in HBM: RS1 / CS1P and GE on the multi-kernel path and beside the dense sweeps.  The inline entity stage
    // keeps S and GE in shared memory; GE holds its S / GE rows when they do not fit there (scg), and the debug dump of GE.
    const bool ent_g = h.ent && (P.dense || lg);
    const bool ge = dbgbuf || (h.ent && (P.dense || P.mode[0].lay.scg || P.mode[1].lay.scg));
    const struct { WsId id; size_t bytes; bool need; } rows[] = {
        {WS_RS1, B * Ne * HD * f, ent_g}, {WS_CS1P, cs1p, ent_g}, {WS_S1, B * Ne * HD * f, dbgbuf},
        {WS_X2, B * Ne * f, dbgbuf}, {WS_NB, B * Nc * 4 * f, dbgbuf}, {WS_PH, B * Nc * HD * f, lg}, {WS_QH, B * Nc * HD * f, lg},
        {WS_RS3, B * Nc * HD * f, dbgbuf}, {WS_CS3P, B * Sc * Nc * HD * f, lg}, {WS_CS3F, B * Nc * HD * f, dbgbuf},
        {WS_PR, B * Nc * HD * f, dbgbuf}, {WS_PC, B * Nc * HD * f, dbgbuf}, {WS_CEP, B * Sc * f, true},
        {WS_RSM, B * Nc * HD * f, lg}, {WS_CSMP, B * Sc * Nc * HD * f, lg}, {WS_LSMP, B * Sc * HD * f, lg},
        {WS_HSP, B * Sc * HD * f, lg}, {WS_DSUMP, B * Sc * f, lg},
        {WS_GRH, B * Nc * HD * f, lg}, {WS_GCH, B * Nc * HD * f, lg},
        {WS_RS3D, B * Nc * HD * f, lg}, {WS_CS3DP, B * Sc * Nc * HD * f, lg}, {WS_LS3P, B * Sc * HD * f, lg},
        {WS_DNB, B * Nc * 4 * f, dbgbuf}, {WS_GE, B * Ne * HD * f, ge}, {WS_DX2, B * Ne * f, dbgbuf},
        {WS_RS1D, B * Ne * HD * f, h.ent && lg}, {WS_CS1DP, B * Se * Ne * HD * f, h.ent && lg}, {WS_LS1P, B * Se * HD * f, h.ent && lg},
        {WS_GPART, 2 * B * (size_t)h.po.total * f, true},       // second half: spare rows of the cluster form (mid2.cuh)
        {WS_GPE, ((size_t)Gb_max + 1) * 4 * HD * f, P.dense}, {WS_FIN_L2, 256 * f, fused}, {WS_FIN_CNT, 16, fused},
        // pack_bits' output for the device entry points taking byte grids
        {WS_EBITS0, B * Ne * (size_t)h.WPe * 4, !h.host_bits}, {WS_EBITS1, B * Ne * (size_t)h.WPe * 4, !h.host_bits},
        {WS_YBITS0, B * Nc * (size_t)h.WPc * 4, !h.host_bits}, {WS_YBITS1, B * Nc * (size_t)h.WPc * 4, !h.host_bits},
        {WS_DBG, B * mid2_dbg_floats(h.Ne, h.Nc) * f, fused && h.debug},
        {WS_CLK, B * 24 * sizeof(long long), fused && h.debug},
        {WS_DLT, B * Nc * (size_t)((h.Nc + 31) / 32 * 32) * f, P.mode[1].fused && !P.mode[1].opt.dlt_smem},
        {WS_TABS, B * (size_t)mid2_tab_floats(h.Nc) * f, fused && P.gt},
        {WS_RSEG, B * Ne * HD * f, P.edge}, {WS_CSEG, B * Ne * HD * f, P.edge}, {WS_REG, B * Ne * HD * f, P.edge},
        {WS_CEG, B * Ne * HD * f, P.edge}, {WS_A1F, B * Ne * (Ne - 1) * f, P.edge}, {WS_PREG, B * Ne * 60 * f, P.edge},
        {WS_RSE, B * Ne * HD * f, h.edge}, {WS_CSEP, B * Se * Ne * HD * f, h.edge}, {WS_CSEF, B * Ne * HD * f, h.edge},
        {WS_PRE, B * Ne * HD * f, h.edge}, {WS_PCE, B * Ne * HD * f, h.edge},
        {WS_SOFT, B * Ne * Ne * 2 * f, h.edge}, {WS_DSOFT, B * Ne * Ne * 2 * f, h.edge},
        {WS_RSME, B * Ne * HD * f, h.edge}, {WS_CSMEP, B * Se * Ne * HD * f, h.edge}, {WS_LSMEP, B * Se * HD * f, h.edge},
        {WS_HSEP, B * Se * HD * f, h.edge}, {WS_DSUMEP, B * Se * f, h.edge},
        {WS_GRE, B * Ne * HD * f, h.edge}, {WS_GCE, B * Ne * HD * f, h.edge},
        {WS_RSED, B * Ne * HD * f, h.edge}, {WS_CSEDP, B * Se * Ne * HD * f, h.edge}, {WS_LSEP, B * Se * HD * f, h.edge},
        // staging slots of the *_host entry points: the wire block [entity bitmaps][hunk bitmaps][x][hmap][L] (16-byte aligned
        // sections), and for byte grids the pitched grids pack_bits reads (+ the un-pitched rows, re-pitched on the device)
        {WS_H_WIRE0, wire_layout(&h, h.cfg.max_batch).total, true}, {WS_H_WIRE1, wire_layout(&h, h.cfg.max_batch).total, true},
        {WS_H_ADJ0, B * Ne * (size_t)h.pe, !h.host_bits}, {WS_H_ADJ1, B * Ne * (size_t)h.pe, !h.host_bits},
        {WS_H_Y0, B * Nc * (size_t)h.pc, !h.host_bits}, {WS_H_Y1, B * Nc * (size_t)h.pc, !h.host_bits},
        {WS_H_ADJ_RAW0, B * Ne * Ne, !h.host_bits && h.pe != h.Ne}, {WS_H_ADJ_RAW1, B * Ne * Ne, !h.host_bits && h.pe != h.Ne},
        {WS_H_Y_RAW0, B * Nc * Nc, !h.host_bits && h.pc != h.Nc}, {WS_H_Y_RAW1, B * Nc * Nc, !h.host_bits && h.pc != h.Nc},
        {WS_H_FLAG, 16, true}, {WS_H_PROBS, B * 2 * Nc * (Nc - 1) * f, true}, {WS_H_LOSS, 4 * f, true}, {WS_H_GRADS, (size_t)h.po.total * f, true},
    };
    std::array<size_t, WS_COUNT> bytes{};
    for (auto& r : rows)
        if (r.need) bytes[r.id] = r.bytes;
    return bytes;
}

}  // namespace

extern "C" {

int hdgnn_param_count(int variant) {
    if (variant < 1 || variant > 4) return HDGNN_E_INVALID;
    return layout(variant).back().second;
}

int hdgnn_param_offset(int variant, const char* name) {
    if (variant < 1 || variant > 4 || !name || !*name) return -1;
    return find_off(layout(variant), name);
}

int hdgnn_pack_label_bits(int N, int n, const uint8_t* grid, int pitch, uint32_t* bits, void* stream) {
    const Call c{"hdgnn_pack_label_bits"};
    if (int rc = c.sizes("N", N, "n", n)) return rc;
    if (pitch < n || (pitch & 15) || pitch > 528) return c.invalid("pitch must be a multiple of 16 in [n, 528]");
    if (int rc = c.pointers({{"grid", grid, 16}, {"bits", bits, 16}})) return rc;
    PackArgs p{};
    p.adj = grid; p.Ne = n; p.pe = pitch; p.WPe = bit_words(n); p.ebits = bits; p.B = N;
    p.Y = nullptr; p.Nc = 0; p.pc = 0; p.WPc = 0; p.ybits = nullptr;
    const long long rows = (long long)N * n;
    if (pitch <= 256) pack_bits_kernel<16><<<(int)((rows + 15) / 16), 256, 0, (cudaStream_t)stream>>>(p);
    else pack_bits_kernel<32><<<(int)((rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(p);
    return c.launched();
}

int hdgnn_bit_words(int n) { return n > 0 && n <= HDGNN_MAX_N ? bit_words(n) : -1; }

int hdgnn_label_pitch(int n) { return n < 1 ? HDGNN_E_INVALID : round_up(n, 16); }

const char* hdgnn_last_error(hdgnn_handle_t h) { return h ? h->err.c_str() : g_error.c_str(); }

int hdgnn_create(const hdgnn_config_t* cfg, hdgnn_handle_t* out) {
    if (!cfg || !out) return fail(nullptr, HDGNN_E_INVALID, "null cfg/out");
    *out = nullptr;
    if (cfg->variant < 1 || cfg->variant > 4) return fail(nullptr, HDGNN_E_INVALID, "variant must be 1..4");
    if (cfg->Ne < 2 || cfg->Nc < 2) return fail(nullptr, HDGNN_E_INVALID, "Ne and Nc must be >= 2");
    if (cfg->Ne > HDGNN_MAX_N || cfg->Nc > HDGNN_MAX_N) return fail(nullptr, HDGNN_E_UNSUPPORTED, "Ne/Nc above HDGNN_MAX_N");
    if (cfg->max_batch < 1) return fail(nullptr, HDGNN_E_INVALID, "max_batch must be >= 1");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return fail(nullptr, HDGNN_E_CUDA, "no CUDA device");
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, HDGNN_E_INVALID, "bad device ordinal");
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess) return fail(nullptr, HDGNN_E_CUDA, "cudaGetDeviceProperties failed");
    if (prop.major != 10) return fail(nullptr, HDGNN_E_UNSUPPORTED, "libhdgnn is built for sm_100a (B200) only");
    if (cudaSetDevice(cfg->device) != cudaSuccess) return fail(nullptr, HDGNN_E_CUDA, "cudaSetDevice failed");

    hdgnn_handle_t h = new hdgnn_handle_s();
    h->cfg = *cfg;
    h->po = make_off(cfg->variant);
    h->Ne = cfg->Ne; h->Nc = cfg->Nc;
    h->pe = round_up(h->Ne, 16); h->pc = round_up(h->Nc, 16);
    h->ent = cfg->variant == 2 || cfg->variant == 4;
    h->edge = cfg->variant == 4;      // model_3's edge branch never reaches the loss (model_3.py:91-97)
    h->ho_hunk = {h->po.hnk_w2, h->po.hnk_b2, h->po.scr_w1, h->po.scr_b1, h->po.scr_w2, h->po.scr_b2};
    h->ho_edge = {h->po.edg_w2, h->po.edg_b2, h->po.eup_w1, h->po.eup_b1, h->po.eup_w2, h->po.eup_b2};
    h->CWe = (h->Ne + 31) / 32; h->CWc = (h->Nc + 31) / 32;
    h->RTe = pick_rt(h->Ne, cfg->max_batch, cfg->rows_per_cta_e);
    h->RTc = pick_rt(h->Nc, cfg->max_batch, cfg->rows_per_cta_c);
    h->Se = (h->Ne + h->RTe - 1) / h->RTe; h->Sc = (h->Nc + h->RTc - 1) / h->RTc;
    h->WPe = bit_words(h->Ne); h->WPc = bit_words(h->Nc);

    const size_t smem_need[] = {pairsum_smem_bytes(h->CWe, h->RTe, 4 * h->WPe, true), score_smem_bytes(h->CWe, h->RTe, 4 * h->WPe, true),
                                pairsum_smem_bytes(h->CWc, h->RTc, 4 * h->WPc, true), score_smem_bytes(h->CWc, h->RTc, 4 * h->WPc, true)};
    for (size_t s : smem_need)
        if (s > (size_t)prop.sharedMemPerBlockOptin) {
            delete h;
            return fail(nullptr, HDGNN_E_UNSUPPORTED, "row tile does not fit in shared memory; lower rows_per_cta");
        }
    h->debug = (cfg->flags & HDGNN_F_DEBUG) != 0;
    h->nsm = prop.multiProcessorCount;
    h->cwt = ent2_cwt(h->Ne);
    cudaError_t e;
    h->plan = plan_fused(*cfg, (int)prop.sharedMemPerBlockOptin, h->nsm, &e);
    h->host_bits = (cfg->flags & HDGNN_F_LABEL_BITS) != 0;
    if (e == cudaSuccess) e = set_attrs(h, (int)prop.sharedMemPerBlockOptin);
    if (e != cudaSuccess) {
        std::string m = std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e);
        delete h;
        return fail(nullptr, HDGNN_E_CUDA, m);
    }
    const std::array<size_t, WS_COUNT> bytes = workspace_bytes(*h);
    for (int i = 0; i < WS_COUNT; ++i) {
        if (!bytes[i]) continue;
        int rc = alloc(h, (WsId)i, bytes[i]);
        if (rc != HDGNN_OK) {
            g_error = h->err;
            hdgnn_destroy(h);
            return rc;
        }
    }
    bool ok = cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking) == cudaSuccess;
    if (ok && cudaHostAlloc((void**)&h->tag_table, 256 * sizeof(uint32_t), cudaHostAllocDefault) == cudaSuccess) {
        for (int i = 0; i < 256; ++i) h->tag_table[i] = (uint32_t)i;
    } else { cudaGetLastError(); h->tag_table = nullptr; }
    for (int i = 0; i < NSLOT && ok; ++i)
        ok = cudaEventCreateWithFlags(&h->ev_copy[i], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&h->ev_done[i], cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
        g_error = "cudaStreamCreate / cudaEventCreate failed";
        hdgnn_destroy(h);
        return HDGNN_E_CUDA;
    }
    *out = h;
    return HDGNN_OK;
}

int hdgnn_destroy(hdgnn_handle_t h) {
    if (!h) return HDGNN_OK;
    cudaSetDevice(h->cfg.device);
    if (h->copy_stream) { cudaStreamSynchronize(h->copy_stream); cudaStreamDestroy(h->copy_stream); }
    for (int i = 0; i < NSLOT; ++i) { if (h->ev_copy[i]) cudaEventDestroy(h->ev_copy[i]); if (h->ev_done[i]) cudaEventDestroy(h->ev_done[i]); }
    for (const Buf& b : h->ws) cudaFree(b.p);
    if (h->tag_table) cudaFreeHost(h->tag_table);
    for (int r = 0; r < PEER_MAX; ++r) if (h->peer_map[r]) cudaIpcCloseMemHandle(h->peer_map[r]);
    if (h->peer_box) cudaFree(h->peer_box);
    delete h;
    return HDGNN_OK;
}

// ---- peer exchange set-up ------------------------------------------------------------------------------------
// mailbox layout (final.cuh): [inbox 2*W*stride u64][lossin 2*W u64]
static void peer_layout(int world, int total, int* stride, int* ncta, size_t* off_loss, size_t* bytes) {
    *ncta = (total + FIN_P - 1) / FIN_P;
    *stride = *ncta * FIN_P;
    *off_loss = (size_t)2 * world * *stride * sizeof(peer_word);
    *bytes = *off_loss + (size_t)2 * world * sizeof(peer_word);
}

int hdgnn_peer_export(hdgnn_handle_t h, int world, unsigned char* ipc_handle_out) {
    if (!h) return HDGNN_E_INVALID;
    if (world < 2 || world > PEER_MAX || !ipc_handle_out) return fail(h, HDGNN_E_INVALID, "world must be 2..8");
    if (!h->plan.mode[1].fused) return fail(h, HDGNN_E_UNSUPPORTED, "the peer exchange is fused into the reduce+Adam kernel of the fused path (Nc <= 256, per-commit state within one SM)");
    static_assert(sizeof(cudaIpcMemHandle_t) == HDGNN_IPC_HANDLE_BYTES, "IPC handle size");
    CK(h, cudaSetDevice(h->cfg.device));
    if (h->peer_box) return fail(h, HDGNN_E_INVALID, "hdgnn_peer_export was already called on this handle");
    int stride, ncta; size_t ol, bytes;
    peer_layout(world, h->po.total, &stride, &ncta, &ol, &bytes);
    CK(h, cudaMalloc(&h->peer_box, bytes));
    CK(h, cudaMemset(h->peer_box, 0, bytes));
    CK(h, cudaDeviceSynchronize());
    h->peer_bytes = bytes; h->peer_world = world;
    cudaIpcMemHandle_t ih;
    CK(h, cudaIpcGetMemHandle(&ih, h->peer_box));
    memcpy(ipc_handle_out, &ih, sizeof(ih));
    return HDGNN_OK;
}

int hdgnn_peer_attach(hdgnn_handle_t h, int rank, int world, const unsigned char* ipc_handles) {
    if (!h) return HDGNN_E_INVALID;
    if (!h->peer_box || world != h->peer_world) return fail(h, HDGNN_E_INVALID, "call hdgnn_peer_export(world) first");
    if (rank < 0 || rank >= world || !ipc_handles) return fail(h, HDGNN_E_INVALID, "bad rank / handles");
    if (h->peer_ready) return fail(h, HDGNN_E_INVALID, "peers are already attached");
    CK(h, cudaSetDevice(h->cfg.device));
    int rc;
    if (!h->ws[WS_PEER_SEQ].p && (rc = alloc(h, WS_PEER_SEQ, 16))) return rc;      // [0] sequence number, [1] error flag
    int stride, ncta; size_t ol, bytes;
    peer_layout(world, h->po.total, &stride, &ncta, &ol, &bytes);
    PeerArgs pa{};
    pa.world = world; pa.rank = rank; pa.stride = stride; pa.ncta = ncta;
    for (int r = 0; r < world; ++r) {
        void* base = h->peer_box;
        if (r != rank) {
            cudaIpcMemHandle_t ih;
            memcpy(&ih, ipc_handles + (size_t)r * sizeof(ih), sizeof(ih));
            CK(h, cudaIpcOpenMemHandle(&h->peer_map[r], ih, cudaIpcMemLazyEnablePeerAccess));
            base = h->peer_map[r];
        }
        pa.inbox[r] = (peer_word*)base;
        pa.lossin[r] = (peer_word*)((char*)base + ol);
    }
    pa.seq = (int*)h->ws[WS_PEER_SEQ].p;
    pa.error = pa.seq + 1;
    {
        const long long ms = env_int("HDGNN_PEER_TIMEOUT_MS", 20000);
        const long long spins = (ms < 1 ? 1 : ms) * 1000;            // ~1 us per poll after the first 64
        pa.max_spins = spins > 0xfffffff0ll ? 0xfffffff0u : (unsigned int)spins;
    }
    pa.stamps = nullptr;
    if (env_int("HDGNN_PEER_STAMPS", 0)) {
        if (!h->ws[WS_PEER_STAMPS].p && (rc = alloc(h, WS_PEER_STAMPS, 4096 * 2 * sizeof(unsigned long long)))) return rc;
        pa.stamps = (unsigned long long*)h->ws[WS_PEER_STAMPS].p;
    }
    h->peer = pa;
    h->peer_ready = true;
    return HDGNN_OK;
}

int hdgnn_set_hits_accumulator(hdgnn_handle_t h, uint64_t* acc) {
    if (!h) return HDGNN_E_INVALID;
    if (acc && !h->plan.mode[1].fused) return fail(h, HDGNN_E_UNSUPPORTED, "the hit counter lives in the fused per-commit kernel (Nc <= 256, per-commit state within one SM); use hdgnn_eval_counts");
    h->hits_acc = (unsigned long long*)acc;
    return HDGNN_OK;
}

int hdgnn_set_eval_counters(hdgnn_handle_t h, int64_t* counts) {
    if (!h) return HDGNN_E_INVALID;
    if (counts && !h->plan.mode[0].fused) return fail(h, HDGNN_E_UNSUPPORTED, "the evaluation counters live in the fused per-commit kernel; use hdgnn_eval_counts");
    if ((uintptr_t)counts & 7) return fail(h, HDGNN_E_INVALID, "counts must be 8-byte aligned");
    h->evc = (unsigned long long*)counts;
    return HDGNN_OK;
}

int hdgnn_set_predictions(hdgnn_handle_t h, uint32_t* pred) {
    if (!h) return HDGNN_E_INVALID;
    if ((uintptr_t)pred & 15) return fail(h, HDGNN_E_INVALID, "pred must be 16-byte aligned");
    h->pred = pred;
    return HDGNN_OK;
}

int hdgnn_peer_status(hdgnn_handle_t h) {
    if (!h) return HDGNN_E_INVALID;
    if (!h->peer_ready) return HDGNN_OK;
    int flag = 0;
    CK(h, cudaMemcpy(&flag, h->peer.error, sizeof(int), cudaMemcpyDeviceToHost));
    if (flag) return fail(h, HDGNN_E_PEER, "a peer's gradient slice did not arrive within HDGNN_PEER_TIMEOUT_MS: the replicas are out of step");
    return HDGNN_OK;
}

// forward [+ backward [+ adam]] on device-resident inputs: the pack step when adj / Y are byte grids (else null, and `in`
// holds the bitmaps), then the fused or the multi-kernel path.
static int run_step(hdgnn_handle_t h, int B, int B_global, const uint8_t* adj, const uint8_t* Y, Inputs in, float* logits,
                    float* probs, float* loss, float* grads, const AdamArgs* adam, cudaStream_t st) {
    const bool train = grads != nullptr, packed = adj != nullptr;
    int rc;
    if (packed && (rc = pack_step(h, B, adj, Y, in, st))) return rc;
    if (h->plan.mode[train].fused) {
        rc = fused_forward(h, B, B_global, in, logits, probs, train, !packed, st);
        if (rc) return rc;

        if (!train) {
            if (loss) {
                PROF_BEGIN(h, st);
                loss_reduce_kernel<<<1, 256, 0, st>>>(F(h, WS_CEP), B, (float)B_global * (float)(h->Nc * (h->Nc - 1)), loss);
                LAUNCH_CHECK(h, "loss_reduce_kernel", st);
            }
            return HDGNN_OK;
        }
        return fused_backward(h, B, B_global, in, loss, grads, adam, st);
    }
    rc = forward_impl(h, B, B_global, in, logits, probs, loss, train, st);
    if (rc || !train) return rc;
    rc = backward_impl(h, B, in, grads, st);
    if (rc || !adam) return rc;
    return adam_impl(h, adam->params, grads, adam->m, adam->v, adam->step, adam->lr, adam->b1, adam->b2, adam->eps,
                     adam->reg, st);
}

// the step of a device entry point whose arguments have been checked
static int device_step(hdgnn_handle_t h, int B, int B_global, const uint8_t* adj, const float* x, const int32_t* hmap,
                       const int32_t* L, const uint8_t* Y, const float* params, float* logits, float* probs, float* loss,
                       float* grads, const AdamArgs* adam, void* stream) {
    h->launches = 0;
    if (h->host_bits) {         // HDGNN_F_LABEL_BITS: adj / Y are the bitmaps
        const Inputs in{(const uint32_t*)adj, (const uint32_t*)Y, x, hmap, L, params};
        return run_step(h, B, B_global, nullptr, nullptr, in, logits, probs, loss, grads, adam, (cudaStream_t)stream);
    }
    const Inputs in{nullptr, nullptr, x, hmap, L, params};
    return run_step(h, B, B_global, adj, Y, in, logits, probs, loss, grads, adam, (cudaStream_t)stream);
}

// the peer-exchange steps: peers attached, equal shards
static int check_peer(hdgnn_handle_t h, int B, int B_global) {
    if (!h->peer_ready) return fail(h, HDGNN_E_INVALID, "hdgnn_peer_attach has not been called");
    if (B_global != B * h->peer.world) return fail(h, HDGNN_E_INVALID, "B_global must be B * world (equal shards)");
    return HDGNN_OK;
}

int hdgnn_forward(hdgnn_handle_t h, int B, const uint8_t* adj, int adj_pitch, const float* x, const int32_t* hmap,
                  const int32_t* L, const uint8_t* Y, int y_pitch, const float* params, float* logits, float* probs,
                  float* loss, void* stream) {
    int rc = check_inputs(h, B, adj, adj_pitch, x, hmap, L, Y, y_pitch, params);
    if (rc) return rc;
    return device_step(h, B, B, adj, x, hmap, L, Y, params, logits, probs, loss, nullptr, nullptr, stream);
}

int hdgnn_forward_backward(hdgnn_handle_t h, int B, int B_global, const uint8_t* adj, int adj_pitch, const float* x,
                           const int32_t* hmap, const int32_t* L, const uint8_t* Y, int y_pitch, const float* params,
                           float* logits, float* probs, float* loss, float* grads, void* stream) {
    int rc = check_inputs(h, B, adj, adj_pitch, x, hmap, L, Y, y_pitch, params);
    if (rc) return rc;
    if (!grads) return fail(h, HDGNN_E_INVALID, "grads is null");
    if (B_global < B) return fail(h, HDGNN_E_INVALID, "B_global < B");
    return device_step(h, B, B_global, adj, x, hmap, L, Y, params, logits, probs, loss, grads, nullptr, stream);
}

int hdgnn_adam_step(hdgnn_handle_t h, float* params, const float* grads, float* m, float* v, int32_t* step_counter,
                    float lr, float beta1, float beta2, float eps, float* reg_losses, void* stream) {
    if (!h) return HDGNN_E_INVALID;
    if (!params || !grads || !m || !v || !step_counter) return fail(h, HDGNN_E_INVALID, "null pointer");
    h->launches = 0;
    return adam_impl(h, params, grads, m, v, step_counter, lr, beta1, beta2, eps, reg_losses, (cudaStream_t)stream);
}

int hdgnn_train_step(hdgnn_handle_t h, int B, const uint8_t* adj, int adj_pitch, const float* x, const int32_t* hmap,
                     const int32_t* L, const uint8_t* Y, int y_pitch, float* params, float* m, float* v,
                     int32_t* step_counter, float lr, float beta1, float beta2, float eps, float* logits, float* probs,
                     float* loss3, void* stream) {
    int rc = check_inputs(h, B, adj, adj_pitch, x, hmap, L, Y, y_pitch, params);
    if (rc) return rc;
    if (!m || !v || !step_counter || !loss3) return fail(h, HDGNN_E_INVALID, "null pointer");
    const AdamArgs ad{params, m, v, step_counter, lr, beta1, beta2, eps, loss3 + 1};
    return device_step(h, B, B, adj, x, hmap, L, Y, params, logits, probs, loss3, F(h, WS_H_GRADS), &ad, stream);
}

// Host buffers -> staging slot `h->cur` (un-pitched rows are re-pitched on the device).  Outside stream capture the
// copies run on the handle's copy stream: slot s is reused only after the kernels that read it (two calls ago)
// have finished, and the step waits for the copies (an event, or the tag mid2 polls), so consecutive calls overlap copy
// and compute.
static int stage_inputs(hdgnn_handle_t h, int B, const uint8_t* adj_host, const float* x_host, const int32_t* hmap_host,
                        const int32_t* L_host, const uint8_t* Y_host, bool train, cudaStream_t st) {
    const size_t Ne = h->Ne, Nc = h->Nc;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cap);
    const bool side = cap == cudaStreamCaptureStatusNone;
    const int slot = h->slot;
    h->cur = slot;
    h->slot = slot ^ 1;
    cudaStream_t cs = side ? h->copy_stream : st;
    if (side && h->done_valid[slot]) CK(h, cudaStreamWaitEvent(cs, h->ev_done[slot], 0));
    h->cur_B = B;
    // one wire block per slot (wire_layout).  Host bitmaps that already sit back to back with x, hmap and L in that layout
    // (one pinned block, what HostBatch builds) are copied with a single DMA, anything else section by section.  Byte grids
    // go to the slot's pitched buffers instead, and pack_bits fills the block's bitmap sections from them (pack_step).
    const WireOff W = wire_layout(h, B);
    char* base = (char*)h->ws[WS_H_WIRE0 + slot].p;
    const char* hb = (const char*)adj_host;
    const bool whole = h->host_bits && (const char*)Y_host == hb + W.yb && (const char*)x_host == hb + W.x &&
                       (const char*)hmap_host == hb + W.hm && (const char*)L_host == hb + W.L;
    if (whole) {
        CK(h, cudaMemcpyAsync(base, hb, W.L + (size_t)B * 4, cudaMemcpyHostToDevice, cs));
    } else if (h->host_bits) {
        CK(h, cudaMemcpyAsync(base + W.eb, adj_host, (size_t)B * Ne * h->WPe * 4, cudaMemcpyHostToDevice, cs));
        CK(h, cudaMemcpyAsync(base + W.yb, Y_host, (size_t)B * Nc * h->WPc * 4, cudaMemcpyHostToDevice, cs));
    } else {
        const uint8_t* srcs[2] = {adj_host, Y_host};
        const WsId raw[2] = {WS_H_ADJ_RAW0, WS_H_Y_RAW0}, dstn[2] = {WS_H_ADJ0, WS_H_Y0};
        const size_t n[2] = {Ne, Nc};
        const int pitch[2] = {h->pe, h->pc};
        for (int t = 0; t < 2; ++t) {
            const size_t rows = (size_t)B * n[t];
            void* dst = h->ws[dstn[t] + slot].p;
            if (pitch[t] == (int)n[t]) {
                CK(h, cudaMemcpyAsync(dst, srcs[t], rows * n[t], cudaMemcpyHostToDevice, cs));
            } else {
                void* rawp = h->ws[raw[t] + slot].p;
                CK(h, cudaMemcpyAsync(rawp, srcs[t], rows * n[t], cudaMemcpyHostToDevice, cs));
                const size_t work = rows * (size_t)pitch[t] / 4;
                int blocks = (int)((work + 255) / 256);
                if (blocks > 148 * 8) blocks = 148 * 8;
                PROF_BEGIN(h, cs);
                repitch_kernel<<<blocks, 256, 0, cs>>>((const uint8_t*)rawp, (uint8_t*)dst, rows, (int)n[t], pitch[t]);
                LAUNCH_CHECK(h, "repitch_kernel", cs);
            }
        }
    }
    if (!whole) {
        CK(h, cudaMemcpyAsync(base + W.x, x_host, (size_t)B * Ne * sizeof(float), cudaMemcpyHostToDevice, cs));
        CK(h, cudaMemcpyAsync(base + W.hm, hmap_host, (size_t)B * Ne * sizeof(int32_t), cudaMemcpyHostToDevice, cs));
        CK(h, cudaMemcpyAsync(base + W.L, L_host, (size_t)B * sizeof(int32_t), cudaMemcpyHostToDevice, cs));
    }
    h->cur_tag = -1;
    if (side) {
        if (h->tag_table && h->host_bits && h->plan.mode[train].fused && h->plan.mid2_first) {
            // mid2 is the first kernel of the step and reads every staged input: order it by a tag instead of an event
            const int tag = (int)(++h->slot_uses[slot] & 0xffu);
            CK(h, cudaMemcpyAsync((int*)h->ws[WS_H_FLAG].p + slot, h->tag_table + tag, sizeof(int), cudaMemcpyHostToDevice, cs));
            h->cur_tag = tag;
        } else {
            CK(h, cudaEventRecord(h->ev_copy[slot], cs));
            CK(h, cudaStreamWaitEvent(st, h->ev_copy[slot], 0));
        }
    }
    return HDGNN_OK;
}

// Device-side views of the staging slot filled by the last stage_inputs call: the sections of its wire block, and, for byte
// grids, the pitched grids (*adj, *Y; null with HDGNN_F_LABEL_BITS) that the pack step turns into the block's bitmaps.
static Inputs staged_inputs(hdgnn_handle_t h, const float* params, const uint8_t** adj, const uint8_t** Y) {
    const int s = h->cur;
    const WireOff W = wire_layout(h, h->cur_B);
    const char* base = (const char*)h->ws[WS_H_WIRE0 + s].p;
    Inputs in{(const uint32_t*)(base + W.eb), (const uint32_t*)(base + W.yb), (const float*)(base + W.x),
              (const int32_t*)(base + W.hm), (const int32_t*)(base + W.L), params};
    if (h->cur_tag >= 0) { in.wait_flag = (const int*)h->ws[WS_H_FLAG].p + s; in.wait_tag = h->cur_tag; }
    *adj = h->host_bits ? nullptr : (const uint8_t*)h->ws[WS_H_ADJ0 + s].p;
    *Y = h->host_bits ? nullptr : (const uint8_t*)h->ws[WS_H_Y0 + s].p;
    return in;
}

// the kernels reading slot h->cur have been enqueued on `st`: the slot may be refilled once they are done
static int release_slot(hdgnn_handle_t h, cudaStream_t st) {
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cap);
    if (cap != cudaStreamCaptureStatusNone) return HDGNN_OK;
    CK(h, cudaEventRecord(h->ev_done[h->cur], st));
    h->done_valid[h->cur] = true;
    return HDGNN_OK;
}

// A pinned (page-locked, UVA-mapped) host buffer can be written by the kernels directly: the three loss floats then
// need no device->host copy at the end of the step (a 12-byte DMA costs several microseconds of stream time and
// breaks the launch overlap with the next step).  Returns the device-visible alias or nullptr.
static float* host_alias(float* host_ptr) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, host_ptr) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    if (at.type != cudaMemoryTypeHost || !at.devicePointer) return nullptr;
    return (float*)at.devicePointer;
}

// argument checks every *_host entry point makes
static int check_host_inputs(hdgnn_handle_t h, int B, const void* adj_host, const void* x_host, const void* hmap_host,
                             const void* L_host, const void* Y_host, const void* params) {
    if (!h) return HDGNN_E_INVALID;
    if (B < 1 || B > h->cfg.max_batch) return fail(h, HDGNN_E_INVALID, "B out of range [1, max_batch]");
    if (!adj_host || !x_host || !hmap_host || !L_host || !Y_host || !params) return fail(h, HDGNN_E_INVALID, "null pointer");
    return HDGNN_OK;
}

// The step of a *_host entry point whose arguments have been checked: stage the host inputs, run the step on the staging
// slot, release the slot, copy the outputs out.
//   to_host = false: probs / loss are device buffers the kernels write;
//   to_host = true:  probs (may be null) and loss are host buffers, filled from H_PROBS / H_LOSS after the step -- except that
//                    the fused optimizer step (reduce_adam; the peer steps always take it) stores the loss floats straight
//                    into a pinned `loss` (host_alias).
// After an optimizer step `loss` holds three floats (the loss, then the two regularisers, adam->reg), else one.
static int host_step(hdgnn_handle_t h, int B, int B_global, const uint8_t* adj_host, const float* x_host,
                     const int32_t* hmap_host, const int32_t* L_host, const uint8_t* Y_host, const float* params,
                     float* probs, float* loss, float* grads, const AdamArgs* adam, bool to_host, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    h->launches = 0;
    int rc = stage_inputs(h, B, adj_host, x_host, hmap_host, L_host, Y_host, grads != nullptr, st);
    if (rc) return rc;
    const uint8_t *adj, *Y;
    const Inputs in = staged_inputs(h, params, &adj, &Y);
    float* probs_d = to_host && probs ? F(h, WS_H_PROBS) : probs;
    float* alias = to_host && adam && h->plan.mode[1].fused ? host_alias(loss) : nullptr;
    float* loss_d = to_host ? (alias ? alias : F(h, WS_H_LOSS)) : loss;
    AdamArgs ad{};
    if (adam) { ad = *adam; ad.reg = loss_d + 1; }
    rc = run_step(h, B, B_global, adj, Y, in, nullptr, probs_d, loss_d, grads, adam ? &ad : nullptr, st);
    if (rc) return rc;
    if ((rc = release_slot(h, st)) || !to_host) return rc;
    if (probs)
        CK(h, cudaMemcpyAsync(probs, probs_d, (size_t)B * 2 * h->Nc * (h->Nc - 1) * sizeof(float), cudaMemcpyDefault, st));
    if (loss && !alias) CK(h, cudaMemcpyAsync(loss, loss_d, (adam ? 3 : 1) * sizeof(float), cudaMemcpyDeviceToHost, st));
    return HDGNN_OK;
}

int hdgnn_train_step_host(hdgnn_handle_t h, int B, const uint8_t* adj_host, const float* x_host,
                          const int32_t* hmap_host, const int32_t* L_host, const uint8_t* Y_host, float* params,
                          float* m, float* v, int32_t* step_counter, float lr, float beta1, float beta2, float eps,
                          float* probs_host, float* loss3_host, void* stream) {
    int rc = check_host_inputs(h, B, adj_host, x_host, hmap_host, L_host, Y_host, params);
    if (rc) return rc;
    if (!m || !v || !step_counter || !loss3_host) return fail(h, HDGNN_E_INVALID, "null pointer");
    const AdamArgs ad{params, m, v, step_counter, lr, beta1, beta2, eps, nullptr};
    return host_step(h, B, B, adj_host, x_host, hmap_host, L_host, Y_host, params, probs_host, loss3_host, F(h, WS_H_GRADS), &ad,
                     true, stream);
}

int hdgnn_train_step_peer(hdgnn_handle_t h, int B, int B_global, const uint8_t* adj, int adj_pitch, const float* x,
                          const int32_t* hmap, const int32_t* L, const uint8_t* Y, int y_pitch, float* params, float* m, float* v,
                          int32_t* step_counter, float lr, float beta1, float beta2, float eps, float* logits, float* probs,
                          float* loss3, void* stream) {
    int rc = check_inputs(h, B, adj, adj_pitch, x, hmap, L, Y, y_pitch, params);
    if (rc) return rc;
    if (!m || !v || !step_counter || !loss3) return fail(h, HDGNN_E_INVALID, "null pointer");
    if ((rc = check_peer(h, B, B_global))) return rc;
    const AdamArgs ad{params, m, v, step_counter, lr, beta1, beta2, eps, loss3 + 1, true};
    return device_step(h, B, B_global, adj, x, hmap, L, Y, params, logits, probs, loss3, F(h, WS_H_GRADS), &ad, stream);
}

int hdgnn_train_step_peer_host(hdgnn_handle_t h, int B, int B_global, const uint8_t* adj_host, const float* x_host,
                               const int32_t* hmap_host, const int32_t* L_host, const uint8_t* Y_host, float* params,
                               float* m, float* v, int32_t* step_counter, float lr, float beta1, float beta2, float eps,
                               float* probs_out, float* loss3_host, void* stream) {
    int rc = check_host_inputs(h, B, adj_host, x_host, hmap_host, L_host, Y_host, params);
    if (rc) return rc;
    if (!m || !v || !step_counter || !loss3_host) return fail(h, HDGNN_E_INVALID, "null pointer");
    if ((rc = check_peer(h, B, B_global))) return rc;
    const AdamArgs ad{params, m, v, step_counter, lr, beta1, beta2, eps, nullptr, true};
    return host_step(h, B, B_global, adj_host, x_host, hmap_host, L_host, Y_host, params, probs_out, loss3_host, F(h, WS_H_GRADS),
                     &ad, true, stream);
}

int hdgnn_forward_backward_host(hdgnn_handle_t h, int B, int B_global, const uint8_t* adj_host, const float* x_host,
                                const int32_t* hmap_host, const int32_t* L_host, const uint8_t* Y_host, const float* params,
                                float* probs, float* loss, float* grads, void* stream) {
    int rc = check_host_inputs(h, B, adj_host, x_host, hmap_host, L_host, Y_host, params);
    if (rc) return rc;
    if (!grads) return fail(h, HDGNN_E_INVALID, "null pointer");
    if (B_global < B) return fail(h, HDGNN_E_INVALID, "B_global < B");
    return host_step(h, B, B_global, adj_host, x_host, hmap_host, L_host, Y_host, params, probs, loss, grads, nullptr, false, stream);
}

int hdgnn_infer_host(hdgnn_handle_t h, int B, const uint8_t* adj_host, const float* x_host, const int32_t* hmap_host,
                     const int32_t* L_host, const uint8_t* Y_host, const float* params, float* probs_host,
                     float* loss_host, void* stream) {
    int rc = check_host_inputs(h, B, adj_host, x_host, hmap_host, L_host, Y_host, params);
    if (rc) return rc;
    return host_step(h, B, B, adj_host, x_host, hmap_host, L_host, Y_host, params, probs_host, loss_host, nullptr, nullptr, true,
                     stream);
}

int hdgnn_workspace(hdgnn_handle_t h, const char* name, void** ptr, size_t* bytes) {
    if (!h || !name) return HDGNN_E_INVALID;
    const Buf* b;
    if (int rc = find_ws(h, name, &b)) return rc;
    if (ptr) *ptr = b->p;
    if (bytes) *bytes = b->bytes;
    return HDGNN_OK;
}

int hdgnn_workspace_copy(hdgnn_handle_t h, const char* name, void* dst, size_t bytes, void* stream) {
    if (!h || !name || !dst) return HDGNN_E_INVALID;
    const Buf* b;
    if (int rc = find_ws(h, name, &b)) return rc;
    if (bytes > b->bytes) return fail(h, HDGNN_E_INVALID, std::string("workspace buffer too small: ") + name);
    CK(h, cudaMemcpyAsync(dst, b->p, bytes, cudaMemcpyDefault, (cudaStream_t)stream));
    return HDGNN_OK;
}

int hdgnn_profile(hdgnn_handle_t h, int enable) {
    if (!h) return HDGNN_E_INVALID;
    for (auto& e : h->prof_ev) { cudaEventDestroy(e.second.first); cudaEventDestroy(e.second.second); }
    h->prof_ev.clear();
    h->prof = enable != 0;
    return HDGNN_OK;
}

int hdgnn_profile_count(hdgnn_handle_t h) { return h ? (int)h->prof_ev.size() : HDGNN_E_INVALID; }

int hdgnn_profile_get(hdgnn_handle_t h, int idx, char* name, int name_cap, float* ms) {
    if (!h || idx < 0 || idx >= (int)h->prof_ev.size() || !ms) return HDGNN_E_INVALID;
    auto& e = h->prof_ev[idx];
    CK(h, cudaEventSynchronize(e.second.second));
    CK(h, cudaEventElapsedTime(ms, e.second.first, e.second.second));
    if (name && name_cap > 0) { strncpy(name, e.first.c_str(), name_cap - 1); name[name_cap - 1] = 0; }
    return HDGNN_OK;
}

int hdgnn_last_launch_count(hdgnn_handle_t h) { return h ? h->launches : HDGNN_E_INVALID; }

}  // extern "C"
