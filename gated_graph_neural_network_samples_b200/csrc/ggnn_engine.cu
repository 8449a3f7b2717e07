// Host side of the GGNN propagation engine + the C ABI declared in include/ggnn_b200.h.
//
// Mirrors the two ChemModel hooks of the reference for this path:
//   ggnn_create / ggnn_set_weights            <- prepare_specific_graph_model        (sparse:63-115, dense:68-91)
//   ggnn_set_graph_* + ggnn_forward           <- compute_final_node_representations  (sparse:117-218, dense:93-117)
// Host work per batch: validate indices, stable counting sort of the type-major message list by
// (target, type) -> CSR, find where the batch can be cut between connected components, pack tiles.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#ifdef _OPENMP
#include <omp.h>
#include <sched.h>
#endif
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/ggnn_b200.h"
#include "ggnn_common.cuh"
#include "ggnn_bwd.cuh"
#include "ggnn_bwd_tc.cuh"
#include "ggnn_readout.cuh"
#include "ggnn_fwd_ffma.cuh"
#include "ggnn_fwd_tc.cuh"
#include "ggnn_fwd_stream.cuh"

using namespace ggnn;

namespace {

std::string g_create_error;

struct DevBuf {
    void* ptr = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (ptr) cudaFree(ptr);
        ptr = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&ptr, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (ptr) cudaFree(ptr); ptr = nullptr; cap = 0; }
};

struct HostPinned {
    void* ptr = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (ptr) cudaFreeHost(ptr);
        ptr = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMallocHost(&ptr, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (ptr) cudaFreeHost(ptr); ptr = nullptr; cap = 0; }
};

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

}  // namespace

struct ggnn_engine {
    // model shape
    int D = 0, T = 0, L = 0;
    int steps[MAX_LAYERS] = {0};
    int nres[MAX_LAYERS] = {0};
    int res[MAX_LAYERS][MAX_RES] = {{0}};
    int step_base[MAX_LAYERS] = {0};
    int total_steps = 0;
    int use_bias = 0, use_avg = 0, cell = 0, act = 0, precision = 0, device = 0;
    int num_sms = 148;
    size_t max_smem = 0;
    bool weights_set = false;
    ggnn_layer_weights w[MAX_LAYERS];

    // batch
    bool graph_set = false;
    int gather_mode = GATHER_SPARSE;
    int V = 0, dense_v = 0;
    int64_t M = 0;
    // plan
    int variant = 0;  // 0: RG=8,CS=1 (64-row tiles)   1: RG=4,CS=2 (32-row tiles)
    int nb1 = 0;
    bool local = false;
    int ntiles = 0;
    int max_span = 0;
    int max_tile_msgs = 0;   // largest number of messages whose target lies in one tile
    std::string plan_text;

    // device memory
    DevBuf graph_buf;   // packed: row_ptr | csr_src | csr_msg | indeg | denom | tile_start | tile_mask | (dense adj)
    HostPinned graph_stage;
    // readout (gated_regression): node -> graph map of the current batch
    DevBuf ro_buf; HostPinned ro_stage; cudaEvent_t ro_stage_done = nullptr;
    int ro_V = -1, ro_G = 0; bool ro_grouped = false, ro_has_mask = false;
    size_t ro_off_graph_of = 0, ro_off_start = 0, ro_off_mask = 0, ro_off_val = 0;
    cudaEvent_t stage_done = nullptr;   // recorded after the staged H2D copy: the next set_graph waits for it before refilling
    size_t off_row_ptr = 0, off_src = 0, off_msg = 0, off_indeg = 0, off_denom = 0, off_tiles = 0, off_mask = 0, off_adj = 0;
    size_t off_trow = 0, off_ttgt = 0;   // source-keyed CSR (rows source*T+type -> targets), built when save_for_backward is on
    bool has_transpose = false;
    int64_t edges_of_type[32] = {0};
    DevBuf state_buf;   // intermediate layer states (L-1) + 2 ping-pong step buffers, each [V][D]
    DevBuf save_bufs;   // 5 (CudnnCompatibleGRUCell: 6) x total_steps x [V][D]
    DevBuf io_buf;      // h0 / h_out staging for ggnn_forward_host
    DevBuf bwd_buf;     // backward scratch
    DevBuf tc_weights;  // pre-split, pre-tiled bf16 copies of the weights (tensor-core path)
    DevBuf tc_respre;   // residual pre-products [ntiles][128][3*DP]
    DevBuf err_flag;    // device int written by kernels on a barrier timeout
    DevBuf dbg_buf;     // optional phase timestamps (GGNN_TC_DEBUG_TIMING=1)
    bool weights_dirty = true;
    int DP = 0;         // hidden size padded to a multiple of 16 (tensor-core path)
    size_t tc_off_edge[MAX_LAYERS] = {0}, tc_off_gate[MAX_LAYERS] = {0}, tc_off_cand[MAX_LAYERS] = {0};
    const float* last_h0 = nullptr;
    float* last_out = nullptr;
    bool save = false;
    bool saved_valid = false;
    // streaming tensor-core plan (ggnn_fwd_stream.cuh): D > 128, or forced with GGNN_TC_STREAM=1
    bool stream = false;
    DevBuf ts_weights, ts_images, ts_u;
    size_t ts_off_edge[MAX_LAYERS] = {0}, ts_off_gate[MAX_LAYERS] = {0}, ts_off_cand[MAX_LAYERS] = {0};
    int ts_nc[2] = {0, 0}, ts_nblk[2] = {0, 0};      // [0]: DP-wide outputs (agg, candidate)  [1]: the 2*DP-wide gate output
    int ts_tiled_nc[2] = {-1, -1};                   // the N-block widths the tiled weights were made for
    size_t off_pair = 0, off_vptr = 0, off_vsrc = 0, off_tvp = 0, off_vinfo = 0;   // streaming plan: (target,type) -> source table, virtual rows (pairs with several messages)
    int ts_nv = 0;                                   // number of virtual rows of the current batch
    DevBuf ts_virt;                                  // their operand image
    int tc_row_budget = 128, tc_kgs = 2048;   // tensor-core plan: no tile has more rows than the budget; <= 64 selects compact operand tiles
    int use_att = 0;                 // use_propagation_attention (sparse:170-196): fp32 path only
    DevBuf att_buf;                  // attention probabilities per target-CSR slot ([steps][M] when saving for backward, else [M])
    size_t off_tslot = 0;            // source-keyed CSR entry -> target-CSR slot (attention backward)
    float drop_keep = 1.0f; unsigned long long drop_seed = 0;          // state dropout for the next forward
    float saved_drop_keep = 1.0f; unsigned long long saved_drop_seed = 0; // ... and what the saved forward used
    int last_launches = 0;
    int bwd_precision = GGNN_PREC_FP32;   // arithmetic of ggnn_backward's GEMMs (ggnn_set_backward_precision), independent of `precision`
    std::vector<int> h_counts, h_diff, h_cursor;   // host scratch of the sparse-graph builder, kept between batches
    struct ggnn_prepared_graph* own_prep = nullptr;   // the prepared graph ggnn_set_graph_sparse builds and uploads from (reused every batch)
    std::string err;

    int fail(int code, const char* fmt, ...) {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof buf, fmt, ap);
        va_end(ap);
        err = buf;
        return code;
    }
};

// The host half of ggnn_set_graph_sparse as an object: `plan` is a shadow engine that carries the model shape in and the batch / tile-plan
// fields out and never touches the device; the packed image (CSR, in-degrees, tiles, streaming tables) sits in pinned memory, or in plain
// memory when no CUDA device is present (host-only construction, CPU test-suite).  Built by a producer thread, uploaded by the engine's
// thread (ggnn_set_graph_prepared) -- the ThreadedIterator overlap of the reference's training loop (chem_tensorflow.py:225, utils.py:16-36).
struct ggnn_prepared_graph {
    ggnn_engine plan;
    HostPinned stage;
    std::vector<char> plain;         // image when !use_cuda
    char* image = nullptr;
    size_t bytes = 0;
    bool use_cuda = true;
    bool valid = false;
    cudaEvent_t uploaded = nullptr;  // recorded after the H2D copy of the image: the next build waits for it before overwriting
};

#define CU_TRY(e, call)                                                                           \
    do {                                                                                          \
        cudaError_t _st = (call);                                                                 \
        if (_st != cudaSuccess) return (e)->fail(GGNN_ECUDA, "%s failed: %s", #call, cudaGetErrorString(_st)); \
    } while (0)

static int ggnn_backward_impl(ggnn_engine* e, const float* d_h_out, const ggnn_layer_grads* grads, int32_t num_layers,
                              float* d_h0, ggnn_stream_t stream);

// ------------------------------------------------------------------------------------------ kernel table
namespace {

typedef void (*FwdKernel)(const FwdParams);

template <int RG, int CS, int NB1, bool LOCAL>
FwdKernel fwd_kernel_ptr() {
    constexpr int NB2 = (2 * NB1 > 8) ? 8 : 2 * NB1;
    constexpr int MINB = (CS == 2 && NB1 <= 2) ? 2 : 1;
    return ggnn_fwd_ffma_kernel<RG, CS, NB1, NB2, LOCAL, MINB>;
}

FwdKernel pick_fwd_kernel(int variant, int nb1, bool local) {
    if (variant == 0) {
        if (nb1 == 1) return local ? fwd_kernel_ptr<8, 1, 1, true>() : fwd_kernel_ptr<8, 1, 1, false>();
        if (nb1 == 2) return local ? fwd_kernel_ptr<8, 1, 2, true>() : fwd_kernel_ptr<8, 1, 2, false>();
        if (nb1 == 4) return local ? fwd_kernel_ptr<8, 1, 4, true>() : fwd_kernel_ptr<8, 1, 4, false>();
    } else {
        if (nb1 == 1) return local ? fwd_kernel_ptr<4, 2, 1, true>() : fwd_kernel_ptr<4, 2, 1, false>();
        if (nb1 == 2) return local ? fwd_kernel_ptr<4, 2, 2, true>() : fwd_kernel_ptr<4, 2, 2, false>();
        if (nb1 == 4) return local ? fwd_kernel_ptr<4, 2, 4, true>() : fwd_kernel_ptr<4, 2, 4, false>();
    }
    return nullptr;
}

int variant_mt(int variant) { return variant == 0 ? 64 : 32; }
int variant_cs(int variant) { return variant == 0 ? 1 : 2; }

int pick_nb1(int variant, int D) {
    const int per = 32 * variant_cs(variant);
    int nb = (D + per - 1) / per;
    if (nb <= 1) return 1;
    if (nb <= 2) return 2;
    if (nb <= 4) return 4;
    return 0;
}

size_t fwd_smem_bytes(int variant, int nb1, int D, int T) {
    const int MT = variant_mt(variant), CS = variant_cs(variant);
    const int nb2 = std::min(8, 2 * nb1);
    const int pw = 32 * nb2 * CS;
    return sizeof(float) * ((size_t)4 * MT * D + (size_t)2 * KC * pw + (size_t)2 * MT * KC + (size_t)T * D);
}

// Decide tile size / mode, then pack tiles greedily between `cuts` (sorted node indices where the batch
// may be split, cuts.front()==0, cuts.back()==V).
int build_plan(ggnn_engine* e, const std::vector<int>& cuts, std::vector<int>& tile_start) {
    const int V = e->V, D = e->D;
    int max_span = 0;
    for (size_t i = 1; i < cuts.size(); ++i) max_span = std::max(max_span, cuts[i] - cuts[i - 1]);
    e->max_span = max_span;
    e->stream = false;
    if (e->precision != GGNN_PREC_FP32) {
        const char* fs = getenv("GGNN_TC_STREAM");
        const char* fgl = getenv("GGNN_FORCE_GLOBAL");
        // a component larger than a tile cannot use the tile-local fused kernel: the streaming plan beats one-launch-per-step of that
        // kernel (cfg5: 0.41 vs 0.57 ms), so it is the default there; GGNN_TC_STREAM=0/1 and GGNN_FORCE_GLOBAL=1 override
        const bool big_component = max_span > tc::TILE_M && e->gather_mode == GATHER_SPARSE && !(fgl && fgl[0] == '1') && !(fs && fs[0] == '0');
        if (e->DP > 128 || big_component || (fs && fs[0] == '1' && e->gather_mode == GATHER_SPARSE)) {
            // streaming plan: fixed 128-row tiles (the gather reads the previous state from L2, so tiles need not respect components),
            // one launch per GEMM of a timestep; N blocks sized so that small batches still spread over the chip
            if (e->gather_mode != GATHER_SPARSE)
                return e->fail(GGNN_EUNSUPPORTED, "hidden_size > 128 on the tensor-core path needs the CSR graph format (a weighted dense adjacency runs on GGNN_PREC_FP32)");
            e->stream = true; e->variant = 3; e->nb1 = 0; e->local = false;
            tile_start.clear(); tile_start.push_back(0);
            for (int r = ts::TILE_M; r < V; r += ts::TILE_M) tile_start.push_back(r);
            if (V > 0) tile_start.push_back(V);
            e->ntiles = (int)tile_start.size() - 1;
            for (int i = 0; i < 2; ++i) {
                const int width = (i + 1) * e->DP;
                int nblk = (width + 255) / 256;
                // a tcgen05.mma costs the same for every N <= 128, so never go below 128 columns per CTA
                while (e->ntiles * nblk <= e->num_sms / 2 && width / (nblk + 1) >= 128) ++nblk;
                e->ts_nblk[i] = nblk;
                e->ts_nc[i] = ((width + nblk - 1) / nblk + 15) / 16 * 16;
            }
            char buf[256];
            int len = snprintf(buf, sizeof buf, "tcgen05-%s STREAM(3 launches per step: gather-GEMM, gate GEMM, candidate GEMM) tiles=%d DP=%d N-blocks agg/cand=%dx%d gate=%dx%d",
                               e->precision == GGNN_PREC_BF16X3 ? "bf16x3" : "bf16", e->ntiles, e->DP, e->ts_nblk[0], e->ts_nc[0], e->ts_nblk[1], e->ts_nc[1]);
            if (e->DP <= 128) snprintf(buf + len, sizeof buf - len, " max_component=%d", max_span);   // (not computed for hidden sizes > 128: fixed tiles)
            e->plan_text = buf;
            return GGNN_OK;
        }
        e->variant = 2;
        e->nb1 = 0;
        e->local = max_span <= tc::TILE_M;
        const char* fg = getenv("GGNN_FORCE_GLOBAL");
        if (fg && fg[0] == '1') e->local = false;
        // Rows per tile: 128 fills the UMMA M dimension, but a small batch then occupies only V/128 SMs and every tile
        // sees every edge type.  When the batch cannot fill the chip, shrink the row budget to the smallest multiple of 8
        // that still fits all tiles in one wave: more SMs, and fewer edge-type blocks per tile (absent types are skipped).
        auto pack = [&](int budget, std::vector<int>& ts) {
            ts.clear(); ts.push_back(0);
            int cur = 0;
            for (size_t i = 1; i < cuts.size(); ++i)
                if (cuts[i] - cur > budget) { ts.push_back(cuts[i - 1]); cur = cuts[i - 1]; }
            if (V > cur) ts.push_back(V);
        };
        int budget = tc::TILE_M;
        if (e->local) {
            pack(tc::TILE_M, tile_start);
            const char* tr = getenv("GGNN_TC_TILE_ROWS");
            if (tr && atoi(tr) >= max_span && atoi(tr) <= tc::TILE_M) { budget = atoi(tr); pack(budget, tile_start); }
            else if ((int)tile_start.size() - 1 < e->num_sms) {
                std::vector<int> trial;
                for (int b = std::max(32, (max_span + 7) / 8 * 8); b < tc::TILE_M; b += 8) {
                    pack(b, trial);
                    if ((int)trial.size() - 1 <= e->num_sms) { budget = b; tile_start = trial; break; }
                }
            }
        } else {
            tile_start.clear(); tile_start.push_back(0);
            for (int r = tc::TILE_M; r < V; r += tc::TILE_M) tile_start.push_back(r);
            if (V > 0) tile_start.push_back(V);
        }
        if (V == 0) tile_start.assign(1, 0);
        e->ntiles = (int)tile_start.size() - 1;
        e->tc_row_budget = e->local ? budget : tc::TILE_M;
        // compact operand tiles when no tile exceeds 64 rows (k-group stride 1024 instead of 2048): half the operand bytes, a ~3x deeper ring
        e->tc_kgs = (e->tc_row_budget <= 64 && !getenv("GGNN_TC_NO_COMPACT")) ? 1024 : 2048;
        char buf[256];
        snprintf(buf, sizeof buf, "tcgen05-%s %s tiles=%d rows/tile<=%d%s DP=%d max_component=%d",
                 e->precision == GGNN_PREC_BF16X3 ? "bf16x3" : "bf16", e->local ? "LOCAL(all layers+steps fused, 1 launch)" : "GLOBAL(1 launch per step)",
                 e->ntiles, budget, e->tc_kgs == 1024 ? " (compact 64-row operand tiles)" : "", e->DP, max_span);
        e->plan_text = buf;
        return GGNN_OK;
    }
    const bool a_ok = pick_nb1(0, D) > 0 && fwd_smem_bytes(0, pick_nb1(0, D), D, e->T) <= e->max_smem;
    const bool b_ok = pick_nb1(1, D) > 0 && fwd_smem_bytes(1, pick_nb1(1, D), D, e->T) <= e->max_smem;
    if (!a_ok && !b_ok) return e->fail(GGNN_EUNSUPPORTED, "hidden_size=%d does not fit any fp32 tile variant", D);
    const char* force = getenv("GGNN_FFMA_VARIANT");
    int variant;
    bool local;
    const bool a_local = a_ok && max_span <= 64, b_local = b_ok && max_span <= 32;
    if (force && (force[0] == '0' || force[0] == '1') && ((force[0] == '0') ? a_ok : b_ok)) {
        variant = force[0] - '0';
        local = variant == 0 ? a_local : b_local;
    } else if (b_local && (!a_local || (long)V <= (long)32 * e->num_sms * 2)) {
        variant = 1; local = true;
    } else if (a_local) {
        variant = 0; local = true;
    } else {
        variant = a_ok ? 0 : 1; local = false;
    }
    const char* force_global = getenv("GGNN_FORCE_GLOBAL");
    if (force_global && force_global[0] == '1') local = false;
    e->variant = variant;
    e->local = local;
    e->nb1 = pick_nb1(variant, D);
    const int MT = variant_mt(variant);
    tile_start.clear();
    tile_start.push_back(0);
    if (local) {
        int cur = 0;
        for (size_t i = 1; i < cuts.size(); ++i) {
            if (cuts[i] - cur > MT) {           // adding this component would overflow: close the tile before it
                tile_start.push_back(cuts[i - 1]);
                cur = cuts[i - 1];
            }
        }
        if (V > cur) tile_start.push_back(V);
    } else {
        for (int r = MT; r < V; r += MT) tile_start.push_back(r);
        if (V > 0) tile_start.push_back(V);
    }
    if (V == 0) tile_start.assign(1, 0);
    e->ntiles = (int)tile_start.size() - 1;
    char buf[256];
    snprintf(buf, sizeof buf, "fp32-ffma%s%s %s tiles=%d rows/tile<=%d warps=8 colsplit=%d nb1=%d max_component=%d smem=%zuB", e->use_att ? "+attention" : "",
             e->cell == CELL_CUDNN_GRU ? "+cudnn-gru" : "",
             local ? "LOCAL(all layers+steps fused, 1 launch)" : "GLOBAL(1 launch per step)", e->ntiles, MT,
             variant_cs(variant), e->nb1, max_span, fwd_smem_bytes(variant, e->nb1, D, e->T));
    e->plan_text = buf;
    return GGNN_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------ backward (host orchestration)
static int ggnn_backward_impl(ggnn_engine* e, const float* d_h_out, const ggnn_layer_grads* grads, int32_t num_layers,
                              float* d_h0, ggnn_stream_t stream) {
    using namespace ggnn::bwd;
    if (!e->graph_set || !e->weights_set) return e->fail(GGNN_ESTATE, "no graph / weights set");
    if (!e->saved_valid) return e->fail(GGNN_ESTATE, "ggnn_backward needs a preceding ggnn_forward with save_for_backward enabled, and no ggnn_set_weights or new graph since");
    if (!e->has_transpose) return e->fail(GGNN_ESTATE, "enable save_for_backward BEFORE ggnn_set_graph_sparse (the source-keyed CSR is built there)");
    if (!grads || num_layers != e->L || (!d_h_out && e->V > 0)) return e->fail(GGNN_EINVAL, "bad backward arguments");
    for (int l = 0; l < e->L; ++l) {   // the weight-gradient kernels use 16-byte vector atomics
        const void* ps[8] = {grads[l].edge_weights, grads[l].edge_biases, grads[l].gate_kernel, grads[l].gate_bias, grads[l].cand_kernel, grads[l].cand_bias,
                             grads[l].edge_type_attention_weights, grads[l].cand_hidden_bias};
        for (const void* q : ps)
            if (q && ((uintptr_t)q & 15)) return e->fail(GGNN_EINVAL, "layer %d: gradient pointers must be 16-byte aligned", l);
    }
    if (((uintptr_t)d_h_out & 15) || ((uintptr_t)d_h0 & 15)) return e->fail(GGNN_EINVAL, "d_h_out / d_h0 must be 16-byte aligned");
    CU_TRY(e, cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    e->last_launches = 0;
    const int V = e->V, D = e->D, T = e->T, L = e->L;
    if (V == 0) return GGNN_OK;
    const size_t vd = (size_t)V * D;
    int maxres = 0;
    for (int l = 0; l < L; ++l) maxres = std::max(maxres, e->nres[l]);
    const int ldx_max = D * (maxres + 2);
    // ---- scratch
    size_t off = 0;
    auto take = [&](size_t floats) { size_t o = off; off = align_up(off + floats * sizeof(float), 256); return o; };
    const size_t o_dstate = take(vd * (L + 1)), o_dha = take(vd), o_dhb = take(vd), o_dpc = take(vd), o_dpg = take(2 * vd);
    const size_t o_dxc = take((size_t)V * ldx_max), o_dxg = take((size_t)V * ldx_max), o_rh = take(vd), o_dxp = take(vd), o_at = take(vd * T), o_gt = take(vd * T);
    const size_t o_pall = take(e->use_att ? vd * T : 0), o_dsa = take(e->use_att ? (size_t)std::max<int64_t>(e->M, 1) : 0);
    // bf16x3: split-reduction workspace of the weight-gradient GEMMs (the largest of their shapes) and per-block attention partials
    const bool tcb = e->bwd_precision == GGNN_PREC_BF16X3;
    size_t ws_floats = 0;
    if (tcb) {
        for (int nseg = 1; nseg <= std::max(maxres + 2, std::min(T, MAX_SEGS)); ++nseg)
            for (int N : {D, 2 * D}) ws_floats = std::max(ws_floats, bwdtc::tn_workspace_floats(V, N, D, nseg, e->num_sms));
        ws_floats = std::max(ws_floats, bwdtc::tn_workspace_floats(V, D, T, 1, e->num_sms));
    }
    const size_t o_ws = take(ws_floats), o_dawp = take(tcb && e->use_att ? (size_t)((V + 7) / 8) * T : 0);
    const size_t o_bpart = take(tcb ? (size_t)((V + bwdtc::COLSUM_ROWS - 1) / bwdtc::COLSUM_ROWS) * 2 * D : 0);
    const size_t o_ptrs = off; off += 256;
    CU_TRY(e, e->bwd_buf.reserve(off));
    char* bb = (char*)e->bwd_buf.ptr;
    float* dstate = (float*)(bb + o_dstate);
    float *dha = (float*)(bb + o_dha), *dhb = (float*)(bb + o_dhb), *dpc = (float*)(bb + o_dpc), *dpg = (float*)(bb + o_dpg);
    float *dxc = (float*)(bb + o_dxc), *dxg = (float*)(bb + o_dxg), *rh = (float*)(bb + o_rh), *dxp = (float*)(bb + o_dxp);
    float *At = (float*)(bb + o_at), *Gt = (float*)(bb + o_gt), *Pall = (float*)(bb + o_pall), *dsa = (float*)(bb + o_dsa);
    float *ws = (float*)(bb + o_ws), *dawp = (float*)(bb + o_dawp), *bpart = (float*)(bb + o_bpart);
    float** d_ptrs = (float**)(bb + o_ptrs);
    if (tcb) CU_TRY(e, bwdtc::configure_tc_gemm());
    CU_TRY(e, cudaMemsetAsync(dstate, 0, vd * L * sizeof(float), st));
    CU_TRY(e, cudaMemcpyAsync(dstate + vd * L, d_h_out, vd * sizeof(float), cudaMemcpyDeviceToDevice, st));
    // forward values of node_states_per_layer
    std::vector<const float*> fstate(L + 1);
    fstate[0] = e->last_h0; fstate[L] = e->last_out;
    for (int l = 1; l < L; ++l) fstate[l] = (const float*)e->state_buf.ptr + (size_t)(l - 1) * vd;
    const float* sv = (const float*)e->save_bufs.ptr;
    const size_t per = vd * (size_t)std::max(e->total_steps, 1);
    const float *sv_h = sv, *sv_x = sv + per, *sv_r = sv + 2 * per, *sv_u = sv + 3 * per, *sv_c = sv + 4 * per, *sv_q = sv + 5 * per;
    char* g = (char*)e->graph_buf.ptr;
    const int* row_ptr = (const int*)(g + e->off_row_ptr);
    const int* csr_src = (const int*)(g + e->off_src);
    const int* trow = (const int*)(g + e->off_trow);
    const int* ttgt = (const int*)(g + e->off_ttgt);
    const int* tslot = (const int*)(g + e->off_tslot);
    const float* dadj = (const float*)(g + e->off_adj);
    const float* indeg = (const float*)(g + e->off_indeg);
    const float* denom = (const float*)(g + e->off_denom);
    const long long n = (long long)vd;
    const int eb = (int)std::min<long long>((n + 255) / 256, 4096);
    // ffma: the FFMA kernel whatever the backward precision (it sums in a fixed order too, without atomics)
    auto gemm_nt = [&](bool acc, const float* A, int lda, int a_stride, const float* B, int ldb, int b_stride, int nseg, float* C, int ldc,
                       int M, int N, int K, bool ffma = false) {
        if (tcb && !ffma) {   // tensor cores: one CTA per 128 x nc tile, the whole reduction in a fixed order
            bwdtc::TcGemmParams p;
            memset(&p, 0, sizeof p);
            p.A = A; p.lda = lda; p.a_stride = a_stride; p.B = B; p.ldb = ldb; p.b_stride = b_stride; p.nseg = nseg;
            p.C = C; p.ldc = ldc; p.M = M; p.N = N; p.K = K; p.nc = bwdtc::pick_nc(N); p.acc = acc ? 1 : 0;
            p.error_flag = (int*)e->err_flag.ptr;
            dim3 grid((N + p.nc - 1) / p.nc, (M + bwdtc::BM - 1) / bwdtc::BM);
            bwdtc::tc_gemm_kernel<bwdtc::MODE_NT><<<grid, bwdtc::NTHREADS, bwdtc::smem_bytes(p.nc), st>>>(p);
            ++e->last_launches;
            return;
        }
        dim3 grid((N + NT_BN - 1) / NT_BN, (M + NT_BM - 1) / NT_BM);
        if (acc) gemm_nt_kernel<true><<<grid, 128, 0, st>>>(A, lda, a_stride, B, ldb, b_stride, nseg, C, ldc, M, N, K);
        else gemm_nt_kernel<false><<<grid, 128, 0, st>>>(A, lda, a_stride, B, ldb, b_stride, nseg, C, ldc, M, N, K);
        ++e->last_launches;
    };
    // C_s[K,N] += A_s^T . B for every segment (C_s = C + s*c_stride), bias[n] += sum_m B[m,n]
    auto gemm_tn = [&](const SegList& segs, int nseg, bool a_vec, const float* B, int ldb, float* C, int ldc, size_t c_stride, float* bias, int M,
                       int N, int K) {
        if (!C && !bias) return;
        if (tcb) {   // tensor cores, S node chunks -> workspace -> chunk-order reduce; no float atomics
            if (bias) {   // its own fixed-order column sum: the same bits whether or not C is requested
                const int nch = (M + bwdtc::COLSUM_ROWS - 1) / bwdtc::COLSUM_ROWS;
                bwdtc::colsum_part_kernel<<<dim3((N + 255) / 256, nch), 256, 0, st>>>(B, ldb, M, N, bpart);
                bwdtc::colsum_det_kernel<<<N, 256, 0, st>>>(bpart, N, nch, bias);
                e->last_launches += 2;
            }
            if (!C) return;
            const bwdtc::TnSplit sp = bwdtc::tn_split(M, N, K, nseg, e->num_sms);
            bwdtc::TcGemmParams p;
            memset(&p, 0, sizeof p);
            p.B = B; p.ldb = ldb; p.nseg = nseg; p.segs = segs; p.C = C; p.ldc = ldc; p.c_stride = (long long)c_stride;
            p.ws = sp.S > 1 ? ws : nullptr; p.M = M; p.N = N; p.K = K; p.nc = sp.nc; p.rows_per_chunk = sp.rows_per_chunk; p.ktiles = sp.ktiles;
            p.error_flag = (int*)e->err_flag.ptr;
            dim3 grid((N + sp.nc - 1) / sp.nc, nseg * sp.ktiles, sp.S);
            bwdtc::tc_gemm_kernel<bwdtc::MODE_TN><<<grid, bwdtc::NTHREADS, bwdtc::smem_bytes(sp.nc), st>>>(p);
            ++e->last_launches;
            if (sp.S > 1) {
                const long long total = (long long)nseg * K * N;
                const int blocks = (int)std::min<long long>((total + 255) / 256, 8 * (long long)e->num_sms);
                bwdtc::tn_reduce_kernel<<<blocks, 256, 0, st>>>(ws, sp.S, nseg, K, N, C, ldc, (long long)c_stride);
                ++e->last_launches;
            }
            return;
        }
        if (C) {
            const int kblocks = (K + 63) / 64;
            const int tiles = ((N + 63) / 64) * nseg * kblocks;
            // ~4 CTAs of 64 threads per SM; every split costs K*N atomics per segment, so keep >= 64 rows per split
            const int want = std::max(1, (4 * e->num_sms + tiles - 1) / tiles);
            const int splits = std::max(1, std::min(want, (M + 63) / 64));
            const int rps = ((M + splits - 1) / splits + GEMM_BK - 1) / GEMM_BK * GEMM_BK;
            dim3 grid((N + 63) / 64, nseg * kblocks, (M + rps - 1) / rps);
            gemm_tn_atomic_kernel<<<grid, 64, 0, st>>>(segs, kblocks, a_vec ? 1 : 0, B, ldb, C, ldc, c_stride, bias, M, N, K, rps);
        } else {   // bias gradient only
            const int rpb = 512;
            dim3 grid((N + 255) / 256, (M + rpb - 1) / rpb);
            colsum_atomic_kernel<<<grid, 256, 0, st>>>(B, ldb, nullptr, 0, bias, M, N, rpb);
        }
        ++e->last_launches;
    };
    const int nodes_blocks = (V + 7) / 8;
    const int TD = T * D;
    for (int l = L - 1; l >= 0; --l) {
        const int R = e->nres[l], din = D * (1 + R), ldx = din + D;
        const ggnn_layer_weights& w = e->w[l];
        const ggnn_layer_grads& gw = grads[l];
        if (R > 0) {
            float* hp[MAX_RES];
            for (int i = 0; i < R; ++i) hp[i] = dstate + (size_t)e->res[l][i] * vd;
            CU_TRY(e, cudaMemcpyAsync(d_ptrs, hp, sizeof(float*) * R, cudaMemcpyHostToDevice, st));
        }
        float* dhn = dstate + (size_t)(l + 1) * vd;   // gradient wrt the state leaving the current step
        float* dh_new = dha;
        for (int s = e->steps[l] - 1; s >= 0; --s) {
            const size_t so = (size_t)(e->step_base[l] + s) * vd;
            const float *h = sv_h + so, *x = sv_x + so;
            if (e->saved_drop_keep < 1.0f) {
                dropout_grad_kernel<<<eb, 256, 0, st>>>(dhn, e->saved_drop_seed, e->step_base[l] + s, V, D, e->saved_drop_keep, n);
                ++e->last_launches;
            }
            // the cell input row [res_0 .. res_{R-1} | x | last], one [V,D] array per piece
            auto cell_segs = [&](const float* last) {
                SegList sl;
                memset(&sl, 0, sizeof sl);
                for (int i = 0; i < R; ++i) { sl.p[i] = fstate[e->res[l][i]]; sl.ld[i] = D; }
                sl.p[R] = x; sl.ld[R] = D;
                sl.p[R + 1] = last; sl.ld[R + 1] = D;
                return sl;
            };
            if (e->cell == CELL_GRU) {
                const float *r = sv_r + so, *u = sv_u + so, *c = sv_c + so;
                gru_bwd1_kernel<<<eb, 256, 0, st>>>(dhn, h, r, u, c, dpc, dpg, dh_new, rh, n, D, e->act); ++e->last_launches;
                gemm_nt(false, dpc, D, 0, w.cand_kernel, D, 0, 1, dxc, ldx, V, ldx, D);
                gemm_tn(cell_segs(rh), R + 2, true, dpc, D, gw.cand_kernel, D, (size_t)D * D, gw.cand_bias, V, D, D);
                gru_bwd2_kernel<<<eb, 256, 0, st>>>(dxc, ldx, (R + 1) * D, h, r, dpg, dh_new, n, D); ++e->last_launches;
                gemm_nt(false, dpg, 2 * D, 0, w.gate_kernel, 2 * D, 0, 1, dxg, ldx, V, ldx, 2 * D);
                gemm_tn(cell_segs(h), R + 2, true, dpg, 2 * D, gw.gate_kernel, 2 * D, (size_t)D * 2 * D, gw.gate_bias, V, 2 * D, D);
                split_input_grad_kernel<<<eb, 256, 0, st>>>(dxc, dxg, ldx, R, d_ptrs, dxp, e->use_avg ? denom : nullptr, dh_new, 0, 1, 1, n, D);
                ++e->last_launches;
            } else if (e->cell == CELL_CUDNN_GRU) {
                // c = act(x.K_in + b_in + r*q), q = h.K_hid + b_hid: the candidate kernel's first din rows see [res.., x], its last D rows see h
                const float *r = sv_r + so, *u = sv_u + so, *c = sv_c + so, *q = sv_q + so;
                float* dq = rh;   // the r*h scratch of the GRU branch is free here
                cudnn_gru_bwd1_kernel<<<eb, 256, 0, st>>>(dhn, h, r, u, c, q, dpc, dq, dpg, dh_new, n, D, e->act); ++e->last_launches;
                gemm_nt(false, dpc, D, 0, w.cand_kernel, D, 0, 1, dxc, ldx, V, din, D);                                  // d[res.., x] = dpc . K_in^T
                gemm_nt(true, dq, D, 0, w.cand_kernel + (size_t)din * D, D, 0, 1, dh_new, D, V, D, D);                   // dh += dq . K_hid^T
                gemm_tn(cell_segs(nullptr), R + 1, true, dpc, D, gw.cand_kernel, D, (size_t)D * D, gw.cand_bias, V, D, D);
                {
                    SegList sl;
                    memset(&sl, 0, sizeof sl);
                    sl.p[0] = h; sl.ld[0] = D;
                    gemm_tn(sl, 1, true, dq, D, gw.cand_kernel ? gw.cand_kernel + (size_t)din * D : nullptr, D, 0, gw.cand_hidden_bias, V, D, D);
                }
                gemm_nt(false, dpg, 2 * D, 0, w.gate_kernel, 2 * D, 0, 1, dxg, ldx, V, ldx, 2 * D);
                gemm_tn(cell_segs(h), R + 2, true, dpg, 2 * D, gw.gate_kernel, 2 * D, (size_t)D * 2 * D, gw.gate_bias, V, 2 * D, D);
                // dxc holds only the din input columns: the recurrent gradient of the candidate went into dh_new through dq above
                split_input_grad_kernel<<<eb, 256, 0, st>>>(dxc, dxg, ldx, R, d_ptrs, dxp, e->use_avg ? denom : nullptr, dh_new, 0, 1, 1, n, D);
                ++e->last_launches;
            } else {
                const float* hnew = (s == e->steps[l] - 1) ? fstate[l + 1] : sv_h + so + vd;
                rnn_bwd1_kernel<<<eb, 256, 0, st>>>(dhn, hnew, dpc, n, e->act, e->saved_drop_keep < 1.0f ? e->saved_drop_keep : 1.0f); ++e->last_launches;
                gemm_nt(false, dpc, D, 0, w.cand_kernel, D, 0, 1, dxc, ldx, V, ldx, D);
                gemm_tn(cell_segs(h), R + 2, true, dpc, D, gw.cand_kernel, D, (size_t)D * D, gw.cand_bias, V, D, D);
                split_input_grad_kernel<<<eb, 256, 0, st>>>(dxc, nullptr, ldx, R, d_ptrs, dxp, e->use_avg ? denom : nullptr, dh_new, 1, 0, 0, n, D);
                ++e->last_launches;
            }
            // ---- messages: all edge types at once.  At[v, t*D..] = sum of h over the type-t sources of v, Gt[s, t*D..] = sum of dx' over
            // the type-t targets of s
            if (e->gather_mode == GATHER_SPARSE) {
                const float* alpha = nullptr;
                if (e->use_att) {   // softmax backward first (it adds to dh_new), then the gathers are weighted by the probabilities
                    alpha = (const float*)e->att_buf.ptr + (size_t)(e->step_base[l] + s) * (size_t)std::max<int64_t>(e->M, 1);
                    // P[v, t*D+k] = <dx'[v], W_t[k, :]>.  Always fp32 FFMA: the softmax backward cancels sum_k alpha_k d alpha_k out of
                    // d alpha, and a bf16x3 P (2^-16 relative) leaves d a_t of a type whose terms nearly cancel outside the gradient bar
                    gemm_nt(false, dxp, D, 0, w.edge_weights, D, 0, 1, Pall, TD, V, TD, D, true);
                    if (tcb) {   // per-block partials of d a_t, added in block order
                        float* part = gw.edge_type_attention_weights ? dawp : nullptr;
                        attention_bwd_target_kernel<true><<<nodes_blocks, 256, 0, st>>>(row_ptr, csr_src, h, Pall, alpha, w.edge_type_attention_weights,
                                                                                        dsa, dh_new, gw.edge_type_attention_weights, V, D, T, part);
                        if (part) { bwdtc::colsum_det_kernel<<<T, 256, 0, st>>>(part, T, nodes_blocks, gw.edge_type_attention_weights); ++e->last_launches; }
                    } else {
                        attention_bwd_target_kernel<false><<<nodes_blocks, 256, 0, st>>>(row_ptr, csr_src, h, Pall, alpha, w.edge_type_attention_weights,
                                                                                         dsa, dh_new, gw.edge_type_attention_weights, V, D, T, nullptr);
                    }
                    attention_bwd_source_kernel<<<nodes_blocks, 256, 0, st>>>(trow, ttgt, tslot, h, dsa, dh_new, V, D, T);
                    e->last_launches += 2;
                }
                GatherJob j0{row_ptr, csr_src, h, At, alpha, nullptr}, j1{trow, ttgt, dxp, Gt, alpha, alpha ? tslot : nullptr};
                csr_gather_all_kernel<<<dim3(nodes_blocks, 2), 256, 0, st>>>(j0, j1, V, D, T);
                ++e->last_launches;
            } else {
                for (int t = 0; t < T; ++t) {
                    dense_gather_sum_kernel<<<nodes_blocks, 256, 0, st>>>(dadj, h, At + (size_t)t * D, TD, V, D, T, t, e->dense_v, 0);
                    dense_gather_sum_kernel<<<nodes_blocks, 256, 0, st>>>(dadj, dxp, Gt + (size_t)t * D, TD, V, D, T, t, e->dense_v, 1);
                    e->last_launches += 2;
                }
            }
            if (e->use_bias && gw.edge_biases) {   // dB[t,:] += sum_v indeg[v,t] dx'[v,:]  =  indeg^T . dx'
                SegList sl;
                memset(&sl, 0, sizeof sl);
                sl.p[0] = indeg; sl.ld[0] = T;
                gemm_tn(sl, 1, false, dxp, D, gw.edge_biases, D, 0, nullptr, V, D, T);
            }
            if (gw.edge_weights) {
                for (int t0 = 0; t0 < T; t0 += MAX_SEGS) {
                    SegList sl;
                    memset(&sl, 0, sizeof sl);
                    const int nt = std::min(MAX_SEGS, T - t0);
                    for (int t = 0; t < nt; ++t) { sl.p[t] = At + (size_t)(t0 + t) * D; sl.ld[t] = TD; }
                    gemm_tn(sl, nt, true, dxp, D, gw.edge_weights + (size_t)t0 * D * D, D, (size_t)D * D, nullptr, V, D, D);
                }
            }
            gemm_nt(true, Gt, TD, D, w.edge_weights, D, D * D, T, dh_new, D, V, D, D);
            dhn = dh_new;
            dh_new = (dh_new == dha) ? dhb : dha;
        }
        if (e->steps[l] > 0) { add_inplace_kernel<<<eb, 256, 0, st>>>(dstate + (size_t)l * vd, dhn, n); ++e->last_launches; }
        else { add_inplace_kernel<<<eb, 256, 0, st>>>(dstate + (size_t)l * vd, dstate + (size_t)(l + 1) * vd, n); ++e->last_launches; }
    }
    if (d_h0) CU_TRY(e, cudaMemcpyAsync(d_h0, dstate, vd * sizeof(float), cudaMemcpyDeviceToDevice, st));
    CU_TRY(e, cudaGetLastError());
    return GGNN_OK;
}

// ------------------------------------------------------------------------------------------ C ABI
extern "C" {

const char* ggnn_last_error(const ggnn_engine* e) { return e ? e->err.c_str() : g_create_error.c_str(); }

// The model shape of a ggnn_config (what prepare_specific_graph_model fixes) -> e; no CUDA.  Shared by ggnn_create and the host-only
// constructor of prepared graphs (which may run in any thread: the text goes to `err`, not to a global).  Returns GGNN_OK or an error code.
static int init_model_shape(ggnn_engine* e, const ggnn_config* cfg, std::string& err) {
    auto bad = [&](const char* msg) { err = msg; return (int)GGNN_EINVAL; };
    if (cfg->hidden_size <= 0 || cfg->hidden_size % 4 != 0) return bad("hidden_size must be a positive multiple of 4");
    if (cfg->hidden_size > 256) { err = "hidden_size > 256 is not supported by this build"; return GGNN_EUNSUPPORTED; }
    if (cfg->num_edge_types <= 0 || cfg->num_edge_types > 32) return bad("num_edge_types must be in 1..32");
    if (cfg->num_layers <= 0 || cfg->num_layers > MAX_LAYERS) return bad("num_layers must be in 1..16");
    if (!cfg->layer_timesteps) return bad("layer_timesteps is null");
    if (cfg->cell != GGNN_CELL_GRU && cfg->cell != GGNN_CELL_RNN && cfg->cell != GGNN_CELL_CUDNN_GRU) return bad("Unknown RNN cell type");   // sparse:112
    if (cfg->cell == GGNN_CELL_CUDNN_GRU && cfg->activation != GGNN_ACT_TANH) return bad("CudnnCompatibleGRUCell requires the tanh activation");   // sparse:106
    if (cfg->activation != GGNN_ACT_TANH && cfg->activation != GGNN_ACT_RELU) return bad("Unknown activation function type");  // sparse:81
    if (cfg->precision != GGNN_PREC_FP32 && cfg->precision != GGNN_PREC_BF16X3 && cfg->precision != GGNN_PREC_BF16) return bad("unknown precision");
    e->D = cfg->hidden_size; e->T = cfg->num_edge_types; e->L = cfg->num_layers;
    e->use_bias = cfg->use_edge_bias != 0; e->use_avg = cfg->use_edge_msg_avg_aggregation != 0;
    e->cell = cfg->cell; e->act = cfg->activation; e->precision = cfg->precision; e->device = cfg->device;
    e->use_att = cfg->use_propagation_attention != 0;
    if (e->use_att && e->T > 16) { err = "propagation attention supports at most 16 edge types"; return GGNN_EUNSUPPORTED; }
    if (e->use_att) e->precision = GGNN_PREC_FP32;   // the softmax-weighted gather lives in the fp32 kernel only (the plan text says so)
    if (e->cell == CELL_CUDNN_GRU) e->precision = GGNN_PREC_FP32;   // so does the reset-after-matmul candidate of CudnnCompatibleGRUCell
    int total = 0;
    for (int l = 0; l < e->L; ++l) {
        if (cfg->layer_timesteps[l] < 0) return bad("negative layer_timesteps entry");
        e->steps[l] = cfg->layer_timesteps[l];
        e->step_base[l] = total;
        total += e->steps[l];
        int nr = 0;
        if (cfg->residual_offsets && cfg->residual_layers) {
            nr = cfg->residual_offsets[l + 1] - cfg->residual_offsets[l];
            if (nr < 0 || nr > MAX_RES) return bad("a layer has more than 4 residual inputs");
            for (int i = 0; i < nr; ++i) {
                int r = cfg->residual_layers[cfg->residual_offsets[l] + i];
                // node_states_per_layer has l+1 entries when layer l is built (sparse:144: IndexError otherwise)
                if (r < 0 || r > l) return bad("residual connection refers to a layer that does not exist yet");
                e->res[l][i] = r;
            }
        }
        e->nres[l] = nr;
    }
    e->total_steps = total;
    e->DP = (e->D + 15) / 16 * 16;
    return GGNN_OK;
}

int ggnn_create(const ggnn_config* cfg, ggnn_engine** out) {
    if (!cfg || !out) { g_create_error = "null argument"; return GGNN_EINVAL; }
    *out = nullptr;
    ggnn_engine* e = new ggnn_engine();
    if (int rc = init_model_shape(e, cfg, g_create_error)) { delete e; return rc; }
    cudaError_t st = cudaSetDevice(e->device);
    cudaDeviceProp prop;
    if (st == cudaSuccess) st = cudaGetDeviceProperties(&prop, e->device);
    if (st != cudaSuccess) {
        g_create_error = std::string("CUDA device unavailable: ") + cudaGetErrorString(st);
        delete e;
        return GGNN_ECUDA;
    }
    e->num_sms = prop.multiProcessorCount;
    e->max_smem = prop.sharedMemPerBlockOptin;
    memset(e->w, 0, sizeof e->w);
    if (e->err_flag.reserve(sizeof(int)) != cudaSuccess || cudaMemset(e->err_flag.ptr, 0, sizeof(int)) != cudaSuccess) {
        g_create_error = "cudaMalloc failed";
        delete e;
        return GGNN_ECUDA;
    }
    *out = e;
    return GGNN_OK;
}

int ggnn_destroy(ggnn_engine* e) {
    if (!e) return GGNN_OK;
    cudaSetDevice(e->device);
    e->graph_buf.release(); e->state_buf.release(); e->save_bufs.release(); e->io_buf.release(); e->bwd_buf.release();
    e->tc_weights.release(); e->tc_respre.release(); e->ts_weights.release(); e->ts_images.release(); e->ts_u.release(); e->ts_virt.release(); e->err_flag.release(); e->dbg_buf.release();
    e->graph_stage.release();
    if (e->own_prep) { ggnn_free_prepared_graph(e->own_prep); e->own_prep = nullptr; }
    if (e->stage_done) cudaEventDestroy(e->stage_done);
    if (e->ro_stage_done) cudaEventDestroy(e->ro_stage_done);
    e->ro_buf.release(); e->ro_stage.release(); e->att_buf.release();
    delete e;
    return GGNN_OK;
}

int ggnn_set_weights(ggnn_engine* e, const ggnn_layer_weights* layers, int32_t num_layers) {
    if (!e) return GGNN_EINVAL;
    // the saved activations belong to the weights they were computed with: a backward after new weights would mix the two
    e->saved_valid = false;
    if (!layers || num_layers != e->L) return e->fail(GGNN_EINVAL, "expected %d layers of weights, got %d", e->L, num_layers);
    for (int l = 0; l < e->L; ++l) {
        const ggnn_layer_weights& w = layers[l];
        if (!w.edge_weights || !w.cand_kernel || !w.cand_bias) return e->fail(GGNN_EINVAL, "layer %d: null edge_weights/cand_kernel/cand_bias", l);
        if (e->use_bias && !w.edge_biases) return e->fail(GGNN_EINVAL, "layer %d: use_edge_bias set but edge_biases is null", l);
        if (e->cell != CELL_RNN && (!w.gate_kernel || !w.gate_bias)) return e->fail(GGNN_EINVAL, "layer %d: GRU needs gate_kernel/gate_bias", l);
        if (e->cell == CELL_CUDNN_GRU && !w.cand_hidden_bias) return e->fail(GGNN_EINVAL, "layer %d: CudnnCompatibleGRUCell needs cand_hidden_bias", l);
        if (e->use_att && !w.edge_type_attention_weights) return e->fail(GGNN_EINVAL, "layer %d: use_propagation_attention set but edge_type_attention_weights is null", l);
        const void* ps[7] = {w.edge_weights, w.edge_biases, w.gate_kernel, w.gate_bias, w.cand_kernel, w.cand_bias, w.cand_hidden_bias};
        for (const void* q : ps)
            if (q && ((uintptr_t)q & 15)) return e->fail(GGNN_EINVAL, "layer %d: weight pointers must be 16-byte aligned", l);
        e->w[l] = w;
    }
    e->weights_set = true;
    e->weights_dirty = true;   // the tensor-core path re-tiles its bf16 copies at the next forward
    return GGNN_OK;
}

static int upload_graph(ggnn_engine* e, size_t bytes, cudaStream_t st) {
    CU_TRY(e, e->graph_buf.reserve(bytes));
    CU_TRY(e, cudaMemcpyAsync(e->graph_buf.ptr, e->graph_stage.ptr, bytes, cudaMemcpyHostToDevice, st));
    if (!e->stage_done) CU_TRY(e, cudaEventCreateWithFlags(&e->stage_done, cudaEventDisableTiming));
    CU_TRY(e, cudaEventRecord(e->stage_done, st));
    return GGNN_OK;
}

static int reserve_states(ggnn_engine* e) {
    const size_t vd = (size_t)std::max(e->V, 1) * e->D * sizeof(float);
    CU_TRY(e, e->state_buf.reserve(vd * (size_t)(e->L + 1)));
    if (e->save) CU_TRY(e, e->save_bufs.reserve(vd * (e->cell == CELL_CUDNN_GRU ? 6 : 5) * (size_t)std::max(e->total_steps, 1)));
    return GGNN_OK;
}

// Stable counting sort of the messages by (target, type): counts[k + 1] holds the number of messages of row k = target*T + type on
// entry (it is reused as the write cursors).  Messages are visited in the reference's order (type-major, then list order,
// sparse:124-129), so within a row they stay in message order -- this IS NumPy's stable argsort by target.
static void fill_target_csr(int V, int T, const int32_t* const* adj, const int32_t* num_edges, std::vector<int>& counts, int* row_ptr,
                            int* csr_src, int* csr_msg) {
    row_ptr[0] = 0;
    for (size_t k = 1; k <= (size_t)V * T; ++k) row_ptr[k] = row_ptr[k - 1] + counts[k];
    std::vector<int>& pos = counts;
    for (size_t k = 0; k < (size_t)V * T; ++k) pos[k] = row_ptr[k];
    int m = 0;
    for (int t = 0; t < T; ++t) {
        const int32_t* a = adj[t];
        for (int i = 0; i < num_edges[t]; ++i, ++m) {
            const int slot = pos[(size_t)a[2 * i + 1] * T + t]++;
            csr_src[slot] = a[2 * i];
            csr_msg[slot] = m;
        }
    }
}

// Streaming plan: number the (target, type) pairs marked -2 ("several messages") in row order, replace the mark by -(2 + vid) and list
// their sources (vinfo: count + the first seven inline; vptr / vsrc: the complete lists).  `pair` already holds -1 / the single source.
static void number_virtual_rows(int ntiles, int T, const int* tile_start, const int* row_ptr, const int* csr_src, int* pair, int* vptr, int* vsrc,
                                int* tvp, int* vinfo) {
    int vid = 0, vm = 0;
    vptr[0] = 0;
    for (int i = 0; i < ntiles; ++i) {
        tvp[i] = vid;
        for (size_t k = (size_t)tile_start[i] * T, kend = (size_t)tile_start[i + 1] * T; k < kend; ++k) {
            if (pair[k] != -2) continue;
            const int b = row_ptr[k], cnt = row_ptr[k + 1] - b;
            pair[k] = -(2 + vid);
            if (vinfo) {
                vinfo[8 * vid] = cnt;
                for (int m = 0; m < 7; ++m) vinfo[8 * vid + 1 + m] = m < cnt ? csr_src[b + m] : 0;
            }
            for (int m = 0; m < cnt; ++m) vsrc[vm++] = csr_src[b + m];
            vptr[++vid] = vm;
        }
    }
    tvp[ntiles] = vid;
}

// The tile plan ggnn_set_graph_sparse would make for this batch, without an engine or a GPU: the cut points (node boundaries no edge
// crosses, from a difference array over the edge spans) and build_plan() on a scratch engine object that never touches CUDA.
int ggnn_host_tile_plan(int32_t hidden_size, int32_t num_edge_types, int32_t precision, int32_t num_sms, int32_t V, const int32_t* const* adj,
                        const int32_t* num_edges, int32_t* tile_start, int32_t tile_capacity, int32_t* num_tiles, char* plan_text,
                        int32_t plan_text_capacity) {
    if (hidden_size <= 0 || num_edge_types <= 0 || V < 0 || !adj || !num_edges || !tile_start || !num_tiles || num_sms <= 0) return GGNN_EINVAL;
    // same cut detection as ggnn_set_graph_sparse: reach[j] = farthest node an edge starting at node j touches
    std::vector<int> reach((size_t)V + 1, 0);
    for (int t = 0; t < num_edge_types; ++t)
        for (int i = 0; i < num_edges[t]; ++i) {
            const int s = adj[t][2 * i], d = adj[t][2 * i + 1];
            if ((unsigned)s >= (unsigned)V || (unsigned)d >= (unsigned)V) return GGNN_ERANGE;
            const int lo = std::min(s, d), hi = std::max(s, d);
            if (hi > reach[lo]) reach[lo] = hi;
        }
    std::vector<int> cuts(1, 0);
    int far = 0;
    for (int i = 1; i < V; ++i) {
        far = std::max(far, reach[i - 1]);
        if (far < i) cuts.push_back(i);
    }
    if (V > 0) cuts.push_back(V);
    ggnn_engine scratch;
    scratch.D = hidden_size; scratch.T = num_edge_types; scratch.precision = precision; scratch.num_sms = num_sms;
    scratch.max_smem = 227 * 1024; scratch.V = V;
    if (precision != GGNN_PREC_FP32) scratch.DP = (hidden_size + 15) / 16 * 16;
    std::vector<int> ts;
    int rc = build_plan(&scratch, cuts, ts);
    if (rc) return rc;
    *num_tiles = scratch.ntiles;
    if ((int)ts.size() > tile_capacity) return GGNN_EINVAL;
    for (size_t i = 0; i < ts.size(); ++i) tile_start[i] = ts[i];
    if (plan_text && plan_text_capacity > 0) snprintf(plan_text, (size_t)plan_text_capacity, "%s", scratch.plan_text.c_str());
    return GGNN_OK;
}

// The same CSR build without an engine or a GPU (host arithmetic only): lets the CPU test-suite pin the integer path bit for bit.
int ggnn_host_target_csr(int32_t V, int32_t T, const int32_t* const* adj, const int32_t* num_edges, int32_t* row_ptr, int32_t* src,
                         int32_t* msg) {
    if (V < 0 || T <= 0 || !adj || !num_edges || !row_ptr) return GGNN_EINVAL;
    std::vector<int> counts((size_t)V * T + 1, 0);
    int64_t M = 0;
    for (int t = 0; t < T; ++t) {
        if (num_edges[t] < 0 || (num_edges[t] > 0 && !adj[t])) return GGNN_EINVAL;
        M += num_edges[t];
        for (int i = 0; i < num_edges[t]; ++i) {
            const int s = adj[t][2 * i], d = adj[t][2 * i + 1];
            if ((unsigned)s >= (unsigned)V || (unsigned)d >= (unsigned)V) return GGNN_ERANGE;
            ++counts[(size_t)d * T + t + 1];
        }
    }
    if (M > 0 && (!src || !msg)) return GGNN_EINVAL;
    fill_target_csr(V, T, adj, num_edges, counts, row_ptr, src, msg);
    return GGNN_OK;
}

int ggnn_host_stream_tables(int32_t V, int32_t T, const int32_t* const* adj, const int32_t* num_edges, int32_t* pair_src, int32_t* vrow_ptr,
                            int32_t vrow_capacity, int32_t* vsrc, int32_t vsrc_capacity, int32_t* tile_vptr, int32_t* num_virtual_rows) {
    if (V < 0 || T <= 0 || !adj || !num_edges || !pair_src || !vrow_ptr || !vsrc || !tile_vptr || !num_virtual_rows) return GGNN_EINVAL;
    std::vector<int> row_ptr((size_t)V * T + 1), src, msg;
    int64_t M = 0;
    for (int t = 0; t < T; ++t) M += num_edges[t];
    src.resize((size_t)std::max<int64_t>(M, 1)); msg.resize((size_t)std::max<int64_t>(M, 1));
    int rc = ggnn_host_target_csr(V, T, adj, num_edges, row_ptr.data(), src.data(), msg.data());
    if (rc) return rc;
    const int ntiles = (V + ts::TILE_M - 1) / ts::TILE_M;
    std::vector<int> tile_start(ntiles + 1);
    for (int i = 0; i <= ntiles; ++i) tile_start[i] = std::min(i * ts::TILE_M, V);
    int nv = 0; int64_t nvm = 0;
    for (size_t k = 0; k < (size_t)V * T; ++k) {
        const int cnt = row_ptr[k + 1] - row_ptr[k];
        pair_src[k] = cnt == 0 ? -1 : (cnt == 1 ? src[row_ptr[k]] : -2);
        if (cnt >= 2) { ++nv; nvm += cnt; }
    }
    for (size_t k = (size_t)V * T; k < (size_t)ntiles * ts::TILE_M * T; ++k) pair_src[k] = -1;
    if (nv + 1 > vrow_capacity || nvm > vsrc_capacity) return GGNN_EINVAL;
    number_virtual_rows(ntiles, T, tile_start.data(), row_ptr.data(), src.data(), pair_src, vrow_ptr, vsrc, tile_vptr, nullptr);
    *num_virtual_rows = nv;
    return GGNN_OK;
}

#ifdef _OPENMP
// Size of the host team for the per-batch graph builders: up to 8 threads, bounded by the cores this process may run on divided by the
// number of ranks on the node (LOCAL_WORLD_SIZE, set by torchrun).  Deliberately NOT omp_get_max_threads(): torchrun exports
// OMP_NUM_THREADS=1 to every rank by default ("to avoid your system being overloaded"), which would silently serialise the builders of
// exactly the multi-GPU runs (measured at N = 2: dense batch e2e 0.77 ms against 0.41 ms at N = 1); 8 ranks x 8 short-lived builder threads
// are far below a GPU host's core count.  GGNN_HOST_THREADS overrides.
static int host_team_size() {
    int avail = 0;
    cpu_set_t set;
    if (sched_getaffinity(0, sizeof set, &set) == 0) avail = CPU_COUNT(&set);
    if (avail <= 0) avail = omp_get_num_procs();
    int ranks = 1;
    if (const char* lws = getenv("LOCAL_WORLD_SIZE")) ranks = std::max(1, atoi(lws));
    return std::max(1, std::min(8, avail / ranks));
}

// One-time probe per process: is a parallel region of `team` threads cheap to enter here?  (Third of three empty regions under 150 us.)
static bool host_team_is_fast(int team) {
    static int verdict[65] = {0};   // 0 unknown, 1 fast, -1 slow; a benign race at worst probes twice
    if (team < 2 || team > 64) return false;
    if (verdict[team] == 0) {
        double us = 0.0;
        for (int rep = 0; rep < 3; ++rep) {
            const auto t0 = std::chrono::steady_clock::now();
            int seen = 0;
#pragma omp parallel num_threads(team) reduction(+ : seen)
            { seen += 1; }
            us = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count();
            if (seen < 1) us = 1e9;
        }
        verdict[team] = us < 150.0 ? 1 : -1;
        if (getenv("GGNN_HOST_TIMING")) fprintf(stderr, "[ggnn host] OpenMP team of %d: region entry %.1f us -> %s\n", team, us, us < 150.0 ? "used" : "not used");
    }
    return verdict[team] > 0;
}
#endif

// ---- the host half of ggnn_set_graph_sparse: validation, tile plan, stable target-sorted CSR, streaming tables -> g->image.
// `e` below is the prepared graph's shadow engine (model shape in, batch / plan fields out): nothing here touches the device except the
// pinned allocation of the image and the wait for the previous upload out of the same image.
static int build_sparse_image(ggnn_prepared_graph* g, int32_t V, const int32_t* const* adj, const int32_t* num_edges, const float* indeg) {
    ggnn_engine* e = &g->plan;
    g->valid = false;
    static const bool host_timing = getenv("GGNN_HOST_TIMING") != nullptr;
    const auto t_begin = std::chrono::steady_clock::now();
    auto lap = [&](const char* what, std::chrono::steady_clock::time_point& t) {
        if (!host_timing) return;
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[ggnn host] %-18s %7.1f us\n", what, std::chrono::duration<double, std::micro>(now - t).count());
        t = now;
    };
    auto t_lap = t_begin;
    e->graph_set = false; e->saved_valid = false;
    if (V < 0 || !adj || !num_edges || (!indeg && V > 0)) return e->fail(GGNN_EINVAL, "null/negative argument");
    const int T = e->T;
    int64_t M = 0;
    for (int t = 0; t < T; ++t) {
        if (num_edges[t] < 0 || (num_edges[t] > 0 && !adj[t])) return e->fail(GGNN_EINVAL, "adjacency list %d is null/negative", t);
        M += num_edges[t];
    }
    if (M > 0x7fffffff || (int64_t)V * T + 1 > 0x7fffffff) return e->fail(GGNN_EUNSUPPORTED, "batch too large for int32 indexing");
    e->V = V; e->M = M; e->gather_mode = GATHER_SPARSE; e->dense_v = 0;

    // ---- host threads.  Every pass below is split over `nth` threads by TARGET ranges (pass 1: equal node ranges; later passes: equal
    // tile ranges): each thread scans the whole edge list (sequential reads) and performs only the scattered writes of its own rows, in the
    // list's order -- so every row keeps the reference's message order and the image is bit-identical for every thread count
    // (tests/test_prepared_graph_cpu.py pins it against the single-pass ggnn_host_target_csr and NumPy's stable sort).
    // Small batches stay on one thread (a cfg2-sized build is ~80 us: less than a team's wake-up).  Large ones use ONE team size per
    // process, and only after host_team_is_fast() has seen that entering a parallel region of that size is cheap here: libgomp's region
    // entry can cost milliseconds in some containers (measured: 8-18 ms per region for 2-3 threads on an 8-CPU box, 2 us for 8).
    int nth = 1;
#ifdef _OPENMP
    if (M >= 24000) {
        const int team = host_team_size();
        if (team > 1 && host_team_is_fast(team)) nth = team;
    }
    if (const char* nt = getenv("GGNN_HOST_THREADS")) nth = std::max(1, std::min(atoi(nt), 64));
#endif
    // ---- pass 1: validate, count per (target,type), mark which node boundaries are spanned by an edge (the cut points of the tile-local
    // plans; the streaming plan of hidden sizes > 128 tiles by fixed 128-row blocks and skips that part)
    std::vector<int>& counts = e->h_counts;
    std::vector<int>& reach = e->h_diff;   // reach[j] = the farthest node an edge whose lower end is node j touches
    const bool need_cuts = !(e->precision != GGNN_PREC_FP32 && e->DP > 128);
    counts.resize((size_t)V * T + 1);
    if (need_cuts) reach.resize((size_t)V + 1);
    std::vector<int64_t> type_base(T + 1, 0);   // position of every type's first message in the reference's type-major message order
    for (int t = 0; t < T; ++t) type_base[t + 1] = type_base[t] + num_edges[t];
    int bad_edge = 0;
    // Pass 1 is split by EDGE ranges: counting is commutative, so the threads add into the shared per-row counts with relaxed atomic
    // increments (and an atomic max for `reach`) -- same totals for every thread count; a single thread uses plain increments.
#ifdef _OPENMP
#pragma omp parallel num_threads(nth) if (nth > 1)
#endif
    {
        int k = 0, n = 1;
#ifdef _OPENMP
        k = omp_get_thread_num(); n = omp_get_num_threads();
#endif
        {   // clear this thread's slice of the scratch arrays
            const size_t nc = (size_t)V * T + 1, c0 = nc * k / n, c1 = nc * (k + 1) / n;
            std::fill(counts.begin() + c0, counts.begin() + c1, 0);
            if (need_cuts) {
                const size_t nr = (size_t)V + 1, r0 = nr * k / n, r1 = nr * (k + 1) / n;
                std::fill(reach.begin() + r0, reach.begin() + r1, 0);
            }
        }
#ifdef _OPENMP
#pragma omp barrier
#endif
        const int64_t e0 = M * k / n, e1 = M * (k + 1) / n;   // this thread's messages, in the type-major order
        int* const cnt = counts.data();
        int* const rch = need_cuts ? reach.data() : nullptr;
        bool bad = false;
        for (int t = 0; t < T && !bad; ++t) {
            const int32_t* a = adj[t];
            const int i0 = (int)(std::max(e0, type_base[t]) - type_base[t]);
            const int i1 = (int)(std::min(e1, type_base[t + 1]) - type_base[t]);
            if (n == 1) {
                for (int i = i0; i < i1; ++i) {
                    const int s = a[2 * i], d = a[2 * i + 1];
                    if ((unsigned)s >= (unsigned)V || (unsigned)d >= (unsigned)V) { bad = true; break; }
                    ++cnt[(size_t)d * T + t + 1];
                    if (need_cuts) {
                        const int lo = std::min(s, d), hi = std::max(s, d);
                        rch[lo] = std::max(rch[lo], hi);   // unconditional store: the compare-and-branch form mispredicts on every other edge
                    }
                }
            } else {
                for (int i = i0; i < i1; ++i) {
                    const int s = a[2 * i], d = a[2 * i + 1];
                    if ((unsigned)s >= (unsigned)V || (unsigned)d >= (unsigned)V) { bad = true; break; }
                    __atomic_fetch_add(cnt + ((size_t)d * T + t + 1), 1, __ATOMIC_RELAXED);
                    if (need_cuts) {
                        const int lo = std::min(s, d), hi = std::max(s, d);
                        int cur = __atomic_load_n(rch + lo, __ATOMIC_RELAXED);
                        while (hi > cur && !__atomic_compare_exchange_n(rch + lo, &cur, hi, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
                    }
                }
            }
        }
        if (bad) {
#ifdef _OPENMP
#pragma omp atomic write
#endif
            bad_edge = 1;
        }
    }
    if (bad_edge) {   // name the first offending edge, like the single pass did
        for (int t = 0; t < T; ++t)
            for (int i = 0; i < num_edges[t]; ++i) {
                const int s = adj[t][2 * i], d = adj[t][2 * i + 1];
                if ((unsigned)s >= (unsigned)V || (unsigned)d >= (unsigned)V)
                    return e->fail(GGNN_ERANGE, "edge %d of type %d = (%d,%d) is out of range for %d nodes", i, t, s, d, V);
            }
    }
    lap("  edges pass 1", t_lap);
    std::vector<int> cuts;
    cuts.push_back(0);
    if (need_cuts) {   // the boundary before node i is crossed by an edge iff max_{j < i} reach[j] >= i
        int far = 0;
        for (int i = 1; i < V; ++i) {
            far = std::max(far, reach[i - 1]);
            if (far < i) cuts.push_back(i);
        }
    }
    if (V > 0) cuts.push_back(V);
    lap("validate+count", t_lap);
    std::vector<int> tile_start;
    int rc = build_plan(e, cuts, tile_start);
    if (rc) return rc;
    const int ntiles = e->ntiles;
    lap("tile plan", t_lap);
    nth = std::max(1, std::min(nth, ntiles));
    // tile ranges of the threads for all later passes: tiles [tb[k], tb[k+1]), i.e. nodes [tile_start[tb[k]], tile_start[tb[k+1]])
    std::vector<int> tb(nth + 1);
    for (int k = 0; k <= nth; ++k) tb[k] = (int)((int64_t)ntiles * k / nth);
    // per-range totals: messages, and (streaming plan) virtual rows = (target, type) pairs with several messages, with their message count
    std::vector<int64_t> part_msgs(nth + 1, 0), part_nv(nth + 1, 0), part_nvm(nth + 1, 0);
#ifdef _OPENMP
#pragma omp parallel for schedule(static, 1) num_threads(nth) if (nth > 1)
#endif
    for (int k = 0; k < nth; ++k) {
        int64_t sm = 0, nv = 0, nvm = 0;
        const size_t k0 = (size_t)tile_start[tb[k]] * T, k1 = (size_t)tile_start[tb[k + 1]] * T;
        if (e->stream) {
            for (size_t r = k0; r < k1; ++r) {
                const int c = counts[r + 1];
                sm += c;
                if (c >= 2) { ++nv; nvm += c; }
            }
        } else {
            for (size_t r = k0; r < k1; ++r) sm += counts[r + 1];
        }
        part_msgs[k + 1] = sm; part_nv[k + 1] = nv; part_nvm[k + 1] = nvm;
    }
    for (int k = 0; k < nth; ++k) { part_msgs[k + 1] += part_msgs[k]; part_nv[k + 1] += part_nv[k]; part_nvm[k + 1] += part_nvm[k]; }

    // ---- layout of the packed upload
    size_t off = 0;
    e->off_row_ptr = off; off = align_up(off + sizeof(int) * ((size_t)V * T + 1), 16);
    e->off_src = off;     off = align_up(off + sizeof(int) * (size_t)std::max<int64_t>(M, 1), 16);
    e->off_msg = off;     off = align_up(off + sizeof(int) * (size_t)std::max<int64_t>(M, 1), 16);
    e->off_indeg = off;   off = align_up(off + sizeof(float) * (size_t)std::max(V, 1) * T, 16);
    e->off_denom = off;   off = align_up(off + sizeof(float) * (size_t)std::max(V, 1), 16);
    e->off_tiles = off;   off = align_up(off + sizeof(int) * (size_t)(ntiles + 1), 16);
    e->off_mask = off;    off = align_up(off + sizeof(unsigned) * (size_t)std::max(ntiles, 1), 16);
    e->off_adj = off;
    e->has_transpose = e->save;
    if (e->has_transpose) {
        e->off_trow = off; off = align_up(off + sizeof(int) * ((size_t)V * T + 1), 16);
        e->off_ttgt = off; off = align_up(off + sizeof(int) * (size_t)std::max<int64_t>(M, 1), 16);
        e->off_tslot = off;
        if (e->use_att) off = align_up(off + sizeof(int) * (size_t)std::max<int64_t>(M, 1), 16);
    }
    // streaming plan: per (target, type) pair the ONE node to copy from (or none / a virtual row), see ggnn_fwd_stream.cuh
    const int nv = (int)part_nv[nth];
    const int64_t nvm = part_nvm[nth];
    if (e->stream) {
        e->off_pair = off; off = align_up(off + sizeof(int) * (size_t)std::max(ntiles, 1) * ts::TILE_M * T, 16);
        e->off_vptr = off; off = align_up(off + sizeof(int) * (size_t)(nv + 1), 16);
        e->off_vsrc = off; off = align_up(off + sizeof(int) * (size_t)std::max<int64_t>(nvm, 1), 16);
        e->off_tvp = off;  off = align_up(off + sizeof(int) * (size_t)(ntiles + 1), 16);
        e->off_vinfo = off; off = align_up(off + sizeof(int) * 8 * (size_t)std::max(nv, 1), 16);
    }
    e->ts_nv = nv;
    for (int t = 0; t < T; ++t) e->edges_of_type[t] = num_edges[t];
    if (g->use_cuda) {
        if (g->uploaded) CU_TRY(e, cudaEventSynchronize(g->uploaded));   // the previous upload may still be reading this image
        CU_TRY(e, g->stage.reserve(off));
        g->image = (char*)g->stage.ptr;
    } else {
        if (g->plain.size() < off) g->plain.resize(off + off / 4 + 256);
        g->image = g->plain.data();
    }
    g->bytes = off;
    char* base = g->image;
    int* row_ptr = (int*)(base + e->off_row_ptr);
    int* csr_src = (int*)(base + e->off_src);
    int* csr_msg = (int*)(base + e->off_msg);
    float* h_indeg = (float*)(base + e->off_indeg);
    float* h_denom = (float*)(base + e->off_denom);
    int* h_tiles = (int*)(base + e->off_tiles);
    unsigned* h_mask = (unsigned*)(base + e->off_mask);
    int* pair = e->stream ? (int*)(base + e->off_pair) : nullptr;   // streaming plan: (target, type) -> its one source / virtual row
    int* vptr = e->stream ? (int*)(base + e->off_vptr) : nullptr;
    int* vsrc = e->stream ? (int*)(base + e->off_vsrc) : nullptr;
    int* tvp = e->stream ? (int*)(base + e->off_tvp) : nullptr;
    int* vinfo = e->stream ? (int*)(base + e->off_vinfo) : nullptr;
    lap("stage reserve", t_lap);

    // ---- pass 2, per thread over its tile range: exclusive scan of the (target, type) rows -> row_ptr, fill cursors, the tiles'
    // edge-type masks and the largest per-tile message count; then the stable fill -- every thread walks the
    // lists in the reference's order (type-major, then list order, sparse:124-129) and places the messages of ITS rows, so within a row
    // they stay in message order: this IS NumPy's stable argsort by target, tests pin it bit for bit; then (streaming plan) the gather
    // table and the virtual rows of its range, numbered from the range's offset; then in-degrees / denominators of its nodes.
    std::vector<int>& cursor = e->h_cursor;   // next free slot of every (target, type) row (its own array: the counts of a range's last
    cursor.resize((size_t)V * T + 1);         // row are read by one thread while the next range's thread already writes cursors)
    int max_tile_msgs = 0;
    row_ptr[0] = 0;
    if (vptr) vptr[0] = 0;
#ifdef _OPENMP
#pragma omp parallel for schedule(static, 1) num_threads(nth) if (nth > 1) reduction(max : max_tile_msgs)
#endif
    for (int k = 0; k < nth; ++k) {
        int run = (int)part_msgs[k];
        for (int i = tb[k]; i < tb[k + 1]; ++i) {
            unsigned mask = 0;
            const int tile_first = run;
            for (size_t r = (size_t)tile_start[i] * T, rend = (size_t)tile_start[i + 1] * T; r < rend; r += T)
                for (int t = 0; t < T; ++t) {
                    const int c = counts[r + t + 1];
                    cursor[r + t] = run;
                    run += c;
                    row_ptr[r + t + 1] = run;
                    mask |= (unsigned)(c > 0) << t;
                }
            h_mask[i] = mask;
            max_tile_msgs = std::max(max_tile_msgs, run - tile_first);
            h_tiles[i] = tile_start[i];
        }
        if (k == nth - 1) h_tiles[ntiles] = tile_start[ntiles];
    }
    e->max_tile_msgs = max_tile_msgs;
    lap("row sweep", t_lap);
#ifdef _OPENMP
#pragma omp parallel for schedule(static, 1) num_threads(nth) if (nth > 1)
#endif
    for (int k = 0; k < nth; ++k) {
        const int v0 = tile_start[tb[k]], v1 = tile_start[tb[k + 1]];
        for (int t = 0; t < T; ++t) {
            const int32_t* a = adj[t];
            const int ne = num_edges[t];
            const int mb = (int)type_base[t];
            if (nth == 1) {
                for (int i = 0; i < ne; ++i) {
                    const int slot = cursor[(size_t)a[2 * i + 1] * T + t]++;
                    csr_src[slot] = a[2 * i];
                    csr_msg[slot] = mb + i;
                }
            } else {
                int dummy_cursor = 0, dummy_src = 0, dummy_msg = 0;   // see pass 1: select, do not branch
                int* const cur = cursor.data();
                const unsigned span = (unsigned)(v1 - v0);
                for (int i = 0; i < ne; ++i) {
                    const int d = a[2 * i + 1];
                    const bool mine = (unsigned)(d - v0) < span;
                    int* pc = mine ? cur + ((size_t)d * T + t) : &dummy_cursor;
                    const int slot = *pc;
                    *pc = slot + 1;
                    *(mine ? csr_src + slot : &dummy_src) = a[2 * i];
                    *(mine ? csr_msg + slot : &dummy_msg) = mb + i;
                }
            }
        }
        if (pair) {   // one sequential pass over the range's rows: no message -> -1, one -> its source, several -> virtual row
            int vid = (int)part_nv[k], vm = (int)part_nvm[k];
            for (int i = tb[k]; i < tb[k + 1]; ++i) {
                tvp[i] = vid;
                size_t r = (size_t)tile_start[i] * T;
                const size_t rend = (size_t)tile_start[i + 1] * T, rpad = (size_t)(i + 1) * ts::TILE_M * T;
                for (; r < rend; ++r) {
                    const int b = row_ptr[r], cnt = row_ptr[r + 1] - b;
                    if (cnt == 0) pair[r] = -1;
                    else if (cnt == 1) pair[r] = csr_src[b];
                    else {
                        pair[r] = -(2 + vid);
                        vinfo[8 * vid] = cnt;
                        for (int m = 0; m < 7; ++m) vinfo[8 * vid + 1 + m] = m < cnt ? csr_src[b + m] : 0;
                        for (int m = 0; m < cnt; ++m) vsrc[vm++] = csr_src[b + m];
                        vptr[++vid] = vm;
                    }
                }
                for (; r < rpad; ++r) pair[r] = -1;   // rows of the last tile beyond V
            }
            if (k == nth - 1) tvp[ntiles] = vid;
        }
        if (v1 > v0) memcpy(h_indeg + (size_t)v0 * T, indeg + (size_t)v0 * T, sizeof(float) * (size_t)(v1 - v0) * T);
        for (int v = v0; v < v1; ++v) {
            const float* row = indeg + (size_t)v * T;
            float s = 0.0f;  // tf.reduce_sum over the type axis in fp32 (sparse:207), then + SMALL_NUMBER (:209)
            for (int t = 0; t < T; ++t) s += row[t];
            h_denom[v] = s + 1e-7f;
        }
    }
    if (ntiles == 0) {
        h_tiles[0] = 0;
        if (pair) { for (size_t r = 0; r < (size_t)ts::TILE_M * T; ++r) pair[r] = -1; tvp[0] = 0; }
    }
    lap("csr fill", t_lap);
    if (e->has_transpose) {   // messages keyed by (source, type): the scatter of the backward pass becomes a gather
        int* trow = (int*)(base + e->off_trow);
        int* ttgt = (int*)(base + e->off_ttgt);
        std::vector<int> cnt((size_t)V * T + 1, 0);
        for (int t = 0; t < T; ++t)
            for (int i = 0; i < num_edges[t]; ++i) ++cnt[(size_t)adj[t][2 * i] * T + t + 1];
        trow[0] = 0;
        for (size_t k = 1; k <= (size_t)V * T; ++k) trow[k] = trow[k - 1] + cnt[k];
        for (size_t k = 0; k < (size_t)V * T; ++k) cnt[k] = trow[k];
        std::vector<int> slot_of_msg;
        int* tslot = e->use_att ? (int*)(base + e->off_tslot) : nullptr;
        if (tslot) {
            slot_of_msg.resize((size_t)std::max<int64_t>(M, 1));
            for (int64_t k = 0; k < M; ++k) slot_of_msg[csr_msg[k]] = (int)k;
        }
        int m = 0;
        for (int t = 0; t < T; ++t)
            for (int i = 0; i < num_edges[t]; ++i, ++m) {
                const int j = cnt[(size_t)adj[t][2 * i] * T + t]++;
                ttgt[j] = adj[t][2 * i + 1];
                if (tslot) tslot[j] = slot_of_msg[m];
            }
    }
    lap("denom+masks+extra", t_lap);
    g->valid = true;
    return GGNN_OK;
}

// Model shape (what ggnn_create fixed) -> the shadow engine of a prepared graph.
static void copy_model_shape(ggnn_engine* dst, const ggnn_engine* src) {
    dst->D = src->D; dst->T = src->T; dst->L = src->L; dst->DP = src->DP;
    memcpy(dst->steps, src->steps, sizeof dst->steps); memcpy(dst->nres, src->nres, sizeof dst->nres);
    memcpy(dst->res, src->res, sizeof dst->res); memcpy(dst->step_base, src->step_base, sizeof dst->step_base);
    dst->total_steps = src->total_steps;
    dst->use_bias = src->use_bias; dst->use_avg = src->use_avg; dst->cell = src->cell; dst->act = src->act;
    dst->precision = src->precision; dst->device = src->device; dst->num_sms = src->num_sms; dst->max_smem = src->max_smem;
    dst->use_att = src->use_att;
    dst->save = src->save;   // decides whether the source-keyed CSR of the backward pass is part of the image
}

// Batch / tile-plan fields (everything build_plan and build_sparse_image derive from a batch) -> the engine that uploads the image.
static void adopt_plan(ggnn_engine* dst, const ggnn_engine* src) {
    dst->V = src->V; dst->M = src->M; dst->gather_mode = src->gather_mode; dst->dense_v = src->dense_v;
    dst->variant = src->variant; dst->nb1 = src->nb1; dst->local = src->local; dst->ntiles = src->ntiles;
    dst->max_span = src->max_span; dst->max_tile_msgs = src->max_tile_msgs; dst->plan_text = src->plan_text;
    dst->stream = src->stream;
    for (int i = 0; i < 2; ++i) { dst->ts_nc[i] = src->ts_nc[i]; dst->ts_nblk[i] = src->ts_nblk[i]; }
    dst->ts_nv = src->ts_nv; dst->tc_row_budget = src->tc_row_budget; dst->tc_kgs = src->tc_kgs;
    dst->off_row_ptr = src->off_row_ptr; dst->off_src = src->off_src; dst->off_msg = src->off_msg; dst->off_indeg = src->off_indeg;
    dst->off_denom = src->off_denom; dst->off_tiles = src->off_tiles; dst->off_mask = src->off_mask; dst->off_adj = src->off_adj;
    dst->has_transpose = src->has_transpose; dst->off_trow = src->off_trow; dst->off_ttgt = src->off_ttgt; dst->off_tslot = src->off_tslot;
    dst->off_pair = src->off_pair; dst->off_vptr = src->off_vptr; dst->off_vsrc = src->off_vsrc; dst->off_tvp = src->off_tvp;
    dst->off_vinfo = src->off_vinfo;
    memcpy(dst->edges_of_type, src->edges_of_type, sizeof dst->edges_of_type);
}

int ggnn_free_prepared_graph(ggnn_prepared_graph* g) {
    if (!g) return GGNN_OK;
    if (g->use_cuda) {
        cudaSetDevice(g->plan.device);
        if (g->uploaded) { cudaEventSynchronize(g->uploaded); cudaEventDestroy(g->uploaded); }
        g->stage.release();
    }
    delete g;
    return GGNN_OK;
}

const char* ggnn_prepared_graph_error(const ggnn_prepared_graph* g) { return g ? g->plan.err.c_str() : "null prepared graph"; }

int ggnn_host_prepare_graph_sparse(const ggnn_config* cfg, int32_t num_sms, int32_t save_for_backward, int32_t V, const int32_t* const* adj,
                                   const int32_t* num_edges, const float* indeg, ggnn_prepared_graph** inout) {
    if (!cfg || !inout || num_sms <= 0) return GGNN_EINVAL;
    ggnn_prepared_graph* g = *inout;
    if (!g) { g = new ggnn_prepared_graph(); *inout = g; }
    g->use_cuda = false;
    g->valid = false;
    if (int rc = init_model_shape(&g->plan, cfg, g->plan.err)) return rc;
    g->plan.num_sms = num_sms; g->plan.max_smem = 227 * 1024;
    g->plan.save = save_for_backward != 0;
    return build_sparse_image(g, V, adj, num_edges, indeg);
}

int ggnn_prepared_graph_info(const ggnn_prepared_graph* g, int32_t* num_nodes, int64_t* num_messages, int32_t* num_tiles, int64_t* image_bytes,
                             int32_t* is_streaming, char* plan_text, int32_t plan_text_capacity) {
    if (!g || !g->valid) return GGNN_ESTATE;
    if (num_nodes) *num_nodes = g->plan.V;
    if (num_messages) *num_messages = g->plan.M;
    if (num_tiles) *num_tiles = g->plan.ntiles;
    if (image_bytes) *image_bytes = (int64_t)g->bytes;
    if (is_streaming) *is_streaming = g->plan.stream ? 1 : 0;
    if (plan_text && plan_text_capacity > 0) snprintf(plan_text, (size_t)plan_text_capacity, "%s", g->plan.plan_text.c_str());
    return GGNN_OK;
}

int ggnn_prepared_graph_arrays(const ggnn_prepared_graph* g, int32_t* row_ptr, int32_t* src, int32_t* msg, int32_t* tile_start, float* denom,
                               int32_t* pair_src) {
    if (!g || !g->valid) return GGNN_ESTATE;
    const ggnn_engine& q = g->plan;
    const char* base = g->image;
    const size_t V = (size_t)q.V, T = (size_t)q.T, M = (size_t)q.M;
    if (row_ptr) memcpy(row_ptr, base + q.off_row_ptr, sizeof(int) * (V * T + 1));
    if (src && M) memcpy(src, base + q.off_src, sizeof(int) * M);
    if (msg && M) memcpy(msg, base + q.off_msg, sizeof(int) * M);
    if (tile_start) memcpy(tile_start, base + q.off_tiles, sizeof(int) * (size_t)(q.ntiles + 1));
    if (denom && V) memcpy(denom, base + q.off_denom, sizeof(float) * V);
    if (pair_src && q.stream) memcpy(pair_src, base + q.off_pair, sizeof(int) * (size_t)std::max(q.ntiles, 1) * ts::TILE_M * T);
    return GGNN_OK;
}

int ggnn_prepared_graph_image(const ggnn_prepared_graph* g, void* dst, int64_t capacity) {
    if (!g || !g->valid || !dst) return GGNN_ESTATE;
    if (capacity < (int64_t)g->bytes) return GGNN_EINVAL;
    memcpy(dst, g->image, g->bytes);
    return GGNN_OK;
}

int ggnn_prepare_graph_sparse(const ggnn_engine* e, int32_t save_for_backward, int32_t V, const int32_t* const* adj, const int32_t* num_edges,
                              const float* indeg, ggnn_prepared_graph** inout) {
    if (!e || !inout) return GGNN_EINVAL;
    ggnn_prepared_graph* g = *inout;
    if (!g) { g = new ggnn_prepared_graph(); *inout = g; }
    g->use_cuda = true;
    copy_model_shape(&g->plan, e);
    if (save_for_backward >= 0) g->plan.save = save_for_backward != 0;   // a producer thread says what the batch will be used for
    if (cudaSetDevice(e->device) != cudaSuccess) return g->plan.fail(GGNN_ECUDA, "cudaSetDevice(%d) failed", e->device);   // this may be a producer thread
    return build_sparse_image(g, V, adj, num_edges, indeg);
}

int ggnn_set_graph_prepared(ggnn_engine* e, ggnn_prepared_graph* g, ggnn_stream_t stream) {
    if (!e) return GGNN_EINVAL;
    e->graph_set = false; e->saved_valid = false;
    if (!g || !g->valid) return e->fail(GGNN_ESTATE, "the prepared graph is empty (its build failed or never ran)");
    const ggnn_engine& q = g->plan;
    if (q.D != e->D || q.T != e->T || q.precision != e->precision || q.DP != e->DP || q.num_sms != e->num_sms || q.cell != e->cell || q.use_att != e->use_att)
        return e->fail(GGNN_EINVAL, "the prepared graph was built for a different engine configuration");
    if (e->save && !q.has_transpose)
        return e->fail(GGNN_ESTATE, "save_for_backward is on but the graph was prepared without it (the source-keyed CSR is built at prepare time)");
    CU_TRY(e, cudaSetDevice(e->device));
    adopt_plan(e, &q);
    cudaStream_t st = (cudaStream_t)stream;
    CU_TRY(e, e->graph_buf.reserve(g->bytes));
    CU_TRY(e, cudaMemcpyAsync(e->graph_buf.ptr, g->image, g->bytes, cudaMemcpyHostToDevice, st));
    if (g->use_cuda) {
        if (!g->uploaded) CU_TRY(e, cudaEventCreateWithFlags(&g->uploaded, cudaEventDisableTiming));
        CU_TRY(e, cudaEventRecord(g->uploaded, st));
    } else {
        CU_TRY(e, cudaStreamSynchronize(st));   // a pageable image (host-only construction) must be consumed before the caller may reuse it
    }
    int rc = reserve_states(e);
    if (rc) return rc;
    e->graph_set = true;
    return GGNN_OK;
}

int ggnn_set_graph_sparse(ggnn_engine* e, int32_t V, const int32_t* const* adj, const int32_t* num_edges,
                          const float* indeg, ggnn_stream_t stream) {
    if (!e) return GGNN_EINVAL;
    e->graph_set = false; e->saved_valid = false;
    // the same two halves a caller can run on two threads: build into the engine's own prepared graph, then upload it
    int rc = ggnn_prepare_graph_sparse(e, -1, V, adj, num_edges, indeg, &e->own_prep);
    if (rc) { if (e->own_prep) e->err = e->own_prep->plan.err; return rc; }
    return ggnn_set_graph_prepared(e, e->own_prep, stream);
}


// The reference only ever feeds 0/1 adjacency (dense:30-36).  A binary adjacency IS an edge list: A_t.(h W_t + b_t) =
// (sum of h over the row's sources) W_t + rowsum(A_t) b_t, which is exactly the sparse path with in-degree = row sums.  One scan of
// [b, T, v, v] -> per-type (source, target) lists in the order (graph, target row, source column) and the row sums; false when an entry is
// neither 0 nor 1 (a weighted matrix keeps the matrix walk).
// The scan is a stream over b*T*v*v floats (4 MB at cfg3) of which ~99 % are zero: memory-bound on one core (~0.5 ms), so the
// graphs are split into contiguous ranges over a few OpenMP threads; every thread appends to its own per-type lists (order inside
// a range: graph, target row, source column) and the ranges are concatenated in order -- the result is the single-thread list.
static bool scan_binary_dense(int T, int b, int v, const float* adjm, std::vector<std::vector<int32_t>>& lists, std::vector<float>& indeg) {
    const int V = b * v;
    bool binary = true;
    lists.assign(T, std::vector<int32_t>());
    {
    indeg.assign((size_t)std::max(V, 1) * T, 0.0f);
    int nthreads = 1;   // graph ranges scanned concurrently
    int team = 1;       // OpenMP team size: ONE size per process (the sparse builder's), used only if its region entry is cheap here
#ifdef _OPENMP
    team = b >= 16 ? host_team_size() : 1;
    if (team > 1 && !host_team_is_fast(team)) team = 1;
    nthreads = std::max(1, std::min(team, b / 8));
    if (const char* nt = getenv("GGNN_HOST_THREADS")) { nthreads = std::max(1, std::min(atoi(nt), std::max(b, 1))); team = nthreads; }
#endif
    std::vector<std::vector<std::vector<int32_t>>> part(nthreads, std::vector<std::vector<int32_t>>(T));
    std::vector<int> bad(nthreads, 0);
    const int chunk = (b + nthreads - 1) / std::max(nthreads, 1);
#ifdef _OPENMP
#pragma omp parallel for schedule(static, 1) num_threads(team) if (team > 1)
#endif
    for (int k = 0; k < nthreads; ++k) {
        std::vector<std::vector<int32_t>>& mine = part[k];
        const int g0 = k * chunk, g1 = std::min(b, g0 + chunk);
        for (int t = 0; t < T; ++t) mine[t].reserve((size_t)std::max(g1 - g0, 0) * v * 3);
        bool ok = true;
        for (int g = g0; g < g1 && ok; ++g)
            for (int t = 0; t < T && ok; ++t) {
                const float* m = adjm + ((size_t)g * T + t) * v * v;
                std::vector<int32_t>& lst = mine[t];
                for (int i = 0; i < v && ok; ++i) {
                    const float* row = m + (size_t)i * v;
                    int cnt = 0;
                    auto visit = [&](int j) {
                        const float a = row[j];
                        if (a != 0.0f) {
                            if (a != 1.0f) { ok = false; return; }
                            lst.push_back(g * v + j);   // source
                            lst.push_back(g * v + i);   // target
                            ++cnt;
                        }
                    };
                    int j = 0;
                    for (; j + 4 <= v && ok; j += 4) {   // test 16 bytes at a time
                        uint64_t w0, w1;
                        memcpy(&w0, row + j, 8); memcpy(&w1, row + j + 2, 8);
                        if ((w0 | w1) == 0) continue;
                        visit(j); visit(j + 1); visit(j + 2); visit(j + 3);
                    }
                    for (; j < v && ok; ++j) visit(j);
                    indeg[((size_t)g * v + i) * T + t] = (float)cnt;
                }
            }
        bad[k] = ok ? 0 : 1;
    }
    for (int k = 0; k < nthreads; ++k) binary = binary && !bad[k];
    if (binary)
        for (int t = 0; t < T; ++t) {
            size_t total = 0;
            for (int k = 0; k < nthreads; ++k) total += part[k][t].size();
            lists[t].resize(total);
            size_t off = 0;
            for (int k = 0; k < nthreads; ++k) {
                if (!part[k][t].empty()) memcpy(lists[t].data() + off, part[k][t].data(), part[k][t].size() * sizeof(int32_t));
                off += part[k][t].size();
            }
        }
    }
    return binary;
}

// Host half of ggnn_set_graph_dense for a 0/1 adjacency: scan -> edge lists -> the sparse builder.  *not_binary tells a weighted matrix
// (GGNN_EUNSUPPORTED) from a real failure.
static int prepare_dense_into(ggnn_prepared_graph* g, int32_t b, int32_t v, const float* adjm, bool* not_binary) {
    ggnn_engine* q = &g->plan;
    g->valid = false;
    *not_binary = false;
    if (b < 0 || v <= 0 || (!adjm && b > 0)) return q->fail(GGNN_EINVAL, "null/negative argument");
    if (q->use_att) return q->fail(GGNN_EUNSUPPORTED, "propagation attention exists only in the sparse model (sparse:170-196)");
    const int T = q->T;
    if ((int64_t)b * v > 0x7fffffff / std::max(T, 1)) return q->fail(GGNN_EUNSUPPORTED, "batch too large for int32 indexing");
    std::vector<std::vector<int32_t>> lists;
    std::vector<float> indeg;
    if (getenv("GGNN_DENSE_KEEP_MATRIX") || !scan_binary_dense(T, b, v, adjm, lists, indeg)) {
        *not_binary = true;
        return q->fail(GGNN_EUNSUPPORTED, "the adjacency matrix is not 0/1: a weighted matrix is fed through ggnn_set_graph_dense (matrix walk)");
    }
    std::vector<const int32_t*> ptrs(T);
    std::vector<int32_t> counts(T);
    for (int t = 0; t < T; ++t) { ptrs[t] = lists[t].data(); counts[t] = (int32_t)(lists[t].size() / 2); }
    int rc = build_sparse_image(g, b * v, ptrs.data(), counts.data(), indeg.data());
    if (rc) return rc;
    q->dense_v = v;
    q->plan_text += " [binary dense adjacency -> CSR]";
    return GGNN_OK;
}

int ggnn_prepare_graph_dense(const ggnn_engine* e, int32_t save_for_backward, int32_t b, int32_t v, const float* adjm, ggnn_prepared_graph** inout) {
    if (!e || !inout) return GGNN_EINVAL;
    ggnn_prepared_graph* g = *inout;
    if (!g) { g = new ggnn_prepared_graph(); *inout = g; }
    g->use_cuda = true;
    copy_model_shape(&g->plan, e);
    if (save_for_backward >= 0) g->plan.save = save_for_backward != 0;
    if (cudaSetDevice(e->device) != cudaSuccess) return g->plan.fail(GGNN_ECUDA, "cudaSetDevice(%d) failed", e->device);
    bool not_binary = false;
    return prepare_dense_into(g, b, v, adjm, &not_binary);
}

int ggnn_host_prepare_graph_dense(const ggnn_config* cfg, int32_t num_sms, int32_t save_for_backward, int32_t b, int32_t v, const float* adjm,
                                  ggnn_prepared_graph** inout) {
    if (!cfg || !inout || num_sms <= 0) return GGNN_EINVAL;
    ggnn_prepared_graph* g = *inout;
    if (!g) { g = new ggnn_prepared_graph(); *inout = g; }
    g->use_cuda = false;
    g->valid = false;
    if (int rc = init_model_shape(&g->plan, cfg, g->plan.err)) return rc;
    g->plan.num_sms = num_sms; g->plan.max_smem = 227 * 1024;
    g->plan.save = save_for_backward != 0;
    bool not_binary = false;
    return prepare_dense_into(g, b, v, adjm, &not_binary);
}

int ggnn_set_graph_dense(ggnn_engine* e, int32_t b, int32_t v, const float* adjm, ggnn_stream_t stream) {
    if (!e) return GGNN_EINVAL;
    e->graph_set = false; e->saved_valid = false;
    if (b < 0 || v <= 0 || (!adjm && b > 0)) return e->fail(GGNN_EINVAL, "null/negative argument");
    if (e->use_att) return e->fail(GGNN_EUNSUPPORTED, "propagation attention exists only in the sparse model (sparse:170-196)");
    CU_TRY(e, cudaSetDevice(e->device));
    const int T = e->T;
    if ((int64_t)b * v > 0x7fffffff / std::max(T, 1)) return e->fail(GGNN_EUNSUPPORTED, "batch too large for int32 indexing");
    const int V = b * v;
    {   // a 0/1 adjacency (all the reference feeds) takes the CSR path: the same two halves as ggnn_set_graph_sparse, on the engine's own prepared graph
        if (!e->own_prep) e->own_prep = new ggnn_prepared_graph();
        ggnn_prepared_graph* g = e->own_prep;
        g->use_cuda = true;
        copy_model_shape(&g->plan, e);
        bool not_binary = false;
        const int rc = prepare_dense_into(g, b, v, adjm, &not_binary);
        if (rc == GGNN_OK) return ggnn_set_graph_prepared(e, g, stream);
        if (!not_binary) { e->err = g->plan.err; return rc; }
    }
    e->V = V; e->M = 0; e->gather_mode = GATHER_DENSE; e->dense_v = v;
    e->has_transpose = true;   // the dense adjacency is its own transpose source
    for (int t = 0; t < T; ++t) e->edges_of_type[t] = 1;
    std::vector<int> cuts;
    for (int g = 0; g <= b; ++g) cuts.push_back(g * v);
    if (b == 0) cuts.assign(1, 0);
    std::vector<int> tile_start;
    int rc = build_plan(e, cuts, tile_start);
    if (rc) return rc;
    const int ntiles = e->ntiles;
    const size_t adj_elems = (size_t)b * T * v * v;
    size_t off = 0;
    e->off_row_ptr = off; off = align_up(off + 16, 16);
    e->off_src = off; e->off_msg = off;
    e->off_indeg = off;   off = align_up(off + sizeof(float) * (size_t)std::max(V, 1) * T, 16);
    e->off_denom = off;   off = align_up(off + sizeof(float) * (size_t)std::max(V, 1), 16);
    e->off_tiles = off;   off = align_up(off + sizeof(int) * (size_t)(ntiles + 1), 16);
    e->off_mask = off;    off = align_up(off + sizeof(unsigned) * (size_t)std::max(ntiles, 1), 16);
    e->off_adj = off;     off = align_up(off + sizeof(float) * std::max<size_t>(adj_elems, 1), 16);
    if (e->stage_done) CU_TRY(e, cudaEventSynchronize(e->stage_done));   // previous upload may still be reading the stage
    CU_TRY(e, e->graph_stage.reserve(off));
    char* base = (char*)e->graph_stage.ptr;
    float* h_indeg = (float*)(base + e->off_indeg);
    float* h_denom = (float*)(base + e->off_denom);
    int* h_tiles = (int*)(base + e->off_tiles);
    unsigned* h_mask = (unsigned*)(base + e->off_mask);
    float* h_adj = (float*)(base + e->off_adj);
    if (adj_elems) memcpy(h_adj, adjm, sizeof(float) * adj_elems);
    // in-degree per type = row sums of A_t (the dense model adds the bias to every source row before A.m,
    // dense:107-112, which equals bias * row-sum after the adjacency product)
    for (int g = 0; g < b; ++g)
        for (int i = 0; i < v; ++i) {
            float tot = 0.0f;
            for (int t = 0; t < T; ++t) {
                const float* row = adjm + (((size_t)g * T + t) * v + i) * v;
                float s = 0.0f;
                for (int j = 0; j < v; ++j) s += row[j];
                h_indeg[((size_t)g * v + i) * T + t] = s;
                tot += s;
            }
            h_denom[(size_t)g * v + i] = tot + 1e-7f;
        }
    for (int i = 0; i <= ntiles; ++i) h_tiles[i] = tile_start[i];
    for (int i = 0; i < ntiles; ++i) {
        unsigned mask = 0;
        for (int n = tile_start[i]; n < tile_start[i + 1]; ++n)
            for (int t = 0; t < T; ++t)
                if (h_indeg[(size_t)n * T + t] != 0.0f) mask |= 1u << t;
        // rows with cancelling +/- entries would have zero row-sum but non-zero entries: scan those rows fully
        if (mask != ((T >= 32) ? 0xffffffffu : ((1u << T) - 1u))) {
            for (int n = tile_start[i]; n < tile_start[i + 1]; ++n) {
                const int g = n / v, ii = n % v;
                for (int t = 0; t < T; ++t) {
                    if (mask & (1u << t)) continue;
                    const float* row = adjm + (((size_t)g * T + t) * v + ii) * v;
                    for (int j = 0; j < v; ++j) if (row[j] != 0.0f) { mask |= 1u << t; break; }
                }
            }
        }
        h_mask[i] = mask;
    }
    rc = upload_graph(e, off, (cudaStream_t)stream);
    if (rc) return rc;
    rc = reserve_states(e);
    if (rc) return rc;
    e->graph_set = true;
    return GGNN_OK;
}

static void fill_params(ggnn_engine* e, FwdParams& p, const float* h0, float* h_out) {
    memset(&p, 0, sizeof p);
    p.V = e->V; p.D = e->D; p.T = e->T; p.L = e->L;
    p.use_bias = e->use_bias; p.use_avg = e->use_avg; p.cell = e->cell; p.act = e->act;
    p.gather_mode = e->gather_mode; p.dense_v = e->dense_v; p.save = e->save ? 1 : 0;
    p.drop_keep = e->drop_keep; p.drop_seed = e->drop_seed;
    p.use_att = e->use_att; p.att = (float*)e->att_buf.ptr; p.att_stride = e->save ? (size_t)std::max<int64_t>(e->M, 1) : 0;
    char* g = (char*)e->graph_buf.ptr;
    p.tile_start = (const int*)(g + e->off_tiles);
    p.tile_mask = (const unsigned*)(g + e->off_mask);
    p.row_ptr = (const int*)(g + e->off_row_ptr);
    p.csr_src = (const int*)(g + e->off_src);
    p.dense_adj = (const float*)(g + e->off_adj);
    p.indeg = (const float*)(g + e->off_indeg);
    p.denom = (const float*)(g + e->off_denom);
    const size_t vd = (size_t)std::max(e->V, 1) * e->D;
    float* sb = (float*)e->state_buf.ptr;
    p.state[0] = h0; p.state_w[0] = nullptr;
    for (int l = 1; l <= e->L; ++l) {
        float* ptr = (l == e->L) ? h_out : sb + (size_t)(l - 1) * vd;
        p.state[l] = ptr; p.state_w[l] = ptr;
    }
    for (int l = 0; l < e->L; ++l) {
        LayerDev& ld = p.layer[l];
        ld.edge_w = e->w[l].edge_weights; ld.edge_b = e->w[l].edge_biases;
        ld.gate_k = e->w[l].gate_kernel; ld.gate_b = e->w[l].gate_bias;
        ld.cand_k = e->w[l].cand_kernel; ld.cand_b = e->w[l].cand_bias;
        ld.att_w = e->use_att ? e->w[l].edge_type_attention_weights : nullptr;
        ld.cand_hb = e->cell == CELL_CUDNN_GRU ? e->w[l].cand_hidden_bias : nullptr;
        ld.steps = e->steps[l]; ld.nres = e->nres[l];
        for (int i = 0; i < MAX_RES; ++i) ld.res[i] = e->res[l][i];
        p.step_base[l] = e->step_base[l];
    }
    if (e->save) {
        float* s = (float*)e->save_bufs.ptr;
        const size_t per = vd * (size_t)std::max(e->total_steps, 1);
        p.save_buf.h_in = s; p.save_buf.agg = s + per; p.save_buf.r = s + 2 * per; p.save_buf.u = s + 3 * per; p.save_buf.c = s + 4 * per;
        p.save_buf.q = e->cell == CELL_CUDNN_GRU ? s + 5 * per : nullptr;
    }
}


// ------------------------------------------------------------------------------------------ tensor-core path (host)
static int tc_prepare_weights(ggnn_engine* e, cudaStream_t st) {
    const int D = e->D, DP = e->DP, T = e->T, NKS = DP / 16;
    size_t off = 0;
    for (int l = 0; l < e->L; ++l) {
        const int nseg = e->nres[l] + 2;
        e->tc_off_edge[l] = off; off += (size_t)T * NKS * 64 * DP;
        e->tc_off_gate[l] = off; off += (size_t)nseg * NKS * 128 * DP;
        e->tc_off_cand[l] = off; off += (size_t)nseg * NKS * 64 * DP;
    }
    if (off > e->tc_weights.cap) e->weights_dirty = true;
    CU_TRY(e, e->tc_weights.reserve(off));
    if (!e->weights_dirty) return GGNN_OK;
    uint8_t* base = (uint8_t*)e->tc_weights.ptr;
    for (int l = 0; l < e->L; ++l) {
        const int nseg = e->nres[l] + 2;
        auto launch = [&](const float* W, uint8_t* out, int segs, int blks, int src_ld, int col0) {
            const long long total = (long long)segs * NKS * 2 * blks * DP;
            const int blocks = (int)std::min<long long>((total + 255) / 256, 1024);
            tc::ggnn_tile_weights_kernel<<<blocks, 256, 0, st>>>(W, out, D, DP, segs, blks, src_ld, col0);
            ++e->last_launches;
        };
        launch(e->w[l].edge_weights, base + e->tc_off_edge[l], T, 1, D, 0);
        if (e->cell == CELL_GRU) launch(e->w[l].gate_kernel, base + e->tc_off_gate[l], nseg, 2, 2 * D, 0);
        launch(e->w[l].cand_kernel, base + e->tc_off_cand[l], nseg, 1, D, 0);
    }
    CU_TRY(e, cudaGetLastError());
    e->weights_dirty = false;
    return GGNN_OK;
}

static int forward_tc(ggnn_engine* e, const float* h0, float* h_out, cudaStream_t st) {
    const int DP = e->DP;
    int rc = tc_prepare_weights(e, st);
    if (rc) return rc;
    bool any_res = false;
    for (int l = 0; l < e->L; ++l) any_res |= e->nres[l] > 0;
    if (any_res) CU_TRY(e, e->tc_respre.reserve((size_t)e->ntiles * tc::TILE_M * 3 * DP * sizeof(float)));
    tc::TcParams p;
    memset(&p, 0, sizeof p);
    p.V = e->V; p.D = e->D; p.DP = DP; p.T = e->T; p.L = e->L;
    p.use_bias = e->use_bias; p.use_avg = e->use_avg; p.cell = e->cell; p.act = e->act;
    p.gather_mode = e->gather_mode; p.dense_v = e->dense_v; p.save = e->save ? 1 : 0;
    p.nparts = e->precision == GGNN_PREC_BF16X3 ? 3 : 1;
    p.drop_keep = e->drop_keep; p.drop_seed = e->drop_seed;
    p.kgs = e->tc_kgs;
    const size_t opb = (size_t)DP * (size_t)p.kgs / 4, stage = (size_t)DP * 128;   // a ring slot = two 64*DP-byte K-step stages
    // tile-local sparse graphs: stage the tile's CSR slice in shared memory when it is small enough
    p.csr_cache = 0; p.csr_cap_msgs = 0;
    size_t csr_b = 0;
    if (e->local && e->gather_mode == GATHER_SPARSE && e->T <= 16 && e->max_tile_msgs <= 4096) {
        p.csr_cache = 1;
        p.csr_cap_msgs = (e->max_tile_msgs + 15) / 16 * 16;
        csr_b = (size_t)((tc::TILE_M * e->T + 1 + 7) & ~7) * 2 + (size_t)p.csr_cap_msgs;
    }
    const size_t bias_b = (size_t)3 * DP * sizeof(float) + csr_b + 64;
    const size_t avail = e->max_smem > 1024 ? e->max_smem - 1024 : 0;
    if (avail < 3 * opb + bias_b + stage) return e->fail(GGNN_EUNSUPPORTED, "not enough shared memory for the tensor-core tile (DP=%d)", DP);
    // two gather buffers; GGNN_TC_GBUFS=4 adds two more compact tiles so that every gather runs ahead of the previous type's MMAs
    // (measured: no gain -- cfg2 0.0870 vs 0.0862 ms, the G1 phase is bound by the gathers themselves, not by the number of buffers; opt-in)
    p.ngbuf = 2;
    if (const char* gb = getenv("GGNN_TC_GBUFS")) p.ngbuf = (atoi(gb) == 4 && e->local && p.kgs == 1024 && avail >= 5 * opb + bias_b + stage) ? 4 : 2;
    const size_t ops = (size_t)(p.ngbuf + 1) * opb;
    p.nstages = (int)std::min<size_t>(tc::MAX_STAGES, (avail - ops - bias_b) / stage);
    if (const char* ns = getenv("GGNN_TC_STAGES")) p.nstages = std::max(1, std::min(p.nstages, atoi(ns)));
    if (p.nstages < 1) return e->fail(GGNN_EUNSUPPORTED, "not enough shared memory for the weight ring (DP=%d)", DP);
    const size_t smem = ops + bias_b + (size_t)p.nstages * stage;
    char* g = (char*)e->graph_buf.ptr;
    p.tile_start = (const int*)(g + e->off_tiles);
    p.tile_mask = (const unsigned*)(g + e->off_mask);
    p.row_ptr = (const int*)(g + e->off_row_ptr);
    p.csr_src = (const int*)(g + e->off_src);
    p.dense_adj = (const float*)(g + e->off_adj);
    p.indeg = (const float*)(g + e->off_indeg);
    p.denom = (const float*)(g + e->off_denom);
    const size_t vd = (size_t)std::max(e->V, 1) * e->D;
    float* sb = (float*)e->state_buf.ptr;
    p.state[0] = h0;
    for (int l = 1; l <= e->L; ++l) {
        float* ptr = (l == e->L) ? h_out : sb + (size_t)(l - 1) * vd;
        p.state[l] = ptr; p.state_w[l] = ptr;
    }
    uint8_t* wb = (uint8_t*)e->tc_weights.ptr;
    for (int l = 0; l < e->L; ++l) {
        tc::TcLayer& ld = p.layer[l];
        ld.w_edge = wb + e->tc_off_edge[l]; ld.w_gate = wb + e->tc_off_gate[l]; ld.w_cand = wb + e->tc_off_cand[l];
        ld.edge_b = e->w[l].edge_biases; ld.gate_b = e->w[l].gate_bias; ld.cand_b = e->w[l].cand_bias;
        ld.steps = e->steps[l]; ld.nres = e->nres[l];
        for (int i = 0; i < MAX_RES; ++i) ld.res[i] = e->res[l][i];
        p.step_base[l] = e->step_base[l];
    }
    if (e->save) {
        float* s = (float*)e->save_bufs.ptr;
        const size_t per = vd * (size_t)std::max(e->total_steps, 1);
        p.save_buf.h_in = s; p.save_buf.agg = s + per; p.save_buf.r = s + 2 * per; p.save_buf.u = s + 3 * per; p.save_buf.c = s + 4 * per;
    }
    p.res_pre = (float*)e->tc_respre.ptr;
    p.error_flag = (int*)e->err_flag.ptr;
    p.dbg = nullptr;
    if (getenv("GGNN_TC_DEBUG_TIMING")) {
        CU_TRY(e, e->dbg_buf.reserve(512 * sizeof(long long)));
        CU_TRY(e, cudaMemsetAsync(e->dbg_buf.ptr, 0, 512 * sizeof(long long), st));
        p.dbg = (long long*)e->dbg_buf.ptr;
    }
    const size_t vd_bytes = (size_t)e->V * e->D * sizeof(float);
    if (e->local) {
        CU_TRY(e, cudaFuncSetAttribute(tc::ggnn_fwd_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tc::ggnn_fwd_tc_kernel<true><<<e->ntiles, tc::NTHREADS, smem, st>>>(p);
        ++e->last_launches;
    } else {
        CU_TRY(e, cudaFuncSetAttribute(tc::ggnn_fwd_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        float* tmp0 = sb + (size_t)(e->L - 1 > 0 ? e->L - 1 : 0) * vd;
        float* tmp1 = tmp0 + vd;
        for (int l = 0; l < e->L; ++l) {
            const float* in = p.state[l];
            if (e->steps[l] == 0) {
                CU_TRY(e, cudaMemcpyAsync(p.state_w[l + 1], in, vd_bytes, cudaMemcpyDeviceToDevice, st));
                continue;
            }
            for (int s = 0; s < e->steps[l]; ++s) {
                float* out = (s == e->steps[l] - 1) ? p.state_w[l + 1] : ((s & 1) ? tmp1 : tmp0);
                p.g_layer = l; p.g_step = s; p.g_in = in; p.g_out = out;
                tc::ggnn_fwd_tc_kernel<false><<<e->ntiles, tc::NTHREADS, smem, st>>>(p);
                ++e->last_launches;
                in = out;
            }
        }
    }
    CU_TRY(e, cudaGetLastError());
    if (e->save) { e->saved_valid = true; e->saved_drop_keep = e->drop_keep; e->saved_drop_seed = e->drop_seed; }
    return GGNN_OK;
}

// ------------------------------------------------------------------------------------------ streaming tensor-core path (host)
static int ts_prepare_weights(ggnn_engine* e, cudaStream_t st) {
    const int D = e->D, DP = e->DP, T = e->T, NKS = DP / 16;
    const int nc0 = e->ts_nc[0], nb0 = e->ts_nblk[0], nc1 = e->ts_nc[1], nb1 = e->ts_nblk[1];
    size_t off = 0;
    for (int l = 0; l < e->L; ++l) {
        const int nseg = e->nres[l] + 2;
        e->ts_off_edge[l] = off; off += (size_t)nb0 * T * NKS * 64 * nc0;
        e->ts_off_gate[l] = off; off += (size_t)nb1 * nseg * NKS * 64 * nc1;
        e->ts_off_cand[l] = off; off += (size_t)nb0 * nseg * NKS * 64 * nc0;
    }
    if (off > e->ts_weights.cap || e->ts_tiled_nc[0] != nc0 || e->ts_tiled_nc[1] != nc1) e->weights_dirty = true;
    CU_TRY(e, e->ts_weights.reserve(off));
    if (!e->weights_dirty) return GGNN_OK;
    uint8_t* base = (uint8_t*)e->ts_weights.ptr;
    for (int l = 0; l < e->L; ++l) {
        const int nseg = e->nres[l] + 2;
        auto launch = [&](const float* W, uint8_t* out, int segs, int ncolblk, int src_ld, int NC, int nblk) {
            const long long total = (long long)nblk * segs * NKS * 2 * NC;
            const int blocks = (int)std::min<long long>((total + 255) / 256, 2048);
            ts::ggnn_tile_weights_stream_kernel<<<blocks, 256, 0, st>>>(W, out, D, DP, segs, ncolblk, src_ld, NC, nblk);
            ++e->last_launches;
        };
        launch(e->w[l].edge_weights, base + e->ts_off_edge[l], T, 1, D, nc0, nb0);
        if (e->cell == CELL_GRU) launch(e->w[l].gate_kernel, base + e->ts_off_gate[l], nseg, 2, 2 * D, nc1, nb1);
        launch(e->w[l].cand_kernel, base + e->ts_off_cand[l], nseg, 1, D, nc0, nb0);
    }
    CU_TRY(e, cudaGetLastError());
    e->weights_dirty = false;
    e->ts_tiled_nc[0] = nc0; e->ts_tiled_nc[1] = nc1;
    return GGNN_OK;
}

static int forward_stream(ggnn_engine* e, const float* h0, float* h_out, cudaStream_t st) {
    const int D = e->D, DP = e->DP, T = e->T, L = e->L, V = e->V, NKS = DP / 16;
    const int ntiles = e->ntiles;
    int rc = ts_prepare_weights(e, st);
    if (rc) return rc;
    const size_t img_b = (size_t)ntiles * NKS * ts::A_STAGE_B;   // one operand image == one chunk-major fp32 copy, in bytes
    const int n_img = L + 1 + 4;    // images: node_states_per_layer, two step temporaries, agg, r*h
    const int n_chk = L + 1 + 3;    // chunk-major fp32: node_states_per_layer, two step temporaries, u
    CU_TRY(e, e->ts_images.reserve(img_b * (n_img + n_chk)));
    uint8_t* ib = (uint8_t*)e->ts_images.ptr;
    auto img_state = [&](int l) { return ib + (size_t)l * img_b; };
    uint8_t* img_tmp[2] = {ib + (size_t)(L + 1) * img_b, ib + (size_t)(L + 2) * img_b};
    uint8_t* img_agg = ib + (size_t)(L + 3) * img_b;
    uint8_t* img_rh = ib + (size_t)(L + 4) * img_b;
    uint8_t* cb = ib + (size_t)n_img * img_b;
    auto chk_state = [&](int l) { return (float*)(cb + (size_t)l * img_b); };
    float* chk_tmp[2] = {(float*)(cb + (size_t)(L + 1) * img_b), (float*)(cb + (size_t)(L + 2) * img_b)};
    float* u_chk = (float*)(cb + (size_t)(L + 3) * img_b);
    const size_t vd = (size_t)std::max(V, 1) * D;
    const size_t vd_bytes = (size_t)V * D * sizeof(float);
    float* sb = (float*)e->state_buf.ptr;
    std::vector<float*> state(L + 1);
    state[0] = const_cast<float*>(h0);
    for (int l = 1; l <= L; ++l) state[l] = (l == L) ? h_out : sb + (size_t)(l - 1) * vd;
    const bool gru = e->cell == CELL_GRU;
    float* sv = (float*)e->save_bufs.ptr;
    const size_t per = vd * (size_t)std::max(e->total_steps, 1);
    char* g = (char*)e->graph_buf.ptr;

    // shared-memory budgets
    const size_t avail = (e->max_smem > 2048 ? e->max_smem - 2048 : 0);
    const size_t csr_b = (size_t)ts::TILE_M * T * 4;   // the tile's (target, type) -> source table
    CU_TRY(e, e->ts_virt.reserve((size_t)((e->ts_nv + ts::TILE_M - 1) / ts::TILE_M + 1) * NKS * ts::A_STAGE_B));
    // a ring stage carries KS = 4 K-steps (the producer thread pays several hundred cycles per bulk copy whatever its size; measured on
    // cfg4 / its 1/8 shard / cfg5: KS = 4 beats 2 beats 1 even where only two 96 KB stages fit)
    const char* env_ks = getenv("GGNN_TS_KSTEPS");
    const char* env_ns = getenv("GGNN_TS_STAGES");
    auto ksteps_for = [&](int NC) { return std::max(1, std::min(env_ks ? atoi(env_ks) : 4, NKS)); };
    auto stage_bytes = [&](int NC) { return (size_t)ksteps_for(NC) * ((size_t)ts::A_STAGE_B + 64 * (size_t)NC); };
    auto stages_for = [&](int NC, size_t budget) { return (int)std::min<size_t>(env_ns ? (size_t)atoi(env_ns) : (size_t)ts::MAX_NS, budget / stage_bytes(NC)); };
    ts::StreamParams base;
    memset(&base, 0, sizeof base);
    base.V = V; base.D = D; base.DP = DP; base.T = T;
    base.nparts = e->precision == GGNN_PREC_BF16X3 ? 3 : 1;
    base.cell = e->cell; base.act = e->act; base.use_bias = e->use_bias; base.use_avg = e->use_avg;
    base.tile_mask = (const unsigned*)(g + e->off_mask);
    base.pair_src = (const int*)(g + e->off_pair); base.vrow_ptr = (const int*)(g + e->off_vptr);
    base.vsrc = (const int*)(g + e->off_vsrc); base.tile_vptr = (const int*)(g + e->off_tvp);
    base.vinfo = (const int4*)(g + e->off_vinfo);
    base.virt_img = (uint8_t*)e->ts_virt.ptr;
    // pairs with several messages are pre-summed into virtual rows by the prologue of every gather launch (GGNN_TS_VIRT=0: summed inside
    // the gather loop instead -- measured slower even on cfg5, where most pairs have two messages: 0.57 vs 0.50 ms)
    base.virt_rows = 1;
    if (const char* vr = getenv("GGNN_TS_VIRT")) base.virt_rows = vr[0] == '1';
    base.indeg = (const float*)(g + e->off_indeg); base.denom = (const float*)(g + e->off_denom);
    base.drop_keep = e->drop_keep; base.drop_seed = e->drop_seed;
    base.error_flag = (int*)e->err_flag.ptr;
    // optional per-CTA phase stamps, one slice per launch (tools/stream_trace.py)
    long long* dbg = nullptr;
    const size_t dbg_slice = (size_t)ntiles * std::max(e->ts_nblk[0], e->ts_nblk[1]) * 16;
    if (getenv("GGNN_TS_DEBUG")) {
        const size_t n = (dbg_slice + 2048) * (size_t)(3 * std::max(e->total_steps, 1));
        CU_TRY(e, e->dbg_buf.reserve(n * sizeof(long long)));
        CU_TRY(e, cudaMemsetAsync(e->dbg_buf.ptr, 0, n * sizeof(long long), st));
        dbg = (long long*)e->dbg_buf.ptr;
    }
    int dbg_launch = 0;
    long long* dbg2_cur = nullptr;   // per launch: [grid][16] phase stamps, then [256][8] K-step timeline of CTA (0,0)
    auto next_dbg = [&]() -> long long* {
        if (!dbg) return nullptr;
        long long* q = dbg + (dbg_slice + 2048) * (size_t)(dbg_launch++);
        dbg2_cur = q + dbg_slice;
        return q;
    };
    auto tmem_cols = [](int cols) { int c = 32; while (c < cols) c *= 2; return c; };
    // a TMA-fed launch whose N blocks would need more than one wave of CTAs lets every CTA compute two N blocks one after the other into two
    // TMEM accumulators: the epilogue of the first runs under the mainloop of the second (the gate GEMM of a full batch: 2 x 256 columns)
    auto passes_for = [&](int NC, int nblk) {
        int np = ((long long)ntiles * nblk > e->num_sms && nblk % 2 == 0 && 2 * NC <= 512) ? 2 : 1;
        if (const char* ev = getenv("GGNN_TS_PASSES")) np = (atoi(ev) == 2 && nblk % 2 == 0 && 2 * NC <= 512) ? 2 : 1;
        return np;
    };
    const int nc0 = e->ts_nc[0], nb0 = e->ts_nblk[0], nc1 = e->ts_nc[1], nb1 = e->ts_nblk[1];
    // one CTA per SM for all three kernels: the whole shared memory is the ring
    const int ns_edge = stages_for(nc0, avail > csr_b ? avail - csr_b : 0);
    const int ns_gate = stages_for(nc1, avail), ns_cand = stages_for(nc0, avail);
    if (ns_edge < 2 || ns_gate < 2 || ns_cand < 2) return e->fail(GGNN_EUNSUPPORTED, "not enough shared memory for the streaming ring (DP=%d)", DP);
    auto smem_of = [&](int NC, int ns, bool gather) { return (size_t)1024 + (size_t)ns * stage_bytes(NC) + (gather ? csr_b : 0); };
    auto k_edge = ts::ggnn_stream_kernel<16, true>;
    auto k_fed = ts::ggnn_stream_kernel<16, false>;   // 16 epilogue warps: the epilogue is bound by the latency of its operand loads
    const size_t sm_edge = smem_of(nc0, ns_edge, true);
    const size_t sm_fed = std::max(smem_of(nc1, ns_gate, false), smem_of(nc0, ns_cand, false));
    CU_TRY(e, cudaFuncSetAttribute(k_edge, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_edge));
    CU_TRY(e, cudaFuncSetAttribute(k_fed, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_fed));

    {   // node_states_per_layer[0] -> operand image
        const long long total = (long long)ntiles * ts::TILE_M * (DP / 8);
        ts::ggnn_image_kernel<<<(int)std::min<long long>((total + 255) / 256, 4096), 256, 0, st>>>(h0, img_state(0), chk_state(0), V, D, DP, ntiles);
        ++e->last_launches;
    }
    const uint8_t* wb = (const uint8_t*)e->ts_weights.ptr;
    for (int l = 0; l < L; ++l) {
        const uint8_t* img_in = img_state(l);
        const float* chk_in = chk_state(l);
        if (e->steps[l] == 0) {   // a layer without timesteps aliases the previous state (sparse:152)
            CU_TRY(e, cudaMemcpyAsync(state[l + 1], state[l], vd_bytes, cudaMemcpyDeviceToDevice, st));
            CU_TRY(e, cudaMemcpyAsync(img_state(l + 1), img_in, img_b, cudaMemcpyDeviceToDevice, st));
            CU_TRY(e, cudaMemcpyAsync(chk_state(l + 1), chk_in, img_b, cudaMemcpyDeviceToDevice, st));
            continue;
        }
        const int R = e->nres[l], nseg = R + 2;
        for (int s = 0; s < e->steps[l]; ++s) {
            const bool last = s == e->steps[l] - 1;
            float* out = last ? state[l + 1] : nullptr;   // the row-major copy exists only for node_states_per_layer entries
            uint8_t* img_out = last ? img_state(l + 1) : img_tmp[s & 1];
            float* chk_out = last ? chk_state(l + 1) : chk_tmp[s & 1];
            const int gs = e->step_base[l] + s;
            const size_t so = (size_t)gs * vd;
            // ---- aggregated messages
            ts::StreamParams p = base;
            p.epi = ts::EPI_AGG; p.NC = nc0; p.nstages = ns_edge; p.ksteps = ksteps_for(nc0); p.npass = 1; p.tmem_cols = tmem_cols(nc0);
            p.g_img = img_in; p.w = wb + e->ts_off_edge[l]; p.kt_all = T * NKS;
            p.bias = e->use_bias ? e->w[l].edge_biases : nullptr;
            p.img_out = img_agg; p.sv_agg = e->save ? sv + per + so : nullptr; p.gstep = gs; p.dbg = next_dbg(); p.dbg2 = dbg2_cur;
            k_edge<<<dim3(ntiles, nb0), 18 * 32, sm_edge, st>>>(p);
            ++e->last_launches;
            auto set_segs = [&](ts::StreamParams& q, const uint8_t* last_img) {
                q.nseg = nseg;
                for (int i = 0; i < R; ++i) q.seg[i] = img_state(e->res[l][i]);
                q.seg[R] = img_agg; q.seg[R + 1] = last_img;
                q.kt_all = nseg * NKS;
            };
            if (gru) {
                ts::StreamParams q = base;
                q.epi = ts::EPI_GATE; q.NC = nc1; q.nstages = ns_gate; q.ksteps = ksteps_for(nc1); q.npass = passes_for(nc1, nb1); q.tmem_cols = tmem_cols(nc1 * q.npass);
                set_segs(q, img_in);
                q.w = wb + e->ts_off_gate[l]; q.bias = e->w[l].gate_bias; q.h_chk = chk_in; q.u_buf = u_chk; q.img_out = img_rh;
                if (e->save) { q.sv_r = sv + 2 * per + so; q.sv_h = sv + so; q.sv_u = sv + 3 * per + so; }
                q.gstep = gs; q.dbg = next_dbg(); q.dbg2 = dbg2_cur;
                k_fed<<<dim3(ntiles, nb1 / q.npass), 18 * 32, smem_of(nc1, ns_gate, false), st>>>(q);
                ++e->last_launches;
            }
            ts::StreamParams c = base;
            c.epi = ts::EPI_CAND; c.NC = nc0; c.nstages = ns_cand; c.ksteps = ksteps_for(nc0); c.npass = passes_for(nc0, nb0); c.tmem_cols = tmem_cols(nc0 * c.npass);
            set_segs(c, gru ? img_rh : img_in);
            c.w = wb + e->ts_off_cand[l]; c.bias = e->w[l].cand_bias; c.h_chk = chk_in; c.u_buf = u_chk; c.h_chk_out = chk_out; c.h_out = out; c.img_out = img_out;
            if (e->save) { if (gru) c.sv_c = sv + 4 * per + so; else c.sv_h = sv + so; }
            c.gstep = gs; c.dbg = next_dbg(); c.dbg2 = dbg2_cur;
            k_fed<<<dim3(ntiles, nb0 / c.npass), 18 * 32, smem_of(nc0, ns_cand, false), st>>>(c);
            ++e->last_launches;
            img_in = img_out; chk_in = chk_out;
        }
    }
    CU_TRY(e, cudaGetLastError());
    if (e->save) { e->saved_valid = true; e->saved_drop_keep = e->drop_keep; e->saved_drop_seed = e->drop_seed; }
    return GGNN_OK;
}

int ggnn_forward(ggnn_engine* e, const float* h0, float* h_out, ggnn_stream_t stream) {
    if (!e) return GGNN_EINVAL;
    if (!e->weights_set) return e->fail(GGNN_ESTATE, "ggnn_set_weights has not been called");
    if (!e->graph_set) return e->fail(GGNN_ESTATE, "no graph set (ggnn_set_graph_sparse/dense)");
    if ((!h0 || !h_out) && e->V > 0) return e->fail(GGNN_EINVAL, "null state pointer");
    if (((uintptr_t)h0 & 15) || ((uintptr_t)h_out & 15)) return e->fail(GGNN_EINVAL, "state pointers must be 16-byte aligned");
    CU_TRY(e, cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    e->last_launches = 0;
    e->last_h0 = h0; e->last_out = h_out; e->saved_valid = false;
    // an empty batch or a model without timesteps saves nothing, but ggnn_backward must still accept it (d_h0 = d_h_out)
    auto mark_saved = [e]() { if (e->save) { e->saved_valid = true; e->saved_drop_keep = e->drop_keep; e->saved_drop_seed = e->drop_seed; } };
    if (e->V == 0) { mark_saved(); return GGNN_OK; }
    if (e->save) { int rc = reserve_states(e); if (rc) return rc; }
    const size_t vd_bytes = (size_t)e->V * e->D * sizeof(float);
    if (e->total_steps == 0) {  // no propagation at all: result is the input (sparse:152 with empty loops)
        if (h_out != h0) CU_TRY(e, cudaMemcpyAsync(h_out, h0, vd_bytes, cudaMemcpyDeviceToDevice, st));
        mark_saved();
        return GGNN_OK;
    }
    if (e->precision != GGNN_PREC_FP32) return e->stream ? forward_stream(e, h0, h_out, st) : forward_tc(e, h0, h_out, st);
    if (e->use_att) {
        if (e->gather_mode != GATHER_SPARSE) return e->fail(GGNN_EUNSUPPORTED, "propagation attention needs the sparse graph format");
        CU_TRY(e, e->att_buf.reserve(sizeof(float) * (size_t)std::max<int64_t>(e->M, 1) * (size_t)(e->save ? std::max(e->total_steps, 1) : 1)));
    }
    FwdParams p;
    fill_params(e, p, h0, h_out);
    FwdKernel k = pick_fwd_kernel(e->variant, e->nb1, e->local);
    if (!k) return e->fail(GGNN_EUNSUPPORTED, "no kernel for variant=%d nb1=%d", e->variant, e->nb1);
    const size_t smem = fwd_smem_bytes(e->variant, e->nb1, e->D, e->T);
    CU_TRY(e, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int threads = 256;
    if (e->local) {
        // layers with zero timesteps just alias the previous state (sparse:152): copy afterwards
        k<<<e->ntiles, threads, smem, st>>>(p);
        ++e->last_launches;
    } else {
        const size_t vd = (size_t)e->V * e->D;
        float* tmp0 = (float*)e->state_buf.ptr + (size_t)(e->L - 1 > 0 ? e->L - 1 : 0) * vd;
        float* tmp1 = tmp0 + vd;
        for (int l = 0; l < e->L; ++l) {
            const float* in = p.state[l];
            if (e->steps[l] == 0) {
                CU_TRY(e, cudaMemcpyAsync(p.state_w[l + 1], in, vd_bytes, cudaMemcpyDeviceToDevice, st));
                continue;
            }
            for (int s = 0; s < e->steps[l]; ++s) {
                float* out = (s == e->steps[l] - 1) ? p.state_w[l + 1] : ((s & 1) ? tmp1 : tmp0);
                p.g_layer = l; p.g_step = s; p.g_in = in; p.g_out = out;
                k<<<e->ntiles, threads, smem, st>>>(p);
                ++e->last_launches;
                in = out;
            }
        }
    }
    CU_TRY(e, cudaGetLastError());
    if (e->save) { e->saved_valid = true; e->saved_drop_keep = e->drop_keep; e->saved_drop_seed = e->drop_seed; }
    return GGNN_OK;
}

int ggnn_forward_host_async(ggnn_engine* e, const float* h0_host, float* h_out_host, ggnn_stream_t stream) {
    if (!e) return GGNN_EINVAL;
    if (!e->graph_set) return e->fail(GGNN_ESTATE, "no graph set (ggnn_set_graph_sparse/dense)");
    if ((!h0_host || !h_out_host) && e->V > 0) return e->fail(GGNN_EINVAL, "null host pointer");
    CU_TRY(e, cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    const size_t bytes = (size_t)e->V * e->D * sizeof(float);
    const size_t slot = align_up(std::max<size_t>(bytes, 16), 256);
    CU_TRY(e, e->io_buf.reserve(2 * slot));
    float* d_in = (float*)e->io_buf.ptr;
    float* d_out = (float*)((char*)e->io_buf.ptr + slot);
    if (bytes) CU_TRY(e, cudaMemcpyAsync(d_in, h0_host, bytes, cudaMemcpyHostToDevice, st));
    int rc = ggnn_forward(e, d_in, d_out, stream);
    if (rc) return rc;
    if (bytes) CU_TRY(e, cudaMemcpyAsync(h_out_host, d_out, bytes, cudaMemcpyDeviceToHost, st));
    return GGNN_OK;
}

int ggnn_forward_host(ggnn_engine* e, const float* h0_host, float* h_out_host, ggnn_stream_t stream) {
    int rc = ggnn_forward_host_async(e, h0_host, h_out_host, stream);
    if (rc) return rc;
    CU_TRY(e, cudaStreamSynchronize((cudaStream_t)stream));
    return GGNN_OK;
}

}  // extern "C"

// One call per batch, the shape of the reference's sess.run(fetch, feed_dict) (chem_tensorflow.py:235): the h0 upload is
// enqueued FIRST so the host-side CSR build of set_graph overlaps it.
template <class SetGraph>
static int run_host(ggnn_engine* e, int64_t V, const float* h0_host, float* h_out_host, cudaStream_t st, SetGraph set_graph) {
    if (!e) return GGNN_EINVAL;
    if (V < 0 || ((!h0_host || !h_out_host) && V > 0)) return e->fail(GGNN_EINVAL, "null host pointer / negative size");
    CU_TRY(e, cudaSetDevice(e->device));
    const size_t bytes = (size_t)V * e->D * sizeof(float);
    const size_t slot = align_up(std::max<size_t>(bytes, 16), 256);
    CU_TRY(e, e->io_buf.reserve(2 * slot));
    float* d_in = (float*)e->io_buf.ptr;
    float* d_out = (float*)((char*)e->io_buf.ptr + slot);
    if (bytes) CU_TRY(e, cudaMemcpyAsync(d_in, h0_host, bytes, cudaMemcpyHostToDevice, st));
    int rc = set_graph();
    if (rc) return rc;
    if ((int64_t)e->V != V) return e->fail(GGNN_EINVAL, "graph has %d nodes, h0 has %lld rows", e->V, (long long)V);
    rc = ggnn_forward(e, d_in, d_out, (ggnn_stream_t)st);
    if (rc) return rc;
    if (bytes) CU_TRY(e, cudaMemcpyAsync(h_out_host, d_out, bytes, cudaMemcpyDeviceToHost, st));
    CU_TRY(e, cudaStreamSynchronize(st));
    return GGNN_OK;
}

extern "C" {

int ggnn_run_sparse_host(ggnn_engine* e, int32_t V, const int32_t* const* adjacency_lists, const int32_t* num_edges,
                         const float* num_incoming_edges_per_type, const float* h0_host, float* h_out_host, ggnn_stream_t stream) {
    return run_host(e, V, h0_host, h_out_host, (cudaStream_t)stream,
                    [&]() { return ggnn_set_graph_sparse(e, V, adjacency_lists, num_edges, num_incoming_edges_per_type, stream); });
}

int ggnn_run_dense_host(ggnn_engine* e, int32_t b, int32_t v, const float* adjacency_matrix, const float* h0_host, float* h_out_host,
                        ggnn_stream_t stream) {
    return run_host(e, (int64_t)b * v, h0_host, h_out_host, (cudaStream_t)stream,
                    [&]() { return ggnn_set_graph_dense(e, b, v, adjacency_matrix, stream); });
}

// ------------------------------------------------------------------------------------------ readout (SURVEY 8f-1)
int ggnn_readout_set_graphs(ggnn_engine* e, int32_t num_nodes, const int32_t* graph_nodes_list, int32_t num_graphs,
                            int32_t nodes_per_graph, const float* node_mask, ggnn_stream_t stream) {
    if (!e) return GGNN_EINVAL;
    e->ro_V = -1;
    if (num_nodes < 0 || num_graphs < 0) return e->fail(GGNN_EINVAL, "negative size");
    if (!graph_nodes_list && (nodes_per_graph <= 0 || (int64_t)nodes_per_graph * num_graphs != num_nodes))
        return e->fail(GGNN_EINVAL, "without a graph_nodes_list the batch must be num_graphs x nodes_per_graph (%d x %d != %d)", num_graphs, nodes_per_graph, num_nodes);
    CU_TRY(e, cudaSetDevice(e->device));
    const int V = num_nodes, G = num_graphs;
    size_t off = 0;
    e->ro_off_graph_of = off; off = align_up(off + sizeof(int) * (size_t)std::max(V, 1), 16);
    e->ro_off_start = off;    off = align_up(off + sizeof(int) * (size_t)(G + 1), 16);
    e->ro_off_mask = off;     off = align_up(off + sizeof(float) * (size_t)std::max(V, 1), 16);
    e->ro_off_val = off;      // device-only scratch: per-node gated value
    const size_t dev_bytes = align_up(off + sizeof(float) * (size_t)std::max(V, 1), 16);
    if (e->ro_stage_done) CU_TRY(e, cudaEventSynchronize(e->ro_stage_done));
    CU_TRY(e, e->ro_stage.reserve(off));
    CU_TRY(e, e->ro_buf.reserve(dev_bytes));
    char* base = (char*)e->ro_stage.ptr;
    int* graph_of = (int*)(base + e->ro_off_graph_of);
    int* start = (int*)(base + e->ro_off_start);
    bool grouped = true;
    for (int v = 0; v < V; ++v) {
        const int g = graph_nodes_list ? graph_nodes_list[v] : v / nodes_per_graph;
        if ((unsigned)g >= (unsigned)G) return e->fail(GGNN_ERANGE, "graph_nodes_list[%d] = %d is out of range for %d graphs", v, g, G);
        if (v > 0 && g < graph_of[v - 1]) grouped = false;
        graph_of[v] = g;
    }
    if (grouped) {   // graph g owns the contiguous node range [start[g], start[g+1])
        int v = 0;
        for (int g = 0; g <= G; ++g) {
            while (v < V && graph_of[v] < g) ++v;
            start[g] = v;
        }
    }
    if (node_mask) memcpy(base + e->ro_off_mask, node_mask, sizeof(float) * (size_t)V);
    cudaStream_t st = (cudaStream_t)stream;
    CU_TRY(e, cudaMemcpyAsync(e->ro_buf.ptr, base, off, cudaMemcpyHostToDevice, st));
    if (!e->ro_stage_done) CU_TRY(e, cudaEventCreateWithFlags(&e->ro_stage_done, cudaEventDisableTiming));
    CU_TRY(e, cudaEventRecord(e->ro_stage_done, st));
    e->ro_V = V; e->ro_G = G; e->ro_grouped = grouped; e->ro_has_mask = node_mask != nullptr;
    return GGNN_OK;
}

static int readout_check(ggnn_engine* e, const void* const* ptrs, int n) {
    if (e->ro_V < 0) return e->fail(GGNN_ESTATE, "ggnn_readout_set_graphs has not been called for this batch");
    if (e->D > 32 * readout::MAX_D_PER_LANE) return e->fail(GGNN_EUNSUPPORTED, "readout supports hidden_size <= %d", 32 * readout::MAX_D_PER_LANE);
    for (int i = 0; i < n; ++i) {
        if (!ptrs[i]) return e->fail(GGNN_EINVAL, "null readout argument %d", i);
        if (i != 3 && i != 5 && ((uintptr_t)ptrs[i] & 15)) return e->fail(GGNN_EINVAL, "readout argument %d must be 16-byte aligned", i);
    }
    return GGNN_OK;
}

int ggnn_readout_forward(ggnn_engine* e, const float* h_last, const float* h0, const float* w_gate, const float* b_gate,
                         const float* w_trans, const float* b_trans, float* out, ggnn_stream_t stream) {
    if (!e) return GGNN_EINVAL;
    const void* ps[7] = {h_last, h0, w_gate, b_gate, w_trans, b_trans, out};
    if (int rc = readout_check(e, ps, e->ro_V > 0 ? 7 : 0)) return rc;
    CU_TRY(e, cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int V = e->ro_V, G = e->ro_G;
    if (G == 0) return GGNN_OK;
    if (!out) return e->fail(GGNN_EINVAL, "null output");
    char* g = (char*)e->ro_buf.ptr;
    const float* mask = e->ro_has_mask ? (const float*)(g + e->ro_off_mask) : nullptr;
    readout::Weights w{w_gate, b_gate, w_trans, b_trans};
    float* val = (float*)(g + e->ro_off_val);
    if (V > 0) readout::readout_node_kernel<<<(V + 7) / 8, 256, 0, st>>>(h_last, h0, w, mask, val, V, e->D);
    if (e->ro_grouped || V == 0) {
        readout::readout_sum_grouped_kernel<<<(G + 127) / 128, 128, 0, st>>>(val, (const int*)(g + e->ro_off_start), out, G);
    } else {
        CU_TRY(e, cudaMemsetAsync(out, 0, sizeof(float) * (size_t)G, st));
        readout::readout_sum_atomic_kernel<<<(V + 255) / 256, 256, 0, st>>>(val, (const int*)(g + e->ro_off_graph_of), out, V);
    }
    CU_TRY(e, cudaGetLastError());
    return GGNN_OK;
}

int ggnn_readout_backward(ggnn_engine* e, const float* h_last, const float* h0, const float* w_gate, const float* b_gate,
                          const float* w_trans, const float* b_trans, const float* d_out, float* d_h_last, float* d_w_gate,
                          float* d_b_gate, float* d_w_trans, float* d_b_trans, ggnn_stream_t stream) {
    if (!e) return GGNN_EINVAL;
    const void* ps[8] = {h_last, h0, w_gate, b_gate, w_trans, b_trans, d_out, d_h_last};
    if (int rc = readout_check(e, ps, e->ro_V > 0 ? 8 : 0)) return rc;
    CU_TRY(e, cudaSetDevice(e->device));
    const int V = e->ro_V;
    if (V == 0) return GGNN_OK;
    char* g = (char*)e->ro_buf.ptr;
    const float* mask = e->ro_has_mask ? (const float*)(g + e->ro_off_mask) : nullptr;
    readout::Weights w{w_gate, b_gate, w_trans, b_trans};
    const int blocks = std::max(1, std::min((V + 7) / 8, 4 * e->num_sms));
    readout::readout_bwd_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(h_last, h0, w, (const int*)(g + e->ro_off_graph_of), mask, d_out, d_h_last,
                                                                         d_w_gate, d_b_gate, d_w_trans, d_b_trans, V, e->D);
    CU_TRY(e, cudaGetLastError());
    return GGNN_OK;
}

int ggnn_run_sparse_host_readout(ggnn_engine* e, int32_t V, const int32_t* const* adjacency_lists, const int32_t* num_edges,
                                 const float* indeg, const float* h0_host, const int32_t* graph_nodes_list, int32_t G, int32_t num_tasks,
                                 const ggnn_readout_task* tasks, const float* target_values, const float* target_mask, float* loss_out,
                                 float* accuracy_out, ggnn_stream_t stream) {
    if (!e) return GGNN_EINVAL;
    if (V < 0 || G < 0 || num_tasks <= 0 || !tasks || !loss_out || !accuracy_out || (V > 0 && (!h0_host || !graph_nodes_list)) ||
        (G > 0 && (!target_values || !target_mask)))
        return e->fail(GGNN_EINVAL, "null / negative argument");
    CU_TRY(e, cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    const size_t bytes = (size_t)V * e->D * sizeof(float);
    const size_t slot = align_up(std::max<size_t>(bytes, 16), 256);
    const size_t tg = (size_t)num_tasks * std::max(G, 1);
    // device scratch behind the two state slots: targets | masks | per-task readout [tasks][G] | results [2*tasks]
    const size_t o_tv = 2 * slot, o_tm = o_tv + align_up(tg * 4, 256), o_ro = o_tm + align_up(tg * 4, 256), o_res = o_ro + align_up(tg * 4, 256);
    CU_TRY(e, e->io_buf.reserve(o_res + align_up((size_t)2 * num_tasks * 4, 256)));
    char* io = (char*)e->io_buf.ptr;
    float *d_in = (float*)io, *d_out = (float*)(io + slot);
    if (bytes) CU_TRY(e, cudaMemcpyAsync(d_in, h0_host, bytes, cudaMemcpyHostToDevice, st));        // overlaps the host-side CSR build below
    if (G > 0) {
        CU_TRY(e, cudaMemcpyAsync(io + o_tv, target_values, tg * 4, cudaMemcpyHostToDevice, st));
        CU_TRY(e, cudaMemcpyAsync(io + o_tm, target_mask, tg * 4, cudaMemcpyHostToDevice, st));
    }
    int rc = ggnn_set_graph_sparse(e, V, adjacency_lists, num_edges, indeg, stream);
    if (rc) return rc;
    rc = ggnn_readout_set_graphs(e, V, graph_nodes_list, G, 0, nullptr, stream);
    if (rc) return rc;
    rc = ggnn_forward(e, d_in, d_out, stream);
    if (rc) return rc;
    for (int t = 0; t < num_tasks; ++t) {
        rc = ggnn_readout_forward(e, d_out, d_in, tasks[t].w_gate, tasks[t].b_gate, tasks[t].w_trans, tasks[t].b_trans,
                                  (float*)(io + o_ro) + (size_t)t * G, stream);
        if (rc) return rc;
    }
    readout::masked_loss_kernel<<<num_tasks, 256, 0, st>>>((const float*)(io + o_ro), (const float*)(io + o_tv), (const float*)(io + o_tm),
                                                           (float*)(io + o_res), G, num_tasks);
    CU_TRY(e, cudaGetLastError());
    std::vector<float> res((size_t)2 * num_tasks);
    CU_TRY(e, cudaMemcpyAsync(res.data(), io + o_res, sizeof(float) * 2 * num_tasks, cudaMemcpyDeviceToHost, st));
    CU_TRY(e, cudaStreamSynchronize(st));
    for (int t = 0; t < num_tasks; ++t) { loss_out[t] = res[t]; accuracy_out[t] = res[num_tasks + t]; }
    return GGNN_OK;
}

int ggnn_sync_check(ggnn_engine* e, ggnn_stream_t stream) {
    if (!e) return GGNN_EINVAL;
    CU_TRY(e, cudaSetDevice(e->device));
    CU_TRY(e, cudaStreamSynchronize((cudaStream_t)stream));
    int flag = 0;
    CU_TRY(e, cudaMemcpy(&flag, e->err_flag.ptr, sizeof(int), cudaMemcpyDeviceToHost));
    if (flag != 0) {
        cudaMemset(e->err_flag.ptr, 0, sizeof(int));
        return e->fail(GGNN_ECUDA, "propagation kernel reported a barrier timeout (role code %d)", flag);
    }
    return GGNN_OK;
}

int ggnn_debug_timestamps(ggnn_engine* e, int64_t* out64) {
    if (!e || !out64) return GGNN_EINVAL;
    if (!e->dbg_buf.ptr) return e->fail(GGNN_ESTATE, "no debug timestamps recorded (set GGNN_TC_DEBUG_TIMING=1)");
    CU_TRY(e, cudaSetDevice(e->device));
    CU_TRY(e, cudaDeviceSynchronize());
    CU_TRY(e, cudaMemcpy(out64, e->dbg_buf.ptr, 64 * sizeof(long long), cudaMemcpyDeviceToHost));   // the phase stamps; ggnn_debug_trace returns everything
    return GGNN_OK;
}

int ggnn_debug_trace(ggnn_engine* e, int64_t* out, int32_t capacity) {
    if (!e || !out || capacity <= 0) return GGNN_EINVAL;
    if (!e->dbg_buf.ptr) return e->fail(GGNN_ESTATE, "no debug trace recorded (set GGNN_TC_DEBUG_TIMING=1)");
    CU_TRY(e, cudaSetDevice(e->device));
    CU_TRY(e, cudaDeviceSynchronize());
    CU_TRY(e, cudaMemcpy(out, e->dbg_buf.ptr, sizeof(long long) * std::min((size_t)capacity, e->dbg_buf.cap / sizeof(long long)), cudaMemcpyDeviceToHost));
    return GGNN_OK;
}

int ggnn_set_save_for_backward(ggnn_engine* e, int32_t enable) {
    if (!e) return GGNN_EINVAL;
    e->save = enable != 0;
    e->saved_valid = false;
    return GGNN_OK;
}

int ggnn_set_backward_precision(ggnn_engine* e, int32_t precision) {
    if (!e) return GGNN_EINVAL;
    if (precision == GGNN_PREC_BF16) return e->fail(GGNN_EUNSUPPORTED, "the backward has no single-MMA bf16 mode (use GGNN_PREC_BF16X3 or GGNN_PREC_FP32)");
    if (precision != GGNN_PREC_FP32 && precision != GGNN_PREC_BF16X3) return e->fail(GGNN_EINVAL, "unknown backward precision %d", (int)precision);
    e->bwd_precision = precision;   // applies to the next ggnn_backward; the saved activations stay valid
    return GGNN_OK;
}

int ggnn_set_state_dropout(ggnn_engine* e, float keep_prob, uint64_t seed) {
    if (!e) return GGNN_EINVAL;
    if (!(keep_prob > 0.0f) || keep_prob > 1.0f) return e->fail(GGNN_EINVAL, "state keep probability must be in (0, 1], got %g", (double)keep_prob);
    e->drop_keep = keep_prob;
    e->drop_seed = (unsigned long long)seed;
    return GGNN_OK;
}

int ggnn_state_dropout_mask(int32_t V, int32_t D, int32_t global_step, float keep_prob, uint64_t seed, uint8_t* mask_out) {
    if (V < 0 || D <= 0 || (!mask_out && V > 0)) return GGNN_EINVAL;
    for (int r = 0; r < V; ++r)
        for (int c = 0; c < D; ++c)
            mask_out[(size_t)r * D + c] = dropout_keeps((unsigned long long)seed, global_step, V, D, r, c, keep_prob) ? 1 : 0;
    return GGNN_OK;
}

int ggnn_backward(ggnn_engine* e, const float* d_h_out, const ggnn_layer_grads* grads, int32_t num_layers,
                  float* d_h0, ggnn_stream_t stream) {
    if (!e) return GGNN_EINVAL;
    return ggnn_backward_impl(e, d_h_out, grads, num_layers, d_h0, stream);
}

int ggnn_num_messages(const ggnn_engine* e, int64_t* out) {
    if (!e || !out) return GGNN_EINVAL;
    *out = e->M;
    return GGNN_OK;
}

int ggnn_get_csr(ggnn_engine* e, int32_t* row_ptr, int32_t* src, int32_t* msg) {
    if (!e) return GGNN_EINVAL;
    if (!e->graph_set || e->gather_mode != GATHER_SPARSE) return e->fail(GGNN_ESTATE, "no sparse graph set");
    CU_TRY(e, cudaSetDevice(e->device));
    CU_TRY(e, cudaDeviceSynchronize());
    char* g = (char*)e->graph_buf.ptr;
    if (row_ptr) CU_TRY(e, cudaMemcpy(row_ptr, g + e->off_row_ptr, sizeof(int) * ((size_t)e->V * e->T + 1), cudaMemcpyDeviceToHost));
    if (src && e->M) CU_TRY(e, cudaMemcpy(src, g + e->off_src, sizeof(int) * (size_t)e->M, cudaMemcpyDeviceToHost));
    if (msg && e->M) CU_TRY(e, cudaMemcpy(msg, g + e->off_msg, sizeof(int) * (size_t)e->M, cudaMemcpyDeviceToHost));
    return GGNN_OK;
}

int ggnn_layer_state(ggnn_engine* e, int32_t layer, const float** dev_ptr) {
    if (!e || !dev_ptr) return GGNN_EINVAL;
    if (layer < 0 || layer > e->L) return e->fail(GGNN_EINVAL, "layer index %d out of range", layer);
    if (!e->last_out) return e->fail(GGNN_ESTATE, "no forward has run");
    const size_t vd = (size_t)std::max(e->V, 1) * e->D;
    if (layer == 0) *dev_ptr = e->last_h0;
    else if (layer == e->L) *dev_ptr = e->last_out;
    else *dev_ptr = (const float*)e->state_buf.ptr + (size_t)(layer - 1) * vd;
    return GGNN_OK;
}

int ggnn_copy_layer_state(ggnn_engine* e, int32_t layer, float* dst, ggnn_stream_t stream) {
    const float* src = nullptr;
    int rc = ggnn_layer_state(e, layer, &src);
    if (rc) return rc;
    if (!dst) return e->fail(GGNN_EINVAL, "null destination");
    CU_TRY(e, cudaSetDevice(e->device));
    if (e->V > 0)
        CU_TRY(e, cudaMemcpyAsync(dst, src, (size_t)e->V * e->D * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return GGNN_OK;
}

int ggnn_last_launch_count(const ggnn_engine* e) { return e ? e->last_launches : 0; }
const char* ggnn_plan_description(const ggnn_engine* e) { return e ? e->plan_text.c_str() : ""; }

}  // extern "C"
