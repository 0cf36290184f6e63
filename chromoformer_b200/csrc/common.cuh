// Shared host/device helpers for libchromo_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/chromoformer_b200.h"

namespace chromo {

// ---------------------------------------------------------------- errors ----
void set_error(const char* fmt, ...);
void count_launch();
#define CHROMO_CHECK_LAUNCH(what)                                              \
    do {                                                                       \
        chromo::count_launch();                                                \
        cudaError_t e__ = cudaGetLastError();                                  \
        if (e__ != cudaSuccess) {                                              \
            chromo::set_error("%s: %s", what, cudaGetErrorString(e__));        \
            return CHROMO_ECUDA;                                               \
        }                                                                      \
    } while (0)
#define CHROMO_TRY(expr)                                                       \
    do {                                                                       \
        int rc__ = (expr);                                                     \
        if (rc__ != CHROMO_OK) return rc__;                                    \
    } while (0)

// --------------------------------------------------- programmatic dependent launch --
// The training step is a chain of ~200 small dependent kernels.  A kernel launched through launch_pdl may be scheduled
// while the kernel in front of it is still running (its launch latency, and for the staged GEMM its TMEM / barrier set-up
// and the staging of the parameter operand, disappear behind that kernel's tail); CHROMO_PDL_ENTER() at the top of the
// kernel blocks until everything in front has completed and its memory is visible, then lets the NEXT kernel start.
#define CHROMO_PDL_ENTER()                                                     \
    do {                                                                       \
        asm volatile("griddepcontrol.wait;" ::: "memory");                     \
        asm volatile("griddepcontrol.launch_dependents;");                     \
    } while (0)
bool pdl_enabled();
template <typename... KArgs, typename... Args>
static inline void launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
    cfg.attrs = attr; cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);        // (errors surface in CHROMO_CHECK_LAUNCH)
}

// --------------------------------------------------- parameter layout -------
// Offsets (in floats) into the flat parameter / gradient buffers.
struct AttnOff {      // MultiHeadAttention (modules.py:8-26) / PairwiseMultiHeadAttention (modules.py:127-148)
    int64_t gamma_f, w_bias, att, p_att, c_att, ffw, ffb, lnw, lnb;
};
struct FfnOff {       // FeedForward (modules.py:91-97)
    int64_t l1w, l1b, l2w, l2b, lnw, lnb;
};
struct EmbedOff {     // EmbeddingTransformer (net.py:9-21)
    int64_t lin_proj;
    AttnOff att[CHROMO_MAX_LAYERS];
    FfnOff ffn[CHROMO_MAX_LAYERS];
};
struct PairOff {      // PairwiseInteractionTransformer (net.py:62-95)
    int64_t lnw, lnb, lin_proj_p, lin_proj_pcre;
    AttnOff att[CHROMO_MAX_LAYERS];
    FfnOff ffn[CHROMO_MAX_LAYERS];
};
struct RegOff {       // RegulationTransformer (net.py:142-150)
    AttnOff att[CHROMO_MAX_LAYERS];
    FfnOff ffn[CHROMO_MAX_LAYERS];
};
struct ParamInfo {
    std::string name;
    int64_t offset, numel;
    bool used;
};
struct ParamLayout {
    EmbedOff embed[CHROMO_MAX_RES];
    PairOff pw[CHROMO_MAX_RES];
    RegOff reg[CHROMO_MAX_RES];
    int64_t fc0w, fc0b, fc2w, fc2b;
    int64_t total, active;
    int64_t embed_stride, pw_stride, reg_stride;   // distance between resolutions
    std::vector<ParamInfo> infos;
};
int validate_config(const chromo_config_t* cfg);
const ParamLayout& get_layout(const chromo_config_t* cfg);

// --------------------------------------------------- workspace layout -------
struct WsLayout {
    int B, I, S, R, T, D;
    int training;
    int64_t res_stride;   // per-resolution block stride (n-independent buffers)
    // embed (single layer)
    int64_t e_hc, e_q, e_qk, e_cbar, e_xbar, e_av, e_preU, e_u, e_f, e_preY;
    // pairwise
    int64_t p_pp;
    int64_t p_slot;       // stride between pairwise layer slots
    int64_t p_q, p_qk, p_cbar, p_xbar, p_av, p_preU, p_u, p_f, p_preY, p_out;
    // regulation
    int64_t r_xin;
    int64_t r_slot;
    int64_t r_proj, r_att, r_prob, r_preU, r_u, r_f, r_preY, r_out;
    // resolution-dependent (probabilities over bins)
    int64_t e_p[CHROMO_MAX_RES];
    int64_t p_p[CHROMO_MAX_RES];      // + slot * p_p_slot[r]
    int64_t p_p_slot[CHROMO_MAX_RES];
    // head
    int64_t h_z, h_h1;
    // BF16 tensor path: packed parameter mirror + packed position tables (float offsets)
    int64_t bf_params, bf_pe[CHROMO_MAX_RES], bf_pet[CHROMO_MAX_RES];
    int64_t bf_win[2];                // W_in as the BF16 B operand of sqa_fused (embed, pairwise), 1024 floats per resolution
    int64_t e_qkt, p_qkt;             // QK rows as BF16 operand tiles for sqa_fused (per-resolution block; p_qkt + slot * p_slot)
    // inference-time folded attention weights (FP32 scratch + packed BF16 mirror, element offsets equal):
    //   M = [W_k[h]^T W_q[h]]_h  ([H*D, D]),  N = [W_o[:,h] W_v[h]]_h  ([D, H*D]);  slot 0 = embed, 1.. = pairwise layers
    int64_t fold_f32, fold_bf, fold_stride, fold_total;
    int64_t fold_slot[CHROMO_MAX_LAYERS + 1];
    int64_t reg_stream;     // packed weight stream of the fused Regulation layers (float offset; 0 = unused)
    int64_t tail_stream;    // packed weight streams of the fused Embedding/Pairwise tails (float offset)
    int tail_fused;         // 1 when the fused row-tail kernel applies
    int reg_fused;          // 1 when the fused Regulation-layer kernel applies to this configuration
    int reg_compact;        // replay layout of the fused path: r_xin, r_att and the r_out parking slots only
    int64_t rg_plan;        // ragged plan of the batch (ragged.cu; float offset, 0 = none)
    // backward scratch (training only)
    int64_t g_base;
    int64_t total;
    int pslots, rslots;
    inline int pslot(int l) const { return training ? l : (l & 1); }
    inline int rslot(int l) const { return training ? l : (l & 1); }
};
// replay: the layout of a Regulation + head replay over `batch` variants (chromo_pcre_subsets): the same batch-independent
// front (the packed BF16 weights), X_in, the Regulation buffers and the head, no Embedding or Pairwise block.  On the fused
// BF16 path the Regulation buffers are the parking rows r_out and the last-layer rows r_att alone.
// pairwise: the layout of a Pairwise replay over `batch` pseudo-genes of ONE pCRE slot each (chromo_pcre_occlusion): the
// same front, then the Pairwise buffers alone (no Embedding, X_in, Regulation or head block; the pass reads and writes
// an X_in the caller places).  The front is that of `cfg` itself, so the packed weights of a gene pass stay valid.
WsLayout make_ws_layout(const chromo_config_t* cfg, int batch, int flags, bool replay = false, bool pairwise = false);

static inline int64_t align4(int64_t x) { return (x + 3) & ~int64_t(3); }

// --------------------------------------------------- per-resolution branches --
// The 2000 / 500 / 100-bp chains of a stage are independent wherever their shapes differ (the single-query attention
// over n bins): between res_fork and res_join resolution r runs on `s[r]` (s[0] is the caller's stream, the others are
// library-owned side streams ordered behind it by an event), so the chains overlap on the device - also inside a captured
// CUDA graph, where the events become plain dependency edges.
struct ResStreams {
    cudaStream_t s[CHROMO_MAX_RES];
    int n;
};
int res_fork(cudaStream_t st, int n, ResStreams& rs);
int res_join(const ResStreams& rs);
// One more side stream, independent of the per-resolution ones (the early weight-gradient launch of backward.cu)
int aux_fork(cudaStream_t st, cudaStream_t* aux);     // *aux == st when side streams are off
int aux_join(cudaStream_t st, cudaStream_t aux);

}  // namespace chromo
