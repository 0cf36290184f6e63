// Argument blocks of the non-GEMM kernels (passed by value).
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"

namespace chromo {

struct CentreEmbedArgs {
    int B, D, F;
    const float* x[CHROMO_MAX_RES];
    const float* pe[CHROMO_MAX_RES];
    int n[CHROMO_MAX_RES];
    const float* w; long long w_stride;
    float* out; long long out_stride;
};

struct AttnRowsArgs {
    int rows, H, n, F, D;
    const float* qk;      // [rows, D]
    float* P;             // [rows, ldp]  in: PE part of the scores, out: probabilities (ldp >= n)
    int ldp = 0;          // row stride of P (0 = n)
    const float* x;       // [regions / x_div, n, F]
    int x_div;
    const uint8_t* mask; long long mask_stride, mask_row_offset;
    const float* w_in;    // [D, F]
    float scale;
    float* xbar;          // [rows, 8]
    float* cbar;          // [rows, D]  <- W_in xbar
    const float* pe = nullptr;   // [n, D] position table: set => the kernel also does both PE GEMMs (n <= 32)
};

struct RegAttnArgs {
    int B, S, H;
    const void* proj; long long proj_zstride;    // [T, 4*dm] FP32, or BF16 when proj_bf16 (stride in elements)
    int proj_bf16;
    const float* gamma_f; long long gamma_zstride;
    const float* freq;
    const uint8_t* imask[CHROMO_MAX_RES];
    float* prob; long long prob_zstride;
    float* out; long long out_zstride;
};

struct HeadGatherArgs {
    int B, S, D, n_res;
    const float* xout; const float* xin; long long zstride;
    float* z;
};

struct RegAttnBwdArgs {
    int B, S, H;
    const float* proj; long long proj_z;
    const float* prob; long long prob_z;
    const float* dout; long long dout_z;
    float* dproj; long long dproj_z;
    const float* freq;
    const uint8_t* imask[CHROMO_MAX_RES];
    float* dgamma_f; long long dgamma_z;
    // d interaction_freq (chromo_backward_inputs with CHROMO_F_FREQ_GRAD): the kernels' FREQ instantiation adds
    // gamma_f[h] * dS into a per-resolution partial (stride dfreq_z); gamma_f has the stride dgamma_z of dgamma_f
    const float* gamma_f;
    float* dfreq; long long dfreq_z;
    int dfreq_add;        // 0: write (top Regulation layer), 1: add (the layers below it)
};

struct AttnRowsBwdArgs {
    int rows, H, n, F, D;
    const float* P;       // [rows, n] probabilities
    float* dS;            // [rows, n] in: dCbar . PE_j, out: d(pre-scale score)
    const float* dcbar;   // [rows, D]
    const float* x;       // [regions, n, F]
    const uint8_t* mask; long long mask_stride, mask_row_offset;
    const float* w_in;    // [D, F]
    float scale;
    float* dU8;           // [rows, 8]
    float* dqk;           // [rows, D] <- W_in dU
};

// single-query attention block (forward)
struct SqaArgs {
    int rows, H, dm, D, n, F;
    const float* q;                 // [rows, dm]
    const float* w_k; const float* w_v;   // [dm, D] each
    const float* w_in;              // [D, F]
    const float* pe;                // [n, D]
    const float* x;                 // [rows, n, F]
    const uint8_t* mask; long long mask_stride, mask_row_offset;
    float* qk; float* P; float* xbar; float* cbar; float* av;
    bool folded = false;                    // caller supplies qk and consumes cbar (folded weights)
    bool tc = false;                        // BF16 training: the four contractions on the staged tcgen05 GEMM
    const __nv_bfloat16* pe_pk = nullptr;   // BF16 tensor path: PE packed as a [n,D] weight
    const __nv_bfloat16* pet_pk = nullptr;  //                   PE^T packed as a [D,n] weight
    long long path_rows = 0;                // the row count that picks the tensor or the FP32 paths (0 = rows)
};

// in-silico pCRE deletion (deletion.cu): B genes -> V = B * (I + 1) variants of the Regulation stage
struct DeletionExpandArgs {
    int B, I, n_res;
    const float* xin; long long xin_z;              // X_in of the genes [B*S, 128] per resolution
    const uint8_t* imask[CHROMO_MAX_RES];           // [B,S,S]
    const float* freq;                              // [B,S,S]
    float* xin_v; long long xin_v_z;                // X_in of the variants [V*S, 128] per resolution
    uint8_t* imask_v[CHROMO_MAX_RES];               // [V,S,S]
    float* freq_v;                                  // [V,S,S]
};
struct DeletionScatterArgs {
    int B, I, n_res, n_out;
    const uint8_t* imask[CHROMO_MAX_RES];           // the genes' masks (which slots are live)
    const float* logits; const float* logits_v;     // [B, n_out], [V, n_out]
    float* without; float* promoter_only;           // [B, I, n_out], [B, n_out]
};
int launch_deletion_expand(const DeletionExpandArgs& a, cudaStream_t st);
int launch_deletion_scatter(const DeletionScatterArgs& a, cudaStream_t st);

// pCRE subsets (subsets.cu): B genes -> V variants of the Regulation stage, variant v = gene var_gene[v] without the live
// slots of var_drop[v]
struct SubsetExpandArgs {
    int B, I, n_res, V;
    const int* var_gene; const uint32_t* var_drop;  // [V]
    const float* xin; long long xin_z;              // X_in of the genes [B*S, 128] per resolution
    const uint8_t* imask[CHROMO_MAX_RES];           // [B,S,S]
    const float* freq;                              // [B,S,S]
    float* xin_v; long long xin_v_z;                // X_in of the variants [V*S, 128] per resolution
    uint8_t* imask_v[CHROMO_MAX_RES];               // [V,S,S]
    float* freq_v;                                  // [V,S,S]
};
struct SubsetGuardArgs {
    int B, I, V, n_out;
    const int* var_gene; const uint32_t* var_drop;  // [V]
    float* logits_v;                                // [V, n_out]: NaN rows for out-of-range descriptors
};
int launch_subset_expand(const SubsetExpandArgs& a, cudaStream_t st);
int launch_subset_guard(const SubsetGuardArgs& a, cudaStream_t st);

// interaction-frequency edits (freq_edits.cu): after subset_expand_kernel with empty drop sets, variant v's freq takes
// the non-NaN entries of var_freq[v]; an invalid variant (gene out of range, a +-inf entry) keeps its freq and gets the
// drop word 0xffffffff, which subset_guard_kernel turns into a NaN logits row
struct FreqSpliceArgs {
    int B, I, V;
    const int* var_gene;                            // [V]
    const float* var_freq;                          // [V,S,S], NaN = keep
    float* freq_v;                                  // [V,S,S] the replay's freq
    uint32_t* var_drop;                             // [V] the (empty) drop sets of subset_expand_kernel
};
int launch_freq_splice(const FreqSpliceArgs& a, cudaStream_t st);

// histone-mark occlusion (occlusion.cu): variant v = gene var_gene[v] with marks var_marks[v] zeroed over the bins
// [var_bins[v, r, 0], var_bins[v, r, 1]) of pCRE slot var_slot[v] at every resolution r
struct OcclusionDesc {
    int B, I, n_res, F, V;
    int n[CHROMO_MAX_RES];                          // bins per region
    const int* gene; const int* slot;               // [V]
    const int* bins;                                // [V, n_res, 2]
    const uint32_t* marks;                          // [V]
    const uint8_t* imask[CHROMO_MAX_RES];           // the genes' interaction masks [B,S,S] (which slots are live)
};
struct OcclusionExpandArgs {
    OcclusionDesc d;
    const float* x_pcre[CHROMO_MAX_RES];            // [B, I, n_r, F]
    const uint8_t* mask_pcre[CHROMO_MAX_RES]; long long mask_stride[CHROMO_MAX_RES], mask_row_offset[CHROMO_MAX_RES];
    const float* xin; long long xin_z;              // X_in of the genes [B*S, 128] per resolution
    float* x_v[CHROMO_MAX_RES];                     // the variant regions [V, n_r, F]
    uint8_t* mask_v[CHROMO_MAX_RES];                // their pad-mask centre rows [V, n_r]
    float* xin_p; long long xin_p_z;                // X_in of the pseudo-genes [V*2, 128] per resolution (token 0 here)
};
struct OcclusionSpliceArgs {
    OcclusionDesc d;
    const float* xin_p; long long xin_p_z;          // the pseudo-genes' X_in: row 2v + 1 is the occluded region's row
    float* xin_v; long long xin_v_z;                // X_in of the Regulation replay [V*S, 128] per resolution
};
struct OcclusionGuardArgs {
    OcclusionDesc d;
    int n_out;
    const float* logits;                            // [B, n_out]
    float* logits_v;                                // [V, n_out]: NaN rows for invalid descriptors, the gene's row on dead slots
};
int launch_occlusion_expand(const OcclusionExpandArgs& a, cudaStream_t st);
int launch_occlusion_splice(const OcclusionSpliceArgs& a, cudaStream_t st);
int launch_occlusion_guard(const OcclusionGuardArgs& a, cudaStream_t st);

int launch_reg_attention(const RegAttnArgs& a, int nz, cudaStream_t st);
int launch_attn_rows(const AttnRowsArgs& a, cudaStream_t st);
int single_query_attention(const SqaArgs& s, cudaStream_t st);

}  // namespace chromo
