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

int launch_reg_attention(const RegAttnArgs& a, int nz, cudaStream_t st);
int launch_attn_rows(const AttnRowsArgs& a, cudaStream_t st);
int single_query_attention(const SqaArgs& s, cudaStream_t st);

}  // namespace chromo
