// Fused Regulation-transformer layer (reg_fused.cu).
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"

namespace chromo {

struct RegFusedArgs {
    int B, S, G, n_tiles;                   // genes, tokens per gene, genes per tile (G*S <= 128), tiles
    const float* x; long long x_z;          // layer input  [B*S, 128] FP32 (z = resolution stride)
    float* y; long long y_z;                // output of the LAST layer [B*S, 128] FP32
    float* y_mid; long long y_mid_z, y_l;   // multi-layer launch: scratch slots y_mid + (li & 1) * y_l, n_tiles * 16384 floats
                                            //   each, where a CTA parks the FP32 residual rows of its tile between layers
    int n_layers; long long p_l;            // layers run back to back by one launch, parameter stride between layers
    const __nv_bfloat16* wstream; long long w_z;   // 14 packed weight chunks per layer, layers contiguous
    const float* gamma_f; const float* bo; const float* ln1w; const float* ln1b;
    const float* b1; const float* b2; const float* ln2w; const float* ln2b; long long p_z;
    const float* freq;                      // [B,S,S]
    const uint8_t* imask[CHROMO_MAX_RES];   // [B,S,S] per resolution
    long long* trace = nullptr;             // profiling hook (chromo_debug_trace): CTA (0,0) logs (event << 48 | clock64) here
    int y_head_only = 0;                    // 1 (with a plan): only token 0 of every gene is stored by the last layer (what fc_head consumes, net.py:377)
    int park_by_sm = 0;                     // 1: a CTA parks its rows in the block of its SM (set by the launcher when the slots allow)
    // ragged plan (ragged.cu): tile t holds plan_tiles[t].y genes (0: the tile is unused - the
    // grid is an upper bound) with their first plan_tiles[t].z tokens each (the others are masked for every token that
    // reaches the head); its rows are gathered from / scattered to rows plan_rows[t][0..128) of the [B*S, 128] layout
    const int4* plan_tiles = nullptr; const int* plan_rows = nullptr;
};

struct RegStreamArgs {
    const float* params; long long p_z;     // flat FP32 parameters, per-resolution stride
    long long att[CHROMO_MAX_LAYERS], ffw[CHROMO_MAX_LAYERS], l1w[CHROMO_MAX_LAYERS], l2w[CHROMO_MAX_LAYERS];
    int n_layers;
    __nv_bfloat16* stream;                  // [res][layer][14][128*128]
};

// ---- fused tail of an Embedding / Pairwise layer (row_tail_fused.cu)
struct RowTailArgs {
    int M, dff;                             // rows, FFN width (128 or 256)
    const float* a; int lda; long long a_z; // Cbar [M, 256] FP32
    const __nv_bfloat16* a_bf16 = nullptr;  // set: Cbar is BF16 at this address instead (lda in elements, resolution stride 2 * a_z elements)
    const float* res; int res_div; long long res_z;   // residual rows [M / res_div, 128]
    float* y; long long y_z; int c_div, c_mul, c_add; // output rows (remapped as in GemmArgs), 128 wide
    const __nv_bfloat16* wstream; long long w_z;
    const float* bo; const float* ln1w; const float* ln1b; const float* b1; const float* b2;
    const float* ln2w; const float* ln2b; long long p_z;
    // ragged plan (device pointers, nullptr = off): only the first *m_dev rows exist; row m takes its residual from row
    // res_rows[m] / res_div and writes output row y_rows[m] (instead of the c_div / c_mul / c_add map)
    const int* m_dev = nullptr; const int* res_rows = nullptr; const int* y_rows = nullptr;
};
struct TailStreamArgs {
    const float* nfold; long long nfold_z;  // folded out-projection N [128, 256] FP32
    const float* params; long long p_z; long long l1w, l2w;
    int dff;
    __nv_bfloat16* stream; long long stream_z;
};
constexpr long long TAIL_SLOT_ELEMS = 6LL * 128 * 128;
int pack_tail_stream(const TailStreamArgs& a, int n_res, cudaStream_t st);
int launch_row_tail_fused(const RowTailArgs& a, int n_res, cudaStream_t st);

long long reg_stream_elems_per_layer();
int pack_reg_stream(const RegStreamArgs& a, int n_res, cudaStream_t st);
void reg_fused_set_trace(long long* buf);
int launch_reg_layer_fused(const RegFusedArgs& a, int n_res, cudaStream_t st);

}  // namespace chromo
