// Ragged plan of a batch (ragged.cu): which pCRE slots can influence the logits at all, and which bins of the others.
#pragma once
#include <cuda_runtime.h>

#include "common.cuh"

namespace chromo {

// Everything is device memory inside the workspace; built once per forward, before the Pairwise stage.
struct RaggedPlan {
    int* live = nullptr;                     // [0] live regions R_live, [1] tiles of 64 live regions, [2] live rows / 128
    int* perm = nullptr;                     // [R] region ids (gene * I + slot): live ones by descending valid length, dead ones last
    int* y_rows = nullptr;                   // [R] token row of region perm[m] in X_in: gene * S + slot + 1
    int* tile_k0[CHROMO_MAX_RES] = {};       // [ceil(R / 64)] first key of tile t's key window (multiple of 8)
    int* tile_ns[CHROMO_MAX_RES] = {};       //                its width (multiple of 16, >= 16)
    // Regulation stage: genes grouped by token class (the smallest S_c of {1 .. 9, i_max + 1} that holds the
    // 1 + n_partners live tokens of the gene); a tile holds floor(128 / S_c) genes of one class, S_c tokens each
    int* gene_list = nullptr;                // [B] gene ids by class (largest class first, stable inside a class)
    int4* reg_tiles = nullptr;               // [reg_tiles_max] (first entry of gene_list, genes, S_c, 0) per tile; genes = 0: unused
    int* reg_rows = nullptr;                 // [reg_tiles_max][128] row of the [B*S, 128] layout behind every tile row
    int* reg_n = nullptr;                    // [0] tiles in use
    int reg_tiles_max = 0;
};

struct RaggedArgs {
    int B, I, n_res;
    int n[CHROMO_MAX_RES], ns[CHROMO_MAX_RES];          // bins per region, bins of the packed position table
    const uint8_t* mask[CHROMO_MAX_RES]; long long mask_stride[CHROMO_MAX_RES], mask_row_offset[CHROMO_MAX_RES];   // pCRE pad masks (centre rows)
    const uint8_t* imask[CHROMO_MAX_RES];               // [B, S, S]
    float* xin; long long xin_z;                        // X_in [B * S, 128] per resolution: token rows of dead slots are zeroed
};

long long ragged_plan_floats(int B, int I, int n_res);            // workspace the plan needs (floats)
int ragged_reg_tiles_max(int B, int I);                           // upper bound of the Regulation tiles of a plan
// carves the plan out of `ws` (ragged_plan_floats floats, 16-byte aligned) and builds it on `st`
int build_ragged_plan(const RaggedArgs& a, float* ws, RaggedPlan* plan, cudaStream_t st);
// The Regulation part of a plan alone (gene_list, reg_tiles, reg_rows, reg_n), from the interaction masks of `a` (B, I,
// n_res, imask; nothing else is read): reg_plan_floats floats of `ws`, 16-byte aligned
long long reg_plan_floats(int B, int I);
int build_reg_plan(const RaggedArgs& a, float* ws, RaggedPlan* plan, cudaStream_t st);

}  // namespace chromo
