// pCRE subsets (chromo_pcre_subsets): the variant batch of a Regulation replay in which each variant is one gene without
// an arbitrary set of its pCREs, and the guard of the variant descriptors.
//
// As for a single deletion (deletion.cu), removing pCREs changes nothing upstream of the Regulation transformer: slot i's
// Pairwise output depends only on the promoter and on pCRE i, so the gene's X_in rows stay valid, and a removed pCRE is
// one whose row and column of every resolution's interaction mask are set.  The Regulation transformer has no token
// positions and a masked key gets softmax weight exactly 0, so a variant may list its tokens in any order as long as X_in,
// freq and the masks follow the same permutation.  Variant v of gene g = var_gene[v] drops the live slots of var_drop[v]
// (bit i: slot i; a dead slot is not there to drop, so its bit changes nothing) and lists
//   token 0, then the tokens it keeps in their order, then the dropped tokens in their order;
// a dropped token has its row and column set in every mask, zero X_in rows and zero freq.  For the block-form masks of
// data.py:200-203 the kept live tokens are then a prefix (the live tokens are a prefix of the gene, and a dead slot sorts
// after every live one), so build_reg_plan puts the variant in token class 1 + (kept live).  A single live slot dropped
// gives exactly the order of deletion_expand_kernel.
// Every row a variant can read is finite (a softmax weight of 0 times NaN would still be NaN, and the fused Regulation
// kernel multiplies a gene's probabilities by the value rows of its tile neighbours).  A descriptor with var_gene outside
// [0, B) or a bit at or above I reads nothing of any gene: it becomes token 0 alone with zero inputs, and
// subset_guard_kernel then sets its logits row to NaN; every other variant is computed as if it were not there.
#include "kernels.cuh"

namespace chromo {

__device__ __forceinline__ bool subset_valid(const int* var_gene, const uint32_t* var_drop, int B, int I, long long v) {
    const int g = var_gene[v];
    return g >= 0 && g < B && (var_drop[v] >> I) == 0u;          // (I <= 16)
}

// one block of 128 threads per variant
__global__ void subset_expand_kernel(SubsetExpandArgs a) {
    CHROMO_PDL_ENTER();
    __shared__ int s_src[32];                       // source token of variant position t
    __shared__ int s_kept;                          // positions [0, s_kept) are kept, the rest dropped
    const int S = a.I + 1, SS = S * S;
    const long long v = blockIdx.x;
    const bool ok = subset_valid(a.var_gene, a.var_drop, a.B, a.I, v);
    const long long g = ok ? a.var_gene[v] : 0;
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x;
        // slot `lane` is live when token lane + 1 is unmasked in row 0 of some resolution's interaction mask
        bool live = false;
#pragma unroll
        for (int r = 0; r < CHROMO_MAX_RES; ++r)        // (unrolled: the pointer array stays in the parameter space)
            if (ok && r < a.n_res && lane < a.I) live |= a.imask[r][g * SS + lane + 1] == 0;
        const uint32_t drop = __ballot_sync(0xffffffffu, live) & (ok ? a.var_drop[v] : 0u);
        const uint32_t dropped_tok = drop << 1;          // bit t: token t dropped
        const int kept = S - __popc(drop);
        if (lane < S) {
            const uint32_t below = (1u << lane) - 1u;
            const bool dr = (dropped_tok >> lane) & 1u;
            s_src[dr ? kept + __popc(dropped_tok & below) : __popc(~dropped_tok & below)] = lane;
        }
        if (lane == 0) s_kept = ok ? kept : 1;
    }
    __syncthreads();
    const int kept = s_kept;
    for (int e = threadIdx.x; e < a.n_res * S * 32; e += blockDim.x) {            // X_in rows, 32 float4 each
        const int r = e / (S * 32), t = (e / 32) % S, c = e % 32;
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ok && t < kept) x = reinterpret_cast<const float4*>(a.xin + r * a.xin_z + (g * S + s_src[t]) * 128)[c];
        reinterpret_cast<float4*>(a.xin_v + r * a.xin_v_z + (v * S + t) * 128)[c] = x;
    }
    for (int e = threadIdx.x; e < SS; e += blockDim.x) {
        const int ta = e / S, tb = e % S;
        const bool keep = ta < kept && tb < kept;
        const long long src = g * SS + s_src[ta] * S + s_src[tb];
        a.freq_v[v * SS + e] = ok && keep ? a.freq[src] : 0.f;
#pragma unroll
        for (int r = 0; r < CHROMO_MAX_RES; ++r)
            if (r < a.n_res) a.imask_v[r][v * SS + e] = keep ? (ok && a.imask[r][src] != 0) : 1;
    }
}

// one thread per variant: the logits row of a descriptor out of range becomes NaN
__global__ void subset_guard_kernel(SubsetGuardArgs a) {
    CHROMO_PDL_ENTER();
    const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= a.V || subset_valid(a.var_gene, a.var_drop, a.B, a.I, v)) return;
    for (int o = 0; o < a.n_out; ++o) a.logits_v[v * a.n_out + o] = __int_as_float(0x7fc00000);
}

int launch_subset_expand(const SubsetExpandArgs& a, cudaStream_t st) {
    launch_pdl(subset_expand_kernel, dim3((unsigned)a.V), dim3(128), 0, st, a);
    CHROMO_CHECK_LAUNCH("subset_expand");
    return CHROMO_OK;
}

int launch_subset_guard(const SubsetGuardArgs& a, cudaStream_t st) {
    launch_pdl(subset_guard_kernel, dim3((unsigned)((a.V + 255) / 256)), dim3(256), 0, st, a);
    CHROMO_CHECK_LAUNCH("subset_guard");
    return CHROMO_OK;
}

}  // namespace chromo
