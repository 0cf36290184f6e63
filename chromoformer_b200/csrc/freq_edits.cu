// Interaction-frequency edits (chromo_freq_edits): the splice of edited pCRE-promoter contact frequencies into the
// Regulation replay of chromo_pcre_subsets.
//
// interaction_freq enters the model in one place: the Regulation attention score, s + gamma_f[r,l,h] * freq[b,i,j],
// added before the interaction mask is applied.  The Embedding and Pairwise stages never read it, so a gene's X_in rows
// serve every frequency variant of that gene.  Variant v of gene g = var_gene[v] is the gene with freq[g, e] replaced by
// var_freq[v, e] wherever that entry is not NaN (NaN: keep the gene's value), e < S * S.  subset_expand_kernel with an
// empty drop set copies the gene's X_in, freq and masks into the replay layout in token order (its s_src is then the
// identity: no token is dropped), and freq_splice_kernel overwrites the edited entries of the variant's freq.
// A variant with var_gene outside [0, B) or a +-inf entry in var_freq is invalid.  Its freq is left as subset_expand_kernel
// wrote it (the gene's own, or zeros for a gene out of range), so every value any tile can read stays finite (the fused
// Regulation kernel multiplies a probability of 0 by its tile neighbours' rows, and 0 * inf is NaN).  The splice marks it
// by setting its drop word to all ones: a bit at or above I, which subset_guard_kernel, after the head, turns into a
// NaN logits row.  The drop words are read by subset_expand_kernel before the splice runs, so the replay is unchanged.
#include "kernels.cuh"

namespace chromo {

// one warp per variant
__global__ void freq_splice_kernel(FreqSpliceArgs a) {
    CHROMO_PDL_ENTER();
    const long long v = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (v >= a.V) return;                                       // (warp-uniform: 32 | blockDim.x)
    const int SS = (a.I + 1) * (a.I + 1);
    const float* src = a.var_freq + v * SS;
    bool inf = false;
    for (int e = lane; e < SS; e += 32) inf |= isinf(src[e]);
    const int g = a.var_gene[v];
    if (__any_sync(0xffffffffu, inf) || g < 0 || g >= a.B) {
        if (lane == 0) a.var_drop[v] = 0xffffffffu;
        return;
    }
    float* dst = a.freq_v + v * SS;
    for (int e = lane; e < SS; e += 32) {
        const float f = src[e];
        if (!isnan(f)) dst[e] = f;
    }
}

int launch_freq_splice(const FreqSpliceArgs& a, cudaStream_t st) {
    launch_pdl(freq_splice_kernel, dim3((unsigned)((a.V + 7) / 8)), dim3(256), 0, st, a);
    CHROMO_CHECK_LAUNCH("freq_splice");
    return CHROMO_OK;
}

}  // namespace chromo
