// Histone-mark occlusion (chromo_pcre_occlusion): the variant regions of a Pairwise replay, the splice of their Pairwise
// rows into the Regulation replay, and the guard of the variant descriptors.
//
// Variant v is gene g = var_gene[v] with pcre_feats[r][g, i, lo_r:hi_r, m] = 0 for i = var_slot[v], every resolution r
// ([lo_r, hi_r) = var_bins[v, r]) and every mark m of var_marks[v]; nothing else changes.  Region i feeds only its own
// Pairwise rows (the Pairwise stage of a slot reads the promoter's Embedding row and that slot's features), so a variant
// needs one Pairwise pass over ONE region, whose query is the gene's Embedding row (X_in token 0, unchanged), and the
// Regulation transformer over the gene's tokens with row i + 1 replaced.  occlusion_expand_kernel writes the V variant
// regions as V pseudo-genes of one slot each: the occluded features, the pad-mask centre rows and the gene's token-0
// rows.  After their Pairwise pass, subset_expand_kernel (empty drop sets) copies every variant's gene X_in, freq and
// masks into the replay layout, and occlusion_splice_kernel overwrites row slot + 1 of every resolution with the
// pseudo-gene's Pairwise row.
// A descriptor with var_gene outside [0, B), var_slot outside [0, I), a range with lo_r < 0, lo_r > hi_r or hi_r > n_r,
// or a mark bit at or above n_feats reads nothing of any gene: its pseudo-gene gets zero inputs (every row any tile can
// read stays finite: the fused kernels multiply a probability of 0 by their tile neighbours' rows) and
// occlusion_guard_kernel writes NaN over its logits row.  A dead slot (no pCRE, as for chromo_pcre_deletion) is computed
// like any other and then gets its gene's logits row, bit for bit.
#include "kernels.cuh"

namespace chromo {

__device__ __forceinline__ bool occlusion_valid(const OcclusionDesc& d, long long v) {
    const int g = d.gene[v], i = d.slot[v];
    bool ok = g >= 0 && g < d.B && i >= 0 && i < d.I && (d.marks[v] >> d.F) == 0u;      // (F <= 8)
#pragma unroll
    for (int r = 0; r < CHROMO_MAX_RES; ++r)
        if (r < d.n_res) {
            const int lo = d.bins[(v * d.n_res + r) * 2], hi = d.bins[(v * d.n_res + r) * 2 + 1];
            ok = ok && lo >= 0 && lo <= hi && hi <= d.n[r];
        }
    return ok;
}

// slot i of gene g is live when token i + 1 is unmasked in row 0 of some resolution's interaction mask
__device__ __forceinline__ bool occlusion_live(const OcclusionDesc& d, int g, int i) {
    const int S = d.I + 1;
    bool live = false;
#pragma unroll
    for (int r = 0; r < CHROMO_MAX_RES; ++r)
        if (r < d.n_res) live |= d.imask[r][(long long)g * S * S + i + 1] == 0;
    return live;
}

// one block of 256 threads per variant
__global__ void occlusion_expand_kernel(OcclusionExpandArgs a) {
    CHROMO_PDL_ENTER();
    const OcclusionDesc& d = a.d;
    const long long v = blockIdx.x;
    const bool ok = occlusion_valid(d, v);
    const long long g = ok ? d.gene[v] : 0, region = ok ? g * d.I + d.slot[v] : 0;
    const uint32_t marks = ok ? d.marks[v] : 0u;
    const int F = d.F;
#pragma unroll
    for (int r = 0; r < CHROMO_MAX_RES; ++r) {
        if (r >= d.n_res) continue;
        const int n = d.n[r];
        const int lo = ok ? d.bins[(v * d.n_res + r) * 2] : 0, hi = ok ? d.bins[(v * d.n_res + r) * 2 + 1] : 0;
        const float* src = a.x_pcre[r] + region * n * F;
        float* dst = a.x_v[r] + v * n * F;
        for (int e = threadIdx.x; e < n * F; e += blockDim.x) {
            const int j = e / F, f = e % F;
            const bool zero = !ok || (j >= lo && j < hi && ((marks >> f) & 1u));
            dst[e] = zero ? 0.f : src[e];
        }
        const uint8_t* msrc = a.mask_pcre[r] + region * a.mask_stride[r] + a.mask_row_offset[r];
        for (int j = threadIdx.x; j < n; j += blockDim.x) a.mask_v[r][v * n + j] = ok ? msrc[j] : 0;
    }
    // token 0 of the pseudo-gene: the gene's Embedding row, the query of every Pairwise layer
    const int S = d.I + 1;
    for (int e = threadIdx.x; e < d.n_res * 32; e += blockDim.x) {
        const int r = e / 32, c = e % 32;
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ok) x = reinterpret_cast<const float4*>(a.xin + r * a.xin_z + g * S * 128)[c];
        reinterpret_cast<float4*>(a.xin_p + r * a.xin_p_z + v * 2 * 128)[c] = x;
    }
}

// one warp per variant: row slot + 1 of every resolution <- the pseudo-gene's Pairwise row (valid, live slots)
__global__ void occlusion_splice_kernel(OcclusionSpliceArgs a) {
    CHROMO_PDL_ENTER();
    const long long v = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (v >= a.d.V || !occlusion_valid(a.d, v)) return;
    const int g = a.d.gene[v], i = a.d.slot[v];
    if (!occlusion_live(a.d, g, i)) return;
    const int S = a.d.I + 1;
    for (int r = 0; r < a.d.n_res; ++r)
        reinterpret_cast<float4*>(a.xin_v + r * a.xin_v_z + (v * S + i + 1) * 128)[lane] =
            reinterpret_cast<const float4*>(a.xin_p + r * a.xin_p_z + (v * 2 + 1) * 128)[lane];
}

// one thread per variant: NaN over the logits row of an invalid descriptor, the gene's row on a dead slot
__global__ void occlusion_guard_kernel(OcclusionGuardArgs a) {
    CHROMO_PDL_ENTER();
    const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= a.d.V) return;
    if (!occlusion_valid(a.d, v)) {
        for (int o = 0; o < a.n_out; ++o) a.logits_v[v * a.n_out + o] = __int_as_float(0x7fc00000);
        return;
    }
    const int g = a.d.gene[v];
    if (occlusion_live(a.d, g, a.d.slot[v])) return;
    for (int o = 0; o < a.n_out; ++o) a.logits_v[v * a.n_out + o] = a.logits[(long long)g * a.n_out + o];
}

int launch_occlusion_expand(const OcclusionExpandArgs& a, cudaStream_t st) {
    launch_pdl(occlusion_expand_kernel, dim3((unsigned)a.d.V), dim3(256), 0, st, a);
    CHROMO_CHECK_LAUNCH("occlusion_expand");
    return CHROMO_OK;
}

int launch_occlusion_splice(const OcclusionSpliceArgs& a, cudaStream_t st) {
    launch_pdl(occlusion_splice_kernel, dim3((unsigned)((a.d.V + 7) / 8)), dim3(256), 0, st, a);
    CHROMO_CHECK_LAUNCH("occlusion_splice");
    return CHROMO_OK;
}

int launch_occlusion_guard(const OcclusionGuardArgs& a, cudaStream_t st) {
    launch_pdl(occlusion_guard_kernel, dim3((unsigned)((a.d.V + 255) / 256)), dim3(256), 0, st, a);
    CHROMO_CHECK_LAUNCH("occlusion_guard");
    return CHROMO_OK;
}

}  // namespace chromo
