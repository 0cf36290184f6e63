// In-silico pCRE deletion (chromo_pcre_deletion): the variant batch of the Regulation replay and the scatter of its logits.
//
// The deletion of pCRE i changes nothing upstream of the Regulation transformer: slot i's Pairwise output depends only on
// the promoter and on pCRE i (net.py:114-125), so the gene's X_in rows stay valid and only row / column i + 1 of every
// resolution's interaction mask changes.  The Regulation transformer has no token positions (the order enters only
// through the masks and interaction_freq), and a masked key gets softmax weight exactly 0, so the variant may list its
// tokens in any order as long as X_in, freq and the masks follow the same permutation.  Variant v = g * (I + 1) + j of
// gene g:
//   j <  I, slot j live: the tokens in their order with token j + 1 moved last, its row and column masked, its X_in rows
//                        zero.  For the block-form masks of data.py:200-203 the live tokens are then a prefix: the variant
//                        lands in the token class below the gene's (ragged.cu).
//   j <  I, slot j dead, and j == I (promoter only): token 0 alone (every other entry of every mask set, the other X_in
//                        rows zero): the 1-token class.  The dead-slot variants' logits are not used.
// Every row a variant can read is finite: a softmax weight of 0 times NaN would still be NaN.
#include "kernels.cuh"

namespace chromo {

// slot j of gene g is live when token j + 1 is unmasked in row 0 of some resolution's interaction mask
__device__ __forceinline__ bool slot_live(const uint8_t* const* imask, int n_res, long long g, int S, int j) {
    bool live = false;
#pragma unroll
    for (int r = 0; r < CHROMO_MAX_RES; ++r)        // (unrolled: the pointer array stays in the parameter space)
        if (r < n_res) live |= imask[r][g * S * S + j + 1] == 0;
    return live;
}

// one block of 128 threads per variant
__global__ void deletion_expand_kernel(DeletionExpandArgs a) {
    CHROMO_PDL_ENTER();
    const int S = a.I + 1, SS = S * S;
    const long long v = blockIdx.x, g = v / S;
    const int j = (int)(v % S);
    const int d = j < a.I && slot_live(a.imask, a.n_res, g, S, j) ? j + 1 : -1;      // the token moved last (-1: none)
    // source token of variant position t
    auto src = [&](int t) { return d < 0 || t < d ? t : (t < S - 1 ? t + 1 : d); };
    // a source token whose rows and columns the variant keeps
    auto kept = [&](int t, int s) { return d < 0 ? t == 0 : s != d; };
    for (int e = threadIdx.x; e < a.n_res * S * 32; e += blockDim.x) {            // X_in rows, 32 float4 each
        const int r = e / (S * 32), t = (e / 32) % S, c = e % 32, s = src(t);
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        if (kept(t, s)) x = reinterpret_cast<const float4*>(a.xin + r * a.xin_z + (g * S + s) * 128)[c];
        reinterpret_cast<float4*>(a.xin_v + r * a.xin_v_z + (v * S + t) * 128)[c] = x;
    }
    for (int e = threadIdx.x; e < SS; e += blockDim.x) {
        const int ta = e / S, tb = e % S, sa = src(ta), sb = src(tb);
        a.freq_v[v * SS + e] = a.freq[g * SS + sa * S + sb];
        const bool keep = kept(ta, sa) && kept(tb, sb);
#pragma unroll
        for (int r = 0; r < CHROMO_MAX_RES; ++r)
            if (r < a.n_res) a.imask_v[r][v * SS + e] = keep ? (a.imask[r][g * SS + sa * S + sb] != 0) : 1;
    }
}

// one thread per output element: without [B, I, n_out], then promoter_only [B, n_out]
__global__ void deletion_scatter_kernel(DeletionScatterArgs a) {
    CHROMO_PDL_ENTER();
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int S = a.I + 1, no = a.n_out;
    const long long nw = (long long)a.B * a.I * no;
    if (idx < nw) {
        const long long g = idx / ((long long)a.I * no);
        const int j = (int)(idx / no % a.I), o = (int)(idx % no);
        a.without[idx] = slot_live(a.imask, a.n_res, g, S, j) ? a.logits_v[(g * S + j) * no + o] : a.logits[g * no + o];
    } else if (idx < nw + (long long)a.B * no) {
        const long long g = (idx - nw) / no;
        const int o = (int)((idx - nw) % no);
        a.promoter_only[g * no + o] = a.logits_v[(g * S + a.I) * no + o];
    }
}

int launch_deletion_expand(const DeletionExpandArgs& a, cudaStream_t st) {
    launch_pdl(deletion_expand_kernel, dim3((unsigned)((long long)a.B * (a.I + 1))), dim3(128), 0, st, a);
    CHROMO_CHECK_LAUNCH("deletion_expand");
    return CHROMO_OK;
}

int launch_deletion_scatter(const DeletionScatterArgs& a, cudaStream_t st) {
    const long long n = (long long)a.B * (a.I + 1) * a.n_out;
    launch_pdl(deletion_scatter_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, st, a);
    CHROMO_CHECK_LAUNCH("deletion_scatter");
    return CHROMO_OK;
}

}  // namespace chromo
