// Forward pass of ChromoformerBase.forward (net.py:332-380), exact-pruned:
//
//  * Embedding (net.py:31-59) and Pairwise-Interaction (net.py:105-139) outputs
//    are consumed only at the centre bin c = n/2 (net.py:59,138) and nothing
//    after the Embedding layer's own attention mixes promoter positions, so only
//    the centre QUERY row is evaluated.
//  * With a single query, K/V = (x W_in^T + PE) W_kv^T never needs to be
//    materialised:   score_j = (W_k^T q) . (W_in x_j + PE_j)
//                    sum_j p_j v_j = W_v (W_in sum_j p_j x_j + sum_j p_j PE_j)
//    i.e. two shared-operand GEMMs against the sinusoid table PE [n,128] plus a
//    rank-n_feats term per region.  Pure re-association of the reference math
//    (modules.py:48-77,159-189): no approximation, differentiable as is.
//
// Everything is FP32 here; the tcgen05 BF16 engine (umma_gemm.cu) replaces the
// large projections when CHROMO_F_BF16 is set.
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"
#include "gemm_simt.cuh"
#include "kernels.cuh"
#include "ragged.cuh"
#include "reg_fused.cuh"
#include "sqa_fused.cuh"
#include "gemm_dispatch.cuh"
#include "umma_gemm.cuh"

namespace chromo {

// --------------------------------------------------------------- kernels ----

// Hc[b,:] = W_lp x_p[b,c,:] + PE[c,:]        (net.py:42,47-53 at the centre bin)
// One thread per output channel, 32 genes per block: the channel's F weights and its position-table entry sit in
// registers, a gene's F features arrive as one broadcast read, the row leaves as 512 contiguous bytes.
constexpr int CE_GENES = 32;
__global__ void __launch_bounds__(128) centre_embed_kernel(CentreEmbedArgs a) {
    CHROMO_PDL_ENTER();
    const int r = blockIdx.y;
    const int n = a.n[r], c = n / 2, D = a.D, F = a.F;
    const float* xr = a.x[r];
    const float* per = a.pe[r];
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
        const float* w = a.w + r * a.w_stride + (long long)d * F;
        float wv[8];
#pragma unroll
        for (int f = 0; f < 8; ++f) wv[f] = f < F ? w[f] : 0.f;
        const float pe = per[(long long)c * D + d];
        const int b1 = min(a.B, (int)(blockIdx.x + 1) * CE_GENES);
        for (int b = blockIdx.x * CE_GENES; b < b1; ++b) {
            const float* x = xr + ((long long)b * n + c) * F;
            float s = pe;
#pragma unroll
            for (int f = 0; f < 8; ++f)
                if (f < F) s = fmaf(wv[f], __ldg(x + f), s);
            a.out[r * a.out_stride + (long long)b * D + d] = s;
        }
    }
}

// Single-query attention row (one warp per (region, head)):
//   s_j = (Spe[j] + u . x_j) * scale, u = W_in^T qk;  masked -> -1e9;  p = softmax(s)
//   xbar = sum_j p_j x_j;   cbar_init = W_in xbar   (the PE part is added by a GEMM)
// modules.py:58-61,71-77 / 170-189 restricted to the centre query.
__global__ void __launch_bounds__(256) attn_rows_kernel(AttnRowsArgs a) {
    CHROMO_PDL_ENTER();
    // W_in [D, F] is read by every row with a stride-F pattern: stage it once per block (coalesced)
    __shared__ float w_s[128 * 8];
    for (int i = threadIdx.x; i < a.D * a.F; i += blockDim.x) w_s[i] = a.w_in[i];
    __syncthreads();
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= a.rows) return;
    const int region = warp / a.H;
    const int n = a.n, F = a.F, D = a.D;
    const float* qk = a.qk + (long long)warp * D;
    float* P = a.P + (long long)warp * (a.ldp ? a.ldp : n);
    const float* x = a.x + (long long)(region / a.x_div) * n * F;
    const uint8_t* mk = a.mask + (long long)region * a.mask_stride + a.mask_row_offset;

    // u[f] = sum_d W[d,f] qk[d]
    float u[8];
#pragma unroll
    for (int f = 0; f < 8; ++f) u[f] = 0.f;
    for (int d = lane; d < D; d += 32) {
        const float q = qk[d];
        const float* w = w_s + d * F;
#pragma unroll
        for (int f = 0; f < 8; ++f)
            if (f < F) u[f] = fmaf(w[f], q, u[f]);
    }
#pragma unroll
    for (int f = 0; f < 8; ++f)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) u[f] += __shfl_xor_sync(0xffffffffu, u[f], o);

    // pass 1: scores + max
    float mx = -INFINITY;
    for (int j = lane; j < n; j += 32) {
        const float* xj = x + (long long)j * F;
        float s = P[j];
#pragma unroll
        for (int f = 0; f < 8; ++f)
            if (f < F) s = fmaf(u[f], xj[f], s);
        s *= a.scale;
        if (mk[j]) s = -1e9f;
        P[j] = s;
        mx = fmaxf(mx, s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    // pass 2: exp + sum
    float sum = 0.f;
    for (int j = lane; j < n; j += 32) {
        const float e = expf(P[j] - mx);
        P[j] = e;
        sum += e;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float inv = 1.f / sum;
    // pass 3: normalise + xbar
    float xb[8];
#pragma unroll
    for (int f = 0; f < 8; ++f) xb[f] = 0.f;
    for (int j = lane; j < n; j += 32) {
        const float p = P[j] * inv;
        P[j] = p;
        const float* xj = x + (long long)j * F;
#pragma unroll
        for (int f = 0; f < 8; ++f)
            if (f < F) xb[f] = fmaf(p, xj[f], xb[f]);
    }
#pragma unroll
    for (int f = 0; f < 8; ++f)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) xb[f] += __shfl_xor_sync(0xffffffffu, xb[f], o);
    if (lane < 8) a.xbar[(long long)warp * 8 + lane] = lane < F ? xb[lane] : 0.f;
    float* cb = a.cbar + (long long)warp * D;
    for (int d = lane; d < D; d += 32) {
        const float* w = w_s + d * F;
        float s = 0.f;
#pragma unroll
        for (int f = 0; f < 8; ++f)
            if (f < F) s = fmaf(w[f], xb[f], s);
        cb[d] = s;
    }
}

// Register-resident variant: one warp per REGION, all heads; the region's features are read from
// HBM once (not once per head and pass) and scores never round-trip through memory.  Every global
// read of the region (features via cp.async, both heads' score rows and W_k^T q vectors) is issued
// up front so that they overlap; NJ = ceil(n/32), F features per bin.
// FUSE_PE (short rows, n <= 32): the two GEMMs against the position table (scores QK.PE^T and
// sum_j p_j PE_j) are done here as well, from a padded copy of the table in shared memory, so the
// whole single-query attention core of a region is this one kernel.
template <int NJ, int H, int F, bool FUSE_PE>
__global__ void __launch_bounds__(128, 3) attn_rows_reg_kernel(AttnRowsArgs a) {
    CHROMO_PDL_ENTER();
    extern __shared__ __align__(16) float xs_all[];
    __shared__ float w_s[128 * F];
    __shared__ float pe_s[FUSE_PE ? 32 * 129 : 1];
    __shared__ __align__(16) float qk_s[FUSE_PE ? 4 * 128 : 4];
    const int nregions = a.rows / H;
    const int lane = threadIdx.x & 31;
    const int n = a.n, D = a.D, ldp = a.ldp ? a.ldp : a.n;
    // block-wide tables once, then every warp walks its share of the regions
    for (int i = threadIdx.x; i < D * F; i += blockDim.x) w_s[i] = a.w_in[i];
    if (FUSE_PE)
        for (int i = threadIdx.x; i < n * D; i += blockDim.x) pe_s[(i >> 7) * 129 + (i & 127)] = a.pe[i];
    __syncthreads();
    const int warps_total = (gridDim.x * blockDim.x) >> 5;
    for (int region = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; region < nregions; region += warps_total) {
    const bool active = true;
    const float* x = a.x + (long long)(region / a.x_div) * n * F;
    const uint8_t* mk = a.mask + (long long)region * a.mask_stride + a.mask_row_offset;
    float* xs = xs_all + (threadIdx.x >> 5) * (NJ * 32 * F);
    const int total = n * F;
    const bool vec = (total & 3) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0;
    if (vec) {
        const uint32_t dst = static_cast<uint32_t>(__cvta_generic_to_shared(xs));
        const float4* src = reinterpret_cast<const float4*>(x);
        for (int i = lane; i < total / 4; i += 32)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + i * 16), "l"(src + i) : "memory");
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
    float sreg[H][NJ], qk[H][4];
    bool msk[NJ];
#pragma unroll
    for (int h = 0; h < H; ++h) {
        const long long rowi = (long long)region * H + h;
#pragma unroll
        for (int jj = 0; jj < NJ; ++jj) {
            const int j = lane + 32 * jj;
            sreg[h][jj] = (!FUSE_PE && j < n) ? a.P[rowi * ldp + j] : 0.f;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) qk[h][k] = a.qk[rowi * D + lane + 32 * k];     // D == 128
    }
#pragma unroll
    for (int jj = 0; jj < NJ; ++jj) {
        const int j = lane + 32 * jj;
        msk[jj] = j < n ? (mk[j] != 0) : true;
    }
    if (vec) asm volatile("cp.async.wait_group 0;" ::: "memory");
    else for (int i = lane; i < total; i += 32) xs[i] = x[i];
    __syncwarp();
    float xr[NJ][F];
#pragma unroll
    for (int jj = 0; jj < NJ; ++jj) {
        const int j = lane + 32 * jj;
#pragma unroll
        for (int f = 0; f < F; ++f) xr[jj][f] = j < n ? xs[j * F + f] : 0.f;
    }
#pragma unroll
    for (int h = 0; h < H; ++h) {
        const long long rowi = (long long)region * H + h;
        float* P = a.P + rowi * ldp;
        float u[F];
#pragma unroll
        for (int f = 0; f < F; ++f) u[f] = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float* w = w_s + (lane + 32 * k) * F;
#pragma unroll
            for (int f = 0; f < F; ++f) u[f] = fmaf(w[f], qk[h][k], u[f]);
        }
#pragma unroll
        for (int f = 0; f < F; ++f)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) u[f] += __shfl_xor_sync(0xffffffffu, u[f], o);
        if (FUSE_PE) {
            // lane j: QK . PE_j over the 128 channels; QK of this (region, head) goes through shared memory
            // (broadcast reads), four independent accumulators
            float* qs = qk_s + (threadIdx.x >> 5) * 128;
            __syncwarp();
#pragma unroll
            for (int k = 0; k < 4; ++k) qs[lane + 32 * k] = qk[h][k];
            __syncwarp();
            const float* per = pe_s + min(lane, n - 1) * 129;
            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 8
            for (int d = 0; d < 128; d += 4) {
                const float4 q4 = *reinterpret_cast<const float4*>(qs + d);
                a0 = fmaf(q4.x, per[d], a0);
                a1 = fmaf(q4.y, per[d + 1], a1);
                a2 = fmaf(q4.z, per[d + 2], a2);
                a3 = fmaf(q4.w, per[d + 3], a3);
            }
            sreg[h][0] = (a0 + a1) + (a2 + a3);
        }
        float s[NJ];
        float mx = -INFINITY;
#pragma unroll
        for (int jj = 0; jj < NJ; ++jj) {
            const int j = lane + 32 * jj;
            s[jj] = -INFINITY;
            if (j < n) {
                float t = sreg[h][jj];
#pragma unroll
                for (int f = 0; f < F; ++f) t = fmaf(u[f], xr[jj][f], t);
                t *= a.scale;
                if (msk[jj]) t = -1e9f;
                s[jj] = t;
                mx = fmaxf(mx, t);
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        float sum = 0.f;
#pragma unroll
        for (int jj = 0; jj < NJ; ++jj) {
            s[jj] = (lane + 32 * jj < n) ? expf(s[jj] - mx) : 0.f;
            sum += s[jj];
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        const float inv = 1.f / sum;
        float xb[F];
#pragma unroll
        for (int f = 0; f < F; ++f) xb[f] = 0.f;
#pragma unroll
        for (int jj = 0; jj < NJ; ++jj) {
            const int j = lane + 32 * jj;
            const float p = s[jj] * inv;
            if (j < n && active) P[j] = p;
#pragma unroll
            for (int f = 0; f < F; ++f) xb[f] = fmaf(p, xr[jj][f], xb[f]);
        }
#pragma unroll
        for (int f = 0; f < F; ++f)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) xb[f] += __shfl_xor_sync(0xffffffffu, xb[f], o);
        float pacc[4] = {0.f, 0.f, 0.f, 0.f};
        if (FUSE_PE) {
            // channels lane + 32k: sum_j p_j PE_j (p_j broadcast from lane j)
            const float pj = s[0] * inv;
            for (int j = 0; j < n; ++j) {
                const float p = __shfl_sync(0xffffffffu, pj, j);
#pragma unroll
                for (int k = 0; k < 4; ++k) pacc[k] = fmaf(p, pe_s[j * 129 + lane + 32 * k], pacc[k]);
            }
        }
        if (active) {
            if (lane < 8) {
                float val = 0.f;
#pragma unroll
                for (int f = 0; f < F; ++f) if (lane == f) val = xb[f];
                a.xbar[rowi * 8 + lane] = val;
            }
            float* cb = a.cbar + rowi * D;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int d = lane + 32 * k;
                const float* w = w_s + d * F;
                float acc = pacc[k];
#pragma unroll
                for (int f = 0; f < F; ++f) acc = fmaf(w[f], xb[f], acc);
                cb[d] = acc;
            }
        }
    }
    __syncwarp();   // xs is re-filled by the next region
    }
}

// Regulation self-attention (modules.py:37-46,58-82): one THREAD per (gene, head, query token).
// The S threads of a (gene, head) group sit in adjacent lanes, so their K/V loads hit the same
// addresses (one transaction, broadcast) and nothing is reduced across lanes:
//   s_j = q.k_j / sqrt(32) + gamma_h * freq[i,j];  masked -> -1e9;  p = softmax_j(s)
//   out = (sum_j p_j v_j) * sigmoid(gate)
// proj = [q | k | v | gate] per token, FP32 or BF16 (PT).
template <typename PT> struct ProjLoad;
template <> struct ProjLoad<float> {
    static __device__ __forceinline__ void load8(const float* p, float* v) {
        const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    }
};
template <> struct ProjLoad<__nv_bfloat16> {
    static __device__ __forceinline__ void load8(const __nv_bfloat16* p, float* v) {
        const uint4 u = *reinterpret_cast<const uint4*>(p);
        const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            v[2 * k] = __uint_as_float(w[k] << 16);
            v[2 * k + 1] = __uint_as_float(w[k] & 0xffff0000u);
        }
    }
};

template <int SMAX, typename PT>
__global__ void __launch_bounds__(128) reg_attention_kernel(RegAttnArgs a) {
    CHROMO_PDL_ENTER();
    const int S = a.S, H = a.H, dm = 32 * H;
    const int gpw = 32 / S;                                   // (gene, head) groups per warp
    const int lane = threadIdx.x & 31;
    const long long warp = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int z = blockIdx.y;
    const long long grp = warp * gpw + lane / S;
    const int i = lane % S;
    if (lane >= gpw * S || grp >= (long long)a.B * H) return;
    const int b = (int)(grp / H), h = (int)(grp % H);
    const PT* base = reinterpret_cast<const PT*>(a.proj) + z * a.proj_zstride + (long long)b * S * 4 * dm + h * 32;
    float q[32];
#pragma unroll
    for (int c = 0; c < 4; ++c) ProjLoad<PT>::load8(base + (long long)i * 4 * dm + c * 8, q + c * 8);
    const float gamma = a.gamma_f[z * a.gamma_zstride + h];
    const float* freq = a.freq + ((long long)b * S + i) * S;
    const uint8_t* mask = a.imask[z] + ((long long)b * S + i) * S;
    const float scale = 0.17677669529663687f;   // 1/sqrt(32)
    float s[SMAX];
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < SMAX; ++j) {
        s[j] = -INFINITY;
        if (j < S) {
            const PT* kj = base + (long long)j * 4 * dm + dm;
            float d0 = 0.f, d1 = 0.f;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                float kv[8];
                ProjLoad<PT>::load8(kj + c * 8, kv);
#pragma unroll
                for (int e = 0; e < 8; e += 2) {
                    d0 = fmaf(q[c * 8 + e], kv[e], d0);
                    d1 = fmaf(q[c * 8 + e + 1], kv[e + 1], d1);
                }
            }
            float t = (d0 + d1) * scale + gamma * freq[j];
            if (mask[j]) t = -1e9f;
            s[j] = t;
            mx = fmaxf(mx, t);
        }
    }
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < SMAX; ++j)
        if (j < S) { s[j] = (sizeof(PT) == 4) ? expf(s[j] - mx) : __expf(s[j] - mx); sum += s[j]; }
    const float inv = 1.f / sum;
    float o[32];
#pragma unroll
    for (int d = 0; d < 32; ++d) o[d] = 0.f;
    float* prob = a.prob ? a.prob + z * a.prob_zstride + (((long long)b * H + h) * S + i) * S : nullptr;
#pragma unroll
    for (int j = 0; j < SMAX; ++j) {
        if (j < S) {
            const float p = s[j] * inv;
            if (prob) prob[j] = p;
            const PT* vj = base + (long long)j * 4 * dm + 2 * dm;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                float vv[8];
                ProjLoad<PT>::load8(vj + c * 8, vv);
#pragma unroll
                for (int e = 0; e < 8; ++e) o[c * 8 + e] = fmaf(p, vv[e], o[c * 8 + e]);
            }
        }
    }
    float* out = a.out + z * a.out_zstride + ((long long)b * S + i) * dm + h * 32;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        float gt[8];
        ProjLoad<PT>::load8(base + (long long)i * 4 * dm + 3 * dm + c * 8, gt);
        float r[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) r[e] = o[c * 8 + e] / (1.f + ((sizeof(PT) == 4) ? expf(-gt[e]) : __expf(-gt[e])));
        *reinterpret_cast<float4*>(out + c * 8) = make_float4(r[0], r[1], r[2], r[3]);
        *reinterpret_cast<float4*>(out + c * 8 + 4) = make_float4(r[4], r[5], r[6], r[7]);
    }
}

// The same attention with one CTA per gene (FP32 projections: the strict path and the training step).  The gene's S rows of
// q | k | v | gate (S x 4 KB) are staged once in shared memory, coalesced; a (head, query) pair is served by four lanes,
// eight channels each: partial dot products against the S keys meet by two shuffles, every lane then holds the whole
// softmax row and accumulates its eight output channels.  (The kernel above reads every key / value row S times from
// L1 with four warps per SM in flight: 23 us at batch 64 against 4 us here.)
constexpr int RA_PAD = 4;          // floats between staged rows: the S query rows of a head fall on different banks
template <int SMAX>
__global__ void __launch_bounds__(SMAX * 32) reg_attention_gene_kernel(RegAttnArgs a) {
    CHROMO_PDL_ENTER();
    extern __shared__ __align__(16) float ra_sm[];
    const int S = a.S, H = a.H, dm = 32 * H, ld = 4 * dm + RA_PAD;
    const int b = blockIdx.x, z = blockIdx.y, tid = threadIdx.x;
    const float* proj = reinterpret_cast<const float*>(a.proj) + z * a.proj_zstride + (long long)b * S * 4 * dm;
    for (int v = tid; v < S * dm; v += blockDim.x) {            // float4 units, rows of 4*dm floats
        const int r = v / dm, c = v % dm;
        *reinterpret_cast<float4*>(ra_sm + r * ld + 4 * c) = __ldg(reinterpret_cast<const float4*>(proj + (long long)r * 4 * dm) + c);
    }
    __syncthreads();
    const int item = tid >> 2, sub = tid & 3;
    if (item >= H * S) return;
    const int h = item / S, i = item % S;
    const int co = h * 32 + sub * 8;                             // this lane's eight channels
    float q[8], s[SMAX];
    {
        const float4 x = *reinterpret_cast<const float4*>(ra_sm + i * ld + co), y = *reinterpret_cast<const float4*>(ra_sm + i * ld + co + 4);
        q[0] = x.x; q[1] = x.y; q[2] = x.z; q[3] = x.w; q[4] = y.x; q[5] = y.y; q[6] = y.z; q[7] = y.w;
    }
#pragma unroll
    for (int j = 0; j < SMAX; ++j) {
        s[j] = 0.f;
        if (j < S) {
            const float4 x = *reinterpret_cast<const float4*>(ra_sm + j * ld + dm + co), y = *reinterpret_cast<const float4*>(ra_sm + j * ld + dm + co + 4);
            s[j] = (q[0] * x.x + q[1] * x.y) + (q[2] * x.z + q[3] * x.w) + (q[4] * y.x + q[5] * y.y) + (q[6] * y.z + q[7] * y.w);
        }
    }
#pragma unroll
    for (int j = 0; j < SMAX; ++j) {
        s[j] += __shfl_xor_sync(0xffffffffu, s[j], 1);
        s[j] += __shfl_xor_sync(0xffffffffu, s[j], 2);
    }
    const float gamma = a.gamma_f[z * a.gamma_zstride + h];
    const float* freq = a.freq + ((long long)b * S + i) * S;
    const uint8_t* mask = a.imask[z] + ((long long)b * S + i) * S;
    const float scale = 0.17677669529663687f;   // 1/sqrt(32)
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < SMAX; ++j) {
        if (j < S) {
            float t = s[j] * scale + gamma * freq[j];
            if (mask[j]) t = -1e9f;
            s[j] = t;
            mx = fmaxf(mx, t);
        }
    }
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < SMAX; ++j)
        if (j < S) { s[j] = expf(s[j] - mx); sum += s[j]; }
    const float inv = 1.f / sum;
    float o[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    float* prob = a.prob ? a.prob + z * a.prob_zstride + (((long long)b * H + h) * S + i) * S : nullptr;
#pragma unroll
    for (int j = 0; j < SMAX; ++j) {
        if (j < S) {
            const float p = s[j] * inv;
            if (prob && sub == (j & 3)) prob[j] = p;
            const float4 x = *reinterpret_cast<const float4*>(ra_sm + j * ld + 2 * dm + co), y = *reinterpret_cast<const float4*>(ra_sm + j * ld + 2 * dm + co + 4);
            o[0] = fmaf(p, x.x, o[0]); o[1] = fmaf(p, x.y, o[1]); o[2] = fmaf(p, x.z, o[2]); o[3] = fmaf(p, x.w, o[3]);
            o[4] = fmaf(p, y.x, o[4]); o[5] = fmaf(p, y.y, o[5]); o[6] = fmaf(p, y.z, o[6]); o[7] = fmaf(p, y.w, o[7]);
        }
    }
    const float4 gx = *reinterpret_cast<const float4*>(ra_sm + i * ld + 3 * dm + co), gy = *reinterpret_cast<const float4*>(ra_sm + i * ld + 3 * dm + co + 4);
    const float g[8] = {gx.x, gx.y, gx.z, gx.w, gy.x, gy.y, gy.z, gy.w};
#pragma unroll
    for (int e = 0; e < 8; ++e) o[e] = o[e] / (1.f + expf(-g[e]));
    float* out = a.out + z * a.out_zstride + ((long long)b * S + i) * dm + co;
    *reinterpret_cast<float4*>(out) = make_float4(o[0], o[1], o[2], o[3]);
    *reinterpret_cast<float4*>(out + 4) = make_float4(o[4], o[5], o[6], o[7]);
}

// z[b, r*D + d] = X_out_r[b, 0, d] + X_in_r[b, 0, d]           (net.py:377-378)
__global__ void head_gather_kernel(HeadGatherArgs a) {
    CHROMO_PDL_ENTER();
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int W = a.n_res * a.D;
    if (idx >= a.B * W) return;
    const int b = idx / W, c = idx % W, r = c / a.D, d = c % a.D;
    const long long row = (long long)b * a.S * a.D + d;
    a.z[idx] = a.xout[r * a.zstride + row] + a.xin[r * a.zstride + row];
}

// ------------------------------------------------------------ launchers -----
int launch_reg_attention(const RegAttnArgs& a, int nz, cudaStream_t st) {
    const int wpb = 4, gpw = 32 / a.S;
    const long long warps = ((long long)a.B * a.H + gpw - 1) / gpw;
    dim3 grid((unsigned)((warps + wpb - 1) / wpb), nz);
    if (a.proj_bf16) {
        if (a.S <= 9) launch_pdl(reg_attention_kernel<9, __nv_bfloat16>, dim3(grid), dim3(wpb * 32), 0, st, a);
        else launch_pdl(reg_attention_kernel<17, __nv_bfloat16>, dim3(grid), dim3(wpb * 32), 0, st, a);
    } else {
        if (a.H == 8 && a.S <= 17) {       // one CTA per gene, rows staged in shared memory
            const size_t smem = (size_t)a.S * (4 * 32 * a.H + RA_PAD) * sizeof(float);
            static bool configured = false;
            if (!configured) {
                cudaFuncSetAttribute(reg_attention_gene_kernel<17>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)(17 * (4 * 32 * 8 + RA_PAD) * sizeof(float)));
                configured = true;
            }
            const int threads = (a.H * a.S * 4 + 31) / 32 * 32;
            if (a.S <= 9) launch_pdl(reg_attention_gene_kernel<9>, dim3(a.B, nz), dim3(threads), smem, st, a);
            else launch_pdl(reg_attention_gene_kernel<17>, dim3(a.B, nz), dim3(threads), smem, st, a);
        } else if (a.S <= 9) launch_pdl(reg_attention_kernel<9, float>, dim3(grid), dim3(wpb * 32), 0, st, a);
        else launch_pdl(reg_attention_kernel<17, float>, dim3(grid), dim3(wpb * 32), 0, st, a);
    }
    CHROMO_CHECK_LAUNCH("reg_attention");
    return CHROMO_OK;
}

int launch_attn_rows(const AttnRowsArgs& a, cudaStream_t st) {
    const int wpb = 8;
    if (a.H == 2 && a.F == 7 && a.D == 128 && a.n <= 416) {
        // one warp per region, every global read issued up front, features staged once, scores in registers
        const int regions = a.rows / 2;
        int blocks = (regions + 3) / 4;
        // persistent (<= 6 blocks per SM, warps loop over regions) where the per-block table staging or the
        // long rows make it pay; one region per warp otherwise
        if ((a.n > 96 || a.n <= 32) && blocks > 148 * 6) blocks = 148 * 6;
        static bool configured = false;
        if (!configured) {
            cudaFuncSetAttribute(attn_rows_reg_kernel<13, 2, 7, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)(4 * 13 * 32 * 7 * sizeof(float)));
            configured = true;
        }
        if (a.n <= 32 && a.pe) launch_pdl(attn_rows_reg_kernel<1, 2, 7, true>, dim3(blocks), dim3(128), 4 * 1 * 32 * 7 * sizeof(float), st, a);
        else if (a.n <= 32) launch_pdl(attn_rows_reg_kernel<1, 2, 7, false>, dim3(blocks), dim3(128), 4 * 1 * 32 * 7 * sizeof(float), st, a);
        else if (a.n <= 96) launch_pdl(attn_rows_reg_kernel<3, 2, 7, false>, dim3(blocks), dim3(128), 4 * 3 * 32 * 7 * sizeof(float), st, a);
        else launch_pdl(attn_rows_reg_kernel<13, 2, 7, false>, dim3(blocks), dim3(128), 4 * 13 * 32 * 7 * sizeof(float), st, a);
        CHROMO_CHECK_LAUNCH("attn_rows_reg");
        return CHROMO_OK;
    }
    launch_pdl(attn_rows_kernel, dim3((a.rows + wpb - 1) / wpb), dim3(wpb * 32), 0, st, a);
    CHROMO_CHECK_LAUNCH("attn_rows");
    return CHROMO_OK;
}

// Single-query attention block shared by Embedding and Pairwise layers:
// Q[rows,dm] -> Av[rows,dm].   w_k / w_v: [dm, D] slices of att/c_att.weight.
int single_query_attention(const SqaArgs& s, cudaStream_t st) {
    const int dh = s.dm / s.H, D = s.D;
    // QK[(row,h), :] = W_k[h]^T Q[row, h]                                  (NN GEMM per head)
    if (!s.folded) {
        GemmArgs g = gemm_args();
        g.A = s.q; g.lda = s.dm; g.sA2 = dh;
        g.B = s.w_k; g.ldb = D; g.sB2 = (long long)dh * D;
        g.C = s.qk; g.ldc = s.H * D; g.sC2 = D;
        g.M = s.rows; g.N = D; g.K = dh; g.zdiv = s.H;
        CHROMO_TRY(gemm_auto(g, true, false, s.H, st, s.tc));
    }
    // Short rows (n <= 32).  BF16 inference: pad the row to 32 bins (the packed position tables carry zero rows /
    // columns there) so that both position-table GEMMs run on the tensor pipe; otherwise the rows kernel does
    // them itself (attn_rows_reg_kernel<.., FUSE_PE>).
    const long long path_rows = (s.path_rows ? s.path_rows : s.rows) * s.H;     // the row count that picks the paths
    const bool pad32 = s.pe_pk && s.folded && s.n <= 32 && path_rows >= 64;
    const int np = pad32 ? 32 : s.n;                       // row stride / GEMM extent of the P buffer
    const bool fuse_pe = !pad32 && s.H == 2 && s.F == 7 && D == 128 && s.n <= 32;
    // Spe[(row,h), j] = QK[(row,h), :] . PE[j, :]                          (NT GEMM vs the table)
    if (!fuse_pe) {
        GemmArgs g = gemm_args();
        g.A = s.qk; g.lda = D;
        g.B = s.pe; g.ldb = D;
        g.C = s.P; g.ldc = np;
        g.M = s.rows * s.H; g.N = np; g.K = D;
        if (s.pe_pk && path_rows >= 64 && np % 16 == 0 && umma_supported(g)) CHROMO_TRY(umma_launch(g, s.pe_pk, 1, st));
        else if (pad32) { set_error("internal: padded short-row path needs the tensor engine"); return CHROMO_EINVAL; }
        else CHROMO_TRY(gemm_auto(g, true, true, 1, st, s.tc));
    }
    {
        AttnRowsArgs a;
        a.rows = s.rows * s.H; a.H = s.H; a.n = s.n; a.F = s.F; a.D = D;
        a.qk = s.qk; a.P = s.P; a.x = s.x; a.x_div = 1;
        a.mask = s.mask; a.mask_stride = s.mask_stride; a.mask_row_offset = s.mask_row_offset;
        a.w_in = s.w_in; a.scale = 1.f / sqrtf((float)dh);
        a.xbar = s.xbar; a.cbar = s.cbar; a.pe = fuse_pe ? s.pe : nullptr; a.ldp = np;
        CHROMO_TRY(launch_attn_rows(a, st));
    }
    // Cbar += P . PE                                                        (NN GEMM, K = n)
    if (!fuse_pe) {
        GemmArgs g = gemm_args();
        g.A = s.P; g.lda = np;
        g.B = s.pe; g.ldb = D;
        g.C = s.cbar; g.ldc = D; g.accumulate = 1;
        g.M = s.rows * s.H; g.N = D; g.K = np;
        if (s.pet_pk && path_rows >= 64 && np % 16 == 0 && umma_supported(g)) CHROMO_TRY(umma_launch(g, s.pet_pk, 1, st));
        else if (pad32) { set_error("internal: padded short-row path needs the tensor engine"); return CHROMO_EINVAL; }
        else CHROMO_TRY(gemm_auto(g, true, false, 1, st, s.tc));   // (no split-K here: the forward stays deterministic)
    }
    // Av[row, h*dh + e] = W_v[h*dh + e, :] . Cbar[(row,h), :]               (NT GEMM per head)
    if (!s.folded) {
        GemmArgs g = gemm_args();
        g.A = s.cbar; g.lda = s.H * D; g.sA2 = D;
        g.B = s.w_v; g.ldb = D; g.sB2 = (long long)dh * D;
        g.C = s.av; g.ldc = s.dm; g.sC2 = dh;
        g.M = s.rows; g.N = dh; g.K = D; g.zdiv = s.H;
        CHROMO_TRY(gemm_auto(g, true, true, s.H, st, s.tc));
    }
    return CHROMO_OK;
}

// BF16 mirror of every weight the tcgen05 engine consumes, in UMMA tile order, at the same
// element offsets as the FP32 parameters; plus the position table as a weight ([n,D]) and
// transposed ([D,n]) for the two shared-operand GEMMs of the single-query attention.
static int pack_all_weights(const chromo_config_t* c, const ParamLayout& L, const float* P, __nv_bfloat16* packed,
                            float* ws, const WsLayout& w, const chromo_batch_t* in, cudaStream_t st) {
    const int D = c->d_emb, NR = c->n_res;
    auto pk = [&](int64_t off, int N, int K, long long zs, int nz) -> int {
        const int nt = umma_tile_n(N);
        if (nt == 0 || K % 16 != 0) return CHROMO_OK;        // this weight stays on the FP32 path
        return pack_weights(P + off, packed + off, N, K, nt, zs, nz, false, K, st);
    };
    const AttnOff& ea = L.embed[0].att[0];
    const FfnOff& ef = L.embed[0].ffn[0];
    CHROMO_TRY(pk(ea.att, c->embed_d_model, D, L.embed_stride, NR));          // W_q rows only
    CHROMO_TRY(pk(ea.ffw, D, c->embed_d_model, L.embed_stride, NR));
    CHROMO_TRY(pk(ef.l1w, c->embed_d_ff, D, L.embed_stride, NR));
    CHROMO_TRY(pk(ef.l2w, D, c->embed_d_ff, L.embed_stride, NR));
    CHROMO_TRY(pk(L.pw[0].lin_proj_p, D, D, L.pw_stride, NR));
    for (int l = 0; l < c->pw_layers; ++l) {
        const AttnOff& a = L.pw[0].att[l];
        const FfnOff& f = L.pw[0].ffn[l];
        CHROMO_TRY(pk(a.p_att, c->pw_d_model, D, L.pw_stride, NR));
        CHROMO_TRY(pk(a.ffw, D, c->pw_d_model, L.pw_stride, NR));
        CHROMO_TRY(pk(f.l1w, c->pw_d_ff, D, L.pw_stride, NR));
        CHROMO_TRY(pk(f.l2w, D, c->pw_d_ff, L.pw_stride, NR));
    }
    for (int l = 0; l < c->reg_layers; ++l) {
        const AttnOff& a = L.reg[0].att[l];
        const FfnOff& f = L.reg[0].ffn[l];
        CHROMO_TRY(pk(a.att, 4 * c->reg_d_model, D, L.reg_stride, NR));
        CHROMO_TRY(pk(a.ffw, D, c->reg_d_model, L.reg_stride, NR));
        CHROMO_TRY(pk(f.l1w, c->reg_d_ff, D, L.reg_stride, NR));
        CHROMO_TRY(pk(f.l2w, D, c->reg_d_ff, L.reg_stride, NR));
    }
    CHROMO_TRY(pk(L.fc0w, c->d_head, NR * D, 0, 1));
    if (w.reg_fused) {
        RegStreamArgs a;
        a.params = P; a.p_z = L.reg_stride; a.n_layers = c->reg_layers;
        for (int l = 0; l < c->reg_layers; ++l) {
            a.att[l] = L.reg[0].att[l].att; a.ffw[l] = L.reg[0].att[l].ffw;
            a.l1w[l] = L.reg[0].ffn[l].l1w; a.l2w[l] = L.reg[0].ffn[l].l2w;
        }
        a.stream = reinterpret_cast<__nv_bfloat16*>(ws + w.reg_stream);
        CHROMO_TRY(pack_reg_stream(a, NR, st));
    }
    if (!w.training) {
        // Folded single-query attention weights (exact re-association, inference only):
        //   QK[(row,h), :] = (W_k[h]^T W_q[h]) x_row        -> one [H*D, D] linear replaces Q and the QK fold
        //   out            = sum_h (W_o[:,h] W_v[h]) cbar_h -> one [D, H*D] linear replaces W_v and the out-projection
        float* F32 = ws + w.fold_f32;
        __nv_bfloat16* FB = reinterpret_cast<__nv_bfloat16*>(ws + w.fold_bf);
        auto fold = [&](int slot, int H, int dm, int64_t wq, int64_t wk, int64_t wv, int64_t wo, long long pz) -> int {
            const int dh = dm / H;
            const int64_t oM = w.fold_slot[slot], oN = oM + (int64_t)H * D * D;
            {   // M[h][d, e] = sum_c W_k[h*dh + c, d] W_q[h*dh + c, e]
                GemmArgs g = gemm_args();
                g.A = P + wk; g.lda = D; g.sA1 = pz; g.sA2 = (long long)dh * D;
                g.B = P + wq; g.ldb = D; g.sB1 = pz; g.sB2 = (long long)dh * D;
                g.C = F32 + oM; g.ldc = D; g.sC1 = w.fold_stride; g.sC2 = (long long)D * D;
                g.M = D; g.N = D; g.K = dh; g.zdiv = H;
                CHROMO_TRY(gemm_launch(g, false, false, NR * H, st));
            }
            {   // N[o, h*D + d] = sum_c W_o[o, h*dh + c] W_v[h*dh + c, d]
                GemmArgs g = gemm_args();
                g.A = P + wo; g.lda = dm; g.sA1 = pz; g.sA2 = dh;
                g.B = P + wv; g.ldb = D; g.sB1 = pz; g.sB2 = (long long)dh * D;
                g.C = F32 + oN; g.ldc = H * D; g.sC1 = w.fold_stride; g.sC2 = D;
                g.M = D; g.N = D; g.K = dh; g.zdiv = H;
                CHROMO_TRY(gemm_launch(g, true, false, NR * H, st));
            }
            CHROMO_TRY(pack_weights(F32 + oM, FB + oM, H * D, D, umma_tile_n(H * D), w.fold_stride, NR, false, D, st));
            CHROMO_TRY(pack_weights(F32 + oN, FB + oN, D, H * D, umma_tile_n(D), w.fold_stride, NR, false, H * D, st));
            return CHROMO_OK;
        };
        const int dme = c->embed_d_model, dmp = c->pw_d_model;
        CHROMO_TRY(fold(0, c->embed_heads, dme, ea.att, ea.att + (int64_t)dme * D, ea.att + (int64_t)2 * dme * D, ea.ffw,
                        L.embed_stride));
        for (int l = 0; l < c->pw_layers; ++l) {
            const AttnOff& a = L.pw[0].att[l];
            CHROMO_TRY(fold(1 + l, c->pw_heads, dmp, a.p_att, a.c_att, a.c_att + (int64_t)dmp * D, a.ffw, L.pw_stride));
        }
        if (w.tail_fused) {
            __nv_bfloat16* TS = reinterpret_cast<__nv_bfloat16*>(ws + w.tail_stream);
            const long long tz = (long long)(1 + c->pw_layers) * TAIL_SLOT_ELEMS;
            for (int slot = 0; slot <= c->pw_layers; ++slot) {
                TailStreamArgs t;
                const int H = slot == 0 ? c->embed_heads : c->pw_heads;
                t.nfold = F32 + w.fold_slot[slot] + (int64_t)H * D * D; t.nfold_z = w.fold_stride;
                t.params = P;
                if (slot == 0) { t.p_z = L.embed_stride; t.l1w = L.embed[0].ffn[0].l1w; t.l2w = L.embed[0].ffn[0].l2w; t.dff = c->embed_d_ff; }
                else { t.p_z = L.pw_stride; t.l1w = L.pw[0].ffn[slot - 1].l1w; t.l2w = L.pw[0].ffn[slot - 1].l2w; t.dff = c->pw_d_ff; }
                t.stream = TS + slot * TAIL_SLOT_ELEMS; t.stream_z = tz;
                CHROMO_TRY(pack_tail_stream(t, NR, st));
            }
        }
    }
    CHROMO_TRY(sqa_pack_w_in(P + L.embed[0].lin_proj, L.embed_stride, reinterpret_cast<__nv_bfloat16*>(ws + w.bf_win[0]), 2048, NR, st));
    CHROMO_TRY(sqa_pack_w_in(P + L.pw[0].lin_proj_pcre, L.pw_stride, reinterpret_cast<__nv_bfloat16*>(ws + w.bf_win[1]), 2048, NR, st));
    for (int r = 0; r < NR; ++r) {
        const int n = c->n_bins[r];
        if (!in->pos_enc[r]) continue;
        const int np = n <= 32 ? 32 : n;                   // short rows are padded to 32 bins with zeros
        if (np % 16 != 0) continue;
        CHROMO_TRY(pack_weights(in->pos_enc[r], reinterpret_cast<__nv_bfloat16*>(ws + w.bf_pe[r]), np, D,
                                umma_tile_n(np), 0, 1, false, D, st, n));
        CHROMO_TRY(pack_weights(in->pos_enc[r], reinterpret_cast<__nv_bfloat16*>(ws + w.bf_pet[r]), D, np,
                                umma_tile_n(D), 0, 1, true, D, st, n));
    }
    return CHROMO_OK;
}

struct RegOnly { int layer; const float* x; float* y; long long xy_stride; };
// The Regulation transformer and the head alone, over the X_in rows already in the workspace (the variants of
// chromo_pcre_deletion and chromo_pcre_subsets); the fused Regulation kernel runs under the token classes of `plan` when
// it is set.  gene_batch: the row count of the gene pass the variants come from; every GEMM takes the path (tcgen05 or
// FP32) the gene pass takes, so a variant is computed the way its gene is, whatever the number of variants.
struct RegReplay { const RaggedPlan* plan; int gene_batch; };
// The Pairwise stage alone over pseudo-genes of one pCRE slot each (the occluded regions of chromo_pcre_occlusion), on a
// make_ws_layout(..., pairwise = true) layout: the PP GEMM reads token 0 of the X_in at `xin` (resolution stride xin_z,
// [B * 2, 128]) and the last layer writes token 1 there; no Embedding, Regulation or head.  Every GEMM takes the path
// the gene pass of gene_batch genes with gene_slots slots takes (its PP GEMM has gene_batch rows, its Pairwise GEMMs
// gene_batch * gene_slots), so an occluded region takes the GEMM paths its gene's region took, whatever the number of
// pseudo-genes.  (The path choice, not the bits: a gene pass under the ragged plan computed its regions over key windows
// shared by a tile.)  No ragged plan here: every region walks the whole position table, so its rows do not depend on
// the others.
struct PwReplay { int gene_batch, gene_slots; float* xin; long long xin_z; };

// The side stream of aux_fork: joined back into `st` by join(), or on leaving the scope when an error return comes first
// (a fork left open invalidates a stream capture).
struct AuxStream {
    cudaStream_t st, aux;
    int join() { const cudaStream_t s = aux; aux = st; return aux_join(st, s); }
    ~AuxStream() { join(); }
};

static int forward_impl(const chromo_config_t* c, const float* P, const chromo_batch_t* in, float* logits,
                        float* ws, const WsLayout& w, int flags, cudaStream_t st, const RegOnly* only = nullptr,
                        const RegReplay* replay = nullptr, const PwReplay* pw = nullptr) {
    const ParamLayout& L = get_layout(c);
    const int B = w.B, I = w.I, S = w.S, R = w.R, T = w.T, D = w.D, F = c->n_feats;
    const int NR = c->n_res;
    const bool train = w.training;
    const long long RS = w.res_stride;
    const bool bf16 = (flags & CHROMO_F_BF16) != 0;
    // a replay picks every path by the gene pass's row count (the rows of a variant GEMM are B or T = B * S, those of
    // the gene pass's gene_batch or gene_batch * S), so the variants are computed the way their genes are
    auto gene_rows = [&](long long M) -> long long {
        return replay ? M / B * replay->gene_batch : pw ? M / B * pw->gene_batch * pw->gene_slots : M;
    };
    const bool proj_bf16 = bf16 && !train && gene_rows(T) >= 64;
    const bool fold = bf16 && !train;           // folded single-query attention weights (see pack_all_weights)      // q|k|v|gate handed to the attention kernel in BF16
    __nv_bfloat16* packed = bf16 ? reinterpret_cast<__nv_bfloat16*>(ws + w.bf_params) : nullptr;
    // Dense projection: tcgen05 BF16 engine when requested and the shape qualifies, FP32 SIMT otherwise.
    // (path_rows: the gene pass's row count when gene_rows cannot tell it from g.M)
    auto lin = [&](const GemmArgs& g, int nz, long long path_rows = -1) -> int {
        if (bf16 && train) {
            // training: parameters change every step, so nothing is packed: FP32 weights are converted while staged
            return gemm_auto(g, true, true, nz, st, true);
        }
        if (bf16 && (path_rows >= 0 ? path_rows : gene_rows(g.M)) >= 64 && g.B >= P && g.B < P + L.total && umma_supported(g))
            return umma_launch(g, packed + (g.B - P), nz, st);
        if (fold && g.B >= ws + w.fold_f32 && g.B < ws + w.fold_f32 + w.fold_total && umma_supported(g))
            return umma_launch(g, reinterpret_cast<const __nv_bfloat16*>(ws + w.fold_bf) + (g.B - (ws + w.fold_f32)), nz, st);
        if (g.c_bf16) { set_error("internal: BF16 output requested on the FP32 path"); return CHROMO_EINVAL; }
        return gemm_launch(g, true, true, nz, st);
    };
    if (bf16 && !train && !(flags & CHROMO_F_PACKED)) CHROMO_TRY(pack_all_weights(c, L, P, packed, ws, w, in, st));
    const bool pe_packed = bf16 && !train;      // the packed position tables exist
    // precision diagnostics (tools/precision_stress.py): keep one stage's contractions on the FP32 CUDA-core GEMM
    const bool reg_fp32 = getenv("CHROMO_REG_FP32") != nullptr, head_fp32 = getenv("CHROMO_HEAD_FP32") != nullptr;
    auto lin_fp32 = [&](const GemmArgs& g, int nz) -> int { return gemm_launch(g, true, true, nz, st); };
    if (w.reg_compact && reg_fp32) { set_error("CHROMO_REG_FP32 set after the replay workspace was sized"); return CHROMO_EINVAL; }

    RaggedPlan plan;                            // (ragged.cu; built next to the Embedding stage when the fused kernels run)
    bool ragged = false, reg_plan = false, reg_y_att = false;
    if (!only && !replay) {
    // ---------------- Embedding transformer, centre query (net.py:31-59) ----
    if (!pw) {
        CentreEmbedArgs a;
        a.B = B; a.D = D; a.F = F;
        for (int r = 0; r < NR; ++r) { a.x[r] = in->x_p[r]; a.pe[r] = in->pos_enc[r]; a.n[r] = c->n_bins[r]; }
        a.w = P + L.embed[0].lin_proj; a.w_stride = L.embed_stride;
        a.out = ws + w.e_hc; a.out_stride = RS;
        dim3 grid((B + CE_GENES - 1) / CE_GENES, NR);
        launch_pdl(centre_embed_kernel, dim3(grid), dim3(128), 0, st, a);
        CHROMO_CHECK_LAUNCH("centre_embed");
    }
    const AttnOff& ea = L.embed[0].att[0];
    const FfnOff& ef = L.embed[0].ffn[0];
    const int dme = c->embed_d_model;
    const int He = c->embed_heads;
    // fused single-query attention core (sqa_fused.cu): all resolutions of a stage in one launch
    auto sqa_fused = [&](int regions, int H, const float* const* x, const uint8_t* const* mask, const int64_t* mstride,
                         const int64_t* moff, int64_t w_in, long long w_in_z, int stage, int dm, float* qk, float* qkt,
                         float* cbar, bool cbar_bf16, bool probe, bool have_tiles, bool* done, const RaggedPlan* rp = nullptr) -> int {
        *done = false;
        if (!fold) return CHROMO_OK;
        SqaFusedArgs f;
        f.n_res = NR; f.regions = regions;
        for (int r = 0; r < NR; ++r) {
            f.n[r] = c->n_bins[r]; f.ns[r] = c->n_bins[r] <= 32 ? 32 : c->n_bins[r]; f.order[r] = r;
            f.x[r] = x[r]; f.mask[r] = mask[r]; f.mask_stride[r] = mstride[r]; f.mask_row_offset[r] = moff[r];
            f.pe_pk[r] = in->pos_enc[r] ? reinterpret_cast<const __nv_bfloat16*>(ws + w.bf_pe[r]) : nullptr;
        }
        for (int i = 1; i < NR; ++i)                       // long rows first
            for (int j = i; j > 0 && f.n[f.order[j]] > f.n[f.order[j - 1]]; --j) std::swap(f.order[j], f.order[j - 1]);
        f.qk_tiles = reinterpret_cast<const __nv_bfloat16*>(qkt); f.qk_tz = 2 * RS;
        f.w_in_pk = reinterpret_cast<const __nv_bfloat16*>(ws + w.bf_win[stage]); f.w_in_pk_z = 2048;
        f.cbar = cbar; f.cbar_z = RS;
        if (cbar_bf16) f.cbar_bf16 = reinterpret_cast<__nv_bfloat16*>(cbar);   // same buffer, BF16 rows (the fused tail reads them)
        f.w_in = P + w_in; f.w_in_z = w_in_z;
        f.scale = 1.f / sqrtf((float)(dm / H));
        if (rp) {
            f.perm = rp->perm; f.live = rp->live;
            for (int r = 0; r < NR; ++r) { f.tile_k0[r] = rp->tile_k0[r]; f.tile_ns[r] = rp->tile_ns[r]; }
        }
        if (!sqa_fused_supported(f, H, F, D)) return CHROMO_OK;
        *done = true;
        if (probe) return CHROMO_OK;
        // QK rows -> BF16 operand tiles, unless the query GEMM's epilogue has written them already
        if (!have_tiles) CHROMO_TRY(sqa_pack_qk(qk, RS, reinterpret_cast<__nv_bfloat16*>(qkt), 2 * RS, regions * H, NR, st));
        return launch_sqa_fused(f, st);
    };
    const bool tail = fold && w.tail_fused;
    const bool cb16 = tail;                     // Cbar handed from sqa_fused to the fused tail in BF16
    // the query GEMM of a stage written as the operand tiles of sqa_fused
    auto qk_tiles = [&](GemmArgs g, float* qkt) { g.c_sqa_tiles = 1; g.C = qkt; g.sC1 = 2 * RS; return g; };
    // the query GEMM of a stage: straight into the operand tiles of sqa_fused when that kernel will run and the tensor
    // GEMM takes the shape, FP32 rows otherwise
    auto qk_gemm = [&](const GemmArgs& g, float* qkt, bool sqa_ok, bool* tiles) -> int {
        const GemmArgs t = qk_tiles(g, qkt);
        *tiles = sqa_ok && umma_supported(t);
        return lin(*tiles ? t : g, NR);
    };
    // the folded query GEMM of Pairwise layer l over its input rows: QK = P_l M^T
    auto pw_qk = [&](int l, const float* pin, int pin_div) {
        GemmArgs g = gemm_args();
        g.A = pin; g.lda = D; g.sA1 = RS; g.a_div = pin_div;
        g.B = ws + w.fold_f32 + w.fold_slot[1 + l]; g.ldb = D; g.sB1 = w.fold_stride;
        g.C = ws + w.p_qk + (long long)w.pslot(l) * w.p_slot; g.ldc = c->pw_heads * D; g.sC1 = RS;
        g.M = R; g.N = c->pw_heads * D; g.K = D;
        return g;
    };
    // Ragged plan (ragged.cu): the Pairwise stage runs over the live pCRE slots only, sorted by valid length, each tile
    // of the attention over its own key window.  Built when every consumer of the stage takes it, as their own predicates
    // say for layer 0: sqa_fused, the fused tail, and the query GEMM in its operand-tile form on the persistent kernel
    // (qk_tiles_kernel).  Later layers differ from layer 0 only by workspace offsets, which keep the 16-byte alignment.
    RaggedArgs ra;
    AuxStream plan_stream{st, st};
    if (tail && w.rg_plan && c->pw_layers > 0 && !(flags & CHROMO_F_DENSE)) {
        bool ok = false;
        CHROMO_TRY(sqa_fused(R, c->pw_heads, in->x_pcre, in->mask_pcre, in->mask_pcre_stride, in->mask_pcre_row_offset,
                             L.pw[0].lin_proj_pcre, L.pw_stride, 1, c->pw_d_model, ws + w.p_qk, ws + w.p_qkt, ws + w.p_cbar, cb16, true, false, &ok));
        const GemmArgs q0 = qk_tiles(pw_qk(0, ws + w.p_pp, I), ws + w.p_qkt);
        if (ok && umma_supported(q0) && umma_qk_persistent(q0)) {
            ra.B = B; ra.I = I; ra.n_res = NR;
            for (int r = 0; r < NR; ++r) {
                ra.n[r] = c->n_bins[r]; ra.ns[r] = c->n_bins[r] <= 32 ? 32 : c->n_bins[r];
                ra.mask[r] = in->mask_pcre[r]; ra.mask_stride[r] = in->mask_pcre_stride[r]; ra.mask_row_offset[r] = in->mask_pcre_row_offset[r];
                ra.imask[r] = in->imask[r];
            }
            ra.xin = ws + w.r_xin; ra.xin_z = RS;
            // on a side stream next to the Embedding stage: forked here, launched behind that stage's kernels (which then
            // come first for the block scheduler; the plan's small latency-bound kernels fill the room they leave), joined
            // in front of the Pairwise stage
            CHROMO_TRY(aux_fork(st, &plan_stream.aux));
            ragged = true;
        }
    }
    const long long tail_z = (long long)(1 + c->pw_layers) * TAIL_SLOT_ELEMS;
    if (!pw) {      // (a Pairwise replay has its token 0 rows already)
    bool e_fused = false, e_tiles = false;
    CHROMO_TRY(sqa_fused(B, c->embed_heads, in->x_p, in->mask_p, in->mask_p_stride, in->mask_p_row_offset,
                         L.embed[0].lin_proj, L.embed_stride, 0, dme, ws + w.e_qk, ws + w.e_qkt, ws + w.e_cbar, cb16, true, false,
                         &e_fused));
    if (fold) {   // QK = Hc M^T  (M = [W_k[h]^T W_q[h]]_h)
        GemmArgs g = gemm_args();
        g.A = ws + w.e_hc; g.lda = D; g.sA1 = RS;
        g.B = ws + w.fold_f32 + w.fold_slot[0]; g.ldb = D; g.sB1 = w.fold_stride;
        g.C = ws + w.e_qk; g.ldc = He * D; g.sC1 = RS;
        g.M = B; g.N = He * D; g.K = D;
        CHROMO_TRY(qk_gemm(g, ws + w.e_qkt, e_fused, &e_tiles));
    } else {      // Q = Hc W_q^T
        GemmArgs g = gemm_args();
        g.A = ws + w.e_hc; g.lda = D; g.sA1 = RS;
        g.B = P + ea.att; g.ldb = D; g.sB1 = L.embed_stride;
        g.C = ws + w.e_q; g.ldc = dme; g.sC1 = RS;
        g.M = B; g.N = dme; g.K = D;
        CHROMO_TRY(lin(g, NR));
    }
    CHROMO_TRY(sqa_fused(B, c->embed_heads, in->x_p, in->mask_p, in->mask_p_stride, in->mask_p_row_offset,
                         L.embed[0].lin_proj, L.embed_stride, 0, dme, ws + w.e_qk, ws + w.e_qkt, ws + w.e_cbar, cb16, false, e_tiles,
                         &e_fused));
    ResStreams ers;
    if (!e_fused) CHROMO_TRY(res_fork(st, NR, ers));
    for (int r = 0; r < NR && !e_fused; ++r) {
        SqaArgs s;
        s.rows = B; s.H = c->embed_heads; s.dm = dme; s.D = D; s.n = c->n_bins[r]; s.F = F;
        s.q = ws + r * RS + w.e_q;
        s.w_k = P + L.embed[r].att[0].att + (long long)dme * D;
        s.w_v = P + L.embed[r].att[0].att + (long long)2 * dme * D;
        s.w_in = P + L.embed[r].lin_proj;
        s.pe = in->pos_enc[r];
        s.x = in->x_p[r];
        s.mask = in->mask_p[r]; s.mask_stride = in->mask_p_stride[r]; s.mask_row_offset = in->mask_p_row_offset[r];
        s.pe_pk = pe_packed ? reinterpret_cast<const __nv_bfloat16*>(ws + w.bf_pe[r]) : nullptr;
        s.pet_pk = pe_packed ? reinterpret_cast<const __nv_bfloat16*>(ws + w.bf_pet[r]) : nullptr;
        s.qk = ws + r * RS + w.e_qk; s.P = ws + w.e_p[r]; s.xbar = ws + r * RS + w.e_xbar;
        s.cbar = ws + r * RS + w.e_cbar; s.av = ws + r * RS + w.e_av; s.folded = fold; s.tc = bf16 && train;
        CHROMO_TRY(single_query_attention(s, ers.s[r]));
    }
    if (!e_fused) CHROMO_TRY(res_join(ers));
    if (tail) {   // out-projection + LN + FFN + LN in one launch (row_tail_fused.cu) -> X_in[b, 0, :]
        RowTailArgs t;
        t.M = B; t.dff = c->embed_d_ff;
        t.a = ws + w.e_cbar; t.lda = He * D; t.a_z = RS;
        if (e_fused && cb16) t.a_bf16 = reinterpret_cast<const __nv_bfloat16*>(ws + w.e_cbar);
        t.res = ws + w.e_hc; t.res_div = 1; t.res_z = RS;
        t.y = ws + w.r_xin; t.y_z = RS; t.c_div = 1; t.c_mul = S; t.c_add = 0;
        t.wstream = reinterpret_cast<const __nv_bfloat16*>(ws + w.tail_stream); t.w_z = tail_z;
        t.bo = P + ea.ffb; t.ln1w = P + ea.lnw; t.ln1b = P + ea.lnb; t.b1 = P + ef.l1b; t.b2 = P + ef.l2b;
        t.ln2w = P + ef.lnw; t.ln2b = P + ef.lnb; t.p_z = L.embed_stride;
        CHROMO_TRY(launch_row_tail_fused(t, NR, st));
    } else {
    {   // U = LN(Hc + Av W_o^T + b_o)                            modules.py:29-30
        GemmArgs g = gemm_args();
        g.A = ws + w.e_av; g.lda = dme; g.sA1 = RS;
        g.B = P + ea.ffw; g.ldb = dme; g.sB1 = L.embed_stride;
        g.C = ws + w.e_u; g.ldc = D; g.sC1 = RS;
        g.M = B; g.N = D; g.K = dme;
        if (fold) {   // ... = LN(Hc + Cbar N^T + b_o),  N = [W_o[:,h] W_v[h]]_h
            g.A = ws + w.e_cbar; g.lda = He * D; g.K = He * D;
            g.B = ws + w.fold_f32 + w.fold_slot[0] + (int64_t)He * D * D; g.ldb = He * D; g.sB1 = w.fold_stride;
        }
        g.epi = EPI_BIAS_RES_LN; g.bias = P + ea.ffb; g.sBias1 = L.embed_stride;
        g.res = ws + w.e_hc; g.ldres = D; g.sRes1 = RS;
        g.gamma = P + ea.lnw; g.beta = P + ea.lnb; g.sLn1 = L.embed_stride;
        if (train) { g.pre = ws + w.e_preU; g.sPre1 = RS; }
        CHROMO_TRY(lin(g, NR));
    }
    {   // F = relu(U W_1^T + b_1)                                modules.py:100-101
        GemmArgs g = gemm_args();
        g.A = ws + w.e_u; g.lda = D; g.sA1 = RS;
        g.B = P + ef.l1w; g.ldb = D; g.sB1 = L.embed_stride;
        g.C = ws + w.e_f; g.ldc = c->embed_d_ff; g.sC1 = RS;
        g.M = B; g.N = c->embed_d_ff; g.K = D;
        g.epi = EPI_BIAS_RELU; g.bias = P + ef.l1b; g.sBias1 = L.embed_stride;
        CHROMO_TRY(lin(g, NR));
    }
    {   // Y = LN(U + F W_2^T + b_2) -> X_in[b, 0, :]              net.py:359-368
        GemmArgs g = gemm_args();
        g.A = ws + w.e_f; g.lda = c->embed_d_ff; g.sA1 = RS;
        g.B = P + ef.l2w; g.ldb = c->embed_d_ff; g.sB1 = L.embed_stride;
        g.C = ws + w.r_xin; g.ldc = D; g.sC1 = RS; g.c_div = 1; g.c_mul = S; g.c_add = 0;
        g.M = B; g.N = D; g.K = c->embed_d_ff;
        g.epi = EPI_BIAS_RES_LN; g.bias = P + ef.l2b; g.sBias1 = L.embed_stride;
        g.res = ws + w.e_u; g.ldres = D; g.sRes1 = RS;
        g.gamma = P + ef.lnw; g.beta = P + ef.lnb; g.sLn1 = L.embed_stride;
        if (train) { g.pre = ws + w.e_preY; g.sPre1 = RS; }
        CHROMO_TRY(lin(g, NR));
    }
    }   // !tail
    }   // !pw

    // ---------------- Pairwise Interaction transformer (net.py:105-139) -----
    const int dmp = c->pw_d_model, Hp = c->pw_heads;
    float* const xin = pw ? pw->xin : ws + w.r_xin;       // token 0 in, the pCRE tokens out
    const long long xin_z = pw ? pw->xin_z : RS;
    {   // PP = Y_c W_lpp^T   (identical for the I slots of a gene, net.py:114-118)
        GemmArgs g = gemm_args();
        g.A = xin; g.lda = S * D; g.sA1 = xin_z;
        g.B = P + L.pw[0].lin_proj_p; g.ldb = D; g.sB1 = L.pw_stride;
        g.C = ws + w.p_pp; g.ldc = D; g.sC1 = RS;
        g.M = B; g.N = D; g.K = D;
        CHROMO_TRY(lin(g, NR, pw ? pw->gene_batch : -1));
    }
    if (ragged) {
        CHROMO_TRY(build_ragged_plan(ra, ws + w.rg_plan, &plan, plan_stream.aux));
        CHROMO_TRY(plan_stream.join());
    }
    const RaggedPlan* rp = ragged ? &plan : nullptr;
    for (int l = 0; l < c->pw_layers; ++l) {
        const AttnOff& pa = L.pw[0].att[l];
        const FfnOff& pf = L.pw[0].ffn[l];
        const long long so = (long long)w.pslot(l) * w.p_slot;
        const float* pin = l == 0 ? ws + w.p_pp : ws + w.p_out + (long long)w.pslot(l - 1) * w.p_slot;
        const int pin_div = l == 0 ? I : 1;
        const bool last = l == c->pw_layers - 1;
        bool p_fused = false, p_tiles = false;
        CHROMO_TRY(sqa_fused(R, Hp, in->x_pcre, in->mask_pcre, in->mask_pcre_stride, in->mask_pcre_row_offset,
                             L.pw[0].lin_proj_pcre, L.pw_stride, 1, dmp, ws + w.p_qk + so, ws + w.p_qkt + so, ws + w.p_cbar + so,
                             cb16, true, false, &p_fused));
        if (fold) {   // QK = P_l M^T
            GemmArgs g = pw_qk(l, pin, pin_div);
            if (rp) { g.m_dev = rp->live; g.a_rows = l == 0 ? rp->perm : nullptr; }   // (later layers read the compacted rows)
            CHROMO_TRY(qk_gemm(g, ws + w.p_qkt + so, p_fused, &p_tiles));
        } else {      // Q = P_l W_q^T                             modules.py:159
            GemmArgs g = gemm_args();
            g.A = pin; g.lda = D; g.sA1 = RS; g.a_div = pin_div;
            g.B = P + pa.p_att; g.ldb = D; g.sB1 = L.pw_stride;
            g.C = ws + w.p_q + so; g.ldc = dmp; g.sC1 = RS;
            g.M = R; g.N = dmp; g.K = D;
            CHROMO_TRY(lin(g, NR));
        }
        CHROMO_TRY(sqa_fused(R, Hp, in->x_pcre, in->mask_pcre, in->mask_pcre_stride, in->mask_pcre_row_offset,
                             L.pw[0].lin_proj_pcre, L.pw_stride, 1, dmp, ws + w.p_qk + so, ws + w.p_qkt + so, ws + w.p_cbar + so,
                             cb16, false, p_tiles, &p_fused, rp));
        ResStreams prs;
        if (!p_fused) CHROMO_TRY(res_fork(st, NR, prs));
        for (int r = 0; r < NR && !p_fused; ++r) {
            SqaArgs s;
            s.rows = R; s.H = Hp; s.dm = dmp; s.D = D; s.n = c->n_bins[r]; s.F = F;
            s.q = ws + r * RS + w.p_q + so;
            s.w_k = P + L.pw[r].att[l].c_att;
            s.w_v = P + L.pw[r].att[l].c_att + (long long)dmp * D;
            s.w_in = P + L.pw[r].lin_proj_pcre;
            s.pe = in->pos_enc[r];
            s.x = in->x_pcre[r];
            s.mask = in->mask_pcre[r]; s.mask_stride = in->mask_pcre_stride[r];
            s.mask_row_offset = in->mask_pcre_row_offset[r];
            s.pe_pk = pe_packed ? reinterpret_cast<const __nv_bfloat16*>(ws + w.bf_pe[r]) : nullptr;
            s.pet_pk = pe_packed ? reinterpret_cast<const __nv_bfloat16*>(ws + w.bf_pet[r]) : nullptr;
            s.qk = ws + r * RS + w.p_qk + so;
            s.P = ws + w.p_p[r] + (long long)w.pslot(l) * w.p_p_slot[r];
            s.xbar = ws + r * RS + w.p_xbar + so;
            s.cbar = ws + r * RS + w.p_cbar + so; s.av = ws + r * RS + w.p_av + so; s.folded = fold; s.tc = bf16 && train;
            s.path_rows = gene_rows(R);
            CHROMO_TRY(single_query_attention(s, prs.s[r]));
        }
        if (!p_fused) CHROMO_TRY(res_join(prs));
        if (tail) {
            RowTailArgs t;
            t.M = R; t.dff = c->pw_d_ff;
            t.a = ws + w.p_cbar + so; t.lda = Hp * D; t.a_z = RS;
            if (p_fused && cb16) t.a_bf16 = reinterpret_cast<const __nv_bfloat16*>(ws + w.p_cbar + so);
            t.res = pin; t.res_div = pin_div; t.res_z = RS;
            if (last) { t.y = xin; t.c_div = I; t.c_mul = S; t.c_add = 1; }
            else { t.y = ws + w.p_out + so; t.c_div = 1; t.c_mul = 1; t.c_add = 0; }
            t.y_z = last ? xin_z : RS;
            t.wstream = reinterpret_cast<const __nv_bfloat16*>(ws + w.tail_stream) + (1 + l) * TAIL_SLOT_ELEMS; t.w_z = tail_z;
            t.bo = P + pa.ffb; t.ln1w = P + pa.lnw; t.ln1b = P + pa.lnb; t.b1 = P + pf.l1b; t.b2 = P + pf.l2b;
            t.ln2w = P + pf.lnw; t.ln2b = P + pf.lnb; t.p_z = L.pw_stride;
            if (rp) { t.m_dev = rp->live; t.res_rows = l == 0 ? rp->perm : nullptr; t.y_rows = last ? rp->y_rows : nullptr; }
            CHROMO_TRY(launch_row_tail_fused(t, NR, st));
            continue;
        }
        {   // U = LN(P_l + Av W_o^T + b_o)                        modules.py:150-152
            GemmArgs g = gemm_args();
            g.A = ws + w.p_av + so; g.lda = dmp; g.sA1 = RS;
            g.B = P + pa.ffw; g.ldb = dmp; g.sB1 = L.pw_stride;
            g.C = ws + w.p_u + so; g.ldc = D; g.sC1 = RS;
            g.M = R; g.N = D; g.K = dmp;
            if (fold) {
                g.A = ws + w.p_cbar + so; g.lda = Hp * D; g.K = Hp * D;
                g.B = ws + w.fold_f32 + w.fold_slot[1 + l] + (int64_t)Hp * D * D; g.ldb = Hp * D; g.sB1 = w.fold_stride;
            }
            g.epi = EPI_BIAS_RES_LN; g.bias = P + pa.ffb; g.sBias1 = L.pw_stride;
            g.res = pin; g.ldres = D; g.res_div = pin_div; g.sRes1 = RS;
            g.gamma = P + pa.lnw; g.beta = P + pa.lnb; g.sLn1 = L.pw_stride;
            if (train) { g.pre = ws + w.p_preU + so; g.sPre1 = RS; }
            CHROMO_TRY(lin(g, NR));
        }
        {
            GemmArgs g = gemm_args();
            g.A = ws + w.p_u + so; g.lda = D; g.sA1 = RS;
            g.B = P + pf.l1w; g.ldb = D; g.sB1 = L.pw_stride;
            g.C = ws + w.p_f + so; g.ldc = c->pw_d_ff; g.sC1 = RS;
            g.M = R; g.N = c->pw_d_ff; g.K = D;
            g.epi = EPI_BIAS_RELU; g.bias = P + pf.l1b; g.sBias1 = L.pw_stride;
            CHROMO_TRY(lin(g, NR));
        }
        {   // P_{l+1} = LN(U + F W_2^T + b_2); the last layer lands in X_in[b, 1+i, :]
            GemmArgs g = gemm_args();
            g.A = ws + w.p_f + so; g.lda = c->pw_d_ff; g.sA1 = RS;
            g.B = P + pf.l2w; g.ldb = c->pw_d_ff; g.sB1 = L.pw_stride;
            if (last) { g.C = xin; g.c_div = I; g.c_mul = S; g.c_add = 1; }
            else g.C = ws + w.p_out + so;
            g.ldc = D; g.sC1 = last ? xin_z : RS;
            g.M = R; g.N = D; g.K = c->pw_d_ff;
            g.epi = EPI_BIAS_RES_LN; g.bias = P + pf.l2b; g.sBias1 = L.pw_stride;
            g.res = ws + w.p_u + so; g.ldres = D; g.sRes1 = RS;
            g.gamma = P + pf.lnw; g.beta = P + pf.lnb; g.sLn1 = L.pw_stride;
            if (train) { g.pre = ws + w.p_preY + so; g.sPre1 = RS; }
            CHROMO_TRY(lin(g, NR));
        }
    }

    if (pw) return CHROMO_OK;
    }   // !only && !replay
    // ---------------- Regulation transformer (net.py:152-153) ---------------
    const int dmr = c->reg_d_model, Hr = c->reg_heads;
    const bool pb16 = proj_bf16 && !reg_fp32;
    const RaggedPlan* rgp = ragged ? &plan : replay ? replay->plan : nullptr;
    auto rlin = [&](const GemmArgs& g, int nz) -> int { return reg_fp32 ? lin_fp32(g, nz) : lin(g, nz); };
    for (int l = 0; l < c->reg_layers; ++l) {
        if (only && only->layer >= 0 && l != only->layer) continue;
        const AttnOff& ra = L.reg[0].att[l];
        const FfnOff& rf = L.reg[0].ffn[l];
        const long long so = (long long)w.rslot(l) * w.r_slot;
        const float* xin = l == 0 ? ws + w.r_xin : ws + w.r_out + (long long)w.rslot(l - 1) * w.r_slot;
        float* xout = ws + w.r_out + so;
        long long x_z = RS, y_z = RS;
        if (only) { xin = only->x; xout = only->y; x_z = y_z = only->xy_stride; }
        if (w.reg_fused && !reg_fp32) {
            // ALL layers in one launch (reg_fused.cu), unless the caller asked for one layer: a CTA keeps its 14 genes on
            // chip from layer to layer (the tokens of a gene only attend to each other)
            const bool all = !only || only->layer < 0;
            if (all && l > 0) continue;
            RegFusedArgs a;
            a.B = B; a.S = S; a.G = 128 / S; a.n_tiles = (B + a.G - 1) / a.G;
            if (rgp && all) {
                // token classes of the plan: a tile holds genes of one class with their live tokens only
                a.plan_tiles = rgp->reg_tiles; a.plan_rows = rgp->reg_rows; a.n_tiles = rgp->reg_tiles_max;
                reg_plan = true;
            }
            a.x = xin; a.x_z = x_z; a.y = xout; a.y_z = y_z;
            a.n_layers = 1; a.y_mid = nullptr; a.y_mid_z = 0; a.y_l = 0; a.p_l = 0;
            if (all) {
                a.n_layers = c->reg_layers;
                a.y_mid = ws + w.r_out; a.y_mid_z = RS; a.y_l = w.rslots > 1 ? w.r_slot : 0;
                if (!only) a.y = ws + w.r_out + (long long)w.rslot(c->reg_layers - 1) * w.r_slot;
                // the rows of the last layer must not land in a parking block of the scratch slots (a persistent CTA parks
                // in the block of its own index, and under a plan a tile's rows are scattered over the [B*S, 128] layout):
                // they go to the (otherwise unused) attention buffer of the layer-by-layer path
                if (!only) { a.y = ws + w.r_att; reg_y_att = true; a.y_head_only = 1; }   // (head_gather reads token 0 only)
                a.p_l = c->reg_layers > 1 ? L.reg[0].att[1].gamma_f - L.reg[0].att[0].gamma_f : 0;
            }
            a.wstream = reinterpret_cast<const __nv_bfloat16*>(ws + w.reg_stream) + (long long)l * reg_stream_elems_per_layer();
            a.w_z = (long long)c->reg_layers * reg_stream_elems_per_layer();
            a.gamma_f = P + ra.gamma_f; a.bo = P + ra.ffb; a.ln1w = P + ra.lnw; a.ln1b = P + ra.lnb;
            a.b1 = P + rf.l1b; a.b2 = P + rf.l2b; a.ln2w = P + rf.lnw; a.ln2b = P + rf.lnb; a.p_z = L.reg_stride;
            a.freq = in->freq;
            for (int r = 0; r < NR; ++r) a.imask[r] = in->imask[r];
            CHROMO_TRY(launch_reg_layer_fused(a, NR, st));
            continue;
        }
        {   // proj = X W_att^T  (q|k|v|gate)                       modules.py:38
            GemmArgs g = gemm_args();
            g.A = xin; g.lda = D; g.sA1 = x_z;
            g.B = P + ra.att; g.ldb = D; g.sB1 = L.reg_stride;
            g.C = ws + w.r_proj + so; g.ldc = 4 * dmr; g.sC1 = RS;
            if (pb16) { g.c_bf16 = 1; g.sC1 = 2 * RS; }
            g.M = T; g.N = 4 * dmr; g.K = D;
            CHROMO_TRY(rlin(g, NR));
        }
        {
            RegAttnArgs a;
            a.B = B; a.S = S; a.H = Hr;
            a.proj = ws + w.r_proj + so; a.proj_zstride = pb16 ? 2 * RS : RS; a.proj_bf16 = pb16 ? 1 : 0;
            a.gamma_f = P + ra.gamma_f; a.gamma_zstride = L.reg_stride;
            a.freq = in->freq;
            for (int r = 0; r < NR; ++r) a.imask[r] = in->imask[r];
            a.prob = train ? ws + w.r_prob + so : nullptr; a.prob_zstride = RS;
            a.out = ws + w.r_att + so; a.out_zstride = RS;
            CHROMO_TRY(launch_reg_attention(a, NR, st));
        }
        {
            GemmArgs g = gemm_args();
            g.A = ws + w.r_att + so; g.lda = dmr; g.sA1 = RS;
            g.B = P + ra.ffw; g.ldb = dmr; g.sB1 = L.reg_stride;
            g.C = ws + w.r_u + so; g.ldc = D; g.sC1 = RS;
            g.M = T; g.N = D; g.K = dmr;
            g.epi = EPI_BIAS_RES_LN; g.bias = P + ra.ffb; g.sBias1 = L.reg_stride;
            g.res = xin; g.ldres = D; g.sRes1 = x_z;
            g.gamma = P + ra.lnw; g.beta = P + ra.lnb; g.sLn1 = L.reg_stride;
            if (train) { g.pre = ws + w.r_preU + so; g.sPre1 = RS; }
            CHROMO_TRY(rlin(g, NR));
        }
        {
            GemmArgs g = gemm_args();
            g.A = ws + w.r_u + so; g.lda = D; g.sA1 = RS;
            g.B = P + rf.l1w; g.ldb = D; g.sB1 = L.reg_stride;
            g.C = ws + w.r_f + so; g.ldc = c->reg_d_ff; g.sC1 = RS;
            g.M = T; g.N = c->reg_d_ff; g.K = D;
            g.epi = EPI_BIAS_RELU; g.bias = P + rf.l1b; g.sBias1 = L.reg_stride;
            CHROMO_TRY(rlin(g, NR));
        }
        {
            GemmArgs g = gemm_args();
            g.A = ws + w.r_f + so; g.lda = c->reg_d_ff; g.sA1 = RS;
            g.B = P + rf.l2w; g.ldb = c->reg_d_ff; g.sB1 = L.reg_stride;
            g.C = xout; g.ldc = D; g.sC1 = y_z;
            g.M = T; g.N = D; g.K = c->reg_d_ff;
            g.epi = EPI_BIAS_RES_LN; g.bias = P + rf.l2b; g.sBias1 = L.reg_stride;
            g.res = ws + w.r_u + so; g.ldres = D; g.sRes1 = RS;
            g.gamma = P + rf.lnw; g.beta = P + rf.lnb; g.sLn1 = L.reg_stride;
            if (train) { g.pre = ws + w.r_preY + so; g.sPre1 = RS; }
            CHROMO_TRY(rlin(g, NR));
        }
    }

    if (only) return CHROMO_OK;
    // ---------------- head (net.py:377-380) ---------------------------------
    {
        HeadGatherArgs a;
        a.B = B; a.S = S; a.D = D; a.n_res = NR;
        a.xout = reg_y_att ? ws + w.r_att : ws + w.r_out + (long long)w.rslot(c->reg_layers - 1) * w.r_slot;
        a.xin = ws + w.r_xin; a.zstride = RS; a.z = ws + w.h_z;
        launch_pdl(head_gather_kernel, dim3((B * NR * D + 255) / 256), dim3(256), 0, st, a);
        CHROMO_CHECK_LAUNCH("head_gather");
    }
    {
        GemmArgs g = gemm_args();
        g.A = ws + w.h_z; g.lda = NR * D;
        g.B = P + L.fc0w; g.ldb = NR * D;
        g.C = ws + w.h_h1; g.ldc = c->d_head;
        g.M = B; g.N = c->d_head; g.K = NR * D;
        g.epi = EPI_BIAS_RELU; g.bias = P + L.fc0b;
        CHROMO_TRY(head_fp32 ? lin_fp32(g, 1) : lin(g, 1));
    }
    {
        GemmArgs g = gemm_args();
        g.A = ws + w.h_h1; g.lda = c->d_head;
        g.B = P + L.fc2w; g.ldb = c->d_head;
        g.C = logits; g.ldc = c->n_out;
        g.M = B; g.N = c->n_out; g.K = c->d_head;
        g.epi = EPI_BIAS; g.bias = P + L.fc2b;
        CHROMO_TRY(head_fp32 ? lin_fp32(g, 1) : lin(g, 1));
    }
    (void)flags;
    return CHROMO_OK;
}

}  // namespace chromo

using namespace chromo;

static int check_forward_args(const chromo_config_t* cfg, const float* params, const chromo_batch_t* in,
                              const float* logits, const float* workspace) {
    CHROMO_TRY(validate_config(cfg));
    if (!params || !in || !logits || !workspace) { set_error("null pointer argument"); return CHROMO_EINVAL; }
    if (in->batch < 1) { set_error("batch must be >= 1"); return CHROMO_EINVAL; }
    for (int r = 0; r < cfg->n_res; ++r) {
        if (!in->x_p[r] || !in->x_pcre[r] || !in->mask_p[r] || !in->mask_pcre[r] || !in->imask[r] ||
            !in->pos_enc[r]) {
            set_error("null input tensor for resolution %d", r);
            return CHROMO_EINVAL;
        }
    }
    if (!in->freq) { set_error("null interaction_freq"); return CHROMO_EINVAL; }
    return CHROMO_OK;
}

extern "C" int chromo_forward(const chromo_config_t* cfg, const float* params, const chromo_batch_t* in,
                              float* logits, float* workspace, int64_t workspace_floats, int32_t flags,
                              void* stream) {
    CHROMO_TRY(check_forward_args(cfg, params, in, logits, workspace));
    WsLayout w = make_ws_layout(cfg, in->batch, flags);
    if (workspace_floats < w.total) {
        set_error("workspace too small: need %lld floats, got %lld", (long long)w.total, (long long)workspace_floats);
        return CHROMO_ENOMEM;
    }
    return forward_impl(cfg, params, in, logits, workspace, w, flags, (cudaStream_t)stream);
}

// ---- in-silico pCRE deletion (deletion.cu) ----
// Workspace: the variant pass's own layout [0, wv.total) (its batch-independent front holds the packed BF16 weights both
// passes read; the gene pass's layout fits inside it), then the gene X_in rows, the variants' freq and masks, their
// logits and the Regulation plan of the variants.
namespace {
struct DeletionWs {
    WsLayout wb, wv;
    int64_t xin_b, freq_v, imask_v, logits_v, plan, total;
    bool plan_on;
};
int deletion_ws(const chromo_config_t* c, int batch, int flags, DeletionWs* d) {
    const int S = c->i_max + 1;
    if ((int64_t)batch * S * S > INT32_MAX) { set_error("chromo_pcre_deletion: batch * (i_max + 1)^2 must fit in int32"); return CHROMO_EINVAL; }
    const int V = batch * S;
    d->wb = make_ws_layout(c, batch, flags);
    d->wv = make_ws_layout(c, V, flags);
    int64_t cur = d->wv.total;
    auto take = [&](int64_t n) { int64_t o = cur; cur = align4(cur + n); return o; };
    d->xin_b = take((int64_t)c->n_res * batch * S * c->d_emb);
    d->freq_v = take((int64_t)V * S * S);
    d->imask_v = take(((int64_t)V * S * S + 3) / 4 * c->n_res);
    d->logits_v = take((int64_t)V * c->n_out);
    d->plan_on = (flags & CHROMO_F_BF16) && d->wv.reg_fused;
    d->plan = d->plan_on ? take(reg_plan_floats(V, c->i_max)) : 0;
    d->total = cur;
    return CHROMO_OK;
}
}  // namespace

extern "C" int64_t chromo_pcre_deletion_workspace_floats(const chromo_config_t* cfg, int32_t batch, int32_t flags) {
    if (validate_config(cfg) != CHROMO_OK) return CHROMO_EINVAL;
    if (batch < 1) { set_error("batch must be >= 1"); return CHROMO_EINVAL; }
    DeletionWs d;
    CHROMO_TRY(deletion_ws(cfg, batch, flags, &d));
    return d.total;
}

extern "C" int chromo_pcre_deletion(const chromo_config_t* cfg, const float* params, const chromo_batch_t* in,
                                    float* logits, float* without, float* promoter_only, float* workspace,
                                    int64_t workspace_floats, int32_t flags, void* stream) {
    CHROMO_TRY(check_forward_args(cfg, params, in, logits, workspace));
    if (!without || !promoter_only) { set_error("chromo_pcre_deletion: null output"); return CHROMO_EINVAL; }
    if (flags & (CHROMO_F_TRAINING | CHROMO_F_REGONLY | CHROMO_F_BWD_HEAD_REG | CHROMO_F_BWD_REST | CHROMO_F_FREQ_GRAD)) {
        set_error("chromo_pcre_deletion: inference only (flags CHROMO_F_BF16, CHROMO_F_PACKED, CHROMO_F_DENSE)");
        return CHROMO_EINVAL;
    }
    DeletionWs d;
    CHROMO_TRY(deletion_ws(cfg, in->batch, flags, &d));
    if (workspace_floats < d.total) {
        set_error("chromo_pcre_deletion: workspace too small: need %lld floats, got %lld", (long long)d.total,
                  (long long)workspace_floats);
        return CHROMO_ENOMEM;
    }
    cudaStream_t st = (cudaStream_t)stream;
    float* ws = workspace;
    const int B = in->batch, I = cfg->i_max, S = I + 1, V = B * S, NR = cfg->n_res, D = cfg->d_emb;
    // the genes: the ordinary forward (it packs the BF16 weights unless CHROMO_F_PACKED), X_in left in the workspace
    CHROMO_TRY(forward_impl(cfg, params, in, logits, ws, d.wb, flags, st));
    // their X_in rows out of the way of the variant layout, which overlaps the gene layout
    const size_t row_bytes = (size_t)B * S * D * sizeof(float);
    if (cudaMemcpy2DAsync(ws + d.xin_b, row_bytes, ws + d.wb.r_xin, (size_t)d.wb.res_stride * sizeof(float), row_bytes, NR,
                          cudaMemcpyDeviceToDevice, st) != cudaSuccess) {
        set_error("chromo_pcre_deletion: X_in copy failed");
        return CHROMO_ECUDA;
    }
    chromo_batch_t vin;
    memset(&vin, 0, sizeof(vin));
    vin.batch = V; vin.freq = ws + d.freq_v;
    {
        DeletionExpandArgs a;
        a.B = B; a.I = I; a.n_res = NR;
        a.xin = ws + d.xin_b; a.xin_z = (long long)B * S * D;
        a.freq = in->freq;
        a.xin_v = ws + d.wv.r_xin; a.xin_v_z = d.wv.res_stride;
        a.freq_v = ws + d.freq_v;
        for (int r = 0; r < NR; ++r) {
            a.imask[r] = in->imask[r];
            a.imask_v[r] = reinterpret_cast<uint8_t*>(ws + d.imask_v) + (long long)r * V * S * S;
            vin.imask[r] = a.imask_v[r];
        }
        CHROMO_TRY(launch_deletion_expand(a, st));
    }
    RaggedPlan plan;
    if (d.plan_on) {
        RaggedArgs ra;
        memset(&ra, 0, sizeof(ra));
        ra.B = V; ra.I = I; ra.n_res = NR;
        for (int r = 0; r < NR; ++r) ra.imask[r] = vin.imask[r];
        CHROMO_TRY(build_reg_plan(ra, ws + d.plan, &plan, st));
    }
    // the variants: Regulation transformer + head, with the weights the gene pass packed
    const RegReplay replay{d.plan_on ? &plan : nullptr, B};
    const int vflags = (flags & ~CHROMO_F_DENSE) | ((flags & CHROMO_F_BF16) ? CHROMO_F_PACKED : 0);
    CHROMO_TRY(forward_impl(cfg, params, &vin, ws + d.logits_v, ws, d.wv, vflags, st, nullptr, &replay));
    DeletionScatterArgs s;
    s.B = B; s.I = I; s.n_res = NR; s.n_out = cfg->n_out;
    for (int r = 0; r < NR; ++r) s.imask[r] = in->imask[r];
    s.logits = logits; s.logits_v = ws + d.logits_v;
    s.without = without; s.promoter_only = promoter_only;
    return launch_deletion_scatter(s, st);
}

// ---- pCRE subsets (subsets.cu) and interaction-frequency edits (freq_edits.cu) ----
// Workspace: the larger of the gene pass's layout and the replay layout of the V variants [0, front) (both start with
// the same batch-independent front, the packed BF16 weights; the replay layout has no Embedding or Pairwise block), then
// the gene X_in rows, the variants' freq and masks and the Regulation plan of the variants.  chromo_freq_edits adds the
// V empty drop sets of subset_expand_kernel behind it.
namespace {
struct SubsetsWs {
    WsLayout wb, wv;
    int64_t xin_b, freq_v, imask_v, plan, total;
    bool plan_on;
};
int subsets_ws(const chromo_config_t* c, int batch, int variants, int flags, SubsetsWs* d, const char* fn) {
    const int S = c->i_max + 1;
    const int64_t row = std::max<int64_t>((int64_t)S * S, (int64_t)c->n_res * c->d_emb);
    if ((int64_t)batch * row > INT32_MAX || (int64_t)variants * row > INT32_MAX) {
        set_error("%s: batch and variants times max((i_max + 1)^2, n_res * d_emb) must fit in int32", fn);
        return CHROMO_EINVAL;
    }
    const int V = variants;
    d->wb = make_ws_layout(c, batch, flags);
    d->wv = make_ws_layout(c, V, flags, true);
    int64_t cur = std::max(d->wb.total, d->wv.total);
    auto take = [&](int64_t n) { int64_t o = cur; cur = align4(cur + n); return o; };
    d->xin_b = take((int64_t)c->n_res * batch * S * c->d_emb);
    d->freq_v = take((int64_t)V * S * S);
    d->imask_v = take(((int64_t)V * S * S + 3) / 4 * c->n_res);
    d->plan_on = (flags & CHROMO_F_BF16) && d->wv.reg_fused;
    d->plan = d->plan_on ? take(reg_plan_floats(V, c->i_max)) : 0;
    d->total = cur;
    return CHROMO_OK;
}

// chromo_freq_edits: the subsets layout, then the V drop words at d.total
int64_t freq_edits_total(const SubsetsWs& d, int variants) { return align4(d.total + variants); }

int check_subsets_args(const chromo_config_t* cfg, const float* params, const chromo_batch_t* in, const void* var_gene,
                       const void* var_desc, int variants, const float* logits, const float* var_logits,
                       const float* workspace, int flags, const char* fn) {
    CHROMO_TRY(check_forward_args(cfg, params, in, logits, workspace));
    if (!var_gene || !var_desc || !var_logits) { set_error("%s: null variant descriptor or output", fn); return CHROMO_EINVAL; }
    if (variants < 1) { set_error("%s: variants must be >= 1", fn); return CHROMO_EINVAL; }
    if (flags & ~(CHROMO_F_BF16 | CHROMO_F_PACKED | CHROMO_F_DENSE)) {
        set_error("%s: inference only (flags CHROMO_F_BF16, CHROMO_F_PACKED, CHROMO_F_DENSE)", fn);
        return CHROMO_EINVAL;
    }
    return CHROMO_OK;
}

// The sequence both entry points run: the gene pass, its X_in set aside, subset_expand_kernel, the splice of the freq
// edits (`splice`, chromo_freq_edits only: its B, I, V and freq_v are filled in here), the variants' Regulation plan,
// the replay of the Regulation transformer and the head, and subset_guard_kernel.
int subsets_run(const chromo_config_t* cfg, const float* params, const chromo_batch_t* in, const int32_t* var_gene,
                const uint32_t* var_drop, int V, float* logits, float* var_logits, float* ws, const SubsetsWs& d,
                int flags, cudaStream_t st, FreqSpliceArgs* splice, const char* fn) {
    const int B = in->batch, I = cfg->i_max, S = I + 1, NR = cfg->n_res, D = cfg->d_emb;
    // the genes: the ordinary forward (it packs the BF16 weights unless CHROMO_F_PACKED), X_in left in the workspace
    CHROMO_TRY(forward_impl(cfg, params, in, logits, ws, d.wb, flags, st));
    // their X_in rows out of the way of the replay layout, which overlaps the gene layout
    const size_t row_bytes = (size_t)B * S * D * sizeof(float);
    if (cudaMemcpy2DAsync(ws + d.xin_b, row_bytes, ws + d.wb.r_xin, (size_t)d.wb.res_stride * sizeof(float), row_bytes, NR,
                          cudaMemcpyDeviceToDevice, st) != cudaSuccess) {
        set_error("%s: X_in copy failed", fn);
        return CHROMO_ECUDA;
    }
    chromo_batch_t vin;
    memset(&vin, 0, sizeof(vin));
    vin.batch = V; vin.freq = ws + d.freq_v;
    {
        SubsetExpandArgs a;
        a.B = B; a.I = I; a.n_res = NR; a.V = V;
        a.var_gene = var_gene; a.var_drop = var_drop;
        a.xin = ws + d.xin_b; a.xin_z = (long long)B * S * D;
        a.freq = in->freq;
        a.xin_v = ws + d.wv.r_xin; a.xin_v_z = d.wv.res_stride;
        a.freq_v = ws + d.freq_v;
        for (int r = 0; r < NR; ++r) {
            a.imask[r] = in->imask[r];
            a.imask_v[r] = reinterpret_cast<uint8_t*>(ws + d.imask_v) + (long long)r * V * S * S;
            vin.imask[r] = a.imask_v[r];
        }
        CHROMO_TRY(launch_subset_expand(a, st));
    }
    if (splice) {
        splice->B = B; splice->I = I; splice->V = V;
        splice->freq_v = ws + d.freq_v;
        CHROMO_TRY(launch_freq_splice(*splice, st));
    }
    RaggedPlan plan;
    if (d.plan_on) {
        RaggedArgs ra;
        memset(&ra, 0, sizeof(ra));
        ra.B = V; ra.I = I; ra.n_res = NR;
        for (int r = 0; r < NR; ++r) ra.imask[r] = vin.imask[r];
        CHROMO_TRY(build_reg_plan(ra, ws + d.plan, &plan, st));
    }
    // the variants: Regulation transformer + head, with the weights the gene pass packed, logits in variant order
    const RegReplay replay{d.plan_on ? &plan : nullptr, B};
    const int vflags = (flags & ~CHROMO_F_DENSE) | ((flags & CHROMO_F_BF16) ? CHROMO_F_PACKED : 0);
    CHROMO_TRY(forward_impl(cfg, params, &vin, var_logits, ws, d.wv, vflags, st, nullptr, &replay));
    SubsetGuardArgs gd;
    gd.B = B; gd.I = I; gd.V = V; gd.n_out = cfg->n_out;
    gd.var_gene = var_gene; gd.var_drop = var_drop; gd.logits_v = var_logits;
    return launch_subset_guard(gd, st);
}
}  // namespace

extern "C" int64_t chromo_pcre_subsets_workspace_floats(const chromo_config_t* cfg, int32_t batch, int32_t variants,
                                                        int32_t flags) {
    if (validate_config(cfg) != CHROMO_OK) return CHROMO_EINVAL;
    if (batch < 1 || variants < 1) { set_error("batch and variants must be >= 1"); return CHROMO_EINVAL; }
    SubsetsWs d;
    CHROMO_TRY(subsets_ws(cfg, batch, variants, flags, &d, "chromo_pcre_subsets"));
    return d.total;
}

extern "C" int chromo_pcre_subsets(const chromo_config_t* cfg, const float* params, const chromo_batch_t* in,
                                   const int32_t* var_gene, const uint32_t* var_drop, int32_t variants, float* logits,
                                   float* var_logits, float* workspace, int64_t workspace_floats, int32_t flags,
                                   void* stream) {
    const char* fn = "chromo_pcre_subsets";
    CHROMO_TRY(check_subsets_args(cfg, params, in, var_gene, var_drop, variants, logits, var_logits, workspace, flags, fn));
    SubsetsWs d;
    CHROMO_TRY(subsets_ws(cfg, in->batch, variants, flags, &d, fn));
    if (workspace_floats < d.total) {
        set_error("%s: workspace too small: need %lld floats, got %lld", fn, (long long)d.total,
                  (long long)workspace_floats);
        return CHROMO_ENOMEM;
    }
    return subsets_run(cfg, params, in, var_gene, var_drop, variants, logits, var_logits, workspace, d, flags,
                       (cudaStream_t)stream, nullptr, fn);
}

extern "C" int64_t chromo_freq_edits_workspace_floats(const chromo_config_t* cfg, int32_t batch, int32_t variants,
                                                      int32_t flags) {
    if (validate_config(cfg) != CHROMO_OK) return CHROMO_EINVAL;
    if (batch < 1 || variants < 1) { set_error("batch and variants must be >= 1"); return CHROMO_EINVAL; }
    SubsetsWs d;
    CHROMO_TRY(subsets_ws(cfg, batch, variants, flags, &d, "chromo_freq_edits"));
    return freq_edits_total(d, variants);
}

extern "C" int chromo_freq_edits(const chromo_config_t* cfg, const float* params, const chromo_batch_t* in,
                                 const int32_t* var_gene, const float* var_freq, int32_t variants, float* logits,
                                 float* var_logits, float* workspace, int64_t workspace_floats, int32_t flags,
                                 void* stream) {
    const char* fn = "chromo_freq_edits";
    CHROMO_TRY(check_subsets_args(cfg, params, in, var_gene, var_freq, variants, logits, var_logits, workspace, flags, fn));
    SubsetsWs d;
    CHROMO_TRY(subsets_ws(cfg, in->batch, variants, flags, &d, fn));
    const int64_t total = freq_edits_total(d, variants);
    if (workspace_floats < total) {
        set_error("%s: workspace too small: need %lld floats, got %lld", fn, (long long)total, (long long)workspace_floats);
        return CHROMO_ENOMEM;
    }
    cudaStream_t st = (cudaStream_t)stream;
    uint32_t* drop = reinterpret_cast<uint32_t*>(workspace + d.total);
    if (cudaMemsetAsync(drop, 0, (size_t)variants * sizeof(uint32_t), st) != cudaSuccess) {
        set_error("%s: memset failed", fn);
        return CHROMO_ECUDA;
    }
    FreqSpliceArgs splice;
    splice.var_gene = var_gene; splice.var_freq = var_freq; splice.var_drop = drop;
    return subsets_run(cfg, params, in, var_gene, drop, variants, logits, var_logits, workspace, d, flags, st, &splice, fn);
}

// ---- histone-mark occlusion (occlusion.cu) ----
// Workspace, three phases on one front (the packed BF16 weights the gene pass writes):
//   [0, front)  the gene pass's layout; then the Pairwise replay's layout (make_ws_layout(..., pairwise = true)) with the
//               variant regions and their pad-mask rows behind it; then the Regulation replay's layout
//   after it    the gene X_in rows, the pseudo-genes' X_in (token 0 in, the occluded region's Pairwise row out), the
//               variants' freq and masks, the empty drop sets of subset_expand_kernel and the Regulation plan.
// The variant regions live only until the Pairwise replay has run, so they share room with the Regulation replay.
namespace {
struct OcclusionWs {
    WsLayout wb, wp, wv;
    int64_t x_v[CHROMO_MAX_RES], mask_v[CHROMO_MAX_RES];
    int64_t xin_b, xin_p, freq_v, imask_v, drop0, plan, total;
    bool plan_on;
};
int occlusion_ws(const chromo_config_t* c, int batch, int variants, int flags, OcclusionWs* d) {
    const int S = c->i_max + 1, NR = c->n_res, V = variants;
    int64_t row = std::max<int64_t>((int64_t)S * S, (int64_t)NR * c->d_emb * 2);
    for (int r = 0; r < NR; ++r) row = std::max<int64_t>(row, (int64_t)c->n_bins[r] * c->n_feats);
    if ((int64_t)batch * row > INT32_MAX || (int64_t)variants * row > INT32_MAX) {
        set_error("chromo_pcre_occlusion: batch and variants times max((i_max + 1)^2, 2 * n_res * d_emb, n_bins * n_feats) "
                  "must fit in int32");
        return CHROMO_EINVAL;
    }
    d->wb = make_ws_layout(c, batch, flags);
    d->wp = make_ws_layout(c, V, flags, false, true);
    d->wv = make_ws_layout(c, V, flags, true);
    int64_t cur = d->wp.total;
    auto take = [&](int64_t n) { int64_t o = cur; cur = align4(cur + n); return o; };
    for (int r = 0; r < NR; ++r) d->x_v[r] = take((int64_t)V * c->n_bins[r] * c->n_feats);
    for (int r = 0; r < NR; ++r) d->mask_v[r] = take(((int64_t)V * c->n_bins[r] + 3) / 4);
    cur = std::max({cur, d->wb.total, d->wv.total});
    d->xin_b = take((int64_t)NR * batch * S * c->d_emb);
    d->xin_p = take((int64_t)NR * V * 2 * c->d_emb);
    d->freq_v = take((int64_t)V * S * S);
    d->imask_v = take(((int64_t)V * S * S + 3) / 4 * NR);
    d->drop0 = take(V);
    d->plan_on = (flags & CHROMO_F_BF16) && d->wv.reg_fused;
    d->plan = d->plan_on ? take(reg_plan_floats(V, c->i_max)) : 0;
    d->total = cur;
    return CHROMO_OK;
}
}  // namespace

extern "C" int64_t chromo_pcre_occlusion_workspace_floats(const chromo_config_t* cfg, int32_t batch, int32_t variants,
                                                          int32_t flags) {
    if (validate_config(cfg) != CHROMO_OK) return CHROMO_EINVAL;
    if (batch < 1 || variants < 1) { set_error("batch and variants must be >= 1"); return CHROMO_EINVAL; }
    OcclusionWs d;
    CHROMO_TRY(occlusion_ws(cfg, batch, variants, flags, &d));
    return d.total;
}

extern "C" int chromo_pcre_occlusion(const chromo_config_t* cfg, const float* params, const chromo_batch_t* in,
                                     int32_t variants, const int32_t* var_gene, const int32_t* var_slot,
                                     const int32_t* var_bins, const uint32_t* var_marks, float* logits, float* var_logits,
                                     float* workspace, int64_t workspace_floats, int32_t flags, void* stream) {
    CHROMO_TRY(check_forward_args(cfg, params, in, logits, workspace));
    if (!var_gene || !var_slot || !var_bins || !var_marks || !var_logits) {
        set_error("chromo_pcre_occlusion: null variant descriptor or output");
        return CHROMO_EINVAL;
    }
    if (variants < 1) { set_error("chromo_pcre_occlusion: variants must be >= 1"); return CHROMO_EINVAL; }
    if (flags & ~(CHROMO_F_BF16 | CHROMO_F_PACKED | CHROMO_F_DENSE)) {
        set_error("chromo_pcre_occlusion: inference only (flags CHROMO_F_BF16, CHROMO_F_PACKED, CHROMO_F_DENSE)");
        return CHROMO_EINVAL;
    }
    OcclusionWs d;
    CHROMO_TRY(occlusion_ws(cfg, in->batch, variants, flags, &d));
    if (workspace_floats < d.total) {
        set_error("chromo_pcre_occlusion: workspace too small: need %lld floats, got %lld", (long long)d.total,
                  (long long)workspace_floats);
        return CHROMO_ENOMEM;
    }
    cudaStream_t st = (cudaStream_t)stream;
    float* ws = workspace;
    const int B = in->batch, I = cfg->i_max, S = I + 1, V = variants, NR = cfg->n_res, D = cfg->d_emb;
    // 1. the genes: the ordinary forward (it packs the BF16 weights unless CHROMO_F_PACKED), X_in set aside
    CHROMO_TRY(forward_impl(cfg, params, in, logits, ws, d.wb, flags, st));
    const size_t row_bytes = (size_t)B * S * D * sizeof(float);
    if (cudaMemcpy2DAsync(ws + d.xin_b, row_bytes, ws + d.wb.r_xin, (size_t)d.wb.res_stride * sizeof(float), row_bytes, NR,
                          cudaMemcpyDeviceToDevice, st) != cudaSuccess) {
        set_error("chromo_pcre_occlusion: X_in copy failed");
        return CHROMO_ECUDA;
    }
    OcclusionDesc desc;
    desc.B = B; desc.I = I; desc.n_res = NR; desc.F = cfg->n_feats; desc.V = V;
    desc.gene = var_gene; desc.slot = var_slot; desc.bins = var_bins; desc.marks = var_marks;
    for (int r = 0; r < CHROMO_MAX_RES; ++r) {
        desc.n[r] = r < NR ? cfg->n_bins[r] : 0;
        desc.imask[r] = r < NR ? in->imask[r] : nullptr;
    }
    // 2. the variant regions as V pseudo-genes of one slot
    chromo_batch_t pin;
    memset(&pin, 0, sizeof(pin));
    pin.batch = V; pin.freq = in->freq;
    const long long xin_p_z = (long long)V * 2 * D;
    {
        OcclusionExpandArgs a;
        a.d = desc;
        a.xin = ws + d.xin_b; a.xin_z = (long long)B * S * D;
        a.xin_p = ws + d.xin_p; a.xin_p_z = xin_p_z;
        for (int r = 0; r < NR; ++r) {
            a.x_pcre[r] = in->x_pcre[r];
            a.mask_pcre[r] = in->mask_pcre[r]; a.mask_stride[r] = in->mask_pcre_stride[r];
            a.mask_row_offset[r] = in->mask_pcre_row_offset[r];
            a.x_v[r] = ws + d.x_v[r];
            a.mask_v[r] = reinterpret_cast<uint8_t*>(ws + d.mask_v[r]);
            pin.x_pcre[r] = a.x_v[r];
            pin.mask_pcre[r] = a.mask_v[r]; pin.mask_pcre_stride[r] = cfg->n_bins[r]; pin.mask_pcre_row_offset[r] = 0;
            pin.pos_enc[r] = in->pos_enc[r];
            pin.imask[r] = in->imask[r];      // (not read: the replay builds no ragged plan and stops before the Regulation stage)
        }
        CHROMO_TRY(launch_occlusion_expand(a, st));
    }
    // 3. their Pairwise pass, on the paths of the gene pass, with the weights it packed
    const int vflags = (flags & ~CHROMO_F_DENSE) | ((flags & CHROMO_F_BF16) ? CHROMO_F_PACKED : 0);
    const PwReplay pw{B, I, ws + d.xin_p, xin_p_z};
    CHROMO_TRY(forward_impl(cfg, params, &pin, nullptr, ws, d.wp, vflags, st, nullptr, nullptr, &pw));
    // 4. the Regulation input: every variant's gene unchanged (empty drop sets), then the occluded region's row
    chromo_batch_t vin;
    memset(&vin, 0, sizeof(vin));
    vin.batch = V; vin.freq = ws + d.freq_v;
    if (cudaMemsetAsync(ws + d.drop0, 0, (size_t)V * sizeof(uint32_t), st) != cudaSuccess) {
        set_error("chromo_pcre_occlusion: memset failed");
        return CHROMO_ECUDA;
    }
    {
        SubsetExpandArgs a;
        a.B = B; a.I = I; a.n_res = NR; a.V = V;
        a.var_gene = var_gene; a.var_drop = reinterpret_cast<const uint32_t*>(ws + d.drop0);
        a.xin = ws + d.xin_b; a.xin_z = (long long)B * S * D;
        a.freq = in->freq;
        a.xin_v = ws + d.wv.r_xin; a.xin_v_z = d.wv.res_stride;
        a.freq_v = ws + d.freq_v;
        for (int r = 0; r < NR; ++r) {
            a.imask[r] = in->imask[r];
            a.imask_v[r] = reinterpret_cast<uint8_t*>(ws + d.imask_v) + (long long)r * V * S * S;
            vin.imask[r] = a.imask_v[r];
        }
        CHROMO_TRY(launch_subset_expand(a, st));
    }
    {
        OcclusionSpliceArgs a;
        a.d = desc;
        a.xin_p = ws + d.xin_p; a.xin_p_z = xin_p_z;
        a.xin_v = ws + d.wv.r_xin; a.xin_v_z = d.wv.res_stride;
        CHROMO_TRY(launch_occlusion_splice(a, st));
    }
    // 5. the Regulation replay and the head, logits in variant order
    RaggedPlan plan;
    if (d.plan_on) {
        RaggedArgs ra;
        memset(&ra, 0, sizeof(ra));
        ra.B = V; ra.I = I; ra.n_res = NR;
        for (int r = 0; r < NR; ++r) ra.imask[r] = vin.imask[r];
        CHROMO_TRY(build_reg_plan(ra, ws + d.plan, &plan, st));
    }
    const RegReplay replay{d.plan_on ? &plan : nullptr, B};
    CHROMO_TRY(forward_impl(cfg, params, &vin, var_logits, ws, d.wv, vflags, st, nullptr, &replay));
    // 6. NaN rows for invalid descriptors, the gene's row for dead slots
    OcclusionGuardArgs gd;
    gd.d = desc; gd.n_out = cfg->n_out;
    gd.logits = logits; gd.logits_v = var_logits;
    return launch_occlusion_guard(gd, st);
}

extern "C" int chromo_regulation_layer(const chromo_config_t* cfg, const float* params, int32_t layer, const float* x,
                                       float* y, int64_t xy_stride, const uint8_t* const* imask, const float* freq,
                                       int32_t batch, float* workspace, int64_t workspace_floats, int32_t flags,
                                       void* stream) {
    CHROMO_TRY(validate_config(cfg));
    if (!params || !x || !y || !imask || !freq || !workspace || batch < 1) { set_error("chromo_regulation_layer: bad argument"); return CHROMO_EINVAL; }
    if (layer >= cfg->reg_layers) { set_error("chromo_regulation_layer: no such layer"); return CHROMO_EINVAL; }
    if (flags & CHROMO_F_TRAINING) { set_error("chromo_regulation_layer: inference only"); return CHROMO_EINVAL; }
    WsLayout w = make_ws_layout(cfg, batch, flags);
    if (workspace_floats < w.total) { set_error("workspace too small"); return CHROMO_ENOMEM; }
    chromo_batch_t in;
    memset(&in, 0, sizeof(in));
    in.batch = batch; in.freq = freq;
    for (int r = 0; r < cfg->n_res; ++r) {
        if (!imask[r]) { set_error("chromo_regulation_layer: null interaction mask"); return CHROMO_EINVAL; }
        in.imask[r] = imask[r];
    }
    if (layer < 0 && !((flags & CHROMO_F_BF16) && w.reg_fused)) {
        set_error("chromo_regulation_layer: layer < 0 (all layers in one launch) needs the fused BF16 kernel");
        return CHROMO_EINVAL;
    }
    RegOnly only{layer, x, y, xy_stride};
    return forward_impl(cfg, params, &in, nullptr, workspace, w, flags | CHROMO_F_REGONLY, (cudaStream_t)stream, &only);
}

extern "C" int chromo_linear(const float* x, const float* w, const float* bias, float* y, int32_t m, int32_t n,
                             int32_t k, int32_t relu, int32_t batches, int64_t x_stride, int64_t w_stride,
                             int64_t bias_stride, int64_t y_stride, int32_t flags, void* stream) {
    if (!x || !w || !y || m < 1 || n < 1 || k < 1 || batches < 1) { set_error("chromo_linear: bad argument"); return CHROMO_EINVAL; }
    GemmArgs g = gemm_args();
    g.A = x; g.lda = k; g.sA1 = x_stride;
    g.B = w; g.ldb = k; g.sB1 = w_stride;
    g.C = y; g.ldc = n; g.sC1 = y_stride;
    g.M = m; g.N = n; g.K = k;
    g.bias = bias; g.sBias1 = bias_stride;
    g.epi = relu ? EPI_BIAS_RELU : (bias ? EPI_BIAS : EPI_PLAIN);
    if (flags & CHROMO_F_BF16) {
        if (!umma_supported(g)) { set_error("chromo_linear: shape not supported by the BF16 tensor path"); return CHROMO_EINVAL; }
        return umma_launch(g, reinterpret_cast<const __nv_bfloat16*>(w), batches, (cudaStream_t)stream);
    }
    return gemm_launch(g, true, true, batches, (cudaStream_t)stream);
}

extern "C" int chromo_single_query_attention(int32_t regions, int32_t n, const float* qk, const float* x,
                                             const uint8_t* mask, const float* w_in, const float* pos_enc, float scale,
                                             float* cbar, float* workspace, int64_t workspace_floats, void* stream) {
    if (!qk || !x || !mask || !w_in || !pos_enc || !cbar || !workspace || regions < 1 || n < 4) {
        set_error("chromo_single_query_attention: bad argument");
        return CHROMO_EINVAL;
    }
    const int ns = n <= 32 ? 32 : (n + 15) / 16 * 16;
    const int64_t tiles = ((int64_t)regions * 2 + 127) / 128;
    if (workspace_floats < (int64_t)ns * 64 + 1024 + tiles * 8192) { set_error("chromo_single_query_attention: workspace too small"); return CHROMO_EINVAL; }
    cudaStream_t st = (cudaStream_t)stream;
    __nv_bfloat16* pk = reinterpret_cast<__nv_bfloat16*>(workspace);
    __nv_bfloat16* wpk = reinterpret_cast<__nv_bfloat16*>(workspace + (int64_t)ns * 64);
    __nv_bfloat16* qkt = reinterpret_cast<__nv_bfloat16*>(workspace + (int64_t)ns * 64 + 1024);
    SqaFusedArgs f;
    f.n_res = 1; f.regions = regions;
    f.n[0] = n; f.ns[0] = ns; f.order[0] = 0;
    f.x[0] = x; f.mask[0] = mask; f.mask_stride[0] = n; f.mask_row_offset[0] = 0;
    f.pe_pk[0] = pk;
    f.qk_tiles = qkt; f.qk_tz = 0; f.cbar = cbar; f.cbar_z = 0;
    f.w_in = w_in; f.w_in_z = 0; f.w_in_pk = wpk; f.w_in_pk_z = 0;
    f.scale = scale;
    if (umma_tile_n(ns) == 0 || (reinterpret_cast<uintptr_t>(qk) & 15) || !sqa_fused_supported(f, 2, 7, 128)) {
        set_error("chromo_single_query_attention: shape / alignment not supported by the fused kernel");
        return CHROMO_EINVAL;
    }
    CHROMO_TRY(pack_weights(pos_enc, pk, ns, 128, umma_tile_n(ns), 0, 1, false, 128, st, n));
    CHROMO_TRY(sqa_pack_w_in(w_in, 0, wpk, 0, 1, st));
    CHROMO_TRY(sqa_pack_qk(qk, 0, qkt, 0, regions * 2, 1, st));
    return launch_sqa_fused(f, st);
}

extern "C" int chromo_pack_linear_weight(const float* w, uint16_t* packed, int32_t n, int32_t k, int32_t batches,
                                         int64_t w_stride, void* stream) {
    if (!w || !packed || n < 1 || k < 1 || batches < 1) { set_error("chromo_pack_linear_weight: bad argument"); return CHROMO_EINVAL; }
    const int nt = umma_tile_n(n);
    if (nt == 0 || k % 16 != 0) { set_error("chromo_pack_linear_weight: n must be a multiple of 16 with a tile <= 256, k a multiple of 16"); return CHROMO_EINVAL; }
    return pack_weights(w, reinterpret_cast<__nv_bfloat16*>(packed), n, k, nt, w_stride, batches, false, k, (cudaStream_t)stream);
}
