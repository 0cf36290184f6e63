// Hand-written backward of the pruned forward in forward.cu (autograd of
// net.py:332-380 as exercised by train.py:195).  Gradients are ACCUMULATED into
// the flat gradient buffer, which shares the parameter layout.
//
// One [rows,128] gradient buffer per stage flows backwards in place through the
// post-LN residual sub-layers:
//     y = LN(x + f(x)):   g <- LN'(g);  (weight grads of f);  g <- g + f'(g)
// Every dense contraction reuses the batched GEMM (data grads: NN form, weight
// grads: A^T form with split-K atomics).
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "gemm_dispatch.cuh"
#include "kernels.cuh"

namespace chromo {

// ------------------------------------------------------------------ kernels --

// LayerNorm backward (dy -> dz, `gout` may alias `gin`); one warp per row of 128.
struct LnBwdArgs {
    int M;
    const float* pre; long long pre_z;
    const float* gin; float* g; long long g_z;
    const float* gamma; float* dgamma; float* dbeta; long long p_z;
};
__global__ void __launch_bounds__(256) ln_bwd_kernel(LnBwdArgs a) {
    CHROMO_PDL_ENTER();
    __shared__ float s_dg[8][128];
    __shared__ float s_db[8][128];
    const int z = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float* pre = a.pre + z * a.pre_z;
    const float* gin = a.gin + z * a.g_z;
    float* g = a.g + z * a.g_z;
    const float4 ga = *reinterpret_cast<const float4*>(a.gamma + z * a.p_z + lane * 4);
    float dg[4] = {0, 0, 0, 0}, db[4] = {0, 0, 0, 0};
    for (int m = blockIdx.x * 8 + warp; m < a.M; m += gridDim.x * 8) {
        const float4 zv = *reinterpret_cast<const float4*>(pre + (long long)m * 128 + lane * 4);
        float4 dy = *reinterpret_cast<const float4*>(gin + (long long)m * 128 + lane * 4);
        float s = zv.x + zv.y + zv.z + zv.w;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        const float mean = s * (1.f / 128.f);
        const float c0 = zv.x - mean, c1 = zv.y - mean, c2 = zv.z - mean, c3 = zv.w - mean;
        float q = c0 * c0 + c1 * c1 + c2 * c2 + c3 * c3;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
        const float rstd = rsqrtf(q * (1.f / 128.f) + 1e-5f);
        const float x0 = c0 * rstd, x1 = c1 * rstd, x2 = c2 * rstd, x3 = c3 * rstd;
        dg[0] += dy.x * x0; dg[1] += dy.y * x1; dg[2] += dy.z * x2; dg[3] += dy.w * x3;
        db[0] += dy.x; db[1] += dy.y; db[2] += dy.z; db[3] += dy.w;
        const float g0 = dy.x * ga.x, g1 = dy.y * ga.y, g2 = dy.z * ga.z, g3 = dy.w * ga.w;
        float sg = g0 + g1 + g2 + g3;
        float sgx = g0 * x0 + g1 * x1 + g2 * x2 + g3 * x3;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            sg += __shfl_xor_sync(0xffffffffu, sg, o);
            sgx += __shfl_xor_sync(0xffffffffu, sgx, o);
        }
        const float mg = sg * (1.f / 128.f), mgx = sgx * (1.f / 128.f);
        dy.x = rstd * (g0 - mg - x0 * mgx);
        dy.y = rstd * (g1 - mg - x1 * mgx);
        dy.z = rstd * (g2 - mg - x2 * mgx);
        dy.w = rstd * (g3 - mg - x3 * mgx);
        *reinterpret_cast<float4*>(g + (long long)m * 128 + lane * 4) = dy;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) { s_dg[warp][lane * 4 + k] = dg[k]; s_db[warp][lane * 4 + k] = db[k]; }
    __syncthreads();
    if (threadIdx.x < 128 && a.dgamma) {     // (no dgamma: data gradient only, chromo_backward_inputs without grads)
        float x = 0.f, y = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) { x += s_dg[w][threadIdx.x]; y += s_db[w][threadIdx.x]; }
        atomicAdd(a.dgamma + z * a.p_z + threadIdx.x, x);
        atomicAdd(a.dbeta + z * a.p_z + threadIdx.x, y);
    }
}

// out[n] += sum_m dY[m, n]      (bias gradients)
__global__ void __launch_bounds__(256) colsum_kernel(const float* dY, int M, int N, int ld, long long dy_z,
                                                     float* out, long long out_z, int rows_per_block) {
    const int z = blockIdx.z;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const int m0 = blockIdx.y * rows_per_block, m1 = min(M, m0 + rows_per_block);
    const float* p = dY + z * dy_z + n;
    float s = 0.f;
    for (int m = m0; m < m1; ++m) s += p[(long long)m * ld];
    atomicAdd(out + z * out_z + n, s);
}

// dst[m, :] (=|+=) src[(m / div) * mul + m % div + add, :]   (128-wide rows)
__global__ void gather_rows_kernel(float* dst, long long dst_z, const float* src, long long src_z, int M, int div,
                                   int mul, int add) {
    CHROMO_PDL_ENTER();
    const int z = blockIdx.y;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // float4 index
    if (i >= (long long)M * 32) return;
    const int m = (int)(i / 32), c = (int)(i % 32);
    const long long srow = (long long)(m / div) * mul + (m % div) + add;
    reinterpret_cast<float4*>(dst + z * dst_z)[i] = reinterpret_cast<const float4*>(src + z * src_z)[srow * 32 + c];
}

// dst[b, :] = sum_i src[b * I + i, :]
__global__ void slot_sum_kernel(float* dst, long long dst_z, const float* src, long long src_z, int B, int I) {
    CHROMO_PDL_ENTER();
    const int z = blockIdx.y;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)B * 32) return;
    const int b = (int)(i / 32), c = (int)(i % 32);
    const float4* s = reinterpret_cast<const float4*>(src + z * src_z) + (long long)b * I * 32 + c;
    float4 acc = make_float4(0, 0, 0, 0);
    for (int k = 0; k < I; ++k) {
        const float4 v = s[(long long)k * 32];
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    reinterpret_cast<float4*>(dst + z * dst_z)[i] = acc;
}

// Head fan-out: g_reg[b*S + 0, :] = dz[b, r*D:(r+1)*D], other rows 0          (net.py:377)
__global__ void head_scatter_kernel(float* g, long long g_z, const float* dz, int B, int S, int D, int n_res) {
    CHROMO_PDL_ENTER();
    const int z = blockIdx.y;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)B * S * D) return;
    const int d = (int)(i % D);
    const long long row = i / D;
    const int b = (int)(row / S), s = (int)(row % S);
    g[z * g_z + i] = s == 0 ? dz[(long long)b * n_res * D + z * D + d] : 0.f;
}
// g[b*S + 0, :] += dz[b, r*D:(r+1)*D]                                        (residual, net.py:378)
__global__ void head_residual_kernel(float* g, long long g_z, const float* dz, int B, int S, int D, int n_res) {
    CHROMO_PDL_ENTER();
    const int z = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * D) return;
    const int b = i / D, d = i % D;
    g[z * g_z + (long long)b * S * D + d] += dz[(long long)b * n_res * D + z * D + d];
}

// dfreq[b, i, j] = sum_r sum_k part_r[(b*K + k), i, j]: the Regulation backward's partials of d interaction_freq (K = 1
// from the gene kernel, K = H per-head slices from the warp kernel), summed in a fixed order; every element is written.
__global__ void freq_grad_sum_kernel(float* dfreq, const float* part, long long part_z, int NR, int K, int B, int SS) {
    CHROMO_PDL_ENTER();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)B * SS) return;
    const long long b = i / SS, e = i % SS;
    float t = 0.f;
    for (int r = 0; r < NR; ++r)
        for (int k = 0; k < K; ++k) t += part[r * part_z + (b * K + k) * SS + e];
    dfreq[i] = t;
}

// Backward of reg_attention_kernel.  One warp per (gene, head), lane = channel.
// FREQ: also gamma_f[h] dS[i, j] (=|+=) into this head's own [S,S] slice of the dfreq partial ([B,H,S,S] per resolution;
// freq_grad_sum_kernel sums the heads), lane j storing column j - no atomics.
template <int SMAX, bool FREQ>
__global__ void __launch_bounds__(256) reg_attention_bwd_kernel(RegAttnBwdArgs a) {
    CHROMO_PDL_ENTER();
    const int warp_in_block = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long gw = (long long)blockIdx.x * (blockDim.x >> 5) + warp_in_block;
    const int z = blockIdx.y;
    const int S = a.S, H = a.H, dm = 32 * H;
    if (gw >= (long long)a.B * H) return;
    const int b = (int)(gw / H), h = (int)(gw % H);
    const float* proj = a.proj + z * a.proj_z + (long long)b * S * 4 * dm + h * 32 + lane;
    float* dproj = a.dproj + z * a.dproj_z + (long long)b * S * 4 * dm + h * 32 + lane;
    const float* dout = a.dout + z * a.dout_z + (long long)b * S * dm + h * 32 + lane;
    const float* prob = a.prob + z * a.prob_z + ((long long)b * H + h) * S * S;
    const float* freq = a.freq + (long long)b * S * S;
    const uint8_t* mask = a.imask[z] + (long long)b * S * S;
    const float scale = 0.17677669529663687f;
    float q[SMAX], k[SMAX], v[SMAX], dk[SMAX], dv[SMAX];
#pragma unroll
    for (int i = 0; i < SMAX; ++i) {
        if (i < S) {
            const float* row = proj + (long long)i * 4 * dm;
            q[i] = row[0]; k[i] = row[dm]; v[i] = row[2 * dm];
        } else { q[i] = k[i] = v[i] = 0.f; }
        dk[i] = 0.f; dv[i] = 0.f;
    }
    float dgam = 0.f;
    const float gam = FREQ ? a.gamma_f[z * a.dgamma_z + h] : 0.f;
    float* dfq = FREQ ? a.dfreq + z * a.dfreq_z + gw * S * S : nullptr;
#pragma unroll
    for (int i = 0; i < SMAX; ++i) {
        if (i >= S) break;
        float p[SMAX], dp[SMAX];
        float av = 0.f;
#pragma unroll
        for (int j = 0; j < SMAX; ++j) {
            p[j] = j < S ? prob[i * S + j] : 0.f;
            av = fmaf(p[j], v[j], av);
        }
        const float gt = proj[(long long)i * 4 * dm + 3 * dm];
        const float sg = 1.f / (1.f + expf(-gt));
        const float d_o = dout[(long long)i * dm];
        const float da = d_o * sg;
        dproj[(long long)i * 4 * dm + 3 * dm] = d_o * av * sg * (1.f - sg);
        float dot = 0.f;
#pragma unroll
        for (int j = 0; j < SMAX; ++j) {
            if (j >= S) { dp[j] = 0.f; continue; }
            float t = da * v[j];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
            dp[j] = t;
            dot = fmaf(p[j], t, dot);
            dv[j] = fmaf(p[j], da, dv[j]);
        }
        float dq = 0.f;
#pragma unroll
        for (int j = 0; j < SMAX; ++j) {
            if (j >= S) continue;
            const float ds = mask[i * S + j] ? 0.f : p[j] * (dp[j] - dot);
            dgam = fmaf(ds, freq[i * S + j], dgam);
            if (FREQ && lane == j) dfq[i * S + j] = a.dfreq_add ? fmaf(gam, ds, dfq[i * S + j]) : gam * ds;
            dq = fmaf(ds, k[j], dq);
            dk[j] = fmaf(ds, q[i], dk[j]);
        }
        dproj[(long long)i * 4 * dm] = dq * scale;
    }
#pragma unroll
    for (int j = 0; j < SMAX; ++j) {
        if (j < S) {
            dproj[(long long)j * 4 * dm + dm] = dk[j] * scale;
            dproj[(long long)j * 4 * dm + 2 * dm] = dv[j];
        }
    }
    if (lane == 0 && a.dgamma_f) atomicAdd(a.dgamma_f + z * a.dgamma_z + h, dgam);
}

// The same backward with one CTA per gene (counterpart of reg_attention_gene_kernel): the gene's rows of q | k | v | gate
// staged once in shared memory; four lanes (eight channels each) per (head, query) for dgate, dq and the score
// gradients - two shuffles per key instead of a 32-lane reduction - then, after a barrier, per (head, key) for dk and dv
// from the staged dS / P / dA.  (The kernel above spends its time in 81 warp-wide reductions per (gene, head).)
// FREQ: also sum_h gamma_f[h] dS[h, i, j] (=|+=) into the gene's [S,S] of the dfreq partial ([B,S,S] per resolution),
// one thread per (i, j) (the block has H*S*4 >= S*S threads), the heads summed in a fixed order.
constexpr int RAB_PAD = 4;
template <int SMAX, bool FREQ>
__global__ void __launch_bounds__(SMAX * 32) reg_attention_gene_bwd_kernel(RegAttnBwdArgs a) {
    CHROMO_PDL_ENTER();
    extern __shared__ __align__(16) float rab_sm[];
    const int S = a.S, H = a.H, dm = 32 * H, ld = 4 * dm + RAB_PAD;
    float* sm_da = rab_sm + S * ld;              // [H*S][32]   dA = dO * sigmoid(gate)
    float* sm_ds = sm_da + S * dm;               // [H*S][S]    gradient wrt the pre-softmax score (before the 1/sqrt(32))
    float* sm_p = sm_ds + H * S * S;             // [H*S][S]    probabilities
    float* sm_gam = sm_p + H * S * S;            // [H*S]       per-query terms of d gamma_f
    const int b = blockIdx.x, z = blockIdx.y, tid = threadIdx.x;
    const float* proj = a.proj + z * a.proj_z + (long long)b * S * 4 * dm;
    for (int v = tid; v < S * dm; v += blockDim.x) {
        const int r = v / dm, c = v % dm;
        *reinterpret_cast<float4*>(rab_sm + r * ld + 4 * c) = __ldg(reinterpret_cast<const float4*>(proj + (long long)r * 4 * dm) + c);
    }
    __syncthreads();
    const int item = tid >> 2, sub = tid & 3;    // blockDim.x == H * S * 4 exactly (H == 8)
    const int h = item / S, i = item % S;        // phase 1: (head, query)
    const int co = h * 32 + sub * 8;
    const float scale = 0.17677669529663687f;
    float* dproj = a.dproj + z * a.dproj_z + (long long)b * S * 4 * dm;
    {
        const float* prob = a.prob + z * a.prob_z + (((long long)b * H + h) * S + i) * S;
        const float* freq = a.freq + ((long long)b * S + i) * S;
        const uint8_t* mask = a.imask[z] + ((long long)b * S + i) * S;
        const float* dout = a.dout + z * a.dout_z + ((long long)b * S + i) * dm + co;
        const float4 d0 = __ldg(reinterpret_cast<const float4*>(dout)), d1 = __ldg(reinterpret_cast<const float4*>(dout) + 1);
        const float d_o[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
        float p[SMAX], dp[SMAX];
        float av[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int j = 0; j < SMAX; ++j) {
            p[j] = j < S ? __ldg(prob + j) : 0.f;
            if (j < S) {
                const float* vj = rab_sm + j * ld + 2 * dm + co;
#pragma unroll
                for (int e = 0; e < 8; ++e) av[e] = fmaf(p[j], vj[e], av[e]);
            }
        }
        float da[8], dg[8];
        {
            const float* gt = rab_sm + i * ld + 3 * dm + co;
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const float sg = 1.f / (1.f + expf(-gt[e]));
                da[e] = d_o[e] * sg;
                dg[e] = d_o[e] * av[e] * sg * (1.f - sg);
            }
        }
        float* drow = dproj + (long long)i * 4 * dm;
        *reinterpret_cast<float4*>(drow + 3 * dm + co) = make_float4(dg[0], dg[1], dg[2], dg[3]);
        *reinterpret_cast<float4*>(drow + 3 * dm + co + 4) = make_float4(dg[4], dg[5], dg[6], dg[7]);
        *reinterpret_cast<float4*>(sm_da + item * 32 + sub * 8) = make_float4(da[0], da[1], da[2], da[3]);
        *reinterpret_cast<float4*>(sm_da + item * 32 + sub * 8 + 4) = make_float4(da[4], da[5], da[6], da[7]);
#pragma unroll
        for (int j = 0; j < SMAX; ++j) {
            dp[j] = 0.f;
            if (j < S) {
                const float* vj = rab_sm + j * ld + 2 * dm + co;
                float t = 0.f;
#pragma unroll
                for (int e = 0; e < 8; ++e) t = fmaf(da[e], vj[e], t);
                dp[j] = t;
            }
        }
        float dot = 0.f;
#pragma unroll
        for (int j = 0; j < SMAX; ++j) {
            dp[j] += __shfl_xor_sync(0xffffffffu, dp[j], 1);
            dp[j] += __shfl_xor_sync(0xffffffffu, dp[j], 2);
            dot = fmaf(p[j], dp[j], dot);
        }
        float dq[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        float dgam = 0.f;
#pragma unroll
        for (int j = 0; j < SMAX; ++j) {
            if (j < S) {
                const float ds = mask[j] ? 0.f : p[j] * (dp[j] - dot);
                dgam = fmaf(ds, freq[j], dgam);
                const float* kj = rab_sm + j * ld + dm + co;
#pragma unroll
                for (int e = 0; e < 8; ++e) dq[e] = fmaf(ds, kj[e], dq[e]);
                if (sub == (j & 3)) { sm_ds[item * S + j] = ds; sm_p[item * S + j] = p[j]; }
            }
        }
        *reinterpret_cast<float4*>(drow + co) = make_float4(dq[0] * scale, dq[1] * scale, dq[2] * scale, dq[3] * scale);
        *reinterpret_cast<float4*>(drow + co + 4) = make_float4(dq[4] * scale, dq[5] * scale, dq[6] * scale, dq[7] * scale);
        if (sub == 0) sm_gam[item] = dgam;
    }
    __syncthreads();
    if (tid < H && a.dgamma_f) {      // one atomic per (gene, head), summed in a fixed order
        float t = 0.f;
        for (int q = 0; q < S; ++q) t += sm_gam[tid * S + q];
        atomicAdd(a.dgamma_f + z * a.dgamma_z + tid, t);
    }
    if (FREQ && tid < S * S) {
        const float* gam = a.gamma_f + z * a.dgamma_z;
        float t = 0.f;
        for (int hh = 0; hh < H; ++hh) t = fmaf(gam[hh], sm_ds[hh * S * S + tid], t);
        float* d = a.dfreq + z * a.dfreq_z + (long long)b * S * S + tid;
        *d = a.dfreq_add ? *d + t : t;
    }
    {   // phase 2: (head, key j = i): dk[j] = scale sum_i dS[i, j] q[i],  dv[j] = sum_i P[i, j] dA[i]
        const int j = i;
        float dk[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, dv[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int q = 0; q < S; ++q) {
            const float ds = sm_ds[(h * S + q) * S + j], pp = sm_p[(h * S + q) * S + j];
            const float* qq = rab_sm + q * ld + co;
            const float* dd = sm_da + (h * S + q) * 32 + sub * 8;
#pragma unroll
            for (int e = 0; e < 8; ++e) { dk[e] = fmaf(ds, qq[e], dk[e]); dv[e] = fmaf(pp, dd[e], dv[e]); }
        }
        float* drow = dproj + (long long)j * 4 * dm;
        *reinterpret_cast<float4*>(drow + dm + co) = make_float4(dk[0] * scale, dk[1] * scale, dk[2] * scale, dk[3] * scale);
        *reinterpret_cast<float4*>(drow + dm + co + 4) = make_float4(dk[4] * scale, dk[5] * scale, dk[6] * scale, dk[7] * scale);
        *reinterpret_cast<float4*>(drow + 2 * dm + co) = make_float4(dv[0], dv[1], dv[2], dv[3]);
        *reinterpret_cast<float4*>(drow + 2 * dm + co + 4) = make_float4(dv[4], dv[5], dv[6], dv[7]);
    }
}

// Backward of attn_rows_kernel; one warp per (region, head).
//   in : dS[j] = dCbar . PE_j (from a GEMM), P, dCbar, x, mask
//   out: dS[j] = gradient wrt the pre-scale score, dU8 = sum_j dS_j x_j,
//        dQK_init = W_in dU  (the PE part is added by a GEMM)
__global__ void __launch_bounds__(256) attn_rows_bwd_kernel(AttnRowsBwdArgs a) {
    CHROMO_PDL_ENTER();
    __shared__ float w_s[128 * 8];
    for (int i = threadIdx.x; i < a.D * a.F; i += blockDim.x) w_s[i] = a.w_in[i];
    __syncthreads();
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= a.rows) return;
    const int region = warp / a.H;
    const int n = a.n, F = a.F, D = a.D;
    const float* P = a.P + (long long)warp * n;
    float* dS = a.dS + (long long)warp * n;
    const float* dcb = a.dcbar + (long long)warp * D;
    const float* x = a.x + (long long)region * n * F;
    const uint8_t* mk = a.mask + (long long)region * a.mask_stride + a.mask_row_offset;
    float dxb[8];
#pragma unroll
    for (int f = 0; f < 8; ++f) dxb[f] = 0.f;
    for (int d = lane; d < D; d += 32) {
        const float c = dcb[d];
        const float* w = w_s + d * F;
#pragma unroll
        for (int f = 0; f < 8; ++f)
            if (f < F) dxb[f] = fmaf(w[f], c, dxb[f]);
    }
#pragma unroll
    for (int f = 0; f < 8; ++f)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) dxb[f] += __shfl_xor_sync(0xffffffffu, dxb[f], o);
    float dot = 0.f;
    for (int j = lane; j < n; j += 32) {
        const float* xj = x + (long long)j * F;
        float dp = dS[j];
#pragma unroll
        for (int f = 0; f < 8; ++f)
            if (f < F) dp = fmaf(dxb[f], xj[f], dp);
        dS[j] = dp;
        dot = fmaf(P[j], dp, dot);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
    float du[8];
#pragma unroll
    for (int f = 0; f < 8; ++f) du[f] = 0.f;
    for (int j = lane; j < n; j += 32) {
        const float ds = mk[j] ? 0.f : P[j] * (dS[j] - dot) * a.scale;
        dS[j] = ds;
        const float* xj = x + (long long)j * F;
#pragma unroll
        for (int f = 0; f < 8; ++f)
            if (f < F) du[f] = fmaf(ds, xj[f], du[f]);
    }
#pragma unroll
    for (int f = 0; f < 8; ++f)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) du[f] += __shfl_xor_sync(0xffffffffu, du[f], o);
    if (lane < 8) a.dU8[(long long)warp * 8 + lane] = lane < F ? du[lane] : 0.f;
    float* dqk = a.dqk + (long long)warp * D;
    for (int d = lane; d < D; d += 32) {
        const float* w = w_s + d * F;
        float s = 0.f;
#pragma unroll
        for (int f = 0; f < 8; ++f)
            if (f < F) s = fmaf(w[f], du[f], s);
        dqk[d] = s;
    }
}

// Gradient with respect to the raw features of single-query attention regions (chromo_backward_inputs).  Keys and values
// are h_j = W_in x_j + PE_j, so with dS as attn_rows_bwd_kernel leaves it (the gradient of the pre-scale score, zero on
// masked bins) and dCbar / qk of the region's H rows:
//     dx[j, :] (=|+=) sum_h P[h, j] a_h + dS[h, j] u_h,   a_h = W_in^T dCbar_h,  u_h = W_in^T qk_h
// plus W_in^T dhc at the centre bin n/2 when `dhc` is set (the promoter's query / residual input).  One warp per region;
// every element of the region is written, so the output needs no memset and no atomics.
struct InputGradArgs {
    int regions, H, n, F, D;
    const float* P;       // [regions * H, n] probabilities
    const float* dS;      // [regions * H, n]
    const float* dcbar;   // [regions * H, D]
    const float* qk;      // [regions * H, D]
    const float* w_in;    // [D, F]
    const float* dhc;     // [regions, D] or nullptr
    float* dx;            // [regions, n, F]
    int accumulate;
};
__global__ void __launch_bounds__(256) input_grad_rows_kernel(InputGradArgs a) {
    CHROMO_PDL_ENTER();
    __shared__ float w_s[128 * 8];
    __shared__ float au_s[8][2 * 8 * 8 + 8];      // per warp: a[h][f], u[h][f], centre term [f]
    for (int i = threadIdx.x; i < a.D * a.F; i += blockDim.x) w_s[i] = a.w_in[i];
    __syncthreads();
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long region = (long long)blockIdx.x * 8 + wib;
    if (region >= a.regions) return;
    const int n = a.n, F = a.F, D = a.D, H = a.H;
    float* au = au_s[wib];
    // W_in^T v for the 2H + 1 vectors v of the region (lanes over d, then a butterfly per feature)
    for (int v = 0; v < 2 * H + 1; ++v) {
        const float* src = v < H ? a.dcbar + (region * H + v) * D
                         : v < 2 * H ? a.qk + (region * H + v - H) * D
                         : a.dhc ? a.dhc + region * D : nullptr;
        float s[8];
#pragma unroll
        for (int f = 0; f < 8; ++f) s[f] = 0.f;
        if (src) {
            for (int d = lane; d < D; d += 32) {
                const float c = src[d];
                const float* w = w_s + d * F;
#pragma unroll
                for (int f = 0; f < 8; ++f)
                    if (f < F) s[f] = fmaf(w[f], c, s[f]);
            }
#pragma unroll
            for (int f = 0; f < 8; ++f)
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) s[f] += __shfl_xor_sync(0xffffffffu, s[f], o);
        }
        const int base = v < H ? v * 8 : v < 2 * H ? 64 + (v - H) * 8 : 128;
        if (lane == 0) {
#pragma unroll
            for (int f = 0; f < 8; ++f) au[base + f] = s[f];
        }
    }
    __syncwarp();
    const float* P = a.P + region * H * n;
    const float* dS = a.dS + region * H * n;
    float* dx = a.dx + region * n * F;
    const int c = n / 2;
    for (int e = lane; e < n * F; e += 32) {       // consecutive lanes, consecutive elements
        const int j = e / F, f = e - j * F;
        float g = 0.f;
        for (int h = 0; h < H; ++h) {
            g = fmaf(P[h * n + j], au[h * 8 + f], g);
            g = fmaf(dS[h * n + j], au[64 + h * 8 + f], g);
        }
        if (j == c) g += au[128 + f];
        if (a.accumulate) g += dx[e];
        dx[e] = g;
    }
}

// ------------------------------------------------------------ host helpers ---
namespace {

// Every gradient tensor of the pass has a buffer of its own (nothing is updated in place), so the weight / bias
// gradients can be taken from them at any later point: on the tensor path they are queued (`q`) and run as ONE
// persistent launch at the end of the pass; the strict FP32 path launches them where they arise.
struct Ctx {
    cudaStream_t st;
    int NR;
    bool tc = false;            // CHROMO_F_BF16: contractions on the tensor pipe (train_gemm.cu)
    WgradQueue* q = nullptr;    // tc: the deferred weight / bias gradients
    bool wgrad = true;          // false: data gradients only (chromo_backward_inputs with grads == NULL)
};

// Split-K factor: the training batch is small (bsz 64 => a few hundred rows), so most gradient
// GEMMs would otherwise run on a handful of CTAs; split the reduction until ~2 waves of CTAs exist.
inline int ksplit_for(int K, int M = 4096, int N = 4096, int nz = 1) {
    const long long ctas = (long long)((M + 63) / 64) * ((N + 63) / 64) * nz;
    long long want = (2 * 148 + ctas - 1) / ctas;
    const int by_k = (K + 31) / 32;
    if (want > by_k) want = by_k;
    if (want > 32) want = 32;
    return want < 1 ? 1 : (int)want;
}

// dX = [res +] mask( dY W )     dY [M,N] (ld ldy), W [N,K] row-major, dX [M,K] (ld lddx); res [M,K] (ld lddx, same batch
// stride as dX) is the gradient arriving over the residual connection, mask [M,K] (ld K) the ReLU output of the forward
struct DataEpi { const float* res = nullptr; const float* mask = nullptr; long long mask_z = 0; };
int bwd_data(const Ctx& c, const float* dY, int ldy, long long dy_z, const float* W, long long w_z, float* dX,
             int lddx, long long dx_z, int M, int N, int K, const DataEpi& e, int nz) {
    if (c.tc && K % 16 == 0) {      // A = dY rows (K-major), B = W rows [n, k] (MN-major: k contiguous)
        TcGemm t = tc_gemm_args();
        t.A = dY; t.lda = ldy; t.a_z = dy_z;
        t.B = W; t.ldb = K; t.b_z = w_z; t.b_t = 1;
        t.C = dX; t.ldc = lddx; t.c_z = dx_z; t.M = M; t.N = K; t.Kc = N;
        if (e.res) { t.epi |= TC_RES; t.res = e.res; t.ldres = lddx; t.res_z = dx_z; }
        if (e.mask) { t.epi |= TC_MASK; t.mask = e.mask; t.ldmask = K; t.mask_z = e.mask_z; }
        if (tc_gemm_supported(t)) return tc_gemm_launch(t, nz, c.st);
    }
    GemmArgs g = gemm_args();
    g.A = dY; g.lda = ldy; g.sA1 = dy_z;
    g.B = W; g.ldb = K; g.sB1 = w_z;
    g.C = dX; g.ldc = lddx; g.sC1 = dx_z;
    g.M = M; g.N = K; g.K = N;
    if (e.res && !e.mask && lddx == K) {
        // strict FP32 path: dX <- res (one strided copy), then dX += dY W with the contraction split over CTAs (atomics):
        // the batch of a training step is a few hundred rows, a handful of CTAs otherwise
        if (cudaMemcpy2DAsync(dX, (size_t)(nz > 1 ? dx_z : (long long)M * K) * sizeof(float), e.res,
                              (size_t)(nz > 1 ? dx_z : (long long)M * K) * sizeof(float), (size_t)M * K * sizeof(float), nz,
                              cudaMemcpyDeviceToDevice, c.st) != cudaSuccess) {
            set_error("bwd_data: residual copy failed");
            return CHROMO_ECUDA;
        }
        g.accumulate = 1;
        g.ksplit = ksplit_for(N, M, K, nz);
        return gemm_launch(g, true, false, nz, c.st);
    }
    if (e.res) { g.res_plain = 1; g.res = e.res; g.ldres = lddx; g.sRes1 = dx_z; }
    if (e.mask) { g.mask = e.mask; g.ldmask = K; g.sMask1 = e.mask_z; }
    return gemm_launch(g, true, false, nz, c.st);
}

// dW += dY^T X          dY [M,N], X [M/x_div rows broadcast, K] (ld ldx), dW [N,K] row-major
int bwd_weight(const Ctx& c, const float* dY, int ldy, long long dy_z, const float* X, int ldx, int x_div,
               long long x_z, float* dW, int lddw, long long dw_z, int M, int N, int K, int nz) {
    if (!c.wgrad) return CHROMO_OK;
    if (c.q) {      // both operands MN-major (rows = tokens = the contraction); runs at the end of the pass
        c.q->add_weight(dY, ldy, dy_z, X, ldx, x_div, x_z, dW, lddw, dw_z, M, N, K, nz);
        return CHROMO_OK;
    }
    GemmArgs g = gemm_args();
    g.A = dY; g.lda = ldy; g.sA1 = dy_z;
    g.B = X; g.ldb = ldx; g.b_div = x_div; g.sB1 = x_z;
    g.C = dW; g.ldc = lddw; g.sC1 = dw_z;
    g.M = N; g.N = K; g.K = M;
    g.ksplit = ksplit_for(M, N, K, nz);
    g.accumulate = 1;
    return gemm_launch(g, false, false, nz, c.st);
}

int bwd_bias(const Ctx& c, const float* dY, int ld, long long dy_z, float* db, long long db_z, int M, int N,
             int nz) {
    if (!c.wgrad) return CHROMO_OK;
    if (c.q) {
        c.q->add_bias(dY, ld, dy_z, db, db_z, M, N, nz);
        return CHROMO_OK;
    }
    const int rpb = 16;
    dim3 grid((N + 127) / 128, (M + rpb - 1) / rpb, nz);
    colsum_kernel<<<grid, 128, 0, c.st>>>(dY, M, N, ld, dy_z, db, db_z, rpb);
    CHROMO_CHECK_LAUNCH("colsum");
    return CHROMO_OK;
}

int ln_bwd(const Ctx& c, const float* pre, long long pre_z, const float* gin, float* gout, long long g_z,
           const float* gamma, float* dgamma, float* dbeta, long long p_z, int M, int nz) {
    LnBwdArgs a{M, pre, pre_z, gin, gout, g_z, gamma, c.wgrad ? dgamma : nullptr, dbeta, p_z};
    int blocks = (M + 7) / 8;
    if (blocks > 296) blocks = 296;
    launch_pdl(ln_bwd_kernel, dim3(dim3(blocks, nz)), dim3(256), 0, c.st, a);
    CHROMO_CHECK_LAUNCH("ln_bwd");
    return CHROMO_OK;
}

// Backward of  y = LN(u + W2 relu(W1 u + b1) + b2):  gin = dy [M,128]  ->  gA = LN'(gin), dF = relu'(gA W2),
// gout = gA + dF W1 (= du).  gA and dF stay untouched afterwards (weight gradients).
int ffn_bwd(const Ctx& c, const float* P, float* G, const FfnOff& f, long long p_z, int dff, const float* u,
            const float* fact, const float* preY, long long act_z, const float* gin, float* gA, float* dF, float* gout,
            long long g_z, int M) {
    const int D = 128, nz = c.NR;
    CHROMO_TRY(ln_bwd(c, preY, act_z, gin, gA, g_z, P + f.lnw, G + f.lnw, G + f.lnb, p_z, M, nz));
    CHROMO_TRY(bwd_weight(c, gA, D, g_z, fact, dff, 1, act_z, G + f.l2w, dff, p_z, M, D, dff, nz));
    CHROMO_TRY(bwd_bias(c, gA, D, g_z, G + f.l2b, p_z, M, D, nz));
    DataEpi relu; relu.mask = fact; relu.mask_z = act_z;
    CHROMO_TRY(bwd_data(c, gA, D, g_z, P + f.l2w, p_z, dF, dff, g_z, M, D, dff, relu, nz));
    CHROMO_TRY(bwd_weight(c, dF, dff, g_z, u, D, 1, act_z, G + f.l1w, D, p_z, M, dff, D, nz));
    CHROMO_TRY(bwd_bias(c, dF, dff, g_z, G + f.l1b, p_z, M, dff, nz));
    DataEpi resid; resid.res = gA;
    CHROMO_TRY(bwd_data(c, dF, dff, g_z, P + f.l1w, p_z, gout, D, g_z, M, dff, D, resid, nz));
    return CHROMO_OK;
}

struct SqaBwd {
    int rows, H, dm, D, n, F;
    const float* q; const float* qk; const float* P; const float* xbar; const float* cbar;
    const float* w_k; const float* w_v; const float* w_in; const float* pe; const float* x;
    const uint8_t* mask; long long mask_stride, mask_row_offset;
    float* g_wk; float* g_wv; float* g_win;
    const float* dAv; float* dQ;
    float* dCbar; float* dQK; float* dU8; float* dS;
};

int sqa_bwd(const Ctx& c, const SqaBwd& s) {
    const int dh = s.dm / s.H, D = s.D, RH = s.rows * s.H;
    Ctx c1 = c; c1.NR = 1;
    {   // dCbar[(r,h), :] = dAv[r, h] W_v[h]
        GemmArgs g = gemm_args();
        g.A = s.dAv; g.lda = s.dm; g.sA2 = dh;
        g.B = s.w_v; g.ldb = D; g.sB2 = (long long)dh * D;
        g.C = s.dCbar; g.ldc = s.H * D; g.sC2 = D;
        g.M = s.rows; g.N = D; g.K = dh; g.zdiv = s.H;
        CHROMO_TRY(gemm_auto(g, true, false, s.H, c.st, c.tc));
    }
    // dW_v[h] += dAv[:, h]^T Cbar[(:,h), :]
    if (c.q) {
        for (int h = 0; h < s.H; ++h)
            CHROMO_TRY(bwd_weight(c1, s.dAv + h * dh, s.dm, 0, s.cbar + (long long)h * D, s.H * D, 1, 0,
                                  s.g_wv + (long long)h * dh * D, D, 0, s.rows, dh, D, 1));
    } else if (c.wgrad) {   // (the queue exists only with wgrad)
        GemmArgs g = gemm_args();
        g.A = s.dAv; g.lda = s.dm; g.sA2 = dh;
        g.B = s.cbar; g.ldb = s.H * D; g.sB2 = D;
        g.C = s.g_wv; g.ldc = D; g.sC2 = (long long)dh * D;
        g.M = dh; g.N = D; g.K = s.rows; g.zdiv = s.H; g.accumulate = 1; g.ksplit = ksplit_for(s.rows, dh, D, s.H);
        CHROMO_TRY(gemm_launch(g, false, false, s.H, c.st));
    }
    {   // dP (PE part) = dCbar PE^T
        GemmArgs g = gemm_args();
        g.A = s.dCbar; g.lda = D; g.B = s.pe; g.ldb = D; g.C = s.dS; g.ldc = s.n;
        g.M = RH; g.N = s.n; g.K = D;
        CHROMO_TRY(gemm_auto(g, true, true, 1, c.st, c.tc));
    }
    {
        AttnRowsBwdArgs a;
        a.rows = RH; a.H = s.H; a.n = s.n; a.F = s.F; a.D = D;
        a.P = s.P; a.dS = s.dS; a.dcbar = s.dCbar; a.x = s.x;
        a.mask = s.mask; a.mask_stride = s.mask_stride; a.mask_row_offset = s.mask_row_offset;
        a.w_in = s.w_in; a.scale = 1.f / sqrtf((float)dh); a.dU8 = s.dU8; a.dqk = s.dQK;
        launch_pdl(attn_rows_bwd_kernel, dim3((RH + 7) / 8), dim3(256), 0, c.st, a);
        CHROMO_CHECK_LAUNCH("attn_rows_bwd");
    }
    // dW_in += dCbar^T xbar + QK^T dU
    CHROMO_TRY(bwd_weight(c1, s.dCbar, D, 0, s.xbar, 8, 1, 0, s.g_win, s.F, 0, RH, D, s.F, 1));
    CHROMO_TRY(bwd_weight(c1, s.qk, D, 0, s.dU8, 8, 1, 0, s.g_win, s.F, 0, RH, D, s.F, 1));
    {   // dQK += dS PE
        GemmArgs g = gemm_args();
        g.A = s.dS; g.lda = s.n; g.B = s.pe; g.ldb = D; g.C = s.dQK; g.ldc = D; g.accumulate = 1;
        g.M = RH; g.N = D; g.K = s.n;
        g.ksplit = ksplit_for(s.n, RH, D, 1);       // K = n bins (up to 400) on a handful of CTAs otherwise
        CHROMO_TRY(gemm_auto(g, true, false, 1, c.st, c.tc));
    }
    {   // dQ[r, h] = W_k[h] dQK[(r,h), :]
        GemmArgs g = gemm_args();
        g.A = s.dQK; g.lda = s.H * D; g.sA2 = D;
        g.B = s.w_k; g.ldb = D; g.sB2 = (long long)dh * D;
        g.C = s.dQ; g.ldc = s.dm; g.sC2 = dh;
        g.M = s.rows; g.N = dh; g.K = D; g.zdiv = s.H;
        CHROMO_TRY(gemm_auto(g, true, true, s.H, c.st, c.tc));
    }
    // dW_k[h] += Q[:, h]^T dQK[(:,h), :]
    if (c.q) {
        for (int h = 0; h < s.H; ++h)
            CHROMO_TRY(bwd_weight(c1, s.q + h * dh, s.dm, 0, s.dQK + (long long)h * D, s.H * D, 1, 0,
                                  s.g_wk + (long long)h * dh * D, D, 0, s.rows, dh, D, 1));
    } else if (c.wgrad) {   // (the queue exists only with wgrad)
        GemmArgs g = gemm_args();
        g.A = s.q; g.lda = s.dm; g.sA2 = dh;
        g.B = s.dQK; g.ldb = s.H * D; g.sB2 = D;
        g.C = s.g_wk; g.ldc = D; g.sC2 = (long long)dh * D;
        g.M = dh; g.N = D; g.K = s.rows; g.zdiv = s.H; g.accumulate = 1; g.ksplit = ksplit_for(s.rows, dh, D, s.H);
        CHROMO_TRY(gemm_launch(g, false, false, s.H, c.st));
    }
    return CHROMO_OK;
}

// dx (=|+=) the feature gradient of the regions sqa_bwd(s) has just run for (its P, dS, dCbar, qk and W_in)
int input_grad(cudaStream_t st, const SqaBwd& s, const float* dhc, float* dx, bool accumulate) {
    InputGradArgs a;
    a.regions = s.rows; a.H = s.H; a.n = s.n; a.F = s.F; a.D = s.D;
    a.P = s.P; a.dS = s.dS; a.dcbar = s.dCbar; a.qk = s.qk; a.w_in = s.w_in; a.dhc = dhc; a.dx = dx;
    a.accumulate = accumulate ? 1 : 0;
    launch_pdl(input_grad_rows_kernel, dim3((unsigned)((s.rows + 7) / 8)), dim3(256), 0, st, a);
    CHROMO_CHECK_LAUNCH("input_grad_rows");
    return CHROMO_OK;
}

}  // namespace

// G == nullptr: no parameter gradient (no weight / bias contraction, no LayerNorm or gamma_f reduction); dx: feature
// gradients to write (nullptr or NULL entries: none); dfreq: d interaction_freq [B,S,S] to write (nullptr: none) -
// chromo_backward passes (G, nullptr, nullptr).
static int backward_impl(const chromo_config_t* c, const float* P, const chromo_batch_t* in, const float* dlogits,
                         float* G, float* ws, const WsLayout& w, cudaStream_t st, bool tc, bool part1, bool part2,
                         const chromo_input_grads_t* dx = nullptr, float* dfreq = nullptr) {
    const ParamLayout& L = get_layout(c);
    const int B = w.B, I = w.I, S = w.S, R = w.R, T = w.T, D = w.D, F = c->n_feats, NR = c->n_res;
    const long long RS = w.res_stride;
    const int dme = c->embed_d_model, He = c->embed_heads, dffe = c->embed_d_ff;
    const int dmp = c->pw_d_model, Hp = c->pw_heads, dffp = c->pw_d_ff;
    const int dmr = c->reg_d_model, Hr = c->reg_heads, dffr = c->reg_d_ff;
    WgradQueue queue;
    const bool wgrad = G != nullptr;
    Ctx cx{st, NR, tc, tc && wgrad ? &queue : nullptr, wgrad};
    Ctx c1 = cx; c1.NR = 1;

    // ---- gradient scratch: one buffer per gradient tensor and layer (see Ctx) -------------------------------------
    int64_t cur = w.g_base;
    auto take = [&](int64_t n) { int64_t o = cur; cur = align4(cur + n); return o; };
    const int64_t blk0 = cur;
    int64_t o_gAr[CHROMO_MAX_LAYERS], o_dFr[CHROMO_MAX_LAYERS], o_gCr[CHROMO_MAX_LAYERS], o_dProj[CHROMO_MAX_LAYERS];
    for (int l = 0; l < c->reg_layers; ++l) {
        o_gAr[l] = take((int64_t)T * D); o_dFr[l] = take((int64_t)T * dffr);
        o_gCr[l] = take((int64_t)T * D); o_dProj[l] = take((int64_t)T * 4 * dmr);
    }
    const int64_t o_tR0 = take((int64_t)T * D), o_tR1 = take((int64_t)T * D), o_dAtt = take((int64_t)T * dmr);
    // The rest of each resolution's block (the Pairwise and Embedding gradient scratch, from o_gAp[0] on) is idle until
    // the Pairwise stage: it holds that resolution's partial of d interaction_freq during the Regulation stage,
    // [B,S,S] (gene kernel) or [B,Hr,S,S] (warp kernel: one slice per head).
    const int64_t o_fq = cur;
    int64_t o_gAp[CHROMO_MAX_LAYERS], o_dFp[CHROMO_MAX_LAYERS], o_gCp[CHROMO_MAX_LAYERS], o_dAvp[CHROMO_MAX_LAYERS],
        o_dQp[CHROMO_MAX_LAYERS], o_dCbP[CHROMO_MAX_LAYERS], o_dQKp[CHROMO_MAX_LAYERS], o_dU8p[CHROMO_MAX_LAYERS];
    for (int l = 0; l < c->pw_layers; ++l) {
        o_gAp[l] = take((int64_t)R * D); o_dFp[l] = take((int64_t)R * dffp); o_gCp[l] = take((int64_t)R * D);
        o_dAvp[l] = take((int64_t)R * dmp); o_dQp[l] = take((int64_t)R * dmp); o_dCbP[l] = take((int64_t)R * Hp * D);
        o_dQKp[l] = take((int64_t)R * Hp * D); o_dU8p[l] = take((int64_t)R * Hp * 8);
    }
    const int64_t o_tP0 = take((int64_t)R * D), o_tP1 = take((int64_t)R * D), o_dPP = take((int64_t)B * D);
    const int64_t o_gAe = take((int64_t)B * D), o_dFe = take((int64_t)B * dffe), o_gCe = take((int64_t)B * D),
                  o_dAve = take((int64_t)B * dme), o_dQe = take((int64_t)B * dme), o_dCbE = take((int64_t)B * He * D),
                  o_dQKe = take((int64_t)B * He * D), o_dU8e = take((int64_t)B * He * 8),
                  o_tE0 = take((int64_t)B * D), o_tE1 = take((int64_t)B * D), o_dHc = take((int64_t)B * D);
    const long long GS = cur - blk0;
    const bool gene_bwd = Hr == 8 && S <= 17;          // reg_attention_gene_bwd_kernel, else reg_attention_bwd_kernel
    const int fq_k = gene_bwd ? 1 : Hr;                // dfreq partials per (resolution, gene)
    if (dfreq && (int64_t)B * fq_k * S * S > blk0 + GS - o_fq) {
        set_error("internal: interaction_freq gradient partials exceed the idle Pairwise scratch");
        return CHROMO_ENOMEM;
    }
    cur = blk0 + GS * NR;
    int64_t o_dSp[CHROMO_MAX_RES], o_dSe[CHROMO_MAX_RES];
    for (int r = 0; r < NR; ++r) {
        o_dSp[r] = take((int64_t)R * Hp * c->n_bins[r]);
        o_dSe[r] = take((int64_t)B * He * c->n_bins[r]);
    }
    const int64_t o_dz = take((int64_t)B * NR * D), o_dh1 = take((int64_t)B * c->d_head);
    if (cur > w.total) { set_error("internal: backward scratch exceeds workspace"); return CHROMO_ENOMEM; }

    float* gcur = ws + o_tR0;           // gradient arriving at the layer's output
    float* gnext = ws + o_tR1;
    cudaStream_t wst = st;
    if (part1) {
    // ---- head (net.py:377-380) ------------------------------------------------
    {
        const int dh = c->d_head, no = c->n_out;
        CHROMO_TRY(bwd_weight(c1, dlogits, no, 0, ws + w.h_h1, dh, 1, 0, G + L.fc2w, dh, 0, B, no, dh, 1));
        CHROMO_TRY(bwd_bias(c1, dlogits, no, 0, G + L.fc2b, 0, B, no, 1));
        DataEpi relu; relu.mask = ws + w.h_h1;
        CHROMO_TRY(bwd_data(c1, dlogits, no, 0, P + L.fc2w, 0, ws + o_dh1, dh, 0, B, no, dh, relu, 1));
        CHROMO_TRY(bwd_weight(c1, ws + o_dh1, dh, 0, ws + w.h_z, NR * D, 1, 0, G + L.fc0w, NR * D, 0, B, dh, NR * D, 1));
        CHROMO_TRY(bwd_bias(c1, ws + o_dh1, dh, 0, G + L.fc0b, 0, B, dh, 1));
        CHROMO_TRY(bwd_data(c1, ws + o_dh1, dh, 0, P + L.fc0w, 0, ws + o_dz, NR * D, 0, B, dh, NR * D, DataEpi(), 1));
        launch_pdl(head_scatter_kernel, dim3(dim3((unsigned)(((long long)T * D + 255) / 256), NR)), dim3(256), 0, st, 
            ws + o_tR0, GS, ws + o_dz, B, S, D, NR);
        CHROMO_CHECK_LAUNCH("head_scatter");
    }

    // ---- Regulation transformer ------------------------------------------------
    for (int l = c->reg_layers - 1; l >= 0; --l) {
        const AttnOff& ra = L.reg[0].att[l];
        const FfnOff& rf = L.reg[0].ffn[l];
        const long long so = (long long)w.rslot(l) * w.r_slot;
        const float* xin = l == 0 ? ws + w.r_xin : ws + w.r_out + (long long)w.rslot(l - 1) * w.r_slot;
        float* gA = ws + o_gAr[l]; float* dF = ws + o_dFr[l]; float* gC = ws + o_gCr[l]; float* dProj = ws + o_dProj[l];
        CHROMO_TRY(ffn_bwd(cx, P, G, rf, L.reg_stride, dffr, ws + w.r_u + so, ws + w.r_f + so, ws + w.r_preY + so, RS,
                           gcur, gA, dF, gnext, GS, T));
        CHROMO_TRY(ln_bwd(cx, ws + w.r_preU + so, RS, gnext, gC, GS, P + ra.lnw, G + ra.lnw, G + ra.lnb, L.reg_stride, T, NR));
        CHROMO_TRY(bwd_weight(cx, gC, D, GS, ws + w.r_att + so, dmr, 1, RS, G + ra.ffw, dmr, L.reg_stride, T, D, dmr, NR));
        CHROMO_TRY(bwd_bias(cx, gC, D, GS, G + ra.ffb, L.reg_stride, T, D, NR));
        CHROMO_TRY(bwd_data(cx, gC, D, GS, P + ra.ffw, L.reg_stride, ws + o_dAtt, dmr, GS, T, D, dmr, DataEpi(), NR));
        {
            RegAttnBwdArgs a;
            a.B = B; a.S = S; a.H = Hr;
            a.proj = ws + w.r_proj + so; a.proj_z = RS;
            a.prob = ws + w.r_prob + so; a.prob_z = RS;
            a.dout = ws + o_dAtt; a.dout_z = GS;
            a.dproj = dProj; a.dproj_z = GS;
            a.freq = in->freq;
            for (int r = 0; r < NR; ++r) a.imask[r] = in->imask[r];
            a.dgamma_f = wgrad ? G + ra.gamma_f : nullptr; a.dgamma_z = L.reg_stride;
            a.gamma_f = P + ra.gamma_f;
            a.dfreq = dfreq ? ws + o_fq : nullptr; a.dfreq_z = GS;
            a.dfreq_add = l != c->reg_layers - 1;       // the layers run in order on st
            dim3 grid((unsigned)(((long long)B * Hr + 7) / 8), NR);
            if (gene_bwd) {       // one CTA per gene, rows staged in shared memory
                const size_t smem = ((size_t)S * (4 * dmr + RAB_PAD) + (size_t)S * dmr + 2 * (size_t)Hr * S * S + Hr * S) * sizeof(float);
                static bool configured = false;
                if (!configured) {
                    const int mx = (17 * (4 * 256 + RAB_PAD) + 17 * 256 + 2 * 8 * 17 * 17 + 8 * 17) * (int)sizeof(float);
                    cudaFuncSetAttribute(reg_attention_gene_bwd_kernel<9, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
                    cudaFuncSetAttribute(reg_attention_gene_bwd_kernel<17, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
                    cudaFuncSetAttribute(reg_attention_gene_bwd_kernel<9, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
                    cudaFuncSetAttribute(reg_attention_gene_bwd_kernel<17, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
                    configured = true;
                }
                auto k = S <= 9 ? (dfreq ? reg_attention_gene_bwd_kernel<9, true> : reg_attention_gene_bwd_kernel<9, false>)
                                : (dfreq ? reg_attention_gene_bwd_kernel<17, true> : reg_attention_gene_bwd_kernel<17, false>);
                launch_pdl(k, dim3(B, NR), dim3(Hr * S * 4), smem, st, a);
            } else {
                auto k = S <= 9 ? (dfreq ? reg_attention_bwd_kernel<9, true> : reg_attention_bwd_kernel<9, false>)
                                : (dfreq ? reg_attention_bwd_kernel<17, true> : reg_attention_bwd_kernel<17, false>);
                launch_pdl(k, dim3(grid), dim3(256), 0, st, a);
            }
            CHROMO_CHECK_LAUNCH("reg_attention_bwd");
        }
        CHROMO_TRY(bwd_weight(cx, dProj, 4 * dmr, GS, xin, D, 1, RS, G + ra.att, D, L.reg_stride, T, 4 * dmr, D, NR));
        DataEpi resid; resid.res = gC;
        CHROMO_TRY(bwd_data(cx, dProj, 4 * dmr, GS, P + ra.att, L.reg_stride, gcur, D, GS, T, 4 * dmr, D, resid, NR));
        // gcur = dX of this layer = the gradient arriving at the output of layer l-1; gnext is free again
        // this layer's weight gradients start now, on the side stream and on 64 SMs, under the next layer's chain
        if (cx.q) {
            CHROMO_TRY(aux_fork(st, &wst));
            if (wst != st) CHROMO_TRY(queue.flush(wst, 64));
        }
    }
    // The Regulation transformer's weight gradients (two thirds of the queue) start now, on a side stream and on two
    // thirds of the SMs, under the Pairwise / Embedding backward; the rest follows at the end.
    launch_pdl(head_residual_kernel, dim3(dim3((B * D + 255) / 256, NR)), dim3(256), 0, st, gcur, GS, ws + o_dz, B, S, D, NR);
    CHROMO_CHECK_LAUNCH("head_residual");
    if (dfreq) {      // before the Pairwise stage reuses the partials' scratch on st
        launch_pdl(freq_grad_sum_kernel, dim3((unsigned)(((long long)B * S * S + 255) / 256)), dim3(256), 0, st, dfreq,
                   (const float*)(ws + o_fq), GS, NR, fq_k, B, S * S);
        CHROMO_CHECK_LAUNCH("freq_grad_sum");
    }
    }   // part1
    float* gR = gcur;                   // dX_in incl. the residual of net.py:378 (the Regulation loop ends in the buffer it began in)
    if (!part2) {
        if (cx.q) CHROMO_TRY(queue.flush(st));
        return aux_join(st, wst);
    }

    // ---- Pairwise Interaction transformer ---------------------------------------
    float* pcur = ws + o_tP0;
    float* pnext = ws + o_tP1;
    launch_pdl(gather_rows_kernel, dim3(dim3((unsigned)(((long long)R * 32 + 255) / 256), NR)), dim3(256), 0, st, pcur, GS, gR, GS, R, I, S, 1);
    CHROMO_CHECK_LAUNCH("gather_pairwise");
    for (int l = c->pw_layers - 1; l >= 0; --l) {
        const AttnOff& pa = L.pw[0].att[l];
        const FfnOff& pf = L.pw[0].ffn[l];
        const long long so = (long long)w.pslot(l) * w.p_slot;
        const float* pin = l == 0 ? ws + w.p_pp : ws + w.p_out + (long long)w.pslot(l - 1) * w.p_slot;
        const int pin_div = l == 0 ? I : 1;
        float* gA = ws + o_gAp[l]; float* dF = ws + o_dFp[l]; float* gC = ws + o_gCp[l];
        CHROMO_TRY(ffn_bwd(cx, P, G, pf, L.pw_stride, dffp, ws + w.p_u + so, ws + w.p_f + so, ws + w.p_preY + so, RS,
                           pcur, gA, dF, pnext, GS, R));
        CHROMO_TRY(ln_bwd(cx, ws + w.p_preU + so, RS, pnext, gC, GS, P + pa.lnw, G + pa.lnw, G + pa.lnb, L.pw_stride, R, NR));
        CHROMO_TRY(bwd_weight(cx, gC, D, GS, ws + w.p_av + so, dmp, 1, RS, G + pa.ffw, dmp, L.pw_stride, R, D, dmp, NR));
        CHROMO_TRY(bwd_bias(cx, gC, D, GS, G + pa.ffb, L.pw_stride, R, D, NR));
        CHROMO_TRY(bwd_data(cx, gC, D, GS, P + pa.ffw, L.pw_stride, ws + o_dAvp[l], dmp, GS, R, D, dmp, DataEpi(), NR));
        ResStreams prs;
        CHROMO_TRY(res_fork(st, NR, prs));
        for (int r = 0; r < NR; ++r) {
            SqaBwd s;
            s.rows = R; s.H = Hp; s.dm = dmp; s.D = D; s.n = c->n_bins[r]; s.F = F;
            s.q = ws + r * RS + w.p_q + so; s.qk = ws + r * RS + w.p_qk + so;
            s.P = ws + w.p_p[r] + (long long)w.pslot(l) * w.p_p_slot[r];
            s.xbar = ws + r * RS + w.p_xbar + so; s.cbar = ws + r * RS + w.p_cbar + so;
            const int64_t catt = L.pw[r].att[l].c_att;
            s.w_k = P + catt; s.w_v = P + catt + (long long)dmp * D; s.w_in = P + L.pw[r].lin_proj_pcre;
            s.pe = in->pos_enc[r]; s.x = in->x_pcre[r];
            s.mask = in->mask_pcre[r]; s.mask_stride = in->mask_pcre_stride[r];
            s.mask_row_offset = in->mask_pcre_row_offset[r];
            s.g_wk = G + catt; s.g_wv = G + catt + (long long)dmp * D; s.g_win = G + L.pw[r].lin_proj_pcre;
            s.dAv = ws + r * GS + o_dAvp[l]; s.dQ = ws + r * GS + o_dQp[l];
            s.dCbar = ws + r * GS + o_dCbP[l]; s.dQK = ws + r * GS + o_dQKp[l]; s.dU8 = ws + r * GS + o_dU8p[l];
            s.dS = ws + o_dSp[r];
            Ctx cr = cx; cr.st = prs.s[r];
            CHROMO_TRY(sqa_bwd(cr, s));
            // both layers read the same pCRE embedding: the last layer writes, lower ones add (before the next layer's
            // sqa_bwd reuses dS on this stream)
            if (dx && dx->x_pcre[r]) CHROMO_TRY(input_grad(prs.s[r], s, nullptr, dx->x_pcre[r], l != c->pw_layers - 1));
        }
        CHROMO_TRY(res_join(prs));
        CHROMO_TRY(bwd_weight(cx, ws + o_dQp[l], dmp, GS, pin, D, pin_div, RS, G + pa.p_att, D, L.pw_stride, R, dmp, D, NR));
        DataEpi resid; resid.res = gC;
        CHROMO_TRY(bwd_data(cx, ws + o_dQp[l], dmp, GS, P + pa.p_att, L.pw_stride, pcur, D, GS, R, dmp, D, resid, NR));
    }
    // pcur = dP_0 per (gene, slot); P_0 = PP[gene] for every slot (net.py:114-118)
    launch_pdl(slot_sum_kernel, dim3(dim3((unsigned)(((long long)B * 32 + 255) / 256), NR)), dim3(256), 0, st, ws + o_dPP, GS, pcur, GS, B, I);
    CHROMO_CHECK_LAUNCH("slot_sum");
    CHROMO_TRY(bwd_weight(cx, ws + o_dPP, D, GS, ws + w.r_xin, S * D, 1, RS, G + L.pw[0].lin_proj_p, D, L.pw_stride, B, D, D, NR));
    {   // dX_in[b, 0, :] += dPP W_lpp
        GemmArgs g = gemm_args();
        g.A = ws + o_dPP; g.lda = D; g.sA1 = GS;
        g.B = P + L.pw[0].lin_proj_p; g.ldb = D; g.sB1 = L.pw_stride;
        g.C = gR; g.ldc = D; g.sC1 = GS; g.c_div = 1; g.c_mul = S; g.c_add = 0; g.accumulate = 1;
        g.M = B; g.N = D; g.K = D;
        CHROMO_TRY(gemm_auto(g, true, false, NR, st, tc));
    }

    if (cx.q) {   // the Pairwise weight gradients follow on the side stream (ordered behind st)
        CHROMO_TRY(aux_fork(st, &wst));
        if (wst != st) CHROMO_TRY(queue.flush(wst, 64));
    }

    // ---- Embedding transformer ----------------------------------------------------
    float* ecur = ws + o_tE0;
    float* enext = ws + o_tE1;
    launch_pdl(gather_rows_kernel, dim3(dim3((unsigned)(((long long)B * 32 + 255) / 256), NR)), dim3(256), 0, st, ecur, GS, gR, GS, B, 1, S, 0);
    CHROMO_CHECK_LAUNCH("gather_embed");
    {
        const AttnOff& ea = L.embed[0].att[0];
        const FfnOff& ef = L.embed[0].ffn[0];
        float* gA = ws + o_gAe; float* dF = ws + o_dFe; float* gC = ws + o_gCe; float* dHc = ws + o_dHc;
        CHROMO_TRY(ffn_bwd(cx, P, G, ef, L.embed_stride, dffe, ws + w.e_u, ws + w.e_f, ws + w.e_preY, RS, ecur, gA, dF,
                           enext, GS, B));
        CHROMO_TRY(ln_bwd(cx, ws + w.e_preU, RS, enext, gC, GS, P + ea.lnw, G + ea.lnw, G + ea.lnb, L.embed_stride, B, NR));
        CHROMO_TRY(bwd_weight(cx, gC, D, GS, ws + w.e_av, dme, 1, RS, G + ea.ffw, dme, L.embed_stride, B, D, dme, NR));
        CHROMO_TRY(bwd_bias(cx, gC, D, GS, G + ea.ffb, L.embed_stride, B, D, NR));
        CHROMO_TRY(bwd_data(cx, gC, D, GS, P + ea.ffw, L.embed_stride, ws + o_dAve, dme, GS, B, D, dme, DataEpi(), NR));
        ResStreams ers;
        CHROMO_TRY(res_fork(st, NR, ers));
        SqaBwd es[CHROMO_MAX_RES];
        for (int r = 0; r < NR; ++r) {
            SqaBwd& s = es[r];
            s.rows = B; s.H = He; s.dm = dme; s.D = D; s.n = c->n_bins[r]; s.F = F;
            s.q = ws + r * RS + w.e_q; s.qk = ws + r * RS + w.e_qk; s.P = ws + w.e_p[r];
            s.xbar = ws + r * RS + w.e_xbar; s.cbar = ws + r * RS + w.e_cbar;
            const int64_t att = L.embed[r].att[0].att;
            s.w_k = P + att + (long long)dme * D; s.w_v = P + att + (long long)2 * dme * D;
            s.w_in = P + L.embed[r].lin_proj;
            s.pe = in->pos_enc[r]; s.x = in->x_p[r];
            s.mask = in->mask_p[r]; s.mask_stride = in->mask_p_stride[r]; s.mask_row_offset = in->mask_p_row_offset[r];
            s.g_wk = G + att + (long long)dme * D; s.g_wv = G + att + (long long)2 * dme * D;
            s.g_win = G + L.embed[r].lin_proj;
            s.dAv = ws + r * GS + o_dAve; s.dQ = ws + r * GS + o_dQe;
            s.dCbar = ws + r * GS + o_dCbE; s.dQK = ws + r * GS + o_dQKe; s.dU8 = ws + r * GS + o_dU8e;
            s.dS = ws + o_dSe[r];
            Ctx cr = cx; cr.st = ers.s[r];
            CHROMO_TRY(sqa_bwd(cr, s));
        }
        CHROMO_TRY(res_join(ers));
        // W_q is rows [0, dme) of att.weight
        CHROMO_TRY(bwd_weight(cx, ws + o_dQe, dme, GS, ws + w.e_hc, D, 1, RS, G + ea.att, D, L.embed_stride, B, dme, D, NR));
        DataEpi resid; resid.res = gC;
        CHROMO_TRY(bwd_data(cx, ws + o_dQe, dme, GS, P + ea.att, L.embed_stride, dHc, D, GS, B, dme, D, resid, NR));
        // Hc = W_lp x_c + PE_c  ->  dW_lp += dHc^T x_p[:, c, :]
        for (int r = 0; r < NR; ++r) {
            const int n = c->n_bins[r];
            CHROMO_TRY(bwd_weight(c1, dHc + r * GS, D, 0, in->x_p[r] + (long long)(n / 2) * F, n * F, 1, 0,
                                  G + L.embed[r].lin_proj, F, 0, B, D, F, 1));
        }
        // promoter features: keys / values of every bin, and the centre bin's Hc through dHc
        for (int r = 0; r < NR; ++r)
            if (dx && dx->x_p[r]) CHROMO_TRY(input_grad(st, es[r], dHc + r * GS, dx->x_p[r], false));
    }
    if (cx.q) CHROMO_TRY(queue.flush(st));
    return aux_join(st, wst);
}

}  // namespace chromo

using namespace chromo;

// The checks both entry points share (`out`: the entry point's required output); fills *w.
static int backward_args(const chromo_config_t* cfg, const float* params, const chromo_batch_t* in, const float* dlogits,
                         const void* out, float* workspace, int64_t workspace_floats, int32_t flags, const char* who,
                         WsLayout* w) {
    CHROMO_TRY(validate_config(cfg));
    if (!params || !in || !dlogits || !out || !workspace) { set_error("null pointer argument"); return CHROMO_EINVAL; }
    if (!(flags & CHROMO_F_TRAINING)) { set_error("%s needs the CHROMO_F_TRAINING workspace", who); return CHROMO_EINVAL; }
    if (in->batch < 1) { set_error("batch must be >= 1"); return CHROMO_EINVAL; }
    *w = make_ws_layout(cfg, in->batch, flags);
    if (workspace_floats < w->total) {
        set_error("workspace too small: need %lld floats, got %lld", (long long)w->total, (long long)workspace_floats);
        return CHROMO_ENOMEM;
    }
    return CHROMO_OK;
}

extern "C" int chromo_backward(const chromo_config_t* cfg, const float* params, const chromo_batch_t* in,
                               const float* dlogits, float* grads, float* workspace, int64_t workspace_floats,
                               int32_t flags, void* stream) {
    WsLayout w;
    CHROMO_TRY(backward_args(cfg, params, in, dlogits, grads, workspace, workspace_floats, flags, "chromo_backward", &w));
    const bool only1 = (flags & CHROMO_F_BWD_HEAD_REG) != 0, only2 = (flags & CHROMO_F_BWD_REST) != 0;
    if (only1 && only2) { set_error("chromo_backward: CHROMO_F_BWD_HEAD_REG and CHROMO_F_BWD_REST are exclusive"); return CHROMO_EINVAL; }
    return backward_impl(cfg, params, in, dlogits, grads, workspace, w, (cudaStream_t)stream,
                         (flags & CHROMO_F_BF16) != 0, !only2, !only1);
}

extern "C" int chromo_backward_inputs(const chromo_config_t* cfg, const float* params, const chromo_batch_t* in,
                                      const float* dlogits, float* grads, const chromo_input_grads_t* dx,
                                      float* workspace, int64_t workspace_floats, int32_t flags, void* stream) {
    WsLayout w;
    CHROMO_TRY(backward_args(cfg, params, in, dlogits, dx, workspace, workspace_floats, flags, "chromo_backward_inputs",
                             &w));
    if (flags & (CHROMO_F_BWD_HEAD_REG | CHROMO_F_BWD_REST)) {
        set_error("chromo_backward_inputs runs the whole pass: CHROMO_F_BWD_HEAD_REG / CHROMO_F_BWD_REST are not accepted");
        return CHROMO_EINVAL;
    }
    float* dfreq = nullptr;             // (dx->freq exists only for callers that set the flag)
    if (flags & CHROMO_F_FREQ_GRAD) {
        if (!dx->freq) { set_error("chromo_backward_inputs: CHROMO_F_FREQ_GRAD with dx->freq == NULL"); return CHROMO_EINVAL; }
        dfreq = dx->freq;
    }
    // Only parameter and feature gradients need the Pairwise / Embedding stages: d interaction_freq alone stops after
    // the Regulation stage.
    bool feats = false;
    for (int r = 0; r < cfg->n_res; ++r) feats |= dx->x_p[r] != nullptr || dx->x_pcre[r] != nullptr;
    return backward_impl(cfg, params, in, dlogits, grads, workspace, w, (cudaStream_t)stream,
                         (flags & CHROMO_F_BF16) != 0, true, grads != nullptr || feats, dx, dfreq);
}
