// BF16 tensor-core engine for the dense projections (sm_100a: tcgen05 + TMEM + TMA bulk).
//
//   C[z][row(m), n] = epi( sum_k bf16(A[z][m, k]) * bf16(W[z][n, k]) )      FP32 accumulate
//
// * A (activations) stays FP32 in HBM: it is converted to BF16 while being staged into
//   shared memory in the canonical K-major no-swizzle UMMA layout (8x8 core matrices).
// * W (nn.Linear weight [N,K]) is pre-packed once per parameter version into that same
//   layout (pack_weights), so one 1-D TMA bulk copy (cp.async.bulk, mbarrier complete_tx)
//   brings a whole [NT x K] tile into shared memory.
// * One CTA = one 128-row M tile x one NT-column N tile: K/16 tcgen05.mma (M=128, N=NT,
//   K=16) issued by a single thread accumulate into TMEM; tcgen05.commit signals the four
//   epilogue warps, which read their 32 TMEM lanes with tcgen05.ld and apply the fused
//   epilogue (bias / ReLU / bias+residual+LayerNorm) straight from registers.
// K is small (128..400) on this path, so there is no K pipeline inside a CTA; overlap comes
// from two resident CTAs per SM (A/B staging of one under the MMA/epilogue of the other).
#include <algorithm>
#include <cuda_bf16.h>

#include "common.cuh"
#include "gemm_simt.cuh"
#include "umma_gemm.cuh"
#include "umma_ptx.cuh"

namespace chromo {

// ------------------------------------------------------------------ weight packing --
// src FP32 [N,K] row-major -> dst BF16, tiles of NT rows, each [NT/8][K/8][8][8].
__global__ void pack_weights_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int N, int K,
                                    int NT, long long z_stride, int transposed, int ld_src, int valid) {
    const int z = blockIdx.y;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // one 8-element K chunk
    const int KC = K / 8;
    if (i >= (long long)N * KC) return;
    const int n = (int)(i / KC), kc = (int)(i % KC);
    const float* s = src + z * z_stride;
    __nv_bfloat16 v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int k = kc * 8 + j;
        // `valid` bounds the source extent along the padded dimension (K when transposed, N otherwise)
        const bool in = transposed ? (k < valid) : (n < valid);
        const float x = !in ? 0.f : (transposed ? s[(long long)k * ld_src + n] : s[(long long)n * ld_src + k]);
        v[j] = __float2bfloat16_rn(x);
    }
    const int t = n / NT, r = n % NT;
    const long long off = (long long)t * NT * K + ((long long)(r / 8) * KC + kc) * 64 + (r % 8) * 8;
    *reinterpret_cast<uint4*>(dst + z * z_stride + off) = *reinterpret_cast<const uint4*>(v);
}

int pack_weights(const float* src, __nv_bfloat16* dst, int N, int K, int NT, long long z_stride, int nz,
                 bool transposed, int ld_src, cudaStream_t st, int valid) {
    if (valid < 0) valid = transposed ? K : N;
    if (K % 8 != 0 || N % NT != 0 || NT % 8 != 0) { set_error("pack_weights: bad shape"); return CHROMO_EINVAL; }
    const long long units = (long long)N * (K / 8);
    pack_weights_kernel<<<dim3((unsigned)((units + 255) / 256), nz), 256, 0, st>>>(src, dst, N, K, NT, z_stride,
                                                                                    transposed ? 1 : 0, ld_src, valid);
    CHROMO_CHECK_LAUNCH("pack_weights");
    return CHROMO_OK;
}

// ------------------------------------------------------------------ the GEMM kernel --
constexpr int UM = 128;           // rows per CTA = UMMA M = TMEM lanes
constexpr int UTHREADS = 256;     // 8 warps: warp w reads TMEM lanes 32*(w%4).., column chunks (c/32)%2 == w/4
constexpr size_t UMMA_SMEM_MAX = 225 * 1024;   // of the 227 KB a CTA may opt in to
constexpr int STAGE_LD = 33;      // padded row of the per-warp 32x32 epilogue staging tile

struct UmmaArgs {
    GemmArgs g;
    const __nv_bfloat16* Bp;      // packed weights (same z strides as g.B)
    int NT;                       // N tile (multiple of 16, <= 256, divides N)
    int tmem_cols;                // power of two >= max(32, NT)
};

// Write one 32x32 FP32 tile held as (lane = row, v[0..31] = columns) to C so that every store
// instruction covers 4 rows x 128 contiguous bytes: transpose through a padded shared tile.
__device__ __forceinline__ void store_tile_f32(float* stage, const float* v, float* C, const long long* crow4,
                                               int ldc, int col0, int ncols, int lane, unsigned rowmask) {
#pragma unroll
    for (int j = 0; j < 32; ++j) stage[lane * STAGE_LD + j] = v[j];
    __syncwarp();
    const int cq = (lane & 7) * 4;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int r = it * 4 + (lane >> 3);
        const float* sp = stage + r * STAGE_LD + cq;
        const float4 o = make_float4(sp[0], sp[1], sp[2], sp[3]);
        const long long cr = __shfl_sync(0xffffffffu, crow4[0], r);     // destination row of tile row r
        if (((rowmask >> r) & 1u) && cq < ncols) *reinterpret_cast<float4*>(C + cr * ldc + col0 + cq) = o;
    }
    __syncwarp();
}

__global__ void __launch_bounds__(UTHREADS) umma_linear_kernel(const UmmaArgs a) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const GemmArgs& g = a.g;
    const int K = g.K, NT = a.NT;
    __nv_bfloat16* sA = reinterpret_cast<__nv_bfloat16*>(smem);
    __nv_bfloat16* sB = reinterpret_cast<__nv_bfloat16*>(smem + (size_t)UM * K * 2);
    size_t ctl = (size_t)(UM + NT) * K * 2;                     // control block sits behind operands AND staging
    if (ctl < (size_t)(UTHREADS / 32) * 32 * STAGE_LD * 4) ctl = (size_t)(UTHREADS / 32) * 32 * STAGE_LD * 4;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + ctl);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);
    float* red = reinterpret_cast<float*>(bars + 4);            // [2][128][2] LayerNorm partial sums

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int m0 = blockIdx.y * UM, nt = blockIdx.x, n0 = nt * NT;
    const int z1 = blockIdx.z / g.zdiv, z2 = blockIdx.z % g.zdiv;
    const float* A = g.A + z1 * g.sA1 + z2 * g.sA2;
    const __nv_bfloat16* Bp = a.Bp + z1 * g.sB1 + z2 * g.sB2 + (long long)nt * NT * K;

    if (warp == 0) tmem_alloc(tmem_slot, a.tmem_cols);
    if (tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (tid == 0) {   // weights: one TMA bulk copy of the pre-packed [NT x K] tile
        const uint32_t bytes = (uint32_t)NT * K * 2;
        mbar_expect_tx(&bars[0], bytes);
        tma_bulk_g2s(sB, Bp, bytes, &bars[0]);
    }

    // activations: FP32 -> BF16 into the canonical layout.  A warp covers 8 rows x 32 columns per
    // unit (lane -> row lane/4, 8-column chunk lane%4): 128-byte coalesced global segments,
    // conflict-free 16-byte shared stores.  Four units are loaded before any is converted so
    // that eight 16-byte loads per thread are in flight.
    {
        const int KC = K / 8;
        const int units = (UM / 8) * ((KC + 3) / 4);
        constexpr int UNR = 4;
        for (int u0 = warp; u0 < units; u0 += (UTHREADS / 32) * UNR) {
            float4 x[UNR][2];
            int r_[UNR], kc_[UNR];
            bool ok_[UNR];
#pragma unroll
            for (int q = 0; q < UNR; ++q) {
                const int u = u0 + q * (UTHREADS / 32);
                const int rg = u % (UM / 8), cg = u / (UM / 8);
                r_[q] = rg * 8 + (lane >> 2);
                kc_[q] = cg * 4 + (lane & 3);
                const int m = m0 + r_[q];
                ok_[q] = u < units && kc_[q] < KC;
                x[q][0] = x[q][1] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (ok_[q] && m < g.M) {
                    const float* p = A + (long long)(m / g.a_div) * g.lda + kc_[q] * 8;
                    x[q][0] = __ldg(reinterpret_cast<const float4*>(p));
                    x[q][1] = __ldg(reinterpret_cast<const float4*>(p + 4));
                }
            }
#pragma unroll
            for (int q = 0; q < UNR; ++q) {
                if (!ok_[q]) continue;
                __nv_bfloat162 b0 = __floats2bfloat162_rn(x[q][0].x, x[q][0].y), b1 = __floats2bfloat162_rn(x[q][0].z, x[q][0].w);
                __nv_bfloat162 b2 = __floats2bfloat162_rn(x[q][1].x, x[q][1].y), b3 = __floats2bfloat162_rn(x[q][1].z, x[q][1].w);
                uint4 packed;
                packed.x = *reinterpret_cast<uint32_t*>(&b0); packed.y = *reinterpret_cast<uint32_t*>(&b1);
                packed.z = *reinterpret_cast<uint32_t*>(&b2); packed.w = *reinterpret_cast<uint32_t*>(&b3);
                *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(sA) + ((size_t)(r_[q] >> 3) * KC + kc_[q]) * 128 +
                                          (r_[q] & 7) * 16) = packed;
            }
        }
    }
    fence_async_smem();
    __syncthreads();

    if (tid == 0) {
        mbar_wait(&bars[0], 0);
        tc_fence_after();
        const uint32_t idesc = umma_idesc_bf16(UM, NT);
        const uint32_t lbo = 128u, sbo = (uint32_t)K * 16;
        const uint32_t a0 = smem_u32(sA), b0 = smem_u32(sB);
        const uint64_t ad = umma_smem_desc(a0, lbo, sbo), bd = umma_smem_desc(b0, lbo, sbo);   // then +256 B = +16 per k step
        for (int k = 0; k < K / 16; ++k) umma_bf16(tmem_base, ad + 16 * k, bd + 16 * k, idesc, k > 0 ? 1u : 0u);
        umma_commit(&bars[1]);
    }
    __syncwarp();
    mbar_wait(&bars[1], 0);
    tc_fence_after();
    // all MMAs have completed: the operand tiles are dead, reuse them as epilogue staging
    float* stage = reinterpret_cast<float*>(smem) + warp * (32 * STAGE_LD);

    // ------------------------------------------------------------------ epilogue ----
    const int lq = warp & 3, ch = warp >> 2;
    const int m = m0 + lq * 32 + lane;                   // this thread's row = its TMEM lane
    const uint32_t trow = tmem_base + ((uint32_t)(lq * 32) << 16);
    const bool ok = m < g.M;
    const unsigned rowmask = __ballot_sync(0xffffffffu, ok);
    const long long crow = ok ? (long long)(m / g.c_div) * g.c_mul + (m % g.c_div) + g.c_add : 0;
    const float* bias = g.bias ? g.bias + z1 * g.sBias1 + z2 * g.sBias2 : nullptr;
    float v[32];
    if (g.epi == EPI_BIAS_RES_LN) {
        // N == NT == 128.  The two warps sharing a lane quarter each own two 32-column chunks of the
        // row: partial sums meet in shared memory, then each normalises and writes its chunks.
        float* C = g.C + z1 * g.sC1 + z2 * g.sC2;
        const float* res = g.res + z1 * g.sRes1 + (ok ? (long long)(m / g.res_div) * g.ldres : 0);
        const float* gamma = g.gamma + z1 * g.sLn1;
        const float* beta = g.beta + z1 * g.sLn1;
        float* pre = (g.pre && ok) ? g.pre + z1 * g.sPre1 + (long long)m * g.N : nullptr;
        float keep[2][32];
        float sum = 0.f, sq = 0.f;
#pragma unroll
        for (int ci = 0; ci < 2; ++ci) {
            const int c = (2 * ci + ch) * 32;
            tmem_ld32(trow + c, v);
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                float4 r4 = make_float4(0, 0, 0, 0);
                if (ok) r4 = *reinterpret_cast<const float4*>(res + c + j);
                const float4 b4 = bias ? *reinterpret_cast<const float4*>(bias + c + j) : make_float4(0, 0, 0, 0);
                const float t0 = v[j] + b4.x + r4.x, t1 = v[j + 1] + b4.y + r4.y;
                const float t2 = v[j + 2] + b4.z + r4.z, t3 = v[j + 3] + b4.w + r4.w;
                keep[ci][j] = t0; keep[ci][j + 1] = t1; keep[ci][j + 2] = t2; keep[ci][j + 3] = t3;
                sum += (t0 + t1) + (t2 + t3);
                sq += (t0 * t0 + t1 * t1) + (t2 * t2 + t3 * t3);
                if (pre) *reinterpret_cast<float4*>(pre + c + j) = make_float4(t0, t1, t2, t3);
            }
        }
        red[(ch * 128 + lq * 32 + lane) * 2] = sum;
        red[(ch * 128 + lq * 32 + lane) * 2 + 1] = sq;
        __syncthreads();
        sum += red[((1 - ch) * 128 + lq * 32 + lane) * 2];
        sq += red[((1 - ch) * 128 + lq * 32 + lane) * 2 + 1];
        const float mean = sum * (1.f / 128.f);
        const float var = fmaxf(sq * (1.f / 128.f) - mean * mean, 0.f);
        const float rstd = rsqrtf(var + 1e-5f);
#pragma unroll
        for (int ci = 0; ci < 2; ++ci) {
            const int c = (2 * ci + ch) * 32;
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                const float4 ga = *reinterpret_cast<const float4*>(gamma + c + j);
                const float4 be = *reinterpret_cast<const float4*>(beta + c + j);
                v[j] = (keep[ci][j] - mean) * rstd * ga.x + be.x;
                v[j + 1] = (keep[ci][j + 1] - mean) * rstd * ga.y + be.y;
                v[j + 2] = (keep[ci][j + 2] - mean) * rstd * ga.z + be.z;
                v[j + 3] = (keep[ci][j + 3] - mean) * rstd * ga.w + be.w;
            }
            store_tile_f32(stage, v, C, &crow, g.ldc, c, 32, lane, rowmask);
        }
    } else {
        const bool sqa_staged = g.c_sqa_tiles && K >= 96;        // (UM + NT) * K * 2 >= 64 KB of dead operand space
        for (int c = ch * 32; c < NT; c += 64) {
            tmem_ld32(trow + c, v);          // columns beyond NT (NT % 32 != 0) are dropped below
            const int ncols = min(32, NT - c);
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                if (j < ncols) {
                    if (g.epi != EPI_PLAIN && bias) {
                        const float4 b4 = *reinterpret_cast<const float4*>(bias + n0 + c + j);
                        v[j] += b4.x; v[j + 1] += b4.y; v[j + 2] += b4.z; v[j + 3] += b4.w;
                    }
                    if (g.epi == EPI_BIAS_RELU) {
                        v[j] = fmaxf(v[j], 0.f); v[j + 1] = fmaxf(v[j + 1], 0.f);
                        v[j + 2] = fmaxf(v[j + 2], 0.f); v[j + 3] = fmaxf(v[j + 3], 0.f);
                    }
                }
            }
            if (g.c_sqa_tiles && sqa_staged) {
                // QK operand tiles of sqa_fused: row 2m + head of the 128-row tiles, 16-byte chunks of 8 channels.  The 128
                // rows of this CTA fill exactly two consecutive tiles (64 KB contiguous in HBM): composed in shared memory
                // (the operands are dead), then written as full lines by everybody (rows past M as zeros)
                const int head = (n0 + c) >> 7, kc0 = ((n0 + c) & 127) >> 3;
                const int Rl = 2 * (lq * 32 + lane) + head, r = Rl & 127;
                uint8_t* sp = smem + (Rl >> 7) * 32768 + (r >> 3) * 2048 + (r & 7) * 16;
#pragma unroll
                for (int j = 0; j < 32; j += 8) {
                    uint4 pk = make_uint4(0u, 0u, 0u, 0u);
                    if (ok) {
                        __nv_bfloat162 p0 = __floats2bfloat162_rn(v[j], v[j + 1]), p1 = __floats2bfloat162_rn(v[j + 2], v[j + 3]);
                        __nv_bfloat162 p2 = __floats2bfloat162_rn(v[j + 4], v[j + 5]), p3 = __floats2bfloat162_rn(v[j + 6], v[j + 7]);
                        pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
                        pk.z = *reinterpret_cast<uint32_t*>(&p2); pk.w = *reinterpret_cast<uint32_t*>(&p3);
                    }
                    *reinterpret_cast<uint4*>(sp + (kc0 + (j >> 3)) * 128) = pk;
                }
            } else if (g.c_sqa_tiles) {
                if (ok) {
                    const int head = (n0 + c) >> 7, kc0 = ((n0 + c) & 127) >> 3;
                    const long long R = 2LL * m + head;
                    const int r = (int)(R & 127);
                    __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(g.C) + z1 * g.sC1 + z2 * g.sC2 + (R >> 7) * 16384 +
                                         (r >> 3) * 1024 + (r & 7) * 8;
#pragma unroll
                    for (int j = 0; j < 32; j += 8) {
                        if (j < ncols) {
                            __nv_bfloat162 p0 = __floats2bfloat162_rn(v[j], v[j + 1]), p1 = __floats2bfloat162_rn(v[j + 2], v[j + 3]);
                            __nv_bfloat162 p2 = __floats2bfloat162_rn(v[j + 4], v[j + 5]), p3 = __floats2bfloat162_rn(v[j + 6], v[j + 7]);
                            uint4 pk;
                            pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
                            pk.z = *reinterpret_cast<uint32_t*>(&p2); pk.w = *reinterpret_cast<uint32_t*>(&p3);
                            *reinterpret_cast<uint4*>(out + (kc0 + (j >> 3)) * 64) = pk;
                        }
                    }
                }
            } else if (g.c_bf16) {
                // BF16 output: the thread's 32 columns are 64 contiguous bytes
                if (ok) {
                    __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(g.C) + z1 * g.sC1 + z2 * g.sC2 +
                                         crow * g.ldc + n0 + c;
#pragma unroll
                    for (int j = 0; j < 32; j += 8) {
                        if (j < ncols) {
                            __nv_bfloat162 p0 = __floats2bfloat162_rn(v[j], v[j + 1]), p1 = __floats2bfloat162_rn(v[j + 2], v[j + 3]);
                            __nv_bfloat162 p2 = __floats2bfloat162_rn(v[j + 4], v[j + 5]), p3 = __floats2bfloat162_rn(v[j + 6], v[j + 7]);
                            uint4 pk;
                            pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
                            pk.z = *reinterpret_cast<uint32_t*>(&p2); pk.w = *reinterpret_cast<uint32_t*>(&p3);
                            *reinterpret_cast<uint4*>(out + j) = pk;
                        }
                    }
                }
            } else {
                float* C = g.C + z1 * g.sC1 + z2 * g.sC2;
                if (g.accumulate) {
                    if (ok) {
                        float* out = C + crow * g.ldc + n0 + c;
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            if (j < ncols) {
                                float4 o = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                                if (g.accumulate) {
                                    const float4 old = *reinterpret_cast<const float4*>(out + j);
                                    o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w;
                                }
                                *reinterpret_cast<float4*>(out + j) = o;
                            }
                        }
                    }
                } else {
                    store_tile_f32(stage, v, C, &crow, g.ldc, n0 + c, ncols, lane, rowmask);
                }
            }
        }
    }
    if (g.c_sqa_tiles && K >= 96) {
        __syncthreads();
        uint8_t* out = reinterpret_cast<uint8_t*>(reinterpret_cast<__nv_bfloat16*>(g.C) + z1 * g.sC1 + z2 * g.sC2) +
                       (long long)blockIdx.y * 65536;
        const int tiles = (2 * g.M - 2 * m0 + 127) / 128;       // 1 when the last CTA's rows end in its first tile
        const int n16 = (tiles >= 2 ? 2 : 1) * 2048;
        for (int i = tid; i < n16; i += UTHREADS)
            reinterpret_cast<uint4*>(out)[i] = reinterpret_cast<const uint4*>(smem)[i];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, a.tmem_cols);
}

// ---------------------------------------------------------------- the query GEMM of a single-query-attention stage ----
// QK[m, (h, :)] = A[m / a_div, :] . M^T  (K = 128, N = 256 = two heads), written as the BF16 operand tiles sqa_fused pulls
// in by TMA (row 2m + head of 128-row tiles: the 128 rows of a step fill two consecutive 32 KB tiles).
// Persistent and warp-specialised, one CTA per SM: the 64 KB weight tile, the barriers and all 512 TMEM columns (two
// accumulators) live for the whole launch;
//   warps 8..15  producers: FP32 rows -> BF16 canonical K-major A stage (two stages), all loads of a thread in flight
//   warp 16      one thread issues the 8 tcgen05.mma (M = 128, N = 256) of a stage and commits them to the barriers
//   warps 0..7   epilogue: accumulator (lane quarter = warp % 4, head = warp / 4) -> BF16 -> 16-byte chunks straight to HBM
// so the staging of tile i+1 and the epilogue of tile i-1 run under the MMAs of tile i.  (The serial one-CTA-per-tile form
// of this GEMM spent ~11 us per tile on set-up and barrier round trips: 1.4 TB/s of output; two such CTAs per SM with 16
// warps each did not change that.)
constexpr int QK_THREADS = 544;
enum { QB_W = 0, QB_AFULL0, QB_AFREE0 = QB_AFULL0 + 2, QB_DFULL0 = QB_AFREE0 + 2, QB_DFREE0 = QB_DFULL0 + 2, QB_COUNT = QB_DFREE0 + 2 };
__device__ __forceinline__ void qk_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__global__ void __launch_bounds__(QK_THREADS, 1) qk_tiles_kernel(const UmmaArgs a) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const GemmArgs& g = a.g;
    constexpr int K = 128, NT = 256, KC = K / 8;
    uint8_t* sB = smem;                                   // 64 KB
    uint8_t* sA = smem + NT * K * 2;                      // 2 x 32 KB
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + NT * K * 2 + 2 * UM * K * 2);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + QB_COUNT);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int z1 = blockIdx.y;
    const float* A = g.A + z1 * g.sA1;
    const __nv_bfloat16* Bp = a.Bp + z1 * g.sB1;
    uint8_t* out_z = reinterpret_cast<uint8_t*>(reinterpret_cast<__nv_bfloat16*>(g.C) + z1 * g.sC1);

    if (warp == 0) tmem_alloc(tmem_slot, 512);
    if (tid == 0) {
        mbar_init(&bars[QB_W], 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bars[QB_AFULL0 + i], 8);           // one arrival per producer warp
            mbar_init(&bars[QB_AFREE0 + i], 1);           // tcgen05.commit
            mbar_init(&bars[QB_DFULL0 + i], 1);           // tcgen05.commit
            mbar_init(&bars[QB_DFREE0 + i], 8);           // one arrival per epilogue warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int M = g.m_dev ? *g.m_dev : g.M;               // ragged plan: the live rows only
    const int m_tiles = (M + UM - 1) / UM;

    if (warp >= 8 && warp < 16) {
        // ================================================= producers ====
        const int pw = warp - 8;
        uint32_t it = 0;
        for (int mt = blockIdx.x; mt < m_tiles; mt += gridDim.x, ++it) {
            const int st = it & 1, m0 = mt * UM;
            if (it >= 2) mbar_wait(&bars[QB_AFREE0 + st], ((it >> 1) - 1) & 1);
            uint8_t* dst = sA + st * (UM * K * 2);
            float4 x[8][2];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int u = pw + q * 8;                         // 64 units: 16 row groups x 4 column groups
                const int r = (u & 15) * 8 + (lane >> 2), kc = (u >> 4) * 4 + (lane & 3);
                const int m = m0 + r;
                x[q][0] = x[q][1] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (m < M) {
                    const float* p = A + (long long)((g.a_rows ? g.a_rows[m] : m) / g.a_div) * g.lda + kc * 8;
                    x[q][0] = __ldg(reinterpret_cast<const float4*>(p));
                    x[q][1] = __ldg(reinterpret_cast<const float4*>(p + 4));
                }
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int u = pw + q * 8;
                const int r = (u & 15) * 8 + (lane >> 2), kc = (u >> 4) * 4 + (lane & 3);
                __nv_bfloat162 b0 = __floats2bfloat162_rn(x[q][0].x, x[q][0].y), b1 = __floats2bfloat162_rn(x[q][0].z, x[q][0].w);
                __nv_bfloat162 b2 = __floats2bfloat162_rn(x[q][1].x, x[q][1].y), b3 = __floats2bfloat162_rn(x[q][1].z, x[q][1].w);
                uint4 pk;
                pk.x = *reinterpret_cast<uint32_t*>(&b0); pk.y = *reinterpret_cast<uint32_t*>(&b1);
                pk.z = *reinterpret_cast<uint32_t*>(&b2); pk.w = *reinterpret_cast<uint32_t*>(&b3);
                *reinterpret_cast<uint4*>(dst + ((size_t)(r >> 3) * KC + kc) * 128 + (r & 7) * 16) = pk;
            }
            fence_async_smem();
            __syncwarp();
            if (lane == 0) qk_arrive(&bars[QB_AFULL0 + st]);
        }
    } else if (warp == 16) {
        // ================================================= MMA issuer ====
        if (lane == 0) {
            mbar_expect_tx(&bars[QB_W], NT * K * 2);
            tma_bulk_g2s(sB, Bp, NT * K * 2, &bars[QB_W]);
            const uint32_t idesc = umma_idesc_bf16(UM, NT);
            const uint64_t bd = umma_smem_desc(smem_u32(sB), 128, K * 16);
            mbar_wait(&bars[QB_W], 0);
            uint32_t it = 0;
            for (int mt = blockIdx.x; mt < m_tiles; mt += gridDim.x, ++it) {
                const int st = it & 1;
                mbar_wait(&bars[QB_AFULL0 + st], (it >> 1) & 1);
                if (it >= 2) mbar_wait(&bars[QB_DFREE0 + st], ((it >> 1) - 1) & 1);
                tc_fence_after();
                const uint64_t ad = umma_smem_desc(smem_u32(sA + st * (UM * K * 2)), 128, K * 16);
#pragma unroll
                for (int k = 0; k < K / 16; ++k) umma_bf16(tmem_base + 256 * st, ad + 16 * k, bd + 16 * k, idesc, k > 0 ? 1u : 0u);
                umma_commit(&bars[QB_AFREE0 + st]);
                umma_commit(&bars[QB_DFULL0 + st]);
            }
        }
    } else if (warp < 8) {
        // ================================================= epilogue ====
        const int lq = warp & 3, head = warp >> 2;
        const int row = lq * 32 + lane;
        const int r = (2 * row + head) & 127, t = row >> 6;
        uint32_t it = 0;
        for (int mt = blockIdx.x; mt < m_tiles; mt += gridDim.x, ++it) {
            const int st = it & 1, m0 = mt * UM;
            mbar_wait(&bars[QB_DFULL0 + st], (it >> 1) & 1);
            tc_fence_after();
            const uint32_t trow = tmem_base + 256 * st + 128 * head + ((uint32_t)(lq * 32) << 16);
            const bool ok = m0 + row < M;
            const bool tile_ok = 2 * m0 + 128 * t < 2 * M;       // (the second tile of the last step may not exist)
            uint8_t* out = out_z + ((long long)mt * 2 + t) * 32768 + (r >> 3) * 2048 + (r & 7) * 16;
            float v[32], w[32];
#pragma unroll
            for (int c2 = 0; c2 < 2; ++c2) {
                tmem_ld32_pair(trow + 64 * c2, v, trow + 64 * c2 + 32, w);
                if (c2 == 1) {                                   // every load of this warp has landed: the accumulator may go
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) qk_arrive(&bars[QB_DFREE0 + st]);
                }
                if (tile_ok) {
#pragma unroll
                    for (int hf = 0; hf < 2; ++hf) {
                        const float* s = hf ? w : v;
#pragma unroll
                        for (int j = 0; j < 32; j += 8) {
                            uint4 pk = make_uint4(0u, 0u, 0u, 0u);
                            if (ok) {
                                __nv_bfloat162 p0 = __floats2bfloat162_rn(s[j], s[j + 1]), p1 = __floats2bfloat162_rn(s[j + 2], s[j + 3]);
                                __nv_bfloat162 p2 = __floats2bfloat162_rn(s[j + 4], s[j + 5]), p3 = __floats2bfloat162_rn(s[j + 6], s[j + 7]);
                                pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
                                pk.z = *reinterpret_cast<uint32_t*>(&p2); pk.w = *reinterpret_cast<uint32_t*>(&p3);
                            }
                            *reinterpret_cast<uint4*>(out + (8 * c2 + 4 * hf + (j >> 3)) * 128) = pk;
                        }
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 512);
}

static size_t umma_smem_bytes(int nt, int K) {
    size_t operands = (size_t)(UM + nt) * K * 2;
    const size_t staging = (size_t)(UTHREADS / 32) * 32 * STAGE_LD * 4;      // reuses the operand area
    if (operands < staging) operands = staging;
    return operands + 32 + 2 * 128 * 2 * 4;                                   // barriers, TMEM slot, LN partials
}

static int choose_nt(int N) {
    if (N % 16 != 0) return 0;
    if (N <= 256) return N;
    for (int nt = 256; nt >= 16; nt -= 16)
        if (N % nt == 0) return nt;
    return 0;
}

int umma_tile_n(int N) { return choose_nt(N); }

bool umma_supported(const GemmArgs& g) {
    if (g.K % 16 != 0 || g.K < 16 || g.ksplit != 1) return false;
    const int nt = choose_nt(g.N);
    if (nt == 0) return false;
    if (umma_smem_bytes(nt, g.K) > UMMA_SMEM_MAX) return false;
    if (g.lda % 4 != 0 || g.ldc % 4 != 0) return false;
    if ((reinterpret_cast<uintptr_t>(g.A) & 15) || (reinterpret_cast<uintptr_t>(g.C) & 15)) return false;
    if (g.epi == EPI_BIAS_RES_LN && (g.N != 128 || g.accumulate || g.c_bf16)) return false;
    if (g.c_bf16 && (g.accumulate || g.N % 8 != 0)) return false;
    if (g.c_sqa_tiles && (g.N != 256 || g.accumulate || g.epi != EPI_PLAIN || g.c_div != 1 || g.c_mul != 1 || g.c_add != 0 ||
                          g.zdiv != 1))
        return false;
    return true;
}

// the persistent query GEMM (qk_tiles_kernel) takes this call: the only GEMM that honours a ragged plan
bool umma_qk_persistent(const GemmArgs& g) {
    return g.c_sqa_tiles && g.K == 128 && g.N == 256 && g.zdiv == 1 && (g.M + UM - 1) / UM >= 8;
}

int umma_launch(const GemmArgs& g, const __nv_bfloat16* Bp, int nz, cudaStream_t st) {
    UmmaArgs a;
    a.g = g; a.Bp = Bp; a.NT = choose_nt(g.N);
    a.tmem_cols = 32;
    while (a.tmem_cols < a.NT) a.tmem_cols *= 2;
    const size_t smem = umma_smem_bytes(a.NT, g.K);
    static size_t configured = 0;
    if (smem > configured) {
        cudaError_t e = cudaFuncSetAttribute(umma_linear_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)UMMA_SMEM_MAX);
        if (e != cudaSuccess) { set_error("umma smem attribute: %s", cudaGetErrorString(e)); return CHROMO_ECUDA; }
        configured = UMMA_SMEM_MAX;
    }
    const bool qk_persistent = umma_qk_persistent(g);
    if ((g.a_rows || g.m_dev) && !qk_persistent) { set_error("internal: ragged plan on a GEMM that does not take it"); return CHROMO_EINVAL; }
    if (qk_persistent) {
        static bool qk_configured = false;
        const size_t qsmem = (size_t)(2 * UM + 256) * 128 * 2 + 128;
        if (!qk_configured) {
            cudaFuncSetAttribute(qk_tiles_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)qsmem);
            cudaFuncSetAttribute(qk_tiles_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            qk_configured = true;
        }
        int sms = 148;
        {
            int dev = 0;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        }
        const int m_tiles = (g.M + UM - 1) / UM;
        const int per_z = std::min(m_tiles, std::max(1, sms / nz));
        qk_tiles_kernel<<<dim3(per_z, nz), QK_THREADS, qsmem, st>>>(a);
        CHROMO_CHECK_LAUNCH("qk_tiles");
        return CHROMO_OK;
    }
    dim3 grid(g.N / a.NT, (g.M + UM - 1) / UM, nz);
    umma_linear_kernel<<<grid, UTHREADS, smem, st>>>(a);
    CHROMO_CHECK_LAUNCH("umma_linear");
    return CHROMO_OK;
}

}  // namespace chromo
