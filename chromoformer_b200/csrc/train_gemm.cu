// Tensor-core contractions of the TRAINING step (train.py:182-196: forward of every nn.Linear, its data gradient, and
// - queued and run in one persistent launch - its weight and bias gradients):
//
//   forward          Y[m, n]   = epi( sum_k X[m, k]  * W[n, k] )         A = X rows  (K-major), B = W rows (K-major)
//   data gradient    dX[m, k]  = epi( sum_n dY[m, n] * W[n, k] )         A = dY rows (K-major), B = W rows (MN-major)
//   weight gradient  dW[n, k] +=      sum_m dY[m, n] * X[m, k]           A = dY rows (MN-major), B = X rows (MN-major)
//
// Activations, gradients and parameters are FP32 in HBM and change every step, so nothing is pre-packed: a CTA converts
// its [128 x 128] A chunk and [NT x 128] B chunk to BF16 while staging them into shared memory in the canonical
// no-swizzle UMMA layout of the wanted major-ness (8 x 8 core matrices of 16-byte rows; the SAME 128-byte cores serve
// the K-major and the MN-major reading, only the instruction descriptor's transpose bits differ), issues the chunk's
// tcgen05.mma (M = 128, N = NT <= 256, K = 16) into a TMEM accumulator and moves on (two shared-memory stages: the
// staging of chunk i+1 runs under the MMAs of chunk i).  Loads are issued eight 32-byte runs per thread ahead of the
// first conversion so that a chunk costs a few memory round trips, not one per row.
//
// Epilogues (tcgen05.ld, thread = accumulator row): bias, residual add, pre-LayerNorm stash + LayerNorm, ReLU, ReLU
// mask of the backward pass; rows leave through a shared-memory transpose as 128-byte segments.
#include <algorithm>
#include <stdlib.h>
#include <string.h>
#include <unordered_map>
#include <cuda_bf16.h>

#include "common.cuh"
#include "train_gemm.cuh"
#include "umma_ptx.cuh"

namespace chromo {

static long long* g_tg_trace = nullptr;        // chromo_debug_trace: phase clocks of CTA 0 of every tc_gemm launch ([2048..))
void tc_gemm_set_trace(long long* buf) { g_tg_trace = buf; }

namespace {

constexpr int TG_THREADS = 512;                // 16 warps: the staging and the epilogue of a tile are latency chains per warp
constexpr int TG_WARPS = TG_THREADS / 32;
constexpr int TG_KCH = 128;                    // contraction elements per chunk
constexpr uint32_t TG_A_BYTES = 128 * TG_KCH * 2;
constexpr int TG_UNR = 8;                      // 32-byte runs per thread in flight
constexpr int STAGE_LD = 33;                   // padded row of the per-warp 32 x 32 epilogue staging tile

__device__ __forceinline__ uint4 pack8(const float4& a, const float4& b) {
    __nv_bfloat162 p0 = __floats2bfloat162_rn(a.x, a.y), p1 = __floats2bfloat162_rn(a.z, a.w);
    __nv_bfloat162 p2 = __floats2bfloat162_rn(b.x, b.y), p3 = __floats2bfloat162_rn(b.z, b.w);
    uint4 pk;
    pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
    pk.z = *reinterpret_cast<uint32_t*>(&p2); pk.w = *reinterpret_cast<uint32_t*>(&p3);
    return pk;
}

// eight consecutive floats at p, the first `n` of them valid (the rest zeros)
__device__ __forceinline__ void load8(const float* __restrict__ p, int n, bool vec, float4& x0, float4& x1) {
    if (n >= 8 && vec) {
        x0 = __ldg(reinterpret_cast<const float4*>(p));
        x1 = __ldg(reinterpret_cast<const float4*>(p + 4));
    } else {
        float t[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) t[j] = j < n ? __ldg(p + j) : 0.f;
        x0 = make_float4(t[0], t[1], t[2], t[3]);
        x1 = make_float4(t[4], t[5], t[6], t[7]);
    }
}

// Stage one operand chunk: `rows` MN-indices (tile, multiple of 16) x TG_KCH contraction indices -> BF16 in `dst`.
//   mn_major == 0: memory is [mn, kc] (kc contiguous)  -> ((mn/8)*16 + kc/8)*128 + (mn%8)*16 + (kc%8)*2
//   mn_major == 1: memory is [kc, mn] (mn contiguous)  -> ((mn/8)*16 + kc/8)*128 + (kc%8)*16 + (mn%8)*2
// Out-of-range elements are zeros.  `div` broadcasts memory ROWS (row index / div).  `vec`: 16-byte loads are legal
// (aligned base, leading dimension a multiple of 4 floats).
__device__ __noinline__ void stage_operand_generic(uint8_t* dst, const float* __restrict__ src, long long ld, int mn_major,
                                                   int div, int rows, int mn0, int mn_lim, int kc0, int kc_lim, bool vec,
                                                   int warp, int lane) {
    const int rg_n = (rows + 31) >> 5;
    const int units = mn_major ? (TG_KCH / 8) * rg_n : (rows >> 3) * 4;
    for (int u0 = warp; u0 < units; u0 += TG_WARPS * TG_UNR) {
        float4 x[TG_UNR][2];
        uint32_t off[TG_UNR];
#pragma unroll
        for (int q = 0; q < TG_UNR; ++q) {
            const int u = u0 + q * TG_WARPS;
            x[q][0] = x[q][1] = make_float4(0.f, 0.f, 0.f, 0.f);
            off[q] = 0xffffffffu;
            if (u >= units) continue;
            if (!mn_major) {                                    // 8 mn rows x 32 kc columns per warp pass
                const int r = (u >> 2) * 8 + (lane >> 2), c8 = (u & 3) * 4 + (lane & 3);
                const int mn = mn0 + r, kc = kc0 + c8 * 8;
                off[q] = (uint32_t)(((r >> 3) * 16 + c8) * 128 + (r & 7) * 16);
                if (mn < mn_lim && kc < kc_lim) load8(src + (long long)(mn / div) * ld + kc, kc_lim - kc, vec, x[q][0], x[q][1]);
            } else {                                            // 8 kc rows x 32 mn columns per warp pass
                const int k = (u / rg_n) * 8 + (lane >> 2), r8 = (u % rg_n) * 4 + (lane & 3);
                if (r8 * 8 >= rows) continue;                   // (tile narrower than the last 32-column group)
                const int kc = kc0 + k, mn = mn0 + r8 * 8;
                off[q] = (uint32_t)((r8 * 16 + (k >> 3)) * 128 + (k & 7) * 16);
                if (kc < kc_lim && mn < mn_lim) load8(src + (long long)(kc / div) * ld + mn, mn_lim - mn, vec, x[q][0], x[q][1]);
            }
        }
#pragma unroll
        for (int q = 0; q < TG_UNR; ++q)
            if (off[q] != 0xffffffffu) *reinterpret_cast<uint4*>(dst + off[q]) = pack8(x[q][0], x[q][1]);
    }
}

// The same staging when no row is broadcast (div == 1) and the tile's 32-column groups divide the 16 warps: the runs of
// a thread then differ by constant strides in memory and in the tile, so that a chunk costs each thread two compares,
// two 16-byte loads, four conversions and one 16-byte store per run - all loads ahead of the first conversion.
__device__ __forceinline__ void stage_operand(uint8_t* dst, const float* __restrict__ src, long long ld, int mn_major, int div,
                                              int rows, int mn0, int mn_lim, int kc0, int kc_lim, bool vec, int warp,
                                              int lane) {
    const int rg_n = (rows + 31) >> 5;
    if (div != 1 || (mn_major && (TG_WARPS % rg_n) != 0)) {
        stage_operand_generic(dst, src, ld, mn_major, div, rows, mn0, mn_lim, kc0, kc_lim, vec, warp, lane);
        return;
    }
    const float* p; long long pstride; uint32_t off, ostride; int idx, istride, ilim, nq, nvalid;
    if (!mn_major) {
        const int units = (rows >> 3) * 4;
        const int r0 = (warp >> 2) * 8 + (lane >> 2), c8 = (warp & 3) * 4 + (lane & 3);
        nq = warp < units ? (units - warp + TG_WARPS - 1) / TG_WARPS : 0;
        p = src + (long long)(mn0 + r0) * ld + kc0 + c8 * 8; pstride = (long long)(TG_WARPS / 4) * 8 * ld;
        off = (uint32_t)(((r0 >> 3) * 16 + c8) * 128 + (r0 & 7) * 16); ostride = (TG_WARPS / 4) * 2048;
        idx = mn0 + r0; istride = (TG_WARPS / 4) * 8; ilim = mn_lim;
        nvalid = kc_lim - (kc0 + c8 * 8);
    } else {
        const int per = TG_WARPS / rg_n;                      // k groups advanced per step
        const int kq = warp / rg_n, r8 = (warp % rg_n) * 4 + (lane & 3), k = kq * 8 + (lane >> 2);
        nq = (r8 * 8 < rows && kq < TG_KCH / 8) ? (TG_KCH / 8 - kq + per - 1) / per : 0;
        p = src + (long long)(kc0 + k) * ld + mn0 + r8 * 8; pstride = (long long)per * 8 * ld;
        off = (uint32_t)((r8 * 16 + (k >> 3)) * 128 + (k & 7) * 16); ostride = per * 128;
        idx = kc0 + k; istride = per * 8; ilim = kc_lim;
        nvalid = mn_lim - (mn0 + r8 * 8);
    }
    nvalid = nvalid < 0 ? 0 : (nvalid > 8 ? 8 : nvalid);
    const bool full = vec && nvalid == 8;
    for (int q0 = 0; q0 < nq; q0 += TG_UNR) {
        float4 x[TG_UNR][2];
        if (full) {
#pragma unroll
            for (int j = 0; j < TG_UNR; ++j) {
                const int q = q0 + j;
                x[j][0] = x[j][1] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (q < nq && idx + q * istride < ilim) {
                    const float* pp = p + q * pstride;
                    x[j][0] = __ldg(reinterpret_cast<const float4*>(pp));
                    x[j][1] = __ldg(reinterpret_cast<const float4*>(pp + 4));
                }
            }
        } else {
#pragma unroll
            for (int j = 0; j < TG_UNR; ++j) {
                const int q = q0 + j;
                x[j][0] = x[j][1] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (q < nq && idx + q * istride < ilim && nvalid > 0) load8(p + q * pstride, nvalid, false, x[j][0], x[j][1]);
            }
        }
#pragma unroll
        for (int j = 0; j < TG_UNR; ++j)
            if (q0 + j < nq) *reinterpret_cast<uint4*>(dst + off + (uint32_t)(q0 + j) * ostride) = pack8(x[j][0], x[j][1]);
    }
}

struct Operands {
    const float* A; long long lda; int a_t, a_div, a_vec, m0, m_lim;
    const float* B; long long ldb; int b_t, b_div, b_vec, n0, n_lim;
    int Kc, NT;                 // contraction range [k_begin, Kc)
    int k_begin = 0;
    int pdl = 0;                // launched as a programmatic dependent: griddepcontrol.wait before the first A access
};

// The contraction of one output tile into TMEM columns [0, NT).  `g` counts the chunks this CTA has pushed through the
// two stages so far (mbarrier parities carry over from tile to tile), `tiles` the tiles it has finished.
__device__ __forceinline__ void contract_tile(const Operands& o, uint8_t* smem, uint32_t stage_bytes, uint64_t* bars,
                                              uint32_t tmem, uint32_t& g, uint32_t tiles, int tid, int warp, int lane,
                                              long long* trace = nullptr) {
    const int chunks = (o.Kc - o.k_begin + TG_KCH - 1) / TG_KCH;
    const uint32_t idesc = umma_idesc_bf16(128, o.NT) | (o.a_t ? (1u << 15) : 0u) | (o.b_t ? (1u << 16) : 0u);
    for (int ci = 0; ci < chunks; ++ci, ++g) {
        const uint32_t st = g & 1;
        uint8_t* sA = smem + st * stage_bytes;
        uint8_t* sB = sA + TG_A_BYTES;
        if (g >= 2) mbar_wait(&bars[st], ((g >> 1) - 1) & 1);           // the MMAs of chunk g-2 have left this stage
        const int kc0 = o.k_begin + ci * TG_KCH;
        // B first: in tc_gemm_kernel it is a parameter / position table, independent of the kernel in front, so its staging
        // (like everything above) runs under that kernel's tail; A is the first dependent access (programmatic dependent launch)
        stage_operand(sB, o.B, o.ldb, o.b_t, o.b_div, o.NT, o.n0, o.n_lim, kc0, o.Kc, o.b_vec, warp, lane);
        if (ci == 0 && trace && tid == 0) trace[2] = clock64();
        if (ci == 0 && o.pdl) asm volatile("griddepcontrol.wait;" ::: "memory");
        stage_operand(sA, o.A, o.lda, o.a_t, o.a_div, 128, o.m0, o.m_lim, kc0, o.Kc, o.a_vec, warp, lane);
        if (ci == 0 && trace && tid == 0) trace[3] = clock64();
        fence_async_smem();
        __syncthreads();
        if (ci == 0 && trace && tid == 0) trace[4] = clock64();
        if (tid == 0) {
            tc_fence_after();
            const int ksteps = (min(TG_KCH, o.Kc - kc0) + 15) / 16;
            const uint64_t ad = umma_smem_desc(smem_u32(sA), 128, 2048), bd = umma_smem_desc(smem_u32(sB), 128, 2048);
            for (int k = 0; k < ksteps; ++k) umma_bf16(tmem, ad + 16 * k, bd + 16 * k, idesc, (ci > 0 || k > 0) ? 1u : 0u);
            umma_commit(&bars[st]);
            if (ci == chunks - 1) umma_commit(&bars[2]);
        }
    }
    if (trace && tid == 0) trace[5] = clock64();
    mbar_wait(&bars[2], tiles & 1);
    tc_fence_after();
}

// Write one 32x32 FP32 tile held as (lane = row, v[0..31] = columns) to C so that every store instruction covers 4 rows
// x 128 contiguous bytes: transpose through a padded shared tile.
__device__ __forceinline__ void store_tile_f32(float* stage, const float* v, float* C, long long crow, long long ldc, int col0,
                                               int ncols, int lane, unsigned rowmask) {
#pragma unroll
    for (int j = 0; j < 32; ++j) stage[lane * STAGE_LD + j] = v[j];
    __syncwarp();
    const int cq = (lane & 7) * 4;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int r = it * 4 + (lane >> 3);
        const float* sp = stage + r * STAGE_LD + cq;
        const float4 o = make_float4(sp[0], sp[1], sp[2], sp[3]);
        const long long cr = __shfl_sync(0xffffffffu, crow, r);          // destination row of tile row r
        if (((rowmask >> r) & 1u) && cq < ncols) *reinterpret_cast<float4*>(C + cr * ldc + col0 + cq) = o;
    }
    __syncwarp();
}

// The reverse: a 32 x 32 tile of a row-major matrix (row of tile row r at element offset `rowoff` of lane r) into
// (lane = row, v[0..31] = columns) through the same padded shared tile: 4 rows x 128 contiguous bytes per load.
__device__ __forceinline__ void load_tile_f32(float* stage, float* v, const float* src, long long rowoff, int col0, int ncols,
                                              int lane, unsigned rowmask) {
    const int cq = (lane & 7) * 4;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int r = it * 4 + (lane >> 3);
        const long long ro = __shfl_sync(0xffffffffu, rowoff, r);
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        if (((rowmask >> r) & 1u) && cq < ncols) x = *reinterpret_cast<const float4*>(src + ro + col0 + cq);
        float* sp = stage + r * STAGE_LD + cq;
        sp[0] = x.x; sp[1] = x.y; sp[2] = x.z; sp[3] = x.w;
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = stage[lane * STAGE_LD + j];
    __syncwarp();
}

// C tile (32 consecutive rows from `C`, leading dimension ldc) += (lane = row, v = columns), coalesced
__device__ __forceinline__ void add_tile_f32(float* stage, const float* v, float* C, long long ldc, int ncols, int nrows,
                                             int lane) {
#pragma unroll
    for (int j = 0; j < 32; ++j) stage[lane * STAGE_LD + j] = v[j];
    __syncwarp();
    const int cq = (lane & 7) * 4;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int r = it * 4 + (lane >> 3);
        if (r < nrows && cq < ncols) {
            const float* sp = stage + r * STAGE_LD + cq;
            float4* out = reinterpret_cast<float4*>(C + (long long)r * ldc + cq);
            float4 x = *out;
            x.x += sp[0]; x.y += sp[1]; x.z += sp[2]; x.w += sp[3];
            *out = x;
        }
    }
    __syncwarp();
}

#define TG_MARK(i) do { if (trace && tid == 0) trace[i] = clock64(); } while (0)

__global__ void __launch_bounds__(TG_THREADS) tc_gemm_kernel(const TcGemm a, long long* trace_buf) {
    extern __shared__ __align__(1024) uint8_t smem[];
    asm volatile("griddepcontrol.launch_dependents;");     // the next kernel of the chain may start its own prologue
    long long* trace = (trace_buf && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) ? trace_buf : nullptr;
    const int NT = a.NT;
    const uint32_t stage_bytes = TG_A_BYTES + (uint32_t)NT * TG_KCH * 2;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * stage_bytes);      // [0,1] stage free, [2] tile done
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3);
    float* red = reinterpret_cast<float*>(bars + 4);                            // [4][128][2] LayerNorm partial sums
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n0 = blockIdx.x * NT, m0 = blockIdx.y * 128, z = blockIdx.z / a.ksplit, split = blockIdx.z % a.ksplit;
    TG_MARK(0);
    int tmem_cols = 32;
    while (tmem_cols < NT) tmem_cols *= 2;

    if (warp == 0) tmem_alloc(tmem_slot, tmem_cols);
    if (tid == 0) {
        mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_init(&bars[2], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    TG_MARK(1);

    Operands o;
    o.A = a.A + z * a.a_z; o.lda = a.lda; o.a_t = a.a_t; o.a_div = a.a_div; o.m0 = m0; o.m_lim = a.M;
    o.B = a.B + z * a.b_z; o.ldb = a.ldb; o.b_t = a.b_t; o.b_div = a.b_div; o.n0 = n0; o.n_lim = a.N;
    o.a_vec = ((reinterpret_cast<uintptr_t>(o.A) & 15) == 0 && (a.lda & 3) == 0) ? 1 : 0;
    o.b_vec = ((reinterpret_cast<uintptr_t>(o.B) & 15) == 0 && (a.ldb & 3) == 0) ? 1 : 0;
    o.Kc = a.Kc; o.NT = NT; o.pdl = 1;
    if (a.ksplit > 1) {
        const int per = ((a.Kc + TG_KCH - 1) / TG_KCH + a.ksplit - 1) / a.ksplit * TG_KCH;
        o.k_begin = split * per;
        o.Kc = min(a.Kc, o.k_begin + per);
                                                        // (the launcher never makes an empty split)
    }
    uint32_t g = 0;
    contract_tile(o, smem, stage_bytes, bars, tmem, g, 0, tid, warp, lane, trace);
    TG_MARK(6);

    // ------------------------------------------------------------------ epilogue ----
    // all MMAs have completed: the operand stages are dead, reuse them as the transpose staging of the stores
    float* stage = reinterpret_cast<float*>(smem) + warp * (32 * STAGE_LD);
    const int lq = warp & 3, ch = warp >> 2;
    const int m = m0 + lq * 32 + lane;                   // this thread's row = its TMEM lane
    const uint32_t trow = tmem + ((uint32_t)(lq * 32) << 16);
    const bool ok = m < a.M;
    const unsigned rowmask = __ballot_sync(0xffffffffu, ok);
    const long long crow = ok ? (long long)(m / a.c_div) * a.c_mul + (m % a.c_div) + a.c_add : 0;
    float* C = a.C + z * a.c_z;
    const float* bias = (a.epi & TC_BIAS) ? a.bias + z * a.bias_z : nullptr;
    const float* res = ((a.epi & TC_RES) && split == 0) ? a.res + z * a.res_z : nullptr;
    const long long res_off = ok ? (long long)(m / a.res_div) * a.ldres : 0;
    float v[32], t[32];
    if (a.epi & TC_LN) {
        // N == NT == 128.  The four warps sharing a lane quarter each own one 32-column chunk of the row: partial sums
        // meet in shared memory, then each normalises and writes its chunk.
        const float* gamma = a.gamma + z * a.ln_z;
        const float* beta = a.beta + z * a.ln_z;
        const int c = ch * 32, rr = lq * 32 + lane;
        float sum = 0.f, sq = 0.f;
        tmem_ld32(trow + c, v);
        if (res) {
            load_tile_f32(stage, t, res, res_off, c, 32, lane, rowmask);
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] += t[j];
        }
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
            const float4 b4 = bias ? *reinterpret_cast<const float4*>(bias + c + j) : make_float4(0, 0, 0, 0);
            v[j] += b4.x; v[j + 1] += b4.y; v[j + 2] += b4.z; v[j + 3] += b4.w;
            sum += (v[j] + v[j + 1]) + (v[j + 2] + v[j + 3]);
        }
        if (a.pre) store_tile_f32(stage, v, a.pre + z * a.pre_z, ok ? (long long)m : 0, a.N, c, 32, lane, rowmask);
        red[(ch * 128 + rr) * 2] = sum;
        __syncthreads();
        sum = (red[rr * 2] + red[(128 + rr) * 2]) + (red[(256 + rr) * 2] + red[(384 + rr) * 2]);
        const float mean = sum * (1.f / 128.f);
#pragma unroll
        for (int j = 0; j < 32; ++j) { const float d = v[j] - mean; sq = fmaf(d, d, sq); }
        red[(ch * 128 + rr) * 2 + 1] = sq;
        __syncthreads();
        sq = (red[rr * 2 + 1] + red[(128 + rr) * 2 + 1]) + (red[(256 + rr) * 2 + 1] + red[(384 + rr) * 2 + 1]);
        const float rstd = rsqrtf(sq * (1.f / 128.f) + 1e-5f);
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
            const float4 ga = *reinterpret_cast<const float4*>(gamma + c + j);
            const float4 be = *reinterpret_cast<const float4*>(beta + c + j);
            v[j] = (v[j] - mean) * rstd * ga.x + be.x;
            v[j + 1] = (v[j + 1] - mean) * rstd * ga.y + be.y;
            v[j + 2] = (v[j + 2] - mean) * rstd * ga.z + be.z;
            v[j + 3] = (v[j + 3] - mean) * rstd * ga.w + be.w;
        }
        store_tile_f32(stage, v, C, crow, a.ldc, c, 32, lane, rowmask);
    } else {
        const float* mask = (a.epi & TC_MASK) ? a.mask + z * a.mask_z : nullptr;
        const long long mask_off = ok ? (long long)m * a.ldmask : 0;
        for (int c = ch * 32; c < NT; c += 128) {
            tmem_ld32(trow + c, v);          // columns beyond NT (NT % 32 != 0) are dropped below
            const int ncols = min(32, NT - c);
            if (res) {
                load_tile_f32(stage, t, res, res_off, n0 + c, ncols, lane, rowmask);
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] += t[j];
            }
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                if (j < ncols) {
                    if (bias) {
                        const float4 b4 = *reinterpret_cast<const float4*>(bias + n0 + c + j);
                        v[j] += b4.x; v[j + 1] += b4.y; v[j + 2] += b4.z; v[j + 3] += b4.w;
                    }
                    if (a.epi & TC_RELU) {
                        v[j] = fmaxf(v[j], 0.f); v[j + 1] = fmaxf(v[j + 1], 0.f);
                        v[j + 2] = fmaxf(v[j + 2], 0.f); v[j + 3] = fmaxf(v[j + 3], 0.f);
                    }
                }
            }
            if (mask) {
                load_tile_f32(stage, t, mask, mask_off, n0 + c, ncols, lane, rowmask);
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (!(t[j] > 0.f)) v[j] = 0.f;
            }
            if (a.ksplit > 1) {             // partial tile: FP32 atomics into the zeroed output
                if (ok) {
                    float* out = C + crow * a.ldc + n0 + c;
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (j < ncols) atomicAdd(out + j, v[j]);
                }
            } else {
                store_tile_f32(stage, v, C, crow, a.ldc, n0 + c, ncols, lane, rowmask);
            }
        }
    }
    TG_MARK(7);
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, tmem_cols);
    TG_MARK(8);
}

// ------------------------------------------------------------------ deferred weight / bias gradients ----
constexpr int WG_MAX_ITEMS = 640;              // 640 x 48 B = 30 KB of kernel parameters (limit 32,764 B)
constexpr int WG_NT_MAX = 256;
struct WgTable {
    int n;
    int pad[3];
    WgItem items[WG_MAX_ITEMS];
};
static_assert(sizeof(WgItem) == 48, "WgItem layout");
static_assert(sizeof(WgTable) <= 32000, "kernel parameter space");

__global__ void __launch_bounds__(TG_THREADS) wgrad_grouped_kernel(const __grid_constant__ WgTable tbl, long long* trace_buf) {
    extern __shared__ __align__(1024) uint8_t smem[];
    long long* trace = (trace_buf && blockIdx.x == 0) ? trace_buf : nullptr;
    int tr_i = 0;
    constexpr uint32_t stage_bytes = TG_A_BYTES + (uint32_t)WG_NT_MAX * TG_KCH * 2;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * stage_bytes);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (warp == 0) tmem_alloc(tmem_slot, WG_NT_MAX);
    if (tid == 0) {
        mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_init(&bars[2], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const int lq = warp & 3, ch = warp >> 2;
    const uint32_t trow = tmem + ((uint32_t)(lq * 32) << 16);
    uint32_t g = 0, tiles = 0;

    if (trace && threadIdx.x == 0) trace[tr_i++] = clock64();
    for (int it = blockIdx.x; it < tbl.n; it += gridDim.x) {
        const WgItem& w = tbl.items[it];
        if (trace && threadIdx.x == 0 && tr_i < 60) { trace[tr_i++] = ((long long)w.tokens << 48) | ((long long)w.n_cols << 36) | (clock64() & 0xfffffffffLL); }
        if (w.kind & 1) {
            // db[n] += sum_t dY[t, n]: one column per thread, four rows in flight
            if (tid < w.n_cols) {
                const float* p = w.A + tid;
                float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
                int t = 0;
                for (; t + 4 <= w.tokens; t += 4) {
                    s0 += __ldg(p + (long long)t * w.lda); s1 += __ldg(p + (long long)(t + 1) * w.lda);
                    s2 += __ldg(p + (long long)(t + 2) * w.lda); s3 += __ldg(p + (long long)(t + 3) * w.lda);
                }
                for (; t < w.tokens; ++t) s0 += __ldg(p + (long long)t * w.lda);
                if (w.kind & 2) atomicAdd(w.C + tid, (s0 + s1) + (s2 + s3));
                else w.C[tid] += (s0 + s1) + (s2 + s3);
            }
            continue;
        }
        Operands o;
        o.A = w.A; o.lda = w.lda; o.a_t = 1; o.a_div = 1; o.m0 = 0; o.m_lim = w.m_rows;
        o.B = w.B; o.ldb = w.ldb; o.b_t = 1; o.b_div = w.b_div; o.n0 = 0; o.n_lim = w.n_cols;
        o.a_vec = ((reinterpret_cast<uintptr_t>(w.A) & 15) == 0 && (w.lda & 3) == 0) ? 1 : 0;
        o.b_vec = ((reinterpret_cast<uintptr_t>(w.B) & 15) == 0 && (w.ldb & 3) == 0) ? 1 : 0;
        o.Kc = w.tokens; o.NT = (w.n_cols + 15) & ~15;
        contract_tile(o, smem, stage_bytes, bars, tmem, g, tiles, tid, warp, lane);
        ++tiles;
        if (trace && threadIdx.x == 0 && tr_i < 60) trace[tr_i++] = clock64() & 0xfffffffffLL;
        // dW tile += accumulator (this CTA owns the tile for the whole launch: plain read-modify-write, through a
        // shared-memory transpose so that every access covers 4 rows x 128 contiguous bytes)
        const int row = lq * 32 + lane;
        const bool vec = (reinterpret_cast<uintptr_t>(w.C) & 15) == 0 && (w.ldc & 3) == 0 && (w.n_cols & 3) == 0;
        float* wstage = reinterpret_cast<float*>(smem) + warp * (32 * STAGE_LD);     // (all MMAs of the tile have completed)
        float v[32];
        for (int c = ch * 32; c < o.NT; c += 128) {
            tmem_ld32(trow + c, v);
            const int ncols = min(32, w.n_cols - c);
            if (vec && !(w.kind & 2)) {
                if (lq * 32 < w.m_rows && ncols > 0)
                    add_tile_f32(wstage, v, w.C + (long long)(lq * 32) * w.ldc + c, w.ldc, ncols, w.m_rows - lq * 32, lane);
            } else if (row < w.m_rows) {
                float* out = w.C + (long long)row * w.ldc + c;
                if (w.kind & 2) {
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (j < ncols) atomicAdd(out + j, v[j]);
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (j < ncols) out[j] += v[j];
                }
            }
        }
        __syncthreads();              // the staging area goes back to the operands of the next tile
        tc_fence_before();            // the next tile's first MMA overwrites these columns: order it behind the loads
        if (trace && threadIdx.x == 0 && tr_i < 60) trace[tr_i++] = clock64() & 0xfffffffffLL;
    }
    if (trace && threadIdx.x == 0) { trace[tr_i++] = clock64() & 0xfffffffffLL; trace[63] = tr_i; }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, WG_NT_MAX);
}

int choose_nt(int N, int M, int nz, bool ln) {
    if (N % 16 != 0) return 0;
    if (ln) return N == 128 ? 128 : 0;
    // the largest tile that still gives a CTA to every third SM: the batch of a training step is a few hundred rows, and
    // every CTA of a row tile stages the same A chunk, so narrower tiles only shorten the B staging and the epilogue
    const int mt = (M + 127) / 128 * nz;
    for (int nt = 256; nt >= 64; nt >>= 1)
        if (N % nt == 0 && (N / nt) * mt >= 48) return nt;
    if (N % 64 == 0) return 64;
    if (N <= 256) return N;
    for (int nt = 240; nt >= 16; nt -= 16)
        if (N % nt == 0) return nt;
    return 0;
}

size_t gemm_smem(int NT) { return 2 * ((size_t)TG_A_BYTES + (size_t)NT * TG_KCH * 2) + 64 + 4 * 128 * 2 * 4; }

}  // namespace

TcGemm tc_gemm_args() {
    TcGemm g;
    memset(&g, 0, sizeof(g));
    g.a_div = g.b_div = g.res_div = g.c_div = g.c_mul = 1;
    return g;
}

bool tc_gemm_supported(const TcGemm& a) {
    if (a.M < 1 || a.Kc < 1 || a.N % 16 != 0) return false;
    if ((a.epi & TC_LN) && a.N != 128) return false;
    if (a.ldc % 4 != 0 || (reinterpret_cast<uintptr_t>(a.C) & 15) || a.c_z % 4 != 0) return false;
    if ((a.epi & TC_RES) && (a.ldres % 4 != 0 || (reinterpret_cast<uintptr_t>(a.res) & 15) || a.res_z % 4 != 0)) return false;
    if ((a.epi & TC_MASK) && (a.ldmask % 4 != 0 || (reinterpret_cast<uintptr_t>(a.mask) & 15) || a.mask_z % 4 != 0)) return false;
    if ((a.epi & TC_BIAS) && ((reinterpret_cast<uintptr_t>(a.bias) & 15) || a.bias_z % 4 != 0)) return false;
    // operands: any alignment (unaligned ones are staged with scalar loads), but batches must keep the alignment class
    if (a.a_z % 4 != 0 || a.b_z % 4 != 0) return false;
    return true;
}

int tc_gemm_launch(const TcGemm& in, int nz, cudaStream_t st) {
    TcGemm a = in;
    a.NT = choose_nt(a.N, a.M, nz, (a.epi & TC_LN) != 0);
    if (a.NT == 0 || !tc_gemm_supported(a)) { set_error("tc_gemm: shape / alignment not supported"); return CHROMO_EINVAL; }
    const size_t smem = gemm_smem(a.NT);
    static size_t configured = 0;
    if (smem > configured) {
        cudaError_t e = cudaFuncSetAttribute(tc_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_smem(256));
        if (e != cudaSuccess) { set_error("tc_gemm smem attribute: %s", cudaGetErrorString(e)); return CHROMO_ECUDA; }
        configured = gemm_smem(256);
    }
    // a long contraction on a handful of row tiles (the data gradient of the fused q|k|v|gate projection, K = 1024; the
    // position-table products over n = 400 bins): split it over CTAs until every SM has one.  Partial tiles are added
    // with FP32 atomics: to the output itself when the call accumulates in place, to a zeroed output otherwise.
    a.ksplit = 1;
    const int chunks = (a.Kc + TG_KCH - 1) / TG_KCH;
    if (chunks >= 4 && (a.epi & ~TC_RES) == 0 && a.c_div == 1 && a.c_mul == 1 && a.c_add == 0) {
        const bool in_place = (a.epi & TC_RES) && a.res == a.C && a.ldres == a.ldc && a.res_z == a.c_z && a.res_div == 1;
        const int ctas = (a.N / a.NT) * ((a.M + 127) / 128) * nz;
        int ks = 1;
        while (ks * 2 <= chunks / 2 && ctas * ks * 2 <= 160) ks *= 2;
        const int per = (chunks + ks - 1) / ks;
        if (ks > 1 && per * (ks - 1) < chunks && (in_place || a.ldc == a.N)) {
            if (in_place) {
                a.epi &= ~TC_RES;
            } else if (cudaMemset2DAsync(a.C, (size_t)(nz > 1 ? a.c_z : (long long)a.M * a.N) * sizeof(float), 0,
                                         (size_t)a.M * a.N * sizeof(float), nz, st) != cudaSuccess) {
                set_error("tc_gemm: cannot zero the split-K output");
                return CHROMO_ECUDA;
            }
            a.ksplit = ks;
        }
    }
    dim3 grid(a.N / a.NT, (a.M + 127) / 128, nz * a.ksplit);
    {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = grid; cfg.blockDim = dim3(TG_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
        cfg.attrs = attr; cfg.numAttrs = 1;
        long long* tb = g_tg_trace ? g_tg_trace + 2048 : nullptr;
        cudaError_t e = cudaLaunchKernelEx(&cfg, tc_gemm_kernel, a, tb);
        if (e != cudaSuccess) { set_error("tc_gemm launch: %s", cudaGetErrorString(e)); return CHROMO_ECUDA; }
    }
    CHROMO_CHECK_LAUNCH("tc_gemm");
    return CHROMO_OK;
}

void WgradQueue::add_weight(const float* dY, int ldy, long long dy_z, const float* X, int ldx, int x_div, long long x_z,
                            float* dW, int lddw, long long dw_z, int tokens, int N, int K, int nz) {
    for (int z = 0; z < nz; ++z)
        for (int m0 = 0; m0 < N; m0 += 128)
            for (int n0 = 0; n0 < K; n0 += WG_NT_MAX) {
                WgItem w;
                w.A = dY + z * dy_z + m0; w.B = X + z * x_z + n0; w.C = dW + z * dw_z + (long long)m0 * lddw + n0;
                w.lda = ldy; w.ldb = ldx; w.ldc = lddw; w.tokens = tokens;
                w.m_rows = (short)std::min(128, N - m0); w.n_cols = (short)std::min(WG_NT_MAX, K - n0);
                w.b_div = (short)x_div; w.kind = 0;
                items_.push_back(w);
            }
}

void WgradQueue::add_bias(const float* dY, int ld, long long dy_z, float* db, long long db_z, int tokens, int N, int nz) {
    for (int z = 0; z < nz; ++z)
        for (int n0 = 0; n0 < N; n0 += TG_THREADS) {
            WgItem w;
            w.A = dY + z * dy_z + n0; w.B = nullptr; w.C = db + z * db_z + n0;
            w.lda = ld; w.ldb = 0; w.ldc = 0; w.tokens = tokens;
            w.m_rows = 0; w.n_cols = (short)std::min(TG_THREADS, N - n0); w.b_div = 1; w.kind = 1;
            items_.push_back(w);
        }
}

int WgradQueue::flush(cudaStream_t st, int max_ctas) {
    if (items_.empty()) return CHROMO_OK;
    // A CTA owns its output tile for the whole launch (plain read-modify-write).  Tiles are either disjoint or
    // identical; the few tensors that receive several products (dW_in: three) take theirs with FP32 atomics instead.
    std::vector<std::vector<WgItem>> waves;
    {
        std::unordered_map<const float*, int> uses;
        uses.reserve(items_.size() * 2);
        for (const WgItem& w : items_) ++uses[w.C];
        for (WgItem w : items_) {
            if (uses[w.C] > 1) w.kind |= 2;
            if (waves.empty() || (int)waves.back().size() >= WG_MAX_ITEMS) waves.emplace_back();
            waves.back().push_back(w);
        }
    }
    items_.clear();
    static bool configured = false;
    const size_t smem = gemm_smem(WG_NT_MAX);
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(wgrad_grouped_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) { set_error("wgrad smem attribute: %s", cudaGetErrorString(e)); return CHROMO_ECUDA; }
        configured = true;
    }
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms < 1) sms = 148;
    }
    for (std::vector<WgItem>& wave : waves) {
        std::stable_sort(wave.begin(), wave.end(), [](const WgItem& x, const WgItem& y) {
            const long long cx = (x.kind & 1) ? x.tokens / 8 : (long long)x.tokens * (128 + x.n_cols);
            const long long cy = (y.kind & 1) ? y.tokens / 8 : (long long)y.tokens * (128 + y.n_cols);
            return cx > cy;
        });
        WgTable tbl;
        tbl.n = (int)wave.size();
        std::copy(wave.begin(), wave.end(), tbl.items);
        const int grid = std::min(tbl.n, max_ctas > 0 ? std::min(max_ctas, sms) : sms);
        wgrad_grouped_kernel<<<grid, TG_THREADS, smem, st>>>(tbl, g_tg_trace ? g_tg_trace + 3072 : nullptr);
        CHROMO_CHECK_LAUNCH("wgrad_grouped");
    }
    return CHROMO_OK;
}

}  // namespace chromo

// C ABI: the general contraction of the training step (see include/chromoformer_b200.h)
extern "C" int chromo_matmul(const float* A, int64_t lda, int32_t a_transposed, const float* B, int64_t ldb, int32_t b_transposed,
                             float* C, int64_t ldc, int32_t M, int32_t N, int32_t K, int32_t accumulate, int32_t ksplit,
                             void* stream) {
    using namespace chromo;
    (void)ksplit;
    if (!A || !B || !C || M < 1 || N < 1 || K < 1) { set_error("chromo_matmul: bad argument"); return CHROMO_EINVAL; }
    if (accumulate && a_transposed && b_transposed) {
        // the weight-gradient form runs through the deferred queue's kernel: tiles of 128 x 256 with their own accumulate
        WgradQueue q;
        q.add_weight(A, (int)lda, 0, B, (int)ldb, 1, 0, C, (int)ldc, 0, K, M, N, 1);
        return q.flush((cudaStream_t)stream);
    }
    TcGemm a = tc_gemm_args();
    a.A = A; a.lda = lda; a.a_t = a_transposed ? 1 : 0;
    a.B = B; a.ldb = ldb; a.b_t = b_transposed ? 1 : 0;
    a.C = C; a.ldc = ldc; a.M = M; a.N = N; a.Kc = K;
    if (accumulate) { a.epi |= TC_RES; a.res = C; a.ldres = ldc; }
    if (!tc_gemm_supported(a)) { set_error("chromo_matmul: shape / alignment not supported by the tensor-core path"); return CHROMO_EINVAL; }
    return tc_gemm_launch(a, 1, (cudaStream_t)stream);
}
