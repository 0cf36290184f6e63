// Regulation-transformer layers (modules.py:28-30,37-88,100-101 with gate=True) as ONE kernel: one layer or all of them.
//
// A CTA owns a tile of G genes (G*S <= 128 token rows) from the first layer of the launch to the last (the tokens of a
// gene only attend to each other); activations never leave the SM inside a layer, and between layers only the FP32
// residual rows go out, to a scratch slot that stays in L2:
//
//   X (FP32, HBM) -> BF16 A-operand in shared memory
//   per layer, for each pair of heads t = 0..3:
//       [q|k] and [v|gate] = X W^T          2 x (8 tcgen05.mma 128x128x16) -> TMEM
//       S = Q K^T on the tensor pipe (q, k in BF16), block-diagonal over the genes of the tile -> TMEM;
//       gamma*freq bias, mask(-1e9), softmax over the gene's own S keys -> P (BF16, TMEM);
//       O = P V on the tensor pipe -> sigmoid gate -> BF16 into the out-proj A-operand
//   out-proj (K = 256, two chunks) -> TMEM -> + bias + residual X -> LayerNorm -> U (registers + BF16 operand)
//   FFN-1 (N = 256, two chunks)    -> TMEM -> + bias, ReLU -> BF16 operand
//   FFN-2 (K = 256, two chunks)    -> TMEM -> + bias + U -> LayerNorm -> Y (next layer's operand; FP32, HBM, coalesced)
//
// The 14 weight chunks of a layer ([128 x 128] BF16 each, 448 KB, pre-packed in consumption
// order by pack_reg_stream) are streamed through a 3-deep ring of 32 KB stages by 1-D TMA bulk
// copies.  Warps 0..15 compute (attention, TMEM epilogues), warp 16 issues the dense tcgen05.mma, warp 17 loads the
// weight stream, warps 18 and 19 issue S = Q K^T and O = P V of one head each.  mbarriers carry every hand-off.
// Under a ragged plan (ragged.cu) a tile holds genes of one token class with their live tokens only.
#include "common.cuh"
#include "kernels.cuh"
#include "reg_fused.cuh"
#include "umma_ptx.cuh"

namespace chromo {

namespace {

constexpr int RF_NSTAGE = 3;
constexpr int RF_CHUNK_ELEMS = 128 * 128;
constexpr uint32_t RF_CHUNK_BYTES = RF_CHUNK_ELEMS * 2;
constexpr int RF_NCHUNK = 14;

// shared-memory map (bytes)
constexpr uint32_t OFF_XB = 0;                              // [128 x 128] BF16 operand (X, later U)
constexpr uint32_t OFF_ATT = 32768;                         // [128 x 256] BF16 operand (att, later F, later store staging)
constexpr uint32_t OFF_STAGE = OFF_ATT + 65536;             // 3 x 32 KB weight ring
constexpr uint32_t OFF_K = OFF_STAGE + RF_NSTAGE * RF_CHUNK_BYTES;   // k of the two heads in flight (BF16, K-major, 8 KB each)
constexpr uint32_t OFF_V = OFF_K + 16384;                   // v of the two heads in flight (BF16, MN-major, 8 KB each)
constexpr uint32_t OFF_CTL = OFF_V + 16384;                 // mbarriers + TMEM slot
constexpr uint32_t OFF_ROWMAP = OFF_CTL + 256;              // ragged plan: [B*S, 128]-layout row of every tile row (128 ints)
constexpr uint32_t RF_SMEM = OFF_ROWMAP + 512;
static_assert(RF_SMEM <= 227 * 1024, "shared memory budget");

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void warp_arrive(uint64_t* bar, int lane) {
    __syncwarp();
    if (lane == 0) mbar_arrive(bar);
}

// sigmoid(g) = 0.5 + 0.5 tanh(g / 2): one MUFU (tanh.approx, abs. error 2^-11, well inside the
// BF16 rounding of the result) instead of ex2 + rcp.  (Rows past the tile's last gene carry finite garbage that only
// reaches their own, never stored, output rows.)
__device__ __forceinline__ float gate_factor(float g) {
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * g));
    return fmaf(0.5f, t, 0.5f);
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}
// byte offset of the 16-byte chunk holding columns [8*kc, 8*kc+8) of `row` in a K-major operand of K columns
__device__ __forceinline__ uint32_t op_chunk(int row, int kc, int K) {
    return (uint32_t)(row >> 3) * (uint32_t)(K * 16) + (uint32_t)kc * 128u + (uint32_t)(row & 7) * 16u;
}

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        :
        : "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
          "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t* r) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        :
        : "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
          "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
          "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
          "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
// A operand in TMEM (lane = row, two BF16 per 32-bit column), B in shared memory
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        :
        : "r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// P row of one (token, head) as packed BF16 pairs for the 64-key window that starts at the warp's first
// gene (rounded down to an even key): entry m holds keys 2m, 2m+1 of the window; only the S keys of the
// thread's own gene (candidate index c relative to the warp's first gene) are non-zero.  The S probabilities are
// packed once in both alignments (gene starting on an even / odd key of the window); a candidate then only decides
// WHICH run of packed registers receives them: one select per (candidate, packed register).
template <int S, int NC, int PAR>
__device__ __forceinline__ void build_p_window(const float* p, int c, uint32_t* W) {
    constexpr int NE = (S + 1) / 2, NO = S / 2 + 1;
    uint32_t ev[NE], od[NO];
#pragma unroll
    for (int i = 0; i < NE; ++i) ev[i] = pack2(p[2 * i], 2 * i + 1 < S ? p[2 * i + 1] : 0.f);
#pragma unroll
    for (int i = 0; i < NO; ++i) od[i] = pack2(i > 0 ? p[2 * i - 1] : 0.f, 2 * i < S ? p[2 * i] : 0.f);
#pragma unroll
    for (int m = 0; m < 32; ++m) W[m] = 0u;
#pragma unroll
    for (int cc = 0; cc < NC; ++cc) {
        constexpr int dummy = 0; (void)dummy;
        const int base = cc * S + PAR;                        // first key of candidate cc's gene inside the window
        const bool mine = c == cc;
        if (base % 2 == 0) {
#pragma unroll
            for (int i = 0; i < NE; ++i)
                if (base / 2 + i < 32) W[base / 2 + i] = mine ? ev[i] : W[base / 2 + i];
        } else {
#pragma unroll
            for (int i = 0; i < NO; ++i)
                if (base / 2 + i < 32) W[base / 2 + i] = mine ? od[i] : W[base / 2 + i];
        }
    }
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// Compute warps.  TMEM lane quarter lq = warp & 3 (hardware rule); role = warp >> 2:
//   role 0, 1  "score" warps of the two heads in flight (ch = role & 1): q -> BF16 A operand in TMEM, k -> shared,
//              issue S = Q K^T, softmax on the gene's own S keys, P -> BF16 A operand in TMEM, issue O = P V;
//   role 2, 3  "value" warps of the same two heads: v -> shared (MN-major), sigmoid(gate) kept in registers,
//              O -> gate -> BF16 out-projection operand.
// The two kinds of warps work on the SAME rows a head pair apart from each other in time: while the value warps gate
// O(t), the score warps already repack q / k of pair t+1 — a software pipeline over the four head pairs of a layer.
// In the epilogue phases (out-projection + LayerNorm, FFN-1, FFN-2 + LayerNorm) role = column quarter: every row is
// served by four threads, 32 columns each (64 of the 256 FFN-1 columns), and FFN-1 / FFN-2 are chained per half of the
// hidden width, so that one half's bias + ReLU epilogue runs under the other half's MMAs.
constexpr int RF_THREADS = 640;            // 16 compute warps + dense-MMA issuer + weight loader + 2 attention issuers
enum { C_FULL0 = 0, C_FREE0 = 3, C_XREADY = 6, C_ATTREADY, C_UREADY, C_FREADY0, C_FREADY1, C_ACCQ, C_ACCVG, C_ACCO, C_ACCF1A,
       C_ACCF1B, C_ACCF2, C_OFREE, C_SR0, C_OR0 = C_SR0 + 2, C_QKS0 = C_OR0 + 2, C_PST0 = C_QKS0 + 2,
       C_VR0 = C_PST0 + 2, C_COUNT = C_VR0 + 2 };
static_assert(C_COUNT * 8 + 8 <= 256, "control block");

// timeline hook: traced threads of CTA (0,0) (dense issuer, one score warp, one value warp) append
// (event id << 48 | clock64) to their own 512-entry lane of a.trace
// (compiled out of the production instantiation: the test of `p` alone, made by every thread at every hand-off, was 7 % of
// the kernel's issued warp instructions)
template <bool ON>
struct Tracer {
    long long* p; int n;
    __device__ __forceinline__ void operator()(int id) {
        if (ON) {
            if (p && n < 512) { p[n++] = ((long long)id << 48) | (clock64() & 0xFFFFFFFFFFFFll); }
        }
    }
};
__device__ __forceinline__ void all_compute_barrier() { asm volatile("bar.sync 1, 512;" ::: "memory"); }
// the four warps that share a TMEM lane quarter (the four column quarters of the same 32 rows)
__device__ __forceinline__ void quarter_barrier(int lq) { asm volatile("bar.sync %0, 128;" ::"r"(4 + lq) : "memory"); }

// Score warps of one layer's attention (four head pairs): scores of a row against the S keys of its own gene -> softmax
// -> P (BF16) over the S tile.  S = tokens per gene in this tile (compile time: the window arithmetic below).
template <int S, int SMAX, bool TRACE>
__device__ __forceinline__ void score_rows(uint64_t* bars, uint32_t trow, int ch, int lq, int lane, int gl, const float* fr,
                                           unsigned mbits, const float* gam, Tracer<TRACE>& tr) {
    const float scale = 0.17677669529663687f;            // 1/sqrt(32)
    {
            // a window of the S tile that starts at the first gene touched by this warp (register indices stay
            // compile-time, the column is warp-uniform)
            constexpr int NC = (31 + S - 1) / S + 1;             // genes a 32-row warp can touch
            constexpr int NW = NC * S;                            // window width in keys (<= 64)
            const int g_lo = (32 * lq) / S;
            const int cand = gl - g_lo;                           // 0 .. NC-1
#pragma unroll 1
            for (int t = 0; t < 4; ++t) {
                const float gamma = t == 0 ? gam[0] : t == 1 ? gam[1] : t == 2 ? gam[2] : gam[3];
                float w[64];
                mbar_wait(&bars[C_SR0 + ch], t & 1);
                tr(24);
                tc_fence_after();
                {
                    const uint32_t sc0 = trow + 128 * ch + S * g_lo;
                    if (NW > 48) tmem_ld32_pair(sc0, w, sc0 + 32, w + 32);
                    else { tmem_ld32(sc0, w); tmem_ld16(sc0 + 32, w + 32); }
                }
                tc_fence_before();
                {   // zeros over the P columns of the tile while the scores are being reduced
                    uint32_t Z[32];
#pragma unroll
                    for (int m = 0; m < 32; ++m) Z[m] = 0u;
                    tmem_st32(trow + 128 * ch, Z);
                    tmem_st32(trow + 128 * ch + 32, Z);
                }
                float s[S];
                float mx = -INFINITY;
#pragma unroll
                for (int j = 0; j < S; ++j) {
                    float sc = w[j];
#pragma unroll
                    for (int c = 1; c < NC; ++c)
                        if (cand == c) sc = w[c * S + j];
                    sc = fmaf(gamma, fr[j], sc * scale);
                    if ((mbits >> j) & 1u) sc = -1e9f;
                    s[j] = sc;
                    mx = fmaxf(mx, sc);
                }
                float sum = 0.f;
#pragma unroll
                for (int j = 0; j < S; ++j) { s[j] = __expf(s[j] - mx); sum += s[j]; }
                const float inv = 1.f / sum;
#pragma unroll
                for (int j = 0; j < S; ++j) s[j] *= inv;
                {   // P (BF16 pairs) over the first 64 columns of the S tile: this warp's window over the zeros
                    uint32_t W[32];
                    const int kb = S * g_lo;
                    if (kb & 1) build_p_window<S, NC, 1>(s, cand, W);
                    else build_p_window<S, NC, 0>(s, cand, W);
                    tmem_st_wait();                                 // (the zeros have landed)
                    tmem_st32(trow + 128 * ch + (kb >> 1), W);
                    tmem_st_wait();
                    tc_fence_before();
                    warp_arrive(&bars[C_PST0 + ch], lane);          // P(t) of this warp's rows is in place
                    tr(25);
                }
            }
    }
}

// the token classes below SMAX (ragged plan): real calls, so that their window arithmetic does not weigh on the register
// allocation of the full-size class
template <int S, int SMAX, bool TRACE>
__device__ __noinline__ void score_rows_call(uint64_t* bars, uint32_t trow, int ch, int lq, int lane, int gl, const float* fr,
                                             unsigned mbits, const float* gam, Tracer<TRACE>& tr) {
    score_rows<S, SMAX, TRACE>(bars, trow, ch, lq, lane, gl, fr, mbits, gam, tr);
}

template <int SMAX, bool TRACE, bool PLAN>
__global__ void __launch_bounds__(RF_THREADS, 1) reg_layer_fused_kernel(const RegFusedArgs a) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_CTL);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + C_COUNT);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int z = blockIdx.y, tile = blockIdx.x;
    // tokens per gene in this tile: SMAX, or the tile's token class under a ragged plan (then the tile's rows are gathered
    // through `rowmap`: row of the [B*SMAX, 128] layout per tile row)
    int S = SMAX, G = a.G;
    long long row0 = (long long)tile * G * S;                  // first token row of this tile (without a plan)
    int rows_valid = min((long long)G * S, (long long)a.B * S - row0);
    const int* rowmap = reinterpret_cast<const int*>(smem + OFF_ROWMAP);
    if (PLAN) {
        int r = 0;
        if (tid < 128) r = __ldg(a.plan_rows + tile * 128 + tid);   // (both loads in flight)
        const int4 tt = __ldg(a.plan_tiles + tile);
        if (tt.y == 0) return;                                // (the grid is an upper bound)
        G = tt.y; S = tt.z; rows_valid = G * S; row0 = 0;
        if (tid < 128) reinterpret_cast<int*>(smem + OFF_ROWMAP)[tid] = r;
    }

    if (warp == 0) tmem_alloc(tmem_slot, 512);
    if (tid == 0) {
        for (int i = 0; i < RF_NSTAGE; ++i) { mbar_init(&bars[C_FULL0 + i], 1); mbar_init(&bars[C_FREE0 + i], 1); }
        mbar_init(&bars[C_XREADY], 16); mbar_init(&bars[C_ATTREADY], 8); mbar_init(&bars[C_UREADY], 16);
        mbar_init(&bars[C_FREADY0], 8); mbar_init(&bars[C_FREADY1], 8);
        mbar_init(&bars[C_ACCQ], 1); mbar_init(&bars[C_ACCVG], 1); mbar_init(&bars[C_ACCO], 1);
        mbar_init(&bars[C_ACCF1A], 1); mbar_init(&bars[C_ACCF1B], 1); mbar_init(&bars[C_ACCF2], 1);
        mbar_init(&bars[C_OFREE], 8);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bars[C_SR0 + i], 1); mbar_init(&bars[C_OR0 + i], 1);
            mbar_init(&bars[C_QKS0 + i], 4); mbar_init(&bars[C_PST0 + i], 4); mbar_init(&bars[C_VR0 + i], 4);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 17) {
        // ===================================================== loader: weight stream through the 3-stage ring ====
        if (lane == 0) {
            const __nv_bfloat16* wsrc = a.wstream + z * a.w_z;
            const int n_chunks = RF_NCHUNK * a.n_layers;   // the layers' chunks follow each other in the stream
            for (int c = 0; c < n_chunks; ++c) {
                const int st = c % RF_NSTAGE;
                if (c >= RF_NSTAGE) mbar_wait(&bars[C_FREE0 + st], ((c / RF_NSTAGE) - 1) & 1);
                mbar_expect_tx(&bars[C_FULL0 + st], RF_CHUNK_BYTES);
                tma_bulk_g2s(smem + OFF_STAGE + st * RF_CHUNK_BYTES, wsrc + (long long)c * RF_CHUNK_ELEMS, RF_CHUNK_BYTES,
                             &bars[C_FULL0 + st]);
            }
        }
    } else if (warp >= 18) {
        // ===================================================== attention issuers: S = Q K^T and O = P V of one head each ====
        // The order per head is fixed - S(0), O(0), S(1), O(1), ... (S(t+1) overwrites the tile P(t) sits in, so it has to
        // follow O(t) in the in-order tensor pipe) - so a dedicated thread per head simply blocks on the hand-offs in that
        // order; nothing else competes for its instruction slots.
        if (lane == 0) {
            const int ch = warp - 18;
            const uint64_t k_d = umma_smem_desc(smem_u32(smem + OFF_K) + ch * 8192, 128, 512);
            const uint64_t v_d = umma_smem_desc(smem_u32(smem + OFF_V) + ch * 8192, 128, 2048);
            const uint32_t idesc_s = umma_idesc_bf16(128, 128), idesc_o = umma_idesc_bf16(128, 32) | (1u << 16);   // O: B MN-major
            const int n_steps = 4 * a.n_layers;
            for (int i = 0; i < n_steps; ++i) {
                const uint32_t par = i & 1;
                mbar_wait(&bars[C_QKS0 + ch], par);                        // q (TMEM, BF16) and k (shared) of this pair staged
                tc_fence_after();
#pragma unroll
                for (int k = 0; k < 2; ++k)
                    umma_bf16_ts(tmem + 128 * ch, tmem + 256 + 32 * ch + 8 * k, k_d + 16 * k, idesc_s, k > 0 ? 1u : 0u);
                umma_commit(&bars[C_SR0 + ch]);
                mbar_wait(&bars[C_PST0 + ch], par);                        // P stored by the score warps
                mbar_wait(&bars[C_VR0 + ch], par);                         // V staged by the value warps
                tc_fence_after();
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    umma_bf16_ts(tmem + 384 + 32 * ch, tmem + 128 * ch + 8 * k, v_d + 16 * k, idesc_o, k > 0 ? 1u : 0u);
                umma_commit(&bars[C_OR0 + ch]);
            }
        }
    } else if (warp == 16) {
        // ===================================================== dense issuer: projections, out-projection, FFN ====
        if (lane == 0) {
            const uint32_t idesc = umma_idesc_bf16(128, 128);
            const uint32_t s_xb = smem_u32(smem + OFF_XB), s_att = smem_u32(smem + OFF_ATT);
            const uint64_t xd = umma_smem_desc(s_xb, 128, 2048), attd = umma_smem_desc(s_att, 128, 4096);
            const uint64_t stage_d = umma_smem_desc(smem_u32(smem + OFF_STAGE), 128, 2048);   // + st * 2048 per ring stage
            Tracer<TRACE> tr{(a.trace && tile == 0 && z == 0) ? a.trace : nullptr, 0};
            auto consume = [&](int c, uint64_t ad, uint32_t col, bool accumulate) {
                const int st = c % RF_NSTAGE;
                mbar_wait(&bars[C_FULL0 + st], (c / RF_NSTAGE) & 1);
                tc_fence_after();
                // descriptors by plain adds (+256 B = +16 in the address field): building them per MMA costs the issuing
                // thread ~120 cycles per instruction against the 64-cycle MMA (tools/bench_micro/mma_rate.cu)
                const uint64_t bd = stage_d + 2048 * st;
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    umma_bf16(tmem + col, ad + 16 * k, bd + 16 * k, idesc, (accumulate || k > 0) ? 1u : 0u);
                umma_commit(&bars[C_FREE0 + st]);                           // (the loader warp refills the stage)
            };
            for (int li = 0; li < a.n_layers; ++li) {
                const int cb = li * RF_NCHUNK;
                const uint32_t lp = li & 1;
                mbar_wait(&bars[C_XREADY], lp);
                tr(1);
                // TMEM [0,128) / [128,256): S, then P (first 64..77 columns) of the two heads in flight; [256,512): projection
                // pair (q0 q1 k0 k1 v0 v1 g0 g1, 32 columns each); O = P V of a head lands in the (by then dead) v columns of
                // that head, so the S tile is free for the next pair's scores as soon as O has been ISSUED (the tensor pipe
                // runs in order).  The next [q | k] goes out when S is done with q / k (the issuer watches the S commit barriers
                // itself), the next [v | gate] when O has been read out of the v columns.
                consume(cb, xd, 256, false);
                umma_commit(&bars[C_ACCQ]);
                tr(2);
                consume(cb + 1, xd, 384, false);
                umma_commit(&bars[C_ACCVG]);
                tr(3);
                for (int t = 0; t < 3; ++t) {
                    mbar_wait(&bars[C_SR0], t & 1);                         // S(t) of both heads complete: q / k columns are dead
                    mbar_wait(&bars[C_SR0 + 1], t & 1);
                    tr(4);
                    consume(cb + 2 * t + 2, xd, 256, false);                // next [q | k]
                    umma_commit(&bars[C_ACCQ]);
                    tr(2);
                    mbar_wait(&bars[C_OFREE], t & 1);
                    tr(5);
                    consume(cb + 2 * t + 3, xd, 384, false);                // next [v | gate]
                    umma_commit(&bars[C_ACCVG]);
                    tr(3);
                }
                mbar_wait(&bars[C_ATTREADY], lp);
                tr(6);
                consume(cb + 8, attd, 0, false);                            // out-projection, K halves
                consume(cb + 9, attd + 128, 0, true);
                umma_commit(&bars[C_ACCO]);
                tr(7);
                mbar_wait(&bars[C_UREADY], lp);
                tr(8);
                consume(cb + 10, xd, 256, false);                           // FFN-1, hidden half A
                umma_commit(&bars[C_ACCF1A]);
                consume(cb + 11, xd, 384, false);                           // FFN-1, hidden half B
                umma_commit(&bars[C_ACCF1B]);
                tr(9);
                mbar_wait(&bars[C_FREADY0], lp);
                consume(cb + 12, attd, 0, false);                           // FFN-2 over hidden half A
                mbar_wait(&bars[C_FREADY1], lp);
                consume(cb + 13, attd + 128, 0, true);                      // ... + half B
                umma_commit(&bars[C_ACCF2]);
                tr(12);
            }   // layers
        }
    } else {
        // ===================================================== compute warps =================
        const int lq = warp & 3, role = warp >> 2;
        const int ch = role & 1;                             // head of the pair (attention)
        const bool score_warp = role < 2;
        const int cq = role;                                 // column quarter (epilogues)
        const int row = lq * 32 + lane;                      // tile row == TMEM lane
        const bool valid = row < rows_valid;
        const long long grow = PLAN ? (long long)rowmap[row] : row0 + row;   // row of the [B*SMAX, 128] layout
        const uint32_t trow = tmem + ((uint32_t)(lq * 32) << 16);
        const float* X = a.x + z * a.x_z;
        float v[32];
        // Parking block of the FP32 residual rows between layers: the block of this SM (one CTA per SM is resident, so the
        // same 148 x 64 KB per slot are written and read back by tile after tile and stay in L2) when the slot has that many
        // blocks, else the tile's own.  (Read where it is used: a value held across the layers costs a register there.)
        auto park_block = [&]() -> long long {
            int idx = tile;
            if (a.park_by_sm) asm volatile("mov.u32 %0, %%smid;" : "=r"(idx));
            return (long long)idx * 4096;
        };

        // ---- phase 0 (first layer only; later layers get their operand from phase 4): X -> BF16 operand
        {
            float4 x[4][2];                                   // all 8 loads of the thread in flight at once
            int r_[4], kc_[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int u = warp + q * 16;                  // 64 (8-row group, 4-chunk group) items
                r_[q] = (u & 15) * 8 + (lane >> 2);
                kc_[q] = (u >> 4) * 4 + (lane & 3);
                x[q][0] = x[q][1] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (r_[q] < rows_valid) {
                    const float* p = X + (PLAN ? (long long)rowmap[r_[q]] : row0 + r_[q]) * 128 + kc_[q] * 8;
                    x[q][0] = __ldg(reinterpret_cast<const float4*>(p));
                    x[q][1] = __ldg(reinterpret_cast<const float4*>(p + 4));
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                uint4 pk;
                pk.x = pack2(x[q][0].x, x[q][0].y); pk.y = pack2(x[q][0].z, x[q][0].w);
                pk.z = pack2(x[q][1].x, x[q][1].y); pk.w = pack2(x[q][1].z, x[q][1].w);
                *reinterpret_cast<uint4*>(smem + OFF_XB + op_chunk(r_[q], kc_[q], 128)) = pk;
            }
            fence_async_smem();
            warp_arrive(&bars[C_XREADY], lane);
        }

        const int gl = row / S;                               // gene within tile
        float fr[SMAX];
        unsigned mbits = 0;
        if (score_warp) {
            // (grow = gene * SMAX + query token: row `grow` of the [B, SMAX, SMAX] bias and mask tensors)
            const float* freq = a.freq + (valid ? grow * SMAX : 0);
            const uint8_t* mask = a.imask[z] + (valid ? grow * SMAX : 0);
#pragma unroll
            for (int j = 0; j < SMAX; ++j) {
                fr[j] = 0.f;
                if (valid && j < S) {
                    fr[j] = freq[j];
                    if (mask[j]) mbits |= 1u << j;
                }
            }
        }
        uint8_t* sk = smem + OFF_K + ch * 8192;
        uint8_t* sv = smem + OFF_V + ch * 8192;
        const uint32_t pb = trow + 256;
        // traced threads: warp 0 lane 0 (score warp, lane 1 of the buffer), warp 8 lane 0 (value warp, lane 2)
        Tracer<TRACE> tr{(a.trace && tile == 0 && z == 0 && lane == 0 && (warp == 0 || warp == 8)) ? a.trace + (warp == 0 ? 512 : 1024) : nullptr, 0};

        for (int li = 0; li < a.n_layers; ++li) {
        const uint32_t lp = li & 1;
        const long long po = z * a.p_z + li * a.p_l;          // this (resolution, layer)'s parameters

        // ---- phase 1: attention, four head pairs.  Score warps: scores of a row against the S keys of its own gene ->
        // softmax -> P; value warps: operand staging (q, k, v), sigmoid(gate), O -> gated out-projection operand.
        if (score_warp) {
            float gam[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) gam[t] = a.gamma_f[po + 2 * t + ch];
            if (!PLAN) score_rows<SMAX, SMAX, TRACE>(bars, trow, ch, lq, lane, gl, fr, mbits, gam, tr);
            else {
                // one instantiation per token class of the plan (the window arithmetic wants S at compile time)
                switch (S) {
                    case 1: score_rows_call<1, SMAX, TRACE>(bars, trow, ch, lq, lane, gl, fr, mbits, gam, tr); break;
                    case 2: score_rows_call<2, SMAX, TRACE>(bars, trow, ch, lq, lane, gl, fr, mbits, gam, tr); break;
                    case 3: score_rows_call<3, SMAX, TRACE>(bars, trow, ch, lq, lane, gl, fr, mbits, gam, tr); break;
                    case 4: score_rows_call<4, SMAX, TRACE>(bars, trow, ch, lq, lane, gl, fr, mbits, gam, tr); break;
                    case 5: score_rows_call<5, SMAX, TRACE>(bars, trow, ch, lq, lane, gl, fr, mbits, gam, tr); break;
                    case 6: score_rows_call<6, SMAX, TRACE>(bars, trow, ch, lq, lane, gl, fr, mbits, gam, tr); break;
                    case 7: score_rows_call<7, SMAX, TRACE>(bars, trow, ch, lq, lane, gl, fr, mbits, gam, tr); break;
                    case 8: score_rows_call<8, SMAX, TRACE>(bars, trow, ch, lq, lane, gl, fr, mbits, gam, tr); break;
                    case 9: if (SMAX > 9) score_rows_call<(SMAX >= 9 ? 9 : SMAX), SMAX, TRACE>(bars, trow, ch, lq, lane, gl, fr, mbits, gam, tr); else score_rows<(SMAX >= 9 ? 9 : SMAX), SMAX, TRACE>(bars, trow, ch, lq, lane, gl, fr, mbits, gam, tr); break;
                    default: score_rows<SMAX, SMAX, TRACE>(bars, trow, ch, lq, lane, gl, fr, mbits, gam, tr); break;
                }
            }
        } else {
            uint32_t gsig[16];
            auto stage_qk = [&](int t) {    // Q -> BF16 back into TMEM in place (A operand of S = Q K^T); K -> shared, K-major
                mbar_wait(&bars[C_ACCQ], t & 1);
                tr(20);
                tc_fence_after();
                uint32_t qp[16];
                float v2[32];
                tmem_ld32_pair(pb + 32 * ch, v, pb + 64 + 32 * ch, v2);    // q and k of this head, both loads in flight
#pragma unroll
                for (int c = 0; c < 16; ++c) qp[c] = pack2(v[2 * c], v[2 * c + 1]);
                tmem_st16(pb + 32 * ch, qp);
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    uint4 pk;
                    pk.x = pack2(v2[8 * c], v2[8 * c + 1]); pk.y = pack2(v2[8 * c + 2], v2[8 * c + 3]);
                    pk.z = pack2(v2[8 * c + 4], v2[8 * c + 5]); pk.w = pack2(v2[8 * c + 6], v2[8 * c + 7]);
                    *reinterpret_cast<uint4*>(sk + op_chunk(row, c, 32)) = pk;
                }
                tmem_st_wait();
                tc_fence_before();
                fence_async_smem();
                warp_arrive(&bars[C_QKS0 + ch], lane);
                tr(21);
            };
            auto stage_vg = [&](int t) {    // v -> shared, MN-major (B operand of O = P V); sigmoid(gate) kept as BF16 pairs
                mbar_wait(&bars[C_ACCVG], t & 1);
                tr(30);
                tc_fence_after();
                float v2[32];
                tmem_ld32_pair(pb + 128 + 32 * ch, v, pb + 192 + 32 * ch, v2);   // v and gate of this head
                tc_fence_before();
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    uint4 pk;
                    pk.x = pack2(v[8 * c], v[8 * c + 1]); pk.y = pack2(v[8 * c + 2], v[8 * c + 3]);
                    pk.z = pack2(v[8 * c + 4], v[8 * c + 5]); pk.w = pack2(v[8 * c + 6], v[8 * c + 7]);
                    *reinterpret_cast<uint4*>(sv + c * 2048 + (row >> 3) * 128 + (row & 7) * 16) = pk;
                }
                fence_async_smem();             // (V must be visible to the tensor pipe before O = P V is issued)
                warp_arrive(&bars[C_VR0 + ch], lane);
                tr(31);
#pragma unroll
                for (int c = 0; c < 16; ++c) gsig[c] = pack2(gate_factor(v2[2 * c]), gate_factor(v2[2 * c + 1]));
            };
            stage_qk(0);
            stage_vg(0);
#pragma unroll 1
            for (int t = 0; t < 4; ++t) {
                if (t < 3) stage_qk(t + 1);                         // (S(t) is complete once [q | k](t+1) has been projected)
                mbar_wait(&bars[C_OR0 + ch], t & 1);
                tr(32);
                tc_fence_after();
                float o[32];
                tmem_ld32(pb + 128 + 32 * ch, o);                 // O = P V (in this head's v columns)
                tc_fence_before();
                warp_arrive(&bars[C_OFREE], lane);                // the v columns may take the next [v | gate]
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    float r[8];
#pragma unroll
                    for (int e = 0; e < 8; e += 2) {
                        const uint32_t gp = gsig[4 * c + (e >> 1)];
                        const float2 g2 = make_float2(__uint_as_float(gp << 16), __uint_as_float(gp & 0xffff0000u));
                        const float2 r2 = __fmul2_rn(make_float2(o[8 * c + e], o[8 * c + e + 1]), g2);
                        r[e] = r2.x; r[e + 1] = r2.y;
                    }
                    uint4 pk;
                    pk.x = pack2(r[0], r[1]); pk.y = pack2(r[2], r[3]); pk.z = pack2(r[4], r[5]); pk.w = pack2(r[6], r[7]);
                    *reinterpret_cast<uint4*>(smem + OFF_ATT + op_chunk(row, 8 * t + 4 * ch + c, 256)) = pk;
                }
                tr(33);
                if (t < 3) stage_vg(t + 1);                         // O(t) is complete: V(t) may be overwritten
            }
            fence_async_smem();
            warp_arrive(&bars[C_ATTREADY], lane);
        }

        // residual rows of phase 2 (FP32), 32 columns per thread: issued now so that their latency hides behind the
        // out-projection MMA; u_keep then carries U and is the residual of phase 4.  First layer: the caller's row-major X.
        // Later layers: what THIS thread parked in the scratch slot at the end of the previous layer, in a lane-major order
        // (float4 index (cq*8 + j/4)*128 + row inside the tile's 64 KB block): every warp access is 512 contiguous bytes.
        float u_keep[32];
        if (li == 0) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                float4 r4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (valid) r4 = __ldg(reinterpret_cast<const float4*>(X + grow * 128 + 32 * cq + j));
                u_keep[j] = r4.x; u_keep[j + 1] = r4.y; u_keep[j + 2] = r4.z; u_keep[j + 3] = r4.w;
            }
        } else {
            const float4* park = reinterpret_cast<const float4*>(a.y_mid + z * a.y_mid_z + ((li - 1) & 1) * a.y_l) +
                                 park_block() + row;
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                const float4 r4 = __ldcg(park + (cq * 8 + (j >> 2)) * 128);
                u_keep[j] = r4.x; u_keep[j + 1] = r4.y; u_keep[j + 2] = r4.z; u_keep[j + 3] = r4.w;
            }
        }
        // small FP32 vectors of the layer -> shared (k, v are dead once every value warp has passed its last O):
        // bo, ln1w, ln1b, b2, ln2w, ln2b, b1[256]
        float* prm = reinterpret_cast<float*>(smem + OFF_V);
        {   // (global loads before the barrier, so that their latency hides behind it)
            const float* srcs[6] = {a.bo, a.ln1w, a.ln1b, a.b2, a.ln2w, a.ln2b};
            const int ct = warp * 32 + lane;                  // 0..511
            float pv[3] = {0.f, 0.f, 0.f};
#pragma unroll
            for (int k = 0; k < 6; ++k)
                if ((ct >> 7) == (k >> 1)) pv[k & 1] = __ldg(srcs[k] + po + (ct & 127));
            if (ct >= 256) pv[2] = __ldg(a.b1 + po + ct - 256);
            tr(40);
            all_compute_barrier();
            tr(41);
            if (ct < 384) { prm[(2 * (ct >> 7)) * 128 + (ct & 127)] = pv[0]; prm[(2 * (ct >> 7) + 1) * 128 + (ct & 127)] = pv[1]; }
            if (ct >= 256) prm[768 + ct - 256] = pv[2];
        }
        all_compute_barrier();
        // ---- phase 2: out-projection epilogue: + bias + residual, LayerNorm -> U
        float* red = reinterpret_cast<float*>(smem + OFF_K);  // [4][128][2] partial sums (k is dead)
        const int c0 = 32 * cq;
        {
            tr(42);
            mbar_wait(&bars[C_ACCO], lp);
            tr(43);
            tc_fence_after();
            const float* bo = prm;
            float sum = 0.f, sq = 0.f;
            tmem_ld32(trow + c0, v);
            tr(50);
            float2 sum2 = make_float2(0.f, 0.f), sq2 = make_float2(0.f, 0.f);      // packed FP32x2 math (sm_100)
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                const float4 b4 = *reinterpret_cast<const float4*>(bo + c0 + j);
                const float2 ta = __fadd2_rn(__fadd2_rn(make_float2(v[j], v[j + 1]), make_float2(b4.x, b4.y)),
                                             make_float2(u_keep[j], u_keep[j + 1]));
                const float2 tb = __fadd2_rn(__fadd2_rn(make_float2(v[j + 2], v[j + 3]), make_float2(b4.z, b4.w)),
                                             make_float2(u_keep[j + 2], u_keep[j + 3]));
                u_keep[j] = ta.x; u_keep[j + 1] = ta.y; u_keep[j + 2] = tb.x; u_keep[j + 3] = tb.y;
                sum2 = __fadd2_rn(sum2, __fadd2_rn(ta, tb));
                sq2 = __ffma2_rn(ta, ta, __ffma2_rn(tb, tb, sq2));
            }
            sum = sum2.x + sum2.y; sq = sq2.x + sq2.y;
            tc_fence_before();
            *reinterpret_cast<float2*>(red + (cq * 128 + row) * 2) = make_float2(sum, sq);
            tr(51);
            quarter_barrier(lq);
            tr(52);
            sum = 0.f; sq = 0.f;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float2 p2 = *reinterpret_cast<const float2*>(red + (k * 128 + row) * 2);
                sum += p2.x; sq += p2.y;
            }
            const float mean = sum * (1.f / 128.f);
            const float rstd = rsqrtf(fmaxf(sq * (1.f / 128.f) - mean * mean, 0.f) + 1e-5f);
            const float* lw = prm + 128;
            const float* lb = prm + 256;
            const float2 nm2 = make_float2(-mean, -mean), rs2 = make_float2(rstd, rstd);
#pragma unroll
            for (int j = 0; j < 32; j += 8) {
                float r[8];
#pragma unroll
                for (int e = 0; e < 8; e += 4) {
                    const float4 w4 = *reinterpret_cast<const float4*>(lw + c0 + j + e);
                    const float4 b4 = *reinterpret_cast<const float4*>(lb + c0 + j + e);
                    const float2 ra = __ffma2_rn(__fadd2_rn(make_float2(u_keep[j + e], u_keep[j + e + 1]), nm2),
                                                 __fmul2_rn(rs2, make_float2(w4.x, w4.y)), make_float2(b4.x, b4.y));
                    const float2 rb = __ffma2_rn(__fadd2_rn(make_float2(u_keep[j + e + 2], u_keep[j + e + 3]), nm2),
                                                 __fmul2_rn(rs2, make_float2(w4.z, w4.w)), make_float2(b4.z, b4.w));
                    r[e] = ra.x; r[e + 1] = ra.y; r[e + 2] = rb.x; r[e + 3] = rb.y;
                    u_keep[j + e] = ra.x; u_keep[j + e + 1] = ra.y; u_keep[j + e + 2] = rb.x; u_keep[j + e + 3] = rb.y;
                }
                uint4 pk;
                pk.x = pack2(r[0], r[1]); pk.y = pack2(r[2], r[3]); pk.z = pack2(r[4], r[5]); pk.w = pack2(r[6], r[7]);
                *reinterpret_cast<uint4*>(smem + OFF_XB + op_chunk(row, (c0 + j) >> 3, 128)) = pk;
            }
            tr(53);
            fence_async_smem();
            warp_arrive(&bars[C_UREADY], lane);
            tr(44);
        }

        // ---- phase 3: FFN-1 epilogue: + bias, ReLU -> BF16 operand (over the dead att tile); 64 hidden columns per thread,
        //      the two halves of the hidden width are committed (and handed to FFN-2) separately
        {
            mbar_wait(&bars[cq < 2 ? C_ACCF1A : C_ACCF1B], lp);
            tr(45);
            tc_fence_after();
            const float* b1 = prm + 768;
            const int h0 = 64 * cq;
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                // (one 32-column load at a time: with the residual row live next to it a pair does not fit the 96 registers)
                tmem_ld32(trow + 256 + h0 + 32 * half, v);
                const float* vv = v;
                const int c = h0 + 32 * half;
#pragma unroll
                for (int j = 0; j < 32; j += 8) {
                    float r[8];
#pragma unroll
                    for (int e = 0; e < 8; e += 4) {
                        const float4 b4 = *reinterpret_cast<const float4*>(b1 + c + j + e);
                        const float2 ra = __fadd2_rn(make_float2(vv[j + e], vv[j + e + 1]), make_float2(b4.x, b4.y));
                        const float2 rb = __fadd2_rn(make_float2(vv[j + e + 2], vv[j + e + 3]), make_float2(b4.z, b4.w));
                        r[e] = fmaxf(ra.x, 0.f); r[e + 1] = fmaxf(ra.y, 0.f); r[e + 2] = fmaxf(rb.x, 0.f); r[e + 3] = fmaxf(rb.y, 0.f);
                    }
                    uint4 pk;
                    pk.x = pack2(r[0], r[1]); pk.y = pack2(r[2], r[3]); pk.z = pack2(r[4], r[5]); pk.w = pack2(r[6], r[7]);
                    *reinterpret_cast<uint4*>(smem + OFF_ATT + op_chunk(row, (c + j) >> 3, 256)) = pk;
                }
            }
            tc_fence_before();
            fence_async_smem();
            warp_arrive(&bars[cq < 2 ? C_FREADY0 : C_FREADY1], lane);
            tr(46);
        }

        // ---- phase 4: FFN-2 epilogue: + bias + U, LayerNorm -> Y (coalesced through shared)
        {
            mbar_wait(&bars[C_ACCF2], lp);
            tr(47);
            tc_fence_after();
            const float* b2 = prm + 384;
            float* red2 = red + 1024;
            float sum = 0.f, sq = 0.f;
            tmem_ld32(trow + c0, v);
            float2 sum2 = make_float2(0.f, 0.f), sq2 = make_float2(0.f, 0.f);
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                const float4 b4 = *reinterpret_cast<const float4*>(b2 + c0 + j);
                const float2 ta = __fadd2_rn(__fadd2_rn(make_float2(v[j], v[j + 1]), make_float2(b4.x, b4.y)),
                                             make_float2(u_keep[j], u_keep[j + 1]));
                const float2 tb = __fadd2_rn(__fadd2_rn(make_float2(v[j + 2], v[j + 3]), make_float2(b4.z, b4.w)),
                                             make_float2(u_keep[j + 2], u_keep[j + 3]));
                u_keep[j] = ta.x; u_keep[j + 1] = ta.y; u_keep[j + 2] = tb.x; u_keep[j + 3] = tb.y;
                sum2 = __fadd2_rn(sum2, __fadd2_rn(ta, tb));
                sq2 = __ffma2_rn(ta, ta, __ffma2_rn(tb, tb, sq2));
            }
            sum = sum2.x + sum2.y; sq = sq2.x + sq2.y;
            tc_fence_before();
            *reinterpret_cast<float2*>(red2 + (cq * 128 + row) * 2) = make_float2(sum, sq);
            quarter_barrier(lq);
            sum = 0.f; sq = 0.f;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float2 p2 = *reinterpret_cast<const float2*>(red2 + (k * 128 + row) * 2);
                sum += p2.x; sq += p2.y;
            }
            const float mean = sum * (1.f / 128.f);
            const float rstd = rsqrtf(fmaxf(sq * (1.f / 128.f) - mean * mean, 0.f) + 1e-5f);
            const float* lw = prm + 512;
            const float* lb = prm + 640;
            const bool more = li + 1 < a.n_layers;
            {
                const float2 nm2 = make_float2(-mean, -mean), rs2 = make_float2(rstd, rstd);
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 w4 = *reinterpret_cast<const float4*>(lw + c0 + j);
                    const float4 b4 = *reinterpret_cast<const float4*>(lb + c0 + j);
                    const float2 ra = __ffma2_rn(__fadd2_rn(make_float2(u_keep[j], u_keep[j + 1]), nm2),
                                                 __fmul2_rn(rs2, make_float2(w4.x, w4.y)), make_float2(b4.x, b4.y));
                    const float2 rb = __ffma2_rn(__fadd2_rn(make_float2(u_keep[j + 2], u_keep[j + 3]), nm2),
                                                 __fmul2_rn(rs2, make_float2(w4.z, w4.w)), make_float2(b4.z, b4.w));
                    u_keep[j] = ra.x; u_keep[j + 1] = ra.y; u_keep[j + 2] = rb.x; u_keep[j + 3] = rb.y;
                }
            }
            if (more) {
                // Y is the next layer's operand (BF16, over X in shared memory) and residual (FP32, parked in the scratch
                // slot by the thread that will read it back, lane-major).  Operand first: the driver starts the next
                // layer's projections on C_XREADY while the rows are being parked.  (No CTA barrier is needed for prm / red:
                // nobody gets past the next all_compute_barrier before every warp has arrived there.)
#pragma unroll
                for (int j = 0; j < 32; j += 8) {
                    uint4 pk;
                    pk.x = pack2(u_keep[j], u_keep[j + 1]); pk.y = pack2(u_keep[j + 2], u_keep[j + 3]);
                    pk.z = pack2(u_keep[j + 4], u_keep[j + 5]); pk.w = pack2(u_keep[j + 6], u_keep[j + 7]);
                    *reinterpret_cast<uint4*>(smem + OFF_XB + op_chunk(row, (c0 + j) >> 3, 128)) = pk;
                }
                fence_async_smem();
                warp_arrive(&bars[C_XREADY], lane);
                tr(48);
                float4* park = reinterpret_cast<float4*>(a.y_mid + z * a.y_mid_z + (li & 1) * a.y_l) + park_block() + row;
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                    __stcg(park + (cq * 8 + (j >> 2)) * 128, make_float4(u_keep[j], u_keep[j + 1], u_keep[j + 2], u_keep[j + 3]));
            } else {
                // last layer: Y row-major to the caller, coalesced through a shared-memory transpose.  16 warps x 4224 B
                // run from the att tile into the (by now idle) weight ring: every MMA of the launch is complete.
                float* Y = a.y + z * a.y_z;
                float* stage = reinterpret_cast<float*>(smem + OFF_ATT) + warp * (32 * 33);
#pragma unroll
                for (int j = 0; j < 32; ++j) stage[lane * 33 + j] = u_keep[j];
                __syncwarp();
                const int cc = (lane & 7) * 4;
#pragma unroll
                for (int it = 0; it < 8; ++it) {
                    const int r = it * 4 + (lane >> 3);
                    const float* sp = stage + r * 33 + cc;
                    const int trw = lq * 32 + r;
                    // (token 0 of a gene: tile rows are whole genes, row0 is a multiple of S)
                    const bool head_row = PLAN ? rowmap[trw] % SMAX == 0 : trw % SMAX == 0;
                    // (under a plan only: in the other instantiation the extra test costs more in registers than the rows in bytes)
                    if (trw < rows_valid && (head_row || !PLAN || !a.y_head_only))
                        *reinterpret_cast<float4*>(Y + (PLAN ? (long long)rowmap[trw] : row0 + trw) * 128 + c0 + cc) = make_float4(sp[0], sp[1], sp[2], sp[3]);
                }
            }
        }
        }   // layers
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

// ---------------------------------------------------------------- weight stream ----
// 14 chunks of [128 rows x 128 k] BF16 per (resolution, layer) in UMMA tile order, in the order
// the kernel consumes them (see the header comment).
__global__ void pack_reg_stream_kernel(RegStreamArgs a) {
    const int z = blockIdx.z, l = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;        // (chunk, row, kc)
    if (i >= RF_NCHUNK * 128 * 16) return;
    const int c = i / (128 * 16), n = (i / 16) % 128, kc = i % 16;
    const float* P = a.params + z * a.p_z;
    const float* src;
    if (c < 8) {                 // fused projection [1024, 128]: q rows 0.., k 256.., v 512.., gate 768..
        const int t = c >> 1, base = (c & 1) ? 512 : 0;
        const int r = base + (n < 64 ? 64 * t + n : 256 + 64 * t + (n - 64));
        src = P + a.att[l] + (long long)r * 128 + kc * 8;
    } else if (c < 10) {         // out-projection [128, 256], K halves
        src = P + a.ffw[l] + (long long)n * 256 + (c - 8) * 128 + kc * 8;
    } else if (c < 12) {         // FFN-1 [256, 128], N halves
        src = P + a.l1w[l] + (long long)((c - 10) * 128 + n) * 128 + kc * 8;
    } else {                     // FFN-2 [128, 256], K halves
        src = P + a.l2w[l] + (long long)n * 256 + (c - 12) * 128 + kc * 8;
    }
    const float4 x0 = *reinterpret_cast<const float4*>(src), x1 = *reinterpret_cast<const float4*>(src + 4);
    uint4 pk;
    pk.x = pack2(x0.x, x0.y); pk.y = pack2(x0.z, x0.w); pk.z = pack2(x1.x, x1.y); pk.w = pack2(x1.z, x1.w);
    __nv_bfloat16* dst = a.stream + ((long long)(z * a.n_layers + l) * RF_NCHUNK + c) * RF_CHUNK_ELEMS +
                         ((n >> 3) * 16 + kc) * 64 + (n & 7) * 8;
    *reinterpret_cast<uint4*>(dst) = pk;
}

long long reg_stream_elems_per_layer() { return (long long)RF_NCHUNK * RF_CHUNK_ELEMS; }

int pack_reg_stream(const RegStreamArgs& a, int n_res, cudaStream_t st) {
    dim3 grid((RF_NCHUNK * 128 * 16 + 255) / 256, a.n_layers, n_res);
    pack_reg_stream_kernel<<<grid, 256, 0, st>>>(a);
    CHROMO_CHECK_LAUNCH("pack_reg_stream");
    return CHROMO_OK;
}

static long long* g_trace = nullptr;
void reg_fused_set_trace(long long* buf) { g_trace = buf; }

int launch_reg_layer_fused(const RegFusedArgs& a, int n_res, cudaStream_t st) {
    static bool configured = false;
    if (!configured) {
        cudaError_t e1 = cudaFuncSetAttribute(reg_layer_fused_kernel<9, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RF_SMEM);
        cudaError_t e2 = cudaFuncSetAttribute(reg_layer_fused_kernel<17, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RF_SMEM);
        cudaError_t e3 = cudaFuncSetAttribute(reg_layer_fused_kernel<9, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RF_SMEM);
        cudaError_t e4 = cudaFuncSetAttribute(reg_layer_fused_kernel<17, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RF_SMEM);
        cudaError_t e5 = cudaFuncSetAttribute(reg_layer_fused_kernel<9, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RF_SMEM);
        cudaError_t e6 = cudaFuncSetAttribute(reg_layer_fused_kernel<17, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RF_SMEM);
        for (cudaError_t e : {e1, e2, e3, e4, e5, e6})
            if (e != cudaSuccess) { set_error("reg_fused smem attribute: %s", cudaGetErrorString(e)); return CHROMO_ECUDA; }
        configured = true;
    }
    dim3 grid(a.n_tiles, n_res);
    RegFusedArgs at = a;
    at.trace = g_trace;
    {
        static int sms = 0;
        if (!sms) {
            int dev = 0;
            if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms < 1) sms = 1 << 30;
        }
        at.park_by_sm = (a.n_layers > 1 && a.n_tiles >= sms) ? 1 : 0;   // (%smid < SM count)
    }
    if (a.n_layers < 1) { set_error("reg_layer_fused: n_layers must be >= 1"); return CHROMO_EINVAL; }
    const bool plan = a.plan_tiles != nullptr;
    if (plan && !a.plan_rows) { set_error("reg_layer_fused: ragged plan without its row map"); return CHROMO_EINVAL; }
    if (plan) at.trace = nullptr;
    if (a.S == 9 && plan) reg_layer_fused_kernel<9, false, true><<<grid, RF_THREADS, RF_SMEM, st>>>(at);
    else if (a.S == 17 && plan) reg_layer_fused_kernel<17, false, true><<<grid, RF_THREADS, RF_SMEM, st>>>(at);
    else if (a.S == 9 && at.trace) reg_layer_fused_kernel<9, true, false><<<grid, RF_THREADS, RF_SMEM, st>>>(at);
    else if (a.S == 17 && at.trace) reg_layer_fused_kernel<17, true, false><<<grid, RF_THREADS, RF_SMEM, st>>>(at);
    else if (a.S == 9) reg_layer_fused_kernel<9, false, false><<<grid, RF_THREADS, RF_SMEM, st>>>(at);
    else if (a.S == 17) reg_layer_fused_kernel<17, false, false><<<grid, RF_THREADS, RF_SMEM, st>>>(at);
    else { set_error("reg_layer_fused: tokens per gene must be 9 or 17"); return CHROMO_EINVAL; }
    CHROMO_CHECK_LAUNCH("reg_layer_fused");
    return CHROMO_OK;
}

}  // namespace chromo
