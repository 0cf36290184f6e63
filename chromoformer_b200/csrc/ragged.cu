// Ragged plan of a batch (BF16 inference): the work the masks make irrelevant is not done.
//
// data.py:156-203 pads every pCRE to w_max / bin_size bins (mask = 1 outside the centred valid span) and every gene to
// i_max pCRE slots (dummy slots: zero features, pad mask all ones, and the interaction mask in block form - token j sees
// token i only when both are <= n_partners).  On the demo set 42 % of the genes have fewer than 8 pCREs and a pCRE fills
// 63 of 400 bins on average.  Two exact eliminations follow from the masks alone:
//   * a masked key has probability exp(-1e9 - max) == 0 in FP32 as soon as its row holds one unmasked key, so the
//     single-query attention of a region only needs the keys from its first to its last unmasked bin;
//   * with a block-form interaction mask the tokens of the slots > n_partners are never attended by the tokens that reach
//     the head (token 0 through the layers), so their Pairwise-Interaction rows need not exist.
// The plan: live slots sorted by descending span length (stable: a dense batch keeps its order) so that 64 regions of a
// tile share one key window; dead slots last, their X_in rows zeroed (they stay masked keys of the Regulation layers and
// must be finite).  A gene whose interaction mask is not in block form keeps all its slots; a live region without any
// unmasked key keeps the whole table (the reference's uniform softmax over the masked row).
#include <cub/block/block_scan.cuh>
#include <cub/device/device_radix_sort.cuh>

#include <algorithm>

#include "ragged.cuh"

namespace chromo {

namespace {

constexpr int DEAD_KEY = 255;

struct Carve {
    int* cls_cnt; int* k_gene; int* keys_in; int* keys_out; int* vals_in; int* span[CHROMO_MAX_RES];
    void* temp; size_t temp_bytes;
};

inline long long a4(long long x) { return (x + 3) & ~3LL; }
inline long long temp_ints(long long R) { return 4 * R + 65536; }

// n_partners of every gene from its interaction masks: k such that mask[j][i] == !(j <= k && i <= k) at every
// resolution (the largest k over the resolutions); I (every slot live) when a mask has another form.  One warp per gene.
constexpr int NCLS = 10;
// token classes of the Regulation stage by descending token count: S, then 9 8 ... 1 below it (0 = class does not exist)
__host__ __device__ __forceinline__ int class_tokens(int c, int S) {
    if (c == 0) return S;
    const int top = S - 1 < 9 ? S - 1 : 9;                        // largest class below S
    const int t = top - (c - 1);
    return t >= 1 ? t : 0;
}
__host__ __device__ __forceinline__ int class_of(int k, int S) {   // the smallest class that holds the 1 + k live tokens
    int c = 0;
    for (int i = 1; i < NCLS; ++i)
        if (class_tokens(i, S) >= k + 1) c = i;
    return c;
}

__global__ void ragged_gene_kernel(RaggedArgs a, int* __restrict__ k_gene, int* __restrict__ cls_cnt) {
    const int b = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (b >= a.B) return;
    const int S = a.I + 1, SS = S * S;
    int k = 0;
    for (int r = 0; r < a.n_res; ++r) {
        const uint8_t* m = a.imask[r] + (long long)b * SS;
        // row 0 sees tokens 0..kr
        const unsigned row0 = __ballot_sync(0xffffffffu, lane < S && m[lane] != 0) | (1u << S);
        const int kr = __ffs(row0) - 2;
        bool ok = kr >= 0;
        for (int e = lane; e < SS; e += 32) {
            const int j = e / S, i = e % S;
            if ((m[e] != 0) != !(j <= kr && i <= kr)) ok = false;
        }
        k = max(k, __all_sync(0xffffffffu, ok) ? kr : a.I);
    }
    if (lane == 0) {
        k_gene[b] = k;
        atomicAdd(&cls_cnt[(b >> 10) * NCLS + class_of(k, S)], 1);      // genes per (run of 1024 genes, class)
    }
}

// one warp per four pCRE regions: [first, last + 1) unmasked bin per resolution, sort key of the region (8 bits: one pass
// of the radix sort; the key windows come from the spans themselves, the key only groups similar lengths)
constexpr int SPAN_RPW = 4;
__global__ void ragged_span_kernel(RaggedArgs a, const int* __restrict__ k_gene, int* __restrict__ keys, int* __restrict__ vals,
                                   Carve c, int r_fine) {
    const int lane = threadIdx.x & 31;
    const int region0 = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * SPAN_RPW;
    const int R = a.B * a.I;
    if (region0 >= R) return;
    int len_fine[SPAN_RPW];
#pragma unroll
    for (int r = 0; r < CHROMO_MAX_RES; ++r) {
        if (r < a.n_res) {
            const int n = a.n[r], nw = n >> 2;
            const uint8_t* base = a.mask[r] + a.mask_row_offset[r];
            {
                constexpr int q0 = 0;                        // (up to 512 bins per region: build_ragged_plan checks)
                uint32_t v[SPAN_RPW][4];
#pragma unroll
                for (int g = 0; g < SPAN_RPW; ++g) {         // every load of the round in flight before the first use
                    const uint32_t* row = reinterpret_cast<const uint32_t*>(base + (long long)min(region0 + g, R - 1) * a.mask_stride[r]);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int w = q0 + lane + 32 * q;
                        v[g][q] = w < nw ? __ldg(row + w) : 0x01010101u;
                    }
                }
#pragma unroll
                for (int g = 0; g < SPAN_RPW; ++g) {
                    int lo = n, hi = 0;
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        // bit 7 of every zero byte: ~(((v & 0x7f..) + 0x7f..) | v) & 0x80..
                        const uint32_t x = v[g][q];
                        const uint32_t zb = ~(((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;
                        if (zb) {
                            const int w4 = 4 * (q0 + lane + 32 * q);
                            lo = min(lo, w4 + ((__ffs(zb) - 1) >> 3));
                            hi = max(hi, w4 + ((31 - __clz(zb)) >> 3) + 1);
                        }
                    }
                    lo = __reduce_min_sync(0xffffffffu, lo);
                    hi = __reduce_max_sync(0xffffffffu, hi);
                    if (hi == 0) { lo = 0; hi = n; }          // no unmasked key: uniform softmax over the whole row
                    if (lane == 0 && region0 + g < R) c.span[r][region0 + g] = lo | (hi << 16);
                    if (r == r_fine) len_fine[g] = hi - lo;
                }
            }
        }
    }
    if (lane < SPAN_RPW && region0 + lane < R) {
        const int region = region0 + lane;
        int lf = len_fine[0];
#pragma unroll
        for (int g = 1; g < SPAN_RPW; ++g) lf = lane == g ? len_fine[g] : lf;
        const bool dead = region % a.I >= k_gene[region / a.I];
        keys[region] = dead ? DEAD_KEY : ((a.n[r_fine] - lf) * (DEAD_KEY - 1)) / a.n[r_fine];
        vals[region] = region;
    }
}

// one warp per tile of 64 sorted regions: key windows, live counts, X_in rows (zeroed for the dead slots)
__global__ void ragged_tile_kernel(RaggedArgs a, Carve c, RaggedPlan p) {
    const int t = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    const int R = a.B * a.I, S = a.I + 1;
    const int first = 64 * t;
    if (first >= R) return;
    const int n_tile = min(64, R - first);
    int reg[2], yrow[2];
    bool live[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int m = first + 32 * h + lane;
        reg[h] = 0; yrow[h] = 0; live[h] = false;
        if (m < R) {
            reg[h] = p.perm[m];
            live[h] = c.keys_out[m] != DEAD_KEY;
            yrow[h] = (reg[h] / a.I) * S + reg[h] % a.I + 1;
            p.y_rows[m] = yrow[h];
        }
    }
    const unsigned lv0 = __ballot_sync(0xffffffffu, live[0]), lv1 = __ballot_sync(0xffffffffu, live[1]);
    const int cnt = __popc(lv0) + __popc(lv1);
    for (int r = 0; r < a.n_res; ++r) {
        int lo = a.n[r], hi = 0;
#pragma unroll
        for (int h = 0; h < 2; ++h)
            if (live[h]) {
                const int s = c.span[r][reg[h]];
                lo = min(lo, s & 0xffff); hi = max(hi, s >> 16);
            }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
            hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
        }
        if (lane == 0) {
            int k0 = 0, ns = 16;
            if (cnt > 0) {
                k0 = lo & ~7;
                ns = max(16, (hi - k0 + 15) & ~15);
                if (k0 + ns > a.ns[r]) k0 = a.ns[r] - ns;   // (both multiples of 16)
            }
            p.tile_k0[r][t] = k0; p.tile_ns[r][t] = ns;
        }
    }
    // the tile that holds the end of the live range publishes the counts
    const bool prev_live = t == 0 || c.keys_out[first - 1] != DEAD_KEY;
    if (lane == 0 && prev_live && (cnt < n_tile || first + n_tile == R)) {
        const int nl = first + cnt;
        p.live[0] = nl; p.live[1] = (nl + 63) / 64; p.live[2] = (nl + 127) / 128;
    }
    // dead slots: zero token rows in X_in (finite values under the masked keys of the Regulation layers)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const unsigned valid = __ballot_sync(0xffffffffu, first + 32 * h + lane < R);
        unsigned dead = valid & ~(h ? lv1 : lv0);
        while (dead) {
            const int j = __ffs(dead) - 1;
            dead &= dead - 1;
            const int row = __shfl_sync(0xffffffffu, yrow[h], j);
            for (int r = 0; r < a.n_res; ++r)
                reinterpret_cast<float4*>(a.xin + r * a.xin_z + (long long)row * 128)[lane] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
}

// Token classes of the Regulation stage: genes grouped by class (stable), tiles of floor(128 / S_c) genes per class.
// Block j ranks its run of 1024 genes; the counts per (run, class) come from ragged_gene_kernel.
__global__ void __launch_bounds__(1024) ragged_class_kernel(int B, int I, const int* __restrict__ k_gene,
                                                            const int* __restrict__ cls_cnt, RaggedPlan p) {
    using Scan = cub::BlockScan<int, 1024>;
    __shared__ typename Scan::TempStorage tmp;
    __shared__ int tot[NCLS], pre[NCLS], start[NCLS], tile0[NCLS + 1];
    const int t = threadIdx.x, S = I + 1, n_blk = gridDim.x;
    if (t < NCLS) {
        int all = 0, before = 0;
        for (int j = 0; j < n_blk; ++j) {
            const int v = cls_cnt[j * NCLS + t];
            all += v;
            if (j < (int)blockIdx.x) before += v;
        }
        tot[t] = all; pre[t] = before;
    }
    __syncthreads();
    if (t == 0) {
        int s0 = 0, n_t = 0;
        for (int c = 0; c < NCLS; ++c) {
            start[c] = s0; s0 += tot[c];
            tile0[c] = n_t;
            const int Sc = class_tokens(c, S);
            if (Sc > 0) n_t += (tot[c] + 128 / Sc - 1) / (128 / Sc);
        }
        tile0[NCLS] = n_t;
        if (blockIdx.x == 0) p.reg_n[0] = n_t;
    }
    __syncthreads();
    const int g = blockIdx.x * 1024 + t;
    const int c = g < B ? class_of(k_gene[g], S) : -1;
#pragma unroll
    for (int i = 0; i < NCLS; ++i) {
        int rank;
        Scan(tmp).ExclusiveSum(c == i ? 1 : 0, rank);
        if (c == i) p.gene_list[start[i] + pre[i] + rank] = g;
        __syncthreads();
    }
    if (blockIdx.x == 0)
        for (int i = t; i < p.reg_tiles_max; i += 1024) {
            int4 e = make_int4(0, 0, S, 0);                    // (unused tile)
            if (i < tile0[NCLS]) {
                int cc = 0;
                while (i >= tile0[cc + 1]) ++cc;
                const int Sc = class_tokens(cc, S), G = 128 / Sc, j = i - tile0[cc];
                e = make_int4(start[cc] + j * G, min(G, tot[cc] - j * G), Sc, 0);
            }
            p.reg_tiles[i] = e;
        }
}

// row of the [B*S, 128] layout behind every row of every Regulation tile (one block per tile)
__global__ void __launch_bounds__(128) ragged_rows_kernel(int I, RaggedPlan p) {
    const int4 e = p.reg_tiles[blockIdx.x];
    const int r = threadIdx.x;
    p.reg_rows[blockIdx.x * 128 + r] = r < e.y * e.z ? p.gene_list[e.x + r / e.z] * (I + 1) + r % e.z : 0;
}

Carve carve(const RaggedArgs& a, float* ws, RaggedPlan* p) {
    const long long R = (long long)a.B * a.I, T = (R + 63) / 64;
    int* cur = reinterpret_cast<int*>(ws);
    auto take = [&](long long n) { int* o = cur; cur += a4(n); return o; };
    Carve c;
    c.cls_cnt = take((long long)((a.B + 1023) / 1024) * NCLS);
    c.k_gene = take(a.B);
    c.keys_in = take(R); c.keys_out = take(R); c.vals_in = take(R);
    p->perm = take(R); p->y_rows = take(R);
    for (int r = 0; r < a.n_res; ++r) { c.span[r] = take(R); p->tile_k0[r] = take(T); p->tile_ns[r] = take(T); }
    p->live = take(4);
    p->gene_list = take(a.B);
    p->reg_n = take(4);
    p->reg_tiles_max = ragged_reg_tiles_max(a.B, a.I);
    p->reg_tiles = reinterpret_cast<int4*>(take(4LL * p->reg_tiles_max));
    p->reg_rows = take(128LL * p->reg_tiles_max);
    uintptr_t t = (reinterpret_cast<uintptr_t>(cur) + 255) & ~uintptr_t(255);
    c.temp = reinterpret_cast<void*>(t);
    c.temp_bytes = (size_t)(temp_ints(R) - 64) * 4;
    return c;
}

// token classes of the Regulation stage from the interaction masks: the counts per (run, class), then the gene list, the
// tiles and their row map
int launch_reg_classes(const RaggedArgs& a, int* k_gene, int* cls_cnt, RaggedPlan* plan, cudaStream_t st) {
    const int n_blk = (a.B + 1023) / 1024;
    if (cudaMemsetAsync(cls_cnt, 0, (size_t)n_blk * NCLS * sizeof(int), st) != cudaSuccess) { set_error("ragged plan: memset failed"); return CHROMO_ECUDA; }
    ragged_gene_kernel<<<(unsigned)(((long long)a.B * 32 + 255) / 256), 256, 0, st>>>(a, k_gene, cls_cnt);
    CHROMO_CHECK_LAUNCH("ragged_gene");
    ragged_class_kernel<<<n_blk, 1024, 0, st>>>(a.B, a.I, k_gene, cls_cnt, *plan);
    CHROMO_CHECK_LAUNCH("ragged_class");
    ragged_rows_kernel<<<plan->reg_tiles_max, 128, 0, st>>>(a.I, *plan);
    CHROMO_CHECK_LAUNCH("ragged_rows");
    return CHROMO_OK;
}

}  // namespace

int ragged_reg_tiles_max(int B, int I) {
    const int G = 128 / (I + 1) > 0 ? 128 / (I + 1) : 1;            // a class has at least this many genes per tile,
    return (B + G - 1) / G + NCLS;                                  // and at most one partly filled tile
}

long long ragged_plan_floats(int B, int I, int n_res) {
    const long long R = (long long)B * I, T = (R + 63) / 64;
    return a4((long long)((B + 1023) / 1024) * NCLS) + 2 * a4(B) + 5 * a4(R) + n_res * (a4(R) + 2 * a4(T)) + 8 + 132LL * ragged_reg_tiles_max(B, I) + temp_ints(R);
}

int build_ragged_plan(const RaggedArgs& a, float* ws, RaggedPlan* plan, cudaStream_t st) {
    const int R = a.B * a.I;
    Carve c = carve(a, ws, plan);
    int r_fine = 0;
    for (int r = 1; r < a.n_res; ++r)
        if (a.n[r] > a.n[r_fine]) r_fine = r;
    if (a.n[r_fine] > 512) { set_error("ragged plan: more than 512 bins per region"); return CHROMO_EINVAL; }
    CHROMO_TRY(launch_reg_classes(a, c.k_gene, c.cls_cnt, plan, st));
    ragged_span_kernel<<<(unsigned)(((long long)(R + SPAN_RPW - 1) / SPAN_RPW * 32 + 255) / 256), 256, 0, st>>>(a, c.k_gene, c.keys_in, c.vals_in, c, r_fine);
    CHROMO_CHECK_LAUNCH("ragged_span");
    size_t need = 0;
    cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, need, c.keys_in, c.keys_out, c.vals_in, plan->perm, R, 0, 8, st);
    if (e != cudaSuccess || need > c.temp_bytes) {
        set_error("ragged plan: sort scratch (%zu bytes needed, %zu reserved): %s", need, c.temp_bytes, cudaGetErrorString(e));
        return CHROMO_ECUDA;
    }
    e = cub::DeviceRadixSort::SortPairs(c.temp, need, c.keys_in, c.keys_out, c.vals_in, plan->perm, R, 0, 8, st);   // stable
    if (e != cudaSuccess) { set_error("ragged plan: sort: %s", cudaGetErrorString(e)); return CHROMO_ECUDA; }
    count_launch();
    const int tiles = (R + 63) / 64;
    ragged_tile_kernel<<<(tiles * 32 + 255) / 256, 256, 0, st>>>(a, c, *plan);
    CHROMO_CHECK_LAUNCH("ragged_tile");
    return CHROMO_OK;
}

// class counts, n_partners per gene, gene list, tile count, tiles, row map
long long reg_plan_floats(int B, int I) {
    return a4((long long)((B + 1023) / 1024) * NCLS) + 2 * a4(B) + 4 + 132LL * ragged_reg_tiles_max(B, I);
}

int build_reg_plan(const RaggedArgs& a, float* ws, RaggedPlan* plan, cudaStream_t st) {
    int* cur = reinterpret_cast<int*>(ws);
    auto take = [&](long long n) { int* o = cur; cur += a4(n); return o; };
    *plan = RaggedPlan();
    int* cls_cnt = take((long long)((a.B + 1023) / 1024) * NCLS);
    int* k_gene = take(a.B);
    plan->gene_list = take(a.B);
    plan->reg_n = take(4);
    plan->reg_tiles_max = ragged_reg_tiles_max(a.B, a.I);
    plan->reg_tiles = reinterpret_cast<int4*>(take(4LL * plan->reg_tiles_max));
    plan->reg_rows = take(128LL * plan->reg_tiles_max);
    return launch_reg_classes(a, k_gene, cls_cnt, plan, st);
}

}  // namespace chromo
