// Input path: ChromoformerDataset._bin_and_pad / _get_region_representation
// (data.py:68-113) for a batch of regions, every resolution in one launch.
//
// HBM-bound byte work: 2 B read per (feature, bp); the per-region FP16 row is
// staged in shared memory ONCE with 16-byte vector loads (a row is re-used by
// all resolutions, where the reference re-loads the .npy per bin size,
// data.py:104) and each warp then reduces whole bins out of shared memory.
#include <cuda_fp16.h>
#include <stdlib.h>

#include "common.cuh"

namespace chromo {

constexpr int BIN_THREADS = 256;
constexpr int BIN_CHUNK = 16384;          // bp staged per pass (32 KB of FP16)
constexpr int BIN_MAX_RES = CHROMO_MAX_RES;

struct BinArgs {
    const __half* raw;
    const chromo_region_t* regions;
    int n_regions, F, n_res;
    int bin[BIN_MAX_RES];
    int nb[BIN_MAX_RES];                  // max bins per resolution
    float* feats[BIN_MAX_RES];
    int* spans;
};

// grid = (F, n_regions); one CTA per (region, feature) row.
__global__ void __launch_bounds__(BIN_THREADS) bin_regions_kernel(BinArgs a) {
    __shared__ __align__(16) __half stage[BIN_CHUNK];
    const int f = blockIdx.x, reg = blockIdx.y;
    const chromo_region_t rg = a.regions[reg];
    const __half* row = a.raw + rg.offset + (long long)f * rg.length + rg.start;
    const int W = rg.width;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = BIN_THREADS / 32;

    // zero-fill the padded output rows + spans first (each CTA owns feature f)
    for (int r = 0; r < a.n_res; ++r) {
        const int n = a.nb[r];
        int nbins = (W + a.bin[r] - 1) / a.bin[r];
        if (nbins > n) nbins = n;
        const int lp = (n - nbins + 1) / 2, rp = (n - nbins) / 2;
        const int first = rg.flip ? rp : lp;      // left pad after the optional flip
        float* out = a.feats[r] + (long long)reg * n * a.F + f;
        for (int p = threadIdx.x; p < n; p += BIN_THREADS)
            if (p < first || p >= first + nbins) out[(long long)p * a.F] = 0.f;
        if (f == 0 && threadIdx.x == 0) {
            a.spans[((long long)r * a.n_regions + reg) * 2 + 0] = first;
            a.spans[((long long)r * a.n_regions + reg) * 2 + 1] = nbins;
        }
    }

    // chunk size is a multiple of every bin size <= BIN_CHUNK we meet in practice
    // (100, 500, 2000 | 16000); compute the largest common multiple that fits.
    int chunk = BIN_CHUNK;
    {
        // lcm of the bin sizes, capped: fall back to per-resolution chunking otherwise
        long long l = 1;
        for (int r = 0; r < a.n_res; ++r) {
            long long x = l, y = a.bin[r];
            while (y) { long long t = x % y; x = y; y = t; }
            l = l / x * a.bin[r];
            if (l > BIN_CHUNK) break;
        }
        if (l <= BIN_CHUNK) chunk = (int)(BIN_CHUNK / l * l);
        else chunk = 0;
    }

    if (chunk > 0) {
        for (int c0 = 0; c0 < W; c0 += chunk) {
            const int len = min(chunk, W - c0);
            const __half* src = row + c0;
            // vectorised staging: 8 halves (16 B) per thread when aligned
            const int mis = (int)((reinterpret_cast<uintptr_t>(src) & 15) / 2);
            const int head = mis ? min(len, 8 - mis) : 0;
            for (int i = threadIdx.x; i < head; i += BIN_THREADS) stage[i] = src[i];
            const int nvec = (len - head) / 8;
            // keep shared destination aligned as well: shift by `head` only if head % 8 == 0
            if (head == 0) {
                const uint4* s4 = reinterpret_cast<const uint4*>(src);
                uint4* d4 = reinterpret_cast<uint4*>(stage);
                for (int i = threadIdx.x; i < nvec; i += BIN_THREADS) d4[i] = __ldg(s4 + i);
            } else {
                for (int i = threadIdx.x; i < nvec * 8; i += BIN_THREADS) stage[head + i] = src[head + i];
            }
            for (int i = head + nvec * 8 + threadIdx.x; i < len; i += BIN_THREADS) stage[i] = src[i];
            __syncthreads();
            for (int r = 0; r < a.n_res; ++r) {
                const int bs = a.bin[r], n = a.nb[r];
                int nbins = (W + bs - 1) / bs;
                if (nbins > n) nbins = n;
                const int lp = (n - nbins + 1) / 2;
                const int b0 = c0 / bs, bcnt = (len + bs - 1) / bs;
                float* out = a.feats[r] + (long long)reg * n * a.F + f;
                for (int b = warp; b < bcnt; b += nwarps) {
                    const int gb = b0 + b;
                    if (gb >= nbins) break;
                    const int s = b * bs, e = min(s + bs, len);
                    float acc = 0.f;
                    for (int i = s + lane; i < e; i += 32) acc += __half2float(stage[i]);
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
                    if (lane == 0) {
                        const float mean = acc / (float)(e - s);
                        int pos = lp + gb;
                        if (rg.flip) pos = n - 1 - pos;
                        out[(long long)pos * a.F] = logf(mean + 1.f);
                    }
                }
            }
            __syncthreads();
        }
    } else {
        // generic bin sizes: straight from global memory, one warp per bin
        for (int r = 0; r < a.n_res; ++r) {
            const int bs = a.bin[r], n = a.nb[r];
            int nbins = (W + bs - 1) / bs;
            if (nbins > n) nbins = n;
            const int lp = (n - nbins + 1) / 2;
            float* out = a.feats[r] + (long long)reg * n * a.F + f;
            for (int b = warp; b < nbins; b += nwarps) {
                const int s = b * bs, e = min(s + bs, W);
                float acc = 0.f;
                for (int i = s + lane; i < e; i += 32) acc += __half2float(row[i]);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
                if (lane == 0) {
                    const float mean = acc / (float)(e - s);
                    int pos = lp + b;
                    if (rg.flip) pos = n - 1 - pos;
                    out[(long long)pos * a.F] = logf(mean + 1.f);
                }
            }
        }
    }
}


// ---------------------------------------------------------------------------------------------
// Fast path (bin sizes that are multiples of the finest one, e.g. 100 | 500 | 2000): one THREAD per
// finest bin reads its bp straight from HBM with 8-byte loads (a warp covers a contiguous
// 32*bin0*2-byte span, every sector is consumed completely), coarser bins are sums of finest-bin
// sums exchanged through shared memory.  Nothing is staged, each byte is read exactly once.
//   grid = (chunks, regions), block = BT threads = one chunk of BT finest bins (all F rows in turn).
struct BinFastArgs {
    BinArgs b;
    int bt;                 // threads per block = finest bins per chunk (multiple of every ratio)
    int ratio[BIN_MAX_RES]; // bin[r] / bin0
    int fine;               // index of the finest resolution
};

__global__ void __launch_bounds__(256) bin_regions_fast_kernel(BinFastArgs fa) {
    // grid = (chunks, regions); the block walks the F feature rows of its span one after the other and
    // writes the [bins x F] outputs of every resolution as contiguous runs (F-interleaved, coalesced).
    __shared__ float sums[8][256];
    extern __shared__ __align__(16) __half span_s[];
    const BinArgs& a = fa.b;
    const int chunk = blockIdx.x, reg = blockIdx.y;
    const chromo_region_t rg = a.regions[reg];
    const int W = rg.width, bin0 = a.bin[fa.fine], F = a.F;
    const int t = threadIdx.x;
    const int fb = chunk * fa.bt + t;                          // finest-bin index within the region
    const int s0 = fb * bin0, e0 = min(s0 + bin0, W);
    const int c0 = chunk * fa.bt * bin0;                       // first bp of the span
    const int clen = min(fa.bt * bin0, W - c0);                // bp in the span (<= 0: only padding to write)
    for (int f = 0; f < F; ++f) {
        float acc = 0.f;
        if (clen > 0) {
            // stage the span of feature f: 16-byte cp.async copies (coalesced, all in flight), element-wise head/tail
            const __half* src = a.raw + rg.offset + (long long)f * rg.length + rg.start + c0;
            const int mis = (int)((reinterpret_cast<uintptr_t>(src) & 15) >> 1);
            const int head = mis ? min(clen, 8 - mis) : 0;
            const int nvec = (clen - head) / 8;
            for (int i = t; i < head; i += blockDim.x) span_s[mis + i] = src[i];
            const uint32_t dst = static_cast<uint32_t>(__cvta_generic_to_shared(span_s + mis + head));
            const __half* body = src + head;
            for (int i = t; i < nvec; i += blockDim.x)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + i * 16), "l"(body + i * 8) : "memory");
            asm volatile("cp.async.commit_group;" ::: "memory");
            for (int i = head + nvec * 8 + t; i < clen; i += blockDim.x) span_s[mis + i] = src[i];
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            __syncthreads();
            if (s0 < W) {
                const __half* p = span_s + mis + (s0 - c0);
                const int len = e0 - s0;
                int i = 0;
                if ((reinterpret_cast<uintptr_t>(p) & 3) == 0) {
                    float a0 = 0.f, a1 = 0.f;
                    for (; i + 2 <= len; i += 2) {
                        const float2 v = __half22float2(*reinterpret_cast<const __half2*>(p + i));
                        a0 += v.x; a1 += v.y;
                    }
                    acc = a0 + a1;
                }
                for (; i < len; ++i) acc += __half2float(p[i]);
            }
        }
        sums[f][t] = acc;
        __syncthreads();                                       // span_s is reused by the next feature
    }
    for (int r = 0; r < a.n_res; ++r) {
        const int ratio = fa.ratio[r], bs = a.bin[r], n = a.nb[r];
        int nbins = (W + bs - 1) / bs;
        if (nbins > n) nbins = n;
        const int lp = (n - nbins + 1) / 2, rp = (n - nbins) / 2;
        const int per_chunk = fa.bt / ratio;
        float* out = a.feats[r] + (long long)reg * n * F;
        for (int idx = t; idx < per_chunk * F; idx += blockDim.x) {
            const int lb = idx / F, f = idx - lb * F;
            const int gb = chunk * per_chunk + lb;
            if (gb < nbins) {
                float sacc = 0.f;
                for (int k = 0; k < ratio; ++k) sacc += sums[f][lb * ratio + k];
                const int s = gb * bs, e = min(s + bs, W);
                int pos = lp + gb;
                if (rg.flip) pos = n - 1 - pos;
                out[(long long)pos * F + f] = logf(sacc / (float)(e - s) + 1.f);
            }
        }
        if (chunk == 0) {   // zero padding + spans
            const int first = rg.flip ? rp : lp;
            for (int idx = t; idx < n * F; idx += blockDim.x) {
                const int pp = idx / F;
                if (pp < first || pp >= first + nbins) out[idx] = 0.f;
            }
            if (t == 0) {
                a.spans[((long long)r * a.n_regions + reg) * 2 + 0] = first;
                a.spans[((long long)r * a.n_regions + reg) * 2 + 1] = nbins;
            }
        }
    }
}

}  // namespace chromo

using namespace chromo;

extern "C" int chromo_bin_regions(const uint16_t* raw, const chromo_region_t* regions, int32_t n_regions,
                                  int32_t n_feats, int32_t n_res, const int32_t* bin_sizes,
                                  const int32_t* n_bins, float* const* feats, int32_t* spans, void* stream) {
    if (!raw || !regions || !bin_sizes || !n_bins || !feats || !spans) { set_error("bin_regions: null argument"); return CHROMO_EINVAL; }
    if (n_res < 1 || n_res > BIN_MAX_RES || n_feats < 1 || n_feats > 65535) { set_error("bin_regions: bad n_res / n_feats"); return CHROMO_EINVAL; }
    if (n_regions < 0 || n_regions > 65535) { set_error("bin_regions: at most 65535 regions per call"); return CHROMO_EINVAL; }
    if (n_regions == 0) return CHROMO_OK;
    BinArgs a;
    a.raw = reinterpret_cast<const __half*>(raw);
    a.regions = regions; a.n_regions = n_regions; a.F = n_feats; a.n_res = n_res; a.spans = spans;
    for (int r = 0; r < n_res; ++r) {
        if (bin_sizes[r] < 1 || n_bins[r] < 1 || !feats[r]) { set_error("bin_regions: bad resolution %d", r); return CHROMO_EINVAL; }
        a.bin[r] = bin_sizes[r]; a.nb[r] = n_bins[r]; a.feats[r] = feats[r];
    }
    // fast path: every bin size is a multiple of the finest one and a chunk of <= 256 finest bins
    // can be cut on a boundary of all of them
    {
        BinFastArgs fa;
        fa.b = a;
        int fine = 0;
        for (int r = 1; r < n_res; ++r) if (a.bin[r] < a.bin[fine]) fine = r;
        long long max_width = 0;      // longer regions are truncated to n_bins anyway (data.py requires L <= w_max)
        for (int r = 0; r < n_res; ++r) max_width = max_width > (long long)a.nb[r] * a.bin[r] ? max_width : (long long)a.nb[r] * a.bin[r];
        bool ok = max_width > 0;
        long long l = 1;
        for (int r = 0; r < n_res && ok; ++r) {
            if (a.bin[r] % a.bin[fine] != 0) { ok = false; break; }
            fa.ratio[r] = a.bin[r] / a.bin[fine];
            long long x = l, y = fa.ratio[r];
            while (y) { long long t = x % y; x = y; y = t; }
            l = l / x * fa.ratio[r];
            if (l > 256) ok = false;
        }
        if (ok) {
            fa.fine = fine;
            fa.bt = (int)(256 / l * l);
            const long long fine_bins = ((long long)max_width + a.bin[fine] - 1) / a.bin[fine];
            const int chunks = (int)((fine_bins + fa.bt - 1) / fa.bt);
            const size_t smem = ((size_t)fa.bt * a.bin[fine] + 16) * sizeof(__half);
            if (chunks >= 1 && n_feats <= 8 && smem <= 200 * 1024) {
                dim3 grid(chunks, n_regions);
                static size_t configured = 0;
                if (smem > configured) {
                    cudaFuncSetAttribute(bin_regions_fast_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                    configured = smem;
                }
                bin_regions_fast_kernel<<<grid, fa.bt, smem, (cudaStream_t)stream>>>(fa);
                CHROMO_CHECK_LAUNCH("bin_regions_fast");
                return CHROMO_OK;
            }
        }
    }
    dim3 grid(n_feats, n_regions);
    bin_regions_kernel<<<grid, BIN_THREADS, 0, (cudaStream_t)stream>>>(a);
    CHROMO_CHECK_LAUNCH("bin_regions");
    return CHROMO_OK;
}

// ------------------------------------------------------------------ FP16 feature wire ----
// Host -> device transport of a gene batch at half the bytes of the reference's (run_demo.py:100-105 ships FP32
// features + n x n boolean masks): features travel as FP16 (the raw depth is FP16 on disk; ln(mean + 1) <= 11 fits
// with 2^-11 relative rounding), pad masks as (first valid bin, count) spans.  One launch widens every feature tensor
// back to the FP32 layout the forward consumes and expands the spans to centre-row masks.
namespace chromo {

constexpr int WIRE_MAX = 8;
struct WireArgs {
    int n_seg, n_sets;
    const __half* src[WIRE_MAX]; float* dst[WIRE_MAX]; long long count[WIRE_MAX];
    const int* spans[WIRE_MAX]; uint8_t* mask[WIRE_MAX]; int rows[WIRE_MAX]; int n[WIRE_MAX];
};

__global__ void __launch_bounds__(256) unpack_wire_kernel(const WireArgs a) {
    const int seg = blockIdx.y;
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x, nthr = (long long)gridDim.x * blockDim.x;
    if (seg < a.n_seg) {
        const __half* src = a.src[seg];
        float* dst = a.dst[seg];
        const long long n8 = a.count[seg] >> 3;
        for (long long i = tid; i < n8; i += nthr) {
            const uint4 h = __ldg(reinterpret_cast<const uint4*>(src) + i);
            const __half2* h2 = reinterpret_cast<const __half2*>(&h);
            const float2 f0 = __half22float2(h2[0]), f1 = __half22float2(h2[1]);
            const float2 f2 = __half22float2(h2[2]), f3 = __half22float2(h2[3]);
            float4* o = reinterpret_cast<float4*>(dst) + 2 * i;
            o[0] = make_float4(f0.x, f0.y, f1.x, f1.y);
            o[1] = make_float4(f2.x, f2.y, f3.x, f3.y);
        }
        for (long long i = (n8 << 3) + tid; i < a.count[seg]; i += nthr) dst[i] = __half2float(src[i]);
    } else {
        const int set = seg - a.n_seg;
        const int n = a.n[set];
        const long long total = (long long)a.rows[set] * n;
        for (long long i = tid; i < total; i += nthr) {
            const int row = (int)(i / n), p = (int)(i - (long long)row * n);
            const int lo = a.spans[set][2 * row], cnt = a.spans[set][2 * row + 1];
            a.mask[set][i] = (p >= lo && p < lo + cnt) ? 0 : 1;
        }
    }
}

// Compact wire of ragged genes: only the valid bins of a region travel (data.py:86-97 pads the rest with zeros).  One warp
// per region row: the row's [lo, lo + cnt) bins come from the FP16 stream at the region's offset, everything else is zero.
struct CompactArgs {
    int n_sets, F;
    const __half* src[WIRE_MAX]; const int* spans[WIRE_MAX]; const int* off[WIRE_MAX]; int base[WIRE_MAX];
    float* dst[WIRE_MAX]; int rows[WIRE_MAX]; int n[WIRE_MAX];
};
__global__ void __launch_bounds__(256) unpack_compact_kernel(const CompactArgs a) {
    const int set = blockIdx.y, lane = threadIdx.x & 31;
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= a.rows[set]) return;
    const int F = a.F, nF = a.n[set] * F;
    const int lo = a.spans[set][2 * row] * F, hi = lo + a.spans[set][2 * row + 1] * F;
    const __half* src = a.src[set] + (long long)(a.off[set][row] - a.base[set]) * F - lo;
    float* dst = a.dst[set] + (long long)row * nF;
    for (int e = lane; e < nF; e += 32) dst[e] = (e >= lo && e < hi) ? __half2float(src[e]) : 0.f;
}

// Zero-suppressed wire: ln(mean + 1) of binned read depth is exactly zero wherever no read fell (37 % of the demo's bins),
// so a feature tensor travels as an occupancy bitmap (one bit per value) + its non-zero FP16 values + the running count of
// non-zeros at every block of 1024 values.  One warp per block: lane = bitmap word, its values start at the block's count
// plus the popcounts of the lanes in front.
struct SparseArgs {
    int n_seg;
    const uint32_t* bits[WIRE_MAX]; const __half* vals[WIRE_MAX]; const int* off[WIRE_MAX]; int base[WIRE_MAX];
    float* dst[WIRE_MAX]; long long count[WIRE_MAX];
};
__global__ void __launch_bounds__(256) unpack_sparse_kernel(const SparseArgs a) {
    const int seg = blockIdx.y, lane = threadIdx.x & 31;
    const long long count = a.count[seg], n_blk = (count + 1023) >> 10;
    const long long stride = (long long)gridDim.x * 8;
    for (long long blk = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); blk < n_blk; blk += stride) {
        const long long v0 = (blk << 10) + 32 * lane;                     // first value of this lane's word
        const uint32_t word = v0 < count ? __ldg(a.bits[seg] + (blk << 5) + lane) : 0u;
        int before = __popc(word);
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, before, o);
            if (lane >= o) before += t;
        }
        before -= __popc(word);                                            // exclusive
        const __half* src = a.vals[seg] + (long long)(__ldg(a.off[seg] + blk) - a.base[seg]) + before;
        float out[32];
        int k = 0;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            const bool on = (word >> j) & 1u;
            out[j] = on ? __half2float(src[k]) : 0.f;
            k += on;
        }
        float* dst = a.dst[seg] + v0;
        if (v0 + 32 <= count) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(dst + j) = make_float4(out[j], out[j + 1], out[j + 2], out[j + 3]);
        } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
                if (v0 + j < count) dst[j] = out[j];
        }
    }
}

}  // namespace chromo

extern "C" int chromo_unpack_sparse(int32_t n_seg, const uint32_t* const* bits, const uint16_t* const* vals,
                                    const int32_t* const* offsets, const int32_t* base, float* const* dst,
                                    const int64_t* counts, void* stream) {
    using namespace chromo;
    if (n_seg < 1 || n_seg > WIRE_MAX) { set_error("unpack_sparse: 1..%d segments", WIRE_MAX); return CHROMO_EINVAL; }
    SparseArgs a;
    a.n_seg = n_seg;
    long long most = 0;
    for (int i = 0; i < n_seg; ++i) {
        if (!bits[i] || !vals[i] || !offsets[i] || !dst[i] || counts[i] < 0) { set_error("unpack_sparse: bad segment %d", i); return CHROMO_EINVAL; }
        if (reinterpret_cast<uintptr_t>(dst[i]) & 15) { set_error("unpack_sparse: segment %d is not 16-byte aligned", i); return CHROMO_EINVAL; }
        a.bits[i] = bits[i]; a.vals[i] = reinterpret_cast<const __half*>(vals[i]); a.off[i] = offsets[i]; a.base[i] = base[i];
        a.dst[i] = dst[i]; a.count[i] = counts[i];
        most = counts[i] > most ? counts[i] : most;
    }
    if (most == 0) return CHROMO_OK;
    long long blocks = ((most + 1023) / 1024 + 7) / 8;
    if (blocks > 148 * 8) blocks = 148 * 8;
    unpack_sparse_kernel<<<dim3((unsigned)blocks, n_seg), 256, 0, (cudaStream_t)stream>>>(a);
    CHROMO_CHECK_LAUNCH("unpack_sparse");
    return CHROMO_OK;
}

extern "C" int chromo_unpack_compact(int32_t n_sets, const uint16_t* const* src, const int32_t* const* spans,
                                     const int32_t* const* offsets, const int32_t* base, float* const* dst,
                                     const int32_t* rows, const int32_t* n_bins, int32_t n_feats, void* stream) {
    using namespace chromo;
    if (n_sets < 1 || n_sets > WIRE_MAX || n_feats < 1) { set_error("unpack_compact: 1..%d sets", WIRE_MAX); return CHROMO_EINVAL; }
    CompactArgs a;
    a.n_sets = n_sets; a.F = n_feats;
    int most = 0;
    for (int i = 0; i < n_sets; ++i) {
        if (!src[i] || !spans[i] || !offsets[i] || !dst[i] || rows[i] < 0 || n_bins[i] < 1) { set_error("unpack_compact: bad set %d", i); return CHROMO_EINVAL; }
        a.src[i] = reinterpret_cast<const __half*>(src[i]); a.spans[i] = spans[i]; a.off[i] = offsets[i]; a.base[i] = base[i];
        a.dst[i] = dst[i]; a.rows[i] = rows[i]; a.n[i] = n_bins[i];
        most = rows[i] > most ? rows[i] : most;
    }
    if (most == 0) return CHROMO_OK;
    unpack_compact_kernel<<<dim3((unsigned)((most + 7) / 8), n_sets), 256, 0, (cudaStream_t)stream>>>(a);
    CHROMO_CHECK_LAUNCH("unpack_compact");
    return CHROMO_OK;
}

extern "C" int chromo_unpack_wire(int32_t n_seg, const uint16_t* const* src, float* const* dst, const int64_t* counts,
                                  int32_t n_sets, const int32_t* const* spans, uint8_t* const* masks,
                                  const int32_t* rows, const int32_t* n_bins, void* stream) {
    using namespace chromo;
    if (n_seg < 0 || n_seg > WIRE_MAX || n_sets < 0 || n_sets > WIRE_MAX) { set_error("unpack_wire: at most %d segments / span sets", WIRE_MAX); return CHROMO_EINVAL; }
    if (n_seg + n_sets == 0) return CHROMO_OK;
    WireArgs a;
    a.n_seg = n_seg; a.n_sets = n_sets;
    long long most = 0;
    for (int i = 0; i < n_seg; ++i) {
        if (!src[i] || !dst[i] || counts[i] < 0) { set_error("unpack_wire: bad segment %d", i); return CHROMO_EINVAL; }
        if ((reinterpret_cast<uintptr_t>(src[i]) | reinterpret_cast<uintptr_t>(dst[i])) & 15) { set_error("unpack_wire: segment %d is not 16-byte aligned", i); return CHROMO_EINVAL; }
        a.src[i] = reinterpret_cast<const __half*>(src[i]); a.dst[i] = dst[i]; a.count[i] = counts[i];
        most = counts[i] / 8 > most ? counts[i] / 8 : most;
    }
    for (int i = 0; i < n_sets; ++i) {
        if (!spans[i] || !masks[i] || rows[i] < 0 || n_bins[i] < 1) { set_error("unpack_wire: bad span set %d", i); return CHROMO_EINVAL; }
        a.spans[i] = spans[i]; a.mask[i] = masks[i]; a.rows[i] = rows[i]; a.n[i] = n_bins[i];
        const long long t = (long long)rows[i] * n_bins[i];
        most = t > most ? t : most;
    }
    long long blocks = (most + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;           // grid-stride: 8 CTAs per SM cover the widest segment
    if (blocks < 1) blocks = 1;
    unpack_wire_kernel<<<dim3((unsigned)blocks, n_seg + n_sets), 256, 0, (cudaStream_t)stream>>>(a);
    CHROMO_CHECK_LAUNCH("unpack_wire");
    return CHROMO_OK;
}
