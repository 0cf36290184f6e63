// Flat parameter layout + workspace layout + error plumbing (host only).
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <map>
#include <mutex>

#include <algorithm>

#include "common.cuh"
#include "ragged.cuh"
#include "reg_fused.cuh"
#include "train_gemm.cuh"

namespace chromo {
long long launch_counter(bool reset);

static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
long long launch_counter(bool reset) { return reset ? g_launches.exchange(0) : g_launches.load(); }

int validate_config(const chromo_config_t* c) {
    if (!c) { set_error("null config"); return CHROMO_EINVAL; }
#define REQ(cond, msg)                                                        \
    if (!(cond)) { set_error("unsupported config: %s", msg); return CHROMO_EINVAL; }
    REQ(c->d_emb == 128, "d_emb must be 128 (LayerNorm/row kernels are specialised for it)");
    REQ(c->n_feats >= 1 && c->n_feats <= 8, "n_feats must be in [1,8]");
    REQ(c->n_res >= 1 && c->n_res <= CHROMO_MAX_RES, "n_res must be in [1,4]");
    REQ(c->i_max >= 1 && c->i_max <= 16, "i_max must be in [1,16]");
    REQ(c->n_out >= 1 && c->n_out <= 16, "n_out must be in [1,16]");
    REQ(c->d_head >= 4 && c->d_head % 4 == 0 && c->d_head <= 1024, "d_head must be a multiple of 4");
    // The Embedding transformer is evaluated for the centre query row only
    // (net.py:59); that is exact for a single layer, which is the only depth the
    // reference configs use (configs/default.yaml:19).
    REQ(c->embed_layers == 1, "embed.n_layers must be 1");
    REQ(c->embed_d_model == c->d_emb, "embed.d_model must equal d_emb (net.py:305)");
    REQ(c->embed_heads >= 1 && c->embed_heads <= 8 && c->embed_d_model % c->embed_heads == 0,
        "embed.n_heads must divide embed.d_model");
    REQ((c->embed_d_model / c->embed_heads) % 4 == 0, "embed head width must be a multiple of 4");
    REQ(c->embed_d_ff % 4 == 0 && c->embed_d_ff >= 4, "embed.d_ff must be a multiple of 4");
    REQ(c->pw_layers >= 1 && c->pw_layers <= CHROMO_MAX_LAYERS, "pairwise.n_layers in [1,8]");
    REQ(c->pw_heads >= 1 && c->pw_heads <= 8 && c->pw_d_model % c->pw_heads == 0,
        "pairwise.n_heads must divide pairwise.d_model");
    REQ(c->pw_d_model == c->d_emb, "pairwise.d_model must equal d_emb (net.py:86-89)");
    REQ((c->pw_d_model / c->pw_heads) % 4 == 0, "pairwise head width must be a multiple of 4");
    REQ(c->pw_d_ff % 4 == 0 && c->pw_d_ff >= 4, "pairwise.d_ff must be a multiple of 4");
    REQ(c->reg_layers >= 1 && c->reg_layers <= CHROMO_MAX_LAYERS, "regulation.n_layers in [1,8]");
    REQ(c->reg_heads >= 1 && c->reg_heads <= 32 && c->reg_d_model == 32 * c->reg_heads,
        "regulation head width (d_model / n_heads) must be 32");
    REQ(c->reg_d_ff % 4 == 0 && c->reg_d_ff >= 4, "regulation.d_ff must be a multiple of 4");
    for (int r = 0; r < c->n_res; ++r)
        REQ(c->n_bins[r] >= 1 && c->n_bins[r] <= 4096, "n_bins must be in [1,4096]");
#undef REQ
    return CHROMO_OK;
}

namespace {

struct Builder {
    ParamLayout* L;
    int pass;            // 0: used tensors, 1: unused tensors
    int64_t cursor;
    void add(const std::string& name, int64_t numel, bool used, int64_t* slot) {
        if ((pass == 0) != used) return;
        *slot = cursor;
        L->infos.push_back({name, cursor, numel, used});
        cursor = (cursor + numel + 7) & ~int64_t(7);   // 16-byte aligned in the BF16 mirror too (TMA bulk)
    }
};

void ffn(Builder& b, const std::string& p, int d_emb, int d_ff, FfnOff* f) {
    b.add(p + "l1.weight", (int64_t)d_ff * d_emb, true, &f->l1w);
    b.add(p + "l1.bias", d_ff, true, &f->l1b);
    b.add(p + "l2.weight", (int64_t)d_emb * d_ff, true, &f->l2w);
    b.add(p + "l2.bias", d_emb, true, &f->l2b);
    b.add(p + "ln.weight", d_emb, true, &f->lnw);
    b.add(p + "ln.bias", d_emb, true, &f->lnb);
}

void build(const chromo_config_t* c, ParamLayout* L) {
    Builder b{L, 0, 0};
    const int D = c->d_emb, F = c->n_feats;
    for (int pass = 0; pass < 2; ++pass) {
        b.pass = pass;
        for (int r = 0; r < c->n_res; ++r) {
            std::string p = "embed." + std::to_string(r) + ".";
            EmbedOff& e = L->embed[r];
            b.add(p + "lin_proj.weight", (int64_t)D * F, true, &e.lin_proj);
            for (int l = 0; l < c->embed_layers; ++l) {
                std::string q = p + "transformer.layers." + std::to_string(l) + ".";
                AttnOff& a = e.att[l];
                b.add(q + "self_att.gamma_f", c->embed_heads, false, &a.gamma_f);
                b.add(q + "self_att.w_bias.weight", 2 * c->embed_heads, false, &a.w_bias);
                b.add(q + "self_att.att.weight", (int64_t)3 * c->embed_d_model * D, true, &a.att);
                b.add(q + "self_att.ff.weight", (int64_t)D * c->embed_d_model, true, &a.ffw);
                b.add(q + "self_att.ff.bias", D, true, &a.ffb);
                b.add(q + "self_att.ln.weight", D, true, &a.lnw);
                b.add(q + "self_att.ln.bias", D, true, &a.lnb);
                ffn(b, q + "ff.", D, c->embed_d_ff, &e.ffn[l]);
            }
        }
        for (int r = 0; r < c->n_res; ++r) {
            std::string p = "pairwise_interaction." + std::to_string(r) + ".";
            PairOff& e = L->pw[r];
            b.add(p + "ln.weight", D, false, &e.lnw);
            b.add(p + "ln.bias", D, false, &e.lnb);
            b.add(p + "lin_proj_p.weight", (int64_t)D * D, true, &e.lin_proj_p);
            b.add(p + "lin_proj_pcre.weight", (int64_t)D * F, true, &e.lin_proj_pcre);
            for (int l = 0; l < c->pw_layers; ++l) {
                std::string q = p + "transformer.layers." + std::to_string(l) + ".";
                AttnOff& a = e.att[l];
                b.add(q + "self_att.gamma_f", c->pw_heads, false, &a.gamma_f);
                b.add(q + "self_att.p_att.weight", (int64_t)c->pw_d_model * D, true, &a.p_att);
                b.add(q + "self_att.c_att.weight", (int64_t)2 * c->pw_d_model * D, true, &a.c_att);
                b.add(q + "self_att.ff.weight", (int64_t)D * c->pw_d_model, true, &a.ffw);
                b.add(q + "self_att.ff.bias", D, true, &a.ffb);
                b.add(q + "self_att.ln.weight", D, true, &a.lnw);
                b.add(q + "self_att.ln.bias", D, true, &a.lnb);
                ffn(b, q + "ff.", D, c->pw_d_ff, &e.ffn[l]);
            }
        }
        for (int r = 0; r < c->n_res; ++r) {
            std::string p = "regulation." + std::to_string(r) + ".";
            RegOff& e = L->reg[r];
            for (int l = 0; l < c->reg_layers; ++l) {
                std::string q = p + "transformer.layers." + std::to_string(l) + ".";
                AttnOff& a = e.att[l];
                b.add(q + "self_att.gamma_f", c->reg_heads, true, &a.gamma_f);
                b.add(q + "self_att.w_bias.weight", 2 * c->reg_heads, false, &a.w_bias);
                b.add(q + "self_att.att.weight", (int64_t)4 * c->reg_d_model * D, true, &a.att);
                b.add(q + "self_att.ff.weight", (int64_t)D * c->reg_d_model, true, &a.ffw);
                b.add(q + "self_att.ff.bias", D, true, &a.ffb);
                b.add(q + "self_att.ln.weight", D, true, &a.lnw);
                b.add(q + "self_att.ln.bias", D, true, &a.lnb);
                ffn(b, q + "ff.", D, c->reg_d_ff, &e.ffn[l]);
            }
        }
        b.add("fc_head.0.weight", (int64_t)c->d_head * c->n_res * D, true, &L->fc0w);
        b.add("fc_head.0.bias", c->d_head, true, &L->fc0b);
        b.add("fc_head.2.weight", (int64_t)c->n_out * c->d_head, true, &L->fc2w);
        b.add("fc_head.2.bias", c->n_out, true, &L->fc2b);
        if (pass == 0) L->active = b.cursor;
    }
    L->total = b.cursor;
    L->embed_stride = c->n_res > 1 ? L->embed[1].lin_proj - L->embed[0].lin_proj : 0;
    L->pw_stride = c->n_res > 1 ? L->pw[1].lin_proj_p - L->pw[0].lin_proj_p : 0;
    L->reg_stride = c->n_res > 1 ? L->reg[1].att[0].att - L->reg[0].att[0].att : 0;
}

struct CfgKey {
    int32_t v[18];
    bool operator<(const CfgKey& o) const { return memcmp(v, o.v, sizeof(v)) < 0; }
};

}  // namespace

const ParamLayout& get_layout(const chromo_config_t* c) {
    // n_bins does not influence the parameter layout.
    static std::mutex mu;
    static std::map<CfgKey, ParamLayout*> cache;
    CfgKey k;
    memcpy(k.v, c, sizeof(k.v));
    std::lock_guard<std::mutex> g(mu);
    auto it = cache.find(k);
    if (it != cache.end()) return *it->second;
    ParamLayout* L = new ParamLayout();
    memset((void*)L->embed, 0, sizeof(L->embed));
    memset((void*)L->pw, 0, sizeof(L->pw));
    memset((void*)L->reg, 0, sizeof(L->reg));
    build(c, L);
    cache[k] = L;
    return *L;
}

WsLayout make_ws_layout(const chromo_config_t* c, int batch, int flags, bool replay, bool pairwise) {
    WsLayout w;
    memset(&w, 0, sizeof(w));
    const int B = batch, I = pairwise ? 1 : c->i_max, S = I + 1, D = c->d_emb;
    const int R = B * I, T = B * S;
    w.B = B; w.I = I; w.S = S; w.R = R; w.T = T; w.D = D;
    w.training = (flags & CHROMO_F_TRAINING) ? 1 : 0;
    w.pslots = w.training ? c->pw_layers : (c->pw_layers < 2 ? c->pw_layers : 2);
    w.rslots = w.training ? c->reg_layers : (c->reg_layers < 2 ? c->reg_layers : 2);
    int64_t cur = 0;
    auto take = [&](int64_t n) { int64_t o = cur; cur = align4(cur + n); return o; };
    const int He = c->embed_heads, Hp = c->pw_heads, Hr = c->reg_heads;
    // Batch-independent part first, so that packed weights survive a change of batch size
    // (CHROMO_F_PACKED).
    if (flags & CHROMO_F_BF16) {
        // BF16 mirror of the flat parameters in UMMA tile order (same element offsets) and
        // the packed position tables (PE [n,D] as a weight, and its transpose).
        w.bf_params = take((get_layout(c).total + 1) / 2 + 8);
        for (int r = 0; r < c->n_res; ++r) {
            const int64_t n16 = c->n_bins[r] <= 32 ? 32 : (c->n_bins[r] + 15) / 16 * 16;
            w.bf_pe[r] = take((n16 * D + 1) / 2 + 8);
            w.bf_pet[r] = take((n16 * D + 1) / 2 + 8);
        }
        w.bf_win[0] = take((int64_t)c->n_res * 1024);
        w.bf_win[1] = take((int64_t)c->n_res * 1024);
        if (!w.training) {
            int64_t off = 0;
            w.fold_slot[0] = off; off += (int64_t)2 * He * D * D;
            for (int l = 0; l < c->pw_layers; ++l) { w.fold_slot[1 + l] = off; off += (int64_t)2 * Hp * D * D; }
            w.fold_stride = off;
            w.fold_total = off * c->n_res;
            w.fold_f32 = take(w.fold_total);
            w.fold_bf = take((w.fold_total + 1) / 2 + 8);
            if (He * D == 256 && Hp * D == 256 && (c->embed_d_ff == 128 || c->embed_d_ff == 256) &&
                (c->pw_d_ff == 128 || c->pw_d_ff == 256)) {
                w.tail_fused = 1;
                w.tail_stream = take(((int64_t)c->n_res * (1 + c->pw_layers) * 6 * 128 * 128 + 1) / 2 + 8);
            }
            // fused Regulation layer: default geometry only (8 heads x 32, d_ff 256), i_max 8 or 16 (kernel is
            // specialised on the exact token count)
            if (c->reg_heads == 8 && c->reg_d_model == 256 && c->reg_d_ff == 256 && D == 128 && (c->i_max == 8 || c->i_max == 16)) {
                w.reg_fused = 1;
                w.reg_stream = take(((int64_t)c->n_res * c->reg_layers * 14 * 128 * 128 + 1) / 2 + 8);
            }
        }
    }
    // ---- per-resolution block
    const int64_t res_base = cur;
    if (!replay) {
    if (!pairwise) {
    w.e_hc = take((int64_t)B * D);
    w.e_q = take((int64_t)B * c->embed_d_model);
    w.e_qk = take((int64_t)B * He * D);
    w.e_qkt = take((int64_t)((B * He + 127) / 128) * 8192);
    w.e_cbar = take((int64_t)B * He * D);
    w.e_xbar = take((int64_t)B * He * 8);
    w.e_av = take((int64_t)B * c->embed_d_model);
    w.e_preU = take((int64_t)B * D);
    w.e_u = take((int64_t)B * D);
    w.e_f = take((int64_t)B * c->embed_d_ff);
    w.e_preY = take((int64_t)B * D);
    }   // !pairwise
    w.p_pp = take((int64_t)B * D);
    {
        int64_t s0 = cur;
        w.p_q = take((int64_t)R * c->pw_d_model) - s0;
        w.p_qk = take((int64_t)R * Hp * D) - s0;
        w.p_qkt = take((int64_t)((R * Hp + 127) / 128) * 8192) - s0;
        w.p_cbar = take((int64_t)R * Hp * D) - s0;
        w.p_xbar = take((int64_t)R * Hp * 8) - s0;
        w.p_av = take((int64_t)R * c->pw_d_model) - s0;
        w.p_preU = take((int64_t)R * D) - s0;
        w.p_u = take((int64_t)R * D) - s0;
        w.p_f = take((int64_t)R * c->pw_d_ff) - s0;
        w.p_preY = take((int64_t)R * D) - s0;
        w.p_out = take((int64_t)R * D) - s0;
        w.p_slot = cur - s0;
        // make offsets absolute for slot 0
        w.p_q += s0; w.p_qk += s0; w.p_qkt += s0; w.p_cbar += s0; w.p_xbar += s0; w.p_av += s0;
        w.p_preU += s0; w.p_u += s0; w.p_f += s0; w.p_preY += s0; w.p_out += s0;
        cur = s0 + w.p_slot * w.pslots;
    }
    }   // !replay
    if (!pairwise) {
    w.r_xin = take((int64_t)T * D);
    // a replay on the fused path (CHROMO_REG_FP32 sends the Regulation stage down the layer-by-layer path instead) needs
    // the last layer's rows (token 0 is what the head reads) and the parking slots of the plan's tiles
    w.reg_compact = replay && w.reg_fused && getenv("CHROMO_REG_FP32") == nullptr;
    if (w.reg_compact) {
        w.r_att = take((int64_t)T * D);
        w.r_out = cur;
        w.r_slot = align4((int64_t)ragged_reg_tiles_max(B, I) * 128 * D);
        cur += w.r_slot * w.rslots;
    } else {
        int64_t s0 = cur;
        w.r_proj = take((int64_t)T * 4 * c->reg_d_model);
        w.r_att = take((int64_t)T * c->reg_d_model);
        w.r_prob = take((int64_t)B * Hr * S * S);
        w.r_preU = take((int64_t)T * D);
        w.r_u = take((int64_t)T * D);
        w.r_f = take((int64_t)T * c->reg_d_ff);
        w.r_preY = take((int64_t)T * D);
        {   // (the fused multi-layer kernel parks whole 128-row tiles of floor(128 / S) genes here between layers)
            const int64_t G = 128 / S > 0 ? 128 / S : 1;
            const int64_t tiles = (B + G - 1) / G + 16;       // (+ the partly filled tiles of a ragged plan's token classes)
            w.r_out = take(std::max((int64_t)T * D, tiles * 128 * D));
        }
        w.r_slot = cur - s0;
        cur = s0 + w.r_slot * w.rslots;
    }
    }   // !pairwise
    w.res_stride = cur - res_base;
    cur = res_base + w.res_stride * c->n_res;
    // ---- resolution-dependent buffers
    for (int r = 0; r < c->n_res && !replay; ++r) {
        // rows may be padded to a multiple of 16 bins (tensor path for short rows, see single_query_attention)
        const int64_t n16 = (c->n_bins[r] + 15) / 16 * 16;
        if (!pairwise) w.e_p[r] = take((int64_t)B * He * n16);
        w.p_p_slot[r] = align4((int64_t)R * Hp * n16);
        w.p_p[r] = take(w.p_p_slot[r] * w.pslots);
    }
    if (!pairwise) {
        w.h_z = take((int64_t)B * c->n_res * D);
        w.h_h1 = take((int64_t)B * c->d_head);
    }
    if (w.tail_fused && !replay && !pairwise) w.rg_plan = take(ragged_plan_floats(B, I, c->n_res));
    w.g_base = cur;
    if (w.training) {
        // backward scratch, carved up in backward.cu: every gradient tensor of every layer has its own buffer (the
        // weight gradients are taken from them in one launch at the end of the pass)
        int64_t per_res = (int64_t)c->reg_layers * T * (4 * c->reg_d_model + c->reg_d_ff + 2 * D) +
                          (int64_t)T * (c->reg_d_model + 2 * D) +
                          (int64_t)c->pw_layers * R * (2 * Hp * D + 2 * c->pw_d_model + c->pw_d_ff + 2 * D + Hp * 8) +
                          (int64_t)R * 2 * D + (int64_t)B * D +
                          (int64_t)B * (2 * He * D + 2 * c->embed_d_model + c->embed_d_ff + 5 * D + He * 8) + 4096;
        int64_t nmax = 0;
        for (int r = 0; r < c->n_res; ++r) nmax = nmax > c->n_bins[r] ? nmax : c->n_bins[r];
        int64_t probs = (int64_t)R * Hp * nmax + (int64_t)B * He * nmax;
        cur += align4(per_res) * c->n_res + align4(probs) * c->n_res +
               (int64_t)B * (c->n_res * D + c->d_head + 64) + 1024;
    }
    w.total = cur;
    return w;
}

bool pdl_enabled() {
    static const bool on = getenv("CHROMO_NO_PDL") == nullptr;
    return on;
}

namespace {
struct SideStreams {
    int device = -1;
    cudaStream_t s[CHROMO_MAX_RES] = {};
    cudaEvent_t fork = nullptr, join[CHROMO_MAX_RES] = {};
};
SideStreams g_side[16];
}  // namespace

static SideStreams* side_streams() {
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 16) return nullptr;
    SideStreams& g = g_side[dev];
    if (g.device != dev) {
        for (int r = 1; r < CHROMO_MAX_RES; ++r) {
            if (cudaStreamCreateWithFlags(&g.s[r], cudaStreamNonBlocking) != cudaSuccess ||
                cudaEventCreateWithFlags(&g.join[r], cudaEventDisableTiming) != cudaSuccess) {
                set_error("cannot create the side streams");
                return nullptr;
            }
        }
        if (cudaEventCreateWithFlags(&g.fork, cudaEventDisableTiming) != cudaSuccess) {
            set_error("cannot create the fork event");
            return nullptr;
        }
        g.device = dev;
    }
    return &g;
}

int res_fork(cudaStream_t st, int n, ResStreams& rs) {
    rs.n = n;
    rs.s[0] = st;
    SideStreams* g = n >= 2 && n < CHROMO_MAX_RES ? side_streams() : nullptr;     // (the last side stream is aux_fork's)
    if (!g) {
        for (int r = 1; r < n; ++r) rs.s[r] = st;
        rs.n = 1;                                   // nothing to join
        return CHROMO_OK;
    }
    if (cudaEventRecord(g->fork, st) != cudaSuccess) { set_error("res_fork: event record failed"); return CHROMO_ECUDA; }
    for (int r = 1; r < n; ++r) {
        rs.s[r] = g->s[r];
        if (cudaStreamWaitEvent(g->s[r], g->fork, 0) != cudaSuccess) { set_error("res_fork: stream wait failed"); return CHROMO_ECUDA; }
    }
    return CHROMO_OK;
}

int aux_fork(cudaStream_t st, cudaStream_t* aux) {
    *aux = st;
    SideStreams* g = side_streams();
    if (!g) return CHROMO_OK;
    if (cudaEventRecord(g->fork, st) != cudaSuccess || cudaStreamWaitEvent(g->s[CHROMO_MAX_RES - 1], g->fork, 0) != cudaSuccess) {
        set_error("aux_fork: event record / wait failed");
        return CHROMO_ECUDA;
    }
    *aux = g->s[CHROMO_MAX_RES - 1];
    return CHROMO_OK;
}

int aux_join(cudaStream_t st, cudaStream_t aux) {
    if (aux == st) return CHROMO_OK;
    int dev = 0;
    cudaGetDevice(&dev);
    SideStreams& g = g_side[dev];
    if (cudaEventRecord(g.join[CHROMO_MAX_RES - 1], aux) != cudaSuccess ||
        cudaStreamWaitEvent(st, g.join[CHROMO_MAX_RES - 1], 0) != cudaSuccess) {
        set_error("aux_join: event record / wait failed");
        return CHROMO_ECUDA;
    }
    return CHROMO_OK;
}

int res_join(const ResStreams& rs) {
    if (rs.n < 2) return CHROMO_OK;
    int dev = 0;
    cudaGetDevice(&dev);
    SideStreams& g = g_side[dev];
    for (int r = 1; r < rs.n; ++r) {
        if (cudaEventRecord(g.join[r], rs.s[r]) != cudaSuccess || cudaStreamWaitEvent(rs.s[0], g.join[r], 0) != cudaSuccess) {
            set_error("res_join: event record / wait failed");
            return CHROMO_ECUDA;
        }
    }
    return CHROMO_OK;
}

}  // namespace chromo

using namespace chromo;

extern "C" {

int chromo_abi_version(void) { return CHROMO_ABI_VERSION; }
int chromo_debug_trace(int64_t* buf) {
    chromo::reg_fused_set_trace(reinterpret_cast<long long*>(buf));
    chromo::tc_gemm_set_trace(reinterpret_cast<long long*>(buf));
    return CHROMO_OK;
}
int64_t chromo_launch_counter(int32_t reset) { return chromo::launch_counter(reset != 0); }
const char* chromo_last_error(void) { return g_err; }

int64_t chromo_param_total(const chromo_config_t* cfg) {
    if (validate_config(cfg) != CHROMO_OK) return CHROMO_EINVAL;
    return get_layout(cfg).total;
}
int64_t chromo_param_active(const chromo_config_t* cfg) {
    if (validate_config(cfg) != CHROMO_OK) return CHROMO_EINVAL;
    return get_layout(cfg).active;
}
int32_t chromo_param_count(const chromo_config_t* cfg) {
    if (validate_config(cfg) != CHROMO_OK) return CHROMO_EINVAL;
    return (int32_t)get_layout(cfg).infos.size();
}
int64_t chromo_param_info(const chromo_config_t* cfg, int32_t idx, char* buf, int32_t buflen,
                          int64_t* numel) {
    if (validate_config(cfg) != CHROMO_OK) return CHROMO_EINVAL;
    const ParamLayout& L = get_layout(cfg);
    if (idx < 0 || idx >= (int32_t)L.infos.size()) { set_error("param index out of range"); return CHROMO_EINVAL; }
    const ParamInfo& p = L.infos[idx];
    if (buf && buflen > 0) { strncpy(buf, p.name.c_str(), buflen - 1); buf[buflen - 1] = 0; }
    if (numel) *numel = p.numel;
    return p.offset;
}
int64_t chromo_workspace_floats(const chromo_config_t* cfg, int32_t batch, int32_t flags) {
    if (validate_config(cfg) != CHROMO_OK) return CHROMO_EINVAL;
    if (batch < 1) { set_error("batch must be >= 1"); return CHROMO_EINVAL; }
    return make_ws_layout(cfg, batch, flags).total;
}

}  // extern "C"
