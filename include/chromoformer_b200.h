/*
 * chromoformer_b200.h — C ABI of libchromo_b200.so (sm_100a).
 *
 * The reference (dohlee/chromoformer) has no FFI layer: its hot path is the
 * PyTorch-eager forward of chromoformer/net.py + chromoformer/modules.py, the
 * autograd backward / torch.optim.AdamW step of chromoformer/train.py and the
 * numpy input path of chromoformer/data.py.  This header is the boundary a
 * maintainer binds instead of those ATen call sites (ctypes stub shown in
 * INTEGRATION.md).  Every entry point
 *   - takes plain device pointers, sizes and a cudaStream_t passed as void*,
 *   - never allocates, never synchronises the device, never touches the host
 *     copy of a tensor: workspaces are caller-owned device buffers,
 *   - returns 0 on success, a negative CHROMO_E* code otherwise
 *     (chromo_last_error() gives the text).
 *
 * All floating point tensors are FP32, row-major, contiguous unless a stride
 * argument says otherwise.  Masks are one byte per element (torch.bool).
 */
#ifndef CHROMOFORMER_B200_H
#define CHROMOFORMER_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CHROMO_ABI_VERSION 1
#define CHROMO_MAX_RES 4      /* resolutions (bin sizes) per model          */
#define CHROMO_MAX_LAYERS 8   /* layers per sub-transformer                 */

#define CHROMO_OK 0
#define CHROMO_EINVAL (-1)    /* unsupported configuration / bad argument   */
#define CHROMO_ENOMEM (-2)    /* workspace too small                        */
#define CHROMO_ECUDA (-3)     /* a CUDA launch failed                       */

/* flags for chromo_forward */
#define CHROMO_F_TRAINING 1   /* keep every activation the backward needs   */
#define CHROMO_F_BF16 2       /* dense projections on tcgen05 (BF16 operands,
                                 FP32 accumulate); default is strict FP32   */
#define CHROMO_F_REGONLY 8    /* internal */
#define CHROMO_F_BWD_HEAD_REG 16 /* chromo_backward: only the head + Regulation-transformer part of the pass (their
                                    gradients - the contiguous tail [first regulation tensor, active) of the flat buffer -
                                    are final when the call's work completes)                                            */
#define CHROMO_F_BWD_REST 32     /* chromo_backward: only the Pairwise + Embedding part; needs the other part first.
                                    Neither bit = the whole pass.  Data-parallel training all-reduces the first bucket
                                    under the second call (trainer.TrainStep).                                           */
#define CHROMO_F_PACKED 4     /* with CHROMO_F_BF16: the workspace already holds
                                 the packed BF16 weights of THESE parameters
                                 (left there by a previous call) - skip packing */
#define CHROMO_F_DENSE 64     /* hint: the batch carries no padding to speak of (every pCRE slot
                                 live, every bin valid), so the ragged plan of the BF16 inference
                                 path - dummy slots of data.py:175-203 leave the Pairwise and
                                 Regulation stages, padded bins of data.py:86-97 leave the attention
                                 windows - is not built.  Results do not depend on the hint.     */
#define CHROMO_F_FREQ_GRAD 128 /* chromo_backward_inputs: also write d interaction_freq to dx->freq */

/* Hyper-parameters: the config.yaml schema of chromoformer/configs/default.yaml:11-32
 * plus the number of bins per resolution (w_max // binsize, data.py:140).     */
typedef struct chromo_config {
    int32_t n_feats;      /* 7 histone marks                         net.py:276 */
    int32_t d_emb;        /* 128                                     net.py:277 */
    int32_t d_head;       /* 128  fc_head hidden width               net.py:278 */
    int32_t n_out;        /* 2 = classifier (net.py:329), 1 = regressor (net.py:427) */
    int32_t n_res;        /* number of bin sizes, 3                  net.py:297 */
    int32_t i_max;        /* pCRE slots per gene, 8                  data.py:30 */
    int32_t embed_layers, embed_heads, embed_d_model, embed_d_ff;   /* net.py:279-284 */
    int32_t pw_layers, pw_heads, pw_d_model, pw_d_ff;               /* net.py:285-290 */
    int32_t reg_layers, reg_heads, reg_d_model, reg_d_ff;           /* net.py:291-296 */
    int32_t n_bins[CHROMO_MAX_RES];   /* 20, 80, 400 for bin sizes 2000, 500, 100 */
} chromo_config_t;

/* One batch of genes as ChromoformerBase.forward receives it (net.py:332-340).
 * Only the centre query row (bin n/2) of each pad mask can influence the
 * logits (net.py:59, net.py:138), so a mask is described by a base pointer, a
 * per-region stride and the byte offset of that row:
 *   full  [B,I,1,n,n] bool tensor : stride = n*n, row_offset = (n/2)*n
 *   compact [B,I,n] centre rows   : stride = n,   row_offset = 0            */
typedef struct chromo_batch {
    int32_t batch;                                   /* genes B                          */
    const float*   x_p[CHROMO_MAX_RES];              /* [B,1,n,F]  promoter_feats[r]     */
    const float*   x_pcre[CHROMO_MAX_RES];           /* [B,I,n,F]  pcre_feats[r]         */
    const uint8_t* mask_p[CHROMO_MAX_RES];           /* promoter_pad_masks[r]            */
    int64_t        mask_p_stride[CHROMO_MAX_RES];
    int64_t        mask_p_row_offset[CHROMO_MAX_RES];
    const uint8_t* mask_pcre[CHROMO_MAX_RES];        /* pcre_pad_masks[r]                */
    int64_t        mask_pcre_stride[CHROMO_MAX_RES];
    int64_t        mask_pcre_row_offset[CHROMO_MAX_RES];
    const uint8_t* imask[CHROMO_MAX_RES];            /* [B,1,S,S]  interaction_masks[r]  */
    const float*   freq;                             /* [B,S,S]    interaction_freq      */
    const float*   pos_enc[CHROMO_MAX_RES];          /* [n,d_emb]  sinusoid table, net.py:23-29 */
} chromo_batch_t;

/* ---- library / layout ---------------------------------------------------- */
int         chromo_abi_version(void);
const char* chromo_last_error(void);

/* Flat FP32 parameter buffer.  Tensors that receive gradients come first
 * ([0, chromo_param_active)), the 36 structurally unused ones (w_bias.weight,
 * embed/pairwise gamma_f, pairwise ln.*; SURVEY A.4) after them.  Names are the
 * reference state_dict keys of the dict layout (SURVEY A.3), e.g.
 * "regulation.2.transformer.layers.0.self_att.att.weight" with the resolution
 * given as its INDEX (0..n_res-1), not its bin size.                          */
int64_t chromo_param_total(const chromo_config_t* cfg);
int64_t chromo_param_active(const chromo_config_t* cfg);
int32_t chromo_param_count(const chromo_config_t* cfg);
/* name of tensor idx into buf; returns its offset (floats), numel in *numel  */
int64_t chromo_param_info(const chromo_config_t* cfg, int32_t idx, char* buf, int32_t buflen,
                          int64_t* numel);

/* ---- forward: net.py:332-380 (and the flat-API twin net.py:228-270) ------- */
int64_t chromo_workspace_floats(const chromo_config_t* cfg, int32_t batch, int32_t flags);
int chromo_forward(const chromo_config_t* cfg, const float* params, const chromo_batch_t* in,
                   float* logits /* [B,n_out] */, float* workspace, int64_t workspace_floats,
                   int32_t flags, void* stream);

/* ---- in-silico pCRE deletion: the exact effect of removing each pCRE of each gene -------------------------------
 * For B genes with I = i_max slots (S = I + 1 tokens).  Slot i of gene g is LIVE when token i + 1 is unmasked in row 0
 * of at least one resolution's interaction mask, DEAD otherwise (the dummy slots of data.py:175-203).
 *   logits[g]          the ordinary forward, bit-identical to chromo_forward with the same flags;
 *   without[g, i]      live slot: the logits with row and column i + 1 of every resolution's interaction mask set, which
 *                      is the gene reassembled without pCRE i; dead slot: logits[g], bit for bit;
 *   promoter_only[g]   the logits with tokens 1..I masked in every resolution (the gene with no pCRE at all).
 * One Embedding + Pairwise pass serves every deletion of a gene (slot i's Pairwise output depends on the promoter and
 * pCRE i only); the Regulation transformer and the head then run over V = B * (I + 1) variants whose live tokens come
 * first, so that the BF16 path's ragged plan packs them into the token class below the gene's.  Every output element is
 * written; no atomics on the floating-point path; identical inputs give identical outputs; no host synchronisation
 * (legal inside a stream capture).  Flags: CHROMO_F_BF16, CHROMO_F_PACKED (as for chromo_forward) and the
 * CHROMO_F_DENSE hint (the gene pass only); any other flag, or a NULL output, is CHROMO_EINVAL.  The workspace must hold
 * chromo_pcre_deletion_workspace_floats floats (CHROMO_ENOMEM otherwise); it is not interchangeable with a
 * chromo_forward workspace, except that it too keeps the packed BF16 weights at its front.                        */
int64_t chromo_pcre_deletion_workspace_floats(const chromo_config_t* cfg, int32_t batch, int32_t flags);
int chromo_pcre_deletion(const chromo_config_t* cfg, const float* params, const chromo_batch_t* in,
                         float* logits /* [B,n_out] */, float* without /* [B,I,n_out] */,
                         float* promoter_only /* [B,n_out] */, float* workspace, int64_t workspace_floats,
                         int32_t flags, void* stream);

/* ---- one Regulation-transformer layer: AttentionBlock with gate (modules.py:104-111 as used by
 * net.py:152-153), for every resolution at once: y[r] = layer(x[r]), x/y = [n_res][B*(i_max+1), d_emb] FP32
 * with `xy_stride` floats between resolutions.  With CHROMO_F_BF16 and the default geometry this is ONE
 * fused tcgen05 kernel per call (reg_fused.cu); otherwise the FP32 kernels.  Inference only.
 * layer < 0 (fused BF16 kernel only): the whole Regulation transformer, y = layer_{L-1}(...layer_0(x)), in ONE
 * launch, as the BF16 forward runs it (a CTA keeps its genes on chip from layer to layer).              */
int chromo_regulation_layer(const chromo_config_t* cfg, const float* params, int32_t layer, const float* x,
                            float* y, int64_t xy_stride, const uint8_t* const* imask /* n_res x [B,S,S] */,
                            const float* freq /* [B,S,S] */, int32_t batch, float* workspace,
                            int64_t workspace_floats, int32_t flags, void* stream);

/* ---- single-query attention core of the Embedding / Pairwise Interaction transformers --------------
 * For every (region, head) row: the attention of ONE query over the n bins of the region, with keys and
 * values W_in x_j + PE_j (net.py:31-59 and 105-139 feed modules.py:16-30 / 150-170 this way; only the
 * centre query is consumed downstream):
 *   s_j = scale * qk[row] . (W_in x[region, j] + PE_j);  masked j -> -1e9;  p = softmax_j(s)
 *   cbar[row] = sum_j p_j (W_in x[region, j] + PE_j)
 * qk [regions*2, 128] (= W_k[h]^T q per head), x [regions, n, 7], mask [regions, n] bytes (non-zero = pad),
 * w_in [128, 7], pos_enc [n, 128], cbar [regions*2, 128]; n % 4 == 0, n <= 400.  BF16 tensor path only
 * (sqa_fused.cu): the kernel the BF16 forward runs per stage, exposed to be tested and timed alone.
 * workspace: at least 64 * max(32, round_up(n, 16)) + 1024 + 8192 * ceil(regions / 64) floats (the position table,
 * W_in and the qk rows as BF16 tensor-core operands).                                                */
int chromo_single_query_attention(int32_t regions, int32_t n, const float* qk, const float* x, const uint8_t* mask,
                                  const float* w_in, const float* pos_enc, float scale, float* cbar,
                                  float* workspace, int64_t workspace_floats, void* stream);

/* ---- one dense layer: nn.Linear (+ReLU) as at modules.py:38,100,159-160, net.py:326-330 --
 * y[z] = act(x[z] W[z]^T + b[z]) for z < batches; x [m,k], W [n,k], y [m,n] row-major.
 * The same kernel the forward uses for every projection; exposed so that a single
 * contraction can be tested and timed in isolation.                                    */
int chromo_linear(const float* x, const float* w, const float* bias, float* y, int32_t m, int32_t n,
                  int32_t k, int32_t relu, int32_t batches, int64_t x_stride, int64_t w_stride,
                  int64_t bias_stride, int64_t y_stride, int32_t flags, void* stream);
/* With CHROMO_F_BF16, `w` of chromo_linear must point at weights packed by this call
 * (BF16, UMMA K-major core-matrix tiles; n*k elements per batch, same strides in elements). */
int chromo_pack_linear_weight(const float* w, uint16_t* packed, int32_t n, int32_t k, int32_t batches,
                              int64_t w_stride, void* stream);

/* Profiling hook: while `buf` (device memory, 1536 int64, zero-filled by the caller) is set, CTA (0,0) of every fused
 * Regulation launch logs (event id << 48 | clock64) for its driver thread ([0,512)), one score warp ([512,1024)) and one
 * value warp ([1024,1536)); NULL switches it off.  tools/reg_timeline.py prints the timeline. */
int chromo_debug_trace(int64_t* buf);

/* Number of kernel launches issued by this library since the last reset (process-wide). */
int64_t chromo_launch_counter(int32_t reset);

/* ---- backward: autograd of the same graph (train.py:195) ------------------
 * `workspace` must be the buffer a CHROMO_F_TRAINING forward of the same batch
 * filled.  grads ([chromo_param_total] floats) is ACCUMULATED into (+=).       */
int chromo_backward(const chromo_config_t* cfg, const float* params, const chromo_batch_t* in,
                    const float* dlogits /* [B,n_out] */, float* grads, float* workspace,
                    int64_t workspace_floats, int32_t flags, void* stream);

/* ---- gradients with respect to the inputs (saliency, integrated gradients) ------------------------------------
 * The same pass as chromo_backward (same CHROMO_F_TRAINING workspace of the same batch, CHROMO_F_BF16 honoured)
 * that also WRITES (=) the gradient of the histone-mark features of every resolution whose pointer is non-NULL:
 * every element, zeros on padded bins and dummy pCRE slots included.  With CHROMO_F_FREQ_GRAD in flags it also
 * WRITES (=) the gradient of interaction_freq to dx->freq (non-NULL then), every element, zeros wherever the
 * interaction mask of every resolution is set; without the flag dx->freq is never read, so callers built against
 * the struct without that member keep working.  grads == NULL: no parameter gradient at all (no weight / bias
 * contraction runs), otherwise grads is accumulated into exactly as by chromo_backward; with grads == NULL and no
 * feature pointer the pass ends after the Regulation transformer.  The masks and the position tables get no
 * gradient.  CHROMO_F_BWD_HEAD_REG / CHROMO_F_BWD_REST are rejected (CHROMO_EINVAL).                           */
typedef struct chromo_input_grads {
    float* x_p[CHROMO_MAX_RES];       /* [B,1,n_r,F], written (=) when non-NULL */
    float* x_pcre[CHROMO_MAX_RES];    /* [B,I,n_r,F], written (=) when non-NULL */
    float* freq;                      /* [B,S,S], written (=) with CHROMO_F_FREQ_GRAD; read only then */
} chromo_input_grads_t;
int chromo_backward_inputs(const chromo_config_t* cfg, const float* params, const chromo_batch_t* in,
                           const float* dlogits /* [B,n_out] */, float* grads /* NULL: no parameter gradient */,
                           const chromo_input_grads_t* dx, float* workspace, int64_t workspace_floats,
                           int32_t flags, void* stream);

/* ---- the contraction of the training step on the tensor pipe (train.py:195: autograd of nn.Linear) --------
 * C[M,N] (=|+=) opA . opB^T with BF16 operands converted on the fly and FP32 accumulation (tcgen05 / TMEM):
 *   a_transposed = 0: A is [M,K] (ld lda); 1: A is [K,M]        b_transposed = 0: B is [N,K] (ld ldb); 1: B is [K,N]
 * data gradient  dX = dY W   : chromo_matmul(dY, ., 0, W, ., 1, dX, ...)    (W [N_out, K_in] as stored by nn.Linear)
 * weight gradient dW += dY^T X: chromo_matmul(dY, ., 1, X, ., 1, dW, ..., accumulate = 1, ksplit = token chunks)
 * chromo_backward routes every qualifying contraction through this kernel when CHROMO_F_BF16 is set.  N % 16 == 0,
 * leading dimensions % 4 == 0, 16-byte aligned pointers; ksplit > 1 needs accumulate (FP32 atomics).            */
int chromo_matmul(const float* A, int64_t lda, int32_t a_transposed, const float* B, int64_t ldb, int32_t b_transposed,
                  float* C, int64_t ldc, int32_t M, int32_t N, int32_t K, int32_t accumulate, int32_t ksplit, void* stream);

/* ---- losses: train.py:156,193 (mean reduction); write loss[0] and dlogits -- */
int chromo_mse_loss(const float* logits, const float* target, int32_t count, float grad_scale,
                    float* loss, float* dlogits, void* stream);
int chromo_ce_loss(const float* logits, const int64_t* labels, int32_t batch, int32_t n_classes,
                   float grad_scale, float* loss, float* dlogits, void* stream);

/* ---- fused AdamW: torch.optim.AdamW as used at train.py:157,196 ------------
 * One launch over a flat range: decoupled weight decay, bias correction from
 * `step` (1-based), grads optionally pre-scaled (DP mean).                    */
int chromo_adamw(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                 int64_t count, float lr, float beta1, float beta2, float eps,
                 float weight_decay, int32_t step, float grad_scale, void* stream);

/* ---- validation metrics on the device: train.py:198-251 (training log) and 286-320 (validation) --------------
 * Replaces out.cpu() + sklearn.metrics.{accuracy_score, roc_auc_score, average_precision_score} / r2_score +
 * scipy.stats.pearsonr.  Rank statistics are exact pair counts (ties as sklearn treats them), sums in FP64.
 * chromo_clf_metrics: logits [n, n_out] (n_out >= 2), labels int64 [n]; writes score[n] = softmax(logits)[:, 1]
 *   (the `val_score` the checkpoint keeps, train.py:322-343) and out[4] = {accuracy, AUROC, average precision,
 *   #positives}; `scratch` = 32 bytes of device memory.
 * chromo_reg_metrics: pred, labels FP32 [n]; out[3] = {r2_score(labels, pred), pearsonr, MSE}.
 * Fractions, not percent.  Asynchronous on `stream`; nothing is copied to the host.                              */
int chromo_clf_metrics(const float* logits, const int64_t* labels, int32_t n, int32_t n_out, float* score,
                       double* out, void* scratch, void* stream);
int chromo_reg_metrics(const float* pred, const float* labels, int32_t n, double* out, void* stream);

/* ---- input path: data.py:68-113 -------------------------------------------
 * Bins raw per-bp depth (FP16 [F,L] per region, regions concatenated in one
 * device buffer) at every resolution: mean over <=bin bp, ln(x+1), centre pad,
 * optional strand flip; writes feats[r] as [regions,n_r,F] and the valid-bin
 * span (left_pad, n_bins) per region and resolution.                          */
typedef struct chromo_region {
    int64_t offset;     /* element offset of this region's [F,L] block in `raw`      */
    int32_t length;     /* L in bp (row stride)                                       */
    int32_t start;      /* first bp used (crop, data.py:106-107)                      */
    int32_t width;      /* bp used after cropping                                     */
    int32_t flip;       /* 1 = '-' strand promoter (data.py:110-113)                  */
} chromo_region_t;
int chromo_bin_regions(const uint16_t* raw /* fp16 bits */, const chromo_region_t* regions,
                       int32_t n_regions, int32_t n_feats, int32_t n_res,
                       const int32_t* bin_sizes, const int32_t* n_bins,
                       float* const* feats /* n_res device ptrs */, int32_t* spans /* [n_res,regions,2] */,
                       void* stream);

/* ---- host -> device transport: run_demo.py:100-105 / train.py:172-177 -------
 * The reference ships every tensor of a batch with `.cuda()`: FP32 features and
 * n x n boolean masks, 1.63 MB per gene.  The wire format of this library is
 * FP16 features (the raw depth is FP16 on disk; ln(mean+1) rounds at 2^-11) and
 * (first valid bin, count) spans instead of pad masks: 64 kB per gene.  This
 * call widens n_seg feature tensors to the FP32 layout chromo_forward consumes
 * and expands n_sets span arrays ([rows,2] int32) to centre-row pad masks
 * ([rows,n_bins] bytes, 1 = padded), all in one launch.  Pointer ARRAYS are
 * host memory; what they point at is device memory, 16-byte aligned.          */
int chromo_unpack_wire(int32_t n_seg, const uint16_t* const* src /* fp16 bits */, float* const* dst,
                       const int64_t* counts, int32_t n_sets, const int32_t* const* spans,
                       uint8_t* const* masks, const int32_t* rows, const int32_t* n_bins, void* stream);

/* Compact wire for ragged genes (run_demo.py:100-105 again): data.py:86-97 pads every region to
 * w_max / bin_size bins with zeros, so only the valid bins need to cross PCIe - 14 kB per gene of the demo
 * set instead of 64 kB.  For each of n_sets feature tensors: `src` holds the valid bins of its regions
 * back to back (FP16 [bins, n_feats], region order), `offsets[row]` the first bin of region `row` in the
 * whole stream and `base` the stream position `src` starts at (a chunk of a longer stream), `spans`
 * ([rows,2] int32: first valid bin, count) where the bins belong.  `dst` (FP32 [rows, n_bins, n_feats]) is
 * written completely: the bins at their place, zeros elsewhere.                                  */
int chromo_unpack_compact(int32_t n_sets, const uint16_t* const* src /* fp16 bits */, const int32_t* const* spans,
                          const int32_t* const* offsets, const int32_t* base, float* const* dst,
                          const int32_t* rows, const int32_t* n_bins, int32_t n_feats, void* stream);

/* Zero-suppressed wire: ln(mean + 1) of binned read depth is exactly 0 wherever no read fell (37 % of
 * the demo's bins; data.py:75-80).  A feature tensor of `count` values travels as `bits` (one bit per
 * value, little-endian in 32-bit words), its non-zero values `vals` (FP16, in order) and `offsets` (the
 * number of non-zeros in front of every block of 1024 values, counted over the whole stream; `base` = that
 * count at the position `vals` starts at).  `dst` (FP32, `count` values, 16-byte aligned) is written
 * completely.  Lossless; 44 kB instead of 64 kB per gene at the demo's statistics.                 */
int chromo_unpack_sparse(int32_t n_seg, const uint32_t* const* bits, const uint16_t* const* vals /* fp16 bits */,
                         const int32_t* const* offsets, const int32_t* base, float* const* dst,
                         const int64_t* counts, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CHROMOFORMER_B200_H */
