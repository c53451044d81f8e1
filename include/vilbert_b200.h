/* vilbert_b200 -- C ABI of the B200-native ViLBERT multi-task forward.
 *
 * The reference has no FFI for this path: its boundary is the Python object protocol that
 * /root/reference/worker.py fixes (SURVEY.md section 8b):
 *     config = BertConfig.from_json_file(...)                          worker.py:495, 506-522
 *     model  = VILBertForVLTasks.from_pretrained(ckpt, config=config,
 *                                                num_labels=3129, ...) worker.py:530-532
 *     model.eval(); model.cuda(0)                                      worker.py:534-536
 *     out10  = model(question, features, spatials, segment_ids, input_mask, image_mask,
 *                    co_attention_mask, task_tokens, output_all_attention_masks=True)
 *                                                                      worker.py:286-289
 * The entry points below are exactly what a binding for that protocol needs, and nothing else:
 * vb200_create <- from_pretrained + cuda(i); vb200_forward <- __call__; vb200_destroy <- del.
 * The Python shim in vilbert-multi-task_b200/ (ctypes) implements the protocol on top of them; see
 * INTEGRATION.md for the stub a maintainer of the reference would add.
 *
 * Conventions: plain pointers and sizes, no C++/torch types; every function returns 0 on success or a
 * negative vb200_status; no exception crosses the boundary; vb200_last_error() returns the message of the
 * last failure on that handle (or of the last failed vb200_create when handle == NULL).
 * vb200_forward is asynchronous on the caller's stream (no hidden synchronisation); input and output
 * buffers are owned by the caller; one handle serves one stream at a time (workspaces are per handle).
 */
#ifndef VILBERT_B200_H
#define VILBERT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VB200_ABI_VERSION 2

typedef struct vb200_engine* vb200_handle;

typedef enum {
    VB200_OK = 0,
    VB200_ERR_INVALID = -1,      /* bad argument / unsupported shape */
    VB200_ERR_CONFIG = -2,       /* config JSON could not be parsed or is unsupported */
    VB200_ERR_CHECKPOINT = -3,   /* missing / unexpected / mis-shaped state_dict entry */
    VB200_ERR_CUDA = -4,         /* CUDA runtime or driver error (message has the detail) */
    VB200_ERR_NO_DEVICE = -5     /* no sm_100 device: there is deliberately no CPU fallback */
} vb200_status;

typedef enum { VB200_F32 = 0, VB200_F16 = 1, VB200_BF16 = 2 } vb200_dtype;

/* One entry of the flat checkpoint state_dict (worker.py:470, 530-532): upstream key name, host pointer. */
typedef struct {
    const char* name;        /* e.g. "bert.encoder.c_layer.3.biattention.query1.weight" ("module." prefix accepted) */
    int32_t dtype;           /* vb200_dtype */
    int32_t ndim;            /* 1 or 2 */
    int64_t shape[2];        /* nn.Linear weights are [out, in] row-major */
    const void* data;        /* host memory, contiguous */
} vb200_tensor;

/* Which elements of the reference's 10-tuple (worker.py:287) to compute. */
enum {
    VB200_OUT_VIL_PREDICTION = 1 << 0,         /* [B, num_labels]  VQA / VG-QA            worker.py:296 */
    VB200_OUT_VIL_PREDICTION_GQA = 1 << 1,     /* [B, 1533]        GQA                    worker.py:313 */
    VB200_OUT_VIL_LOGIT = 1 << 2,              /* [B, 1]           retrieval              worker.py:359 */
    VB200_OUT_VIL_BINARY_PREDICTION = 1 << 3,  /* [B/2, 2] (B even) / [B, 2] (B odd)  NLVR2  worker.py:329 */
    VB200_OUT_VIL_TRI_PREDICTION = 1 << 4,     /* [B, 3]           SNLI-VE                worker.py:345 */
    VB200_OUT_VISION_PREDICTION = 1 << 5,      /* [B, V, v_target_size]  pre-training head, unused by the worker */
    VB200_OUT_VISION_LOGIT = 1 << 6,           /* [B, V, 1]        grounding              worker.py:374 */
    VB200_OUT_LINGUISIC_PREDICTION = 1 << 7,   /* [B, T, vocab]    pre-training head, unused by the worker */
    VB200_OUT_LINGUISIC_LOGIT = 1 << 8,        /* [B, T, 1]        never read by the worker */
    VB200_OUT_TASK_HEADS = 0x15F,              /* the seven task heads (everything but the two pre-training heads) */
    VB200_OUT_ALL = 0x1FF,
    VB200_OUT_ATTENTION = 1 << 9               /* element 9 of the tuple, attn_data_list: the attention probabilities of all 24 layers
                                                  (worker.py:287-288; the reference returns them because config.visualization is set,
                                                  worker.py:522, and never reads them).  Off unless requested: see
                                                  vb200_attention_layout and vb200_outputs.attention_probs. */
};

/* Inputs of one forward, in the dtypes the worker builds them (worker.py:416-419, 452-455).
 * T = Tin + 1 when config.task_specific_tokens (worker.py:516-517).  co_attention_mask is accepted for
 * signature compatibility and ignored, as upstream ignores it (worker passes zeros, worker.py:455). */
typedef struct {
    int32_t batch;                 /* B  */
    int32_t n_tokens;              /* Tin */
    int32_t n_regions;             /* V  */
    const int64_t* question;       /* [B, Tin] token ids */
    const float* features;         /* [B, V, v_feature_size] */
    const float* spatials;         /* [B, V, 5] */
    const int64_t* segment_ids;    /* [B, Tin] */
    const int64_t* input_mask;     /* [B, Tin] */
    const uint8_t* image_mask;     /* [B, V] */
    const float* co_attention_mask;/* [B, V, Tin] or NULL; ignored */
    const int64_t* task_tokens;    /* [B, 1] */
} vb200_inputs;

/* Caller-allocated fp32 outputs; a NULL pointer (or a cleared select bit) skips that output. */
typedef struct {
    float* vil_prediction;         /* [B, num_labels] */
    float* vil_prediction_gqa;     /* [B, gqa_labels] */
    float* vil_logit;              /* [B, 1] */
    float* vil_binary_prediction;  /* [B/2, 2] if B even else [B, 2] */
    float* vil_tri_prediction;     /* [B, 3] */
    float* vision_prediction;      /* [B, V, v_target_size] */
    float* vision_logit;           /* [B, V, 1] */
    float* linguisic_prediction;   /* [B, T, vocab] */
    float* linguisic_logit;        /* [B, T, 1] */
    float* sequence_output_t;      /* optional debug tap: final text stream  [B, T, hidden]   (fp32) */
    float* sequence_output_v;      /* optional debug tap: final image stream [B, V, v_hidden] (fp32).  Without a per-row head or
                                      a sequence tap of a stream, its last layer (when it follows the last connection layer) runs
                                      on row 0 of each sample only -- all the poolers read; asking for a tap keeps the full layer */
    float* pooled_output;          /* optional debug tap: pooled_t * pooled_v [B, bi_hidden] */
    float* attention_probs;        /* VB200_OUT_ATTENTION: one flat fp32 buffer holding every layer's softmax probabilities
                                      [B, heads, Lq, Lk] back to back in execution order (vb200_attention_layout gives the
                                      offsets); NULL skips the copy */
} vb200_outputs;

/* Engine options (all optional; zero-initialise for defaults).  Flags are tri-state: 0 default, 1 on, -1 off. */
typedef struct {
    int32_t device;                /* CUDA ordinal */
    int32_t num_labels;            /* vil_prediction width; 0 -> taken from the checkpoint (worker.py:523: 3129) */
    int32_t use_cuda_graph;        /* default on: each (B,Tin,V,select) plan is captured once and replayed */
    int32_t use_pdl;               /* programmatic dependent launch: 0 default (= every kernel), > 0 every kernel, < 0 none */
    int32_t strict;                /* default on: unexpected checkpoint keys are an error */
    int32_t act_fp16;              /* 16-bit format of the tensor-core operands (weights AND activations; tcgen05 kind::f16
                                      needs matching A/B formats).  default on: IEEE fp16 (11-bit significand; activations
                                      are LayerNorm-bounded, converts saturate); -1: bf16.  Accumulation, residual stream,
                                      LayerNorm, softmax and logits are fp32 either way. */
    int32_t fused_layernorm;       /* default off: LayerNorm(dense(x) + residual) runs as GEMM (fp32 out) + an L2-resident row
                                      kernel; 1: cluster-LayerNorm GEMM epilogue (N tiles of a row-panel form a thread-block
                                      cluster and exchange (mean, M2) through distributed shared memory).  Both are
                                      parity-tested; the split form measured faster on B200 at every batch tried. */
    int32_t split_fp32;            /* 1: fp32-parity mode ("fp32x").  Every GEMM operand travels as TWO fp16 numbers (hi = fp16(x),
                                      lo = fp16(x - hi), 22 significand bits); operand buffers hold hi | lo | hi (weights hi | hi |
                                      lo) per 64 columns, so an ordinary tcgen05 GEMM over K' = 3K adds hi.hi + lo.hi + hi.lo in its
                                      fp32 accumulator; attention runs in fp32 on CUDA cores; GELU uses the 1.5e-7 erf.  3x the
                                      tensor work of the default mode -- for logit parity with the reference's fp32 forward
                                      (<= 1e-3 per logit, BASELINE.json north_star), not for throughput.  Implies act_fp16. */
    int32_t ln_fold;               /* 1: LayerNorm folded into the GEMMs around it (default off).  The GEMM that produces
                                      u = dense(x) + residual writes u (fp32 + 16-bit) and per-row (mean, M2) statistics instead of
                                      LayerNorm(u); the next GEMM runs on u with weights pre-scaled by gamma and finishes with
                                      rstd * (acc - mean * s) + c; residual readers rebuild LayerNorm(u) on the fly.  Same math,
                                      57 of a forward's 62 LayerNorm launches gone -- but measured SLOWER on B200 at batch 64
                                      (the extra epilogue work exceeds the row kernels it replaces, profiles/r2_ln_fold.md), so
                                      it is an option, parity-tested, not the default.  Ignored in split_fp32 / fused_layernorm. */
    int32_t max_plans;             /* plan-cache bound: plans (workspace + CUDA graph per (batch, tokens, regions, select, slot))
                                      beyond this are evicted least-recently-used; 0 -> 24 */
} vb200_options;

int vb200_abi_version(void);

/* from_pretrained + cuda(device): parse the BertConfig JSON, audit the state_dict against the upstream key list,
 * repack weights to device (16-bit GEMM operands in the format vb200_options::act_fp16 selects -- fp16 by default, bf16, or the
 * fp16 hi/lo pairs of split_fp32 -- and fp32 LayerNorm / bias / embedding tables). */
int vb200_create(const char* config_json, int64_t n_tensors, const vb200_tensor* tensors, const vb200_options* opt,
                 vb200_handle* out);
int vb200_destroy(vb200_handle h);
const char* vb200_last_error(vb200_handle h);

/* Device-pointer forward (what worker.py:286-289 does): all vb200_inputs / vb200_outputs pointers are device
 * memory on the engine's device; enqueued on `cuda_stream` (a cudaStream_t passed as void*).
 * Synchronisation: a call whose (batch, n_tokens, n_regions, select, slot) plan already exists only enqueues work and returns.
 * The FIRST call of a shape builds its plan: cudaMalloc of the workspace, one eager validation pass with a stream
 * synchronisation, and the CUDA-graph capture -- it blocks the host for some milliseconds and may synchronise the device (also
 * when the plan cache evicts an old plan, vb200_options::max_plans).  Warm a server's shapes up before taking traffic. */
int vb200_forward(vb200_handle h, const vb200_inputs* in, const vb200_outputs* out, uint32_t select, void* cuda_stream);

/* Same with an explicit workspace slot (0..15): forwards on DIFFERENT slots may run concurrently on different streams (each
 * slot owns its workspace, TMA descriptors and captured graph; weights are shared) -- how a server keeps more than one batch in
 * flight so kernels of one batch fill the SMs another leaves idle.  vb200_forward is slot 0. */
int vb200_forward_slot(vb200_handle h, const vb200_inputs* in, const vb200_outputs* out, uint32_t select, int32_t slot,
                       void* cuda_stream);

/* Host-pointer forward: same, but every pointer is HOST memory (pinned for full speed); copies in, runs, copies
 * the selected outputs back and synchronises the stream before returning. */
int vb200_forward_host(vb200_handle h, const vb200_inputs* in, const vb200_outputs* out, uint32_t select,
                       void* cuda_stream);

/* Same on workspace slot `slot`; synchronize = 0 returns right after enqueueing (H2D copies, kernels and D2H copies are
 * ordered on `cuda_stream`; the host buffers must stay valid and the outputs are complete once the caller has synchronised
 * that stream).  Two slots on two streams overlap one batch's copies with the other's kernels. */
int vb200_forward_host_slot(vb200_handle h, const vb200_inputs* in, const vb200_outputs* out, uint32_t select, int32_t slot,
                            int32_t synchronize, void* cuda_stream);

/* Introspection used by the tests / bench: number of kernels one forward of this shape launches,
 * FLOPs it executes (a pruned tail counts its B-row work), model dimensions. */
int vb200_plan_info(vb200_handle h, int32_t batch, int32_t n_tokens, int32_t n_regions, uint32_t select,
                    int64_t* n_launches, double* flops);
int vb200_model_dim(vb200_handle h, const char* key, int64_t* value);
/* Run-time knobs: "max_plans" (plan-cache bound); "profile_grid_pct" (0 or 10..100): the NEXT vb200_profile_ops call launches every
 * GEMM with this percentage of the resident CTA slots as its persistent grid (production: two thirds, profiles/r2_grid_size.md) --
 * for reporting what a launch does when it has the GPU to itself; forwards are never affected.  "chain_ffn" (0/1): issue every
 * FFN-in -> FFN-out pair as ONE chained persistent launch (csrc/gemm_chain.cu: dynamic tile list + per-row-panel dependency counters;
 * same bits, measured slower at batch 64, profiles/r2_chain.md -> off by default); changing it drains the device and drops cached plans.
 * "prune_tail" (0/1, default 1, env VB200_PRUNE=0): run a stream's last layer after the last connection layer on the pooled rows only
 * when no selected output reads that stream's sequence (same bits; for A/B runs); changing it drains the device and drops cached plans. */
int vb200_set_option(vb200_handle h, const char* key, int64_t value);
/* Profiling: after vb200_set_option(h, "timeline", 1) every tcgen05 GEMM launch of a forward records 16 stamps per CTA (0: clock64 at
 * entry, 1: setup done, 2: first k-block landed [-DVB200_STAMPS builds], 8 / 9: %globaltimer ns at entry / exit, 10: last MMA committed,
 * 11: tiles walked, 12: SM id).  Copies the stamps of the LAST forward run on (shape, select, slot): stamps[n_ops][304][16],
 * dims[n_ops][4] = M, N, K, graph branch.  Synchronises the device.  scripts/step_timeline.py turns two slots' worth into per-SM
 * occupancy figures. */
int vb200_timeline(vb200_handle h, int32_t batch, int32_t n_tokens, int32_t n_regions, uint32_t select, int32_t slot, int32_t max_ops,
                   int32_t* n_ops, int32_t* dims, int64_t* stamps);
/* Per-launch device time of one forward of this shape (after at least one vb200_forward of it): every kernel of the plan is
 * captured 8x into its own CUDA graph and replayed `iters` times between two CUDA events (no host launch gaps).  kinds: 0 GEMM, 1 self-attention,
 * 2 co-attention, 3 narrow head, 4 LayerNorm; dims[4*i..] = {M, N, K, act|16*fusedLN} for GEMMs.  Profiling aid for bench.py. */
int vb200_profile_ops(vb200_handle h, int32_t batch, int32_t n_tokens, int32_t n_regions, uint32_t select, int32_t iters,
                      int32_t max_ops, int32_t* n_ops, int32_t* kinds, double* ms, double* flops, int32_t* dims);

/* Layout of vb200_outputs.attention_probs for a shape: entry i is a [batch, dims[4i], dims[4i+1], dims[4i+2]] fp32 tensor
 * (heads, query length, key length) at float offset offsets[i]; dims[4i+3] is the layer kind: 0 text layer, 1 image layer,
 * 2 connection layer, text queries over image keys, 3 connection layer, image queries over text keys (kinds 2 and 3 of one layer
 * are adjacent: the reference's per-layer tuple).  *n_entries receives the entry count (30 for the 12/6/6 configuration: 24
 * layers, two tensors per connection layer), total_floats the buffer size.  Arrays may be NULL to query the count only. */
int vb200_attention_layout(vb200_handle h, int32_t batch, int32_t n_tokens, int32_t n_regions, int32_t max_entries,
                           int32_t* n_entries, int32_t* dims, int64_t* offsets, int64_t* total_floats);

/* custom_prediction()'s tensor construction fused into the forward (worker.py:422-455): instead of features [B, V, F] /
 * spatials [B, V, 5] / image_mask the caller passes what the detector produced -- box features, pixel boxes, image sizes -- and one
 * kernel writes the image-embedding GEMM's 16-bit operand rows directly: global mean row first, 5-d normalised locations
 * ([0,0,1,1,1] for the global row), masks.  n_regions of the forward is n_boxes + 1. */
typedef struct {
    int32_t batch;                 /* images (= rows of the forward) */
    int32_t n_tokens;              /* Tin */
    int32_t n_boxes;               /* detector boxes per image (rows of box_features per image); n_regions = n_boxes + 1 */
    const int64_t* question;       /* [B, Tin]   (text already repeated per image for pair / retrieval tasks, worker.py:266-284) */
    const int64_t* segment_ids;    /* [B, Tin] */
    const int64_t* input_mask;     /* [B, Tin] */
    const int64_t* task_tokens;    /* [B, 1] */
    const float* box_features;     /* [B, n_boxes, v_feature_size] fp32, as the detector returns them (worker.py:213) */
    const float* boxes;            /* [B, n_boxes, 4] pixel x1, y1, x2, y2 (infos[i]['bbox'], worker.py:434) */
    const float* image_wh;         /* [B, 2] image_width, image_height */
    const int32_t* num_boxes;      /* [B] valid boxes per image or NULL (= n_boxes); padded boxes are zeroed, masked and left out
                                      of the mean */
    float* spatials_out;           /* optional [B, n_boxes + 1, 5]: the spatials tensor the reference would have built (the
                                      grounding decode reads spatials[0], worker.py:379) */
} vb200_region_inputs;
int vb200_forward_regions(vb200_handle h, const vb200_region_inputs* in, const vb200_outputs* out, uint32_t select, int32_t slot,
                          void* cuda_stream);

/* ---- Caption-image retrieval with reuse (SURVEY.md section 8e; reference semantics worker.py:278-284, 359).  Everything ahead of
 * the first connection layer depends on the caption alone or on the image alone: encode each caption / image ONCE, then score
 * pairs from the cached states.  Same kernels on the same rows as the full forward: scores are bit-identical to vb200_forward.
 * State buffers are caller-allocated device memory: fp32 [n, L, hidden], 16-bit [n, L, hidden * operand_width_factor] (2 bytes per
 * element; vb200_model_dim "operand_width_factor" is 1, or 3 in split_fp32 mode) and the additive mask fp32 [n, L], with
 * L = n_tokens + 1 (task token) for text and L = n_regions for images. */
int vb200_encode_text(vb200_handle h, int32_t n, int32_t n_tokens, const int64_t* question, const int64_t* segment_ids,
                      const int64_t* input_mask, const int64_t* task_tokens, float* state_f32, void* state_16, float* state_mask,
                      void* cuda_stream);
int vb200_encode_image(vb200_handle h, int32_t n, int32_t n_regions, const float* features, const float* spatials,
                       const uint8_t* image_mask, float* state_f32, void* state_16, float* state_mask, void* cuda_stream);
/* Pair b = (caption text_index[b], image image_index[b]); index arrays are device int32. */
int vb200_forward_cached(vb200_handle h, int32_t batch, int32_t n_tokens, int32_t n_regions, const int32_t* text_index,
                         int32_t n_text, const float* text_f32, const void* text_16, const float* text_mask,
                         const int32_t* image_index, int32_t n_image, const float* image_f32, const void* image_16,
                         const float* image_mask, const vb200_outputs* out, uint32_t select, int32_t slot, void* cuda_stream);

/* ---- Kernel-level entry points (device pointers), used by the parity tests and the roofline bench.  ---- */
/* y = epilogue(x[M,K] (16-bit) . w[N,K]^T (16-bit)); act: 0 none, 1 GELU(erf), 2 ReLU; LayerNorm applied when gamma != NULL.
 * act_fp16 != 0: x, w and the 16-bit output y are fp16, else bf16 (parameter names keep the historical _bf16 suffix).
 * act 3 = GELU with the 1.5e-7 erf (fp32-parity mode).  variant 0: persistent kernel (gemm_persistent.cuh, what the engine
 * uses); 2: CTA-pair kernel (gemm_pair.cu, cta_group::2); 3: persistent kernel with three CTAs per SM (128-wide tile, PCfg MODE 6);
 * 4: persistent kernel with one CTA per SM and a 6-stage ring (128- or 64-wide tile, PCfg MODE 7 -- what the engine uses for forwards
 * of <= 320 rows).  Variants 0, 3 and 4 produce the same bits.
 * timing: NULL, or a device buffer of 16 int64 per CTA that receives clock64() / %globaltimer stamps (profiling aid, variants 0, 3, 4). */
int vb200_linear(const void* x_bf16, int64_t ld_x, const void* w_bf16, int64_t ld_w, const float* bias,
                 const float* residual, int64_t ld_res, const float* gamma, const float* beta, float eps, int32_t act,
                 void* y_bf16, int64_t ld_y_bf16, float* y_f32, int64_t ld_y_f32, int64_t M, int64_t N, int64_t K,
                 int32_t block_n, int32_t use_pdl, int32_t act_fp16, int32_t variant, long long* timing, void* cuda_stream);
/* The same GEMM on fp32-parity-mode operands (fp16 only): x16 holds hi | lo | hi and w16 hi | hi | lo per 64 logical columns, K3 is
 * the PHYSICAL contraction length (3x the logical one), y16 (optional) is written in the activation split layout (stride ld_y16 of
 * the 3x wider buffer), y_f32 (optional) as usual. */
int vb200_linear_split(const void* x16, int64_t ld_x, const void* w16, int64_t ld_w, const float* bias, int32_t act, void* y16,
                       int64_t ld_y16, float* y_f32, int64_t ld_y_f32, int64_t M, int64_t N, int64_t K3, void* cuda_stream);
/* ctx = softmax(Q K^T / sqrt(d) + mask) V, qkv rows = [Q | K | V] (bf16), mask_add fp32 [B, L]. */
/* out = LayerNorm(y + residual) * gamma + beta over rows of N (N % 128 == 0, N <= 2048); fp32 and/or 16-bit outputs. */
int vb200_layernorm(const float* y, int64_t ld_y, const float* residual, int64_t ld_res, const float* gamma, const float* beta,
                    float eps, float* out_f32, int64_t ld_f32, void* out_16, int64_t ld_16, int64_t M, int64_t N,
                    int32_t act_fp16, void* cuda_stream);
/* Two dependent GEMMs in one launch (vilbert-multi-task_b200/csrc/gemm_chain.cu): h = act(x w1^T + b1) (16-bit, [M, N1]) and
 * y = h w2^T + b2 ([M, N2], 16-bit and/or fp32).  sync_ints: device memory, M / 128 (rounded up) + 2 ints, zero before the first
 * call (the kernel leaves it zeroed).  Results are bit-identical to two vb200_linear calls. */
int vb200_linear_chain(const void* x16, int64_t ld_x, const void* w1, int64_t ld_w1, const float* b1, int32_t act, void* h16, int64_t ld_h,
                       const void* w2, int64_t ld_w2, const float* b2, void* y16, int64_t ld_y16, float* y_f32, int64_t ld_y_f32, int64_t M,
                       int64_t N1, int64_t K1, int64_t N2, int32_t act_fp16, void* sync_ints, void* cuda_stream);
/* The GEMM with the LayerNorm fold epilogues (vilbert-multi-task_b200/csrc/gemm_persistent.cuh, row_stats).  Statistics arrays are
 * float2 (mean, M2 = sum (x - mean)^2) per row and 32-column chunk, laid out [N_src / 32][stats_ld].
 * mode 5 (producer): u = x w^T + bias + residual, where the residual is res, or LayerNorm_{res_gamma,res_beta}(res) rebuilt from
 *         res_stats when that is non-NULL; writes u to y_f32 AND y16, and its statistics to out_stats.
 * mode 4 (consumer): x holds such a u, w = gamma o W (16-bit), fold_s[n] = sum_k w[n,k], bias = c;
 *         y = act(rstd * (x w^T - mean * s) + c), mean / rstd from a_stats (a_parts = K_logical / 32). */
int vb200_linear_ln(const void* x16, int64_t ld_x, const void* w16, int64_t ld_w, const float* bias, int32_t mode, const void* a_stats,
                    int32_t a_parts, const float* fold_s, const float* res, int64_t ld_res, const void* res_stats, int32_t res_parts,
                    const float* res_gamma, const float* res_beta, void* out_stats, int32_t stats_ld, float eps, int32_t act, void* y16,
                    int64_t ld_y16, float* y_f32, int64_t ld_y_f32, int64_t M, int64_t N, int64_t K, int32_t act_fp16, void* cuda_stream);
/* split16 != 0: out_16 is the fp16 hi | lo | hi operand (stride ld_16 of the 3x wider buffer). */
int vb200_layernorm_split(const float* y, int64_t ld_y, const float* residual, int64_t ld_res, const float* gamma, const float* beta,
                          float eps, float* out_f32, int64_t ld_f32, void* out_16, int64_t ld_16, int64_t M, int64_t N, void* cuda_stream);
/* fp32 CUDA-core attention (attention_f32.cu): q / k / v point at head 0 of sample 0 (row strides ld_q, ld_kv; the three may alias
 * one QKV buffer), in_kind 0 fp32 / 1 fp16 / 2 bf16; ctx_mode 0 no context / 1 fp16 / 2 bf16 / 3 fp16 hi | lo | hi;
 * probs optional [B, heads, Lq, Lk]. */
int vb200_attention_f32(const void* q, int64_t ld_q, const void* k, const void* v, int64_t ld_kv, int32_t in_kind,
                        const float* key_mask_add, int32_t B, int32_t Lq, int32_t Lk, int32_t heads, int32_t head_dim, void* ctx,
                        int64_t ld_ctx, int32_t ctx_mode, float* probs, void* cuda_stream);
int vb200_self_attention(const void* qkv_bf16, int64_t ld_qkv, int32_t hidden, const float* mask_add, void* ctx_bf16,
                         int64_t ld_ctx, int32_t B, int32_t L, int32_t heads, int32_t head_dim, int32_t act_fp16,
                         void* cuda_stream);
int vb200_co_attention(const void* qkv_img_bf16, int64_t ld_img, const void* qkv_txt_bf16, int64_t ld_txt,
                       int32_t hidden, const float* img_mask_add, const float* txt_mask_add, void* ctx_txt_bf16,
                       int64_t ld_ctx_txt, void* ctx_img_bf16, int64_t ld_ctx_img, int32_t B, int32_t T, int32_t V,
                       int32_t heads, int32_t head_dim, int32_t act_fp16, void* cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* VILBERT_B200_H */
