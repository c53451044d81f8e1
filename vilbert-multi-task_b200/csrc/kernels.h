// Internal launch interface of the vilbert_b200 sm_100a kernels (not part of the C ABI; see include/vilbert_b200.h).
#pragma once
#include "common.cuh"

namespace vb {

enum Act : int { kActNone = 0, kActGelu = 1, kActRelu = 2, kActGeluExact = 3 };   // 3: erf to 1.5e-7 (fp32-parity mode)

// Epilogue of the tcgen05 GEMM:  x = act(acc + bias + res) * mul ; LN variant: y = LayerNorm(x) * gamma + beta.
struct GemmEpilogue {
    int M, N, K;
    const float* bias;            // [N] or null
    const float* res;             // fp32 [M, ld_res] residual or null (may alias out_f32)
    int ld_res;
    const float* mul;             // fp32 [M, ld_mul] multiplicand (pooled_t * pooled_v fusion) or null
    int ld_mul;
    const float* gamma;           // LN only
    const float* beta;
    float eps;
    __nv_bfloat16* out_bf16;      // optional
    int ld_bf16;
    float* out_f32;               // optional
    int ld_f32;
    int act;
    int pdl;                      // in-kernel griddepcontrol.wait / launch_dependents; 1 = also LAUNCHED with programmatic stream
                                  // serialization, 2 = trigger only (this GEMM waits for its predecessor the normal way, but
                                  // lets a light dependent -- LayerNorm, attention -- start under its epilogue),
                                  // 5 = as 1, and the producer puts the first ring pass of WEIGHT tiles in flight before
                                  // griddepcontrol.wait (weights do not depend on the previous kernel)
    int a_f16;                    // both GEMM operands (activations A, weights W) are fp16 instead of bf16
    int out_f16;                  // 16-bit output is fp16 instead of bf16
    int split16;                  // fp32-parity mode: the 16-bit output is written as fp16 hi | lo | hi per 64 columns
                                  // (common.cuh split_col; ld_bf16 is the stride of that 3x wider buffer); plain kernel only
    long long* timing;            // optional (profiling): 8 clock64 stamps per CTA, see gemm_persistent.cu; null in production
    const void* tmap_c_host;      // host pointer to the CUtensorMap of the output (launchers copy it into a kernel parameter)
    int tma_store;                // 0: register/LSU stores only; 1: 16-bit output, 2: fp32 output may leave through a TMA store
                                  // (plain persistent kernel: the LAST tile of every CTA is staged in the idle operand ring)
    // LayerNorm fold (gemm_persistent.cuh, PCfg MODE 4 / 5).  stats arrays: [N_src / 32][stats_ld] float2 (mean, M2) per 32 columns
    const float2* a_stats;        // MODE 4: statistics of the A operand's rows (its LayerNorm is pending); bias then holds c
    int a_parts;                  //         N_src / 32
    const float* fold_s;          //         s_n = sum_k W'[n, k]   [N]
    const float2* res_stats;      // MODE 5: statistics of the residual's rows, or null when the residual holds final values
    int res_parts;
    const float* res_gamma;       //         the residual's pending LayerNorm parameters [N]
    const float* res_beta;
    float2* out_stats;            // MODE 5: this GEMM's own row statistics, [N / 32][stats_ld]
    int stats_ld;                 // row capacity of every stats array of this launch (>= M)
    int grid_pct;                 // 0: default persistent grid (2/3 of the CTA slots, launch_p); 10..100: this percentage of them
    int ln_mode;                  // 0 none, 4 fold-in (consumer), 5 pre-LayerNorm output + statistics (producer)
    int tri;                      // plain 128-wide tile only: three CTAs per SM (gemm_persistent.cuh PCfg MODE 6)
    int lone;                     // plain 128-wide tile only: one CTA per SM, 6-stage ring (PCfg MODE 7; small-batch latency)
    int debug;                    // timing decomposition only (VB200_DEBUG through vb200_linear): 1 = issue no MMA, 2 = no epilogue
                                  // stores, 4 = no operand loads (the ring is "filled" by plain arrives); results are garbage
};                                //   every GEMM starts on HBM misses (weights never survive in the 126 MB L2 until the next step)

// v2: persistent CTAs / clusters, TMEM double-buffered accumulators, single-exchange LayerNorm (gemm_persistent.cu)
int gemm_p_pick_block_n(int N, bool ln);
int gemm_p_max_clusters(int block_n, int cluster);
cudaError_t launch_gemm_persistent(const CUtensorMap& tmap_a, const CUtensorMap& tmap_b, const GemmEpilogue& ep,
                                   int block_n, bool ln, cudaStream_t st);
int num_sms_host();          // SM count of the current device (148 on B200)
// CTA-pair kernel (gemm_pair.cu, tcgen05 cta_group::2, 256 x block_n tile per pair); tmap_b box rows = block_n / 2
cudaError_t launch_gemm_pair(const CUtensorMap& tmap_a, const CUtensorMap& tmap_b, const GemmEpilogue& ep, int block_n,
                             cudaStream_t stream);
// Two dependent GEMMs (FFN-in -> FFN-out) in one persistent launch with a dynamic tile list (gemm_chain.cu); sync: (M tiles + 2) zeroed ints
cudaError_t launch_gemm_chain(const CUtensorMap& ta0, const CUtensorMap& tb0, const GemmEpilogue& ep0, const CUtensorMap& ta1,
                              const CUtensorMap& tb1, const GemmEpilogue& ep1, int* sync, cudaStream_t st);
cudaError_t launch_gemm_persistent_plain(const CUtensorMap& tmap_a, const CUtensorMap& tmap_b, const GemmEpilogue& ep,
                                         int block_n, cudaStream_t st);

// 16-bit activation buffers are typed __nv_bfloat16* throughout; `f16` says the bits are IEEE fp16 instead.
// K4: softmax(Q K^T / sqrt(d) + mask) V per (sample, head); qkv row = [Q | K | V], each `hidden` wide.  Context rows are
// computed for the first nq (1..L) query rows of each sample, in place at rows b*L .. b*L + nq - 1 of ctx.
cudaError_t launch_self_attention(const __nv_bfloat16* qkv, int ld_qkv, int hidden, const float* key_mask_add,
                                  __nv_bfloat16* ctx, int ld_ctx, int B, int L, int nq, int heads, int head_dim, int pdl,
                                  int f16, cudaStream_t st);
// K5: both co-attention directions in one kernel.  qkv_img rows = [Q1|K1|V1], qkv_txt rows = [Q2|K2|V2].
//   ctx_txt[b,t] = softmax(Q2 K1^T / sqrt(d) + img_mask) V1      ctx_img[b,v] = softmax(Q1 K2^T / sqrt(d) + txt_mask) V2
cudaError_t launch_co_attention(const __nv_bfloat16* qkv_img, int ld_img, const __nv_bfloat16* qkv_txt, int ld_txt,
                                int hidden, const float* img_mask_add, const float* txt_mask_add,
                                __nv_bfloat16* ctx_txt, int ld_ctx_txt, __nv_bfloat16* ctx_img, int ld_ctx_img, int B,
                                int T, int V, int heads, int head_dim, int pdl, int f16, cudaStream_t st);

// un-fused LayerNorm(y + res): fp32 stream out + 16-bit operand out (layernorm.cu); split16: hi | lo | hi operand (fp32-parity mode)
struct LnPending {                // a residual whose own LayerNorm is still pending (LayerNorm fold): statistics + parameters
    const float2* stats;          // [parts][ld] (mean, M2) per 32 columns
    int parts, ld;
    const float *gamma, *beta;
};
cudaError_t launch_ln_residual(const float* y, int ld_y, const float* res, int ld_res, const float* gamma, const float* beta,
                               float eps, float* out_f32, int ld_f32, __nv_bfloat16* out16, int ld16, int M, int N, int f16,
                               int split16, int pdl, cudaStream_t st, const LnPending* res_pending = nullptr);
// K2: word + position + token-type gather, task-token row at index 1, LayerNorm; also builds the additive text mask.
cudaError_t launch_text_embed(const int64_t* ids, const int64_t* seg, const int64_t* input_mask, const int64_t* task,
                              const float* word, const float* pos, const float* type, const float* task_tab,
                              const float* gamma, const float* beta, float eps, float* out_f32,
                              __nv_bfloat16* out_bf16, float* mask_add, int B, int Tin, int H, int vocab, int max_pos,
                              int n_type, int n_task, int task_tokens, int f16, int split16, cudaStream_t st);
// K1 (input half): fp32 region features + 5-d boxes -> bf16 GEMM operand [B*V, Kp] = [feat | loc | 0], additive image mask.
cudaError_t launch_image_pack(const float* feats, const float* loc, const uint8_t* image_mask, __nv_bfloat16* a_out,
                              float* mask_add, int rows, int F, int Kp, int f16, int split16, cudaStream_t st);
// custom_prediction()'s tensor construction on the device (worker.py:422-455): box features [B, n, F] + pixel boxes [B, n, 4] +
// image sizes [B, 2] (+ optional valid-box counts) -> operand rows [B * (n + 1), Kp] with the global mean row first, masks, spatials.
cudaError_t launch_region_pack(const float* box_feats, const float* boxes, const float* image_wh, const int32_t* num_boxes,
                               __nv_bfloat16* a_out, float* mask_add, float* spatials_out, int B, int n, int F, int Kp, int f16,
                               int split16, cudaStream_t st);
// retrieval reuse: cached encoder state rows idx[b] -> sample b of a pair plan (fp32 stream [L, H], 16-bit operand [L, H16], mask [L])
cudaError_t launch_gather_state(const int32_t* idx, int n_src, const float* src_f32, const void* src_16, const float* src_mask,
                                float* dst_f32, void* dst_16, float* dst_mask, int B, int L, int H, int H16, cudaStream_t st);
// fp32 CUDA-core attention (attention_f32.cu): in_kind 0 fp32 / 1 fp16 / 2 bf16 Q, K, V; ctx_mode 0 none / 1 fp16 / 2 bf16 /
// 3 fp16 hi | lo | hi; probs: optional [B, heads, Lq, Lk] fp32 attention probabilities.
cudaError_t launch_attention_f32(const void* q, int ld_q, const void* k, const void* v, int ld_kv, int in_kind,
                                 const float* key_mask_add, int B, int Lq, int Lk, int heads, int D, __nv_bfloat16* ctx, int ld_ctx,
                                 int ctx_mode, float* probs, int pdl, cudaStream_t st);
// K8 (narrow heads): out[m, j] = dot(x[m, :K], W[j, :K]) + b[j] + (add ? add[m] : 0), j < n_out <= 4.
cudaError_t launch_rowdot(const float* x, int ld_x, const float* W, const float* b, const float* add, float* out,
                          int ld_out, int M, int K, int n_out, int pdl, cudaStream_t st);

// ---- shared host-side launch helpers
template <typename K>
inline cudaError_t set_smem(K kern, size_t bytes) {
    // opt in to > 48 KB dynamic shared memory (host-side attribute; launches are replayed from a CUDA graph,
    // so this runs at capture time only)
    if (bytes <= 48 * 1024) return cudaSuccess;
    return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes));
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_ex(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, int pdl, cudaStream_t st,
                             Args&&... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    if (pdl) {
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
    }
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

}  // namespace vb
