// Host side of the vilbert_b200 engine: BertConfig JSON, state_dict audit + weight repack, per-shape plans
// (workspace, TMA descriptors, launch list, CUDA graph) and the C ABI of include/vilbert_b200.h.
//
// Mirrors what the reference does at /root/reference/worker.py:495-536 (config + from_pretrained + cuda)
// and worker.py:286-289 (the forward call); the layer schedule and module wiring follow the [UPSTREAM]
// vilbert/vilbert.py restated in SURVEY.md section 3C / 8a.
#include "../../include/vilbert_b200.h"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <set>
#include <stdexcept>
#include <string>
#include <vector>

#include <nvtx3/nvToolsExt.h>      // header-only NVTX v3: ranges per layer / per forward for nsys and ncu --nvtx (SURVEY.md section 5)

#include "kernels.h"

namespace {

using vb::GemmEpilogue;
typedef __nv_bfloat16 bf16;

struct VbError : std::runtime_error {
    int status;
    VbError(int s, const std::string& m) : std::runtime_error(m), status(s) {}
};

[[noreturn]] void fail(int status, const char* fmt, ...) {
    char buf[2048];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    throw VbError(status, buf);
}

#define CUDA_CHECK(expr)                                                                                    \
    do {                                                                                                    \
        cudaError_t _e = (expr);                                                                            \
        if (_e != cudaSuccess) fail(VB200_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                                    __FILE__, __LINE__);                                                    \
    } while (0)

std::string g_create_error;   // last failed vb200_create (no handle to hang it on)

// ------------------------------------------------------------------------------------------ tiny JSON
struct JVal {
    enum Kind { NUM, STR, BOOL, ARR, NUL, OBJ } kind = NUL;
    double num = 0;
    bool b = false;
    std::string str;
    std::vector<double> arr;
};

struct JsonParser {
    const char* p;
    explicit JsonParser(const char* s) : p(s) {}
    void ws() { while (*p == ' ' || *p == '\n' || *p == '\t' || *p == '\r') ++p; }
    std::string parse_string() {
        if (*p != '"') fail(VB200_ERR_CONFIG, "config JSON: expected string");
        ++p;
        std::string s;
        while (*p && *p != '"') {
            if (*p != '\\') { s.push_back(*p++); continue; }
            ++p;                                                   // escape sequence (RFC 8259 section 7)
            switch (*p) {
                case 'n': s.push_back('\n'); break;
                case 't': s.push_back('\t'); break;
                case 'r': s.push_back('\r'); break;
                case 'b': s.push_back('\b'); break;
                case 'f': s.push_back('\f'); break;
                case 'u': {                                        // \uXXXX -> UTF-8 (basic multilingual plane; surrogates kept as-is)
                    unsigned cp = 0;
                    for (int i = 1; i <= 4; ++i) {
                        const char c = p[i];
                        const int d = (c >= '0' && c <= '9') ? c - '0' : (c >= 'a' && c <= 'f') ? c - 'a' + 10 : (c >= 'A' && c <= 'F') ? c - 'A' + 10 : -1;
                        if (d < 0) fail(VB200_ERR_CONFIG, "config JSON: bad \\u escape");
                        cp = cp * 16 + static_cast<unsigned>(d);
                    }
                    p += 4;
                    if (cp < 0x80) s.push_back(static_cast<char>(cp));
                    else if (cp < 0x800) { s.push_back(static_cast<char>(0xC0 | (cp >> 6))); s.push_back(static_cast<char>(0x80 | (cp & 0x3F))); }
                    else { s.push_back(static_cast<char>(0xE0 | (cp >> 12))); s.push_back(static_cast<char>(0x80 | ((cp >> 6) & 0x3F))); s.push_back(static_cast<char>(0x80 | (cp & 0x3F))); }
                    break;
                }
                case '\0': fail(VB200_ERR_CONFIG, "config JSON: unterminated string");
                default: s.push_back(*p);                          // \" \\ \/
            }
            ++p;
        }
        if (*p != '"') fail(VB200_ERR_CONFIG, "config JSON: unterminated string");
        ++p;
        return s;
    }
    void skip_value();
    JVal parse_value() {
        ws();
        JVal v;
        if (*p == '"') { v.kind = JVal::STR; v.str = parse_string(); }
        else if (*p == '[') {
            v.kind = JVal::ARR;
            ++p; ws();
            while (*p && *p != ']') {
                JVal e = parse_value();
                if (e.kind == JVal::NUM) v.arr.push_back(e.num);
                ws();
                if (*p == ',') { ++p; ws(); }
            }
            if (*p != ']') fail(VB200_ERR_CONFIG, "config JSON: unterminated array");
            ++p;
        } else if (*p == '{') {            // nested objects are skipped (none carry model dimensions)
            v.kind = JVal::OBJ;
            int depth = 0;
            do {
                if (*p == '"') { parse_string(); continue; }
                if (*p == '{') ++depth;
                if (*p == '}') --depth;
                ++p;
            } while (*p && depth > 0);
        } else if (!strncmp(p, "true", 4)) { v.kind = JVal::BOOL; v.b = true; p += 4; }
        else if (!strncmp(p, "false", 5)) { v.kind = JVal::BOOL; v.b = false; p += 5; }
        else if (!strncmp(p, "null", 4)) { v.kind = JVal::NUL; p += 4; }
        else {
            char* end = nullptr;
            v.num = strtod(p, &end);
            if (end == p) fail(VB200_ERR_CONFIG, "config JSON: unexpected character '%c'", *p);
            v.kind = JVal::NUM;
            p = end;
        }
        return v;
    }
    std::map<std::string, JVal> parse_object() {
        std::map<std::string, JVal> m;
        ws();
        if (*p != '{') fail(VB200_ERR_CONFIG, "config JSON: expected '{'");
        ++p; ws();
        while (*p && *p != '}') {
            std::string k = parse_string();
            ws();
            if (*p != ':') fail(VB200_ERR_CONFIG, "config JSON: expected ':' after \"%s\"", k.c_str());
            ++p;
            m[k] = parse_value();
            ws();
            if (*p == ',') { ++p; ws(); }
        }
        if (*p != '}') fail(VB200_ERR_CONFIG, "config JSON: unterminated object");
        return m;
    }
};

struct Config {
    int hidden = 768, layers = 12, heads = 12, inter = 3072, max_pos = 512, type_vocab = 2, vocab = 30522;
    int v_feat = 2048, v_target = 1601, v_hidden = 1024, v_layers = 6, v_heads = 8, v_inter = 1024;
    int bi_hidden = 1024, bi_heads = 8;
    int task_tokens = 1, n_task = 20;
    std::vector<int> v_bi_id{0, 1, 2, 3, 4, 5}, t_bi_id{6, 7, 8, 9, 10, 11};
    std::string hidden_act = "gelu", v_hidden_act = "gelu", fusion = "mul";
    float ln_eps = 1e-12f;
};

Config parse_config(const char* json) {
    Config c;
    if (json == nullptr) fail(VB200_ERR_CONFIG, "config JSON is NULL");
    JsonParser jp(json);
    auto m = jp.parse_object();
    auto geti = [&](const char* k, int& dst) {
        auto it = m.find(k);
        if (it == m.end()) return;
        if (it->second.kind == JVal::NUM) dst = static_cast<int>(it->second.num);
        else if (it->second.kind == JVal::BOOL) dst = it->second.b ? 1 : 0;
    };
    geti("hidden_size", c.hidden); geti("num_hidden_layers", c.layers); geti("num_attention_heads", c.heads);
    geti("intermediate_size", c.inter); geti("max_position_embeddings", c.max_pos);
    geti("type_vocab_size", c.type_vocab); geti("vocab_size", c.vocab); geti("v_feature_size", c.v_feat);
    geti("v_target_size", c.v_target); geti("v_hidden_size", c.v_hidden); geti("v_num_hidden_layers", c.v_layers);
    geti("v_num_attention_heads", c.v_heads); geti("v_intermediate_size", c.v_inter);
    geti("bi_hidden_size", c.bi_hidden); geti("bi_num_attention_heads", c.bi_heads);
    geti("task_specific_tokens", c.task_tokens); geti("num_task_tokens", c.n_task);
    auto geta = [&](const char* k, std::vector<int>& dst) {
        auto it = m.find(k);
        if (it == m.end() || it->second.kind != JVal::ARR) return;
        dst.clear();
        for (double d : it->second.arr) dst.push_back(static_cast<int>(d));
    };
    geta("v_biattention_id", c.v_bi_id); geta("t_biattention_id", c.t_bi_id);
    auto gets = [&](const char* k, std::string& dst) {
        auto it = m.find(k);
        if (it != m.end() && it->second.kind == JVal::STR) dst = it->second.str;
    };
    gets("hidden_act", c.hidden_act); gets("v_hidden_act", c.v_hidden_act); gets("fusion_method", c.fusion);
    int dyn = 0;
    geti("dynamic_attention", dyn);
    // ---- what this engine implements (everything the worker configures, worker.py:509-522)
    if (dyn) fail(VB200_ERR_CONFIG, "dynamic_attention=true is not supported (worker.py:484 sets it false)");
    if (c.hidden_act != "gelu" || c.v_hidden_act != "gelu") fail(VB200_ERR_CONFIG, "only hidden_act = gelu is supported");
    if (c.fusion != "mul") fail(VB200_ERR_CONFIG, "only fusion_method = mul is supported");
    if (c.v_bi_id.size() != c.t_bi_id.size()) fail(VB200_ERR_CONFIG, "v_biattention_id / t_biattention_id length mismatch");
    auto head_ok = [](int hid, int heads) { return heads > 0 && hid % heads == 0 && (hid / heads == 64 || hid / heads == 128); };
    if (!head_ok(c.hidden, c.heads) || !head_ok(c.v_hidden, c.v_heads) || !head_ok(c.bi_hidden, c.bi_heads))
        fail(VB200_ERR_CONFIG, "attention head size must be 64 or 128");
    for (int d : {c.hidden, c.v_hidden, c.bi_hidden, c.inter, c.v_inter})
        if (d % 128 != 0) fail(VB200_ERR_CONFIG, "hidden/intermediate sizes must be multiples of 128 (got %d)", d);
    if (c.hidden > 1024 || c.v_hidden > 1024 || c.bi_hidden > 1024)
        fail(VB200_ERR_CONFIG, "hidden sizes above 1024 need a wider LayerNorm cluster than 8 CTAs");
    if (c.v_feat % 8 != 0) fail(VB200_ERR_CONFIG, "v_feature_size must be a multiple of 8");
    return c;
}

// ------------------------------------------------------------------------------------------ device memory
struct Arena {   // owns every device allocation of an engine / plan
    std::vector<void*> ptrs;
    size_t total = 0;
    void* alloc(size_t bytes) {
        void* p = nullptr;
        bytes = (bytes + 255) & ~size_t(255);
        CUDA_CHECK(cudaMalloc(&p, bytes ? bytes : 256));
        ptrs.push_back(p);
        total += bytes;
        return p;
    }
    template <typename T> T* alloc_n(size_t n) { return static_cast<T*>(alloc(n * sizeof(T))); }
    ~Arena() { for (void* p : ptrs) cudaFree(p); }
};

inline uint16_t f32_to_f16_bits(float f) {          // IEEE half, round to nearest even, saturating to +-65504
    const __half h = __float2half_rn(f);            // host-callable conversion from cuda_fp16.h
    uint16_t b;
    memcpy(&b, &h, 2);
    if ((b & 0x7fffu) == 0x7c00u) b = static_cast<uint16_t>((b & 0x8000u) | 0x7bffu);
    return b;
}
inline uint16_t f32_to_bf16_bits(float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return static_cast<uint16_t>((u >> 16) | 0x40);   // NaN
    u += 0x7fffu + ((u >> 16) & 1u);                                                          // round to nearest even
    return static_cast<uint16_t>(u >> 16);
}
inline float bf16_bits_to_f32(uint16_t h) { uint32_t u = static_cast<uint32_t>(h) << 16; float f; memcpy(&f, &u, 4); return f; }
inline float half_bits_to_f32(uint16_t h) {
    const uint32_t sign = (h & 0x8000u) << 16, exp = (h >> 10) & 0x1f, man = h & 0x3ff;
    uint32_t u;
    if (exp == 0) {
        if (man == 0) u = sign;
        else {
            int e = -1; uint32_t m = man;
            do { ++e; m <<= 1; } while (!(m & 0x400));
            u = sign | ((127 - 15 - e) << 23) | ((m & 0x3ff) << 13);
        }
    } else if (exp == 31) u = sign | 0x7f800000u | (man << 13);
    else u = sign | ((exp + 112) << 23) | (man << 13);
    float f; memcpy(&f, &u, 4); return f;
}

struct HostTensor {
    int dtype = 0, ndim = 0;
    int64_t shape[2] = {0, 0};
    const void* data = nullptr;
    bool used = false;
    int64_t numel() const { return ndim == 1 ? shape[0] : shape[0] * shape[1]; }
    float at(int64_t i) const {
        switch (dtype) {
            case VB200_F32: return static_cast<const float*>(data)[i];
            case VB200_F16: return half_bits_to_f32(static_cast<const uint16_t*>(data)[i]);
            default: { uint32_t u = static_cast<uint32_t>(static_cast<const uint16_t*>(data)[i]) << 16; float f; memcpy(&f, &u, 4); return f; }
        }
    }
};

struct LinearW {            // nn.Linear [N, K] -> bf16 [N, ldw] (K zero-padded to a multiple of 64), fp32 bias
    bf16* w = nullptr;
    float* bias = nullptr;
    int N = 0, K = 0, ldw = 0;
    // LayerNorm fold (gemm_persistent.cuh row_stats): this Linear's input is LayerNorm_{g,b}(u) of a pending LayerNorm; then
    // w = g o W (16-bit), bias = c = sum_k b_k W[n,k] + bias_n, fold_s = s = sum_k w[n,k]; fold_g identifies that LayerNorm
    float* fold_s = nullptr;
    const float* fold_g = nullptr;
};
struct LNW { float* g = nullptr; float* b = nullptr; int n = 0; std::vector<float> hg, hb; };   // hg / hb: host copies (fold)
struct RowW { float* w = nullptr; float* b = nullptr; int n_out = 0, K = 0; };   // narrow fp32 heads
struct LayerW { LinearW qkv, attn_out, inter, out; LNW ln1, ln2; };
struct ConnW { LinearW qkv_img, qkv_txt, dense1, dense2, v_inter, v_out, t_inter, t_out; LNW ln1, ln2, v_ln, t_ln; };
struct ClsW { LinearW fc0, fc3; LNW ln; RowW fc3_row; };

// ------------------------------------------------------------------------------------------ TMA descriptors
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (fn) return fn;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qr;
    CUDA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr));
    if (qr != cudaDriverEntryPointSuccess || p == nullptr) fail(VB200_ERR_CUDA, "cuTensorMapEncodeTiled not available in this driver");
    fn = reinterpret_cast<EncodeTiledFn>(p);
    return fn;
}
// bf16 matrix [rows, cols] with row stride ld (elements); box = 64 columns x box_rows rows, 128-byte swizzle,
// out-of-bounds elements read as zero.
CUtensorMap make_tmap(const void* base, int64_t rows, int64_t cols, int64_t ld, int box_rows, bool f16 = false) {
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (ld * 2) % 16 != 0)
        fail(VB200_ERR_INVALID, "TMA operand must be 16-byte aligned with a 16-byte-multiple row stride (ld=%lld)", (long long)ld);
    if (box_rows < 1 || box_rows > 256) fail(VB200_ERR_INVALID, "TMA box rows %d out of range", box_rows);
    CUtensorMap m;
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * 2};
    cuuint32_t box[2] = {64, static_cast<cuuint32_t>(box_rows)};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = get_encode_fn()(&m, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box,
                                 estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                 CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) fail(VB200_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld cols=%lld ld=%lld box_rows=%d)",
                                (int)r, (long long)rows, (long long)cols, (long long)ld, box_rows);
    return m;
}

// Output tile map for the TMA-store epilogue: [rows, cols] row-major with leading dimension ld (elements), boxes of 128 rows x
// 128 bytes (64 16-bit or 32 fp32 columns), SWIZZLE_128B.  Returns false when the buffer does not meet the TMA's alignment rules.
bool make_tmap_out(CUtensorMap* m, const void* base, int64_t rows, int64_t cols, int64_t ld, bool fp32, bool f16) {
    const int esz = fp32 ? 4 : 2;
    if (base == nullptr || (reinterpret_cast<uintptr_t>(base) & 15) || (ld * esz) % 16 != 0 || rows < 1 || cols < 1) return false;
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * esz};
    cuuint32_t box[2] = {static_cast<cuuint32_t>(128 / esz), 128};
    cuuint32_t estr[2] = {1, 1};
    const CUtensorMapDataType dt = fp32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                        : (f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
    return get_encode_fn()(m, dt, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// Decide whether a plain GEMM may use the TMA-store epilogue and build its output map (exactly one output, aligned).
void setup_tma_store(CUtensorMap* tc, GemmEpilogue& e) {
    e.tma_store = 0;
    if (e.split16 || e.gamma != nullptr) return;
    if (e.out_bf16 != nullptr && e.out_f32 == nullptr) {
        if (make_tmap_out(tc, e.out_bf16, e.M, e.N, e.ld_bf16, false, e.out_f16 != 0)) e.tma_store = 1;
    } else if (e.out_f32 != nullptr && e.out_bf16 == nullptr) {
        if (make_tmap_out(tc, e.out_f32, e.M, e.N, e.ld_f32, true, false)) e.tma_store = 2;
    }
}

// ------------------------------------------------------------------------------------------ launch list
struct Op {
    enum Kind { GEMM, SELF_ATTN, CO_ATTN, ROWDOT, LAYERNORM, ATTN_F32 } kind;
    int stream = 0;                // 0 main, 1 side (image branch) inside the captured graph
    // GEMM
    CUtensorMap ta, tb, tc;        // operands, and the output (TMA-store epilogue, ep.tma_store != 0)
    GemmEpilogue ep;
    int block_n = 128;
    bool ln = false;
    bool pair = false;             // CTA-pair kernel (cta_group::2); tb then has box rows block_n / 2
    // chained GEMM (gemm_chain.cu): this GEMM's 16-bit output is the A operand of a second one issued from the same launch
    CUtensorMap ta2, tb2;
    GemmEpilogue ep2;
    int* chain_sync = nullptr;
    double flops2 = 0;
    // fp32 attention (attention_f32.cu): fp32-parity mode and the attention-probability output
    const void* a_ptr = nullptr;   // GEMM: the A operand (chain detection)
    const void *f_q = nullptr, *f_k = nullptr, *f_v = nullptr;
    int f_ld_q = 0, f_ld_kv = 0, f_in = 0, f_Lq = 0, f_Lk = 0, f_ctx_mode = 0, f_ld_ctx = 0;
    const float* f_mask = nullptr;
    bf16* f_ctx = nullptr;
    float* f_probs = nullptr;
    // attention
    const bf16 *qkv_a = nullptr, *qkv_b = nullptr;
    int ld_a = 0, ld_b = 0, hidden = 0;
    const float *mask_a = nullptr, *mask_b = nullptr;
    bf16 *ctx_a = nullptr, *ctx_b = nullptr;
    int ld_ctx_a = 0, ld_ctx_b = 0, B = 0, La = 0, Lb = 0, heads = 0, head_dim = 0;   // SELF_ATTN: Lb = query rows per sample
                                                                                       //   when fewer than La (pruned tail), else 0
    // layernorm (un-fused): out = LN(ln_y + ln_res)
    const float *ln_y = nullptr, *ln_res = nullptr, *ln_g = nullptr, *ln_b = nullptr;
    float* ln_out_f = nullptr;
    bf16* ln_out_h = nullptr;
    int ln_ld = 0, ln_M = 0, ln_N = 0;
    vb::LnPending ln_pend{nullptr, 0, 0, nullptr, nullptr};   // residual whose own LayerNorm is still pending (LayerNorm fold)
    // rowdot
    const float *x = nullptr, *W = nullptr, *bias = nullptr, *add = nullptr;
    float* out = nullptr;
    int ld_x = 0, ld_out = 0, M = 0, K = 0, n_out = 0;
    // fork/join markers for the two-stream graph
    enum Sync { NONE, FORK, JOIN } sync = NONE;
    double flops = 0;
    const char* tag = nullptr;     // layer this launch belongs to ("T3", "V0", "C2", "embed", "heads"): NVTX range name
};

struct OutBuf { float* p = nullptr; int rows = 0, cols = 0, ld = 0; };

struct Plan {
    int B = 0, Tin = 0, T = 0, V = 0;
    uint32_t select = 0;
    Arena mem;
    // input-side buffers
    bf16* img_a = nullptr; int kp = 0;
    float *mask_t = nullptr, *mask_v = nullptr;
    float* t_f32[2]; bf16* t_b16[2];
    float* v_f32[2]; bf16* v_b16[2];
    float* y_scratch[2] = {nullptr, nullptr};   // per-stream fp32 GEMM output feeding the un-fused LayerNorm kernel
    float2* t_stats[2] = {nullptr, nullptr};    // LayerNorm fold: per-row (mean, M2) per 32 columns of t_f32[i] / v_f32[i],
    float2* v_stats[2] = {nullptr, nullptr};    //   [hidden / 32][stats_ld] (gemm_persistent.cuh row_stats)
    int stats_ld_t = 0, stats_ld_v = 0;
    int t_cur = 0, v_cur = 0;
    std::vector<Op> ops;
    OutBuf outs[12];
    struct AttnOut { float* p; int heads, Lq, Lk; };   // attention probabilities [B, heads, Lq, Lk] in schedule order
    std::vector<AttnOut> attn;                         //   (T / V layers: one entry; connection layers: text->image, image->text)
    uint64_t last_use = 0;                             // plan-cache LRU stamp
    long long* timeline = nullptr;                     // profiling (set_option "timeline"): [GEMM op][kTimelineCtas][16] stamps of the LAST replay
    double flops = 0;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    // host-API staging (device copies of the inputs)
    int64_t *d_q = nullptr, *d_seg = nullptr, *d_mask = nullptr, *d_task = nullptr;
    float *d_feat = nullptr, *d_loc = nullptr;
    uint8_t* d_imask = nullptr;
    float* d_out[12] = {nullptr};
    ~Plan() {
        if (exec) cudaGraphExecDestroy(exec);
        if (graph) cudaGraphDestroy(graph);
    }
};

}  // namespace

// =========================================================================================== engine
struct vb200_engine {
    Config cfg;
    vb200_options opt{};
    int num_labels = 0, gqa_labels = 0;
    bool dry = false;          // audit pass: check names / shapes / dtypes only, touch no device
    bool ln_fold = false;      // LayerNorm folded into the neighbouring GEMMs (row_stats in gemm_persistent.cuh); opt-in
                               // (vb200_options::ln_fold = 1 / VB200_LNFOLD=1): 57 fewer launches per forward, but the heavier
                               // GEMM epilogues cost more than the row kernels they replace (measured: 36.9 k vs 40.8 k pairs/s
                               // at batch 64, profiles/r2_ln_fold.md) -- default stays GEMM (fp32 out) + row LayerNorm kernel
    std::set<std::string> fold_out_t, fold_out_v;   // stages ("T3", "C0", "E", ...) whose OUTPUT LayerNorm stays pending
    bool chain_ffn = false;    // VB200_CHAIN=1 / vb200_set_option("chain_ffn", 1): FFN-in and FFN-out as ONE chained launch (gemm_chain.cu);
                               // bit-identical, measured slower at batch 64 (profiles/r2_chain.md) -> opt-in
    bool wide192 = false;      // VB200_BN192=1: 128x192 tiles for GEMMs that need more than one wave of 128-wide ones.  Faster per
                               // launch (FFN-in 18.5 -> 16.2 us, image QKV 16.9 -> 14.9 us, 973 TFLOP/s) but the STEP is 3 % slower
                               // with them (38.8 k vs 40.1 k pairs/s, profiles/r2_tile192.md) -- opt-in
    int tri_min_tiles = 0;     // VB200_TRI=<tiles> (0 = off): plain 128-wide GEMMs with at least this many tiles run THREE CTAs per SM
                               // (PCfg MODE 6: 2-stage ring, one accumulator, four epilogue warps)
    int lone_rows = 320;       // VB200_LONE_ROWS (0 = off): forwards with at most this many rows in either stream (batch <= 8 at the default
                               // shapes) run their plain 128-wide GEMMs one CTA per SM with a 6-stage ring (PCfg MODE 7): nothing else is
                               // there to share the SM, and a lone CTA's k loop is 1.5x faster with six stages in flight
    bool x3 = false;           // fp32-parity mode (vb200_options::split_fp32): fp16 hi/lo split operands, K' = 3K GEMMs, fp32 attention
    // Programmatic dependent launch.  Default: every kernel ("full": each kernel triggers its dependents once its main work is
    // issued; a dependent GEMM's producer puts its first weight tiles in flight before griddepcontrol.wait).  Measured with two
    // batches in flight, per step: off 1.597-1.604 ms | full 1.567 | "mediumplus" (everything except edges across a fork / join)
    // 1.571-1.581 | "medium" (into LayerNorm / attention and into the GEMM that follows one) 1.557-1.566 on another box whose
    // off was 1.601; with ONE batch in flight 1.83 (full) vs 1.96 ms (off).
    // VB200_PDL=off|light|medium|mediumplus|full; use_pdl < 0 = off, > 0 = full.
    bool pdl_light = true;
    bool pdl_medium = true;
    bool tma_store_enabled = true;  // VB200_TMASTORE=0: every tile leaves through the register / LSU epilogue
    bool early_w = true;            // VB200_EARLYW=0: no weight loads ahead of griddepcontrol.wait
    bool pdl_gemm_gemm = false;     // VB200_PDL=mediumplus: also GEMM -> GEMM edges of one graph branch (FFN-in -> FFN-out)
    int light_pdl() const { return (pdl_light || opt.use_pdl) ? 1 : 0; }
    // CTA-pair GEMM (cta_group::2, gemm_pair.cu).  -1 = auto: 256-wide pair tiles where a GEMM has >= 4 waves of them (large
    // batches: +6 % at batch 512); below that the single-CTA kernel wins -- one or two tiles per CTA, where the pair's extra
    // cluster syncs and coarser tiles cost more than the halved W traffic saves (profiles/README.md).  VB200_PAIR=0|128|256
    // forces it off / on for every plain GEMM with >= 256 rows.
    int pair_bn = -1;
    int pair_min_waves = 0;    // automatic CTA-pair selection: at least this many waves of 256 x 256 pair tiles.  0 = measured rule
                               // (profiles/r2_b512.md): 2 waves when the GEMM has >= 20 row panels of 256 (batch >= ~160: 512: +5.7 %,
                               // 384: +2 %, 192: +1 %, 256: =), else 4 (batch 128 loses 4.5 % with 2).  VB200_PAIR_MIN_WAVES overrides.
    bool fused_ln = false;     // VB200_FUSED_LN=1: cluster-LayerNorm GEMM epilogue instead of GEMM(fp32) + row LayerNorm kernel
    bool prune_tail = true;    // VB200_PRUNE=0 / vb200_set_option("prune_tail", 0): the last layer of a stream runs at full size even
                               // when nothing reads its rows beyond row 0 of each sample (A/B runs; get_plan, tail_prunable)
    Arena weights;
    std::string last_error;
    // embeddings
    float *word = nullptr, *pos = nullptr, *type = nullptr, *task = nullptr;
    bf16* word_b16 = nullptr;   // tied LM decoder operand
    LNW emb_ln, vemb_ln;
    LinearW img_emb;            // [v_hidden, v_feat + 64]: image_embeddings | image_location_embeddings | 0, bias = b_img + b_loc
    std::vector<LayerW> t_layers, v_layers;
    std::vector<ConnW> c_layers;
    LinearW t_pool, v_pool;
    ClsW vqa, gqa, binary;
    RowW vil_logit, vil_tri, vision_logit, ling_logit, seq_rel;
    // pre-training heads
    LinearW lm_transform, img_transform, img_decoder, lm_decoder;
    LNW lm_ln, img_ln;
    float* lm_bias = nullptr;
    std::map<std::string, HostTensor> sd;
    std::map<std::vector<int64_t>, std::unique_ptr<Plan>> plans;
    bool timeline = false;          // vb200_set_option("timeline", 1): plans built from now on record per-CTA stamps (vb200_timeline)
    int profile_grid_pct = 0;       // vb200_set_option("profile_grid_pct"): persistent-grid override for vb200_profile_ops only
    uint64_t use_clock = 0;         // LRU clock of the plan cache
    size_t max_plans = 24;          // VB200_MAX_PLANS: least-recently-used plans beyond this are destroyed (workspace + graph)
    cudaStream_t side_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    std::vector<std::string> schedule;

    ~vb200_engine() {
        plans.clear();
        if (side_stream) cudaStreamDestroy(side_stream);
        if (ev_fork) cudaEventDestroy(ev_fork);
        if (ev_join) cudaEventDestroy(ev_join);
    }

    // ---------------------------------------------------------------- checkpoint ingestion
    HostTensor& need(const std::string& name, int ndim, int64_t d0, int64_t d1 = 0) {
        auto it = sd.find(name);
        if (it == sd.end()) fail(VB200_ERR_CHECKPOINT, "checkpoint is missing key \"%s\"", name.c_str());
        HostTensor& t = it->second;
        if (t.ndim != ndim || t.shape[0] != d0 || (ndim == 2 && t.shape[1] != d1))
            fail(VB200_ERR_CHECKPOINT, "checkpoint key \"%s\" has shape [%lld,%lld] (ndim %d), expected [%lld,%lld] (ndim %d)",
                 name.c_str(), (long long)t.shape[0], (long long)t.shape[1], t.ndim, (long long)d0, (long long)d1, ndim);
        t.used = true;
        return t;
    }
    float* upload_f32(const std::vector<float>& h) {
        if (dry) return nullptr;
        float* d = weights.alloc_n<float>(h.size());
        CUDA_CHECK(cudaMemcpy(d, h.data(), h.size() * 4, cudaMemcpyHostToDevice));
        return d;
    }
    float* load_vec(const std::string& name, int64_t n) {
        HostTensor& t = need(name, 1, n);
        if (dry) return nullptr;
        std::vector<float> h(n);
        for (int64_t i = 0; i < n; ++i) h[i] = t.at(i);
        return upload_f32(h);
    }
    float* load_mat_f32(const std::string& name, int64_t r, int64_t c) {
        HostTensor& t = need(name, 2, r, c);
        if (dry) return nullptr;
        std::vector<float> h(r * c);
        if (t.dtype == VB200_F32) memcpy(h.data(), t.data, h.size() * 4);
        else for (int64_t i = 0; i < r * c; ++i) h[i] = t.at(i);
        return upload_f32(h);
    }
    std::map<std::string, LNW> ln_cache;        // every LayerNorm is loaded once (a fold source is needed before its own layer)
    LNW load_ln(const std::string& prefix, int n) {
        auto it = ln_cache.find(prefix);
        if (it != ln_cache.end()) return it->second;
        LNW l; l.n = n;
        HostTensor& tg = need(prefix + ".weight", 1, n);
        HostTensor& tb = need(prefix + ".bias", 1, n);
        if (!dry) {
            l.hg.resize(n); l.hb.resize(n);
            for (int i = 0; i < n; ++i) { l.hg[i] = tg.at(i); l.hb[i] = tb.at(i); }
            l.g = upload_f32(l.hg);
            l.b = upload_f32(l.hb);
        }
        ln_cache[prefix] = l;
        return l;
    }
    // one or several nn.Linear stacked along N (fused QKV), optional extra K columns from a second weight
    LinearW load_linear(const std::vector<std::string>& prefixes, int64_t n_each, int64_t k,
                        const std::string& extra_k_prefix = "", int64_t extra_k = 0, const LNW* fold = nullptr) {
        LinearW L;
        L.N = static_cast<int>(n_each * prefixes.size());
        L.K = static_cast<int>(k + (extra_k ? 64 : 0));
        L.ldw = (L.K + 63) / 64 * 64;
        if (dry) {
            for (const std::string& p : prefixes) { need(p + ".weight", 2, n_each, k); need(p + ".bias", 1, n_each); }
            if (extra_k) { need(extra_k_prefix + ".weight", 2, n_each, extra_k); need(extra_k_prefix + ".bias", 1, n_each); }
            return L;
        }
        const bool f16 = opt.act_fp16 != 0;     // weights are stored in the same 16-bit format as the activations
        if (x3) { load_linear_split(L, prefixes, n_each, k, extra_k_prefix, extra_k); return L; }
        std::vector<uint16_t> h(static_cast<size_t>(L.N) * L.ldw, 0);
        std::vector<float> hb(L.N, 0.0f);
        if (fold != nullptr) {
            // LayerNorm fold: W' = g o W in 16 bits, s_n = sum of the ROUNDED W'[n,:] (so the mean term cancels exactly against
            // what the tensor cores multiply), c_n = sum_k b_k W[n,k] + bias_n
            if (extra_k || static_cast<int64_t>(fold->hg.size()) != k) fail(VB200_ERR_INVALID, "LayerNorm fold: width mismatch");
            std::vector<float> hs(L.N, 0.0f);
            for (size_t pi = 0; pi < prefixes.size(); ++pi) {
                HostTensor& w = need(prefixes[pi] + ".weight", 2, n_each, k);
                HostTensor& b = need(prefixes[pi] + ".bias", 1, n_each);
                for (int64_t n = 0; n < n_each; ++n) {
                    uint16_t* dst = &h[(pi * n_each + n) * L.ldw];
                    double sn = 0.0, cn = 0.0;
                    for (int64_t j = 0; j < k; ++j) {
                        const float wv = w.at(n * k + j);
                        dst[j] = cvt16(wv * fold->hg[j]);
                        sn += static_cast<double>(f16 ? half_bits_to_f32(dst[j]) : bf16_bits_to_f32(dst[j]));
                        cn += static_cast<double>(fold->hb[j]) * static_cast<double>(wv);
                    }
                    hs[pi * n_each + n] = static_cast<float>(sn);
                    hb[pi * n_each + n] = static_cast<float>(cn + static_cast<double>(b.at(n)));
                }
            }
            L.w = weights.alloc_n<bf16>(h.size());
            CUDA_CHECK(cudaMemcpy(L.w, h.data(), h.size() * 2, cudaMemcpyHostToDevice));
            L.bias = upload_f32(hb);
            L.fold_s = upload_f32(hs);
            L.fold_g = fold->g;
            return L;
        }
        for (size_t pi = 0; pi < prefixes.size(); ++pi) {
            HostTensor& w = need(prefixes[pi] + ".weight", 2, n_each, k);
            HostTensor& b = need(prefixes[pi] + ".bias", 1, n_each);
            for (int64_t n = 0; n < n_each; ++n) {
                uint16_t* dst = &h[(pi * n_each + n) * L.ldw];
                if (w.dtype == VB200_F32) {
                    const float* src = static_cast<const float*>(w.data) + n * k;
                    if (f16) for (int64_t j = 0; j < k; ++j) dst[j] = f32_to_f16_bits(src[j]);
                    else for (int64_t j = 0; j < k; ++j) dst[j] = f32_to_bf16_bits(src[j]);
                } else {
                    for (int64_t j = 0; j < k; ++j) dst[j] = cvt16(w.at(n * k + j));
                }
                hb[pi * n_each + n] = b.at(n);
            }
        }
        if (extra_k) {
            HostTensor& w = need(extra_k_prefix + ".weight", 2, n_each, extra_k);
            HostTensor& b = need(extra_k_prefix + ".bias", 1, n_each);
            for (int64_t n = 0; n < n_each; ++n) {
                for (int64_t j = 0; j < extra_k; ++j) h[n * L.ldw + k + j] = cvt16(w.at(n * extra_k + j));
                hb[n] += b.at(n);
            }
        }
        L.w = weights.alloc_n<bf16>(h.size());
        CUDA_CHECK(cudaMemcpy(L.w, h.data(), h.size() * 2, cudaMemcpyHostToDevice));
        L.bias = upload_f32(hb);
        return L;
    }
    uint16_t cvt16(float f) const { return opt.act_fp16 ? f32_to_f16_bits(f) : f32_to_bf16_bits(f); }
    // fp32-parity mode: every weight is stored as fp16 hi | hi | lo per 64 columns of K (activations are hi | lo | hi), so the
    // K' = 3K GEMM adds hi.hi + lo.hi + hi.lo; physical row stride 3 * ldw.
    static void put_split_w(uint16_t* row, int64_t j, float w) {
        const uint16_t hi = f32_to_f16_bits(w);
        const uint16_t lo = f32_to_f16_bits(w - half_bits_to_f32(hi));
        uint16_t* d = row + (j >> 6) * 192 + (j & 63);
        d[0] = hi; d[64] = hi; d[128] = lo;
    }
    void load_linear_split(LinearW& L, const std::vector<std::string>& prefixes, int64_t n_each, int64_t k,
                           const std::string& extra_k_prefix, int64_t extra_k) {
        std::vector<uint16_t> h(static_cast<size_t>(L.N) * L.ldw * 3, 0);
        std::vector<float> hb(L.N, 0.0f);
        for (size_t pi = 0; pi < prefixes.size(); ++pi) {
            HostTensor& w = need(prefixes[pi] + ".weight", 2, n_each, k);
            HostTensor& b = need(prefixes[pi] + ".bias", 1, n_each);
            for (int64_t n = 0; n < n_each; ++n) {
                uint16_t* dst = &h[(pi * n_each + n) * L.ldw * 3];
                for (int64_t j = 0; j < k; ++j) put_split_w(dst, j, w.at(n * k + j));
                hb[pi * n_each + n] = b.at(n);
            }
        }
        if (extra_k) {
            HostTensor& w = need(extra_k_prefix + ".weight", 2, n_each, extra_k);
            HostTensor& b = need(extra_k_prefix + ".bias", 1, n_each);
            for (int64_t n = 0; n < n_each; ++n) {
                for (int64_t j = 0; j < extra_k; ++j) put_split_w(&h[n * L.ldw * 3], k + j, w.at(n * extra_k + j));
                hb[n] += b.at(n);
            }
        }
        L.w = weights.alloc_n<bf16>(h.size());
        CUDA_CHECK(cudaMemcpy(L.w, h.data(), h.size() * 2, cudaMemcpyHostToDevice));
        L.bias = upload_f32(hb);
    }
    LinearW load_linear1(const std::string& prefix, int64_t n, int64_t k, const LNW* fold = nullptr) {
        return load_linear({prefix}, n, k, "", 0, fold);
    }
    RowW load_row(const std::string& prefix, int n_out, int k) {
        RowW r; r.n_out = n_out; r.K = k;
        r.w = load_mat_f32(prefix + ".weight", n_out, k);
        r.b = load_vec(prefix + ".bias", n_out);
        return r;
    }
    // src: the pending LayerNorm of this layer's input (previous stage of the stream) when that one is folded, else null
    LayerW load_layer(const std::string& p, int hid, int inter, const LNW* src) {
        LayerW L;
        L.ln1 = load_ln(p + ".attention.output.LayerNorm", hid);
        L.ln2 = load_ln(p + ".output.LayerNorm", hid);
        L.qkv = load_linear({p + ".attention.self.query", p + ".attention.self.key", p + ".attention.self.value"}, hid, hid, "", 0, src);
        L.attn_out = load_linear1(p + ".attention.output.dense", hid, hid);
        L.inter = load_linear1(p + ".intermediate.dense", inter, hid, ln_fold ? &L.ln1 : nullptr);
        L.out = load_linear1(p + ".output.dense", hid, inter);
        return L;
    }
    ClsW load_cls(const std::string& p, int in_dim, int hid, int out_dim, bool narrow) {
        ClsW c;
        c.fc0 = load_linear1(p + ".logit_fc.0", hid, in_dim);
        c.ln = load_ln(p + ".logit_fc.2", hid);
        if (narrow) c.fc3_row = load_row(p + ".logit_fc.3", out_dim, hid);
        else c.fc3 = load_linear1(p + ".logit_fc.3", out_dim, hid);
        return c;
    }

    void ingest(int64_t n_tensors, const vb200_tensor* tensors) {
        for (int64_t i = 0; i < n_tensors; ++i) {
            const vb200_tensor& t = tensors[i];
            if (t.name == nullptr || t.data == nullptr) fail(VB200_ERR_CHECKPOINT, "state_dict entry %lld has a NULL name or data pointer", (long long)i);
            if (t.ndim < 1 || t.ndim > 2 || t.dtype < 0 || t.dtype > 2)
                fail(VB200_ERR_CHECKPOINT, "state_dict entry \"%s\": unsupported ndim %d / dtype %d", t.name, t.ndim, t.dtype);
            std::string name = t.name;
            if (name.rfind("module.", 0) == 0) name = name.substr(7);          // DataParallel prefix
            // old checkpoints: LayerNorm gamma/beta -> weight/bias
            auto ends = [&](const char* s) { size_t n = strlen(s); return name.size() >= n && name.compare(name.size() - n, n, s) == 0; };
            if (ends(".gamma")) name = name.substr(0, name.size() - 6) + ".weight";
            else if (ends(".beta")) name = name.substr(0, name.size() - 5) + ".bias";
            HostTensor h; h.dtype = t.dtype; h.ndim = t.ndim; h.shape[0] = t.shape[0]; h.shape[1] = t.ndim == 2 ? t.shape[1] : 0; h.data = t.data;
            sd[name] = h;
        }
        const Config& c = cfg;
        // vil_prediction width comes from the checkpoint unless the caller pins it (worker.py:523 passes 3129)
        {
            auto it = sd.find("vil_prediction.logit_fc.3.weight");
            if (it == sd.end()) fail(VB200_ERR_CHECKPOINT, "checkpoint is missing key \"vil_prediction.logit_fc.3.weight\"");
            const int ck = static_cast<int>(it->second.shape[0]);
            if (opt.num_labels > 0 && opt.num_labels != ck)
                fail(VB200_ERR_CHECKPOINT, "num_labels=%d but the checkpoint's vil_prediction head has %d outputs", opt.num_labels, ck);
            num_labels = ck;
            auto ig = sd.find("vil_prediction_gqa.logit_fc.3.weight");
            if (ig == sd.end()) fail(VB200_ERR_CHECKPOINT, "checkpoint is missing key \"vil_prediction_gqa.logit_fc.3.weight\"");
            gqa_labels = static_cast<int>(ig->second.shape[0]);
        }
        word = load_mat_f32("bert.embeddings.word_embeddings.weight", c.vocab, c.hidden);
        pos = load_mat_f32("bert.embeddings.position_embeddings.weight", c.max_pos, c.hidden);
        type = load_mat_f32("bert.embeddings.token_type_embeddings.weight", c.type_vocab, c.hidden);
        if (c.task_tokens) task = load_mat_f32("bert.embeddings.task_embeddings.weight", c.n_task, c.hidden);
        emb_ln = load_ln("bert.embeddings.LayerNorm", c.hidden);
        img_emb = load_linear({"bert.v_embeddings.image_embeddings"}, c.v_hidden, c.v_feat,
                              "bert.v_embeddings.image_location_embeddings", 5);
        vemb_ln = load_ln("bert.v_embeddings.LayerNorm", c.v_hidden);
        // [UPSTREAM] BertEncoder.forward schedule
        {
            int v_start = 0, t_start = 0;
            for (size_t i = 0; i < c.v_bi_id.size(); ++i) {
                const int v_end = c.v_bi_id[i], t_end = c.t_bi_id[i];
                for (int k = t_start; k < t_end; ++k) schedule.push_back("T" + std::to_string(k));
                for (int k = v_start; k < v_end; ++k) schedule.push_back("V" + std::to_string(k));
                schedule.push_back("C" + std::to_string(i));
                v_start = v_end; t_start = t_end;
            }
            for (int k = v_start; k < c.v_layers; ++k) schedule.push_back("V" + std::to_string(k));
            for (int k = t_start; k < c.layers; ++k) schedule.push_back("T" + std::to_string(k));
        }
        // LayerNorm fold map (gemm_persistent.cuh row_stats).  Each stream is a chain of stages (text: T layers and the text half of
        // the connection layers; image: the embedding, V layers, the image half of the connection layers).  A stage's OUTPUT
        // LayerNorm stays pending -- folded into the next stage's first GEMM and rebuilt in its residual -- unless the stage is the
        // stream's last one (poolers, heads and the output taps read real values) or the last one ahead of the first connection
        // layer (that is where the retrieval path caches per-caption / per-image states, and every plan mode must compute the same
        // bits).  The LayerNorm INSIDE a stage (after the attention / co-attention output projection) always folds.
        std::vector<std::string> t_st, v_st{"E"};
        for (const std::string& st : schedule) {
            if (st[0] == 'T' || st[0] == 'C') t_st.push_back(st);
            if (st[0] == 'V' || st[0] == 'C') v_st.push_back(st);
        }
        auto stage_ln = [&](const std::string& st, bool text) -> std::pair<std::string, int> {
            const std::string i = st.substr(st[0] == 'E' ? 0 : 1);
            if (st[0] == 'E') return {"bert.v_embeddings.LayerNorm", c.v_hidden};
            if (st[0] == 'T') return {"bert.encoder.layer." + i + ".output.LayerNorm", c.hidden};
            if (st[0] == 'V') return {"bert.encoder.v_layer." + i + ".output.LayerNorm", c.v_hidden};
            return text ? std::make_pair("bert.encoder.c_layer." + i + ".t_output.LayerNorm", c.hidden)
                        : std::make_pair("bert.encoder.c_layer." + i + ".v_output.LayerNorm", c.v_hidden);
        };
        // src_of[stage] = the previous stage's output LayerNorm if it folds, else nothing; fold_out[stage] as above
        std::map<std::string, LNW> src_t, src_v;
        auto walk = [&](const std::vector<std::string>& stages, bool text, std::map<std::string, LNW>& src, std::set<std::string>& folds) {
            int first_c = -1;
            for (size_t i = 0; i < stages.size(); ++i) if (stages[i][0] == 'C') { first_c = static_cast<int>(i); break; }
            for (size_t i = 0; i < stages.size(); ++i) {
                const bool fo = ln_fold && i + 1 < stages.size() && static_cast<int>(i) != first_c - 1;
                if (fo) {
                    folds.insert(stages[i]);
                    auto nm = stage_ln(stages[i], text);
                    src[stages[i + 1]] = load_ln(nm.first, nm.second);
                }
            }
        };
        walk(t_st, true, src_t, fold_out_t);
        walk(v_st, false, src_v, fold_out_v);
        auto src_ptr = [](std::map<std::string, LNW>& m, const std::string& st) -> const LNW* {
            auto it = m.find(st);
            return it == m.end() ? nullptr : &it->second;
        };
        for (int i = 0; i < c.layers; ++i)
            t_layers.push_back(load_layer("bert.encoder.layer." + std::to_string(i), c.hidden, c.inter, src_ptr(src_t, "T" + std::to_string(i))));
        for (int i = 0; i < c.v_layers; ++i)
            v_layers.push_back(load_layer("bert.encoder.v_layer." + std::to_string(i), c.v_hidden, c.v_inter, src_ptr(src_v, "V" + std::to_string(i))));
        for (size_t i = 0; i < c.v_bi_id.size(); ++i) {
            const std::string p = "bert.encoder.c_layer." + std::to_string(i);
            const std::string cs = "C" + std::to_string(i);
            ConnW w;
            w.ln1 = load_ln(p + ".biOutput.LayerNorm1", c.v_hidden);
            w.ln2 = load_ln(p + ".biOutput.LayerNorm2", c.hidden);
            w.v_ln = load_ln(p + ".v_output.LayerNorm", c.v_hidden);
            w.t_ln = load_ln(p + ".t_output.LayerNorm", c.hidden);
            w.qkv_img = load_linear({p + ".biattention.query1", p + ".biattention.key1", p + ".biattention.value1"}, c.bi_hidden, c.v_hidden,
                                    "", 0, src_ptr(src_v, cs));
            w.qkv_txt = load_linear({p + ".biattention.query2", p + ".biattention.key2", p + ".biattention.value2"}, c.bi_hidden, c.hidden,
                                    "", 0, src_ptr(src_t, cs));
            w.dense1 = load_linear1(p + ".biOutput.dense1", c.v_hidden, c.bi_hidden);
            w.dense2 = load_linear1(p + ".biOutput.dense2", c.hidden, c.bi_hidden);
            w.v_inter = load_linear1(p + ".v_intermediate.dense", c.v_inter, c.v_hidden, ln_fold ? &w.ln1 : nullptr);
            w.v_out = load_linear1(p + ".v_output.dense", c.v_hidden, c.v_inter);
            w.t_inter = load_linear1(p + ".t_intermediate.dense", c.inter, c.hidden, ln_fold ? &w.ln2 : nullptr);
            w.t_out = load_linear1(p + ".t_output.dense", c.hidden, c.inter);
            c_layers.push_back(w);
            // [UPSTREAM] present in the checkpoint, never applied in forward
            for (const char* u : {".biOutput.q_dense1.weight", ".biOutput.q_dense1.bias", ".biOutput.q_dense2.weight", ".biOutput.q_dense2.bias"}) {
                auto it = sd.find(p + u);
                if (it != sd.end()) it->second.used = true;
            }
        }
        t_pool = load_linear1("bert.t_pooler.dense", c.bi_hidden, c.hidden);
        v_pool = load_linear1("bert.v_pooler.dense", c.bi_hidden, c.v_hidden);
        vqa = load_cls("vil_prediction", c.bi_hidden, 2 * c.bi_hidden, num_labels, false);
        gqa = load_cls("vil_prediction_gqa", c.bi_hidden, 2 * c.bi_hidden, gqa_labels, false);
        binary = load_cls("vil_binary_prediction", 2 * c.bi_hidden, 2 * c.bi_hidden, 2, true);
        vil_logit = load_row("vil_logit", 1, c.bi_hidden);
        vil_tri = load_row("vil_tri_prediction", 3, c.bi_hidden);
        vision_logit = load_row("vision_logit", 1, c.v_hidden);
        ling_logit = load_row("linguisic_logit", 1, c.hidden);
        seq_rel = load_row("cls.bi_seq_relationship", 2, c.bi_hidden);
        lm_transform = load_linear1("cls.predictions.transform.dense", c.hidden, c.hidden);
        lm_ln = load_ln("cls.predictions.transform.LayerNorm", c.hidden);
        lm_bias = load_vec("cls.predictions.bias", c.vocab);
        img_transform = load_linear1("cls.imagePredictions.transform.dense", c.v_hidden, c.v_hidden);
        img_ln = load_ln("cls.imagePredictions.transform.LayerNorm", c.v_hidden);
        img_decoder = load_linear1("cls.imagePredictions.decoder", c.v_target, c.v_hidden);
        {   // tied LM decoder: bf16 copy of the word-embedding table as a [vocab, hidden] GEMM operand
            HostTensor& w = need("bert.embeddings.word_embeddings.weight", 2, c.vocab, c.hidden);
            if (!dry) {
                std::vector<uint16_t> h(static_cast<size_t>(c.vocab) * c.hidden * (x3 ? 3 : 1));
                if (x3) {
                    for (int64_t n = 0; n < c.vocab; ++n)
                        for (int64_t j = 0; j < c.hidden; ++j) put_split_w(&h[static_cast<size_t>(n) * c.hidden * 3], j, w.at(n * c.hidden + j));
                } else {
                    for (size_t i = 0; i < h.size(); ++i) h[i] = cvt16(w.at(i));
                }
                word_b16 = weights.alloc_n<bf16>(h.size());
                CUDA_CHECK(cudaMemcpy(word_b16, h.data(), h.size() * 2, cudaMemcpyHostToDevice));
            }
            lm_decoder.w = word_b16; lm_decoder.bias = lm_bias; lm_decoder.N = c.vocab; lm_decoder.K = c.hidden; lm_decoder.ldw = c.hidden;
            auto it = sd.find("cls.predictions.decoder.weight");   // tied duplicate of the word table
            if (it != sd.end()) it->second.used = true;
            auto ip = sd.find("bert.embeddings.position_ids");
            if (ip != sd.end()) ip->second.used = true;
        }
        if (opt.strict) {
            std::string extra;
            int n = 0;
            for (auto& kv : sd) if (!kv.second.used) { if (n++ < 8) extra += " \"" + kv.first + "\""; }
            if (n) fail(VB200_ERR_CHECKPOINT, "checkpoint has %d unexpected key(s):%s%s", n, extra.c_str(), n > 8 ? " ..." : "");
        }
        sd.clear();   // host pointers are the caller's; do not keep them
        ln_cache.clear();
    }

    // ---------------------------------------------------------------- plan construction
    // One nn.Linear (+ activation, + residual LayerNorm) -> one or two launch-list entries on `stream`.
    //   fused_ln:  a single cluster-LayerNorm GEMM (epilogue normalises across the N tiles of a cluster)
    //   default :  GEMM (+bias, +activation) writing fp32 to the stream's scratch, then the row LayerNorm kernel
    //              (adds the residual) -- measured faster at every batch size tried (profiles/).
    // All sizes are LOGICAL (elements of the mathematical matrices).  In fp32-parity mode (x3) every 16-bit operand buffer is
    // physically 3x as wide (fp16 hi | lo | hi per 64 columns), so operand strides, the contraction length and the 16-bit
    // output stride are multiplied by S = 3 here and nowhere else.
    // LayerNorm fold (row_stats in gemm_persistent.cuh): what add_linear needs to know beyond the plain call
    struct FoldArgs {
        const float2* a_stats = nullptr;   // the A operand's LayerNorm is pending: its row statistics (W must be a folded Linear)
        int a_parts = 0;
        const float2* res_stats = nullptr; // the residual's LayerNorm is pending: its statistics and parameters
        int res_parts = 0;
        const LNW* res_ln = nullptr;
        float2* out_stats = nullptr;       // keep THIS Linear's LayerNorm pending: write u (fp32 + 16-bit) and its statistics here
        int stats_ld = 0;
    };
    void add_linear(Plan& pl, const bf16* A, int64_t a_rows, int64_t lda, const LinearW& W, int act, const float* res, int ld_res,
                    const LNW* ln, bf16* out_b, int ld_b, float* out_f, int ld_f, int stream = 0, Op::Sync sync = Op::NONE,
                    const float* mul = nullptr, int ld_mul = 0, const FoldArgs* fa = nullptr) {
        const int S = x3 ? 3 : 1;
        const bool keep_pending = ln != nullptr && fa != nullptr && fa->out_stats != nullptr;
        const bool fold_in = fa != nullptr && fa->a_stats != nullptr;
        if ((W.fold_s != nullptr) != fold_in)
            fail(VB200_ERR_INVALID, "LayerNorm fold: Linear N=%d K=%d was %s with a pending LayerNorm but its input is %s", W.N, W.K,
                 W.fold_s ? "folded" : "not folded", fold_in ? "pending" : "final");
        const bool split_ln = ln != nullptr && !fused_ln && !keep_pending;
        if (x3 && act == vb::kActGelu) act = vb::kActGeluExact;
        Op op{};
        op.kind = Op::GEMM;
        op.stream = stream;
        op.sync = sync;
        op.ln = ln != nullptr && !split_ln && !keep_pending;      // cluster-LayerNorm epilogue (fused_layernorm option)
        op.block_n = vb::gemm_p_pick_block_n(W.N, op.ln);
        if (op.block_n == 0) fail(VB200_ERR_INVALID, "no LayerNorm-fused GEMM tiling for N=%d", W.N);
        if (!x3 && !op.ln && !keep_pending && !fold_in && a_rows >= 256) {
            if (pair_bn > 0) op.pair = W.N % pair_bn == 0;
            else if (pair_bn < 0) {
                const long long panels = (a_rows + 255) / 256;
                const int waves = pair_min_waves > 0 ? pair_min_waves : (panels >= 20 ? 2 : 4);
                op.pair = W.N % 256 == 0 && panels * (W.N / 256) >= static_cast<long long>(waves) * (vb::num_sms_host() / 2);
            }
            if (op.pair) op.block_n = pair_bn > 0 ? pair_bn : 256;
        }
        if (wide192 && !x3 && !op.ln && !op.pair && !keep_pending && !fold_in && W.N % 192 == 0 && op.block_n == 128) {
            // 128x192 tiles when 128-wide ones need more than one wave of the 2-per-SM CTA slots and 192-wide ones fit in one
            // (the N = 3072 GEMMs at batch 64).  The tile width never changes an element's accumulation order: results are the same bits.
            const long long slots = 2LL * vb::num_sms_host(), mt = (a_rows + 127) / 128;
            if (mt * ((W.N + 127) / 128) > slots && mt * (W.N / 192) <= slots) op.block_n = 192;
        }
        // Small forwards (<= lone_rows rows in either stream, batch <= 8): one CTA per SM with a 6-stage ring (PCfg MODE 7), and 64-wide
        // tiles while they still fit one per SM -- twice the CTAs, half the epilogue each (batch 1: 0.932 -> 0.869 ms per forward,
        // profiles/r2_small_batch_latency.md).  Neither changes an element's accumulation order.
        bool lone = false;
        if (lone_rows > 0 && tri_min_tiles == 0 && !x3 && !op.ln && !op.pair && !keep_pending && !fold_in && (op.block_n == 128 || op.block_n == 64) &&
            std::max(pl.B * pl.T, pl.B * pl.V) <= lone_rows) {
            const long long mt = (a_rows + 127) / 128;
            if (mt * ((W.N + 127) / 128) <= vb::num_sms_host()) {
                lone = true;
                if (W.N % 64 == 0 && mt * (W.N / 64) <= vb::num_sms_host()) op.block_n = 64;
            }
        }
        op.ta = make_tmap(A, a_rows, static_cast<int64_t>(W.ldw) * S, lda * S, 128, opt.act_fp16 != 0);
        op.tb = make_tmap(W.w, W.N, static_cast<int64_t>(W.ldw) * S, static_cast<int64_t>(W.ldw) * S, op.pair ? op.block_n / 2 : op.block_n,
                          opt.act_fp16 != 0);
        GemmEpilogue& e = op.ep;
        if (tri_min_tiles > 0 && !x3 && !op.ln && !op.pair && !keep_pending && !fold_in && op.block_n == 128 &&
            ((a_rows + 127) / 128) * ((W.N + 127) / 128) >= tri_min_tiles) e.tri = 1;
        if (lone) e.lone = 1;
        e.M = static_cast<int>(a_rows); e.N = W.N; e.K = W.ldw * S;
        e.bias = W.bias; e.mul = mul; e.ld_mul = ld_mul; e.eps = cfg.ln_eps; e.act = act; e.pdl = pdl_light ? 2 : (opt.use_pdl ? (early_w ? 5 : 1) : 0);
        e.a_f16 = opt.act_fp16; e.out_f16 = opt.act_fp16;
        if (fold_in) {
            e.ln_mode = 4; e.a_stats = fa->a_stats; e.a_parts = fa->a_parts; e.fold_s = W.fold_s; e.stats_ld = fa->stats_ld;
        }
        if (split_ln) {
            e.out_f32 = pl.y_scratch[stream]; e.ld_f32 = W.N;
        } else if (keep_pending) {
            // producer of a pending LayerNorm: u = acc + bias + residual in fp32 and 16 bits, plus the row statistics
            e.ln_mode = 5; e.res = res; e.ld_res = ld_res;
            e.res_stats = fa->res_stats; e.res_parts = fa->res_parts;
            e.res_gamma = fa->res_ln ? fa->res_ln->g : nullptr; e.res_beta = fa->res_ln ? fa->res_ln->b : nullptr;
            e.out_stats = fa->out_stats; e.stats_ld = fa->stats_ld;
            e.out_bf16 = out_b; e.ld_bf16 = ld_b; e.out_f32 = out_f; e.ld_f32 = ld_f;
        } else {
            e.res = res; e.ld_res = ld_res;
            e.gamma = ln ? ln->g : nullptr; e.beta = ln ? ln->b : nullptr;
            e.out_bf16 = out_b; e.ld_bf16 = ld_b * S; e.out_f32 = out_f; e.ld_f32 = ld_f;
            e.split16 = (x3 && out_b != nullptr) ? 1 : 0;
            if (e.split16 && (W.N & 63)) fail(VB200_ERR_INVALID, "fp32-parity mode: 16-bit GEMM output of width %d is not a multiple of 64", W.N);
        }
        if (tma_store_enabled && !op.pair && !op.ln) setup_tma_store(&op.tc, e);
        op.flops = 2.0 * a_rows * W.N * W.K;
        op.a_ptr = A;
        pl.flops += op.flops;
        pl.ops.push_back(op);
        if (split_ln) {
            Op l{};
            l.kind = Op::LAYERNORM;
            l.stream = stream;
            l.ln_y = pl.y_scratch[stream]; l.ln_res = res; l.ld_x = ld_res;
            l.ln_g = ln->g; l.ln_b = ln->b; l.ln_out_f = out_f; l.ln_out_h = out_b; l.ln_ld = W.N;
            l.ld_out = out_f ? ld_f : 0; l.ld_a = out_b ? ld_b * S : 0;
            l.ln_M = static_cast<int>(a_rows); l.ln_N = W.N;
            if (fa != nullptr && fa->res_stats != nullptr)
                l.ln_pend = vb::LnPending{fa->res_stats, fa->res_parts, fa->stats_ld, fa->res_ln->g, fa->res_ln->b};
            pl.ops.push_back(l);
        }
    }
    // softmax(Q K^T / sqrt(d) + mask) V of one stream (self) or one direction of a connection layer.  Default: the tensor-core
    // kernel writes the context (callers push that op themselves); this adds the fp32 kernel -- as THE attention in fp32-parity
    // mode (context out as hi | lo | hi), and/or as the producer of the attention-probability output.
    void add_attn_f32(Plan& pl, const void* q, int ld_q, const void* k, const void* v, int ld_kv, const float* mask, int Lq, int Lk,
                      int heads, int hid, bf16* ctx, bool want_probs, int stream) {
        Op a{};
        a.kind = Op::ATTN_F32;
        a.stream = stream;
        a.f_q = q; a.f_k = k; a.f_v = v; a.f_ld_q = ld_q; a.f_ld_kv = ld_kv; a.f_mask = mask; a.f_Lq = Lq; a.f_Lk = Lk;
        a.f_in = x3 ? 0 : (opt.act_fp16 ? 1 : 2);
        a.B = pl.B; a.heads = heads; a.head_dim = hid / heads;
        a.f_ctx = x3 ? ctx : nullptr; a.f_ctx_mode = x3 ? 3 : 0; a.f_ld_ctx = x3 ? 3 * hid : 0;
        if (want_probs) {
            a.f_probs = pl.mem.alloc_n<float>(static_cast<size_t>(pl.B) * heads * Lq * Lk);
            pl.attn.push_back(Plan::AttnOut{a.f_probs, heads, Lq, Lk});
        }
        if (x3) { a.flops = 4.0 * pl.B * heads * Lq * Lk * (hid / heads); pl.flops += a.flops; }
        pl.ops.push_back(a);
    }
    Op rowdot_op(const float* x, int ld_x, const RowW& w, const float* add, float* out, int ld_out, int M) {
        Op op{};
        op.kind = Op::ROWDOT;
        op.x = x; op.ld_x = ld_x; op.W = w.w; op.bias = w.b; op.add = add; op.out = out; op.ld_out = ld_out;
        op.M = M; op.K = w.K; op.n_out = w.n_out;
        op.flops = 2.0 * M * w.K * w.n_out;
        return op;
    }
    OutBuf make_out(Plan& pl, int rows, int cols) {
        OutBuf o; o.rows = rows; o.cols = cols; o.ld = (cols + 3) / 4 * 4;
        o.p = pl.mem.alloc_n<float>(static_cast<size_t>(rows) * o.ld);
        return o;
    }

    // Plan modes.  FULL is the reference's forward (worker.py:286-289).  The other three split it at the first connection layer
    // for caption-image retrieval (SURVEY.md section 8e): everything before it depends on the caption alone (text embeddings +
    // the text layers scheduled ahead of C0) or on the image alone (image embedding + any image layer ahead of C0), so a
    // 1000 x 1000 score matrix computes those once per caption / per image and runs only the SUFFIX per pair -- the same kernels on
    // the same rows, hence bit-identical scores.
    enum PlanMode { FULL = 0, TEXT_PREFIX = 1, IMAGE_PREFIX = 2, SUFFIX = 3 };

    // Pruned tail.  When a stream's last step is a single-stream layer after the last connection layer and nothing selected reads
    // that stream's sequence (no per-row head, no sequence-output tap, no attention maps), the only reader of the layer's output is
    // the pooler, which takes row 0 of each sample.  Then everything after the QKV projection (keys and values are still needed for
    // every row) runs on those B rows alone.  Every kernel computes a row from that row alone in a fixed order, so the pooled
    // outputs keep their bits.  Returns bit 0 for the text stream, bit 1 for the image stream.  seq_out: the same two bits for the
    // sequence outputs the caller asks for.  The opt-in fp32-parity, LayerNorm-fold, fused-LayerNorm and chained-FFN modes keep the
    // full tail.
    int tail_prunable(uint32_t select, int mode, bool want_attn, int seq_out) const {
        if (!prune_tail || x3 || ln_fold || fused_ln || chain_ffn || want_attn || mode == TEXT_PREFIX || mode == IMAGE_PREFIX) return 0;
        int last_t = -1, last_v = -1, last_c = -1;
        for (size_t i = 0; i < schedule.size(); ++i) {
            const int k = static_cast<int>(i);
            if (schedule[i][0] == 'T') last_t = k; else if (schedule[i][0] == 'V') last_v = k; else last_c = k;
        }
        int bits = 0;
        if (last_t > last_c && !(seq_out & 1) && !(select & (VB200_OUT_LINGUISIC_PREDICTION | VB200_OUT_LINGUISIC_LOGIT))) bits |= 1;
        if (last_v > last_c && !(seq_out & 2) && !(select & (VB200_OUT_VISION_PREDICTION | VB200_OUT_VISION_LOGIT))) bits |= 2;
        return bits;
    }

    // seq_out: bit 0 / bit 1 = the caller reads the final text / image sequence (vb200_outputs::sequence_output_t / _v)
    Plan* get_plan(int B, int Tin, int V, uint32_t select, int slot = 0, int mode = FULL, bool want_attn = false, int seq_out = 0) {
        if (slot < 0 || slot > 15) fail(VB200_ERR_INVALID, "slot %d out of range (0..15)", slot);
        if (slot > 0 && !opt.use_cuda_graph) fail(VB200_ERR_INVALID, "concurrent slots need CUDA-graph plans (use_cuda_graph)");
        if (mode == TEXT_PREFIX || mode == IMAGE_PREFIX) { select = 0; want_attn = false; }
        const int prune = tail_prunable(select, mode, want_attn, seq_out);
        std::vector<int64_t> key{B, Tin, V, static_cast<int64_t>(select), slot, mode, want_attn ? 1 : 0, prune};
        auto it = plans.find(key);
        if (it != plans.end()) { it->second->last_use = ++use_clock; return it->second.get(); }
        std::unique_ptr<Plan> up(new Plan());
        Plan& pl = *up;
        const Config& c = cfg;
        const int T = Tin + (c.task_tokens ? 1 : 0);
        if (B < 1 || Tin < 1 || V < 1) fail(VB200_ERR_INVALID, "batch, n_tokens and n_regions must be positive");
        if (T > 256 || V > 256) fail(VB200_ERR_INVALID, "sequence too long for the small-sequence attention kernels (T=%d, V=%d, max 256)", T, V);
        if (Tin > c.max_pos) fail(VB200_ERR_INVALID, "n_tokens %d exceeds max_position_embeddings %d", Tin, c.max_pos);
        pl.B = B; pl.Tin = Tin; pl.T = T; pl.V = V; pl.select = select;
        const int Mt = B * T, Mv = B * V, H = c.hidden, Hv = c.v_hidden, Hb = c.bi_hidden;
        const size_t S = x3 ? 3 : 1;                 // physical width factor of the 16-bit operand buffers (fp32-parity mode)
        const bool do_t = mode == FULL || mode == TEXT_PREFIX, do_v = mode == FULL || mode == IMAGE_PREFIX;
        const bool do_s = mode == FULL || mode == SUFFIX;
        pl.kp = img_emb.ldw;
        pl.img_a = pl.mem.alloc_n<bf16>(static_cast<size_t>(Mv) * pl.kp * S);
        pl.mask_t = pl.mem.alloc_n<float>(Mt);
        pl.mask_v = pl.mem.alloc_n<float>(Mv);
        for (int i = 0; i < 2; ++i) {
            pl.t_f32[i] = pl.mem.alloc_n<float>(static_cast<size_t>(Mt) * H);
            pl.t_b16[i] = pl.mem.alloc_n<bf16>(static_cast<size_t>(Mt) * H * S);
            pl.v_f32[i] = pl.mem.alloc_n<float>(static_cast<size_t>(Mv) * Hv);
            pl.v_b16[i] = pl.mem.alloc_n<bf16>(static_cast<size_t>(Mv) * Hv * S);
        }
        if (!fused_ln) {
            const size_t n0 = std::max({static_cast<size_t>(Mt) * H, static_cast<size_t>(Mv) * Hv, static_cast<size_t>(B) * 2 * Hb});
            pl.y_scratch[0] = pl.mem.alloc_n<float>(n0);
            pl.y_scratch[1] = pl.mem.alloc_n<float>(static_cast<size_t>(Mv) * Hv);
        }
        const int qt = 3 * std::max(H, Hb), qv = 3 * std::max(Hv, Hb);
        // Q | K | V projections: 16-bit for the tensor-core attention kernel, fp32 in fp32-parity mode
        const size_t qe = x3 ? 4 : 2;
        uint8_t* qkv_t = static_cast<uint8_t*>(pl.mem.alloc(static_cast<size_t>(Mt) * qt * qe));
        uint8_t* qkv_v = static_cast<uint8_t*>(pl.mem.alloc(static_cast<size_t>(Mv) * qv * qe));
        bf16* ctx_t = pl.mem.alloc_n<bf16>(static_cast<size_t>(Mt) * std::max(H, Hb) * S);
        bf16* ctx_v = pl.mem.alloc_n<bf16>(static_cast<size_t>(Mv) * std::max(Hv, Hb) * S);
        bf16* inter_t = pl.mem.alloc_n<bf16>(static_cast<size_t>(Mt) * c.inter * S);
        bf16* inter_v = pl.mem.alloc_n<bf16>(static_cast<size_t>(Mv) * c.v_inter * S);
        auto& ops = pl.ops;
        auto qkv_out = [&](uint8_t* q, bf16*& ob, float*& of) {       // where a QKV GEMM writes
            ob = x3 ? nullptr : reinterpret_cast<bf16*>(q);
            of = x3 ? reinterpret_cast<float*>(q) : nullptr;
        };
        auto qkv_at = [&](const uint8_t* q, int col) -> const void* { return q + static_cast<size_t>(col) * qe; };

        // ---- LayerNorm fold state of the two streams: `pend` = the LayerNorm still to be applied to buffers [cur] (null: the
        // buffers hold final values), its row statistics live in stats[cur]
        struct StreamSt {
            float** f32; bf16** b16; float2** stats; int cur; const LNW* pend; int hid, rows, stats_ld, stream; const float* mask; int seq;
            uint8_t* qkv; bf16* ctx; bf16* inter;
        };
        if (ln_fold) {
            pl.stats_ld_t = (Mt + 31) & ~31; pl.stats_ld_v = (Mv + 31) & ~31;
            for (int i = 0; i < 2; ++i) {
                pl.t_stats[i] = static_cast<float2*>(pl.mem.alloc(static_cast<size_t>(H / 32) * pl.stats_ld_t * sizeof(float2)));
                pl.v_stats[i] = static_cast<float2*>(pl.mem.alloc(static_cast<size_t>(Hv / 32) * pl.stats_ld_v * sizeof(float2)));
            }
        }
        StreamSt ts{pl.t_f32, pl.t_b16, pl.t_stats, 0, nullptr, H, Mt, pl.stats_ld_t, 0, pl.mask_t, T, qkv_t, ctx_t, inter_t};
        StreamSt vs{pl.v_f32, pl.v_b16, pl.v_stats, 0, nullptr, Hv, Mv, pl.stats_ld_v, 1, pl.mask_v, V, qkv_v, ctx_v, inter_v};
        auto fold_in_args = [&](const StreamSt& st, int which) {          // consume buffers[which] of a stream as a GEMM's A operand
            FoldArgs fa;
            fa.a_stats = st.stats[which]; fa.a_parts = st.hid / 32; fa.stats_ld = st.stats_ld;
            return fa;
        };
        // GEMM + LayerNorm whose residual is buffers[rwhich] of stream st (its own LayerNorm possibly pending: res_pend);
        // the result lands in buffers[owhich]; keep == true leaves THIS LayerNorm pending (statistics in stats[owhich]).
        // M rows of A; the residual and the result are M rows of the stream buffers ld elements apart (pruned tail: row 0 of each sample)
        auto ln_linear = [&](StreamSt& st, const bf16* A, int64_t M, int64_t lda, const LinearW& W, const LNW& ln, int rwhich,
                             const LNW* res_pend, int owhich, bool keep, Op::Sync sync, int ld) {
            FoldArgs fa;
            fa.stats_ld = st.stats_ld;
            if (res_pend != nullptr) { fa.res_stats = st.stats[rwhich]; fa.res_parts = st.hid / 32; fa.res_ln = res_pend; }
            if (keep) fa.out_stats = st.stats[owhich];
            add_linear(pl, A, M, lda, W, vb::kActNone, st.f32[rwhich], ld, &ln, st.b16[owhich], ld, st.f32[owhich], ld,
                       st.stream, sync, nullptr, 0, (res_pend != nullptr || keep) ? &fa : nullptr);
        };

        // ---- image embedding: LayerNorm(feat.W_img^T + loc.W_loc^T + b) as ONE GEMM over K = v_feat + 64
        if (do_v) {
            const bool keep = ln_fold && fold_out_v.count("E") != 0;
            FoldArgs fa;
            fa.stats_ld = vs.stats_ld;
            if (keep) fa.out_stats = vs.stats[0];
            add_linear(pl, pl.img_a, Mv, pl.kp, img_emb, vb::kActNone, nullptr, 0, &vemb_ln, pl.v_b16[0], Hv, pl.v_f32[0], Hv,
                       1, Op::NONE, nullptr, 0, keep ? &fa : nullptr);   // side stream: overlaps the text layers ahead of the first co-attention
        }
        if (do_v && ln_fold && fold_out_v.count("E") != 0) vs.pend = &vemb_ln;

        // one BertLayer / BertImageLayer.  keep_out: this stage's output LayerNorm stays pending (LayerNorm fold map, ingest()).
        // tail: pruned last layer of the stream (tail_prunable) -- QKV over every row, then attention, the output projection, the
        // FFN and both LayerNorms for row 0 of each sample only, in place (rows b * seq of the stream buffers, row stride seq * hid;
        // the FFN intermediate is compact [B, inter]).  The other rows of the stream buffers keep the layer's input.
        auto single_layer = [&](const LayerW& L, StreamSt& st, int inter, int heads, bool keep_out, bool tail) {
            const int hid = st.hid, cur = st.cur, stream = st.stream;
            const int M = tail ? B : st.rows, ld = tail ? st.seq * hid : hid, nq = tail ? 1 : st.seq;
            bf16* qb; float* qf;
            qkv_out(st.qkv, qb, qf);
            {
                FoldArgs fa = fold_in_args(st, cur);
                add_linear(pl, st.b16[cur], st.rows, hid, L.qkv, vb::kActNone, nullptr, 0, nullptr, qb, 3 * hid, qf, 3 * hid, stream, Op::NONE,
                           nullptr, 0, st.pend ? &fa : nullptr);
            }
            if (!x3) {
                Op a{};
                a.kind = Op::SELF_ATTN;
                a.stream = stream;
                a.qkv_a = qb; a.ld_a = 3 * hid; a.hidden = hid; a.mask_a = st.mask; a.ctx_a = st.ctx; a.ld_ctx_a = hid;
                a.B = B; a.La = st.seq; a.Lb = nq < st.seq ? nq : 0; a.heads = heads; a.head_dim = hid / heads;
                a.flops = 4.0 * B * heads * nq * st.seq * (hid / heads);
                pl.flops += a.flops;
                ops.push_back(a);
            }
            if (x3 || want_attn)
                add_attn_f32(pl, qkv_at(st.qkv, 0), 3 * hid, qkv_at(st.qkv, hid), qkv_at(st.qkv, 2 * hid), 3 * hid, st.mask, st.seq, st.seq,
                             heads, hid, st.ctx, want_attn, stream);
            // attention output + LayerNorm1 (residual: the layer input) -> buffers [1 - cur]
            ln_linear(st, st.ctx, M, ld, L.attn_out, L.ln1, cur, st.pend, 1 - cur, ln_fold, Op::NONE, ld);
            {
                FoldArgs fa = fold_in_args(st, 1 - cur);
                add_linear(pl, st.b16[1 - cur], M, ld, L.inter, vb::kActGelu, nullptr, 0, nullptr, st.inter, inter, nullptr, 0, stream,
                           Op::NONE, nullptr, 0, ln_fold ? &fa : nullptr);
            }
            // FFN output + LayerNorm2 (residual: LayerNorm1's output) -> buffers [cur]
            ln_linear(st, st.inter, M, inter, L.out, L.ln2, 1 - cur, ln_fold ? &L.ln1 : nullptr, cur, keep_out, Op::NONE, ld);
            st.pend = keep_out ? &L.ln2 : nullptr;
        };

        for (Op& op : ops) op.tag = "embed";
        bool in_suffix = false;
        size_t tagged = ops.size();
        const std::string* tail_t = nullptr, *tail_v = nullptr;          // the layers tail_prunable prunes (last T / last V step)
        for (const std::string& step : schedule) {
            if (step[0] == 'T' && (prune & 1)) tail_t = &step;
            if (step[0] == 'V' && (prune & 2)) tail_v = &step;
        }
        for (const std::string& step : schedule) {
            for (; tagged < ops.size(); ++tagged) if (ops[tagged].tag == nullptr) ops[tagged].tag = "?";
            const int idx = atoi(step.c_str() + 1);
            if (step[0] == 'C') in_suffix = true;
            struct Tagger {          // names the launches this step appends after its layer (engine.schedule outlives every plan)
                std::vector<Op>& ops; size_t from; const char* name;
                ~Tagger() { for (size_t i = from; i < ops.size(); ++i) ops[i].tag = name; }
            } tagger{ops, ops.size(), step.c_str()};
            if (step[0] == 'T') {
                if (in_suffix ? do_s : do_t)
                    single_layer(t_layers[idx], ts, c.inter, c.heads, ln_fold && fold_out_t.count(step) != 0, &step == tail_t);
            } else if (step[0] == 'V') {
                if (in_suffix ? do_s : do_v)
                    single_layer(v_layers[idx], vs, c.v_inter, c.v_heads, ln_fold && fold_out_v.count(step) != 0, &step == tail_v);
            } else if (do_s) {
                const ConnW& W = c_layers[idx];
                const int tcur = ts.cur, vcur = vs.cur;
                bf16 *qvb, *qtb; float *qvf, *qtf;
                qkv_out(qkv_v, qvb, qvf);
                qkv_out(qkv_t, qtb, qtf);
                {
                    FoldArgs fv = fold_in_args(vs, vcur), ft = fold_in_args(ts, tcur);
                    add_linear(pl, pl.v_b16[vcur], Mv, Hv, W.qkv_img, vb::kActNone, nullptr, 0, nullptr, qvb, 3 * Hb, qvf, 3 * Hb, 1, Op::NONE,
                               nullptr, 0, vs.pend ? &fv : nullptr);
                    add_linear(pl, pl.t_b16[tcur], Mt, H, W.qkv_txt, vb::kActNone, nullptr, 0, nullptr, qtb, 3 * Hb, qtf, 3 * Hb, 0, Op::NONE,
                               nullptr, 0, ts.pend ? &ft : nullptr);
                }
                const size_t first_co = ops.size();
                if (!x3) {
                    Op a{};
                    a.kind = Op::CO_ATTN;
                    a.qkv_a = qvb; a.ld_a = 3 * Hb; a.qkv_b = qtb; a.ld_b = 3 * Hb; a.hidden = Hb;
                    a.mask_a = pl.mask_v; a.mask_b = pl.mask_t; a.ctx_a = ctx_t; a.ld_ctx_a = Hb; a.ctx_b = ctx_v; a.ld_ctx_b = Hb;
                    a.B = B; a.La = T; a.Lb = V; a.heads = c.bi_heads; a.head_dim = Hb / c.bi_heads;
                    a.flops = 8.0 * B * c.bi_heads * T * V * (Hb / c.bi_heads);
                    pl.flops += a.flops;
                    ops.push_back(a);
                }
                if (x3 || want_attn) {
                    // text queries (Q2) over image keys / values (K1, V1) -> text context; then image queries (Q1) over K2, V2
                    add_attn_f32(pl, qkv_at(qkv_t, 0), 3 * Hb, qkv_at(qkv_v, Hb), qkv_at(qkv_v, 2 * Hb), 3 * Hb, pl.mask_v, T, V,
                                 c.bi_heads, Hb, ctx_t, want_attn, 0);
                    add_attn_f32(pl, qkv_at(qkv_v, 0), 3 * Hb, qkv_at(qkv_t, Hb), qkv_at(qkv_t, 2 * Hb), 3 * Hb, pl.mask_t, V, T,
                                 c.bi_heads, Hb, ctx_v, want_attn, 0);
                }
                ops[first_co].sync = Op::JOIN;              // needs both projections
                const bool keep_v = ln_fold && fold_out_v.count(step) != 0, keep_t = ln_fold && fold_out_t.count(step) != 0;
                // image branch (side stream; forks from the co-attention): biOutput.dense1 + LayerNorm1, v_intermediate, v_output + LayerNorm
                ln_linear(vs, ctx_v, Mv, Hb, W.dense1, W.ln1, vcur, vs.pend, 1 - vcur, ln_fold, Op::FORK, Hv);
                {
                    FoldArgs fa = fold_in_args(vs, 1 - vcur);
                    add_linear(pl, pl.v_b16[1 - vcur], Mv, Hv, W.v_inter, vb::kActGelu, nullptr, 0, nullptr, inter_v, c.v_inter, nullptr, 0, 1,
                               Op::NONE, nullptr, 0, ln_fold ? &fa : nullptr);
                }
                ln_linear(vs, inter_v, Mv, c.v_inter, W.v_out, W.v_ln, 1 - vcur, ln_fold ? &W.ln1 : nullptr, vcur, keep_v, Op::NONE, Hv);
                vs.pend = keep_v ? &W.v_ln : nullptr;
                // text branch (main stream)
                ln_linear(ts, ctx_t, Mt, Hb, W.dense2, W.ln2, tcur, ts.pend, 1 - tcur, ln_fold, Op::NONE, H);
                {
                    FoldArgs fa = fold_in_args(ts, 1 - tcur);
                    add_linear(pl, pl.t_b16[1 - tcur], Mt, H, W.t_inter, vb::kActGelu, nullptr, 0, nullptr, inter_t, c.inter, nullptr, 0, 0,
                               Op::NONE, nullptr, 0, ln_fold ? &fa : nullptr);
                }
                ln_linear(ts, inter_t, Mt, c.inter, W.t_out, W.t_ln, 1 - tcur, ln_fold ? &W.ln2 : nullptr, tcur, keep_t, Op::NONE, H);
                ts.pend = keep_t ? &W.t_ln : nullptr;
            }
        }
        if ((do_s || do_t) && ts.pend != nullptr) fail(VB200_ERR_INVALID, "LayerNorm fold: the text stream ends with a pending LayerNorm");
        if ((do_s || do_v) && vs.pend != nullptr) fail(VB200_ERR_INVALID, "LayerNorm fold: the image stream ends with a pending LayerNorm");
        const int tc = ts.cur, vc = vs.cur;
        pl.t_cur = tc; pl.v_cur = vc;
        // a pruned stream holds final values in row 0 of each sample only: its sequence output stays unavailable
        if (!(prune & 1)) pl.outs[9] = OutBuf{pl.t_f32[tc], Mt, H, H};
        if (!(prune & 2)) pl.outs[10] = OutBuf{pl.v_f32[vc], Mv, Hv, Hv};

        const size_t n_before_heads = ops.size();
        if (do_s) build_heads(pl, select);
        for (size_t i = n_before_heads; i < ops.size(); ++i) ops[i].tag = "heads";
        for (Op& op : ops) if (op.kind == Op::ROWDOT) pl.flops += op.flops;

        link_chains(pl);
        link_pdl(pl);
        if (timeline) attach_timeline(pl);
        // One eager pass first: opts kernels into their shared-memory sizes and surfaces launch-configuration
        // errors with a real message (errors inside a capture only invalidate the capture).
        if (!ops.empty()) {
            cudaStream_t ws;
            CUDA_CHECK(cudaStreamCreateWithFlags(&ws, cudaStreamNonBlocking));
            try { run_ops(pl, ws); } catch (...) { cudaStreamSynchronize(ws); cudaStreamDestroy(ws); throw; }
            cudaError_t e = cudaStreamSynchronize(ws);
            cudaStreamDestroy(ws);
            CUDA_CHECK(e);
            if (opt.use_cuda_graph) capture(pl);
        }
        Plan* raw = up.get();
        raw->last_use = ++use_clock;
        plans[key] = std::move(up);
        evict_plans(raw);
        return raw;
    }

    // Profiling: every plain persistent GEMM of the plan writes its per-CTA stamps (gemm_persistent.cuh: entry / exit %globaltimer, SM id,
    // clock64 at setup done, first k-block landed, last MMA committed, epilogue done) into a plan-owned buffer; a replay overwrites the
    // previous one, so after a run the buffer holds the LAST forward of this plan (scripts/step_timeline.py reads two slots' worth).
    static constexpr int kTimelineCtas = 304;
    void attach_timeline(Plan& pl) {
        size_t n = 0;
        for (const Op& op : pl.ops) if (op.kind == Op::GEMM && !op.pair && !op.ln && !op.chain_sync) ++n;
        if (n == 0) return;
        pl.timeline = pl.mem.alloc_n<long long>(n * kTimelineCtas * 16);
        CUDA_CHECK(cudaMemset(pl.timeline, 0, n * kTimelineCtas * 16 * sizeof(long long)));
        size_t i = 0;
        for (Op& op : pl.ops) if (op.kind == Op::GEMM && !op.pair && !op.ln && !op.chain_sync) op.ep.timing = pl.timeline + (i++) * kTimelineCtas * 16;
    }

    // Plan cache bound (a MicroBatchWorker produces many (batch, length, regions) combinations): beyond max_plans the least
    // recently used plan -- its workspace (about 1 MB per pair) and CUDA graph -- is destroyed.  Rare, so the device is drained
    // first: a plan may still be executing on some stream.
    void evict_plans(const Plan* keep) {
        while (plans.size() > max_plans) {
            auto victim = plans.end();
            for (auto it = plans.begin(); it != plans.end(); ++it)
                if (it->second.get() != keep && (victim == plans.end() || it->second->last_use < victim->second->last_use)) victim = it;
            if (victim == plans.end()) break;
            cudaDeviceSynchronize();
            plans.erase(victim);
        }
    }

    // ---- poolers + heads (main stream, after joining the image branch)
    void build_heads(Plan& pl, uint32_t select) {
        const Config& c = cfg;
        const int B = pl.B, T = pl.T, V = pl.V, tc = pl.t_cur, vc = pl.v_cur;
        const int Mt = B * T, Mv = B * V, H = c.hidden, Hv = c.v_hidden, Hb = c.bi_hidden;
        const size_t S = x3 ? 3 : 1;
        auto& ops = pl.ops;
        float* pooled_t = pl.mem.alloc_n<float>(static_cast<size_t>(B) * Hb);
        float* pooled = pl.mem.alloc_n<float>(static_cast<size_t>(B) * Hb);
        bf16* pooled_b = pl.mem.alloc_n<bf16>(static_cast<size_t>(B) * Hb * S);
        {
            add_linear(pl, pl.t_b16[tc], B, static_cast<int64_t>(T) * H, t_pool, vb::kActRelu, nullptr, 0, nullptr, nullptr, 0, pooled_t, Hb, 0, Op::JOIN);
            add_linear(pl, pl.v_b16[vc], B, static_cast<int64_t>(V) * Hv, v_pool, vb::kActRelu, nullptr, 0, nullptr, pooled_b, Hb, pooled, Hb, 0, Op::NONE, pooled_t, Hb);
        }
        pl.outs[11] = OutBuf{pooled, B, Hb, Hb};
        auto cls_head = [&](const ClsW& w, int n_out, int slot) {
            bf16* hid = pl.mem.alloc_n<bf16>(static_cast<size_t>(B) * 2 * Hb * S);
            add_linear(pl, pooled_b, B, Hb, w.fc0, vb::kActGelu, nullptr, 0, &w.ln, hid, 2 * Hb, nullptr, 0);
            pl.outs[slot] = make_out(pl, B, n_out);
            add_linear(pl, hid, B, 2 * Hb, w.fc3, vb::kActNone, nullptr, 0, nullptr, nullptr, 0, pl.outs[slot].p, pl.outs[slot].ld);
        };
        if (select & VB200_OUT_VIL_PREDICTION) cls_head(vqa, num_labels, 0);
        if (select & VB200_OUT_VIL_PREDICTION_GQA) cls_head(gqa, gqa_labels, 1);
        if (select & VB200_OUT_VIL_LOGIT) {
            pl.outs[2] = make_out(pl, B, 1);
            ops.push_back(rowdot_op(pooled, Hb, vil_logit, nullptr, pl.outs[2].p, pl.outs[2].ld, B));
        }
        if (select & VB200_OUT_VIL_BINARY_PREDICTION) {
            if (B % 2 == 0) {
                // pooled.view(-1, 2*bi_hidden): adjacent samples form one NLVR2 pair (worker.py:266-276)
                float* hid_f = pl.mem.alloc_n<float>(static_cast<size_t>(B / 2) * 2 * Hb);
                add_linear(pl, pooled_b, B / 2, 2 * Hb, binary.fc0, vb::kActGelu, nullptr, 0, &binary.ln, nullptr, 0, hid_f, 2 * Hb);
                pl.outs[3] = make_out(pl, B / 2, 2);
                ops.push_back(rowdot_op(hid_f, 2 * Hb, binary.fc3_row, nullptr, pl.outs[3].p, pl.outs[3].ld, B / 2));
            } else {
                // [UPSTREAM] odd batch: element 3 stays the pre-training bi_seq_relationship score
                pl.outs[3] = make_out(pl, B, 2);
                ops.push_back(rowdot_op(pooled, Hb, seq_rel, nullptr, pl.outs[3].p, pl.outs[3].ld, B));
            }
        }
        if (select & VB200_OUT_VIL_TRI_PREDICTION) {
            pl.outs[4] = make_out(pl, B, 3);
            ops.push_back(rowdot_op(pooled, Hb, vil_tri, nullptr, pl.outs[4].p, pl.outs[4].ld, B));
        }
        if (select & VB200_OUT_VISION_PREDICTION) {
            bf16* hid = pl.mem.alloc_n<bf16>(static_cast<size_t>(Mv) * Hv * S);
            add_linear(pl, pl.v_b16[vc], Mv, Hv, img_transform, vb::kActGelu, nullptr, 0, &img_ln, hid, Hv, nullptr, 0);
            pl.outs[5] = make_out(pl, Mv, c.v_target);
            add_linear(pl, hid, Mv, Hv, img_decoder, vb::kActNone, nullptr, 0, nullptr, nullptr, 0, pl.outs[5].p, pl.outs[5].ld);
        }
        if (select & VB200_OUT_VISION_LOGIT) {
            pl.outs[6] = make_out(pl, Mv, 1);
            ops.push_back(rowdot_op(pl.v_f32[vc], Hv, vision_logit, pl.mask_v, pl.outs[6].p, pl.outs[6].ld, Mv));
        }
        if (select & VB200_OUT_LINGUISIC_PREDICTION) {
            bf16* hid = pl.mem.alloc_n<bf16>(static_cast<size_t>(Mt) * H * S);
            add_linear(pl, pl.t_b16[tc], Mt, H, lm_transform, vb::kActGelu, nullptr, 0, &lm_ln, hid, H, nullptr, 0);
            pl.outs[7] = make_out(pl, Mt, c.vocab);
            add_linear(pl, hid, Mt, H, lm_decoder, vb::kActNone, nullptr, 0, nullptr, nullptr, 0, pl.outs[7].p, pl.outs[7].ld);
        }
        if (select & VB200_OUT_LINGUISIC_LOGIT) {
            pl.outs[8] = make_out(pl, Mt, 1);
            ops.push_back(rowdot_op(pl.t_f32[tc], H, ling_logit, nullptr, pl.outs[8].p, pl.outs[8].ld, Mt));
        }
    }

    // ---------------------------------------------------------------- execution
    void launch_op(const Op& op, cudaStream_t st) {
        switch (op.kind) {
            case Op::GEMM:
                if (op.chain_sync != nullptr) {
                    const cudaError_t le = vb::launch_gemm_chain(op.ta, op.tb, op.ep, op.ta2, op.tb2, op.ep2, op.chain_sync, st);
                    if (le != cudaSuccess)
                        fail(VB200_ERR_CUDA, "chained GEMM launch failed: %s (layer %s, M=%d N1=%d K1=%d N2=%d)", cudaGetErrorString(le),
                             op.tag ? op.tag : "?", op.ep.M, op.ep.N, op.ep.K, op.ep2.N);
                } else if (op.pair) CUDA_CHECK(vb::launch_gemm_pair(op.ta, op.tb, op.ep, op.block_n, st));
                else {
                    GemmEpilogue e = op.ep;
                    e.tmap_c_host = e.tma_store ? &op.tc : nullptr;       // Op objects move when the list grows: bind here
                    e.grid_pct = profile_grid_pct;                        // 0 outside vb200_profile_ops
                    const cudaError_t le = vb::launch_gemm_persistent(op.ta, op.tb, e, op.block_n, op.ln, st);
                    if (le != cudaSuccess)
                        fail(VB200_ERR_CUDA, "GEMM launch failed: %s (layer %s, M=%d N=%d K=%d act=%d block_n=%d cluster_ln=%d ln_mode=%d split16=%d tma_store=%d)",
                             cudaGetErrorString(le), op.tag ? op.tag : "?", e.M, e.N, e.K, e.act, op.block_n, (int)op.ln, e.ln_mode, e.split16, e.tma_store);
                }
                break;
            case Op::SELF_ATTN:
                CUDA_CHECK(vb::launch_self_attention(op.qkv_a, op.ld_a, op.hidden, op.mask_a, op.ctx_a, op.ld_ctx_a, op.B, op.La,
                                                     op.Lb > 0 ? op.Lb : op.La, op.heads, op.head_dim, light_pdl(), opt.act_fp16, st));
                break;
            case Op::CO_ATTN:
                CUDA_CHECK(vb::launch_co_attention(op.qkv_a, op.ld_a, op.qkv_b, op.ld_b, op.hidden, op.mask_a, op.mask_b, op.ctx_a,
                                                   op.ld_ctx_a, op.ctx_b, op.ld_ctx_b, op.B, op.La, op.Lb, op.heads, op.head_dim,
                                                   light_pdl(), opt.act_fp16, st));
                break;
            case Op::LAYERNORM:
                CUDA_CHECK(vb::launch_ln_residual(op.ln_y, op.ln_ld, op.ln_res, op.ld_x, op.ln_g, op.ln_b, cfg.ln_eps, op.ln_out_f,
                                                  op.ld_out, op.ln_out_h, op.ld_a, op.ln_M, op.ln_N, opt.act_fp16, x3 ? 1 : 0,
                                                  light_pdl(), st, op.ln_pend.stats ? &op.ln_pend : nullptr));
                break;
            case Op::ATTN_F32:
                CUDA_CHECK(vb::launch_attention_f32(op.f_q, op.f_ld_q, op.f_k, op.f_v, op.f_ld_kv, op.f_in, op.f_mask, op.B, op.f_Lq,
                                                    op.f_Lk, op.heads, op.head_dim, op.f_ctx, op.f_ld_ctx, op.f_ctx_mode, op.f_probs,
                                                    light_pdl(), st));
                break;
            case Op::ROWDOT:
                CUDA_CHECK(vb::launch_rowdot(op.x, op.ld_x, op.W, op.bias, op.add, op.out, op.ld_out, op.M, op.K, op.n_out, opt.use_pdl, st));
                break;
        }
    }
    // Text-stream ops go to `st`, image-stream ops to the side stream so the two ViLBERT streams overlap
    // (T_k || V_k between co-attentions, and the two halves of a connection layer).  Dependencies across the
    // two are explicit: a side op marked FORK (and the first side op) waits for everything enqueued on `st`
    // so far; a main op marked JOIN waits for the side stream.  Under capture these become graph edges.
    void run_ops(Plan& pl, cudaStream_t st) {
        bool side_started = false, side_dirty = false;
        const char* open_tag = nullptr;
        struct RangeGuard { const char*& t; ~RangeGuard() { if (t) nvtxRangePop(); } } guard{open_tag};
        for (const Op& op : pl.ops) {
            if (op.tag != open_tag) {              // one NVTX range per layer of the schedule (enqueue side)
                if (open_tag) nvtxRangePop();
                open_tag = op.tag;
                if (open_tag) nvtxRangePushA(open_tag);
            }
            if (op.stream == 1) {
                if (!side_started || op.sync == Op::FORK) {
                    CUDA_CHECK(cudaEventRecord(ev_fork, st));
                    CUDA_CHECK(cudaStreamWaitEvent(side_stream, ev_fork, 0));
                    side_started = true;
                }
                launch_op(op, side_stream);
                side_dirty = true;
            } else {
                if (op.sync == Op::JOIN && side_dirty) {
                    CUDA_CHECK(cudaEventRecord(ev_join, side_stream));
                    CUDA_CHECK(cudaStreamWaitEvent(st, ev_join, 0));
                    side_dirty = false;
                }
                launch_op(op, st);
            }
        }
        if (side_dirty) {
            CUDA_CHECK(cudaEventRecord(ev_join, side_stream));
            CUDA_CHECK(cudaStreamWaitEvent(st, ev_join, 0));
        }
    }
    // Per-op device time: each launch-list entry is captured `kRep` times into its own CUDA graph and the graph replayed
    // between two CUDA events on the launching stream, so the number is the kernel's duration (incl. the grid launch
    // latency every launch pays inside the captured forward as well) without host launch gaps.  Every op is idempotent on
    // the plan's workspace, which must hold a previous forward's data.  Used by bench.py for the per-kernel roofline.
    void profile_ops(Plan& pl, int iters, std::vector<double>& ms_out) {
        constexpr int kRep = 8;
        cudaStream_t st;
        CUDA_CHECK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        cudaEvent_t e0, e1;
        CUDA_CHECK(cudaEventCreate(&e0));
        CUDA_CHECK(cudaEventCreate(&e1));
        const size_t n = pl.ops.size();
        ms_out.assign(n, 0.0);
        cudaGraph_t g = nullptr;
        cudaGraphExec_t ge = nullptr;
        try {
            for (size_t i = 0; i < n; ++i) {
                CUDA_CHECK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
                for (int r = 0; r < kRep; ++r) launch_op(pl.ops[i], st);
                CUDA_CHECK(cudaStreamEndCapture(st, &g));
                CUDA_CHECK(cudaGraphInstantiate(&ge, g, 0));
                CUDA_CHECK(cudaGraphLaunch(ge, st));                    // warm-up
                CUDA_CHECK(cudaEventRecord(e0, st));
                for (int it = 0; it < iters; ++it) CUDA_CHECK(cudaGraphLaunch(ge, st));
                CUDA_CHECK(cudaEventRecord(e1, st));
                CUDA_CHECK(cudaStreamSynchronize(st));
                float ms = 0.0f;
                CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
                ms_out[i] = ms / (static_cast<double>(iters) * kRep);
                cudaGraphExecDestroy(ge); ge = nullptr;
                cudaGraphDestroy(g); g = nullptr;
            }
        } catch (...) {
            if (ge) cudaGraphExecDestroy(ge);
            if (g) cudaGraphDestroy(g);
            cudaEventDestroy(e0); cudaEventDestroy(e1); cudaStreamDestroy(st);
            throw;
        }
        cudaEventDestroy(e0); cudaEventDestroy(e1); cudaStreamDestroy(st);
    }
    // FFN-in -> FFN-out (and every other producer / consumer pair of plain 128-wide GEMMs that sit next to each other on one graph
    // branch, the first writing only the 16-bit operand the second reads) become ONE chained launch (gemm_chain.cu).
    void link_chains(Plan& pl) {
        if (!chain_ffn || x3) return;
        std::vector<Op> out;
        out.reserve(pl.ops.size());
        for (size_t i = 0; i < pl.ops.size(); ++i) {
            Op a = pl.ops[i];
            if (i + 1 < pl.ops.size() && a.kind == Op::GEMM && !a.chain_sync) {
                const Op& b = pl.ops[i + 1];
                auto plain = [](const Op& o) {
                    const GemmEpilogue& e = o.ep;
                    return o.kind == Op::GEMM && !o.pair && !o.ln && o.block_n == 128 && e.ln_mode == 0 && !e.split16 && e.res == nullptr &&
                           e.mul == nullptr && e.gamma == nullptr && (e.N & 31) == 0 && e.act != vb::kActGeluExact;
                };
                if (plain(a) && plain(b) && a.stream == b.stream && b.sync == Op::NONE && a.ep.M == b.ep.M && a.ep.M >= 256 &&
                    a.ep.out_bf16 != nullptr && a.ep.out_f32 == nullptr && (a.ep.ld_bf16 & 7) == 0 && b.a_ptr == a.ep.out_bf16 &&
                    b.ep.K == a.ep.N && (b.ep.out_bf16 == nullptr || (b.ep.ld_bf16 & 7) == 0) && (b.ep.out_f32 == nullptr || (b.ep.ld_f32 & 3) == 0)) {
                    a.ta2 = b.ta; a.tb2 = b.tb; a.ep2 = b.ep; a.flops2 = b.flops;
                    const int m_tiles = (a.ep.M + 127) / 128;
                    a.chain_sync = pl.mem.alloc_n<int>(m_tiles + 2);
                    CUDA_CHECK(cudaMemset(a.chain_sync, 0, sizeof(int) * (m_tiles + 2)));
                    a.ep.tma_store = 0; a.ep2.tma_store = 0;
                    out.push_back(a);
                    ++i;                       // b is issued by the same launch
                    continue;
                }
            }
            out.push_back(a);
        }
        pl.ops.swap(out);
    }

    // PDL "medium" (default): additionally launch a GEMM programmatically when the kernel before it on its graph branch is a light one
    // (LayerNorm / attention trigger their dependents right after loading their inputs, so the GEMM's prologue -- barrier init,
    // TMEM allocation, descriptor prefetch -- overlaps the light kernel's math instead of following it).
    void link_pdl(Plan& pl) {
        if (!pdl_medium) return;
        int prev_kind[2] = {-1, -1};
        for (Op& op : pl.ops) {
            const int st = op.stream & 1;
            if (op.kind == Op::GEMM && op.ep.pdl == 2 &&
                (prev_kind[st] == Op::LAYERNORM || prev_kind[st] == Op::SELF_ATTN || prev_kind[st] == Op::CO_ATTN ||
                 prev_kind[st] == Op::ATTN_F32 ||
                 (pdl_gemm_gemm && prev_kind[st] == Op::GEMM)))
                op.ep.pdl = early_w ? 5 : 1;
            prev_kind[st] = op.kind;
            if (op.sync != Op::NONE) prev_kind[0] = prev_kind[1] = -1;      // fork / join: the predecessor set is not one kernel
        }
    }

    void capture(Plan& pl) {
        cudaStream_t cs;
        CUDA_CHECK(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
        cudaError_t e = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
        if (e != cudaSuccess) { cudaStreamDestroy(cs); CUDA_CHECK(e); }
        try {
            run_ops(pl, cs);
        } catch (...) {
            cudaGraph_t g = nullptr;
            cudaStreamEndCapture(cs, &g);
            if (g) cudaGraphDestroy(g);
            cudaStreamDestroy(cs);
            throw;
        }
        e = cudaStreamEndCapture(cs, &pl.graph);
        cudaStreamDestroy(cs);
        CUDA_CHECK(e);
        CUDA_CHECK(cudaGraphInstantiate(&pl.exec, pl.graph, 0));
    }

    void forward_device(Plan& pl, const vb200_inputs& in, cudaStream_t st) {
        const Config& c = cfg;
        if (!in.question || !in.features || !in.spatials || !in.segment_ids || !in.input_mask || !in.image_mask ||
            (c.task_tokens && !in.task_tokens))
            fail(VB200_ERR_INVALID, "vb200_inputs has a NULL required pointer");
        CUDA_CHECK(vb::launch_text_embed(in.question, in.segment_ids, in.input_mask, in.task_tokens, word, pos, type, task,
                                         emb_ln.g, emb_ln.b, c.ln_eps, pl.t_f32[0], pl.t_b16[0], pl.mask_t, pl.B, pl.Tin,
                                         c.hidden, c.vocab, c.max_pos, c.type_vocab, c.n_task, c.task_tokens, opt.act_fp16, x3 ? 1 : 0, st));
        CUDA_CHECK(vb::launch_image_pack(in.features, in.spatials, in.image_mask, pl.img_a, pl.mask_v, pl.B * pl.V, c.v_feat, pl.kp,
                                         opt.act_fp16, x3 ? 1 : 0, st));
        run_plan(pl, st);
    }
    void run_plan(Plan& pl, cudaStream_t st) {
        if (pl.ops.empty()) return;
        struct R { R(const Plan& p) { char b[96]; snprintf(b, sizeof(b), "vb200 forward B=%d T=%d V=%d", p.B, p.T, p.V); nvtxRangePushA(b); }
                   ~R() { nvtxRangePop(); } } range(pl);
        if (pl.exec) CUDA_CHECK(cudaGraphLaunch(pl.exec, st));
        else run_ops(pl, st);
    }
    // worker.py:422-455 on the device: detector output -> operand rows / masks, then the same plan as forward_device
    void forward_regions(Plan& pl, const vb200_region_inputs& in, cudaStream_t st) {
        const Config& c = cfg;
        if (!in.question || !in.segment_ids || !in.input_mask || (c.task_tokens && !in.task_tokens) || !in.box_features || !in.boxes ||
            !in.image_wh)
            fail(VB200_ERR_INVALID, "vb200_region_inputs has a NULL required pointer");
        CUDA_CHECK(vb::launch_text_embed(in.question, in.segment_ids, in.input_mask, in.task_tokens, word, pos, type, task,
                                         emb_ln.g, emb_ln.b, c.ln_eps, pl.t_f32[0], pl.t_b16[0], pl.mask_t, pl.B, pl.Tin,
                                         c.hidden, c.vocab, c.max_pos, c.type_vocab, c.n_task, c.task_tokens, opt.act_fp16, x3 ? 1 : 0, st));
        CUDA_CHECK(vb::launch_region_pack(in.box_features, in.boxes, in.image_wh, in.num_boxes, pl.img_a, pl.mask_v, in.spatials_out,
                                          pl.B, pl.V - 1, c.v_feat, pl.kp, opt.act_fp16, x3 ? 1 : 0, st));
        run_plan(pl, st);
    }
    // ---- retrieval reuse (PlanMode): per-caption / per-image prefixes and the pair suffix
    void encode_text(int n, int Tin, const int64_t* q, const int64_t* seg, const int64_t* im, const int64_t* tk, float* st_f32,
                     void* st_16, float* st_mask, cudaStream_t st) {
        const Config& c = cfg;
        if (!q || !seg || !im || (c.task_tokens && !tk) || !st_f32 || !st_16 || !st_mask) fail(VB200_ERR_INVALID, "vb200_encode_text: NULL pointer");
        Plan& pl = *get_plan(n, Tin, 1, 0, 0, TEXT_PREFIX);
        CUDA_CHECK(vb::launch_text_embed(q, seg, im, tk, word, pos, type, task, emb_ln.g, emb_ln.b, c.ln_eps, pl.t_f32[0], pl.t_b16[0],
                                         pl.mask_t, pl.B, pl.Tin, c.hidden, c.vocab, c.max_pos, c.type_vocab, c.n_task, c.task_tokens,
                                         opt.act_fp16, x3 ? 1 : 0, st));
        run_plan(pl, st);
        const size_t rows = static_cast<size_t>(pl.B) * pl.T, S = x3 ? 3 : 1;
        CUDA_CHECK(cudaMemcpyAsync(st_f32, pl.t_f32[pl.t_cur], rows * c.hidden * 4, cudaMemcpyDeviceToDevice, st));
        CUDA_CHECK(cudaMemcpyAsync(st_16, pl.t_b16[pl.t_cur], rows * c.hidden * S * 2, cudaMemcpyDeviceToDevice, st));
        CUDA_CHECK(cudaMemcpyAsync(st_mask, pl.mask_t, rows * 4, cudaMemcpyDeviceToDevice, st));
    }
    void encode_image(int n, int V, const float* feats, const float* loc, const uint8_t* vmask, float* st_f32, void* st_16,
                      float* st_mask, cudaStream_t st) {
        const Config& c = cfg;
        if (!feats || !loc || !vmask || !st_f32 || !st_16 || !st_mask) fail(VB200_ERR_INVALID, "vb200_encode_image: NULL pointer");
        Plan& pl = *get_plan(n, 1, V, 0, 0, IMAGE_PREFIX);
        CUDA_CHECK(vb::launch_image_pack(feats, loc, vmask, pl.img_a, pl.mask_v, pl.B * pl.V, c.v_feat, pl.kp, opt.act_fp16, x3 ? 1 : 0, st));
        run_plan(pl, st);
        const size_t rows = static_cast<size_t>(pl.B) * pl.V, S = x3 ? 3 : 1;
        CUDA_CHECK(cudaMemcpyAsync(st_f32, pl.v_f32[pl.v_cur], rows * c.v_hidden * 4, cudaMemcpyDeviceToDevice, st));
        CUDA_CHECK(cudaMemcpyAsync(st_16, pl.v_b16[pl.v_cur], rows * c.v_hidden * S * 2, cudaMemcpyDeviceToDevice, st));
        CUDA_CHECK(cudaMemcpyAsync(st_mask, pl.mask_v, rows * 4, cudaMemcpyDeviceToDevice, st));
    }
    void forward_cached(Plan& pl, const int32_t* t_idx, int n_text, const float* t_f32, const void* t_16, const float* t_mask,
                        const int32_t* v_idx, int n_img, const float* v_f32, const void* v_16, const float* v_mask, cudaStream_t st) {
        const Config& c = cfg;
        if (!t_idx || !t_f32 || !t_16 || !t_mask || !v_idx || !v_f32 || !v_16 || !v_mask) fail(VB200_ERR_INVALID, "vb200_forward_cached: NULL pointer");
        const int S = x3 ? 3 : 1;
        CUDA_CHECK(vb::launch_gather_state(t_idx, n_text, t_f32, t_16, t_mask, pl.t_f32[0], pl.t_b16[0], pl.mask_t, pl.B, pl.T,
                                           c.hidden, c.hidden * S, st));
        CUDA_CHECK(vb::launch_gather_state(v_idx, n_img, v_f32, v_16, v_mask, pl.v_f32[0], pl.v_b16[0], pl.mask_v, pl.B, pl.V,
                                           c.v_hidden, c.v_hidden * S, st));
        run_plan(pl, st);
    }
    static int seq_out(const vb200_outputs& o) {       // get_plan's seq_out bits for the sequence outputs the caller reads
        return (o.sequence_output_t != nullptr ? 1 : 0) | (o.sequence_output_v != nullptr ? 2 : 0);
    }
    static float* out_ptr(const vb200_outputs& o, int slot) {
        switch (slot) {
            case 0: return o.vil_prediction; case 1: return o.vil_prediction_gqa; case 2: return o.vil_logit;
            case 3: return o.vil_binary_prediction; case 4: return o.vil_tri_prediction; case 5: return o.vision_prediction;
            case 6: return o.vision_logit; case 7: return o.linguisic_prediction; case 8: return o.linguisic_logit;
            case 9: return o.sequence_output_t; case 10: return o.sequence_output_v; case 11: return o.pooled_output;
        }
        return nullptr;
    }
    void copy_outputs(Plan& pl, const vb200_outputs& out, cudaStream_t st, cudaMemcpyKind kind) {
        for (int s = 0; s < 12; ++s) {
            float* dst = out_ptr(out, s);
            const OutBuf& o = pl.outs[s];
            if (dst == nullptr) continue;
            if (o.p == nullptr) fail(VB200_ERR_INVALID, "output slot %d requested but not %s", s,
                                     s >= 9 && s <= 10 ? "available from this plan" : "selected in the `select` mask");
            CUDA_CHECK(cudaMemcpy2DAsync(dst, static_cast<size_t>(o.cols) * 4, o.p, static_cast<size_t>(o.ld) * 4,
                                         static_cast<size_t>(o.cols) * 4, o.rows, kind, st));
        }
        if (out.attention_probs != nullptr) {
            if (pl.attn.empty()) fail(VB200_ERR_INVALID, "attention_probs requested but VB200_OUT_ATTENTION is not set in `select`");
            float* dst = out.attention_probs;
            for (const Plan::AttnOut& a : pl.attn) {
                const size_t n = static_cast<size_t>(pl.B) * a.heads * a.Lq * a.Lk;
                CUDA_CHECK(cudaMemcpyAsync(dst, a.p, n * 4, kind, st));
                dst += n;
            }
        }
    }
};

namespace {
int guard(vb200_handle h, const std::function<void()>& body) {
    try {
        body();
        return VB200_OK;
    } catch (const VbError& e) {
        if (h) h->last_error = e.what(); else g_create_error = e.what();
        return e.status;
    } catch (const std::exception& e) {
        if (h) h->last_error = e.what(); else g_create_error = e.what();
        return VB200_ERR_INVALID;
    }
}

void require_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        fail(VB200_ERR_NO_DEVICE, "no CUDA device visible (%s); vilbert_b200 has no CPU fallback", e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= n) fail(VB200_ERR_INVALID, "device ordinal %d out of range (0..%d)", device, n - 1);
    cudaDeviceProp p;
    CUDA_CHECK(cudaGetDeviceProperties(&p, device));
    if (p.major != 10) fail(VB200_ERR_NO_DEVICE, "device %d is sm_%d%d; the kernels are built for sm_100a only", device, p.major, p.minor);
    CUDA_CHECK(cudaSetDevice(device));
}
}  // namespace

// =========================================================================================== C ABI
extern "C" {

int vb200_abi_version(void) { return VB200_ABI_VERSION; }

int vb200_create(const char* config_json, int64_t n_tensors, const vb200_tensor* tensors, const vb200_options* opt,
                 vb200_handle* out) {
    if (out == nullptr) { g_create_error = "vb200_create: out handle pointer is NULL"; return VB200_ERR_INVALID; }
    *out = nullptr;
    vb200_engine* eng = nullptr;
    int rc = guard(nullptr, [&] {
        if (tensors == nullptr || n_tensors <= 0) fail(VB200_ERR_CHECKPOINT, "empty state_dict");
        vb200_options o{};
        if (opt) o = *opt;
        // tri-state flags: 0 = default, 1 = on, -1 = off
        o.use_cuda_graph = o.use_cuda_graph >= 0 ? 1 : 0;
        o.strict = o.strict >= 0 ? 1 : 0;
        const int pdl_req = o.use_pdl;
        o.use_pdl = o.use_pdl > 0 ? 1 : 0;
        o.split_fp32 = o.split_fp32 > 0 ? 1 : 0;
        o.act_fp16 = (o.act_fp16 >= 0 || o.split_fp32) ? 1 : 0;
        o.fused_layernorm = (o.fused_layernorm > 0 && !o.split_fp32) ? 1 : 0;
        Config c = parse_config(config_json);
        {   // audit the state_dict (names, shapes, dtypes, strictness) before touching any device
            vb200_engine audit;
            audit.cfg = c; audit.opt = o; audit.dry = true; audit.x3 = o.split_fp32 != 0; audit.ln_fold = false;
            audit.ingest(n_tensors, tensors);
        }
        require_device(o.device);
        eng = new vb200_engine();
        eng->cfg = c;
        eng->opt = o;
        eng->x3 = o.split_fp32 != 0;
        eng->fused_ln = o.fused_layernorm != 0;
        if (const char* v = getenv("VB200_FUSED_LN")) eng->fused_ln = (strcmp(v, "1") == 0) && !eng->x3;
        if (const char* v = getenv("VB200_BN192")) eng->wide192 = (strcmp(v, "0") != 0);
        if (const char* v = getenv("VB200_TRI")) eng->tri_min_tiles = std::max(0, atoi(v));
        if (const char* v = getenv("VB200_LONE_ROWS")) eng->lone_rows = std::max(0, atoi(v));
        if (const char* v = getenv("VB200_CHAIN")) eng->chain_ffn = (strcmp(v, "0") != 0);
        if (const char* v = getenv("VB200_PRUNE")) eng->prune_tail = (strcmp(v, "0") != 0);
        eng->ln_fold = o.ln_fold > 0;
        if (const char* v = getenv("VB200_LNFOLD")) eng->ln_fold = (strcmp(v, "0") != 0);
        if (eng->x3 || eng->fused_ln) eng->ln_fold = false;      // those modes keep every LayerNorm as its own step
        eng->max_plans = o.max_plans > 0 ? static_cast<size_t>(o.max_plans) : 24;
        if (const char* v = getenv("VB200_MAX_PLANS")) { const int n = atoi(v); if (n > 0) eng->max_plans = static_cast<size_t>(n); }
        eng->pdl_light = eng->pdl_medium = false;
        if (pdl_req == 0) eng->opt.use_pdl = 1;               // default: full
        if (const char* v = getenv("VB200_PDL")) {
            eng->pdl_gemm_gemm = strcmp(v, "mediumplus") == 0;
            eng->pdl_light = strcmp(v, "light") == 0 || strcmp(v, "medium") == 0 || eng->pdl_gemm_gemm;
            eng->pdl_medium = strcmp(v, "medium") == 0 || eng->pdl_gemm_gemm;
            if (strcmp(v, "full") == 0) eng->opt.use_pdl = 1;
            if (strcmp(v, "off") == 0) eng->opt.use_pdl = 0;
        }
        if (const char* v = getenv("VB200_TMASTORE")) eng->tma_store_enabled = (strcmp(v, "0") != 0);
        if (const char* v = getenv("VB200_EARLYW")) eng->early_w = (strcmp(v, "0") != 0);
        if (const char* v = getenv("VB200_PAIR_MIN_WAVES")) eng->pair_min_waves = std::max(0, atoi(v));
        if (const char* v = getenv("VB200_PAIR")) { const int b = atoi(v); eng->pair_bn = (b == 128 || b == 256) ? b : (strcmp(v, "auto") == 0 ? -1 : 0); }
        CUDA_CHECK(cudaStreamCreateWithFlags(&eng->side_stream, cudaStreamNonBlocking));
        CUDA_CHECK(cudaEventCreateWithFlags(&eng->ev_fork, cudaEventDisableTiming));
        CUDA_CHECK(cudaEventCreateWithFlags(&eng->ev_join, cudaEventDisableTiming));
        eng->ingest(n_tensors, tensors);
        CUDA_CHECK(cudaDeviceSynchronize());
    });
    if (rc != VB200_OK) { delete eng; return rc; }
    *out = eng;
    return VB200_OK;
}

int vb200_destroy(vb200_handle h) {
    if (h == nullptr) return VB200_OK;
    cudaSetDevice(h->opt.device);
    cudaDeviceSynchronize();
    delete h;
    return VB200_OK;
}

const char* vb200_last_error(vb200_handle h) { return h ? h->last_error.c_str() : g_create_error.c_str(); }

int vb200_forward(vb200_handle h, const vb200_inputs* in, const vb200_outputs* out, uint32_t select, void* cuda_stream) {
    return vb200_forward_slot(h, in, out, select, 0, cuda_stream);
}

int vb200_forward_slot(vb200_handle h, const vb200_inputs* in, const vb200_outputs* out, uint32_t select, int32_t slot,
                       void* cuda_stream) {
    if (h == nullptr) return VB200_ERR_INVALID;
    return guard(h, [&] {
        if (in == nullptr || out == nullptr) fail(VB200_ERR_INVALID, "inputs/outputs struct is NULL");
        CUDA_CHECK(cudaSetDevice(h->opt.device));
        Plan* pl = h->get_plan(in->batch, in->n_tokens, in->n_regions, select & VB200_OUT_ALL, slot, vb200_engine::FULL,
                               (select & VB200_OUT_ATTENTION) != 0, vb200_engine::seq_out(*out));
        cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
        h->forward_device(*pl, *in, st);
        h->copy_outputs(*pl, *out, st, cudaMemcpyDeviceToDevice);
    });
}

int vb200_forward_regions(vb200_handle h, const vb200_region_inputs* in, const vb200_outputs* out, uint32_t select, int32_t slot,
                          void* cuda_stream) {
    if (h == nullptr) return VB200_ERR_INVALID;
    return guard(h, [&] {
        if (in == nullptr || out == nullptr) fail(VB200_ERR_INVALID, "inputs/outputs struct is NULL");
        if (in->n_boxes < 1) fail(VB200_ERR_INVALID, "n_boxes must be positive");
        CUDA_CHECK(cudaSetDevice(h->opt.device));
        Plan* pl = h->get_plan(in->batch, in->n_tokens, in->n_boxes + 1, select & VB200_OUT_ALL, slot, vb200_engine::FULL,
                               (select & VB200_OUT_ATTENTION) != 0, vb200_engine::seq_out(*out));
        cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
        h->forward_regions(*pl, *in, st);
        h->copy_outputs(*pl, *out, st, cudaMemcpyDeviceToDevice);
    });
}

int vb200_encode_text(vb200_handle h, int32_t n, int32_t n_tokens, const int64_t* question, const int64_t* segment_ids,
                      const int64_t* input_mask, const int64_t* task_tokens, float* state_f32, void* state_16, float* state_mask,
                      void* cuda_stream) {
    if (h == nullptr) return VB200_ERR_INVALID;
    return guard(h, [&] {
        CUDA_CHECK(cudaSetDevice(h->opt.device));
        h->encode_text(n, n_tokens, question, segment_ids, input_mask, task_tokens, state_f32, state_16, state_mask,
                       static_cast<cudaStream_t>(cuda_stream));
    });
}

int vb200_encode_image(vb200_handle h, int32_t n, int32_t n_regions, const float* features, const float* spatials,
                       const uint8_t* image_mask, float* state_f32, void* state_16, float* state_mask, void* cuda_stream) {
    if (h == nullptr) return VB200_ERR_INVALID;
    return guard(h, [&] {
        CUDA_CHECK(cudaSetDevice(h->opt.device));
        h->encode_image(n, n_regions, features, spatials, image_mask, state_f32, state_16, state_mask,
                        static_cast<cudaStream_t>(cuda_stream));
    });
}

int vb200_forward_cached(vb200_handle h, int32_t batch, int32_t n_tokens, int32_t n_regions, const int32_t* text_index,
                         int32_t n_text, const float* text_f32, const void* text_16, const float* text_mask,
                         const int32_t* image_index, int32_t n_image, const float* image_f32, const void* image_16,
                         const float* image_mask, const vb200_outputs* out, uint32_t select, int32_t slot, void* cuda_stream) {
    if (h == nullptr) return VB200_ERR_INVALID;
    return guard(h, [&] {
        if (out == nullptr) fail(VB200_ERR_INVALID, "outputs struct is NULL");
        if (n_text < 1 || n_image < 1) fail(VB200_ERR_INVALID, "cached state counts must be positive");
        CUDA_CHECK(cudaSetDevice(h->opt.device));
        Plan* pl = h->get_plan(batch, n_tokens, n_regions, select & VB200_OUT_ALL, slot, vb200_engine::SUFFIX,
                               (select & VB200_OUT_ATTENTION) != 0, vb200_engine::seq_out(*out));
        cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
        h->forward_cached(*pl, text_index, n_text, text_f32, text_16, text_mask, image_index, n_image, image_f32, image_16,
                          image_mask, st);
        h->copy_outputs(*pl, *out, st, cudaMemcpyDeviceToDevice);
    });
}

int vb200_attention_layout(vb200_handle h, int32_t batch, int32_t n_tokens, int32_t n_regions, int32_t max_entries,
                           int32_t* n_entries, int32_t* dims, int64_t* offsets, int64_t* total_floats) {
    if (h == nullptr || n_entries == nullptr) return VB200_ERR_INVALID;
    return guard(h, [&] {
        // derived from the layer schedule alone (no plan is built): the order add_attn_f32 is called in by get_plan
        const Config& c = h->cfg;
        const int T = n_tokens + (c.task_tokens ? 1 : 0), V = n_regions;
        int n = 0;
        int64_t off = 0;
        auto put = [&](int heads, int lq, int lk, int kind) {
            if (n < max_entries) {
                if (dims) { dims[4 * n] = heads; dims[4 * n + 1] = lq; dims[4 * n + 2] = lk; dims[4 * n + 3] = kind; }
                if (offsets) offsets[n] = off;
            }
            off += static_cast<int64_t>(batch) * heads * lq * lk;
            ++n;
        };
        for (const std::string& step : h->schedule) {
            if (step[0] == 'T') put(c.heads, T, T, 0);
            else if (step[0] == 'V') put(c.v_heads, V, V, 1);
            else { put(c.bi_heads, T, V, 2); put(c.bi_heads, V, T, 3); }
        }
        *n_entries = n;
        if (total_floats) *total_floats = off;
    });
}

int vb200_forward_host(vb200_handle h, const vb200_inputs* in, const vb200_outputs* out, uint32_t select, void* cuda_stream) {
    return vb200_forward_host_slot(h, in, out, select, 0, 1, cuda_stream);
}

int vb200_forward_host_slot(vb200_handle h, const vb200_inputs* in, const vb200_outputs* out, uint32_t select, int32_t slot,
                            int32_t synchronize, void* cuda_stream) {
    if (h == nullptr) return VB200_ERR_INVALID;
    return guard(h, [&] {
        if (in == nullptr || out == nullptr) fail(VB200_ERR_INVALID, "inputs/outputs struct is NULL");
        CUDA_CHECK(cudaSetDevice(h->opt.device));
        Plan* pl = h->get_plan(in->batch, in->n_tokens, in->n_regions, select & VB200_OUT_ALL, slot, vb200_engine::FULL,
                               (select & VB200_OUT_ATTENTION) != 0, vb200_engine::seq_out(*out));
        cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
        const size_t B = pl->B, Tin = pl->Tin, V = pl->V, F = h->cfg.v_feat;
        if (pl->d_q == nullptr) {
            pl->d_q = pl->mem.alloc_n<int64_t>(B * Tin); pl->d_seg = pl->mem.alloc_n<int64_t>(B * Tin);
            pl->d_mask = pl->mem.alloc_n<int64_t>(B * Tin); pl->d_task = pl->mem.alloc_n<int64_t>(B);
            pl->d_feat = pl->mem.alloc_n<float>(B * V * F); pl->d_loc = pl->mem.alloc_n<float>(B * V * 5);
            pl->d_imask = pl->mem.alloc_n<uint8_t>(B * V);
        }
        if (!in->question || !in->features || !in->spatials || !in->segment_ids || !in->input_mask || !in->image_mask ||
            (h->cfg.task_tokens && !in->task_tokens))
            fail(VB200_ERR_INVALID, "vb200_inputs has a NULL required pointer");
        CUDA_CHECK(cudaMemcpyAsync(pl->d_q, in->question, B * Tin * 8, cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaMemcpyAsync(pl->d_seg, in->segment_ids, B * Tin * 8, cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaMemcpyAsync(pl->d_mask, in->input_mask, B * Tin * 8, cudaMemcpyHostToDevice, st));
        if (in->task_tokens) CUDA_CHECK(cudaMemcpyAsync(pl->d_task, in->task_tokens, B * 8, cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaMemcpyAsync(pl->d_feat, in->features, B * V * F * 4, cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaMemcpyAsync(pl->d_loc, in->spatials, B * V * 5 * 4, cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaMemcpyAsync(pl->d_imask, in->image_mask, B * V, cudaMemcpyHostToDevice, st));
        vb200_inputs dev = *in;
        dev.question = pl->d_q; dev.segment_ids = pl->d_seg; dev.input_mask = pl->d_mask; dev.task_tokens = pl->d_task;
        dev.features = pl->d_feat; dev.spatials = pl->d_loc; dev.image_mask = pl->d_imask; dev.co_attention_mask = nullptr;
        h->forward_device(*pl, dev, st);
        h->copy_outputs(*pl, *out, st, cudaMemcpyDeviceToHost);
        if (synchronize) CUDA_CHECK(cudaStreamSynchronize(st));
    });
}

int vb200_plan_info(vb200_handle h, int32_t batch, int32_t n_tokens, int32_t n_regions, uint32_t select,
                    int64_t* n_launches, double* flops) {
    if (h == nullptr) return VB200_ERR_INVALID;
    return guard(h, [&] {
        CUDA_CHECK(cudaSetDevice(h->opt.device));
        Plan* pl = h->get_plan(batch, n_tokens, n_regions, select & VB200_OUT_ALL);
        if (n_launches) *n_launches = static_cast<int64_t>(pl->ops.size()) + 2;   // + text-embed + image-pack
        if (flops) *flops = pl->flops;
    });
}

int vb200_profile_ops(vb200_handle h, int32_t batch, int32_t n_tokens, int32_t n_regions, uint32_t select, int32_t iters,
                      int32_t max_ops, int32_t* n_ops, int32_t* kinds, double* ms, double* flops, int32_t* dims) {
    if (h == nullptr || n_ops == nullptr) return VB200_ERR_INVALID;
    return guard(h, [&] {
        CUDA_CHECK(cudaSetDevice(h->opt.device));
        Plan* pl = h->get_plan(batch, n_tokens, n_regions, select & VB200_OUT_ALL);
        std::vector<double> t;
        struct Reset { vb200_engine* e; int keep; ~Reset() { e->profile_grid_pct = keep; } } reset{h, h->profile_grid_pct};
        h->profile_ops(*pl, iters < 1 ? 1 : iters, t);
        h->profile_grid_pct = 0;          // the override never leaks into forwards (plans are captured without it anyway)
        reset.keep = 0;
        const int n = static_cast<int>(pl->ops.size());
        *n_ops = n;
        for (int i = 0; i < n && i < max_ops; ++i) {
            const Op& op = pl->ops[i];
            if (kinds) kinds[i] = static_cast<int>(op.kind);
            if (ms) ms[i] = t[i];
            if (flops) flops[i] = op.flops + op.flops2;
            if (dims) {
                dims[4 * i + 0] = op.kind == Op::GEMM ? op.ep.M : (op.kind == Op::LAYERNORM ? op.ln_M : op.B);
                dims[4 * i + 1] = op.kind == Op::GEMM ? op.ep.N : (op.kind == Op::LAYERNORM ? op.ln_N : op.La);
                dims[4 * i + 2] = op.kind == Op::GEMM ? op.ep.K : op.Lb;
                dims[4 * i + 3] = op.kind == Op::GEMM ? (op.ep.act | (op.ln ? 16 : 0) | (op.ep.ln_mode == 4 ? 32 : 0) | (op.ep.ln_mode == 5 ? 64 : 0) |
                                                         (op.chain_sync ? 128 : 0))
                                                      : op.heads;
            }
        }
    });
}

int vb200_set_option(vb200_handle h, const char* key, int64_t value) {
    if (h == nullptr || key == nullptr) return VB200_ERR_INVALID;
    return guard(h, [&] {
        const std::string k = key;
        if (k == "profile_grid_pct") {
            if (value != 0 && (value < 10 || value > 100)) fail(VB200_ERR_INVALID, "profile_grid_pct must be 0 or 10..100");
            h->profile_grid_pct = static_cast<int>(value);
        } else if (k == "max_plans") {
            if (value < 1) fail(VB200_ERR_INVALID, "max_plans must be positive");
            h->max_plans = static_cast<size_t>(value);
        } else if (k == "timeline") {
            if ((value != 0) != h->timeline) {
                CUDA_CHECK(cudaDeviceSynchronize());
                h->plans.clear();
                h->timeline = value != 0;
            }
        } else if (k == "chain_ffn") {
            // changes how plans are built: drop the cached ones (the device is drained first, a plan may still be executing)
            if ((value != 0) != h->chain_ffn) {
                CUDA_CHECK(cudaDeviceSynchronize());
                h->plans.clear();
                h->chain_ffn = value != 0;
            }
        } else if (k == "prune_tail") {
            if ((value != 0) != h->prune_tail) {           // as chain_ffn: plans are built differently
                CUDA_CHECK(cudaDeviceSynchronize());
                h->plans.clear();
                h->prune_tail = value != 0;
            }
        } else fail(VB200_ERR_INVALID, "unknown option \"%s\"", key);
    });
}

int vb200_timeline(vb200_handle h, int32_t batch, int32_t n_tokens, int32_t n_regions, uint32_t select, int32_t slot, int32_t max_ops,
                   int32_t* n_ops, int32_t* dims, int64_t* stamps) {
    if (h == nullptr || n_ops == nullptr) return VB200_ERR_INVALID;
    return guard(h, [&] {
        CUDA_CHECK(cudaSetDevice(h->opt.device));
        if (!h->timeline) fail(VB200_ERR_INVALID, "vb200_timeline: set_option(\"timeline\", 1) first");
        Plan* pl = h->get_plan(batch, n_tokens, n_regions, select & VB200_OUT_ALL, slot);
        CUDA_CHECK(cudaDeviceSynchronize());
        int n = 0;
        for (const Op& op : pl->ops) {
            if (op.ep.timing == nullptr || op.kind != Op::GEMM) continue;
            if (n < max_ops) {
                if (dims) { dims[4 * n] = op.ep.M; dims[4 * n + 1] = op.ep.N; dims[4 * n + 2] = op.ep.K; dims[4 * n + 3] = op.stream; }
                if (stamps) CUDA_CHECK(cudaMemcpy(stamps + static_cast<size_t>(n) * vb200_engine::kTimelineCtas * 16, op.ep.timing,
                                                  sizeof(long long) * vb200_engine::kTimelineCtas * 16, cudaMemcpyDeviceToHost));
            }
            ++n;
        }
        *n_ops = n;
    });
}

int vb200_model_dim(vb200_handle h, const char* key, int64_t* value) {
    if (h == nullptr || key == nullptr || value == nullptr) return VB200_ERR_INVALID;
    return guard(h, [&] {
        const Config& c = h->cfg;
        const std::string k = key;
        if (k == "hidden_size") *value = c.hidden; else if (k == "v_hidden_size") *value = c.v_hidden;
        else if (k == "bi_hidden_size") *value = c.bi_hidden; else if (k == "vocab_size") *value = c.vocab;
        else if (k == "v_target_size") *value = c.v_target; else if (k == "v_feature_size") *value = c.v_feat;
        else if (k == "num_labels") *value = h->num_labels; else if (k == "gqa_labels") *value = h->gqa_labels;
        else if (k == "task_specific_tokens") *value = c.task_tokens;
        else if (k == "weight_bytes") *value = static_cast<int64_t>(h->weights.total);
        else if (k == "operand_width_factor") *value = h->x3 ? 3 : 1;
        else if (k == "ln_fold") *value = h->ln_fold ? 1 : 0;
        else if (k == "n_plans") *value = static_cast<int64_t>(h->plans.size());
        else if (k == "n_layers_scheduled") *value = static_cast<int64_t>(h->schedule.size());
        else fail(VB200_ERR_INVALID, "unknown model dimension \"%s\"", key);
    });
}

// ---------------------------------------------------------------- kernel-level entry points
static std::string g_op_error;
static int op_guard(const std::function<void()>& body) {
    try { body(); return VB200_OK; }
    catch (const VbError& e) { g_create_error = e.what(); return e.status; }
    catch (const std::exception& e) { g_create_error = e.what(); return VB200_ERR_INVALID; }
}

int vb200_linear(const void* x_bf16, int64_t ld_x, const void* w_bf16, int64_t ld_w, const float* bias,
                 const float* residual, int64_t ld_res, const float* gamma, const float* beta, float eps, int32_t act,
                 void* y_bf16, int64_t ld_y_bf16, float* y_f32, int64_t ld_y_f32, int64_t M, int64_t N, int64_t K,
                 int32_t block_n, int32_t use_pdl, int32_t act_fp16, int32_t variant, long long* timing, void* cuda_stream) {
    return op_guard([&] {
        const bool ln = gamma != nullptr;
        const bool pair = variant == 2;                                    // CTA-pair kernel: block_n 128 (default) or 256
        if (variant != 0 && variant != 2 && variant != 3 && variant != 4)
            fail(VB200_ERR_INVALID, "vb200_linear: variant %d does not exist (0 persistent, 2 CTA pair, 3 three CTAs per SM, 4 one CTA per SM with a 6-stage ring)", variant);
        int bn = block_n > 0 ? block_n : (pair ? 128 : vb::gemm_p_pick_block_n(static_cast<int>(N), ln));
        if (bn == 0) fail(VB200_ERR_INVALID, "no tiling for N=%lld with LayerNorm", (long long)N);
        CUtensorMap ta = make_tmap(x_bf16, M, K, ld_x, 128, act_fp16 != 0);
        CUtensorMap tb = make_tmap(w_bf16, N, K, ld_w, pair ? bn / 2 : bn, act_fp16 != 0);
        GemmEpilogue e{};
        e.M = (int)M; e.N = (int)N; e.K = (int)K; e.bias = bias; e.res = residual; e.ld_res = (int)ld_res;
        e.gamma = gamma; e.beta = beta; e.eps = eps; e.out_bf16 = static_cast<bf16*>(y_bf16); e.ld_bf16 = (int)ld_y_bf16;
        e.out_f32 = y_f32; e.ld_f32 = (int)ld_y_f32; e.act = act; e.pdl = use_pdl;
        e.a_f16 = act_fp16 ? 1 : 0; e.out_f16 = e.a_f16; e.timing = timing;
        if (const char* dbg = getenv("VB200_DEBUG")) e.debug = atoi(dbg);          // timing decomposition (kernels.h), op entry only
        CUtensorMap tc;
        const char* ts = getenv("VB200_TMASTORE");
        if (variant == 3 || variant == 4) {
            if (ln || (bn != 128 && !(variant == 4 && bn == 64))) fail(VB200_ERR_INVALID, "vb200_linear: variant 3 is the plain 128-wide tile, variant 4 the 128- or 64-wide one");
            if (variant == 3) e.tri = 1; else e.lone = 1;
        }
        if (variant != 2 && !ln && !(ts && strcmp(ts, "0") == 0)) { setup_tma_store(&tc, e); e.tmap_c_host = e.tma_store ? &tc : nullptr; }
        if (pair) CUDA_CHECK(vb::launch_gemm_pair(ta, tb, e, bn, static_cast<cudaStream_t>(cuda_stream)));
        else CUDA_CHECK(vb::launch_gemm_persistent(ta, tb, e, bn, ln, static_cast<cudaStream_t>(cuda_stream)));
    });
}

int vb200_layernorm(const float* y, int64_t ld_y, const float* residual, int64_t ld_res, const float* gamma, const float* beta,
                    float eps, float* out_f32, int64_t ld_f32, void* out_16, int64_t ld_16, int64_t M, int64_t N,
                    int32_t act_fp16, void* cuda_stream) {
    return op_guard([&] {
        CUDA_CHECK(vb::launch_ln_residual(y, (int)ld_y, residual, (int)ld_res, gamma, beta, eps, out_f32, (int)ld_f32,
                                          static_cast<bf16*>(out_16), (int)ld_16, (int)M, (int)N, act_fp16 ? 1 : 0, 0, 0,
                                          static_cast<cudaStream_t>(cuda_stream)));
    });
}

int vb200_layernorm_split(const float* y, int64_t ld_y, const float* residual, int64_t ld_res, const float* gamma, const float* beta,
                          float eps, float* out_f32, int64_t ld_f32, void* out_16, int64_t ld_16, int64_t M, int64_t N, void* cuda_stream) {
    return op_guard([&] {
        CUDA_CHECK(vb::launch_ln_residual(y, (int)ld_y, residual, (int)ld_res, gamma, beta, eps, out_f32, (int)ld_f32,
                                          static_cast<bf16*>(out_16), (int)ld_16, (int)M, (int)N, 1, 1, 0,
                                          static_cast<cudaStream_t>(cuda_stream)));
    });
}

int vb200_linear_split(const void* x16, int64_t ld_x, const void* w16, int64_t ld_w, const float* bias, int32_t act, void* y16,
                       int64_t ld_y16, float* y_f32, int64_t ld_y_f32, int64_t M, int64_t N, int64_t K3, void* cuda_stream) {
    return op_guard([&] {
        if (K3 % 192 != 0) fail(VB200_ERR_INVALID, "vb200_linear_split: K3 = %lld is not 3 x a multiple of 64", (long long)K3);
        const int bn = vb::gemm_p_pick_block_n(static_cast<int>(N), false);
        CUtensorMap ta = make_tmap(x16, M, K3, ld_x, 128, true);
        CUtensorMap tb = make_tmap(w16, N, K3, ld_w, bn, true);
        GemmEpilogue e{};
        e.M = (int)M; e.N = (int)N; e.K = (int)K3; e.bias = bias; e.eps = 0.0f; e.out_bf16 = static_cast<bf16*>(y16);
        e.ld_bf16 = (int)ld_y16; e.out_f32 = y_f32; e.ld_f32 = (int)ld_y_f32; e.act = act; e.a_f16 = 1; e.out_f16 = 1;
        e.split16 = y16 != nullptr ? 1 : 0;
        CUDA_CHECK(vb::launch_gemm_persistent(ta, tb, e, bn, false, static_cast<cudaStream_t>(cuda_stream)));
    });
}

int vb200_linear_ln(const void* x16, int64_t ld_x, const void* w16, int64_t ld_w, const float* bias, int32_t mode, const void* a_stats,
                    int32_t a_parts, const float* fold_s, const float* res, int64_t ld_res, const void* res_stats, int32_t res_parts,
                    const float* res_gamma, const float* res_beta, void* out_stats, int32_t stats_ld, float eps, int32_t act, void* y16,
                    int64_t ld_y16, float* y_f32, int64_t ld_y_f32, int64_t M, int64_t N, int64_t K, int32_t act_fp16, void* cuda_stream) {
    return op_guard([&] {
        if (mode != 4 && mode != 5) fail(VB200_ERR_INVALID, "vb200_linear_ln: mode must be 4 (fold-in) or 5 (pre-LayerNorm output)");
        CUtensorMap ta = make_tmap(x16, M, K, ld_x, 128, act_fp16 != 0);
        CUtensorMap tb = make_tmap(w16, N, K, ld_w, 128, act_fp16 != 0);
        GemmEpilogue e{};
        e.M = (int)M; e.N = (int)N; e.K = (int)K; e.bias = bias; e.eps = eps; e.act = act; e.a_f16 = act_fp16 ? 1 : 0; e.out_f16 = e.a_f16;
        e.out_bf16 = static_cast<bf16*>(y16); e.ld_bf16 = (int)ld_y16; e.out_f32 = y_f32; e.ld_f32 = (int)ld_y_f32;
        e.ln_mode = mode; e.stats_ld = stats_ld;
        e.a_stats = static_cast<const float2*>(a_stats); e.a_parts = a_parts; e.fold_s = fold_s;
        e.res = res; e.ld_res = (int)ld_res; e.res_stats = static_cast<const float2*>(res_stats); e.res_parts = res_parts;
        e.res_gamma = res_gamma; e.res_beta = res_beta; e.out_stats = static_cast<float2*>(out_stats);
        CUDA_CHECK(vb::launch_gemm_persistent(ta, tb, e, 128, false, static_cast<cudaStream_t>(cuda_stream)));
    });
}

int vb200_linear_chain(const void* x16, int64_t ld_x, const void* w1, int64_t ld_w1, const float* b1, int32_t act, void* h16, int64_t ld_h,
                       const void* w2, int64_t ld_w2, const float* b2, void* y16, int64_t ld_y16, float* y_f32, int64_t ld_y_f32, int64_t M,
                       int64_t N1, int64_t K1, int64_t N2, int32_t act_fp16, void* sync_ints, void* cuda_stream) {
    return op_guard([&] {
        CUtensorMap ta0 = make_tmap(x16, M, K1, ld_x, 128, act_fp16 != 0), tb0 = make_tmap(w1, N1, K1, ld_w1, 128, act_fp16 != 0);
        CUtensorMap ta1 = make_tmap(h16, M, N1, ld_h, 128, act_fp16 != 0), tb1 = make_tmap(w2, N2, N1, ld_w2, 128, act_fp16 != 0);
        GemmEpilogue e0{}, e1{};
        e0.M = e1.M = (int)M; e0.N = (int)N1; e0.K = (int)K1; e1.N = (int)N2; e1.K = (int)N1;
        e0.bias = b1; e1.bias = b2; e0.act = act; e0.a_f16 = e0.out_f16 = e1.a_f16 = e1.out_f16 = act_fp16 ? 1 : 0;
        e0.out_bf16 = static_cast<bf16*>(h16); e0.ld_bf16 = (int)ld_h;
        e1.out_bf16 = static_cast<bf16*>(y16); e1.ld_bf16 = (int)ld_y16; e1.out_f32 = y_f32; e1.ld_f32 = (int)ld_y_f32;
        CUDA_CHECK(vb::launch_gemm_chain(ta0, tb0, e0, ta1, tb1, e1, static_cast<int*>(sync_ints), static_cast<cudaStream_t>(cuda_stream)));
    });
}

int vb200_attention_f32(const void* q, int64_t ld_q, const void* k, const void* v, int64_t ld_kv, int32_t in_kind,
                        const float* key_mask_add, int32_t B, int32_t Lq, int32_t Lk, int32_t heads, int32_t head_dim, void* ctx,
                        int64_t ld_ctx, int32_t ctx_mode, float* probs, void* cuda_stream) {
    return op_guard([&] {
        CUDA_CHECK(vb::launch_attention_f32(q, (int)ld_q, k, v, (int)ld_kv, in_kind, key_mask_add, B, Lq, Lk, heads, head_dim,
                                            static_cast<bf16*>(ctx), (int)ld_ctx, ctx_mode, probs, 0,
                                            static_cast<cudaStream_t>(cuda_stream)));
    });
}

int vb200_self_attention(const void* qkv_bf16, int64_t ld_qkv, int32_t hidden, const float* mask_add, void* ctx_bf16,
                         int64_t ld_ctx, int32_t B, int32_t L, int32_t heads, int32_t head_dim, int32_t act_fp16,
                         void* cuda_stream) {
    return op_guard([&] {
        CUDA_CHECK(vb::launch_self_attention(static_cast<const bf16*>(qkv_bf16), (int)ld_qkv, hidden, mask_add,
                                             static_cast<bf16*>(ctx_bf16), (int)ld_ctx, B, L, L, heads, head_dim, 0,
                                             act_fp16 ? 1 : 0, static_cast<cudaStream_t>(cuda_stream)));
    });
}

int vb200_co_attention(const void* qkv_img_bf16, int64_t ld_img, const void* qkv_txt_bf16, int64_t ld_txt,
                       int32_t hidden, const float* img_mask_add, const float* txt_mask_add, void* ctx_txt_bf16,
                       int64_t ld_ctx_txt, void* ctx_img_bf16, int64_t ld_ctx_img, int32_t B, int32_t T, int32_t V,
                       int32_t heads, int32_t head_dim, int32_t act_fp16, void* cuda_stream) {
    return op_guard([&] {
        CUDA_CHECK(vb::launch_co_attention(static_cast<const bf16*>(qkv_img_bf16), (int)ld_img,
                                           static_cast<const bf16*>(qkv_txt_bf16), (int)ld_txt, hidden, img_mask_add,
                                           txt_mask_add, static_cast<bf16*>(ctx_txt_bf16), (int)ld_ctx_txt,
                                           static_cast<bf16*>(ctx_img_bf16), (int)ld_ctx_img, B, T, V, heads, head_dim, 0,
                                           act_fp16 ? 1 : 0, static_cast<cudaStream_t>(cuda_stream)));
    });
}

}  // extern "C"
