// K4 / K5: small-sequence attention for the two ViLBERT streams and the bidirectional co-attention.
//
// Replaces, per layer, the reference's 2 batched SGEMMs + scale + mask-add + softmax kernels of
// BertSelfAttention / BertImageSelfAttention, and the 4 bmm + 2 softmax of BertBiAttention
// ([UPSTREAM] vilbert/vilbert.py; anchor /root/reference/worker.py:286-289).
//
// Sequences are tiny (T <= 129, V <= 101) and attention is < 1 % of the FLOPs, so the goals are fusion, launch
// count and instruction count -- not tcgen05 throughput (a 128-row UMMA tile would be 75 % padding at T = 31).
// One CTA owns one (sample, head): Q/K/V head slices are staged once in shared memory (16-bit, rows padded by
// 16 B so ldmatrix is conflict-free); each warp owns 16 query rows and runs a register-resident flash-attention
// pass over the keys in blocks of 64: S = Q K^T on warp-level tensor-core MMAs (mma.sync m16n8k16, fp32
// accumulate), additive key mask, online softmax with quad shuffles in fp32, P V again on mma.sync.
// The co-attention kernel produces BOTH directions of a (sample, head) in one launch (text-query x image-key -> text
// context, then image-query x text-key -> image context), re-using one Q/K/V buffer set so five CTAs fit per SM.
#include <cstdlib>
#include "kernels.h"

namespace vb {

constexpr int kKeyBlock = 64;             // keys per online-softmax block
constexpr float kLog2e = 1.4426950408889634f;

template <int D>
struct AttnTile {
    static constexpr int kStride = D + 8;                 // 16-bit elements per padded row (row = D*2 + 16 bytes)
    static size_t bytes(int rows) { return static_cast<size_t>(rows) * kStride * 2; }
};

__host__ __device__ inline int pad16(int n) { return (n + 15) & ~15; }

// rows x D 16-bit tile: global (row stride ld elements, 16-byte aligned) -> padded shared with cp.async (every 16-byte
// copy of every tile is in flight before anyone waits); rows [rows, rows_pad) are zero-filled (src-size 0).
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, bool valid) {
    const uint32_t sz = valid ? 16u : 0u;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}
template <int D>
__device__ __forceinline__ void load_tile(uint16_t* dst, const uint16_t* src, int rows, int rows_pad, int ld) {
    constexpr int kVec = D / 8;
    constexpr int kStride = AttnTile<D>::kStride;
    for (int i = threadIdx.x; i < rows_pad * kVec; i += blockDim.x) {
        const int r = i / kVec, c = i % kVec;
        const bool ok = r < rows;
        cp_async16(dst + r * kStride + c * 8, src + (ok ? static_cast<size_t>(r) * ld + c * 8 : 0), ok);
    }
}

__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(p)));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t (&r)[4], const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(p)));
}
template <bool F16>
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    if constexpr (F16) {
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                     : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                     : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
    } else {
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                     : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                     : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
    }
}

// One warp: 16 query rows [r0, r0+16) of Qs against nk keys (Ks/Vs zero-padded to a multiple of 16 rows), output columns
// [oc0, oc0 + OW) of the head.  D = 128 is split into two 64-column work items (S is recomputed by both): 32 instead of 64
// accumulator registers per thread keep the kernel under 128 registers, i.e. five CTAs per SM and one wave at batch 64
// (at 170 registers: two CTAs per SM, 1.7 waves -- profiles/r1_attention_ncu.txt).
// mask_l2[j] = additive key mask * log2(e).  out: 16-bit global, already offset to this head's first column.
template <int D, int OW, bool F16>
__device__ __forceinline__ void attend_tile(const uint16_t* Qs, const uint16_t* Ks, const uint16_t* Vs, int r0, int nq,
                                            int nk, const float* mask_l2, float scale_l2, uint16_t* out, int ld_out,
                                            int lane, int oc0) {
    constexpr int kStride = AttnTile<D>::kStride;
    constexpr int kKSteps = D / 16;         // k-steps of Q K^T
    constexpr int kONTiles = OW / 8;        // 8-wide output column tiles of this work item
    const int g = lane >> 2, tq = lane & 3;  // row within 8, column pair within 8

    uint32_t qa[kKSteps][4];
#pragma unroll
    for (int ks = 0; ks < kKSteps; ++ks)
        ldsm_x4(qa[ks], Qs + (r0 + (lane & 15)) * kStride + ks * 16 + (lane >> 4) * 8);

    float o[kONTiles][4];
#pragma unroll
    for (int i = 0; i < kONTiles; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.0f;
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.0f, l1 = 0.0f;   // running max / sum for rows g and g+8

    const int nk_pad = pad16(nk);
    for (int kb = 0; kb < nk_pad; kb += kKeyBlock) {
        const int nkeys = min(kKeyBlock, nk_pad - kb);            // multiple of 16
        float s[kKeyBlock / 8][4];
        // ---- S = Q K^T for this key block
#pragma unroll
        for (int nt = 0; nt < kKeyBlock / 8; ++nt) {
            s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.0f;
            if (nt * 8 < nkeys) {
#pragma unroll
                for (int ks2 = 0; ks2 < kKSteps / 2; ++ks2) {
                    uint32_t kf[4];   // keys nt*8..+8: k-cols [ks2*32, +8), [+8,+16), [+16,+24), [+24,+32)
                    ldsm_x4(kf, Ks + (kb + nt * 8 + (lane & 7)) * kStride + ks2 * 32 + (lane >> 3) * 8);
                    mma16816<F16>(s[nt], qa[2 * ks2], kf[0], kf[1]);
                    mma16816<F16>(s[nt], qa[2 * ks2 + 1], kf[2], kf[3]);
                }
            }
        }
        // ---- scale + mask (log2 domain), block row max
        float bm0 = -INFINITY, bm1 = -INFINITY;
#pragma unroll
        for (int nt = 0; nt < kKeyBlock / 8; ++nt) {
            if (nt * 8 < nkeys) {
                const int j = kb + nt * 8 + tq * 2;
                const float ma = j < nk ? mask_l2[j] : -INFINITY;
                const float mb = j + 1 < nk ? mask_l2[j + 1] : -INFINITY;
                s[nt][0] = fmaf(s[nt][0], scale_l2, ma); s[nt][1] = fmaf(s[nt][1], scale_l2, mb);
                s[nt][2] = fmaf(s[nt][2], scale_l2, ma); s[nt][3] = fmaf(s[nt][3], scale_l2, mb);
                bm0 = fmaxf(bm0, fmaxf(s[nt][0], s[nt][1]));
                bm1 = fmaxf(bm1, fmaxf(s[nt][2], s[nt][3]));
            }
        }
        bm0 = fmaxf(bm0, __shfl_xor_sync(0xffffffffu, bm0, 1)); bm0 = fmaxf(bm0, __shfl_xor_sync(0xffffffffu, bm0, 2));
        bm1 = fmaxf(bm1, __shfl_xor_sync(0xffffffffu, bm1, 1)); bm1 = fmaxf(bm1, __shfl_xor_sync(0xffffffffu, bm1, 2));
        const float nm0 = fmaxf(m0, bm0), nm1 = fmaxf(m1, bm1);   // finite: every block holds >= 1 real key
        const float c0 = exp2f(m0 - nm0), c1 = exp2f(m1 - nm1);   // exp2f(-inf) = 0 on the first block
        m0 = nm0; m1 = nm1;
        float bs0 = 0.0f, bs1 = 0.0f;
#pragma unroll
        for (int nt = 0; nt < kKeyBlock / 8; ++nt) {
            if (nt * 8 < nkeys) {
                s[nt][0] = exp2f(s[nt][0] - nm0); s[nt][1] = exp2f(s[nt][1] - nm0);
                s[nt][2] = exp2f(s[nt][2] - nm1); s[nt][3] = exp2f(s[nt][3] - nm1);
                bs0 += s[nt][0] + s[nt][1];
                bs1 += s[nt][2] + s[nt][3];
            }
        }
        l0 = l0 * c0 + bs0;                  // per-lane partial sums; reduced over the quad at the end
        l1 = l1 * c1 + bs1;
#pragma unroll
        for (int i = 0; i < kONTiles; ++i) { o[i][0] *= c0; o[i][1] *= c0; o[i][2] *= c1; o[i][3] *= c1; }
        // ---- O += P V   (P: C fragments of two adjacent key tiles form one A fragment)
#pragma unroll
        for (int kk = 0; kk < kKeyBlock / 16; ++kk) {
            if (kk * 16 < nkeys) {
                uint32_t pa[4];
                pa[0] = pack16x2<F16>(s[2 * kk][0], s[2 * kk][1]);
                pa[1] = pack16x2<F16>(s[2 * kk][2], s[2 * kk][3]);
                pa[2] = pack16x2<F16>(s[2 * kk + 1][0], s[2 * kk + 1][1]);
                pa[3] = pack16x2<F16>(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
                for (int nt2 = 0; nt2 < kONTiles / 2; ++nt2) {
                    uint32_t vf[4];   // V[keys kk*16..+16][cols nt2*16..+16] transposed on load
                    ldsm_x4_trans(vf, Vs + (kb + kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * kStride + oc0 + nt2 * 16 + (lane >> 4) * 8);
                    mma16816<F16>(o[2 * nt2], pa, vf[0], vf[1]);
                    mma16816<F16>(o[2 * nt2 + 1], pa, vf[2], vf[3]);
                }
            }
        }
    }
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float i0 = 1.0f / l0, i1 = 1.0f / l1;
    const int row0 = r0 + g, row1 = r0 + g + 8;
#pragma unroll
    for (int nt = 0; nt < kONTiles; ++nt) {
        const int col = oc0 + nt * 8 + tq * 2;
        if (row0 < nq) *reinterpret_cast<uint32_t*>(out + static_cast<size_t>(row0) * ld_out + col) = pack16x2<F16>(o[nt][0] * i0, o[nt][1] * i0);
        if (row1 < nq) *reinterpret_cast<uint32_t*>(out + static_cast<size_t>(row1) * ld_out + col) = pack16x2<F16>(o[nt][2] * i1, o[nt][3] * i1);
    }
}

// Short key sequences (nk <= 64: every default ViLBERT shape) need no online softmax: one warp computes S = Q K^T and the
// probabilities ONCE for its 16 query rows and then walks the head's 64-column output slices (the general routine above would
// recompute S and the softmax per slice).  Same arithmetic, same order of operations per output element.
template <int D, bool F16>
__device__ __forceinline__ void attend_tile_short(const uint16_t* Qs, const uint16_t* Ks, const uint16_t* Vs, int r0, int nq,
                                                  int nk, const float* mask_l2, float scale_l2, uint16_t* out, int ld_out,
                                                  int lane) {
    constexpr int kStride = AttnTile<D>::kStride;
    constexpr int kKSteps = D / 16;
    const int g = lane >> 2, tq = lane & 3;
    const int nkeys = pad16(nk);                                  // <= 64, multiple of 16
    float s[kKeyBlock / 8][4];
    {
        uint32_t qa[kKSteps][4];
#pragma unroll
        for (int ks = 0; ks < kKSteps; ++ks)
            ldsm_x4(qa[ks], Qs + (r0 + (lane & 15)) * kStride + ks * 16 + (lane >> 4) * 8);
#pragma unroll
        for (int nt = 0; nt < kKeyBlock / 8; ++nt) {
            s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.0f;
            if (nt * 8 < nkeys) {
#pragma unroll
                for (int ks2 = 0; ks2 < kKSteps / 2; ++ks2) {
                    uint32_t kf[4];
                    ldsm_x4(kf, Ks + (nt * 8 + (lane & 7)) * kStride + ks2 * 32 + (lane >> 3) * 8);
                    mma16816<F16>(s[nt], qa[2 * ks2], kf[0], kf[1]);
                    mma16816<F16>(s[nt], qa[2 * ks2 + 1], kf[2], kf[3]);
                }
            }
        }
    }
    float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < kKeyBlock / 8; ++nt) {
        if (nt * 8 < nkeys) {
            const int j = nt * 8 + tq * 2;
            const float ma = j < nk ? mask_l2[j] : -INFINITY;
            const float mb = j + 1 < nk ? mask_l2[j + 1] : -INFINITY;
            s[nt][0] = fmaf(s[nt][0], scale_l2, ma); s[nt][1] = fmaf(s[nt][1], scale_l2, mb);
            s[nt][2] = fmaf(s[nt][2], scale_l2, ma); s[nt][3] = fmaf(s[nt][3], scale_l2, mb);
            m0 = fmaxf(m0, fmaxf(s[nt][0], s[nt][1]));
            m1 = fmaxf(m1, fmaxf(s[nt][2], s[nt][3]));
        }
    }
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1)); m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1)); m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
    float l0 = 0.0f, l1 = 0.0f;
    uint32_t pa[kKeyBlock / 16][4];                               // probabilities as A fragments (16 keys each)
#pragma unroll
    for (int nt = 0; nt < kKeyBlock / 8; ++nt) {
        if (nt * 8 < nkeys) {
            s[nt][0] = exp2f(s[nt][0] - m0); s[nt][1] = exp2f(s[nt][1] - m0);
            s[nt][2] = exp2f(s[nt][2] - m1); s[nt][3] = exp2f(s[nt][3] - m1);
            l0 += s[nt][0] + s[nt][1];
            l1 += s[nt][2] + s[nt][3];
        }
    }
#pragma unroll
    for (int kk = 0; kk < kKeyBlock / 16; ++kk) {
        pa[kk][0] = pack16x2<F16>(s[2 * kk][0], s[2 * kk][1]);
        pa[kk][1] = pack16x2<F16>(s[2 * kk][2], s[2 * kk][3]);
        pa[kk][2] = pack16x2<F16>(s[2 * kk + 1][0], s[2 * kk + 1][1]);
        pa[kk][3] = pack16x2<F16>(s[2 * kk + 1][2], s[2 * kk + 1][3]);
    }
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float i0 = 1.0f / l0, i1 = 1.0f / l1;
    const int row0 = r0 + g, row1 = r0 + g + 8;
#pragma unroll
    for (int oc0 = 0; oc0 < D; oc0 += 64) {                       // 64 output columns at a time: 32 accumulator registers
        float o[8][4];
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.0f;
#pragma unroll
        for (int kk = 0; kk < kKeyBlock / 16; ++kk) {
            if (kk * 16 < nkeys) {
#pragma unroll
                for (int nt2 = 0; nt2 < 4; ++nt2) {
                    uint32_t vf[4];
                    ldsm_x4_trans(vf, Vs + (kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * kStride + oc0 + nt2 * 16 + (lane >> 4) * 8);
                    mma16816<F16>(o[2 * nt2], pa[kk], vf[0], vf[1]);
                    mma16816<F16>(o[2 * nt2 + 1], pa[kk], vf[2], vf[3]);
                }
            }
        }
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const int col = oc0 + nt * 8 + tq * 2;
            if (row0 < nq) *reinterpret_cast<uint32_t*>(out + static_cast<size_t>(row0) * ld_out + col) = pack16x2<F16>(o[nt][0] * i0, o[nt][1] * i0);
            if (row1 < nq) *reinterpret_cast<uint32_t*>(out + static_cast<size_t>(row1) * ld_out + col) = pack16x2<F16>(o[nt][2] * i1, o[nt][3] * i1);
        }
    }
}

template <int D, bool F16>
__global__ void __launch_bounds__(256, 2)     // <= 128 registers: 5 CTAs of 3-4 warps per SM -> one wave at batch 64
self_attention_kernel(const uint16_t* __restrict__ qkv, int ld_qkv, int hidden, const float* __restrict__ key_mask_add,
                      uint16_t* __restrict__ ctx, int ld_ctx, int L, int nq, float scale_l2, int pdl) {
    // nq <= L: only the first nq query rows of each sample are computed (the last layer of a stream whose consumers read row 0
    // alone); keys and values are always the sample's L rows, so a computed row has the same bits as in the full pass
    extern __shared__ __align__(16) uint8_t smem_attn[];
    constexpr int kStride = AttnTile<D>::kStride;
    const int h = blockIdx.x, b = blockIdx.y;
    const int Lp = pad16(L), Qp = pad16(nq);
    uint16_t* Qs = reinterpret_cast<uint16_t*>(smem_attn);
    uint16_t* Ks = Qs + Qp * kStride;
    uint16_t* Vs = Ks + Lp * kStride;
    float* mask_s = reinterpret_cast<float*>(Vs + Lp * kStride);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;

    if (pdl) pdl_wait();

    const uint16_t* base = qkv + static_cast<size_t>(b) * L * ld_qkv + h * D;
    load_tile<D>(Qs, base, nq, Qp, ld_qkv);
    load_tile<D>(Ks, base + hidden, L, Lp, ld_qkv);
    load_tile<D>(Vs, base + 2 * hidden, L, Lp, ld_qkv);
    for (int j = threadIdx.x; j < L; j += blockDim.x) mask_s[j] = key_mask_add[b * L + j] * kLog2e;
    cp_async_wait_all();
    __syncthreads();
    if (pdl) pdl_launch_dependents();       // tiles are staged: the next kernel's prologue may overlap the math
    uint16_t* outp = ctx + static_cast<size_t>(b) * L * ld_ctx + h * D;
    constexpr int kSplit = D / 64, kOW = D / kSplit;             // work item = (16-row tile, 64-column slice of the head)
    if (L <= kKeyBlock) {                                        // one key block: S and the softmax once per row tile
        for (int t = warp; t * 16 < nq; t += nwarps)
            attend_tile_short<D, F16>(Qs, Ks, Vs, t * 16, nq, L, mask_s, scale_l2, outp, ld_ctx, lane);
        return;
    }
    for (int w = warp; (w / kSplit) * 16 < nq; w += nwarps)
        attend_tile<D, kOW, F16>(Qs, Ks, Vs, (w / kSplit) * 16, nq, L, mask_s, scale_l2, outp, ld_ctx, lane, (w % kSplit) * kOW);
}

template <int D, bool F16>
__global__ void __launch_bounds__(256, 2)
co_attention_kernel(const uint16_t* __restrict__ qkv_img, int ld_img, const uint16_t* __restrict__ qkv_txt, int ld_txt,
                    int hidden, const float* __restrict__ img_mask_add, const float* __restrict__ txt_mask_add,
                    uint16_t* __restrict__ ctx_txt, int ld_ctx_txt, uint16_t* __restrict__ ctx_img, int ld_ctx_img, int T,
                    int V, float scale_l2, int pdl) {
    // Two phases over ONE set of Q/K/V buffers sized for the longer sequence (39 KB at T=31/V=36 instead of 65 KB for all
    // six tiles: 5 CTAs per SM, so the 512 (sample, head) CTAs of a batch-64 layer are resident in a single wave).
    //   phase 1: text queries (Q2) over image keys/values (K1, V1) -> context for the text stream
    //   phase 2: image queries (Q1) over text keys/values (K2, V2)  -> context for the image stream
    extern __shared__ __align__(16) uint8_t smem_attn[];
    constexpr int kStride = AttnTile<D>::kStride;
    const int h = blockIdx.x, b = blockIdx.y;
    const int Tp = pad16(T), Vp = pad16(V);
    const int Lp = Tp > Vp ? Tp : Vp;
    uint16_t* Qs = reinterpret_cast<uint16_t*>(smem_attn);
    uint16_t* Ks = Qs + Lp * kStride;
    uint16_t* Vs = Ks + Lp * kStride;
    float* mask_img = reinterpret_cast<float*>(Vs + Lp * kStride);
    float* mask_txt = mask_img + V;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;

    if (pdl) pdl_wait();

    const uint16_t* bi = qkv_img + static_cast<size_t>(b) * V * ld_img + h * D;
    const uint16_t* bt = qkv_txt + static_cast<size_t>(b) * T * ld_txt + h * D;
    load_tile<D>(Qs, bt, T, Tp, ld_txt);                         // Q2
    load_tile<D>(Ks, bi + hidden, V, Vp, ld_img);                // K1
    load_tile<D>(Vs, bi + 2 * hidden, V, Vp, ld_img);            // V1
    for (int j = threadIdx.x; j < V; j += blockDim.x) mask_img[j] = img_mask_add[b * V + j] * kLog2e;
    for (int j = threadIdx.x; j < T; j += blockDim.x) mask_txt[j] = txt_mask_add[b * T + j] * kLog2e;
    cp_async_wait_all();
    __syncthreads();
    uint16_t* out_t = ctx_txt + static_cast<size_t>(b) * T * ld_ctx_txt + h * D;
    constexpr int kSplit = D / 64, kOW = D / kSplit;
    if (V <= kKeyBlock) {
        for (int t = warp; t * 16 < T; t += nwarps)
            attend_tile_short<D, F16>(Qs, Ks, Vs, t * 16, T, V, mask_img, scale_l2, out_t, ld_ctx_txt, lane);
    } else {
        for (int w = warp; (w / kSplit) * 16 < T; w += nwarps)
            attend_tile<D, kOW, F16>(Qs, Ks, Vs, (w / kSplit) * 16, T, V, mask_img, scale_l2, out_t, ld_ctx_txt, lane, (w % kSplit) * kOW);
    }
    __syncthreads();                                             // everyone is done reading phase-1 tiles
    load_tile<D>(Qs, bi, V, Vp, ld_img);                         // Q1
    load_tile<D>(Ks, bt + hidden, T, Tp, ld_txt);                // K2
    load_tile<D>(Vs, bt + 2 * hidden, T, Tp, ld_txt);            // V2
    cp_async_wait_all();
    __syncthreads();
    if (pdl) pdl_launch_dependents();
    uint16_t* out_v = ctx_img + static_cast<size_t>(b) * V * ld_ctx_img + h * D;
    if (T <= kKeyBlock) {
        for (int t = warp; t * 16 < V; t += nwarps)
            attend_tile_short<D, F16>(Qs, Ks, Vs, t * 16, V, T, mask_txt, scale_l2, out_v, ld_ctx_img, lane);
    } else {
        for (int w = warp; (w / kSplit) * 16 < V; w += nwarps)
            attend_tile<D, kOW, F16>(Qs, Ks, Vs, (w / kSplit) * 16, V, T, mask_txt, scale_l2, out_v, ld_ctx_img, lane, (w % kSplit) * kOW);
    }
}

template <int D, bool F16>
static cudaError_t launch_self(const __nv_bfloat16* qkv, int ld_qkv, int hidden, const float* key_mask_add,
                               __nv_bfloat16* ctx, int ld_ctx, int B, int L, int nq, int heads, int pdl, cudaStream_t st) {
    const int Lp = pad16(L), Qp = pad16(nq);
    const size_t smem = AttnTile<D>::bytes(Qp) + 2 * AttnTile<D>::bytes(Lp) + sizeof(float) * L;
    if (smem > 227 * 1024) return cudaErrorInvalidValue;
    cudaError_t e = set_smem(self_attention_kernel<D, F16>, smem);
    if (e != cudaSuccess) return e;
    static const int split_warps = [] { const char* e = getenv("VB200_ATTN_SPLIT_WARPS"); return e ? atoi(e) : 0; }();
    // one warp per 16-row tile, walking its D / 64 column slices in turn (measured better than one warp per slice: 3-warp CTAs
    // of the 128-wide heads fit five per SM -> one wave; VB200_ATTN_SPLIT_WARPS=1 for the other layout)
    const int nwarps = min(8, (Qp / 16) * (split_warps ? D / 64 : 1));
    const float scale_l2 = kLog2e / sqrtf(static_cast<float>(D));
    return launch_ex(self_attention_kernel<D, F16>, dim3(heads, B), dim3(32 * nwarps), smem, pdl, st,
                     reinterpret_cast<const uint16_t*>(qkv), ld_qkv, hidden, key_mask_add, reinterpret_cast<uint16_t*>(ctx),
                     ld_ctx, L, nq, scale_l2, pdl);
}

cudaError_t launch_self_attention(const __nv_bfloat16* qkv, int ld_qkv, int hidden, const float* key_mask_add,
                                  __nv_bfloat16* ctx, int ld_ctx, int B, int L, int nq, int heads, int head_dim, int pdl,
                                  int f16, cudaStream_t st) {
    if (L < 1 || nq < 1 || nq > L || (head_dim != 64 && head_dim != 128) || (ld_qkv & 7) || (ld_ctx & 1) || (hidden & 7))
        return cudaErrorInvalidValue;
#define VB_SELF(D, F) launch_self<D, F>(qkv, ld_qkv, hidden, key_mask_add, ctx, ld_ctx, B, L, nq, heads, pdl, st)
    if (head_dim == 64) return f16 ? VB_SELF(64, true) : VB_SELF(64, false);
    return f16 ? VB_SELF(128, true) : VB_SELF(128, false);
#undef VB_SELF
}

template <int D, bool F16>
static cudaError_t launch_co(const __nv_bfloat16* qkv_img, int ld_img, const __nv_bfloat16* qkv_txt, int ld_txt, int hidden,
                             const float* img_mask_add, const float* txt_mask_add, __nv_bfloat16* ctx_txt, int ld_ctx_txt,
                             __nv_bfloat16* ctx_img, int ld_ctx_img, int B, int T, int V, int heads, int pdl,
                             cudaStream_t st) {
    const int Tp = pad16(T), Vp = pad16(V);
    const int Lp = Tp > Vp ? Tp : Vp;
    const size_t smem = 3 * AttnTile<D>::bytes(Lp) + sizeof(float) * (T + V);
    if (smem > 227 * 1024) return cudaErrorInvalidValue;     // sequence too long for one CTA's shared memory
    cudaError_t e = set_smem(co_attention_kernel<D, F16>, smem);
    if (e != cudaSuccess) return e;
    static const int split_warps = [] { const char* e = getenv("VB200_ATTN_SPLIT_WARPS"); return e ? atoi(e) : 0; }();
    const int nwarps = max(4, min(8, (Lp / 16) * (split_warps ? D / 64 : 1)));  // >= 4 warps: cp.async staging over 128 threads
    const float scale_l2 = kLog2e / sqrtf(static_cast<float>(D));
    return launch_ex(co_attention_kernel<D, F16>, dim3(heads, B), dim3(32 * nwarps), smem, pdl, st,
                     reinterpret_cast<const uint16_t*>(qkv_img), ld_img, reinterpret_cast<const uint16_t*>(qkv_txt), ld_txt,
                     hidden, img_mask_add, txt_mask_add, reinterpret_cast<uint16_t*>(ctx_txt), ld_ctx_txt,
                     reinterpret_cast<uint16_t*>(ctx_img), ld_ctx_img, T, V, scale_l2, pdl);
}

cudaError_t launch_co_attention(const __nv_bfloat16* qkv_img, int ld_img, const __nv_bfloat16* qkv_txt, int ld_txt,
                                int hidden, const float* img_mask_add, const float* txt_mask_add,
                                __nv_bfloat16* ctx_txt, int ld_ctx_txt, __nv_bfloat16* ctx_img, int ld_ctx_img, int B,
                                int T, int V, int heads, int head_dim, int pdl, int f16, cudaStream_t st) {
    if (T < 1 || V < 1 || (head_dim != 64 && head_dim != 128) || (ld_img & 7) || (ld_txt & 7) || (hidden & 7) ||
        (ld_ctx_txt & 1) || (ld_ctx_img & 1))
        return cudaErrorInvalidValue;
#define VB_CO(D, F) launch_co<D, F>(qkv_img, ld_img, qkv_txt, ld_txt, hidden, img_mask_add, txt_mask_add, ctx_txt, ld_ctx_txt, \
                                    ctx_img, ld_ctx_img, B, T, V, heads, pdl, st)
    if (head_dim == 64) return f16 ? VB_CO(64, true) : VB_CO(64, false);
    return f16 ? VB_CO(128, true) : VB_CO(128, false);
#undef VB_CO
}

}  // namespace vb
