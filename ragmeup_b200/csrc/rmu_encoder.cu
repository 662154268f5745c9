// Post-LN BERT encoder forward for sm_100a: sentence embeddings and cross-encoder logits.
//
// Stands behind HuggingFaceEmbeddings.embed_documents / embed_query (reference call sites
// server/RAGHelper_local.py:114-117, server/RAGHelper_cloud.py:101-103; arithmetic = transformers
// BertModel + sentence-transformers Pooling/Normalize, SURVEY.md H2-H4) and behind
// HuggingFaceCrossEncoder.score (server/RAGHelper.py:484, server/ScoredCrossEncoderReranker.py:42;
// BertForSequenceClassification, H8-H9).  SURVEY.md §8 rows a2-a5, a9, a10.
//
// Batches are RAGGED (cu_seqlens): no padding token is ever computed.  The reference pads to the
// longest sequence of each 32-batch and masks padded keys with finfo.min, which contributes exactly
// 0 to every softmax, so the packed computation returns the same numbers.
//
// Activations between kernels are split fp16 planes (see rmu_gemm.cuh); LayerNorm, softmax, GELU,
// residual adds, pooling and the classifier head are fp32.
#include <algorithm>
#include <mutex>
#include <vector>

#include "rmu_gemm.cuh"

namespace rmu {

// ------------------------------------------------------------------------------------ small kernels
__global__ void split_planes_kernel(const float* __restrict__ src, __half* __restrict__ hi, __half* __restrict__ lo, size_t n) {
    size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) {
        __half h, l;
        split_f16(src[i], h, l);
        hi[i] = h;
        lo[i] = l;
    }
}

constexpr int kMaxPerLane = 32;  // hidden <= 1024

// LayerNorm of one row (H % 128 == 0).  Lane l holds float4 chunks l, l + 32, l + 64 ... of the row
// (element v[i] is column ((i / 4) * 32 + l) * 4 + i % 4), so every warp load is one contiguous 512-byte
// segment and every plane store one contiguous 256-byte segment.  Biased variance, eps inside the sqrt
// (nn.LayerNorm).
__device__ __forceinline__ void warp_layernorm_store(float (&v)[kMaxPerLane], int per_lane, int H, float eps,
                                                     const float* __restrict__ g, const float* __restrict__ b,
                                                     __half* __restrict__ hi, __half* __restrict__ lo) {
    const unsigned lane = lane_id();
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < kMaxPerLane; ++i) if (i < per_lane) s += v[i];
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = s / static_cast<float>(H);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < kMaxPerLane; ++i) if (i < per_lane) { const float d = v[i] - mean; q = fmaf(d, d, q); }
    for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
    const float rstd = 1.0f / sqrtf(q / static_cast<float>(H) + eps);
#pragma unroll
    for (int i = 0; i < kMaxPerLane; i += 4) {
        if (i < per_lane) {
            const int col = (i * 8 + static_cast<int>(lane)) * 4;      // (i / 4) * 32 + lane, in float4 units
            const float4 gg = *reinterpret_cast<const float4*>(g + col);
            const float4 bb = *reinterpret_cast<const float4*>(b + col);
            const float y0 = (v[i] - mean) * rstd * gg.x + bb.x, y1 = (v[i + 1] - mean) * rstd * gg.y + bb.y;
            const float y2 = (v[i + 2] - mean) * rstd * gg.z + bb.z, y3 = (v[i + 3] - mean) * rstd * gg.w + bb.w;
            __half h0, l0, h1, l1, h2, l2, h3, l3;
            split_f16(y0, h0, l0); split_f16(y1, h1, l1); split_f16(y2, h2, l2); split_f16(y3, h3, l3);
            __half2 ha = __halves2half2(h0, h1), hb = __halves2half2(h2, h3);
            __half2 la = __halves2half2(l0, l1), lb = __halves2half2(l2, l3);
            uint2 ph, pl;
            ph.x = *reinterpret_cast<uint32_t*>(&ha); ph.y = *reinterpret_cast<uint32_t*>(&hb);
            pl.x = *reinterpret_cast<uint32_t*>(&la); pl.y = *reinterpret_cast<uint32_t*>(&lb);
            *reinterpret_cast<uint2*>(hi + col) = ph;
            *reinterpret_cast<uint2*>(lo + col) = pl;
        }
    }
}

// word + position + token-type embedding sum -> LayerNorm -> split planes.  One warp per token.
__global__ void embed_ln_kernel(const int* __restrict__ ids, const int* __restrict__ type_ids,
                                const int* __restrict__ cu, int B, int T, int H, int vocab, int max_pos, int type_vocab,
                                const float* __restrict__ word, const float* __restrict__ pos,
                                const float* __restrict__ typ, const float* __restrict__ g, const float* __restrict__ b,
                                float eps, __half* __restrict__ hi, __half* __restrict__ lo) {
    const int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (t >= T) return;
    // sequence of token t: last b with cu[b] <= t
    int lo_b = 0, hi_b = B;
    while (hi_b - lo_b > 1) {
        const int mid = (lo_b + hi_b) >> 1;
        if (cu[mid] <= t) lo_b = mid; else hi_b = mid;
    }
    int p = t - cu[lo_b];
    p = p < max_pos ? p : max_pos - 1;
    int id = ids[t];
    id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
    int ty = type_ids ? type_ids[t] : 0;
    ty = ty < 0 ? 0 : (ty >= type_vocab ? type_vocab - 1 : ty);
    const int per_lane = H >> 5;
    const int l4 = static_cast<int>(lane_id()) * 4;
    const float* w = word + static_cast<size_t>(id) * H + l4;
    const float* pp = pos + static_cast<size_t>(p) * H + l4;
    const float* tt = typ + static_cast<size_t>(ty) * H + l4;
    float v[kMaxPerLane];
#pragma unroll
    for (int i = 0; i < kMaxPerLane; i += 4) {
        if (i < per_lane) {
            const float4 a = *reinterpret_cast<const float4*>(w + i * 32);
            const float4 c = *reinterpret_cast<const float4*>(tt + i * 32);
            const float4 e = *reinterpret_cast<const float4*>(pp + i * 32);
            // HF: inputs_embeds + token_type_embeddings, then + position_embeddings
            v[i] = (a.x + c.x) + e.x; v[i + 1] = (a.y + c.y) + e.y; v[i + 2] = (a.z + c.z) + e.z; v[i + 3] = (a.w + c.w) + e.w;
        }
    }
    warp_layernorm_store(v, per_lane, H, eps, g, b, hi + static_cast<size_t>(t) * H, lo + static_cast<size_t>(t) * H);
}

// LayerNorm(pre) -> split planes.  One warp per token.
__global__ void ln_kernel(const float* __restrict__ pre, int T, int H, const float* __restrict__ g,
                          const float* __restrict__ b, float eps, __half* __restrict__ hi, __half* __restrict__ lo) {
    const int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (t >= T) return;
    const int per_lane = H >> 5;
    const float* row = pre + static_cast<size_t>(t) * H + lane_id() * 4;
    float v[kMaxPerLane];
#pragma unroll
    for (int i = 0; i < kMaxPerLane; i += 4) {
        if (i < per_lane) {
            const float4 a = *reinterpret_cast<const float4*>(row + i * 32);
            v[i] = a.x; v[i + 1] = a.y; v[i + 2] = a.z; v[i + 3] = a.w;
        }
    }
    warp_layernorm_store(v, per_lane, H, eps, g, b, hi + static_cast<size_t>(t) * H, lo + static_cast<size_t>(t) * H);
}

__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

__device__ __forceinline__ void split_pack(float x, float y, uint32_t& hi, uint32_t& lo) {
    __half hx, lx, hy, ly;
    split_f16(x, hx, lx);
    split_f16(y, hy, ly);
    __half2 h = __halves2half2(hx, hy), l = __halves2half2(lx, ly);
    hi = *reinterpret_cast<uint32_t*>(&h);
    lo = *reinterpret_cast<uint32_t*>(&l);
}

constexpr int kKeySB = 256;   // keys resident in shared memory at a time

// ---------------------------------------------------------------------------------------------------
// attention_planes_kernel (mma.sync; sequences the tcgen05 kernel does not take): Q (pre-scaled), K and V arrive as
// split fp16 planes [T, 3H] written by the QKV GEMM epilogue, so this kernel does no conversion work:
// K / V tiles are 16-byte copies into shared memory ([key][d] for both) and the P V operand is fetched
// with ldmatrix.trans.  One CTA = (sequence, head, block of 16 * kAttWarps query rows), one warp = 16 rows.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], const void* smem_row) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(smem_u32(smem_row)));
}

__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void* smem_row) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(smem_u32(smem_row)));
}

constexpr int kAttWarps = 10;   // 160 query rows per CTA (a 147-token rerank pair fits one CTA)

__device__ __forceinline__ float fast_exp2(float x) {   // ex2.approx: 2 ulp, exp2(-inf) = +0
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// MINB = CTAs per SM the register allocation is bounded for (d_h = 32: 2 -> 95 registers, no spills; bounding it
// to 3 CTAs / 64 registers spills in the key loop and measured 541 us instead of 352 us per layer call).
// Grid = (heads, sequences, row blocks): the heads of one sequence run together, so the 64-byte (d_h = 32)
// K / V row segments of neighbouring heads are fetched from DRAM as whole lines.
template <int DH, int MINB>
__global__ void __launch_bounds__(kAttWarps * 32, MINB) attention_planes_kernel(const __half* __restrict__ ph, const __half* __restrict__ pl,
                                                                          const int* __restrict__ cu, int H, int ksb,
                                                                          __half* __restrict__ ctx_hi, __half* __restrict__ ctx_lo) {
    constexpr int KSTR = DH + 8;
    constexpr int KS = DH / 16;
    constexpr int NT = DH / 8;
    extern __shared__ __align__(16) unsigned char att_smem[];
    __half* Kh = reinterpret_cast<__half*>(att_smem);
    __half* Kl = Kh + ksb * KSTR;           // ksb = keys resident at a time (multiple of 32, <= kKeySB)
    __half* Vh = Kl + ksb * KSTR;
    __half* Vl = Vh + ksb * KSTR;

    const int b = blockIdx.y, h = blockIdx.x;
    const int t0 = cu[b], S = cu[b + 1] - t0;
    const int rbase = blockIdx.z * (kAttWarps * 16);
    if (rbase >= S) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    const size_t ld = static_cast<size_t>(3) * H;
    const __half* qh_base = ph + static_cast<size_t>(t0) * ld + h * DH;
    const __half* ql_base = pl + static_cast<size_t>(t0) * ld + h * DH;
    const int r0 = rbase + warp * 16;
    const bool warp_live = r0 < S;

    uint32_t qh[KS][4], ql[KS][4];
    {
        const int ra = r0 + g, rb = r0 + g + 8;
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
#pragma unroll
            for (int i = 0; i < 4; ++i) { qh[ks][i] = 0u; ql[ks][i] = 0u; }
            if (warp_live && ra < S) {
                qh[ks][0] = *reinterpret_cast<const uint32_t*>(qh_base + ra * ld + ks * 16 + 2 * t);
                ql[ks][0] = *reinterpret_cast<const uint32_t*>(ql_base + ra * ld + ks * 16 + 2 * t);
                qh[ks][2] = *reinterpret_cast<const uint32_t*>(qh_base + ra * ld + ks * 16 + 2 * t + 8);
                ql[ks][2] = *reinterpret_cast<const uint32_t*>(ql_base + ra * ld + ks * 16 + 2 * t + 8);
            }
            if (warp_live && rb < S) {
                qh[ks][1] = *reinterpret_cast<const uint32_t*>(qh_base + rb * ld + ks * 16 + 2 * t);
                ql[ks][1] = *reinterpret_cast<const uint32_t*>(ql_base + rb * ld + ks * 16 + 2 * t);
                qh[ks][3] = *reinterpret_cast<const uint32_t*>(qh_base + rb * ld + ks * 16 + 2 * t + 8);
                ql[ks][3] = *reinterpret_cast<const uint32_t*>(ql_base + rb * ld + ks * 16 + 2 * t + 8);
            }
        }
    }
    float oacc[NT][4];
#pragma unroll
    for (int n = 0; n < NT; ++n) oacc[n][0] = oacc[n][1] = oacc[n][2] = oacc[n][3] = 0.f;
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;

    for (int sb0 = 0; sb0 < S; sb0 += ksb) {
        const int nk = min(ksb, S - sb0);
        const int nk16 = (nk + 15) & ~15;
        __syncthreads();
        for (int e = threadIdx.x; e < nk16 * (DH / 8); e += blockDim.x) {
            const int j = e / (DH / 8), c8 = (e % (DH / 8)) * 8;
            uint4 kh = make_uint4(0, 0, 0, 0), kl = kh, vh = kh, vl = kh;
            if (j < nk) {
                const size_t o = static_cast<size_t>(t0 + sb0 + j) * ld + h * DH + c8;
                kh = *reinterpret_cast<const uint4*>(ph + o + H);
                kl = *reinterpret_cast<const uint4*>(pl + o + H);
                vh = *reinterpret_cast<const uint4*>(ph + o + 2 * H);
                vl = *reinterpret_cast<const uint4*>(pl + o + 2 * H);
            }
            *reinterpret_cast<uint4*>(Kh + j * KSTR + c8) = kh;
            *reinterpret_cast<uint4*>(Kl + j * KSTR + c8) = kl;
            *reinterpret_cast<uint4*>(Vh + j * KSTR + c8) = vh;
            *reinterpret_cast<uint4*>(Vl + j * KSTR + c8) = vl;
        }
        __syncthreads();
        if (!warp_live) continue;
        for (int kb0 = 0; kb0 < nk16; kb0 += 32) {
            float sacc[4][4];
#pragma unroll
            for (int n = 0; n < 4; ++n) sacc[n][0] = sacc[n][1] = sacc[n][2] = sacc[n][3] = 0.f;
            const bool full_blk = kb0 + 32 <= nk16;      // else only the first two n-tiles hold keys
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {
                // K fragments of four key tiles through two ldmatrix.x4 per plane: matrices (keys a, d lo),
                // (keys a, d hi), (keys a+1, d lo), (keys a+1, d hi); rows past nk16 are stale smem, masked below
                uint32_t bh[4][2], bl[4][2];
                const int lrow = (lane & 7) + ((lane >> 4) << 3);
                const int lcol = ks * 16 + ((lane >> 3) & 1) * 8;
#pragma unroll
                for (int n2 = 0; n2 < 2; ++n2) {
                    uint32_t th[4], tl[4];
                    ldmatrix_x4(th, Kh + (kb0 + n2 * 16 + lrow) * KSTR + lcol);
                    ldmatrix_x4(tl, Kl + (kb0 + n2 * 16 + lrow) * KSTR + lcol);
                    bh[2 * n2][0] = th[0]; bh[2 * n2][1] = th[1]; bh[2 * n2 + 1][0] = th[2]; bh[2 * n2 + 1][1] = th[3];
                    bl[2 * n2][0] = tl[0]; bl[2 * n2][1] = tl[1]; bl[2 * n2 + 1][0] = tl[2]; bl[2 * n2 + 1][1] = tl[3];
                }
#pragma unroll
                for (int n = 0; n < 4; ++n) if (n < 2 || full_blk) mma16816(sacc[n], qh[ks], bh[n]);
#pragma unroll
                for (int n = 0; n < 4; ++n) if (n < 2 || full_blk) mma16816(sacc[n], ql[ks], bh[n]);
#pragma unroll
                for (int n = 0; n < 4; ++n) if (n < 2 || full_blk) mma16816(sacc[n], qh[ks], bl[n]);
            }
            float bm0 = -INFINITY, bm1 = -INFINITY;
            if (kb0 + 32 > nk) {                     // only the last key block holds keys past the sequence end
#pragma unroll
                for (int n = 0; n < 4; ++n) {
                    const int k0 = kb0 + n * 8 + 2 * t;
                    if (k0 >= nk) { sacc[n][0] = -INFINITY; sacc[n][2] = -INFINITY; }
                    if (k0 + 1 >= nk) { sacc[n][1] = -INFINITY; sacc[n][3] = -INFINITY; }
                }
            }
#pragma unroll
            for (int n = 0; n < 4; ++n) {
                bm0 = fmaxf(bm0, fmaxf(sacc[n][0], sacc[n][1]));
                bm1 = fmaxf(bm1, fmaxf(sacc[n][2], sacc[n][3]));
            }
            bm0 = fmaxf(bm0, __shfl_xor_sync(0xffffffffu, bm0, 1));
            bm0 = fmaxf(bm0, __shfl_xor_sync(0xffffffffu, bm0, 2));
            bm1 = fmaxf(bm1, __shfl_xor_sync(0xffffffffu, bm1, 1));
            bm1 = fmaxf(bm1, __shfl_xor_sync(0xffffffffu, bm1, 2));
            const float mn0 = fmaxf(m0, bm0), mn1 = fmaxf(m1, bm1);
            const float c0 = fast_exp2(m0 - mn0), c1 = fast_exp2(m1 - mn1);   // scores are pre-scaled by log2(e)
            m0 = mn0; m1 = mn1;
            float ps0 = 0.f, ps1 = 0.f;
#pragma unroll
            for (int n = 0; n < 4; ++n) {
                sacc[n][0] = fast_exp2(sacc[n][0] - mn0); sacc[n][1] = fast_exp2(sacc[n][1] - mn0);
                sacc[n][2] = fast_exp2(sacc[n][2] - mn1); sacc[n][3] = fast_exp2(sacc[n][3] - mn1);
                ps0 += sacc[n][0] + sacc[n][1];
                ps1 += sacc[n][2] + sacc[n][3];
            }
            l0 = l0 * c0 + ps0;
            l1 = l1 * c1 + ps1;
#pragma unroll
            for (int n = 0; n < NT; ++n) { oacc[n][0] *= c0; oacc[n][1] *= c0; oacc[n][2] *= c1; oacc[n][3] *= c1; }
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
                if (kb0 + kk * 16 < nk16) {
                    uint32_t pfh[4], pfl[4];
                    split_pack(sacc[2 * kk][0], sacc[2 * kk][1], pfh[0], pfl[0]);
                    split_pack(sacc[2 * kk][2], sacc[2 * kk][3], pfh[1], pfl[1]);
                    split_pack(sacc[2 * kk + 1][0], sacc[2 * kk + 1][1], pfh[2], pfl[2]);
                    split_pack(sacc[2 * kk + 1][2], sacc[2 * kk + 1][3], pfh[3], pfl[3]);
                    // ldmatrix.x4.trans: matrices (keys 0-7, d-tile n), (keys 8-15, n), (keys 0-7, n+1), (keys 8-15, n+1)
                    const int krow = kb0 + kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
                    const int dsel = (lane >> 4) * 8;
                    uint32_t vh4[NT / 2][4], vl4[NT / 2][4];
#pragma unroll
                    for (int n2 = 0; n2 < NT / 2; ++n2) {
                        ldmatrix_x4_trans(vh4[n2], Vh + krow * KSTR + n2 * 16 + dsel);
                        ldmatrix_x4_trans(vl4[n2], Vl + krow * KSTR + n2 * 16 + dsel);
                    }
#pragma unroll
                    for (int n2 = 0; n2 < NT / 2; ++n2) {
                        const uint32_t a_[2] = {vh4[n2][0], vh4[n2][1]}, b_[2] = {vh4[n2][2], vh4[n2][3]};
                        mma16816(oacc[2 * n2], pfh, a_);
                        mma16816(oacc[2 * n2 + 1], pfh, b_);
                    }
#pragma unroll
                    for (int n2 = 0; n2 < NT / 2; ++n2) {
                        const uint32_t a_[2] = {vh4[n2][0], vh4[n2][1]}, b_[2] = {vh4[n2][2], vh4[n2][3]};
                        mma16816(oacc[2 * n2], pfl, a_);
                        mma16816(oacc[2 * n2 + 1], pfl, b_);
                    }
#pragma unroll
                    for (int n2 = 0; n2 < NT / 2; ++n2) {
                        const uint32_t a_[2] = {vl4[n2][0], vl4[n2][1]}, b_[2] = {vl4[n2][2], vl4[n2][3]};
                        mma16816(oacc[2 * n2], pfh, a_);
                        mma16816(oacc[2 * n2 + 1], pfh, b_);
                    }
                }
            }
        }
    }
    if (!warp_live) return;
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
    l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float i0 = 1.0f / l0, i1 = 1.0f / l1;
    const int ra = r0 + g, rb = r0 + g + 8;
#pragma unroll
    for (int n = 0; n < NT; ++n) {
        const int col = h * DH + n * 8 + 2 * t;
        uint32_t hi, lo;
        if (ra < S) {
            split_pack(oacc[n][0] * i0, oacc[n][1] * i0, hi, lo);
            *reinterpret_cast<uint32_t*>(ctx_hi + static_cast<size_t>(t0 + ra) * H + col) = hi;
            *reinterpret_cast<uint32_t*>(ctx_lo + static_cast<size_t>(t0 + ra) * H + col) = lo;
        }
        if (rb < S) {
            split_pack(oacc[n][2] * i1, oacc[n][3] * i1, hi, lo);
            *reinterpret_cast<uint32_t*>(ctx_hi + static_cast<size_t>(t0 + rb) * H + col) = hi;
            *reinterpret_cast<uint32_t*>(ctx_lo + static_cast<size_t>(t0 + rb) * H + col) = lo;
        }
    }
}

// sentence-transformers Pooling (mean | cls) + optional Normalize -> out [B, H]
__global__ void __launch_bounds__(256) pool_kernel(const __half* __restrict__ hi, const __half* __restrict__ lo,
                                                   const int* __restrict__ cu, int H, int mode, int normalize,
                                                   float* __restrict__ out) {
    __shared__ float red[32];
    const int b = blockIdx.x;
    const int t0 = cu[b], S = cu[b + 1] - t0;
    float ss = 0.f;
    float vals[4];   // H <= 1024 with 256 threads
    int nv = 0;
    for (int d = threadIdx.x; d < H; d += blockDim.x, ++nv) {
        float v = 0.f;
        if (mode == RMU_POOL_CLS) {
            if (S > 0) v = __half2float(hi[static_cast<size_t>(t0) * H + d]) + __half2float(lo[static_cast<size_t>(t0) * H + d]);
        } else {
            for (int t = 0; t < S; ++t) {
                const size_t o = static_cast<size_t>(t0 + t) * H + d;
                v += __half2float(hi[o]) + __half2float(lo[o]);
            }
            v = v / fmaxf(static_cast<float>(S), 1e-9f);
        }
        vals[nv] = v;
        ss = fmaf(v, v, ss);
    }
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
    __syncthreads();
    float tot = 0.f;
    for (int i = 0; i < (blockDim.x >> 5); ++i) tot += red[i];
    const float inv = normalize ? 1.0f / fmaxf(sqrtf(tot), 1e-12f) : 1.0f;
    nv = 0;
    for (int d = threadIdx.x; d < H; d += blockDim.x, ++nv) out[static_cast<size_t>(b) * H + d] = vals[nv] * inv;
}

// BertPooler (tanh(W_p h_cls + b_p)) + classifier -> logits [B, num_labels]
__global__ void __launch_bounds__(256) cls_head_kernel(const __half* __restrict__ hi, const __half* __restrict__ lo,
                                                       const int* __restrict__ cu, int H, int num_labels,
                                                       const float* __restrict__ pw, const float* __restrict__ pb,
                                                       const float* __restrict__ cw, const float* __restrict__ cb,
                                                       float* __restrict__ out) {
    extern __shared__ float sh[];   // h[H], pooled[H]
    float* hcls = sh;
    float* pooled = sh + H;
    const int b = blockIdx.x;
    const size_t o = static_cast<size_t>(cu[b]) * H;
    for (int d = threadIdx.x; d < H; d += blockDim.x) hcls[d] = __half2float(hi[o + d]) + __half2float(lo[o + d]);
    __syncthreads();
    const int warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int j = warp; j < H; j += nw) {
        const float* wr = pw + static_cast<size_t>(j) * H;
        float s = 0.f;
        for (int d = lane_id(); d < H; d += 32) s = fmaf(wr[d], hcls[d], s);
        for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
        if (lane_id() == 0) pooled[j] = tanhf(s + pb[j]);
    }
    __syncthreads();
    for (int c = warp; c < num_labels; c += nw) {
        const float* wr = cw + static_cast<size_t>(c) * H;
        float s = 0.f;
        for (int d = lane_id(); d < H; d += 32) s = fmaf(wr[d], pooled[d], s);
        for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
        if (lane_id() == 0) out[static_cast<size_t>(b) * num_labels + c] = s + cb[c];
    }
}

__global__ void join_planes_kernel(const __half* __restrict__ hi, const __half* __restrict__ lo, float* __restrict__ out, size_t n) {
    size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) out[i] = __half2float(hi[i]) + __half2float(lo[i]);
}

#include "rmu_attention.cuh"

}  // namespace rmu

using namespace rmu;

struct EncLayer {
    SplitOperand Wqkv, Wo, W1, W2;
    float *bqkv = nullptr, *bo = nullptr, *b1 = nullptr, *b2 = nullptr;
    float *ln1g = nullptr, *ln1b = nullptr, *ln2g = nullptr, *ln2b = nullptr;
};

struct rmu_encoder {
    rmu_bert_config cfg{};
    int has_head = 0, sms = 0, device = 0;
    std::vector<void*> allocs;
    float *word = nullptr, *pos = nullptr, *typ = nullptr, *eg = nullptr, *eb = nullptr;
    std::vector<EncLayer> layers;
    float *pw = nullptr, *pb = nullptr, *cw = nullptr, *cb = nullptr;
    // activations
    int tok_cap = 0, seq_cap = 0;
    std::vector<void*> act_allocs;
    SplitOperand X, CTX, X1, FF, QKVP;   // QKVP: q (pre-scaled) | k | v as split planes [T, 3H]
    CUtensorMap att_q_hi{}, att_q_lo{}, att_k_hi{}, att_k_lo{};   // tcgen05 attention: boxes {d_h, 128 rows} / {d_h, 64 rows} of QKVP
    __half* QKVI = nullptr;                                       // [T, 6H]: q | k | v with every head's hi and lo halves interleaved
    CUtensorMap att_qkvi{};                                       // head-pair attention (d_h = 32): boxes {64 halves, 32 rows} of QKVI
    float* PRE = nullptr;                 // fp32 pre-LayerNorm rows (hidden sizes the fused GEMM+LN kernel does not cover)
    // staging of the *_host entry points: owned by host_mu alone (NOT part of the activation workspace, which a
    // concurrent device-pointer caller may free and re-allocate under mu)
    int *d_ids = nullptr, *d_typ = nullptr, *d_cu = nullptr;
    float* d_out = nullptr;
    int stage_tok_cap = 0, stage_seq_cap = 0;
    cudaEvent_t ws_done = nullptr;   // last use of the shared activation workspace (callers on other streams wait on it)
    std::mutex mu;
    std::mutex host_mu;   // the *_host entry points share the staging buffers above: one at a time per handle
};

template <typename T>
static int dev_alloc(std::vector<void*>& keep, T** p, size_t count) {
    void* q = nullptr;
    RMU_CUDA(cudaMalloc(&q, std::max<size_t>(count, 1) * sizeof(T)));
    keep.push_back(q);
    *p = static_cast<T*>(q);
    return RMU_OK;
}

static int upload(rmu_encoder* e, float** dst, const float* src_h, size_t n) {
    int rc = dev_alloc(e->allocs, dst, n);
    if (rc != RMU_OK) return rc;
    RMU_CUDA(cudaMemcpy(*dst, src_h, n * sizeof(float), cudaMemcpyHostToDevice));
    return RMU_OK;
}

// upload a [rows, cols] fp32 weight (optionally a vertical concat of several) as split fp16 planes
static int upload_split(rmu_encoder* e, SplitOperand* op, const std::vector<const float*>& parts, int rows_each, int cols) {
    const size_t rows = static_cast<size_t>(rows_each) * parts.size();
    const size_t n = rows * cols;
    float* tmp = nullptr;
    RMU_CUDA(cudaMalloc(reinterpret_cast<void**>(&tmp), n * sizeof(float)));
    for (size_t i = 0; i < parts.size(); ++i)
        RMU_CUDA(cudaMemcpy(tmp + i * rows_each * cols, parts[i], static_cast<size_t>(rows_each) * cols * sizeof(float), cudaMemcpyHostToDevice));
    __half *hi = nullptr, *lo = nullptr;
    int rc = dev_alloc(e->allocs, &hi, n);
    if (rc == RMU_OK) rc = dev_alloc(e->allocs, &lo, n);
    if (rc != RMU_OK) { cudaFree(tmp); return rc; }
    split_planes_kernel<<<static_cast<unsigned>((n + 255) / 256), 256>>>(tmp, hi, lo, n);
    count_launch();
    cudaError_t err = cudaDeviceSynchronize();
    cudaFree(tmp);
    if (err != cudaSuccess) { set_error(std::string("split_planes: ") + cudaGetErrorString(err)); return RMU_ERR_CUDA; }
    return make_split_operand(op, hi, lo, static_cast<int64_t>(rows), cols, /*is_activation=*/false);
}

static void free_acts(rmu_encoder* e) {
    for (void* p : e->act_allocs) cudaFree(p);
    e->act_allocs.clear();
    e->tok_cap = 0;
}

static int ensure_tokens(rmu_encoder* e, int T, int B) {
    if (T <= e->tok_cap && B + 1 <= e->seq_cap) return RMU_OK;
    RMU_CUDA(cudaDeviceSynchronize());
    free_acts(e);
    const int H = e->cfg.hidden, F = e->cfg.ffn;
    int cap = std::max(T, 1024);
    cap = (cap + 127) / 128 * 128;
    const int scap = std::max(B + 1, 1024);
    auto planes = [&](SplitOperand* op, int cols) -> int {
        __half *hi = nullptr, *lo = nullptr;
        int rc = dev_alloc(e->act_allocs, &hi, static_cast<size_t>(cap) * cols);
        if (rc == RMU_OK) rc = dev_alloc(e->act_allocs, &lo, static_cast<size_t>(cap) * cols);
        if (rc != RMU_OK) return rc;
        RMU_CUDA(cudaMemset(hi, 0, static_cast<size_t>(cap) * cols * sizeof(__half)));
        RMU_CUDA(cudaMemset(lo, 0, static_cast<size_t>(cap) * cols * sizeof(__half)));
        return make_split_operand(op, hi, lo, cap, cols, /*is_activation=*/true);
    };
    int rc = planes(&e->X, H);
    if (rc == RMU_OK) rc = planes(&e->CTX, H);
    if (rc == RMU_OK) rc = planes(&e->X1, H);
    if (rc == RMU_OK) rc = planes(&e->FF, F);
    if (rc == RMU_OK) rc = planes(&e->QKVP, 3 * H);
    if (rc == RMU_OK) {
        const int DH = H / e->cfg.heads;
        const uint64_t pitch = static_cast<uint64_t>(3) * H * sizeof(__half);
        rc = make_tmap_2d(&e->att_q_hi, e->QKVP.hi, cap, 3 * H, pitch, DH, kAtcRows, 2);
        if (rc == RMU_OK) rc = make_tmap_2d(&e->att_q_lo, e->QKVP.lo, cap, 3 * H, pitch, DH, kAtcRows, 2);
        if (rc == RMU_OK) rc = make_tmap_2d(&e->att_k_hi, e->QKVP.hi, cap, 3 * H, pitch, DH, 64, 2);
        if (rc == RMU_OK) rc = make_tmap_2d(&e->att_k_lo, e->QKVP.lo, cap, 3 * H, pitch, DH, 64, 2);
        if (rc == RMU_OK && DH == 32) {
            rc = dev_alloc(e->act_allocs, &e->QKVI, static_cast<size_t>(cap) * 6 * H);
            if (rc == RMU_OK) RMU_CUDA(cudaMemset(e->QKVI, 0, static_cast<size_t>(cap) * 6 * H * sizeof(__half)));
            if (rc == RMU_OK) rc = make_tmap_2d(&e->att_qkvi, e->QKVI, cap, 6 * H, 2 * pitch, 64, 32, 2);
        }
    }
    if (rc == RMU_OK) rc = dev_alloc(e->act_allocs, &e->PRE, static_cast<size_t>(cap) * H);
    if (rc != RMU_OK) { free_acts(e); return rc; }
    e->tok_cap = cap;
    e->seq_cap = scap;
    return RMU_OK;
}

// the encoder stack: leaves the last hidden state in e->X (split planes)
static int run_encoder(rmu_encoder* e, const int32_t* ids, const int32_t* type_ids, const int32_t* cu, int B, int T,
                       int max_seqlen, cudaStream_t st) {
    const rmu_bert_config& c = e->cfg;
    const int H = c.hidden, F = c.ffn, DH = H / c.heads;
    if (max_seqlen > c.max_pos) { set_error("sequence longer than max_position_embeddings"); return RMU_ERR_ARG; }
    int rc = ensure_tokens(e, T, B);
    if (rc != RMU_OK) return rc;
    RMU_CUDA(cudaStreamWaitEvent(st, e->ws_done, 0));    // the activation workspace is shared by all callers
    const int wpb = 8;
    const unsigned tok_blocks = static_cast<unsigned>((T + wpb - 1) / wpb);
    { ProfScope _ps(PROF_EMBED, st);
    embed_ln_kernel<<<tok_blocks, wpb * 32, 0, st>>>(ids, type_ids, cu, B, T, H, c.vocab_size, c.max_pos, c.type_vocab,
                                                     e->word, e->pos, e->typ, e->eg, e->eb, c.ln_eps, e->X.hi, e->X.lo); }
    count_launch();
    RMU_CHECK_LAUNCH();
    const float scale = 1.0f / sqrtf(static_cast<float>(DH));
    for (int l = 0; l < c.layers; ++l) {
        EncLayer& L = e->layers[l];
        GemmParams g{};
        g.M = T; g.N = 3 * H; g.K = H; g.bias = L.bqkv;
        // q (scaled by 1/sqrt(dh)), k, v leave the GEMM as split fp16 planes: attention does no conversions
        // (the softmax runs in base 2: q also carries log2(e))
        g.out_hi = e->QKVP.hi; g.out_lo = e->QKVP.lo; g.qcols = H; g.qscale = scale * 1.4426950408889634f;
        // the head-pair attention kernel reads q / k / v with hi and lo of a head interleaved in one 128-byte line
        const bool pair_attn = DH == 32 && c.heads % 2 == 0 && max_seqlen <= kApMaxKeys;
        if (pair_attn) { g.out_hi = e->QKVI; g.out_lo = nullptr; g.interleave32 = 1; }
        rc = launch_gemm(GEMM_BIAS_SPLIT_QSCALE, e->X, L.Wqkv, g, e->sms, st);
        if (rc != RMU_OK) return rc;
        {
            ProfScope _ps(PROF_ATTN, st);
            // tcgen05 attention: all keys of a sequence in one TMEM score tile (<= 256 - d_h keys) and at least two operand
            // slots in shared memory; longer sequences take the mma.sync kernel
            const int kp = (max_seqlen + 63) / 64 * 64;
            const int slot_bytes = 2 * kAtcRows * DH * 2 + 4 * kp * DH * 2;
            const int nslots = std::min(kAtcMaxSlots, (227 * 1024 - 1024 - kAtcStateBytes) / slot_bytes);
            if (pair_attn) {
                // head-pair kernel: 128-byte operand rows, K / V shared by the query-row tiles of a sequence
                ApParams ap{};
                ap.cu = cu; ap.B = B; ap.heads = c.heads; ap.H = H; ap.kp = (max_seqlen + 31) / 32 * 32;
                ap.ctx_hi = e->CTX.hi; ap.ctx_lo = e->CTX.lo;
                // no alignment pad: the dynamic shared array is declared __align__(1024) and the kernel traps if the base is not
                const size_t smem = 2 * static_cast<size_t>(4 * ap.kp * kApRowB) + 2 * kApQSlot + kApStateBytes;
                const long long nwork = static_cast<long long>(B) * (c.heads / 2);
                const unsigned grid = static_cast<unsigned>(std::min<long long>(e->sms, nwork));
                RMU_CUDA(cudaFuncSetAttribute(attention_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
                attention_pair_kernel<<<grid, kApThreads, smem, st>>>(e->att_qkvi, ap);
            } else if (max_seqlen <= kAtcBufCols - DH && nslots >= 2) {
                AtcParams ap{};
                ap.cu = cu; ap.B = B; ap.heads = c.heads; ap.H = H; ap.row_tiles = (max_seqlen + kAtcRows - 1) / kAtcRows;
                ap.kp = kp; ap.nslots = nslots; ap.ctx_hi = e->CTX.hi; ap.ctx_lo = e->CTX.lo;
                ap.nacc = (max_seqlen + 31) / 32 * 32 <= kAtcBufCols - 3 * DH ? 3 : 1;
                const size_t smem = 1024 + static_cast<size_t>(nslots) * slot_bytes + kAtcStateBytes;
                const long long nunits = static_cast<long long>(B) * ap.row_tiles * c.heads;
                const unsigned grid = static_cast<unsigned>(std::min<long long>(e->sms, nunits));
                if (DH == 32) {
                    // always the device maximum: concurrent callers (other handles, other sequence lengths) must never lower it
                    RMU_CUDA(cudaFuncSetAttribute(attention_tc_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
                    attention_tc_kernel<32><<<grid, kAtcThreads, smem, st>>>(e->att_q_hi, e->att_q_lo, e->att_k_hi, e->att_k_lo, ap);
                } else {
                    RMU_CUDA(cudaFuncSetAttribute(attention_tc_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
                    attention_tc_kernel<64><<<grid, kAtcThreads, smem, st>>>(e->att_q_hi, e->att_q_lo, e->att_k_hi, e->att_k_lo, ap);
                }
            } else {
                dim3 pg(static_cast<unsigned>(c.heads), static_cast<unsigned>(B),
                        static_cast<unsigned>((max_seqlen + kAttWarps * 16 - 1) / (kAttWarps * 16)));
                // keys resident per CTA: the whole (longest) sequence when it fits, else super-blocks of kKeySB
                const int ksb = std::min(kKeySB, (max_seqlen + 31) / 32 * 32);
                const size_t smem_max = 4 * sizeof(__half) * static_cast<size_t>(kKeySB) * (DH + 8);
                const size_t smem = 4 * sizeof(__half) * static_cast<size_t>(ksb) * (DH + 8);
                auto kern = DH == 32 ? attention_planes_kernel<32, 2> : attention_planes_kernel<64, 1>;   // d_h = 64 needs > 96 registers
                RMU_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem_max)));
                kern<<<pg, kAttWarps * 32, smem, st>>>(e->QKVP.hi, e->QKVP.lo, cu, H, ksb, e->CTX.hi, e->CTX.lo);
            }
        }
        count_launch();
        RMU_CHECK_LAUNCH();
        if (gemm_ln_supported(L.Wo, H)) {
            // attention-output projection + residual + LayerNorm in one kernel (cluster of H / 192 CTAs per row block)
            GemmLnParams gl{};
            gl.M = T; gl.N = H; gl.K = H; gl.bias = L.bo; gl.res_hi = e->X.hi; gl.res_lo = e->X.lo;
            gl.gamma = L.ln1g; gl.beta = L.ln1b; gl.eps = c.ln_eps; gl.out_hi = e->X1.hi; gl.out_lo = e->X1.lo;
            rc = launch_gemm_ln(e->CTX, L.Wo, gl, e->sms, st);
            if (rc != RMU_OK) return rc;
        } else {
            g = GemmParams{};
            g.M = T; g.N = H; g.K = H; g.bias = L.bo; g.out_f32 = e->PRE; g.res_hi = e->X.hi; g.res_lo = e->X.lo;
            rc = launch_gemm(GEMM_BIAS_RESID_F32, e->CTX, L.Wo, g, e->sms, st);
            if (rc != RMU_OK) return rc;
            { ProfScope _ps(PROF_LN, st);
            ln_kernel<<<tok_blocks, wpb * 32, 0, st>>>(e->PRE, T, H, L.ln1g, L.ln1b, c.ln_eps, e->X1.hi, e->X1.lo); }
            count_launch();
            RMU_CHECK_LAUNCH();
        }
        g = GemmParams{};
        g.M = T; g.N = F; g.K = H; g.bias = L.b1; g.out_hi = e->FF.hi; g.out_lo = e->FF.lo;
        rc = launch_gemm(GEMM_BIAS_GELU_SPLIT, e->X1, L.W1, g, e->sms, st);
        if (rc != RMU_OK) return rc;
        if (gemm_ln_supported(L.W2, H)) {
            GemmLnParams gl{};
            gl.M = T; gl.N = H; gl.K = F; gl.bias = L.b2; gl.res_hi = e->X1.hi; gl.res_lo = e->X1.lo;
            gl.gamma = L.ln2g; gl.beta = L.ln2b; gl.eps = c.ln_eps; gl.out_hi = e->X.hi; gl.out_lo = e->X.lo;
            rc = launch_gemm_ln(e->FF, L.W2, gl, e->sms, st);
            if (rc != RMU_OK) return rc;
        } else {
            g = GemmParams{};
            g.M = T; g.N = H; g.K = F; g.bias = L.b2; g.out_f32 = e->PRE; g.res_hi = e->X1.hi; g.res_lo = e->X1.lo;
            rc = launch_gemm(GEMM_BIAS_RESID_F32, e->FF, L.W2, g, e->sms, st);
            if (rc != RMU_OK) return rc;
            { ProfScope _ps(PROF_LN, st);
            ln_kernel<<<tok_blocks, wpb * 32, 0, st>>>(e->PRE, T, H, L.ln2g, L.ln2b, c.ln_eps, e->X.hi, e->X.lo); }
            count_launch();
            RMU_CHECK_LAUNCH();
        }
    }
    return RMU_OK;
}

static int check_batch(const rmu_encoder* e, const void* ids, const void* cu, int B, int T, const void* out) {
    if (!e || !ids || !cu || !out || B <= 0 || T <= 0) { set_error("encoder: bad argument"); return RMU_ERR_ARG; }
    return RMU_OK;
}

extern "C" {

int rmu_encoder_create(const rmu_bert_config* cfg, const float* const* w, int n_weights, int has_head, rmu_encoder** out) {
    if (!cfg || !w || !out) { set_error("rmu_encoder_create: bad argument"); return RMU_ERR_ARG; }
    const int H = cfg->hidden, F = cfg->ffn, L = cfg->layers;
    const int expect = 5 + 16 * L + (has_head ? 4 : 0);
    if (n_weights != expect) { set_error("rmu_encoder_create: expected " + std::to_string(expect) + " weight tensors"); return RMU_ERR_ARG; }
    if (H % 128 != 0 || F % 128 != 0 || H > 1024 || cfg->heads <= 0 || H % cfg->heads != 0 ||
        (H / cfg->heads != 32 && H / cfg->heads != 64)) {
        set_error("rmu_encoder_create: unsupported shape (hidden/ffn multiples of 128, hidden <= 1024, head_dim 32 or 64)");
        return RMU_ERR_UNSUPPORTED;
    }
    rmu_encoder* e = new rmu_encoder();
    e->cfg = *cfg;
    e->has_head = has_head;
    if (cudaGetDevice(&e->device) != cudaSuccess || (e->sms = device_sm_count()) <= 0 ||
        cudaEventCreateWithFlags(&e->ws_done, cudaEventDisableTiming) != cudaSuccess) {
        set_error("rmu_encoder_create: no CUDA device (this library has no CPU path)");
        delete e;
        return RMU_ERR_CUDA;
    }
    int rc = RMU_OK;
    int i = 0;
    auto up = [&](float** dst, size_t n) { if (rc == RMU_OK) rc = upload(e, dst, w[i], n); ++i; };
    up(&e->word, static_cast<size_t>(cfg->vocab_size) * H);
    up(&e->pos, static_cast<size_t>(cfg->max_pos) * H);
    up(&e->typ, static_cast<size_t>(cfg->type_vocab) * H);
    up(&e->eg, H);
    up(&e->eb, H);
    e->layers.resize(L);
    for (int l = 0; l < L && rc == RMU_OK; ++l) {
        EncLayer& Ly = e->layers[l];
        const float *qw = w[i], *qb = w[i + 1], *kw = w[i + 2], *kb = w[i + 3], *vw = w[i + 4], *vb = w[i + 5];
        i += 6;
        rc = upload_split(e, &Ly.Wqkv, {qw, kw, vw}, H, H);
        if (rc == RMU_OK) {
            std::vector<float> bcat(3 * static_cast<size_t>(H));
            std::copy(qb, qb + H, bcat.begin());
            std::copy(kb, kb + H, bcat.begin() + H);
            std::copy(vb, vb + H, bcat.begin() + 2 * H);
            rc = upload(e, &Ly.bqkv, bcat.data(), bcat.size());
        }
        if (rc == RMU_OK) rc = upload_split(e, &Ly.Wo, {w[i]}, H, H);
        ++i;
        up(&Ly.bo, H);
        up(&Ly.ln1g, H);
        up(&Ly.ln1b, H);
        if (rc == RMU_OK) rc = upload_split(e, &Ly.W1, {w[i]}, F, H);
        ++i;
        up(&Ly.b1, F);
        if (rc == RMU_OK) rc = upload_split(e, &Ly.W2, {w[i]}, H, F);
        ++i;
        up(&Ly.b2, H);
        up(&Ly.ln2g, H);
        up(&Ly.ln2b, H);
    }
    if (has_head) {
        up(&e->pw, static_cast<size_t>(H) * H);
        up(&e->pb, H);
        up(&e->cw, static_cast<size_t>(cfg->num_labels) * H);
        up(&e->cb, cfg->num_labels);
    }
    if (rc != RMU_OK) { rmu_encoder_destroy(e); return rc; }
    *out = e;
    return RMU_OK;
}

void rmu_encoder_destroy(rmu_encoder* e) {
    if (!e) return;
    cudaDeviceSynchronize();
    free_acts(e);
    cudaFree(e->d_ids); cudaFree(e->d_typ); cudaFree(e->d_cu); cudaFree(e->d_out);
    for (void* p : e->allocs) cudaFree(p);
    if (e->ws_done) cudaEventDestroy(e->ws_done);
    delete e;
}

int rmu_encoder_embed(rmu_encoder* e, const int32_t* ids, const int32_t* type_ids, const int32_t* cu, int B, int T,
                      int max_seqlen, int pool_mode, int normalize, float* out, void* stream) {
    int rc = check_batch(e, ids, cu, B, T, out);
    if (rc != RMU_OK) return rc;
    if (pool_mode != RMU_POOL_MEAN && pool_mode != RMU_POOL_CLS) { set_error("bad pool_mode"); return RMU_ERR_ARG; }
    std::lock_guard<std::mutex> g(e->mu);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    rc = run_encoder(e, ids, type_ids, cu, B, T, max_seqlen, st);
    if (rc != RMU_OK) return rc;
    ProfScope _ps(PROF_POOL_HEAD, st);
    pool_kernel<<<B, 256, 0, st>>>(e->X.hi, e->X.lo, cu, e->cfg.hidden, pool_mode, normalize, out);
    count_launch();
    RMU_CHECK_LAUNCH();
    RMU_CUDA(cudaEventRecord(e->ws_done, st));
    return RMU_OK;
}

int rmu_encoder_classify(rmu_encoder* e, const int32_t* ids, const int32_t* type_ids, const int32_t* cu, int B, int T,
                         int max_seqlen, float* out, void* stream) {
    int rc = check_batch(e, ids, cu, B, T, out);
    if (rc != RMU_OK) return rc;
    if (!e->has_head) { set_error("rmu_encoder_classify: encoder was created without a classification head"); return RMU_ERR_ARG; }
    std::lock_guard<std::mutex> g(e->mu);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    rc = run_encoder(e, ids, type_ids, cu, B, T, max_seqlen, st);
    if (rc != RMU_OK) return rc;
    const int H = e->cfg.hidden;
    ProfScope _ps(PROF_POOL_HEAD, st);
    cls_head_kernel<<<B, 256, 2 * H * sizeof(float), st>>>(e->X.hi, e->X.lo, cu, H, e->cfg.num_labels, e->pw, e->pb,
                                                            e->cw, e->cb, out);
    count_launch();
    RMU_CHECK_LAUNCH();
    RMU_CUDA(cudaEventRecord(e->ws_done, st));
    return RMU_OK;
}

int rmu_encoder_hidden(rmu_encoder* e, const int32_t* ids, const int32_t* type_ids, const int32_t* cu, int B, int T,
                       int max_seqlen, float* out, void* stream) {
    int rc = check_batch(e, ids, cu, B, T, out);
    if (rc != RMU_OK) return rc;
    std::lock_guard<std::mutex> g(e->mu);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    rc = run_encoder(e, ids, type_ids, cu, B, T, max_seqlen, st);
    if (rc != RMU_OK) return rc;
    const size_t n = static_cast<size_t>(T) * e->cfg.hidden;
    join_planes_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(e->X.hi, e->X.lo, out, n);
    count_launch();
    RMU_CHECK_LAUNCH();
    RMU_CUDA(cudaEventRecord(e->ws_done, st));
    return RMU_OK;
}

// host_mu held: the staging buffers belong to the *_host entry points only
static int stage_batch(rmu_encoder* e, const int32_t* ids_h, const int32_t* typ_h, const int32_t* cu_h, int B, int T,
                       cudaStream_t st) {
    if (T > e->stage_tok_cap || B + 1 > e->stage_seq_cap) {
        RMU_CUDA(cudaStreamSynchronize(st));              // earlier *_host calls on this stream are complete (they synchronise)
        cudaFree(e->d_ids); cudaFree(e->d_typ); cudaFree(e->d_cu); cudaFree(e->d_out);
        e->d_ids = e->d_typ = e->d_cu = nullptr; e->d_out = nullptr;
        e->stage_tok_cap = e->stage_seq_cap = 0;
        const int cap = (std::max(T, 1024) + 127) / 128 * 128, scap = std::max(B + 1, 1024);
        RMU_CUDA(cudaMalloc(reinterpret_cast<void**>(&e->d_ids), static_cast<size_t>(cap) * sizeof(int)));
        RMU_CUDA(cudaMalloc(reinterpret_cast<void**>(&e->d_typ), static_cast<size_t>(cap) * sizeof(int)));
        RMU_CUDA(cudaMalloc(reinterpret_cast<void**>(&e->d_cu), static_cast<size_t>(scap) * sizeof(int)));
        RMU_CUDA(cudaMalloc(reinterpret_cast<void**>(&e->d_out), static_cast<size_t>(scap) * std::max(e->cfg.hidden, e->cfg.num_labels) * sizeof(float)));
        e->stage_tok_cap = cap;
        e->stage_seq_cap = scap;
    }
    RMU_CUDA(cudaMemcpyAsync(e->d_ids, ids_h, static_cast<size_t>(T) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    if (typ_h) RMU_CUDA(cudaMemcpyAsync(e->d_typ, typ_h, static_cast<size_t>(T) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    RMU_CUDA(cudaMemcpyAsync(e->d_cu, cu_h, static_cast<size_t>(B + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    return RMU_OK;
}

int rmu_encoder_embed_host(rmu_encoder* e, const int32_t* ids_h, const int32_t* typ_h, const int32_t* cu_h, int B, int T,
                           int max_seqlen, int pool_mode, int normalize, float* out_h, void* stream) {
    int rc = check_batch(e, ids_h, cu_h, B, T, out_h);
    if (rc != RMU_OK) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    std::lock_guard<std::mutex> hg(e->host_mu);
    rc = stage_batch(e, ids_h, typ_h, cu_h, B, T, st);
    if (rc != RMU_OK) return rc;
    rc = rmu_encoder_embed(e, e->d_ids, typ_h ? e->d_typ : nullptr, e->d_cu, B, T, max_seqlen, pool_mode, normalize, e->d_out, st);
    if (rc != RMU_OK) return rc;
    RMU_CUDA(cudaMemcpyAsync(out_h, e->d_out, static_cast<size_t>(B) * e->cfg.hidden * sizeof(float), cudaMemcpyDeviceToHost, st));
    RMU_CUDA(cudaStreamSynchronize(st));
    return RMU_OK;
}

int rmu_encoder_classify_host(rmu_encoder* e, const int32_t* ids_h, const int32_t* typ_h, const int32_t* cu_h, int B,
                              int T, int max_seqlen, float* out_h, void* stream) {
    int rc = check_batch(e, ids_h, cu_h, B, T, out_h);
    if (rc != RMU_OK) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    std::lock_guard<std::mutex> hg(e->host_mu);
    rc = stage_batch(e, ids_h, typ_h, cu_h, B, T, st);
    if (rc != RMU_OK) return rc;
    rc = rmu_encoder_classify(e, e->d_ids, typ_h ? e->d_typ : nullptr, e->d_cu, B, T, max_seqlen, e->d_out, st);
    if (rc != RMU_OK) return rc;
    RMU_CUDA(cudaMemcpyAsync(out_h, e->d_out, static_cast<size_t>(B) * e->cfg.num_labels * sizeof(float), cudaMemcpyDeviceToHost, st));
    RMU_CUDA(cudaStreamSynchronize(st));
    return RMU_OK;
}

}  // extern "C"
