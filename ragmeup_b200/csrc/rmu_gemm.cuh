// fp32-accurate GEMM on the 16-bit tensor path of sm_100a.
//
//   C[M,N] = A[M,K] * W[N,K]^T      (both operands K-major, as nn.Linear stores W)
//
// The reference runs these contractions in fp32 (torch nn.Linear inside transformers' BertModel;
// SURVEY.md H3/H9) and BASELINE.json demands 1e-3 parity on logits, which neither TF32 nor bf16
// operands hold on trained-like weights (measured in DESIGN.md).  Operands are therefore carried as
// SPLIT fp16 PLANES, v = hi + lo with hi = fp16(v), lo = fp16(v - hi) (22 mantissa bits), and each
// K step issues three tcgen05.mma kind::f16: hi*hi + lo*hi + hi*lo, fp32 accumulate in TMEM.
//
// Kernel shape: persistent, 1 CTA/SM, 192 threads = TMA producer warp, MMA issuer warp (one lane)
// + TMEM allocator, 8 epilogue warps.  128x128 output tiles, K blocks of 64 (one 128-byte swizzled
// row per operand row), 3-stage smem ring (4 planes x 16 KB per stage), two TMEM accumulator
// buffers so the epilogue of tile i overlaps the MMAs of tile i+1.
#pragma once
#include "rmu_common.h"
#include "rmu_ptx.cuh"

namespace rmu {

constexpr int kGemmBM = 128, kGemmBK = 64;
constexpr int kGemmPlaneBytes = 128 * 128;                 // one A plane of a stage: 128 rows x 128 B
constexpr int kGemmEpiWarps = 8;                           // two per TMEM lane quadrant, each takes half the columns
constexpr int kGemmThreads = 64 + 32 * kGemmEpiWarps;      // + TMA producer warp + MMA issuer warp
constexpr int kGemmStageRow = 33;                          // padded row of the per-warp [32][32] staging tile
constexpr size_t kGemmStagingBytes = static_cast<size_t>(kGemmEpiWarps) * 32 * kGemmStageRow * sizeof(float);
constexpr size_t kGemmSmem = 196608 + kGemmStagingBytes + 256 + 1024;   // stages never exceed 192 KB

enum GemmMode {
    GEMM_BIAS_GELU_SPLIT = 1, // out planes = split(gelu_erf(acc + bias))
    GEMM_BIAS_RESID_F32 = 2,  // out_f32 = acc + bias + (res_hi + res_lo)
    GEMM_BIAS_SPLIT_QSCALE = 3, // out planes = split((acc + bias) * (col < qcols ? qscale : 1))   (QKV projection)
};

struct GemmParams {
    int M, N, K;
    const float* bias;                    // [N]
    float* out_f32;                       // [M, N]
    __half* out_hi; __half* out_lo;       // [M, N]
    const __half* res_hi; const __half* res_lo;  // [M, N]
    int qcols; float qscale;              // GEMM_BIAS_SPLIT_QSCALE
    int interleave32;                     // GEMM_BIAS_SPLIT_QSCALE: out_hi is ONE buffer [M, 2N] where every 32-column group
                                          // (a d_h = 32 head) is stored as 32 hi halves followed by its 32 lo halves: a head's
                                          // q / k / v row is one 128-byte line (what attention_pair_kernel's TMA boxes fetch)
};

__device__ __forceinline__ void split_f16(float v, __half& hi, __half& lo) {
    hi = __float2half_rn(v);
    lo = __float2half_rn(v - __half2float(hi));
}

// erf by Abramowitz & Stegun 7.1.26 (|error| <= 1.5e-7, the fp32 noise floor of the erf-GELU the
// reference computes with torch.erf) on the fast exp / reciprocal units: the FFN-in epilogue is ALU-bound.
__device__ __forceinline__ float erf_as(float x) {
    const float ax = fabsf(x);
    const float t = __fdividef(1.0f, fmaf(0.3275911f, ax, 1.0f));
    float p = fmaf(1.061405429f, t, -1.453152027f);
    p = fmaf(p, t, 1.421413741f);
    p = fmaf(p, t, -0.284496736f);
    p = fmaf(p, t, 0.254829592f);
    const float y = 1.0f - p * t * __expf(-ax * ax);
    return copysignf(y, x);
}
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erf_as(x * 0.70710678118654752440f)); }

// Packed fp32 pairs (FFMA2 / FMUL2 / FADD2 of sm_100): one issue slot for a lane's two adjacent output columns.  The
// FFN-in epilogue is issue-bound (ncu: 74 % of issue slots, 42 instructions per output element before this), not
// FMA-pipe bound, so halving the count of its fp32 instructions is what pays.
__device__ __forceinline__ float2 f2_fma(float2 a, float2 b, float2 c) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
        "fma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return d;
}
__device__ __forceinline__ float2 f2_mul(float2 a, float2 b) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
        "mul.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}
__device__ __forceinline__ float2 f2_add(float2 a, float2 b) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
        "add.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}
__device__ __forceinline__ float2 f2_sub(float2 a, float2 b) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
        "sub.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}
__device__ __forceinline__ float2 f2_splat(float v) { return make_float2(v, v); }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// gelu_erf of two values: the same A&S 7.1.26 polynomial; the minus sign of 1 - p t e is folded into the coefficients
__device__ __forceinline__ float2 gelu_erf2(float2 v) {
    const float2 x = f2_mul(v, f2_splat(0.70710678118654752440f));
    const float2 ax = make_float2(fabsf(x.x), fabsf(x.y));
    const float2 d = f2_fma(ax, f2_splat(0.3275911f), f2_splat(1.0f));
    const float2 t = make_float2(rcp_approx(d.x), rcp_approx(d.y));
    float2 q = f2_fma(t, f2_splat(-1.061405429f), f2_splat(1.453152027f));      // -p
    q = f2_fma(q, t, f2_splat(-1.421413741f));
    q = f2_fma(q, t, f2_splat(0.284496736f));
    q = f2_fma(q, t, f2_splat(-0.254829592f));
    q = f2_mul(q, t);                                                           // -p t
    float2 e = f2_mul(f2_mul(ax, ax), f2_splat(-1.4426950408889634f));          // exp(-x^2) = 2^(-x^2 log2 e)
    e = make_float2(ex2_approx(e.x), ex2_approx(e.y));
    const float2 y = f2_fma(q, e, f2_splat(1.0f));                              // |erf|
    const float2 er = make_float2(copysignf(y.x, x.x), copysignf(y.y, x.y));
    const float2 h = f2_mul(v, f2_splat(0.5f));
    return f2_fma(h, er, h);
}
// (a, b) -> fp16 pair of the high parts and fp16 pair of the residuals
__device__ __forceinline__ void split_f16x2(float2 v, __half2& hi, __half2& lo) {
    hi = __floats2half2_rn(v.x, v.y);
    const float2 r = f2_sub(v, __half22float2(hi));
    lo = __floats2half2_rn(r.x, r.y);
}

// BN = output-tile width (MMA N): 128 (3 stages of 64 KB), 192 (2 x 80 KB) or 256 (2 x 96 KB).  Wider tiles read
// the A slab once for more columns: L2->SM bytes per MMA cycle 85 -> 69 -> 62, smem operand reads 128 -> 104 -> 94.
// The erf-GELU epilogue (FFN-in) is ALU / issue bound: with 192-wide tiles it runs 12 epilogue warps (three per
// TMEM lane quadrant, two column chunks each) instead of 8.
template <int MODE, int BN>
__host__ __device__ constexpr int gemm_epi_warps() { return (MODE == GEMM_BIAS_GELU_SPLIT && BN == 192) ? 12 : kGemmEpiWarps; }

template <int MODE, int BN>
__global__ void __launch_bounds__(64 + 32 * gemm_epi_warps<MODE, BN>(), 1)
gemm_f16x3_kernel(const __grid_constant__ CUtensorMap tAh, const __grid_constant__ CUtensorMap tAl,
                  const __grid_constant__ CUtensorMap tWh, const __grid_constant__ CUtensorMap tWl,
                  const GemmParams p) {
    constexpr uint32_t IDESC = umma_idesc(0 /*f16*/, kGemmBM, BN);
    constexpr int kGemmBN = BN;
    constexpr int kGemmStages = BN == 128 ? 3 : 2;
    constexpr int kWPlane = BN * 128;                              // one W plane of a stage
    constexpr int kGemmStageBytes = 2 * kGemmPlaneBytes + 2 * kWPlane;
    constexpr int kTmemCols = BN == 128 ? 256 : 512;
    constexpr int kEpi = gemm_epi_warps<MODE, BN>();
    constexpr int kChunksPerWarp = (BN / 32) / (kEpi / 4);
    constexpr size_t kStagingBytes = static_cast<size_t>(kEpi) * 32 * kGemmStageRow * sizeof(float);
    static_assert(static_cast<size_t>(kGemmStages) * kGemmStageBytes + kStagingBytes + 256 + 1024 <= kGemmSmem, "smem budget");
    extern __shared__ uint8_t gemm_smem_raw[];
    // 1024-byte alignment by OFFSET into the shared array: a pointer round-trip through an integer would lose the
    // shared address space and turn every staging access into a generic LD/ST
    uint8_t* smem = gemm_smem_raw + ((1024u - (smem_u32(gemm_smem_raw) & 1023u)) & 1023u);
    float* staging = reinterpret_cast<float*>(smem + kGemmStages * kGemmStageBytes);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + kGemmStages * kGemmStageBytes + kStagingBytes);
    uint64_t* empty = full + kGemmStages;
    uint64_t* acc_full = empty + kGemmStages;
    uint64_t* acc_empty = acc_full + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

    const int warp = threadIdx.x >> 5;
    const unsigned lane = lane_id();
    if (threadIdx.x == 0) {
        for (int i = 0; i < kGemmStages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 32 * kEpi); }
        fence_mbar_init();
        prefetch_tmap(&tAh); prefetch_tmap(&tAl); prefetch_tmap(&tWh); prefetch_tmap(&tWl);
    }
    if (warp == 1) tmem_alloc<kTmemCols>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int m_blks = (p.M + kGemmBM - 1) / kGemmBM;
    const int n_blks = p.N / kGemmBN;
    const int k_blks = p.K / kGemmBK;
    const int tiles = m_blks * n_blks;

    if (warp == 0) {
        if (elect_one()) {
            int slot = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
                const int mb = tile / n_blks, nb = tile % n_blks;
                for (int kb = 0; kb < k_blks; ++kb) {
                    mbar_wait(&empty[slot], phase ^ 1);
                    uint8_t* st = smem + slot * kGemmStageBytes;
                    mbar_arrive_expect_tx(&full[slot], kGemmStageBytes);
                    tma_load_2d(st, &tAh, kb * kGemmBK, mb * kGemmBM, &full[slot], kEvictNormal);
                    tma_load_2d(st + kGemmPlaneBytes, &tAl, kb * kGemmBK, mb * kGemmBM, &full[slot], kEvictNormal);
                    tma_load_2d(st + 2 * kGemmPlaneBytes, &tWh, kb * kGemmBK, nb * kGemmBN, &full[slot], kEvictLast);
                    tma_load_2d(st + 2 * kGemmPlaneBytes + kWPlane, &tWl, kb * kGemmBK, nb * kGemmBN, &full[slot], kEvictLast);
                    if (++slot == kGemmStages) { slot = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (elect_one()) {
            int slot = 0;
            uint32_t phase = 0;
            int i = 0;
            for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++i) {
                const int buf = i & 1;
                const uint32_t use = static_cast<uint32_t>(i >> 1);
                mbar_wait(&acc_empty[buf], (use & 1) ^ 1);
                tc_fence_after();
                const uint32_t d_addr = tmem_base + buf * kGemmBN;
                for (int kb = 0; kb < k_blks; ++kb) {
                    mbar_wait(&full[slot], phase);
                    tc_fence_after();
                    const uint32_t sbase = smem_u32(smem + slot * kGemmStageBytes);
                    const uint64_t dAh = umma_desc_sw128_kmajor(sbase);
                    const uint64_t dAl = umma_desc_sw128_kmajor(sbase + kGemmPlaneBytes);
                    const uint64_t dWh = umma_desc_sw128_kmajor(sbase + 2 * kGemmPlaneBytes);
                    const uint64_t dWl = umma_desc_sw128_kmajor(sbase + 2 * kGemmPlaneBytes + kWPlane);
#pragma unroll
                    for (int k = 0; k < kGemmBK / 16; ++k) {
                        const uint64_t off = static_cast<uint64_t>(k * 2);   // 16 halves = 32 B = 2 x 16 B units
                        mma_f16_ss(d_addr, dAh + off, dWh + off, IDESC, (kb | k) != 0 ? 1u : 0u);
                        mma_f16_ss(d_addr, dAl + off, dWh + off, IDESC, 1u);
                        mma_f16_ss(d_addr, dAh + off, dWl + off, IDESC, 1u);
                    }
                    tc_commit(&empty[slot]);
                    if (++slot == kGemmStages) { slot = 0; phase ^= 1; }
                }
                tc_commit(&acc_full[buf]);
            }
        }
    } else {
        // ---- epilogue: warp (2 + ew) reads TMEM lanes of quadrant (warp & 3); ew < 4 takes column chunks 0-1
        //      of the tile, ew >= 4 chunks 2-3.  Values are staged through a per-warp smem tile so that every
        //      global access (output rows, residual rows) is a fully used, coalesced row segment.
        const int ew = warp - 2;
        const int quad = warp & 3;
        const int chalf = ew >> 2;
        float* stg = staging + ew * (32 * kGemmStageRow);
        const int rsub = static_cast<int>(lane) >> 4, cp = (static_cast<int>(lane) & 15) * 2;
        int i = 0;
        for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++i) {
            const int mb = tile / n_blks, nb = tile % n_blks;
            const int buf = i & 1;
            const uint32_t use = static_cast<uint32_t>(i >> 1);
            mbar_wait(&acc_full[buf], use & 1);
            tc_fence_after();
            const int row_base = mb * kGemmBM + quad * 32;
#pragma unroll 1
            for (int cc = 0; cc < kChunksPerWarp; ++cc) {
                const int c = chalf * kChunksPerWarp + cc;
                const int col0 = nb * kGemmBN + c * 32;
                // residual rows of this chunk: issued first so their latency hides behind the TMEM read
                __half2 rsh[16], rsl[16];
                if (MODE == GEMM_BIAS_RESID_F32) {
#pragma unroll
                    for (int q = 0; q < 16; ++q) {
                        const int grow = row_base + 2 * q + rsub;
                        if (grow < p.M) {
                            const size_t o = static_cast<size_t>(grow) * p.N + col0 + cp;
                            rsh[q] = *reinterpret_cast<const __half2*>(p.res_hi + o);
                            rsl[q] = *reinterpret_cast<const __half2*>(p.res_lo + o);
                        }
                    }
                }
                const float2 bia2 = __ldg(reinterpret_cast<const float2*>(p.bias + col0 + cp));
                uint32_t r[32];
                tmem_ld32(tmem_addr(tmem_base, quad * 32, buf * kGemmBN + c * 32), r);
                tmem_ld_wait();
                if (cc == kChunksPerWarp - 1) {      // last TMEM read of this warp for the tile
                    tc_fence_before();
                    mbar_arrive(&acc_empty[buf]);
                }
                const float sc = (MODE == GEMM_BIAS_SPLIT_QSCALE && col0 < p.qcols) ? p.qscale : 1.0f;
#pragma unroll
                for (int j = 0; j < 32; ++j) stg[lane * kGemmStageRow + j] = __uint_as_float(r[j]);
                __syncwarp();
#pragma unroll
                for (int rr = 0; rr < 32; rr += 2) {
                    const int rl = rr + rsub;
                    const int grow = row_base + rl;
                    if (grow < p.M) {
                        // lane = column pair: the bias is a per-lane constant of the chunk
                        float2 v = f2_add(make_float2(stg[rl * kGemmStageRow + cp], stg[rl * kGemmStageRow + cp + 1]), bia2);
                        if (MODE == GEMM_BIAS_GELU_SPLIT) v = gelu_erf2(v);
                        if (MODE == GEMM_BIAS_SPLIT_QSCALE) v = f2_mul(v, f2_splat(sc));
                        const size_t o = static_cast<size_t>(grow) * p.N + col0 + cp;
                        if (MODE == GEMM_BIAS_RESID_F32)
                            v = f2_add(v, f2_add(__half22float2(rsh[rr >> 1]), __half22float2(rsl[rr >> 1])));
                        if (MODE == GEMM_BIAS_RESID_F32) {
                            *reinterpret_cast<float2*>(p.out_f32 + o) = v;
                        } else {
                            __half2 h2, l2;
                            split_f16x2(v, h2, l2);
                            if (MODE == GEMM_BIAS_SPLIT_QSCALE && p.interleave32) {
                                const size_t oi = static_cast<size_t>(grow) * (2 * p.N) + 2 * col0 + cp;   // col0 is a multiple of 32
                                *reinterpret_cast<__half2*>(p.out_hi + oi) = h2;
                                *reinterpret_cast<__half2*>(p.out_hi + oi + 32) = l2;
                            } else {
                                *reinterpret_cast<__half2*>(p.out_hi + o) = h2;
                                *reinterpret_cast<__half2*>(p.out_lo + o) = l2;
                            }
                        }
                    }
                }
                __syncwarp();
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 1) tmem_dealloc<kTmemCols>(tmem_base);
}


// ---------------------------------------------------------------------------------------------------
// GEMM + bias + residual + LayerNorm -> split planes in ONE kernel (attention-output and FFN-output
// projections of a post-LN BERT block: transformers BertSelfOutput / BertOutput, modeling_bert.py:287-357).
//
// A LayerNorm row spans the whole N = hidden, i.e. CL = N / 192 output tiles.  The CL CTAs of a thread-block
// CLUSTER take the CL column tiles of the same 128-row block at the same time; every epilogue warp computes
// (mean, M2) of its 96 columns of y = acc + bias + residual per row, publishes them into the shared memory of
// all CL CTAs (st.async whose completion bytes are credited to the destination CTA's mbarrier), and each CTA combines the 2*CL partials per row
// with Chan's parallel-variance formula (exact two-pass statistics, no E[x^2] - E[x]^2 cancellation).  y never
// leaves the SM: it is written back into the TMEM accumulator columns between the passes.  Compared with
// GEMM(RESID_F32) + ln_kernel this removes one fp32 write and one fp32 read of [M, N] per LayerNorm.
// ---------------------------------------------------------------------------------------------------
struct GemmLnParams {
    int M, N, K;
    const float* bias;                            // [N]
    const __half* res_hi; const __half* res_lo;   // [M, N] residual stream (planes)
    const float* gamma; const float* beta;        // [N]
    float eps;
    __half* out_hi; __half* out_lo;               // [M, N] LayerNorm output (planes)
};

constexpr int kLnBN = 192;
constexpr int kLnMaxCL = 4;                       // hidden <= 768
constexpr int kLnStages = 2;
constexpr int kLnStageBytes = 2 * kGemmPlaneBytes + 2 * kLnBN * 128;
// 12 epilogue warps only with clusters of 2 (hidden 384): 6 column slices; 8 warps: up to 2 * kLnMaxCL = 8 slices
__host__ __device__ constexpr int ln_max_parts(int epi_warps) { return epi_warps == 12 ? 6 : 2 * kLnMaxCL; }
__host__ __device__ constexpr size_t ln_stats_bytes(int epi_warps) { return 2ull * ln_max_parts(epi_warps) * kGemmBM * sizeof(float2); }
__host__ __device__ constexpr size_t ln_staging_bytes(int epi_warps) { return static_cast<size_t>(epi_warps) * 32 * kGemmStageRow * sizeof(float); }
constexpr size_t kLnVecBytes = 3 * kLnBN * sizeof(float);      // this CTA's bias | gamma | beta columns
__host__ __device__ constexpr size_t ln_smem_bytes(int epi_warps) {
    return static_cast<size_t>(kLnStages) * kLnStageBytes + ln_staging_bytes(epi_warps) + ln_stats_bytes(epi_warps) + kLnVecBytes + 256 + 1024;
}
static_assert(ln_smem_bytes(8) <= 232448 && ln_smem_bytes(12) <= 232448, "shared memory budget");

template <int EPI_WARPS>      // 8 (two warps per TMEM lane quadrant, 96 columns each) or 12 (three, 64 columns each; clusters of 2)
__global__ void __launch_bounds__(64 + 32 * EPI_WARPS, 1)
gemm_f16x3_ln_kernel(const __grid_constant__ CUtensorMap tAh, const __grid_constant__ CUtensorMap tAl,
                     const __grid_constant__ CUtensorMap tWh, const __grid_constant__ CUtensorMap tWl,
                     const GemmLnParams p) {
    static_assert(EPI_WARPS == 8 || EPI_WARPS == 12, "two or three epilogue warps per TMEM lane quadrant");
    constexpr int kWQ = EPI_WARPS / 4;            // warps per lane quadrant = column slices (parts) per CTA
    constexpr int kChunks = 6 / kWQ;              // 32-column chunks per warp
    constexpr size_t kStagingBytes = ln_staging_bytes(EPI_WARPS);
    constexpr int kMaxParts = ln_max_parts(EPI_WARPS);
    constexpr uint32_t IDESC = umma_idesc(0 /*f16*/, kGemmBM, kLnBN);
    constexpr int kWPlane = kLnBN * 128;
    constexpr int kPartCols = kLnBN / kWQ;        // columns per epilogue warp
    extern __shared__ uint8_t gemm_smem_raw[];
    // 1024-byte alignment by OFFSET into the shared array: a pointer round-trip through an integer would lose the
    // shared address space and turn every staging access into a generic LD/ST
    uint8_t* smem = gemm_smem_raw + ((1024u - (smem_u32(gemm_smem_raw) & 1023u)) & 1023u);
    float* staging = reinterpret_cast<float*>(smem + kLnStages * kLnStageBytes);
    float2* stats = reinterpret_cast<float2*>(smem + kLnStages * kLnStageBytes + kStagingBytes);   // [2][2*CLmax][128]
    // bias | gamma | beta of this CTA's 192 columns: the cluster-scope acquire of every tile invalidates L1, so
    // re-reading them from global memory would miss each time
    float* svec = reinterpret_cast<float*>(smem + kLnStages * kLnStageBytes + kStagingBytes + ln_stats_bytes(EPI_WARPS));
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + kLnStages * kLnStageBytes + kStagingBytes + ln_stats_bytes(EPI_WARPS) + kLnVecBytes);
    uint64_t* empty = full + kLnStages;
    uint64_t* acc_full = empty + kLnStages;
    uint64_t* acc_empty = acc_full + 2;
    uint64_t* stat_full = acc_empty + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(stat_full + 2);

    const int warp = threadIdx.x >> 5;
    const unsigned lane = lane_id();
    const uint32_t CL = cluster_nctarank();
    const uint32_t rank = cluster_ctarank();
    if (threadIdx.x == 0) {
        for (int i = 0; i < kLnStages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&acc_full[i], 1);
            mbar_init(&acc_empty[i], 32 * EPI_WARPS);
            mbar_init(&stat_full[i], 1);                        // armed per tile with the bytes of all 2*CL column slices
        }
        fence_mbar_init();
        prefetch_tmap(&tAh); prefetch_tmap(&tAl); prefetch_tmap(&tWh); prefetch_tmap(&tWl);
    }
    if (warp == 1) tmem_alloc<512>(tmem_slot);
    for (int j = threadIdx.x; j < kLnBN; j += blockDim.x) {
        const int col = static_cast<int>(cluster_ctarank()) * kLnBN + j;
        svec[j] = p.bias[col];
        svec[kLnBN + j] = p.gamma[col];
        svec[2 * kLnBN + j] = p.beta[col];
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                           // every CTA's barriers exist before any remote arrive
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int m_blks = (p.M + kGemmBM - 1) / kGemmBM;
    const int k_blks = p.K / kGemmBK;
    const int cluster_id = blockIdx.x / CL, n_clusters = gridDim.x / CL;
    const int nb = static_cast<int>(rank);        // this CTA's column tile of every row block

    if (warp == 0) {
        if (elect_one()) {
            int slot = 0;
            uint32_t phase = 0;
            for (int mb = cluster_id; mb < m_blks; mb += n_clusters) {
                for (int kb = 0; kb < k_blks; ++kb) {
                    mbar_wait(&empty[slot], phase ^ 1);
                    uint8_t* st = smem + slot * kLnStageBytes;
                    mbar_arrive_expect_tx(&full[slot], kLnStageBytes);
                    tma_load_2d(st, &tAh, kb * kGemmBK, mb * kGemmBM, &full[slot], kEvictNormal);
                    tma_load_2d(st + kGemmPlaneBytes, &tAl, kb * kGemmBK, mb * kGemmBM, &full[slot], kEvictNormal);
                    tma_load_2d(st + 2 * kGemmPlaneBytes, &tWh, kb * kGemmBK, nb * kLnBN, &full[slot], kEvictLast);
                    tma_load_2d(st + 2 * kGemmPlaneBytes + kWPlane, &tWl, kb * kGemmBK, nb * kLnBN, &full[slot], kEvictLast);
                    if (++slot == kLnStages) { slot = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (elect_one()) {
            int slot = 0;
            uint32_t phase = 0;
            int i = 0;
            for (int mb = cluster_id; mb < m_blks; mb += n_clusters, ++i) {
                const int buf = i & 1;
                const uint32_t use = static_cast<uint32_t>(i >> 1);
                mbar_wait(&acc_empty[buf], (use & 1) ^ 1);
                tc_fence_after();
                const uint32_t d_addr = tmem_base + buf * kLnBN;
                for (int kb = 0; kb < k_blks; ++kb) {
                    mbar_wait(&full[slot], phase);
                    tc_fence_after();
                    const uint32_t sbase = smem_u32(smem + slot * kLnStageBytes);
                    const uint64_t dAh = umma_desc_sw128_kmajor(sbase);
                    const uint64_t dAl = umma_desc_sw128_kmajor(sbase + kGemmPlaneBytes);
                    const uint64_t dWh = umma_desc_sw128_kmajor(sbase + 2 * kGemmPlaneBytes);
                    const uint64_t dWl = umma_desc_sw128_kmajor(sbase + 2 * kGemmPlaneBytes + kWPlane);
#pragma unroll
                    for (int k = 0; k < kGemmBK / 16; ++k) {
                        const uint64_t off = static_cast<uint64_t>(k * 2);
                        mma_f16_ss(d_addr, dAh + off, dWh + off, IDESC, (kb | k) != 0 ? 1u : 0u);
                        mma_f16_ss(d_addr, dAl + off, dWh + off, IDESC, 1u);
                        mma_f16_ss(d_addr, dAh + off, dWl + off, IDESC, 1u);
                    }
                    tc_commit(&empty[slot]);
                    if (++slot == kLnStages) { slot = 0; phase ^= 1; }
                }
                tc_commit(&acc_full[buf]);
            }
        }
    } else {
        // ---- epilogue warp (quad, chalf): rows quad*32 .. +32 of the tile (thread = row in TMEM), columns
        //      chalf*96 .. +96 of the tile.  part = rank*2 + chalf identifies its 96-column slice of the LN row.
        const int ew = warp - 2;
        const int quad = warp & 3;
        const int chalf = ew >> 2;
        const int part = static_cast<int>(rank) * kWQ + chalf;
        const int nparts = kWQ * static_cast<int>(CL);
        float* stg = staging + ew * (32 * kGemmStageRow);
        const int rsub = static_cast<int>(lane) >> 4, cp = (static_cast<int>(lane) & 15) * 2;
        const int trow = quad * 32 + static_cast<int>(lane);           // this thread's row of the tile
        const float inv_n = 1.0f / static_cast<float>(p.N);
        // residual rows of chunk (chalf*3 + cc), coalesced: lane = column pair, 16 row pairs
        auto load_res = [&](int row_base_, int cc_, __half2 (&h)[16], __half2 (&l)[16]) {
            const int col0_ = nb * kLnBN + (chalf * kChunks + cc_) * 32;
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const int grow = row_base_ + 2 * q + rsub;
                if (grow < p.M) {
                    const size_t o = static_cast<size_t>(grow) * p.N + col0_ + cp;
                    h[q] = *reinterpret_cast<const __half2*>(p.res_hi + o);
                    l[q] = *reinterpret_cast<const __half2*>(p.res_lo + o);
                } else {
                    h[q] = __float2half2_rn(0.f);
                    l[q] = __float2half2_rn(0.f);
                }
            }
        };
        int i = 0;
        __half2 rsh[16], rsl[16];
        if (cluster_id < m_blks) load_res(cluster_id * kGemmBM + quad * 32, 0, rsh, rsl);
        for (int mb = cluster_id; mb < m_blks; mb += n_clusters, ++i) {
            const int buf = i & 1;
            const uint32_t use = static_cast<uint32_t>(i >> 1);
            const int row_base = mb * kGemmBM + quad * 32;
            // ---- pass A: y = acc + (bias + residual).  The residual chunk is loaded coalesced (lane = column pair,
            //      one chunk ahead; the first chunk of a row block is fetched during the previous block's pass C), parked with the bias in the
            //      staging tile, and picked up in the thread = row layout next to the tcgen05.ld registers; y goes back
            //      into the accumulator columns and the statistics of this warp's 96 columns are formed from registers
            //      (per-chunk mean / M2, chunks merged with Chan's formula).
            float m_loc = 0.f, m2 = 0.f;
#pragma unroll
            for (int cc = 0; cc < kChunks; ++cc) {
                const int c = chalf * kChunks + cc;
                const float2 bia2 = *reinterpret_cast<const float2*>(svec + c * 32 + cp);
#pragma unroll
                for (int rr = 0; rr < 32; rr += 2) {
                    const int rl = rr + rsub;
                    const float2 br = f2_add(bia2, f2_add(__half22float2(rsh[rr >> 1]), __half22float2(rsl[rr >> 1])));
                    stg[rl * kGemmStageRow + cp] = br.x;
                    stg[rl * kGemmStageRow + cp + 1] = br.y;
                }
                if (cc + 1 < kChunks) load_res(row_base, cc + 1, rsh, rsl);      // in flight during the rest of this chunk
                __syncwarp();
                if (cc == 0) {
                    mbar_wait(&acc_full[buf], use & 1);
                    tc_fence_after();
                }
                uint32_t r[32];
                const uint32_t taddr = tmem_addr(tmem_base, quad * 32, buf * kLnBN + c * 32);
                tmem_ld32(taddr, r);
                tmem_ld_wait();
                float2 s2 = make_float2(0.f, 0.f);                        // two interleaved partial sums (packed adds)
#pragma unroll
                for (int j = 0; j < 32; j += 2) {
                    const float2 y = f2_add(make_float2(__uint_as_float(r[j]), __uint_as_float(r[j + 1])),
                                            make_float2(stg[lane * kGemmStageRow + j], stg[lane * kGemmStageRow + j + 1]));
                    r[j] = __float_as_uint(y.x);
                    r[j + 1] = __float_as_uint(y.y);
                    s2 = f2_add(s2, y);
                }
                tmem_st32(taddr, r);
                __syncwarp();                                            // staging tile free for the next chunk
                const float mc = (s2.x + s2.y) * (1.0f / 32.0f);
                float2 q2 = make_float2(0.f, 0.f);
#pragma unroll
                for (int j = 0; j < 32; j += 2) {
                    const float2 d = f2_sub(make_float2(__uint_as_float(r[j]), __uint_as_float(r[j + 1])), f2_splat(mc));
                    q2 = f2_fma(d, d, q2);
                }
                const float qc = q2.x + q2.y;
                // merge (32 * cc columns: m_loc, m2) with (32 columns: mc, qc)
                const float na = 32.0f * static_cast<float>(cc), nn = na + 32.0f;
                const float delta = mc - m_loc;
                m_loc += delta * (32.0f / nn);
                m2 += qc + delta * delta * (na * 32.0f / nn);
            }
            tmem_st_wait();
            // first residual chunk of the NEXT row block: in flight during the exchange and pass C
            if (mb + n_clusters < m_blks) load_res((mb + n_clusters) * kGemmBM + quad * 32, 0, rsh, rsl);
            // ---- exchange (mean, M2) of (row, part) with every CTA of the cluster
            const int sbuf = i & 1;
            float2* my = stats + (static_cast<size_t>(sbuf) * kMaxParts + part) * kGemmBM + trow;
            if (ew == 0 && lane == 0) mbar_arrive_expect_tx(&stat_full[sbuf], static_cast<uint32_t>(kGemmBM * nparts * sizeof(float2)));
            for (uint32_t c = 0; c < CL; ++c) st_async_cluster_f2(my, &stat_full[sbuf], c, make_float2(m_loc, m2));
            mbar_wait(&stat_full[sbuf], use & 1);
            float mean = 0.f;
            for (int q = 0; q < nparts; ++q) mean += stats[(static_cast<size_t>(sbuf) * kMaxParts + q) * kGemmBM + trow].x;
            mean /= static_cast<float>(nparts);
            float M2 = 0.f;
            for (int q = 0; q < nparts; ++q) {
                const float2 s2 = stats[(static_cast<size_t>(sbuf) * kMaxParts + q) * kGemmBM + trow];
                const float d = s2.x - mean;
                M2 += s2.y + static_cast<float>(kPartCols) * d * d;
            }
            const float rstd = 1.0f / sqrtf(M2 * inv_n + p.eps);
            // ---- pass C: normalise, gamma / beta in the column-pair layout, split, coalesced plane stores
#pragma unroll 1
            for (int cc = 0; cc < kChunks; ++cc) {
                const int c = chalf * kChunks + cc;
                const int col0 = nb * kLnBN + c * 32;
                const float2 g2 = *reinterpret_cast<const float2*>(svec + kLnBN + c * 32 + cp);
                const float2 b2 = *reinterpret_cast<const float2*>(svec + 2 * kLnBN + c * 32 + cp);
                uint32_t r[32];
                tmem_ld32(tmem_addr(tmem_base, quad * 32, buf * kLnBN + c * 32), r);
                tmem_ld_wait();
                if (cc == kChunks - 1) {                       // last TMEM read of this warp for the tile
                    tc_fence_before();
                    mbar_arrive(&acc_empty[buf]);
                }
#pragma unroll
                for (int j = 0; j < 32; j += 2) {
                    const float2 z = f2_mul(f2_sub(make_float2(__uint_as_float(r[j]), __uint_as_float(r[j + 1])), f2_splat(mean)), f2_splat(rstd));
                    stg[lane * kGemmStageRow + j] = z.x;
                    stg[lane * kGemmStageRow + j + 1] = z.y;
                }
                __syncwarp();
#pragma unroll
                for (int rr = 0; rr < 32; rr += 2) {
                    const int rl = rr + rsub;
                    const int grow = row_base + rl;
                    if (grow < p.M) {
                        const float2 v = f2_fma(make_float2(stg[rl * kGemmStageRow + cp], stg[rl * kGemmStageRow + cp + 1]), g2, b2);
                        const size_t o = static_cast<size_t>(grow) * p.N + col0 + cp;
                        __half2 h2, l2;
                        split_f16x2(v, h2, l2);
                        *reinterpret_cast<__half2*>(p.out_hi + o) = h2;
                        *reinterpret_cast<__half2*>(p.out_lo + o) = l2;
                    }
                }
                __syncwarp();
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 1) tmem_dealloc<512>(tmem_base);
    cluster_sync_all();                           // no CTA leaves while a peer could still address its shared memory
}

// A K-major fp16 operand carried as two planes, with the TMA maps of both
struct SplitOperand {
    __half* hi = nullptr;
    __half* lo = nullptr;
    int64_t rows = 0;     // rows covered by the tensor maps (allocation rows)
    int cols = 0;
    CUtensorMap map_hi{}, map_lo{};          // box {64 halves, 128 rows}, SWIZZLE_128B  (A side and BN = 128 weights)
    CUtensorMap map192_hi{}, map192_lo{};    // weights only: box {64, 192}
    CUtensorMap map256_hi{}, map256_lo{};    // weights only: box {64, 256}
    bool is_weight = false;                  // weights carry the wider boxes
};

// is_activation: operand is the A side of the GEMMs (128-row boxes only) rather than a weight
int make_split_operand(SplitOperand* op, __half* hi, __half* lo, int64_t rows, int cols, bool is_activation);
// C = A * W^T with the epilogue `mode`; A rows used = p.M (<= A.rows)
int launch_gemm(int mode, const SplitOperand& A, const SplitOperand& W, const GemmParams& p, int sms, cudaStream_t st);
// fused GEMM + bias + residual + LayerNorm -> planes; supported when N is 384 or 768 (gemm_ln_supported)
bool gemm_ln_supported(const SplitOperand& W, int N);
int launch_gemm_ln(const SplitOperand& A, const SplitOperand& W, const GemmLnParams& p, int sms, cudaStream_t st);

}  // namespace rmu
