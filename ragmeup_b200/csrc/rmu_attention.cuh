// Self-attention on tcgen05 / TMEM / TMA (sm_100a).  Included by rmu_encoder.cu inside namespace rmu.
//
// Stands behind the eager attention of the reference's encoders (transformers BertSelfAttention,
// modeling_bert.py:114-140,168-208: softmax(Q K^T / sqrt(d_h)) V per head), reached through
// HuggingFaceEmbeddings.embed_* (server/RAGHelper_local.py:114-117) and HuggingFaceCrossEncoder.score
// (server/RAGHelper.py:483-486, server/ScoredCrossEncoderReranker.py:42).
//
// One work unit = (sequence, head, block of 128 query rows); all keys of the sequence (<= 256 - d_h) are handled
// in ONE score tile, so the softmax is the plain two-pass form (no running rescale).  Q (pre-scaled by
// log2(e) / sqrt(d_h)), K and V arrive as the split fp16 planes [T, 3H] the QKV GEMM epilogue wrote; every
// product keeps the 3-term split (hi*hi + lo*hi + hi*lo, fp32 accumulate) that holds 1e-3 parity with fp32.
//
//   S[128 x keys] = Q K^T     tcgen05.mma.kind::f16, M = 128, N = keys (16-aligned), K = d_h; operands are TMA boxes of
//                             {d_h halves, rows} (SWIZZLE_64B for d_h = 32, SWIZZLE_128B for 64); S lives in TMEM.
//   P = exp2(S - rowmax)      softmax warps, thread = row = TMEM lane: two passes of tcgen05.ld over S; P is split into
//                             fp16 hi / lo, packed two keys per 32-bit column and written back IN PLACE with tcgen05.st:
//                             the 32 fp32 columns of a 32-key chunk become 16 columns of P_hi + 16 columns of P_lo.
//   O[128 x d_h] = P V        A operand straight from TMEM (no shared-memory round trip for P), B = the V box as it
//                             landed ([key][d_h], i.e. MN-major: no transposed copy of V is ever made), O in TMEM.
//   ctx = O / rowsum          read back with tcgen05.ld, split to planes, stored as 64/128-byte row segments.
//
// Persistent CTAs (one per SM) keep TWO units in flight: while softmax group g works on unit i, the tensor core
// already computes S of unit i+1 into the other TMEM buffer and the TMA warp prefetches units i+2.. into a ring of
// operand slots, so the CUDA-core softmax (the real cost: exp2, hi/lo split, ~8 instructions per score) never waits
// for loads or MMAs.
// The S = Q K^T and O = P V instruction streams are issued by two different threads: S of unit i+2 only waits for the
// TMEM buffer (P V of unit i done), P V of unit i only for its softmax; issued by one thread in program order, each P V
// sat behind the other group's read-out and the two groups ran in lockstep (measured: 390 us per layer call, the same
// as the mma.sync kernel, with 38 % of all warp samples waiting for O).
//   warp 0: TMA producer   warp 1: S issuer + TMEM allocator   warp 2: P V issuer   warps 3-10: softmax group 0   warps 11-18: group 1
#pragma once

constexpr int kAtcThreads = 608;             // 3 control warps + 2 in-flight units x 8 softmax warps
constexpr int kAtcRows = 128;                 // query rows per unit = MMA M
constexpr int kAtcBufCols = 256;              // TMEM columns per in-flight unit: S / P from 0, O in the last d_h columns
constexpr int kAtcMaxSlots = 3;
constexpr int kAtcMaxChunks = 8;             // 32-key chunks of a score tile (<= 256 keys)
constexpr int kAtcStateBytes = 512 + 4 * 128 * 4;   // mbarriers + the row max / row sum exchange of the softmax warps

struct AtcParams {
    const int* cu;          // [B + 1] token offsets
    int B, heads, H;        // H = hidden = heads * d_h
    int row_tiles;          // ceil(max_seqlen / 128)
    int kp;                 // keys per operand slot: max_seqlen rounded up to 64
    int nslots;             // operand slots in shared memory (1..3)
    int nacc;               // O accumulators per unit: 3 (one per product term; needs keys <= 256 - 3 d_h) or 1
    __half* ctx_hi; __half* ctx_lo;   // [T, H]
};

// shared-memory matrix descriptor, 8-row (or 8-key) groups `sbo` bytes apart; layout 2 = SWIZZLE_128B, 4 = SWIZZLE_64B
__device__ __forceinline__ uint64_t atc_desc(uint32_t smem_addr, uint32_t sbo, uint32_t layout) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
    d |= static_cast<uint64_t>(1) << 16;
    d |= static_cast<uint64_t>(sbo >> 4) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(layout) << 61;
    return d;
}

// D[tmem] (+)= A[tmem, fp16 packed two per column] * B[smem], fp32 accumulate
__device__ __forceinline__ void mma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
          "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}

__device__ __forceinline__ float atc_exp2(float x) {   // ex2.approx: 2 ulp, exp2(-inf) = +0
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// (a, b) -> packed fp16 pair of the high parts and of the residuals (a - hi(a), b - hi(b))
__device__ __forceinline__ void atc_split_pack(float a, float b, uint32_t& hi, uint32_t& lo) {
    const __half2 h = __floats2half2_rn(a, b);
    const float2 hf = __half22float2(h);
    const __half2 l = __floats2half2_rn(a - hf.x, b - hf.y);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}

// unit u of the grid-stride enumeration -> (sequence, row tile, head); false when the row tile lies past the sequence
struct AtcUnit { int b, rt, h, t0, S; };
__device__ __forceinline__ bool atc_unit(const AtcParams& p, int u, AtcUnit& o) {
    o.h = u % p.heads;
    const int br = u / p.heads;
    o.rt = br % p.row_tiles;
    o.b = br / p.row_tiles;
    o.t0 = __ldg(p.cu + o.b);
    o.S = __ldg(p.cu + o.b + 1) - o.t0;
    return o.rt * kAtcRows < o.S;
}

template <int DH>
__global__ void __launch_bounds__(kAtcThreads, 1)
attention_tc_kernel(const __grid_constant__ CUtensorMap tq_hi, const __grid_constant__ CUtensorMap tq_lo,
                    const __grid_constant__ CUtensorMap tk_hi, const __grid_constant__ CUtensorMap tk_lo, const AtcParams p) {
    constexpr int ROWB = DH * 2;                           // bytes of one operand row (64 or 128)
    constexpr uint32_t LAYOUT = DH == 32 ? 4u : 2u;        // SWIZZLE_64B / SWIZZLE_128B
    constexpr uint32_t SBO = 8 * ROWB;                     // 8 rows (or 8 keys) per swizzle group
    constexpr int QBYTES = kAtcRows * ROWB;                // one plane of the Q tile
    constexpr int KS = DH / 16;                            // MMA K steps over d_h
    // O accumulators sit at the end of a TMEM buffer: one per product term (P_hi V_hi, P_lo V_hi, P_hi V_lo) when the
    // columns allow it, added up by the read-out.  (Measured since: an N = 32 TS-form MMA costs 17.6 cycles and MMAs into
    // one accumulator run at that rate, tools/micro/mma_cost.cu, so one accumulator would do as well.)
    const int OCOL = kAtcBufCols - p.nacc * DH;
    const int OCOL_C = OCOL;
    // O = P V: A from TMEM (K-major), B = V as it lies in shared memory ([key][d_h]): MN-major -> bit 16
    constexpr uint32_t IDESC_O = umma_idesc(0 /*f16*/, kAtcRows, DH) | (1u << 16);

    extern __shared__ uint8_t atc_smem_raw[];
    uint8_t* smem = atc_smem_raw + ((1024u - (smem_u32(atc_smem_raw) & 1023u)) & 1023u);
    const int kbytes = p.kp * ROWB;                        // one plane of K (or V) of a slot
    const int slot_bytes = 2 * QBYTES + 4 * kbytes;        // Qh Ql Kh Kl Vh Vl
    uint8_t* state = smem + p.nslots * slot_bytes;
    uint64_t* load_full = reinterpret_cast<uint64_t*>(state);
    uint64_t* load_empty = load_full + kAtcMaxSlots;
    uint64_t* s_full = load_empty + kAtcMaxSlots;          // [2] S of buffer g is complete
    uint64_t* p_full = s_full + 2;                         // [2][8] 32-key chunk c of P in buffer g is written (one barrier per chunk:
                                                           // a group that runs ahead of the P V issuer cannot lap a phase)
    uint64_t* o_full = p_full + 2 * kAtcMaxChunks;         // [2] O of buffer g is complete
    uint64_t* s_free = o_full + 2;                         // [2] the P V MMAs that read buffer g have completed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_free + 2);
    float* xch = reinterpret_cast<float*>(state + 512);    // [2 groups][2 halves][128 rows]

    const int warp = threadIdx.x >> 5;
    const unsigned lane = lane_id();
    const int nunits = p.B * p.row_tiles * p.heads;

    if (threadIdx.x == 0) {
        for (int i = 0; i < p.nslots; ++i) { mbar_init(&load_full[i], 1); mbar_init(&load_empty[i], 1); }
        for (int g = 0; g < 2; ++g) { mbar_init(&s_full[g], 1); for (int c = 0; c < kAtcMaxChunks; ++c) mbar_init(&p_full[g * kAtcMaxChunks + c], 1); mbar_init(&o_full[g], 1); mbar_init(&s_free[g], 1); }
        fence_mbar_init();
        prefetch_tmap(&tq_hi); prefetch_tmap(&tq_lo); prefetch_tmap(&tk_hi); prefetch_tmap(&tk_lo);
    }
    if (warp == 1) tmem_alloc<512>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // =========================== TMA producer ===========================
        if (elect_one()) {
            int i = 0;
            for (int u = blockIdx.x; u < nunits; u += gridDim.x) {
                AtcUnit un;
                if (!atc_unit(p, u, un)) continue;
                const int slot = i % p.nslots;
                const uint32_t use = static_cast<uint32_t>(i / p.nslots);
                mbar_wait(&load_empty[slot], (use & 1) ^ 1);
                const int nkb = (un.S + 63) >> 6;                       // 64-key boxes of this sequence
                uint8_t* sb = smem + slot * slot_bytes;
                mbar_arrive_expect_tx(&load_full[slot], static_cast<uint32_t>(2 * QBYTES + 4 * nkb * 64 * ROWB));
                const int qrow = un.t0 + un.rt * kAtcRows, qcol = un.h * DH;
                tma_load_2d(sb, &tq_hi, qcol, qrow, &load_full[slot], kEvictNormal);
                tma_load_2d(sb + QBYTES, &tq_lo, qcol, qrow, &load_full[slot], kEvictNormal);
                for (int kb = 0; kb < nkb; ++kb) {
                    const int krow = un.t0 + kb * 64;
                    uint8_t* kd = sb + 2 * QBYTES + kb * 64 * ROWB;
                    tma_load_2d(kd, &tk_hi, p.H + qcol, krow, &load_full[slot], kEvictNormal);
                    tma_load_2d(kd + kbytes, &tk_lo, p.H + qcol, krow, &load_full[slot], kEvictNormal);
                    tma_load_2d(kd + 2 * kbytes, &tk_hi, 2 * p.H + qcol, krow, &load_full[slot], kEvictNormal);
                    tma_load_2d(kd + 3 * kbytes, &tk_lo, 2 * p.H + qcol, krow, &load_full[slot], kEvictNormal);
                }
                ++i;
            }
        }
    } else if (warp == 1) {
        // =========================== S = Q K^T issuer ===========================
        if (elect_one()) {
            int i = 0;
            for (int u = blockIdx.x; u < nunits; u += gridDim.x) {
                AtcUnit un;
                if (!atc_unit(p, u, un)) continue;
                const int g = i & 1;
                const uint32_t use = static_cast<uint32_t>(i >> 1);
                const int slot = i % p.nslots;
                mbar_wait(&load_full[slot], static_cast<uint32_t>(i / p.nslots) & 1);
                mbar_wait(&s_free[g], (use & 1) ^ 1);            // P V of the unit two back no longer reads this buffer
                tc_fence_after();
                const uint8_t* sb = smem + slot * slot_bytes;
                const uint32_t qh = smem_u32(sb), ql = qh + QBYTES, kh = qh + 2 * QBYTES, kl = kh + kbytes;
                const uint32_t idesc_s = umma_idesc(0 /*f16*/, kAtcRows, ((un.S + 15) >> 4) << 4);
                const uint32_t d_addr = tmem_base + g * kAtcBufCols;
#pragma unroll
                for (int term = 0; term < 3; ++term) {
                    const uint32_t a = term == 1 ? ql : qh, b = term == 2 ? kl : kh;
#pragma unroll
                    for (int k = 0; k < KS; ++k)
                        mma_f16_ss(d_addr, atc_desc(a + k * 32, SBO, LAYOUT), atc_desc(b + k * 32, SBO, LAYOUT), idesc_s,
                                   (term | k) != 0 ? 1u : 0u);
                }
                tc_commit(&s_full[g]);
                ++i;
            }
        }
    } else if (warp == 2) {
        // =========================== O = P V issuer ===========================
        if (elect_one()) {
            int i = 0;
            uint32_t ppar[2] = {0u, 0u};                         // bit c = parity the next wait on p_full[g][c] uses
            for (int u = blockIdx.x; u < nunits; u += gridDim.x) {
                AtcUnit un;
                if (!atc_unit(p, u, un)) continue;
                const int g = i & 1;
                const int slot = i % p.nslots;
                const uint8_t* sb = smem + slot * slot_bytes;
                const uint32_t vh = smem_u32(sb + 2 * QBYTES + 2 * kbytes), vl = vh + kbytes;
                const uint32_t pbase = tmem_base + g * kAtcBufCols;
                const uint32_t d_addr = pbase + OCOL;
                const uint32_t d1 = p.nacc == 3 ? d_addr + DH : d_addr, d2 = p.nacc == 3 ? d_addr + 2 * DH : d_addr;
                const int nk16 = (un.S + 15) >> 4;
                const int nchunk = (un.S + 31) >> 5;
                // P arrives 32 keys at a time (the same warps read O of the unit two back out before they wrote any of it):
                // the MMAs of a chunk are issued while the softmax warps are still working on the next one
                for (int c = 0; c < nchunk; ++c) {
                    mbar_wait(&p_full[g * kAtcMaxChunks + c], (ppar[g] >> c) & 1u);   // per-barrier parity: sequences differ in chunks
                    ppar[g] ^= 1u << c;
                    tc_fence_after();
                    for (int j16 = 2 * c; j16 < min(2 * c + 2, nk16); ++j16) {
                        const uint32_t a_hi = pbase + 32 * c + 8 * (j16 & 1), a_lo = a_hi + 16;
                        const uint64_t bh = atc_desc(vh + j16 * 16 * ROWB, SBO, LAYOUT), bl = atc_desc(vl + j16 * 16 * ROWB, SBO, LAYOUT);
                        const uint32_t acc = j16 != 0 ? 1u : 0u;
                        mma_f16_ts(d_addr, a_hi, bh, IDESC_O, acc);
                        mma_f16_ts(d1, a_lo, bh, IDESC_O, p.nacc == 3 ? acc : 1u);
                        mma_f16_ts(d2, a_hi, bl, IDESC_O, p.nacc == 3 ? acc : 1u);
                    }
                }
                tc_commit(&o_full[g]);
                tc_commit(&s_free[g]);
                tc_commit(&load_empty[slot]);                    // the operand slot is free once these MMAs have read it
                ++i;
            }
        }
    } else {
        // =========================== softmax + output: thread = query row, two warps per row ===========================
        // Each in-flight unit has EIGHT warps: the two warps of a TMEM lane quadrant own the same 32 rows and split the
        // 32-key chunks (even / odd); row maxima and row sums are exchanged through shared memory.  With one warp per
        // quadrant a unit's softmax was a 5-chunk serial chain of tcgen05.ld -> exp2 / split -> tcgen05.st -> barrier
        // latencies (~9900 cycles from S ready to O stored, measured) and two units in flight could not hide it.
        const int grp = (warp - 3) >> 3;                         // which of the two in-flight units this warp serves
        const int half = ((warp - 3) >> 2) & 1;                  // which chunks (c & 1) and which half of O's columns
        const int quad = warp & 3;                               // TMEM lane quadrant this warp may touch
        const int r = quad * 32 + static_cast<int>(lane);        // row of the unit
        const int htid = ((warp - 3) & 3) * 32 + static_cast<int>(lane);       // thread index inside the (group, half)
        float* xm = xch + (grp * 2 + half) * kAtcRows;           // my partial row maxima, then my partial row sums
        const float* xo = xch + (grp * 2 + (half ^ 1)) * kAtcRows;   // the other warp's
        int i = 0;
        for (int u = blockIdx.x; u < nunits; u += gridDim.x) {
            AtcUnit un;
            if (!atc_unit(p, u, un)) continue;
            if ((i & 1) != grp) { ++i; continue; }
            const uint32_t use = static_cast<uint32_t>(i >> 1);
            ++i;
            const uint32_t tb = tmem_addr(tmem_base, quad * 32, grp * kAtcBufCols);
            const int S = un.S;
            const int nchunk = (S + 31) >> 5;
            const bool warp_live = un.rt * kAtcRows + quad * 32 < S;      // any row of this warp inside the sequence
            mbar_wait(&s_full[grp], use & 1);
            tc_fence_after();
            // ---- pass 1: row maximum over my chunks, then over both warps of the row
            float m = -INFINITY;
            if (warp_live) {
                for (int c = half; c < nchunk; c += 2) {
                    uint32_t s[32];
                    tmem_ld32(tb + c * 32, s);
                    tmem_ld_wait();
                    if (c * 32 + 32 <= S) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) m = fmaxf(m, __uint_as_float(s[j]));
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j) m = fmaxf(m, c * 32 + j < S ? __uint_as_float(s[j]) : -INFINITY);
                    }
                }
            }
            xm[r] = m;
            bar_sync_named(1 + grp, 256);
            m = fmaxf(m, xo[r]);
            bar_sync_named(1 + grp, 256);                        // both warps have read the maxima: the slots may take the sums
            // ---- pass 2: P = exp2(S - m) (scores are pre-scaled by log2 e), split, packed back in place; every chunk is
            // handed to the P V issuer as soon as the four warps that own it have written it
            float l = 0.f;
            for (int c = half; c < nchunk; c += 2) {
                if (warp_live) {
                    uint32_t s[32];
                    tmem_ld32(tb + c * 32, s);
                    tmem_ld_wait();
                    uint32_t ph[16], pl[16];
                    const bool tail = c * 32 + 32 > S;
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        float a = atc_exp2(__uint_as_float(s[2 * j]) - m), b = atc_exp2(__uint_as_float(s[2 * j + 1]) - m);
                        if (tail) {                                  // keys past the sequence end: stale columns, P = 0
                            if (c * 32 + 2 * j >= S) a = 0.f;
                            if (c * 32 + 2 * j + 1 >= S) b = 0.f;
                        }
                        l += a + b;
                        atc_split_pack(a, b, ph[j], pl[j]);
                    }
                    tmem_st16(tb + c * 32, ph);
                    tmem_st16(tb + c * 32 + 16, pl);
                    tmem_st_wait();
                }
                tc_fence_before();
                bar_sync_named(3 + grp * 2 + half, 128);
                if (htid == 0) mbar_arrive(&p_full[grp * kAtcMaxChunks + c]);
            }
            xm[r] = l;
            // ---- O / l -> split planes; this warp takes half of the d_h columns of its rows
            mbar_wait(&o_full[grp], use & 1);
            tc_fence_after();
            bar_sync_named(1 + grp, 256);
            l += xo[r];
            const int row = un.rt * kAtcRows + r;
            if (warp_live) {
                constexpr int CE = DH / 2;                       // columns per warp: 16 or 32
                const float inv = 1.0f / l;
                uint32_t o[CE];
                if constexpr (CE == 32) tmem_ld32(tb + OCOL_C + half * CE, o); else tmem_ld16(tb + OCOL_C + half * CE, o);
                tmem_ld_wait();
                if (p.nacc == 3) {                               // the three product terms were accumulated separately
#pragma unroll 1
                    for (int t = 1; t < 3; ++t) {
                        uint32_t o1[CE];
                        if constexpr (CE == 32) tmem_ld32(tb + OCOL_C + t * DH + half * CE, o1); else tmem_ld16(tb + OCOL_C + t * DH + half * CE, o1);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < CE; ++j) o[j] = __float_as_uint(__uint_as_float(o[j]) + __uint_as_float(o1[j]));
                    }
                }
                if (row < S) {
                    uint32_t oh[CE / 2], ol[CE / 2];
#pragma unroll
                    for (int j = 0; j < CE / 2; ++j)
                        atc_split_pack(__uint_as_float(o[2 * j]) * inv, __uint_as_float(o[2 * j + 1]) * inv, oh[j], ol[j]);
                    const size_t off = static_cast<size_t>(un.t0 + row) * p.H + un.h * DH + half * CE;
                    uint4* dh = reinterpret_cast<uint4*>(p.ctx_hi + off);
                    uint4* dl = reinterpret_cast<uint4*>(p.ctx_lo + off);
#pragma unroll
                    for (int q4 = 0; q4 < CE / 8; ++q4) {
                        dh[q4] = make_uint4(oh[4 * q4], oh[4 * q4 + 1], oh[4 * q4 + 2], oh[4 * q4 + 3]);
                        dl[q4] = make_uint4(ol[4 * q4], ol[4 * q4 + 1], ol[4 * q4 + 2], ol[4 * q4 + 3]);
                    }
                }
            }
            bar_sync_named(1 + grp, 256);                        // the sums have been read: the exchange slots are free again
        }
    }

    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 1) tmem_dealloc<512>(tmem_base);
}

// =====================================================================================================================
// attention_pair_kernel (d_h = 32): the same arithmetic, organised around what measurements of attention_tc_kernel showed
// to be its limit: the TMA engine delivers about one box ROW (<= 128 B) per 5 cycles per SM, whatever the row length
// (13.2 B/clk/SM with the 64-byte rows of one d_h = 32 head; 25.6 B/clk/SM in the scan's 128-byte rows), and the kernel
// spent its 367 us per layer call fetching 19.7 M such rows (K and V twice per sequence, once per query-row tile; 192 rows
// for 147 keys) while tensor pipe, MUFU and issue slots idled.  Here
//   * the QKV GEMM writes every head's q / k / v row as ONE 128-byte line [32 hi halves | 32 lo halves] (GemmParams::
//     interleave32), so all TMA boxes are 128 bytes wide (SWIZZLE_128B) and the hi / lo parts of an operand are the two
//     64-byte halves of its swizzled rows; a work item is (sequence, PAIR of adjacent heads), the two heads are the two
//     in-flight units (TMEM buffer g = head 2*hp + g);
//   * O = P V takes TWO MMAs per 16 keys instead of three: P_hi x [V_hi | V_lo] is one N = 64 MMA (V's row IS hi | lo),
//     P_lo x V_hi one N = 32 MMA that accumulates into the V_hi half of the same 64 columns;
//   * K and V of a work item are loaded once and serve all its query-row tiles; boxes are 32 rows, so 147 keys fetch
//     160 rows, and a 19-row last tile fetches 32 Q rows;
// i.e. 480 box rows per (sequence, head) instead of 2048.  Roles: warp 0 TMA, warp 1 S = Q K^T issuer (both heads),
// warps 2 / 3 the P V issuers of head 0 / 1, warps 4-7 output (O and row sums -> context planes), then 8 softmax warps
// per head.
// =====================================================================================================================
constexpr int kApThreads = 768;                // 4 role warps + 4 output warps + 2 heads x 8 softmax warps
constexpr int kApMaxKeys = 160;                // keys (16-aligned); the O accumulator (64 columns) sits at column 160 of the buffer
constexpr int kApRowB = 128;                   // operand row: two heads x 32 halves
constexpr int kApQSlot = 2 * kAtcRows * kApRowB;   // the Q tiles (hi | lo rows) of both heads
constexpr int kApStateBytes = 512 + 4 * 128 * 4;   // barriers | per (head, half, row) exchange slot: row max during pass 1, then the row sum

struct ApParams {
    const int* cu;
    int B, heads, H;
    int kp;                 // rows per K / V plane of a slot: max_seqlen rounded up to 32 (<= kApMaxKeys)
    __half* ctx_hi; __half* ctx_lo;
};

// packed fp32 pairs (FADD2 / FFMA2 of sm_100): one issue slot for two lanes' worth of softmax arithmetic
__device__ __forceinline__ void ap_add2(float& x0, float& x1, float y0, float y1) {
    asm("{\n\t.reg .b64 a, b;\n\tmov.b64 a, {%0, %1};\n\tmov.b64 b, {%2, %3};\n\tadd.rn.f32x2 a, a, b;\n\tmov.b64 {%0, %1}, a;\n\t}"
        : "+f"(x0), "+f"(x1) : "f"(y0), "f"(y1));
}
__device__ __forceinline__ void ap_sub2(float& x0, float& x1, float y0, float y1) {
    asm("{\n\t.reg .b64 a, b;\n\tmov.b64 a, {%0, %1};\n\tmov.b64 b, {%2, %3};\n\tsub.rn.f32x2 a, a, b;\n\tmov.b64 {%0, %1}, a;\n\t}"
        : "+f"(x0), "+f"(x1) : "f"(y0), "f"(y1));
}
__device__ __forceinline__ void ap_mul2(float& x0, float& x1, float y0, float y1) {
    asm("{\n\t.reg .b64 a, b;\n\tmov.b64 a, {%0, %1};\n\tmov.b64 b, {%2, %3};\n\tmul.rn.f32x2 a, a, b;\n\tmov.b64 {%0, %1}, a;\n\t}"
        : "+f"(x0), "+f"(x1) : "f"(y0), "f"(y1));
}
__device__ __forceinline__ void ap_split_pack(float a, float b, uint32_t& hi, uint32_t& lo) {
    const __half2 h = __floats2half2_rn(a, b);
    const float2 hf = __half22float2(h);
    ap_sub2(a, b, hf.x, hf.y);
    const __half2 l = __floats2half2_rn(a, b);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}

// The softmax warps of a head run a serial chain per query-row tile (row max, exp + split + write-back, then -- in the
// first version of this kernel -- the wait for O and its read-out): 7400 cycles per tile of which they computed 45 %,
// the rest latency, and with TMEM allowing only two heads in flight nothing hid it.  Here the O read-out belongs to four
// OUTPUT warps (one per TMEM lane quadrant, serving both heads): a softmax warp leaves its row sums in shared memory and
// goes straight to the next tile's scores, so a head's chain is row max -> exp -> (P V tail -> next S), and the read-out
// of tile n overlaps the softmax of tile n + 1.
__global__ void __launch_bounds__(kApThreads, 1)
attention_pair_kernel(const __grid_constant__ CUtensorMap t_qkv, const ApParams p) {
    constexpr int DH = 32;
    constexpr uint32_t LAYOUT = 2u;                        // SWIZZLE_128B
    constexpr uint32_t SBO = 8 * kApRowB;
    constexpr int OCOL = kAtcBufCols - 3 * DH;             // 160
    constexpr uint32_t IDESC_O64 = umma_idesc(0 /*f16*/, kAtcRows, 2 * DH) | (1u << 16);   // B = [V_hi | V_lo], MN-major
    constexpr uint32_t IDESC_O32 = umma_idesc(0 /*f16*/, kAtcRows, DH) | (1u << 16);       // B = V_hi

    extern __shared__ __align__(1024) uint8_t ap_smem_raw[];     // two K / V slots + two Q slots use nearly all 227 KB at 160 keys:
    uint8_t* smem = ap_smem_raw;                                  // no room for an alignment pad, the declaration must deliver it
    if ((smem_u32(ap_smem_raw) & 1023u) != 0u) __trap();
    const int kvplane = p.kp * kApRowB;                    // K (or V) of one head: kp rows of [hi | lo]
    const int kvslot = 4 * kvplane;
    uint8_t* kvring = smem;                                // 2 slots
    uint8_t* qring = smem + 2 * kvslot;                    // 2 slots
    uint8_t* state = qring + 2 * kApQSlot;
    uint64_t* kv_full = reinterpret_cast<uint64_t*>(state);
    uint64_t* kv_empty = kv_full + 2;
    uint64_t* q_full = kv_empty + 2;
    uint64_t* q_empty = q_full + 2;
    uint64_t* s_full = q_empty + 2;                        // [2] S of head g is complete
    uint64_t* p_full = s_full + 2;                         // [2][8] chunk c of P of head g is written
    uint64_t* o_full = p_full + 2 * kAtcMaxChunks;         // [2] all P V MMAs of head g's tile have completed (output warps)
    uint64_t* s_free = o_full + 2;                         // [2] the same event, for the S issuer: buffer g may be overwritten
    uint64_t* l_full = s_free + 2;                         // [2] the 8 softmax warps of head g have left their row sums
    uint64_t* o_free = l_full + 2;                         // [2] the 4 output warps have read O of head g
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_free + 2);
    float* xch = reinterpret_cast<float*>(state + 512);    // [2 heads][2 halves][128 rows]: row max (pass 1), then the row sum

    const int warp = threadIdx.x >> 5;
    const unsigned lane = lane_id();
    const int hpairs = p.heads >> 1;
    const int nwork = p.B * hpairs;

    if (threadIdx.x == 0) {
        for (int i = 0; i < 2; ++i) {
            mbar_init(&kv_full[i], 1); mbar_init(&kv_empty[i], 2); mbar_init(&q_full[i], 1); mbar_init(&q_empty[i], 1);
            mbar_init(&s_full[i], 1); mbar_init(&o_full[i], 1); mbar_init(&s_free[i], 1);
            mbar_init(&l_full[i], 8 * 32); mbar_init(&o_free[i], 4 * 32);   // every lane arrives: compute-sanitizer racecheck
            // models mbarrier ordering per arriving thread (an elected lane after __syncwarp is flagged on the exchange slots)
            for (int c = 0; c < kAtcMaxChunks; ++c) mbar_init(&p_full[i * kAtcMaxChunks + c], 4);   // the four warps that own the chunk
        }
        fence_mbar_init();
        prefetch_tmap(&t_qkv);
    }
    if (warp == 1) tmem_alloc<512>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // =========================== TMA producer ===========================
        if (elect_one()) {
            int kvi = 0, qi = 0;
            for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
                const int b = w / hpairs, hp = w % hpairs;
                const int t0 = __ldg(p.cu + b), S = __ldg(p.cu + b + 1) - t0;
                const int col = hp * 128;                        // interleaved layout: a head is 64 halves, a pair 128
                const int kvs = kvi & 1;
                mbar_wait(&kv_empty[kvs], ((kvi >> 1) & 1) ^ 1);
                const int nkb = (S + 31) >> 5;
                uint8_t* kb0 = kvring + kvs * kvslot;
                mbar_arrive_expect_tx(&kv_full[kvs], static_cast<uint32_t>(4 * nkb * 32 * kApRowB));
                for (int kb = 0; kb < nkb; ++kb) {
                    uint8_t* d = kb0 + kb * 32 * kApRowB;
                    tma_load_2d(d, &t_qkv, 2 * p.H + col, t0 + kb * 32, &kv_full[kvs], kEvictNormal);                  // K, head 0
                    tma_load_2d(d + kvplane, &t_qkv, 2 * p.H + col + 64, t0 + kb * 32, &kv_full[kvs], kEvictNormal);   // K, head 1
                    tma_load_2d(d + 2 * kvplane, &t_qkv, 4 * p.H + col, t0 + kb * 32, &kv_full[kvs], kEvictNormal);    // V, head 0
                    tma_load_2d(d + 3 * kvplane, &t_qkv, 4 * p.H + col + 64, t0 + kb * 32, &kv_full[kvs], kEvictNormal);
                }
                for (int r0 = 0; r0 < S; r0 += kAtcRows, ++qi) {
                    const int qs = qi & 1;
                    mbar_wait(&q_empty[qs], ((qi >> 1) & 1) ^ 1);
                    const int nqb = (min(kAtcRows, S - r0) + 31) >> 5;
                    uint8_t* q0 = qring + qs * kApQSlot;
                    mbar_arrive_expect_tx(&q_full[qs], static_cast<uint32_t>(2 * nqb * 32 * kApRowB));
                    for (int qb = 0; qb < nqb; ++qb) {
                        tma_load_2d(q0 + qb * 32 * kApRowB, &t_qkv, col, t0 + r0 + qb * 32, &q_full[qs], kEvictNormal);
                        tma_load_2d(q0 + kAtcRows * kApRowB + qb * 32 * kApRowB, &t_qkv, col + 64, t0 + r0 + qb * 32, &q_full[qs], kEvictNormal);
                    }
                }
                ++kvi;
            }
        }
    } else if (warp == 1) {
        // =========================== S = Q K^T issuer, both heads ===========================
        if (elect_one()) {
            int kvi = 0, qi = 0;
            uint32_t cnt = 0;                                    // tiles issued so far (the same for both heads)
            for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
                const int b = w / hpairs;
                const int S = __ldg(p.cu + b + 1) - __ldg(p.cu + b);
                const int kvs = kvi & 1;
                mbar_wait(&kv_full[kvs], (kvi >> 1) & 1);
                const uint32_t kbase = smem_u32(kvring + kvs * kvslot);
                const uint32_t idesc_s = umma_idesc(0 /*f16*/, kAtcRows, ((S + 15) >> 4) << 4);
                for (int r0 = 0; r0 < S; r0 += kAtcRows, ++qi, ++cnt) {
                    const int qs = qi & 1;
                    mbar_wait(&q_full[qs], (qi >> 1) & 1);
                    const uint32_t qbase = smem_u32(qring + qs * kApQSlot);
#pragma unroll
                    for (int g = 0; g < 2; ++g) {
                        mbar_wait(&s_free[g], (cnt & 1) ^ 1);    // P V of this head's previous tile no longer reads the buffer
                        tc_fence_after();
                        const uint32_t d_addr = tmem_base + g * kAtcBufCols;
                        const uint32_t qg = qbase + g * kAtcRows * kApRowB, kg = kbase + g * kvplane;   // rows = [hi 64 B | lo 64 B]
#pragma unroll
                        for (int term = 0; term < 3; ++term) {
                            const uint32_t a = qg + (term == 1 ? 64 : 0), bb = kg + (term == 2 ? 64 : 0);
#pragma unroll
                            for (int k = 0; k < 2; ++k)
                                mma_f16_ss(d_addr, atc_desc(a + k * 32, SBO, LAYOUT), atc_desc(bb + k * 32, SBO, LAYOUT), idesc_s,
                                           (term | k) != 0 ? 1u : 0u);
                        }
                        tc_commit(&s_full[g]);
                    }
                    tc_commit(&q_empty[qs]);                     // the Q tile has been read by both heads' MMAs
                }
                ++kvi;
            }
        }
    } else if (warp < 4) {
        // =========================== O = P V issuer of head g ===========================
        if (elect_one()) {
            const int g = warp - 2;
            int kvi = 0;
            uint32_t cnt = 0;
            uint32_t ppar = 0u;                                  // bit c = parity the next wait on p_full[g][c] uses
            for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
                const int b = w / hpairs;
                const int S = __ldg(p.cu + b + 1) - __ldg(p.cu + b);
                const int kvs = kvi & 1;
                const uint32_t vg = smem_u32(kvring + kvs * kvslot + (2 + g) * kvplane);      // V rows of this head: [hi | lo]
                const uint32_t pbase = tmem_base + g * kAtcBufCols;
                const uint32_t d0 = pbase + OCOL;                    // [P_hi V_hi + P_lo V_hi | P_hi V_lo] (64 columns)
                const int nk16 = (S + 15) >> 4, nchunk = (S + 31) >> 5;
                for (int r0 = 0; r0 < S; r0 += kAtcRows, ++cnt) {
                    for (int c = 0; c < nchunk; ++c) {
                        mbar_wait(&p_full[g * kAtcMaxChunks + c], (ppar >> c) & 1u);
                        ppar ^= 1u << c;
                        if (c == 0) mbar_wait(&o_free[g], (cnt & 1) ^ 1);   // the output warps have read the previous tile's O
                        tc_fence_after();
                        for (int j16 = 2 * c; j16 < min(2 * c + 2, nk16); ++j16) {
                            const uint32_t a_hi = pbase + 32 * c + 8 * (j16 & 1), a_lo = a_hi + 16;
                            const uint64_t bv = atc_desc(vg + j16 * 16 * kApRowB, SBO, LAYOUT);
                            const uint32_t acc = j16 != 0 ? 1u : 0u;
                            mma_f16_ts(d0, a_hi, bv, IDESC_O64, acc);
                            mma_f16_ts(d0, a_lo, bv, IDESC_O32, 1u);      // N = 32: lands on the V_hi half of the same accumulator
                        }
                    }
                    tc_commit(&o_full[g]);
                    tc_commit(&s_free[g]);
                    if (r0 + kAtcRows >= S) tc_commit(&kv_empty[kvs]);   // last tile of the work item: K / V slot free (both heads commit)
                }
                ++kvi;
            }
        }
    } else if (warp < 8) {
        // =========================== output warps: O / l of both heads -> context planes ===========================
        const int quad = warp & 3;
        const int r = quad * 32 + static_cast<int>(lane);
        uint32_t cnt = 0;
        for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
            const int b = w / hpairs, hp = w % hpairs;
            const int t0 = __ldg(p.cu + b), S = __ldg(p.cu + b + 1) - t0;
            for (int r0 = 0; r0 < S; r0 += kAtcRows, ++cnt) {
                const bool warp_live = r0 + quad * 32 < S;
                const int row = r0 + r;
#pragma unroll 1
                for (int g = 0; g < 2; ++g) {
                    mbar_wait(&l_full[g], cnt & 1);
                    const float* lp = xch + g * 2 * kAtcRows;
                    const float inv = 1.0f / (lp[r] + lp[kAtcRows + r]);
                    mbar_wait(&o_full[g], cnt & 1);
                    tc_fence_after();
                    const uint32_t ob = tmem_addr(tmem_base, quad * 32, g * kAtcBufCols + OCOL);
                    uint32_t oh[16], ol[16];
                    if (warp_live) {
#pragma unroll
                        for (int hc = 0; hc < 2; ++hc) {             // 16 output columns at a time
                            uint32_t o0[16], o1[16];
                            tmem_ld16(ob + hc * 16, o0);                 // (P_hi + P_lo) V_hi
                            tmem_ld16(ob + DH + hc * 16, o1);            // P_hi V_lo
                            tmem_ld_wait();
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                float a = __uint_as_float(o0[2 * j]), bq = __uint_as_float(o0[2 * j + 1]);
                                ap_add2(a, bq, __uint_as_float(o1[2 * j]), __uint_as_float(o1[2 * j + 1]));
                                ap_mul2(a, bq, inv, inv);
                                ap_split_pack(a, bq, oh[hc * 8 + j], ol[hc * 8 + j]);
                            }
                        }
                    }
                    tc_fence_before();
                    mbar_arrive(&o_free[g]);
                    if (warp_live && row < S) {
                        const size_t off = static_cast<size_t>(t0 + row) * p.H + (2 * hp + g) * DH;
                        uint4* dh = reinterpret_cast<uint4*>(p.ctx_hi + off);
                        uint4* dl = reinterpret_cast<uint4*>(p.ctx_lo + off);
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            dh[q] = make_uint4(oh[4 * q], oh[4 * q + 1], oh[4 * q + 2], oh[4 * q + 3]);
                            dl[q] = make_uint4(ol[4 * q], ol[4 * q + 1], ol[4 * q + 2], ol[4 * q + 3]);
                        }
                    }
                }
            }
        }
    } else {
        // =========================== softmax of head g: thread = query row, two warps per row ===========================
        const int g = (warp - 8) >> 3;
        const int half = ((warp - 8) >> 2) & 1;                  // which chunks (c & 1)
        const int quad = warp & 3;
        const int r = quad * 32 + static_cast<int>(lane);
        const int htid = ((warp - 8) & 3) * 32 + static_cast<int>(lane);
        float* xm = xch + (g * 2 + half) * kAtcRows;
        const float* xo = xch + (g * 2 + (half ^ 1)) * kAtcRows;
        const uint32_t tb = tmem_addr(tmem_base, quad * 32, g * kAtcBufCols);
        uint32_t cnt = 0;
        for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
            const int b = w / hpairs;
            const int S = __ldg(p.cu + b + 1) - __ldg(p.cu + b);
            const int nchunk = (S + 31) >> 5;
            for (int r0 = 0; r0 < S; r0 += kAtcRows, ++cnt) {
                const bool warp_live = r0 + quad * 32 < S;
                mbar_wait(&s_full[g], cnt & 1);
                tc_fence_after();
                float m = -INFINITY;
                if (warp_live) {
                    float m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;   // four independent chains: fmaxf does not reassociate
                    for (int c = half; c < nchunk; c += 2) {
                        uint32_t sv[32];
                        tmem_ld32(tb + c * 32, sv);
                        tmem_ld_wait();
                        if (c * 32 + 32 > S) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) if (c * 32 + j >= S) sv[j] = 0xFF800000u;   // -inf
                        }
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            m = fmaxf(m, __uint_as_float(sv[j])); m1 = fmaxf(m1, __uint_as_float(sv[j + 1]));
                            m2 = fmaxf(m2, __uint_as_float(sv[j + 2])); m3 = fmaxf(m3, __uint_as_float(sv[j + 3]));
                        }
                    }
                    m = fmaxf(fmaxf(m, m1), fmaxf(m2, m3));
                }
                mbar_wait(&o_free[g], (cnt & 1) ^ 1);          // the output warps have taken the previous tile's row sums out of xch
                xm[r] = m;                                       // (they did so while S of this tile was being computed: no stall)
                bar_sync_named(1 + g * 4 + quad, 64);            // the two warps that share these 32 rows (same SM sub-partition)
                m = fmaxf(m, xo[r]);
                bar_sync_named(1 + g * 4 + quad, 64);
                float l0 = 0.f, l1 = 0.f;
                for (int c = half; c < nchunk; c += 2) {
                    if (warp_live) {
                        uint32_t sv[32];
                        tmem_ld32(tb + c * 32, sv);
                        tmem_ld_wait();
                        if (c * 32 + 32 > S) {                       // ragged last chunk (warp-uniform): keys past the end weigh nothing
#pragma unroll
                            for (int j = 0; j < 32; ++j) if (c * 32 + j >= S) sv[j] = 0xFF800000u;   // exp2(-inf) = +0
                        }
#pragma unroll
                        for (int hc = 0; hc < 2; ++hc) {             // 16 keys at a time: 8 packed hi + 8 packed lo columns
                            uint32_t ph[8], pl[8];
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                float a = __uint_as_float(sv[hc * 16 + 2 * j]), bq = __uint_as_float(sv[hc * 16 + 2 * j + 1]);
                                ap_sub2(a, bq, m, m);
                                a = atc_exp2(a); bq = atc_exp2(bq);
                                ap_add2(l0, l1, a, bq);
                                ap_split_pack(a, bq, ph[j], pl[j]);
                            }
                            tmem_st8(tb + c * 32 + hc * 8, ph);
                            tmem_st8(tb + c * 32 + 16 + hc * 8, pl);
                        }
                        tmem_st_wait();
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&p_full[g * kAtcMaxChunks + c]);     // one arrival per owning warp: no CTA-level barrier
                }
                xm[r] = l0 + l1;                                 // row sum for the output warps (every warp of the head is past pass 1)
                mbar_arrive(&l_full[g]);
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 1) tmem_dealloc<512>(tmem_base);
}
