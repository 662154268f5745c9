// Coarse top-k scan of the flat index (sm_100a) and its selection kernel.  Included by rmu_index.cu inside
// namespace rmu, after exact_metric / block_bitonic_desc / block_radix_select / warp_bitonic_desc.
//
// Stands behind the reference's brute-force search (col.search of the retriever built at
// server/RAGHelper.py:497-499; Milvus-lite FLAT / pgvector sequential scan on the CPU).
//
// Geometry.  The fp32 corpus streams HBM -> smem through TMA exactly once as 16 KB boxes (128 rows x 32
// floats, SWIZZLE_128B) and is consumed in place as the **A operand** of tcgen05.mma.kind::tf32.  The kernel runs
// as CTA PAIRS (cta_group::2, M = 256): each CTA of a pair streams its OWN 128-row tile, the queries are the B
// operand (N = NQ <= 128 of them per launch), and -- the point of the pairing -- each CTA keeps only HALF of the
// query block resident in shared memory ([K block][NQ/2 rows x 128 B], loaded once by TMA, zero filled past
// nq / dim); the tensor core reads both halves.  At 64 queries x 384 dims that is 48 KB per SM instead of 96 KB,
// which leaves 176 KB of every SM's shared memory for corpus boxes in flight: measured on this part, the HBM
// stream needs ~190 KB in flight per SM to saturate (128 KB: 5.3-5.7 TB/s; TMA-multicast clusters, which make
// every SM of a cluster hold the SAME bytes, fall to 1/cluster-size of that).
// The accumulator D[128 rows x NQ queries] of each CTA takes NQ TMEM columns, so 512 / NQ accumulators fit: the
// MMA issuer runs up to eight tiles ahead of the epilogue and neither waits for the other in steady state (the
// round-1 kernel kept the queries in TMEM, had room for one accumulator, and was bound by MMA and epilogue
// taking turns).
//
// Epilogue: thread = corpus row (TMEM lane), column = query.  Each score is compared with the query's running
// threshold tau; the few that pass are appended (shared-memory counter, global list) to the (CTA, query)
// candidate list.  At tile boundaries lists past 95 entries are sorted by one warp each (warp-shuffle bitonic network)
// and cut to their best 64; the 64th key becomes the list's floor.
// Threshold exchange without a second launch: whenever a list is sorted, its 16th best key is published with an
// atomicMax into gmax[query][cluster % groups].  If every one of `groups` disjoint groups of clusters contains a
// cluster with >= 16 keys >= v, then >= 16 * groups rows score >= v: tau = min over groups of the group maxima is
// a valid lower bound of the (16 * groups)-th best key of the whole corpus.  groups = KSEL / 16, so nothing that
// belongs to the global best KSEL is ever rejected (ties at tau are covered by the certificate's bound).
// gmax entries are tagged with a per-search epoch in their high word, so they never need clearing.
#pragma once

constexpr int kTileRows = 128;                   // corpus rows per CTA tile = TMEM lanes (the pair's MMA has M = 256)
constexpr int kBoxBytes = kTileRows * 128;       // one TMA box: 128 rows x 32 fp32
constexpr int kScanMaxThreads = 320;             // warp 0 TMA, warp 1 MMA + TMEM alloc, then 4 or 8 epilogue warps
__host__ __device__ constexpr int scan_epi_warps(int nq) { return nq >= 64 ? 8 : 4; }   // two warps per TMEM lane quadrant split the queries
constexpr int kAccBufsMax = 8;                   // TMEM accumulators (NQ columns each): min(8, 512 / NQ)
constexpr int kListCap = 256;                    // slots of a (CTA, query) candidate list
constexpr int kListKeep = 64;                    // entries a list keeps when it is sorted and cut
constexpr int kListTrig = 95;                    // a list longer than this at a tile boundary is sorted and cut
                                                 // (one tile adds <= 128 entries to a list: 95 + 128 < kListCap)
constexpr int kPubRank = 16;                     // the published key of a list: its 16th best
constexpr int kGroupsMax = 16;                   // gmax row length; KSEL <= 16 * kPubRank = 256
constexpr int kScanStateBytes = 2048;            // mbarriers + per-query state behind the ring
constexpr int kScanQOpMax = 96 * 1024;           // shared memory the resident half of the query operand may take
constexpr int kScanMaxStages = 16;
constexpr int kScanKD = 2;                       // TMA boxes (K blocks) per pipeline stage
constexpr int kScanMaxQ = 128;                   // queries per launch (MMA N)

struct ScanParams {
    int nq;                    // live queries of this launch (<= NQ); query j = row j of tmap_q
    int dim;
    long long n;               // rows in the index
    int ntiles;                // ceil(n / 128)
    int nstages;               // ring depth, in stages of kScanKD boxes
    int metric;
    const float* rscale;       // [n] 1/||x|| (cosine), used unless the corpus is unit-norm
    const float* rbias;        // [n] -0.5 ||x||^2 (L2), used unless the corpus is unit-norm
    const unsigned* stats_bits;   // [1] = max over rows of | ||x||^2 - 1 | (float bits): < 1e-6 => unit rows
    unsigned long long* lists; // [grid][NQ][kListCap]
    int* counts;               // [grid][NQ] entries valid in each list when the launch ends
    float* floors;             // [grid][NQ] largest score the list ever cut away (-inf: never cut)
    unsigned long long* gmax;  // [NQ][kGroupsMax]  (epoch << 32 | ordered score), see above
    unsigned epoch;
    int groups;                // 0: no exchange (grids smaller than the group count)
    float* dbg;                // diagnostics: raw accumulators of the first 256 rows, [NQ][256]
    // second pass for queries whose certificate failed ("pool mode", fixed_tau != nullptr): every row whose coarse key
    // beats the query's FIXED threshold is appended to a per-query pool; no lists, no exchange
    const float* fixed_tau;    // [NQ] thresholds of the launch's query slots
    unsigned long long* pool;  // [NQ][pool_cap]
    int* pool_cnt;             // [NQ] entries appended (may exceed pool_cap: overflow, the query stays flagged)
    int pool_cap;
    const int* nq_dev;         // nullable: live queries of the pass (device count of flagged queries)
    int q_off;                 // this launch serves slots q_off .. q_off + nq - 1 of them
};

// sort one candidate list (n <= 32 * E entries) descending, keep its best kListKeep, publish its kPubRank-th key
template <int E>
__device__ __forceinline__ void scan_sort_list(unsigned long long* b, int n, int& cnt, float& floor_v,
                                               unsigned long long* gslot, unsigned epoch) {
    const unsigned lane = lane_id();
    unsigned long long v[E];
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const int i = e * 32 + static_cast<int>(lane);
        v[e] = (i < n) ? b[i] : 0ull;
    }
    warp_bitonic_desc<E>(v);
    b[lane] = v[0];
    b[32 + lane] = v[1];
    const unsigned long long k_pub = __shfl_sync(0xffffffffu, v[0], kPubRank - 1);
    const unsigned long long k_keep = __shfl_sync(0xffffffffu, v[1], 31);
    if (lane == 0) {
        if (n > kListKeep) { cnt = kListKeep; floor_v = fmaxf(floor_v, key_score(k_keep)); }
        if (n >= kPubRank && gslot != nullptr)
            atomicMax(gslot, (static_cast<unsigned long long>(epoch) << 32) | (k_pub >> 32));
    }
}

// D[tmem of both CTAs] (+)= A[smem of both: 2 x 128 rows] * B[smem of both: 2 x N/2 rows]^T, tf32
__device__ __forceinline__ void mma_tf32_ss_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                 uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// PAIR = true: clusters of two CTAs, cta_group::2 (the protocol of gemm_f16x3_pair_kernel):
//   full[s]  (the leader's is the one waited on): the leader's arrive.expect_tx with the bytes of BOTH CTAs; the
//            cta_group::2 loads of both CTAs credit the leader's barrier (the peer cannot run a phase ahead on a slot:
//            it refills the slot only after the leader's commit released it);
//   empty[s], acc_full[b]: per CTA, signalled by the leader's tcgen05.commit multicast to both CTAs;
//   acc_empty[b] (leader's): one arrival per epilogue warp of either CTA;
//   qbar (leader's): the resident query halves of both CTAs, same scheme as full[].
// PAIR = false: one CTA, cta_group::1, the whole query block resident.
template <int NQ, bool PAIR>
__global__ void __launch_bounds__(64 + 32 * scan_epi_warps(NQ), 1)
scan_rows_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_q, const ScanParams p) {
    constexpr int NCTA = PAIR ? 2 : 1;
    constexpr int NQH = NQ / NCTA;                       // query rows resident in THIS CTA
    constexpr int STAGE_BYTES = kScanKD * kBoxBytes;
    constexpr int QBLK_BYTES = NQH * 128;                // one K block of this CTA's part of the query operand
    constexpr int CW = NQ < 32 ? NQ : 32;                // accumulator columns per TMEM load
    constexpr int EPW = scan_epi_warps(NQ);              // epilogue warps: with 8, each TMEM lane quadrant has two, half the queries each
    constexpr int CPW = NQ / (EPW / 4);                  // query columns one warp looks at
    constexpr int ETH = 32 * EPW;
    constexpr int NBUF = 512 / NQ < kAccBufsMax ? 512 / NQ : kAccBufsMax;
    constexpr uint32_t IDESC = umma_idesc(2 /*tf32*/, NCTA * kTileRows, NQ);
    static_assert(NQ == 16 || NQ == 32 || NQ == 64 || NQ == 128, "queries per launch");

    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment by OFFSET (a pointer round-trip through an integer loses the shared address space)
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const int KB = (p.dim + 31) / 32;                    // 128-byte K blocks
    const int NST = (KB + kScanKD - 1) / kScanKD;        // pipeline stages per tile
    uint8_t* qop = smem;
    uint8_t* ring = smem + KB * QBLK_BYTES;
    uint8_t* state = ring + p.nstages * STAGE_BYTES;
    uint64_t* full = reinterpret_cast<uint64_t*>(state);
    uint64_t* empty = full + kScanMaxStages;
    uint64_t* acc_full = empty + kScanMaxStages;
    uint64_t* acc_empty = acc_full + kAccBufsMax;
    uint64_t* qbar = acc_empty + kAccBufsMax;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(qbar + 1);
    float* tau_s = reinterpret_cast<float*>(state + 512);       // [NQ] running threshold of each query
    int* cnt_s = reinterpret_cast<int*>(state + 1024);          // [NQ] entries in each list of this CTA
    float* floor_s = reinterpret_cast<float*>(state + 1536);    // [NQ] largest score each list ever cut away

    int nq_live = p.nq;
    if (p.nq_dev != nullptr) {                           // second pass: nothing flagged in this launch's range -> nothing to do
        nq_live = min(p.nq, __ldg(p.nq_dev) - p.q_off);
        if (nq_live <= 0) return;                        // uniform over the grid: no barrier, no TMEM allocation yet
    }
    const bool pool_mode = p.fixed_tau != nullptr;
    const int warp = threadIdx.x >> 5;
    const unsigned lane = lane_id();
    const int rank = PAIR ? static_cast<int>(cluster_ctarank()) : 0;   // 0 = leader (issues the MMAs)
    const int cta = blockIdx.x;
    const int unit = blockIdx.x / NCTA, nunits = gridDim.x / NCTA;     // CTA or CTA pair
    const int nutiles = (p.ntiles + NCTA - 1) / NCTA;    // tiles of NCTA * 128 rows; CTA `rank` takes tile NCTA * u + rank

    if (threadIdx.x == 0) {
        for (int i = 0; i < p.nstages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        for (int i = 0; i < NBUF; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], EPW * NCTA); }
        mbar_init(qbar, 1);
        fence_mbar_init();
        prefetch_tmap(&tmap_x);
        prefetch_tmap(&tmap_q);
    }
    if (PAIR) cluster_sync_all();                        // barriers of both CTAs exist before anyone signals them
    if (warp == 1) {
        if (PAIR) tmem_alloc_pair<512>(tmem_slot);
        else tmem_alloc<512>(tmem_slot);
    }
    tc_fence_before();
    if (PAIR) cluster_sync_all();
    else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // =========================== TMA producer ===========================
        if (elect_one()) {
            if (rank == 0) mbar_arrive_expect_tx(qbar, static_cast<uint32_t>(NCTA * KB * QBLK_BYTES));
            for (int kb = 0; kb < KB; ++kb) {
                if (PAIR) tma_load_2d_pair(qop + kb * QBLK_BYTES, &tmap_q, kb * 32, rank * NQH, qbar, kEvictLast);
                else tma_load_2d(qop + kb * QBLK_BYTES, &tmap_q, kb * 32, 0, qbar, kEvictLast);
            }
            int slot = 0;
            uint32_t phase = 0;
            for (int u = unit; u < nutiles; u += nunits) {
                const int t = NCTA * u + rank;                   // this CTA's 128-row tile (past the end: zeros)
                for (int s = 0; s < NST; ++s) {
                    mbar_wait(&empty[slot], phase ^ 1);
                    if (rank == 0) mbar_arrive_expect_tx(&full[slot], NCTA * STAGE_BYTES);
#pragma unroll
                    for (int kk = 0; kk < kScanKD; ++kk) {
                        // K blocks past the row end are out of bounds: they arrive as zeros and still count their bytes
                        uint8_t* dst = ring + slot * STAGE_BYTES + kk * kBoxBytes;
                        if (PAIR) tma_load_2d_pair(dst, &tmap_x, (s * kScanKD + kk) * 32, t * kTileRows, &full[slot], kEvictFirst);
                        else tma_load_2d(dst, &tmap_x, (s * kScanKD + kk) * 32, t * kTileRows, &full[slot], kEvictFirst);
                    }
                    if (++slot == p.nstages) { slot = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // =========================== MMA issuer (leader only) ===========================
        if (rank == 0 && elect_one()) {
            mbar_wait(qbar, 0);                                  // the query operand is resident (both halves)
            tc_fence_after();
            int slot = 0;
            uint32_t phase = 0;
            int i = 0;
            for (int u = unit; u < nutiles; u += nunits, ++i) {
                const int buf = i % NBUF;
                const uint32_t use = static_cast<uint32_t>(i / NBUF);
                mbar_wait(&acc_empty[buf], (use & 1) ^ 1);
                tc_fence_after();
                const uint32_t d_addr = tmem_base + buf * NQ;
                for (int s = 0; s < NST; ++s) {
                    mbar_wait(&full[slot], phase);
                    tc_fence_after();
#pragma unroll
                    for (int kk = 0; kk < kScanKD; ++kk) {
                        const int kb = s * kScanKD + kk;
                        if (kb < KB) {
                            const uint64_t adesc = umma_desc_sw128_kmajor(smem_u32(ring + slot * STAGE_BYTES + kk * kBoxBytes));
                            const uint64_t bdesc = umma_desc_sw128_kmajor(smem_u32(qop + kb * QBLK_BYTES));
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                if (kb * 32 + k * 8 < p.dim) {
                                    const uint64_t ko = static_cast<uint64_t>(k * 2);
                                    if (PAIR) mma_tf32_ss_pair(d_addr, adesc + ko, bdesc + ko, IDESC, (kb | k) != 0 ? 1u : 0u);
                                    else mma_tf32_ss(d_addr, adesc + ko, bdesc + ko, IDESC, (kb | k) != 0 ? 1u : 0u);
                                }
                            }
                        }
                    }
                    if (PAIR) tc_commit_pair(&empty[slot]);      // both CTAs' ring slots are free again
                    else tc_commit(&empty[slot]);
                    if (++slot == p.nstages) { slot = 0; phase ^= 1; }
                }
                if (PAIR) tc_commit_pair(&acc_full[buf]);
                else tc_commit(&acc_full[buf]);
            }
        }
    } else {
        // =========================== epilogue: thread = corpus row ===========================
        const int quad = warp & 3;                               // TMEM lane quadrant this warp may touch
        const int er = quad * 32 + static_cast<int>(lane);       // row of the tile
        const int ew = warp - 2;
        const int et = ew * 32 + static_cast<int>(lane);         // 0..ETH-1: per-query duties
        const int c0 = (ew >> 2) * (CPW / CW);                   // first 32-column chunk of this warp
        unsigned long long* mylists = p.lists + static_cast<size_t>(cta) * NQ * kListCap;
        const bool unit_rows = __uint_as_float(__ldg(p.stats_bits + 1)) < 1e-6f;
        const bool has_sc = p.metric == RMU_METRIC_COSINE && !unit_rows;
        const bool has_bi = p.metric == RMU_METRIC_L2 && !unit_rows;
        const bool qlive = et < NQ && et < nq_live;
        if (et < NQ) {
            tau_s[et] = qlive ? (pool_mode ? __ldg(p.fixed_tau + et) : -INFINITY) : INFINITY;
            cnt_s[et] = 0;
            floor_s[et] = -INFINITY;
        }
        bar_sync_named(1, ETH);
        bool mine = false;                                       // this thread pushed a list past kListTrig
        int i = 0;
        for (int u = unit; u < nutiles; u += nunits, ++i) {
            const int buf = i % NBUF;
            const uint32_t use = static_cast<uint32_t>(i / NBUF);
            const long long row = (static_cast<long long>(NCTA) * u + rank) * kTileRows + er;
            const bool valid = row < p.n;
            float sc = 1.f, bi = 0.f;
            if (has_sc && valid) sc = __ldg(p.rscale + row);
            if (has_bi && valid) bi = __ldg(p.rbias + row);
            mbar_wait(&acc_full[buf], use & 1);
            tc_fence_after();
#pragma unroll
            for (int cc = 0; cc < CPW / CW; ++cc) {
                const int c = c0 + cc;
                uint32_t r[CW];
                if constexpr (CW == 32) tmem_ld32(tmem_addr(tmem_base, quad * 32, buf * NQ + c * CW), r);
                else tmem_ld16(tmem_addr(tmem_base, quad * 32, buf * NQ + c * CW), r);
                tmem_ld_wait();
                if (cc == CPW / CW - 1) {                        // last TMEM read of this tile: hand the accumulator back
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {                             // the leader's MMA thread owns the hand-back
                        if (PAIR) mbar_arrive_cluster(&acc_empty[buf], 0);
                        else mbar_arrive(&acc_empty[buf]);
                    }
                }
                if (p.dbg != nullptr && i == 0 && NCTA * unit + rank < 2) {     // tiles 0 and 1 = the first 256 rows
#pragma unroll
                    for (int j = 0; j < CW; ++j) p.dbg[(c * CW + j) * 2 * kTileRows + (NCTA * unit + rank) * kTileRows + er] = __uint_as_float(r[j]);
                }
                float v[CW];
                unsigned m = 0u;
#pragma unroll
                for (int j4 = 0; j4 < CW / 4; ++j4) {
                    const float4 tq = *reinterpret_cast<const float4*>(tau_s + c * CW + j4 * 4);   // broadcast read
                    v[4 * j4 + 0] = fmaf(__uint_as_float(r[4 * j4 + 0]), sc, bi);
                    v[4 * j4 + 1] = fmaf(__uint_as_float(r[4 * j4 + 1]), sc, bi);
                    v[4 * j4 + 2] = fmaf(__uint_as_float(r[4 * j4 + 2]), sc, bi);
                    v[4 * j4 + 3] = fmaf(__uint_as_float(r[4 * j4 + 3]), sc, bi);
                    m |= (v[4 * j4 + 0] > tq.x) ? (1u << (4 * j4 + 0)) : 0u;
                    m |= (v[4 * j4 + 1] > tq.y) ? (1u << (4 * j4 + 1)) : 0u;
                    m |= (v[4 * j4 + 2] > tq.z) ? (1u << (4 * j4 + 2)) : 0u;
                    m |= (v[4 * j4 + 3] > tq.w) ? (1u << (4 * j4 + 3)) : 0u;
                }
                if (!valid) m = 0u;
                if (__any_sync(0xffffffffu, m != 0u)) {          // rare once the thresholds have risen
#pragma unroll
                    for (int j = 0; j < CW; ++j) {
                        if (m & (1u << j)) {
                            const int ql = c * CW + j;
                            if (pool_mode) {
                                const int pos = atomicAdd(p.pool_cnt + ql, 1);
                                if (pos < p.pool_cap) p.pool[static_cast<size_t>(ql) * p.pool_cap + pos] = make_key(v[j], static_cast<uint32_t>(row));
                            } else {
                                const int pos = atomicAdd(&cnt_s[ql], 1);
                                mylists[ql * kListCap + pos] = make_key(v[j], static_cast<uint32_t>(row));
                                mine |= pos >= kListTrig;
                            }
                        }
                    }
                }
            }
            if (pool_mode) continue;
            // ---- tile boundary: sort + cut the lists that grew past kListTrig (every sort publishes the list's 16th key, so
            // the thresholds of all CTAs rise together: ~5 sorts per list over a 10M-row scan, most of them in the first tiles)
            const bool any = bar_red_or_named(1, ETH, mine);
            mine = false;
            if (any) {
                for (int ql = ew; ql < NQ; ql += EPW) {
                    const int n = cnt_s[ql];
                    if (n > kListTrig) {
                        unsigned long long* gslot = p.groups > 0 ? p.gmax + static_cast<size_t>(ql) * kGroupsMax + (cta % p.groups) : nullptr;
                        if (n <= 128) scan_sort_list<4>(mylists + ql * kListCap, n, cnt_s[ql], floor_s[ql], gslot, p.epoch);
                        else scan_sort_list<8>(mylists + ql * kListCap, n, cnt_s[ql], floor_s[ql], gslot, p.epoch);
                    }
                }
                bar_sync_named(1, ETH);
            }
            // ---- refresh this query's threshold from what the other CTAs published
            if (qlive) {
                float tg = -INFINITY;
                if (p.groups > 0) {
                    tg = INFINITY;
                    const ulonglong2* g2 = reinterpret_cast<const ulonglong2*>(p.gmax + static_cast<size_t>(et) * kGroupsMax);
                    for (int g = 0; g < p.groups; g += 2) {
                        const ulonglong2 w = __ldcg(g2 + (g >> 1));
                        const float s0 = static_cast<unsigned>(w.x >> 32) == p.epoch ? ordered_to_f32(static_cast<uint32_t>(w.x)) : -INFINITY;
                        const float s1 = static_cast<unsigned>(w.y >> 32) == p.epoch ? ordered_to_f32(static_cast<uint32_t>(w.y)) : -INFINITY;
                        tg = fminf(tg, fminf(s0, g + 1 < p.groups ? s1 : INFINITY));
                    }
                }
                tau_s[et] = fmaxf(tg, floor_s[et]);
            }
        }
        if (et < NQ && !pool_mode) {
            p.counts[cta * NQ + et] = cnt_s[et];
            p.floors[cta * NQ + et] = floor_s[et];
        }
    }

    tc_fence_before();
    if (PAIR) cluster_sync_all();                        // both CTAs are done with TMEM and each other's smem
    else __syncthreads();
    tc_fence_after();
    if (warp == 1) {
        if (PAIR) tmem_dealloc_pair<512>(tmem_base);
        else tmem_dealloc<512>(tmem_base);
    }
}

// =====================================================================================================
// selection: union of the (cluster, query) lists -> best KSEL coarse candidates -> exact fp32 re-score ->
// sort -> top-k + certificate.  One CTA per query.
// =====================================================================================================
constexpr int kSel2Threads = 512;
constexpr int kSel2Cap = 16384;                  // candidates gathered into shared memory (128 KB); more -> radix select over the lists
constexpr int kSel2Max = 1024;                   // coarse candidates re-scored exactly, at most

struct SelectParams {
    const unsigned long long* lists; const int* counts; const float* floors; const unsigned long long* gmax;
    int ncl, qb;               // lists per query (CTAs of the scan launch), list blocks per CTA (NQ)
    unsigned epoch; int groups;
    int ksel;                  // coarse candidates re-scored exactly (<= kSel2Max)
    const float* x; long long n; int dim; int metric;
    const float* q;            // [launch queries, dim]
    int q0;                    // index of the launch's first query in the outputs
    int k; long long id_offset;
    const unsigned* stats_bits;   // [0] max ||x|| , [1] max | ||x||^2 - 1 |
    float eps_rel;
    float* out_scores; long long* out_ids; int* flags;
    float* tau2;               // [nq] per query: the coarse-key threshold a second pass must use when the query is flagged
};

// exact_metric with the four fmaf chains of one (query, row) pair spread over the four lanes of a quad (lane & 3 = chain):
// every chain sees the same elements in the same order and the partial sums are combined as (a0 + a1) + (a2 + a3), so the
// result is bit-identical to exact_metric.  All four lanes return the value.
__device__ __forceinline__ float exact_metric_quad(const float* __restrict__ q, const float* __restrict__ x, int D, int metric,
                                                   float qnorm) {
    const int c = static_cast<int>(lane_id() & 3u);
    const int D4 = D & ~3;
    float a = 0.f, nn = 0.f;
    if (metric == RMU_METRIC_L2) {
        for (int d = c; d < D4; d += 4) { const float e = q[d] - x[d]; a = fmaf(e, e, a); }
        if (c == 0) for (int d = D4; d < D; ++d) { const float e = q[d] - x[d]; a = fmaf(e, e, a); }
    } else {
        for (int d = c; d < D4; d += 4) {
            const float xv = x[d];
            a = fmaf(q[d], xv, a);
            if (metric == RMU_METRIC_COSINE) nn = fmaf(xv, xv, nn);
        }
        if (c == 0) for (int d = D4; d < D; ++d) {
            a = fmaf(q[d], x[d], a);
            if (metric == RMU_METRIC_COSINE) nn = fmaf(x[d], x[d], nn);
        }
    }
    const unsigned qb = lane_id() & ~3u;
    const float a0 = __shfl_sync(0xffffffffu, a, qb), a1 = __shfl_sync(0xffffffffu, a, qb + 1);
    const float a2 = __shfl_sync(0xffffffffu, a, qb + 2), a3 = __shfl_sync(0xffffffffu, a, qb + 3);
    const float s = (a0 + a1) + (a2 + a3);
    if (metric != RMU_METRIC_COSINE) return s;
    const float n0 = __shfl_sync(0xffffffffu, nn, qb), n1 = __shfl_sync(0xffffffffu, nn, qb + 1);
    const float n2 = __shfl_sync(0xffffffffu, nn, qb + 2), n3 = __shfl_sync(0xffffffffu, nn, qb + 3);
    const float xn = sqrtf((n0 + n1) + (n2 + n3));
    const float den = qnorm * xn;
    return den > 0.f ? s / den : 0.f;
}

__global__ void __launch_bounds__(kSel2Threads) select_rescore_kernel(const SelectParams p) {
    __shared__ unsigned long long sel[kSel2Max];
    __shared__ int hist[256];
    __shared__ float red[32];
    __shared__ int s_n, s_nsel;
    __shared__ unsigned long long s_prefix;
    __shared__ int s_remaining, s_ties;
    __shared__ float s_tau;
    extern __shared__ unsigned long long sel_dyn[];  // cand [kSel2Cap], then the query [dim] floats
    unsigned long long* cand = sel_dyn;
    float* qs = reinterpret_cast<float*>(sel_dyn + kSel2Cap);

    const int f = blockIdx.x;
    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;

    // ||q|| in the summation order of exact_scan_kernel (256 threads, stride 256), so that cosine scores of the
    // two paths are bit-identical
    float part = 0.f;
    if (tid < 256) {
        for (int d = tid; d < p.dim; d += 256) {
            const float v = p.q[static_cast<long long>(f) * p.dim + d];
            qs[d] = v;
            part = fmaf(v, v, part);
        }
    }
    const float qnorm = sqrtf(block_sum(part, red));

    // ---- what the scan may have rejected: everything <= tau (exchange) or <= a list's floor (cuts)
    if (tid == 0) {
        float tg = -INFINITY;
        if (p.groups > 0) {
            tg = INFINITY;
            for (int g = 0; g < p.groups; ++g) {
                const unsigned long long w = p.gmax[static_cast<size_t>(f) * kGroupsMax + g];
                tg = fminf(tg, static_cast<unsigned>(w >> 32) == p.epoch ? ordered_to_f32(static_cast<uint32_t>(w)) : -INFINITY);
            }
        }
        s_tau = tg;
        s_n = 0;
        s_nsel = 0;
    }
    float fl = -INFINITY;
    for (int c = tid; c < p.ncl; c += blockDim.x) fl = fmaxf(fl, p.floors[c * p.qb + f]);
    for (int o = 16; o > 0; o >>= 1) fl = fmaxf(fl, __shfl_xor_sync(0xffffffffu, fl, o));
    __syncthreads();
    if (lane == 0) red[warp] = fl;
    __syncthreads();
    fl = red[0];
    for (int w = 1; w < kSel2Threads / 32; ++w) fl = fmaxf(fl, red[w]);
    const float tau = s_tau;
    float bound = fmaxf(tau, fl);                // coarse upper bound of every row that is in no list
    __syncthreads();

    // ---- gather the entries above tau (two lists per warp step: the count loads of both are in flight together)
    for (int c = 2 * warp; c < p.ncl; c += 2 * (kSel2Threads / 32)) {
        const int n0 = p.counts[c * p.qb + f];
        const int n1 = c + 1 < p.ncl ? p.counts[(c + 1) * p.qb + f] : 0;
        const unsigned long long* b0 = p.lists + static_cast<size_t>(c * p.qb + f) * kListCap;
        const unsigned long long* b1 = b0 + static_cast<size_t>(p.qb) * kListCap;
        for (int e = lane; e < n0 + n1; e += 32) {
            const unsigned long long key = e < n0 ? b0[e] : b1[e - n0];
            if (key_score(key) > tau) {
                const int pos = atomicAdd(&s_n, 1);
                if (pos < kSel2Cap) cand[pos] = key;
            }
        }
    }
    __syncthreads();
    const int n = s_n;
    int ncand;
    if (n <= p.ksel) {                           // every survivor is re-scored
        for (int i = tid; i < n; i += blockDim.x) sel[i] = cand[i];
        ncand = n;
    } else {
        // the ksel-th best key by radix select (shared memory when the survivors fit, else over the lists), then collect
        unsigned long long T;
        if (n <= kSel2Cap) {
            auto load_key = [&](long long idx) -> unsigned long long { return cand[idx]; };
            T = block_radix_select(load_key, n, p.ksel, hist, &s_prefix, &s_remaining, &s_ties);
            __syncthreads();
            for (int i = tid; i < n; i += blockDim.x) {
                const unsigned long long key = cand[i];
                if (key >= T) { const int pos = atomicAdd(&s_nsel, 1); if (pos < kSel2Max) sel[pos] = key; }
            }
        } else {
            const long long total = static_cast<long long>(p.ncl) * kListCap;
            auto load_key = [&](long long idx) -> unsigned long long {
                const int c = static_cast<int>(idx / kListCap), e = static_cast<int>(idx % kListCap);
                if (e >= p.counts[c * p.qb + f]) return 0ull;
                const unsigned long long key = p.lists[static_cast<size_t>(c * p.qb + f) * kListCap + e];
                return key_score(key) > tau ? key : 0ull;
            };
            T = block_radix_select(load_key, total, p.ksel, hist, &s_prefix, &s_remaining, &s_ties);
            __syncthreads();
            for (long long idx = tid; idx < total; idx += blockDim.x) {
                const unsigned long long key = load_key(idx);
                if (key != 0ull && key >= T) { const int pos = atomicAdd(&s_nsel, 1); if (pos < kSel2Max) sel[pos] = key; }
            }
        }
        __syncthreads();
        ncand = min(s_nsel, p.ksel);
        bound = fmaxf(bound, key_score(T));      // list entries that were not selected are below T
    }
    __syncthreads();

    // ---- exact re-score, a quad of lanes per candidate (the same arithmetic as the exact scan: bit-identical scores)
    for (int c0 = 0; c0 < ncand; c0 += kSel2Threads / 4) {
        const int c = c0 + (tid >> 2);
        const bool live = c < ncand;
        const uint32_t row = live ? key_row(sel[c]) : 0u;
        const float v = exact_metric_quad(qs, p.x + static_cast<long long>(row) * p.dim, p.dim, p.metric, qnorm);
        __syncwarp();
        if (live && (tid & 3) == 0) sel[c] = make_key(metric_to_rank(v, p.metric), row);
    }
    int m2 = 32;
    while (m2 < ncand) m2 <<= 1;
    __syncthreads();
    for (int i = ncand + tid; i < m2; i += blockDim.x) sel[i] = 0ull;
    block_bitonic_desc(sel, m2);

    // ---- outputs
    const int qg = p.q0 + f;
    const float missing = p.metric == RMU_METRIC_L2 ? INFINITY : -INFINITY;
    for (int j = tid; j < p.k; j += blockDim.x) {
        float s = missing;
        long long id = -1;
        if (j < ncand) {
            const float rk = key_score(sel[j]);
            s = p.metric == RMU_METRIC_L2 ? -rk : rk;
            id = p.id_offset + key_row(sel[j]);
        }
        p.out_scores[static_cast<long long>(qg) * p.k + j] = s;
        p.out_ids[static_cast<long long>(qg) * p.k + j] = id;
    }
    // ---- certificate: every row outside the candidate set has coarse key <= bound; its exact key is at
    //      most eps above.  The k-th exact candidate must beat that strictly.
    if (tid == 0 && p.flags != nullptr) {
        int flag = 0;
        if (bound > -INFINITY) {
            if (ncand < p.k) flag = 1;
            else {
                const float rk = key_score(sel[p.k - 1]);    // rank value of the k-th exact result
                const float xmax = __uint_as_float(p.stats_bits[0]);
                const bool unit = __uint_as_float(p.stats_bits[1]) < 1e-6f && p.metric != RMU_METRIC_IP;
                float kth_key, scale;                        // in the units of the coarse key
                if (p.metric == RMU_METRIC_IP) { kth_key = rk; scale = qnorm * xmax; }
                else if (p.metric == RMU_METRIC_COSINE) { kth_key = rk * qnorm; scale = qnorm; }
                else { kth_key = 0.5f * (qnorm * qnorm + rk) + (unit ? 0.5f : 0.f); scale = qnorm * xmax; }  // rk = -dist
                // unit rows: cosine / L2 keys were scanned as inner products, exact to 1e-6 (||x||^2 = 1 +- 1e-6)
                const float eps = p.eps_rel * scale + 1e-6f * (1.f + fabsf(kth_key)) + (unit ? 4e-6f * (1.f + qnorm) : 0.f);
                if (!(bound + eps < kth_key)) flag = 1;
                // every row whose exact score reaches the k-th candidate's has a coarse key above this:
                if (p.tau2 != nullptr) p.tau2[qg] = kth_key - eps - 1e-6f * (1.f + fabsf(kth_key));
            }
            if (flag && ncand < p.k && p.tau2 != nullptr) p.tau2[qg] = -INFINITY;   // not even k candidates: everything qualifies
        }
        p.flags[qg] = flag;
    }
}


// =====================================================================================================
// second pass for flagged queries: gather them, then (after the pool-mode scan) re-score their pools exactly
// =====================================================================================================
// block j < *nsel: copy flagged query qmap[j] into slot j of qbuf, its threshold into taubuf[j], clear its pool counter
__global__ void pool_prepare_kernel(const float* __restrict__ q, const int* __restrict__ qmap, const int* __restrict__ nsel, int dim,
                                    const float* __restrict__ tau2, float* __restrict__ qbuf, float* __restrict__ taubuf,
                                    int* __restrict__ pool_cnt) {
    const int j = blockIdx.x;
    if (j >= *nsel) return;
    const int qg = qmap[j];
    for (int d = threadIdx.x; d < dim; d += blockDim.x) qbuf[static_cast<size_t>(j) * dim + d] = q[static_cast<size_t>(qg) * dim + d];
    if (threadIdx.x == 0) { taubuf[j] = tau2[qg]; pool_cnt[j] = 0; }
}

struct PoolParams {
    unsigned long long* pool; const int* pool_cnt; int pool_cap;
    const int* qmap; const int* nsel; int max_slots;   // flagged queries beyond max_slots stay flagged
    const float* x; int dim; int metric;
    const float* q;            // all queries [nq, dim]
    int k; long long id_offset;
    float* out_scores; long long* out_ids; int* flags;
};

// block j: every row of the pool (a superset of the rows whose exact score can reach the k-th) is re-scored exactly in
// place, the best k are selected; the result is the exact top-k.  A pool that overflowed leaves the query flagged.
__global__ void __launch_bounds__(kSel2Threads) pool_rescore_kernel(const PoolParams p) {
    __shared__ unsigned long long sel[kSel2Max];
    __shared__ int hist[256];
    __shared__ float red[32];
    __shared__ int s_nsel;
    __shared__ unsigned long long s_prefix;
    __shared__ int s_remaining, s_ties;
    extern __shared__ float pqs[];               // [dim]
    const int j = blockIdx.x;
    if (j >= *p.nsel) return;
    const int qg = p.qmap[j];
    const int tid = threadIdx.x;
    if (j >= p.max_slots) return;                // never scanned: stays flagged
    const int n = p.pool_cnt[j];
    if (n > p.pool_cap) return;                  // overflow: stays flagged, the exact scan answers
    float part = 0.f;
    if (tid < 256) {
        for (int d = tid; d < p.dim; d += 256) {
            const float v = p.q[static_cast<size_t>(qg) * p.dim + d];
            pqs[d] = v;
            part = fmaf(v, v, part);
        }
    }
    const float qnorm = sqrtf(block_sum(part, red));
    if (tid == 0) s_nsel = 0;
    unsigned long long* pool = p.pool + static_cast<size_t>(j) * p.pool_cap;
    for (int c0 = 0; c0 < n; c0 += kSel2Threads / 4) {
        const int c = c0 + (tid >> 2);
        const bool live = c < n;
        const uint32_t row = live ? key_row(pool[c]) : 0u;
        const float v = exact_metric_quad(pqs, p.x + static_cast<long long>(row) * p.dim, p.dim, p.metric, qnorm);
        __syncwarp();
        if (live && (tid & 3) == 0) pool[c] = make_key(metric_to_rank(v, p.metric), row);
    }
    __syncthreads();
    auto load_key = [&](long long idx) -> unsigned long long { return pool[idx]; };
    const unsigned long long T = block_radix_select(load_key, n, p.k, hist, &s_prefix, &s_remaining, &s_ties);
    __syncthreads();
    for (int i = tid; i < n; i += blockDim.x) {
        const unsigned long long key = pool[i];
        if (key >= T) { const int pos = atomicAdd(&s_nsel, 1); if (pos < kSel2Max) sel[pos] = key; }
    }
    __syncthreads();
    const int ncand = min(s_nsel, p.k);
    int m2 = 32;
    while (m2 < min(s_nsel, kSel2Max)) m2 <<= 1;
    for (int i = min(s_nsel, kSel2Max) + tid; i < m2; i += blockDim.x) sel[i] = 0ull;
    block_bitonic_desc(sel, m2);
    const float missing = p.metric == RMU_METRIC_L2 ? INFINITY : -INFINITY;
    for (int jj = tid; jj < p.k; jj += blockDim.x) {
        float sc = missing;
        long long id = -1;
        if (jj < ncand) {
            const float rk = key_score(sel[jj]);
            sc = p.metric == RMU_METRIC_L2 ? -rk : rk;
            id = p.id_offset + key_row(sel[jj]);
        }
        p.out_scores[static_cast<long long>(qg) * p.k + jj] = sc;
        p.out_ids[static_cast<long long>(qg) * p.k + jj] = id;
    }
    if (tid == 0) p.flags[qg] = 0;               // answered exactly
}
