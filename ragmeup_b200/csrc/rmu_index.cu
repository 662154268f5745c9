// Flat (brute-force) vector index for sm_100a.
//
// Stands behind the reference's vector store (Milvus-lite FLAT / pgvector seq-scan, CPU) as it is
// driven from server/RAGHelper.py:388-404 (ctor), :431,:525 (add_documents) and :497-499
// (retriever -> col.search).  SURVEY.md §8 rows a6, a7 (+ gather for a8).
//
// Search = (1) tcgen05 coarse scan: the fp32 corpus streams HBM -> smem through TMA exactly once,
//              is consumed in place as TF32 by tcgen05.mma (queries resident in TMEM as the A
//              operand, scores accumulate in TMEM), and the epilogue keeps, per query, the best
//              KEEP rows of this CTA's row range (running threshold + warp-shuffle bitonic
//              compaction);
//          (2) finalize: radix-select the global best KEEP coarse candidates of every query,
//              re-score them exactly in fp32, sort, and CERTIFY that no excluded row can belong to
//              the top-k (coarse bound + TF32 error bound < exact k-th score);
//          (3) queries that fail the certificate (and corpora too small / shapes the tensor scan
//              does not take) run the exact fp32 CUDA-core scan.
// The ids and scores returned are therefore those of an exact fp32 brute-force search.
#include <algorithm>
#include <mutex>
#include <vector>

#include "rmu_common.h"
#include "rmu_ptx.cuh"

namespace rmu {

// =====================================================================================================
// exact fp32 metric — ONE definition, used by the finalize re-score and by the exact scan, so both
// paths return bit-identical scores.  Fixed summation order: four interleaved fmaf chains.
// =====================================================================================================
__device__ __forceinline__ float exact_metric(const float* __restrict__ q, const float* __restrict__ x, int D,
                                              int metric, float qnorm) {
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    float n0 = 0.f, n1 = 0.f, n2 = 0.f, n3 = 0.f;
    const int D4 = D & ~3;
    if (metric == RMU_METRIC_L2) {
        for (int d = 0; d < D4; d += 4) {
            float e0 = q[d] - x[d], e1 = q[d + 1] - x[d + 1], e2 = q[d + 2] - x[d + 2], e3 = q[d + 3] - x[d + 3];
            a0 = fmaf(e0, e0, a0); a1 = fmaf(e1, e1, a1); a2 = fmaf(e2, e2, a2); a3 = fmaf(e3, e3, a3);
        }
        for (int d = D4; d < D; ++d) { float e = q[d] - x[d]; a0 = fmaf(e, e, a0); }
        return (a0 + a1) + (a2 + a3);
    }
    if (metric == RMU_METRIC_IP) {
        for (int d = 0; d < D4; d += 4) {
            a0 = fmaf(q[d], x[d], a0); a1 = fmaf(q[d + 1], x[d + 1], a1);
            a2 = fmaf(q[d + 2], x[d + 2], a2); a3 = fmaf(q[d + 3], x[d + 3], a3);
        }
        for (int d = D4; d < D; ++d) a0 = fmaf(q[d], x[d], a0);
        return (a0 + a1) + (a2 + a3);
    }
    // cosine
    for (int d = 0; d < D4; d += 4) {
        float x0 = x[d], x1 = x[d + 1], x2 = x[d + 2], x3 = x[d + 3];
        a0 = fmaf(q[d], x0, a0); a1 = fmaf(q[d + 1], x1, a1); a2 = fmaf(q[d + 2], x2, a2); a3 = fmaf(q[d + 3], x3, a3);
        n0 = fmaf(x0, x0, n0); n1 = fmaf(x1, x1, n1); n2 = fmaf(x2, x2, n2); n3 = fmaf(x3, x3, n3);
    }
    for (int d = D4; d < D; ++d) { a0 = fmaf(q[d], x[d], a0); n0 = fmaf(x[d], x[d], n0); }
    float ip = (a0 + a1) + (a2 + a3);
    float xn = sqrtf((n0 + n1) + (n2 + n3));
    float den = qnorm * xn;
    return den > 0.f ? ip / den : 0.f;
}

// The same arithmetic as exact_metric (same four fmaf chains per (query,row), so bit-identical results)
// for QT queries at once: the row is read once for all of them.
template <int QT>
__device__ __forceinline__ void exact_metric_multi(const float* __restrict__ qs /*[QT][D]*/, const float* __restrict__ x,
                                                   int D, int metric, const float* __restrict__ qnorm, float (&out)[QT]) {
    float a[QT][4];
#pragma unroll
    for (int i = 0; i < QT; ++i) a[i][0] = a[i][1] = a[i][2] = a[i][3] = 0.f;
    float n0 = 0.f, n1 = 0.f, n2 = 0.f, n3 = 0.f;
    const int D4 = D & ~3;
    if (metric == RMU_METRIC_L2) {
        for (int d = 0; d < D4; d += 4) {
            const float x0 = x[d], x1 = x[d + 1], x2 = x[d + 2], x3 = x[d + 3];
#pragma unroll
            for (int i = 0; i < QT; ++i) {
                const float* q = qs + i * D;
                const float e0 = q[d] - x0, e1 = q[d + 1] - x1, e2 = q[d + 2] - x2, e3 = q[d + 3] - x3;
                a[i][0] = fmaf(e0, e0, a[i][0]); a[i][1] = fmaf(e1, e1, a[i][1]);
                a[i][2] = fmaf(e2, e2, a[i][2]); a[i][3] = fmaf(e3, e3, a[i][3]);
            }
        }
        for (int d = D4; d < D; ++d) {
#pragma unroll
            for (int i = 0; i < QT; ++i) { const float e = qs[i * D + d] - x[d]; a[i][0] = fmaf(e, e, a[i][0]); }
        }
#pragma unroll
        for (int i = 0; i < QT; ++i) out[i] = (a[i][0] + a[i][1]) + (a[i][2] + a[i][3]);
        return;
    }
    for (int d = 0; d < D4; d += 4) {
        const float x0 = x[d], x1 = x[d + 1], x2 = x[d + 2], x3 = x[d + 3];
        if (metric == RMU_METRIC_COSINE) { n0 = fmaf(x0, x0, n0); n1 = fmaf(x1, x1, n1); n2 = fmaf(x2, x2, n2); n3 = fmaf(x3, x3, n3); }
#pragma unroll
        for (int i = 0; i < QT; ++i) {
            const float* q = qs + i * D;
            a[i][0] = fmaf(q[d], x0, a[i][0]); a[i][1] = fmaf(q[d + 1], x1, a[i][1]);
            a[i][2] = fmaf(q[d + 2], x2, a[i][2]); a[i][3] = fmaf(q[d + 3], x3, a[i][3]);
        }
    }
    for (int d = D4; d < D; ++d) {
        if (metric == RMU_METRIC_COSINE) n0 = fmaf(x[d], x[d], n0);
#pragma unroll
        for (int i = 0; i < QT; ++i) a[i][0] = fmaf(qs[i * D + d], x[d], a[i][0]);
    }
    const float xn = sqrtf((n0 + n1) + (n2 + n3));
#pragma unroll
    for (int i = 0; i < QT; ++i) {
        const float ip = (a[i][0] + a[i][1]) + (a[i][2] + a[i][3]);
        if (metric == RMU_METRIC_IP) out[i] = ip;
        else { const float den = qnorm[i] * xn; out[i] = den > 0.f ? ip / den : 0.f; }
    }
}

// "larger is better" key of a metric value
__device__ __forceinline__ float metric_to_rank(float v, int metric) { return metric == RMU_METRIC_L2 ? -v : v; }

__device__ __forceinline__ float block_sum(float v, float* red /*[32]*/) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    int w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[w] = v;
    __syncthreads();
    float t = 0.f;
    for (int i = 0; i < nw; ++i) t += red[i];
    return t;
}

// =====================================================================================================
// per-row statistics at insert time: cosine scale 1/||x||, L2 bias -0.5||x||^2, running max ||x||
// =====================================================================================================
__global__ void row_stats_kernel(const float* __restrict__ x, long long row0, long long n, int D, int metric,
                                 float* __restrict__ rscale, float* __restrict__ rbias, unsigned* __restrict__ max_norm_bits,
                                 unsigned* __restrict__ max_dev_bits) {
    int warps_per_block = blockDim.x >> 5;
    long long r = static_cast<long long>(blockIdx.x) * warps_per_block + (threadIdx.x >> 5);
    if (r >= n) return;
    const float* p = x + (row0 + r) * D;
    float s = 0.f;
    for (int d = lane_id(); d < D; d += 32) s = fmaf(p[d], p[d], s);
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane_id() == 0) {
        float nrm = sqrtf(s);
        if (metric == RMU_METRIC_COSINE) rscale[row0 + r] = nrm > 0.f ? 1.f / nrm : 0.f;
        if (metric == RMU_METRIC_L2) rbias[row0 + r] = -0.5f * s;
        atomicMax(max_norm_bits, __float_as_uint(nrm));  // non-negative floats order like uints
        atomicMax(max_dev_bits, __float_as_uint(fabsf(s - 1.0f)));   // how far from unit norm the corpus gets
    }
}

// overwrite existing rows (upsert of a vector store): one warp per row copies the vector and refreshes its statistics
// (the running maxima only grow: conservative for the certificate)
__global__ void set_rows_kernel(float* __restrict__ x, const long long* __restrict__ rows, const float* __restrict__ vecs,
                                long long n_rows, long long n, int D, int metric, float* __restrict__ rscale,
                                float* __restrict__ rbias, unsigned* __restrict__ max_norm_bits, unsigned* __restrict__ max_dev_bits) {
    const long long i = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (i >= n_rows) return;
    const long long r = rows[i];
    if (r < 0 || r >= n) return;
    const float* src = vecs + i * D;
    float* dst = x + r * D;
    float s = 0.f;
    for (int d = lane_id(); d < D; d += 32) { const float v = src[d]; dst[d] = v; s = fmaf(v, v, s); }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane_id() == 0) {
        const float nrm = sqrtf(s);
        if (metric == RMU_METRIC_COSINE) rscale[r] = nrm > 0.f ? 1.f / nrm : 0.f;
        if (metric == RMU_METRIC_L2) rbias[r] = -0.5f * s;
        atomicMax(max_norm_bits, __float_as_uint(nrm));
        atomicMax(max_dev_bits, __float_as_uint(fabsf(s - 1.0f)));
    }
}

// =====================================================================================================
// warp-shuffle bitonic sort, descending, of 32*E u64 keys (element i = e*32 + lane)
// =====================================================================================================
template <int E>
__device__ __forceinline__ void warp_bitonic_desc(unsigned long long (&v)[E]) {
    const unsigned lane = lane_id();
#pragma unroll
    for (int k = 2; k <= 32 * E; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (j >= 32) {
                const int je = j >> 5;
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    if ((e & je) == 0) {
                        const int e2 = e | je;
                        const bool desc = (((e << 5) & k) == 0);
                        unsigned long long a = v[e], b = v[e2];
                        const bool sw = desc ? (a < b) : (a > b);
                        v[e] = sw ? b : a;
                        v[e2] = sw ? a : b;
                    }
                }
            } else {
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    const unsigned i = (static_cast<unsigned>(e) << 5) | lane;
                    unsigned long long o = __shfl_xor_sync(0xffffffffu, v[e], j);
                    const bool lower = (lane & j) == 0;
                    const bool desc = ((i & k) == 0);
                    const bool keepmax = (lower == desc);
                    v[e] = keepmax ? (v[e] > o ? v[e] : o) : (v[e] < o ? v[e] : o);
                }
            }
        }
    }
}

// =====================================================================================================
// (3) exact fp32 scan: one CTA = one chunk of rows x one (flagged) query -> sorted top list
// =====================================================================================================
constexpr int kChunk = 2048;

__device__ __forceinline__ void block_bitonic_desc(unsigned long long* s, int n /*pow2*/) {
    for (int k = 2; k <= n; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            __syncthreads();
            for (int t = threadIdx.x; t < n / 2; t += blockDim.x) {
                const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));  // index with bit j clear
                const int l = i | j;
                const bool desc = ((i & k) == 0);
                unsigned long long a = s[i], b = s[l];
                const bool sw = desc ? (a < b) : (a > b);
                if (sw) { s[i] = b; s[l] = a; }
            }
        }
    }
    __syncthreads();
}

struct ExactParams {
    const float* x; long long n; int dim; int metric;
    const float* q;            // [nq_total, dim]
    const int* qmap;           // [*nsel] query indices to process (nullable = identity over nq_total)
    const int* nsel;           // device count of selected queries (nullable -> nq_total)
    int nq_total;
    unsigned long long* lists; // [nchunks][nq_total][keep]
    int keep;                  // pow2 <= kChunk
    int nchunks;               // ceil(n / kChunk); the grid strides over them
};

constexpr int kExactQT = 8;    // queries scored per pass over a chunk of rows

__global__ void __launch_bounds__(256) exact_scan_kernel(const ExactParams p) {
    __shared__ unsigned long long keys[kChunk];
    __shared__ float red[32];
    __shared__ float qn[kExactQT];
    extern __shared__ float esm[];                 // qs [QT][dim], then sc [QT][kChunk]
    float* qs = esm;
    float* sc = esm + kExactQT * p.dim;
    const int nsel = p.nsel ? *p.nsel : p.nq_total;
    const int ngroups = (nsel + kExactQT - 1) / kExactQT;
    for (int chunk = blockIdx.x; chunk < p.nchunks; chunk += gridDim.x) {
    const long long row0 = static_cast<long long>(chunk) * kChunk;
    for (int grp = blockIdx.y; grp < ngroups; grp += gridDim.y) {
        const int f0 = grp * kExactQT;
        const int nq = min(kExactQT, nsel - f0);
        __syncthreads();
        for (int i = 0; i < kExactQT; ++i) {
            float part = 0.f;
            if (i < nq) {
                const int qg = p.qmap ? p.qmap[f0 + i] : f0 + i;
                for (int d = threadIdx.x; d < p.dim; d += blockDim.x) {
                    const float v = p.q[static_cast<long long>(qg) * p.dim + d];
                    qs[i * p.dim + d] = v;
                    part = fmaf(v, v, part);
                }
            } else {
                for (int d = threadIdx.x; d < p.dim; d += blockDim.x) qs[i * p.dim + d] = 0.f;
            }
            const float nrm = sqrtf(block_sum(part, red));
            if (threadIdx.x == 0) qn[i] = nrm;
        }
        __syncthreads();
        for (int r = threadIdx.x; r < kChunk; r += blockDim.x) {
            const long long row = row0 + r;
            if (row < p.n) {
                float v[kExactQT];
                exact_metric_multi<kExactQT>(qs, p.x + row * p.dim, p.dim, p.metric, qn, v);
#pragma unroll
                for (int i = 0; i < kExactQT; ++i) sc[i * kChunk + r] = v[i];
            }
        }
        __syncthreads();
        for (int i = 0; i < nq; ++i) {
            for (int r = threadIdx.x; r < kChunk; r += blockDim.x) {
                const long long row = row0 + r;
                keys[r] = row < p.n ? make_key(metric_to_rank(sc[i * kChunk + r], p.metric), static_cast<uint32_t>(row)) : 0ull;
            }
            block_bitonic_desc(keys, kChunk);
            unsigned long long* out = p.lists + (static_cast<long long>(chunk) * p.nq_total + f0 + i) * p.keep;
            for (int e = threadIdx.x; e < p.keep; e += blockDim.x) out[e] = keys[e];
            __syncthreads();
        }
    }
    }
}

// threads of the selection kernels (select_tau, finalize): their 8 radix passes over nlists * len keys are latency-bound,
// one CTA per query
constexpr int kSelThreads = 512;

// Block-wide radix select (8 bits per pass, most significant first) over passes [pass0, pass1): after pass 8 the
// state holds the ksel-th largest non-zero key among load_key(0..total); after pass 4 its 32 score bits (the low
// word still zero) and, in *s_ties, how many keys share those score bits.  *s_remaining < 0 means fewer than ksel
// keys exist ("keep everything").  pass0 == 0 initialises the state.  All threads call.
template <typename LoadKey>
__device__ __forceinline__ void block_radix_passes(LoadKey load_key, long long total, int ksel, int pass0, int pass1, int* hist,
                                                   unsigned long long* s_prefix, int* s_remaining, int* s_ties) {
    const int tid = threadIdx.x;
    if (pass0 == 0) {
        if (tid == 0) { *s_prefix = 0ull; *s_remaining = ksel; *s_ties = 0; }
        __syncthreads();
    }
    for (int pass = pass0; pass < pass1; ++pass) {
        const int shift = 56 - 8 * pass;
        for (int i = tid; i < 256; i += blockDim.x) hist[i] = 0;
        __syncthreads();
        const unsigned long long prefix = *s_prefix;
        const int remaining = *s_remaining;         // < 0: fewer than ksel keys exist, keep all
        const unsigned long long himask = pass == 0 ? 0ull : (~0ull << (shift + 8));
        if (remaining >= 0) {
            for (long long idx = tid; idx < total; idx += blockDim.x) {
                const unsigned long long key = load_key(idx);
                if (key != 0ull && (key & himask) == prefix) atomicAdd(&hist[(key >> shift) & 0xFF], 1);
            }
        }
        __syncthreads();
        if (tid == 0 && remaining >= 0) {
            int rem = remaining;
            int b = 255;
            for (; b >= 0; --b) {
                if (hist[b] >= rem) break;
                rem -= hist[b];
            }
            if (b < 0) { *s_remaining = -1; }
            else { *s_prefix = prefix | (static_cast<unsigned long long>(b) << shift); *s_remaining = rem; *s_ties = hist[b]; }
        }
        __syncthreads();
    }
}

// the ksel-th largest non-zero key, or 1 ("keep everything") when fewer than ksel exist.  Ties on the 32 score bits
// are rare: when the keys that share the selected score are all needed (s_ties == s_remaining after four passes) the
// threshold is that score with a zero row word and the four passes over the row bits are skipped.
template <typename LoadKey>
__device__ __forceinline__ unsigned long long block_radix_select(LoadKey load_key, long long total, int ksel, int* hist,
                                                                 unsigned long long* s_prefix, int* s_remaining, int* s_ties) {
    block_radix_passes(load_key, total, ksel, 0, 4, hist, s_prefix, s_remaining, s_ties);
    if (*s_remaining >= 0 && *s_ties != *s_remaining)        // uniform: shared state, read after the barrier
        block_radix_passes(load_key, total, ksel, 4, 8, hist, s_prefix, s_remaining, s_ties);
    return *s_remaining < 0 ? 1ull : *s_prefix;
}

// =====================================================================================================
// (3b) merge of the exact scan's per-chunk lists: select the best `ksel` keys, sort, write the top-k
// =====================================================================================================
struct FinalizeParams {
    const unsigned long long* lists;   // [nlists][nq_total][len] exact keys, sorted per chunk, zero padded
    int nlists;        // lists per query
    int qstride;       // queries per list block
    int len;           // entries per list, pow2
    int ksel;          // keys to keep (<= 1024)
    int metric;
    const int* qmap;   // blockIdx.x -> query through qmap (nullable: identity)
    const int* nsel;   // number of valid blockIdx.x (nullable: all)
    int k;
    long long id_offset;
    float* out_scores; long long* out_ids;   // [nq_total, k]
};

__global__ void __launch_bounds__(kSelThreads) finalize_kernel(const FinalizeParams p) {
    __shared__ unsigned long long cand[1024];
    __shared__ int hist[256];
    __shared__ int s_ncand;
    __shared__ unsigned long long s_prefix;
    __shared__ int s_remaining, s_ties;

    const int f = blockIdx.x;
    if (p.nsel != nullptr && f >= *p.nsel) return;
    const int qg = p.qmap ? p.qmap[f] : f;
    const int tid = threadIdx.x;

    const long long total = static_cast<long long>(p.nlists) * p.len;
    const int len_shift = __ffs(p.len) - 1;
    auto load_key = [&](long long idx) -> unsigned long long {
        const long long l = idx >> len_shift;
        const int e = static_cast<int>(idx & (p.len - 1));
        return p.lists[(l * p.qstride + f) * p.len + e];
    };
    const unsigned long long T = block_radix_select(load_key, total, p.ksel, hist, &s_prefix, &s_remaining, &s_ties);
    if (tid == 0) s_ncand = 0;
    __syncthreads();
    for (long long idx = tid; idx < total; idx += blockDim.x) {
        const unsigned long long key = load_key(idx);
        if (key != 0ull && key >= T) {
            const int pos = atomicAdd(&s_ncand, 1);
            if (pos < 1024) cand[pos] = key;
        }
    }
    __syncthreads();
    const int ncand = min(s_ncand, p.ksel);
    for (int c = ncand + tid; c < 1024; c += blockDim.x) cand[c] = 0ull;
    int n2 = 32;
    while (n2 < ncand) n2 <<= 1;
    block_bitonic_desc(cand, n2);
    const float missing = p.metric == RMU_METRIC_L2 ? INFINITY : -INFINITY;
    for (int j = tid; j < p.k; j += blockDim.x) {
        float s = missing;
        long long id = -1;
        if (j < ncand) {
            const float rk = key_score(cand[j]);
            s = p.metric == RMU_METRIC_L2 ? -rk : rk;
            id = p.id_offset + key_row(cand[j]);
        }
        p.out_scores[static_cast<long long>(qg) * p.k + j] = s;
        p.out_ids[static_cast<long long>(qg) * p.k + j] = id;
    }
}

#include "rmu_scan.cuh"

// flags[nq] -> qmap (ordered, compacted indices of flagged queries) + nsel; launched with one warp
__global__ void compact_flags_kernel(const int* __restrict__ flags, int nq, int* __restrict__ qmap, int* __restrict__ nsel) {
    int count = 0;
    for (int base = 0; base < nq; base += 32) {
        const int i = base + static_cast<int>(lane_id());
        const bool f = i < nq && flags[i] != 0;
        const unsigned m = __ballot_sync(0xffffffffu, f);
        if (f) qmap[count + __popc(m & ((1u << lane_id()) - 1u))] = i;
        count += __popc(m);
    }
    if (lane_id() == 0) *nsel = count;
}

// =====================================================================================================
// shard merge (after the all-gather of per-shard results): [R, nq, k] -> [nq, k]
// =====================================================================================================
__global__ void __launch_bounds__(256) merge_kernel(const float* __restrict__ scores, const long long* __restrict__ ids,
                                                    long long rstride_s, long long rstride_i,   // elements between ranks
                                                    int R, int nq, int k, int metric, float* __restrict__ out_s,
                                                    long long* __restrict__ out_i) {
    extern __shared__ unsigned char sm[];
    // entries sorted by (rank desc, id asc); ids are 64-bit so keep them beside a (rank, slot) key
    const int n = R * k;
    int n2 = 32;
    while (n2 < n) n2 <<= 1;
    unsigned long long* keys = reinterpret_cast<unsigned long long*>(sm);   // [n2] (ordered rank << 32 | ~slot)
    long long* sid = reinterpret_cast<long long*>(keys + n2);               // [n]
    float* sval = reinterpret_cast<float*>(sid + n);                        // [n]
    const int qi = blockIdx.x;
    // stable rule shared with the oracle: rank desc, then global id asc.  Slots are ordered by id
    // inside equal ranks by a final fix-up pass below (ties across shards are rare: duplicates).
    for (int t = threadIdx.x; t < n2; t += blockDim.x) {
        unsigned long long key = 0ull;
        if (t < n) {
            const int r = t / k, j = t % k;
            const long long src = static_cast<long long>(qi) * k + j;
            const long long id = ids[r * rstride_i + src];
            const float v = scores[r * rstride_s + src];
            sid[t] = id;
            sval[t] = v;
            if (id >= 0) key = (static_cast<unsigned long long>(f32_to_ordered(metric_to_rank(v, metric))) << 32) |
                               static_cast<unsigned long long>(0xFFFFFFFFu - static_cast<unsigned>(t));
        }
        keys[t] = key;
    }
    block_bitonic_desc(keys, n2);
    // fix-up: within runs of equal rank order by id ascending (insertion sort by one thread; runs are tiny)
    if (threadIdx.x == 0) {
        int a = 0;
        while (a < n && keys[a] != 0ull) {
            int b = a + 1;
            while (b < n && keys[b] != 0ull && (keys[b] >> 32) == (keys[a] >> 32)) ++b;
            for (int i = a + 1; i < b; ++i) {
                unsigned long long ki = keys[i];
                long long idi = sid[0xFFFFFFFFu - static_cast<unsigned>(ki)];
                int j = i - 1;
                while (j >= a && sid[0xFFFFFFFFu - static_cast<unsigned>(keys[j])] > idi) { keys[j + 1] = keys[j]; --j; }
                keys[j + 1] = ki;
            }
            a = b;
        }
    }
    __syncthreads();
    const float missing = metric == RMU_METRIC_L2 ? INFINITY : -INFINITY;
    for (int j = threadIdx.x; j < k; j += blockDim.x) {
        float s = missing;
        long long id = -1;
        if (j < n && keys[j] != 0ull) {
            const unsigned slot = 0xFFFFFFFFu - static_cast<unsigned>(keys[j]);
            s = sval[slot];
            id = sid[slot];
        }
        out_s[static_cast<long long>(qi) * k + j] = s;
        out_i[static_cast<long long>(qi) * k + j] = id;
    }
}

__global__ void gather_rows_kernel(const float* __restrict__ x, long long n, int dim, const long long* __restrict__ rows,
                                   int nrows, float* __restrict__ out) {
    const int r = blockIdx.x;
    if (r >= nrows) return;
    const long long row = rows[r];
    for (int d = threadIdx.x; d < dim; d += blockDim.x)
        out[static_cast<long long>(r) * dim + d] = (row >= 0 && row < n) ? x[row * dim + d] : 0.f;
}

// SemanticChunker (langchain_experimental.text_splitter, built at server/RAGHelper.py:329-341) embeds every sentence
// group and takes 1 - cosine_similarity of consecutive embeddings with numpy on float64 copies of the float32 vectors:
// dot / (|a| |b|).  One warp per pair, float64 accumulation, lanes stride the row (coalesced).
__global__ void adjacent_cosine_kernel(const float* __restrict__ x, long long pairs, int dim, double* __restrict__ out) {
    const long long pair = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (pair >= pairs) return;
    const unsigned lane = threadIdx.x & 31;
    const float* a = x + pair * dim;
    const float* b = a + dim;
    double dot = 0.0, na = 0.0, nb = 0.0;
    for (int j = static_cast<int>(lane); j < dim; j += 32) {
        const double u = static_cast<double>(a[j]), v = static_cast<double>(b[j]);
        dot = fma(u, v, dot); na = fma(u, u, na); nb = fma(v, v, nb);
    }
    for (int o = 16; o > 0; o >>= 1) {
        dot += __shfl_xor_sync(0xffffffffu, dot, o);
        na += __shfl_xor_sync(0xffffffffu, na, o);
        nb += __shfl_xor_sync(0xffffffffu, nb, o);
    }
    if (lane == 0) out[pair] = 1.0 - dot / (sqrt(na) * sqrt(nb));
}

// =====================================================================================================
// greedy MMR (langchain_core.vectorstores.utils.maximal_marginal_relevance), fp64 like numpy on
// python-float embeddings.  One CTA per query; fetch_k is small (20 by default).
// =====================================================================================================
__global__ void __launch_bounds__(128) mmr_kernel(const float* __restrict__ q, const float* __restrict__ cand,
                                                  const int* __restrict__ n_cand, int fetch_k, int dim, int k,
                                                  double lambda_mult, int* __restrict__ out_sel) {
    extern __shared__ double sh[];
    double* sim_q = sh;                    // [fetch_k]
    double* norms = sim_q + fetch_k;       // [fetch_k]
    double* simmat = norms + fetch_k;      // [fetch_k * fetch_k]
    double* best_sel = simmat + fetch_k * fetch_k;  // [fetch_k] running max similarity to the selected set
    __shared__ int s_sel[1];
    const int qi = blockIdx.x;
    const int n = n_cand ? min(n_cand[qi], fetch_k) : fetch_k;
    const float* qv = q + static_cast<long long>(qi) * dim;
    const float* E = cand + static_cast<long long>(qi) * fetch_k * dim;
    const int warp = threadIdx.x >> 5, nw = blockDim.x >> 5, lane = lane_id();
    // norms, <q, e_i>, <e_i, e_j>
    double qn = 0.0;
    for (int d = lane; d < dim; d += 32) qn += static_cast<double>(qv[d]) * qv[d];
    for (int o = 16; o > 0; o >>= 1) qn += __shfl_xor_sync(0xffffffffu, qn, o);
    qn = sqrt(qn);
    for (int i = warp; i < n; i += nw) {
        double s = 0.0, nn = 0.0;
        for (int d = lane; d < dim; d += 32) {
            const double e = E[static_cast<long long>(i) * dim + d];
            s += e * qv[d];
            nn += e * e;
        }
        for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); nn += __shfl_xor_sync(0xffffffffu, nn, o); }
        if (lane == 0) { norms[i] = sqrt(nn); sim_q[i] = s; }
    }
    __syncthreads();
    for (int pq = warp; pq < n * n; pq += nw) {
        const int i = pq / n, j = pq % n;
        double s = 0.0;
        for (int d = lane; d < dim; d += 32) s += static_cast<double>(E[static_cast<long long>(i) * dim + d]) * E[static_cast<long long>(j) * dim + d];
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) {
            const double den = norms[i] * norms[j];
            double c = den > 0.0 ? s / den : 0.0;
            if (isnan(c) || isinf(c)) c = 0.0;
            simmat[i * fetch_k + j] = c;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 0; i < n; ++i) {
            const double den = qn * norms[i];
            double c = den > 0.0 ? sim_q[i] / den : 0.0;
            if (isnan(c) || isinf(c)) c = 0.0;
            sim_q[i] = c;
            best_sel[i] = -1e300;
        }
        int nsel = 0;
        const int kk = min(k, n);
        unsigned long long chosen = 0ull;  // fetch_k <= 64
        if (kk > 0) {
            int first = 0;
            for (int i = 1; i < n; ++i) if (sim_q[i] > sim_q[first]) first = i;   // np.argmax: first maximum
            out_sel[static_cast<long long>(qi) * k + nsel++] = first;
            chosen |= 1ull << first;
            for (int i = 0; i < n; ++i) best_sel[i] = simmat[i * fetch_k + first];
        }
        while (nsel < kk) {
            double best = -INFINITY;
            int add = -1;
            for (int i = 0; i < n; ++i) {
                if (chosen & (1ull << i)) continue;
                const double sc = lambda_mult * sim_q[i] - (1.0 - lambda_mult) * best_sel[i];
                if (sc > best) { best = sc; add = i; }
            }
            if (add < 0) break;
            out_sel[static_cast<long long>(qi) * k + nsel++] = add;
            chosen |= 1ull << add;
            for (int i = 0; i < n; ++i) best_sel[i] = fmax(best_sel[i], simmat[i * fetch_k + add]);
        }
        for (int j = nsel; j < k; ++j) out_sel[static_cast<long long>(qi) * k + j] = -1;
        s_sel[0] = nsel;
    }
}

}  // namespace rmu

// =====================================================================================================
// host side
// =====================================================================================================
using namespace rmu;

struct rmu_index {
    int dim = 0, metric = 0, device = 0, sms = 0;
    int64_t n = 0, cap = 0;
    float* x = nullptr;
    float* rscale = nullptr;
    float* rbias = nullptr;
    unsigned* max_norm_bits = nullptr;   // [0] max ||x||, [1] max | ||x||^2 - 1 |
    CUtensorMap tmap{};
    int64_t tmap_rows = -1;
    unsigned long long* gmax = nullptr;  // [256][kGroupsMax] threshold exchange of the scan, epoch-tagged (never cleared)
    unsigned epoch = 0;                  // bumped once per scan launch (under mu)
    // scratch
    void* ws = nullptr;
    size_t ws_bytes = 0;
    void* hbuf = nullptr;          // device staging of the *_host entry points (queries, scores, ids)
    size_t hbuf_bytes = 0;
    cudaEvent_t ws_done = nullptr;
    std::mutex mu;
    std::mutex host_mu;            // serialises the *_host entry points (they share hbuf and synchronise anyway)
};

static int ensure_ws(rmu_index* idx, size_t bytes) {
    if (bytes <= idx->ws_bytes) return RMU_OK;
    if (idx->ws) {
        RMU_CUDA(cudaDeviceSynchronize());
        RMU_CUDA(cudaFree(idx->ws));
        idx->ws = nullptr;
        idx->ws_bytes = 0;
    }
    size_t want = bytes + bytes / 4;
    RMU_CUDA(cudaMalloc(&idx->ws, want));
    idx->ws_bytes = want;
    return RMU_OK;
}

static int keep_for_k(int k) {
    // coarse candidates re-scored exactly per query: >= 3k where that fits, never above 256
    if (3 * k <= 64) return 64;
    if (3 * k <= 128) return 128;
    return 256;
}

// one scan launch: NQ queries (MMA N); CTA pairs keep NQ/2 query rows resident per CTA, single CTAs all NQ
struct ScanGeom { int nq, nstages, pair; size_t smem; };
constexpr int kPass2MaxQ = 256;         // flagged queries the second pass takes per search (more stay flagged)
constexpr int kPass2PoolCap = 16384;    // rows a flagged query may collect; more -> the exact scan answers

template <int NQ, bool PAIR>
static int scan_launch_t(const CUtensorMap& tx, const CUtensorMap& tq, const ScanParams& p, int grid, size_t smem, cudaStream_t st) {
    auto kern = scan_rows_kernel<NQ, PAIR>;
    // per device and cheap: set on every launch (a process may drive several GPUs); always the device maximum, so that
    // concurrent callers on other handles never lower it under a launch that needs more
    RMU_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(static_cast<unsigned>(grid));
    cfg.blockDim = dim3(64 + 32 * scan_epi_warps(NQ));
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = PAIR ? 2 : 1; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    ProfScope _ps(p.fixed_tau != nullptr ? PROF_SCAN_LEAD : PROF_SCAN, st);   // second-pass launches are timed apart
    RMU_CUDA(cudaLaunchKernelEx(&cfg, kern, tx, tq, p));
    count_launch();
    return RMU_OK;
}

static int scan_dispatch(const ScanGeom& g, const CUtensorMap& tx, const CUtensorMap& tq, const ScanParams& p, int grid, cudaStream_t st) {
#define SCAN_CASE(NQ)                                                                                            \
    if (g.nq == NQ) return g.pair ? scan_launch_t<NQ, true>(tx, tq, p, grid, g.smem, st) : scan_launch_t<NQ, false>(tx, tq, p, grid, g.smem, st);
    SCAN_CASE(128) SCAN_CASE(64) SCAN_CASE(32) SCAN_CASE(16)
#undef SCAN_CASE
    set_error("scan: unsupported geometry");
    return RMU_ERR_UNSUPPORTED;
}

// largest query block (MMA N) whose resident part fits shared memory at this dimension; 0: dim too large
static int scan_block_cap(int dim, bool pair) {
    const int KB = (dim + 31) / 32;
    int cap = pair ? kScanMaxQ : 64;
    while (cap >= 16 && KB * (cap / (pair ? 2 : 1)) * 128 > kScanQOpMax) cap >>= 1;
    return cap >= 16 ? cap : 0;
}
static int scan_max_block(int dim) { return std::max(scan_block_cap(dim, false), scan_block_cap(dim, true)); }

// geometry for `rem` queries still to scan.  Single CTAs keep the whole query block resident (<= 64 queries at 384
// dims) and are the faster kernel per pass (measured 10M x 384, Q = 64: 2.26 ms vs 2.36 ms); CTA pairs keep half a
// block per CTA, so they take twice the queries (or twice the dimension) per pass: 5M x 768, Q = 64: one pass of 2.19 ms
// instead of two of 2.15 ms; 10M x 384, Q = 128: 3.0 ms instead of 4.5 ms.
static ScanGeom scan_geometry(int dim, int rem) {
    const int KB = (dim + 31) / 32;
    const int cap1 = scan_block_cap(dim, false), cap2 = scan_block_cap(dim, true);
    ScanGeom g{};
    g.pair = cap1 == 0 || (rem > cap1 && cap2 > cap1);
    const int cap = g.pair ? cap2 : cap1;
    int nq = 16;
    while (nq < cap && nq < rem) nq <<= 1;
    const size_t qop = static_cast<size_t>(KB) * (nq / (g.pair ? 2 : 1)) * 128;
    const size_t stage = static_cast<size_t>(kScanKD) * kBoxBytes;
    const size_t budget = 227 * 1024 - 1024 - kScanStateBytes - qop;
    g.nq = nq;
    g.nstages = static_cast<int>(std::min<size_t>(budget / stage, kScanMaxStages));
    g.smem = 1024 + qop + static_cast<size_t>(g.nstages) * stage + kScanStateBytes;
    return g;
}

// one scan launch over the first `ntiles` corpus tiles for the nq queries at qbase (row pitch = dim), one CTA per SM.
// `sp` comes with the fields of the caller's pass set; the ones every launch shares are filled here.  Grids too small
// for the threshold exchange run without it (sp.groups = 0).  *grid_out (if given) receives the grid.
static int scan_launch(rmu_index* idx, const ScanGeom& geo, const float* qbase, int nq, int ntiles, ScanParams& sp,
                       cudaStream_t st, int* grid_out = nullptr) {
    const int D = idx->dim;
    const int grid = geo.pair ? 2 * std::min(idx->sms / 2, (ntiles + 1) / 2) : std::min(idx->sms, ntiles);
    CUtensorMap tq;
    const int rc = make_tmap_2d(&tq, qbase, static_cast<uint64_t>(nq), static_cast<uint64_t>(D),
                                static_cast<uint64_t>(D) * sizeof(float), 32, static_cast<uint32_t>(geo.nq / (geo.pair ? 2 : 1)), 4);
    if (rc != RMU_OK) return rc;
    sp.nq = nq; sp.dim = D; sp.n = idx->n; sp.ntiles = ntiles; sp.nstages = geo.nstages; sp.metric = idx->metric;
    sp.rscale = idx->rscale; sp.rbias = idx->rbias; sp.stats_bits = idx->max_norm_bits; sp.gmax = idx->gmax;
    if (grid < 2 * sp.groups) sp.groups = 0;         // small grids: lists are cut only by their own floors
    if (grid_out) *grid_out = grid;
    return scan_dispatch(geo, idx->tmap, tq, sp, grid, st);
}

extern "C" {

int rmu_index_create(int dim, int metric, rmu_index** out) {
    if (!out || dim <= 0 || metric < 0 || metric > 2) { set_error("rmu_index_create: bad argument"); return RMU_ERR_ARG; }
    rmu_index* idx = new rmu_index();
    idx->dim = dim;
    idx->metric = metric;
    if (cudaGetDevice(&idx->device) != cudaSuccess || (idx->sms = device_sm_count()) <= 0) {
        set_error("rmu_index_create: no CUDA device (this library has no CPU path)");
        delete idx;
        return RMU_ERR_CUDA;
    }
    cudaError_t e = cudaMalloc(&idx->max_norm_bits, 2 * sizeof(unsigned));
    if (e == cudaSuccess) e = cudaMemset(idx->max_norm_bits, 0, 2 * sizeof(unsigned));
    if (e == cudaSuccess) e = cudaMalloc(&idx->gmax, sizeof(unsigned long long) * 256 * kGroupsMax);
    if (e == cudaSuccess) e = cudaMemset(idx->gmax, 0, sizeof(unsigned long long) * 256 * kGroupsMax);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&idx->ws_done, cudaEventDisableTiming);
    if (e != cudaSuccess) { set_error(std::string("rmu_index_create: ") + cudaGetErrorString(e)); delete idx; return RMU_ERR_CUDA; }
    *out = idx;
    return RMU_OK;
}

void rmu_index_destroy(rmu_index* idx) {
    if (!idx) return;
    cudaDeviceSynchronize();
    cudaFree(idx->x); cudaFree(idx->rscale); cudaFree(idx->rbias); cudaFree(idx->max_norm_bits); cudaFree(idx->ws); cudaFree(idx->hbuf); cudaFree(idx->gmax);
    if (idx->ws_done) cudaEventDestroy(idx->ws_done);
    delete idx;
}

}  // extern "C"

// grow the corpus allocation to `rows` rows; idx->mu must be held
static int reserve_locked(rmu_index* idx, int64_t rows) {
    if (rows <= idx->cap) return RMU_OK;
    RMU_CUDA(cudaDeviceSynchronize());
    float* nx = nullptr; float* ns = nullptr; float* nb = nullptr;
    cudaError_t e = cudaMalloc(&nx, static_cast<size_t>(rows) * idx->dim * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&ns, static_cast<size_t>(rows) * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&nb, static_cast<size_t>(rows) * sizeof(float));
    if (e == cudaSuccess && idx->n > 0) {
        e = cudaMemcpy(nx, idx->x, static_cast<size_t>(idx->n) * idx->dim * sizeof(float), cudaMemcpyDeviceToDevice);
        if (e == cudaSuccess) e = cudaMemcpy(ns, idx->rscale, static_cast<size_t>(idx->n) * sizeof(float), cudaMemcpyDeviceToDevice);
        if (e == cudaSuccess) e = cudaMemcpy(nb, idx->rbias, static_cast<size_t>(idx->n) * sizeof(float), cudaMemcpyDeviceToDevice);
    }
    if (e != cudaSuccess) {
        cudaFree(nx); cudaFree(ns); cudaFree(nb);            // the index keeps its old storage
        set_error(std::string("rmu_index_reserve: ") + cudaGetErrorString(e));
        return RMU_ERR_CUDA;
    }
    cudaFree(idx->x); cudaFree(idx->rscale); cudaFree(idx->rbias);
    idx->x = nx; idx->rscale = ns; idx->rbias = nb;
    idx->cap = rows;
    idx->tmap_rows = -1;
    return RMU_OK;
}

extern "C" {

int rmu_index_reserve(rmu_index* idx, int64_t rows) {
    if (!idx || rows < 0) { set_error("rmu_index_reserve: bad argument"); return RMU_ERR_ARG; }
    std::lock_guard<std::mutex> g(idx->mu);
    return reserve_locked(idx, rows);
}

int rmu_index_add(rmu_index* idx, const float* vecs, int64_t n, int src_is_host, void* stream) {
    if (!idx || (n > 0 && !vecs) || n < 0) { set_error("rmu_index_add: bad argument"); return RMU_ERR_ARG; }
    if (n == 0) return RMU_OK;
    std::lock_guard<std::mutex> g(idx->mu);      // size check, growth and append are one critical section
    if (idx->n + n > static_cast<int64_t>(0xFFFFFFF0u)) { set_error("rmu_index_add: more than 2^32 rows per shard"); return RMU_ERR_UNSUPPORTED; }
    if (idx->n + n > idx->cap) {
        int64_t want = std::max<int64_t>(idx->n + n, idx->cap + idx->cap / 2);
        int rc = reserve_locked(idx, std::max<int64_t>(want, 1024));
        if (rc != RMU_OK) return rc;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    RMU_CUDA(cudaMemcpyAsync(idx->x + idx->n * idx->dim, vecs, static_cast<size_t>(n) * idx->dim * sizeof(float),
                             src_is_host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, st));
    const int wpb = 8;
    const long long blocks = (n + wpb - 1) / wpb;
    row_stats_kernel<<<static_cast<unsigned>(blocks), wpb * 32, 0, st>>>(idx->x, idx->n, n, idx->dim, idx->metric,
                                                                          idx->rscale, idx->rbias, idx->max_norm_bits,
                                                                          idx->max_norm_bits + 1);
    count_launch();
    RMU_CHECK_LAUNCH();
    idx->n += n;
    idx->tmap_rows = -1;
    return RMU_OK;
}

int rmu_index_set_rows(rmu_index* idx, const int64_t* rows, const float* vecs, int64_t n, void* stream) {
    if (!idx || n < 0 || (n > 0 && (!rows || !vecs))) { set_error("rmu_index_set_rows: bad argument"); return RMU_ERR_ARG; }
    if (n == 0) return RMU_OK;
    std::lock_guard<std::mutex> g(idx->mu);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int wpb = 8;
    set_rows_kernel<<<static_cast<unsigned>((n + wpb - 1) / wpb), wpb * 32, 0, st>>>(
        idx->x, reinterpret_cast<const long long*>(rows), vecs, n, idx->n, idx->dim, idx->metric, idx->rscale, idx->rbias,
        idx->max_norm_bits, idx->max_norm_bits + 1);
    count_launch();
    RMU_CHECK_LAUNCH();
    return RMU_OK;
}

int64_t rmu_index_size(const rmu_index* idx) { return idx ? idx->n : -1; }
int rmu_index_dim(const rmu_index* idx) { return idx ? idx->dim : -1; }
int rmu_index_metric(const rmu_index* idx) { return idx ? idx->metric : -1; }
const float* rmu_index_data(const rmu_index* idx) { return idx ? idx->x : nullptr; }

int rmu_index_clear(rmu_index* idx) {
    if (!idx) return RMU_ERR_ARG;
    std::lock_guard<std::mutex> g(idx->mu);
    RMU_CUDA(cudaDeviceSynchronize());
    idx->n = 0;
    idx->tmap_rows = -1;
    RMU_CUDA(cudaMemset(idx->max_norm_bits, 0, 2 * sizeof(unsigned)));
    return RMU_OK;
}

// corpus tensor map: boxes of {32 floats, 128 rows}, 128-byte swizzle; idx->mu held
static int ensure_corpus_tmap(rmu_index* idx) {
    if (idx->tmap_rows == idx->n) return RMU_OK;
    int rc = make_tmap_2d(&idx->tmap, idx->x, static_cast<uint64_t>(idx->n), static_cast<uint64_t>(idx->dim),
                          static_cast<uint64_t>(idx->dim) * sizeof(float), 32, kTileRows, 4);
    if (rc != RMU_OK) return rc;
    idx->tmap_rows = idx->n;
    return RMU_OK;
}

int rmu_index_search(rmu_index* idx, const float* queries, int nq, int k, int64_t id_offset, int mode,
                     float* out_scores, int64_t* out_ids, int32_t* stats_h, void* stream) {
    if (!idx || nq < 0 || k <= 0 || (nq > 0 && (!queries || !out_scores || !out_ids))) {
        set_error("rmu_index_search: bad argument");
        return RMU_ERR_ARG;
    }
    if (k > 1024) { set_error("rmu_index_search: k > 1024 is not supported"); return RMU_ERR_UNSUPPORTED; }
    if (stats_h) { stats_h[0] = stats_h[1] = stats_h[2] = stats_h[3] = 0; }
    if (nq == 0) return RMU_OK;
    std::lock_guard<std::mutex> g(idx->mu);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    RMU_CUDA(cudaStreamWaitEvent(st, idx->ws_done, 0));   // scratch is shared by all callers of this handle

    const int D = idx->dim;
    const long long N = idx->n;
    // tensor scan eligibility: TMA row pitch multiple of 16 B (queries too: they are loaded by TMA), the resident
    // query operand fits shared memory (dim <= 3072), enough rows, k small
    const bool tensor_ok = (D % 4 == 0) && scan_max_block(D) > 0 && N >= 16384 && k <= 128 && mode != RMU_SEARCH_EXACT &&
                           (reinterpret_cast<uintptr_t>(queries) & 15) == 0 && idx->sms >= 2;
    const int keep = keep_for_k(k);                       // tensor: coarse candidates re-scored per query (>= 2k)
    int keepx = 32; while (keepx < k) keepx <<= 1;        // exact: per-chunk list length (>= k)
    const int nchunks = static_cast<int>((N + kChunk - 1) / kChunk);

    // ---- scratch layout
    const int max_lists = idx->sms * kScanMaxQ;           // (CTA, query) lists of one scan launch
    size_t off = 0;
    auto carve = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~size_t(255); return o; };
    const size_t o_flags = carve(sizeof(int) * nq);
    const size_t o_qmap = carve(sizeof(int) * nq);
    const size_t o_nsel = carve(sizeof(int) * 4);
    const size_t o_scan = tensor_ok ? carve(sizeof(unsigned long long) * max_lists * kListCap) : 0;
    const size_t o_cnt = tensor_ok ? carve(sizeof(int) * max_lists) : 0;
    const size_t o_floor = tensor_ok ? carve(sizeof(float) * max_lists) : 0;
    // second pass (flagged queries, AUTO mode): compacted queries + thresholds + per-query pools
    const int p2max = (tensor_ok && mode == RMU_SEARCH_AUTO) ? std::min(nq, kPass2MaxQ) : 0;
    const size_t o_tau2 = carve(sizeof(float) * nq);
    const size_t o_qbuf = carve(sizeof(float) * static_cast<size_t>(p2max) * D);
    const size_t o_taub = carve(sizeof(float) * std::max(p2max, 1));
    const size_t o_pcnt = carve(sizeof(int) * std::max(p2max, 1));
    const size_t o_pool = carve(sizeof(unsigned long long) * static_cast<size_t>(p2max) * kPass2PoolCap);
    const size_t o_qmap2 = carve(sizeof(int) * nq);
    const size_t o_exact = carve(sizeof(unsigned long long) * std::max(nchunks, 1) * static_cast<size_t>(nq) * keepx);
    int rc = ensure_ws(idx, off);
    if (rc != RMU_OK) return rc;
    uint8_t* ws = static_cast<uint8_t*>(idx->ws);
    int* d_flags = reinterpret_cast<int*>(ws + o_flags);
    int* d_qmap = reinterpret_cast<int*>(ws + o_qmap);
    int* d_nsel = reinterpret_cast<int*>(ws + o_nsel);
    unsigned long long* d_scan = reinterpret_cast<unsigned long long*>(ws + o_scan);
    unsigned long long* d_exact = reinterpret_cast<unsigned long long*>(ws + o_exact);
    int* d_cnt = reinterpret_cast<int*>(ws + o_cnt);
    float* d_floor = reinterpret_cast<float*>(ws + o_floor);
    float* d_tau2 = reinterpret_cast<float*>(ws + o_tau2);
    float* d_qbuf = reinterpret_cast<float*>(ws + o_qbuf);
    float* d_taub = reinterpret_cast<float*>(ws + o_taub);
    int* d_pcnt = reinterpret_cast<int*>(ws + o_pcnt);
    unsigned long long* d_pool = reinterpret_cast<unsigned long long*>(ws + o_pool);
    int* d_qmap2 = reinterpret_cast<int*>(ws + o_qmap2);
    int* d_nsel2 = d_nsel + 1;                               // queries still flagged after the second pass

    int scan_launches = 0;

    if (tensor_ok) {
        rc = ensure_corpus_tmap(idx);
        if (rc != RMU_OK) return rc;
        const int ntiles = static_cast<int>((N + kTileRows - 1) / kTileRows);
        for (int q0 = 0; q0 < nq;) {
            const ScanGeom geo = scan_geometry(D, nq - q0);
            const int nql = std::min(nq - q0, geo.nq);
            const float* qbase = queries + static_cast<size_t>(q0) * D;
            ScanParams sp{};
            sp.lists = d_scan; sp.counts = d_cnt; sp.floors = d_floor;
            sp.epoch = ++idx->epoch;
            if (idx->epoch == 0xFFFFFFFFu) {                 // epoch wrap: start over from clean tags
                RMU_CUDA(cudaMemsetAsync(idx->gmax, 0, sizeof(unsigned long long) * 256 * kGroupsMax, st));
                idx->epoch = 0;
                sp.epoch = ++idx->epoch;
            }
            sp.groups = keep / kPubRank;                      // 16 * groups >= keep rows score >= the exchanged threshold
            int grid = 0;
            rc = scan_launch(idx, geo, qbase, nql, ntiles, sp, st, &grid);
            if (rc != RMU_OK) return rc;
            ++scan_launches;
            SelectParams fp{};
            fp.lists = d_scan; fp.counts = d_cnt; fp.floors = d_floor; fp.gmax = idx->gmax;
            fp.ncl = grid; fp.qb = geo.nq; fp.epoch = sp.epoch; fp.groups = sp.groups; fp.ksel = keep;
            fp.x = idx->x; fp.n = N; fp.dim = D; fp.metric = idx->metric; fp.q = qbase; fp.q0 = q0;
            fp.k = k; fp.id_offset = id_offset; fp.stats_bits = idx->max_norm_bits;
            fp.eps_rel = 2.2e-3f;   // > 2^-9: both TF32 operands truncated to 10 mantissa bits
            fp.out_scores = out_scores; fp.out_ids = reinterpret_cast<long long*>(out_ids); fp.flags = d_flags; fp.tau2 = d_tau2;
            const size_t sel_smem = sizeof(unsigned long long) * kSel2Cap + static_cast<size_t>(D) * sizeof(float);
            RMU_CUDA(cudaFuncSetAttribute(select_rescore_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
            { ProfScope _ps(PROF_FINALIZE, st);
            select_rescore_kernel<<<nql, kSel2Threads, sel_smem, st>>>(fp); }
            count_launch();
            RMU_CHECK_LAUNCH();
            q0 += nql;
        }
        compact_flags_kernel<<<1, 32, 0, st>>>(d_flags, nq, d_qmap, d_nsel);
        count_launch();
        RMU_CHECK_LAUNCH();
        if (p2max > 0) {
            // ---- second pass for the queries whose certificate failed (near-duplicate heavy neighbourhoods): one more
            // tensor scan that collects EVERY row whose coarse key can still reach the k-th exact score of the first pass
            // (threshold = that score - eps), exact re-score of those pools -> exact top-k.  Worst case = 2 scans instead of
            // the 8+ CUDA-core passes of the exact scan; when nothing is flagged the launches below exit at once.
            pool_prepare_kernel<<<p2max, 128, 0, st>>>(queries, d_qmap, d_nsel, D, d_tau2, d_qbuf, d_taub, d_pcnt);
            count_launch();
            RMU_CHECK_LAUNCH();
            for (int j0 = 0; j0 < p2max;) {
                const ScanGeom geo = scan_geometry(D, p2max - j0);
                const int nql = std::min(p2max - j0, geo.nq);
                ScanParams sp{};                              // pool mode: no lists, no exchange
                sp.fixed_tau = d_taub + j0; sp.pool = d_pool + static_cast<size_t>(j0) * kPass2PoolCap; sp.pool_cnt = d_pcnt + j0;
                sp.pool_cap = kPass2PoolCap; sp.nq_dev = d_nsel; sp.q_off = j0;
                rc = scan_launch(idx, geo, d_qbuf + static_cast<size_t>(j0) * D, nql, ntiles, sp, st);
                if (rc != RMU_OK) return rc;
                j0 += nql;
            }
            PoolParams pp{};
            pp.pool = d_pool; pp.pool_cnt = d_pcnt; pp.pool_cap = kPass2PoolCap; pp.qmap = d_qmap; pp.nsel = d_nsel; pp.max_slots = p2max;
            pp.x = idx->x; pp.dim = D; pp.metric = idx->metric; pp.q = queries; pp.k = k; pp.id_offset = id_offset;
            pp.out_scores = out_scores; pp.out_ids = reinterpret_cast<long long*>(out_ids); pp.flags = d_flags;
            { ProfScope _ps(PROF_FINALIZE, st);
            pool_rescore_kernel<<<p2max, kSel2Threads, static_cast<size_t>(D) * sizeof(float), st>>>(pp); }
            count_launch();
            RMU_CHECK_LAUNCH();
            compact_flags_kernel<<<1, 32, 0, st>>>(d_flags, nq, d_qmap2, d_nsel2);
            count_launch();
            RMU_CHECK_LAUNCH();
        }
    }

    if (!tensor_ok || mode == RMU_SEARCH_AUTO) {
        FinalizeParams fp{};
        fp.lists = d_exact; fp.qstride = nq; fp.len = keepx; fp.ksel = keepx; fp.metric = idx->metric;
        fp.k = k; fp.id_offset = id_offset;
        fp.out_scores = out_scores; fp.out_ids = reinterpret_cast<long long*>(out_ids);
        if (N > 0) {
            ExactParams ep{};
            ep.x = idx->x; ep.n = N; ep.dim = D; ep.metric = idx->metric; ep.q = queries;
            ep.qmap = tensor_ok ? (p2max > 0 ? d_qmap2 : d_qmap) : nullptr;
            ep.nsel = tensor_ok ? (p2max > 0 ? d_nsel2 : d_nsel) : nullptr; ep.nq_total = nq;
            ep.lists = d_exact; ep.keep = keepx; ep.nchunks = nchunks;
            const int ngroups = (nq + kExactQT - 1) / kExactQT;
            int gy = tensor_ok ? 1 : std::min(ngroups, std::max(1, (2 * idx->sms + nchunks - 1) / nchunks));
            gy = std::min(gy, 65535);
            // behind the tensor scan only flagged queries run here (usually none): a small grid strides over the chunks
            dim3 eg(static_cast<unsigned>(tensor_ok ? std::min(nchunks, 4 * idx->sms) : nchunks), static_cast<unsigned>(gy));
            const size_t esmem = sizeof(float) * kExactQT * (static_cast<size_t>(D) + kChunk);
            if (esmem > 200 * 1024) { set_error("rmu_index_search: dim too large for the exact scan"); return RMU_ERR_UNSUPPORTED; }
            RMU_CUDA(cudaFuncSetAttribute(exact_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
            { ProfScope _ps(PROF_EXACT, st);
            exact_scan_kernel<<<eg, 256, esmem, st>>>(ep); }
            count_launch();
            RMU_CHECK_LAUNCH();
            fp.nlists = nchunks; fp.qmap = ep.qmap; fp.nsel = ep.nsel;
        } else {
            fp.nlists = 0;                                // nothing to search: all results missing
        }
        { ProfScope _ps(PROF_EXACT, st);
        finalize_kernel<<<nq, kSelThreads, 0, st>>>(fp); }
        count_launch();
        RMU_CHECK_LAUNCH();
    }

    if (stats_h) {
        int nsel[2] = {tensor_ok ? 0 : nq, tensor_ok ? 0 : nq};
        if (tensor_ok) {
            RMU_CUDA(cudaMemcpyAsync(nsel, d_nsel, (p2max > 0 ? 2 : 1) * sizeof(int), cudaMemcpyDeviceToHost, st));
            RMU_CUDA(cudaStreamSynchronize(st));
            if (p2max == 0) nsel[1] = nsel[0];
        }
        stats_h[0] = nsel[0];          // certificate failed in the first pass
        stats_h[1] = scan_launches;
        stats_h[2] = nsel[1];          // still unanswered after the second pass: went to the exact CUDA-core scan
    }
    RMU_CUDA(cudaEventRecord(idx->ws_done, st));
    return RMU_OK;
}

// diagnostics: raw TF32 accumulators of the first 256 rows (one pair tile), out [nq <= 64, 256] device fp32
int rmu_debug_scan_tile(rmu_index* idx, const float* queries, int nq, float* out, void* stream) {
    if (!idx || !queries || !out || nq <= 0 || nq > 64 || idx->n <= 0 || idx->dim % 4 != 0 || idx->dim > 384 ||
        (reinterpret_cast<uintptr_t>(queries) & 15) != 0) {
        set_error("rmu_debug_scan_tile: bad argument");
        return RMU_ERR_ARG;
    }
    std::lock_guard<std::mutex> g(idx->mu);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    RMU_CUDA(cudaStreamWaitEvent(st, idx->ws_done, 0));
    const size_t lists = sizeof(unsigned long long) * 2 * 64 * kListCap;
    int rc = ensure_ws(idx, lists + 4 * sizeof(int) * 64 + 1024);
    if (rc != RMU_OK) return rc;
    rc = ensure_corpus_tmap(idx);
    if (rc != RMU_OK) return rc;
    ScanParams sp{};
    sp.lists = static_cast<unsigned long long*>(idx->ws);
    sp.counts = reinterpret_cast<int*>(static_cast<uint8_t*>(idx->ws) + lists);
    sp.floors = reinterpret_cast<float*>(sp.counts + 128);
    sp.epoch = ++idx->epoch;
    sp.dbg = out;
    rc = scan_launch(idx, scan_geometry(idx->dim, 64), queries, nq, 2, sp, st);   // two tiles: grid 2
    RMU_CUDA(cudaEventRecord(idx->ws_done, st));
    return rc;
}

int rmu_index_search_host(rmu_index* idx, const float* queries_h, int nq, int k, int64_t id_offset, int mode,
                          float* out_scores_h, int64_t* out_ids_h, void* stream) {
    if (!idx || nq <= 0 || k <= 0 || !queries_h || !out_scores_h || !out_ids_h) {
        set_error("rmu_index_search_host: bad argument");
        return RMU_ERR_ARG;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    std::lock_guard<std::mutex> hg(idx->host_mu);
    const size_t qb = (static_cast<size_t>(nq) * idx->dim * sizeof(float) + 255) & ~size_t(255);
    const size_t sb = (static_cast<size_t>(nq) * k * sizeof(float) + 255) & ~size_t(255);
    const size_t ib = static_cast<size_t>(nq) * k * sizeof(int64_t);
    {
        // handle-owned staging (a cudaMallocAsync/free pair per call costs milliseconds once the pool is trimmed)
        std::lock_guard<std::mutex> g(idx->mu);
        if (qb + sb + ib > idx->hbuf_bytes) {
            RMU_CUDA(cudaStreamSynchronize(st));
            if (idx->hbuf) RMU_CUDA(cudaFree(idx->hbuf));
            idx->hbuf = nullptr;
            idx->hbuf_bytes = 0;
            RMU_CUDA(cudaMalloc(&idx->hbuf, 2 * (qb + sb + ib)));
            idx->hbuf_bytes = 2 * (qb + sb + ib);
        }
    }
    uint8_t* hb = static_cast<uint8_t*>(idx->hbuf);
    float* dq = reinterpret_cast<float*>(hb);
    float* ds = reinterpret_cast<float*>(hb + qb);
    int64_t* di = reinterpret_cast<int64_t*>(hb + qb + sb);
    RMU_CUDA(cudaMemcpyAsync(dq, queries_h, static_cast<size_t>(nq) * idx->dim * sizeof(float), cudaMemcpyHostToDevice, st));
    int rc = rmu_index_search(idx, dq, nq, k, id_offset, mode, ds, di, nullptr, st);
    if (rc == RMU_OK) {
        RMU_CUDA(cudaMemcpyAsync(out_scores_h, ds, static_cast<size_t>(nq) * k * sizeof(float), cudaMemcpyDeviceToHost, st));
        RMU_CUDA(cudaMemcpyAsync(out_ids_h, di, ib, cudaMemcpyDeviceToHost, st));
    }
    RMU_CUDA(cudaStreamSynchronize(st));
    return rc;
}

int rmu_index_gather(rmu_index* idx, const int64_t* rows, int n, float* out, void* stream) {
    if (!idx || n < 0 || (n > 0 && (!rows || !out))) { set_error("rmu_index_gather: bad argument"); return RMU_ERR_ARG; }
    if (n == 0) return RMU_OK;
    std::lock_guard<std::mutex> g(idx->mu);      // a concurrent add may grow (free + reallocate) the corpus
    gather_rows_kernel<<<n, 128, 0, static_cast<cudaStream_t>(stream)>>>(idx->x, idx->n, idx->dim,
                                                                          reinterpret_cast<const long long*>(rows), n, out);
    count_launch();
    RMU_CHECK_LAUNCH();
    return RMU_OK;
}

int rmu_topk_merge_strided(const float* scores, const int64_t* ids, int64_t rank_stride_scores, int64_t rank_stride_ids,
                           int R, int nq, int k, int metric, float* out_scores, int64_t* out_ids, void* stream) {
    if (R <= 0 || nq < 0 || k <= 0 || !scores || !ids || !out_scores || !out_ids || metric < 0 || metric > 2) {
        set_error("rmu_topk_merge: bad argument");
        return RMU_ERR_ARG;
    }
    if (nq == 0) return RMU_OK;
    const int n = R * k;
    if (n > 4096) { set_error("rmu_topk_merge: R*k > 4096"); return RMU_ERR_UNSUPPORTED; }
    int n2 = 32; while (n2 < n) n2 <<= 1;
    const size_t smem = static_cast<size_t>(n2) * 8 + static_cast<size_t>(n) * 8 + static_cast<size_t>(n) * 4;
    RMU_CUDA(cudaFuncSetAttribute(merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    ProfScope _ps(PROF_MERGE, static_cast<cudaStream_t>(stream));
    merge_kernel<<<nq, 256, smem, static_cast<cudaStream_t>(stream)>>>(scores, reinterpret_cast<const long long*>(ids),
                                                                       rank_stride_scores, rank_stride_ids, R, nq, k,
                                                                       metric, out_scores, reinterpret_cast<long long*>(out_ids));
    count_launch();
    RMU_CHECK_LAUNCH();
    return RMU_OK;
}

int rmu_topk_merge(const float* scores, const int64_t* ids, int R, int nq, int k, int metric, float* out_scores,
                   int64_t* out_ids, void* stream) {
    return rmu_topk_merge_strided(scores, ids, static_cast<int64_t>(nq) * k, static_cast<int64_t>(nq) * k, R, nq, k, metric,
                                  out_scores, out_ids, stream);
}

/* cosine distance between consecutive rows (SemanticChunker: sentence group i vs i + 1), float64 like the numpy code the
 * reference's chunker runs on the embedding lists */
int rmu_adjacent_cosine_distance(const float* x, int64_t n, int dim, double* out, void* stream) {
    if (!x || !out || n < 0 || dim <= 0) { set_error("rmu_adjacent_cosine_distance: bad argument"); return RMU_ERR_ARG; }
    if (n < 2) return RMU_OK;
    const int64_t pairs = n - 1;
    const int warps_per_block = 8;
    const unsigned grid = static_cast<unsigned>((pairs + warps_per_block - 1) / warps_per_block);
    adjacent_cosine_kernel<<<grid, warps_per_block * 32, 0, static_cast<cudaStream_t>(stream)>>>(x, pairs, dim, out);
    count_launch();
    RMU_CHECK_LAUNCH();
    return RMU_OK;
}

int rmu_mmr_select(const float* q, const float* cand, const int32_t* n_cand, int nq, int fetch_k, int dim, int k,
                   float lambda_mult, int32_t* out_sel, void* stream) {
    if (!q || !cand || !out_sel || nq < 0 || fetch_k <= 0 || fetch_k > 64 || dim <= 0 || k <= 0) {
        set_error("rmu_mmr_select: bad argument (fetch_k must be in 1..64)");
        return RMU_ERR_ARG;
    }
    if (nq == 0) return RMU_OK;
    const size_t smem = sizeof(double) * (3 * static_cast<size_t>(fetch_k) + static_cast<size_t>(fetch_k) * fetch_k);
    mmr_kernel<<<nq, 128, smem, static_cast<cudaStream_t>(stream)>>>(q, cand, n_cand, fetch_k, dim, k,
                                                                     static_cast<double>(lambda_mult), out_sel);
    count_launch();
    RMU_CHECK_LAUNCH();
    return RMU_OK;
}

}  // extern "C"
