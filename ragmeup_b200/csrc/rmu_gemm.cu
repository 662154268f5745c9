#include <algorithm>

#include "rmu_gemm.cuh"

namespace rmu {

int make_split_operand(SplitOperand* op, __half* hi, __half* lo, int64_t rows, int cols, bool is_activation) {
    if (cols % kGemmBK != 0) { set_error("make_split_operand: K must be a multiple of 64"); return RMU_ERR_ARG; }
    op->hi = hi; op->lo = lo; op->rows = rows; op->cols = cols;
    const uint64_t pitch = static_cast<uint64_t>(cols) * sizeof(__half);
    int rc = make_tmap_2d(&op->map_hi, hi, static_cast<uint64_t>(rows), static_cast<uint64_t>(cols), pitch, kGemmBK, 128, 2);
    if (rc == RMU_OK) rc = make_tmap_2d(&op->map_lo, lo, static_cast<uint64_t>(rows), static_cast<uint64_t>(cols), pitch, kGemmBK, 128, 2);
    op->is_weight = !is_activation;
    if (!is_activation) {
        if (rc == RMU_OK) rc = make_tmap_2d(&op->map192_hi, hi, static_cast<uint64_t>(rows), static_cast<uint64_t>(cols), pitch, 64, 192, 2);
        if (rc == RMU_OK) rc = make_tmap_2d(&op->map192_lo, lo, static_cast<uint64_t>(rows), static_cast<uint64_t>(cols), pitch, 64, 192, 2);
        if (rc == RMU_OK) rc = make_tmap_2d(&op->map256_hi, hi, static_cast<uint64_t>(rows), static_cast<uint64_t>(cols), pitch, 64, 256, 2);
        if (rc == RMU_OK) rc = make_tmap_2d(&op->map256_lo, lo, static_cast<uint64_t>(rows), static_cast<uint64_t>(cols), pitch, 64, 256, 2);
    }
    return rc;
}

template <int MODE, int BN>
static int launch_bn(const SplitOperand& A, const SplitOperand& W, const GemmParams& p, int sms, cudaStream_t st) {
    auto kern = gemm_f16x3_kernel<MODE, BN>;
    // the attribute is per device and the call is cheap: set it on every launch (one process may drive several GPUs)
    RMU_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kGemmSmem)));
    const int tiles = ((p.M + kGemmBM - 1) / kGemmBM) * (p.N / BN);
    const int grid = tiles < sms ? tiles : sms;
    ProfScope _ps(PROF_GEMM, st);
    const CUtensorMap& wh = BN == 128 ? W.map_hi : BN == 192 ? W.map192_hi : W.map256_hi;
    const CUtensorMap& wl = BN == 128 ? W.map_lo : BN == 192 ? W.map192_lo : W.map256_lo;
    kern<<<grid, 64 + 32 * gemm_epi_warps<MODE, BN>(), kGemmSmem, st>>>(A.map_hi, A.map_lo, wh, wl, p);
    count_launch();
    RMU_CHECK_LAUNCH();
    return RMU_OK;
}

// tile width: 192 when it divides N, else 256, else 128
template <int MODE>
static int launch_mode(const SplitOperand& A, const SplitOperand& W, const GemmParams& p, int sms, cudaStream_t st) {
    int bn = 128;
    if (p.N % 192 == 0) bn = 192;           // measured best on the MiniLM / bge shapes (768, 1152, 1536, 2304, 3072 ...)
    else if (p.N % 256 == 0) bn = 256;
    if (!W.is_weight) bn = 128;              // operand without the wide weight maps
    if (bn == 256) return launch_bn<MODE, 256>(A, W, p, sms, st);
    if (bn == 192) return launch_bn<MODE, 192>(A, W, p, sms, st);
    return launch_bn<MODE, 128>(A, W, p, sms, st);
}

bool gemm_ln_supported(const SplitOperand& W, int N) {
    return W.is_weight && (N == 2 * kLnBN || N == 4 * kLnBN);
}

int launch_gemm_ln(const SplitOperand& A, const SplitOperand& W, const GemmLnParams& p_in, int sms, cudaStream_t st) {
    const GemmLnParams& p = p_in;
    if (p.M <= 0) return RMU_OK;
    if (!gemm_ln_supported(W, p.N) || p.K % kGemmBK != 0 || A.cols != p.K || W.cols != p.K || W.rows < p.N || A.rows < p.M) {
        set_error("launch_gemm_ln: shape not supported (N = 384 or 768, K % 64)");
        return RMU_ERR_UNSUPPORTED;
    }
    const int CL = p.N / kLnBN;
    // three epilogue warps per TMEM lane quadrant when the projection is short (K <= 512: its epilogue, not its MMAs,
    // bounds it: 158 -> 145 us at K = 384) and the cluster is a pair (shared-memory budget)
    const bool epi12 = CL == 2 && p.K <= 512;
    if (epi12) RMU_CUDA(cudaFuncSetAttribute(gemm_f16x3_ln_kernel<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(ln_smem_bytes(12))));
    else RMU_CUDA(cudaFuncSetAttribute(gemm_f16x3_ln_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(ln_smem_bytes(8))));
    const int m_blks = (p.M + kGemmBM - 1) / kGemmBM;
    const int clusters = std::max(1, std::min(m_blks, sms / CL));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(static_cast<unsigned>(clusters * CL));
    cfg.blockDim = dim3(64 + 32 * (epi12 ? 12 : 8));
    cfg.dynamicSmemBytes = ln_smem_bytes(epi12 ? 12 : 8);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = static_cast<unsigned>(CL);
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    ProfScope _ps(PROF_GEMM, st);
    if (epi12) RMU_CUDA(cudaLaunchKernelEx(&cfg, gemm_f16x3_ln_kernel<12>, A.map_hi, A.map_lo, W.map192_hi, W.map192_lo, p));
    else RMU_CUDA(cudaLaunchKernelEx(&cfg, gemm_f16x3_ln_kernel<8>, A.map_hi, A.map_lo, W.map192_hi, W.map192_lo, p));
    count_launch();
    RMU_CHECK_LAUNCH();
    return RMU_OK;
}

int launch_gemm(int mode, const SplitOperand& A, const SplitOperand& W, const GemmParams& p, int sms, cudaStream_t st) {
    if (p.M <= 0) return RMU_OK;
    if (p.N % 128 != 0 || p.K % kGemmBK != 0 || A.cols != p.K || W.cols != p.K || W.rows < p.N || A.rows < p.M) {
        set_error("launch_gemm: shape not supported (N % 128, K % 64)");
        return RMU_ERR_UNSUPPORTED;
    }
    switch (mode) {
        case GEMM_BIAS_GELU_SPLIT: return launch_mode<GEMM_BIAS_GELU_SPLIT>(A, W, p, sms, st);
        case GEMM_BIAS_RESID_F32: return launch_mode<GEMM_BIAS_RESID_F32>(A, W, p, sms, st);
        case GEMM_BIAS_SPLIT_QSCALE: return launch_mode<GEMM_BIAS_SPLIT_QSCALE>(A, W, p, sms, st);
    }
    set_error("launch_gemm: bad mode");
    return RMU_ERR_ARG;
}

}  // namespace rmu
