// C-ABI entry points that are thin argument-checking shims over the internal launchers.
#include "../../include/gpgp.h"
#include "gp_common.cuh"
#include "gp_internal.h"

extern "C" {

int gp_abi_version(void) { return 100; }

int64_t gp_padded_size(int64_t n) { return n <= 0 ? 0 : ((n + GP_TILE - 1) / GP_TILE) * GP_TILE; }

int gp_dgemm_f64(int at, int bt, double* C, int64_t ldc, const double* A, int64_t lda, const double* B,
                 int64_t ldb, int64_t M, int64_t N, int64_t K, double alpha, double beta, int krange, int tmask,
                 void* stream) {
    if (M > INT32_MAX || N > INT32_MAX || K > INT32_MAX) return -1;
    return gp::launch_dgemm(at, bt, C, ldc, A, lda, B, ldb, (int)M, (int)N, (int)K, alpha, beta, krange, tmask,
                            (cudaStream_t)stream);
}

int gp_dgemm_ktab_f64(int at, int bt, double* C, int64_t ldc, const double* A, int64_t lda, const double* B, int64_t ldb,
                      int64_t M, int64_t N, int64_t K, double alpha, double beta, const int* kbeg_tab, const int* kend_tab,
                      void* stream) {
    if (M > INT32_MAX || N > INT32_MAX || K > INT32_MAX) return -1;
    return gp::launch_dgemm_ktab(at, bt, C, ldc, A, lda, B, ldb, (int)M, (int)N, (int)K, alpha, beta, kbeg_tab, kend_tab,
                                 (cudaStream_t)stream);
}

unsigned long long gp_launch_count(void) { return gp::g_launch_count.load(std::memory_order_relaxed); }

int gp_gemm_profile_enable(int on) { return gp::profile_enable(on); }

int gp_gemm_profile_read(double* ms_sum_host, double* ms_union_host, double* flops_host, long long* launches_host) {
    if (!ms_sum_host || !ms_union_host || !flops_host || !launches_host) return -1;
    return gp::profile_read(ms_sum_host, ms_union_host, flops_host, launches_host);
}

}  // extern "C"
