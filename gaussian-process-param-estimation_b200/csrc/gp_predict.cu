// Kriging at new points (gaussian_proc/_predict.py). With the cross block P (npad x mc: training rows, test columns),
// W = inv(L) from gp_trtri_f64 and S = Kn^-1 [X z] from gp_potrs_f64, everything n-sized the mean, the variance and the
// covariance need comes from
//   V = W P                    one DMMA GEMM (W lower: k < m0 + 128, the operand layout of W21 = -W22 T in trtri)
//   out[j][c] = P[:, j]^T S[:, c]   (c < p)     out[j][p] = ||V[:, j]||^2
// The second line is one pass over P and V in 2048-row chunks (per-column partials) and a fixed-order sum over the chunks:
// a column's result does not depend on how many columns are predicted together.
#include "../../include/gpgp.h"
#include "gp_common.cuh"
#include "gp_internal.h"

namespace gp {

constexpr int PRED_MAXP = 16;
constexpr int PRED_ROWS = 2048;   // rows per partial chunk

// partial[kc][j][0..p) = sum_{k in chunk kc} P[k][j] S[k][:], partial[kc][j][p] = sum_{k in chunk kc} V[k][j]^2.
// 128 columns per CTA, two threads per column (even / odd rows), S staged 128 rows at a time.
template <int PP>
__global__ void __launch_bounds__(256)
predict_partial_kernel(const double* __restrict__ P, int64_t ldp, const double* __restrict__ V, int64_t ldv,
                       const double* __restrict__ S, int p, int npad, int mcpad, double* __restrict__ partial) {
    constexpr int SP = PP + 1;
    __shared__ double ss[128 * SP];
    __shared__ double comb[128 * SP];
    const int tid = threadIdx.x, jl = tid & 127, half = tid >> 7;
    const int j = blockIdx.x * 128 + jl, kc = blockIdx.y;
    const int kbeg = kc * PRED_ROWS, kend = min(npad, kbeg + PRED_ROWS);
    double acc[PP], nrm = 0.0;
#pragma unroll
    for (int c = 0; c < PP; ++c) acc[c] = 0.0;
    for (int k0 = kbeg; k0 < kend; k0 += 128) {
        __syncthreads();
        for (int idx = tid; idx < 128 * p; idx += 256) {
            int r = idx / p, c = idx - r * p;
            ss[r * SP + c] = S[(int64_t)(k0 + r) * p + c];
        }
        __syncthreads();
#pragma unroll 4
        for (int kk = half; kk < 128; kk += 2) {
            const double pv = P[(int64_t)(k0 + kk) * ldp + j];
            const double vv = V[(int64_t)(k0 + kk) * ldv + j];
            nrm += vv * vv;
#pragma unroll
            for (int c = 0; c < PP; ++c)
                if (c < p) acc[c] += pv * ss[kk * SP + c];
        }
    }
    __syncthreads();
    if (half == 1) {
#pragma unroll
        for (int c = 0; c < PP; ++c) comb[jl * SP + c] = acc[c];
        comb[jl * SP + PP] = nrm;
    }
    __syncthreads();
    if (half == 0) {
        double* dst = partial + ((int64_t)kc * mcpad + j) * (p + 1);
#pragma unroll
        for (int c = 0; c < PP; ++c)
            if (c < p) dst[c] = acc[c] + comb[jl * SP + c];
        dst[p] = nrm + comb[jl * SP + PP];
    }
}

// out[t] = sum over the chunks, in chunk order, of partial[kc][t] (t < mc * (p + 1))
__global__ void predict_reduce_kernel(const double* __restrict__ partial, int nchunks, int64_t stride, int64_t width,
                                      double* __restrict__ out) {
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= width) return;
    double s = 0.0;
    for (int kc = 0; kc < nchunks; ++kc) s += partial[(int64_t)kc * stride + t];
    out[t] = s;
}

}  // namespace gp

using namespace gp;

extern "C" {

int64_t gp_predict_workspace_bytes(int64_t npad, int64_t mc, int64_t p) {
    if (npad <= 0 || (npad % 128) || mc <= 0 || p <= 0 || p > PRED_MAXP) return -1;
    int64_t nchunks = (npad + PRED_ROWS - 1) / PRED_ROWS, mcpad = gp_padded_size(mc);
    return (int64_t)sizeof(double) * nchunks * mcpad * (p + 1);
}

int gp_predict_dense(const double* W, int64_t n, int64_t npad, const double* S, int64_t p, const double* P, int64_t mc,
                     int64_t ldp, double* V, int64_t ldv, double* out, void* ws, void* stream) {
    if (!W || !S || !P || !V || !out || !ws || n <= 0 || npad != gp_padded_size(n) || npad > INT32_MAX || p <= 0 ||
        p > PRED_MAXP || mc <= 0)
        return -1;
    const int64_t mcpad = gp_padded_size(mc);
    if (mcpad > INT32_MAX || ldp < mcpad || ldv < mcpad || (ldp & 1) || (ldv & 1)) return -2;
    if (((uintptr_t)W | (uintptr_t)P | (uintptr_t)V) & 15) return -3;
    cudaStream_t s = (cudaStream_t)stream;
    int rc = launch_dgemm(0, 1, V, ldv, W, npad, P, ldp, (int)npad, (int)mcpad, (int)npad, 1.0, 0.0, KR_A_LOWER, TM_ALL, s);
    if (rc) return rc;
    const int nchunks = (int)((npad + PRED_ROWS - 1) / PRED_ROWS);
    double* partial = (double*)ws;
    dim3 grid((unsigned)(mcpad / 128), (unsigned)nchunks);
    if (p <= 8) predict_partial_kernel<8><<<grid, 256, 0, s>>>(P, ldp, V, ldv, S, (int)p, (int)npad, (int)mcpad, partial);
    else predict_partial_kernel<PRED_MAXP><<<grid, 256, 0, s>>>(P, ldp, V, ldv, S, (int)p, (int)npad, (int)mcpad, partial);
    const int64_t width = mc * (p + 1);
    predict_reduce_kernel<<<(unsigned)((width + 255) / 256), 256, 0, s>>>(partial, nchunks, mcpad * (p + 1), width, out);
    GP_COUNT(2);
    GP_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
