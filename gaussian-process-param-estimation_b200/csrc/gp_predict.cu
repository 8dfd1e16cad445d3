// Kriging at new points (gaussian_proc/_predict.py). With the cross block P (npad x mc: training rows, test columns),
// W = inv(L) from gp_trtri_f64 and S = Kn^-1 [X z] from gp_potrs_f64, everything n-sized the mean, the variance and the
// covariance need comes from
//   V = W P                    one DMMA GEMM (W lower: k < m0 + 128, the operand layout of W21 = -W22 T in trtri)
//   out[j][c] = P[:, j]^T S[:, c]   (c < p)     out[j][p] = ||V[:, j]||^2
// The second line is one pass over P and V in 2048-row chunks (per-column partials) and a fixed-order sum over the chunks:
// a column's result does not depend on how many columns are predicted together.
//
// Gradients with respect to the test-point coordinates (gp_predict_grad_dense): with G_k[i][j] = dP[i][j]/dq_jk,
//   out[(j d + k)(p+1) + c] = G_k[:, j]^T S[:, c]  (c < p)     out[(j d + k)(p+1) + p] = G_k[:, j]^T U[:, j]
// where U = W^T V = Kn^-1 P is one more gp_dgemm_ktab_f64 by the caller. G is regenerated from the points in the same
// 2048-row chunks and never stored; the partials are summed over the chunks by predict_reduce_kernel.
#include "../../include/gpgp.h"
#include "gp_common.cuh"
#include "gp_internal.h"
#include "gp_matern.cuh"

namespace gp {

constexpr int PRED_MAXP = 16;
constexpr int PRED_ROWS = 2048;   // rows per partial chunk
constexpr int GRAD_MAXD = 8;      // spatial dimensions (gp_matern_cross_points' limit)
constexpr int GRAD_COLS = 64;     // test columns per CTA (threadIdx.x); threadIdx.y picks a group of dimensions

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

// Dimensions per thread: DK (PP + 1) accumulators, 36 for p <= 8 and 34 for p <= 16. With d <= DK (d <= 4 for p <= 8,
// d <= 2 for p <= 16) one thread owns every dimension of its column and x, h(x) are evaluated once per pair; a larger d
// takes ceil(d / DK) thread rows, each evaluating the pair again.
template <int PP>
struct GradDims { static constexpr int DK = PP <= 8 ? 4 : 2; };

// partial[kc][(j d + k)(p+1) + c] over the rows i < n of chunk kc; one thread per (column j, dimension group), rows in order.
// The training points and the S rows of a 128-row slab are staged in shared memory; U is read coalesced across columns.
template <int MODE, int PP>
__global__ void __launch_bounds__(256)
predict_grad_partial_kernel(const double* __restrict__ pts, int n, const double* __restrict__ q, int mc, int d,
                            MaternParams mp, const double* __restrict__ S, int p, const double* __restrict__ U,
                            int64_t ldu, double* __restrict__ partial) {
    constexpr int DK = GradDims<PP>::DK;
    __shared__ double sp[GRAD_MAXD][128];
    __shared__ double ss[128 * PP];
    const int tid = threadIdx.y * GRAD_COLS + threadIdx.x, nthr = GRAD_COLS * blockDim.y;
    const int j = blockIdx.x * GRAD_COLS + threadIdx.x, kc = blockIdx.y;
    const int k0 = threadIdx.y * DK;
    const int ibeg = kc * PRED_ROWS, iend = min(n, ibeg + PRED_ROWS);
    const bool live = j < mc;
    double qj[GRAD_MAXD], qo[DK], so[DK], acc[DK][PP + 1];
#pragma unroll
    for (int k = 0; k < GRAD_MAXD; ++k) qj[k] = (live && k < d) ? q[(int64_t)j * d + k] : 0.0;
#pragma unroll
    for (int kk = 0; kk < DK; ++kk) {
        const bool own = live && k0 + kk < d;
        qo[kk] = own ? q[(int64_t)j * d + k0 + kk] : 0.0;
        so[kk] = 0.0;
#pragma unroll
        for (int k = 0; k < GRAD_MAXD; ++k)
            if (k == k0 + kk && own) so[kk] = mp.inv_scale[k];
#pragma unroll
        for (int c = 0; c <= PP; ++c) acc[kk][c] = 0.0;
    }
    for (int i0 = ibeg; i0 < iend; i0 += 128) {
        const int rows = min(128, iend - i0);
        __syncthreads();
        for (int idx = tid; idx < rows * d; idx += nthr) {
            int r = idx / d, k = idx - r * d;
            sp[k][r] = pts[(int64_t)(i0 + r) * d + k];
        }
        for (int idx = tid; idx < rows * p; idx += nthr) {
            int r = idx / p, c = idx - r * p;
            ss[r * PP + c] = S[(int64_t)(i0 + r) * p + c];
        }
        __syncthreads();
        if (!live) continue;
        for (int r = 0; r < rows; ++r) {
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < GRAD_MAXD; ++k)
                if (k < d) {
                    double t = (sp[k][r] - qj[k]) * mp.inv_scale[k];
                    s += t * t;
                }
            const double h = matern_h<MODE>(sqrt(s), mp);
            const double u = U ? U[(int64_t)(i0 + r) * ldu + j] : 0.0;
#pragma unroll
            for (int kk = 0; kk < DK; ++kk) {
                // dP/dq_k = h t_k / scale_k with t_k = (p_k - q_k) / scale_k (0 for a dimension this thread does not own)
                const double g = h * ((sp[k0 + kk < d ? k0 + kk : 0][r] - qo[kk]) * so[kk]) * so[kk];
#pragma unroll
                for (int c = 0; c < PP; ++c)
                    if (c < p) acc[kk][c] += g * ss[r * PP + c];
                acc[kk][PP] += g * u;
            }
        }
    }
    if (!live) return;
    double* dst = partial + (int64_t)kc * mc * d * (p + 1) + (int64_t)j * d * (p + 1);
#pragma unroll
    for (int kk = 0; kk < DK; ++kk)
        if (k0 + kk < d) {
#pragma unroll
            for (int c = 0; c < PP; ++c)
                if (c < p) dst[(k0 + kk) * (p + 1) + c] = acc[kk][c];
            dst[(k0 + kk) * (p + 1) + p] = acc[kk][PP];
        }
}

template <int MODE>
static void launch_grad_partial(const double* pts, int n, const double* q, int mc, int d, const MaternParams& mp,
                                const double* S, int p, const double* U, int64_t ldu, double* partial, cudaStream_t s) {
    const int dk = p <= 8 ? GradDims<8>::DK : GradDims<PRED_MAXP>::DK;
    dim3 grid((unsigned)((mc + GRAD_COLS - 1) / GRAD_COLS), (unsigned)((n + PRED_ROWS - 1) / PRED_ROWS));
    dim3 block(GRAD_COLS, (unsigned)((d + dk - 1) / dk));
    if (p <= 8) predict_grad_partial_kernel<MODE, 8><<<grid, block, 0, s>>>(pts, n, q, mc, d, mp, S, p, U, ldu, partial);
    else predict_grad_partial_kernel<MODE, PRED_MAXP><<<grid, block, 0, s>>>(pts, n, q, mc, d, mp, S, p, U, ldu, partial);
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

int64_t gp_predict_grad_workspace_bytes(int64_t n, int64_t mc, int64_t d, int64_t p) {
    if (n <= 0 || mc <= 0 || d <= 0 || d > GRAD_MAXD || p <= 0 || p > PRED_MAXP) return -1;
    int64_t nchunks = (n + PRED_ROWS - 1) / PRED_ROWS;
    return (int64_t)sizeof(double) * nchunks * mc * d * (p + 1);
}

int gp_predict_grad_dense(const double* points, int64_t n, const double* q, int64_t mc, int64_t d, const double* scale_host,
                          double nu, const double* S, int64_t p, const double* U, int64_t ldu, double* out, void* ws,
                          void* stream) {
    if (!points || !q || !scale_host || !S || !out || !ws || n <= 0 || mc <= 0 || d <= 0 || d > GRAD_MAXD || p <= 0 ||
        p > PRED_MAXP)
        return -1;
    if (gp_padded_size(n) > INT32_MAX || gp_padded_size(mc) > INT32_MAX || (U && ldu < mc)) return -2;
    MaternParams mp;
    int mode;
    if (int rc = matern_params(scale_host, d, nu, false, &mp, &mode)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    double* partial = (double*)ws;
    with_matern_mode(mode, [&](auto tag) {
        launch_grad_partial<decltype(tag)::value>(points, (int)n, q, (int)mc, (int)d, mp, S, (int)p, U, ldu, partial, s);
    });
    const int nchunks = (int)((n + PRED_ROWS - 1) / PRED_ROWS);
    const int64_t width = mc * d * (p + 1);
    predict_reduce_kernel<<<(unsigned)((width + 255) / 256), 256, 0, s>>>(partial, nchunks, width, width, out);
    GP_COUNT(2);
    GP_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
