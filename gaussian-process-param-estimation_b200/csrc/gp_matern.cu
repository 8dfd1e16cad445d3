// Dense Matern correlation generator (and optional dK/drho) -- replaces
// gaussian_proc/generate_correlation/_generate_dense_correlation.pyx:23-91 (OpenMP row loop over i, j >= i with
// mirror store) by 128x128 output tiles: the two point tiles are staged in shared memory, lower tiles are
// evaluated once and stored twice (direct rows as 32-byte per-thread segments, the mirror through a padded
// shared-memory transpose so both stores are fully coalesced). HBM-write bound: 8 n^2 bytes (16 n^2 with dK).
#include "../../include/gpgp.h"
#include "gp_common.cuh"
#include "gp_matern.cuh"
#include "gp_internal.h"

namespace gp {

constexpr int MT = 128;          // tile edge
constexpr int MAXD = 8;          // max spatial dimension staged in shared memory
constexpr int CH = 32;           // rows per transpose chunk
constexpr int PITCH = MT + 1;    // padded pitch of the transpose buffer (doubles)

#ifndef GP_MATERN_MINB
#define GP_MATERN_MINB 2
#endif
template <int MODE, bool WITH_DK>
__global__ void __launch_bounds__(256, WITH_DK ? 2 : GP_MATERN_MINB)
matern_dense_kernel(const double* __restrict__ pts, int n, int d, int npad, double* __restrict__ K,
                    double* __restrict__ dK, MaternParams mp) {
    extern __shared__ double dyn_smem[];
    double (*pr)[MT] = reinterpret_cast<double (*)[MT]>(dyn_smem);           // row points, coordinate-major [d][MT]
    double (*pc)[MT] = reinterpret_cast<double (*)[MT]>(dyn_smem + d * MT);  // column points [d][MT]
    double* tbuf = dyn_smem + 2 * d * MT;                                     // [(1|2)][CH][PITCH]
    __shared__ double isc[MAXD];

    // lower-triangular tile enumeration
    int b = blockIdx.x;
    int tm = (int)((sqrt(8.0 * b + 1.0) - 1.0) * 0.5);
    while ((tm + 1) * (tm + 2) / 2 <= b) ++tm;
    while (tm * (tm + 1) / 2 > b) --tm;
    int tn = b - tm * (tm + 1) / 2;
    const int m0 = tm * MT, n0 = tn * MT;
    const int tid = threadIdx.x;

    if (tid < d) isc[tid] = mp.inv_scale[tid];
    for (int idx = tid; idx < MT * d; idx += 256) {
        int r = idx / d, k = idx - r * d;
        int gr = m0 + r, gc = n0 + r;
        pr[k][r] = (gr < n) ? pts[(int64_t)gr * d + k] : 0.0;
        pc[k][r] = (gc < n) ? pts[(int64_t)gc * d + k] : 0.0;
    }
    __syncthreads();

    const int tx = tid & 31, ty = tid >> 5;  // tx: 4 consecutive columns; ty: rows ty + 8*rr
    double cx[MAXD][4];
#pragma unroll
    for (int k = 0; k < MAXD; ++k)
        if (k < d)
#pragma unroll
            for (int e = 0; e < 4; ++e) cx[k][e] = pc[k][tx * 4 + e];

    for (int chunk = 0; chunk < MT / CH; ++chunk) {
        // (the values go straight to the global row and to the transpose buffer: only 4 of them are live per thread, which
        // keeps the kernel at 3 CTAs per SM - it is bound by instruction issue of the FP64 sqrt / exp sequences, not by HBM)
        if (tm != tn && chunk > 0) __syncthreads();          // the previous chunk's mirror reads are done
#pragma unroll
        for (int rr = 0; rr < 4; ++rr) {
            const int rl = ty + 8 * rr;
            const int r = chunk * CH + rl;
            const int gi = m0 + r;
            double v[4], dv[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                int gj = n0 + tx * 4 + e;
                double val, dval = 0.0;
                if (gi >= n || gj >= n) {
                    val = (gi == gj) ? 1.0 : 0.0;
                } else if (gi == gj) {
                    val = 1.0;
                } else {
                    double s = 0.0;
#pragma unroll
                    for (int k = 0; k < MAXD; ++k)
                        if (k < d) {
                            double t = (pr[k][r] - cx[k][e]) * isc[k];
                            s += t * t;
                        }
                    double x = sqrt(s);
                    if (WITH_DK) matern_value_drho<MODE>(x, mp, &val, &dval);
                    else val = matern_value<MODE>(x, mp);
                }
                v[e] = val;
                dv[e] = dval;
            }
            // direct store: 4 doubles = 32 bytes per thread, a warp covers one full 1 KB tile row
            double* dst = K + (int64_t)gi * npad + n0 + tx * 4;
            reinterpret_cast<double2*>(dst)[0] = make_double2(v[0], v[1]);
            reinterpret_cast<double2*>(dst)[1] = make_double2(v[2], v[3]);
            if (WITH_DK) {
                double* dd = dK + (int64_t)gi * npad + n0 + tx * 4;
                reinterpret_cast<double2*>(dd)[0] = make_double2(dv[0], dv[1]);
                reinterpret_cast<double2*>(dd)[1] = make_double2(dv[2], dv[3]);
            }
            if (tm != tn) {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    tbuf[rl * PITCH + tx * 4 + e] = v[e];
                    if (WITH_DK) tbuf[CH * PITCH + rl * PITCH + tx * 4 + e] = dv[e];
                }
            }
        }
        if (tm != tn) {
            // mirror store through shared memory: lane -> local row (32 consecutive doubles = 256 B of the mirrored row),
            // warp -> column
            __syncthreads();
            for (int c = ty; c < MT; c += 8) {
                int64_t o = (int64_t)(n0 + c) * npad + m0 + chunk * CH + tx;
                K[o] = tbuf[tx * PITCH + c];
                if (WITH_DK) dK[o] = tbuf[CH * PITCH + tx * PITCH + c];
            }
        }
    }
}

template <int MODE>
static int launch_mode(const double* pts, int n, int d, int npad, double* K, double* dK, const MaternParams& mp,
                       cudaStream_t s) {
    int T = npad / MT;
    int tiles = T * (T + 1) / 2;
    size_t smem = sizeof(double) * (2 * d * MT + (dK ? 2 : 1) * CH * PITCH);
    if (dK) {
        if (int rc = configure_once((const void*)matern_dense_kernel<MODE, true>, 96 * 1024)) return rc;
        matern_dense_kernel<MODE, true><<<tiles, 256, smem, s>>>(pts, n, d, npad, K, dK, mp);
    } else {
        if (int rc = configure_once((const void*)matern_dense_kernel<MODE, false>, 96 * 1024)) return rc;
        matern_dense_kernel<MODE, false><<<tiles, 256, smem, s>>>(pts, n, d, npad, K, nullptr, mp);
    }
    GP_COUNT(1);
    GP_LAUNCH_CHECK();
    return 0;
}

// ---- rectangular cross-correlation block K(P_rows, P_cols) for distributed (block-cyclic) layouts -----------------
// Global indices decide the special cases: identity padding for indices >= n, exactly 1 (+ eta) on the diagonal.
template <int MODE, bool DK>
__global__ void __launch_bounds__(256)
matern_cross_kernel(const double* __restrict__ prow, const double* __restrict__ pcol, const int* __restrict__ rg,
                    const int* __restrict__ cg, int n, int d, int64_t ld, double* __restrict__ out, double eta, MaternParams mp) {
    __shared__ double sr[MAXD][64];
    __shared__ double sc[MAXD][128];
    __shared__ int gr[64], gc[128];
    const int r0 = blockIdx.y * 64, c0 = blockIdx.x * 128, tid = threadIdx.x;
    for (int idx = tid; idx < 64 * d; idx += 256) { int r = idx / d, k = idx - r * d; sr[k][r] = prow[(int64_t)(r0 + r) * d + k]; }
    for (int idx = tid; idx < 128 * d; idx += 256) { int r = idx / d, k = idx - r * d; sc[k][r] = pcol[(int64_t)(c0 + r) * d + k]; }
    if (tid < 64) gr[tid] = rg[r0 + tid];
    if (tid < 128) gc[tid] = cg[c0 + tid];
    __syncthreads();
    const int tx = tid & 31, ty = tid >> 5;
    for (int rr = ty; rr < 64; rr += 8) {
        const int gi = gr[rr];
        double v[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int cl = tx * 4 + e, gj = gc[cl];
            double val;
            if (gi >= n || gj >= n) val = (gi == gj && !DK) ? 1.0 : 0.0;
            else if (gi == gj) val = DK ? 0.0 : 1.0 + eta;
            else {
                double s = 0.0;
#pragma unroll
                for (int k = 0; k < MAXD; ++k)
                    if (k < d) { double t = (sr[k][rr] - sc[k][cl]) * mp.inv_scale[k]; s += t * t; }
                if (DK) {
                    double kv;
                    matern_value_drho<MODE>(sqrt(s), mp, &kv, &val);      // d/d rho of an isotropic correlation scale
                } else {
                    val = matern_value<MODE>(sqrt(s), mp);
                }
            }
            v[e] = val;
        }
        double* dst = out + (int64_t)(r0 + rr) * ld + c0 + tx * 4;
        reinterpret_cast<double2*>(dst)[0] = make_double2(v[0], v[1]);
        reinterpret_cast<double2*>(dst)[1] = make_double2(v[2], v[3]);
    }
}

template <int MODE>
static int launch_cross(const double* prow, const double* pcol, const int* rg, const int* cg, int nr, int nc, int n, int d,
                        int64_t ld, double* out, double eta, const MaternParams& mp, cudaStream_t s, bool dk = false) {
    dim3 grid(nc / 128, nr / 64);
    if (dk) matern_cross_kernel<MODE, true><<<grid, 256, 0, s>>>(prow, pcol, rg, cg, n, d, ld, out, eta, mp);
    else matern_cross_kernel<MODE, false><<<grid, 256, 0, s>>>(prow, pcol, rg, cg, n, d, ld, out, eta, mp);
    GP_COUNT(1);
    GP_LAUNCH_CHECK();
    return 0;
}

// ---- cross-correlation P[i][j] = K(p_i, q_j) between two point sets (prediction at new points) ---------------------
// Same distance expression and k order as matern_dense_kernel, so P(points, points) equals the dense K bit for bit.
// Nothing can be mirrored: every 64 x 128 tile is evaluated. Entries with i >= n or j >= m are exactly 0.
template <int MODE>
__global__ void __launch_bounds__(256)
matern_cross_points_kernel(const double* __restrict__ p, int n, const double* __restrict__ q, int m, int d, int64_t ldp,
                           double* __restrict__ P, MaternParams mp) {
    __shared__ double sr[MAXD][64];
    __shared__ double sc[MAXD][128];
    const int r0 = blockIdx.y * 64, c0 = blockIdx.x * 128, tid = threadIdx.x;
    for (int idx = tid; idx < 64 * d; idx += 256) {
        int r = idx / d, k = idx - r * d;
        sr[k][r] = (r0 + r < n) ? p[(int64_t)(r0 + r) * d + k] : 0.0;
    }
    for (int idx = tid; idx < 128 * d; idx += 256) {
        int r = idx / d, k = idx - r * d;
        sc[k][r] = (c0 + r < m) ? q[(int64_t)(c0 + r) * d + k] : 0.0;
    }
    __syncthreads();
    const int tx = tid & 31, ty = tid >> 5;   // tx: 4 consecutive columns; ty: rows ty + 8*rr
    double cx[MAXD][4];
#pragma unroll
    for (int k = 0; k < MAXD; ++k)
        if (k < d)
#pragma unroll
            for (int e = 0; e < 4; ++e) cx[k][e] = sc[k][tx * 4 + e];
    for (int rr = ty; rr < 64; rr += 8) {
        const int gi = r0 + rr;
        double v[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int gj = c0 + tx * 4 + e;
            double val = 0.0;
            if (gi < n && gj < m) {
                double s = 0.0;
#pragma unroll
                for (int k = 0; k < MAXD; ++k)
                    if (k < d) {
                        double t = (sr[k][rr] - cx[k][e]) * mp.inv_scale[k];
                        s += t * t;
                    }
                val = matern_value<MODE>(sqrt(s), mp);
            }
            v[e] = val;
        }
        double* dst = P + (int64_t)gi * ldp + c0 + tx * 4;
        reinterpret_cast<double2*>(dst)[0] = make_double2(v[0], v[1]);
        reinterpret_cast<double2*>(dst)[1] = make_double2(v[2], v[3]);
    }
}

template <int MODE>
static int launch_cross_points(const double* p, int n, const double* q, int m, int d, int64_t ldp, double* P,
                               const MaternParams& mp, cudaStream_t s) {
    dim3 grid((unsigned)(gp_padded_size(m) / 128), (unsigned)(gp_padded_size(n) / 64));
    matern_cross_points_kernel<MODE><<<grid, 256, 0, s>>>(p, n, q, m, d, ldp, P, mp);
    GP_COUNT(1);
    GP_LAUNCH_CHECK();
    return 0;
}

}  // namespace gp

extern "C" int gp_matern_dense(const double* points, int64_t n, int64_t d, const double* scale_host, double nu,
                               double* K, int64_t ldk, double* dK, void* stream) {
    using namespace gp;
    if (n <= 0 || d <= 0 || d > MAXD || !points || !K || !scale_host) return -1;
    int64_t npad = gp_padded_size(n);
    if (ldk != npad || npad > INT32_MAX) return -2;
    cudaStream_t s = (cudaStream_t)stream;
    MaternParams mp;
    for (int k = 0; k < d; ++k) {
        if (!(scale_host[k] > 0.0)) return -3;
        if (dK && scale_host[k] != scale_host[0]) return -4;  // d/drho is defined for an isotropic scale only
        mp.inv_scale[k] = 1.0 / scale_host[k];
    }
    mp.nu = nu;
    mp.coef = 0.0;
    mp.sq2nu = 0.0;
    mp.inv_rho = 1.0 / scale_host[0];
    int mode = matern_mode_of(nu);
    if (mode == MAT_GENERAL) {
        if (!(nu > 0.0)) return -5;
        mp.coef = pow(2.0, 1.0 - nu) / tgamma(nu);
        mp.sq2nu = sqrt(2.0 * nu);
    }
    switch (mode) {
        case MAT_05: return launch_mode<MAT_05>(points, (int)n, (int)d, (int)npad, K, dK, mp, s);
        case MAT_15: return launch_mode<MAT_15>(points, (int)n, (int)d, (int)npad, K, dK, mp, s);
        case MAT_25: return launch_mode<MAT_25>(points, (int)n, (int)d, (int)npad, K, dK, mp, s);
        case MAT_GAUSS: return launch_mode<MAT_GAUSS>(points, (int)n, (int)d, (int)npad, K, dK, mp, s);
        default: return launch_mode<MAT_GENERAL>(points, (int)n, (int)d, (int)npad, K, dK, mp, s);
    }
}

// out[r][c] = K(p_row[r], p_col[c]) (+ eta on the global diagonal) for nr x nc blocks of a larger padded matrix;
// row_gidx / col_gidx are the global indices of the rows / columns (device int32), n the unpadded global size.
static int matern_cross_impl(const double* prow, const double* pcol, const int* row_gidx, const int* col_gidx, int64_t nr,
                             int64_t nc, int64_t n, int64_t d, const double* scale_host, double nu, double eta, double* out,
                             int64_t ld, void* stream, bool dk) {
    using namespace gp;
    if (!prow || !pcol || !row_gidx || !col_gidx || !out || !scale_host || nr <= 0 || nc <= 0 || (nr % 64) || (nc % 128) || d <= 0 ||
        d > MAXD || (ld & 1))
        return -1;
    MaternParams mp;
    for (int k = 0; k < d; ++k) {
        if (!(scale_host[k] > 0.0)) return -3;
        if (dk && scale_host[k] != scale_host[0]) return -4;
        mp.inv_scale[k] = 1.0 / scale_host[k];
    }
    mp.nu = nu; mp.coef = 0.0; mp.sq2nu = 0.0; mp.inv_rho = 1.0 / scale_host[0];
    int mode = matern_mode_of(nu);
    if (mode == MAT_GENERAL) {
        if (!(nu > 0.0)) return -5;
        mp.coef = pow(2.0, 1.0 - nu) / tgamma(nu);
        mp.sq2nu = sqrt(2.0 * nu);
    }
    cudaStream_t s = (cudaStream_t)stream;
    switch (mode) {
        case MAT_05: return launch_cross<MAT_05>(prow, pcol, row_gidx, col_gidx, (int)nr, (int)nc, (int)n, (int)d, ld, out, eta, mp, s, dk);
        case MAT_15: return launch_cross<MAT_15>(prow, pcol, row_gidx, col_gidx, (int)nr, (int)nc, (int)n, (int)d, ld, out, eta, mp, s, dk);
        case MAT_25: return launch_cross<MAT_25>(prow, pcol, row_gidx, col_gidx, (int)nr, (int)nc, (int)n, (int)d, ld, out, eta, mp, s, dk);
        case MAT_GAUSS: return launch_cross<MAT_GAUSS>(prow, pcol, row_gidx, col_gidx, (int)nr, (int)nc, (int)n, (int)d, ld, out, eta, mp, s, dk);
        default: return launch_cross<MAT_GENERAL>(prow, pcol, row_gidx, col_gidx, (int)nr, (int)nc, (int)n, (int)d, ld, out, eta, mp, s, dk);
    }
}

extern "C" int gp_matern_cross(const double* prow, const double* pcol, const int* row_gidx, const int* col_gidx, int64_t nr,
                               int64_t nc, int64_t n, int64_t d, const double* scale_host, double nu, double eta, double* out,
                               int64_t ld, void* stream) {
    return matern_cross_impl(prow, pcol, row_gidx, col_gidx, nr, nc, n, d, scale_host, nu, eta, out, ld, stream, false);
}

// the same block of dK/d rho (isotropic correlation scale): zero on the global diagonal and in the padding
extern "C" int gp_matern_cross_dk(const double* prow, const double* pcol, const int* row_gidx, const int* col_gidx, int64_t nr,
                                  int64_t nc, int64_t n, int64_t d, const double* scale_host, double nu, double* out,
                                  int64_t ld, void* stream) {
    return matern_cross_impl(prow, pcol, row_gidx, col_gidx, nr, nc, n, d, scale_host, nu, 0.0, out, ld, stream, true);
}

extern "C" int gp_matern_cross_points(const double* p, int64_t n, const double* q, int64_t m, int64_t d,
                                      const double* scale_host, double nu, double* P, int64_t ldp, void* stream) {
    using namespace gp;
    if (!p || !q || !P || !scale_host || n <= 0 || m <= 0 || d <= 0 || d > MAXD) return -1;
    int64_t npad = gp_padded_size(n), mpad = gp_padded_size(m);
    if (ldp < mpad || (ldp & 1) || ((uintptr_t)P & 15) || npad > INT32_MAX || mpad > INT32_MAX) return -2;
    MaternParams mp;
    for (int k = 0; k < d; ++k) {
        if (!(scale_host[k] > 0.0)) return -3;
        mp.inv_scale[k] = 1.0 / scale_host[k];
    }
    mp.nu = nu; mp.coef = 0.0; mp.sq2nu = 0.0; mp.inv_rho = 1.0 / scale_host[0];
    int mode = matern_mode_of(nu);
    if (mode == MAT_GENERAL) {
        if (!(nu > 0.0)) return -5;
        mp.coef = pow(2.0, 1.0 - nu) / tgamma(nu);
        mp.sq2nu = sqrt(2.0 * nu);
    }
    cudaStream_t s = (cudaStream_t)stream;
    switch (mode) {
        case MAT_05: return launch_cross_points<MAT_05>(p, (int)n, q, (int)m, (int)d, ldp, P, mp, s);
        case MAT_15: return launch_cross_points<MAT_15>(p, (int)n, q, (int)m, (int)d, ldp, P, mp, s);
        case MAT_25: return launch_cross_points<MAT_25>(p, (int)n, q, (int)m, (int)d, ldp, P, mp, s);
        case MAT_GAUSS: return launch_cross_points<MAT_GAUSS>(p, (int)n, q, (int)m, (int)d, ldp, P, mp, s);
        default: return launch_cross_points<MAT_GENERAL>(p, (int)n, q, (int)m, (int)d, ldp, P, mp, s);
    }
}
