// Fused dense log-likelihood (+ gradient ingredients) evaluator: one Cholesky per (rho, eta) instead of the 4-9
// fresh O(n^3) solves the reference spends per evaluation (SURVEY 3.3).
//
// It produces every n-sized reduction that gaussian_proc/_likelihood/_direct_likelihood.py:31-157 and
// _profile_likelihood.py:38-132 need, leaving only (m+1)x(m+1) algebra to the host:
//   logdet(Kn), tr Kn^-1, tr Kn^-2, tr(Kn^-1 dK/drho), and with R = [X z], S = Kn^-1 R:
//   G = R^T S, H = S^T S, Q = S^T (dK/drho) S.
// dK/drho is never stored: its tiles are re-evaluated from the points inside the reductions.
#include "../../include/gpgp.h"
#include "gp_common.cuh"
#include "gp_internal.h"
#include "gp_matern.cuh"

namespace gp {

constexpr int MAXP = 16;
constexpr int LMAXD = 8;

// ---- Gram of two tall-skinny blocks: out[a][b] = sum_r A[r][a] * B[r][b]  (rows < nrows) ----------------
__global__ void __launch_bounds__(256)
gram_partial_kernel(const double* __restrict__ A, const double* __restrict__ B, int nrows, int p, int64_t ld,
                    double* partial) {
    __shared__ double sa[64 * MAXP], sb[64 * MAXP];
    const int tid = threadIdx.x;
    const int a = tid / p, b = tid - a * p;
    double acc = 0.0;
    int rows_per_cta = (nrows + gridDim.x - 1) / gridDim.x;
    int r0 = blockIdx.x * rows_per_cta, r1 = min(nrows, r0 + rows_per_cta);
    for (int base = r0; base < r1; base += 64) {
        int cnt = min(64, r1 - base);
        __syncthreads();
        for (int idx = tid; idx < cnt * p; idx += 256) {
            int r = idx / p, c = idx - r * p;
            sa[idx] = A[(int64_t)(base + r) * ld + c];
            sb[idx] = B[(int64_t)(base + r) * ld + c];
        }
        __syncthreads();
        if (tid < p * p)
            for (int r = 0; r < cnt; ++r) acc += sa[r * p + a] * sb[r * p + b];
    }
    if (tid < p * p) partial[(int64_t)blockIdx.x * p * p + tid] = acc;
}

__global__ void sum_partials_kernel(const double* partial, int nparts, int width, double* out) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= width) return;
    double s = 0.0;
    for (int i = 0; i < nparts; ++i) s += partial[(int64_t)i * width + t];
    out[t] = s;
}

// ---- traces over the lower tiles of the symmetric inverse: tr, ||.||_F^2, <Ainv, dK> ---------------------
template <int MODE, bool WITH_DK>
__global__ void __launch_bounds__(256)
trace_tiles_kernel(const double* __restrict__ Ainv, int n, int npad, const double* __restrict__ pts, int d,
                   MaternParams mp, double* partial) {
    __shared__ double pr[LMAXD][128], pc[LMAXD][128];
    __shared__ double red[32];
    int b = blockIdx.x;
    int tm = (int)((sqrt(8.0 * b + 1.0) - 1.0) * 0.5);
    while ((tm + 1) * (tm + 2) / 2 <= b) ++tm;
    while (tm * (tm + 1) / 2 > b) --tm;
    int tn = b - tm * (tm + 1) / 2;
    const int m0 = tm * 128, n0 = tn * 128, tid = threadIdx.x;
    if (WITH_DK) {
        for (int idx = tid; idx < 128 * d; idx += 256) {
            int r = idx / d, k = idx - r * d;
            pr[k][r] = (m0 + r < n) ? pts[(int64_t)(m0 + r) * d + k] : 0.0;
            pc[k][r] = (n0 + r < n) ? pts[(int64_t)(n0 + r) * d + k] : 0.0;
        }
        __syncthreads();
    }
    double t1 = 0.0, t2 = 0.0, t3 = 0.0;
    const int tx = tid & 63, ty = tid >> 6;  // tx: column pair; ty: row phase
    for (int r = ty; r < 128; r += 4) {
        int gi = m0 + r;
        if (gi >= n) break;
        double2 v = *reinterpret_cast<const double2*>(Ainv + (int64_t)gi * npad + n0 + 2 * tx);
        double vals[2] = {v.x, v.y};
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            int gj = n0 + 2 * tx + e;
            if (gj > gi || gj >= n) continue;
            double a = vals[e];
            if (gj == gi) {
                t1 += a;
                t2 += a * a;
            } else {
                t2 += 2.0 * a * a;
                if (WITH_DK) {
                    double s = 0.0, ud = 0.0;
#pragma unroll
                    for (int k = 0; k < LMAXD; ++k)
                        if (k < d) {
                            double t = (pr[k][r] - pc[k][2 * tx + e]) * mp.inv_scale[k];
                            s += t * t;
                            if (k == mp.ddim) ud = t * t;
                        }
                    double val, dval;
                    matern_value_drho<MODE>(sqrt(s), mp, &val, &dval);
                    // d/d scale[ddim]: the isotropic g(x) / rho becomes g(x) u_ddim^2 / (x^2 scale[ddim])
                    if (mp.ddim >= 0) dval = (s > 0.0) ? dval * (ud / s) * mp.inv_scale[mp.ddim] : 0.0;
                    t3 += 2.0 * a * dval;
                }
            }
        }
    }
    t1 = block_sum(t1, red);
    t2 = block_sum(t2, red);
    t3 = block_sum(t3, red);
    if (tid == 0) {
        partial[(int64_t)b * 3 + 0] = t1;
        partial[(int64_t)b * 3 + 1] = t2;
        partial[(int64_t)b * 3 + 2] = t3;
    }
}

// ||W||_F^2 over the lower tiles of the triangular inverse (= tr Kn^-1 without forming the inverse)
__global__ void __launch_bounds__(256)
frob_lower_kernel(const double* __restrict__ W, int n, int npad, double* partial) {
    __shared__ double red[32];
    int tm = blockIdx.y, tn = blockIdx.x;
    double s = 0.0;
    if (tn <= tm) {
        int m0 = tm * 128, n0 = tn * 128;
        for (int idx = threadIdx.x; idx < 128 * 64; idx += 256) {
            int r = idx >> 6, c = (idx & 63) * 2;
            int gi = m0 + r;
            if (gi >= n) break;
            double2 v = *reinterpret_cast<const double2*>(W + (int64_t)gi * npad + n0 + c);
            if (n0 + c <= gi) s += v.x * v.x;
            if (n0 + c + 1 <= gi) s += v.y * v.y;
        }
    }
    s = block_sum(s, red);
    if (threadIdx.x == 0) partial[blockIdx.y * gridDim.x + blockIdx.x] = s;
}

// ---- V = dK * S for S (n x p): 16 rows per CTA (2 per warp), all column tiles streamed through shared memory ---------
// A lane evaluates its 4 columns of the 128-column tile for both rows of its warp; 5 shuffles per accumulator at the end.
// PP = p padded to 8 or 16 at compile time: the accumulators stay in registers. (Round 1 mapped 64 rows to a CTA: n / 64
// CTAs - 125 at n = 8000, less than one per SM - with the accumulators on the stack; 1.57 ms at n = 8000, 5.0 ms at n = 20 000.)
constexpr int SSP = MAXP + 1;  // padded row pitch of a staged skinny tile
constexpr int DKR = 16;        // rows per CTA
template <int MODE, int PP>
__global__ void __launch_bounds__(256)
dk_apply_kernel(const double* __restrict__ pts, int n, int d, MaternParams mp, const double* __restrict__ S, int p,
                int64_t lds, double* __restrict__ V) {
    constexpr int SP = PP + 1;
    __shared__ double pcs[LMAXD][128];
    __shared__ double ss[128 * SP];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g0 = blockIdx.x * DKR + warp * 2;
    double pi[2][LMAXD];
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int k = 0; k < LMAXD; ++k) pi[r][k] = (k < d && g0 + r < n) ? pts[(int64_t)(g0 + r) * d + k] : 0.0;
    double acc[2][PP];
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int c = 0; c < PP; ++c) acc[r][c] = 0.0;
    for (int j0 = 0; j0 < n; j0 += 128) {
        __syncthreads();
        for (int idx = tid; idx < 128 * d; idx += 256) {
            int r = idx / d, k = idx - r * d;
            pcs[k][r] = (j0 + r < n) ? pts[(int64_t)(j0 + r) * d + k] : 0.0;
        }
        for (int idx = tid; idx < 128 * p; idx += 256) {
            int r = idx / p, c = idx - r * p;
            ss[r * SP + c] = (j0 + r < n) ? S[(int64_t)(j0 + r) * lds + c] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int jj = t * 32 + lane;
            const int gj = j0 + jj;
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const int gi = g0 + r;
                if (gi >= n || gj >= n || gj == gi) continue;
                double s2 = 0.0, ud = 0.0;
#pragma unroll
                for (int k = 0; k < LMAXD; ++k)
                    if (k < d) {
                        double u = (pi[r][k] - pcs[k][jj]) * mp.inv_scale[k];
                        s2 += u * u;
                        if (k == mp.ddim) ud = u * u;
                    }
                double val, dval;
                matern_value_drho<MODE>(sqrt(s2), mp, &val, &dval);
                if (mp.ddim >= 0) dval = (s2 > 0.0) ? dval * (ud / s2) * mp.inv_scale[mp.ddim] : 0.0;
#pragma unroll
                for (int c = 0; c < PP; ++c)
                    if (c < p) acc[r][c] += dval * ss[jj * SP + c];
            }
        }
    }
    const int rows128 = ((n + 127) / 128) * 128;
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int c = 0; c < PP; ++c)
            if (c < p) {
                const double v = warp_sum(acc[r][c]);
                if (lane == 0 && g0 + r < rows128) V[(int64_t)(g0 + r) * lds + c] = (g0 + r < n) ? v : 0.0;
            }
}

template <int MODE>
static void launch_dk_apply(const double* pts, int n, int d, const MaternParams& mp, const double* S, int p, int64_t lds,
                            double* V, cudaStream_t s) {
    const unsigned grid = (unsigned)((((n + 127) / 128) * 128) / DKR);
    if (p <= 8) dk_apply_kernel<MODE, 8><<<grid, 256, 0, s>>>(pts, n, d, mp, S, p, lds, V);
    else dk_apply_kernel<MODE, MAXP><<<grid, 256, 0, s>>>(pts, n, d, mp, S, p, lds, V);
}

// ---- Y = K X for a skinny X (n x p): 32 rows per CTA, 4 rows per warp, X tile staged in shared memory ----
__global__ void __launch_bounds__(256)
symm_skinny_kernel(const double* __restrict__ K, int n, int npad, const double* __restrict__ X, int p, double* __restrict__ Y) {
    __shared__ double xs[128 * SSP];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int r0 = blockIdx.x * 32 + warp * 4;
    double acc[4][MAXP];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < MAXP; ++c) acc[r][c] = 0.0;
    for (int j0 = 0; j0 < npad; j0 += 128) {
        __syncthreads();
        for (int idx = tid; idx < 128 * p; idx += 256) {
            int r = idx / p, c = idx - r * p;
            xs[r * SSP + c] = (j0 + r < n) ? X[(int64_t)(j0 + r) * p + c] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            int j = lane + 32 * q;
            double kv[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) kv[r] = K[(int64_t)(r0 + r) * npad + j0 + j];
#pragma unroll
            for (int c = 0; c < MAXP; ++c)
                if (c < p) {
                    double x = xs[j * SSP + c];
#pragma unroll
                    for (int r = 0; r < 4; ++r) acc[r][c] += kv[r] * x;
                }
        }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < MAXP; ++c)
            if (c < p) {
                double v = warp_sum(acc[r][c]);
                if (lane == 0) Y[(int64_t)(r0 + r) * p + c] = (r0 + r < n) ? v : 0.0;
            }
}

// ---- solves through the explicit triangular inverse: S = W^T (W R), W = inv(L) lower ----------------------------
// Y = W X : like symm_skinny_kernel but only columns j <= i are read (32 rows per CTA, 4 rows per warp).
// PP = p padded to 8 or 16 at compile time (4 x 16 accumulators were 170 registers: one CTA per SM); the CTAs take the row
// blocks from the bottom up - the long rows first, the short ones fill the tail.
template <int PP>
__global__ void __launch_bounds__(256)
tril_skinny_kernel(const double* __restrict__ W, int npad, const double* __restrict__ X, int p, double* __restrict__ Y) {
    constexpr int SP = PP + 1;
    __shared__ double xs[128 * SP];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int rb = ((int)gridDim.x - 1 - (int)blockIdx.x) * 32, r0 = rb + warp * 4;
    double acc[4][PP];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < PP; ++c) acc[r][c] = 0.0;
    for (int j0 = 0; j0 < rb + 32; j0 += 128) {
        __syncthreads();
        for (int idx = tid; idx < 128 * p; idx += 256) {
            int r = idx / p, c = idx - r * p;
            xs[r * SP + c] = X[(int64_t)(j0 + r) * p + c];
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            int j = lane + 32 * q;
            double kv[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) kv[r] = (j0 + j <= r0 + r) ? W[(int64_t)(r0 + r) * npad + j0 + j] : 0.0;
#pragma unroll
            for (int c = 0; c < PP; ++c)
                if (c < p) {
                    double x = xs[j * SP + c];
#pragma unroll
                    for (int r = 0; r < 4; ++r) acc[r][c] += kv[r] * x;
                }
        }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < PP; ++c)
            if (c < p) {
                double v = warp_sum(acc[r][c]);
                if (lane == 0) Y[(int64_t)(r0 + r) * p + c] = v;
            }
}

// partial[kc][i][c] = sum_{k in chunk kc, k >= i} W[k][i] X[k][c]; 128 columns i per CTA, 1024-row k chunks
constexpr int TCH = 1024;
template <int PP>
__global__ void __launch_bounds__(256)
trilT_skinny_partial_kernel(const double* __restrict__ W, int npad, const double* __restrict__ X, int p, double* __restrict__ partial) {
    constexpr int SP = PP + 1;
    __shared__ double xs[128 * SP];
    __shared__ double comb[128 * SP];
    const int tid = threadIdx.x;
    const int i0 = blockIdx.x * 128, kc = blockIdx.y;
    const int il = tid & 127, half = tid >> 7, i = i0 + il;
    int kbeg = kc * TCH, kend = min(npad, kbeg + TCH);
    double acc[PP];
#pragma unroll
    for (int c = 0; c < PP; ++c) acc[c] = 0.0;
    if (kend > i0) {   // uniform per CTA
        if (kbeg < i0) kbeg = i0;
        for (int k0 = kbeg; k0 < kend; k0 += 128) {
            __syncthreads();
            for (int idx = tid; idx < 128 * p; idx += 256) {
                int r = idx / p, c = idx - r * p;
                xs[r * SP + c] = X[(int64_t)(k0 + r) * p + c];
            }
            __syncthreads();
#pragma unroll 4
            for (int kk = half; kk < 128; kk += 2) {
                int k = k0 + kk;
                double w = (k >= i) ? W[(int64_t)k * npad + i] : 0.0;
#pragma unroll
                for (int c = 0; c < PP; ++c)
                    if (c < p) acc[c] += w * xs[kk * SP + c];
            }
        }
    }
    __syncthreads();
    if (half == 1)
#pragma unroll
        for (int c = 0; c < PP; ++c) comb[il * SP + c] = acc[c];
    __syncthreads();
    if (half == 0)
        for (int c = 0; c < p; ++c) partial[((int64_t)kc * npad + i) * p + c] = acc[c] + comb[il * SP + c];
}

__global__ void trilT_reduce_kernel(const double* __restrict__ partial, int npad, int p, int nchunks, double* __restrict__ Y) {
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)npad * p) return;
    int i = (int)(t / p);
    double s = 0.0;
    for (int kc = i / TCH; kc < nchunks; ++kc) s += partial[(int64_t)kc * npad * p + t];
    Y[t] = s;
}

__global__ void __launch_bounds__(256)
finalize_out_kernel(double* out, const double* logdet, const double* tr_parts, int ntiles, const double* frob_parts,
                    int nfrob, const int* info, int flags) {
    // one CTA, fixed strided order + fixed tree -> bit-reproducible across runs and rank counts
    __shared__ double red[32];
    double t1 = 0.0, t2 = 0.0, t3 = 0.0;
    if (flags & 2) {
        for (int i = threadIdx.x; i < ntiles; i += 256) {
            t1 += tr_parts[3 * i];
            t2 += tr_parts[3 * i + 1];
            t3 += tr_parts[3 * i + 2];
        }
    } else if (flags & 1) {
        for (int i = threadIdx.x; i < nfrob; i += 256) t1 += frob_parts[i];
    }
    t1 = block_sum(t1, red);
    t2 = block_sum(t2, red);
    t3 = block_sum(t3, red);
    if (threadIdx.x == 0) {
        out[0] = *logdet;
        out[1] = t1;
        out[2] = t2;
        out[3] = t3;
        out[4] = (double)(*info);
        out[5] = out[6] = out[7] = 0.0;      // reserved
    }
}

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

struct LoglikWs {
    double* S;        // npad x p
    double* V;        // npad x p
    double* V2;       // npad x p (Kn^-1 S of the third-moment flag)
    double* logdet;   // 1
    double* gram;     // nparts x p^2
    double* tr;       // ntiles x 3
    double* frob;     // T x T
    int* info;
    double* tpart;    // (npad / 1024 + 1) x npad x MAXP
    void* potri;
    size_t total;
};

static LoglikWs carve(void* ws, int64_t npad, int p) {
    LoglikWs w;
    char* base = (char*)ws;
    size_t off = 0;
    int64_t T = npad / 128;
    auto take = [&](size_t bytes) { size_t o = off; off += align256(bytes); return base ? base + o : (char*)nullptr; };
    w.S = (double*)take(sizeof(double) * npad * MAXP);
    w.V = (double*)take(sizeof(double) * npad * MAXP);
    w.V2 = (double*)take(sizeof(double) * npad * MAXP);
    w.logdet = (double*)take(sizeof(double) * 4);
    w.gram = (double*)take(sizeof(double) * 296 * MAXP * MAXP);
    w.tr = (double*)take(sizeof(double) * (T * (T + 1) / 2) * 3);
    w.frob = (double*)take(sizeof(double) * T * T);
    w.info = (int*)take(sizeof(int) * 4);
    w.tpart = (double*)take(sizeof(double) * (npad / TCH + 1) * npad * MAXP);
    w.potri = (void*)take((size_t)gp_potri_workspace_bytes(npad));
    w.total = off;
    (void)p;
    return w;
}

static int gram(const double* A, const double* B, int nrows, int p, int64_t ld, double* partial, double* out, cudaStream_t s) {
    int parts = 296;
    gram_partial_kernel<<<parts, 256, 0, s>>>(A, B, nrows, p, ld, partial);
    sum_partials_kernel<<<(p * p + 127) / 128, 128, 0, s>>>(partial, parts, p * p, out);
    GP_COUNT(2);
    GP_LAUNCH_CHECK();
    return 0;
}

// S := W^T (W S) in place (S: npad x p), tmp: npad x p
static int solve_with_inverse(const double* W, int npad, double* S, double* tmp, int p, double* tpart, cudaStream_t s) {
    int nchunks = (npad + TCH - 1) / TCH;
    if (p <= 8) {
        tril_skinny_kernel<8><<<npad / 32, 256, 0, s>>>(W, npad, S, p, tmp);
        trilT_skinny_partial_kernel<8><<<dim3(npad / 128, nchunks), 256, 0, s>>>(W, npad, tmp, p, tpart);
    } else {
        tril_skinny_kernel<MAXP><<<npad / 32, 256, 0, s>>>(W, npad, S, p, tmp);
        trilT_skinny_partial_kernel<MAXP><<<dim3(npad / 128, nchunks), 256, 0, s>>>(W, npad, tmp, p, tpart);
    }
    trilT_reduce_kernel<<<(unsigned)(((int64_t)npad * p + 255) / 256), 256, 0, s>>>(tpart, npad, p, nchunks, S);
    GP_COUNT(3);
    GP_LAUNCH_CHECK();
    return 0;
}

template <int MODE>
static int grad_reductions(const double* Ainv, int n, int npad, const double* pts, int d, const MaternParams& mp, bool with_dk,
                           const LoglikWs& w, int p, double* outQ, cudaStream_t s) {
    int T = npad / 128, tiles = T * (T + 1) / 2;
    if (with_dk) {
        trace_tiles_kernel<MODE, true><<<tiles, 256, 0, s>>>(Ainv, n, npad, pts, d, mp, w.tr);
        launch_dk_apply<MODE>(pts, n, d, mp, w.S, p, p, w.V, s);
        GP_COUNT(2);
        GP_LAUNCH_CHECK();
        return gram(w.S, w.V, n, p, p, w.gram, outQ, s);
    }
    trace_tiles_kernel<MODE, false><<<tiles, 256, 0, s>>>(Ainv, n, npad, pts, d, mp, w.tr);
    GP_COUNT(1);
    GP_LAUNCH_CHECK();
    return 0;
}

}  // namespace gp

using namespace gp;

extern "C" {

int gp_symm_skinny(const double* K, int64_t n, int64_t npad, const double* X, int64_t p, double* Y, void* stream) {
    if (!K || !X || !Y || n <= 0 || npad != gp_padded_size(n) || p <= 0 || p > MAXP) return -1;
    symm_skinny_kernel<<<(unsigned)(npad / 32), 256, 0, (cudaStream_t)stream>>>(K, (int)n, (int)npad, X, (int)p, Y);
    GP_COUNT(1);
    GP_LAUNCH_CHECK();
    return 0;
}

// V = dK/drho S with dK regenerated from the points (never stored): the device half of Q = S^T dK S for callers that
// assemble the evaluation themselves (the distributed path, gaussian_proc/_blockcyclic.py)
int gp_dk_apply(const double* points, int64_t n, int64_t d, const double* scale_host, double nu, const double* S, int64_t p,
                int64_t lds, double* V, void* stream) {
    if (!points || !scale_host || !S || !V || n <= 0 || d <= 0 || d > LMAXD || p <= 0 || p > MAXP || lds < p) return -1;
    MaternParams mp;
    int mode;
    if (int rc = matern_params(scale_host, d, nu, true, &mp, &mode)) return rc;
    with_matern_mode(mode, [&](auto tag) {
        launch_dk_apply<decltype(tag)::value>(points, (int)n, (int)d, mp, S, (int)p, lds, V, (cudaStream_t)stream);
    });
    GP_COUNT(1);
    GP_LAUNCH_CHECK();
    return 0;
}

int64_t gp_traces_workspace_bytes(int64_t npad) {
    int64_t T = npad / 128;
    return (int64_t)sizeof(double) * (T * (T + 1) / 2 * 3 + T * T + 64);
}

int gp_inverse_traces(const double* M, int64_t n, int64_t npad, int kind, double* out_dev, void* ws, void* stream) {
    // kind 0: M = inv(L) lower triangular -> out[1] = ||M||_F^2 (= tr Kn^-1);  kind 1: M = Kn^-1 (lower stored)
    // -> out[1] = tr, out[2] = ||.||_F^2 (= tr Kn^-2). out_dev follows the gp_loglik_dense layout (>= 5 doubles).
    if (!M || !out_dev || !ws || n <= 0 || npad != gp_padded_size(n) || (kind != 0 && kind != 1)) return -1;
    cudaStream_t s = (cudaStream_t)stream;
    int T = (int)(npad / 128), tiles = T * (T + 1) / 2;
    double* tr = (double*)ws;
    double* frob = tr + (int64_t)tiles * 3;
    double* misc = frob + (int64_t)T * T;
    GP_CUDA_CHECK(cudaMemsetAsync(misc, 0, sizeof(double) * 8, s));
    MaternParams mp;
    mp.nu = 0; mp.coef = 0; mp.sq2nu = 0; mp.inv_rho = 0;
    if (kind == 0) frob_lower_kernel<<<dim3(T, T), 256, 0, s>>>(M, (int)n, (int)npad, frob);
    else trace_tiles_kernel<MAT_05, false><<<tiles, 256, 0, s>>>(M, (int)n, (int)npad, nullptr, 0, mp, tr);
    finalize_out_kernel<<<1, 256, 0, s>>>(out_dev, misc, tr, tiles, frob, T * T, (const int*)(misc + 2), kind == 0 ? 1 : 2);
    GP_COUNT(2);
    GP_LAUNCH_CHECK();
    return 0;
}

__global__ void sum_trace3_kernel(const double* __restrict__ tr, int tiles, double* out) {
    __shared__ double red[32];
    double s = 0.0;
    for (int i = threadIdx.x; i < tiles; i += blockDim.x) s += tr[(int64_t)i * 3 + 2];
    s = block_sum(s, red);
    if (threadIdx.x == 0) out[0] = s;
}

// Anisotropic gradient: after gp_loglik_dense(flags & 2) on the same (Ainv = A, ws), out_dim[0] = tr(Kn^-1 dK/d scale[dim])
// and out_dim[1 .. p^2] = S^T (dK/d scale[dim]) S, with dK regenerated from the points (reference kernel:
// generate_correlation/_kernels.pyx:107-136, one scale per dimension).
int gp_loglik_dense_dscale(const double* Ainv, int64_t n, int64_t npad, int64_t p, const double* points, int64_t d,
                           const double* scale_host, double nu, int64_t dim, void* ws, double* out_dim, void* stream) {
    if (!Ainv || !points || !scale_host || !ws || !out_dim || n <= 0 || npad != gp_padded_size(n) || p <= 0 || p > MAXP ||
        d <= 0 || d > LMAXD || dim < 0 || dim >= d)
        return -1;
    MaternParams mp;
    int mode;
    if (int rc = matern_params(scale_host, d, nu, false, &mp, &mode)) return rc;
    mp.inv_rho = 1.0;
    mp.ddim = (int)dim;
    cudaStream_t s = (cudaStream_t)stream;
    LoglikWs w = carve(ws, npad, (int)p);
    const int NP = (int)npad;
    int rc = with_matern_mode(mode, [&](auto tag) {
        return grad_reductions<decltype(tag)::value>(Ainv, (int)n, NP, points, (int)d, mp, true, w, (int)p, out_dim + 1, s);
    });
    if (rc) return rc;
    int T = NP / 128;
    sum_trace3_kernel<<<1, 256, 0, s>>>(w.tr, T * (T + 1) / 2, out_dim);
    GP_COUNT(1);
    GP_LAUNCH_CHECK();
    return 0;
}

int64_t gp_loglik_workspace_bytes(int64_t npad) { return (int64_t)carve(nullptr, npad, MAXP).total; }

int64_t gp_loglik_out_len(int64_t p) { return 8 + 4 * p * p; }

int gp_loglik_dense(const double* K, int64_t n, int64_t npad, const double* R, int64_t p, double eta, int flags,
                    const double* points, int64_t d, const double* scale_host, double nu, double* A, double* W,
                    void* potrf_ws, void* ws, double* out, void* stream) {
    if (!K || !R || !A || !potrf_ws || !ws || !out || n <= 0 || npad != gp_padded_size(n) || p <= 0 || p > MAXP) return -1;
    if ((flags & 3) && !W) return -2;
    if ((flags & 4) && (!(flags & 2) || !points || !scale_host || d <= 0 || d > LMAXD)) return -8;
    if ((flags & 8) && !(flags & 3)) return -9;
    const bool with_dk = (flags & 4) != 0;
    MaternParams mp{};     // without flag 4 the reductions do not read it
    int mode = MAT_05;
    if (with_dk)
        if (int rc = matern_params(scale_host, d, nu, true, &mp, &mode)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    LoglikWs w = carve(ws, npad, (int)p);
    const int N = (int)n, NP = (int)npad, P = (int)p;
    int rc;
    if ((rc = gp_shift_copy(K, n, npad, eta, A, stream))) return rc;
    if ((rc = gp_potrf_f64(A, n, npad, w.info, potrf_ws, stream))) return rc;
    if ((rc = gp_logdet_from_chol(A, n, npad, w.logdet, stream))) return rc;
    GP_CUDA_CHECK(cudaMemcpyAsync(w.S, R, sizeof(double) * npad * p, cudaMemcpyDeviceToDevice, s));
    int T = NP / 128;
    if (flags & 3) {
        // the triangular inverse is needed anyway: solve through it (two skinny triangular products) instead of
        // the latency-bound block substitution
        if ((rc = gp_trtri_f64(A, W, npad, potrf_ws, w.potri, stream))) return rc;
        if ((rc = solve_with_inverse(W, NP, w.S, w.V, P, w.tpart, s))) return rc;
    } else {
        if ((rc = gp_potrs_f64(A, npad, potrf_ws, w.S, p, p, stream))) return rc;
    }
    double* G = out + 8;
    double* H = G + p * p;
    double* Q = H + p * p;
    if ((rc = gram(R, w.S, N, P, p, w.gram, G, s))) return rc;
    if ((rc = gram(w.S, w.S, N, P, p, w.gram, H, s))) return rc;
    double* T3 = Q + p * p;
    GP_CUDA_CHECK(cudaMemsetAsync(Q, 0, sizeof(double) * 2 * p * p, s));
    if (flags & 8) {
        // third moments (Hessian, second eta-derivative): T3 = S^T Kn^-1 S = R^T Kn^-3 R from one more skinny solve batch
        GP_CUDA_CHECK(cudaMemcpyAsync(w.V2, w.S, sizeof(double) * npad * p, cudaMemcpyDeviceToDevice, s));
        if ((rc = solve_with_inverse(W, NP, w.V2, w.V, P, w.tpart, s))) return rc;
        if ((rc = gram(w.S, w.V2, N, P, p, w.gram, T3, s))) return rc;
    }
    if (flags & 2) {
        if ((rc = gp_lauum_f64(W, A, npad, stream))) return rc;
        rc = with_matern_mode(mode, [&](auto tag) {
            return grad_reductions<decltype(tag)::value>(A, N, NP, points, (int)d, mp, with_dk, w, P, Q, s);
        });
        if (rc) return rc;
    } else if (flags & 1) {
        frob_lower_kernel<<<dim3(T, T), 256, 0, s>>>(W, N, NP, w.frob);
        GP_COUNT(1);
        GP_LAUNCH_CHECK();
    }
    finalize_out_kernel<<<1, 256, 0, s>>>(out, w.logdet, w.tr, T * (T + 1) / 2, w.frob, T * T, w.info, flags);
    GP_COUNT(1);
    GP_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
