// Blocked FP64 Cholesky, triangular solves, inverse and log-determinant on the padded matrix K + eta*I.
// Replaces what the reference obtains from scipy.linalg.solve(assume_a='pos') (LAPACK dposv, one fresh O(n^3)
// factorisation per call: gaussian_proc/_mixed_correlation/mixed_correlation.py:280-299, _linear_solver.py:71)
// and from imate's 'cholesky' logdet / traceinv (mixed_correlation.py:183-191,250-261).
//
// potrf : right-looking, two-level blocking (outer panel 512, inner 128). The 128x128 diagonal block is factored
//         AND inverted by one CTA in shared memory; the panel solve is a GEMM with that inverse and all trailing
//         updates are DMMA GEMMs (gp_gemm.cu), lower tiles only.
// potrs : block forward/back substitution that reuses the inverted diagonal blocks.
// potri : W = inv(L) by recursive halving (two triangular GEMMs per level), then inv(A) = W^T W (one TN GEMM).
#include "../../include/gpgp.h"
#include "gp_common.cuh"
#include "gp_internal.h"
#include <map>
#include <mutex>
#include <utility>
#include <vector>

namespace gp {

constexpr int DB = 128;         // diagonal block
constexpr int DPITCH = DB + 1;  // shared pitch (odd -> conflict-free column walks)
constexpr int DIAG_THREADS = 256;  // 255 registers per thread: the unrolled warp-level factorisation must not spill
constexpr int OUTER_NB = 512;  // outer panel width (multiple of 128)

// Factor the 128x128 diagonal block at `Ajj` (lower, in place) and write inv(L_jj) (lower, zero above) to `Linv`.
//
// Shared array S[128][129]: the lower triangle holds A / L; W = inv(L) is kept transposed in the strict upper
// triangle (W[i][c], c <= i, lives at S[c][i+1]) so that one 132 KB array serves both. Algorithm, 32-wide sub-blocks:
//   for each block column J: (1) warp 0 factors the 32x32 diagonal sub-block in registers (lane = row) with
//   warp shuffles, (2) one thread per row below solves its 32 unknowns against that sub-block (axpy form, the
//   L_D entries are shared-memory broadcasts), (3) all threads apply the rank-32 update to the trailing part with
//   4x4 register micro-tiles.  Then inv(L): (4) four warps invert the four diagonal sub-blocks, (5) the
//   off-diagonal blocks follow by block distance d = 1, 2, 3:  W_IJ = -inv(L_II) * sum_K L_IK W_KJ.
constexpr int SB = 32;
constexpr int TPITCH = SB + 1;

#ifdef GP_DIAG_TIMING
__device__ long long g_diag_clk[32];
#define DIAG_T(i) do { if (tid == 0) g_diag_clk[i] = clock64(); } while (0)
#else
#define DIAG_T(i)
#endif


// Warp-level Cholesky of a 32x32 block (lane = row, a[] = this lane's row, a[0] = current column).
// The column loop stays ROLLED and the register array is rotated by one each step so that every register index is
// static: a single warp running ~3000 straight-line instructions is instruction-fetch bound (measured 1100 cycles per
// column fully unrolled vs ~250 rolled). Column j is broadcast through `cb` with all loads issued before the FMAs.
__device__ __forceinline__ int chol32_warp(double (&a)[SB], int lane, double* cb, double* dinv_out, double* Srow) {
    int badcol = -1;
#pragma unroll 1
    for (int j = 0; j < SB; ++j) {
        double ajj = __shfl_sync(0xffffffffu, a[0], j);
        if (!(ajj > 0.0) && badcol < 0) badcol = j;   // also catches NaN
        double inv = rsqrt(ajj);
        double lj = (lane == j) ? ajj * inv : a[0] * inv;   // l_ij for lanes i >= j
        if (lane >= j) Srow[j] = lj;
        if (lane == j) dinv_out[j] = inv;
        double* c = cb + (j & 1) * 2 * SB;
        c[lane] = lj;
        __syncwarp();
        double t[SB - 1];
#pragma unroll
        for (int k = 0; k < SB - 1; ++k) t[k] = c[j + 1 + k];          // entries past 31 are never used by a valid lane
#pragma unroll
        for (int k = 0; k < SB - 1; ++k) a[k] = a[k + 1] - lj * t[k];  // update + rotate: new a[0] is column j + 1
    }
    return badcol;
}

__global__ void __launch_bounds__(DIAG_THREADS, 1)
chol_diag_block_kernel(double* Ajj, int64_t lda, double* Linv, int* info, int j0, int nvalid) {
    extern __shared__ double S[];                  // [128][129]
    double* dinv = S + DB * DPITCH;                // [128]   1 / L_ii
    double* T = dinv + DB;                         // [3][32][33] scratch for the inverse assembly
    double* colbuf = T;                            // [2][32] column broadcast buffer of the warp-level factorisation
    __shared__ int bad;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) bad = 0;
    DIAG_T(0);
    // 8 independent loads per thread in flight (the block usually sits in L2: latency, not bandwidth, matters)
    for (int base = 0; base < DB * DB; base += 8 * DIAG_THREADS) {
        double v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            int idx = base + u * DIAG_THREADS + tid, i = idx >> 7, k = idx & 127;
            v[u] = (k <= i) ? Ajj[(int64_t)i * lda + k] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            int idx = base + u * DIAG_THREADS + tid, i = idx >> 7, k = idx & 127;
            S[i * DPITCH + k] = v[u];
        }
    }
    if (tid < DB) S[tid * DPITCH + DB] = 0.0;
    __syncthreads();

    DIAG_T(1);
    for (int J = 0; J < DB / SB; ++J) {
        const int J0 = J * SB;
        DIAG_T(2 + 4 * J);
        // ---- (1) 32x32 diagonal sub-block: lane = row, registers hold the row, columns broadcast by shuffle
        if (warp == 0) {
            double a[SB];
            const int row = J0 + lane;
#pragma unroll
            for (int k = 0; k < SB; ++k) a[k] = S[row * DPITCH + J0 + k];
            int badcol = chol32_warp(a, lane, colbuf, dinv + J0, S + row * DPITCH + J0);
            if (lane == 0 && badcol >= 0 && !bad) {
                bad = 1;
                if (j0 + J0 + badcol < nvalid) atomicCAS(info, 0, j0 + J0 + badcol + 1);
            }
        }
        __syncthreads();
        DIAG_T(3 + 4 * J);
        const int r = DB - J0 - SB;   // rows below the sub-block
        if (r == 0) break;
        // ---- (2) panel solve, one thread per row: x = p * inv(L_D)^T in axpy form
        if (tid < r) {
            const int i = J0 + SB + tid;
            double pr[SB];
#pragma unroll
            for (int c = 0; c < SB; ++c) pr[c] = S[i * DPITCH + J0 + c];
#pragma unroll
            for (int c = 0; c < SB; ++c) {
                double x = pr[c] * dinv[J0 + c];
                pr[c] = x;
#pragma unroll
                for (int k = c + 1; k < SB; ++k) pr[k] -= x * S[(J0 + k) * DPITCH + J0 + c];
            }
#pragma unroll
            for (int c = 0; c < SB; ++c) S[i * DPITCH + J0 + c] = pr[c];
        }
        __syncthreads();
        DIAG_T(4 + 4 * J);
        // ---- (3) trailing rank-32 update on lower 8x4 register micro-tiles (tile row mi holds 2 mi + 2 tiles)
        {
            const int mr = r / 8, cnt = mr * (mr + 1);
            if (tid < cnt) {
                int mi = (int)((sqrtf(4.0f * tid + 1.0f) - 1.0f) * 0.5f);
                while ((mi + 1) * (mi + 2) <= tid) ++mi;
                while (mi * (mi + 1) > tid) --mi;
                const int mk = tid - mi * (mi + 1);
                const int i0 = J0 + SB + 8 * mi, k0 = J0 + SB + 4 * mk;
                double acc[8][4];
#pragma unroll
                for (int e = 0; e < 8; ++e)
#pragma unroll
                    for (int f = 0; f < 4; ++f) acc[e][f] = 0.0;
#pragma unroll 4
                for (int c = 0; c < SB; ++c) {
                    double av[8], bv[4];
#pragma unroll
                    for (int e = 0; e < 8; ++e) av[e] = S[(i0 + e) * DPITCH + J0 + c];
#pragma unroll
                    for (int f = 0; f < 4; ++f) bv[f] = S[(k0 + f) * DPITCH + J0 + c];
#pragma unroll
                    for (int e = 0; e < 8; ++e)
#pragma unroll
                        for (int f = 0; f < 4; ++f) acc[e][f] += av[e] * bv[f];
                }
#pragma unroll
                for (int e = 0; e < 8; ++e)
#pragma unroll
                    for (int f = 0; f < 4; ++f)
                        if (k0 + f <= i0 + e) S[(i0 + e) * DPITCH + k0 + f] -= acc[e][f];
            }
        }
        __syncthreads();
    }

    DIAG_T(18);
    // ---- (4) inverses of the four diagonal sub-blocks: warp J, lane = column c of inv(L_JJ)
    if (warp < DB / SB) {
        const int J0 = warp * SB;
        double acc[SB];
#pragma unroll
        for (int i = 0; i < SB; ++i) acc[i] = (i == lane) ? 1.0 : 0.0;
#pragma unroll
        for (int k = 0; k < SB; ++k) {
            double w = acc[k] * dinv[J0 + k];
            acc[k] = w;
#pragma unroll
            for (int i = k + 1; i < SB; ++i) acc[i] -= S[(J0 + i) * DPITCH + J0 + k] * w;
        }
#pragma unroll
        for (int i = 0; i < SB; ++i)
            if (i >= lane) S[(J0 + lane) * DPITCH + J0 + i + 1] = acc[i];   // W[J0+i][J0+lane]
    }
    __syncthreads();
    DIAG_T(19);
    // ---- (5) off-diagonal blocks of W by block distance
    for (int d = 1; d < DB / SB; ++d) {
        const int nblk = DB / SB - d;
        const int i0 = 2 * (tid >> 4), c0 = 2 * (tid & 15);   // 256 threads x (2 x 2) = one 32 x 32 block
        // T_b = sum_K L_IK W_KJ over g in [32 J, 32 I): W[g][col] lives at S[col][g + 1] and is zero for g < col
        // (those slots of the shared array hold L, hence the explicit mask)
        for (int b = 0; b < nblk; ++b) {
            const int Jb = b, Ib = b + d;
            const double* l0p = S + (Ib * SB + i0) * DPITCH;
            const double* l1p = l0p + DPITCH;
            const int col0 = Jb * SB + c0;
            const double* w0p = S + col0 * DPITCH + 1;
            const double* w1p = w0p + DPITCH;
            double a00 = 0.0, a01 = 0.0, a10 = 0.0, a11 = 0.0;
#pragma unroll 4
            for (int g = Jb * SB; g < Ib * SB; ++g) {
                double l0 = l0p[g], l1 = l1p[g];
                double w0 = (g >= col0) ? w0p[g] : 0.0;
                double w1 = (g >= col0 + 1) ? w1p[g] : 0.0;
                a00 += l0 * w0; a01 += l0 * w1; a10 += l1 * w0; a11 += l1 * w1;
            }
            double* tp = T + (b * SB + i0) * TPITCH + c0;
            tp[0] = a00; tp[1] = a01; tp[TPITCH] = a10; tp[TPITCH + 1] = a11;
        }
        __syncthreads();
        // W_IJ[i][c] = - sum_{k <= i} inv(L_II)[i][k] T[k][c];  inv(L_II)[i][k] lives at S[32 I + k][32 I + i + 1]
        for (int b = 0; b < nblk; ++b) {
            const int Jb = b, Ib = b + d;
            const double* dp = S + (Ib * SB) * DPITCH + Ib * SB + i0 + 1;
            const double* tp = T + (b * SB) * TPITCH + c0;
            double a00 = 0.0, a01 = 0.0, a10 = 0.0, a11 = 0.0;
#pragma unroll 4
            for (int k = 0; k <= i0 + 1; ++k) {
                double d0 = (k <= i0) ? dp[k * DPITCH] : 0.0, d1 = dp[k * DPITCH + 1];
                double t0 = tp[k * TPITCH], t1 = tp[k * TPITCH + 1];
                a00 += d0 * t0; a01 += d0 * t1; a10 += d1 * t0; a11 += d1 * t1;
            }
            double* wp = S + (Jb * SB + c0) * DPITCH + Ib * SB + i0 + 1;
            wp[0] = -a00; wp[1] = -a10; wp[DPITCH] = -a01; wp[DPITCH + 1] = -a11;
        }
        __syncthreads();
    }

    DIAG_T(20);
    for (int idx = tid; idx < DB * DB; idx += DIAG_THREADS) {
        int i = idx >> 7, k = idx & 127;
        if (k <= i) {
            Ajj[(int64_t)i * lda + k] = S[i * DPITCH + k];
            Linv[i * DB + k] = S[k * DPITCH + i + 1];
        } else {
            Linv[i * DB + k] = 0.0;
        }
    }
    DIAG_T(21);
}

__global__ void logdet_kernel(const double* L, int n, int64_t ld, double* out) {
    __shared__ double red[32];
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) s += log(L[(int64_t)i * ld + i]);
    s = block_sum(s, red);
    if (threadIdx.x == 0) *out = 2.0 * s;
}

__global__ void shift_copy_kernel(const double* __restrict__ K, int n, int npad, double eta, double* __restrict__ A) {
    // lower tiles only (the factorisation never references the strict upper triangle)
    int tm = blockIdx.y, tn = blockIdx.x;
    if (tn > tm) return;
    int r0 = tm * 128, c0 = tn * 128;
    for (int idx = threadIdx.x; idx < 128 * 64; idx += blockDim.x) {
        int r = idx >> 6, c2 = (idx & 63) * 2;
        int64_t o = (int64_t)(r0 + r) * npad + c0 + c2;
        double2 v = *reinterpret_cast<const double2*>(K + o);
        int gi = r0 + r, gj = c0 + c2;
        if (gi < n) {
            if (gi == gj) v.x += eta;
            if (gi == gj + 1) v.y += eta;
        }
        *reinterpret_cast<double2*>(A + o) = v;
    }
}

// ---- substitution kernels -------------------------------------------------------------------------------

constexpr int MAX_RHS = 16;

// y = op(Linv_j) * b_j for one 128-row block (in place in B). TRANS: use Linv^T.
// Linv is row-major [i][k]: the plain product walks rows with a warp (coalesced), the transposed one assigns a
// thread per output row so that consecutive threads read consecutive columns.
template <bool TRANS>
__global__ void __launch_bounds__(256)
diag_apply_kernel(const double* __restrict__ Linv, double* Bj, int nrhs, int64_t ldb) {
    __shared__ double bs[DB * MAX_RHS];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int idx = tid; idx < DB * nrhs; idx += 256) bs[idx] = Bj[(int64_t)(idx / nrhs) * ldb + idx % nrhs];
    __syncthreads();
    if (!TRANS) {
        for (int i = warp; i < DB; i += 8) {
            double l[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) { int k = lane + 32 * q; l[q] = (k <= i) ? Linv[i * DB + k] : 0.0; }
            for (int c = 0; c < nrhs; ++c) {
                double s = 0.0;
#pragma unroll
                for (int q = 0; q < 4; ++q) s += l[q] * bs[(lane + 32 * q) * nrhs + c];
                s = warp_sum(s);
                if (lane == 0) Bj[(int64_t)i * ldb + c] = s;
            }
        }
    } else {
        // two threads per output row split the k range
        int i = tid & 127, half = tid >> 7;
        __shared__ double part[DB * MAX_RHS];
        int kb = half ? (i + DB) / 2 + 1 : i, ke = half ? DB : (i + DB) / 2 + 1;
        for (int c = 0; c < nrhs; ++c) {
            double s = 0.0;
            for (int k = kb; k < ke; ++k) s += Linv[k * DB + i] * bs[k * nrhs + c];
            if (half) part[i * nrhs + c] = s;
            __syncthreads();
            if (!half) Bj[(int64_t)i * ldb + c] = s + part[i * nrhs + c];
            __syncthreads();
        }
    }
}

// forward: B[r] -= L[r, j:j+128] * Y_j   for rows r in [row0, npad); one warp per row, 8 rows per CTA
template <int NR>
__global__ void __launch_bounds__(256)
fwd_update_kernel(const double* __restrict__ L, int64_t ldl, int row0, int j0, const double* Yj, double* B, int64_t ldb,
                  int nrows, int nrhs) {
    __shared__ double ys[DB * NR];
    for (int idx = threadIdx.x; idx < DB * NR; idx += 256) {
        int k = idx / NR, c = idx - k * NR;
        ys[idx] = (c < nrhs) ? Yj[(int64_t)k * ldb + c] : 0.0;
    }
    __syncthreads();
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int r = blockIdx.x * 8 + warp; r < nrows; r += gridDim.x * 8) {
        const double* lrow = L + (int64_t)(row0 + r) * ldl + j0;
        double acc[NR];
#pragma unroll
        for (int c = 0; c < NR; ++c) acc[c] = 0.0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            int k = lane + 32 * q;
            double l = lrow[k];
#pragma unroll
            for (int c = 0; c < NR; ++c) acc[c] += l * ys[k * NR + c];
        }
#pragma unroll
        for (int c = 0; c < NR; ++c) acc[c] = warp_sum(acc[c]);
        if (lane == 0) {
            double* b = B + (int64_t)(row0 + r) * ldb;
            for (int c = 0; c < nrhs; ++c) b[c] -= acc[c];
        }
    }
}

// backward: Y[c] -= sum_r L[j0 + r][c] * Z_j[r]   for c in [0, j0); thread per column c
template <int NR>
__global__ void __launch_bounds__(256)
bwd_update_kernel(const double* __restrict__ L, int64_t ldl, int j0, const double* Zj, double* Y, int64_t ldb, int nrhs) {
    __shared__ double zs[DB * NR];
    for (int idx = threadIdx.x; idx < DB * NR; idx += 256) {
        int k = idx / NR, c = idx - k * NR;
        zs[idx] = (c < nrhs) ? Zj[(int64_t)k * ldb + c] : 0.0;
    }
    __syncthreads();
    int c = blockIdx.x * 256 + threadIdx.x;
    if (c >= j0) return;
    double acc[NR];
#pragma unroll
    for (int q = 0; q < NR; ++q) acc[q] = 0.0;
    const double* lp = L + (int64_t)j0 * ldl + c;
#pragma unroll 4
    for (int r = 0; r < DB; ++r) {
        double l = lp[(int64_t)r * ldl];
#pragma unroll
        for (int q = 0; q < NR; ++q) acc[q] += l * zs[r * NR + q];
    }
    double* y = Y + (int64_t)c * ldb;
    for (int q = 0; q < nrhs; ++q) y[q] -= acc[q];
}

__global__ void place_diag_inverse_kernel(const double* __restrict__ Linv, double* W, int64_t ldw) {
    int b = blockIdx.x;
    const double* src = Linv + (int64_t)b * DB * DB;
    double* dst = W + (int64_t)b * DB * ldw + b * DB;
    for (int idx = threadIdx.x; idx < DB * DB; idx += blockDim.x) dst[(int64_t)(idx >> 7) * ldw + (idx & 127)] = src[idx];
}

// ---- helper streams (one process drives one GPU): independent sub-problems of the recursive inverse and the
// look-ahead panel of the factorisation run beside the caller's stream, ordered with events ---------------------
struct SidePool {
    cudaStream_t s[3];
    // ordering events of this pool, reused round-robin: an event is re-recorded only after EVENT_RING later orderings
    // have been enqueued on the same caller stream, by which time the earlier wait has long been submitted (a
    // cudaStreamWaitEvent captures the event's state at submission, so re-recording afterwards is safe)
    std::vector<cudaEvent_t> events;
    size_t next = 0;
};
constexpr size_t EVENT_RING = 64;
// one pool per (device, caller stream): two evaluations driven on two streams (a sweep keeps two cells in flight to fill
// the latency-bound phases of each other) must not serialise on shared helper streams, and a second device in the same
// process gets its own streams. The map is guarded by a mutex; a pool itself is only used by the host thread that drives
// its caller stream.
static std::mutex g_pools_mutex;
static std::map<std::pair<int, cudaStream_t>, SidePool*> g_pools;
static thread_local SidePool* g_side_ptr = nullptr;
#define g_side (*g_side_ptr)

static int side_streams_init(cudaStream_t caller) {
    int dev = 0;
    GP_CUDA_CHECK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_pools_mutex);
    auto key = std::make_pair(dev, caller);
    auto it = g_pools.find(key);
    if (it == g_pools.end()) {
        int lo = 0, hi = 0;
        GP_CUDA_CHECK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        SidePool* p = new SidePool();
        for (int i = 0; i < 3; ++i) GP_CUDA_CHECK(cudaStreamCreateWithPriority(&p->s[i], cudaStreamNonBlocking, hi));
        p->events.resize(EVENT_RING);
        for (size_t i = 0; i < EVENT_RING; ++i) GP_CUDA_CHECK(cudaEventCreateWithFlags(&p->events[i], cudaEventDisableTiming));
        it = g_pools.insert(std::make_pair(key, p)).first;
    }
    g_side_ptr = it->second;
    return 0;
}

// make `to` wait for everything enqueued on `from` so far (event from the pool's ring: no create / destroy per call)
static int stream_order(cudaStream_t from, cudaStream_t to) {
    cudaEvent_t e = g_side.events[g_side.next];
    g_side.next = (g_side.next + 1) % EVENT_RING;
    GP_CUDA_CHECK(cudaEventRecord(e, from));
    GP_CUDA_CHECK(cudaStreamWaitEvent(to, e, 0));
    return 0;
}

static int64_t trtri_need(int nb) { return (int64_t)(nb / 2) * (nb - nb / 2) * DB * DB; }

// recursive inverse of the lower-triangular L over block range [lo, hi) (units of 128); T = scratch of
// trtri_need(hi - lo) doubles. The two halves are independent: down to depth 2 the right half runs on a side stream.
static int trtri_rec(const double* L, double* W, int64_t ld, int lo, int hi, double* T, cudaStream_t s, int depth, int slot) {
    if (hi - lo <= 1) return 0;
    int mid = lo + (hi - lo) / 2;  // first half has floor((hi-lo)/2) blocks
    int rc;
    bool fork = depth < 2 && (hi - lo) >= 8;
    double* Tr = T + trtri_need(mid - lo);
    if (fork) {
        cudaStream_t side = g_side.s[slot];
        if ((rc = stream_order(s, side))) return rc;
        if ((rc = trtri_rec(L, W, ld, mid, hi, Tr, side, depth + 1, slot == 0 ? 2 : slot))) return rc;
        if ((rc = trtri_rec(L, W, ld, lo, mid, T, s, depth + 1, 1))) return rc;
        if ((rc = stream_order(side, s))) return rc;
    } else {
        if ((rc = trtri_rec(L, W, ld, lo, mid, T, s, 2, slot))) return rc;
        if ((rc = trtri_rec(L, W, ld, mid, hi, Tr, s, 2, slot))) return rc;
    }
    int M = (hi - mid) * DB, N = (mid - lo) * DB;
    // T (M x N) = L21 * W11      (W11 lower: k >= n0)
    rc = launch_dgemm(0, 1, T, N, L + (int64_t)mid * DB * ld + (int64_t)lo * DB, ld,
                      W + (int64_t)lo * DB * ld + (int64_t)lo * DB, ld, M, N, N, 1.0, 0.0, KR_B_LOWER, TM_ALL, s);
    if (rc) return rc;
    // W21 = -W22 * T             (W22 lower: k < m0 + 128)
    rc = launch_dgemm(0, 1, W + (int64_t)mid * DB * ld + (int64_t)lo * DB, ld,
                      W + (int64_t)mid * DB * ld + (int64_t)mid * DB, ld, T, N, M, N, M, -1.0, 0.0, KR_A_LOWER, TM_ALL, s);
    return rc;
}

template <int NR>
static void launch_fwd(const double* L, int64_t npad, int row0, int j0, const double* Yj, double* B, int64_t ldb, int nrows,
                       int nrhs, cudaStream_t s) {
    int grid = (nrows + 7) / 8;
    if (grid > 148 * 8) grid = 148 * 8;
    fwd_update_kernel<NR><<<grid, 256, 0, s>>>(L, npad, row0, j0, Yj, B, ldb, nrows, nrhs);
}
template <int NR>
static void launch_bwd(const double* L, int64_t npad, int j0, const double* Zj, double* Y, int64_t ldb, int nrhs, cudaStream_t s) {
    bwd_update_kernel<NR><<<(j0 + 255) / 256, 256, 0, s>>>(L, npad, j0, Zj, Y, ldb, nrhs);
}

}  // namespace gp

using namespace gp;

extern "C" {

#ifdef GP_DIAG_TIMING
int gp_diag_timing_read(long long* out32) {
    return (int)cudaMemcpyFromSymbol(out32, gp::g_diag_clk, sizeof(long long) * 32);
}
#endif

int gp_shift_copy(const double* K, int64_t n, int64_t npad, double eta, double* A, void* stream) {
    if (!K || !A || n <= 0 || npad != gp_padded_size(n)) return -1;
    dim3 grid((unsigned)(npad / 128), (unsigned)(npad / 128));
    shift_copy_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(K, (int)n, (int)npad, eta, A);
    GP_COUNT(1);
    GP_LAUNCH_CHECK();
    return 0;
}

int64_t gp_potrf_workspace_bytes(int64_t npad) { return (npad / DB) * (int64_t)DB * DB * sizeof(double); }

// factor one outer panel [J, Jend): diagonal blocks, panel solves and the updates that stay inside the panel
static int factor_panel(double* A, int64_t npad, int n, int J, int Jend, double* linv, int* info_dev, int diag_smem,
                        cudaStream_t s) {
    const int N = (int)npad;
    for (int j = J; j < Jend; j += DB) {
        double* Ajj = A + (int64_t)j * npad + j;
        double* Lj = linv + (int64_t)(j / DB) * DB * DB;
        chol_diag_block_kernel<<<1, DIAG_THREADS, diag_smem, s>>>(Ajj, npad, Lj, info_dev, j, n);
        GP_COUNT(1);
        GP_LAUNCH_CHECK();
        int below = N - (j + DB);
        if (below <= 0) continue;
        double* A21 = A + (int64_t)(j + DB) * npad + j;
        // panel solve L21 = A21 * inv(L_jj)^T  (in place: each CTA reads exactly the tile it overwrites)
        int rc = launch_dgemm(0, 0, A21, npad, A21, npad, Lj, DB, below, DB, DB, 1.0, 0.0, KR_FULL, TM_ALL, s);
        if (rc) return rc;
        int ncols = Jend - (j + DB);
        if (ncols > 0) {
            rc = launch_dgemm(0, 0, A + (int64_t)(j + DB) * npad + (j + DB), npad, A21, npad, A21, npad, below, ncols, DB,
                              -1.0, 1.0, KR_FULL, TM_LOWER, s);
            if (rc) return rc;
        }
    }
    return 0;
}

int gp_potrf_f64(double* A, int64_t n, int64_t npad, int* info_dev, void* ws, void* stream) {
    if (!A || !info_dev || !ws || npad <= 0 || (npad % DB) || npad > INT32_MAX || n > npad) return -1;
    cudaStream_t s = (cudaStream_t)stream;
    double* linv = (double*)ws;
    const int diag_smem = (DB * DPITCH + DB + 3 * SB * TPITCH) * sizeof(double);
    if (int rc0 = configure_once((const void*)chol_diag_block_kernel, diag_smem)) return rc0;
    int rc = side_streams_init(s);
    if (rc) return rc;
    cudaStream_t ps = g_side.s[0];  // high-priority panel stream (look-ahead)
    GP_CUDA_CHECK(cudaMemsetAsync(info_dev, 0, sizeof(int), s));
    const int N = (int)npad;
    // Right-looking with look-ahead 1: after panel J, the trailing update is split into (i) the block column of the
    // next panel and (ii) the rest; panel J+1 is factored on the panel stream while (ii) still runs on `s`.
    if ((rc = factor_panel(A, npad, (int)n, 0, OUTER_NB < N ? OUTER_NB : N, linv, info_dev, diag_smem, s))) return rc;
    for (int J = 0; J < N; J += OUTER_NB) {
        int Jend = (J + OUTER_NB < N) ? J + OUTER_NB : N;
        int rows = N - Jend;
        if (rows <= 0) break;
        int K = Jend - J;
        int nextw = (OUTER_NB < rows) ? OUTER_NB : rows;           // width of panel J+1
        const double* P = A + (int64_t)Jend * npad + J;              // L[Jend:, J:Jend]
        // (i) block column of the next panel: rows x nextw, lower-masked
        rc = launch_dgemm(0, 0, A + (int64_t)Jend * npad + Jend, npad, P, npad, P, npad, rows, nextw, K, -1.0, 1.0, KR_FULL,
                          TM_LOWER, s);
        if (rc) return rc;
        int rest = rows - nextw;
        if (rest > 0) {
            if ((rc = stream_order(s, ps))) return rc;
            if ((rc = factor_panel(A, npad, (int)n, Jend, Jend + nextw, linv, info_dev, diag_smem, ps))) return rc;
            // (ii) the remaining trailing matrix
            const double* P2 = A + (int64_t)(Jend + nextw) * npad + J;
            rc = launch_dgemm(0, 0, A + (int64_t)(Jend + nextw) * npad + (Jend + nextw), npad, P2, npad, P2, npad, rest, rest,
                              K, -1.0, 1.0, KR_FULL, TM_LOWER, s);
            if (rc) return rc;
            if ((rc = stream_order(ps, s))) return rc;
        } else {
            if ((rc = factor_panel(A, npad, (int)n, Jend, Jend + nextw, linv, info_dev, diag_smem, s))) return rc;
        }
    }
    return 0;
}

int gp_logdet_from_chol(const double* L, int64_t n, int64_t npad, double* out_dev, void* stream) {
    if (!L || !out_dev || n <= 0 || n > npad) return -1;
    logdet_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(L, (int)n, npad, out_dev);
    GP_COUNT(1);
    GP_LAUNCH_CHECK();
    return 0;
}

int gp_potrs_f64(const double* L, int64_t npad, const void* potrf_ws, double* B, int64_t nrhs, int64_t ldb, void* stream) {
    if (!L || !potrf_ws || !B || nrhs <= 0 || nrhs > MAX_RHS || ldb < nrhs || (npad % DB)) return -1;
    cudaStream_t s = (cudaStream_t)stream;
    const double* linv = (const double*)potrf_ws;
    const int N = (int)npad, nb = N / DB, nr = (int)nrhs;
    for (int b = 0; b < nb; ++b) {
        int j = b * DB;
        double* Bj = B + (int64_t)j * ldb;
        diag_apply_kernel<false><<<1, 256, 0, s>>>(linv + (int64_t)b * DB * DB, Bj, nr, ldb);
        int below = N - (j + DB);
        GP_COUNT(below > 0 ? 2 : 1);
        if (below > 0) {
            if (nr <= 8) launch_fwd<8>(L, npad, j + DB, j, Bj, B, ldb, below, nr, s);
            else launch_fwd<16>(L, npad, j + DB, j, Bj, B, ldb, below, nr, s);
        }
    }
    for (int b = nb - 1; b >= 0; --b) {
        int j = b * DB;
        double* Bj = B + (int64_t)j * ldb;
        diag_apply_kernel<true><<<1, 256, 0, s>>>(linv + (int64_t)b * DB * DB, Bj, nr, ldb);
        GP_COUNT(j > 0 ? 2 : 1);
        if (j > 0) {
            if (nr <= 8) launch_bwd<8>(L, npad, j, Bj, B, ldb, nr, s);
            else launch_bwd<16>(L, npad, j, Bj, B, ldb, nr, s);
        }
    }
    GP_LAUNCH_CHECK();
    return 0;
}

int64_t gp_potri_workspace_bytes(int64_t npad) {
    int64_t nb = npad / DB, h1 = nb / 2, h2 = nb - h1;
    return h1 * h2 * (int64_t)DB * DB * sizeof(double) + 256;
}

int gp_trtri_f64(const double* L, double* W, int64_t npad, const void* potrf_ws, void* ws, void* stream) {
    if (!L || !W || !potrf_ws || !ws || (npad % DB)) return -1;
    cudaStream_t s = (cudaStream_t)stream;
    int nb = (int)(npad / DB);
    place_diag_inverse_kernel<<<nb, 256, 0, s>>>((const double*)potrf_ws, W, npad);
    GP_COUNT(1);
    GP_LAUNCH_CHECK();
    int rc = side_streams_init(s);
    if (rc) return rc;
    return trtri_rec(L, W, npad, 0, nb, (double*)ws, s, 0, 0);
}

int gp_lauum_f64(const double* W, double* Ainv, int64_t npad, void* stream) {
    if (!W || !Ainv || (npad % DB)) return -1;
    // Ainv_lower[i][j] = sum_{k >= i} W[k][i] W[k][j]
    return launch_dgemm(1, 1, Ainv, npad, W, npad, W, npad, (int)npad, (int)npad, (int)npad, 1.0, 0.0, KR_TN_LOWER, TM_LOWER,
                        (cudaStream_t)stream);
}

int gp_potri_f64(double* A, double* W, int64_t npad, const void* potrf_ws, void* ws, void* stream) {
    int rc = gp_trtri_f64(A, W, npad, potrf_ws, ws, stream);
    if (rc) return rc;
    return gp_lauum_f64(W, A, npad, stream);
}

}  // extern "C"
