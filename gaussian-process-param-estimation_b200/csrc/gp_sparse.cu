// Kernel-threshold sparse Matern correlation in CSR -- replaces the brute-force O(n^2) OpenMP COO fill + coo->csr of
// gaussian_proc/generate_correlation/_generate_sparse_correlation.pyx:35-201,472-594 by a uniform cell list (cell edge =
// taper radius; points of a cell kept in index order by a stable radix sort), a count pass, a device scan of the row
// pointer, a fill pass and - on demand (gp_csr_sort_rows / sort_rows = 1) - a per-row sort into the canonical CSR.
//
// Bit-exact pattern: the keep rule is the reference's strict `K_ij > tau` (:160). The scaled distance is evaluated
// in the reference's operation order with IEEE division/sqrt and no FMA contraction (this file is compiled with
// -fmad=false); only exp() can differ from glibc by an ulp, so pairs with |K - tau| <= 8 ulp are not decided on the
// device: they are listed, re-evaluated on the host with libm in the reference's arithmetic, and the accepted ones
// are appended to their rows (in that rare case the row pointer is rebuilt on the host).
#include "../../include/gpgp.h"
#include "gp_common.cuh"
#include "gp_internal.h"
#include "gp_matern.cuh"
#include <math.h>
#include <vector>

namespace gp {

constexpr int SMAXD = 3;             // cell list for d <= 3 (higher d: a single cell = brute force)
constexpr int BORDER_CAP = 1 << 20;  // max borderline ordered pairs
constexpr int SORT_CAP = 2048;       // max entries per row handled by the shared-memory sort

struct CellGrid {
    int d;
    int nc[SMAXD];
    double lo[SMAXD];
    double inv_size[SMAXD];
    int ncells;
};

// ---- host-side restatement of the scalar pieces (bit-following the reference) ---------------------------------
static double gamma_half_int(int dimension) {  // Gamma(d/2 + 1), _generate_sparse_correlation.pyx:208-233
    double g, k;
    if (dimension % 2 == 0) {
        k = 0.5 * dimension; g = 1.0;
        while (k > 0.0) { g *= k; k -= 1.0; }
    } else {
        k = ceil(0.5 * dimension); g = sqrt(M_PI);
        while (k > 0.0) { g *= k - 0.5; k -= 1.0; }
    }
    return g;
}

static double matern_host(double x, double nu) {  // _kernels.pyx:17-100, glibc exp/sqrt/pow
    if (x == 0) return 1.0;
    if (nu == 0.5) return exp(-x);
    if (nu == 1.5) return (1.0 + sqrt(3.0) * x) * exp(-sqrt(3.0) * x);
    if (nu == 2.5) return (1.0 + sqrt(5.0) * x + (5.0 / 3.0) * pow(x, 2.0)) * exp(-sqrt(5.0) * x);
    if (nu < 100) {
        double y = sqrt(2.0 * nu) * x, k, k1;
        bessel_k_pair(nu, y, &k, &k1);
        return (pow(2.0, 1.0 - nu) / tgamma(nu)) * pow(y, nu) * k;
    }
    return exp(-0.5 * pow(x, 2.0));
}

static double distance_host(const double* a, const double* b, const double* scale, int d) {
    double s = 0;
    for (int k = 0; k < d; ++k) s += pow((a[k] - b[k]) / scale[k], 2.0);
    return sqrt(s);
}

// scaled taper radius x_tau: K(x) > tau only if x < x_tau (K is decreasing); bisection, returned with a safety margin
static double support_radius(double tau, double nu) {
    if (!(tau > 0.0)) return 1e300;
    if (tau >= 1.0) return 0.0;
    double lo = 0.0, hi = 1.0;
    while (matern_host(hi, nu) > tau && hi < 1e6) hi *= 2.0;
    for (int it = 0; it < 200; ++it) {
        double mid = 0.5 * (lo + hi);
        if (matern_host(mid, nu) > tau) lo = mid; else hi = mid;
    }
    return hi * (1.0 + 1e-9) + 1e-300;
}

// ---- device pieces ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int cell_of_point(const double* p, const CellGrid& g) {
    int id = 0;
#pragma unroll
    for (int k = 0; k < SMAXD; ++k)
        if (k < g.d) {
            int c = (int)floor((p[k] - g.lo[k]) * g.inv_size[k]);
            c = c < 0 ? 0 : (c >= g.nc[k] ? g.nc[k] - 1 : c);
            id = id * g.nc[k] + c;
        }
    return id;
}

__global__ void cell_histogram_kernel(const double* __restrict__ pts, int n, int d, CellGrid g, int* cell_of, int* cell_cnt) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double p[SMAXD] = {0, 0, 0};
    for (int k = 0; k < d && k < SMAXD; ++k) p[k] = pts[(int64_t)i * d + k];
    int id = (g.ncells == 1) ? 0 : cell_of_point(p, g);
    cell_of[i] = id;
    atomicAdd(&cell_cnt[id], 1);
}

// bounding box of the points on the device: order-preserving 64-bit keys, atomicMin / atomicMax per coordinate
__device__ __forceinline__ unsigned long long dkey(double x) {
    unsigned long long b = (unsigned long long)__double_as_longlong(x);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
static double dkey_decode(unsigned long long k) {
    unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
    double x;
    memcpy(&x, &b, sizeof(double));
    return x;
}
__global__ void bbox_kernel(const double* __restrict__ pts, int64_t n, int d, unsigned long long* keys /* [8] min, [8] max */) {
    __shared__ unsigned long long smin[8], smax[8];
    if (threadIdx.x < 8) { smin[threadIdx.x] = ~0ull; smax[threadIdx.x] = 0ull; }
    __syncthreads();
    // block-uniform trip count: every lane takes part in the shuffles, out-of-range lanes carry the identities
    for (int64_t base = (int64_t)blockIdx.x * blockDim.x; base < n; base += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = base + threadIdx.x;
        for (int k = 0; k < d; ++k) {
            unsigned long long mn = ~0ull, mx = 0ull;
            if (i < n) mn = mx = dkey(pts[i * d + k]);
            for (int o = 16; o > 0; o >>= 1) {
                unsigned long long a = __shfl_xor_sync(0xffffffffu, mn, o), b = __shfl_xor_sync(0xffffffffu, mx, o);
                mn = a < mn ? a : mn;
                mx = b > mx ? b : mx;
            }
            if ((threadIdx.x & 31) == 0) { atomicMin(&smin[k], mn); atomicMax(&smax[k], mx); }
        }
    }
    __syncthreads();
    if (threadIdx.x < d) { atomicMin(&keys[threadIdx.x], smin[threadIdx.x]); atomicMax(&keys[8 + threadIdx.x], smax[threadIdx.x]); }
}

__global__ void sum64_kernel(const int* __restrict__ v, int n, unsigned long long* out) {
    unsigned long long acc = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) acc += (unsigned)v[i];
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

// The points of a cell are kept in ORIGINAL index order (stable radix sort of the cell ids): the generation order of
// every row - and with it the row-blocked operator and every estimate - is the same in every run.
// cell ids as 64-bit sort keys (gp_sort_keys_u64 works on 64-bit keys)
__global__ void widen_keys_kernel(const int* __restrict__ in, int n, unsigned long long* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (unsigned long long)(unsigned)in[i];
}

__global__ void gather_points_kernel(const double* __restrict__ pts, int n, int d, const int* __restrict__ sorted_idx,
                                     double* sorted_pts) {
    int pos = blockIdx.x * blockDim.x + threadIdx.x;
    if (pos >= n) return;
    int i = sorted_idx[pos];
    for (int k = 0; k < d; ++k) sorted_pts[(int64_t)pos * d + k] = pts[(int64_t)i * d + k];
}

struct SparseParams {
    double tau, band;         // keep rule K > tau; |K - tau| <= band -> host decides
    double r2_lo, r2_hi;      // squared scaled distance certainly inside / outside the support (quick classification)
    int quick;                // 0: no quick classification (tau <= 0 or tau >= 1)
    double scale[8];
    MaternParams mp;
    int d, n;
    // row filter of the row-slab engine (one slab of the ordered operator per GPU): only rows i with
    // row_first <= row_pos[i] < row_last are generated, the others stay empty. row_pos == nullptr: every row.
    const int* row_pos;
    int row_first, row_last;
};

// reference arithmetic: divide-then-square, k-ordered sum, IEEE sqrt (_kernels.pyx:130-136)
__device__ __forceinline__ double scaled_distance(const double* a, const double* b, const SparseParams& sp) {
    double s = 0.0;
    for (int k = 0; k < sp.d; ++k) {
        double t = (a[k] - b[k]) / sp.scale[k];
        s += t * t;
    }
    return sqrt(s);
}

// One warp per (cell-sorted) point. PASS 0 counts kept entries and lists borderline pairs; PASS 1 writes (col, value
// [, dvalue]) into the row's segment (any order: the rows are sorted afterwards).
// Candidates are first classified by their squared scaled distance (multiply-by-reciprocal, no sqrt / exp): further than
// the support radius by a 1e-7 margin -> dropped; closer by the same margin -> kept (PASS 0 just counts them). Only the
// others are evaluated in the reference's arithmetic (IEEE divide, sqrt, exp) - in PASS 0 a vanishing fraction, in
// PASS 1 the kept third of the candidates, which are compacted through a per-warp queue so that the expensive
// evaluation always runs on full warps.
template <int MODE, int PASS, bool WITH_DK>
__global__ void __launch_bounds__(256)
sparse_rows_kernel(SparseParams sp, CellGrid g, const int* __restrict__ cell_start, const int* __restrict__ sorted_idx,
                   const double* __restrict__ sorted_pts, int* devcount, int* border_cnt, int2* border,
                   const int* __restrict__ indptr, int* indices, double* data, double* ddata) {
    __shared__ int queue_s[8][64];
    const int lane = threadIdx.x & 31;
    int* queue = queue_s[threadIdx.x >> 5];
    const int wpos = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (wpos >= sp.n) return;
    const int i = sorted_idx[wpos];
    if (sp.row_pos) {
        const int pos = sp.row_pos[i];
        if (pos < sp.row_first || pos >= sp.row_last) {      // another rank's row
            if (PASS == 0 && lane == 0) devcount[i] = 0;
            return;
        }
    }
    double pi[8];
    for (int k = 0; k < sp.d; ++k) pi[k] = sorted_pts[(int64_t)wpos * sp.d + k];
    int cc[SMAXD] = {0, 0, 0};
    if (g.ncells > 1) {
        int id = cell_of_point(pi, g);
        for (int k = g.d - 1; k >= 0; --k) { cc[k] = id % g.nc[k]; id /= g.nc[k]; }
    }
    int count = 0;
    int qn = 0;                                   // queued candidates (warp-uniform)
    const int64_t base = (PASS == 1) ? (int64_t)indptr[i] : 0;

    // exact evaluation of candidate q (sorted position) by the lanes with act = true
    auto evaluate = [&](int q, bool act) {
        bool keep = false;
        double val = 0.0, dval = 0.0;
        int j = -1;
        if (act) {
            j = sorted_idx[q];
            double pj[8];
            for (int k = 0; k < sp.d; ++k) pj[k] = sorted_pts[(int64_t)q * sp.d + k];
            double x = (i <= j) ? scaled_distance(pi, pj, sp) : scaled_distance(pj, pi, sp);
            if (WITH_DK && PASS == 1) matern_value_drho<MODE>(x, sp.mp, &val, &dval);
            else val = matern_value<MODE>(x, sp.mp);
            bool borderline = (i != j) && fabs(val - sp.tau) <= sp.band;
            keep = !borderline && (val > sp.tau);
            if (PASS == 0 && borderline) {
                int slot = atomicAdd(border_cnt, 1);
                if (slot < BORDER_CAP) border[slot] = make_int2(i, j);
            }
        }
        unsigned m = __ballot_sync(0xffffffffu, keep);
        if (PASS == 1 && keep) {
            int64_t o = base + count + __popc(m & ((1u << lane) - 1u));
            indices[o] = j;
            data[o] = val;
            if (WITH_DK) ddata[o] = dval;
        }
        count += __popc(m);
    };

    const int span = (g.ncells > 1) ? 3 : 1;
    const int nnb = (g.ncells > 1) ? (g.d == 1 ? 3 : (g.d == 2 ? 9 : 27)) : 1;
    for (int nb = 0; nb < nnb; ++nb) {
        int id = 0;
        bool ok = true;
        if (g.ncells > 1) {
            int r = nb;
            int off[SMAXD];
            for (int k = g.d - 1; k >= 0; --k) { off[k] = r % span - 1; r /= span; }
            for (int k = 0; k < g.d; ++k) {
                int c = cc[k] + off[k];
                if (c < 0 || c >= g.nc[k]) ok = false;
                id = id * g.nc[k] + c;
            }
        }
        if (!ok) continue;
        const int s0 = cell_start[id], s1 = cell_start[id + 1];
        for (int q0 = s0; q0 < s1; q0 += 32) {
            const int q = q0 + lane;
            if (!sp.quick) { evaluate(q, q < s1); continue; }
            bool need = false, sure = false;
            if (q < s1) {
                double s2 = 0.0;
                for (int k = 0; k < sp.d; ++k) {
                    double t = (pi[k] - sorted_pts[(int64_t)q * sp.d + k]) * sp.mp.inv_scale[k];
                    s2 += t * t;
                }
                if (PASS == 0 && s2 < sp.r2_lo) sure = true;          // certainly K > tau
                else if (!(s2 > sp.r2_hi)) need = true;               // kept entry (PASS 1) or inside the margin
            }
            if (PASS == 0) count += __popc(__ballot_sync(0xffffffffu, sure));
            const unsigned mn = __ballot_sync(0xffffffffu, need);
            if (need) queue[qn + __popc(mn & ((1u << lane) - 1u))] = q;
            qn += __popc(mn);
            __syncwarp();
            if (qn >= 32) {
                const int qq = queue[lane];
                const int rest = (lane < qn - 32) ? queue[32 + lane] : 0;
                __syncwarp();
                if (lane < qn - 32) queue[lane] = rest;
                qn -= 32;
                __syncwarp();
                evaluate(qq, true);
            }
        }
    }
    if (qn > 0) evaluate(lane < qn ? queue[lane] : 0, lane < qn);
    if (PASS == 0 && lane == 0) devcount[i] = count;
}

__global__ void place_extras_kernel(int nextra, const int* __restrict__ ei, const int* __restrict__ ej,
                                    const double* __restrict__ ev, const double* __restrict__ edv, const int* __restrict__ eslot,
                                    const int* __restrict__ indptr, const int* __restrict__ devcount, int* indices, double* data,
                                    double* ddata) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nextra) return;
    int i = ei[t];
    int64_t o = (int64_t)indptr[i] + devcount[i] + eslot[t];
    indices[o] = ej[t];
    data[o] = ev[t];
    if (ddata) ddata[o] = edv[t];
}

// One WARP per row (rows of <= WSORT_CAP entries, i.e. practically all of them): bitonic sort of packed (col, position)
// words in shared memory with warp-level barriers only, then the values are permuted through their staged copies.
// Longer rows are flagged and left to the CTA-wide kernel below.
constexpr int WSORT_CAP = 512;
__global__ void __launch_bounds__(128)
sort_rows_warp_kernel(int n, const int* __restrict__ indptr, int* indices, double* data, double* ddata, int* has_long) {
    __shared__ unsigned long long sk[4][WSORT_CAP];
    __shared__ double sv[4][WSORT_CAP];
    __shared__ double sd[4][WSORT_CAP];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    unsigned long long* k = sk[w];
    double* v = sv[w];
    double* dv = sd[w];
    for (int row = blockIdx.x * 4 + w; row < n; row += gridDim.x * 4) {
        const int s0 = indptr[row], len = indptr[row + 1] - s0;
        if (len <= 1) continue;
        if (len > WSORT_CAP) { if (lane == 0) atomicExch(has_long, 1); continue; }
        int m = 32;
        while (m < len) m <<= 1;
        bool sorted = true;
        for (int t = lane; t < m; t += 32) {
            const int key = (t < len) ? indices[s0 + t] : 0x7fffffff;
            if (t + 1 < len && indices[s0 + t + 1] < key) sorted = false;
            k[t] = ((unsigned long long)(unsigned)key << 32) | (unsigned)t;
            if (t < len) {
                v[t] = data[s0 + t];
                if (ddata) dv[t] = ddata[s0 + t];
            }
        }
        if (__all_sync(0xffffffffu, sorted)) { __syncwarp(); continue; }
        __syncwarp();
        for (int kk = 2; kk <= m; kk <<= 1)
            for (int j = kk >> 1; j > 0; j >>= 1) {
                for (int i = lane; i < (m >> 1); i += 32) {
                    const int t = 2 * i - (i & (j - 1));      // lower index of the pair (bit j clear)
                    const int p = t + j;
                    const bool up = ((t & kk) == 0);
                    const unsigned long long a = k[t], b = k[p];
                    if ((a > b) == up) { k[t] = b; k[p] = a; }
                }
                __syncwarp();
            }
        for (int t = lane; t < len; t += 32) {
            const unsigned long long e = k[t];
            const int pos = (int)(e & 0xffffffffu);
            indices[s0 + t] = (int)(e >> 32);
            data[s0 + t] = v[pos];
            if (ddata) ddata[s0 + t] = dv[pos];
        }
        __syncwarp();
    }
}

// one CTA per row (grid-stride): bitonic sort of (col, value[, dvalue]) by col in shared memory
__global__ void __launch_bounds__(256)
sort_rows_kernel(int n, const int* __restrict__ indptr, int* indices, double* data, double* ddata, int* overflow) {
    __shared__ int keys[SORT_CAP];
    __shared__ double vals[SORT_CAP];
    __shared__ double dvals[SORT_CAP];
    for (int row = blockIdx.x; row < n; row += gridDim.x) {
        const int s0 = indptr[row], len = indptr[row + 1] - s0;
        if (len <= WSORT_CAP) continue;      // sorted by sort_rows_warp_kernel
        if (len > SORT_CAP) { if (threadIdx.x == 0) atomicExch(overflow, row + 1); continue; }
        int m = 1;
        while (m < len) m <<= 1;
        __syncthreads();
        for (int t = threadIdx.x; t < m; t += blockDim.x) {
            keys[t] = (t < len) ? indices[s0 + t] : 0x7fffffff;
            vals[t] = (t < len) ? data[s0 + t] : 0.0;
            if (ddata) dvals[t] = (t < len) ? ddata[s0 + t] : 0.0;
        }
        __syncthreads();
        for (int k = 2; k <= m; k <<= 1)
            for (int jj = k >> 1; jj > 0; jj >>= 1) {
                for (int t = threadIdx.x; t < m; t += blockDim.x) {
                    int p = t ^ jj;
                    if (p > t) {
                        bool up = ((t & k) == 0);
                        int a = keys[t], b = keys[p];
                        if ((a > b) == up) {
                            keys[t] = b; keys[p] = a;
                            double v = vals[t]; vals[t] = vals[p]; vals[p] = v;
                            if (ddata) { double w = dvals[t]; dvals[t] = dvals[p]; dvals[p] = w; }
                        }
                    }
                }
                __syncthreads();
            }
        for (int t = threadIdx.x; t < len; t += blockDim.x) {
            indices[s0 + t] = keys[t];
            data[s0 + t] = vals[t];
            if (ddata) ddata[s0 + t] = dvals[t];
        }
    }
}

// workspace carving (all int32 / f64 device arrays)
struct SparseWs {
    int *cell_of, *cell_start, *cell_fill, *sorted_idx, *devcount, *border_cnt, *overflow;
    unsigned long long* keys64;
    void* sort_temp;
    size_t sort_temp_bytes;
    unsigned long long* bbox_keys;   // [8] min keys, [8] max keys, [16] total nnz
    double* bbox;                    // lo[8], hi[8] (decoded, for the fill call)
    int2* border;
    int *ei, *ej, *eslot;
    double *ev, *edv, *sorted_pts;
    size_t total;
};
static size_t al(size_t x) { return (x + 255) & ~(size_t)255; }
static SparseWs carve_sparse(void* ws, int64_t n, int64_t d) {
    SparseWs w;
    char* base = (char*)ws;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += al(bytes); return base ? base + o : (char*)nullptr; };
    int64_t maxcells = 2 * n + 64;
    w.cell_of = (int*)take(sizeof(int) * n);
    w.cell_start = (int*)take(sizeof(int) * (maxcells + 1));
    w.cell_fill = (int*)take(sizeof(int) * maxcells);
    w.sorted_idx = (int*)take(sizeof(int) * n);
    w.devcount = (int*)take(sizeof(int) * n);
    w.border_cnt = (int*)take(sizeof(int) * 4);
    w.overflow = (int*)take(sizeof(int) * 4);
    w.border = (int2*)take(sizeof(int2) * BORDER_CAP);
    w.ei = (int*)take(sizeof(int) * BORDER_CAP);
    w.ej = (int*)take(sizeof(int) * BORDER_CAP);
    w.eslot = (int*)take(sizeof(int) * BORDER_CAP);
    w.ev = (double*)take(sizeof(double) * BORDER_CAP);
    w.edv = (double*)take(sizeof(double) * BORDER_CAP);
    w.sorted_pts = (double*)take(sizeof(double) * n * d);
    w.keys64 = (unsigned long long*)take(sizeof(unsigned long long) * n);
    w.sort_temp_bytes = (size_t)n * 16 + (8u << 20);      // radix sort scratch (alternate key/value buffers + histograms)
    w.sort_temp = (void*)take(w.sort_temp_bytes);
    w.bbox_keys = (unsigned long long*)take(sizeof(unsigned long long) * 24);
    w.bbox = (double*)take(sizeof(double) * 16);
    w.total = off;
    return w;
}

static int make_params(int64_t n, int64_t d, const double* scale_host, double nu, double tau, const MaternParams& mp,
                       const double* bbox_lo, const double* bbox_hi, SparseParams* sp, CellGrid* g) {
    sp->tau = tau;
    sp->band = 8.0 * 2.220446049250313e-16 * fabs(tau);
    sp->d = (int)d;
    sp->n = (int)n;
    sp->row_pos = nullptr;
    sp->row_first = sp->row_last = 0;
    for (int k = 0; k < d; ++k) sp->scale[k] = scale_host[k];
    sp->mp = mp;
    double xr = support_radius(tau, nu);
    sp->quick = (tau > 0.0 && tau < 1.0 && xr > 0.0 && xr < 1e100) ? 1 : 0;
    sp->r2_lo = xr * xr * (1.0 - 4e-7);
    sp->r2_hi = xr * xr * (1.0 + 4e-7);
    g->d = (int)d;
    g->ncells = 1;
    for (int k = 0; k < SMAXD; ++k) { g->nc[k] = 1; g->lo[k] = 0.0; g->inv_size[k] = 0.0; }
    if (d <= SMAXD && xr < 1e200) {
        double cells = 1.0;
        int nc[SMAXD] = {1, 1, 1};
        for (int k = 0; k < d; ++k) {
            double size = xr * scale_host[k];
            double extent = bbox_hi[k] - bbox_lo[k];
            double c = (size > 0.0) ? floor(extent / size) : 1e9;
            if (c < 1.0) c = 1.0;
            if (c > 4096.0) c = 4096.0;
            nc[k] = (int)c;
            cells *= c;
        }
        // cap the total at ~2n cells by coarsening (cells may only get larger than the radius, never smaller)
        while (cells > 2.0 * (double)n + 32.0) {
            cells = 1.0;
            for (int k = 0; k < d; ++k) { nc[k] = (nc[k] + 1) / 2; cells *= nc[k]; }
        }
        for (int k = 0; k < d; ++k) {
            double extent = bbox_hi[k] - bbox_lo[k];
            g->nc[k] = nc[k];
            g->lo[k] = bbox_lo[k];
            g->inv_size[k] = (extent > 0.0) ? nc[k] / extent : 0.0;   // cell edge = extent / nc >= radius
        }
        g->ncells = (int)cells;
    }
    return 0;
}

template <int MODE>
static void launch_rows(int pass, bool with_dk, const SparseParams& sp, const CellGrid& g, const SparseWs& w, const int* indptr,
                        int* indices, double* data, double* ddata, cudaStream_t s) {
    int blocks = (int)(((int64_t)sp.n * 32 + 255) / 256);
    if (pass == 0)
        sparse_rows_kernel<MODE, 0, false><<<blocks, 256, 0, s>>>(sp, g, w.cell_start, w.sorted_idx, w.sorted_pts, w.devcount,
                                                                  w.border_cnt, w.border, nullptr, nullptr, nullptr, nullptr);
    else if (with_dk)
        sparse_rows_kernel<MODE, 1, true><<<blocks, 256, 0, s>>>(sp, g, w.cell_start, w.sorted_idx, w.sorted_pts, w.devcount,
                                                                 w.border_cnt, w.border, indptr, indices, data, ddata);
    else
        sparse_rows_kernel<MODE, 1, false><<<blocks, 256, 0, s>>>(sp, g, w.cell_start, w.sorted_idx, w.sorted_pts, w.devcount,
                                                                  w.border_cnt, w.border, indptr, indices, data, nullptr);
    GP_COUNT(1);
}

struct MortonParams {
    double lo[3], mul[3];
    int nd, d, bits;
};

__global__ void morton_keys_kernel(const double* __restrict__ points, int64_t n, MortonParams mp, int64_t* keys) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long qmax = (1ull << mp.bits) - 1ull;
    unsigned long long q[3] = {0ull, 0ull, 0ull};
    for (int k = 0; k < mp.nd; ++k) {
        double t = (points[i * mp.d + k] - mp.lo[k]) * mp.mul[k];
        unsigned long long v = (t > 0.0) ? (unsigned long long)t : 0ull;
        q[k] = v > qmax ? qmax : v;
    }
    unsigned long long key = 0ull;
    if (mp.nd == 2) {
        // Hilbert curve index (no long jumps between consecutive keys: consecutive rows of the sorted order are always
        // spatial neighbours, which keeps the fill-in of the 8 x 1 row blocks low)
        unsigned long long x = q[0], y = q[1];
        for (unsigned long long s = 1ull << (mp.bits - 1); s > 0; s >>= 1) {
            const unsigned long long rx = (x & s) ? 1ull : 0ull, ry = (y & s) ? 1ull : 0ull;
            key += s * s * ((3ull * rx) ^ ry);
            if (!ry) {
                if (rx) { x = (s << 1) - 1ull - (x & ((s << 1) - 1ull)); y = (s << 1) - 1ull - (y & ((s << 1) - 1ull)); }
                const unsigned long long t = x; x = y; y = t;
            }
            x &= (s << 1) - 1ull;
            y &= (s << 1) - 1ull;
        }
    } else {
        for (int b = mp.bits - 1; b >= 0; --b)
            for (int k = 0; k < mp.nd; ++k) key = (key << 1) | ((q[k] >> b) & 1ull);
    }
    keys[i] = (int64_t)key;
}

}  // namespace gp

using namespace gp;

extern "C" {

int gp_kernel_threshold(int64_t n, int64_t d, double density, const double* scale_host, double nu, double* tau_host) {
    // _estimate_kernel_threshold, _generate_sparse_correlation.pyx:294-413 (with _ball_volume given its dimension)
    if (!scale_host || !tau_host || n <= 0 || d <= 0) return -1;
    if (int rc = matern_check(scale_host, d, nu, false)) return rc;
    double adjacency_volume = density * (double)n;
    if (adjacency_volume < 1.0) return -10;  // -> ValueError in the Python layer (:378-383)
    double prod = 1.0;
    for (int k = 0; k < d; ++k) prod *= scale_host[k];
    double geometric_mean_radius = pow(prod, 1.0 / (double)d);
    double ellipsoid_volume = pow(geometric_mean_radius * sqrt(M_PI), (double)d) / gamma_half_int((int)d);
    adjacency_volume /= ellipsoid_volume;
    double adjacency_radius = pow(gamma_half_int((int)d) * adjacency_volume, 1.0 / (double)d) / sqrt(M_PI);
    double grid_axis_num_points = pow((double)n, 1.0 / (double)d);
    double grid_size = 1.0 / (grid_axis_num_points - 1.0);
    double kernel_radius = grid_size * adjacency_radius;
    *tau_host = matern_host(kernel_radius, nu);
    return 0;
}

int64_t gp_sparse_workspace_bytes(int64_t n, int64_t d) { return (int64_t)carve_sparse(nullptr, n, d).total; }

}  // extern "C"

// Bounding box, cell grid (cell edge >= support radius), cell-sorted point list: everything the row / row-block kernels
// enumerate candidates from. Leaves the bounding box in w.bbox for the fill call.
static int sparse_prepare(const double* points, int64_t n, int64_t d, const double* scale_host, double nu, double tau,
                          const MaternParams& mp, const SparseWs& w, cudaStream_t s, SparseParams* sp_out, CellGrid* g_out) {
    const int N = (int)n, D = (int)d;
    double lo[8], hi[8], bb[16];
    {
        unsigned long long init[24], got[16];
        for (int k = 0; k < 8; ++k) { init[k] = ~0ull; init[8 + k] = 0ull; init[16 + k] = 0ull; }
        GP_CUDA_CHECK(cudaMemcpyAsync(w.bbox_keys, init, sizeof(init), cudaMemcpyHostToDevice, s));
        bbox_kernel<<<296, 256, 0, s>>>(points, n, D, w.bbox_keys);
        GP_COUNT(1);
        GP_CUDA_CHECK(cudaMemcpyAsync(got, w.bbox_keys, sizeof(got), cudaMemcpyDeviceToHost, s));
        GP_CUDA_CHECK(cudaStreamSynchronize(s));
        for (int k = 0; k < 8; ++k) {
            lo[k] = (k < d) ? dkey_decode(got[k]) : 0.0;
            hi[k] = (k < d) ? dkey_decode(got[8 + k]) : 0.0;
            bb[k] = lo[k];
            bb[8 + k] = hi[k];
        }
        GP_CUDA_CHECK(cudaMemcpyAsync(w.bbox, bb, sizeof(bb), cudaMemcpyHostToDevice, s));
    }
    SparseParams& sp = *sp_out;
    CellGrid& g = *g_out;
    make_params(n, d, scale_host, nu, tau, mp, lo, hi, &sp, &g);
    GP_CUDA_CHECK(cudaMemsetAsync(w.cell_start, 0, sizeof(int) * (g.ncells + 1), s));
    GP_CUDA_CHECK(cudaMemsetAsync(w.border_cnt, 0, sizeof(int) * 4, s));
    GP_CUDA_CHECK(cudaMemsetAsync(w.overflow, 0, sizeof(int) * 4, s));
    cell_histogram_kernel<<<(N + 255) / 256, 256, 0, s>>>(points, N, D, g, w.cell_of, w.cell_start + 1);
    GP_COUNT(1);
    // host exclusive scan of the cell histogram
    std::vector<int> cs(g.ncells + 1);
    GP_CUDA_CHECK(cudaMemcpyAsync(cs.data(), w.cell_start, sizeof(int) * (g.ncells + 1), cudaMemcpyDeviceToHost, s));
    GP_CUDA_CHECK(cudaStreamSynchronize(s));
    for (int c = 0; c < g.ncells; ++c) cs[c + 1] += cs[c];
    GP_CUDA_CHECK(cudaMemcpyAsync(w.cell_start, cs.data(), sizeof(int) * (g.ncells + 1), cudaMemcpyHostToDevice, s));
    {
        int bits = 1;
        while ((1 << bits) < g.ncells && bits < 31) ++bits;
        // stable radix sort of the cell ids (own kernels, csrc/gp_index.cu): the points of a cell stay in index order
        if ((size_t)gp_sort_workspace_bytes(N) > w.sort_temp_bytes) return -24;
        widen_keys_kernel<<<(N + 255) / 256, 256, 0, s>>>(w.cell_of, N, w.keys64);
        if (int rc = gp_sort_keys_u64(w.keys64, N, bits, w.sorted_idx, w.sort_temp, s)) return rc;
        gather_points_kernel<<<(N + 255) / 256, 256, 0, s>>>(points, N, D, w.sorted_idx, w.sorted_pts);
        GP_COUNT(2);
    }
    return 0;
}

extern "C" {

int gp_matern_sparse_count(const double* points, const double* points_host, int64_t n, int64_t d, const double* scale_host,
                           double nu, double tau, void* ws, int* indptr_dev, int64_t* nnz_host, const int* row_pos_dev,
                           int64_t row_first, int64_t row_last, void* stream) {
    if (!points || !points_host || !scale_host || !ws || !indptr_dev || !nnz_host || n <= 0 || d <= 0 || d > 8 || n > INT32_MAX)
        return -1;
    if (row_pos_dev && (row_first < 0 || row_last < row_first || row_last > n)) return -1;
    MaternParams mp;
    int mode;
    if (int rc = matern_params(scale_host, d, nu, false, &mp, &mode)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    SparseWs w = carve_sparse(ws, n, d);
    SparseParams sp;
    CellGrid g;
    if (int rc = sparse_prepare(points, n, d, scale_host, nu, tau, mp, w, s, &sp, &g)) return rc;
    sp.row_pos = row_pos_dev;
    sp.row_first = (int)row_first;
    sp.row_last = (int)row_last;
    const int N = (int)n;
    with_matern_mode(mode, [&](auto tag) {
        launch_rows<decltype(tag)::value>(0, false, sp, g, w, nullptr, nullptr, nullptr, nullptr, s);
    });
    GP_LAUNCH_CHECK();
    int nb = 0;
    unsigned long long total = 0;
    sum64_kernel<<<296, 256, 0, s>>>(w.devcount, N, w.bbox_keys + 16);
    GP_COUNT(1);
    GP_CUDA_CHECK(cudaMemcpyAsync(&nb, w.border_cnt, sizeof(int), cudaMemcpyDeviceToHost, s));
    GP_CUDA_CHECK(cudaMemcpyAsync(&total, w.bbox_keys + 16, sizeof(total), cudaMemcpyDeviceToHost, s));
    GP_CUDA_CHECK(cudaStreamSynchronize(s));
    if (nb > BORDER_CAP) return -21;
    if (nb == 0) {
        // the common case: no borderline pair -> the row pointer is an exclusive scan on the device
        if (total > (unsigned long long)INT32_MAX) return -22;
        if (int rc = gp_scan_counts_i32(w.devcount, N, indptr_dev, s)) return rc;
        int meta0[4] = {0, 0, 0, 0};
        GP_CUDA_CHECK(cudaMemcpyAsync(w.border_cnt, meta0, sizeof(int) * 4, cudaMemcpyHostToDevice, s));
        GP_CUDA_CHECK(cudaStreamSynchronize(s));
        *nnz_host = (int64_t)total;
        return 0;
    }
    std::vector<int> cnt(n);
    GP_CUDA_CHECK(cudaMemcpyAsync(cnt.data(), w.devcount, sizeof(int) * n, cudaMemcpyDeviceToHost, s));
    GP_CUDA_CHECK(cudaStreamSynchronize(s));
    // borderline pairs: decide with the reference's host arithmetic
    std::vector<int> ei, ej, eslot;
    std::vector<double> ev, edv;
    if (nb > 0) {
        std::vector<int2> bl(nb);
        GP_CUDA_CHECK(cudaMemcpy(bl.data(), w.border, sizeof(int2) * nb, cudaMemcpyDeviceToHost));
        std::vector<int> extra(n, 0);
        for (int t = 0; t < nb; ++t) {
            int i = bl[t].x, j = bl[t].y;
            const double* a = points_host + (int64_t)(i <= j ? i : j) * d;
            const double* b = points_host + (int64_t)(i <= j ? j : i) * d;
            double x = distance_host(a, b, scale_host, (int)d);
            double v = matern_host(x, nu);
            if (v > tau) {
                ei.push_back(i); ej.push_back(j); ev.push_back(v); eslot.push_back(extra[i]++);
                edv.push_back(0.0);  // filled on the device side convention: derivative of borderline entries is recomputed below
            }
        }
        for (int64_t i = 0; i < n; ++i) cnt[i] += extra[i];
    }
    std::vector<int> ip(n + 1);
    int64_t run = 0;
    for (int64_t i = 0; i < n; ++i) { ip[i] = (int)run; run += cnt[i]; }
    if (run > INT32_MAX) return -22;
    ip[n] = (int)run;
    *nnz_host = run;
    GP_CUDA_CHECK(cudaMemcpyAsync(indptr_dev, ip.data(), sizeof(int) * (n + 1), cudaMemcpyHostToDevice, s));
    int ne = (int)ei.size();
    int meta[4] = {ne, 0, 0, 0};
    GP_CUDA_CHECK(cudaMemcpyAsync(w.border_cnt, meta, sizeof(int) * 4, cudaMemcpyHostToDevice, s));
    if (ne > 0) {
        GP_CUDA_CHECK(cudaMemcpyAsync(w.ei, ei.data(), sizeof(int) * ne, cudaMemcpyHostToDevice, s));
        GP_CUDA_CHECK(cudaMemcpyAsync(w.ej, ej.data(), sizeof(int) * ne, cudaMemcpyHostToDevice, s));
        GP_CUDA_CHECK(cudaMemcpyAsync(w.eslot, eslot.data(), sizeof(int) * ne, cudaMemcpyHostToDevice, s));
        GP_CUDA_CHECK(cudaMemcpyAsync(w.ev, ev.data(), sizeof(double) * ne, cudaMemcpyHostToDevice, s));
    }
    GP_CUDA_CHECK(cudaStreamSynchronize(s));  // host vectors go out of scope
    return 0;
}

// Space-filling-curve keys of the points over their bounding box (2-D: Hilbert index, 31 bits per coordinate; otherwise
// Z-order / Morton over the first min(d, 3) coordinates, 63 / min(d, 3) bits each): a stable sort by this key gives a deterministic, spatially local ordering of the points. The sparse operator
// uses it internally (row-blocked form, gp_bcsr_*): consecutive rows then have nearly identical patterns.
int gp_spatial_keys(const double* points, int64_t n, int64_t d, const double* lo_host, const double* hi_host,
                    int64_t* keys_dev, void* stream) {
    if (!points || !lo_host || !hi_host || !keys_dev || n <= 0 || d <= 0) return -1;
    MortonParams mp;
    mp.nd = (int)(d < 3 ? d : 3);
    mp.d = (int)d;
    mp.bits = 63 / mp.nd;
    if (mp.bits > 31) mp.bits = 31;
    for (int k = 0; k < 3; ++k) { mp.lo[k] = 0.0; mp.mul[k] = 0.0; }
    for (int k = 0; k < mp.nd; ++k) {
        double extent = hi_host[k] - lo_host[k];
        mp.lo[k] = lo_host[k];
        mp.mul[k] = (extent > 0.0) ? ldexp(1.0, mp.bits) / extent : 0.0;
    }
    morton_keys_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(points, n, mp, keys_dev);
    GP_COUNT(1);
    GP_LAUNCH_CHECK();
    return 0;
}

static int sort_rows_run(int64_t n, const int* indptr_dev, int* indices_dev, double* data_dev, double* ddata_dev, int* flags,
                         cudaStream_t s) {
    GP_CUDA_CHECK(cudaMemsetAsync(flags, 0, sizeof(int) * 2, s));
    sort_rows_warp_kernel<<<148 * 4, 128, 0, s>>>((int)n, indptr_dev, indices_dev, data_dev, ddata_dev, flags + 1);
    GP_COUNT(1);
    GP_LAUNCH_CHECK();
    int ovf[2] = {0, 0};
    GP_CUDA_CHECK(cudaMemcpyAsync(ovf, flags, sizeof(int) * 2, cudaMemcpyDeviceToHost, s));
    GP_CUDA_CHECK(cudaStreamSynchronize(s));
    if (ovf[1]) {   // rows longer than WSORT_CAP exist: CTA-wide sort for those
        sort_rows_kernel<<<148 * 8, 256, 0, s>>>((int)n, indptr_dev, indices_dev, data_dev, ddata_dev, flags);
        GP_COUNT(1);
        GP_LAUNCH_CHECK();
        GP_CUDA_CHECK(cudaMemcpyAsync(ovf, flags, sizeof(int), cudaMemcpyDeviceToHost, s));
        GP_CUDA_CHECK(cudaStreamSynchronize(s));
    }
    if (ovf[0]) return -23;  // a row longer than SORT_CAP
    return 0;
}

// Sorts every row of a CSR matrix by column index (values and optional derivative values follow): the canonical form.
// flags_dev: 2 device ints of scratch.
int gp_csr_sort_rows(int64_t n, const int* indptr_dev, int* indices_dev, double* data_dev, double* ddata_dev, int* flags_dev,
                     void* stream) {
    if (!indptr_dev || !indices_dev || !data_dev || !flags_dev || n <= 0 || n > INT32_MAX) return -1;
    return sort_rows_run(n, indptr_dev, indices_dev, data_dev, ddata_dev, flags_dev, (cudaStream_t)stream);
}

int gp_matern_sparse_fill(const double* points, const double* points_host, int64_t n, int64_t d, const double* scale_host,
                          double nu, double tau, void* ws, const int* indptr_dev, int* indices_dev, double* data_dev,
                          double* ddata_dev, int sort_rows, const int* row_pos_dev, int64_t row_first, int64_t row_last,
                          void* stream) {
    if (!points || !points_host || !scale_host || !ws || !indptr_dev || !indices_dev || !data_dev || n <= 0 || d <= 0 || d > 8)
        return -1;
    if (row_pos_dev && (row_first < 0 || row_last < row_first || row_last > n)) return -1;
    MaternParams mp;
    int mode;
    if (int rc = matern_params(scale_host, d, nu, ddata_dev != nullptr, &mp, &mode)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    SparseWs w = carve_sparse(ws, n, d);
    double bb[16];
    int meta[4];
    GP_CUDA_CHECK(cudaMemcpyAsync(bb, w.bbox, sizeof(bb), cudaMemcpyDeviceToHost, s));      // left by the count call
    GP_CUDA_CHECK(cudaMemcpyAsync(meta, w.border_cnt, sizeof(int) * 4, cudaMemcpyDeviceToHost, s));
    GP_CUDA_CHECK(cudaStreamSynchronize(s));
    SparseParams sp;
    CellGrid g;
    make_params(n, d, scale_host, nu, tau, mp, bb, bb + 8, &sp, &g);
    sp.row_pos = row_pos_dev;
    sp.row_first = (int)row_first;
    sp.row_last = (int)row_last;
    int ne = meta[0];
    with_matern_mode(mode, [&](auto tag) {
        launch_rows<decltype(tag)::value>(1, ddata_dev != nullptr, sp, g, w, indptr_dev, indices_dev, data_dev, ddata_dev, s);
    });
    if (ne > 0) {
        if (ddata_dev) {
            // derivative values of the host-decided entries (any ulp-level value is fine here: only the pattern and
            // the K values are pinned)
            std::vector<int> ei(ne), ej(ne);
            std::vector<double> edv(ne);
            GP_CUDA_CHECK(cudaMemcpy(ei.data(), w.ei, sizeof(int) * ne, cudaMemcpyDeviceToHost));
            GP_CUDA_CHECK(cudaMemcpy(ej.data(), w.ej, sizeof(int) * ne, cudaMemcpyDeviceToHost));
            double rho = scale_host[0], h = 1e-6 * rho;
            std::vector<double> sc(d);
            for (int t = 0; t < ne; ++t) {
                const double* a = points_host + (int64_t)ei[t] * d;
                const double* b = points_host + (int64_t)ej[t] * d;
                for (int k = 0; k < d; ++k) sc[k] = rho + h;
                double vp = matern_host(distance_host(a, b, sc.data(), (int)d), nu);
                for (int k = 0; k < d; ++k) sc[k] = rho - h;
                double vm = matern_host(distance_host(a, b, sc.data(), (int)d), nu);
                edv[t] = (vp - vm) / (2 * h);
            }
            GP_CUDA_CHECK(cudaMemcpy(w.edv, edv.data(), sizeof(double) * ne, cudaMemcpyHostToDevice));
        }
        place_extras_kernel<<<(ne + 255) / 256, 256, 0, s>>>(ne, w.ei, w.ej, w.ev, w.edv, w.eslot, indptr_dev, w.devcount,
                                                             indices_dev, data_dev, ddata_dev);
        GP_COUNT(1);
    }
    GP_LAUNCH_CHECK();
    if (sort_rows) return sort_rows_run(n, indptr_dev, indices_dev, data_dev, ddata_dev, w.overflow, s);
    GP_CUDA_CHECK(cudaStreamSynchronize(s));
    return 0;
}

}  // extern "C"


// =====================================================================================================================
// Direct generation of the ROW-BLOCKED operator (16-row blocks of the spatially ordered matrix, the SpMM's storage,
// gp_sparse_la.cu) without the CSR round trip: one warp per row block enumerates the candidate points of the cells its 16
// rows touch ONCE, classifies every (row, candidate) pair by the squared scaled distance, and keeps a candidate as a
// block-column when any of the 16 entries is in the pattern. PASS 0 counts block-columns (and the entries, = nnz);
// PASS 1 evaluates the kept entries in the reference's arithmetic (the same device functions as the CSR generator: same
// values, same pattern rule K > tau) and writes index + 16 values (zeros where an entry is outside the pattern) in the
// SpMM's fragment order - no memset, no hash build, no second read of a CSR.
// A pair inside the borderline band (|K - tau| <= 8 ulp: the host decides those in the CSR path) makes PASS 0 report it; the
// caller then takes the CSR path for this matrix.

// DIM > 0: the dimension is a compile-time constant (coordinates stay in registers, loops unrolled); DIM = 0: sp.d at run time
template <int DIM>
__device__ __forceinline__ double scaled_distance_dim(const double* a, const double* b, const SparseParams& sp) {
    const int dd = DIM > 0 ? DIM : sp.d;
    double s = 0.0;     // the reference's arithmetic: divide, square, sum in coordinate order, IEEE sqrt (_kernels.pyx:130-136)
#pragma unroll
    for (int k = 0; k < (DIM > 0 ? DIM : 8); ++k)
        if (k < dd) {
            const double t = (a[k] - b[k]) / sp.scale[k];
            s += t * t;
        }
    return sqrt(s);
}

template <int MODE, bool WITH_DK, int DIM>
__device__ __forceinline__ void block_entry(const SparseParams& sp, int i, const double* pi, int j, const double* pj, double* val,
                                            double* dval) {
    const double x = (i <= j) ? scaled_distance_dim<DIM>(pi, pj, sp) : scaled_distance_dim<DIM>(pj, pi, sp);
    if (WITH_DK) matern_value_drho<MODE>(x, sp.mp, val, dval);
    else { *val = matern_value<MODE>(x, sp.mp); *dval = 0.0; }
}

template <int MODE, int PASS, bool WITH_DK, int DIM>
__global__ void __launch_bounds__(128)
sparse_blocks_kernel(SparseParams sp, CellGrid g, const int* __restrict__ cell_start, const int* __restrict__ sorted_idx,
                     const double* __restrict__ sorted_pts, const double* __restrict__ pts, const int* __restrict__ order,
                     const int* __restrict__ inv_order, int row_first, int nrows, int* __restrict__ nblk,
                     unsigned long long* stats, const int64_t* __restrict__ bptr, int* __restrict__ bidx,
                     double* __restrict__ bvals, double* __restrict__ bdvals) {
    __shared__ double rowp_s[4][BCSR_ROWS][8];
    __shared__ int rowid_s[4][BCSR_ROWS];
    __shared__ int queue_s[4][64];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int rb = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (rb * BCSR_ROWS >= nrows) return;
    double (*rowp)[8] = rowp_s[w];
    int* rowid = rowid_s[w];
    int* queue = queue_s[w];
    // the block's rows: original point ids and coordinates
    int cmin[SMAXD] = {1 << 30, 1 << 30, 1 << 30}, cmax[SMAXD] = {-1, -1, -1};
    if (lane < BCSR_ROWS) {
        const int r = rb * BCSR_ROWS + lane;
        const int id = (r < nrows) ? order[row_first + r] : -1;
        rowid[lane] = id;
        double p[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        if (id >= 0)
            for (int k = 0; k < sp.d; ++k) p[k] = pts[(int64_t)id * sp.d + k];
        for (int k = 0; k < 8; ++k) rowp[lane][k] = p[k];
        if (id >= 0 && g.ncells > 1) {
            int c = cell_of_point(p, g);
            for (int k = g.d - 1; k >= 0; --k) { cmin[k] = cmax[k] = c % g.nc[k]; c /= g.nc[k]; }
        }
    }
#pragma unroll
    for (int k = 0; k < SMAXD; ++k)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            cmin[k] = min(cmin[k], __shfl_xor_sync(0xffffffffu, cmin[k], o));
            cmax[k] = max(cmax[k], __shfl_xor_sync(0xffffffffu, cmax[k], o));
        }
    __syncwarp();
    int nvalid = nrows - rb * BCSR_ROWS;
    if (nvalid > BCSR_ROWS) nvalid = BCSR_ROWS;
    // cell box of the block: the cells of its rows, one cell of margin (cell edge >= support radius)
    int blo[SMAXD] = {0, 0, 0}, bsz[SMAXD] = {1, 1, 1};
    int ncell_box = 1;
    if (g.ncells > 1) {
        for (int k = 0; k < g.d; ++k) {
            const int a = max(cmin[k] - 1, 0), b = min(cmax[k] + 1, g.nc[k] - 1);
            blo[k] = a;
            bsz[k] = b - a + 1;
            ncell_box *= bsz[k];
        }
    }
    const int64_t base = (PASS == 1) ? bptr[rb] : 0;
    int ncols = 0;                 // block-columns so far (warp-uniform)
    unsigned long long nent = 0;   // entries in the pattern (this lane)
    unsigned border = 0;
    int qn = 0;
    const int dd = DIM > 0 ? DIM : sp.d;
    constexpr int PD = DIM > 0 ? DIM : 8;
    // squared scaled distance for the quick classification (multiply by the reciprocal scale, as the CSR generator does)
    auto sq_dist = [&](const double* a, const double* b) {
        double s2 = 0.0;
#pragma unroll
        for (int k = 0; k < PD; ++k)
            if (k < dd) {
                const double t = (a[k] - b[k]) * sp.mp.inv_scale[k];
                s2 += t * t;
            }
        return s2;
    };

    // PASS 1: the lanes with act take one queued candidate each. First the keep decision (exactly PASS 0's: an entry is in
    // the pattern when it is certainly inside the support radius, or inside the margin with K > tau), then - the slot being
    // known - one loop over the 16 rows that evaluates the entries and stores them (zeros outside the pattern). The loop is
    // NOT unrolled: 16 inlined copies of the FP64 sqrt / exp sequences do not fit the instruction cache (first version:
    // 145 ms, issue slots 4 % busy, `no_instruction` stalls).
    auto emit = [&](int q, bool act) {
        bool kept = false;
        int j = -1;
        double pj[PD];
        if (act) {
            j = sorted_idx[q];
#pragma unroll
            for (int k = 0; k < PD; ++k)
                if (k < dd) pj[k] = sorted_pts[(int64_t)q * dd + k];
#pragma unroll 1
            for (int r = 0; r < nvalid && !kept; ++r) {
                const double s2 = sq_dist(rowp[r], pj);
                if (s2 < sp.r2_lo) kept = true;
                else if (!(s2 > sp.r2_hi)) {
                    double val, dval;
                    block_entry<MODE, false, DIM>(sp, rowid[r], rowp[r], j, pj, &val, &dval);
                    if (val > sp.tau) kept = true;
                }
            }
        }
        const unsigned m = __ballot_sync(0xffffffffu, kept);
        if (kept) {
            const int64_t slot = base + ncols + __popc(m & ((1u << lane) - 1u));
            bidx[slot] = inv_order[j];
            const int64_t o = bval_group(slot);
#pragma unroll 1
            for (int r = 0; r < BCSR_ROWS; ++r) {
                double val = 0.0, dval = 0.0;
                if (r < nvalid) {
                    const double s2 = sq_dist(rowp[r], pj);
                    if (!(s2 > sp.r2_hi)) {
                        block_entry<MODE, WITH_DK, DIM>(sp, rowid[r], rowp[r], j, pj, &val, &dval);
                        if (!(val > sp.tau)) { val = 0.0; dval = 0.0; }
                    }
                }
                bvals[bval_pos(o, r)] = val;
                if (WITH_DK) bdvals[bval_pos(o, r)] = dval;
            }
        }
        ncols += __popc(m);
    };

    for (int cb = 0; cb < ncell_box; ++cb) {
        int id = 0;
        if (g.ncells > 1) {
            int r = cb;
            int cc[SMAXD] = {0, 0, 0};
            for (int k = g.d - 1; k >= 0; --k) { cc[k] = blo[k] + r % bsz[k]; r /= bsz[k]; }
            for (int k = 0; k < g.d; ++k) id = id * g.nc[k] + cc[k];
        }
        const int s0 = cell_start[id], s1 = cell_start[id + 1];
        for (int q0 = s0; q0 < s1; q0 += 32) {
            const int q = q0 + lane;
            bool cand = false;       // PASS 0: the column is kept; PASS 1: some entry may be in the pattern
            if (q < s1) {
                double pj[PD];
#pragma unroll
                for (int k = 0; k < PD; ++k)
                    if (k < dd) pj[k] = sorted_pts[(int64_t)q * dd + k];
                int j = -1;
                for (int r = 0; r < nvalid; ++r) {
                    const double s2 = sq_dist(rowp[r], pj);
                    if (PASS == 1) {
                        if (!(s2 > sp.r2_hi)) { cand = true; break; }
                    } else {
                        if (s2 < sp.r2_lo) { cand = true; ++nent; }
                        else if (!(s2 > sp.r2_hi)) {      // inside the margin of the support radius: exact value decides
                            if (j < 0) j = sorted_idx[q];
                            double val, dval;
                            block_entry<MODE, false, DIM>(sp, rowid[r], rowp[r], j, pj, &val, &dval);
                            if (rowid[r] != j && fabs(val - sp.tau) <= sp.band) ++border;
                            if (val > sp.tau) { cand = true; ++nent; }
                        }
                    }
                }
            }
            const unsigned m = __ballot_sync(0xffffffffu, cand);
            if (PASS == 0) {
                ncols += __popc(m);
            } else {
                if (cand) queue[qn + __popc(m & ((1u << lane) - 1u))] = q;
                qn += __popc(m);
                __syncwarp();
                if (qn >= 32) {
                    const int qq = queue[lane];
                    const int rest = (lane < qn - 32) ? queue[32 + lane] : 0;
                    __syncwarp();
                    if (lane < qn - 32) queue[lane] = rest;
                    qn -= 32;
                    __syncwarp();
                    emit(qq, true);
                }
            }
        }
    }
    if (PASS == 1 && qn > 0) emit(lane < qn ? queue[lane] : 0, lane < qn);
    const int padded = (ncols + 3) & ~3;
    if (PASS == 0) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            nent += __shfl_xor_sync(0xffffffffu, nent, o);
            border += __shfl_xor_sync(0xffffffffu, border, o);
        }
        if (lane == 0) {
            nblk[rb] = padded;
            if (nent) atomicAdd(stats, nent);
            if (border) atomicAdd(stats + 1, (unsigned long long)border);
        }
    } else if (lane < padded - ncols) {          // pad the block to a multiple of 4 block-columns (zero values, a valid index)
        const int64_t slot = base + ncols + lane;
        bidx[slot] = inv_order[rowid[0]];
        const int64_t o = bval_group(slot);
#pragma unroll
        for (int r = 0; r < BCSR_ROWS; ++r) {
            bvals[bval_pos(o, r)] = 0.0;
            if (WITH_DK) bdvals[bval_pos(o, r)] = 0.0;
        }
    }
}

template <int MODE>
static void launch_blocks(int pass, bool with_dk, const SparseParams& sp, const CellGrid& g, const SparseWs& w, const double* pts,
                          const int* order, const int* inv_order, int row_first, int nrows, int* nblk, unsigned long long* stats,
                          const int64_t* bptr, int* bidx, double* bvals, double* bdvals, cudaStream_t s) {
    const int nrb = (nrows + BCSR_ROWS - 1) / BCSR_ROWS;
    const unsigned blocks = (unsigned)((nrb + 3) / 4);
#define GP_BLOCKS_LAUNCH(PASS, DK, DIM)                                                                                         \
    sparse_blocks_kernel<MODE, PASS, DK, DIM><<<blocks, 128, 0, s>>>(sp, g, w.cell_start, w.sorted_idx, w.sorted_pts, pts, order, \
                                                                       inv_order, row_first, nrows, nblk, stats, bptr, bidx, bvals, bdvals)
    if (sp.d == 2) {      // the common case (spatial data in the plane) with the dimension compiled in
        if (pass == 0) GP_BLOCKS_LAUNCH(0, false, 2);
        else if (with_dk) GP_BLOCKS_LAUNCH(1, true, 2);
        else GP_BLOCKS_LAUNCH(1, false, 2);
    } else {
        if (pass == 0) GP_BLOCKS_LAUNCH(0, false, 0);
        else if (with_dk) GP_BLOCKS_LAUNCH(1, true, 0);
        else GP_BLOCKS_LAUNCH(1, false, 0);
    }
#undef GP_BLOCKS_LAUNCH
    GP_COUNT(1);
}

// Per-dimension derivative streams of a built row-blocked operator: stream k holds dK/d scale[k] at the positions of bvals and
// 0 where bvals is 0 (K > tau > 0 on the pattern, so this is the pattern whichever path built the blocks). With u_k = Delta_k /
// scale[k], x = ||u|| and g(x) = -x K'(x) (matern_value_drho with inv_rho = 1): dK/d scale[k] = g(x) u_k^2 / (x^2 scale[k]),
// 0 at x = 0 - the formula of gp_loglik_dense_dscale. x is computed in scaled_distance_dim's arithmetic with block_entry's
// (i <= j) ordering; g(x) is evaluated once per entry and all d streams are written from it. One warp per row block, one
// lane per block-column; the 16-row loop is not unrolled, for the reason given at sparse_blocks_kernel's emit.
template <int MODE, int DIM>
__global__ void __launch_bounds__(128)
bcsr_dscale_kernel(const int64_t* __restrict__ bptr, const int* __restrict__ bidx, const double* __restrict__ bvals, int rows,
                   int row_first, int64_t stream_len, const int* __restrict__ order, const double* __restrict__ pts,
                   SparseParams sp, double* __restrict__ dvals) {
    __shared__ double rowp_s[4][BCSR_ROWS][8];
    __shared__ int rowid_s[4][BCSR_ROWS];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int rb = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (rb * BCSR_ROWS >= rows) return;
    const int dd = DIM > 0 ? DIM : sp.d;
    constexpr int PD = DIM > 0 ? DIM : 8;
    double (*rowp)[8] = rowp_s[w];
    int* rowid = rowid_s[w];
    if (lane < BCSR_ROWS) {
        const int r = rb * BCSR_ROWS + lane;
        const int id = (r < rows) ? order[row_first + r] : -1;
        rowid[lane] = id;
        for (int k = 0; k < 8; ++k) rowp[lane][k] = (id >= 0 && k < dd) ? pts[(int64_t)id * dd + k] : 0.0;
    }
    __syncwarp();
    const int64_t s1 = bptr[rb + 1];
    for (int64_t slot = bptr[rb] + lane; slot < s1; slot += 32) {
        const int j = order[bidx[slot]];
        double pj[PD];
#pragma unroll
        for (int k = 0; k < PD; ++k) pj[k] = (k < dd) ? pts[(int64_t)j * dd + k] : 0.0;
        const int64_t o = bval_group(slot);
#pragma unroll 1
        for (int r = 0; r < BCSR_ROWS; ++r) {
            const int64_t pos = bval_pos(o, r);
            double u2[PD];
            double s = 0.0, g = 0.0;
#pragma unroll
            for (int k = 0; k < PD; ++k) u2[k] = 0.0;
            if (bvals[pos] != 0.0) {
                const bool i_first = rowid[r] <= j;
#pragma unroll
                for (int k = 0; k < PD; ++k)
                    if (k < dd) {
                        const double t = (i_first ? rowp[r][k] - pj[k] : pj[k] - rowp[r][k]) / sp.scale[k];
                        u2[k] = t * t;
                        s += u2[k];
                    }
                double val;
                matern_value_drho<MODE>(sqrt(s), sp.mp, &val, &g);
            }
#pragma unroll
            for (int k = 0; k < PD; ++k)
                if (k < dd) dvals[k * stream_len + pos] = (s > 0.0) ? g * (u2[k] / s) * sp.mp.inv_scale[k] : 0.0;
        }
    }
}

extern "C" {

// Pass 0 of the direct row-blocked generation for the operator rows [row_first, row_last) (row_first a multiple of 16;
// the whole matrix: 0, n). order / inv_order: the spatial order of the points and its inverse (device int32).
// nblk_dev[rb] = block-columns of row block rb, padded to a multiple of 4. stats_host[0] = entries in the pattern (nnz of
// these rows), stats_host[1] = pairs inside the borderline band. Returns 3 when the direct path does not apply (borderline
// pairs present, or a threshold without a finite support radius): use gp_matern_sparse_count / fill + gp_bcsr_* then.
int gp_matern_blocks_count(const double* points, int64_t n, int64_t d, const double* scale_host, double nu, double tau, void* ws,
                           const int* order_dev, const int* inv_order_dev, int64_t row_first, int64_t row_last, int* nblk_dev,
                           int64_t* stats_host, void* stream) {
    if (!points || !scale_host || !ws || !order_dev || !inv_order_dev || !nblk_dev || !stats_host || n <= 0 || d <= 0 || d > 8 ||
        n > INT32_MAX || row_first < 0 || row_last <= row_first || row_last > n || (row_first % BCSR_ROWS))
        return -1;
    MaternParams mp;
    int mode;
    if (int rc = matern_params(scale_host, d, nu, false, &mp, &mode)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    SparseWs w = carve_sparse(ws, n, d);
    SparseParams sp;
    CellGrid g;
    if (int rc = sparse_prepare(points, n, d, scale_host, nu, tau, mp, w, s, &sp, &g)) return rc;
    stats_host[0] = stats_host[1] = 0;
    if (!sp.quick) return 3;
    unsigned long long* stats = w.bbox_keys + 16;
    GP_CUDA_CHECK(cudaMemsetAsync(stats, 0, 2 * sizeof(unsigned long long), s));
    with_matern_mode(mode, [&](auto tag) {
        launch_blocks<decltype(tag)::value>(0, false, sp, g, w, points, order_dev, inv_order_dev, (int)row_first,
                                            (int)(row_last - row_first), nblk_dev, stats, nullptr, nullptr, nullptr, nullptr, s);
    });
    GP_LAUNCH_CHECK();
    unsigned long long h[2] = {0, 0};
    GP_CUDA_CHECK(cudaMemcpyAsync(h, stats, sizeof(h), cudaMemcpyDeviceToHost, s));
    GP_CUDA_CHECK(cudaStreamSynchronize(s));
    stats_host[0] = (int64_t)h[0];
    stats_host[1] = (int64_t)h[1];
    return h[1] ? 3 : 0;
}

// Pass 1: after the exclusive scan of nblk (gp_scan_counts) and the allocation of bidx (total), bvals [, bdvals] (16 total).
int gp_matern_blocks_fill(const double* points, int64_t n, int64_t d, const double* scale_host, double nu, double tau, void* ws,
                          const int* order_dev, const int* inv_order_dev, int64_t row_first, int64_t row_last,
                          const int64_t* bptr_dev, int* bidx_dev, double* bvals_dev, double* bdvals_dev, void* stream) {
    if (!points || !scale_host || !ws || !order_dev || !inv_order_dev || !bptr_dev || !bidx_dev || !bvals_dev || n <= 0 ||
        d <= 0 || d > 8 || row_first < 0 || row_last <= row_first || row_last > n || (row_first % BCSR_ROWS))
        return -1;
    MaternParams mp;
    int mode;
    if (int rc = matern_params(scale_host, d, nu, bdvals_dev != nullptr, &mp, &mode)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    SparseWs w = carve_sparse(ws, n, d);
    double bb[16];
    GP_CUDA_CHECK(cudaMemcpyAsync(bb, w.bbox, sizeof(bb), cudaMemcpyDeviceToHost, s));      // left by the count call
    GP_CUDA_CHECK(cudaStreamSynchronize(s));
    SparseParams sp;
    CellGrid g;
    make_params(n, d, scale_host, nu, tau, mp, bb, bb + 8, &sp, &g);
    with_matern_mode(mode, [&](auto tag) {
        launch_blocks<decltype(tag)::value>(1, bdvals_dev != nullptr, sp, g, w, points, order_dev, inv_order_dev, (int)row_first,
                                            (int)(row_last - row_first), nullptr, nullptr, bptr_dev, bidx_dev, bvals_dev,
                                            bdvals_dev, s);
    });
    GP_LAUNCH_CHECK();
    return 0;
}

// d streams of 16 * nblocks doubles (stream k at dvals_dev + 16 * nblocks * k): dK/d scale[k] on the row blocks of the
// operator rows [row_first, row_first + rows) (bidx: operator positions, before gp_slab_encode_columns). Any scale with
// positive entries is accepted (never -4).
int gp_bcsr_dscale_fill(const int64_t* bptr_dev, const int* bidx_dev, const double* bvals_dev, int64_t nblocks, int64_t row_first,
                        int64_t rows, const int* order_dev, const double* points, int64_t n, int64_t d, const double* scale_host,
                        double nu, double* dvals_dev, void* stream) {
    if (!bptr_dev || !bidx_dev || !bvals_dev || !order_dev || !points || !scale_host || !dvals_dev || d < 1 || d > 8 || n <= 0 ||
        n > INT32_MAX || nblocks < 0 || row_first < 0 || (row_first % BCSR_ROWS) || rows <= 0 || row_first + rows > n)
        return -1;
    SparseParams sp{};
    int mode;
    if (int rc = matern_params(scale_host, d, nu, false, &sp.mp, &mode)) return rc;
    sp.mp.inv_rho = 1.0;
    sp.d = (int)d;
    for (int k = 0; k < d; ++k) sp.scale[k] = scale_host[k];
    if (nblocks == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    const unsigned blocks = (unsigned)(((rows + BCSR_ROWS - 1) / BCSR_ROWS + 3) / 4);
    with_matern_mode(mode, [&](auto tag) {
        constexpr int MODE = decltype(tag)::value;
        if (d == 2)
            bcsr_dscale_kernel<MODE, 2><<<blocks, 128, 0, s>>>(bptr_dev, bidx_dev, bvals_dev, (int)rows, (int)row_first,
                                                               16 * nblocks, order_dev, points, sp, dvals_dev);
        else
            bcsr_dscale_kernel<MODE, 0><<<blocks, 128, 0, s>>>(bptr_dev, bidx_dev, bvals_dev, (int)rows, (int)row_first,
                                                               16 * nblocks, order_dev, points, sp, dvals_dev);
    });
    GP_COUNT(1);
    GP_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
