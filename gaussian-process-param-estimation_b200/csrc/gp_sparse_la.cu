// Sparse operator K + eta*I (plain CSR, or the row-blocked form whose SpMM runs on the FP64 tensor cores) on blocks of
// probe / right-hand-side columns: SpMM, batched Lanczos (stochastic
// Lanczos quadrature for logdet and trace of the inverse) and batched CG (solves, Hutchinson tr(Kn^-1 dK)).
// Replaces what the reference reaches through imate's 'slq' / 'hutchinson' methods and scipy.sparse.linalg.cg
// (gaussian_proc/_mixed_correlation/mixed_correlation.py:193-209,263-268; _linear_solver.py:49-68, tol = 1e-6).
// All column blocks are n x B row-major with B in {1,2,4,8,16,32}; HBM-bound: 12 nnz + 4 (n+1) + 16 n B bytes / SpMM.
#include "../../include/gpgp.h"
#include "gp_common.cuh"
#include "gp_internal.h"
#include "gp_peer.cuh"

namespace gp {

constexpr int RED_PARTS = 592;  // CTAs of the column reductions (4 per SM)

// ---- Y = (K + eta I) X, one warp per row; lane = (q, c): q-th nonzero of the current group, column c ---------
template <int B>
__global__ void __launch_bounds__(256)
csr_spmm_kernel(const int* __restrict__ indptr, const int* __restrict__ indices, const double* __restrict__ data, int n,
                double eta, const double* __restrict__ X, const double* __restrict__ scale, double* __restrict__ Y) {
    constexpr int NQ = 32 / B;
    const int lane = threadIdx.x & 31;
    const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= n) return;
    const int q = lane / B, c = lane % B;
    const int s0 = indptr[row], s1 = indptr[row + 1];
    double acc = 0.0;
    for (int p = s0 + q; p < s1; p += NQ) acc += data[p] * X[(int64_t)indices[p] * B + c];
#pragma unroll
    for (int o = B; o < 32; o <<= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (q == 0) Y[(int64_t)row * B + c] = (acc + eta * X[(int64_t)row * B + c]) * (scale ? scale[c] : 1.0);
}

// ---- column reductions: partial[cta][c] = sum over the CTA's elements of column c --------------------------------
// mode 0: x*y   mode 1: (lanczos) u_next = w - a u - b u_prev (Z; may be u_prev's buffer), accumulate u_next^2
// mode 2: (cg) x += a p, r -= a ap, accumulate r*r
template <int MODE>
__global__ void __launch_bounds__(256)
col_fused_kernel(int64_t total, int B, const double* __restrict__ X, const double* Y, double* W,
                 double* Z, const double* __restrict__ a, const double* __restrict__ b, double* partial,
                 double* Z2 = nullptr) {
    __shared__ double red[256];
    const int64_t stride = (int64_t)gridDim.x * 256;  // multiple of 32 >= B: a thread stays in one column
    const int c = threadIdx.x % B;
    double acc = 0.0;
    double ac = (MODE != 0) ? a[c] : 0.0, bc = (MODE == 1) ? b[c] : 0.0;
    for (int64_t idx = (int64_t)blockIdx.x * 256 + threadIdx.x; idx < total; idx += stride) {
        if (MODE == 0) {
            acc += X[idx] * Y[idx];
        } else if (MODE == 1) {
            double w = W[idx] - ac * X[idx] - bc * Y[idx];   // X = u_j, Y = u_{j-1}, Z = u_{j+1} (may alias Y)
            Z[idx] = w;
            if (Z2) Z2[idx] = w;                              // row-slab operator: the copy the peers' SpMM gathers from
            acc += w * w;
        } else {
            Z[idx] += ac * X[idx];                            // Z = solution, X = p
            double r = W[idx] - ac * Y[idx];                  // W = residual, Y = A p
            W[idx] = r;
            acc += r * r;
        }
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    // threads t, t+B, t+2B, ... share column t % B (256 % B == 0)
    if (threadIdx.x < B) {
        double s = 0.0;
        for (int t = threadIdx.x; t < 256; t += B) s += red[t];
        partial[(int64_t)blockIdx.x * B + threadIdx.x] = s;
    }
}

// first stage for long partial lists (the SpMM epilogue leaves one row per CTA): CTA b sums rows [256 b, 256 b + 256)
__global__ void __launch_bounds__(256)
col_partial_reduce_kernel(const double* __restrict__ partial, int nparts, int B, double* __restrict__ out) {
    __shared__ double red[256];
    const int c = threadIdx.x % B, sl = threadIdx.x / B, nsl = 256 / B;
    const int i0 = blockIdx.x * 256, i1 = min(nparts, i0 + 256);
    double s = 0.0;
#pragma unroll 4
    for (int i = i0 + sl; i < i1; i += nsl) s += partial[(int64_t)i * B + c];
    red[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x >= B) return;
    s = 0.0;
    for (int k = 0; k < nsl; ++k) s += red[k * B + c];
    out[(int64_t)blockIdx.x * B + c] = s;
}

// final stage + the scalar recurrences: 256 threads sum the partials in a fixed order (reproducible), then one thread
// per column applies the recurrence.
// op 0: out = sum
// op 1 (lanczos alpha): alpha = s_cur * sum -> out; s2 = a1 = alpha * s_cur; s3 = b1 = beta_prev * s_prev
//                       (sc layout, 32 doubles each: s1 = {s_cur, s_prev, beta_prev} at s1, s1+32, s1+64)
// op 2 (lanczos beta):  beta = sqrt(sum) -> out; beta_prev = beta; s_prev = s_cur; s_cur = beta > tiny ? 1/beta : 0
// op 3 (cg pAp):        alpha[c] = active ? rr/sum : 0
// op 4 (cg rr_new):     beta[c] = active ? sum/rr : 0; rr = sum; active &= rr > tol2*bb
__global__ void __launch_bounds__(256)
col_final_kernel(const double* __restrict__ partial, int nparts, int B, int op, double* out, double* s1, double* s2,
                 double* s3, double tol2, const __grid_constant__ PeerComm pc) {
    __shared__ double red[256];
    const int c = threadIdx.x % B, sl = threadIdx.x / B, nsl = 256 / B;
    double s = 0.0;
    for (int i = sl; i < nparts; i += nsl) s += partial[(int64_t)i * B + c];
    red[threadIdx.x] = s;
    __syncthreads();
    s = 0.0;
    if (threadIdx.x < B)
        for (int k = 0; k < nsl; ++k) s += red[k * B + c];
    s = peer_block_sum(pc, s, B);      // row-slab operator: the sum over the ranks' slabs (no-op on one GPU)
    if (threadIdx.x >= B) return;
    if (op == 0) {
        out[c] = s;
    } else if (op == 1) {
        double* s_cur = s1; double* s_prev = s1 + 32; double* beta_prev = s1 + 64;
        const double al = s_cur[c] * s;
        out[c] = al;
        s2[c] = al * s_cur[c];
        s3[c] = beta_prev[c] * s_prev[c];
    } else if (op == 2) {
        double* s_cur = s1; double* s_prev = s1 + 32; double* beta_prev = s1 + 64;
        const double bt = sqrt(s);
        out[c] = bt;
        beta_prev[c] = bt;
        s_prev[c] = s_cur[c];
        s_cur[c] = (bt > 1e-300) ? 1.0 / bt : 0.0;
    } else if (op == 3) {
        // s1 = rr, s2 = active flag (1/0), s3 = breakdown flag, out = alpha
        if (s2[c] != 0.0 && !(s > 0.0)) { s3[0] = 1.0; s2[c] = 0.0; }   // p^T A p <= 0: A is not positive definite
        out[c] = (s2[c] != 0.0) ? s1[c] / s : 0.0;
    } else {
        // s1 = rr (updated), s2 = active, s3 = bb, out = beta
        double rr_old = s1[c];
        out[c] = (s2[c] != 0.0 && rr_old != 0.0) ? s / rr_old : 0.0;
        s1[c] = s;
        if (!(s > tol2 * s3[c])) s2[c] = 0.0;
    }
}

// p = r + beta p
__global__ void cg_direction_kernel(int64_t total, int B, const double* __restrict__ R, const double* __restrict__ beta, double* P) {
    int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    P[idx] = R[idx] + beta[idx % B] * P[idx];
}

// Rademacher probes from a counter-based hash of (seed, probe id, row): independent of batching and rank count
__global__ void rademacher_kernel(int64_t n, int B, uint64_t seed, int64_t probe0, const int* __restrict__ row_map, double* V) {
    int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n * B) return;
    int64_t r = idx / B;
    uint64_t row = (uint64_t)(row_map ? row_map[r] : r), pid = (uint64_t)(probe0 + idx % B);
    uint64_t z = seed * 0x9E3779B97F4A7C15ull + pid * 0xBF58476D1CE4E5B9ull + row * 0x94D049BB133111EBull + 0x2545F4914F6CDD1Dull;
    z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ull;
    z ^= z >> 27; z *= 0x94D049BB133111EBull;
    z ^= z >> 31;
    V[idx] = (z & 1ull) ? 1.0 : -1.0;
}

// ---- row-blocked operator: BCSR_ROWS = 16 consecutive rows share one column list (16 x 1 blocks, zero filled) ----------
// Rows that are neighbours in a spatially sorted order have almost the same pattern, so one gathered row of X serves
// 16 rows of K: gather traffic (the L1/L2-bound part of a multi-column SpMM) drops ~16-fold and the column index is
// amortised over 16 values. Block-columns of a row block: [all columns of row 0][columns of row 1 not in row 0]...
// (each segment in the source row's order); any order is valid for the product.
__device__ __forceinline__ int find_col(const int* __restrict__ row, int len, int c) {
    int lo = 0, hi = len;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (row[mid] < c) lo = mid + 1; else hi = mid;
    }
    return (lo < len && row[lo] == c) ? lo : -1;
}

// One warp per row block. PASS 0: nblk[rb] = number of distinct columns rounded up to a multiple of 4 (the k extent of
// one DMMA); PASS 1: fill (bidx, bvals[, bdvals]; the value arrays are zeroed by the caller); padding block-columns
// repeat the block's first column with zeros. New row r = old row order[r]; new column = inv_order[old column]; the
// source CSR must have sorted rows.
// Columns get their block-column slot in order of first appearance (row 0's entries, then the new ones of row 1, ...).
// Fast path: a per-warp open-addressing hash table (column -> slot) in shared memory, one probe sequence per entry.
// If a block has more than HMAX distinct columns the warp redoes it with binary searches in the (sorted) source rows:
// the same layout, so both paths write identical output.
constexpr int HCAP = 2048, HMAX = 1536;

template <int PASS>
__device__ __forceinline__ int bcsr_block_search(int lane, int rb, const int* s, const int* len, const int* __restrict__ inv_order,
                                                 const int* __restrict__ indices, const double* __restrict__ data,
                                                 const double* __restrict__ ddata, int64_t base, int* bidx, double* bvals,
                                                 double* bdvals) {
    int running = 0;
#pragma unroll
    for (int k = 0; k < BCSR_ROWS; ++k) {
        for (int t0 = 0; t0 < len[k]; t0 += 32) {
            const int t = t0 + lane;
            const bool valid = t < len[k];
            const int c = valid ? indices[s[k] + t] : -1;
            bool owned = valid;
#pragma unroll
            for (int kk = 0; kk < k; ++kk)
                if (owned && find_col(indices + s[kk], len[kk], c) >= 0) owned = false;
            const unsigned m = __ballot_sync(0xffffffffu, owned);
            if (PASS == 1 && owned) {
                const int64_t slot = base + running + __popc(m & ((1u << lane) - 1u));
                bidx[slot] = inv_order ? inv_order[c] : c;
                double v[BCSR_ROWS], dv[BCSR_ROWS];
#pragma unroll
                for (int kk = 0; kk < BCSR_ROWS; ++kk) { v[kk] = 0.0; dv[kk] = 0.0; }
                v[k] = data[s[k] + t];
                if (ddata) dv[k] = ddata[s[k] + t];
#pragma unroll
                for (int kk = k + 1; kk < BCSR_ROWS; ++kk) {
                    int pos = find_col(indices + s[kk], len[kk], c);
                    if (pos >= 0) {
                        v[kk] = data[s[kk] + pos];
                        if (ddata) dv[kk] = ddata[s[kk] + pos];
                    }
                }
#pragma unroll
                for (int kk = 0; kk < BCSR_ROWS; ++kk) bvals[bval_pos(bval_group(slot), kk)] = v[kk];
                if (ddata) {
#pragma unroll
                    for (int kk = 0; kk < BCSR_ROWS; ++kk) bdvals[bval_pos(bval_group(slot), kk)] = dv[kk];
                }
            }
            running += __popc(m);
        }
    }
    return running;
}

template <int PASS>
__global__ void __launch_bounds__(128)
bcsr_build_kernel(int n, const int* __restrict__ order, const int* __restrict__ inv_order, const int* __restrict__ indptr,
                  const int* __restrict__ indices, const double* __restrict__ data, const double* __restrict__ ddata,
                  int* nblk, const int64_t* __restrict__ bptr, int* bidx, double* bvals, double* bdvals, int* searched) {
    __shared__ int hkey[4][HCAP];
    __shared__ unsigned short hslot[4][HCAP];      // slots < HMAX + 32
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int rb = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (rb * BCSR_ROWS >= n) return;
    int* hk = hkey[w];
    unsigned short* hs = hslot[w];
    for (int i = lane; i < HCAP; i += 32) hk[i] = -1;
    int s[BCSR_ROWS], len[BCSR_ROWS];
#pragma unroll
    for (int k = 0; k < BCSR_ROWS; ++k) {
        int r = rb * BCSR_ROWS + k;
        if (r < n) {
            int o = order ? order[r] : r;
            s[k] = indptr[o];
            len[k] = indptr[o + 1] - s[k];
        } else {
            s[k] = 0;
            len[k] = 0;
        }
    }
    const int64_t base = (PASS == 1) ? bptr[rb] : 0;
    __syncwarp();
    int running = 0;
    bool overflow = false;
#pragma unroll
    for (int k = 0; k < BCSR_ROWS; ++k) {
        for (int t0 = 0; t0 < len[k] && !overflow; t0 += 32) {
            const int t = t0 + lane;
            const bool valid = t < len[k];
            const int c = valid ? indices[s[k] + t] : -1;
            int slot = -1;
            bool isnew = false;
            unsigned h = ((unsigned)c * 2654435761u) >> 21;      // 11 bits = HCAP
            if (valid) {
                while (true) {
                    const int kk = hk[h];
                    if (kk == c) { slot = hs[h]; break; }
                    if (kk == -1) { isnew = true; break; }
                    h = (h + 1) & (HCAP - 1);
                }
            }
            const unsigned m = __ballot_sync(0xffffffffu, isnew);
            if (isnew) {
                slot = running + __popc(m & ((1u << lane) - 1u));
                while (true) {      // claim the first free cell from h on (other lanes insert other columns concurrently)
                    const int old = atomicCAS(&hk[h], -1, c);
                    if (old == -1) { hs[h] = (unsigned short)slot; break; }
                    h = (h + 1) & (HCAP - 1);
                }
            }
            running += __popc(m);
            __syncwarp();
            if (running > HMAX) overflow = true;
            if (PASS == 1 && valid && !overflow) {
                const int64_t o = bval_pos(bval_group(base + slot), k);
                bvals[o] = data[s[k] + t];
                if (ddata) bdvals[o] = ddata[s[k] + t];
                if (isnew) bidx[base + slot] = inv_order ? inv_order[c] : c;
            }
        }
    }
    if (overflow) {
        if (searched && lane == 0) atomicExch(searched, 1);
        if (PASS == 1) {      // clear what the hash path wrote, then redo the block by searching
            const int64_t cnt = (bptr[rb + 1] - base) * BCSR_ROWS;
            for (int64_t i = lane; i < cnt; i += 32) {
                bvals[base * BCSR_ROWS + i] = 0.0;
                if (ddata) bdvals[base * BCSR_ROWS + i] = 0.0;
            }
            __syncwarp();
        }
        running = bcsr_block_search<PASS>(lane, rb, s, len, inv_order, indices, data, ddata, base, bidx, bvals, bdvals);
    }
    const int padded = (running + 3) & ~3;
    if (PASS == 0 && lane == 0) nblk[rb] = padded;
    if (PASS == 1 && lane < padded - running) {
        const int64_t slot = base + running + lane;
        const int c0 = (len[0] > 0) ? indices[s[0]] : (order ? order[rb * BCSR_ROWS] : rb * BCSR_ROWS);
        bidx[slot] = inv_order ? inv_order[c0] : c0;
#pragma unroll
        for (int kk = 0; kk < BCSR_ROWS; ++kk) {
            bvals[bval_pos(bval_group(slot), kk)] = 0.0;
            if (ddata) bdvals[bval_pos(bval_group(slot), kk)] = 0.0;
        }
    }
}

// Y = (K + eta I) X on the row-blocked operator with FP64 tensor-core MMAs. One warp per row block. Four
// block-columns form one DMMA.8x8x4: A (8 rows x 4 block-columns) is exactly 256 contiguous bytes of the value stream
// (one 8-byte load per lane, no broadcast), B (4 x 8) holds the four gathered rows of X restricted to 8 columns, and the
// 8 x 8 accumulator stays in two registers per lane for the whole row block - no cross-lane reduction. For B = 16 / 32
// the 2 / 4 MMAs of a step share A; their column sets are interleaved (tile j owns columns j, j + NT, ...) so that a
// lane's B operands are NT consecutive doubles of one X row (one 16-byte load for B = 16) and its results are 2 NT
// consecutive columns of one Y row. Index and values are streamed past L1 (ld.global.cs): L1 is kept for X.
// Epilogue: Y = scale[c] (A X + eta X) (scale optional) and, with DOT, partial[cta][c] = sum over the CTA's 64 rows
// of X[i][c] Y[i][c] (fixed order) - the Lanczos alpha / CG p^T A p reduction without another pass over the vectors.
// A 16-row block is H = 2 fragments: two A fragments and two MMAs per gathered B fragment.
// PEER (row-slab operator on several GPUs): the rows of this rank's slab; a block-column index carries the owner rank in its
// top 4 bits and the row within the owner's slab below (gp_slab_encode_columns), and the gather goes to the owner's copy of
// the exchange vector - local HBM for the own slab, a load over NVLink from the mapped arena of a peer for the halo.
constexpr int PEER_SHIFT = 28;
constexpr int SPMM_MINB = 4;      // CTAs per SM (launch bounds)
constexpr int SPMM_U = 4;         // steps in flight per warp for B <= 16
template <int B, bool DOT, bool PEER = false>
__global__ void __launch_bounds__(256, SPMM_MINB)
bcsr8_spmm_dmma_kernel(const int64_t* __restrict__ bptr, const int* __restrict__ bidx, const double* __restrict__ bvals, int n,
                       double eta, const double* __restrict__ X, const double* __restrict__ scale, double* __restrict__ Y,
                       double* __restrict__ partial, const __grid_constant__ PeerVec pv) {
    constexpr int H = BCSR_ROWS / 8;           // 8-row A fragments per row block
    constexpr int NT = (B >= 8) ? B / 8 : 1;   // 8-column MMA tiles per step
    const int lane = threadIdx.x & 31;
    const int g = lane >> 2, t = lane & 3;     // DMMA.8x8x4 fragments: A[g][t], B[t][g], D[g][2t .. 2t+1]
    // PEER: the CTAs alternate between the two ends of the slab, where the halo rows (NVLink latency) are - the slow row
    // blocks start first and the interior ones fill the tail
    const int bx = PEER ? ((blockIdx.x & 1) ? (int)gridDim.x - 1 - (int)(blockIdx.x >> 1) : (int)(blockIdx.x >> 1)) : (int)blockIdx.x;
    const int rb = (bx * blockDim.x + threadIdx.x) >> 5;
    const bool live = rb * BCSR_ROWS < n;
    if (!DOT && !live) return;
    const int64_t p0 = live ? bptr[rb] : 0, p1 = live ? bptr[rb + 1] : 0;   // p1 - p0 is a multiple of 4
    double acc[H][NT][2];
#pragma unroll
    for (int h = 0; h < H; ++h)
#pragma unroll
        for (int j = 0; j < NT; ++j) acc[h][j][0] = acc[h][j][1] = 0.0;
    const bool colok = (B >= 8) || (g < B);
    const int coff = (B >= 8) ? g * NT : (colok ? g : 0);
    const double* aptr = bvals + lane;          // A fragment order: element (row g, block-column t) at 4 g + t = lane
    // B = 16: a gathered X row is 128 bytes = one L1 line. In the fragment layout (lane 4 g + t holds row t, columns 2 g,
    // 2 g + 1) a quarter-warp - the unit a 16-byte load is served in - touches FOUR rows: 16 line accesses (wavefronts) per
    // load instruction, and the L1 data pipe, not HBM, bounds the kernel (ncu, profiles/r01_spmm_ncu_summary.md).
    auto load_x = [&](int col, double* x) {
        const double* xr;
        if (PEER) {
            // Interior row blocks (almost all of them: the halo is ~1 % of the block-columns) only reference this rank's
            // rows: one warp vote keeps them on the single-GPU addressing (X = this rank's copy); the pointer-table lookup -
            // a dependent constant-bank load in front of every gather - is taken only by steps that touch a peer.
            const unsigned owner = (unsigned)col >> PEER_SHIFT;
            const int64_t local = (int64_t)(col & ((1 << PEER_SHIFT) - 1));
            if (__any_sync(0xffffffffu, owner != (unsigned)pv.rank)) xr = pv.base[owner] + local * B + coff;
            else xr = X + local * B + coff;
        } else {
            xr = X + (int64_t)col * B + coff;
        }
        if (NT == 1) {
            x[0] = colok ? *xr : 0.0;
        } else {
#pragma unroll
            for (int j = 0; j < NT; j += 2) {
                double2 v = *reinterpret_cast<const double2*>(xr + j);
                x[j] = v.x;
                x[j + (NT > 1 ? 1 : 0)] = v.y;
            }
        }
    };
    constexpr int U = (NT <= 2) ? SPMM_U : 2;          // steps in flight per warp: all loads of U steps are issued before their MMAs
    int64_t p = p0;
    for (; p + 4 * U <= p1; p += 4 * U) {
        int col[U];
        double a[U][H], x[U][NT];
#pragma unroll
        for (int u = 0; u < U; ++u) col[u] = __ldcs(bidx + p + 4 * u + t);
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int h = 0; h < H; ++h) a[u][h] = __ldcs(aptr + (p + 4 * u) * BCSR_ROWS + 32 * h);
#pragma unroll
        for (int u = 0; u < U; ++u) load_x(col[u], x[u]);
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int h = 0; h < H; ++h)
#pragma unroll
                for (int j = 0; j < NT; ++j) dmma884(acc[h][j][0], acc[h][j][1], a[u][h], x[u][j]);
    }
    for (; p < p1; p += 4) {
        const int col = __ldcs(bidx + p + t);
        double a[H], x[NT];
#pragma unroll
        for (int h = 0; h < H; ++h) a[h] = __ldcs(aptr + p * BCSR_ROWS + 32 * h);
        load_x(col, x);
#pragma unroll
        for (int h = 0; h < H; ++h)
#pragma unroll
            for (int j = 0; j < NT; ++j) dmma884(acc[h][j][0], acc[h][j][1], a[h], x[j]);
    }
    constexpr int NC = (B >= 8) ? 2 * NT : 2;               // result columns of this lane, from column c0
    const int c0 = (B >= 8) ? 2 * t * NT : 2 * t;
    double dsum[NC];
#pragma unroll
    for (int k = 0; k < NC; ++k) dsum[k] = 0.0;
#pragma unroll
    for (int h = 0; h < H; ++h) {
        const int row = rb * BCSR_ROWS + h * 8 + g;
        if (live && row < n) {
#pragma unroll
            for (int k = 0; k < NC; ++k) {
                // tile j, fragment column cc in {2t, 2t+1} is the true column cc * NT + j: k = i * NT + j
                const int i = (B >= 8) ? k / NT : k, j = (B >= 8) ? k % NT : 0;
                if (B >= 8 || c0 + k < B) {
                    const int64_t o = (int64_t)row * B + c0 + k;
                    const double xv = X[o];
                    double y = acc[h][j][i] + eta * xv;
                    if (scale) y *= scale[c0 + k];
                    Y[o] = y;
                    if (DOT) dsum[k] += xv * y;
                }
            }
        }
    }
    if (DOT) {
        __shared__ double red[8][32];
#pragma unroll
        for (int k = 0; k < NC; ++k) {
            double v = dsum[k];
            v += __shfl_xor_sync(0xffffffffu, v, 4);
            v += __shfl_xor_sync(0xffffffffu, v, 8);
            v += __shfl_xor_sync(0xffffffffu, v, 16);
            if (g == 0 && (B >= 8 || c0 + k < B)) red[threadIdx.x >> 5][c0 + k] = v;
        }
        __syncthreads();
        if (threadIdx.x < B) {
            double v = 0.0;
#pragma unroll
            for (int w = 0; w < 8; ++w) v += red[w][threadIdx.x];
            partial[(int64_t)blockIdx.x * B + threadIdx.x] = v;
        }
    }
}

// the operator a Krylov routine works on: plain CSR or the row-blocked form
struct SparseOp {
    bool blocked;          // false: CSR (ptr32, idx, val); true: row-blocked (ptr64, idx, val)
    const int* ptr32;
    const int64_t* ptr64;
    const int* idx;
    const double* val;
    int n;
};

// CTAs of the row-blocked SpMM (8 warps = 8 row blocks each) = rows of its dot partials
static int bcsr_parts(int n) { return ((n + BCSR_ROWS - 1) / BCSR_ROWS + 7) / 8; }

template <int B>
static void bcsr8_spmm_launch_b(const SparseOp& A, double eta, const double* X, const double* scale, double* Y,
                                double* partial, cudaStream_t s, const PeerVec* pvp) {
    const int blocks = bcsr_parts(A.n);
    PeerVec pv = {};
    if (pvp) pv = *pvp;
#define SPMM_LAUNCH(DOT, PEER) \
    bcsr8_spmm_dmma_kernel<B, DOT, PEER><<<blocks, 256, 0, s>>>(A.ptr64, A.idx, A.val, A.n, eta, X, scale, Y, partial, pv)
    if (pvp) {       // row-slab operator
        if (partial) SPMM_LAUNCH(true, true); else SPMM_LAUNCH(false, true);
    } else {
        if (partial) SPMM_LAUNCH(true, false); else SPMM_LAUNCH(false, false);
    }
#undef SPMM_LAUNCH
}

// Y = scale (.) ((A + eta I) X); with `partial` also the per-column partial sums of X (.) Y: *nparts rows of B doubles
// `pv` (row-slab operator): X is this rank's copy of the exchange vector (epilogue rows), the gathers go through pv
static int spmm(const SparseOp& A, double eta, const double* X, int B, double* Y, cudaStream_t s,
                const double* scale = nullptr, double* partial = nullptr, int* nparts = nullptr, const PeerVec* pv = nullptr) {
    const int n = A.n;
    if (!A.blocked) {
        int blocks = (int)(((int64_t)n * 32 + 255) / 256);
        switch (B) {
            case 1: csr_spmm_kernel<1><<<blocks, 256, 0, s>>>(A.ptr32, A.idx, A.val, n, eta, X, scale, Y); break;
            case 2: csr_spmm_kernel<2><<<blocks, 256, 0, s>>>(A.ptr32, A.idx, A.val, n, eta, X, scale, Y); break;
            case 4: csr_spmm_kernel<4><<<blocks, 256, 0, s>>>(A.ptr32, A.idx, A.val, n, eta, X, scale, Y); break;
            case 8: csr_spmm_kernel<8><<<blocks, 256, 0, s>>>(A.ptr32, A.idx, A.val, n, eta, X, scale, Y); break;
            case 16: csr_spmm_kernel<16><<<blocks, 256, 0, s>>>(A.ptr32, A.idx, A.val, n, eta, X, scale, Y); break;
            case 32: csr_spmm_kernel<32><<<blocks, 256, 0, s>>>(A.ptr32, A.idx, A.val, n, eta, X, scale, Y); break;
            default: return -2;
        }
        GP_COUNT(1);
        if (partial) {   // plain CSR keeps the separate reduction pass
            col_fused_kernel<0><<<RED_PARTS, 256, 0, s>>>((int64_t)n * B, B, X, Y, nullptr, nullptr, nullptr, nullptr, partial);
            *nparts = RED_PARTS;
            GP_COUNT(1);
        }
    } else {
        switch (B) {
            case 1: bcsr8_spmm_launch_b<1>(A, eta, X, scale, Y, partial, s, pv); break;
            case 2: bcsr8_spmm_launch_b<2>(A, eta, X, scale, Y, partial, s, pv); break;
            case 4: bcsr8_spmm_launch_b<4>(A, eta, X, scale, Y, partial, s, pv); break;
            case 8: bcsr8_spmm_launch_b<8>(A, eta, X, scale, Y, partial, s, pv); break;
            case 16: bcsr8_spmm_launch_b<16>(A, eta, X, scale, Y, partial, s, pv); break;
            case 32: bcsr8_spmm_launch_b<32>(A, eta, X, scale, Y, partial, s, pv); break;
            default: return -2;
        }
        if (partial) *nparts = bcsr_parts(n);
        GP_COUNT(1);
    }
    GP_LAUNCH_CHECK();
    return 0;
}

// partial (nparts x B) -> scalar recurrence `op`; long lists go through col_partial_reduce_kernel into `scratch`
// `px` (row-slab operator): the sums are all-reduced over the ranks inside the final kernel (peer_block_sum)
static void col_final(const double* partial, int nparts, int B, int op, double* out, double* s1, double* s2, double* s3,
                      double tol2, double* scratch, cudaStream_t s, PeerCtx* px = nullptr) {
    if (nparts > 1024) {
        const int nb = (nparts + 255) / 256;
        col_partial_reduce_kernel<<<nb, 256, 0, s>>>(partial, nparts, B, scratch);
        col_final_kernel<<<1, 256, 0, s>>>(scratch, nb, B, op, out, s1, s2, s3, tol2, peer_next(px));
        GP_COUNT(2);
    } else {
        col_final_kernel<<<1, 256, 0, s>>>(partial, nparts, B, op, out, s1, s2, s3, tol2, peer_next(px));
        GP_COUNT(1);
    }
}

static SparseOp csr_op(const int* indptr, const int* indices, const double* data, int64_t n) {
    SparseOp A = {false, indptr, nullptr, indices, data, (int)n};
    return A;
}
static SparseOp bcsr_op(const int64_t* bptr, const int* bidx, const double* bvals, int64_t n) {
    SparseOp A = {true, nullptr, bptr, bidx, bvals, (int)n};
    return A;
}

// X = sum_j coef[j][c] U_j (elementwise per column): one pass over the m kept Lanczos vectors. The coefficients are
// staged in shared memory mc degrees at a time (mc = min(m, COMBINE_DEGREES)); the accumulators stay in registers across
// the chunks, so the sum runs over j = 0 .. m - 1 in order whatever m is.
constexpr int COMBINE_DEGREES = 256;    // 64 KB of coefficients at B = 32
__global__ void __launch_bounds__(256)
block_combine_kernel(const double* __restrict__ basis, int64_t total, int B, int m, int mc, const double* __restrict__ coef,
                     double* __restrict__ X) {
    extern __shared__ double cf[];      // mc x B: degrees [j0, j0 + mc)
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t e = (B == 1) ? idx : idx * 2;     // B > 1: two adjacent columns of one row (B is even)
    const bool live = e < total;
    const int c = (int)(e % B);
    double a0 = 0.0, a1 = 0.0;
    for (int j0 = 0; j0 < m; j0 += mc) {
        const int mj = min(mc, m - j0);
        if (j0 > 0) __syncthreads();    // every thread is done with the previous chunk
        for (int i = threadIdx.x; i < mj * B; i += blockDim.x) cf[i] = coef[(int64_t)j0 * B + i];
        __syncthreads();
        if (!live) continue;
        const double* bj = basis + (int64_t)j0 * total + e;
        if (B == 1) {
            for (int j = 0; j < mj; ++j) a0 += cf[j] * bj[(int64_t)j * total];
        } else {
#pragma unroll 4
            for (int j = 0; j < mj; ++j) {
                const double2 u = *reinterpret_cast<const double2*>(bj + (int64_t)j * total);
                a0 += cf[j * B + c] * u.x;
                a1 += cf[j * B + c + 1] * u.y;
            }
        }
    }
    if (!live) return;
    if (B == 1) X[e] = a0;
    else *reinterpret_cast<double2*>(X + e) = make_double2(a0, a1);
}

// ---- skinny Gram matrix: out[a][b] = sum_i X[i][a] Y[i][b] for two n x B blocks (B <= 16) ----------------------
// Each CTA walks a contiguous slice of rows in tiles of 64 rows staged in shared memory (coalesced loads); thread
// (pair (a, b), slice) accumulates its pair over every (256 / B^2)-th row of the tile; partial[cta][a][b], then a
// fixed-order final sum.
constexpr int GRAM_PARTS = 1184;
constexpr int GRAM_TILE = 64;
__global__ void __launch_bounds__(256)
gram_skinny_partial_kernel(const double* __restrict__ X, const double* __restrict__ Y, int64_t n, int B, double* partial) {
    __shared__ double sx[GRAM_TILE * 16], sy[GRAM_TILE * 16];
    __shared__ double red[256];
    const int BB = B * B;
    const int nsl = 256 / BB;                 // row slices (>= 1 since B <= 16)
    const int pair = threadIdx.x % BB, sl = threadIdx.x / BB;
    const int a = pair / B, b = pair % B;
    const int64_t per = (n + gridDim.x - 1) / gridDim.x;
    const int64_t i0 = blockIdx.x * per, i1 = min(n, i0 + per);
    double acc = 0.0;
    for (int64_t r0 = i0; r0 < i1; r0 += GRAM_TILE) {
        const int rows = (int)min((int64_t)GRAM_TILE, i1 - r0);
        for (int e = threadIdx.x; e < rows * B; e += 256) {
            sx[e] = X[r0 * B + e];
            sy[e] = Y[r0 * B + e];
        }
        __syncthreads();
        if (sl < nsl)
            for (int r = sl; r < rows; r += nsl) acc += sx[r * B + a] * sy[r * B + b];
        __syncthreads();
    }
    red[threadIdx.x] = (sl < nsl) ? acc : 0.0;
    __syncthreads();
    if (threadIdx.x < BB) {
        double s = 0.0;
        for (int k = 0; k < nsl; ++k) s += red[k * BB + threadIdx.x];
        partial[(int64_t)blockIdx.x * BB + threadIdx.x] = s;
    }
}
__global__ void gram_skinny_final_kernel(const double* __restrict__ partial, int nparts, int BB, double* out) {
    const int t = threadIdx.x;
    if (t >= BB) return;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    int i = 0;
    for (; i + 3 < nparts; i += 4) {
        s0 += partial[(int64_t)i * BB + t];
        s1 += partial[(int64_t)(i + 1) * BB + t];
        s2 += partial[(int64_t)(i + 2) * BB + t];
        s3 += partial[(int64_t)(i + 3) * BB + t];
    }
    for (; i < nparts; ++i) s0 += partial[(int64_t)i * BB + t];
    out[t] = (s0 + s1) + (s2 + s3);
}

static size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

}  // namespace gp

using namespace gp;

extern "C" {

int gp_csr_spmm(const int* indptr, const int* indices, const double* data, int64_t n, double eta, const double* X, int64_t B,
                double* Y, void* stream) {
    if (!indptr || !indices || !data || !X || !Y || n <= 0 || n > INT32_MAX) return -1;
    return spmm(csr_op(indptr, indices, data, n), eta, X, (int)B, Y, (cudaStream_t)stream);
}

// Y = (K + eta I) X restricted to the rows of the operator. Row-slab operator (`peer`): X (this rank's rows) is first copied
// into exchange vector 2; a barrier before (every rank's copy is in place) and after (nobody overwrites it while a peer
// still gathers) the SpMM.
int gp_bcsr_spmm(void* peer, const int64_t* bptr, const int* bidx, const double* bvals, int64_t n, double eta, const double* X,
                 int64_t B, double* Y, void* stream) {
    if (!bptr || !bidx || !bvals || !X || !Y || n <= 0 || n > INT32_MAX) return -1;
    cudaStream_t s = (cudaStream_t)stream;
    PeerCtx* px = (PeerCtx*)peer;
    if (!px) return spmm(bcsr_op(bptr, bidx, bvals, n), eta, X, (int)B, Y, s);
    double* E = peer_local_vec(px, 2);
    PeerVec pv = peer_vec(px, 2);
    GP_CUDA_CHECK(cudaMemcpyAsync(E, X, sizeof(double) * n * B, cudaMemcpyDeviceToDevice, s));
    if (int rc = peer_barrier_launch(px, s)) return rc;
    if (int rc = spmm(bcsr_op(bptr, bidx, bvals, n), eta, E, (int)B, Y, s, nullptr, nullptr, nullptr, &pv)) return rc;
    return peer_barrier_launch(px, s);
}

}  // extern "C"

static int bcsr_build(int pass, int64_t n, const int* order, const int* inv_order, const int* indptr, const int* indices,
                      const double* data, const double* ddata, int* nblk, const int64_t* bptr, int* bidx, double* bvals,
                      double* bdvals, int* searched, void* stream) {
    cudaStream_t s = (cudaStream_t)stream;
    if (!indptr || !indices || n <= 0 || n > INT32_MAX || ((order == nullptr) != (inv_order == nullptr))) return -1;
    const int nrb = (int)((n + BCSR_ROWS - 1) / BCSR_ROWS);
    const unsigned blocks = (unsigned)(((int64_t)nrb * 32 + 127) / 128);
    if (pass == 0)
        bcsr_build_kernel<0><<<blocks, 128, 0, s>>>((int)n, order, inv_order, indptr, indices, data, ddata, nblk, bptr, bidx, bvals, bdvals, searched);
    else
        bcsr_build_kernel<1><<<blocks, 128, 0, s>>>((int)n, order, inv_order, indptr, indices, data, ddata, nblk, bptr, bidx, bvals, bdvals, searched);
    GP_COUNT(1);
    GP_LAUNCH_CHECK();
    return 0;
}

extern "C" {

int gp_bcsr_count(int64_t n, const int* order, const int* inv_order, const int* indptr, const int* indices, int* nblk,
                  int* needs_sorted_dev, void* stream) {
    if (!nblk) return -1;
    if (needs_sorted_dev) GP_CUDA_CHECK(cudaMemsetAsync(needs_sorted_dev, 0, sizeof(int), (cudaStream_t)stream));
    return bcsr_build(0, n, order, inv_order, indptr, indices, nullptr, nullptr, nblk, nullptr, nullptr, nullptr, nullptr,
                      needs_sorted_dev, stream);
}

int gp_bcsr_fill(int64_t n, const int* order, const int* inv_order, const int* indptr, const int* indices, const double* data,
                 const double* ddata, const int64_t* bptr, int64_t nblocks, int* bidx, double* bvals, double* bdvals,
                 void* stream) {
    if (!data || !bptr || !bidx || !bvals || (ddata && !bdvals) || nblocks < 0) return -1;
    GP_CUDA_CHECK(cudaMemsetAsync(bvals, 0, sizeof(double) * nblocks * BCSR_ROWS, (cudaStream_t)stream));
    if (ddata) GP_CUDA_CHECK(cudaMemsetAsync(bdvals, 0, sizeof(double) * nblocks * BCSR_ROWS, (cudaStream_t)stream));
    return bcsr_build(1, n, order, inv_order, indptr, indices, data, ddata, nullptr, bptr, bidx, bvals, bdvals, nullptr, stream);
}

int gp_rademacher(double* V, int64_t n, int64_t B, uint64_t seed, int64_t probe_offset, const int* row_map, void* stream) {
    if (!V || n <= 0 || B <= 0) return -1;
    rademacher_kernel<<<(unsigned)((n * B + 255) / 256), 256, 0, (cudaStream_t)stream>>>(n, (int)B, seed, probe_offset, row_map, V);
    GP_COUNT(1);
    GP_LAUNCH_CHECK();
    return 0;
}

static size_t partial_rows(int64_t n) {
    int64_t parts = bcsr_parts((int)n);
    return (size_t)(parts < RED_PARTS ? RED_PARTS : parts);
}
// reduction partials: the main list followed by the first-stage scratch (1/256 of it)
static size_t partial_bytes(int64_t n) {
    return al256(sizeof(double) * partial_rows(n) * 32) + al256(sizeof(double) * (partial_rows(n) / 256 + 1) * 32);
}

// workspace: 4 vectors of n x B, the reduction partials, 16 x 32 scalars
int64_t gp_krylov_workspace_bytes(int64_t n, int64_t B) {
    return (int64_t)(4 * al256(sizeof(double) * n * B) + partial_bytes(n) + 16 * al256(sizeof(double) * 32));
}

// out[c] = sum_i X[i][c] * Y[i][c]; row-slab operator (`peer`): X, Y are this rank's rows and out holds the dot products
// over ALL rows (identical on every rank)
int gp_col_dot(void* peer, const double* X, const double* Y, int64_t n, int64_t B, double* out_dev, void* ws, void* stream) {
    if (!X || !Y || !out_dev || !ws || B <= 0 || B > 32 || (32 % B)) return -1;
    cudaStream_t s = (cudaStream_t)stream;
    double* partial = (double*)ws;
    col_fused_kernel<0><<<RED_PARTS, 256, 0, s>>>(n * B, (int)B, X, Y, nullptr, nullptr, nullptr, nullptr, partial);
    col_final_kernel<<<1, 256, 0, s>>>(partial, RED_PARTS, (int)B, 0, out_dev, nullptr, nullptr, nullptr, 0.0,
                                       peer_next((PeerCtx*)peer));
    GP_COUNT(2);
    GP_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"

// m Lanczos steps of A = K + eta I started from the columns of V.
// alpha_dev, beta_dev: (m x B) row-major; beta[j] is the norm of the (j+1)-th unnormalised vector.
// The Lanczos vectors are kept UNNORMALISED (u_j = beta_{j-1} q_j) with their scales s_j = 1 / ||u_j|| on the device:
//   W = s_j (A u_j) (scale applied in the SpMM epilogue, which also reduces u_j . W), alpha_j = s_j (u_j . W),
//   u_{j+1} = W - (alpha_j s_j) u_j - (beta_{j-1} s_{j-1}) u_{j-1}  (written over u_{j-1}),  beta_j = ||u_{j+1}||
// so a step is two passes over the vectors (the SpMM and one fused update) and four launches.
// With `basis` (m x n x B doubles) the vectors u_0 .. u_{m-1} are kept: q_j = u_j / beta_{j-1} (beta_{-1} = ||v||) is the
// Krylov basis from which the caller forms (K + eta I)^-1 v = ||v|| Q T^-1 e_1 without a separate CG solve.
// Row-slab operator (`px`): A holds this rank's rows, every vector is the rank's slab, the reductions are summed over the
// ranks inside col_final_kernel, and u_j additionally lives in exchange vector (j mod 2) of the rank's arena - the copy the
// other ranks' SpMM gathers its halo rows from. Hazards: u_{j+1} is written by the update kernel BEFORE this rank
// contributes to the beta_j exchange, and a peer starts its SpMM j+1 only after that exchange (read after write); the
// buffer it overwrites held u_{j-1}, which the peers finished reading before they contributed to alpha_{j-1} (write after
// read). No barrier beyond the two reductions a Lanczos step has anyway.
static int lanczos_run(const SparseOp& A, double eta, const double* V, int64_t B, int64_t m, double* alpha_dev,
                       double* beta_dev, double* basis, void* ws, void* stream, PeerCtx* px = nullptr) {
    const int64_t n = A.n;
    if (!A.idx || !A.val || !V || !alpha_dev || !beta_dev || !ws || n <= 0 || m <= 0) return -1;
    if (B <= 0 || B > 32 || (32 % B)) return -2;
    cudaStream_t s = (cudaStream_t)stream;
    const int Bc = (int)B;
    const int64_t total = n * B;
    char* base = (char*)ws;
    size_t vb = al256(sizeof(double) * total);
    double* U0 = (double*)base;
    double* U1 = (double*)(base + vb);
    double* W = (double*)(base + 2 * vb);
    double* partial = (double*)(base + 4 * vb);
    double* scratch = partial + partial_rows(n) * 32;
    double* sc = (double*)(base + 4 * vb + partial_bytes(n));
    double* E[2] = {nullptr, nullptr};      // row-slab operator: the exchange copies of u_j (j even / odd)
    PeerVec pv[2];
    if (px) {
        for (int k = 0; k < 2; ++k) { E[k] = peer_local_vec(px, k); pv[k] = peer_vec(px, k); }
        if (!basis) { U0 = E[0]; U1 = E[1]; }      // no kept vectors: the two-buffer rotation runs in the exchange vectors
    }
    double* st = sc;           // s_cur, s_prev (+32), beta_prev (+64)
    double* a1 = sc + 96;      // alpha_j s_j
    double* b1 = sc + 128;     // beta_{j-1} s_{j-1}
    double* tmp = sc + 160;
    // u_0 = v, s_0 = 1 / ||v||, u_{-1} = 0
    auto vec = [&](int64_t j) -> double* {      // storage of u_j
        if (basis) return (j >= 0 && j < m) ? basis + j * total : U1;
        return (j & 1) ? U1 : U0;
    };
    GP_CUDA_CHECK(cudaMemcpyAsync(vec(0), V, sizeof(double) * total, cudaMemcpyDeviceToDevice, s));
    if (px && basis) GP_CUDA_CHECK(cudaMemcpyAsync(E[0], V, sizeof(double) * total, cudaMemcpyDeviceToDevice, s));
    GP_CUDA_CHECK(cudaMemsetAsync(U1, 0, sizeof(double) * total, s));
    GP_CUDA_CHECK(cudaMemsetAsync(st, 0, sizeof(double) * 96, s));
    col_fused_kernel<0><<<RED_PARTS, 256, 0, s>>>(total, Bc, V, V, nullptr, nullptr, nullptr, nullptr, partial);
    col_final_kernel<<<1, 256, 0, s>>>(partial, RED_PARTS, Bc, 2, tmp, st, nullptr, nullptr, 0.0, peer_next(px));
    GP_CUDA_CHECK(cudaMemsetAsync(st + 32, 0, sizeof(double) * 64, s));    // s_prev = beta_prev = 0 for the first step
    GP_COUNT(2);
    for (int64_t j = 0; j < m; ++j) {
        double* u = vec(j);
        int nparts = 0;
        int rc = spmm(A, eta, px ? E[j & 1] : u, Bc, W, s, st, partial, &nparts, px ? &pv[j & 1] : nullptr);
        if (rc) return rc;
        col_final(partial, nparts, Bc, 1, alpha_dev + j * B, st, a1, b1, 0.0, scratch, s, px);
        col_fused_kernel<1><<<RED_PARTS, 256, 0, s>>>(total, Bc, u, vec(j - 1), W, vec(j + 1), a1, b1, partial,
                                                      (px && basis) ? E[(j + 1) & 1] : nullptr);
        col_final_kernel<<<1, 256, 0, s>>>(partial, RED_PARTS, Bc, 2, beta_dev + j * B, st, nullptr, nullptr, 0.0,
                                           peer_next(px));
        GP_COUNT(2);
    }
    GP_LAUNCH_CHECK();
    return 0;
}

// Batched CG for (K + eta I) X = R0, all B columns at once, stop per column at ||r|| <= tol ||b|| (the reference's
// scipy cg tol=1e-6, atol=0). X: in = initial guess is ignored (zero start), out = solution. R0 is overwritten.
// iters_host receives the number of iterations performed. Returns 0, or 1 if maxiter was hit before convergence.
// Row-slab operator (`px`): the direction p lives in exchange vector 2 of the rank's arena; it is rewritten AFTER the last
// reduction of an iteration, so a cross-GPU barrier follows the direction kernel (the peers' next SpMM gathers from it).
static int cg_run(const SparseOp& A, double eta, double* R0, double* X, int64_t B, double tol, int64_t maxiter,
                  int64_t* iters_host, void* ws, void* stream, PeerCtx* px = nullptr) {
    const int64_t n = A.n;
    if (!A.idx || !A.val || !R0 || !X || !ws || n <= 0) return -1;
    if (B <= 0 || B > 32 || (32 % B)) return -2;
    cudaStream_t s = (cudaStream_t)stream;
    const int Bc = (int)B;
    const int64_t total = n * B;
    char* base = (char*)ws;
    size_t vb = al256(sizeof(double) * total);
    double* Pd = px ? peer_local_vec(px, 2) : (double*)base;
    PeerVec pv;
    if (px) pv = peer_vec(px, 2);
    double* AP = (double*)(base + vb);
    double* partial = (double*)(base + 4 * vb);
    double* scratch = partial + partial_rows(n) * 32;
    double* sc = (double*)(base + 4 * vb + partial_bytes(n));
    double *rr = sc, *active = sc + 32, *bb = sc + 64, *alpha = sc + 96, *beta = sc + 128, *flag = sc + 160;
    const unsigned eb = (unsigned)((total + 255) / 256);
    const double tol2 = tol * tol;
    GP_CUDA_CHECK(cudaMemsetAsync(X, 0, sizeof(double) * total, s));
    GP_CUDA_CHECK(cudaMemsetAsync(flag, 0, sizeof(double) * 32, s));
    GP_CUDA_CHECK(cudaMemcpyAsync(Pd, R0, sizeof(double) * total, cudaMemcpyDeviceToDevice, s));
    col_fused_kernel<0><<<RED_PARTS, 256, 0, s>>>(total, Bc, R0, R0, nullptr, nullptr, nullptr, nullptr, partial);
    // (the exchange of ||r0||^2 also orders the copy of p_0 above before the peers' first SpMM)
    col_final_kernel<<<1, 256, 0, s>>>(partial, RED_PARTS, Bc, 0, rr, nullptr, nullptr, nullptr, 0.0, peer_next(px));
    GP_CUDA_CHECK(cudaMemcpyAsync(bb, rr, sizeof(double) * 32, cudaMemcpyDeviceToDevice, s));
    double ones[32], act[32];
    GP_CUDA_CHECK(cudaMemcpyAsync(ones, rr, sizeof(double) * B, cudaMemcpyDeviceToHost, s));
    GP_CUDA_CHECK(cudaStreamSynchronize(s));
    for (int c = 0; c < 32; ++c) act[c] = (c < B && ones[c] > 0.0) ? 1.0 : 0.0;
    GP_CUDA_CHECK(cudaMemcpyAsync(active, act, sizeof(double) * 32, cudaMemcpyHostToDevice, s));
    GP_COUNT(2);
    int64_t it = 0;
    bool converged = false;
    const int check_every = 8;
    while (it < maxiter) {
        int nparts = 0;
        int rc = spmm(A, eta, Pd, Bc, AP, s, nullptr, partial, &nparts, px ? &pv : nullptr);
        if (rc) return rc;
        col_final(partial, nparts, Bc, 3, alpha, rr, active, flag, 0.0, scratch, s, px);
        col_fused_kernel<2><<<RED_PARTS, 256, 0, s>>>(total, Bc, Pd, AP, R0, X, alpha, nullptr, partial);
        col_final_kernel<<<1, 256, 0, s>>>(partial, RED_PARTS, Bc, 4, beta, rr, active, bb, tol2, peer_next(px));
        cg_direction_kernel<<<eb, 256, 0, s>>>(total, Bc, R0, beta, Pd);
        GP_COUNT(3);
        if (px) { if (int rb = peer_barrier_launch(px, s)) return rb; }
        ++it;
        if (it % check_every == 0 || it == maxiter) {
            double brk = 0.0;
            GP_CUDA_CHECK(cudaMemcpyAsync(act, active, sizeof(double) * 32, cudaMemcpyDeviceToHost, s));
            GP_CUDA_CHECK(cudaMemcpyAsync(&brk, flag, sizeof(double), cudaMemcpyDeviceToHost, s));
            GP_CUDA_CHECK(cudaStreamSynchronize(s));
            if (brk != 0.0) { if (iters_host) *iters_host = it; return 2; }
            bool any = false;
            for (int c = 0; c < B; ++c) any = any || (act[c] != 0.0);
            if (!any) { converged = true; break; }
        }
    }
    GP_LAUNCH_CHECK();
    if (iters_host) *iters_host = it;
    return converged ? 0 : 1;  // 2 (above): negative curvature met, K + eta I is not positive definite
}

extern "C" {

int gp_lanczos(const int* indptr, const int* indices, const double* data, int64_t n, double eta, const double* V, int64_t B,
               int64_t m, double* alpha_dev, double* beta_dev, double* basis_dev, void* ws, void* stream) {
    if (!indptr || n <= 0 || n > INT32_MAX) return -1;
    return lanczos_run(csr_op(indptr, indices, data, n), eta, V, B, m, alpha_dev, beta_dev, basis_dev, ws, stream);
}

int gp_bcsr_lanczos(void* peer, const int64_t* bptr, const int* bidx, const double* bvals, int64_t n, double eta,
                    const double* V, int64_t B, int64_t m, double* alpha_dev, double* beta_dev, double* basis_dev, void* ws,
                    void* stream) {
    if (!bptr || n <= 0 || n > INT32_MAX) return -1;
    return lanczos_run(bcsr_op(bptr, bidx, bvals, n), eta, V, B, m, alpha_dev, beta_dev, basis_dev, ws, stream,
                       (PeerCtx*)peer);
}

// X[i][c] = sum_j coef[j][c] basis[j][i][c]: the Lanczos solution ||v|| Q T^-1 e_1 from the kept vectors
int gp_block_combine(const double* basis, int64_t n, int64_t B, int64_t m, const double* coef_dev, double* X, void* stream) {
    if (!basis || !coef_dev || !X || n <= 0 || B <= 0 || B > 32 || (32 % B) || m <= 0 || m > INT32_MAX) return -1;
    const int64_t total = n * B;
    const int64_t work = (B == 1) ? total : total / 2;
    const int64_t mc = m < COMBINE_DEGREES ? m : COMBINE_DEGREES;
    // mc B coefficients in dynamic shared memory: up to 64 KB (mc = 256, B = 32), above the 48 KB default
    if (mc * B * (int64_t)sizeof(double) > 48 * 1024)
        if (int rc = configure_once((const void*)block_combine_kernel, 64 * 1024)) return rc;
    block_combine_kernel<<<(unsigned)((work + 255) / 256), 256, (size_t)(mc * B * sizeof(double)), (cudaStream_t)stream>>>(
        basis, total, (int)B, (int)m, (int)mc, coef_dev, X);
    GP_COUNT(1);
    GP_LAUNCH_CHECK();
    return 0;
}

int gp_cg_solve(const int* indptr, const int* indices, const double* data, int64_t n, double eta, double* R0, double* X,
                int64_t B, double tol, int64_t maxiter, int64_t* iters_host, void* ws, void* stream) {
    if (!indptr || n <= 0 || n > INT32_MAX) return -1;
    return cg_run(csr_op(indptr, indices, data, n), eta, R0, X, B, tol, maxiter, iters_host, ws, stream);
}

int gp_bcsr_cg_solve(void* peer, const int64_t* bptr, const int* bidx, const double* bvals, int64_t n, double eta, double* R0,
                     double* X, int64_t B, double tol, int64_t maxiter, int64_t* iters_host, void* ws, void* stream) {
    if (!bptr || n <= 0 || n > INT32_MAX) return -1;
    return cg_run(bcsr_op(bptr, bidx, bvals, n), eta, R0, X, B, tol, maxiter, iters_host, ws, stream, (PeerCtx*)peer);
}

// ---- row-slab operator on several GPUs (one process per GPU, peers' arenas mapped: gp_peer_*) ---------------------------------
// Every rank holds the 16-row blocks of ITS rows [rank * slab, ...) of the (spatially ordered) operator; bidx carries
// (owner << 28 | row within the owner's slab). Vectors are the rank's rows; results of reductions are identical on all ranks.

__global__ void encode_columns_kernel(int* __restrict__ bidx, int64_t total, int slab, int rank, unsigned long long* halo,
                                      unsigned* seen) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool ok = i < total;
    int owner = rank;
    if (ok) {
        const int col = bidx[i];
        owner = col / slab;
        bidx[i] = (owner << PEER_SHIFT) | (col - owner * slab);
        if (seen && owner != rank) atomicOr(seen + (col >> 5), 1u << (col & 31));
    }
    const unsigned remote = __ballot_sync(0xffffffffu, ok && owner != rank);
    if (halo && (threadIdx.x & 31) == 0 && remote) atomicAdd(halo, (unsigned long long)__popc(remote));
}

__global__ void popcount_kernel(const unsigned* __restrict__ words, int64_t nwords, unsigned long long* out) {
    unsigned long long c = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nwords; i += (int64_t)gridDim.x * blockDim.x)
        c += __popc(words[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}

// global operator-space column (< n) -> (owner, local row) for uniform slabs of `slab` rows (slab < 2^28, owner < 8).
// halo_host (optional, 2 entries; needs ws >= 16 + 4 * ceil(n / 32) bytes; synchronises the stream): [0] block-columns owned
// by another rank than `rank` = rows of X gathered over NVLink per SpMM; [1] DISTINCT remote rows among them = the halo a
// bulk exchange would move.
int gp_slab_encode_columns(int* bidx, int64_t total, int64_t slab, int64_t rank, int64_t n, int64_t* halo_host, void* ws,
                           void* stream) {
    if (!bidx || total < 0 || slab <= 0 || slab >= (1 << PEER_SHIFT) || rank < 0 || rank >= PEER_MAX || n <= 0) return -1;
    if (halo_host && !ws) return -1;
    if (halo_host) halo_host[0] = halo_host[1] = 0;
    if (total == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long* cnt = nullptr;
    unsigned* seen = nullptr;
    const int64_t nwords = (n + 31) / 32;
    if (halo_host) {
        cnt = (unsigned long long*)ws;
        seen = (unsigned*)(cnt + 2);
        GP_CUDA_CHECK(cudaMemsetAsync(ws, 0, 16 + nwords * sizeof(unsigned), s));
    }
    encode_columns_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(bidx, total, (int)slab, (int)rank, cnt, seen);
    GP_COUNT(1);
    GP_LAUNCH_CHECK();
    if (halo_host) {
        popcount_kernel<<<148, 256, 0, s>>>(seen, nwords, cnt + 1);
        GP_COUNT(1);
        unsigned long long h[2] = {0, 0};
        GP_CUDA_CHECK(cudaMemcpyAsync(h, cnt, sizeof(h), cudaMemcpyDeviceToHost, s));
        GP_CUDA_CHECK(cudaStreamSynchronize(s));
        halo_host[0] = (int64_t)h[0];
        halo_host[1] = (int64_t)h[1];
    }
    return 0;
}

}  // extern "C"

extern "C" {

int64_t gp_gram_workspace_bytes(int64_t B) { return (int64_t)(sizeof(double) * GRAM_PARTS * B * B); }

int gp_gram_skinny(const double* X, const double* Y, int64_t n, int64_t B, double* out_dev, void* ws, void* stream) {
    if (!X || !Y || !out_dev || !ws || n <= 0 || B <= 0 || B > 16) return -1;
    cudaStream_t s = (cudaStream_t)stream;
    gram_skinny_partial_kernel<<<GRAM_PARTS, 256, 0, s>>>(X, Y, n, (int)B, (double*)ws);
    gram_skinny_final_kernel<<<1, 256, 0, s>>>((const double*)ws, GRAM_PARTS, (int)(B * B), out_dev);
    GP_COUNT(2);
    GP_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
