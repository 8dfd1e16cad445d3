// FP64 tensor-core (DMMA) GEMM for the Cholesky / inverse hot path: C = beta C + alpha op(A) op(B).
//
// One 128 x BN output tile per CTA, warp tile 64 x 32 built from m8n8k4 DMMA fragments. The k-slabs (16 deep) are moved
// by ONE producer warp with cp.async.bulk.tensor (SASS: UTMALDG) into a ring of 128-byte-swizzled shared tiles guarded
// by full/empty mbarriers, so the consumer warps never meet in a CTA barrier inside the main loop. Both operand layouts
// are read bank-conflict free (see the shared layouts below), which lets one kernel serve
//   NT: trailing SYRK/GEMM update and the panel TRSM-by-inverse   (potrf)
//   NN: triangular products of the recursive inverse               (trtri)
//   TN: W^T W                                                      (lauum)
// Triangular operands are exploited by restricting each tile's k-range, never by element masks.
//
// Shared layouts (hardware SWIZZLE_128B: 16-byte chunk index ^= row & 7 inside 1024-byte groups):
//   K-major operand  ([mn][k], T = 0): one 2-D box {16 k, ROWS mn}; row = mn (128 B each).
//   MN-major operand ([k][mn], T = 1): ROWS/16 boxes of a 5-D view {16 mn, kbit1, kbit0, k>>3, kbit2} (2 KB each); the box
//                    row is r = kbit1 | kbit0<<1 | kbit3<<2 | kbit2<<3.
// Inside a slab of 16 k the MMA step kk (0..3) gives lane t (0..3) the logical k = (t&1) | kk<<1 | (t>>1)<<3 - the same
// permutation for A and B, so the product is unchanged - which makes the 8-byte fragment loads of both layouts
// bank-conflict free (each half-warp covers 16 distinct 8-byte bank groups).
#include "gp_common.cuh"
#include "gp_internal.h"
#include <cuda.h>
#include <algorithm>
#include <mutex>
#include <set>
#include <utility>
#include <vector>

namespace gp {

std::atomic<unsigned long long> g_launch_count{0};

// optional per-launch timing of the DMMA GEMM (bench.py's roofline leg): events around every launch
struct GemmProfile {
    bool on = false;
    std::vector<cudaEvent_t> pool;
    size_t used = 0;
    double flops = 0.0;       // executed tile flops (2 * 128 * BN * k per computed tile)
    long long launches = 0;
    cudaEvent_t ref = nullptr;  // time origin for the union of the (possibly concurrent) launch intervals
};
static GemmProfile g_prof;
static std::mutex g_prof_mutex;

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is a per-device property of a kernel: done once per (device, kernel)
static std::mutex g_cfg_mutex;
static std::set<std::pair<int, const void*>> g_cfg_done;

int configure_once(const void* func, int smem_bytes) {
    int dev = 0;
    GP_CUDA_CHECK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_cfg_mutex);
    std::pair<int, const void*> key(dev, func);
    if (g_cfg_done.count(key)) return 0;
    GP_CUDA_CHECK(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    g_cfg_done.insert(key);
    return 0;
}

// when profiling is on: records the start event on `stream`, books the flops and returns the stop event to record
// after the launch (nullptr when profiling is off)
static cudaEvent_t profile_begin(double flops, cudaStream_t stream) {
    if (!g_prof.on) return nullptr;
    std::lock_guard<std::mutex> lock(g_prof_mutex);
    while (g_prof.pool.size() < g_prof.used + 2) {
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
        g_prof.pool.push_back(e);
    }
    cudaEvent_t e0 = g_prof.pool[g_prof.used++];
    cudaEvent_t e1 = g_prof.pool[g_prof.used++];
    g_prof.flops += flops;
    g_prof.launches++;
    cudaEventRecord(e0, stream);
    return e1;
}

static double tile_flops(int tiles_m, int tiles_n, int bn, int K, int krange, int tmask) {
    double kt = 0.0;  // sum over computed tiles of their k extent
    for (int tm = 0; tm < tiles_m; ++tm) {
        int lim = ((tm + 1) * 128) / bn;  // tiles with n0 < m0 + 128
        int ncols = (tmask == TM_LOWER) ? (lim < tiles_n ? lim : tiles_n) : tiles_n;
        if (krange == KR_FULL) kt += (double)ncols * K;
        else if (krange == KR_A_LOWER) kt += (double)ncols * ((tm + 1) * 128 < K ? (tm + 1) * 128 : K);
        else for (int tn = 0; tn < ncols; ++tn) {
            int kb = (krange == KR_B_LOWER) ? tn * bn : (tm * 128 > tn * bn ? tm * 128 : tn * bn);
            kt += (double)(K - (kb < K ? kb : K));
        }
    }
    return 2.0 * 128.0 * bn * kt;
}

constexpr int BM = 128, WM = 64, WN = 32, MI = WM / 8, NI = WN / 8;
constexpr int RASTER_GROUP = 8;

// Two tile shapes share one kernel body:
//   BN = 64 : 4 consumer warps, 4 stages (96 KB), TWO CTAs per SM: while one CTA sits in its prologue or its C
//             read-modify-write epilogue, the other keeps the FP64 tensor pipe busy. Every product but the one below.
//   BN = 128: 8 consumer warps, 6 stages (192 KB), one CTA per SM. Only for the in-place panel solve, where C aliases A
//             and a CTA must own the full row block it overwrites (see check_args).
template <int BN_>
struct TCfg {
    static constexpr int BN = BN_;
    static constexpr int BK = 16;
    static constexpr int STAGES = (BN_ == 128) ? 6 : 4;
    static constexpr int WARPS_N = BN_ / WN;
    static constexpr int CONSUMER_WARPS = (BM / WM) * WARPS_N;
    static constexpr int THREADS = (CONSUMER_WARPS + 1) * 32;            // + the TMA producer warp
    static constexpr int A_BYTES = BM * BK * 8, B_BYTES = BN_ * BK * 8, STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int SMEM = STAGES * STAGE_BYTES + 2048;   // tiles + 1 KB alignment slack + barriers (whole KB)
    static constexpr int MIN_CTAS = (BN_ == 128) ? 1 : 2;
};

__device__ __forceinline__ void mbar_init(uint32_t bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar) : "memory");
}
// arrive with a data dependence on `value` that the assembler cannot fold away: both predicated copies arrive once
__device__ __forceinline__ void mbar_arrive_after(uint32_t bar, uint32_t value) {
    asm volatile(
        "{\n"
        ".reg .pred q;\n"
        "setp.ne.u32 q, %1, 0x7ff7a5c3;\n"
        "@q mbarrier.arrive.shared::cta.b64 _, [%0];\n"
        "@!q mbarrier.arrive.shared::cta.b64 _, [%0];\n"
        "}\n" ::"r"(bar), "r"(value) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n" : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2,
                                            int c3, int c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];\n"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4) : "memory");
}

// byte offset of the fragment element (tile-local mn, MMA step kk, lane column t) inside an operand tile
template <int T>
__device__ __forceinline__ uint32_t frag_off(int mn, int kk, int t) {
    if (T == 0) {
        int chunk = (kk | ((t >> 1) << 2)) ^ (mn & 7);
        return (uint32_t)(mn * 128 + (chunk << 4) + ((t & 1) << 3));
    }
    int r = (kk & 1) | ((t & 1) << 1) | ((t >> 1) << 2) | ((kk >> 1) << 3);
    int ml = mn & 15;
    int chunk = (ml >> 1) ^ (r & 7);
    return (uint32_t)((mn >> 4) * 2048 + r * 128 + (chunk << 4) + ((ml & 1) << 3));
}

__device__ __forceinline__ double lds_f64(uint32_t addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];\n" : "=d"(v) : "r"(addr));
    return v;
}

template <int AT, int BT, int BN_>
__global__ void __launch_bounds__(TCfg<BN_>::THREADS, TCfg<BN_>::MIN_CTAS)
dgemm_tma_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, double* C, int64_t ldc,
                 int tiles_m, int tiles_n, int K, double alpha, double beta, int krange, int tmask,
                 const int* __restrict__ kbeg_tab, const int* __restrict__ kend_tab) {
    using G = TCfg<BN_>;
    constexpr int BN = G::BN, BK = G::BK, STAGES = G::STAGES;
    extern __shared__ __align__(16) unsigned char smem_raw[];

    // grouped rasterisation: RASTER_GROUP tile-rows share each B tile while it is hot in L2
    int bid = blockIdx.x;
    int group_sz = RASTER_GROUP * tiles_n;
    int grp = bid / group_sz;
    int first_m = grp * RASTER_GROUP;
    int rows_in_grp = min(RASTER_GROUP, tiles_m - first_m);
    int rem = bid - grp * group_sz;
    int tm = first_m + rem % rows_in_grp;
    int tn = rem / rows_in_grp;
    const int m0 = tm * BM, n0 = tn * BN;
    if (tmask == TM_LOWER && n0 >= m0 + BM) return;

    int kbeg = 0, kend = K;
    if (krange == KR_A_LOWER) kend = min(K, m0 + BM);
    else if (krange == KR_B_LOWER) kbeg = min(n0, K);
    else if (krange == KR_TN_LOWER) kbeg = min(max(m0, n0), K);
    // optional per-row-tile k ranges (staircase operands of the distributed inverse, _blockcyclic.py)
    if (kbeg_tab) kbeg = max(kbeg, min(kbeg_tab[tm], K));
    if (kend_tab) kend = min(kend, kend_tab[tm]);
    kbeg = (kbeg / BK) * BK;
    const int KT = max(0, (kend - kbeg) / BK);

    const uint32_t base = ((uint32_t)__cvta_generic_to_shared(smem_raw) + 1023u) & ~1023u;
    const uint32_t bars = base + STAGES * G::STAGE_BYTES;      // full[s] at bars + 8 s, empty[s] at bars + 8 (STAGES + s)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(bars + 8 * s, 1);
            mbar_init(bars + 8 * (STAGES + s), G::CONSUMER_WARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncthreads();

    if (warp == G::CONSUMER_WARPS) {
        // ===== producer warp: one lane issues the bulk tensor copies =====
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];\n" ::"l"(reinterpret_cast<uint64_t>(&mapA)) : "memory");
            asm volatile("prefetch.tensormap [%0];\n" ::"l"(reinterpret_cast<uint64_t>(&mapB)) : "memory");
            for (int kt = 0; kt < KT; ++kt) {
                const int s = kt % STAGES;
                if (kt >= STAGES) mbar_wait(bars + 8 * (STAGES + s), ((kt / STAGES) - 1) & 1);
                const uint32_t full = bars + 8 * s;
                const uint32_t sa = base + s * G::STAGE_BYTES, sb = sa + G::A_BYTES;
                const int k0 = kbeg + kt * BK;
                mbar_expect_tx(full, G::STAGE_BYTES);
                if (AT == 0) {
                    tma_load_2d(sa, &mapA, full, k0, m0);
                } else {
#pragma unroll
                    for (int j = 0; j < BM / 16; ++j) tma_load_5d(sa + j * 2048, &mapA, full, m0 + 16 * j, 0, 0, k0 >> 3, 0);
                }
                if (BT == 0) {
                    tma_load_2d(sb, &mapB, full, k0, n0);
                } else {
#pragma unroll
                    for (int j = 0; j < BN / 16; ++j) tma_load_5d(sb + j * 2048, &mapB, full, n0 + 16 * j, 0, 0, k0 >> 3, 0);
                }
            }
        }
        return;
    }

    // ===== consumer warps =====
    const int g = lane >> 2, t = lane & 3;
    const int wm = (warp / G::WARPS_N) * WM, wn = (warp % G::WARPS_N) * WN;

    double acc[MI][NI][2];
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
        for (int j = 0; j < NI; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    if (beta != 0.0) {
        // the epilogue read-modify-writes a tile of C that streams from HBM: pull it into L2 now so those loads cost
        // an L2 hit instead of a DRAM round trip each (128 rows x BN/16 lines of 128 B)
        constexpr int LINES = BM * BN / 16;
        constexpr int CT = G::CONSUMER_WARPS * 32;
#pragma unroll
        for (int i = 0; i < LINES / CT; ++i) {
            int line = tid + i * CT;
            const double* pc = C + (int64_t)(m0 + line / (BN / 16)) * ldc + n0 + ((line % (BN / 16)) << 4);
            asm volatile("prefetch.global.L2 [%0];" ::"l"(pc));
        }
    }

    // per-thread fragment offsets (bytes) inside the A and B tiles for the four MMA steps of a slab
    uint32_t aoff[4], boff[4];
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
        aoff[kk] = frag_off<AT>(wm + g, kk, t);
        boff[kk] = frag_off<BT>(wn + g, kk, t);
    }
    // fragment i sits 8 mn further: K-major +8 rows = +1024 B; MN-major +8 mn = half a box: chunk bit 2 flips (+/- 64 B)
    // for odd i and every second i moves one box (2048 B) on
    for (int kt = 0; kt < KT; ++kt) {
        const int s = kt % STAGES;
        mbar_wait(bars + 8 * s, (kt / STAGES) & 1);
        const uint32_t sa = base + s * G::STAGE_BYTES, sb = sa + G::A_BYTES;
        uint32_t dep = 0;        // data dependence of the release on every fragment load of this slab (see mbar_arrive_after)
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            double a[MI], b[NI];
#pragma unroll
            for (int i = 0; i < MI; ++i) {
                uint32_t o = (AT == 0) ? aoff[kk] + i * 1024 : ((aoff[kk] ^ ((i & 1) << 6)) + (i >> 1) * 2048);
                a[i] = lds_f64(sa + o);
            }
#pragma unroll
            for (int j = 0; j < NI; ++j) {
                uint32_t o = (BT == 0) ? boff[kk] + j * 1024 : ((boff[kk] ^ ((j & 1) << 6)) + (j >> 1) * 2048);
                b[j] = lds_f64(sb + o);
            }
#pragma unroll
            for (int i = 0; i < MI; ++i) dep ^= (uint32_t)__double2hiint(a[i]);
#pragma unroll
            for (int j = 0; j < NI; ++j) dep ^= (uint32_t)__double2hiint(b[j]);
#pragma unroll
            for (int i = 0; i < MI; ++i)
#pragma unroll
                for (int j = 0; j < NI; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
        // Release of the stage. The arrive must not be ISSUED before every fragment load of this warp has RETURNED its
        // data: the hardware does not order an outstanding LDS before a later SYNCS.ARRIVE of the same warp, and the
        // assembler is free to hoist the arrive right behind the last LDS issue (measured: with the load / store unit
        // busy - two CTAs per SM, C read-modify-write epilogues - the producer's next TMA write then overtook pending
        // loads and single fragment rows were read from the wrong slab). The arrive is therefore predicated on a value
        // computed from ALL loaded registers of the slab (it is skipped only for one exact bit pattern that is then
        // replaced), a data dependence the assembler cannot remove.
        dep = __reduce_xor_sync(0xffffffffu, dep);
        if (lane == 0) mbar_arrive_after(bars + 8 * (STAGES + s), dep);
    }

    // epilogue: each thread owns (row, 2 consecutive cols) of every 8x8 fragment -> 16-byte accesses
    const bool diag = (tmask == TM_LOWER) && (n0 + BN - 1 > m0);   // tile crosses the diagonal: mask col > row
    if (beta != 0.0 && !diag) {
        // full tile with accumulate: issue all loads of a row group before using them (memory-level parallelism)
#pragma unroll
        for (int i = 0; i < MI; i += 2) {
            double2 o[2][NI];
#pragma unroll
            for (int ii = 0; ii < 2; ++ii)
#pragma unroll
                for (int j = 0; j < NI; ++j)
                    o[ii][j] = *reinterpret_cast<const double2*>(C + (int64_t)(m0 + wm + (i + ii) * 8 + g) * ldc + n0 + wn + j * 8 + 2 * t);
#pragma unroll
            for (int ii = 0; ii < 2; ++ii)
#pragma unroll
                for (int j = 0; j < NI; ++j) {
                    double2 v;
                    v.x = alpha * acc[i + ii][j][0] + beta * o[ii][j].x;
                    v.y = alpha * acc[i + ii][j][1] + beta * o[ii][j].y;
                    *reinterpret_cast<double2*>(C + (int64_t)(m0 + wm + (i + ii) * 8 + g) * ldc + n0 + wn + j * 8 + 2 * t) = v;
                }
        }
        return;
    }
#pragma unroll
    for (int i = 0; i < MI; ++i) {
        const int grow = m0 + wm + i * 8 + g;
        double* crow = C + (int64_t)grow * ldc;
#pragma unroll
        for (int j = 0; j < NI; ++j) {
            const int gcol = n0 + wn + j * 8 + 2 * t;
            if (diag && gcol > grow) continue;
            double2 v;
            v.x = alpha * acc[i][j][0];
            v.y = alpha * acc[i][j][1];
            double2* p = reinterpret_cast<double2*>(crow + gcol);
            if (beta != 0.0) {
                double2 o = *p;
                v.x += beta * o.x;
                v.y += beta * o.y;
            }
            if (diag && gcol + 1 > grow) {
                crow[gcol] = v.x;  // keep the strictly-upper neighbour untouched
            } else {
                *p = v;
            }
        }
    }
}

// ---- tensor maps --------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;
static int g_encode_state = 0;   // 0 unknown, 1 ready, -1 unavailable

static int encode_init() {
    if (g_encode_state) return g_encode_state;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn ||
        q != cudaDriverEntryPointSuccess) {
        (void)cudaGetLastError();
        g_encode_state = -1;
        return -1;
    }
    g_encode = (EncodeTiledFn)fn;
    g_encode_state = 1;
    return 1;
}

// operand `P` (logical rows = mn extent, K columns) with leading dimension ld; T = 0: stored [mn][k], T = 1: stored [k][mn]
static int make_map(CUtensorMap* map, int T, const double* P, int64_t ld, int mn, int K, int rows_per_box) {
    cuuint32_t es[5] = {1, 1, 1, 1, 1};
    CUresult r;
    if (T == 0) {
        cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)mn};
        cuuint64_t strides[1] = {(cuuint64_t)ld * 8};
        cuuint32_t box[2] = {16, (cuuint32_t)rows_per_box};
        r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, (void*)P, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    } else {
        cuuint64_t dims[5] = {(cuuint64_t)mn, 2, 2, (cuuint64_t)(K / 8), 2};
        cuuint64_t strides[4] = {(cuuint64_t)ld * 16, (cuuint64_t)ld * 8, (cuuint64_t)ld * 64, (cuuint64_t)ld * 32};
        cuuint32_t box[5] = {16, 2, 2, 2, 2};
        r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 5, (void*)P, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    }
    return r == CUDA_SUCCESS ? 0 : -(int)r - 2000;
}

template <int AT, int BT, int BN_>
static int launch_tma_inst(double* C, int64_t ldc, const double* A, int64_t lda, const double* B, int64_t ldb,
                           int M, int N, int K, double alpha, double beta, int krange, int tmask, cudaStream_t stream,
                           const int* kbeg_tab, const int* kend_tab) {
    using G = TCfg<BN_>;
    if (K % G::BK) return -1;
    int tiles_m = M / BM, tiles_n = N / BN_;
    if (tiles_m == 0 || tiles_n == 0) return 0;
    int rc = configure_once((const void*)dgemm_tma_kernel<AT, BT, BN_>, G::SMEM);
    if (rc) return rc;
    // K == 0 (C = beta C): the driver refuses a zero extent, so the maps get a dummy one that no load touches (KT = 0)
    const int Kmap = K > 0 ? K : 32;
    CUtensorMap mapA, mapB;
    if ((rc = make_map(&mapA, AT, A, lda, M, Kmap, BM))) return rc;
    if ((rc = make_map(&mapB, BT, B, ldb, N, Kmap, BN_))) return rc;
    cudaEvent_t e1 = profile_begin(tile_flops(tiles_m, tiles_n, BN_, K, krange, tmask), stream);
    dgemm_tma_kernel<AT, BT, BN_><<<tiles_m * tiles_n, G::THREADS, G::SMEM, stream>>>(
        mapA, mapB, C, ldc, tiles_m, tiles_n, K, alpha, beta, krange, tmask, kbeg_tab, kend_tab);
    if (e1) cudaEventRecord(e1, stream);
    GP_COUNT(1);
    GP_LAUNCH_CHECK();
    return 0;
}

static int launch_tma_bn64(int at, int bt, double* C, int64_t ldc, const double* A, int64_t lda, const double* B, int64_t ldb,
                           int M, int N, int K, double alpha, double beta, int krange, int tmask, cudaStream_t stream,
                           const int* kbeg_tab, const int* kend_tab) {
    if (at == 0 && bt == 0) return launch_tma_inst<0, 0, 64>(C, ldc, A, lda, B, ldb, M, N, K, alpha, beta, krange, tmask, stream, kbeg_tab, kend_tab);
    if (at == 0 && bt == 1) return launch_tma_inst<0, 1, 64>(C, ldc, A, lda, B, ldb, M, N, K, alpha, beta, krange, tmask, stream, kbeg_tab, kend_tab);
    if (at == 1 && bt == 1) return launch_tma_inst<1, 1, 64>(C, ldc, A, lda, B, ldb, M, N, K, alpha, beta, krange, tmask, stream, kbeg_tab, kend_tab);
    if (at == 1 && bt == 0) return launch_tma_inst<1, 0, 64>(C, ldc, A, lda, B, ldb, M, N, K, alpha, beta, krange, tmask, stream, kbeg_tab, kend_tab);
    return -4;
}

// Argument checks shared by launch_dgemm and launch_dgemm_ktab, all made before any launch. Returns the tile width to
// launch (64, or 128 for the in-place form below) or a negative error code.
// The one aliased form allowed is the in-place panel solve of factor_panel (gp_chol.cu): C == A with the same leading
// dimension, at = bt = 0, a single 128-wide column tile and no k tables. There each BN = 128 CTA reads exactly the row
// block it overwrites. In every other aliased form CTAs read rows or columns that other CTAs write, and the result
// would depend on their timing: -6.
static int check_args(int at, int bt, const double* C, int64_t ldc, const double* A, int64_t lda, const double* B,
                      int64_t ldb, int M, int N, int K, bool ktab) {
    if (M < 0 || N < 0 || K < 0 || (M % BM) || (N % 128) || (K % 32)) return -1;
    if ((lda & 1) || (ldb & 1) || (ldc & 1)) return -2;
    if (((uintptr_t)A | (uintptr_t)B | (uintptr_t)C) & 15) return -3;
    const bool in_place = !ktab && C == A && C != B && ldc == lda && at == 0 && bt == 0 && N == 128;
    if ((C == A || C == B) && !in_place) return -6;
    if (encode_init() != 1) return -7;
    return in_place ? 128 : 64;
}

int launch_dgemm(int at, int bt, double* C, int64_t ldc, const double* A, int64_t lda, const double* B, int64_t ldb,
                 int M, int N, int K, double alpha, double beta, int krange, int tmask, cudaStream_t stream) {
    const int bn = check_args(at, bt, C, ldc, A, lda, B, ldb, M, N, K, false);
    if (bn < 0) return bn;
    if (bn == 128)
        return launch_tma_inst<0, 0, 128>(C, ldc, A, lda, B, ldb, M, N, K, alpha, beta, krange, tmask, stream, nullptr, nullptr);
    return launch_tma_bn64(at, bt, C, ldc, A, lda, B, ldb, M, N, K, alpha, beta, krange, tmask, stream, nullptr, nullptr);
}

// GEMM with per-row-tile k ranges: tile row tm (128 rows) uses k in [kbeg_tab[tm], kend_tab[tm]) (device int arrays, either
// may be null; entries multiples of 16, the k-slab of the kernel).
int launch_dgemm_ktab(int at, int bt, double* C, int64_t ldc, const double* A, int64_t lda, const double* B, int64_t ldb,
                      int M, int N, int K, double alpha, double beta, const int* kbeg_tab, const int* kend_tab,
                      cudaStream_t stream) {
    const int bn = check_args(at, bt, C, ldc, A, lda, B, ldb, M, N, K, true);
    if (bn < 0) return bn;
    return launch_tma_bn64(at, bt, C, ldc, A, lda, B, ldb, M, N, K, alpha, beta, KR_FULL, TM_ALL, stream, kbeg_tab, kend_tab);
}


int profile_enable(int on) {
    g_prof.on = on != 0;
    g_prof.used = 0;
    g_prof.flops = 0.0;
    g_prof.launches = 0;
    if (g_prof.on) {
        if (!g_prof.ref) GP_CUDA_CHECK(cudaEventCreate(&g_prof.ref));
        GP_CUDA_CHECK(cudaDeviceSynchronize());
        GP_CUDA_CHECK(cudaEventRecord(g_prof.ref, 0));
        GP_CUDA_CHECK(cudaDeviceSynchronize());
    }
    return 0;
}

// synchronises the device; returns the summed GEMM kernel milliseconds, the length of the UNION of the launch
// intervals (launches on different streams overlap), the executed tile flops and the launch count since enable
int profile_read(double* ms_sum, double* ms_union, double* flops, long long* launches) {
    GP_CUDA_CHECK(cudaDeviceSynchronize());
    std::vector<std::pair<float, float>> iv;
    double total = 0.0;
    for (size_t i = 0; i + 1 < g_prof.used; i += 2) {
        float t0 = 0.f, t1 = 0.f;
        GP_CUDA_CHECK(cudaEventElapsedTime(&t0, g_prof.ref, g_prof.pool[i]));
        GP_CUDA_CHECK(cudaEventElapsedTime(&t1, g_prof.ref, g_prof.pool[i + 1]));
        total += (double)t1 - (double)t0;
        iv.push_back(std::make_pair(t0, t1));
    }
    std::sort(iv.begin(), iv.end());
    double uni = 0.0;
    float cur0 = 0.f, cur1 = -1.f;
    for (size_t i = 0; i < iv.size(); ++i) {
        if (cur1 < cur0 || iv[i].first > cur1) {
            if (cur1 >= cur0) uni += (double)cur1 - (double)cur0;
            cur0 = iv[i].first;
            cur1 = iv[i].second;
        } else if (iv[i].second > cur1) {
            cur1 = iv[i].second;
        }
    }
    if (cur1 >= cur0) uni += (double)cur1 - (double)cur0;
    *ms_sum = total;
    *ms_union = uni;
    *flops = g_prof.flops;
    *launches = g_prof.launches;
    return 0;
}

}  // namespace gp
