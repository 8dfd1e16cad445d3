// Internal (non-ABI) declarations shared between the gpgp translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace gp {

// k-range restriction of one 128x128 output tile at (m0, n0); exploits triangular operands
enum KRange {
    KR_FULL = 0,      // k in [0, K)
    KR_A_LOWER = 1,   // A(m,k) lower triangular: k in [0, m0 + 128)
    KR_B_LOWER = 2,   // B(k,n) lower triangular: k in [n0, K)
    KR_TN_LOWER = 3,  // A(m,k)=W[k][m], B(k,n)=W[k][n], W lower: k in [max(m0,n0), K)
};
enum TileMask {
    TM_ALL = 0,
    TM_LOWER = 1,  // only tiles with n0 <= m0; diagonal tiles store col <= row only
};

// C[M x N] (row-major, ldc) = beta*C + alpha * op(A) * op(B)
//   at == 0: A(m,k) = A[m*lda + k]   at == 1: A(m,k) = A[k*lda + m]
//   bt == 0: B(k,n) = B[n*ldb + k]   bt == 1: B(k,n) = B[k*ldb + n]
// M, N multiples of 128; K multiple of 32; all ld even; pointers 16-byte aligned. C may alias an operand only in the
// in-place panel solve (C == A, lda == ldc, at == bt == 0, N == 128); any other aliasing returns -6.
int launch_dgemm(int at, int bt, double* C, int64_t ldc, const double* A, int64_t lda,
                 const double* B, int64_t ldb, int M, int N, int K, double alpha, double beta,
                 int krange, int tmask, cudaStream_t stream);

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (device, kernel); thread-safe
int configure_once(const void* func, int smem_bytes);

int launch_dgemm_ktab(int at, int bt, double* C, int64_t ldc, const double* A, int64_t lda, const double* B, int64_t ldb,
                      int M, int N, int K, double alpha, double beta, const int* kbeg_tab, const int* kend_tab,
                      cudaStream_t stream);

int profile_enable(int on);
int profile_read(double* ms_sum, double* ms_union, double* flops, long long* launches);

// ---- row-slab (multi-GPU) sparse operator: every rank maps its peers' arenas through CUDA IPC (csrc/gp_peer.cu) ------------
constexpr int PEER_MAX = 8;         // ranks of one NVSwitch domain
constexpr int PEER_SLOTS = 8;       // mailbox ring (a peer is never more than one exchange ahead; see peer_block_sum)
constexpr int PEER_PAYLOAD = 256;   // doubles per (slot, rank): up to a 16 x 16 Gram block
constexpr int PEER_VECS = 3;        // exchange vectors per arena (the SpMM inputs peers gather from)

struct PeerComm {                   // one exchange, passed to the kernel by value
    int rank, world;                // world <= 1: no exchange
    unsigned long long seq;         // sequence number of this exchange (1, 2, ...), the same on every rank
    double* mail[PEER_MAX];         // mail[p]: rank p's mailbox: payload[SLOTS][MAX][PAYLOAD] doubles, then flags[SLOTS][MAX] u64
    int* err;                       // local flag: a wait timed out
};
struct PeerVec {                    // one exchange vector as mapped on this rank: base[p] = rank p's copy (its own rows)
    const double* base[PEER_MAX];
    int rank;                       // this rank (base[rank] is local memory)
};
struct PeerCtx;                     // host side (gp_peer.cu)
PeerComm peer_next(PeerCtx* ctx);                  // the next exchange (advances the sequence number); world 1 without ctx
PeerVec peer_vec(PeerCtx* ctx, int k);             // exchange vector k on every rank
double* peer_local_vec(PeerCtx* ctx, int k);       // this rank's copy of exchange vector k
int peer_world(const PeerCtx* ctx);
int peer_barrier_launch(PeerCtx* ctx, cudaStream_t s);

}  // namespace gp
