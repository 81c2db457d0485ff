// Launchers of the solve-phase kernels (linalg.cu).
#pragma once
#include "internal.h"

namespace bemb {
// Row-sharded solve over peer memory (one process per GPU, buffers mapped with CUDA IPC), in
// flag-in-data form: element i of the work vector is two uint4 {lo32, epoch, hi32, epoch} (re, im).
// PeerOut  - every rank's buffer (own rank included), offset to MY first row, for the ZGEMV epilogue;
// PeerWait - the local buffer a consumer kernel reads, spinning per element until the epoch matches.
constexpr int MAX_PEERS = 8;
struct PeerOut {
    uint4* ll[MAX_PEERS];
    uint32_t epoch;
    int npeers;
};
struct PeerWait {
    const uint4* ll = nullptr;  // nullptr: plain work vector, nothing to wait for
    uint32_t epoch = 0;
    int* err = nullptr;         // mapped host int, set to 1 when a wait timed out
    unsigned long long timeout_ns = 4000000000ull;  // BEMB200_PEER_TIMEOUT_MS
};
cudaError_t launch_zgemv_peer(const cplx* A, uint64_t lda, uint64_t nrows, uint64_t ncols, const cplx* x, const PeerOut& po,
                              cudaStream_t s);
bool mgs_peer_wait_capable(uint64_t n, uint32_t restart);
cudaError_t launch_zgemv(const cplx* A, uint64_t lda, uint64_t nrows, uint64_t ncols, const cplx* x, cplx* y, cudaStream_t s);
cudaError_t launch_zgemv_t(const cplx* A, uint64_t lda, uint64_t nrows, uint64_t ncols, const cplx* x, cplx* y, cudaStream_t s);
// Lmat (may be NULL): (ldl x ldl) scratch for the Gram triangle of the current restart cycle (low-sync kernel)
cudaError_t launch_mgs(const cplx* V, uint64_t ldv, cplx* w, int j, uint64_t n, cplx* hcol, cplx* vnext, const cplx* pinv,
                       int direct_scale, cplx* Lmat, int ldl, cplx* scratch, cplx* hcol_host, bool* wrote_host,
                       const PeerWait& pw, bool strict, cudaStream_t s);  // strict: one rank of a row-sharded solve, no per-rank kernel fallback  // hcol_host: mapped pinned copy of the column (written by the kernel when *wrote_host)
size_t mgs_scratch_elems();  // cplx elements of scratch launch_mgs needs after the ldl*ldl Gram triangle
cudaError_t launch_residual(const cplx* b, const cplx* ax, cplx* r, uint64_t n, double* out, const cplx* pinv, cudaStream_t s);
// BiCGSTAB vector kernels: out = device scratch of >= 2 complex numbers
cudaError_t launch_bicg_dot(const cplx* a, const cplx* b, uint64_t n, cplx* out, cudaStream_t s);
cudaError_t launch_bicg_p(const cplx* r, cplx* p, const cplx* v, cplx beta, cplx omega, uint64_t n, cudaStream_t s);
cudaError_t launch_bicg_s(const cplx* r, const cplx* v, cplx alpha, cplx* sv, uint64_t n, cplx* out, cudaStream_t s);
cudaError_t launch_bicg_tt(const cplx* t, const cplx* sv, uint64_t n, cplx* out, cudaStream_t s);
cudaError_t launch_bicg_update(cplx* x, const cplx* p, const cplx* sv, const cplx* t, cplx* r, const cplx* r0, cplx alpha, cplx omega,
                               uint64_t n, cplx* out, cudaStream_t s);
cudaError_t launch_bicg_axpy(cplx* x, const cplx* p, cplx alpha, uint64_t n, cudaStream_t s);
// CGS (cgs.rs:71-140)
cudaError_t launch_cgs_q(const cplx* u, const cplx* v, cplx alpha, cplx* q, cplx* uq, uint64_t n, cudaStream_t s);
cudaError_t launch_cgs_update(cplx* x, const cplx* uq, const cplx* w, cplx* r, const cplx* r0, cplx alpha, uint64_t n, cplx* out,
                              cudaStream_t s);
cudaError_t launch_cgs_p(const cplx* r, const cplx* q, cplx beta, cplx* u, cplx* p, uint64_t n, cudaStream_t s);
// block_matvec.cu: Y = A X for nrhs = 8, 16, 24 or 32 right-hand sides (X interleaved [k][S], Y interleaved [row][S]);
// DMMA.8x8x4 kernel with shared-memory staging and a stream-K decomposition
cudaError_t launch_zgemm_block(const cplx* A, uint64_t lda, uint64_t nrows, uint64_t ncols, const cplx* X, cplx* Y, int nrhs,
                               cudaStream_t s);
cudaError_t launch_mgs_batched(int nrhs, const cplx* Vall, uint64_t ldv, uint64_t vstride, const cplx* Yblk, int j, uint64_t n,
                               cplx* hcol_all, uint64_t hstride, cplx* Xblk, const unsigned char* active, cudaStream_t s);
cudaError_t launch_block_residual(const cplx* B, const cplx* AX, cplx* R, uint64_t n, int nrhs, double* out, cudaStream_t s);
cudaError_t launch_block_scale(const cplx* R, const double* scale, cplx* Vall, uint64_t vstride, cplx* Xblk, uint64_t n, int nrhs,
                               cudaStream_t s);
cudaError_t launch_block_update_x(cplx* Xsol, const cplx* Vall, uint64_t ldv, uint64_t vstride, const cplx* ycoef, int ldy,
                                  const int* cnt, uint64_t n, int nrhs, cudaStream_t s);
cudaError_t launch_interleave(const cplx* src, cplx* dst, uint64_t n, int nsrc, int nrhs, int to_block, cudaStream_t s);
cudaError_t launch_scale(const cplx* r, double sc, cplx* v, uint64_t n, cudaStream_t s);
cudaError_t launch_update_x(cplx* x, const cplx* V, uint64_t ldv, const cplx* ycoef, int cnt, uint64_t n, cudaStream_t s);
cudaError_t launch_row_sum(cplx* A, uint64_t lda, uint64_t nloc, uint64_t ncols, uint64_t r0, cplx* rowsums, cudaStream_t s);
cudaError_t launch_dfma_peak(double* out, int iters, cudaStream_t s);
cudaError_t launch_math_selftest(uint64_t n, double xmax, double* err, cudaStream_t s);
}  // namespace bemb
