// Test-only C entry points over the solve-phase launchers of linalg.cu and block_matvec.cu, so that the tests can call
// every dispatch branch of one Arnoldi step, of the GEMV pair and of the stream-K block product with chosen sizes and
// compare it with an extended-precision reference (tests/solve_kernels_reference.py).  Linked against the library's own
// sources, compiled with the library's flags; nothing here changes what the kernels do.
//
// Every wrapper takes raw device pointers, runs on the legacy default stream and returns the cudaError_t of the launcher
// as an int.  launch_mgs runs without a mapped host column (hcol_host = NULL), without a peer wait and not strict, which
// is how a one-GPU solve calls it.
#include "linalg.h"

using namespace bemb;

extern "C" {

int shim_zgemv(const void* A, uint64_t lda, uint64_t nrows, uint64_t ncols, const void* x, void* y) {
    return (int)launch_zgemv((const cplx*)A, lda, nrows, ncols, (const cplx*)x, (cplx*)y, 0);
}

int shim_zgemv_t(const void* A, uint64_t lda, uint64_t nrows, uint64_t ncols, const void* x, void* y) {
    return (int)launch_zgemv_t((const cplx*)A, lda, nrows, ncols, (const cplx*)x, (cplx*)y, 0);
}

int shim_zgemm_block(const void* A, uint64_t lda, uint64_t nrows, uint64_t ncols, const void* X, void* Y, int nrhs) {
    return (int)launch_zgemm_block((const cplx*)A, lda, nrows, ncols, (const cplx*)X, (cplx*)Y, nrhs, 0);
}

int shim_mgs(const void* V, uint64_t ldv, void* w, int j, uint64_t n, void* hcol, void* vnext, const void* pinv, int direct_scale,
             void* Lmat, int ldl, void* scratch) {
    bool wrote_host = false;
    const PeerWait pw;
    return (int)launch_mgs((const cplx*)V, ldv, (cplx*)w, j, n, (cplx*)hcol, (cplx*)vnext, (const cplx*)pinv, direct_scale,
                           (cplx*)Lmat, ldl, (cplx*)scratch, nullptr, &wrote_host, pw, false, 0);
}

uint64_t shim_mgs_scratch_elems() { return (uint64_t)mgs_scratch_elems(); }

int shim_mgs_batched(int nrhs, const void* Vall, uint64_t ldv, uint64_t vstride, const void* Yblk, int j, uint64_t n, void* hcol_all,
                     uint64_t hstride, void* Xblk, const void* active) {
    return (int)launch_mgs_batched(nrhs, (const cplx*)Vall, ldv, vstride, (const cplx*)Yblk, j, n, (cplx*)hcol_all, hstride,
                                   (cplx*)Xblk, (const unsigned char*)active, 0);
}

int shim_residual(const void* b, const void* ax, void* r, uint64_t n, void* out, const void* pinv) {
    return (int)launch_residual((const cplx*)b, (const cplx*)ax, (cplx*)r, n, (double*)out, (const cplx*)pinv, 0);
}

int shim_interleave(const void* src, void* dst, uint64_t n, int nsrc, int nrhs, int to_block) {
    return (int)launch_interleave((const cplx*)src, (cplx*)dst, n, nsrc, nrhs, to_block, 0);
}

int shim_sync() { return (int)cudaStreamSynchronize(0); }

}  // extern "C"
