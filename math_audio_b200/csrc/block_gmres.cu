// block_gmres.cu -- multi-RHS solve (BASELINE config 5): nrhs independent restarted GMRES solves
// advanced in LOCKSTEP so that they share one block matvec per iteration (A is read once for all
// right-hand sides: FP64 tensor-core ZGEMM instead of nrhs HBM-bound ZGEMVs).
//
// Semantics = the reference's: every right-hand side goes through exactly the operations of its
// own `gmres(operator, b_s, config)` call (math-solvers/src/iterative/gmres.rs:96-277): own
// Krylov basis, Hessenberg matrix, Givens rotations, convergence test, restart counter.  A
// right-hand side that has converged simply stops taking part (its column of the block still
// rides along in the matvec).  There is no coupling between the right-hand sides (this is
// "batched GMRES", not block-Krylov), so results are those of nrhs separate solves.  The host
// arithmetic of each right-hand side's cycle is the single-RHS solver's (GmresCycle, gmres_host.h).
#include <cmath>
#include <cstring>
#include <vector>

#include "api_internal.h"
#include "gmres_host.h"
#include "linalg.h"
#include "schwarz.h"

using namespace bemb;

namespace bemb {
int nccl_allgather_bytes(bemb200_ctx* ctx, const void* send, void* recv, size_t count_bytes);
}

namespace {

struct Rhs {
    bool active = false;   // still iterating
    bool done = false;     // result final
    double b_norm = 0.0;
    GmresCycle cycle;
    bemb200_gmres_info info{0, 0, 0.0, 0};
};

// Workspace of one call: stream-ordered allocations from the device's (cached) memory pool -- cudaMalloc / cudaFree of half a
// gigabyte of Krylov bases per call synchronise the device and were measured to cost anything between 1 and 200 ms.
struct DevBuf {
    cudaStream_t stream = nullptr;
    std::vector<void*> ptrs;
    explicit DevBuf(cudaStream_t s) : stream(s) {}
    template <class T>
    cudaError_t alloc(T** p, size_t count) {
        cudaError_t e = cudaMallocAsync((void**)p, (count ? count : 1) * sizeof(T), stream);
        if (e == cudaSuccess) ptrs.push_back(*p);
        return e;
    }
    ~DevBuf() {
        for (void* p : ptrs) cudaFreeAsync(p, stream);
    }
};

}  // namespace

// `sp` != NULL: nrhs independent gmres_preconditioned() solves (gmres.rs:282-585) with the block-Jacobi preconditioner: M^-1 acts on
// the rank's slab of the block product before the exchange, residuals are M^-1 (B - A X), norms relative to ||M^-1 b||.
// `device_io`: b_all / x_all are device arrays of the matrix's device; B is interleaved straight from b_all and X
// de-interleaved straight into x_all (no staging copy, no host round trip).
static int gmres_batched_impl(const bemb200_matrix* cm, const bemb200_precond* sp, const double* b_all, uint32_t nrhs,
                              uint32_t max_iterations, uint32_t restart, double tolerance, double* x_all, bemb200_gmres_info* infos,
                              double* block_matvec_ms, uint64_t* block_matvecs, bool device_io = false) {
    bemb200_matrix* m = const_cast<bemb200_matrix*>(cm);
    if (!m || !b_all || !x_all || !infos) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    bemb200_ctx* ctx = m->ctx;
    if (device_io && (!device_ptr_on(ctx->device, b_all) || !device_ptr_on(ctx->device, x_all)))
        return set_error(ctx, BEMB200_EINVAL, "b_dev / x_dev are not device memory of the matrix's device");
    if (sp && (sp->ctx != ctx || sp->n != m->n_rows || sp->r0 != m->r0 || sp->r1 != m->r1))
        return set_error(ctx, BEMB200_EINVAL, "preconditioner was built for another operator shape / context");
    if (sp && !sp->disjoint)
        return set_error(ctx, BEMB200_EUNSUPPORTED, "batched GMRES takes block-Jacobi (disjoint subdomains covering every row) only");
    if (m->n_rows != m->n_cols) return set_error(ctx, BEMB200_EINVAL, "gmres needs a square operator");
    if (restart == 0 || nrhs == 0 || nrhs > 32) return set_error(ctx, BEMB200_EINVAL, "need 1 <= nrhs <= 32 and restart >= 1");
    const uint64_t n = m->n_rows;
    if (n > 196608) return set_error(ctx, BEMB200_EUNSUPPORTED, "batched GMRES supports up to 196608 unknowns in this version");
    {
        uint64_t b = 0, e = 0;
        bemb200_partition(n, ctx->nranks, ctx->rank, &b, &e);
        if (m->r0 != b || m->r1 != e) return set_error(ctx, BEMB200_EINVAL, "matrix slab is not this rank's canonical row block");
    }
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const int S = (int)((nrhs + 7) / 8 * 8);  // padded block width
    const int mm = (int)restart;
    const uint64_t chunk = (n + ctx->nranks - 1) / ctx->nranks;
    const uint64_t npad = chunk * ctx->nranks;
    const uint64_t nloc = m->r1 - m->r0;
    const uint64_t ldv = npad, vstride = (uint64_t)(mm + 1) * npad;
    const uint64_t hstride = (uint64_t)(mm + 2);

    DevBuf buf(s);
    cplx *Vall, *Xblk, *Yblk, *Bblk, *Rblk, *Xsol, *stage, *hcol_d, *ycoef_d;
    double *scal_d;
    int* cnt_d;
    unsigned char* active_d;
    BEMB_CUDA(ctx, buf.alloc(&Vall, (size_t)S * vstride));
    BEMB_CUDA(ctx, buf.alloc(&Xblk, npad * S));
    BEMB_CUDA(ctx, buf.alloc(&Yblk, npad * S));
    BEMB_CUDA(ctx, buf.alloc(&Bblk, npad * S));
    BEMB_CUDA(ctx, buf.alloc(&Rblk, npad * S));
    BEMB_CUDA(ctx, buf.alloc(&Xsol, npad * S));
    BEMB_CUDA(ctx, buf.alloc(&stage, device_io ? 0 : (size_t)nrhs * n));
    cplx* Pslab = nullptr;  // this rank's slab of a block before M^-1
    if (sp) BEMB_CUDA(ctx, buf.alloc(&Pslab, (nloc ? nloc : 1) * (size_t)S));
    BEMB_CUDA(ctx, buf.alloc(&hcol_d, (size_t)S * hstride));
    BEMB_CUDA(ctx, buf.alloc(&ycoef_d, (size_t)S * mm));
    BEMB_CUDA(ctx, buf.alloc(&scal_d, (size_t)S));
    BEMB_CUDA(ctx, buf.alloc(&cnt_d, (size_t)S));
    BEMB_CUDA(ctx, buf.alloc(&active_d, (size_t)S));
    std::vector<cplx> hcol_h((size_t)S * hstride), ycoef_h((size_t)S * mm);
    std::vector<double> scal_h(S);
    std::vector<int> cnt_h(S);
    std::vector<unsigned char> active_h(S);
    struct EvGuard { cudaEvent_t a = nullptr, b = nullptr; ~EvGuard() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); } } evg;
    BEMB_CUDA(ctx, cudaEventCreate(&evg.a));  // the guard owns both events from the start: nothing leaks if the second create fails
    BEMB_CUDA(ctx, cudaEventCreate(&evg.b));
    const cudaEvent_t e0 = evg.a, e1 = evg.b;
    double mv_ms = 0.0;
    uint64_t mv_count = 0;

    BEMB_CUDA(ctx, cudaMemsetAsync(Vall, 0, (size_t)S * vstride * sizeof(cplx), s));
    BEMB_CUDA(ctx, cudaMemsetAsync(Xblk, 0, npad * S * sizeof(cplx), s));
    BEMB_CUDA(ctx, cudaMemsetAsync(Yblk, 0, npad * S * sizeof(cplx), s));
    BEMB_CUDA(ctx, cudaMemsetAsync(Xsol, 0, npad * S * sizeof(cplx), s));
    if (device_io) {
        BEMB_CUDA(ctx, launch_interleave((const cplx*)b_all, Bblk, n, (int)nrhs, S, 1, s));
    } else {
        BEMB_CUDA(ctx, cudaMemcpyAsync(stage, b_all, (size_t)nrhs * n * sizeof(cplx), cudaMemcpyHostToDevice, s));
        BEMB_CUDA(ctx, launch_interleave(stage, Bblk, n, (int)nrhs, S, 1, s));
    }

    bool precond_in_matvec = false;  // on inside the Arnoldi loop; the residual products need the bare A X
    // Z (npad x S) = M^-1 R for a whole block: every rank solves on its slab, the slabs are gathered
    auto precond_full = [&](const cplx* R, cplx* Z) -> int {
        const uint64_t off = (ctx->nranks > 1 ? (uint64_t)ctx->rank * chunk : m->r0) * S;
        BEMB_CUDA(ctx, schwarz_apply_block_local(sp, R + m->r0 * S, Z + off, S, s));
        if (ctx->nranks > 1) return nccl_allgather_bytes(ctx, Z + off, Z, chunk * S * sizeof(cplx));
        return BEMB200_OK;
    };
    auto block_matvec = [&](const cplx* X, cplx* Y) -> int {
        cplx* yloc = Y + (ctx->nranks > 1 ? (uint64_t)ctx->rank * chunk : m->r0) * S;
        BEMB_CUDA(ctx, cudaEventRecord(e0, s));
        BEMB_CUDA(ctx, launch_zgemm_block(m->A, m->n_cols, nloc, m->n_cols, X, precond_in_matvec ? Pslab : yloc, S, s));
        BEMB_CUDA(ctx, cudaEventRecord(e1, s));
        if (precond_in_matvec) BEMB_CUDA(ctx, schwarz_apply_block_local(sp, Pslab, yloc, S, s));  // w = M^-1 (A v) on this rank's rows
        if (ctx->nranks > 1) {
            int rc = nccl_allgather_bytes(ctx, yloc, Y, chunk * S * sizeof(cplx));
            if (rc != BEMB200_OK) return rc;
        }
        mv_count += 1;
        return BEMB200_OK;
    };
    auto add_mv_time = [&]() {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, e0, e1) == cudaSuccess) mv_ms += ms;
        else cudaGetLastError();
    };
    auto norms = [&](const cplx* B, const cplx* AX, cplx* R) -> int {
        BEMB_CUDA(ctx, launch_block_residual(B, AX, R, n, S, scal_d, s));
        BEMB_CUDA(ctx, cudaMemcpyAsync(scal_h.data(), scal_d, S * sizeof(double), cudaMemcpyDeviceToHost, s));
        BEMB_CUDA(ctx, cudaStreamSynchronize(s));
        return BEMB200_OK;
    };
    auto apply_updates = [&]() -> int {  // X[:, s] += V_s y_s for every s with cnt_h[s] > 0
        bool any = false;
        for (int q = 0; q < S; ++q) any = any || cnt_h[q] > 0;
        if (!any) return BEMB200_OK;
        BEMB_CUDA(ctx, cudaMemcpyAsync(ycoef_d, ycoef_h.data(), ycoef_h.size() * sizeof(cplx), cudaMemcpyHostToDevice, s));
        BEMB_CUDA(ctx, cudaMemcpyAsync(cnt_d, cnt_h.data(), S * sizeof(int), cudaMemcpyHostToDevice, s));
        BEMB_CUDA(ctx, launch_block_update_x(Xsol, Vall, ldv, vstride, ycoef_d, mm, cnt_d, n, S, s));
        BEMB_CUDA(ctx, cudaStreamSynchronize(s));
        return BEMB200_OK;
    };

    std::vector<Rhs> R(S);
    int rc = BEMB200_OK;
    if (sp) {  // ||M^-1 b|| (gmres.rs:455-457)
        rc = precond_full(Bblk, Yblk);
        if (rc == BEMB200_OK) rc = norms(Yblk, nullptr, nullptr);
    } else {
        rc = norms(Bblk, nullptr, nullptr);
    }
    if (rc != BEMB200_OK) return rc;
    for (int q = 0; q < S; ++q) {
        R[q].b_norm = std::sqrt(scal_h[q]);
        if (q >= (int)nrhs) { R[q].done = true; continue; }
        if (R[q].b_norm < 1e-15) {  // gmres.rs:125-135
            R[q].done = true;
            R[q].info = bemb200_gmres_info{0, 0, 0.0, 1};
        }
    }
    auto all_done = [&]() {
        for (int q = 0; q < (int)nrhs; ++q)
            if (!R[q].done) return false;
        return true;
    };

    for (uint32_t outer = 0; outer < max_iterations && !all_done(); ++outer) {
        precond_in_matvec = false;
        rc = block_matvec(Xsol, Yblk);
        if (rc != BEMB200_OK) return rc;
        rc = norms(Bblk, Yblk, Rblk);
        if (rc == BEMB200_OK && sp) {  // r = M^-1 (b - A x) (gmres.rs:473-476)
            rc = precond_full(Rblk, Yblk);
            if (rc == BEMB200_OK) rc = norms(Yblk, nullptr, Rblk);
        }
        if (rc != BEMB200_OK) return rc;
        add_mv_time();
        precond_in_matvec = sp != nullptr;
        for (int q = 0; q < S; ++q) R[q].active = false;
        std::vector<double> scale(S, 0.0);
        for (int q = 0; q < S; ++q) {
            Rhs& r = R[q];
            if (r.done) continue;
            const double beta = std::sqrt(scal_h[q]);
            const double rel = beta / r.b_norm;
            if (rel < tolerance) {  // gmres.rs:148-157
                r.done = true;
                r.info.residual = rel;
                r.info.converged = 1;
                continue;
            }
            r.active = true;
            r.cycle.start(mm, beta);
            scale[q] = 1.0 / beta;
        }
        if (all_done()) break;
        BEMB_CUDA(ctx, cudaMemcpyAsync(scal_d, scale.data(), S * sizeof(double), cudaMemcpyHostToDevice, s));
        BEMB_CUDA(ctx, launch_block_scale(Rblk, scal_d, Vall, vstride, Xblk, n, S, s));  // inactive columns become 0
        for (int q = 0; q < S; ++q) active_h[q] = R[q].active ? 1 : 0;
        BEMB_CUDA(ctx, cudaMemcpyAsync(active_d, active_h.data(), S, cudaMemcpyHostToDevice, s));
        BEMB_CUDA(ctx, cudaStreamSynchronize(s));  // `scale` lives on the host stack
        for (int j = 0; j < mm; ++j) {
            bool any_active = false;
            for (int q = 0; q < S; ++q) any_active = any_active || R[q].active;
            if (!any_active) break;
            rc = block_matvec(Xblk, Yblk);
            if (rc != BEMB200_OK) return rc;
            BEMB_CUDA(ctx, launch_mgs_batched(S, Vall, ldv, vstride, Yblk, j, n, hcol_d, hstride, Xblk, active_d, s));
            BEMB_CUDA(ctx, cudaMemcpyAsync(hcol_h.data(), hcol_d, (size_t)S * hstride * sizeof(cplx), cudaMemcpyDeviceToHost, s));
            BEMB_CUDA(ctx, cudaStreamSynchronize(s));
            add_mv_time();
            std::fill(cnt_h.begin(), cnt_h.end(), 0);
            bool changed = false;
            for (int q = 0; q < S; ++q) {
                Rhs& r = R[q];
                if (!r.active) continue;
                r.info.iterations += 1;
                bool breakdown = false;
                const double rel_res = r.cycle.add_column(j, hcol_h.data() + (size_t)q * hstride, r.b_norm, &breakdown);
                if (rel_res < tolerance || breakdown) {
                    std::vector<cplx> y;
                    r.cycle.solve(j + 1, y);
                    for (int i = 0; i < (int)y.size(); ++i) ycoef_h[(size_t)q * mm + i] = y[i];
                    cnt_h[q] = (int)y.size();
                    r.active = false;
                    r.done = true;
                    r.info.residual = rel_res;
                    r.info.converged = 1;
                    changed = true;
                }
            }
            if (changed) {
                rc = apply_updates();
                if (rc != BEMB200_OK) return rc;
                for (int q = 0; q < S; ++q) active_h[q] = R[q].active ? 1 : 0;
                BEMB_CUDA(ctx, cudaMemcpyAsync(active_d, active_h.data(), S, cudaMemcpyHostToDevice, s));
                BEMB_CUDA(ctx, cudaStreamSynchronize(s));
            }
        }
        // cycle exhausted for the still-active right-hand sides: x += V y, restart (gmres.rs:255-262)
        std::fill(cnt_h.begin(), cnt_h.end(), 0);
        for (int q = 0; q < S; ++q) {
            Rhs& r = R[q];
            if (!r.active) continue;
            std::vector<cplx> y;
            r.cycle.solve(mm, y);
            for (int i = 0; i < (int)y.size(); ++i) ycoef_h[(size_t)q * mm + i] = y[i];
            cnt_h[q] = (int)y.size();
            r.info.restarts += 1;
            r.active = false;
        }
        rc = apply_updates();
        if (rc != BEMB200_OK) return rc;
    }
    if (!all_done()) {  // budget exhausted: true residual, converged = false (gmres.rs:264-276)
        precond_in_matvec = false;
        rc = block_matvec(Xsol, Yblk);
        if (rc != BEMB200_OK) return rc;
        rc = norms(Bblk, Yblk, Rblk);
        if (rc == BEMB200_OK && sp) {
            rc = precond_full(Rblk, Yblk);
            if (rc == BEMB200_OK) rc = norms(Yblk, nullptr, Rblk);
        }
        if (rc != BEMB200_OK) return rc;
        add_mv_time();
        for (int q = 0; q < (int)nrhs; ++q)
            if (!R[q].done) {
                R[q].info.residual = std::sqrt(scal_h[q]) / R[q].b_norm;
                R[q].info.converged = 0;
                R[q].done = true;
            }
    }
    if (device_io) {
        BEMB_CUDA(ctx, launch_interleave(Xsol, (cplx*)x_all, n, (int)nrhs, S, 0, s));
    } else {
        BEMB_CUDA(ctx, launch_interleave(Xsol, stage, n, (int)nrhs, S, 0, s));
        BEMB_CUDA(ctx, cudaMemcpyAsync(x_all, stage, (size_t)nrhs * n * sizeof(cplx), cudaMemcpyDeviceToHost, s));
    }
    BEMB_CUDA(ctx, cudaStreamSynchronize(s));
    for (uint32_t q = 0; q < nrhs; ++q) infos[q] = R[q].info;
    if (block_matvec_ms) *block_matvec_ms = mv_ms;
    if (block_matvecs) *block_matvecs = mv_count;
    return BEMB200_OK;
}

extern "C" int bemb200_gmres_batched(const bemb200_matrix* cm, const double* b_all, uint32_t nrhs, uint32_t max_iterations,
                                     uint32_t restart, double tolerance, double* x_all, bemb200_gmres_info* infos,
                                     double* block_matvec_ms, uint64_t* block_matvecs) {
    return gmres_batched_impl(cm, nullptr, b_all, nrhs, max_iterations, restart, tolerance, x_all, infos, block_matvec_ms, block_matvecs);
}

extern "C" int bemb200_gmres_batched_schwarz(const bemb200_matrix* cm, const bemb200_precond* precond, const double* b_all, uint32_t nrhs,
                                             uint32_t max_iterations, uint32_t restart, double tolerance, double* x_all,
                                             bemb200_gmres_info* infos, double* block_matvec_ms, uint64_t* block_matvecs) {
    if (!precond) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    return gmres_batched_impl(cm, precond, b_all, nrhs, max_iterations, restart, tolerance, x_all, infos, block_matvec_ms, block_matvecs);
}

extern "C" int bemb200_gmres_batched_device(const bemb200_matrix* cm, const bemb200_precond* precond, const double* b_dev, uint32_t nrhs,
                                            uint32_t max_iterations, uint32_t restart, double tolerance, double* x_dev,
                                            bemb200_gmres_info* infos, double* block_matvec_ms, uint64_t* block_matvecs) {
    return gmres_batched_impl(cm, precond, b_dev, nrhs, max_iterations, restart, tolerance, x_dev, infos, block_matvec_ms, block_matvecs,
                              true);
}

// Y = A X for a block of nrhs right-hand sides (each contiguous on the host): the tensor-core
// block matvec on its own (LinearOperator::apply applied to nrhs vectors at once).
extern "C" int bemb200_apply_block(const bemb200_matrix* cm, const double* x_all, uint32_t nrhs, double* y_all, double* kernel_ms) {
    bemb200_matrix* m = const_cast<bemb200_matrix*>(cm);
    if (!m || !x_all || !y_all) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    bemb200_ctx* ctx = m->ctx;
    if (nrhs == 0 || nrhs > 32) return set_error(ctx, BEMB200_EINVAL, "need 1 <= nrhs <= 32");
    {
        uint64_t b = 0, e = 0;  // row-sharded operator: every rank multiplies its canonical row block, the slabs are gathered
        bemb200_partition(m->n_rows, ctx->nranks, ctx->rank, &b, &e);
        if (m->r0 != b || m->r1 != e) return set_error(ctx, BEMB200_EINVAL, "apply_block needs the whole operator (every rank its canonical row block)");
    }
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const int S = (int)((nrhs + 7) / 8 * 8);
    const uint64_t nc = m->n_cols, nr = m->n_rows, nloc = m->r1 - m->r0;
    const uint64_t chunk = (nr + ctx->nranks - 1) / ctx->nranks, npad = chunk * ctx->nranks;
    DevBuf buf(s);
    cplx *Xb, *Yb, *stage;
    BEMB_CUDA(ctx, buf.alloc(&Xb, nc * S));
    BEMB_CUDA(ctx, buf.alloc(&Yb, npad * S));
    BEMB_CUDA(ctx, buf.alloc(&stage, (size_t)nrhs * (nc > nr ? nc : nr)));
    struct EvGuard { cudaEvent_t a = nullptr, b = nullptr; ~EvGuard() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); } } evg;
    BEMB_CUDA(ctx, cudaEventCreate(&evg.a));
    BEMB_CUDA(ctx, cudaEventCreate(&evg.b));
    const cudaEvent_t e0 = evg.a, e1 = evg.b;
    BEMB_CUDA(ctx, cudaMemcpyAsync(stage, x_all, (size_t)nrhs * nc * sizeof(cplx), cudaMemcpyHostToDevice, s));
    BEMB_CUDA(ctx, launch_interleave(stage, Xb, nc, (int)nrhs, S, 1, s));
    cplx* yloc = Yb + m->r0 * S;  // r0 = rank * chunk
    BEMB_CUDA(ctx, launch_zgemm_block(m->A, nc, nloc, nc, Xb, yloc, S, s));  // warm-up
    BEMB_CUDA(ctx, cudaEventRecord(e0, s));
    BEMB_CUDA(ctx, launch_zgemm_block(m->A, nc, nloc, nc, Xb, yloc, S, s));
    BEMB_CUDA(ctx, cudaEventRecord(e1, s));
    if (ctx->nranks > 1) {
        int rc = nccl_allgather_bytes(ctx, yloc, Yb, chunk * S * sizeof(cplx));
        if (rc != BEMB200_OK) return rc;
    }
    BEMB_CUDA(ctx, launch_interleave(Yb, stage, nr, (int)nrhs, S, 0, s));
    BEMB_CUDA(ctx, cudaMemcpyAsync(y_all, stage, (size_t)nrhs * nr * sizeof(cplx), cudaMemcpyDeviceToHost, s));
    BEMB_CUDA(ctx, cudaStreamSynchronize(s));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    if (kernel_ms) *kernel_ms = ms;
    return BEMB200_OK;
}
