// gmres.cu -- operator application and restarted GMRES on a device-resident, row-sharded
// matrix.  Host control flow restates math-solvers/src/iterative/gmres.rs:105-277 (restart
// semantics, iteration counting, relative residual vs ||b||, zero-RHS early return); the
// Hessenberg / Givens arithmetic of a cycle (conj(c), conj(s), breakdown 1e-14) is GmresCycle
// of gmres_host.h, shared with the batched solver.  All O(N) and O(N^2) work runs in the
// kernels of linalg.cu.
//
// Multi-GPU layout ("sharded matvec, replicated Arnoldi"): rank p owns rows
// [p*chunk,(p+1)*chunk) of A; after the local GEMV the slices of y are all-gathered (NCCL,
// 16*N bytes) and EVERY rank runs the same deterministic cluster MGS kernel on the full
// vectors, so all ranks hold bit-identical Krylov bases and Hessenberg columns and take the
// same convergence decisions without any all-reduce.
#include <chrono>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <vector>

#include "api_internal.h"
#include "gmres_fused.h"
#include "gmres_host.h"
#include "linalg.h"
#include "schwarz.h"

using namespace bemb;

namespace bemb {
int nccl_allgather_bytes(bemb200_ctx* ctx, const void* send, void* recv, size_t count_bytes);
}

struct GmresWorkspace {
    uint64_t n = 0, npad = 0, chunk = 0;
    uint32_t restart = 0;
    cplx* V = nullptr;      // (restart+1) x npad
    cplx* w = nullptr;      // npad  (matvec output / Arnoldi work vector)
    cplx* r = nullptr;      // npad
    cplx* xin = nullptr;    // npad  staging for host-pointer calls
    cplx* bin = nullptr;    // npad
    cplx* xout = nullptr;   // npad
    cplx* hcol_d = nullptr; // (restart+1) slots x (restart+2): one Hessenberg column per in-flight iteration
    cplx* ycoef_d = nullptr;
    cplx* lmat_d = nullptr;  // (restart+1)^2 Gram triangle of the current cycle (low-sync MGS kernel)
    double* scal_d = nullptr;
    cplx* hcol_h = nullptr;   // pinned, same shape as hcol_d
    double* scal_h = nullptr; // pinned
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // per-iteration events: matvec start/stop and "column j is on the host"
    std::vector<cudaEvent_t> it_ev0, it_ev1, it_done;
    std::vector<char> launched;
    uint32_t ldh_slot = 0;
};

static void destroy_workspace(GmresWorkspace* ws) {
    if (!ws) return;
    cudaFree(ws->V); cudaFree(ws->w); cudaFree(ws->r); cudaFree(ws->xin); cudaFree(ws->bin); cudaFree(ws->xout);
    cudaFree(ws->hcol_d); cudaFree(ws->ycoef_d); cudaFree(ws->scal_d); cudaFree(ws->lmat_d);
    if (ws->hcol_h) cudaFreeHost(ws->hcol_h);
    if (ws->scal_h) cudaFreeHost(ws->scal_h);
    if (ws->ev0) cudaEventDestroy(ws->ev0);
    if (ws->ev1) cudaEventDestroy(ws->ev1);
    for (auto* v : {&ws->it_ev0, &ws->it_ev1, &ws->it_done})
        for (cudaEvent_t e : *v)
            if (e) cudaEventDestroy(e);
    delete ws;
    cudaGetLastError();
}

namespace bemb {
void free_workspace(bemb200_matrix* m) {
    destroy_workspace(m->ws);
    m->ws = nullptr;
}
}  // namespace bemb

// ---- peer-memory exchange (row-sharded solve) ----------------------------------------------
// Collective over the ranks of ctx (called at the start of a solve, the same sequence on every
// rank).  On success the Arnoldi matvec stores its slab of y directly into every rank's work
// vector (ZGEMV epilogue over NVLink) and the Gram-Schmidt kernel waits for the per-rank epoch
// flags: the NCCL all-gather and its two kernel boundaries leave the iteration.  Any failure
// (no peer access, IPC refused by the platform) is agreed on by all ranks and leaves the NCCL
// all-gather path in place.  BEMB200_PEER_FUSED=0 disables it.
constexpr size_t PX_HEADER = 256;
constexpr size_t PX_RPART_BYTES = 2 * (size_t)MAX_PEERS * FUSED_KMAX * 2 * sizeof(uint4);
static inline size_t px_bytes(uint64_t npad) { return PX_HEADER + 2 * npad * 2 * sizeof(uint4) + PX_RPART_BYTES; }
namespace bemb {
void free_peer_exchange(bemb200_ctx* ctx, bool collective) {
    PeerExchange& px = ctx->px;
    if (!ctx->group)  // (ranks of one process share plain pointers: nothing to unmap)
        for (int p = 0; p < ctx->nranks && p < 8; ++p)
            if (p != ctx->rank && px.base[p]) cudaIpcCloseMemHandle(px.base[p]);
    bool may_free = true;
    if (px.ok) {
        // nobody frees exported memory while a peer may still have it mapped
        if (collective && ctx->nccl_comm) {
            unsigned char* tok = nullptr;
            if (cudaMalloc((void**)&tok, (size_t)ctx->nranks) == cudaSuccess) {
                nccl_allgather_bytes(ctx, tok + ctx->rank, tok, 1);
                cudaStreamSynchronize(ctx->stream);
                cudaFree(tok);
            }
        } else {
            // context destruction is not a collective call (a peer may already be gone, and waiting for it could
            // hang this process): keep the few MB alive until the process exits rather than risk either
            may_free = false;
        }
    }
    if (px.local && may_free) cudaFree(px.local);
    if (px.err_h) cudaFreeHost(px.err_h);
    px = PeerExchange();
    FusedLocal& fx = ctx->fx;
    if (fx.cpart) cudaFree(fx.cpart);
    if (fx.hbuf) cudaFree(fx.hbuf);
    if (fx.trace_d) cudaFree(fx.trace_d);
    if (fx.row_off_d) cudaFree(fx.row_off_d);
    if (fx.frag) cudaFree(fx.frag);
    if (fx.result_h) cudaFreeHost(fx.result_h);
    fx = FusedLocal();
    cudaGetLastError();
}
}  // namespace bemb

static int ensure_peer_exchange(bemb200_ctx* ctx, uint64_t npad) {
    PeerExchange& px = ctx->px;
    static const bool enabled = []() { const char* v = std::getenv("BEMB200_PEER_FUSED"); return v ? std::atoi(v) != 0 : true; }();
    if (!enabled || ctx->nranks < 2 || ctx->nranks > MAX_PEERS || !ctx->nccl_comm) return BEMB200_OK;
    if (px.tried && (!px.ok || px.npad >= npad)) return BEMB200_OK;
    if (px.tried) free_peer_exchange(ctx, true);  // a larger operator: re-establish (collective, same on every rank)
    px.tried = true;
    px.npad = npad;
    const int P = ctx->nranks;
    const size_t bytes = px_bytes(npad);  // two epochs x npad elements x 32 B + the fused kernel's inbox of rank partials
    int ok = 1;
    cudaIpcMemHandle_t mine;
    std::memset(&mine, 0, sizeof(mine));
    if (cudaMalloc((void**)&px.local, bytes) != cudaSuccess) { ok = 0; px.local = nullptr; }
    if (ok && cudaMemsetAsync(px.local, 0, bytes, ctx->stream) != cudaSuccess) ok = 0;
    if (ok && cudaIpcGetMemHandle(&mine, px.local) != cudaSuccess) ok = 0;
    if (ok && cudaHostAlloc((void**)&px.err_h, sizeof(int), cudaHostAllocMapped) != cudaSuccess) { ok = 0; px.err_h = nullptr; }
    if (px.err_h) *px.err_h = 0;
    cudaGetLastError();
    // exchange {handle, ok} through the communicator
    struct Slot { cudaIpcMemHandle_t h; int ok; int pad[3]; char uuid[16]; };
    static_assert(sizeof(Slot) % 16 == 0, "slot alignment");
    std::vector<Slot> all(P);
    Slot me{};
    me.h = mine;
    me.ok = ok;
    {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, ctx->device) == cudaSuccess) std::memcpy(me.uuid, prop.uuid.bytes, 16);
        else { cudaGetLastError(); me.ok = ok = 0; }
    }
    unsigned char* stage = nullptr;
    BEMB_CUDA(ctx, cudaMalloc((void**)&stage, sizeof(Slot) * P));
    BEMB_CUDA(ctx, cudaMemcpyAsync(stage + sizeof(Slot) * ctx->rank, &me, sizeof(Slot), cudaMemcpyHostToDevice, ctx->stream));
    int rc = nccl_allgather_bytes(ctx, stage + sizeof(Slot) * ctx->rank, stage, sizeof(Slot));
    if (rc != BEMB200_OK) { cudaFree(stage); return rc; }
    BEMB_CUDA(ctx, cudaMemcpyAsync(all.data(), stage, sizeof(Slot) * P, cudaMemcpyDeviceToHost, ctx->stream));
    BEMB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int p = 0; p < P; ++p) ok &= all[p].ok;
    // two ranks on ONE device cannot run the spinning consumer and the producer ZGEMV side by side (separate
    // processes time-slice a GPU): such a job keeps the NCCL all-gather
    for (int p = 0; p < P; ++p)
        for (int q = p + 1; q < P; ++q)
            if (std::memcmp(all[p].uuid, all[q].uuid, 16) == 0) ok = 0;
    if (ok) {
        for (int p = 0; p < P; ++p) {
            if (p == ctx->rank) { px.base[p] = px.local; continue; }
            void* ptr = nullptr;
            if (cudaIpcOpenMemHandle(&ptr, all[p].h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { ok = 0; cudaGetLastError(); break; }
            px.base[p] = static_cast<unsigned char*>(ptr);
        }
    }
    // second round: did every rank map every peer?
    me.ok = ok;
    BEMB_CUDA(ctx, cudaMemcpyAsync(stage + sizeof(Slot) * ctx->rank, &me, sizeof(Slot), cudaMemcpyHostToDevice, ctx->stream));
    rc = nccl_allgather_bytes(ctx, stage + sizeof(Slot) * ctx->rank, stage, sizeof(Slot));
    if (rc != BEMB200_OK) { cudaFree(stage); return rc; }
    BEMB_CUDA(ctx, cudaMemcpyAsync(all.data(), stage, sizeof(Slot) * P, cudaMemcpyDeviceToHost, ctx->stream));
    BEMB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaFree(stage);
    for (int p = 0; p < P; ++p) ok &= all[p].ok;
    px.ok = ok != 0;
    px.epoch = 0;
    if (!px.ok) {
        for (int p = 0; p < P; ++p)
            if (p != ctx->rank && px.base[p]) { cudaIpcCloseMemHandle(px.base[p]); px.base[p] = nullptr; }
        if (px.local) { cudaFree(px.local); px.local = nullptr; }
        cudaGetLastError();
    }
    return BEMB200_OK;
}

static inline uint4* px_work(const PeerExchange& px, int p, unsigned long long epoch) {
    return reinterpret_cast<uint4*>(px.base[p] + PX_HEADER) + (epoch & 1ull) * 2 * px.npad;
}

// The workspace is built in a local object and attached to the matrix only when EVERY allocation has
// succeeded: a failed attempt (OOM next to a slab that nearly fills HBM is realistic) leaves the handle
// without a workspace instead of a half-built one that later calls would dereference.
static int build_workspace(bemb200_matrix* m, uint32_t restart, GmresWorkspace* ws) {
    bemb200_ctx* ctx = m->ctx;
    ws->n = m->n_rows;
    ws->chunk = (m->n_rows + ctx->nranks - 1) / ctx->nranks;
    ws->npad = ws->chunk * ctx->nranks;
    if (m->n_cols > ws->npad) ws->npad = m->n_cols;
    ws->restart = restart;
    const size_t vb = ws->npad * sizeof(cplx);
    BEMB_CUDA(ctx, cudaMalloc((void**)&ws->V, (size_t)(restart + 1) * vb));
    BEMB_CUDA(ctx, cudaMalloc((void**)&ws->w, vb));
    BEMB_CUDA(ctx, cudaMalloc((void**)&ws->r, vb));
    BEMB_CUDA(ctx, cudaMalloc((void**)&ws->xin, vb));
    BEMB_CUDA(ctx, cudaMalloc((void**)&ws->bin, vb));
    BEMB_CUDA(ctx, cudaMalloc((void**)&ws->xout, vb));
    ws->ldh_slot = restart + 2;
    BEMB_CUDA(ctx, cudaMalloc((void**)&ws->hcol_d, (size_t)(restart + 1) * ws->ldh_slot * sizeof(cplx)));
    BEMB_CUDA(ctx, cudaMalloc((void**)&ws->ycoef_d, (restart + 2) * sizeof(cplx)));
    BEMB_CUDA(ctx, cudaMalloc((void**)&ws->lmat_d, ((size_t)(restart + 1) * (restart + 1) + mgs_scratch_elems()) * sizeof(cplx)));
    BEMB_CUDA(ctx, cudaMalloc((void**)&ws->scal_d, 4 * sizeof(double)));
    BEMB_CUDA(ctx, cudaMallocHost((void**)&ws->hcol_h, (size_t)(restart + 1) * ws->ldh_slot * sizeof(cplx)));
    ws->it_ev0.assign(restart + 1, nullptr); ws->it_ev1.assign(restart + 1, nullptr); ws->it_done.assign(restart + 1, nullptr);
    ws->launched.assign(restart + 1, 0);
    for (uint32_t i = 0; i <= restart; ++i) {
        BEMB_CUDA(ctx, cudaEventCreate(&ws->it_ev0[i]));
        BEMB_CUDA(ctx, cudaEventCreate(&ws->it_ev1[i]));
        BEMB_CUDA(ctx, cudaEventCreate(&ws->it_done[i]));
    }
    BEMB_CUDA(ctx, cudaMallocHost((void**)&ws->scal_h, 4 * sizeof(double)));
    BEMB_CUDA(ctx, cudaEventCreate(&ws->ev0));
    BEMB_CUDA(ctx, cudaEventCreate(&ws->ev1));
    BEMB_CUDA(ctx, cudaMemsetAsync(ws->w, 0, vb, ctx->stream));
    return BEMB200_OK;
}

static int ensure_workspace(bemb200_matrix* m, uint32_t restart) {
    if (m->ws && m->ws->restart >= restart) return BEMB200_OK;
    free_workspace(m);
    if ((uint64_t)restart + 1 > (1ull << 40) / ((m->n_rows + 1) * sizeof(cplx)))  // > 1 TiB of basis vectors: refuse before asking CUDA
        return set_error(m->ctx, BEMB200_ENOMEM, "GMRES workspace: restart x n does not fit any device");
    GmresWorkspace* ws = new GmresWorkspace();
    const int rc = build_workspace(m, restart, ws);
    if (rc != BEMB200_OK) {
        destroy_workspace(ws);
        return rc;
    }
    m->ws = ws;
    return BEMB200_OK;
}

// y_full = A x  (x: n_cols on device, y_full: npad on device, valid in [0, n_rows))
static int matvec(bemb200_matrix* m, const cplx* x, cplx* y_full, bool timed) {
    bemb200_ctx* ctx = m->ctx;
    GmresWorkspace* ws = m->ws;
    const uint64_t nloc = m->r1 - m->r0;
    cplx* yloc = y_full + (ctx->nranks > 1 ? (uint64_t)ctx->rank * ws->chunk : m->r0);
    if (timed) BEMB_CUDA(ctx, cudaEventRecord(ws->ev0, ctx->stream));
    BEMB_CUDA(ctx, launch_zgemv(m->A, m->n_cols, nloc, m->n_cols, x, yloc, ctx->stream));
    if (timed) BEMB_CUDA(ctx, cudaEventRecord(ws->ev1, ctx->stream));
    m->last_launches += 1;
    m->last_matvecs += 1;
    if (ctx->nranks > 1) {
        int rc = nccl_allgather_bytes(ctx, yloc, y_full, ws->chunk * sizeof(cplx));
        if (rc != BEMB200_OK) return rc;
    }
    return BEMB200_OK;
}

static void accumulate_matvec_time(bemb200_matrix* m) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, m->ws->ev0, m->ws->ev1) == cudaSuccess) m->last_matvec_ms += ms;
    else cudaGetLastError();
}

static int norm_of(bemb200_matrix* m, const cplx* b, const cplx* ax, cplx* r, double* out, const cplx* pinv = nullptr) {
    bemb200_ctx* ctx = m->ctx;
    GmresWorkspace* ws = m->ws;
    BEMB_CUDA(ctx, launch_residual(b, ax, r, m->n_rows, ws->scal_d, pinv, ctx->stream));
    m->last_launches += 1;
    BEMB_CUDA(ctx, cudaMemcpyAsync(ws->scal_h, ws->scal_d, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    BEMB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *out = std::sqrt(ws->scal_h[0]);
    return BEMB200_OK;
}

// ---- user preconditioner (bemb200_gmres_callback): Preconditioner::apply (traits.rs:366-371) supplied by the caller as a host
// function.  The Arnoldi process stays on the device; only M^-1 makes the round trip through two pinned host vectors.
struct UserPrecond {
    bemb200_precond_fn fn = nullptr;
    void* user = nullptr;
    cplx* r_h = nullptr;  // pinned, n
    cplx* z_h = nullptr;  // pinned, n
    uint64_t calls = 0;
};

// The left preconditioner of gmres_preconditioned_with_guess (gmres.rs:434-585); `left` = false is plain gmres_with_guess.
// With `left`, at most one of the other members is set, and none of them means IdentityPreconditioner.
struct LeftPrecond {
    bool left = false;
    const cplx* pinv = nullptr;                // DiagonalPreconditioner: inverse diagonal on the device, applied inside the
                                               // residual and Gram-Schmidt kernels
    const bemb200_precond* schwarz = nullptr;  // additive Schwarz / block-Jacobi (schwarz.cu)
    UserPrecond* user = nullptr;               // the caller's host function
    // M^-1 is a step of its own between the matvec and the exchange; the fused kernel and peer mode have no room for it
    bool own_step() const { return schwarz || user; }
};

// dst (npad, device) = M^-1 src for a preconditioner with a step of its own; src_loc points at this rank's rows of src.
// Schwarz: every rank solves on its slab, then the slabs are gathered.  Callback: single rank only (checked by the entry
// point), so the slab is the whole vector; src_loc == dst allowed.
static int precond_apply(bemb200_matrix* m, const LeftPrecond& P, const cplx* src_loc, cplx* dst) {
    bemb200_ctx* ctx = m->ctx;
    GmresWorkspace* ws = m->ws;
    if (P.schwarz) {
        const uint64_t off = ctx->nranks > 1 ? (uint64_t)ctx->rank * ws->chunk : m->r0;
        BEMB_CUDA(ctx, schwarz_apply_local(P.schwarz, src_loc, dst + off, ctx->stream));
        m->last_launches += schwarz_apply_launches(P.schwarz);
        if (ctx->nranks > 1) return nccl_allgather_bytes(ctx, dst + off, dst, ws->chunk * sizeof(cplx));
        return BEMB200_OK;
    }
    UserPrecond* up = P.user;
    const size_t nb = m->n_rows * sizeof(cplx);
    BEMB_CUDA(ctx, cudaMemcpyAsync(up->r_h, src_loc, nb, cudaMemcpyDeviceToHost, ctx->stream));
    BEMB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    up->calls += 1;
    const int urc = up->fn(up->user, reinterpret_cast<const double*>(up->r_h), reinterpret_cast<double*>(up->z_h), m->n_rows);
    if (urc != 0) return set_error(ctx, BEMB200_ECALLBACK, "the preconditioner callback returned a non-zero code");
    // z_h is not touched again before the next call has synchronised the stream, i.e. after this copy has completed
    BEMB_CUDA(ctx, cudaMemcpyAsync(dst, up->z_h, nb, cudaMemcpyHostToDevice, ctx->stream));
    return BEMB200_OK;
}

// *out = ||M^-1 (b - A x)|| with A x in ax = ws->w, and M^-1 (b - A x) left in ws->r (gmres.rs:473-476); with ax = nullptr
// *out = ||M^-1 b|| (gmres.rs:455-457).  M = I without a left preconditioner.
static int residual_norm(bemb200_matrix* m, const LeftPrecond& P, const cplx* b, const cplx* ax, double* out) {
    bemb200_ctx* ctx = m->ctx;
    GmresWorkspace* ws = m->ws;
    cplx* r = ax ? ws->r : nullptr;
    if (!P.own_step()) return norm_of(m, b, ax, r, out, P.pinv);
    const cplx* src = b;
    if (ax) {
        BEMB_CUDA(ctx, launch_residual(b, ax, ws->r, m->n_rows, ws->scal_d, nullptr, ctx->stream));  // r = b - A x
        m->last_launches += 1;
        src = ws->r;
    }
    int rc = precond_apply(m, P, src + m->r0, ws->w);
    if (rc != BEMB200_OK) return rc;
    return norm_of(m, ws->w, nullptr, r, out);
}

static int update_x(bemb200_matrix* m, cplx* x, const std::vector<cplx>& y) {
    bemb200_ctx* ctx = m->ctx;
    GmresWorkspace* ws = m->ws;
    if (y.empty()) return BEMB200_OK;
    BEMB_CUDA(ctx, cudaMemcpyAsync(ws->ycoef_d, y.data(), y.size() * sizeof(cplx), cudaMemcpyHostToDevice, ctx->stream));
    BEMB_CUDA(ctx, launch_update_x(x, ws->V, ws->npad, ws->ycoef_d, (int)y.size(), m->n_rows, ctx->stream));
    m->last_launches += 1;
    BEMB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // y lives on the host stack
    return BEMB200_OK;
}

// ---- persistent fused solve (gmres_fused.cu) ----------------------------------------------------------------
// BEMB200_GMRES_FUSED: 0 never, 1 whenever the kernel applies, unset = auto: the ranks of a single-process group always;
// process-per-GPU jobs from 2 ranks on when the solver owns the GPU.  Measured with the final kernel (DESIGN.md section 4.4,
// s/frequency of the config-2 sweep, sequential schedule): 2 GPUs 57.3 ms fused against 61.7 ms for the pipelined per-iteration
// path; 1 GPU 110.3 fused against 103.9 sequential / 101.0 pipelined per-iteration -- on one GPU the hardware-scheduled ZGEMV
// (perfect load balance for free) outweighs the saved launches, from two ranks on the sharded Gram-Schmidt and the single
// exchange per iteration win.
static const int g_fused_mode = []() { const char* v = std::getenv("BEMB200_GMRES_FUSED"); return v ? (std::atoi(v) != 0 ? 1 : 0) : -1; }();

// BEMB200_PEER_TIMEOUT_MS (default 4000): bound of every device-side wait for data of another rank or CTA
static unsigned long long peer_timeout_ns() {
    static const unsigned long long ns = []() {
        const char* v = std::getenv("BEMB200_PEER_TIMEOUT_MS");
        const long long ms = v ? std::atoll(v) : 4000;
        return (unsigned long long)(ms > 0 ? ms : 4000) * 1000000ull;
    }();
    return ns;
}

static double g_fused_total_ms = 0.0, g_fused_matvec_ms = 0.0, g_fused_round_ms = 0.0;
static unsigned long long g_fused_rounds = 0;

// Exchange vectors for the fused kernel.  One rank: a plain local allocation in the PeerExchange layout; several
// ranks: the IPC-mapped allocation of ensure_peer_exchange (collective).  Returns with *ok = false when the
// platform refused peer mappings (the caller then stays on the per-iteration kernels -- agreed by all ranks).
bool bemb::PeerGroup::exchange(int rank, unsigned char* mine, unsigned char** all) {
    std::unique_lock<std::mutex> lk(mu);
    posted[rank] = mine;
    const unsigned long long gen = generation;
    if (++arrived == nranks) {
        for (int p = 0; p < nranks; ++p) snap[p] = posted[p];
        arrived = 0;
        generation += 1;
        cv.notify_all();
    } else if (!cv.wait_for(lk, std::chrono::seconds(60), [&] { return generation != gen; })) {
        arrived -= 1;
        return false;
    }
    for (int p = 0; p < nranks; ++p) all[p] = snap[p];
    return true;
}

static int ensure_fused_exchange(bemb200_ctx* ctx, uint64_t npad, bool* ok) {
    *ok = false;
    PeerExchange& px = ctx->px;
    if (ctx->nranks > 1 && ctx->group) {
        // ranks of one process: plain pointers, exchanged through the group table (collective: every rank of the group is
        // inside the same solve call on its own host thread)
        if (!px.local || px.npad < npad) {
            if (px.local) { cudaFree(px.local); px.local = nullptr; }
            unsigned char* mine = nullptr;
            if (ctx->group->peer_ok && cudaMalloc((void**)&mine, px_bytes(npad)) == cudaSuccess) {
                if (cudaMemsetAsync(mine, 0, px_bytes(npad), ctx->stream) != cudaSuccess || cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
                    cudaFree(mine);
                    mine = nullptr;
                }
            }
            cudaGetLastError();
            unsigned char* all[MAX_GROUP_RANKS];
            if (!ctx->group->exchange(ctx->rank, mine, all)) {
                if (mine) cudaFree(mine);
                return set_error(ctx, BEMB200_ENCCL, "multi-GPU group: a rank never reached the exchange set-up");
            }
            bool every = true;
            for (int p = 0; p < ctx->nranks; ++p) every = every && all[p] != nullptr;
            // second barrier: nobody frees or writes before everybody has taken the table
            unsigned char* dummy[MAX_GROUP_RANKS];
            ctx->group->exchange(ctx->rank, mine, dummy);
            if (!every) {
                if (mine) cudaFree(mine);
                return set_error(ctx, BEMB200_EUNSUPPORTED, "multi-GPU group: peer access between the devices is not available");
            }
            px.local = mine;
            px.npad = npad;
            for (int p = 0; p < ctx->nranks; ++p) px.base[p] = all[p];
        }
    } else if (ctx->nranks > 1) {
        int rc = ensure_peer_exchange(ctx, npad);
        if (rc != BEMB200_OK) return rc;
        if (!px.ok || px.npad < npad) return BEMB200_OK;
    } else if (!px.local || px.npad < npad) {
        if (px.local) { cudaFree(px.local); px.local = nullptr; }
        BEMB_CUDA(ctx, cudaMalloc((void**)&px.local, px_bytes(npad)));
        BEMB_CUDA(ctx, cudaMemsetAsync(px.local, 0, px_bytes(npad), ctx->stream));
        px.npad = npad;
        px.base[0] = px.local;
        // (the epochs keep counting: the CTA inboxes and broadcast slots are older than this allocation)
    }
    FusedLocal& fx = ctx->fx;
    int grid = ctx->fused_grid;
    if (grid <= 0) {
        int sms = 0;
        BEMB_CUDA(ctx, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device));
        grid = sms;
    }
    if (!fx.cpart || fx.grid != grid) {
        if (fx.cpart) cudaFree(fx.cpart);
        if (fx.hbuf) cudaFree(fx.hbuf);
        if (fx.trace_d) cudaFree(fx.trace_d);
        if (fx.row_off_d) cudaFree(fx.row_off_d);
        if (fx.frag) cudaFree(fx.frag);
        fx.frag = nullptr;
        fx.cpart = fx.hbuf = nullptr;
        fx.trace_d = nullptr;
        fx.row_off_d = nullptr;
        fx.speed.clear();
        fx.smid.clear();
        fx.calib_runs = 0;
        BEMB_CUDA(ctx, cudaMalloc((void**)&fx.trace_d, (size_t)grid * 4 * sizeof(unsigned long long)));
        BEMB_CUDA(ctx, cudaMalloc((void**)&fx.row_off_d, ((size_t)grid + 1) * sizeof(uint32_t)));
        BEMB_CUDA(ctx, cudaMalloc((void**)&fx.frag, 2 * ((size_t)grid + 1) * 2 * sizeof(uint4)));
        BEMB_CUDA(ctx, cudaMemsetAsync(fx.frag, 0, 2 * ((size_t)grid + 1) * 2 * sizeof(uint4), ctx->stream));
        const size_t cb = 2 * (size_t)grid * FUSED_KMAX * 2 * sizeof(uint4), hb = 2 * (size_t)FUSED_KMAX * 2 * sizeof(uint4);
        BEMB_CUDA(ctx, cudaMalloc((void**)&fx.cpart, cb));
        BEMB_CUDA(ctx, cudaMalloc((void**)&fx.hbuf, hb));
        BEMB_CUDA(ctx, cudaMemsetAsync(fx.cpart, 0, cb, ctx->stream));
        BEMB_CUDA(ctx, cudaMemsetAsync(fx.hbuf, 0, hb, ctx->stream));
        fx.grid = grid;
        // epochs of the old buffers mean nothing for the new ones, but the inbox of rank partials is older: keep counting
    }
    if (!fx.result_h) {
        BEMB_CUDA(ctx, cudaHostAlloc(&fx.result_h, sizeof(FusedResult), cudaHostAllocMapped));
        BEMB_CUDA(ctx, cudaHostGetDevicePointer(&fx.result_d, fx.result_h, 0));
    }
    *ok = true;
    return BEMB200_OK;
}

// *used = false: the fused kernel does not apply here (restart too long, shared-memory budget, no peer mapping) and
// nothing was done; otherwise the solve is complete and *info is set.
static int gmres_fused_solve(bemb200_matrix* m, const cplx* b, cplx* x, uint32_t max_iterations, uint32_t restart, double tol,
                             bemb200_gmres_info* info, bool precond, const cplx* pinv, bool* used) {
    *used = false;
    bemb200_ctx* ctx = m->ctx;
    GmresWorkspace* ws = m->ws;
    if (g_fused_mode == 0 || ctx->fx.disabled || restart > (uint32_t)FUSED_MAX_RESTART || m->n_rows > 0x7fffffffull) return BEMB200_OK;
    const bool polite = ctx->shared_gpu.load() != 0;  // a background assembly shares the SMs: 96-register build
    if (g_fused_mode < 0 && !ctx->group && (ctx->nranks < 2 || polite)) return BEMB200_OK;
    if (ctx->nranks > 1 && !ctx->group && !ctx->nccl_comm) return BEMB200_OK;
    if (ctx->nranks > MAX_PEERS) return BEMB200_OK;
    bool ok = false;
    int rc = ensure_fused_exchange(ctx, ws->npad, &ok);
    if (rc != BEMB200_OK) return rc;
    if (!ok) return BEMB200_OK;
    FusedLocal& fx = ctx->fx;
    PeerExchange& px = ctx->px;
    FusedParams p{};
    p.A = m->A;
    p.lda = m->n_cols;
    p.n = (uint32_t)m->n_rows;
    p.row0 = (uint32_t)m->r0;
    p.nloc = (uint32_t)(m->r1 - m->r0);
    p.npad = (uint32_t)px.npad;
    p.rank = ctx->rank;
    p.nranks = ctx->nranks;
    p.b = b;
    p.x = x;
    p.V = ws->V;
    p.ldv = ws->npad;
    p.pinv = pinv;
    p.direct_scale = precond ? 1 : 0;
    for (int r = 0; r < ctx->nranks; ++r) {
        p.xbuf[r] = reinterpret_cast<uint4*>(px.base[r] + PX_HEADER);
        p.rpart[r] = p.xbuf[r] + 4 * (size_t)px.npad;
    }
    p.cpart = fx.cpart;
    p.hbuf = fx.hbuf;
    p.restart = restart;
    p.max_cycles = max_iterations;
    p.tol = tol;
    p.ex0 = (uint32_t)px.epoch;
    p.er0 = fx.er;
    p.timeout_ns = peer_timeout_ns();
    p.result = static_cast<FusedResult*>(fx.result_d);
    const uint32_t G = (uint32_t)fx.grid;
    p.S = (p.nloc + G - 1) / G;
    if (p.S == 0) p.S = 1;
    // Row ownership.  SMs do not stream from HBM equally fast (the SMs of fuller GPCs share their path to L2: 86 ... 103 ms per
    // 100 matvecs at 20 480 unknowns), and the slowest CTA sets the pace of every iteration.  The first sizeable solve of a context
    // runs with equal shares and measures rows/ns per CTA (and the SM it sat on); later solves split the slab proportionally.
    // One refinement, then the table is frozen (same inputs -> same bits from then on).
    p.row_off = nullptr;
    p.unit_off = nullptr;
    p.units_per_row = 0;
    p.frag = fx.frag;
    std::vector<uint32_t> off;
    const bool have_speed = fx.speed.size() == G;
    if (p.nloc >= 4 * G) {
        // CTA boundaries in units of (row, segment): shares proportional to the measured speeds (equal before the calibration)
        const uint32_t nsegu = (p.n + FUSED_SEGMENT_WIDTH - 1) / FUSED_SEGMENT_WIDTH;
        const uint64_t total_units = (uint64_t)p.nloc * nsegu;
        double tot = 0.0;
        for (uint32_t c = 0; c < G; ++c) tot += have_speed ? fx.speed[c] : 1.0;
        off.assign(G + 1, 0);
        double cum = 0.0;
        uint32_t smax = 0;
        bool ok_units = total_units < 0xffffffffull;
        for (uint32_t c = 0; c < G && ok_units; ++c) {
            cum += (have_speed ? fx.speed[c] : 1.0) / tot;
            uint64_t e = c + 1 == G ? total_units : (uint64_t)std::llround(cum * (double)total_units);
            if (e > total_units) e = total_units;
            if (e < (uint64_t)off[c] + 2ull * nsegu) ok_units = false;  // every CTA keeps at least two whole rows of work
            off[c + 1] = (uint32_t)e;
            const uint32_t own0 = (off[c] + nsegu - 1) / nsegu, own1 = (off[c + 1] + nsegu - 1) / nsegu;
            if (own1 - own0 + 1 > smax) smax = own1 - own0 + 1;  // + 1: the head-fragment slot
        }
        if (ok_units && smax <= 256) {
            p.S = smax;
            p.units_per_row = nsegu;
            BEMB_CUDA(ctx, cudaMemcpyAsync(fx.row_off_d, off.data(), (G + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
            BEMB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // `off` is pageable host memory
            p.unit_off = fx.row_off_d;
        }
    }
    if (!p.unit_off && have_speed && p.nloc >= 8 * G) {
        double tot = 0.0;
        for (double v : fx.speed) tot += v;
        off.assign(G + 1, 0);
        double cum = 0.0;
        uint32_t smax = 0;
        for (uint32_t c = 0; c < G; ++c) {
            cum += fx.speed[c] / tot;
            uint32_t e = c + 1 == G ? p.nloc : (uint32_t)std::llround(cum * (double)p.nloc);
            if (e < off[c]) e = off[c];
            if (e > p.nloc) e = p.nloc;
            off[c + 1] = e;
            if (e - off[c] > smax) smax = e - off[c];
        }
        p.S = smax ? smax : 1;
        BEMB_CUDA(ctx, cudaMemcpyAsync(fx.row_off_d, off.data(), (G + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
        BEMB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // `off` is pageable host memory
        p.row_off = fx.row_off_d;
    }
    p.rblk = fused_pick_rblk(p.S);
    const size_t smem = fused_smem_bytes(p.S, p.rblk, restart);
    if (smem > 200 * 1024) return BEMB200_OK;
    p.trace = fx.trace_d;
    FusedResult* res = static_cast<FusedResult*>(fx.result_h);
    std::memset(res, 0, sizeof(FusedResult));
    cudaStream_t s = ctx->stream;
    BEMB_CUDA(ctx, cudaEventRecord(ws->ev0, s));
    cudaError_t le = launch_gmres_fused(p, (int)G, smem, polite, s);
    if (le != cudaSuccess) {
        // e.g. cooperative launch too large for what is free on this device: not an error of the solve
        cudaGetLastError();
        if (ctx->nranks > 1) return cuda_fail(ctx, le, "fused GMRES launch (row-sharded solve: no per-rank fallback)");
        fx.disabled = true;
        return BEMB200_OK;
    }
    BEMB_CUDA(ctx, cudaEventRecord(ws->ev1, s));
    BEMB_CUDA(ctx, cudaStreamSynchronize(s));
    *used = true;
    if (res->done && !res->error) {
        std::vector<unsigned long long> tr((size_t)G * 4);
        BEMB_CUDA(ctx, cudaMemcpy(tr.data(), fx.trace_d, tr.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        bool same_map = fx.smid.size() == G;
        for (uint32_t c = 0; c < G && same_map; ++c) same_map = fx.smid[c] == (unsigned)tr[4 * c + 3];
        const bool sizeable = p.nloc >= 16 * G && res->matvecs >= 10;
        if (sizeable && (fx.calib_runs < 2 || !same_map)) {
            if (!same_map) fx.calib_runs = 0;
            std::vector<double> sp(G, 0.0);
            bool good = true;
            for (uint32_t c = 0; c < G; ++c) {
                if (tr[4 * c + 2] == 0 || tr[4 * c] == 0) { good = false; break; }
                sp[c] = (double)tr[4 * c + 2] / (double)tr[4 * c];
            }
            if (good) {
                fx.speed = sp;
                fx.smid.resize(G);
                for (uint32_t c = 0; c < G; ++c) fx.smid[c] = (unsigned)tr[4 * c + 3];
                fx.calib_runs += 1;
            }
        }
    }
    if (res->error || !res->done) {
        fx.disabled = true;
        px.epoch += 1u << 20;  // whatever the aborted kernel left in the buffers is older than anything written from now on
        fx.er += 1u << 20;
        if (ctx->nranks > 1) px.ok = false;
        return set_error(ctx, BEMB200_ENCCL, "fused GMRES kernel: a bounded wait timed out (a rank or a CTA never delivered its data)");
    }
    px.epoch = res->ex_final;
    fx.er = res->er_final;
    *info = bemb200_gmres_info{res->iterations, res->restarts, res->residual, res->converged};
    m->last_launches += 1;
    m->last_matvecs += res->matvecs;
    m->last_matvec_ms += (double)res->t_matvec_ns * 1e-6;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ws->ev0, ws->ev1) == cudaSuccess) m->last_solve_ms = ms;
    else cudaGetLastError();
    g_fused_total_ms += (double)res->t_total_ns * 1e-6;
    g_fused_matvec_ms += (double)res->t_matvec_ns * 1e-6;
    g_fused_round_ms += (double)res->t_round_ns * 1e-6;
    g_fused_rounds += res->iterations + res->restarts + 1;
    return BEMB200_OK;
}

extern "C" void bemb200_debug_fused_times(double* total_ms, double* matvec_ms, double* round_ms, unsigned long long* rounds) {
    *total_ms = g_fused_total_ms; *matvec_ms = g_fused_matvec_ms; *round_ms = g_fused_round_ms; *rounds = g_fused_rounds;
    g_fused_total_ms = g_fused_matvec_ms = g_fused_round_ms = 0.0;
    g_fused_rounds = 0;
}

// gmres_with_guess (gmres.rs:105-277) with device vectors b, x (x holds x0 on entry), or with P.left its left-preconditioned
// variant.  A Schwarz or callback preconditioner acts on the rank's slab of A v between the ZGEMV and the exchange; the
// Gram-Schmidt kernel then sees an already preconditioned vector.  A diagonal one is applied by that kernel (pinv).
static int gmres_core(bemb200_matrix* m, const cplx* b, cplx* x, uint32_t max_iterations, uint32_t restart, double tol,
                      bemb200_gmres_info* info, const LeftPrecond& P) {
    bemb200_ctx* ctx = m->ctx;
    GmresWorkspace* ws = m->ws;
    const uint64_t n = m->n_rows;
    const int mm = (int)restart;
    cudaStream_t s = ctx->stream;
    if (!P.own_step()) {
        bool used = false;
        int frc = gmres_fused_solve(m, b, x, max_iterations, restart, tol, info, P.left, P.pinv, &used);
        if (frc != BEMB200_OK || used) return frc;
    }
    double b_norm = 0.0;
    int rc = residual_norm(m, P, b, nullptr, &b_norm);  // ||b|| resp. ||M^-1 b||
    if (rc != BEMB200_OK) return rc;
    const int direct_scale = P.left ? 1 : 0;
    if (b_norm < 1e-15) {
        *info = bemb200_gmres_info{0, 0, 0.0, 1};
        return BEMB200_OK;
    }
    uint64_t total_iterations = 0, restarts = 0;
    GmresCycle cycle;
    std::vector<cplx> y;
    const bool allow_grid = ctx->shared_gpu.load() == 0;
    if (allow_grid) {  // same value on every rank (collective call sequence)
        rc = ensure_peer_exchange(ctx, ws->npad);
        if (rc != BEMB200_OK) return rc;
    }
    // (with assembly kernels of another stream on the GPU the spinning consumer measured slower than NCCL: keep it for
    //  the solver-owns-the-GPU case)
    if (ctx->nranks > 1 && ctx->px.tried && ctx->nccl_comm) {
        // a rank whose consumer kernel once timed out has left peer mode; the ranks agree on the path of THIS solve
        // (one 4-byte all-gather per solve) so that nobody waits in a protocol the others no longer speak
        int* st = reinterpret_cast<int*>(ws->hcol_d);
        const int mine = ctx->px.ok ? 1 : 0;
        std::vector<int> all(ctx->nranks, 0);
        BEMB_CUDA(ctx, cudaMemcpyAsync(st + ctx->rank, &mine, sizeof(int), cudaMemcpyHostToDevice, s));
        rc = nccl_allgather_bytes(ctx, st + ctx->rank, st, sizeof(int));
        if (rc != BEMB200_OK) return rc;
        BEMB_CUDA(ctx, cudaMemcpyAsync(all.data(), st, sizeof(int) * ctx->nranks, cudaMemcpyDeviceToHost, s));
        BEMB_CUDA(ctx, cudaStreamSynchronize(s));
        bool every = true;
        for (int v : all) every = every && v != 0;
        if (!every) ctx->px.ok = false;
        if (ctx->px.err_h) *ctx->px.err_h = 0;
    }
    const bool peer_fused = !P.own_step() && allow_grid && ctx->nranks > 1 && ctx->px.ok && ctx->px.npad >= ws->npad && ws->npad == ws->chunk * (uint64_t)ctx->nranks &&
                            mgs_peer_wait_capable(n, restart);
    struct PeerErrCheck {  // a consumer kernel that gave up waiting for a peer poisons the solve: report it
        bemb200_ctx* c; bool on;
        int check() const { return (on && c->px.err_h && *c->px.err_h) ? 1 : 0; }
    } peer_err{ctx, peer_fused};
    for (uint32_t outer = 0; outer < max_iterations; ++outer) {
        rc = matvec(m, x, ws->w, true);
        if (rc != BEMB200_OK) return rc;
        double beta = 0.0;
        rc = residual_norm(m, P, b, ws->w, &beta);
        if (rc != BEMB200_OK) return rc;
        accumulate_matvec_time(m);
        double rel = beta / b_norm;
        if (rel < tol) {
            *info = bemb200_gmres_info{total_iterations, restarts, rel, 1};
            return BEMB200_OK;
        }
        BEMB_CUDA(ctx, launch_scale(ws->r, 1.0 / beta, ws->V, n, s));
        m->last_launches += 1;
        cycle.start(mm, beta);
        // One Arnoldi iteration = ZGEMV (+ all-gather) + ONE cluster MGS kernel + a (j+2)-number
        // D2H copy.  Iteration j+1 is enqueued BEFORE the host waits for column j, so the GPU never
        // idles on the host round trip; if column j turns out to converge, the speculative
        // iteration j+1 is simply ignored (it only touches V[j+2], w and its own column slot).
        for (int j = 0; j < mm; ++j) ws->launched[j] = 0;
        auto enqueue_iteration = [&](int j) -> int {
            BEMB_CUDA(ctx, cudaEventRecord(ws->it_ev0[j], s));
            const uint64_t nloc = m->r1 - m->r0;
            const cplx* wvec = ws->w;
            PeerWait pw;
            if (peer_fused) {
                // ZGEMV epilogue stores this rank's slab into every rank's work vector; no all-gather
                PeerExchange& px = ctx->px;
                unsigned long long epoch = ++px.epoch;
                if ((uint32_t)epoch == 0) epoch = ++px.epoch;  // 0 is the "never written" flag
                PeerOut po{};
                po.npeers = ctx->nranks;
                po.epoch = (uint32_t)epoch;
                for (int p = 0; p < ctx->nranks; ++p) po.ll[p] = px_work(px, p, epoch) + 2 * (uint64_t)ctx->rank * ws->chunk;
                BEMB_CUDA(ctx, launch_zgemv_peer(m->A, m->n_cols, nloc, m->n_cols, ws->V + (uint64_t)j * ws->npad, po, s));
                BEMB_CUDA(ctx, cudaEventRecord(ws->it_ev1[j], s));
                pw.ll = px_work(px, ctx->rank, epoch);
                pw.epoch = (uint32_t)epoch;
                pw.err = px.err_h;
                pw.timeout_ns = peer_timeout_ns();
            } else {
                cplx* yloc = ws->w + (ctx->nranks > 1 ? (uint64_t)ctx->rank * ws->chunk : m->r0);
                cplx* av = P.schwarz ? P.schwarz->tmp : yloc;  // Schwarz: A v_j into scratch, M^-1 writes the rank's rows of w
                BEMB_CUDA(ctx, launch_zgemv(m->A, m->n_cols, nloc, m->n_cols, ws->V + (uint64_t)j * ws->npad, av, s));
                BEMB_CUDA(ctx, cudaEventRecord(ws->it_ev1[j], s));
                int rc2 = BEMB200_OK;
                if (P.own_step()) rc2 = precond_apply(m, P, av, ws->w);  // w = M^-1 (A v_j) (gmres.rs:513-514)
                else if (ctx->nranks > 1) rc2 = nccl_allgather_bytes(ctx, yloc, ws->w, ws->chunk * sizeof(cplx));
                if (rc2 != BEMB200_OK) return rc2;
            }
            cplx* hd = ws->hcol_d + (size_t)j * ws->ldh_slot;
            bool wrote_host = false;
            BEMB_CUDA(ctx, launch_mgs(ws->V, ws->npad, const_cast<cplx*>(wvec), j, n, hd, ws->V + (uint64_t)(j + 1) * ws->npad, P.pinv,
                                      direct_scale, ws->lmat_d, (int)ws->restart + 1,
                                      ws->lmat_d + (size_t)(ws->restart + 1) * (ws->restart + 1),
                                      ws->hcol_h + (size_t)j * ws->ldh_slot, &wrote_host, pw, ctx->nranks > 1, s));
            if (!wrote_host)
                BEMB_CUDA(ctx, cudaMemcpyAsync(ws->hcol_h + (size_t)j * ws->ldh_slot, hd, (j + 2) * sizeof(cplx),
                                               cudaMemcpyDeviceToHost, s));
            BEMB_CUDA(ctx, cudaEventRecord(ws->it_done[j], s));
            ws->launched[j] = 1;
            m->last_launches += 2;  // every launch counts, also a speculative iteration that ends up unused
            return BEMB200_OK;
        };
        for (int j = 0; j < mm; ++j) {
            total_iterations += 1;
            if (!ws->launched[j]) {
                rc = enqueue_iteration(j);
                if (rc != BEMB200_OK) return rc;
            }
            // (never with a callback: the caller's apply runs exactly as often as in the reference)
            if (!P.user && j + 1 < mm && !ws->launched[j + 1]) {
                rc = enqueue_iteration(j + 1);
                if (rc != BEMB200_OK) return rc;
            }
            BEMB_CUDA(ctx, cudaEventSynchronize(ws->it_done[j]));
            {
                float ms = 0.f;
                if (cudaEventElapsedTime(&ms, ws->it_ev0[j], ws->it_ev1[j]) == cudaSuccess) m->last_matvec_ms += ms;
                else cudaGetLastError();
                m->last_matvecs += 1;  // matvecs whose duration is in last_matvec_ms
            }
            if (peer_err.check()) {
                // this solve is lost (the peers run into their own bounded waits); later solves of this context use the
                // NCCL all-gather, which the ranks agree on at the start of the next solve
                ctx->px.ok = false;
                *ctx->px.err_h = 0;
                return set_error(ctx, BEMB200_ENCCL, "peer-memory exchange timed out waiting for another rank's slab of A v");
            }
            bool breakdown = false;
            const double rel_res = cycle.add_column(j, ws->hcol_h + (size_t)j * ws->ldh_slot, b_norm, &breakdown);
            if (rel_res < tol || breakdown) {
                cycle.solve(j + 1, y);
                rc = update_x(m, x, y);
                if (rc != BEMB200_OK) return rc;
                *info = bemb200_gmres_info{total_iterations, restarts, rel_res, 1};
                return BEMB200_OK;
            }
        }
        cycle.solve(mm, y);
        rc = update_x(m, x, y);
        if (rc != BEMB200_OK) return rc;
        restarts += 1;
    }
    rc = matvec(m, x, ws->w, true);
    if (rc != BEMB200_OK) return rc;
    double rn = 0.0;
    rc = residual_norm(m, P, b, ws->w, &rn);
    if (rc != BEMB200_OK) return rc;
    accumulate_matvec_time(m);
    *info = bemb200_gmres_info{total_iterations, restarts, rn / b_norm, 0};
    return BEMB200_OK;
}

// ---- bicgstab (math-solvers/src/iterative/bicgstab.rs:53-215) with device vectors --------------
// Complex / Complex as num-complex 0.4 evaluates it: (a conj(b)) / |b|^2
static inline cplx cdiv(cplx a, cplx b) {
    const double ns = norm_sqr(b);
    return C((a.re * b.re + a.im * b.im) / ns, (a.im * b.re - a.re * b.im) / ns);
}

// the first cnt device scalars of BiCGSTAB / CGS (ws->hcol_d) into their pinned mirror (ws->hcol_h)
static int fetch_scalars(bemb200_matrix* m, int cnt) {
    bemb200_ctx* ctx = m->ctx;
    BEMB_CUDA(ctx, cudaMemcpyAsync(m->ws->hcol_h, m->ws->hcol_d, cnt * sizeof(cplx), cudaMemcpyDeviceToHost, ctx->stream));
    BEMB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return BEMB200_OK;
}

// b, x: device vectors of n (x = 0 on entry, as the reference starts).  Workspace rows
// V[0..6] hold r, r0, p, v, s, t; two A-products per iteration through the same (row-sharded)
// matvec as GMRES; every vector update is fused with the inner products that follow it and the
// scalars (4 small D2H reads per iteration) drive the reference's control flow on the host.
static int bicgstab_core(bemb200_matrix* m, const cplx* b, cplx* x, uint32_t max_iterations, double tol, bemb200_gmres_info* info) {
    bemb200_ctx* ctx = m->ctx;
    GmresWorkspace* ws = m->ws;
    const uint64_t n = m->n_rows;
    cudaStream_t s = ctx->stream;
    cplx* r = ws->V;
    cplx* r0 = ws->V + 1 * ws->npad;
    cplx* p = ws->V + 2 * ws->npad;
    cplx* v = ws->V + 3 * ws->npad;
    cplx* sv = ws->V + 4 * ws->npad;
    cplx* t = ws->V + 5 * ws->npad;
    cplx* dsc = ws->hcol_d;                 // device scalars
    cplx* hsc = ws->hcol_h;                 // pinned mirror
    // r = r0 = b, p = v = 0; (b, b) gives ||b|| and the first rho_new = (r0, r)
    BEMB_CUDA(ctx, cudaMemcpyAsync(r, b, n * sizeof(cplx), cudaMemcpyDeviceToDevice, s));
    BEMB_CUDA(ctx, cudaMemcpyAsync(r0, b, n * sizeof(cplx), cudaMemcpyDeviceToDevice, s));
    BEMB_CUDA(ctx, cudaMemsetAsync(p, 0, ws->npad * sizeof(cplx), s));
    BEMB_CUDA(ctx, cudaMemsetAsync(v, 0, ws->npad * sizeof(cplx), s));
    BEMB_CUDA(ctx, launch_bicg_dot(b, b, n, dsc, s));
    m->last_launches += 1;
    int rc = fetch_scalars(m, 1);
    if (rc != BEMB200_OK) return rc;
    const double b_norm = std::sqrt(hsc[0].re);
    if (b_norm < 1e-15) {
        *info = bemb200_gmres_info{0, 0, 0.0, 1};
        return BEMB200_OK;
    }
    cplx rho = C(1, 0), alpha = C(1, 0), omega = C(1, 0);
    cplx rho_new = hsc[0];
    double r_norm = b_norm;
    for (uint32_t iter = 0; iter < max_iterations; ++iter) {
        if (tnorm(rho_new) < 1e-30) {
            *info = bemb200_gmres_info{iter, 0, r_norm / b_norm, 0};
            return BEMB200_OK;
        }
        const cplx beta = cdiv(rho_new, rho) * cdiv(alpha, omega);
        rho = rho_new;
        BEMB_CUDA(ctx, launch_bicg_p(r, p, v, beta, omega, n, s));
        rc = matvec(m, p, v, true);
        if (rc != BEMB200_OK) return rc;
        BEMB_CUDA(ctx, launch_bicg_dot(r0, v, n, dsc, s));
        m->last_launches += 2;
        rc = fetch_scalars(m, 1);
        if (rc != BEMB200_OK) return rc;
        accumulate_matvec_time(m);
        const cplx r0v = hsc[0];
        if (tnorm(r0v) < 1e-30) {
            *info = bemb200_gmres_info{iter, 0, r_norm / b_norm, 0};
            return BEMB200_OK;
        }
        alpha = cdiv(rho, r0v);
        BEMB_CUDA(ctx, launch_bicg_s(r, v, alpha, sv, n, dsc, s));
        m->last_launches += 1;
        rc = fetch_scalars(m, 1);
        if (rc != BEMB200_OK) return rc;
        const double s_norm = std::sqrt(hsc[0].re);
        if (s_norm / b_norm < tol) {
            BEMB_CUDA(ctx, launch_bicg_axpy(x, p, alpha, n, s));
            m->last_launches += 1;
            BEMB_CUDA(ctx, cudaStreamSynchronize(s));
            *info = bemb200_gmres_info{(uint64_t)iter + 1, 0, s_norm / b_norm, 1};
            return BEMB200_OK;
        }
        rc = matvec(m, sv, t, true);
        if (rc != BEMB200_OK) return rc;
        BEMB_CUDA(ctx, launch_bicg_tt(t, sv, n, dsc, s));
        m->last_launches += 1;
        rc = fetch_scalars(m, 2);
        if (rc != BEMB200_OK) return rc;
        accumulate_matvec_time(m);
        const cplx tt = hsc[0];
        if (tnorm(tt) < 1e-30) {
            *info = bemb200_gmres_info{iter, 0, r_norm / b_norm, 0};
            return BEMB200_OK;
        }
        omega = cdiv(hsc[1], tt);
        BEMB_CUDA(ctx, launch_bicg_update(x, p, sv, t, r, r0, alpha, omega, n, dsc, s));
        m->last_launches += 1;
        rc = fetch_scalars(m, 2);
        if (rc != BEMB200_OK) return rc;
        r_norm = std::sqrt(hsc[0].re);
        rho_new = hsc[1];
        const double rel = r_norm / b_norm;
        if (rel < tol) {
            *info = bemb200_gmres_info{(uint64_t)iter + 1, 0, rel, 1};
            return BEMB200_OK;
        }
        if (tnorm(omega) < 1e-30) {
            *info = bemb200_gmres_info{(uint64_t)iter + 1, 0, rel, 0};
            return BEMB200_OK;
        }
    }
    *info = bemb200_gmres_info{max_iterations, 0, r_norm / b_norm, 0};
    return BEMB200_OK;
}

// ---- cgs (math-solvers/src/iterative/cgs.rs:46-155) with device vectors ------------------------
// x = 0 on entry.  Workspace rows V[0..7] hold r, r0, p, u, q, v, u+q, w; two A-products per iteration; three fused
// vector kernels; 2 scalar read-backs per iteration drive the reference's control flow on the host
// (including its test of the OLD rho after rho_new has been formed, cgs.rs:122).
static int cgs_core(bemb200_matrix* m, const cplx* b, cplx* x, uint32_t max_iterations, double tol, bemb200_gmres_info* info) {
    bemb200_ctx* ctx = m->ctx;
    GmresWorkspace* ws = m->ws;
    const uint64_t n = m->n_rows;
    cudaStream_t s = ctx->stream;
    cplx* r = ws->V;
    cplx* r0 = ws->V + 1 * ws->npad;
    cplx* p = ws->V + 2 * ws->npad;
    cplx* u = ws->V + 3 * ws->npad;
    cplx* q = ws->V + 4 * ws->npad;
    cplx* v = ws->V + 5 * ws->npad;
    cplx* uq = ws->V + 6 * ws->npad;
    cplx* w = ws->V + 7 * ws->npad;
    cplx* dsc = ws->hcol_d;
    cplx* hsc = ws->hcol_h;
    // r = r0 = p = u = b; (b, b) gives ||b|| and the first rho = (r0, r)
    for (cplx* dst : {r, r0, p, u}) {
        BEMB_CUDA(ctx, cudaMemsetAsync(dst, 0, ws->npad * sizeof(cplx), s));
        BEMB_CUDA(ctx, cudaMemcpyAsync(dst, b, n * sizeof(cplx), cudaMemcpyDeviceToDevice, s));
    }
    BEMB_CUDA(ctx, cudaMemsetAsync(uq, 0, ws->npad * sizeof(cplx), s));
    BEMB_CUDA(ctx, launch_bicg_dot(b, b, n, dsc, s));
    m->last_launches += 1;
    int rc = fetch_scalars(m, 1);
    if (rc != BEMB200_OK) return rc;
    const double b_norm = std::sqrt(hsc[0].re);
    if (b_norm < 1e-15) {
        *info = bemb200_gmres_info{0, 0, 0.0, 1};
        return BEMB200_OK;
    }
    cplx rho = hsc[0];
    double r_norm = b_norm;
    for (uint32_t iter = 0; iter < max_iterations; ++iter) {
        rc = matvec(m, p, v, true);
        if (rc != BEMB200_OK) return rc;
        BEMB_CUDA(ctx, launch_bicg_dot(r0, v, n, dsc, s));
        m->last_launches += 1;
        rc = fetch_scalars(m, 1);
        if (rc != BEMB200_OK) return rc;
        accumulate_matvec_time(m);
        const cplx sigma = hsc[0];
        if (tnorm(sigma) < 1e-30) {
            *info = bemb200_gmres_info{iter, 0, r_norm / b_norm, 0};
            return BEMB200_OK;
        }
        const cplx alpha = cdiv(rho, sigma);
        BEMB_CUDA(ctx, launch_cgs_q(u, v, alpha, q, uq, n, s));
        rc = matvec(m, uq, w, true);
        if (rc != BEMB200_OK) return rc;
        BEMB_CUDA(ctx, launch_cgs_update(x, uq, w, r, r0, alpha, n, dsc, s));
        m->last_launches += 2;
        rc = fetch_scalars(m, 2);
        if (rc != BEMB200_OK) return rc;
        accumulate_matvec_time(m);
        r_norm = std::sqrt(hsc[0].re);
        const cplx rho_new = hsc[1];
        const double rel = r_norm / b_norm;
        if (rel < tol) {
            *info = bemb200_gmres_info{(uint64_t)iter + 1, 0, rel, 1};
            return BEMB200_OK;
        }
        if (tnorm(rho) < 1e-30) {
            *info = bemb200_gmres_info{(uint64_t)iter + 1, 0, rel, 0};
            return BEMB200_OK;
        }
        const cplx beta = cdiv(rho_new, rho);
        rho = rho_new;
        BEMB_CUDA(ctx, launch_cgs_p(r, q, beta, u, p, n, s));
        m->last_launches += 1;
    }
    *info = bemb200_gmres_info{max_iterations, 0, r_norm / b_norm, 0};
    return BEMB200_OK;
}

// the solver needs the whole operator: every row owned by exactly one rank, canonical split
static int check_partition(bemb200_matrix* m) {
    bemb200_ctx* ctx = m->ctx;
    uint64_t b = 0, e = 0;
    bemb200_partition(m->n_rows, ctx->nranks, ctx->rank, &b, &e);
    if (m->r0 != b || m->r1 != e)
        return set_error(ctx, BEMB200_EINVAL,
                         "matrix slab is not this rank's canonical row block (see bemb200_partition); apply/gmres need the whole operator");
    return BEMB200_OK;
}

static void reset_stats(bemb200_matrix* m) {
    m->last_launches = 0;
    m->last_matvecs = 0;
    m->last_matvec_ms = 0.0;
    m->last_solve_ms = 0.0;
}

// workspace rows V[0..7] of BiCGSTAB and CGS (what GMRES sizes by its restart length)
constexpr uint32_t BICG_ROWS = 8;

// Argument checks of the solver entry points: `args` = every pointer argument the call needs is non-NULL; `restart` = the
// GMRES restart length (BICG_ROWS for BiCGSTAB / CGS).
static int check_solver_args(const bemb200_matrix* m, bool args, const char* solver, uint32_t restart) {
    if (!m || !args) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    if (m->n_rows != m->n_cols) return set_error(m->ctx, BEMB200_EINVAL, std::string(solver) + " needs a square operator");
    if (restart == 0) return set_error(m->ctx, BEMB200_EINVAL, "restart must be >= 1");
    return BEMB200_OK;
}

// The start of a solver or operator call after its argument checks, with ctx->mu held: device, partition check, a
// workspace for `restart` Krylov vectors, fresh statistics.
static int begin_call(bemb200_matrix* m, uint32_t restart) {
    bemb200_ctx* ctx = m->ctx;
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = check_partition(m);
    if (rc != BEMB200_OK) return rc;
    rc = ensure_workspace(m, restart);
    if (rc != BEMB200_OK) return rc;
    reset_stats(m);
    return BEMB200_OK;
}

// A solve on host vectors: b and x0 (NULL: x = 0) into the workspace, core(b, x) on the device, x back to x_out.
// `b_kind` = cudaMemcpyDeviceToDevice: b is a device vector (the sweep's right-hand sides formed on the device).
template <class Core>
static int solve_host_vectors(bemb200_matrix* m, const double* b, const double* x0, double* x_out, Core core,
                              cudaMemcpyKind b_kind = cudaMemcpyHostToDevice) {
    bemb200_ctx* ctx = m->ctx;
    GmresWorkspace* ws = m->ws;
    const size_t nb = m->n_rows * sizeof(cplx);
    BEMB_CUDA(ctx, cudaMemcpyAsync(ws->bin, b, nb, b_kind, ctx->stream));
    if (x0) BEMB_CUDA(ctx, cudaMemcpyAsync(ws->xout, x0, nb, cudaMemcpyHostToDevice, ctx->stream));
    else BEMB_CUDA(ctx, cudaMemsetAsync(ws->xout, 0, nb, ctx->stream));
    const int rc = core(ws->bin, ws->xout);
    if (rc != BEMB200_OK) return rc;
    BEMB_CUDA(ctx, cudaMemcpyAsync(x_out, ws->xout, nb, cudaMemcpyDeviceToHost, ctx->stream));
    BEMB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return BEMB200_OK;
}

extern "C" {

int bemb200_gmres_device(const bemb200_matrix* cm, const double* b_dev, const double* x0_dev, uint32_t max_iterations,
                         uint32_t restart, double tolerance, double* x_dev, bemb200_gmres_info* info) {
    bemb200_matrix* m = const_cast<bemb200_matrix*>(cm);
    int rc = check_solver_args(m, b_dev && x_dev && info, "gmres", restart);
    if (rc != BEMB200_OK) return rc;
    bemb200_ctx* ctx = m->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    rc = begin_call(m, restart);
    if (rc != BEMB200_OK) return rc;
    const size_t nb = m->n_rows * sizeof(cplx);
    if (x0_dev) {
        if ((const void*)x0_dev != (const void*)x_dev)
            BEMB_CUDA(ctx, cudaMemcpyAsync(x_dev, x0_dev, nb, cudaMemcpyDeviceToDevice, ctx->stream));
    } else {
        BEMB_CUDA(ctx, cudaMemsetAsync(x_dev, 0, nb, ctx->stream));
    }
    rc = gmres_core(m, (const cplx*)b_dev, (cplx*)x_dev, max_iterations, restart, tolerance, info, LeftPrecond{});
    cudaStreamSynchronize(ctx->stream);
    return rc;
}

int bemb200_gmres(const bemb200_matrix* cm, const double* b, const double* x0, uint32_t max_iterations, uint32_t restart,
                  double tolerance, double* x_out, bemb200_gmres_info* info) {
    bemb200_matrix* m = const_cast<bemb200_matrix*>(cm);
    int rc = check_solver_args(m, b && x_out && info, "gmres", restart);
    if (rc != BEMB200_OK) return rc;
    std::lock_guard<std::mutex> lk(m->ctx->mu);
    rc = begin_call(m, restart);
    if (rc != BEMB200_OK) return rc;
    return solve_host_vectors(m, b, x0, x_out, [&](const cplx* bd, cplx* xd) {
        return gmres_core(m, bd, xd, max_iterations, restart, tolerance, info, LeftPrecond{});
    });
}

int bemb200_bicgstab(const bemb200_matrix* cm, const double* b, uint32_t max_iterations, double tolerance, double* x_out,
                     bemb200_gmres_info* info) {
    bemb200_matrix* m = const_cast<bemb200_matrix*>(cm);
    int rc = check_solver_args(m, b && x_out && info, "bicgstab", BICG_ROWS);
    if (rc != BEMB200_OK) return rc;
    std::lock_guard<std::mutex> lk(m->ctx->mu);
    rc = begin_call(m, BICG_ROWS);
    if (rc != BEMB200_OK) return rc;
    return solve_host_vectors(m, b, nullptr, x_out, [&](const cplx* bd, cplx* xd) {
        return bicgstab_core(m, bd, xd, max_iterations, tolerance, info);
    });
}

int bemb200_cgs(const bemb200_matrix* cm, const double* b, uint32_t max_iterations, double tolerance, double* x_out,
                bemb200_gmres_info* info) {
    bemb200_matrix* m = const_cast<bemb200_matrix*>(cm);
    int rc = check_solver_args(m, b && x_out && info, "cgs", BICG_ROWS);
    if (rc != BEMB200_OK) return rc;
    std::lock_guard<std::mutex> lk(m->ctx->mu);
    rc = begin_call(m, BICG_ROWS);
    if (rc != BEMB200_OK) return rc;
    return solve_host_vectors(m, b, nullptr, x_out, [&](const cplx* bd, cplx* xd) {
        return cgs_core(m, bd, xd, max_iterations, tolerance, info);
    });
}

int bemb200_gmres_preconditioned(const bemb200_matrix* cm, const double* inv_diag, const double* b, const double* x0,
                                 uint32_t max_iterations, uint32_t restart, double tolerance, double* x_out,
                                 bemb200_gmres_info* info) {
    bemb200_matrix* m = const_cast<bemb200_matrix*>(cm);
    int rc = check_solver_args(m, b && x_out && info, "gmres", restart);
    if (rc != BEMB200_OK) return rc;
    bemb200_ctx* ctx = m->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    rc = begin_call(m, restart);
    if (rc != BEMB200_OK) return rc;
    return solve_host_vectors(m, b, x0, x_out, [&](const cplx* bd, cplx* xd) {
        LeftPrecond P{true};  // inv_diag == NULL: IdentityPreconditioner
        if (inv_diag) {
            BEMB_CUDA(ctx, cudaMemcpyAsync(m->ws->xin, inv_diag, m->n_rows * sizeof(cplx), cudaMemcpyHostToDevice, ctx->stream));
            P.pinv = m->ws->xin;
        }
        return gmres_core(m, bd, xd, max_iterations, restart, tolerance, info, P);
    });
}

int bemb200_gmres_schwarz(const bemb200_matrix* cm, const bemb200_precond* precond, const double* b, const double* x0,
                          uint32_t max_iterations, uint32_t restart, double tolerance, double* x_out, bemb200_gmres_info* info) {
    bemb200_matrix* m = const_cast<bemb200_matrix*>(cm);
    int rc = check_solver_args(m, precond && b && x_out && info, "gmres", restart);
    if (rc != BEMB200_OK) return rc;
    bemb200_ctx* ctx = m->ctx;
    if (precond->ctx != ctx || precond->n != m->n_rows || precond->r0 != m->r0 || precond->r1 != m->r1)
        return set_error(ctx, BEMB200_EINVAL, "preconditioner was built for another operator shape / context");
    std::lock_guard<std::mutex> lk(ctx->mu);
    rc = begin_call(m, restart);
    if (rc != BEMB200_OK) return rc;
    return solve_host_vectors(m, b, x0, x_out, [&](const cplx* bd, cplx* xd) {
        return gmres_core(m, bd, xd, max_iterations, restart, tolerance, info, LeftPrecond{true, nullptr, precond});
    });
}

int bemb200_gmres_callback(const bemb200_matrix* cm, bemb200_precond_fn apply, void* user, const double* b, const double* x0,
                           uint32_t max_iterations, uint32_t restart, double tolerance, double* x_out, bemb200_gmres_info* info,
                           uint64_t* precond_calls) {
    bemb200_matrix* m = const_cast<bemb200_matrix*>(cm);
    int rc = check_solver_args(m, apply && b && x_out && info, "gmres", restart);
    if (rc != BEMB200_OK) return rc;
    bemb200_ctx* ctx = m->ctx;
    if (ctx->nranks != 1 || m->r0 != 0 || m->r1 != m->n_rows)
        return set_error(ctx, BEMB200_EUNSUPPORTED, "bemb200_gmres_callback: a host preconditioner acts on whole vectors -- single-rank operators only");
    std::lock_guard<std::mutex> lk(ctx->mu);
    rc = begin_call(m, restart);
    if (rc != BEMB200_OK) return rc;
    const size_t nb = m->n_rows * sizeof(cplx);
    struct Pinned {  // the two host vectors of the round trip
        cplx* p = nullptr;
        ~Pinned() { if (p) cudaFreeHost(p); }
    } rbuf, zbuf;
    if (cudaMallocHost((void**)&rbuf.p, nb ? nb : sizeof(cplx)) != cudaSuccess || cudaMallocHost((void**)&zbuf.p, nb ? nb : sizeof(cplx)) != cudaSuccess) {
        cudaGetLastError();
        return set_error(ctx, BEMB200_ENOMEM, "pinned host vectors for the preconditioner callback");
    }
    UserPrecond up;
    up.fn = apply;
    up.user = user;
    up.r_h = rbuf.p;
    up.z_h = zbuf.p;
    rc = solve_host_vectors(m, b, x0, x_out, [&](const cplx* bd, cplx* xd) {
        return gmres_core(m, bd, xd, max_iterations, restart, tolerance, info, LeftPrecond{true, nullptr, nullptr, &up});
    });
    if (precond_calls) *precond_calls = up.calls;
    if (rc != BEMB200_OK) cudaStreamSynchronize(ctx->stream);  // nothing of this solve may still be reading the pinned vectors when they go
    return rc;
}

int bemb200_matrix_diagonal(const bemb200_matrix* cm, double* out) {
    bemb200_matrix* m = const_cast<bemb200_matrix*>(cm);
    if (!m || !out) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    bemb200_ctx* ctx = m->ctx;
    if (m->n_rows != m->n_cols) return set_error(ctx, BEMB200_EINVAL, "diagonal needs a square matrix");
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = check_partition(m);
    if (rc != BEMB200_OK) return rc;
    rc = ensure_workspace(m, 1);
    if (rc != BEMB200_OK) return rc;
    GmresWorkspace* ws = m->ws;
    const uint64_t nloc = m->r1 - m->r0;
    cplx* loc = ws->r + (ctx->nranks > 1 ? (uint64_t)ctx->rank * ws->chunk : m->r0);
    // strided gather of A[i, r0 + i]
    if (nloc)
        BEMB_CUDA(ctx, cudaMemcpy2DAsync(loc, sizeof(cplx), m->A + m->r0, (m->n_cols + 1) * sizeof(cplx), sizeof(cplx), nloc,
                                         cudaMemcpyDeviceToDevice, ctx->stream));
    rc = nccl_allgather_bytes(ctx, loc, ws->r, ws->chunk * sizeof(cplx));
    if (rc != BEMB200_OK) return rc;
    BEMB_CUDA(ctx, cudaMemcpyAsync(out, ws->r, m->n_rows * sizeof(cplx), cudaMemcpyDeviceToHost, ctx->stream));
    BEMB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return BEMB200_OK;
}

int bemb200_apply_device(const bemb200_matrix* cm, const double* x_dev, double* y_dev) {
    bemb200_matrix* m = const_cast<bemb200_matrix*>(cm);
    if (!m || !x_dev || !y_dev) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    bemb200_ctx* ctx = m->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    int rc = begin_call(m, 1);
    if (rc != BEMB200_OK) return rc;
    GmresWorkspace* ws = m->ws;
    if (ctx->nranks == 1) {
        // write straight into the caller's vector
        BEMB_CUDA(ctx, cudaEventRecord(ws->ev0, ctx->stream));
        BEMB_CUDA(ctx, launch_zgemv(m->A, m->n_cols, m->r1 - m->r0, m->n_cols, (const cplx*)x_dev, (cplx*)y_dev + m->r0, ctx->stream));
        BEMB_CUDA(ctx, cudaEventRecord(ws->ev1, ctx->stream));
        m->last_launches = 1;
        m->last_matvecs = 1;
    } else {
        rc = matvec(m, (const cplx*)x_dev, ws->w, true);
        if (rc != BEMB200_OK) return rc;
        BEMB_CUDA(ctx, cudaMemcpyAsync(y_dev, ws->w, m->n_rows * sizeof(cplx), cudaMemcpyDeviceToDevice, ctx->stream));
    }
    BEMB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    accumulate_matvec_time(m);
    return BEMB200_OK;
}

int bemb200_apply(const bemb200_matrix* cm, const double* x, double* y) {
    bemb200_matrix* m = const_cast<bemb200_matrix*>(cm);
    if (!m || !x || !y) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    bemb200_ctx* ctx = m->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    int rc = begin_call(m, 1);
    if (rc != BEMB200_OK) return rc;
    GmresWorkspace* ws = m->ws;
    BEMB_CUDA(ctx, cudaMemcpyAsync(ws->xin, x, m->n_cols * sizeof(cplx), cudaMemcpyHostToDevice, ctx->stream));
    rc = matvec(m, ws->xin, ws->w, true);
    if (rc != BEMB200_OK) return rc;
    BEMB_CUDA(ctx, cudaMemcpyAsync(y, ws->w, m->n_rows * sizeof(cplx), cudaMemcpyDeviceToHost, ctx->stream));
    BEMB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    accumulate_matvec_time(m);
    return BEMB200_OK;
}

int bemb200_apply_transpose(const bemb200_matrix* cm, const double* x, double* y) {
    bemb200_matrix* m = const_cast<bemb200_matrix*>(cm);
    if (!m || !x || !y) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    bemb200_ctx* ctx = m->ctx;
    if (ctx->nranks > 1) return set_error(ctx, BEMB200_EUNSUPPORTED, "apply_transpose on a row-sharded matrix is not implemented");
    std::lock_guard<std::mutex> lk(ctx->mu);
    int rc = begin_call(m, 1);
    if (rc != BEMB200_OK) return rc;
    GmresWorkspace* ws = m->ws;
    // y = A^T x : x has num_rows entries, y has num_cols entries
    BEMB_CUDA(ctx, cudaMemcpyAsync(ws->xin, x, m->n_rows * sizeof(cplx), cudaMemcpyHostToDevice, ctx->stream));
    BEMB_CUDA(ctx, launch_zgemv_t(m->A, m->n_cols, m->r1 - m->r0, m->n_cols, ws->xin + m->r0, ws->w, ctx->stream));
    m->last_launches = 1;
    BEMB_CUDA(ctx, cudaMemcpyAsync(y, ws->w, m->n_cols * sizeof(cplx), cudaMemcpyDeviceToHost, ctx->stream));
    BEMB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return BEMB200_OK;
}

int bemb200_row_sum_correction(bemb200_matrix* m, double* avg) {
    if (!m) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    bemb200_ctx* ctx = m->ctx;
    if (m->n_rows != m->n_cols) return set_error(ctx, BEMB200_EINVAL, "row-sum correction needs a square matrix");
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint64_t nloc = m->r1 - m->r0;
    cplx* d_sums = nullptr;
    BEMB_CUDA(ctx, cudaMalloc((void**)&d_sums, (nloc + 1) * sizeof(cplx)));
    cudaError_t e = launch_row_sum(m->A, m->n_cols, nloc, m->n_cols, m->r0, d_sums, ctx->stream);
    std::vector<cplx> sums(nloc);
    if (e == cudaSuccess && nloc) e = cudaMemcpyAsync(sums.data(), d_sums, nloc * sizeof(cplx), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d_sums);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "row_sum_correction");
    cplx total = C(0, 0);
    for (uint64_t i = 0; i < nloc; ++i) total += sums[i];
    if (ctx->nranks > 1) {
        // gather the per-rank partial totals (16 bytes each) and add them in rank order
        cplx* d_part = nullptr;
        BEMB_CUDA(ctx, cudaMalloc((void**)&d_part, ctx->nranks * sizeof(cplx)));
        BEMB_CUDA(ctx, cudaMemcpyAsync(d_part + ctx->rank, &total, sizeof(cplx), cudaMemcpyHostToDevice, ctx->stream));
        int rc = nccl_allgather_bytes(ctx, d_part + ctx->rank, d_part, sizeof(cplx));
        std::vector<cplx> parts(ctx->nranks);
        if (rc == BEMB200_OK) {
            e = cudaMemcpyAsync(parts.data(), d_part, ctx->nranks * sizeof(cplx), cudaMemcpyDeviceToHost, ctx->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        }
        cudaFree(d_part);
        if (rc != BEMB200_OK) return rc;
        if (e != cudaSuccess) return cuda_fail(ctx, e, "row_sum_correction gather");
        total = C(0, 0);
        for (int p = 0; p < ctx->nranks; ++p) total += parts[p];
    }
    if (avg) *avg = std::hypot(total.re, total.im) / (double)m->n_rows;
    return BEMB200_OK;
}

int bemb200_rhs_download_full(const bemb200_matrix* cm, double* out) {
    bemb200_matrix* m = const_cast<bemb200_matrix*>(cm);
    if (!m || !out) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    return rhs_full(m, out, cudaMemcpyDeviceToHost);
}

}  // extern "C"

int bemb::rhs_full(bemb200_matrix* m, double* out, cudaMemcpyKind kind) {
    bemb200_ctx* ctx = m->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = check_partition(m);
    if (rc != BEMB200_OK) return rc;
    rc = ensure_workspace(m, 1);
    if (rc != BEMB200_OK) return rc;
    GmresWorkspace* ws = m->ws;
    cplx* loc = ws->r + (ctx->nranks > 1 ? (uint64_t)ctx->rank * ws->chunk : m->r0);
    BEMB_CUDA(ctx, cudaMemcpyAsync(loc, m->rhs, (m->r1 - m->r0) * sizeof(cplx), cudaMemcpyDeviceToDevice, ctx->stream));
    rc = nccl_allgather_bytes(ctx, loc, ws->r, ws->chunk * sizeof(cplx));
    if (rc != BEMB200_OK) return rc;
    BEMB_CUDA(ctx, cudaMemcpyAsync(out, ws->r, m->n_rows * sizeof(cplx), kind, ctx->stream));
    BEMB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return BEMB200_OK;
}

int bemb::gmres_solve_device_b(bemb200_matrix* m, const bemb200_precond* pc, const double* b_dev, uint32_t max_iterations,
                               uint32_t restart, double tolerance, double* x_out, bemb200_gmres_info* info) {
    int rc = check_solver_args(m, b_dev && x_out && info, "gmres", restart);
    if (rc != BEMB200_OK) return rc;
    bemb200_ctx* ctx = m->ctx;
    if (pc && (pc->ctx != ctx || pc->n != m->n_rows || pc->r0 != m->r0 || pc->r1 != m->r1))
        return set_error(ctx, BEMB200_EINVAL, "preconditioner was built for another operator shape / context");
    std::lock_guard<std::mutex> lk(ctx->mu);
    rc = begin_call(m, restart);
    if (rc != BEMB200_OK) return rc;
    return solve_host_vectors(
        m, b_dev, nullptr, x_out,
        [&](const cplx* bd, cplx* xd) {
            return gmres_core(m, bd, xd, max_iterations, restart, tolerance, info, pc ? LeftPrecond{true, nullptr, pc} : LeftPrecond{});
        },
        cudaMemcpyDeviceToDevice);
}

extern "C" {

int bemb200_solver_stats(const bemb200_matrix* m, uint64_t* kernel_launches, double* matvec_ms, uint64_t* matvecs) {
    if (!m) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    if (kernel_launches) *kernel_launches = m->last_launches;
    if (matvec_ms) *matvec_ms = m->last_matvec_ms;
    if (matvecs) *matvecs = m->last_matvecs;
    return BEMB200_OK;
}

int bemb200_measure_fp64_peak(bemb200_ctx* ctx, double* tflops) {
    if (!ctx || !tflops) return set_error(ctx, BEMB200_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    double* d = nullptr;
    BEMB_CUDA(ctx, cudaMalloc((void**)&d, sizeof(double)));
    cudaEvent_t a, b;
    BEMB_CUDA(ctx, cudaEventCreate(&a));
    BEMB_CUDA(ctx, cudaEventCreate(&b));
    const int iters = 4096;
    double best = 0.0;
    cudaError_t e = launch_dfma_peak(d, 256, ctx->stream);  // warm-up
    for (int rep = 0; rep < 5 && e == cudaSuccess; ++rep) {
        cudaEventRecord(a, ctx->stream);
        e = launch_dfma_peak(d, iters, ctx->stream);
        cudaEventRecord(b, ctx->stream);
        if (e == cudaSuccess) e = cudaEventSynchronize(b);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, a, b);
        const double flops = 2.0 * 64.0 * (double)iters * 256.0 * 148.0 * 8.0;  // 8 chains x 8 unrolled FMAs per iteration
        if (ms > 0.f && flops / (ms * 1e-3) > best) best = flops / (ms * 1e-3);
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    cudaFree(d);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "dfma peak kernel");
    *tflops = best * 1e-12;
    return BEMB200_OK;
}

int bemb200_measure_allgather(bemb200_ctx* ctx, uint64_t bytes_per_rank, int iters, int sync_each, double* usec_per_call) {
    if (!ctx || !usec_per_call || iters < 1) return set_error(ctx, BEMB200_EINVAL, "bad argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    unsigned char* buf = nullptr;
    BEMB_CUDA(ctx, cudaMalloc((void**)&buf, bytes_per_rank * ctx->nranks + 16));
    BEMB_CUDA(ctx, cudaMemsetAsync(buf, 0, bytes_per_rank * ctx->nranks, ctx->stream));
    int rc = BEMB200_OK;
    for (int i = 0; i < 5 && rc == BEMB200_OK; ++i) rc = nccl_allgather_bytes(ctx, buf + bytes_per_rank * ctx->rank, buf, bytes_per_rank);
    cudaStreamSynchronize(ctx->stream);
    auto t0 = std::chrono::steady_clock::now();
    for (int i = 0; i < iters && rc == BEMB200_OK; ++i) {
        rc = nccl_allgather_bytes(ctx, buf + bytes_per_rank * ctx->rank, buf, bytes_per_rank);
        if (sync_each) cudaStreamSynchronize(ctx->stream);
    }
    cudaStreamSynchronize(ctx->stream);
    auto t1 = std::chrono::steady_clock::now();
    cudaFree(buf);
    if (rc != BEMB200_OK) return rc;
    *usec_per_call = std::chrono::duration<double, std::micro>(t1 - t0).count() / iters;
    return BEMB200_OK;
}

int bemb200_selftest_math(bemb200_ctx* ctx, uint64_t n, double xmax, double* sincos_err, double* rsqrt_relerr) {
    if (!ctx) return set_error(ctx, BEMB200_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    double* d = nullptr;
    BEMB_CUDA(ctx, cudaMalloc((void**)&d, 2 * sizeof(double)));
    cudaError_t e = cudaMemsetAsync(d, 0, 2 * sizeof(double), ctx->stream);
    if (e == cudaSuccess) e = launch_math_selftest(n, xmax, d, ctx->stream);
    double h[2] = {0, 0};
    if (e == cudaSuccess) e = cudaMemcpyAsync(h, d, sizeof h, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "math selftest");
    if (sincos_err) *sincos_err = h[0];
    if (rsqrt_relerr) *rsqrt_relerr = h[1];
    return BEMB200_OK;
}

}  // extern "C"
