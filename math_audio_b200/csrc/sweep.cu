// sweep.cu -- two host-side orchestrations behind the C ABI (no kernels of their own):
//
//   bemb200_sweep_*   the pipelined frequency sweep (reference shape: math-bem/examples/audio_frequency_sweep.rs, the
//                     per-frequency body of BemSolver::solve, bem_solver.rs:273-322): the mesh is staged once and the FP64
//                     assembly of frequency f+1 runs on a second context / stream / matrix buffer -- as a polite background
//                     grid -- underneath the HBM-bound solve of frequency f.  Every frequency is still exactly
//                     build_tbem_system_with_beta + gmres; only the schedule changes.
//
//   bemb200_multi_*   ONE process driving P devices (SURVEY 8b "Threading": every reference caller is one process).  The
//                     group owns one rank context per device; collective entry points run the per-rank calls on P host
//                     threads; the ranks exchange Krylov vectors and reduction partials through peer-mapped memory
//                     (cudaDeviceEnablePeerAccess, plain pointers: no CUDA IPC, no NCCL) inside the fused GMRES kernel.
#include <condition_variable>
#include <cstring>
#include <deque>
#include <memory>
#include <string>
#include <thread>

#include "api_internal.h"

using namespace bemb;

// =============================================================================================================
// sweep
// =============================================================================================================
// bemb200_assembly_options with the admittance owned (empty: none)
struct AssemblyOptionsCopy {
    int32_t dg_dn_sign = 0, consistent_beta = 0;
    std::vector<double> admittance;
    bemb200_assembly_options view() const { return {dg_dn_sign, consistent_beta, admittance.empty() ? nullptr : admittance.data()}; }
};

struct SweepJob {
    bemb200_physics phys;
    double beta_re, beta_im;
    AssemblyOptionsCopy opts;  // bemb200_sweep_set_assembly_options current at submit
    std::vector<double> rhs_extra;  // 2 n doubles or empty
    // bemb200_sweep_submit_incident: nrhs > 0 incident right-hand sides, built by the worker into the slot's device buffer
    uint32_t nrhs = 0;
    std::vector<uint32_t> src_ptr;
    std::vector<int32_t> kinds;
    std::vector<double> vecs, amps;
    uint32_t max_iterations, restart;
    double tolerance;
    int slot = 0;
    int rc = BEMB200_OK;
    std::string err;
    bool assembled = false;
};

struct bemb200_sweep {
    bemb200_ctx* ctx_solve = nullptr;
    bemb200_ctx* ctx_asm = nullptr;  // == ctx_solve when overlap is off
    bemb200_staged_mesh* staged = nullptr;
    bemb200_matrix* buf[2] = {nullptr, nullptr};
    bool buf_handed[2] = {false, false};
    uint64_t n = 0, r0 = 0, r1 = 0;
    bool overlap = true;
    int background = 1;
    std::thread worker;
    std::mutex mu;
    std::condition_variable cv;
    std::deque<std::shared_ptr<SweepJob>> queue;     // submitted, not yet returned by next()
    size_t next_to_assemble = 0;                      // index into queue of the next job the worker takes
    bool slot_busy[2] = {false, false};               // a matrix buffer is owned by a job (assembling or waiting for / in its solve)
    bool solving = false;                             // a solve is in flight on ctx_solve
    bool stop = false;
    uint64_t submitted = 0, boosts = 0;
    std::string err;
    // optional block-Jacobi / additive Schwarz preconditioner of every solve (bemb200_sweep_set_block_jacobi)
    bool precond = false;
    uint32_t pc_subdomains = 0;
    std::vector<uint64_t> pc_ptr, pc_idx;
    double pc_setup_ms = 0.0;  // device time of the last preconditioner set-up
    AssemblyOptionsCopy opts;  // assembly options of every frequency submitted from now on (bemb200_sweep_set_assembly_options)
    // per matrix slot: the incident block of the job owning the slot (nrhs x n complex128, device of ctx_asm, grow-only)
    bemb::cplx* inc[2] = {nullptr, nullptr};
    size_t inc_cap[2] = {0, 0};
};

// The incident block of `job` into its slot's buffer, on the assembly context right after the job's assembly (the worker
// thread): next_batch() then only adds TbemSystem.rhs and never waits for the assembly context behind the next frequency.
static int build_incident_block(bemb200_sweep* sw, SweepJob* job) {
    const size_t need = (size_t)job->nrhs * sw->n;
    if (sw->inc_cap[job->slot] < need) {
        cudaFree(sw->inc[job->slot]);
        sw->inc[job->slot] = nullptr;
        sw->inc_cap[job->slot] = 0;
        cudaError_t e = cudaMalloc((void**)&sw->inc[job->slot], (need ? need : 1) * sizeof(bemb::cplx));
        if (e != cudaSuccess) return cuda_fail(sw->ctx_asm, e, "sweep incident block");
        sw->inc_cap[job->slot] = need;
    }
    return bemb200_incident_rhs_batch(sw->staged, &job->phys, job->beta_re, job->beta_im, job->nrhs, job->src_ptr.data(), job->kinds.data(),
                                      job->vecs.data(), job->amps.data(), nullptr, nullptr, (double*)sw->inc[job->slot]);
}

static void sweep_worker(bemb200_sweep* sw) {
    cudaSetDevice(sw->ctx_asm->device);
    for (;;) {
        std::shared_ptr<SweepJob> job;
        bool foreground;
        {
            std::unique_lock<std::mutex> lk(sw->mu);
            sw->cv.wait(lk, [&] {
                if (sw->stop) return true;
                if (sw->next_to_assemble >= sw->queue.size()) return false;
                return !sw->slot_busy[sw->queue[sw->next_to_assemble]->slot];
            });
            if (sw->stop) return;
            job = sw->queue[sw->next_to_assemble];
            sw->next_to_assemble += 1;
            sw->slot_busy[job->slot] = true;
            // only the job at the head of the queue has nothing to hide behind (its own solve cannot start before it is
            // assembled): full speed.  Every other job is assembled underneath the solve of its predecessor: polite grid.
            foreground = job == sw->queue.front();
        }
        bemb200_ctx_set_background(sw->ctx_asm, (sw->overlap && !foreground) ? sw->background : 0);
        const bemb200_assembly_options opts = job->opts.view();
        int rc = bemb200_assemble_staged_opts(sw->ctx_asm, sw->staged, &job->phys, job->beta_re, job->beta_im, &opts, sw->r0, sw->r1,
                                              &sw->buf[job->slot]);
        if (rc == BEMB200_OK && sw->overlap && !sw->buf_handed[job->slot]) {
            rc = bemb200_matrix_set_context(sw->buf[job->slot], sw->ctx_solve);  // the solver owns the handle from now on
            sw->buf_handed[job->slot] = rc == BEMB200_OK;
        }
        if (rc == BEMB200_OK && job->nrhs > 0) rc = build_incident_block(sw, job.get());
        {
            std::lock_guard<std::mutex> lk(sw->mu);
            job->rc = rc;
            if (rc != BEMB200_OK) job->err = bemb200_last_error(sw->ctx_asm);
            job->assembled = true;
        }
        sw->cv.notify_all();
    }
}

extern "C" {

int bemb200_sweep_create(int device, int rank, int nranks, const uint8_t* nccl_id, const bemb200_mesh* mesh, int overlap,
                         int background_blocks_per_sm, bemb200_sweep** out) {
    if (!out || !mesh) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    *out = nullptr;
    std::unique_ptr<bemb200_sweep> sw(new bemb200_sweep());
    sw->overlap = overlap != 0;
    sw->background = background_blocks_per_sm > 0 ? background_blocks_per_sm : 1;
    int rc = bemb200_ctx_create_ex(device, rank, nranks, nccl_id, nullptr, &sw->ctx_solve);
    if (rc != BEMB200_OK) return rc;
    if (sw->overlap) {
        rc = bemb200_ctx_create_ex(device, rank, nranks, nullptr, nullptr, &sw->ctx_asm);  // assembly needs no communicator
        if (rc != BEMB200_OK) { bemb200_ctx_destroy(sw->ctx_solve); return rc; }
    } else {
        sw->ctx_asm = sw->ctx_solve;
    }
    rc = bemb200_mesh_stage(sw->ctx_asm, mesh, &sw->staged);
    if (rc != BEMB200_OK) {
        const std::string msg = bemb200_last_error(sw->ctx_asm);
        if (sw->overlap) bemb200_ctx_destroy(sw->ctx_asm);
        bemb200_ctx_destroy(sw->ctx_solve);
        return set_error(nullptr, rc, msg);
    }
    sw->n = bemb200_staged_num_dofs(sw->staged);
    bemb200_partition(sw->n, nranks, rank, &sw->r0, &sw->r1);
    bemb200_sweep* raw = sw.release();
    raw->worker = std::thread(sweep_worker, raw);
    *out = raw;
    return BEMB200_OK;
}

uint64_t bemb200_sweep_num_dofs(const bemb200_sweep* sw) { return sw ? sw->n : 0; }

int bemb200_sweep_submit(bemb200_sweep* sw, const bemb200_physics* phys, double beta_re, double beta_im, const double* rhs_extra,
                         uint32_t max_iterations, uint32_t restart, double tolerance) {
    if (!sw || !phys) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    if (restart == 0) return set_error(sw->ctx_solve, BEMB200_EINVAL, "restart must be >= 1");
    auto job = std::make_shared<SweepJob>();
    job->phys = *phys;
    job->beta_re = beta_re;
    job->beta_im = beta_im;
    if (rhs_extra) job->rhs_extra.assign(rhs_extra, rhs_extra + 2 * sw->n);
    job->max_iterations = max_iterations;
    job->restart = restart;
    job->tolerance = tolerance;
    {
        std::lock_guard<std::mutex> lk(sw->mu);
        job->opts = sw->opts;
        job->slot = (int)(sw->submitted & 1u);
        sw->submitted += 1;
        sw->queue.push_back(job);
    }
    sw->cv.notify_all();
    return BEMB200_OK;
}

int bemb200_sweep_submit_incident(bemb200_sweep* sw, const bemb200_physics* phys, double beta_re, double beta_im, uint32_t nrhs,
                                  const uint32_t* src_ptr, const int32_t* kinds, const double* vecs, const double* amps,
                                  uint32_t max_iterations, uint32_t restart, double tolerance) {
    if (!sw || !phys || !src_ptr || !kinds || !vecs || !amps) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    if (restart == 0) return set_error(sw->ctx_solve, BEMB200_EINVAL, "restart must be >= 1");
    if (nrhs == 0 || nrhs > 32) return set_error(sw->ctx_solve, BEMB200_EINVAL, "need 1..32 right-hand sides per frequency");
    if (src_ptr[0] != 0) return set_error(sw->ctx_solve, BEMB200_EINVAL, "src_ptr[0] must be 0");
    for (uint32_t s = 0; s < nrhs; ++s)
        if (src_ptr[s + 1] < src_ptr[s]) return set_error(sw->ctx_solve, BEMB200_EINVAL, "src_ptr must be non-decreasing");
    const uint32_t ns = src_ptr[nrhs];
    if (ns > 65536) return set_error(sw->ctx_solve, BEMB200_EINVAL, "at most 65536 sources in all");
    for (uint32_t s = 0; s < ns; ++s)
        if (kinds[s] != 0 && kinds[s] != 1) return set_error(sw->ctx_solve, BEMB200_EINVAL, "source kind must be 0 (plane wave) or 1 (point source)");
    auto job = std::make_shared<SweepJob>();
    job->phys = *phys;
    job->beta_re = beta_re;
    job->beta_im = beta_im;
    job->nrhs = nrhs;
    job->src_ptr.assign(src_ptr, src_ptr + nrhs + 1);
    job->kinds.assign(kinds, kinds + ns);
    job->vecs.assign(vecs, vecs + 3 * (size_t)ns);
    job->amps.assign(amps, amps + 2 * (size_t)ns);
    job->max_iterations = max_iterations;
    job->restart = restart;
    job->tolerance = tolerance;
    {
        std::lock_guard<std::mutex> lk(sw->mu);
        job->opts = sw->opts;
        job->slot = (int)(sw->submitted & 1u);
        sw->submitted += 1;
        sw->queue.push_back(job);
    }
    sw->cv.notify_all();
    return BEMB200_OK;
}

}  // extern "C"

// The oldest queued job: wait for its assembly, solve it, hand its slot back.  A job of more than `capacity` right-hand
// sides stays queued (BEMB200_EINVAL).  x_out / infos hold `capacity` solutions; rhs_out (may be NULL) receives b of a
// single right-hand side.
static int sweep_take(bemb200_sweep* sw, uint32_t capacity, double* x_out, bemb200_gmres_info* infos, uint32_t* nrhs_out,
                      bemb200_assembly_stats* stats, double* rhs_out) {
    std::shared_ptr<SweepJob> job;
    {
        std::unique_lock<std::mutex> lk(sw->mu);
        if (sw->queue.empty()) return set_error(sw->ctx_solve, BEMB200_EINVAL, "bemb200_sweep_next: nothing submitted");
        job = sw->queue.front();
        const uint32_t nrhs = job->nrhs > 0 ? job->nrhs : 1;
        if (nrhs > capacity)
            return set_error(sw->ctx_solve, BEMB200_EINVAL,
                             "the oldest job has " + std::to_string(nrhs) + " right-hand sides, more than the " + std::to_string(capacity) +
                                 " the caller has room for (bemb200_sweep_next_batch takes it)");
        sw->cv.wait(lk, [&] { return job->assembled; });
        if (job->rc != BEMB200_OK) {
            sw->queue.pop_front();
            sw->next_to_assemble -= 1;
            sw->slot_busy[job->slot] = false;
            sw->cv.notify_all();
            return set_error(sw->ctx_solve, job->rc, job->err);
        }
        sw->solving = true;
        // kernels of the assembly context run beside this solve whenever another job is queued behind this one
        bemb200_ctx_set_shared_gpu(sw->ctx_solve, (sw->overlap && sw->queue.size() > 1) ? 1 : 0);
    }
    if (nrhs_out) *nrhs_out = job->nrhs > 0 ? job->nrhs : 1;
    bemb200_matrix* m = sw->buf[job->slot];
    int rc = BEMB200_OK;
    if (stats) rc = bemb200_assembly_stats_get(m, stats);
    bool use_pc;
    uint32_t nsub;
    std::vector<uint64_t> pptr, pidx;
    {
        std::lock_guard<std::mutex> lk(sw->mu);
        use_pc = sw->precond; nsub = sw->pc_subdomains; pptr = sw->pc_ptr; pidx = sw->pc_idx;
    }
    // solve(pc): the job's solve, pc = NULL or the block-Jacobi preconditioner of THIS frequency's matrix
    auto with_precond = [&](auto solve) -> int {
        if (!use_pc) return solve((const bemb200_precond*)nullptr);
        bemb200_precond* pc = nullptr;  // gmres_preconditioned with the block-Jacobi preconditioner of THIS frequency's matrix
        int r = bemb200_schwarz_create(m, nsub, pptr.empty() ? nullptr : pptr.data(), pptr.empty() ? nullptr : pidx.data(), &pc);
        if (r == BEMB200_OK) {
            bemb200_precond_stats st{};
            if (bemb200_precond_stats_get(pc, &st) == BEMB200_OK) sw->pc_setup_ms = st.factor_ms;
            r = solve(pc);
        }
        bemb200_precond_free(pc);
        return r;
    };
    if (rc == BEMB200_OK && job->nrhs == 0) {  // bemb200_sweep_submit: b = TbemSystem.rhs + rhs_extra on the host
        std::vector<double> b(2 * sw->n);
        rc = bemb200_rhs_download_full(m, b.data());  // TbemSystem.rhs (all rows)
        if (rc == BEMB200_OK) {
            if (!job->rhs_extra.empty())
                for (size_t i = 0; i < b.size(); ++i) b[i] += job->rhs_extra[i];
            if (rhs_out) std::memcpy(rhs_out, b.data(), b.size() * sizeof(double));
            rc = with_precond([&](const bemb200_precond* pc) {
                return pc ? bemb200_gmres_schwarz(m, pc, b.data(), nullptr, job->max_iterations, job->restart, job->tolerance, x_out, infos)
                          : bemb200_gmres(m, b.data(), nullptr, job->max_iterations, job->restart, job->tolerance, x_out, infos);
            });
        }
    } else if (rc == BEMB200_OK) {  // bemb200_sweep_submit_incident: b = TbemSystem.rhs + incident block, formed on the device
        bemb200_ctx* ctx = sw->ctx_solve;
        cplx* bdev = sw->inc[job->slot];
        const size_t nb = (size_t)job->nrhs * sw->n * sizeof(cplx);
        // stream-ordered: a cudaFree would wait for the next frequency's assembly running beside this solve
        struct DevMem {
            cudaStream_t s;
            void* p = nullptr;
            ~DevMem() { if (p) cudaFreeAsync(p, s); }
        } sysv{ctx->stream}, xdev{ctx->stream};
        cudaError_t e = cudaSetDevice(ctx->device);
        if (e == cudaSuccess) e = cudaMallocAsync(&sysv.p, (sw->n ? sw->n : 1) * sizeof(cplx), ctx->stream);
        if (e == cudaSuccess && job->nrhs > 1) e = cudaMallocAsync(&xdev.p, nb ? nb : 1, ctx->stream);
        if (e != cudaSuccess) rc = cuda_fail(ctx, e, "sweep right-hand side block");
        if (rc == BEMB200_OK) rc = rhs_full(m, (double*)sysv.p, cudaMemcpyDeviceToDevice);  // TbemSystem.rhs (all rows)
        if (rc == BEMB200_OK) {
            std::lock_guard<std::mutex> lk(ctx->mu);
            e = launch_add_system_rhs((const cplx*)sysv.p, bdev, sw->n, job->nrhs, bdev, ctx->stream);
            if (e == cudaSuccess && rhs_out) e = cudaMemcpyAsync(rhs_out, bdev, nb, cudaMemcpyDeviceToHost, ctx->stream);
            if (e == cudaSuccess && rhs_out) e = cudaStreamSynchronize(ctx->stream);
            if (e != cudaSuccess) rc = cuda_fail(ctx, e, "sweep right-hand side block");
        }
        if (rc == BEMB200_OK && job->nrhs == 1) {
            rc = with_precond([&](const bemb200_precond* pc) {
                return gmres_solve_device_b(m, pc, (const double*)bdev, job->max_iterations, job->restart, job->tolerance, x_out, infos);
            });
        } else if (rc == BEMB200_OK) {
            rc = with_precond([&](const bemb200_precond* pc) {
                return bemb200_gmres_batched_device(m, pc, (const double*)bdev, job->nrhs, job->max_iterations, job->restart, job->tolerance,
                                                    (double*)xdev.p, infos, nullptr, nullptr);
            });
            if (rc == BEMB200_OK) {
                std::lock_guard<std::mutex> lk(ctx->mu);
                e = cudaMemcpyAsync(x_out, xdev.p, nb, cudaMemcpyDeviceToHost, ctx->stream);
                if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
                if (e != cudaSuccess) rc = cuda_fail(ctx, e, "sweep solution block");
            }
        }
    }
    bool boost = false;
    {
        std::lock_guard<std::mutex> lk(sw->mu);
        sw->solving = false;
        bemb200_ctx_set_shared_gpu(sw->ctx_solve, 0);
        sw->queue.pop_front();
        sw->next_to_assemble -= 1;
        sw->slot_busy[job->slot] = false;
        // the solver has left the GPU: a background assembly still in flight is joined by full-speed helper blocks
        boost = sw->overlap && !sw->queue.empty() && !sw->queue.front()->assembled && sw->buf[sw->queue.front()->slot] != nullptr;
    }
    sw->cv.notify_all();
    if (boost) {
        std::shared_ptr<SweepJob> nxt;
        {
            std::lock_guard<std::mutex> lk(sw->mu);
            if (!sw->queue.empty()) nxt = sw->queue.front();
        }
        if (nxt && sw->buf[nxt->slot] && bemb200_matrix_boost_assembly(sw->buf[nxt->slot], sw->ctx_solve) == BEMB200_OK) sw->boosts += 1;
    }
    return rc;
}

extern "C" {

int bemb200_sweep_next(bemb200_sweep* sw, double* x_out, bemb200_gmres_info* info, bemb200_assembly_stats* stats, double* rhs_out) {
    if (!sw || !x_out || !info) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    return sweep_take(sw, 1, x_out, info, nullptr, stats, rhs_out);
}

int bemb200_sweep_next_batch(bemb200_sweep* sw, uint32_t capacity, double* x_out, bemb200_gmres_info* infos, uint32_t* nrhs_out,
                             bemb200_assembly_stats* stats) {
    if (!sw || !x_out || !infos || !nrhs_out) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    return sweep_take(sw, capacity, x_out, infos, nrhs_out, stats, nullptr);
}

uint64_t bemb200_sweep_boosts(const bemb200_sweep* sw) { return sw ? sw->boosts : 0; }

int bemb200_sweep_set_block_jacobi(bemb200_sweep* sw, uint32_t num_subdomains, const uint64_t* sub_ptr, const uint64_t* sub_idx) {
    if (!sw) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    if ((sub_ptr == nullptr) != (sub_idx == nullptr)) return set_error(sw->ctx_solve, BEMB200_EINVAL, "sub_ptr and sub_idx go together");
    std::lock_guard<std::mutex> lk(sw->mu);
    sw->precond = num_subdomains > 0;
    sw->pc_subdomains = num_subdomains;
    sw->pc_ptr.clear(); sw->pc_idx.clear();
    if (sw->precond && sub_ptr) {
        sw->pc_ptr.assign(sub_ptr, sub_ptr + num_subdomains + 1);
        sw->pc_idx.assign(sub_idx, sub_idx + sub_ptr[num_subdomains]);
    }
    return BEMB200_OK;
}

int bemb200_sweep_set_assembly_options(bemb200_sweep* sw, const bemb200_assembly_options* opts) {
    if (!sw) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    if (check_assembly_options(sw->ctx_solve, sw->staged, opts) != BEMB200_OK) return BEMB200_EINVAL;
    AssemblyOptionsCopy c;
    if (opts) {
        c.dg_dn_sign = opts->dg_dn_sign;
        c.consistent_beta = opts->consistent_beta;
        if (opts->admittance) c.admittance.assign(opts->admittance, opts->admittance + 2 * sw->n);
    }
    std::lock_guard<std::mutex> lk(sw->mu);
    sw->opts = std::move(c);
    return BEMB200_OK;
}

void bemb200_sweep_destroy(bemb200_sweep* sw) {
    if (!sw) return;
    {
        std::lock_guard<std::mutex> lk(sw->mu);
        sw->stop = true;
    }
    sw->cv.notify_all();
    if (sw->worker.joinable()) sw->worker.join();
    if (sw->inc[0] || sw->inc[1]) {
        cudaSetDevice(sw->ctx_asm->device);
        for (int i = 0; i < 2; ++i) cudaFree(sw->inc[i]);
    }
    for (int i = 0; i < 2; ++i)
        if (sw->buf[i]) bemb200_matrix_free(sw->buf[i]);
    if (sw->staged) bemb200_staged_mesh_free(sw->staged);
    if (sw->overlap && sw->ctx_asm) bemb200_ctx_destroy(sw->ctx_asm);
    if (sw->ctx_solve) bemb200_ctx_destroy(sw->ctx_solve);
    delete sw;
}

}  // extern "C"

// =============================================================================================================
// single-process multi-GPU group
// =============================================================================================================
struct bemb200_multi {
    int n = 0;
    std::vector<int> devices;
    std::vector<bemb200_ctx*> ctx;
    std::shared_ptr<bemb::PeerGroup> group;
    std::string err;
};
struct bemb200_multi_matrix {
    bemb200_multi* mg = nullptr;
    std::vector<bemb200_matrix*> m;
    uint64_t n = 0;
};

// run fn(rank) on one host thread per rank; first non-zero return code wins
template <class F>
static int on_all_ranks(bemb200_multi* mg, F fn) {
    std::vector<int> rc(mg->n, BEMB200_OK);
    std::vector<std::thread> th;
    for (int p = 0; p < mg->n; ++p) th.emplace_back([&, p] { rc[p] = fn(p); });
    for (auto& t : th) t.join();
    for (int p = 0; p < mg->n; ++p)
        if (rc[p] != BEMB200_OK) {
            mg->err = bemb200_last_error(mg->ctx[p]);
            return set_error(nullptr, rc[p], mg->err);
        }
    return BEMB200_OK;
}

extern "C" {

int bemb200_multi_create(const int* devices, int n, bemb200_multi** out) {
    if (!devices || !out || n < 1 || n > MAX_GROUP_RANKS) return set_error(nullptr, BEMB200_EINVAL, "bemb200_multi_create: 1..8 devices");
    *out = nullptr;
    std::unique_ptr<bemb200_multi> mg(new bemb200_multi());
    mg->n = n;
    mg->devices.assign(devices, devices + n);
    mg->group = std::make_shared<bemb::PeerGroup>();
    mg->group->nranks = n;
    for (int p = 0; p < n; ++p) mg->group->device[p] = devices[p];
    for (int p = 0; p < n; ++p) {
        bemb200_ctx* c = nullptr;
        int rc = bemb200_ctx_create_ex(devices[p], p, n, nullptr, nullptr, &c);  // no NCCL communicator: the group exchanges through peer memory
        if (rc != BEMB200_OK) {
            for (bemb200_ctx* q : mg->ctx) bemb200_ctx_destroy(q);
            return rc;
        }
        c->group = mg->group;
        int same = 0;  // ranks sharing this device split its SMs between their persistent solver kernels
        for (int q = 0; q < n; ++q) same += devices[q] == devices[p] ? 1 : 0;
        if (same > 1) {
            int sms = 0;
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, devices[p]);
            c->fused_grid = sms / same;
        }
        mg->ctx.push_back(c);
    }
    // peer access between distinct devices (both directions); a refusal is reported by the first solve
    for (int p = 0; p < n; ++p)
        for (int q = 0; q < n; ++q)
            if (devices[p] != devices[q]) {
                cudaSetDevice(devices[p]);
                cudaError_t e = cudaDeviceEnablePeerAccess(devices[q], 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) mg->group->peer_ok = false;
                cudaGetLastError();
            }
    *out = mg.release();
    return BEMB200_OK;
}

void bemb200_multi_destroy(bemb200_multi* mg) {
    if (!mg) return;
    for (bemb200_ctx* c : mg->ctx) bemb200_ctx_destroy(c);
    delete mg;
}

int bemb200_multi_num_ranks(const bemb200_multi* mg) { return mg ? mg->n : 0; }
const char* bemb200_multi_last_error(const bemb200_multi* mg) { return mg ? mg->err.c_str() : ""; }

int bemb200_multi_assemble(bemb200_multi* mg, const bemb200_mesh* mesh, const bemb200_physics* phys, double beta_re, double beta_im,
                           bemb200_multi_matrix** out) {
    if (!mg || !mesh || !phys || !out) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    *out = nullptr;
    std::unique_ptr<bemb200_multi_matrix> mm(new bemb200_multi_matrix());
    mm->mg = mg;
    mm->m.assign(mg->n, nullptr);
    uint64_t ndof = 0;
    for (uint64_t e = 0; e < mesh->n_elem; ++e) ndof += mesh->is_eval[e] ? 0 : 1;
    mm->n = ndof;
    int rc = on_all_ranks(mg, [&](int p) {
        uint64_t b = 0, e = 0;
        bemb200_partition(ndof, mg->n, p, &b, &e);
        return bemb200_assemble(mg->ctx[p], mesh, phys, beta_re, beta_im, b, e, &mm->m[p]);
    });
    if (rc != BEMB200_OK) {
        for (bemb200_matrix* m : mm->m)
            if (m) bemb200_matrix_free(m);
        return rc;
    }
    *out = mm.release();
    return BEMB200_OK;
}

void bemb200_multi_matrix_free(bemb200_multi_matrix* mm) {
    if (!mm) return;
    for (bemb200_matrix* m : mm->m)
        if (m) bemb200_matrix_free(m);
    delete mm;
}

uint64_t bemb200_multi_num_rows(const bemb200_multi_matrix* mm) { return mm ? mm->n : 0; }

int bemb200_multi_rhs_download(const bemb200_multi_matrix* mm, double* out) {
    if (!mm || !out) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    for (int p = 0; p < mm->mg->n; ++p) {
        const uint64_t b = bemb200_local_row_begin(mm->m[p]);
        int rc = bemb200_rhs_download(mm->m[p], out + 2 * b);
        if (rc != BEMB200_OK) return rc;
    }
    return BEMB200_OK;
}

int bemb200_multi_matrix_download(const bemb200_multi_matrix* mm, uint64_t row_begin, uint64_t row_end, double* out) {
    if (!mm || !out || row_begin > row_end || row_end > mm->n) return set_error(nullptr, BEMB200_EINVAL, "bad argument");
    for (int p = 0; p < mm->mg->n; ++p) {
        const uint64_t b = bemb200_local_row_begin(mm->m[p]), e = bemb200_local_row_end(mm->m[p]);
        const uint64_t lo = row_begin > b ? row_begin : b, hi = row_end < e ? row_end : e;
        if (lo >= hi) continue;
        int rc = bemb200_matrix_download(mm->m[p], lo, hi, out + 2 * (lo - row_begin) * mm->n);
        if (rc != BEMB200_OK) return rc;
    }
    return BEMB200_OK;
}

int bemb200_multi_gmres(const bemb200_multi_matrix* mm, const double* b, const double* x0, uint32_t max_iterations, uint32_t restart,
                        double tolerance, double* x_out, bemb200_gmres_info* info) {
    if (!mm || !b || !x_out || !info) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    bemb200_multi* mg = mm->mg;
    std::vector<bemb200_gmres_info> infos(mg->n);
    std::vector<std::vector<double>> xs(mg->n);
    int rc = on_all_ranks(mg, [&](int p) {
        xs[p].resize(p == 0 ? 0 : 2 * mm->n);
        return bemb200_gmres(mm->m[p], b, x0, max_iterations, restart, tolerance, p == 0 ? x_out : xs[p].data(), &infos[p]);
    });
    if (rc != BEMB200_OK) return rc;
    *info = infos[0];
    return BEMB200_OK;
}

}  // extern "C"
