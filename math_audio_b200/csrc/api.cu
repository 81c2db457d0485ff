// api.cu -- C ABI of libbemb200: context, mesh staging, assembly, matrix handle.
// (operator / GMRES entry points live in gmres.cu)
#include <cmath>
#include <cstdio>
#include <cstring>
#include <dlfcn.h>

#include "api_internal.h"

using namespace bemb;

namespace {
std::string g_last_error;
std::mutex g_err_mu;
}  // namespace

namespace bemb {
int set_error(bemb200_ctx* ctx, int code, const std::string& msg) {
    {
        std::lock_guard<std::mutex> lk(g_err_mu);
        g_last_error = msg;
    }
    if (ctx) ctx->err = msg;
    return code;
}
int cuda_fail(bemb200_ctx* ctx, cudaError_t e, const char* what) {
    cudaGetLastError();  // clear sticky-less errors
    return set_error(ctx, e == cudaErrorMemoryAllocation ? BEMB200_ENOMEM : BEMB200_ECUDA,
                     std::string("CUDA error '") + cudaGetErrorString(e) + "' in " + what);
}
}  // namespace bemb

// ---- NCCL through dlopen (only needed for nranks > 1) ----------------------------------
namespace ncclshim {
typedef struct { char internal[128]; } UniqueId;
typedef int (*GetUniqueId_t)(UniqueId*);
typedef int (*CommInitRank_t)(void**, int, UniqueId, int);
typedef int (*CommDestroy_t)(void*);
typedef int (*AllGather_t)(const void*, void*, size_t, int, void*, cudaStream_t);
typedef const char* (*GetErrorString_t)(int);
void* handle = nullptr;
GetUniqueId_t GetUniqueId = nullptr;
CommInitRank_t CommInitRank = nullptr;
CommDestroy_t CommDestroy = nullptr;
AllGather_t AllGather = nullptr;
GetErrorString_t GetErrorString = nullptr;
bool load(std::string& why) {
    if (handle) return true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
        handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (handle) break;
    }
    if (!handle) {
        why = std::string("cannot dlopen libnccl.so.2: ") + dlerror();
        return false;
    }
    GetUniqueId = (GetUniqueId_t)dlsym(handle, "ncclGetUniqueId");
    CommInitRank = (CommInitRank_t)dlsym(handle, "ncclCommInitRank");
    CommDestroy = (CommDestroy_t)dlsym(handle, "ncclCommDestroy");
    AllGather = (AllGather_t)dlsym(handle, "ncclAllGather");
    GetErrorString = (GetErrorString_t)dlsym(handle, "ncclGetErrorString");
    if (!GetUniqueId || !CommInitRank || !CommDestroy || !AllGather) {
        why = "libnccl is missing required symbols";
        return false;
    }
    return true;
}
}  // namespace ncclshim

namespace bemb {
// all-gather `count_bytes` bytes per rank (in-stream); used by gmres.cu
int nccl_allgather_bytes(bemb200_ctx* ctx, const void* send, void* recv, size_t count_bytes) {
    if (ctx->nranks == 1) return BEMB200_OK;
    if (!ctx->nccl_comm) return set_error(ctx, BEMB200_ENCCL, "this context was created without a communicator (assembly only)");
    int rc = ncclshim::AllGather(send, recv, count_bytes, /*ncclInt8=*/0, ctx->nccl_comm, ctx->stream);
    if (rc != 0)
        return set_error(ctx, BEMB200_ENCCL, std::string("ncclAllGather failed: ") +
                                                 (ncclshim::GetErrorString ? ncclshim::GetErrorString(rc) : "?"));
    return BEMB200_OK;
}
}  // namespace bemb

// ---- staging ------------------------------------------------------------------------------
template <class T>
static int dev_alloc_copy(bemb200_staged_mesh* sm, T** dst, const std::vector<T>& src) {
    size_t bytes = src.size() * sizeof(T);
    if (bytes == 0) bytes = sizeof(T);
    BEMB_CUDA(sm->ctx, cudaMallocAsync((void**)dst, bytes, sm->ctx->stream));
    sm->allocs.push_back(*dst);
    if (!src.empty()) BEMB_CUDA(sm->ctx, cudaMemcpyAsync(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice, sm->ctx->stream));
    return BEMB200_OK;
}
template <class T>
static int dev_alloc(bemb200_staged_mesh* sm, T** dst, size_t count) {
    BEMB_CUDA(sm->ctx, cudaMallocAsync((void**)dst, (count ? count : 1) * sizeof(T), sm->ctx->stream));
    sm->allocs.push_back(*dst);
    return BEMB200_OK;
}

extern "C" {

int bemb200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

static int ctx_create_common(int device, void* ext_stream, bemb200_ctx** out) {
    if (!out) return set_error(nullptr, BEMB200_EINVAL, "out is NULL");
    *out = nullptr;
    int n = bemb200_device_count();
    if (n <= 0) return set_error(nullptr, BEMB200_ENODEVICE, "no CUDA device visible (libbemb200 has no CPU fallback)");
    if (device < 0 || device >= n) return set_error(nullptr, BEMB200_EINVAL, "device index out of range");
    bemb200_ctx* c = new bemb200_ctx();
    c->device = device;
    BEMB_CUDA(c, cudaSetDevice(device));
    cudaDeviceProp prop;
    BEMB_CUDA(c, cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        std::string msg = std::string("device '") + prop.name + "' is not sm_100 (libbemb200 ships sm_100a code only)";
        delete c;
        return set_error(nullptr, BEMB200_EUNSUPPORTED, msg);
    }
    {
        // keep stream-ordered (cudaMallocAsync) staging memory cached between calls
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            unsigned long long thr = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
        }
        cudaGetLastError();
    }
    if (ext_stream) {
        c->stream = (cudaStream_t)ext_stream;
        c->own_stream = false;
    } else {
        BEMB_CUDA(c, cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    }
    *out = c;
    return BEMB200_OK;
}

int bemb200_ctx_create(int device, bemb200_ctx** out) { return ctx_create_common(device, nullptr, out); }

int bemb200_nccl_unique_id(uint8_t out[128]) {
    std::string why;
    if (!ncclshim::load(why)) return set_error(nullptr, BEMB200_ENCCL, why);
    ncclshim::UniqueId id;
    int rc = ncclshim::GetUniqueId(&id);
    if (rc != 0) return set_error(nullptr, BEMB200_ENCCL, "ncclGetUniqueId failed");
    std::memcpy(out, id.internal, 128);
    return BEMB200_OK;
}

int bemb200_ctx_create_dist(int device, int rank, int nranks, const uint8_t nccl_id[128], bemb200_ctx** out) {
    return bemb200_ctx_create_ex(device, rank, nranks, nccl_id, nullptr, out);
}

int bemb200_ctx_create_ex(int device, int rank, int nranks, const uint8_t* nccl_id, void* cuda_stream, bemb200_ctx** out) {
    if (nranks < 1 || rank < 0 || rank >= nranks) return set_error(nullptr, BEMB200_EINVAL, "bad rank/nranks");
    int rc = ctx_create_common(device, cuda_stream, out);
    if (rc != BEMB200_OK) return rc;
    bemb200_ctx* c = *out;
    c->rank = rank;
    c->nranks = nranks;
    if (nranks > 1 && nccl_id) {
        std::string why;
        if (!ncclshim::load(why)) {
            bemb200_ctx_destroy(c);
            *out = nullptr;
            return set_error(nullptr, BEMB200_ENCCL, why);
        }
        ncclshim::UniqueId id;
        std::memcpy(id.internal, nccl_id, 128);
        int nrc = ncclshim::CommInitRank(&c->nccl_comm, nranks, id, rank);
        if (nrc != 0) {
            bemb200_ctx_destroy(c);
            *out = nullptr;
            return set_error(nullptr, BEMB200_ENCCL, "ncclCommInitRank failed");
        }
    }
    return BEMB200_OK;
}

void bemb200_ctx_destroy(bemb200_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    free_peer_exchange(ctx, false);
    if (ctx->nccl_comm && ncclshim::CommDestroy) ncclshim::CommDestroy(ctx->nccl_comm);
    if (ctx->stream && ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char* bemb200_last_error(const bemb200_ctx* ctx) {
    if (ctx) return ctx->err.c_str();
    return g_last_error.c_str();
}

void bemb200_partition(uint64_t n, int nranks, int rank, uint64_t* row_begin, uint64_t* row_end) {
    uint64_t chunk = (n + (uint64_t)nranks - 1) / (uint64_t)nranks;
    uint64_t b = chunk * (uint64_t)rank, e = b + chunk;
    if (b > n) b = n;
    if (e > n) e = n;
    *row_begin = b;
    *row_end = e;
}

void bemb200_staged_mesh_free(bemb200_staged_mesh* sm) {
    if (!sm) return;
    cudaSetDevice(sm->ctx->device);
    // stream-ordered frees (no device-wide synchronisation, unlike cudaFree)
    for (void* p : sm->allocs) cudaFreeAsync(p, sm->ctx->stream);
    delete sm;
}

uint64_t bemb200_staged_num_dofs(const bemb200_staged_mesh* sm) { return sm ? sm->dm.n : 0; }

int bemb200_mesh_stage(bemb200_ctx* ctx, const bemb200_mesh* mesh, bemb200_staged_mesh** out) {
    if (!ctx) return set_error(nullptr, BEMB200_EINVAL, "ctx is NULL");
    if (!mesh || !out) return set_error(ctx, BEMB200_EINVAL, "mesh/out is NULL");
    *out = nullptr;
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint64_t ne = mesh->n_elem;
    // count_dofs(): tbem.rs:225-231
    uint64_t ndof = 0;
    for (uint64_t e = 0; e < ne; ++e) ndof += mesh->is_eval[e] ? 0 : 1;
    if (ndof == 0) return set_error(ctx, BEMB200_EINVAL, "mesh has no boundary (non-evaluation) element");
    if (ndof > 0x7fffffffull) return set_error(ctx, BEMB200_EINVAL, "too many DOFs");
    std::vector<int64_t> elem_of_dof(ndof, -1);
    for (uint64_t e = 0; e < ne; ++e) {
        if (mesh->is_eval[e]) continue;
        uint64_t d = mesh->dof[e];
        if (d >= ndof || elem_of_dof[d] != -1)
            return set_error(ctx, BEMB200_EINVAL, "dof addresses of boundary elements must be a permutation of 0..ndof-1");
        elem_of_dof[d] = (int64_t)e;
        int et = mesh->etype[e];
        if (et != 3 && et != 4) return set_error(ctx, BEMB200_EINVAL, "etype must be 3 (Tri3) or 4 (Quad4)");
        for (int v = 0; v < et; ++v)
            if (mesh->conn[4 * e + v] >= mesh->n_nodes) return set_error(ctx, BEMB200_EINVAL, "connectivity index out of range");
        if (mesh->bc_len[e] < 1 || mesh->bc_len[e] > 4) return set_error(ctx, BEMB200_EINVAL, "bc_len must be 1..4");
    }
    bemb200_staged_mesh* sm = new bemb200_staged_mesh();
    sm->ctx = ctx;
    DeviceMesh& dm = sm->dm;
    dm.n = (uint32_t)ndof;
    dm.ntiles = (uint32_t)((ndof + TILE - 1) / TILE);
    std::vector<double> coords(ndof * 12, 0.0), area(ndof), src(ndof * 8, 0.0);
    std::vector<uint8_t> etype(ndof), bclen(ndof), nz(ndof);
    std::vector<int32_t> bctype(ndof);
    std::vector<cplx> bcval(ndof * 4);
    for (uint64_t d = 0; d < ndof; ++d) {
        const uint64_t e = (uint64_t)elem_of_dof[d];
        const int et = mesh->etype[e];
        etype[d] = (uint8_t)et;
        for (int v = 0; v < et; ++v)
            for (int c = 0; c < 3; ++c) coords[12 * d + 3 * v + c] = mesh->nodes[3 * (uint64_t)mesh->conn[4 * e + v] + c];
        area[d] = mesh->area[e];
        for (int c = 0; c < 3; ++c) {
            src[8 * d + c] = mesh->center[3 * e + c];
            src[8 * d + 3 + c] = mesh->normal[3 * e + c];
        }
        bctype[d] = mesh->bc_type[e];
        bclen[d] = mesh->bc_len[e];
        bool nonzero = false;
        for (int i = 0; i < 4; ++i) {
            cplx v = C(0, 0);
            if (i < mesh->bc_len[e]) v = C(mesh->bc_val[8 * e + 2 * i], mesh->bc_val[8 * e + 2 * i + 1]);
            bcval[4 * d + i] = v;
            if (i < mesh->bc_len[e] && std::hypot(v.re, v.im) > 1e-15) nonzero = true;  // has_nonzero_bc: tbem.rs:247
        }
        nz[d] = nonzero ? 1 : 0;
    }
    // avg radius of the first <=100 ELEMENTS in element order (tbem.rs:108-117)
    {
        double avg = 0.0;
        uint64_t n_calc = ne < 100 ? ne : 100;
        for (uint64_t e = 0; e < n_calc; ++e) {
            const double* c = mesh->center + 3 * e;
            double s = 0.0;
            s = s + c[0] * c[0];
            s = s + c[1] * c[1];
            s = s + c[2] * c[2];
            avg += std::sqrt(s);
        }
        if (n_calc > 0) avg /= (double)n_calc;
        dm.avg_radius_first100 = avg;
    }
    int rc;
#define STAGE_TRY(x)                         \
    do {                                     \
        rc = (x);                            \
        if (rc != BEMB200_OK) {              \
            bemb200_staged_mesh_free(sm);    \
            return rc;                       \
        }                                    \
    } while (0)
    STAGE_TRY(dev_alloc_copy(sm, &dm.coords, coords));
    STAGE_TRY(dev_alloc_copy(sm, &dm.etype, etype));
    STAGE_TRY(dev_alloc_copy(sm, &dm.area, area));
    STAGE_TRY(dev_alloc_copy(sm, &dm.src, src));
    STAGE_TRY(dev_alloc_copy(sm, &dm.bc_type, bctype));
    sm->bc_type = bctype;
    STAGE_TRY(dev_alloc_copy(sm, &dm.bc_len, bclen));
    STAGE_TRY(dev_alloc_copy(sm, &dm.bc_val, bcval));
    STAGE_TRY(dev_alloc_copy(sm, &dm.nonzero_bc, nz));
    STAGE_TRY(dev_alloc(sm, &dm.esize, ndof));
    STAGE_TRY(dev_alloc(sm, &dm.far_k, (size_t)dm.ntiles * NQ_MAX * TILE));
    STAGE_TRY(dev_alloc(sm, &dm.far_c, (size_t)dm.ntiles * FAR_NCONST * TILE));
    STAGE_TRY(dev_alloc(sm, &dm.col_class, (size_t)dm.ntiles * TILE));
    cudaError_t e = launch_prep(dm, ctx->stream);
    if (e != cudaSuccess) {
        bemb200_staged_mesh_free(sm);
        return cuda_fail(ctx, e, "prep_kernel launch");
    }
    std::vector<uint8_t> cls((size_t)dm.ntiles * TILE);
    e = cudaMemcpyAsync(cls.data(), dm.col_class, cls.size(), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        bemb200_staged_mesh_free(sm);
        return cuda_fail(ctx, e, "prep_kernel");
    }
    std::vector<uint32_t> special, rhs_tri, rhs_quad;
    for (uint32_t j = 0; j < dm.n; ++j) {
        if (cls[j] == COL_SPECIAL) special.push_back(j);
        else if (cls[j] == COL_FLAT_TRI) { dm.n_flat_tri++; if (nz[j]) rhs_tri.push_back(j); }
        else if (cls[j] == COL_FLAT_QUAD) { dm.n_flat_quad++; if (nz[j]) rhs_quad.push_back(j); }
    }
    dm.n_special = (uint32_t)special.size();
    dm.n_rhs_tri = (uint32_t)rhs_tri.size();
    dm.n_rhs_quad = (uint32_t)rhs_quad.size();
    STAGE_TRY(dev_alloc_copy(sm, &dm.special_cols, special));
    STAGE_TRY(dev_alloc_copy(sm, &dm.rhs_cols_tri, rhs_tri));
    STAGE_TRY(dev_alloc_copy(sm, &dm.rhs_cols_quad, rhs_quad));
    e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        bemb200_staged_mesh_free(sm);
        return cuda_fail(ctx, e, "stage sync");
    }
#undef STAGE_TRY
    *out = sm;
    return BEMB200_OK;
}

double bemb200_dg_dn_sign(const bemb200_staged_mesh* sm, double wave_number) {
    if (!sm) return 0.0;
    double ka = wave_number * sm->dm.avg_radius_first100;  // tbem.rs:118-123
    return ka < 0.5 ? 1.0 : -1.0;
}

// ---- matrix handle ----------------------------------------------------------------------------
static int matrix_alloc(bemb200_ctx* ctx, uint64_t n_rows, uint64_t n_cols, uint64_t r0, uint64_t r1, bool with_near,
                        bemb200_matrix** out) {
    bemb200_matrix* m = new bemb200_matrix();
    m->ctx = ctx;
    m->n_rows = n_rows;
    m->n_cols = n_cols;
    m->r0 = r0;
    m->r1 = r1;
    const uint64_t nloc = r1 - r0;
    cudaError_t e = cudaMalloc((void**)&m->A, (nloc * n_cols + 1) * sizeof(cplx));
    if (e == cudaSuccess) e = cudaMalloc((void**)&m->rhs, (nloc + 1) * sizeof(cplx));
    if (e == cudaSuccess) e = cudaMemsetAsync(m->rhs, 0, (nloc + 1) * sizeof(cplx), ctx->stream);
    if (e == cudaSuccess && with_near) {
        m->near_cap = (unsigned int)(nloc * 64 + 4096);
        e = cudaMalloc((void**)&m->near_list, (size_t)m->near_cap * sizeof(uint2));
        if (e == cudaSuccess) e = cudaMalloc((void**)&m->near_count, sizeof(unsigned int));
        if (e == cudaSuccess) e = cudaMalloc((void**)&m->work_counters, 2 * sizeof(unsigned int));
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&m->far_ready_ev, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&m->boost_ev, cudaEventDisableTiming);
    }
    for (int i = 0; i < 4 && e == cudaSuccess; ++i) e = cudaEventCreate(&m->ev[i]);
    if (e != cudaSuccess) {
        bemb200_matrix_free(m);
        return cuda_fail(ctx, e, "matrix allocation");
    }
    *out = m;
    return BEMB200_OK;
}

}  // extern "C" (reopened below)
namespace bemb {
int matrix_alloc_plain(bemb200_ctx* ctx, uint64_t n_rows, uint64_t n_cols, uint64_t r0, uint64_t r1, bemb200_matrix** out) {
    return matrix_alloc(ctx, n_rows, n_cols, r0, r1, false, out);
}
}  // namespace bemb
extern "C" {

void bemb200_matrix_free(bemb200_matrix* m) {
    if (!m) return;
    cudaSetDevice(m->ctx->device);
    free_workspace(m);
    if (m->A) cudaFree(m->A);
    if (m->rhs) cudaFree(m->rhs);
    if (m->adm) cudaFree(m->adm);
    if (m->near_list) cudaFree(m->near_list);
    if (m->near_count) cudaFree(m->near_count);
    if (m->work_counters) cudaFree(m->work_counters);
    if (m->far_ready_ev) cudaEventDestroy(m->far_ready_ev);
    if (m->boost_ev) cudaEventDestroy(m->boost_ev);
    for (int i = 0; i < 4; ++i)
        if (m->ev[i]) cudaEventDestroy(m->ev[i]);
    delete m;
}

}  // extern "C" (reopened below)
namespace bemb {
int check_assembly_options(bemb200_ctx* ctx, const bemb200_staged_mesh* sm, const bemb200_assembly_options* opts) {
    if (!opts) return BEMB200_OK;
    if (opts->dg_dn_sign != 0 && opts->dg_dn_sign != 1 && opts->dg_dn_sign != -1)
        return set_error(ctx, BEMB200_EINVAL, "dg_dn_sign must be 0 (heuristic), +1 or -1");
    if (opts->consistent_beta != 0 && opts->consistent_beta != 1) return set_error(ctx, BEMB200_EINVAL, "consistent_beta must be 0 or 1");
    if (opts->admittance)
        for (uint32_t j = 0; j < sm->dm.n; ++j)
            if (sm->bc_type[j] != 0 && (opts->admittance[2 * j] != 0.0 || opts->admittance[2 * j + 1] != 0.0))
                return set_error(ctx, BEMB200_EINVAL, "admittance is allowed on velocity-BC elements only (DOF " + std::to_string(j) +
                                                          " has bc_type " + std::to_string(sm->bc_type[j]) + ")");
    return BEMB200_OK;
}
}  // namespace bemb
extern "C" {

int bemb200_assemble_staged(bemb200_ctx* ctx, const bemb200_staged_mesh* sm, const bemb200_physics* phys, double beta_re,
                            double beta_im, uint64_t row_begin, uint64_t row_end, bemb200_matrix** inout) {
    return bemb200_assemble_staged_opts(ctx, sm, phys, beta_re, beta_im, nullptr, row_begin, row_end, inout);
}

int bemb200_assemble_staged_opts(bemb200_ctx* ctx, const bemb200_staged_mesh* sm, const bemb200_physics* phys, double beta_re,
                                 double beta_im, const bemb200_assembly_options* opts, uint64_t row_begin, uint64_t row_end,
                                 bemb200_matrix** inout) {
    if (!ctx) return set_error(nullptr, BEMB200_EINVAL, "ctx is NULL");
    if (!sm || !phys || !inout) return set_error(ctx, BEMB200_EINVAL, "NULL argument");
    const DeviceMesh& dm = sm->dm;
    if (row_begin > row_end || row_end > dm.n) return set_error(ctx, BEMB200_EINVAL, "row range outside [0, num_dofs]");
    if (!(phys->wave_number > 0.0)) return set_error(ctx, BEMB200_EINVAL, "wave_number must be > 0");
    if (check_assembly_options(ctx, sm, opts) != BEMB200_OK) return BEMB200_EINVAL;
    bool has_adm = false;
    if (opts && opts->admittance)
        for (uint64_t j = 0; j < 2ull * dm.n && !has_adm; ++j) has_adm = opts->admittance[j] != 0.0;
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    bemb200_matrix* m = *inout;
    if (m) {
        if (m->n_rows != dm.n || m->n_cols != dm.n || m->r0 != row_begin || m->r1 != row_end || !m->near_list)
            return set_error(ctx, BEMB200_EINVAL, "matrix handle to reuse has a different shape / row range");
    } else {
        int rc = matrix_alloc(ctx, dm.n, dm.n, row_begin, row_end, true, &m);
        if (rc != BEMB200_OK) return rc;
    }
    Phys ph;
    ph.k = phys->wave_number;
    ph.wavruim = phys->harmonic_factor * phys->wave_number;
    ph.k2 = phys->wave_number * phys->wave_number;
    ph.tau = phys->tau;
    ph.gamma = phys->gamma;
    ph.sign = bemb200_dg_dn_sign(sm, phys->wave_number);
    ph.beta = C(beta_re, beta_im);
    ph.beta_unscaled = phys->tau > 0.0 ? C(0.0, phys->harmonic_factor / phys->wave_number) : C(0.0, 0.0);  // types.rs:64-70
    ph.adm = nullptr;
    if (opts && opts->dg_dn_sign != 0) ph.sign = (double)opts->dg_dn_sign;
    if (opts && opts->consistent_beta) ph.beta_unscaled = ph.beta;
    const uint64_t nloc = row_end - row_begin;
    cudaStream_t s = ctx->stream;
    int rc = BEMB200_OK;
    unsigned int count = 0;
    auto fail = [&](int code) {
        if (!*inout) bemb200_matrix_free(m);
        return code;
    };
#define ASM_CUDA(call)                                                 \
    do {                                                               \
        cudaError_t _e = (call);                                       \
        if (_e != cudaSuccess) return fail(cuda_fail(ctx, _e, #call)); \
    } while (0)
    ASM_CUDA(cudaMemsetAsync(m->rhs, 0, (nloc + 1) * sizeof(cplx), s));
    if (has_adm) {  // an all-zero admittance launches exactly the kernels of an assembly without one
        if (!m->adm) ASM_CUDA(cudaMalloc((void**)&m->adm, (size_t)dm.n * sizeof(cplx)));
        ASM_CUDA(cudaMemcpyAsync(m->adm, opts->admittance, (size_t)dm.n * sizeof(cplx), cudaMemcpyHostToDevice, s));
        ph.adm = m->adm;
    }
    if (dm.n_special) ASM_CUDA(cudaMemsetAsync(m->A, 0, nloc * dm.n * sizeof(cplx), s));  // transfer-BC columns stay 0
    ASM_CUDA(cudaEventRecord(m->ev[0], s));
    for (int attempt = 0; attempt < 2; ++attempt) {
        ASM_CUDA(cudaMemsetAsync(m->near_count, 0, sizeof(unsigned int), s));
        const int bg = ctx->background_blocks_per_sm.load();
        const bool boostable = bg > 0 && attempt == 0 && m->work_counters;
        if (boostable) {
            ASM_CUDA(cudaMemsetAsync(m->work_counters, 0, 2 * sizeof(unsigned int), s));
            ASM_CUDA(cudaEventRecord(m->far_ready_ev, s));  // everything the far pass depends on is enqueued before this
        }
        ASM_CUDA(cudaEventRecord(m->ev[1], s));
        {
            std::lock_guard<std::mutex> bl(m->boost_mu);
            m->relaunch.clear();
            m->boost_pending = false;
            cudaError_t fe = launch_far(dm, ph, row_begin, row_end, m->A, dm.n, m->near_list, m->near_cap, m->near_count, bg,
                                        boostable ? m->work_counters : nullptr, boostable ? &m->relaunch : nullptr, s);
            if (fe != cudaSuccess) return fail(cuda_fail(ctx, fe, "launch_far"));
            m->far_running = boostable;
        }
        ASM_CUDA(cudaEventRecord(m->ev[2], s));
        ASM_CUDA(cudaMemcpyAsync(&count, m->near_count, sizeof(unsigned int), cudaMemcpyDeviceToHost, s));
        ASM_CUDA(cudaStreamSynchronize(s));
        {
            // the persistent blocks are done; helper blocks of a boost may still hold their last items
            bool pending;
            {
                std::lock_guard<std::mutex> bl(m->boost_mu);
                m->far_running = false;
                pending = m->boost_pending;
                m->boost_pending = false;
                m->relaunch.clear();
            }
            if (pending) {
                ASM_CUDA(cudaEventSynchronize(m->boost_ev));
                ASM_CUDA(cudaMemcpyAsync(&count, m->near_count, sizeof(unsigned int), cudaMemcpyDeviceToHost, s));
                ASM_CUDA(cudaStreamSynchronize(s));
            }
        }
        if (count <= m->near_cap) break;
        // list overflow (pathological mesh): grow and redo the far pass once
        cudaFree(m->near_list);
        m->near_list = nullptr;
        m->near_cap = count + 1024;
        ASM_CUDA(cudaMalloc((void**)&m->near_list, (size_t)m->near_cap * sizeof(uint2)));
    }
    if (count > m->near_cap) {  // still overflowing after the regrown second pass: never index past the list
        if (!*inout) bemb200_matrix_free(m);
        return set_error(ctx, BEMB200_ENOMEM, "near-field pair list overflowed twice (pathological mesh: more near pairs than the list can hold)");
    }
    ASM_CUDA(launch_near_list(dm, ph, row_begin, m->A, dm.n, m->rhs, m->near_list, count, s));
    ASM_CUDA(launch_rhs_far(dm, ph, row_begin, row_end, m->rhs, s));
    ASM_CUDA(launch_special(dm, ph, row_begin, row_end, m->A, dm.n, m->rhs, s));
    ASM_CUDA(launch_self(dm, ph, row_begin, row_end, m->A, dm.n, m->rhs, s));
    ASM_CUDA(cudaEventRecord(m->ev[3], s));
    ASM_CUDA(cudaStreamSynchronize(s));
#undef ASM_CUDA
    float far_ms = 0.f, tot_ms = 0.f;
    cudaEventElapsedTime(&far_ms, m->ev[1], m->ev[2]);
    cudaEventElapsedTime(&tot_ms, m->ev[0], m->ev[3]);
    m->stats.near_pairs = count;
    m->stats.special_pairs = (uint64_t)dm.n_special * nloc;
    m->stats.far_kernel_launches = (uint64_t)far_kernel_launch_count(dm);
    m->stats.total_launches = m->stats.far_kernel_launches + (count ? 1 : 0) + (dm.n_special ? 1 : 0) + 1 +
                              (dm.n_rhs_tri ? 1 : 0) + (dm.n_rhs_quad ? 1 : 0);
    m->stats.far_ms = far_ms;
    m->stats.total_ms = tot_ms;
    *inout = m;
    return rc;
}

int bemb200_assemble(bemb200_ctx* ctx, const bemb200_mesh* mesh, const bemb200_physics* phys, double beta_re,
                     double beta_im, uint64_t row_begin, uint64_t row_end, bemb200_matrix** out) {
    if (!out) return set_error(ctx, BEMB200_EINVAL, "out is NULL");
    *out = nullptr;
    bemb200_staged_mesh* sm = nullptr;
    int rc = bemb200_mesh_stage(ctx, mesh, &sm);
    if (rc != BEMB200_OK) return rc;
    rc = bemb200_assemble_staged(ctx, sm, phys, beta_re, beta_im, row_begin, row_end, out);
    bemb200_staged_mesh_free(sm);
    return rc;
}

int bemb200_assembly_stats_get(const bemb200_matrix* m, bemb200_assembly_stats* out) {
    if (!m || !out) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    *out = m->stats;
    return BEMB200_OK;
}

int bemb200_matrix_from_host(bemb200_ctx* ctx, const double* a_rows, uint64_t n_rows_global, uint64_t n_cols,
                             uint64_t row_begin, uint64_t row_end, bemb200_matrix** out) {
    if (!ctx) return set_error(nullptr, BEMB200_EINVAL, "ctx is NULL");
    if (!a_rows || !out || row_begin > row_end || row_end > n_rows_global || n_cols == 0)
        return set_error(ctx, BEMB200_EINVAL, "bad argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    bemb200_matrix* m = nullptr;
    int rc = matrix_alloc(ctx, n_rows_global, n_cols, row_begin, row_end, false, &m);
    if (rc != BEMB200_OK) return rc;
    cudaError_t e = cudaMemcpyAsync(m->A, a_rows, (row_end - row_begin) * n_cols * sizeof(cplx), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        bemb200_matrix_free(m);
        return cuda_fail(ctx, e, "matrix upload");
    }
    *out = m;
    return BEMB200_OK;
}

int bemb200_ctx_set_background(bemb200_ctx* ctx, int blocks_per_sm) {
    if (!ctx || blocks_per_sm < 0 || blocks_per_sm > 8) return set_error(ctx, BEMB200_EINVAL, "blocks_per_sm must be 0..8");
    // lock-free on purpose: may be flipped by another thread WHILE an assembly call of this context
    // is in flight (the call re-reads it between row slabs)
    ctx->background_blocks_per_sm.store(blocks_per_sm);
    return BEMB200_OK;
}

int bemb200_ctx_set_shared_gpu(bemb200_ctx* ctx, int shared) {
    if (!ctx) return set_error(ctx, BEMB200_EINVAL, "NULL context");
    ctx->shared_gpu.store(shared ? 1 : 0);
    return BEMB200_OK;
}

int bemb200_matrix_boost_assembly(bemb200_matrix* m, bemb200_ctx* ctx) {
    if (!m || !ctx) return set_error(ctx, BEMB200_EINVAL, "NULL argument");
    if (ctx->device != m->ctx->device) return set_error(ctx, BEMB200_EINVAL, "contexts must share the device");
    std::lock_guard<std::mutex> lk(ctx->mu);
    std::lock_guard<std::mutex> bl(m->boost_mu);
    if (!m->far_running || m->relaunch.empty() || m->boost_pending) return BEMB200_OK;  // nothing in flight (or already boosted)
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    BEMB_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, m->far_ready_ev, 0));
    for (auto& fn : m->relaunch) BEMB_CUDA(ctx, fn(ctx->stream));
    BEMB_CUDA(ctx, cudaEventRecord(m->boost_ev, ctx->stream));
    m->boost_pending = true;
    return BEMB200_OK;
}

int bemb200_ctx_peer_exchange_active(const bemb200_ctx* ctx, int* active) {
    if (!ctx || !active) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    *active = ctx->px.ok ? 1 : 0;
    return BEMB200_OK;
}

int bemb200_matrix_set_context(bemb200_matrix* m, bemb200_ctx* ctx) {
    if (!m || !ctx) return set_error(ctx, BEMB200_EINVAL, "NULL argument");
    if (ctx->device != m->ctx->device || ctx->nranks != m->ctx->nranks || ctx->rank != m->ctx->rank)
        return set_error(ctx, BEMB200_EINVAL, "contexts must share device, rank and nranks");
    std::lock_guard<std::mutex> lk(m->ctx->mu);
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(m->ctx->stream);
    free_workspace(m);  // the solver workspace is re-created lazily on the new context's stream
    m->ctx = ctx;
    return BEMB200_OK;
}

uint64_t bemb200_num_rows(const bemb200_matrix* m) { return m ? m->n_rows : 0; }
uint64_t bemb200_num_cols(const bemb200_matrix* m) { return m ? m->n_cols : 0; }
uint64_t bemb200_local_row_begin(const bemb200_matrix* m) { return m ? m->r0 : 0; }
uint64_t bemb200_local_row_end(const bemb200_matrix* m) { return m ? m->r1 : 0; }
void* bemb200_matrix_device_ptr(const bemb200_matrix* m) { return m ? (void*)m->A : nullptr; }

int bemb200_matrix_download(const bemb200_matrix* m, uint64_t row_begin, uint64_t row_end, double* out) {
    if (!m || !out) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    bemb200_ctx* ctx = m->ctx;
    if (row_begin > row_end || row_begin < m->r0 || row_end > m->r1) return set_error(ctx, BEMB200_EINVAL, "rows outside the local slab");
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    BEMB_CUDA(ctx, cudaMemcpyAsync(out, m->A + (row_begin - m->r0) * m->n_cols, (row_end - row_begin) * m->n_cols * sizeof(cplx),
                                   cudaMemcpyDeviceToHost, ctx->stream));
    BEMB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return BEMB200_OK;
}

int bemb200_rhs_download(const bemb200_matrix* m, double* out) {
    if (!m || !out) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    bemb200_ctx* ctx = m->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    BEMB_CUDA(ctx, cudaMemcpyAsync(out, m->rhs, (m->r1 - m->r0) * sizeof(cplx), cudaMemcpyDeviceToHost, ctx->stream));
    BEMB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return BEMB200_OK;
}

}  // extern "C"
