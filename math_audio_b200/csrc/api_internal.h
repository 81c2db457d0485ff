// Handle definitions behind the opaque C types of include/bemb200.h.
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <condition_variable>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/bemb200.h"
#include "internal.h"

// Peer-memory exchange of the row-sharded solve: one buffer per rank (two flag-in-data work vectors,
// alternating by epoch), exported with CUDA IPC and mapped by every other rank of the node.
struct PeerExchange {
    bool tried = false, ok = false;
    uint64_t npad = 0;                 // elements per work vector
    unsigned char* local = nullptr;    // [256 B header][w0: npad x 2 uint4][w1: npad x 2 uint4]  (flag-in-data work vectors)
    unsigned char* base[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // every rank's buffer
    unsigned long long epoch = 0;      // last epoch published (identical on all ranks: collective call sequence)
    int* err_h = nullptr;              // mapped pinned int: a consumer kernel timed out waiting for a peer
};

// Ranks of ONE process (bemb200_multi_*): the exchange buffers are plain device pointers shared through this table instead
// of CUDA IPC handles; `exchange` is a reusable barrier that hands every rank the pointers of all ranks.
namespace bemb {
constexpr int MAX_GROUP_RANKS = 8;
struct PeerGroup {
    int nranks = 0;
    int device[MAX_GROUP_RANKS] = {0, 0, 0, 0, 0, 0, 0, 0};
    bool peer_ok = true;  // cudaDeviceEnablePeerAccess worked for every pair of distinct devices
    std::mutex mu;
    std::condition_variable cv;
    unsigned char* posted[MAX_GROUP_RANKS] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    unsigned char* snap[MAX_GROUP_RANKS] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    int arrived = 0;
    unsigned long long generation = 0;
    // every rank posts `mine` (may be NULL = "I failed"); returns false on a time-out (a rank never arrived)
    bool exchange(int rank, unsigned char* mine, unsigned char** all);
};
}  // namespace bemb

// Buffers of the persistent fused GMRES kernel (gmres_fused.cu) that stay local to the rank: the inbox of CTA
// partials, the broadcast slots and the result record.  The exchange vectors and the inbox of rank partials live in the
// PeerExchange allocation (they are written by other ranks).
struct FusedLocal {
    uint4* cpart = nullptr;
    uint4* hbuf = nullptr;
    void* result_h = nullptr;   // FusedResult, mapped pinned
    void* result_d = nullptr;   // device alias of result_h
    int grid = 0;               // CTAs the buffers were sized for
    uint32_t er = 0;            // last reduction-round epoch used
    bool disabled = false;      // a solve timed out: stay on the per-iteration kernels
    // row ownership weighted by the measured streaming speed of the SM under every CTA (see gmres_fused_solve)
    unsigned long long* trace_d = nullptr;  // [grid][4]
    uint32_t* row_off_d = nullptr;          // [grid + 1] CTA boundaries (rows, or (row, segment) units)
    uint4* frag = nullptr;                  // [2][grid] flag-in-data slots for boundary-row partial sums
    std::vector<double> speed;              // rows per ns of CTA c's SM (empty: not calibrated)
    std::vector<unsigned> smid;             // SM id CTA c ran on when `speed` was measured
    int calib_runs = 0;
};

struct bemb200_ctx {
    int device = 0;
    int rank = 0, nranks = 1;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    std::atomic<int> shared_gpu{0};  // != 0: another stream shares the GPU -> solver avoids whole-GPU cooperative kernels
    std::atomic<int> background_blocks_per_sm{0};  // > 0: assembly kernels use a small persistent grid (sweep pipelining)
    void* nccl_comm = nullptr;  // ncclComm_t when nranks > 1
    PeerExchange px;
    FusedLocal fx;
    std::shared_ptr<bemb::PeerGroup> group;  // set for the rank contexts of a bemb200_multi (one process, several devices)
    int fused_grid = 0;  // > 0: CTAs of the fused GMRES kernel (several ranks sharing one device); 0: one per SM
    std::string err;
    std::mutex mu;  // LinearOperator is Send + Sync: serialise stream submission per context
};

struct bemb200_staged_mesh {
    bemb200_ctx* ctx = nullptr;
    bemb::DeviceMesh dm;
    std::vector<void*> allocs;
    std::vector<int32_t> bc_type;  // host copy, DOF order: admittance is allowed on velocity-BC elements only
};

struct GmresWorkspace;  // gmres.cu

struct bemb200_matrix {
    bemb200_ctx* ctx = nullptr;
    uint64_t n_rows = 0, n_cols = 0;  // global shape
    uint64_t r0 = 0, r1 = 0;          // local rows
    bemb::cplx* A = nullptr;          // (r1-r0) x n_cols, row-major
    bemb::cplx* rhs = nullptr;        // r1-r0
    bemb::cplx* adm = nullptr;        // n_cols: admittance of the last assembly with options (allocated on first use)
    uint2* near_list = nullptr;
    unsigned int near_cap = 0;
    unsigned int* near_count = nullptr;
    bemb200_assembly_stats stats{};
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    GmresWorkspace* ws = nullptr;
    // background assembly that a second stream may join (bemb200_matrix_boost_assembly)
    unsigned int* work_counters = nullptr;  // 2 device counters (Tri3 / Quad4 far pass)
    std::mutex boost_mu;
    bool far_running = false;               // the far pass of an assembly into this matrix is in flight
    bool boost_pending = false;             // helper blocks were started: wait for boost_ev before using the far results
    bemb::FarRelaunch relaunch;
    cudaEvent_t far_ready_ev = nullptr, boost_ev = nullptr;
    // solver statistics of the last call
    uint64_t last_launches = 0, last_matvecs = 0;
    double last_matvec_ms = 0.0;
    double last_solve_ms = 0.0;  // fused kernel: CUDA-event duration of the one launch
};

namespace bemb {
int set_error(bemb200_ctx* ctx, int code, const std::string& msg);
int cuda_fail(bemb200_ctx* ctx, cudaError_t e, const char* what);
// BEMB200_OK, or the error (set on ctx) for options bemb200_assemble_staged_opts would refuse
int check_assembly_options(bemb200_ctx* ctx, const bemb200_staged_mesh* sm, const bemb200_assembly_options* opts);
void free_workspace(bemb200_matrix* m);
void free_peer_exchange(bemb200_ctx* ctx, bool collective);
// true when p is device (or managed) memory of `device` (postprocess.cu)
bool device_ptr_on(int device, const void* p);
// out[s n + i] = sys[i] + inc[s n + i] for s < nrhs (out may be inc) on stream s (postprocess.cu)
cudaError_t launch_add_system_rhs(const cplx* sys, const cplx* inc, uint64_t n, uint32_t nrhs, cplx* out, cudaStream_t s);
// TbemSystem.rhs of every row (local slices all-gathered; collective on a row-sharded operator) to `out`, a host
// (cudaMemcpyDeviceToHost) or device (cudaMemcpyDeviceToDevice) vector of num_rows complex128 (gmres.cu)
int rhs_full(bemb200_matrix* m, double* out, cudaMemcpyKind kind);
// bemb200_gmres (pc == NULL) / bemb200_gmres_schwarz with b already on the device: the same operations, only the copy of b
// into the workspace is device to device (gmres.cu)
int gmres_solve_device_b(bemb200_matrix* m, const bemb200_precond* pc, const double* b_dev, uint32_t max_iterations, uint32_t restart,
                         double tolerance, double* x_out, bemb200_gmres_info* info);
}  // namespace bemb

#define BEMB_CUDA(ctx, call)                                          \
    do {                                                              \
        cudaError_t _e = (call);                                      \
        if (_e != cudaSuccess) return bemb::cuda_fail(ctx, _e, #call); \
    } while (0)
