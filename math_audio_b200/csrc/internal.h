// Internal structures of libbemb200 shared between translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <functional>
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"

namespace bemb {

// Staged mesh: everything in DOF order (column j / row i of the matrix <-> the
// non-evaluation element whose dof_addresses[0] == j).  Frequency independent.
struct DeviceMesh {
    uint32_t n = 0;        // number of DOFs
    uint32_t ntiles = 0;   // ceil(n / TILE)
    double* coords = nullptr;    // [n][12]  gathered node coordinates (4th node zero for Tri3)
    uint8_t* etype = nullptr;    // [n]      3 | 4
    double* area = nullptr;      // [n]      Element.area (mesh supplied)
    double* src = nullptr;       // [n][8]   collocation point xyz, stored normal xyz, 2 pad
    int32_t* bc_type = nullptr;  // [n]
    uint8_t* bc_len = nullptr;   // [n]
    cplx* bc_val = nullptr;      // [n][4]
    uint8_t* nonzero_bc = nullptr;  // [n]   has_nonzero_bc (tbem.rs:247)
    double* esize = nullptr;     // [n]      estimate_element_size (singular.rs:730-745)
    double* far_k = nullptr;     // [ntiles][NQ_MAX][TILE]     kappa_q = |y_q - y_0|^2
    double* far_c = nullptr;     // [ntiles][FAR_NCONST][TILE] per-column constants
    uint8_t* col_class = nullptr;   // [ntiles*TILE]
    uint32_t* special_cols = nullptr;  // [n_special]
    uint32_t n_special = 0;
    uint32_t n_flat_tri = 0, n_flat_quad = 0;
    // flat velocity-BC columns with a NON-ZERO prescribed velocity: the matrix entry does not depend on the BC value, so they
    // stay in the far kernel; only their right-hand-side term (regular.rs:157-177) is added by rhs_far_kernel
    uint32_t* rhs_cols_tri = nullptr;   // [n_rhs_tri]
    uint32_t* rhs_cols_quad = nullptr;  // [n_rhs_quad]
    uint32_t n_rhs_tri = 0, n_rhs_quad = 0;
    double avg_radius_first100 = 0.0;  // mean |center| of the first <=100 ELEMENTS (tbem.rs:108-117)
};

struct Phys {
    double k;        // wave_number
    double wavruim;  // harmonic_factor * wave_number
    double k2;       // k*k
    double tau, gamma;
    double sign;     // dg_dn_sign (tbem.rs:118-123)
    cplx beta;       // coupling passed to build_tbem_system_with_beta
    cplx beta_unscaled;  // physics.burton_miller_beta() (types.rs:64-70), used inside integrators
    // admittance Y_j of velocity-BC column j (DOF order, device) or NULL: v_j = vbar_j + Y_j p_j moves
    // -Y_j (gamma tau G_ij + beta H^T_ij) into A[i,j] and -Y_i beta tau / 2 into A[i,i] (DESIGN.md 4.8)
    const cplx* adm;
};

struct AssemblyStats {
    unsigned long long near_pairs = 0;
    unsigned long long far_pairs = 0;      // pairs evaluated by the far kernel
    unsigned long long special_pairs = 0;  // pairs through the dense generic path
    unsigned int near_overflow = 0;
};

// launchers (assembly_exact.cu / assembly_far.cu)
cudaError_t launch_prep(const DeviceMesh& m, cudaStream_t s);
// work_counters (may be NULL): two pre-zeroed device counters (Tri3 / Quad4 pass); with them a background launch pulls its
// work items dynamically and `relaunch` receives one closure per pass that starts additional blocks on another stream
// pulling from the same counter ("boost": finish the assembly at full speed once the solver has left the GPU).
typedef std::vector<std::function<cudaError_t(cudaStream_t)>> FarRelaunch;
cudaError_t launch_far(const DeviceMesh& m, const Phys& ph, uint64_t row_begin, uint64_t row_end, cplx* A, uint64_t lda,
                       uint2* near_list, unsigned int near_cap, unsigned int* near_count, int background_blocks_per_sm,
                       unsigned int* work_counters, FarRelaunch* relaunch, cudaStream_t s);
// ph.adm != NULL launches the admittance instantiation of the far kernel (its Y = 0 columns keep the bits of the plain one)
// right-hand-side term of the un-subdivided (row, non-zero-velocity column) pairs; same near/far split as launch_far
cudaError_t launch_rhs_far(const DeviceMesh& m, const Phys& ph, uint64_t row_begin, uint64_t row_end, cplx* rhs, cudaStream_t s);
cudaError_t launch_near_list(const DeviceMesh& m, const Phys& ph, uint64_t row_begin, cplx* A, uint64_t lda, cplx* rhs,
                             const uint2* near_list, unsigned int count, cudaStream_t s);
cudaError_t launch_special(const DeviceMesh& m, const Phys& ph, uint64_t row_begin, uint64_t row_end, cplx* A,
                           uint64_t lda, cplx* rhs, cudaStream_t s);
cudaError_t launch_self(const DeviceMesh& m, const Phys& ph, uint64_t row_begin, uint64_t row_end, cplx* A, uint64_t lda,
                        cplx* rhs, cudaStream_t s);
int far_kernel_launch_count(const DeviceMesh& m);

}  // namespace bemb
