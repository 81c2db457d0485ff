/* bemb200.h -- C ABI of libbemb200: B200 (sm_100a) backend for the dense Helmholtz BEM
 * assemble + GMRES path of math-bem / math-solvers.
 *
 * Every entry point below is what a Rust `extern "C"` block (or cgo / ctypes) binds;
 * each one names the reference interface it replaces (paths relative to the
 * reference repository).  Conventions:
 *   - plain pointers and sizes only; complex numbers are interleaved (re, im) doubles,
 *     layout-identical to num_complex::Complex64 and cuDoubleComplex;
 *   - inputs are COPIED during the call, no pointer is retained after return;
 *   - every function returns 0 on success or a negative BEMB200_E* code and never
 *     throws/aborts; bemb200_last_error() gives the message of the last failure;
 *   - handles are opaque and owned by the library; free them with the matching call;
 *   - there is no CPU fallback: without a CUDA device every compute call fails with
 *     BEMB200_ENODEVICE.
 */
#ifndef BEMB200_H
#define BEMB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BEMB200_OK 0
#define BEMB200_EINVAL (-1)     /* bad argument / shape mismatch (the reference panics) */
#define BEMB200_ENODEVICE (-2)  /* no usable CUDA device */
#define BEMB200_ECUDA (-3)      /* CUDA runtime error, see bemb200_last_error */
#define BEMB200_ENOMEM (-4)     /* device or host allocation failed */
#define BEMB200_ENCCL (-5)      /* NCCL error / NCCL not loadable */
#define BEMB200_EUNSUPPORTED (-6)
#define BEMB200_ESINGULAR (-7)   /* LuError::SingularMatrix (math-solvers/src/direct/lu.rs:15-21) */
#define BEMB200_ECALLBACK (-8)   /* a caller-supplied function (bemb200_precond_fn) reported failure */

typedef struct bemb200_ctx bemb200_ctx;
typedef struct bemb200_staged_mesh bemb200_staged_mesh;
typedef struct bemb200_matrix bemb200_matrix;

/* SoA view of `&[Element]` + `nodes: Array2<f64>` (math-bem/src/core/types.rs:329-351,
 * 371-373).  One DOF per non-evaluation element (types.rs:359-363). */
typedef struct bemb200_mesh {
    uint64_t n_nodes;
    uint64_t n_elem;
    const double* nodes;      /* [n_nodes*3]  Mesh.nodes, row-major                         */
    const uint32_t* conn;     /* [n_elem*4]   Element.connectivity, Tri3 padded 0xFFFFFFFF  */
    const uint8_t* etype;     /* [n_elem]     3 = Tri3, 4 = Quad4 (Element.element_type)     */
    const double* center;     /* [n_elem*3]   Element.center  (collocation point)           */
    const double* normal;     /* [n_elem*3]   Element.normal  (n_x; may be flipped outward) */
    const double* area;       /* [n_elem]     Element.area    (drives the subdivision test) */
    const int32_t* bc_type;   /* [n_elem]     get_bc_type_and_value(): 0 velocity, 1 pressure, 2 transfer (tbem.rs:234-244) */
    const uint8_t* bc_len;    /* [n_elem]     number of per-node BC values supplied (1..4)  */
    const double* bc_val;     /* [n_elem*4*2] per-node complex BC values                     */
    const uint32_t* dof;      /* [n_elem]     Element.dof_addresses[0]                       */
    const uint8_t* is_eval;   /* [n_elem]     ElementProperty::Evaluation (skipped)          */
} bemb200_mesh;

/* PhysicsParams (types.rs:16-58, 216-218) -- the four fields the path reads. */
typedef struct bemb200_physics {
    double wave_number;
    double harmonic_factor; /* +1 => exp(+ikr) */
    double tau;             /* +1 exterior, -1 interior */
    double gamma;           /* 1.0 */
} bemb200_physics;

/* GmresSolution minus x (math-solvers/src/iterative/gmres.rs:74-85). */
typedef struct bemb200_gmres_info {
    uint64_t iterations; /* Arnoldi matvecs (gmres.rs:178) */
    uint64_t restarts;
    double residual;     /* relative to ||b|| */
    int32_t converged;
} bemb200_gmres_info;

typedef struct bemb200_assembly_stats {
    uint64_t near_pairs;    /* pairs re-integrated with adaptive subdivision */
    uint64_t special_pairs; /* pairs through the generic path (pressure BC, non-zero BC, warped Quad4) */
    uint64_t far_kernel_launches;
    uint64_t total_launches;
    double far_ms;   /* device time of the far-field kernel(s), CUDA events */
    double total_ms; /* device time of the whole assembly */
} bemb200_assembly_stats;

/* ---- context -------------------------------------------------------------------- */
int bemb200_device_count(void);
/* single-GPU context on `device` */
int bemb200_ctx_create(int device, bemb200_ctx** out);
/* one rank of a row-sharded job: one process per GPU; `nccl_id` is the 128-byte
 * ncclUniqueId produced by bemb200_nccl_unique_id() on rank 0 and distributed by the
 * host program (MPI, torch.distributed, a file ...). */
int bemb200_nccl_unique_id(uint8_t out[128]);
int bemb200_ctx_create_dist(int device, int rank, int nranks, const uint8_t nccl_id[128], bemb200_ctx** out);
/* general form: `cuda_stream` (a cudaStream_t, may be NULL) makes the library submit all its
 * work to a stream owned by the caller, so that the caller's CUDA events bracket it;
 * nranks == 1 ignores nccl_id; nranks > 1 with nccl_id == NULL creates a context WITHOUT a
 * communicator (assembly only: row-block assembly needs no communication). */
int bemb200_ctx_create_ex(int device, int rank, int nranks, const uint8_t* nccl_id, void* cuda_stream, bemb200_ctx** out);
void bemb200_ctx_destroy(bemb200_ctx* ctx);
/* blocks_per_sm > 0 turns the FP64 assembly kernel of this context into a "background" kernel: a
 * persistent grid of 148*blocks_per_sm blocks that leaves registers/shared memory to kernels of
 * other streams (assembly of frequency f+1 underneath the solve of frequency f); 0 = normal. */
int bemb200_ctx_set_background(bemb200_ctx* ctx, int blocks_per_sm);
/* shared != 0 tells the SOLVER of this context that kernels of other streams run beside it (the
 * background assembly above): the Gram-Schmidt step then uses its 16-CTA cluster kernel instead
 * of the whole-GPU cooperative kernel, whose grid barriers stall behind foreign warps. */
int bemb200_ctx_set_shared_gpu(bemb200_ctx* ctx, int shared);
/* While an assembly into `m` runs as a background grid on another context/stream (another thread is
 * inside bemb200_assemble_staged), start additional far-kernel blocks on `ctx`'s stream that pull
 * work items from the same counter: the assembly then finishes at full speed.  Meant for the
 * moment the solver of a pipelined sweep has finished and the GPU would otherwise idle behind the
 * polite background grid.  No-op when nothing is in flight. */
int bemb200_matrix_boost_assembly(bemb200_matrix* m, bemb200_ctx* ctx);
/* Row-sharded solves (nranks > 1): *active = 1 once the ranks have mapped each other's work
 * vectors (CUDA IPC over NVLink) and the Arnoldi matvec stores its slab of A v straight into
 * every rank's memory from the ZGEMV epilogue -- no all-gather kernel; 0 = NCCL all-gather
 * (before the first solve, when the platform refuses peer mappings, or BEMB200_PEER_FUSED=0). */
int bemb200_ctx_peer_exchange_active(const bemb200_ctx* ctx, int* active);
/* Hand a matrix to another context of the SAME device (e.g. a solve context with its own stream
 * while an assembly context fills the next matrix of a frequency sweep).  The caller orders the
 * use of one matrix by the two contexts. */
int bemb200_matrix_set_context(bemb200_matrix* m, bemb200_ctx* ctx);
const char* bemb200_last_error(const bemb200_ctx* ctx); /* ctx may be NULL: last global error */
/* canonical row partition used by the distributed solver: rank r owns
 * [r*ceil(n/nranks), min(n,(r+1)*ceil(n/nranks))) */
void bemb200_partition(uint64_t n, int nranks, int rank, uint64_t* row_begin, uint64_t* row_end);

/* ---- assembly: replaces build_tbem_system_with_beta (assembly/tbem.rs:96-222) ------ */
/* Frequency-independent staging (gather to DOF order, quadrature points, ratio-test
 * data); reuse across a frequency sweep. */
int bemb200_mesh_stage(bemb200_ctx* ctx, const bemb200_mesh* mesh, bemb200_staged_mesh** out);
void bemb200_staged_mesh_free(bemb200_staged_mesh* sm);
uint64_t bemb200_staged_num_dofs(const bemb200_staged_mesh* sm);
/* Assemble matrix rows [row_begin,row_end) (all columns) and the matching rhs entries.
 * If *inout is NULL a matrix is allocated, otherwise the handle is reused (same shape
 * required). */
int bemb200_assemble_staged(bemb200_ctx* ctx, const bemb200_staged_mesh* sm, const bemb200_physics* phys, double beta_re,
                            double beta_im, uint64_t row_begin, uint64_t row_end, bemb200_matrix** inout);
/* stage + assemble in one call (the drop-in for one build_tbem_system_with_beta call) */
int bemb200_assemble(bemb200_ctx* ctx, const bemb200_mesh* mesh, const bemb200_physics* phys, double beta_re,
                     double beta_im, uint64_t row_begin, uint64_t row_end, bemb200_matrix** out);
int bemb200_assembly_stats_get(const bemb200_matrix* m, bemb200_assembly_stats* out);
/* dg_dn_sign heuristic of tbem.rs:108-123 for this mesh and wave number */
double bemb200_dg_dn_sign(const bemb200_staged_mesh* sm, double wave_number);

/* Options of one assembly (DESIGN.md 4.8); all zero / NULL is bemb200_assemble_staged.
 *   dg_dn_sign       0: the heuristic above (the reference's); +1 / -1: that sign at every frequency.  The sign-consistent
 *                    formulation (+1 with consistent_beta = 1) converges to the exact solution at every ka.
 *   consistent_beta  0: the prescribed-velocity right-hand-side integrals use the unscaled beta = i/k (the reference's);
 *                    1: they use the beta passed to the assembly, as the free term does.
 *   admittance       NULL, or num_dofs complex128 in DOF order: the admittance Y_j (1/m, constant over the element) of an
 *                    absorbing velocity-BC element, v_j = vbar_j + Y_j p_j with v = dp/dn_y.  Passive surfaces have
 *                    Im Y <= 0 for harmonic_factor = +1.  A non-zero Y on a pressure or transfer element is BEMB200_EINVAL. */
typedef struct bemb200_assembly_options {
    int32_t dg_dn_sign;
    int32_t consistent_beta;
    const double* admittance;
} bemb200_assembly_options;
/* bemb200_assemble_staged with options (NULL: the same call); row-sharded ranks as there */
int bemb200_assemble_staged_opts(bemb200_ctx* ctx, const bemb200_staged_mesh* sm, const bemb200_physics* phys, double beta_re,
                                 double beta_im, const bemb200_assembly_options* opts, uint64_t row_begin, uint64_t row_end,
                                 bemb200_matrix** inout);

/* ---- matrix handle: TbemSystem (tbem.rs:13-31) / DenseOperator (solver/fmm_interface.rs:25-52) */
/* wrap an existing host matrix: DenseOperator::new(Array2) -- rows [row_begin,row_end) of an n x n_cols matrix */
int bemb200_matrix_from_host(bemb200_ctx* ctx, const double* a_rows, uint64_t n_rows_global, uint64_t n_cols,
                             uint64_t row_begin, uint64_t row_end, bemb200_matrix** out);
void bemb200_matrix_free(bemb200_matrix* m);
uint64_t bemb200_num_rows(const bemb200_matrix* m);   /* LinearOperator::num_rows (global) */
uint64_t bemb200_num_cols(const bemb200_matrix* m);   /* LinearOperator::num_cols */
uint64_t bemb200_local_row_begin(const bemb200_matrix* m);
uint64_t bemb200_local_row_end(const bemb200_matrix* m);
/* copy local rows [row_begin,row_end) (must lie inside the local slab) to the host */
int bemb200_matrix_download(const bemb200_matrix* m, uint64_t row_begin, uint64_t row_end, double* out);
/* rhs entries of the local rows (TbemSystem.rhs) */
int bemb200_rhs_download(const bemb200_matrix* m, double* out);
/* the full rhs vector (num_rows entries) on every rank: local slices all-gathered */
int bemb200_rhs_download_full(const bemb200_matrix* m, double* out);
/* apply_row_sum_correction (tbem.rs:500-520); returns |sum of all row sums| / n in *avg */
int bemb200_row_sum_correction(bemb200_matrix* m, double* avg);

/* LinearOperator::apply / apply_transpose (math-solvers/src/traits.rs:316-364):
 * x has num_cols entries, y has num_rows entries (all ranks receive the full y). */
int bemb200_apply(const bemb200_matrix* m, const double* x, double* y);
int bemb200_apply_transpose(const bemb200_matrix* m, const double* x, double* y);
/* same with DEVICE pointers (x: num_cols, y: num_rows complex128), asynchronous on the
 * context stream followed by a stream synchronise */
int bemb200_apply_device(const bemb200_matrix* m, const double* x_dev, double* y_dev);

/* gmres / gmres_with_guess (math-solvers/src/iterative/gmres.rs:96-277): restarted
 * GMRES(m), modified Gram-Schmidt, complex Givens; `max_iterations` counts restart
 * cycles, info->iterations counts Arnoldi matvecs; residual is relative to ||b||;
 * ||b|| < 1e-15 returns x0 at once; breakdown threshold 1e-14.  b, x0 (may be NULL),
 * x_out: num_rows complex128 on the HOST. */
int bemb200_gmres(const bemb200_matrix* m, const double* b, const double* x0, uint32_t max_iterations, uint32_t restart,
                  double tolerance, double* x_out, bemb200_gmres_info* info);
/* gmres_preconditioned / gmres_preconditioned_with_guess (gmres.rs:282-585): LEFT preconditioning,
 * residual relative to ||M^-1 b||.  The preconditioners of the reference that make sense for a
 * dense operator at scale are built in: inv_diag == NULL is IdentityPreconditioner
 * (traits.rs:377-385); otherwise inv_diag (num_rows complex128, host) is the inverse diagonal of
 * DiagonalPreconditioner (math-solvers/src/preconditioners/diagonal.rs:20-58). */
int bemb200_gmres_preconditioned(const bemb200_matrix* m, const double* inv_diag, const double* b, const double* x0,
                                 uint32_t max_iterations, uint32_t restart, double tolerance, double* x_out,
                                 bemb200_gmres_info* info);
/* diagonal of the (square) matrix, all ranks receive all num_rows entries */
int bemb200_matrix_diagonal(const bemb200_matrix* m, double* out);
/* Block-Jacobi / additive Schwarz preconditioner built on the device from the assembled operator:
 * AdditiveSchwarzPreconditioner::from_csr(matrix, num_subdomains, overlap)
 * (math-solvers/src/preconditioners/schwarz.rs:66-125) with the local solve of schwarz.rs:252-380 -- ILU(0) of the
 * extracted block, which for the dense block of a BEM operator is LU without pivoting, then forward / backward
 * substitution -- and the weighted combination of schwarz.rs:399-417.
 *   sub_ptr == NULL: the reference's contiguous partition into num_subdomains blocks (overlap 0, i.e. block-Jacobi on the
 *                    diagonal blocks: the near field of consecutive DOF clusters, cf. compute_near_block,
 *                    math-bem/src/core/assembly/slfmm.rs:538-608);
 *   otherwise subdomain k holds the global DOF indices sub_idx[sub_ptr[k] .. sub_ptr[k+1]) in the order that becomes its
 *   local numbering (the reference keeps them ascending, schwarz.rs:199-202); sets may overlap (weights 1 / multiplicity).
 * A subdomain holds at most 4096 unknowns.  On a row-sharded operator every rank passes the same subdomains and each must
 * lie inside one rank's row block (BEMB200_EINVAL otherwise): M^-1 then acts on a rank's slab without communication.
 * The handle is independent of the matrix after creation (it stores the inverse blocks) but, like a matrix handle, belongs to
 * the matrix's context: free it before bemb200_ctx_destroy (its device memory returns to the context's stream-ordered pool). */
typedef struct bemb200_precond bemb200_precond;
typedef struct bemb200_precond_stats {
    uint32_t num_subdomains;   /* stats() of schwarz.rs:135-158: count, min / max / average size */
    uint32_t local_subdomains; /* owned by this rank */
    uint32_t min_size, max_size;
    double avg_size;
    uint64_t inverse_bytes;    /* bytes one application streams on this rank */
    double factor_ms;          /* device time of gather + factorisation + inversion */
    int32_t disjoint;          /* 1: every local row in exactly one subdomain (block-Jacobi) */
} bemb200_precond_stats;
int bemb200_schwarz_create(const bemb200_matrix* m, uint32_t num_subdomains, const uint64_t* sub_ptr, const uint64_t* sub_idx,
                           bemb200_precond** out);
void bemb200_precond_free(bemb200_precond* p);
int bemb200_precond_stats_get(const bemb200_precond* p, bemb200_precond_stats* out);
/* Preconditioner::apply (math-solvers/src/traits.rs:366-371): z = M^-1 r, num_rows complex128 on the HOST (collective on a
 * row-sharded operator; every rank receives the whole z) */
int bemb200_precond_apply(const bemb200_precond* p, const double* r, double* z);
/* gmres_preconditioned_with_guess (gmres.rs:434-585) with that preconditioner: per Arnoldi step the ZGEMV, the block
 * solve on the rank's slab, the exchange, one Gram-Schmidt kernel.  Arguments as bemb200_gmres_preconditioned. */
int bemb200_gmres_schwarz(const bemb200_matrix* m, const bemb200_precond* precond, const double* b, const double* x0,
                          uint32_t max_iterations, uint32_t restart, double tolerance, double* x_out, bemb200_gmres_info* info);
/* gmres_preconditioned_with_guess (gmres.rs:434-585) with ANY implementation of the reference's `Preconditioner` trait
 * (math-solvers/src/traits.rs:366-371: `fn apply(&self, r: &Array1<T>) -> Array1<T>`) -- ILU, AMG, hierarchical, a caller's own.
 * `apply(user, r, z, n)` must write z = M^-1 r (n complex128, interleaved, HOST memory owned by the library for the duration
 * of the call) and return 0; any other value ends the solve with BEMB200_ECALLBACK.  The Arnoldi process (ZGEMV, Gram-Schmidt,
 * update) stays on the device; one vector goes down and one comes up per application.  `apply` is called exactly where the
 * reference calls `precond.apply`: once for M^-1 b, once per restart cycle for M^-1 (b - A x), once per Arnoldi step for
 * M^-1 (A v_j) (`*precond_calls`, may be NULL, returns the count).  It runs on the calling thread with the context's lock
 * held: it must not call into the same context.  Single-rank operators only (BEMB200_EUNSUPPORTED otherwise): the trait acts
 * on whole vectors.  Other arguments as bemb200_gmres_preconditioned. */
typedef int (*bemb200_precond_fn)(void* user, const double* r, double* z, uint64_t n);
int bemb200_gmres_callback(const bemb200_matrix* m, bemb200_precond_fn apply, void* user, const double* b, const double* x0,
                           uint32_t max_iterations, uint32_t restart, double tolerance, double* x_out, bemb200_gmres_info* info,
                           uint64_t* precond_calls);
/* same with DEVICE pointers (b_dev, x0_dev or NULL, x_dev) */
int bemb200_gmres_device(const bemb200_matrix* m, const double* b_dev, const double* x0_dev, uint32_t max_iterations,
                         uint32_t restart, double tolerance, double* x_dev, bemb200_gmres_info* info);
/* lu_solve (math-solvers/src/direct/lu.rs:136-161; LAPACK zgesv in the reference's native build),
 * the SolverMethod::Direct branch of BemSolver::solve_dense_system (bem_solver.rs:435-441): LU
 * with partial pivoting + two triangular solves through cuSOLVER (zgetrf / zgetrs, loaded at run
 * time).  Needs the whole matrix on one GPU.  overwrite_matrix = 0 factors a copy (the reference
 * borrows `a`), 1 factors in place (the handle then holds L\U).  factor_ms (may be NULL): device
 * time of the factorisation.  BEMB200_ESINGULAR = LuError::SingularMatrix. */
int bemb200_lu_solve(const bemb200_matrix* m, const double* b, double* x_out, int overwrite_matrix, double* factor_ms);
/* bicgstab (math-solvers/src/iterative/bicgstab.rs:46-187), the iterative solver of
 * BemSolver::solve_dense_system (bem_solver.rs:435-463): x0 = 0, two operator applications per
 * iteration, breakdown thresholds 1e-30, early exit on ||s||/||b|| < tol.  info->restarts = 0;
 * `converged` false on breakdown / stagnation / exhausted budget (the reference never errors). */
int bemb200_bicgstab(const bemb200_matrix* m, const double* b, uint32_t max_iterations, double tolerance, double* x_out,
                     bemb200_gmres_info* info);
/* cgs (math-solvers/src/iterative/cgs.rs:46-155), reached through solve_cgs / solve_with_ilu /
 * solve_tbem_with_ilu (math-bem/src/core/solver/fmm_interface.rs:360-366,389-447; the "ILU"
 * variants run this unpreconditioned solver on the dense TBEM matrix): x0 = 0, two operator
 * applications per iteration, breakdown thresholds 1e-30 (sigma, and the previous rho as in
 * cgs.rs:122).  info->restarts = 0; `converged` false on breakdown / exhausted budget. */
int bemb200_cgs(const bemb200_matrix* m, const double* b, uint32_t max_iterations, double tolerance, double* x_out,
                bemb200_gmres_info* info);
/* Multi-RHS solve (BASELINE config 5): `nrhs` (<= 32) independent gmres() solves -- the reference
 * would loop `gmres(operator, b_s, config)` over the right-hand sides -- advanced in lockstep so
 * that they share ONE FP64 tensor-core block matvec per iteration (A is streamed once for all
 * right-hand sides).  Per-RHS semantics (iterations, restarts, residual, converged) are exactly
 * those of the single-RHS call.  b_all / x_all: nrhs vectors of num_rows complex128, each
 * contiguous; infos[nrhs].  block_matvec_ms / block_matvecs (may be NULL): device time and count
 * of the block matvec kernel. */
int bemb200_gmres_batched(const bemb200_matrix* m, const double* b_all, uint32_t nrhs, uint32_t max_iterations,
                          uint32_t restart, double tolerance, double* x_all, bemb200_gmres_info* infos,
                          double* block_matvec_ms, uint64_t* block_matvecs);
/* The same with nrhs independent gmres_preconditioned() solves (gmres.rs:282) sharing the block-Jacobi preconditioner of
 * bemb200_schwarz_create (disjoint subdomains covering every row; BEMB200_EUNSUPPORTED for overlapping ones). */
int bemb200_gmres_batched_schwarz(const bemb200_matrix* m, const bemb200_precond* precond, const double* b_all, uint32_t nrhs,
                                  uint32_t max_iterations, uint32_t restart, double tolerance, double* x_all,
                                  bemb200_gmres_info* infos, double* block_matvec_ms, uint64_t* block_matvecs);
/* bemb200_gmres_batched (precond == NULL) / bemb200_gmres_batched_schwarz with DEVICE vectors: b_dev and x_dev are nrhs
 * vectors of num_rows complex128, each contiguous, in memory of the matrix's device (BEMB200_EINVAL otherwise).  Same
 * limits and the same results; B is interleaved straight from b_dev and X written straight to x_dev. */
int bemb200_gmres_batched_device(const bemb200_matrix* m, const bemb200_precond* precond, const double* b_dev, uint32_t nrhs,
                                 uint32_t max_iterations, uint32_t restart, double tolerance, double* x_dev,
                                 bemb200_gmres_info* infos, double* block_matvec_ms, uint64_t* block_matvecs);
/* Y = A X for nrhs (<= 32) vectors at once with the tensor-core block kernel; kernel_ms (may be
 * NULL) receives the device time of one block matvec.  Row-sharded operators: collective, every rank multiplies its row
 * block and receives the whole Y.  (bemb200_gmres_batched: up to 196 608 unknowns, also row-sharded.) */
int bemb200_apply_block(const bemb200_matrix* m, const double* x_all, uint32_t nrhs, double* y_all, double* kernel_ms);
/* number of kernels launched and device milliseconds spent inside the zgemv kernel by
 * the last bemb200_gmres* / bemb200_apply* call on this matrix */
int bemb200_solver_stats(const bemb200_matrix* m, uint64_t* kernel_launches, double* matvec_ms, uint64_t* matvecs);

/* ---- neighbours of the hot path (device-resident sweep): incident RHS and field evaluation ---- */
/* IncidentField::compute_rhs_with_beta (math-bem/src/core/incident.rs:317-342) at the collocation
 * points / normals of the staged mesh, in DOF order: rhs_i = -(gamma p_inc + beta tau dp_inc/dn),
 * summed over n_sources sources (MultiplePlaneWaves / MultiplePointSources, incident.rs:136-165).
 * kinds[s]: 0 plane wave (vecs[3s..] = unit direction), 1 point source (vecs = position);
 * amps[2s..] complex amplitude / strength.  Result to rhs_host and/or rhs_dev (either may be NULL). */
int bemb200_incident_rhs(const bemb200_staged_mesh* sm, const bemb200_physics* phys, double beta_re, double beta_im,
                         uint32_t n_sources, const int32_t* kinds, const double* vecs, const double* amps, double* rhs_host,
                         double* rhs_dev);
/* compute_scattered_field (math-bem/src/core/postprocess/pressure.rs:81-259): 7-point rule per
 * element (Quad4 = its first triangle, as the reference).  eval_pts [n_eval*3]; surface_pressure /
 * surface_velocity (may be NULL): num_dofs complex128 in DOF order; out [n_eval] complex128. */
int bemb200_scattered_field(const bemb200_staged_mesh* sm, const bemb200_physics* phys, uint64_t n_eval, const double* eval_pts,
                            const double* surface_pressure, const double* surface_velocity, double* out);
/* compute_rcs (math-bem/src/core/postprocess/pressure.rs:438-478) for n_dirs unit directions
 * dirs[3*n_dirs]: F(d) = sum_j p_j exp(-i k c_j.d) A_j (i k)(n_j.d) with Element.center / normal /
 * area as staged, rcs_out[d] = 4 pi |F(d)|^2.  surface_pressure: num_dofs complex128 in DOF order
 * (the reference indexes it by boundary-element enumeration, identical for sequential dof maps). */
int bemb200_compute_rcs(const bemb200_staged_mesh* sm, const bemb200_physics* phys, uint32_t n_dirs, const double* dirs,
                        const double* surface_pressure, double* rcs_out);
/* ---- several right-hand sides / solutions of one mesh (plane waves from many directions, point sources) ----------------
 * Block layout: nrhs (or nsol) vectors of num_dofs complex128, each contiguous, in DOF order (that of bemb200_gmres_batched).
 * Device arrays belong to the staged mesh's device (BEMB200_EINVAL otherwise).  Row s of every result has the bits of the
 * single-vector call on vector s. */
/* nrhs (1..4096) calls of bemb200_incident_rhs: right-hand side s sums the sources [src_ptr[s], src_ptr[s+1]) (src_ptr[0] = 0,
 * non-decreasing, src_ptr[nrhs] <= 65536 sources in all; kinds / vecs / amps as there).  system != NULL (a matrix of the staged
 * mesh's device) adds TbemSystem.rhs -- b = TbemSystem.rhs + incident, the b of bemb200_sweep_next; on a row-sharded operator
 * the rhs is gathered as bemb200_rhs_download_full gathers it, so the call is collective.  Result [nrhs * num_dofs] to b_host
 * and/or b_dev (either may be NULL). */
int bemb200_incident_rhs_batch(const bemb200_staged_mesh* sm, const bemb200_physics* phys, double beta_re, double beta_im,
                               uint32_t nrhs, const uint32_t* src_ptr, const int32_t* kinds, const double* vecs, const double* amps,
                               const bemb200_matrix* system, double* b_host, double* b_dev);
/* bemb200_compute_rcs for nsol (1..4096) surface solutions at once (on_device = 0: host array, 1: device array);
 * rcs_out [nsol * n_dirs] (host), solution-major. */
int bemb200_compute_rcs_batch(const bemb200_staged_mesh* sm, const bemb200_physics* phys, uint32_t nsol,
                              const double* surface_pressure, int on_device, uint32_t n_dirs, const double* dirs,
                              double* rcs_out);
/* bemb200_scattered_field for nsol (1..4096) surface solutions at once (surface_velocity may be NULL; on_device as above);
 * out [nsol * n_eval] complex128 (host), solution-major. */
int bemb200_scattered_field_batch(const bemb200_staged_mesh* sm, const bemb200_physics* phys, uint32_t nsol,
                                  const double* surface_pressure, const double* surface_velocity, int on_device,
                                  uint64_t n_eval, const double* eval_pts, double* out);
/* Complex far-field amplitude F(d) of nsol (1..4096) surface solutions in n_dirs (>= 1) unit directions dirs[3*n_dirs]
 * (finite, | |d| - 1 | <= 1e-9), defined by p_scat(R d) = F(d) exp(i s k R) / R + O(1/R^2) with s = harmonic_factor:
 *   F(d) = 1/(4 pi) sum_j [-i s k (d.n_j) p_j - v_j] int_{E_j} exp(-i s k d.y) dS_y
 * from the representation of bemb200_scattered_field (v = dp/dn), over the whole element: Tri3 with the field kernel's
 * 7-point rule, Quad4 with 3 x 3 Gauss-Legendre on the bilinear map (its Jacobian, and its normal at each point).
 * surface_pressure / surface_velocity (may be NULL: v = 0): [nsol * num_dofs] complex128 in DOF order, host (on_device = 0)
 * or device memory of the staged mesh's device (on_device = 1).  out [nsol * n_dirs] complex128 (host), solution-major.
 * Row s has the bits of the nsol = 1 call on solution s, for host and device input alike.  Bad arguments return
 * BEMB200_EINVAL before the staged mesh or a device is touched. */
int bemb200_far_field(const bemb200_staged_mesh* sm, const bemb200_physics* phys, uint32_t nsol, const double* surface_pressure,
                      const double* surface_velocity, int on_device, uint32_t n_dirs, const double* dirs, double* out);
/* Accurate scattered (or radiated) pressure of nsol (1..4096) surface solutions at n_eval (1..2^31-1) points
 * eval_pts[3*n_eval] (finite), from the representation of bemb200_scattered_field over the whole element:
 *   p_sc(x) = sum_j p_j int_{E_j} dG/dn_y dS - v_j int_{E_j} G dS,  G = exp(i s k r) / (4 pi r),  v = dp/dn
 * Tri3: the flat triangle; Quad4: the bilinear element (its Jacobian and its normal at each point), so far_field is the
 * R -> infinity limit of this field on both element types.  Pairs with |x - c_j| >= 4 rho_j (c_j node mean, rho_j largest
 * centroid-to-node distance) take the far-field rules (Tri3 7 points, Quad4 3 x 3 Gauss); nearer pairs are subdivided in the
 * element's parameter domain until every piece is at least 3 sqrt(piece area) from x (TR13 / 4 x 4 Gauss per piece), with no
 * cap short of depth 30.  A point within about 2^-30 element sizes of the surface (on it, in particular) gets NaN for every
 * solution; the other points of the call are not affected.  At points where every pair is regular on a Tri3 mesh the result
 * is bemb200_scattered_field's up to summation order.
 * surface_pressure / surface_velocity (may be NULL: v = 0): [nsol * num_dofs] complex128 in DOF order, host (on_device = 0)
 * or device memory of the staged mesh's device (on_device = 1).  out [nsol * n_eval] complex128 (host), solution-major.
 * Row s has the bits of the nsol = 1 call on solution s, for host and device input alike.  Bad arguments return
 * BEMB200_EINVAL before the staged mesh or a device is touched. */
int bemb200_evaluate_field(const bemb200_staged_mesh* sm, const bemb200_physics* phys, uint32_t nsol, const double* surface_pressure,
                           const double* surface_velocity, int on_device, uint64_t n_eval, const double* eval_pts, double* out);

/* ---- room-acoustics dense path (SURVEY 8f rank 3): math-bem/src/room_acoustics/solver.rs -------
 * Point collocation on a RoomMesh (math-xem-common/src/types.rs:185-192): nodes [n_nodes*3],
 * conn [n_elem*4] node indices (triangles: conn[4e+3] = 0xFFFFFFFF).  Staging computes
 * element_center_and_normal / element_area (solver.rs:38-122) on the device, once per mesh. */
typedef struct bemb200_room_mesh bemb200_room_mesh;
int bemb200_room_mesh_stage(bemb200_ctx* ctx, const double* nodes, uint64_t n_nodes, const uint32_t* conn, uint64_t n_elem,
                            bemb200_room_mesh** out);
void bemb200_room_mesh_free(bemb200_room_mesh* rm);
uint64_t bemb200_room_mesh_num_elements(const bemb200_room_mesh* rm);
/* staged element data back to the host (any pointer may be NULL): center[3n], normal[3n], area[n] */
int bemb200_room_mesh_geometry(const bemb200_room_mesh* rm, double* center, double* normal, double* area);
/* build_bem_matrix_parallel (solver.rs:448-493): rows [row_begin, row_end) of
 * A[i,j] = dG/dn(|c_i - c_j|, k, (c_i - c_j).n_i / r) area_j, A[j,j] = (0, -k/2pi) area_j, into a
 * bemb200_matrix handle (NULL *inout: allocate; else reuse) that bemb200_apply / bemb200_gmres accept
 * (solve_bem_system, solver.rs:412-445 = gmres(100 cycles, restart 50, tol 1e-6) on it).
 * kernel_ms (may be NULL): device time of the assembly kernel. */
int bemb200_room_assemble(bemb200_ctx* ctx, const bemb200_room_mesh* rm, double k, uint64_t row_begin, uint64_t row_end,
                          bemb200_matrix** inout, double* kernel_ms);
/* Source (math-xem-common/src/source.rs:160-219) as the device needs it: amplitude already
 * multiplied by crossover.amplitude_at_frequency(f); directivity = DirectivityPattern.magnitude,
 * row-major [n_vertical][n_horizontal], sampled every 10 degrees, or NULL for omnidirectional. */
typedef struct bemb200_room_source {
    double position[3];
    double amplitude;
    const double* directivity;
    uint32_t n_horizontal, n_vertical;
} bemb200_room_source;
/* calculate_incident_field_derivative_parallel (solver.rs:638-679):
 * rhs_i = - sum_s dG/dn(|c_i - x_s|, k, (c_i - x_s).n_i / r) amplitude_towards_s(c_i).
 * Result (num_elements complex128) to rhs_host and/or rhs_dev (either may be NULL). */
int bemb200_room_incident_rhs(const bemb200_room_mesh* rm, double k, uint32_t n_sources, const bemb200_room_source* sources,
                              double* rhs_host, double* rhs_dev);
/* calculate_field_pressure_bem_parallel (solver.rs:687-748) at points [n_points*3]:
 * out_p = sum_s G(|x - x_s|) amplitude_towards_s(x) + sum_j dG/dn(|x - c_j|, k, (x - c_j).n_j / r) p_j area_j */
int bemb200_room_field_pressure(const bemb200_room_mesh* rm, double k, uint32_t n_sources, const bemb200_room_source* sources,
                                uint64_t n_points, const double* points, const double* surface_pressure, double* out);

/* ---- pipelined frequency sweep (reference shape: math-bem/examples/audio_frequency_sweep.rs; the per-frequency body of
 * BemSolver::solve, math-bem/src/core/bem_solver.rs:273-322) ------------------------------------------------------------
 * The mesh is staged once; with overlap != 0 the FP64 assembly of frequency f+1 runs as a polite background grid
 * (background_blocks_per_sm persistent blocks per SM, 0 = default 1) on a second stream / matrix buffer underneath the
 * HBM-bound solve of frequency f, and is joined by full-speed helper blocks when the solve ends first.  Every frequency
 * is still exactly build_tbem_system_with_beta + gmres.  submit() queues a frequency (any number may be queued; two
 * matrix buffers exist), next() blocks until the OLDEST queued frequency is solved.  One rank of a row-sharded job:
 * rank / nranks / nccl_id as for bemb200_ctx_create_ex (every rank submits the same sequence). */
typedef struct bemb200_sweep bemb200_sweep;
int bemb200_sweep_create(int device, int rank, int nranks, const uint8_t* nccl_id, const bemb200_mesh* mesh, int overlap,
                         int background_blocks_per_sm, bemb200_sweep** out);
uint64_t bemb200_sweep_num_dofs(const bemb200_sweep* sw);
/* rhs_extra (host, num_dofs complex128, may be NULL) is added to TbemSystem.rhs to form b -- the incident-field term a
 * caller computes with IncidentField::compute_rhs_with_beta; max_iterations / restart / tolerance = GmresConfig */
int bemb200_sweep_submit(bemb200_sweep* sw, const bemb200_physics* phys, double beta_re, double beta_im, const double* rhs_extra,
                         uint32_t max_iterations, uint32_t restart, double tolerance);
/* x_out: num_dofs complex128 (host); stats and rhs_out (the b that was solved) may be NULL */
int bemb200_sweep_next(bemb200_sweep* sw, double* x_out, bemb200_gmres_info* info, bemb200_assembly_stats* stats, double* rhs_out);
/* Queue a frequency with nrhs (1..32) incident right-hand sides (sources as bemb200_incident_rhs_batch).  The incident block
 * is built on the device right after the frequency's assembly; b = TbemSystem.rhs + incident is formed on the device.
 * nrhs = 1 solves as bemb200_sweep_submit with rhs_extra = that incident vector (same bits); nrhs > 1 with the batched solver
 * (bemb200_gmres_batched / _schwarz; overlapping subdomains fail in next_batch with BEMB200_EUNSUPPORTED and the frequency is
 * consumed).  bemb200_sweep_next on a frequency with nrhs > 1 returns BEMB200_EINVAL and leaves it queued. */
int bemb200_sweep_submit_incident(bemb200_sweep* sw, const bemb200_physics* phys, double beta_re, double beta_im, uint32_t nrhs,
                                  const uint32_t* src_ptr, const int32_t* kinds, const double* vecs, const double* amps,
                                  uint32_t max_iterations, uint32_t restart, double tolerance);
/* Solve the oldest queued frequency, whichever call submitted it: x_out [capacity * num_dofs] complex128 and infos[capacity]
 * (host) receive its *nrhs_out (1 for bemb200_sweep_submit) solutions.  A frequency of more than `capacity` right-hand sides
 * returns BEMB200_EINVAL and stays queued.  stats may be NULL. */
int bemb200_sweep_next_batch(bemb200_sweep* sw, uint32_t capacity, double* x_out, bemb200_gmres_info* infos, uint32_t* nrhs_out,
                             bemb200_assembly_stats* stats);
uint64_t bemb200_sweep_boosts(const bemb200_sweep* sw);
/* Solve every frequency returned from now on with gmres_preconditioned (gmres.rs:282) and the block-Jacobi / additive Schwarz
 * preconditioner of bemb200_schwarz_create, rebuilt from each frequency's matrix (arguments as there; num_subdomains = 0
 * switches back to plain gmres).  The subdomains are copied. */
int bemb200_sweep_set_block_jacobi(bemb200_sweep* sw, uint32_t num_subdomains, const uint64_t* sub_ptr, const uint64_t* sub_idx);
/* Assemble every frequency submitted from now on (through either submit call) with these options; NULL restores the
 * defaults.  The admittance is copied here and each submit takes the options current at that moment, so every frequency can
 * carry its own Y(f). */
int bemb200_sweep_set_assembly_options(bemb200_sweep* sw, const bemb200_assembly_options* opts);
void bemb200_sweep_destroy(bemb200_sweep* sw);

/* ---- one process, several devices (SURVEY 8b "Threading": every reference caller -- BemSolver::solve, qa_suite -- is one
 * process) ----------------------------------------------------------------------------------------------------------------
 * The group owns one rank context per entry of devices[] (1..8; the same device may be listed more than once: its SMs are
 * then split between the ranks -- used by the single-GPU test of the sharded solver).  Rows are block partitioned
 * (bemb200_partition); assembly needs no communication; bemb200_multi_gmres runs the persistent fused GMRES kernel on every
 * device, the ranks exchanging Krylov vectors and reduction partials through peer-mapped memory
 * (cudaDeviceEnablePeerAccess; no CUDA IPC, no NCCL).  Calls on one group must not overlap. */
typedef struct bemb200_multi bemb200_multi;
typedef struct bemb200_multi_matrix bemb200_multi_matrix;
int bemb200_multi_create(const int* devices, int n, bemb200_multi** out);
void bemb200_multi_destroy(bemb200_multi* mg);
int bemb200_multi_num_ranks(const bemb200_multi* mg);
const char* bemb200_multi_last_error(const bemb200_multi* mg);
/* build_tbem_system_with_beta (tbem.rs:96-222), every device assembling its own row block */
int bemb200_multi_assemble(bemb200_multi* mg, const bemb200_mesh* mesh, const bemb200_physics* phys, double beta_re, double beta_im,
                           bemb200_multi_matrix** out);
void bemb200_multi_matrix_free(bemb200_multi_matrix* mm);
uint64_t bemb200_multi_num_rows(const bemb200_multi_matrix* mm);
int bemb200_multi_rhs_download(const bemb200_multi_matrix* mm, double* out);  /* TbemSystem.rhs, all rows */
int bemb200_multi_matrix_download(const bemb200_multi_matrix* mm, uint64_t row_begin, uint64_t row_end, double* out);
/* gmres / gmres_with_guess (gmres.rs:96-277) on the sharded operator; b, x0 (may be NULL), x_out on the host */
int bemb200_multi_gmres(const bemb200_multi_matrix* mm, const double* b, const double* x0, uint32_t max_iterations, uint32_t restart,
                        double tolerance, double* x_out, bemb200_gmres_info* info);

/* ---- measurement helpers ----------------------------------------------------------- */
/* register-resident DFMA peak of this device in TFLOP/s (2 flop per DFMA) */
int bemb200_measure_fp64_peak(bemb200_ctx* ctx, double* tflops);
/* max abs error of the far kernel's sincos / rsqrt against the CUDA math library over
 * `n` sample arguments in [0, xmax] */
int bemb200_selftest_math(bemb200_ctx* ctx, uint64_t n, double xmax, double* sincos_err, double* rsqrt_relerr);
/* latency probe of the in-stream all-gather used by the distributed solver: microseconds per
 * call for `iters` all-gathers of `bytes_per_rank` bytes, stream-ordered (sync_each = 0) or
 * with a host synchronisation after each one (sync_each = 1) */
int bemb200_measure_allgather(bemb200_ctx* ctx, uint64_t bytes_per_rank, int iters, int sync_each, double* usec_per_call);
/* device pointer of the local matrix slab / device stream, for callers that own a CUDA
 * context in the same process (bench harness) */
void* bemb200_matrix_device_ptr(const bemb200_matrix* m);

#ifdef __cplusplus
}
#endif
#endif /* BEMB200_H */
