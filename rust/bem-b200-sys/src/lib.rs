//! Raw FFI declarations of `include/bemb200.h` -- nothing else.  This crate depends on NO crate of the math-audio
//! workspace (so nothing in the workspace can form a cycle through it); build.rs compiles the CUDA sources with nvcc
//! for sm_100a.  The safe wrappers with the reference's signatures live in the sibling crate `math-bem-b200`, which
//! depends on this crate, on `math-solvers` and on `math-bem`.  Written without a Rust toolchain at hand (see
//! INTEGRATION.md); the executable twin of these declarations is math_audio_b200/_capi.py.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_double, c_int, c_void};

#[repr(C)] pub struct bemb200_ctx { _p: [u8; 0] }
#[repr(C)] pub struct bemb200_staged_mesh { _p: [u8; 0] }
#[repr(C)] pub struct bemb200_matrix { _p: [u8; 0] }
#[repr(C)] pub struct bemb200_sweep { _p: [u8; 0] }
#[repr(C)] pub struct bemb200_precond { _p: [u8; 0] }
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct bemb200_precond_stats { pub num_subdomains: u32, pub local_subdomains: u32, pub min_size: u32, pub max_size: u32,
                                   pub avg_size: f64, pub inverse_bytes: u64, pub factor_ms: f64, pub disjoint: i32 }
#[repr(C)] pub struct bemb200_multi { _p: [u8; 0] }
#[repr(C)] pub struct bemb200_multi_matrix { _p: [u8; 0] }
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct bemb200_assembly_stats { pub near_pairs: u64, pub special_pairs: u64, pub far_kernel_launches: u64,
                                    pub total_launches: u64, pub far_ms: f64, pub total_ms: f64 }

#[repr(C)]
pub struct bemb200_mesh {
    pub n_nodes: u64, pub n_elem: u64,
    pub nodes: *const f64, pub conn: *const u32, pub etype: *const u8,
    pub center: *const f64, pub normal: *const f64, pub area: *const f64,
    pub bc_type: *const i32, pub bc_len: *const u8, pub bc_val: *const f64,
    pub dof: *const u32, pub is_eval: *const u8,
}
#[repr(C)] #[derive(Clone, Copy)]
pub struct bemb200_physics { pub wave_number: f64, pub harmonic_factor: f64, pub tau: f64, pub gamma: f64 }
/// `int apply(void* user, const double* r, double* z, uint64_t n)`: z = M^-1 r on host memory, 0 = success (`Preconditioner::apply`).
pub type bemb200_precond_fn = Option<unsafe extern "C" fn(user: *mut c_void, r: *const f64, z: *mut f64, n: u64) -> c_int>;
/// `bemb200_assembly_options`: admittance boundaries and the sign-consistent formulation (DESIGN.md 4.8).
#[repr(C)] #[derive(Clone, Copy)]
pub struct bemb200_assembly_options { pub dg_dn_sign: i32, pub consistent_beta: i32, pub admittance: *const f64 }
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct bemb200_gmres_info { pub iterations: u64, pub restarts: u64, pub residual: f64, pub converged: i32 }

extern "C" {
    pub fn bemb200_ctx_create(device: c_int, out: *mut *mut bemb200_ctx) -> c_int;
    pub fn bemb200_ctx_create_ex(device: c_int, rank: c_int, nranks: c_int, nccl_id: *const u8,
                                 cuda_stream: *mut c_void, out: *mut *mut bemb200_ctx) -> c_int;
    pub fn bemb200_nccl_unique_id(out: *mut u8) -> c_int;
    pub fn bemb200_ctx_destroy(ctx: *mut bemb200_ctx);
    pub fn bemb200_ctx_set_background(ctx: *mut bemb200_ctx, blocks_per_sm: c_int) -> c_int;
    pub fn bemb200_ctx_set_shared_gpu(ctx: *mut bemb200_ctx, shared: c_int) -> c_int;
    pub fn bemb200_ctx_peer_exchange_active(ctx: *const bemb200_ctx, active: *mut c_int) -> c_int;
    pub fn bemb200_last_error(ctx: *const bemb200_ctx) -> *const c_char;
    pub fn bemb200_partition(n: u64, nranks: c_int, rank: c_int, row_begin: *mut u64, row_end: *mut u64);
    pub fn bemb200_mesh_stage(ctx: *mut bemb200_ctx, mesh: *const bemb200_mesh, out: *mut *mut bemb200_staged_mesh) -> c_int;
    pub fn bemb200_staged_mesh_free(sm: *mut bemb200_staged_mesh);
    pub fn bemb200_assemble_staged(ctx: *mut bemb200_ctx, sm: *const bemb200_staged_mesh, phys: *const bemb200_physics,
                                   beta_re: c_double, beta_im: c_double, row_begin: u64, row_end: u64,
                                   inout: *mut *mut bemb200_matrix) -> c_int;
    pub fn bemb200_assemble_staged_opts(ctx: *mut bemb200_ctx, sm: *const bemb200_staged_mesh, phys: *const bemb200_physics,
                                        beta_re: c_double, beta_im: c_double, opts: *const bemb200_assembly_options, row_begin: u64,
                                        row_end: u64, inout: *mut *mut bemb200_matrix) -> c_int;
    pub fn bemb200_assemble(ctx: *mut bemb200_ctx, mesh: *const bemb200_mesh, phys: *const bemb200_physics,
                            beta_re: c_double, beta_im: c_double, row_begin: u64, row_end: u64,
                            out: *mut *mut bemb200_matrix) -> c_int;
    pub fn bemb200_matrix_from_host(ctx: *mut bemb200_ctx, a_rows: *const f64, n_rows_global: u64, n_cols: u64,
                                    row_begin: u64, row_end: u64, out: *mut *mut bemb200_matrix) -> c_int;
    pub fn bemb200_matrix_free(m: *mut bemb200_matrix);
    pub fn bemb200_num_rows(m: *const bemb200_matrix) -> u64;
    pub fn bemb200_num_cols(m: *const bemb200_matrix) -> u64;
    pub fn bemb200_matrix_download(m: *const bemb200_matrix, row_begin: u64, row_end: u64, out: *mut f64) -> c_int;
    pub fn bemb200_rhs_download_full(m: *const bemb200_matrix, out: *mut f64) -> c_int;
    pub fn bemb200_row_sum_correction(m: *mut bemb200_matrix, avg: *mut f64) -> c_int;
    pub fn bemb200_apply(m: *const bemb200_matrix, x: *const f64, y: *mut f64) -> c_int;
    pub fn bemb200_apply_transpose(m: *const bemb200_matrix, x: *const f64, y: *mut f64) -> c_int;
    pub fn bemb200_bicgstab(m: *const bemb200_matrix, b: *const f64, max_iterations: u32, tolerance: f64, x_out: *mut f64,
                            info: *mut bemb200_gmres_info) -> c_int;
    pub fn bemb200_cgs(m: *const bemb200_matrix, b: *const f64, max_iterations: u32, tolerance: f64, x_out: *mut f64,
                       info: *mut bemb200_gmres_info) -> c_int;
    pub fn bemb200_lu_solve(m: *const bemb200_matrix, b: *const f64, x_out: *mut f64, overwrite_matrix: c_int,
                            factor_ms: *mut f64) -> c_int;
    pub fn bemb200_compute_rcs(sm: *const bemb200_staged_mesh, phys: *const bemb200_physics, n_dirs: u32, dirs: *const f64,
                               surface_pressure: *const f64, rcs_out: *mut f64) -> c_int;
    pub fn bemb200_gmres_preconditioned(m: *const bemb200_matrix, inv_diag: *const f64, b: *const f64, x0: *const f64,
                                        max_iterations: u32, restart: u32, tolerance: f64, x_out: *mut f64,
                                        info: *mut bemb200_gmres_info) -> c_int;
    pub fn bemb200_matrix_diagonal(m: *const bemb200_matrix, out: *mut f64) -> c_int;
    // block-Jacobi / additive Schwarz preconditioner (schwarz.rs) built on the device
    pub fn bemb200_schwarz_create(m: *const bemb200_matrix, num_subdomains: u32, sub_ptr: *const u64, sub_idx: *const u64,
                                  out: *mut *mut bemb200_precond) -> c_int;
    pub fn bemb200_precond_free(p: *mut bemb200_precond);
    pub fn bemb200_precond_stats_get(p: *const bemb200_precond, out: *mut bemb200_precond_stats) -> c_int;
    pub fn bemb200_precond_apply(p: *const bemb200_precond, r: *const f64, z: *mut f64) -> c_int;
    pub fn bemb200_gmres_schwarz(m: *const bemb200_matrix, precond: *const bemb200_precond, b: *const f64, x0: *const f64,
                                 max_iterations: u32, restart: u32, tolerance: f64, x_out: *mut f64,
                                 info: *mut bemb200_gmres_info) -> c_int;
    // gmres_preconditioned with a caller-supplied Preconditioner (host function), Arnoldi process on the device
    pub fn bemb200_gmres_callback(m: *const bemb200_matrix, apply: bemb200_precond_fn, user: *mut c_void, b: *const f64, x0: *const f64,
                                  max_iterations: u32, restart: u32, tolerance: f64, x_out: *mut f64, info: *mut bemb200_gmres_info,
                                  precond_calls: *mut u64) -> c_int;
    pub fn bemb200_gmres_batched(m: *const bemb200_matrix, b_all: *const f64, nrhs: u32, max_iterations: u32, restart: u32,
                                 tolerance: f64, x_all: *mut f64, infos: *mut bemb200_gmres_info, block_matvec_ms: *mut f64,
                                 block_matvecs: *mut u64) -> c_int;
    pub fn bemb200_gmres_batched_schwarz(m: *const bemb200_matrix, precond: *const bemb200_precond, b_all: *const f64, nrhs: u32,
                                         max_iterations: u32, restart: u32, tolerance: f64, x_all: *mut f64,
                                         infos: *mut bemb200_gmres_info, block_matvec_ms: *mut f64, block_matvecs: *mut u64) -> c_int;
    pub fn bemb200_gmres_batched_device(m: *const bemb200_matrix, precond: *const bemb200_precond, b_dev: *const f64, nrhs: u32,
                                        max_iterations: u32, restart: u32, tolerance: f64, x_dev: *mut f64,
                                        infos: *mut bemb200_gmres_info, block_matvec_ms: *mut f64, block_matvecs: *mut u64) -> c_int;
    pub fn bemb200_incident_rhs_batch(sm: *const bemb200_staged_mesh, phys: *const bemb200_physics, beta_re: f64, beta_im: f64,
                                      nrhs: u32, src_ptr: *const u32, kinds: *const i32, vecs: *const f64, amps: *const f64,
                                      system: *const bemb200_matrix, b_host: *mut f64, b_dev: *mut f64) -> c_int;
    pub fn bemb200_compute_rcs_batch(sm: *const bemb200_staged_mesh, phys: *const bemb200_physics, nsol: u32,
                                     surface_pressure: *const f64, on_device: c_int, n_dirs: u32, dirs: *const f64,
                                     rcs_out: *mut f64) -> c_int;
    pub fn bemb200_scattered_field_batch(sm: *const bemb200_staged_mesh, phys: *const bemb200_physics, nsol: u32,
                                         surface_pressure: *const f64, surface_velocity: *const f64, on_device: c_int,
                                         n_eval: u64, eval_pts: *const f64, out: *mut f64) -> c_int;
    pub fn bemb200_far_field(sm: *const bemb200_staged_mesh, phys: *const bemb200_physics, nsol: u32, surface_pressure: *const f64,
                             surface_velocity: *const f64, on_device: c_int, n_dirs: u32, dirs: *const f64, out: *mut f64) -> c_int;
    pub fn bemb200_evaluate_field(sm: *const bemb200_staged_mesh, phys: *const bemb200_physics, nsol: u32, surface_pressure: *const f64,
                                  surface_velocity: *const f64, on_device: c_int, n_eval: u64, eval_pts: *const f64, out: *mut f64) -> c_int;
    pub fn bemb200_evaluate_field_gradient(sm: *const bemb200_staged_mesh, phys: *const bemb200_physics, nsol: u32,
                                           surface_pressure: *const f64, surface_velocity: *const f64, on_device: c_int, n_eval: u64,
                                           eval_pts: *const f64, out_p: *mut f64, out_grad: *mut f64) -> c_int;
    pub fn bemb200_incident_rhs(sm: *const bemb200_staged_mesh, phys: *const bemb200_physics, beta_re: f64, beta_im: f64,
                                n_sources: u32, kinds: *const i32, vecs: *const f64, amps: *const f64, rhs_host: *mut f64,
                                rhs_dev: *mut f64) -> c_int;
    pub fn bemb200_scattered_field(sm: *const bemb200_staged_mesh, phys: *const bemb200_physics, n_eval: u64, eval_pts: *const f64,
                                   surface_pressure: *const f64, surface_velocity: *const f64, out: *mut f64) -> c_int;
    pub fn bemb200_gmres(m: *const bemb200_matrix, b: *const f64, x0: *const f64, max_iterations: u32, restart: u32,
                         tolerance: f64, x_out: *mut f64, info: *mut bemb200_gmres_info) -> c_int;
    // pipelined frequency sweep behind the C ABI
    pub fn bemb200_sweep_create(device: c_int, rank: c_int, nranks: c_int, nccl_id: *const u8, mesh: *const bemb200_mesh,
                                overlap: c_int, background_blocks_per_sm: c_int, out: *mut *mut bemb200_sweep) -> c_int;
    pub fn bemb200_sweep_num_dofs(sw: *const bemb200_sweep) -> u64;
    pub fn bemb200_sweep_submit(sw: *mut bemb200_sweep, phys: *const bemb200_physics, beta_re: c_double, beta_im: c_double,
                                rhs_extra: *const f64, max_iterations: u32, restart: u32, tolerance: f64) -> c_int;
    pub fn bemb200_sweep_next(sw: *mut bemb200_sweep, x_out: *mut f64, info: *mut bemb200_gmres_info,
                              stats: *mut bemb200_assembly_stats, rhs_out: *mut f64) -> c_int;
    pub fn bemb200_sweep_submit_incident(sw: *mut bemb200_sweep, phys: *const bemb200_physics, beta_re: f64, beta_im: f64, nrhs: u32,
                                         src_ptr: *const u32, kinds: *const i32, vecs: *const f64, amps: *const f64,
                                         max_iterations: u32, restart: u32, tolerance: f64) -> c_int;
    pub fn bemb200_sweep_next_batch(sw: *mut bemb200_sweep, capacity: u32, x_out: *mut f64, infos: *mut bemb200_gmres_info,
                                    nrhs_out: *mut u32, stats: *mut bemb200_assembly_stats) -> c_int;
    pub fn bemb200_sweep_boosts(sw: *const bemb200_sweep) -> u64;
    pub fn bemb200_sweep_set_block_jacobi(sw: *mut bemb200_sweep, num_subdomains: u32, sub_ptr: *const u64, sub_idx: *const u64) -> c_int;
    pub fn bemb200_sweep_set_assembly_options(sw: *mut bemb200_sweep, opts: *const bemb200_assembly_options) -> c_int;
    pub fn bemb200_sweep_destroy(sw: *mut bemb200_sweep);
    // one process, several devices
    pub fn bemb200_multi_create(devices: *const c_int, n: c_int, out: *mut *mut bemb200_multi) -> c_int;
    pub fn bemb200_multi_destroy(mg: *mut bemb200_multi);
    pub fn bemb200_multi_last_error(mg: *const bemb200_multi) -> *const c_char;
    pub fn bemb200_multi_assemble(mg: *mut bemb200_multi, mesh: *const bemb200_mesh, phys: *const bemb200_physics,
                                  beta_re: c_double, beta_im: c_double, out: *mut *mut bemb200_multi_matrix) -> c_int;
    pub fn bemb200_multi_matrix_free(mm: *mut bemb200_multi_matrix);
    pub fn bemb200_multi_num_rows(mm: *const bemb200_multi_matrix) -> u64;
    pub fn bemb200_multi_rhs_download(mm: *const bemb200_multi_matrix, out: *mut f64) -> c_int;
    pub fn bemb200_multi_gmres(mm: *const bemb200_multi_matrix, b: *const f64, x0: *const f64, max_iterations: u32, restart: u32,
                               tolerance: f64, x_out: *mut f64, info: *mut bemb200_gmres_info) -> c_int;
}
