// admittance_oracle.cpp -- CPU oracle of bemb200_assemble_staged_opts (DESIGN.md 4.8): admittance boundaries, a forced
// dg_dn_sign and the consistent beta of the prescribed-velocity right-hand side.
//
// TEST INFRASTRUCTURE ONLY.  The reference-faithful oracle (oracle/bem_oracle.cpp) is compiled into this translation unit
// unchanged, so orc_assemble_opts integrates every pair with the very same regular_integration / singular_integration and
// follows orc_assemble line by line; the options only add the terms below.  With default options and no admittance it is
// orc_assemble, bit for bit.
//
//   A[i,j] -= Y_j (gamma tau G_ij + beta H^T_ij)      every row i, including i = j (no dg_dn_sign on G / H^T)
//   A[i,i] -= Y_i beta tau / 2
//
// consistent_beta: the integrators take the unscaled beta0 = i harmonic / k from Physics.  Their velocity right-hand side
// is sum_q (zg gamma tau + zht beta0) zb; a second call with gamma = 0 isolates the beta0 part, which is then rescaled to
// the assembly's beta.  That needs beta0 != 0 (tau > 0): other cases return -2.
#include "../../oracle/bem_oracle.cpp"

extern "C" {

// Returns the number of kernel evaluations, -1 for options the library refuses (dg_dn_sign not in {-1, 0, 1},
// consistent_beta not in {0, 1}, non-zero Y on a pressure / transfer element), -2 for consistent_beta with tau <= 0.
// admittance: NULL or ndof complex128 in DOF order.
long orc_assemble_opts(const orc_mesh* m, double k, double harmonic, double tau, double beta_re, double beta_im,
                       int dg_dn_sign, int consistent_beta, const double* admittance, uint64_t row_begin, uint64_t row_end,
                       double* A_out, double* rhs_out, int nthreads) {
    if (dg_dn_sign < -1 || dg_dn_sign > 1 || consistent_beta < 0 || consistent_beta > 1) return -1;
    if (consistent_beta && !(tau > 0.0)) return -2;
    const uint64_t ndof = orc_count_dofs(m);
    const cplx* Y = (const cplx*)admittance;
    if (Y)
        for (uint64_t e = 0; e < m->n_elem; ++e)
            if (!m->is_eval[e] && m->bc_type[e] != 0 && (Y[m->dof[e]].re != 0.0 || Y[m->dof[e]].im != 0.0)) return -1;
    const uint64_t nrows = row_end - row_begin;
    cplx* A = (cplx*)A_out;
    cplx* rhs = (cplx*)rhs_out;
    std::memset(A, 0, sizeof(cplx) * nrows * ndof);
    std::memset(rhs, 0, sizeof(cplx) * nrows);
    Physics ph{k, harmonic, tau, 1.0};
    Physics ph_nog{k, harmonic, tau, 0.0};  // consistent_beta: the beta0 part of the velocity right-hand side alone
    const cplx gamma = C(ph.gamma, 0.0), ctau = C(tau, 0.0), beta = C(beta_re, beta_im);
    const cplx beta_rescale = consistent_beta ? beta / ph.beta_unscaled() : C(1.0, 0.0);
    const double sign = dg_dn_sign == 0 ? orc_dg_dn_sign(m, k) : (double)dg_dn_sign;
    std::vector<long> qp_per_thread(resolve_threads(nthreads) + 1, 0);
    parallel_for((int64_t)m->n_elem, nthreads, 4, [&](int64_t iel, int tid) {
        if (m->is_eval[iel]) return;
        const uint64_t sdof = m->dof[iel];
        if (sdof < row_begin || sdof >= row_end) return;
        const double* src = m->center + 3 * iel;
        const double* nx = m->normal + 3 * iel;
        cplx* Arow = A + (sdof - row_begin) * ndof;
        cplx& rhs_i = rhs[sdof - row_begin];
        // get_bc_type_and_value(): tbem.rs:234-244
        const int bct = m->bc_type[iel];
        const cplx* bcv = (const cplx*)(m->bc_val + 8 * iel);
        const int bcl = m->bc_len[iel];
        // add_free_terms(): tbem.rs:273-304
        {
            cplx sum = C(0, 0);
            for (int i = 0; i < bcl; ++i) sum += bcv[i];
            cplx avg = sum / (double)bcl;
            if (bct == 0) {
                Arow[sdof] -= gamma * 0.5;
                rhs_i += avg * beta * ctau * 0.5;
            } else if (bct == 1) {
                Arow[sdof] -= beta * ctau * 0.5;
                rhs_i += avg * ctau * 0.5;
            }
        }
        long nq = 0;
        for (uint64_t jel = 0; jel < m->n_elem; ++jel) {
            if (m->is_eval[jel]) continue;
            const int et = m->etype[jel];
            double coords[12];
            for (int v = 0; v < et; ++v)
                for (int c = 0; c < 3; ++c) coords[3 * v + c] = m->nodes[3 * (uint64_t)m->conn[4 * jel + v] + c];
            const uint64_t fdof = m->dof[jel];
            const int fbct = m->bc_type[jel];
            const cplx* fbcv = (const cplx*)(m->bc_val + 8 * jel);
            const int fbcl = m->bc_len[jel];
            bool compute_rhs = false;  // has_nonzero_bc(): tbem.rs:247
            for (int i = 0; i < fbcl; ++i) compute_rhs = compute_rhs || (cnorm(fbcv[i]) > 1e-15);
            IntegrationResult r;
            if ((int64_t)jel == iel)
                r = singular_integration(src, nx, coords, et, ph, compute_rhs ? fbcv : nullptr, fbcl, fbct, compute_rhs, &nq);
            else
                r = regular_integration(src, nx, coords, et, m->area[jel], ph, compute_rhs ? fbcv : nullptr, fbcl, fbct,
                                        compute_rhs, &nq);
            if (consistent_beta && compute_rhs && fbct == 0) {
                IntegrationResult r0;
                long nq0 = 0;
                if ((int64_t)jel == iel)
                    r0 = singular_integration(src, nx, coords, et, ph_nog, fbcv, fbcl, fbct, true, &nq0);
                else
                    r0 = regular_integration(src, nx, coords, et, m->area[jel], ph_nog, fbcv, fbcl, fbct, true, &nq0);
                r.rhs = (r.rhs - r0.rhs) + r0.rhs * beta_rescale;
            }
            r.dg_dn = r.dg_dn * sign;
            // assemble_tbem(): tbem.rs:311-345
            cplx coeff;
            if (fbct == 0) coeff = r.dg_dn * gamma * ctau + r.d2g * beta;
            else if (fbct == 1) coeff = -(r.g * gamma * ctau + r.dg_dnx * beta);
            else coeff = C(0, 0);
            if (Y && (Y[fdof].re != 0.0 || Y[fdof].im != 0.0)) {
                coeff -= Y[fdof] * (r.g * gamma * ctau + r.dg_dnx * beta);
                if ((int64_t)jel == iel) coeff -= Y[fdof] * beta * ctau * 0.5;
            }
            Arow[fdof] += coeff;
            if (compute_rhs) rhs_i += r.rhs;
        }
        qp_per_thread[tid] += nq;
    });
    long total_qp = 0;
    for (long q : qp_per_thread) total_qp += q;
    return total_qp;
}

}  // extern "C"
