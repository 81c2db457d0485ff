// gmres_host.h -- the host side of one GMRES restart cycle (math-solvers/src/iterative/gmres.rs): the Hessenberg matrix,
// the Givens rotations and g, updated column by column as the Arnoldi steps on the device deliver them.  Shared by the
// single-RHS driver (gmres.cu) and the batched one (block_gmres.cu).  The order of every operation is the reference's:
// it fixes the bits of the iterates, the convergence decisions and so the iteration counts.
#pragma once
#include <cmath>
#include <vector>

#include "internal.h"

namespace bemb {

inline double tnorm(cplx a) { return std::sqrt(norm_sqr(a)); }  // ComplexField::norm (traits.rs:93-95)

inline void givens_rotation(cplx a, cplx b, cplx* c, cplx* s) {  // gmres.rs:589-603
    const double tol = 1e-30;
    if (tnorm(b) < tol) { *c = C(1, 0); *s = C(0, 0); return; }
    if (tnorm(a) < tol) { *c = C(0, 0); *s = C(1, 0); return; }
    double r = std::sqrt(norm_sqr(a) + norm_sqr(b));
    *c = a * C(1.0 / r, 0.0);
    *s = b * C(1.0 / r, 0.0);
}

inline void solve_upper_triangular(const std::vector<cplx>& h, int ldh, const std::vector<cplx>& g, int k,
                                   std::vector<cplx>& y) {  // gmres.rs:606-621
    y.assign(k, C(0, 0));
    for (int i = k - 1; i >= 0; --i) {
        cplx sum = g[i];
        for (int j = i + 1; j < k; ++j) sum -= h[i * ldh + j] * y[j];
        cplx d = h[i * ldh + i];
        if (tnorm(d) > 1e-30) {
            double ns = norm_sqr(d);
            y[i] = sum * C(d.re / ns, -d.im / ns);
        }
    }
}

struct GmresCycle {
    int ldh = 0;                   // restart length: H is (ldh + 1) x ldh, row-major
    std::vector<cplx> h, cs, sn, g;

    // v_0 = r / beta, H = 0, g = [beta, 0, ...]  (gmres.rs:160-172)
    void start(int restart, double beta) {
        ldh = restart;
        h.assign((size_t)(ldh + 1) * ldh, C(0, 0));
        cs.clear(); sn.clear();
        g.assign(ldh + 1, C(0, 0));
        g[0] = C(beta, 0.0);
    }

    // Column j as the Arnoldi step left it (hcol[0..j]: the projections, hcol[j + 1].re: ||w||): store it, apply the earlier
    // rotations, form and apply rotation j, update g (gmres.rs:205-222).  Returns |g[j + 1]| / b_norm; *breakdown is set when
    // ||w|| < 1e-14, i.e. v_{j+1} was not formed (gmres.rs:194-202).
    double add_column(int j, const cplx* hcol, double b_norm, bool* breakdown) {
        for (int i = 0; i <= j; ++i) h[i * ldh + j] = hcol[i];
        const double w_norm = hcol[j + 1].re;
        h[(j + 1) * ldh + j] = C(w_norm, 0.0);
        *breakdown = w_norm < 1e-14;
        for (int i = 0; i < j; ++i) {
            cplx temp = conj(cs[i]) * h[i * ldh + j] + conj(sn[i]) * h[(i + 1) * ldh + j];
            h[(i + 1) * ldh + j] = C(0, 0) - sn[i] * h[i * ldh + j] + cs[i] * h[(i + 1) * ldh + j];
            h[i * ldh + j] = temp;
        }
        cplx c, s;
        givens_rotation(h[j * ldh + j], h[(j + 1) * ldh + j], &c, &s);
        cs.push_back(c); sn.push_back(s);
        h[j * ldh + j] = conj(c) * h[j * ldh + j] + conj(s) * h[(j + 1) * ldh + j];
        h[(j + 1) * ldh + j] = C(0, 0);
        cplx temp = conj(c) * g[j] + conj(s) * g[j + 1];
        g[j + 1] = C(0, 0) - s * g[j] + c * g[j + 1];
        g[j] = temp;
        return tnorm(g[j + 1]) / b_norm;
    }

    // y = H[0..k, 0..k]^-1 g[0..k], the coefficients of x += V y
    void solve(int k, std::vector<cplx>& y) const { solve_upper_triangular(h, ldh, g, k, y); }
};

}  // namespace bemb
