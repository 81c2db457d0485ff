// postprocess.cu -- the O(N) / O(M N) neighbours of the hot path (SURVEY.md 8f ranks 1-2):
//   incident_rhs_kernel      IncidentField::compute_rhs_with_beta   math-bem/src/core/incident.rs:93-342
//   scattered_field_kernel   compute_scattered_field                 math-bem/src/core/postprocess/pressure.rs:81-259
//   rcs_kernel               compute_rcs                             math-bem/src/core/postprocess/pressure.rs:438-478
//   far_field_kernel         the complex far-field amplitude with the surface-velocity term (DESIGN.md section 4.9; no
//                            reference counterpart)
// All work on the staged (DOF-ordered) mesh so that a frequency sweep never leaves the device.
//
// The *_batch kernels serve several right-hand sides / solutions of one mesh (plane waves from many directions, DESIGN.md
// section 4.7).  What depends only on the geometry -- sincos(-k c.d) and n.d of the RCS, the 7-point Green's function of the
// field -- is evaluated once and applied to every solution of a chunk.  Per solution they repeat the single kernels'
// expressions, thread-to-element mapping and reduction order, so row s of a batch has the bits of the single call on
// solution s (this unit is compiled with -fmad=false: no contraction can differ between the two).
#include <algorithm>
#include <cmath>
#include <vector>

#include "api_internal.h"

using namespace bemb;

namespace {

struct Source {
    int kind;       // 0 plane wave (vec = unit direction), 1 point source (vec = position)
    double v[3];
    cplx amp;
};

// rhs_i = -(gamma p_inc + beta tau dp_inc/dn) summed over the sources (incident.rs:317-342)
__global__ void incident_rhs_kernel(const double* __restrict__ src, uint32_t n, const Source* __restrict__ sources, int ns, double k,
                                    double gamma, double tau, cplx beta, cplx* __restrict__ rhs) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double* p = src + 8ull * i;
    const double* nr = p + 3;
    cplx pinc = C(0, 0), dpdn = C(0, 0);
    for (int s = 0; s < ns; ++s) {
        const Source sc = sources[s];
        if (sc.kind == 0) {  // incident.rs:103-118, 191-211
            const double kdotx = k * (sc.v[0] * p[0] + sc.v[1] * p[1] + sc.v[2] * p[2]);
            const double kdotn = k * (sc.v[0] * nr[0] + sc.v[1] * nr[1] + sc.v[2] * nr[2]);
            double sn, cs;
            sincos(kdotx, &sn, &cs);
            const cplx pw = sc.amp * C(cs, sn);
            pinc += pw;
            dpdn += C(0.0, kdotn) * pw;
        } else {  // incident.rs:120-134, 213-238
            const double dx = p[0] - sc.v[0], dy = p[1] - sc.v[1], dz = p[2] - sc.v[2];
            const double r = sqrt(dx * dx + dy * dy + dz * dz);
            if (r > 1e-10) {
                double sn, cs;
                sincos(k * r, &sn, &cs);
                const cplx g = C(cs, sn) / (4.0 * PI * r);
                pinc += sc.amp * g;
                const cplx dgdr = (C(0.0, k) - C(1.0 / r, 0.0)) * g;
                const double drdn = (dx * nr[0] + dy * nr[1] + dz * nr[2]) / r;
                dpdn += sc.amp * dgdr * drdn;
            }
        }
    }
    const cplx v = -(pinc * gamma + beta * C(tau, 0.0) * dpdn);
    rhs[i] = v;
}

__device__ __constant__ double d_tr7[7][3] = {
    {0.333333333333333, 0.333333333333333, 0.225},
    {0.797426985353087, 0.101286507323456, 0.125939180544827},
    {0.101286507323456, 0.797426985353087, 0.125939180544827},
    {0.101286507323456, 0.101286507323456, 0.125939180544827},
    {0.470142064105115, 0.059715871789770, 0.132394152788506},
    {0.059715871789770, 0.470142064105115, 0.132394152788506},
    {0.470142064105115, 0.470142064105115, 0.132394152788506},
};

// p_scat(x) = sum_j  p_j int dG/dn_y - v_j int G  with the 7-point rule on the element's FIRST
// triangle (Quad4 is approximated by its first three nodes exactly as pressure.rs:184-198 does).
// One block per evaluation point, threads over elements, deterministic block reduction.
__global__ void __launch_bounds__(256)
scattered_field_kernel(const double* __restrict__ coords, uint32_t n, const double* __restrict__ eval, const cplx* __restrict__ ps,
                       const cplx* __restrict__ vs, double wavruim, cplx* __restrict__ out) {
    __shared__ double red[2][8];
    const double x0 = eval[3 * blockIdx.x], x1 = eval[3 * blockIdx.x + 1], x2 = eval[3 * blockIdx.x + 2];
    cplx acc = C(0, 0);
    for (uint32_t j = threadIdx.x; j < n; j += blockDim.x) {
        const double* c = coords + 12ull * j;
        const double e1[3] = {c[3] - c[0], c[4] - c[1], c[5] - c[2]};
        const double e2[3] = {c[6] - c[0], c[7] - c[1], c[8] - c[2]};
        const double nv[3] = {e1[1] * e2[2] - e1[2] * e2[1], e1[2] * e2[0] - e1[0] * e2[2], e1[0] * e2[1] - e1[1] * e2[0]};
        const double jac = sqrt(nv[0] * nv[0] + nv[1] * nv[1] + nv[2] * nv[2]);
        if (jac < 1e-15) continue;
        const double en[3] = {nv[0] / jac, nv[1] / jac, nv[2] / jac};
        const cplx p_surf = ps[j];
        const cplx v_surf = vs ? vs[j] : C(0, 0);
        const bool has_v = sqrt(v_surf.re * v_surf.re + v_surf.im * v_surf.im) > 1e-15;
        cplx res = C(0, 0);
#pragma unroll
        for (int q = 0; q < 7; ++q) {
            const double xi = d_tr7[q][0], eta = d_tr7[q][1], wq = d_tr7[q][2] * 0.5;
            const double l0 = 1.0 - xi - eta;
            const double rv[3] = {l0 * c[0] + xi * c[3] + eta * c[6] - x0, l0 * c[1] + xi * c[4] + eta * c[7] - x1,
                                  l0 * c[2] + xi * c[5] + eta * c[8] - x2};
            const double r = sqrt(rv[0] * rv[0] + rv[1] * rv[1] + rv[2] * rv[2]);
            if (r < 1e-15) continue;
            const double vjacwe = jac * wq;
            double sn, cs;
            sincos(wavruim * r, &sn, &cs);
            const double re1 = 4.0 * PI * r;
            const cplx zg = C(cs / re1, sn / re1);
            const cplx zgikr = zg * C(-1.0 / r, wavruim);
            const double drdn = (rv[0] * en[0] + rv[1] * en[1] + rv[2] * en[2]) / r;
            res += p_surf * (zgikr * drdn) * vjacwe;
            if (has_v) res -= v_surf * zg * vjacwe;
        }
        acc += res;
    }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) {
        acc.re += __shfl_xor_sync(0xffffffffu, acc.re, m);
        acc.im += __shfl_xor_sync(0xffffffffu, acc.im, m);
    }
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = acc.re; red[1][threadIdx.x >> 5] = acc.im; }
    __syncthreads();
    if (threadIdx.x == 0) {
        cplx t = C(0, 0);
        for (int w = 0; w < 8; ++w) { t.re += red[0][w]; t.im += red[1][w]; }
        out[blockIdx.x] = t;
    }
}

// compute_rcs (pressure.rs:438-478): F(d) = sum_j p_j exp(-i k c_j.d) A_j (i k)(n_j.d), RCS = 4 pi |F|^2.
// One block per direction, threads over elements, deterministic block reduction.
__global__ void __launch_bounds__(256)
rcs_kernel(const double* __restrict__ src, const double* __restrict__ area, uint32_t n, const double* __restrict__ dirs,
           const cplx* __restrict__ ps, double k, double* __restrict__ out) {
    __shared__ double red[2][8];
    const double d0 = dirs[3 * blockIdx.x], d1 = dirs[3 * blockIdx.x + 1], d2 = dirs[3 * blockIdx.x + 2];
    cplx acc = C(0, 0);
    for (uint32_t j = threadIdx.x; j < n; j += blockDim.x) {
        const double* c = src + 8ull * j;
        const double phase = -k * (c[0] * d0 + c[1] * d1 + c[2] * d2);
        double sn, cs;
        sincos(phase, &sn, &cs);
        const double n_dot_d = c[3] * d0 + c[4] * d1 + c[5] * d2;
        const cplx t = ((ps[j] * C(cs, sn)) * area[j]) * C(0.0, k);
        acc += t * n_dot_d;
    }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) {
        acc.re += __shfl_xor_sync(0xffffffffu, acc.re, m);
        acc.im += __shfl_xor_sync(0xffffffffu, acc.im, m);
    }
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = acc.re; red[1][threadIdx.x >> 5] = acc.im; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double tr = 0.0, ti = 0.0;
        for (int w = 0; w < 8; ++w) { tr += red[0][w]; ti += red[1][w]; }
        out[blockIdx.x] = 4.0 * 3.14159265358979323846 * (tr * tr + ti * ti);
    }
}

// Column s of a batch: incident_rhs_kernel over the sources [grp[s], grp[s+1]) (same per-entry arithmetic and source order);
// `sys` != NULL (TbemSystem.rhs, all rows) adds it as one IEEE add, sys + incident, the b of bemb200_sweep_next.
__global__ void incident_rhs_batch_kernel(const double* __restrict__ src, uint32_t n, const Source* __restrict__ sources,
                                          const uint32_t* __restrict__ grp, double k, double gamma, double tau, cplx beta,
                                          const cplx* __restrict__ sys, cplx* __restrict__ rhs) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t s0 = grp[blockIdx.y], s1 = grp[blockIdx.y + 1];
    const double* p = src + 8ull * i;
    const double* nr = p + 3;
    cplx pinc = C(0, 0), dpdn = C(0, 0);
    for (uint32_t s = s0; s < s1; ++s) {
        const Source sc = sources[s];
        if (sc.kind == 0) {
            const double kdotx = k * (sc.v[0] * p[0] + sc.v[1] * p[1] + sc.v[2] * p[2]);
            const double kdotn = k * (sc.v[0] * nr[0] + sc.v[1] * nr[1] + sc.v[2] * nr[2]);
            double sn, cs;
            sincos(kdotx, &sn, &cs);
            const cplx pw = sc.amp * C(cs, sn);
            pinc += pw;
            dpdn += C(0.0, kdotn) * pw;
        } else {
            const double dx = p[0] - sc.v[0], dy = p[1] - sc.v[1], dz = p[2] - sc.v[2];
            const double r = sqrt(dx * dx + dy * dy + dz * dz);
            if (r > 1e-10) {
                double sn, cs;
                sincos(k * r, &sn, &cs);
                const cplx g = C(cs, sn) / (4.0 * PI * r);
                pinc += sc.amp * g;
                const cplx dgdr = (C(0.0, k) - C(1.0 / r, 0.0)) * g;
                const double drdn = (dx * nr[0] + dy * nr[1] + dz * nr[2]) / r;
                dpdn += sc.amp * dgdr * drdn;
            }
        }
    }
    const cplx v = -(pinc * gamma + beta * C(tau, 0.0) * dpdn);
    rhs[(uint64_t)blockIdx.y * n + i] = sys ? sys[i] + v : v;
}

constexpr int SOL_CHUNK = 8;  // solutions per block of the batch kernels (grid dimension y runs over chunks)

// Warp shuffle + 8-warp sum of every solution of the chunk, in the order of the single kernels; thread c < cnt returns
// the block total of solution c (other threads: undefined).
__device__ __forceinline__ cplx block_sum_chunk(cplx (&acc)[SOL_CHUNK], int cnt) {
    __shared__ double red[2][SOL_CHUNK][8];
#pragma unroll
    for (int c = 0; c < SOL_CHUNK; ++c) {
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) {
            acc[c].re += __shfl_xor_sync(0xffffffffu, acc[c].re, m);
            acc[c].im += __shfl_xor_sync(0xffffffffu, acc[c].im, m);
        }
        if ((threadIdx.x & 31) == 0) { red[0][c][threadIdx.x >> 5] = acc[c].re; red[1][c][threadIdx.x >> 5] = acc[c].im; }
    }
    __syncthreads();
    cplx t = C(0, 0);
    if ((int)threadIdx.x < cnt)
        for (int w = 0; w < 8; ++w) { t.re += red[0][threadIdx.x][w]; t.im += red[1][threadIdx.x][w]; }
    return t;
}

// scattered_field_kernel for solutions [SOL_CHUNK * blockIdx.y, +SOL_CHUNK) of ps / vs ([nsol][n], DOF order): the geometry
// and Green's function of a (point, element, quadrature point) are computed once for the whole chunk.
__global__ void __launch_bounds__(256)
scattered_field_batch_kernel(const double* __restrict__ coords, uint32_t n, const double* __restrict__ eval, uint32_t n_eval,
                             uint32_t nsol, const cplx* __restrict__ ps, const cplx* __restrict__ vs, double wavruim,
                             cplx* __restrict__ out) {
    const double x0 = eval[3 * blockIdx.x], x1 = eval[3 * blockIdx.x + 1], x2 = eval[3 * blockIdx.x + 2];
    const uint32_t s0 = blockIdx.y * SOL_CHUNK;
    const int cnt = (int)min((uint32_t)SOL_CHUNK, nsol - s0);
    cplx acc[SOL_CHUNK];
#pragma unroll
    for (int c = 0; c < SOL_CHUNK; ++c) acc[c] = C(0, 0);
    for (uint32_t j = threadIdx.x; j < n; j += blockDim.x) {
        const double* c_ = coords + 12ull * j;
        const double e1[3] = {c_[3] - c_[0], c_[4] - c_[1], c_[5] - c_[2]};
        const double e2[3] = {c_[6] - c_[0], c_[7] - c_[1], c_[8] - c_[2]};
        const double nv[3] = {e1[1] * e2[2] - e1[2] * e2[1], e1[2] * e2[0] - e1[0] * e2[2], e1[0] * e2[1] - e1[1] * e2[0]};
        const double jac = sqrt(nv[0] * nv[0] + nv[1] * nv[1] + nv[2] * nv[2]);
        if (jac < 1e-15) continue;
        const double en[3] = {nv[0] / jac, nv[1] / jac, nv[2] / jac};
        cplx p_surf[SOL_CHUNK], v_surf[SOL_CHUNK];
        bool has_v[SOL_CHUNK];
#pragma unroll
        for (int c = 0; c < SOL_CHUNK; ++c) {
            const uint64_t at = (uint64_t)(s0 + c) * n + j;
            p_surf[c] = c < cnt ? ps[at] : C(0, 0);
            v_surf[c] = (vs && c < cnt) ? vs[at] : C(0, 0);
            has_v[c] = sqrt(v_surf[c].re * v_surf[c].re + v_surf[c].im * v_surf[c].im) > 1e-15;
        }
        cplx res[SOL_CHUNK];
#pragma unroll
        for (int c = 0; c < SOL_CHUNK; ++c) res[c] = C(0, 0);
#pragma unroll
        for (int q = 0; q < 7; ++q) {
            const double xi = d_tr7[q][0], eta = d_tr7[q][1], wq = d_tr7[q][2] * 0.5;
            const double l0 = 1.0 - xi - eta;
            const double rv[3] = {l0 * c_[0] + xi * c_[3] + eta * c_[6] - x0, l0 * c_[1] + xi * c_[4] + eta * c_[7] - x1,
                                  l0 * c_[2] + xi * c_[5] + eta * c_[8] - x2};
            const double r = sqrt(rv[0] * rv[0] + rv[1] * rv[1] + rv[2] * rv[2]);
            if (r < 1e-15) continue;
            const double vjacwe = jac * wq;
            double sn, cs;
            sincos(wavruim * r, &sn, &cs);
            const double re1 = 4.0 * PI * r;
            const cplx zg = C(cs / re1, sn / re1);
            const cplx zgikr = zg * C(-1.0 / r, wavruim);
            const double drdn = (rv[0] * en[0] + rv[1] * en[1] + rv[2] * en[2]) / r;
            const cplx dgdn = zgikr * drdn;
#pragma unroll
            for (int c = 0; c < SOL_CHUNK; ++c) {
                res[c] += p_surf[c] * dgdn * vjacwe;
                if (has_v[c]) res[c] -= v_surf[c] * zg * vjacwe;
            }
        }
#pragma unroll
        for (int c = 0; c < SOL_CHUNK; ++c) acc[c] += res[c];
    }
    const cplx t = block_sum_chunk(acc, cnt);
    if ((int)threadIdx.x < cnt) out[(uint64_t)(s0 + threadIdx.x) * n_eval + blockIdx.x] = t;
}

// rcs_kernel for solutions [SOL_CHUNK * blockIdx.y, +SOL_CHUNK): sincos(-k c_j.d) and n_j.d once per (element, direction).
__global__ void __launch_bounds__(256, 2)  // (256) alone lets ptxas cap it at 64 registers and spill the accumulators
rcs_batch_kernel(const double* __restrict__ src, const double* __restrict__ area, uint32_t n, const double* __restrict__ dirs,
                 uint32_t n_dirs, uint32_t nsol, const cplx* __restrict__ ps, double k, double* __restrict__ out) {
    const double d0 = dirs[3 * blockIdx.x], d1 = dirs[3 * blockIdx.x + 1], d2 = dirs[3 * blockIdx.x + 2];
    const uint32_t s0 = blockIdx.y * SOL_CHUNK;
    const int cnt = (int)min((uint32_t)SOL_CHUNK, nsol - s0);
    cplx acc[SOL_CHUNK];
#pragma unroll
    for (int c = 0; c < SOL_CHUNK; ++c) acc[c] = C(0, 0);
    for (uint32_t j = threadIdx.x; j < n; j += blockDim.x) {
        const double* c_ = src + 8ull * j;
        const double phase = -k * (c_[0] * d0 + c_[1] * d1 + c_[2] * d2);
        double sn, cs;
        sincos(phase, &sn, &cs);
        const double n_dot_d = c_[3] * d0 + c_[4] * d1 + c_[5] * d2;
        const double a = area[j];
#pragma unroll
        for (int c = 0; c < SOL_CHUNK; ++c) {
            if (c < cnt) {
                const cplx t = ((ps[(uint64_t)(s0 + c) * n + j] * C(cs, sn)) * a) * C(0.0, k);
                acc[c] += t * n_dot_d;
            }
        }
    }
    const cplx t = block_sum_chunk(acc, cnt);
    if ((int)threadIdx.x < cnt) out[(uint64_t)(s0 + threadIdx.x) * n_dirs + blockIdx.x] = 4.0 * 3.14159265358979323846 * (t.re * t.re + t.im * t.im);
}

// ---- far-field amplitude (DESIGN.md section 4.9) -------------------------------------------------------------------------
// F(d) = 1/(4 pi) sum_j [-i w (d.n) p_j - v_j] int_{E_j} exp(-i w d.y) dS_y with w = harmonic_factor * k: the R -> infinity
// limit of R exp(-i w R) p_scat(R d) of the field kernel's representation, over the whole element (Quad4: bilinear map,
// 3 x 3 Gauss-Legendre; Tri3: the field kernel's 7-point rule).  The geometry-only sums a_j(d) = sum_q w_q J_q exp(-i w d.y_q)
// and b_j(d) = sum_q w_q J_q (d.n_q) exp(-i w d.y_q) are formed once per (direction, element) for a chunk of solutions;
// each solution then adds p_j (-i w b_j) - v_j a_j.
constexpr int FF_DIRS = 8;   // directions per block: warp w serves direction FF_DIRS * blockIdx.x + w
constexpr int FF_TILE = 32;  // elements per shared-memory tile: lane e of every warp serves element e of the tile
constexpr int FF_NQ = 9;     // quadrature points per element: 7 (Tri3) or 3 x 3 (Quad4)

// Quadrature point q of the element with gathered coordinates c and type et: position y, weight x Jacobian wj and weight x
// the unnormalised normal of the map, wn = wj n (Tri3: e1 x e2 of the field kernel; Quad4: dy/dxi x dy/deta at the point).
__device__ __forceinline__ void far_field_point(const double* c, int et, int q, double y[3], double& wj, double wn[3]) {
    double nv[3], w;
    if (et == 3) {
        const double xi = d_tr7[q][0], eta = d_tr7[q][1], l0 = 1.0 - xi - eta;
        w = d_tr7[q][2] * 0.5;
        const double e1[3] = {c[3] - c[0], c[4] - c[1], c[5] - c[2]};
        const double e2[3] = {c[6] - c[0], c[7] - c[1], c[8] - c[2]};
        nv[0] = e1[1] * e2[2] - e1[2] * e2[1];
        nv[1] = e1[2] * e2[0] - e1[0] * e2[2];
        nv[2] = e1[0] * e2[1] - e1[1] * e2[0];
        for (int k = 0; k < 3; ++k) y[k] = l0 * c[k] + xi * c[3 + k] + eta * c[6 + k];
    } else {  // nodes at (xi, eta) = (-1,-1), (1,-1), (1,1), (-1,1)
        const double xi = BEMQ_GL3_X[q / 3], eta = BEMQ_GL3_X[q % 3];
        w = BEMQ_GL3_W[q / 3] * BEMQ_GL3_W[q % 3];
        const double n0 = 0.25 * (1.0 - xi) * (1.0 - eta), n1 = 0.25 * (1.0 + xi) * (1.0 - eta);
        const double n2 = 0.25 * (1.0 + xi) * (1.0 + eta), n3 = 0.25 * (1.0 - xi) * (1.0 + eta);
        double dxi[3], deta[3];
        for (int k = 0; k < 3; ++k) {
            y[k] = n0 * c[k] + n1 * c[3 + k] + n2 * c[6 + k] + n3 * c[9 + k];
            dxi[k] = 0.25 * ((1.0 - eta) * (c[3 + k] - c[k]) + (1.0 + eta) * (c[6 + k] - c[9 + k]));
            deta[k] = 0.25 * ((1.0 - xi) * (c[9 + k] - c[k]) + (1.0 + xi) * (c[6 + k] - c[3 + k]));
        }
        nv[0] = dxi[1] * deta[2] - dxi[2] * deta[1];
        nv[1] = dxi[2] * deta[0] - dxi[0] * deta[2];
        nv[2] = dxi[0] * deta[1] - dxi[1] * deta[0];
    }
    wj = sqrt(nv[0] * nv[0] + nv[1] * nv[1] + nv[2] * nv[2]) * w;
    for (int k = 0; k < 3; ++k) wn[k] = nv[k] * w;
}

// Partial far field of elements [per_split * blockIdx.z, +per_split) for solutions [SOL_CHUNK * blockIdx.y, +SOL_CHUNK) and
// directions [FF_DIRS * blockIdx.x, +FF_DIRS): part[z][s][d], without the 1/(4 pi).  The block stages the quadrature points of a
// tile of FF_TILE elements and the chunk's surface values in shared memory; lane e of warp w forms a_j, b_j of (direction w,
// element e).  The lane sums are reduced by a fixed butterfly, so a solution's bits depend neither on nsol nor on its chunk.
__global__ void __launch_bounds__(256)
far_field_kernel(const double* __restrict__ coords, const uint8_t* __restrict__ etype, uint32_t n, uint32_t per_split,
                 const double* __restrict__ dirs, uint32_t n_dirs, uint32_t nsol, const cplx* __restrict__ ps,
                 const cplx* __restrict__ vs, double wavruim, cplx* __restrict__ part) {
    __shared__ double sy[3][FF_NQ * FF_TILE], swj[FF_NQ * FF_TILE], swn[3][FF_NQ * FF_TILE];
    __shared__ cplx sp[SOL_CHUNK][FF_TILE], sv[SOL_CHUNK][FF_TILE];
    __shared__ int snq[FF_TILE];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t dir = blockIdx.x * FF_DIRS + warp;
    const bool dir_ok = dir < n_dirs;
    const double d0 = dir_ok ? dirs[3ull * dir] : 0.0, d1 = dir_ok ? dirs[3ull * dir + 1] : 0.0, d2 = dir_ok ? dirs[3ull * dir + 2] : 0.0;
    const uint32_t s0 = blockIdx.y * SOL_CHUNK;
    const int cnt = (int)min((uint32_t)SOL_CHUNK, nsol - s0);
    const uint32_t j_begin = blockIdx.z * per_split, j_end = min(n, j_begin + per_split);
    cplx acc[SOL_CHUNK];
#pragma unroll
    for (int c = 0; c < SOL_CHUNK; ++c) acc[c] = C(0, 0);
    for (uint32_t t0 = j_begin; t0 < j_end; t0 += FF_TILE) {
        for (int i = threadIdx.x; i < FF_NQ * FF_TILE; i += blockDim.x) {
            const int q = i / FF_TILE, e = i % FF_TILE;
            const uint32_t j = t0 + e;
            double y[3] = {0.0, 0.0, 0.0}, wj = 0.0, wn[3] = {0.0, 0.0, 0.0};
            const int et = j < j_end ? etype[j] : 3;
            if (j < j_end && (et == 4 || q < 7)) far_field_point(coords + 12ull * j, et, q, y, wj, wn);
            if (q == 0) snq[e] = et == 4 ? 9 : 7;
            for (int k = 0; k < 3; ++k) { sy[k][i] = y[k]; swn[k][i] = wn[k]; }
            swj[i] = wj;
        }
        for (int i = threadIdx.x; i < SOL_CHUNK * FF_TILE; i += blockDim.x) {
            const int c = i / FF_TILE, e = i % FF_TILE;
            const uint32_t j = t0 + e;
            const bool ok = c < cnt && j < j_end;
            const uint64_t at = (uint64_t)(s0 + c) * n + j;
            sp[c][e] = ok ? ps[at] : C(0, 0);
            sv[c][e] = (ok && vs) ? vs[at] : C(0, 0);
        }
        __syncthreads();
        if (dir_ok && t0 + lane < j_end) {
            double ar = 0.0, ai = 0.0, br = 0.0, bi = 0.0;
            const int nq = snq[lane];
            for (int q = 0; q < nq; ++q) {
                const int at = q * FF_TILE + lane;
                double sn, cs;
                sincos(-wavruim * (d0 * sy[0][at] + d1 * sy[1][at] + d2 * sy[2][at]), &sn, &cs);
                const double wj = swj[at], dn = d0 * swn[0][at] + d1 * swn[1][at] + d2 * swn[2][at];
                ar += wj * cs;
                ai += wj * sn;
                br += dn * cs;
                bi += dn * sn;
            }
            const cplx a = C(ar, ai), mikb = C(wavruim * bi, -(wavruim * br));  // -i w b
#pragma unroll
            for (int c = 0; c < SOL_CHUNK; ++c) {
                if (c < cnt) {
                    acc[c] += sp[c][lane] * mikb;
                    if (vs) acc[c] -= sv[c][lane] * a;
                }
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int c = 0; c < SOL_CHUNK; ++c) {
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) {
            acc[c].re += __shfl_xor_sync(0xffffffffu, acc[c].re, m);
            acc[c].im += __shfl_xor_sync(0xffffffffu, acc[c].im, m);
        }
    }
    if (lane == 0 && dir_ok) {
        const uint64_t base = (uint64_t)blockIdx.z * nsol;
#pragma unroll
        for (int c = 0; c < SOL_CHUNK; ++c)
            if (c < cnt) part[(base + s0 + c) * n_dirs + dir] = acc[c];
    }
}

// out[s][d] = (sum over the element splits z in order of part[z][s][d]) / (4 pi)
__global__ void far_field_reduce_kernel(const cplx* __restrict__ part, uint32_t nsplit, uint64_t total, cplx* __restrict__ out) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= total) return;
    cplx t = part[i];
    for (uint32_t z = 1; z < nsplit; ++z) t += part[z * total + i];
    out[i] = t / (4.0 * PI);
}

// ---- accurate field evaluation (DESIGN.md section 4.10) ------------------------------------------------------------------
// p_sc(x) = sum_j p_j int_{E_j} dG/dn_y - v_j int_{E_j} G over the whole element (Tri3: the flat triangle; Quad4: the bilinear
// map with its Jacobian and normal, as far_field_point), G = exp(i w r) / (4 pi r).  A (point, element) pair is regular when
// |x - c_e| >= FE_ETA rho_e (c_e: node mean, rho_e: largest centroid-to-node distance) and takes far_field_point's rule.  A
// near pair is split 4 ways in the element's parameter domain until |x - y(sub-centre)| >= FE_ACCEPT sqrt(sub-area); accepted
// pieces take TR13 (Tri3) or 4 x 4 Gauss-Legendre (Quad4).  A piece still refused at depth FE_LMAX means the point lies within
// about 2^-FE_LMAX element sizes of the surface: that pair's integrals are NaN, and so is the point's value for every solution.
constexpr double FE_ETA = 4.0;     // regular pair: |x - c_e|^2 >= FE_ETA^2 rho_e^2
constexpr double FE_ACCEPT = 3.0;  // accepted piece: |x - y(sub-centre)|^2 >= FE_ACCEPT^2 sub-area
constexpr int FE_LMAX = 30;        // subdivision depth limit (2 bits per level of the piece's path fit a uint64)
constexpr int FE_POINTS = 8;       // evaluation points per block of the regular pass: warp w serves point FE_POINTS * blockIdx.x + w

// elem[j] = (node mean, FE_ETA^2 x largest squared centroid-to-node distance) of element j
__global__ void field_element_kernel(const double* __restrict__ coords, const uint8_t* __restrict__ etype, uint32_t n,
                                     double4* __restrict__ elem) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const double* c = coords + 12ull * j;
    const int et = etype[j];
    double m[3];
    for (int k = 0; k < 3; ++k) m[k] = ((et == 4 ? (c[k] + c[3 + k]) + c[6 + k] + c[9 + k] : (c[k] + c[3 + k]) + c[6 + k])) / et;
    double rho2 = 0.0;
    for (int v = 0; v < et; ++v) {
        const double d0 = c[3 * v] - m[0], d1 = c[3 * v + 1] - m[1], d2 = c[3 * v + 2] - m[2];
        rho2 = fmax(rho2, d0 * d0 + d1 * d1 + d2 * d2);
    }
    elem[j] = make_double4(m[0], m[1], m[2], FE_ETA * FE_ETA * rho2);
}

__device__ __forceinline__ bool field_pair_regular(double x0, double x1, double x2, double4 e) {
    const double d0 = x0 - e.x, d1 = x1 - e.y, d2 = x2 - e.z;
    return d0 * d0 + d1 * d1 + d2 * d2 >= e.w;
}

// counts[m] = number of near pairs of point m (one warp per point)
__global__ void field_near_count_kernel(const double4* __restrict__ elem, uint32_t n, const double* __restrict__ eval, uint32_t n_eval,
                                        uint32_t* __restrict__ counts) {
    const uint32_t m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (m >= n_eval) return;
    const double x0 = eval[3ull * m], x1 = eval[3ull * m + 1], x2 = eval[3ull * m + 2];
    uint32_t cnt = 0;
    for (uint32_t j = lane; j < n; j += 32) cnt += field_pair_regular(x0, x1, x2, elem[j]) ? 0u : 1u;
    for (int o = 16; o >= 1; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (lane == 0) counts[m] = cnt;
}

// the near pairs of point m at [off[m], off[m + 1]), elements ascending (one warp per point)
__global__ void field_near_fill_kernel(const double4* __restrict__ elem, uint32_t n, const double* __restrict__ eval, uint32_t n_eval,
                                       const uint64_t* __restrict__ off, uint32_t* __restrict__ pair_pt, uint32_t* __restrict__ pair_el) {
    const uint32_t m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (m >= n_eval) return;
    const double x0 = eval[3ull * m], x1 = eval[3ull * m + 1], x2 = eval[3ull * m + 2];
    uint64_t at = off[m];
    for (uint32_t t0 = 0; t0 < n; t0 += 32) {
        const uint32_t j = t0 + lane;
        const bool near = j < n && !field_pair_regular(x0, x1, x2, elem[j]);
        const uint32_t mask = __ballot_sync(0xffffffffu, near);
        if (near) {
            const uint64_t i = at + __popc(mask & ((1u << lane) - 1u));
            pair_pt[i] = m;
            pair_el[i] = j;
        }
        at += __popc(mask);
    }
}

// Regular pass: partial fields of elements [per_split * blockIdx.z, +per_split) for solutions [SOL_CHUNK * blockIdx.y, +SOL_CHUNK)
// and points [FE_POINTS * blockIdx.x, +FE_POINTS): part[z][s][m].  The layout of far_field_kernel: the block stages a tile's
// quadrature points, element data and the chunk's surface values in shared memory; lane e of warp w forms the geometry-only
// a = sum w J G and b = sum w dG/dn_y of (point w, element e) when the pair is regular, and each solution adds p b - v a.
__global__ void __launch_bounds__(256)
field_regular_kernel(const double* __restrict__ coords, const uint8_t* __restrict__ etype, const double4* __restrict__ elem, uint32_t n,
                     uint32_t per_split, const double* __restrict__ eval, uint32_t n_eval, uint32_t nsol, const cplx* __restrict__ ps,
                     const cplx* __restrict__ vs, double wavruim, cplx* __restrict__ part) {
    __shared__ double sy[3][FF_NQ * FF_TILE], swj[FF_NQ * FF_TILE], swn[3][FF_NQ * FF_TILE];
    __shared__ double4 sel[FF_TILE];
    __shared__ cplx sp[SOL_CHUNK][FF_TILE], sv[SOL_CHUNK][FF_TILE];
    __shared__ int snq[FF_TILE];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t m = blockIdx.x * FE_POINTS + warp;
    const bool pt_ok = m < n_eval;
    const double x0 = pt_ok ? eval[3ull * m] : 0.0, x1 = pt_ok ? eval[3ull * m + 1] : 0.0, x2 = pt_ok ? eval[3ull * m + 2] : 0.0;
    const uint32_t s0 = blockIdx.y * SOL_CHUNK;
    const int cnt = (int)min((uint32_t)SOL_CHUNK, nsol - s0);
    const uint32_t j_begin = blockIdx.z * per_split, j_end = min(n, j_begin + per_split);
    cplx acc[SOL_CHUNK];
#pragma unroll
    for (int c = 0; c < SOL_CHUNK; ++c) acc[c] = C(0, 0);
    for (uint32_t t0 = j_begin; t0 < j_end; t0 += FF_TILE) {
        for (int i = threadIdx.x; i < FF_NQ * FF_TILE; i += blockDim.x) {
            const int q = i / FF_TILE, e = i % FF_TILE;
            const uint32_t j = t0 + e;
            double y[3] = {0.0, 0.0, 0.0}, wj = 0.0, wn[3] = {0.0, 0.0, 0.0};
            const int et = j < j_end ? etype[j] : 3;
            if (j < j_end && (et == 4 || q < 7)) far_field_point(coords + 12ull * j, et, q, y, wj, wn);
            if (q == 0) {
                snq[e] = et == 4 ? 9 : 7;
                sel[e] = j < j_end ? elem[j] : make_double4(0.0, 0.0, 0.0, 0.0);
            }
            for (int k = 0; k < 3; ++k) { sy[k][i] = y[k]; swn[k][i] = wn[k]; }
            swj[i] = wj;
        }
        for (int i = threadIdx.x; i < SOL_CHUNK * FF_TILE; i += blockDim.x) {
            const int c = i / FF_TILE, e = i % FF_TILE;
            const uint32_t j = t0 + e;
            const bool ok = c < cnt && j < j_end;
            const uint64_t at = (uint64_t)(s0 + c) * n + j;
            sp[c][e] = ok ? ps[at] : C(0, 0);
            sv[c][e] = (ok && vs) ? vs[at] : C(0, 0);
        }
        __syncthreads();
        if (pt_ok && t0 + lane < j_end && field_pair_regular(x0, x1, x2, sel[lane])) {
            double ar = 0.0, ai = 0.0, br = 0.0, bi = 0.0;
            const int nq = snq[lane];
            for (int q = 0; q < nq; ++q) {
                const int at = q * FF_TILE + lane;
                const double rv[3] = {sy[0][at] - x0, sy[1][at] - x1, sy[2][at] - x2};
                const double r = sqrt(rv[0] * rv[0] + rv[1] * rv[1] + rv[2] * rv[2]);
                double sn, cs;
                sincos(wavruim * r, &sn, &cs);
                const double re1 = 4.0 * PI * r;
                const cplx zg = C(cs / re1, sn / re1);
                const cplx zgikr = zg * C(-1.0 / r, wavruim);
                const double wj = swj[at], dn = (rv[0] * swn[0][at] + rv[1] * swn[1][at] + rv[2] * swn[2][at]) / r;
                ar += wj * zg.re;
                ai += wj * zg.im;
                br += dn * zgikr.re;
                bi += dn * zgikr.im;
            }
            const cplx a = C(ar, ai), b = C(br, bi);
#pragma unroll
            for (int c = 0; c < SOL_CHUNK; ++c) {
                if (c < cnt) {
                    acc[c] += sp[c][lane] * b;
                    if (vs) acc[c] -= sv[c][lane] * a;
                }
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int c = 0; c < SOL_CHUNK; ++c) {
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) {
            acc[c].re += __shfl_xor_sync(0xffffffffu, acc[c].re, o);
            acc[c].im += __shfl_xor_sync(0xffffffffu, acc[c].im, o);
        }
    }
    if (lane == 0 && pt_ok) {
        const uint64_t base = (uint64_t)blockIdx.z * nsol;
#pragma unroll
        for (int c = 0; c < SOL_CHUNK; ++c)
            if (c < cnt) part[(base + s0 + c) * n_eval + m] = acc[c];
    }
}

// A piece of a near pair: Tri3 -- its vertices in the parameter triangle (u[0..5], (xi, eta) per vertex); Quad4 -- its
// sub-square [u0, u0 + u2] x [u1, u1 + u2] of [-1, 1]^2.  The piece at depth `lvl` is reached from the whole element by the
// children path[2 (l - 1) .. 2 l) of levels l = 1..lvl: Tri3 children are the corner triangles at vertices 0, 1, 2 and the
// centre triangle; Quad4 children the sub-squares (xi low, eta low), (high, low), (low, high), (high, high).  Every parameter
// coordinate is a multiple of 2^-FE_LMAX, so the pieces are exact.
struct FieldPiece {
    double u[6];
    int lvl;
};

__device__ __forceinline__ FieldPiece field_piece(int et, uint64_t path, int lvl) {
    FieldPiece p;
    p.lvl = lvl;
    if (et == 3) {
        double u[6] = {0.0, 0.0, 1.0, 0.0, 0.0, 1.0};
        for (int l = 0; l < lvl; ++l) {
            const int ch = (int)((path >> (2 * l)) & 3u);
            const double m01[2] = {(u[0] + u[2]) / 2, (u[1] + u[3]) / 2}, m12[2] = {(u[2] + u[4]) / 2, (u[3] + u[5]) / 2},
                         m20[2] = {(u[4] + u[0]) / 2, (u[5] + u[1]) / 2};
            if (ch == 0) { u[2] = m01[0]; u[3] = m01[1]; u[4] = m20[0]; u[5] = m20[1]; }
            else if (ch == 1) { u[0] = m01[0]; u[1] = m01[1]; u[4] = m12[0]; u[5] = m12[1]; }
            else if (ch == 2) { u[0] = m20[0]; u[1] = m20[1]; u[2] = m12[0]; u[3] = m12[1]; }
            else { u[0] = m01[0]; u[1] = m01[1]; u[2] = m12[0]; u[3] = m12[1]; u[4] = m20[0]; u[5] = m20[1]; }
        }
        for (int k = 0; k < 6; ++k) p.u[k] = u[k];
    } else {
        double xi0 = -1.0, eta0 = -1.0, h = 2.0;
        for (int l = 0; l < lvl; ++l) {
            const int ch = (int)((path >> (2 * l)) & 3u);
            h *= 0.5;
            if (ch & 1) xi0 += h;
            if (ch & 2) eta0 += h;
        }
        p.u[0] = xi0; p.u[1] = eta0; p.u[2] = h;
        p.u[3] = p.u[4] = p.u[5] = 0.0;
    }
    return p;
}

// position y and N = dy/dxi x dy/deta of the bilinear map at (xi, eta) (far_field_point's expressions)
__device__ __forceinline__ void quad_map(const double* c, double xi, double eta, double y[3], double nv[3]) {
    const double n0 = 0.25 * (1.0 - xi) * (1.0 - eta), n1 = 0.25 * (1.0 + xi) * (1.0 - eta);
    const double n2 = 0.25 * (1.0 + xi) * (1.0 + eta), n3 = 0.25 * (1.0 - xi) * (1.0 + eta);
    double dxi[3], deta[3];
    for (int k = 0; k < 3; ++k) {
        y[k] = n0 * c[k] + n1 * c[3 + k] + n2 * c[6 + k] + n3 * c[9 + k];
        dxi[k] = 0.25 * ((1.0 - eta) * (c[3 + k] - c[k]) + (1.0 + eta) * (c[6 + k] - c[9 + k]));
        deta[k] = 0.25 * ((1.0 - xi) * (c[9 + k] - c[k]) + (1.0 + xi) * (c[6 + k] - c[3 + k]));
    }
    nv[0] = dxi[1] * deta[2] - dxi[2] * deta[1];
    nv[1] = dxi[2] * deta[0] - dxi[0] * deta[2];
    nv[2] = dxi[0] * deta[1] - dxi[1] * deta[0];
}

// Is the piece far enough from x for its rule: |x - y(sub-centre)|^2 >= FE_ACCEPT^2 sub-area (Tri3: area / 4^lvl; Quad4: the
// map's |N| at the sub-centre x side^2, the exact area of a sub-parallelogram)?  tri_area: the Tri3 element's area.
__device__ __forceinline__ bool field_piece_accepted(const double* c, int et, const FieldPiece& p, double tri_area, const double x[3]) {
    double y[3], sub_area;
    if (et == 3) {
        const double a = (p.u[0] + p.u[2] + p.u[4]) / 3.0, b = (p.u[1] + p.u[3] + p.u[5]) / 3.0, l0 = 1.0 - a - b;
        for (int k = 0; k < 3; ++k) y[k] = l0 * c[k] + a * c[3 + k] + b * c[6 + k];
        sub_area = tri_area * ldexp(1.0, -2 * p.lvl);
    } else {
        double nv[3];
        quad_map(c, p.u[0] + 0.5 * p.u[2], p.u[1] + 0.5 * p.u[2], y, nv);
        sub_area = sqrt(nv[0] * nv[0] + nv[1] * nv[1] + nv[2] * nv[2]) * p.u[2] * p.u[2];
    }
    const double d0 = y[0] - x[0], d1 = y[1] - x[1], d2 = y[2] - x[2];
    return d0 * d0 + d1 * d1 + d2 * d2 >= FE_ACCEPT * FE_ACCEPT * sub_area;
}

// Adds quadrature point q (TR13: q < 13; 4 x 4 Gauss: q < 16) of piece p to the lane's (int G, int dG/dn_y) sums.
// en, jac: the Tri3 element's unit normal and |e1 x e2|.
__device__ __forceinline__ void field_piece_point(const double* c, int et, const FieldPiece& p, int q, const double en[3], double jac,
                                                  const double x[3], double wavruim, double& ar, double& ai, double& br, double& bi) {
    double y[3], wj, wn[3];
    if (et == 3) {
        const double xi = BEMQ_TR13[q][0], eta = BEMQ_TR13[q][1];
        const double a = p.u[0] + xi * (p.u[2] - p.u[0]) + eta * (p.u[4] - p.u[0]);
        const double b = p.u[1] + xi * (p.u[3] - p.u[1]) + eta * (p.u[5] - p.u[1]);
        const double l0 = 1.0 - a - b;
        for (int k = 0; k < 3; ++k) y[k] = l0 * c[k] + a * c[3 + k] + b * c[6 + k];
        wj = BEMQ_TR13[q][2] * 0.5 * (jac * ldexp(1.0, -2 * p.lvl));
        for (int k = 0; k < 3; ++k) wn[k] = wj * en[k];
    } else {
        const double g = 0.5 * p.u[2];
        const double w = BEMQ_GL4_W[q >> 2] * BEMQ_GL4_W[q & 3] * g * g;
        double nv[3];
        quad_map(c, p.u[0] + g + g * BEMQ_GL4_X[q >> 2], p.u[1] + g + g * BEMQ_GL4_X[q & 3], y, nv);
        wj = w * sqrt(nv[0] * nv[0] + nv[1] * nv[1] + nv[2] * nv[2]);
        for (int k = 0; k < 3; ++k) wn[k] = w * nv[k];
    }
    const double rv[3] = {y[0] - x[0], y[1] - x[1], y[2] - x[2]};
    const double r = sqrt(rv[0] * rv[0] + rv[1] * rv[1] + rv[2] * rv[2]);
    double sn, cs;
    sincos(wavruim * r, &sn, &cs);
    const double re1 = 4.0 * PI * r;
    const cplx zg = C(cs / re1, sn / re1);
    const cplx zgikr = zg * C(-1.0 / r, wavruim);
    const double dn = (rv[0] * wn[0] + rv[1] * wn[1] + rv[2] * wn[2]) / r;
    ar += wj * zg.re;
    ai += wj * zg.im;
    br += dn * zgikr.re;
    bi += dn * zgikr.im;
}

// Near pass: one warp per near pair i walks the subdivision tree of its element depth first (children in order), every lane
// taking the same decisions, without a stack: the current piece is (path, depth).  Accepted pieces are evaluated two at a time,
// the earlier on lanes 0-15 and the later on lanes 16-31, one quadrature point per lane; a fixed butterfly reduces the lanes.
// ab[i] = (int G, int dG/dn_y) of the pair, NaN when a piece reaches FE_LMAX unaccepted.
__global__ void __launch_bounds__(256)
field_near_kernel(const double* __restrict__ coords, const uint8_t* __restrict__ etype, const double* __restrict__ eval,
                  const uint32_t* __restrict__ pair_pt, const uint32_t* __restrict__ pair_el, uint64_t npairs, double wavruim,
                  cplx* __restrict__ ab) {
    const uint64_t i = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (i >= npairs) return;
    const uint32_t m = pair_pt[i], j = pair_el[i];
    const double x[3] = {eval[3ull * m], eval[3ull * m + 1], eval[3ull * m + 2]};
    double c[12];
    for (int k = 0; k < 12; ++k) c[k] = coords[12ull * j + k];
    const int et = etype[j];
    double en[3] = {0.0, 0.0, 0.0}, jac = 0.0;
    if (et == 3) {
        const double e1[3] = {c[3] - c[0], c[4] - c[1], c[5] - c[2]};
        const double e2[3] = {c[6] - c[0], c[7] - c[1], c[8] - c[2]};
        const double nv[3] = {e1[1] * e2[2] - e1[2] * e2[1], e1[2] * e2[0] - e1[0] * e2[2], e1[0] * e2[1] - e1[1] * e2[0]};
        jac = sqrt(nv[0] * nv[0] + nv[1] * nv[1] + nv[2] * nv[2]);
        for (int k = 0; k < 3; ++k) en[k] = nv[k] / jac;
    }
    const int nq = et == 3 ? 13 : 16;
    const int half = lane >> 4, q = lane & 15;
    double ar = 0.0, ai = 0.0, br = 0.0, bi = 0.0;
    bool failed = false, have_pending = false;
    FieldPiece pending{};
    uint64_t path = 0;
    int lvl = 0;
    for (;;) {
        const FieldPiece cur = field_piece(et, path, lvl);
        if (field_piece_accepted(c, et, cur, 0.5 * jac, x)) {
            if (have_pending) {
                if (q < nq) field_piece_point(c, et, half ? cur : pending, q, en, jac, x, wavruim, ar, ai, br, bi);
                have_pending = false;
            } else {
                pending = cur;
                have_pending = true;
            }
            // next piece: the next sibling, or that of the nearest ancestor that has one
            while (lvl > 0 && ((path >> (2 * (lvl - 1))) & 3u) == 3u) {
                path &= ~(3ull << (2 * (lvl - 1)));
                --lvl;
            }
            if (lvl == 0) break;
            path += 1ull << (2 * (lvl - 1));
        } else if (lvl == FE_LMAX) {
            failed = true;
            break;
        } else {
            ++lvl;  // first child: digit 0
        }
    }
    if (have_pending && !failed && half == 0 && q < nq) field_piece_point(c, et, pending, q, en, jac, x, wavruim, ar, ai, br, bi);
    for (int o = 16; o >= 1; o >>= 1) {
        ar += __shfl_xor_sync(0xffffffffu, ar, o);
        ai += __shfl_xor_sync(0xffffffffu, ai, o);
        br += __shfl_xor_sync(0xffffffffu, br, o);
        bi += __shfl_xor_sync(0xffffffffu, bi, o);
    }
    if (lane == 0) {
        const double nan = __longlong_as_double(0x7ff8000000000000ll);
        ab[2 * i] = failed ? C(nan, nan) : C(ar, ai);
        ab[2 * i + 1] = failed ? C(nan, nan) : C(br, bi);
    }
}

// out[s][m] = (sum over the element splits z in order of part[z][s][m]) + sum over the near pairs of m in list order of
// p_j int dG/dn_y - v_j int G
__global__ void field_combine_kernel(const cplx* __restrict__ part, uint32_t nsplit, uint32_t nsol, uint32_t n_eval, uint32_t n,
                                     const uint64_t* __restrict__ off, const uint32_t* __restrict__ pair_el, const cplx* __restrict__ ab,
                                     const cplx* __restrict__ ps, const cplx* __restrict__ vs, cplx* __restrict__ out) {
    const uint64_t total = (uint64_t)nsol * n_eval;
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= total) return;
    const uint64_t s = i / n_eval, m = i % n_eval;
    cplx t = part[i];
    for (uint32_t z = 1; z < nsplit; ++z) t += part[z * total + i];
    for (uint64_t k = off[m]; k < off[m + 1]; ++k) {
        const uint64_t at = s * n + pair_el[k];
        t += ps[at] * ab[2 * k + 1];
        if (vs) t -= vs[at] * ab[2 * k];
    }
    out[i] = t;
}

// b[s] = sys + inc[s] for the nrhs columns of a block (in place: out may be inc), the one IEEE add of bemb200_sweep_next
__global__ void add_system_rhs_kernel(const cplx* __restrict__ sys, const cplx* inc, uint64_t n, uint64_t total, cplx* out) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x)
        out[i] = sys[i % n] + inc[i];
}

}  // namespace

cudaError_t bemb::launch_add_system_rhs(const cplx* sys, const cplx* inc, uint64_t n, uint32_t nrhs, cplx* out, cudaStream_t s) {
    const uint64_t total = n * nrhs;
    if (total == 0) return cudaSuccess;
    const uint64_t blocks = (total + 255) / 256;
    add_system_rhs_kernel<<<(unsigned)(blocks < 148 * 16 ? blocks : 148 * 16), 256, 0, s>>>(sys, inc, n, total, out);
    return cudaGetLastError();
}

// true when p is device (or managed) memory of `device`
bool bemb::device_ptr_on(int device, const void* p) {
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) && a.device == device;
}

extern "C" int bemb200_incident_rhs(const bemb200_staged_mesh* sm, const bemb200_physics* phys, double beta_re, double beta_im,
                                    uint32_t n_sources, const int32_t* kinds, const double* vecs, const double* amps,
                                    double* rhs_host, double* rhs_dev) {
    if (!sm || !phys || !kinds || !vecs || !amps || (!rhs_host && !rhs_dev)) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    bemb200_ctx* ctx = sm->ctx;
    if (n_sources == 0 || n_sources > 4096) return set_error(ctx, BEMB200_EINVAL, "need 1..4096 sources");
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint32_t n = sm->dm.n;
    std::vector<Source> hs(n_sources);
    for (uint32_t s = 0; s < n_sources; ++s) {
        if (kinds[s] != 0 && kinds[s] != 1) return set_error(ctx, BEMB200_EINVAL, "source kind must be 0 (plane wave) or 1 (point source)");
        hs[s].kind = kinds[s];
        for (int d = 0; d < 3; ++d) hs[s].v[d] = vecs[3 * s + d];
        hs[s].amp = C(amps[2 * s], amps[2 * s + 1]);
    }
    Source* dsrc = nullptr;
    cplx* dout = (cplx*)rhs_dev;
    cplx* tmp = nullptr;
    BEMB_CUDA(ctx, cudaMallocAsync((void**)&dsrc, n_sources * sizeof(Source), ctx->stream));
    if (!dout) {
        BEMB_CUDA(ctx, cudaMallocAsync((void**)&tmp, (size_t)n * sizeof(cplx), ctx->stream));
        dout = tmp;
    }
    cudaError_t e = cudaMemcpyAsync(dsrc, hs.data(), n_sources * sizeof(Source), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) {
        incident_rhs_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(sm->dm.src, n, dsrc, (int)n_sources, phys->wave_number, phys->gamma,
                                                                      phys->tau, C(beta_re, beta_im), dout);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess && rhs_host) e = cudaMemcpyAsync(rhs_host, dout, (size_t)n * sizeof(cplx), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFreeAsync(dsrc, ctx->stream);
    if (tmp) cudaFreeAsync(tmp, ctx->stream);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "incident_rhs");
    return BEMB200_OK;
}

extern "C" int bemb200_scattered_field(const bemb200_staged_mesh* sm, const bemb200_physics* phys, uint64_t n_eval, const double* eval_pts,
                                       const double* surface_pressure, const double* surface_velocity, double* out) {
    if (!sm || !phys || !eval_pts || !surface_pressure || !out) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    bemb200_ctx* ctx = sm->ctx;
    if (n_eval == 0) return BEMB200_OK;
    if (n_eval > 0x7fffffffull) return set_error(ctx, BEMB200_EINVAL, "too many evaluation points");
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint32_t n = sm->dm.n;
    double* dev = nullptr;
    cplx *dps = nullptr, *dvs = nullptr, *dout = nullptr;
    cudaStream_t s = ctx->stream;
    BEMB_CUDA(ctx, cudaMallocAsync((void**)&dev, n_eval * 3 * sizeof(double), s));
    BEMB_CUDA(ctx, cudaMallocAsync((void**)&dps, (size_t)n * sizeof(cplx), s));
    BEMB_CUDA(ctx, cudaMallocAsync((void**)&dout, n_eval * sizeof(cplx), s));
    if (surface_velocity) BEMB_CUDA(ctx, cudaMallocAsync((void**)&dvs, (size_t)n * sizeof(cplx), s));
    cudaError_t e = cudaMemcpyAsync(dev, eval_pts, n_eval * 3 * sizeof(double), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dps, surface_pressure, (size_t)n * sizeof(cplx), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess && dvs) e = cudaMemcpyAsync(dvs, surface_velocity, (size_t)n * sizeof(cplx), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) {
        scattered_field_kernel<<<(unsigned)n_eval, 256, 0, s>>>(sm->dm.coords, n, dev, dps, dvs, phys->wave_number * phys->harmonic_factor, dout);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, dout, n_eval * sizeof(cplx), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    cudaFreeAsync(dev, s); cudaFreeAsync(dps, s); cudaFreeAsync(dout, s);
    if (dvs) cudaFreeAsync(dvs, s);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "scattered_field");
    return BEMB200_OK;
}

extern "C" int bemb200_compute_rcs(const bemb200_staged_mesh* sm, const bemb200_physics* phys, uint32_t n_dirs, const double* dirs,
                                   const double* surface_pressure, double* rcs_out) {
    if (!sm || !phys || !dirs || !surface_pressure || !rcs_out) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    bemb200_ctx* ctx = sm->ctx;
    if (n_dirs == 0) return BEMB200_OK;
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint32_t n = sm->dm.n;
    double *ddirs = nullptr, *dout = nullptr;
    cplx* dps = nullptr;
    cudaStream_t s = ctx->stream;
    BEMB_CUDA(ctx, cudaMallocAsync((void**)&ddirs, (size_t)n_dirs * 3 * sizeof(double), s));
    BEMB_CUDA(ctx, cudaMallocAsync((void**)&dout, (size_t)n_dirs * sizeof(double), s));
    BEMB_CUDA(ctx, cudaMallocAsync((void**)&dps, (size_t)(n ? n : 1) * sizeof(cplx), s));
    cudaError_t e = cudaMemcpyAsync(ddirs, dirs, (size_t)n_dirs * 3 * sizeof(double), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess && n) e = cudaMemcpyAsync(dps, surface_pressure, (size_t)n * sizeof(cplx), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) {
        rcs_kernel<<<n_dirs, 256, 0, s>>>(sm->dm.src, sm->dm.area, n, ddirs, dps, phys->wave_number, dout);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(rcs_out, dout, (size_t)n_dirs * sizeof(double), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    cudaFreeAsync(ddirs, s); cudaFreeAsync(dout, s); cudaFreeAsync(dps, s);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "compute_rcs");
    return BEMB200_OK;
}

namespace {

// Surface values of nsol solutions ([nsol][n] complex128, DOF order) on the device: the caller's device array, or an upload of
// the host array into *tmp.
cudaError_t solutions_on_device(const double* values, int on_device, size_t count, cudaStream_t s, cplx** tmp, const cplx** out) {
    if (on_device) {
        *out = (const cplx*)values;
        return cudaSuccess;
    }
    cudaError_t e = cudaMallocAsync((void**)tmp, (count ? count : 1) * sizeof(cplx), s);
    if (e == cudaSuccess && count) e = cudaMemcpyAsync(*tmp, values, count * sizeof(cplx), cudaMemcpyHostToDevice, s);
    *out = *tmp;
    return e;
}

}  // namespace

extern "C" int bemb200_incident_rhs_batch(const bemb200_staged_mesh* sm, const bemb200_physics* phys, double beta_re, double beta_im,
                                          uint32_t nrhs, const uint32_t* src_ptr, const int32_t* kinds, const double* vecs,
                                          const double* amps, const bemb200_matrix* system, double* b_host, double* b_dev) {
    if (!sm || !phys || !src_ptr || !kinds || !vecs || !amps || (!b_host && !b_dev)) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    bemb200_ctx* ctx = sm->ctx;
    if (nrhs == 0 || nrhs > 4096) return set_error(ctx, BEMB200_EINVAL, "need 1..4096 right-hand sides");
    if (src_ptr[0] != 0) return set_error(ctx, BEMB200_EINVAL, "src_ptr[0] must be 0");
    for (uint32_t s = 0; s < nrhs; ++s)
        if (src_ptr[s + 1] < src_ptr[s]) return set_error(ctx, BEMB200_EINVAL, "src_ptr must be non-decreasing");
    const uint32_t n_sources = src_ptr[nrhs];
    if (n_sources > 65536) return set_error(ctx, BEMB200_EINVAL, "at most 65536 sources in all");
    for (uint32_t s = 0; s < n_sources; ++s)
        if (kinds[s] != 0 && kinds[s] != 1) return set_error(ctx, BEMB200_EINVAL, "source kind must be 0 (plane wave) or 1 (point source)");
    const uint32_t n = sm->dm.n;
    if (system) {
        if (system->n_rows != n || system->n_cols != n) return set_error(ctx, BEMB200_EINVAL, "system does not match the staged mesh");
        if (system->ctx->device != ctx->device) return set_error(ctx, BEMB200_EINVAL, "system lives on another device than the staged mesh");
    }
    if (b_dev && !device_ptr_on(ctx->device, b_dev)) return set_error(ctx, BEMB200_EINVAL, "b_dev is not device memory of the staged mesh's device");
    std::vector<Source> hs(n_sources ? n_sources : 1);
    for (uint32_t s = 0; s < n_sources; ++s) {
        hs[s].kind = kinds[s];
        for (int d = 0; d < 3; ++d) hs[s].v[d] = vecs[3 * s + d];
        hs[s].amp = C(amps[2 * s], amps[2 * s + 1]);
    }
    // TbemSystem.rhs of every row, gathered as bemb200_rhs_download_full gathers it (collective on a row-sharded operator)
    struct DevMem {
        cudaStream_t s;
        void* p = nullptr;
        ~DevMem() { if (p) cudaFreeAsync(p, s); }  // after the kernel on the staged mesh's stream
    } sys{ctx->stream};
    if (system) {
        BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
        BEMB_CUDA(ctx, cudaMallocAsync(&sys.p, (size_t)(n ? n : 1) * sizeof(cplx), ctx->stream));
        BEMB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // the system's stream writes it next
        int rc = rhs_full(const_cast<bemb200_matrix*>(system), (double*)sys.p, cudaMemcpyDeviceToDevice);
        if (rc != BEMB200_OK) return set_error(ctx, rc, bemb200_last_error(system->ctx));
    }
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t total = (size_t)nrhs * n;
    cudaStream_t st = ctx->stream;
    Source* dsrc = nullptr;
    uint32_t* dgrp = nullptr;
    cplx* dout = (cplx*)b_dev;
    cplx* tmp = nullptr;
    BEMB_CUDA(ctx, cudaMallocAsync((void**)&dsrc, hs.size() * sizeof(Source), st));
    BEMB_CUDA(ctx, cudaMallocAsync((void**)&dgrp, (nrhs + 1) * sizeof(uint32_t), st));
    if (!dout) {
        BEMB_CUDA(ctx, cudaMallocAsync((void**)&tmp, (total ? total : 1) * sizeof(cplx), st));
        dout = tmp;
    }
    cudaError_t e = cudaMemcpyAsync(dsrc, hs.data(), hs.size() * sizeof(Source), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dgrp, src_ptr, (nrhs + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && n) {
        incident_rhs_batch_kernel<<<dim3((n + 255) / 256, nrhs), 256, 0, st>>>(sm->dm.src, n, dsrc, dgrp, phys->wave_number, phys->gamma,
                                                                            phys->tau, C(beta_re, beta_im), (const cplx*)sys.p, dout);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess && b_host && total) e = cudaMemcpyAsync(b_host, dout, total * sizeof(cplx), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFreeAsync(dsrc, st);
    cudaFreeAsync(dgrp, st);
    if (tmp) cudaFreeAsync(tmp, st);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "incident_rhs_batch");
    return BEMB200_OK;
}

extern "C" int bemb200_compute_rcs_batch(const bemb200_staged_mesh* sm, const bemb200_physics* phys, uint32_t nsol,
                                         const double* surface_pressure, int on_device, uint32_t n_dirs, const double* dirs,
                                         double* rcs_out) {
    if (!sm || !phys || !surface_pressure || !dirs || !rcs_out) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    bemb200_ctx* ctx = sm->ctx;
    if (nsol == 0 || nsol > 4096) return set_error(ctx, BEMB200_EINVAL, "need 1..4096 solutions");
    if (on_device != 0 && on_device != 1) return set_error(ctx, BEMB200_EINVAL, "on_device must be 0 (host arrays) or 1 (device arrays)");
    if (n_dirs > 0x7fffffffu) return set_error(ctx, BEMB200_EINVAL, "too many directions");
    if (on_device && !device_ptr_on(ctx->device, surface_pressure))
        return set_error(ctx, BEMB200_EINVAL, "surface_pressure is not device memory of the staged mesh's device");
    if (n_dirs == 0) return BEMB200_OK;
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint32_t n = sm->dm.n;
    const size_t nout = (size_t)nsol * n_dirs;
    double *ddirs = nullptr, *dout = nullptr;
    cplx* tmp = nullptr;
    const cplx* dps = nullptr;
    cudaStream_t s = ctx->stream;
    BEMB_CUDA(ctx, cudaMallocAsync((void**)&ddirs, (size_t)n_dirs * 3 * sizeof(double), s));
    BEMB_CUDA(ctx, cudaMallocAsync((void**)&dout, nout * sizeof(double), s));
    cudaError_t e = solutions_on_device(surface_pressure, on_device, (size_t)nsol * n, s, &tmp, &dps);
    if (e == cudaSuccess) e = cudaMemcpyAsync(ddirs, dirs, (size_t)n_dirs * 3 * sizeof(double), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) {
        rcs_batch_kernel<<<dim3(n_dirs, (nsol + SOL_CHUNK - 1) / SOL_CHUNK), 256, 0, s>>>(sm->dm.src, sm->dm.area, n, ddirs, n_dirs, nsol,
                                                                                         dps, phys->wave_number, dout);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(rcs_out, dout, nout * sizeof(double), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    cudaFreeAsync(ddirs, s); cudaFreeAsync(dout, s);
    if (tmp) cudaFreeAsync(tmp, s);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "compute_rcs_batch");
    return BEMB200_OK;
}

extern "C" int bemb200_scattered_field_batch(const bemb200_staged_mesh* sm, const bemb200_physics* phys, uint32_t nsol,
                                             const double* surface_pressure, const double* surface_velocity, int on_device,
                                             uint64_t n_eval, const double* eval_pts, double* out) {
    if (!sm || !phys || !surface_pressure || !eval_pts || !out) return set_error(nullptr, BEMB200_EINVAL, "NULL argument");
    bemb200_ctx* ctx = sm->ctx;
    if (nsol == 0 || nsol > 4096) return set_error(ctx, BEMB200_EINVAL, "need 1..4096 solutions");
    if (on_device != 0 && on_device != 1) return set_error(ctx, BEMB200_EINVAL, "on_device must be 0 (host arrays) or 1 (device arrays)");
    if (n_eval > 0x7fffffffull) return set_error(ctx, BEMB200_EINVAL, "too many evaluation points");
    if (on_device && (!device_ptr_on(ctx->device, surface_pressure) || (surface_velocity && !device_ptr_on(ctx->device, surface_velocity))))
        return set_error(ctx, BEMB200_EINVAL, "surface values are not device memory of the staged mesh's device");
    if (n_eval == 0) return BEMB200_OK;
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint32_t n = sm->dm.n;
    const size_t nout = (size_t)nsol * n_eval;
    double* dev = nullptr;
    cplx *dout = nullptr, *tmp_p = nullptr, *tmp_v = nullptr;
    const cplx *dps = nullptr, *dvs = nullptr;
    cudaStream_t s = ctx->stream;
    BEMB_CUDA(ctx, cudaMallocAsync((void**)&dev, n_eval * 3 * sizeof(double), s));
    BEMB_CUDA(ctx, cudaMallocAsync((void**)&dout, nout * sizeof(cplx), s));
    cudaError_t e = solutions_on_device(surface_pressure, on_device, (size_t)nsol * n, s, &tmp_p, &dps);
    if (e == cudaSuccess && surface_velocity) e = solutions_on_device(surface_velocity, on_device, (size_t)nsol * n, s, &tmp_v, &dvs);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dev, eval_pts, n_eval * 3 * sizeof(double), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) {
        scattered_field_batch_kernel<<<dim3((unsigned)n_eval, (nsol + SOL_CHUNK - 1) / SOL_CHUNK), 256, 0, s>>>(
            sm->dm.coords, n, dev, (uint32_t)n_eval, nsol, dps, dvs, phys->wave_number * phys->harmonic_factor, dout);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, dout, nout * sizeof(cplx), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    cudaFreeAsync(dev, s); cudaFreeAsync(dout, s);
    if (tmp_p) cudaFreeAsync(tmp_p, s);
    if (tmp_v) cudaFreeAsync(tmp_v, s);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "scattered_field_batch");
    return BEMB200_OK;
}

extern "C" int bemb200_far_field(const bemb200_staged_mesh* sm, const bemb200_physics* phys, uint32_t nsol, const double* surface_pressure,
                                 const double* surface_velocity, int on_device, uint32_t n_dirs, const double* dirs, double* out) {
    // every argument is checked before a device is touched (the staged mesh last, so each check answers for itself)
    bemb200_ctx* ctx = sm ? sm->ctx : nullptr;
    if (!phys || !surface_pressure || !dirs || !out) return set_error(ctx, BEMB200_EINVAL, "NULL argument");
    if (nsol == 0 || nsol > 4096) return set_error(ctx, BEMB200_EINVAL, "need 1..4096 solutions");
    if (on_device != 0 && on_device != 1) return set_error(ctx, BEMB200_EINVAL, "on_device must be 0 (host arrays) or 1 (device arrays)");
    if (n_dirs == 0 || n_dirs > 0x7fffffffu) return set_error(ctx, BEMB200_EINVAL, "need 1..2^31-1 directions");
    for (uint32_t d = 0; d < n_dirs; ++d) {
        const double x = dirs[3ull * d], y = dirs[3ull * d + 1], z = dirs[3ull * d + 2];
        const double len = std::sqrt(x * x + y * y + z * z);
        if (!std::isfinite(x) || !std::isfinite(y) || !std::isfinite(z) || !(std::fabs(len - 1.0) <= 1e-9))
            return set_error(ctx, BEMB200_EINVAL, "direction " + std::to_string(d) + " is not a finite unit vector (|d| - 1 within 1e-9)");
    }
    if (!sm) return set_error(nullptr, BEMB200_EINVAL, "NULL staged mesh");
    if (on_device && (!device_ptr_on(ctx->device, surface_pressure) || (surface_velocity && !device_ptr_on(ctx->device, surface_velocity))))
        return set_error(ctx, BEMB200_EINVAL, "surface values are not device memory of the staged mesh's device");
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint32_t n = sm->dm.n;
    // Split the elements (at most 32 ways) so that about 1184 blocks (four waves of two 256-thread blocks per SM of a B200)
    // serve one chunk of solutions when there are few directions.  The split depends on n_dirs and n only, so a solution's bits do not depend on nsol.
    const uint32_t dir_blocks = (n_dirs + FF_DIRS - 1) / FF_DIRS, tiles = (n + FF_TILE - 1) / FF_TILE;
    uint32_t nsplit = (1184u + dir_blocks - 1) / dir_blocks;
    nsplit = std::max(1u, std::min({nsplit, 32u, tiles}));
    const uint32_t per_split = (tiles + nsplit - 1) / nsplit * FF_TILE;
    nsplit = (n + per_split - 1) / per_split;
    const size_t nout = (size_t)nsol * n_dirs;
    double* ddirs = nullptr;
    cplx *part = nullptr, *dout = nullptr, *tmp_p = nullptr, *tmp_v = nullptr;
    const cplx *dps = nullptr, *dvs = nullptr;
    cudaStream_t s = ctx->stream;
    BEMB_CUDA(ctx, cudaMallocAsync((void**)&ddirs, (size_t)n_dirs * 3 * sizeof(double), s));
    BEMB_CUDA(ctx, cudaMallocAsync((void**)&part, nout * nsplit * sizeof(cplx), s));
    BEMB_CUDA(ctx, cudaMallocAsync((void**)&dout, nout * sizeof(cplx), s));
    cudaError_t e = solutions_on_device(surface_pressure, on_device, (size_t)nsol * n, s, &tmp_p, &dps);
    if (e == cudaSuccess && surface_velocity) e = solutions_on_device(surface_velocity, on_device, (size_t)nsol * n, s, &tmp_v, &dvs);
    if (e == cudaSuccess) e = cudaMemcpyAsync(ddirs, dirs, (size_t)n_dirs * 3 * sizeof(double), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) {
        far_field_kernel<<<dim3(dir_blocks, (nsol + SOL_CHUNK - 1) / SOL_CHUNK, nsplit), 256, 0, s>>>(
            sm->dm.coords, sm->dm.etype, n, per_split, ddirs, n_dirs, nsol, dps, dvs, phys->wave_number * phys->harmonic_factor, part);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) {
        far_field_reduce_kernel<<<(unsigned)((nout + 255) / 256), 256, 0, s>>>(part, nsplit, nout, dout);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, dout, nout * sizeof(cplx), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    cudaFreeAsync(ddirs, s); cudaFreeAsync(part, s); cudaFreeAsync(dout, s);
    if (tmp_p) cudaFreeAsync(tmp_p, s);
    if (tmp_v) cudaFreeAsync(tmp_v, s);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "far_field");
    return BEMB200_OK;
}

extern "C" int bemb200_evaluate_field(const bemb200_staged_mesh* sm, const bemb200_physics* phys, uint32_t nsol, const double* surface_pressure,
                                      const double* surface_velocity, int on_device, uint64_t n_eval, const double* eval_pts, double* out) {
    // every argument is checked before a device is touched (the staged mesh last, so each check answers for itself)
    bemb200_ctx* ctx = sm ? sm->ctx : nullptr;
    if (!phys || !surface_pressure || !eval_pts || !out) return set_error(ctx, BEMB200_EINVAL, "NULL argument");
    if (nsol == 0 || nsol > 4096) return set_error(ctx, BEMB200_EINVAL, "need 1..4096 solutions");
    if (on_device != 0 && on_device != 1) return set_error(ctx, BEMB200_EINVAL, "on_device must be 0 (host arrays) or 1 (device arrays)");
    if (n_eval == 0 || n_eval > 0x7fffffffull) return set_error(ctx, BEMB200_EINVAL, "need 1..2^31-1 evaluation points");
    for (uint64_t m = 0; m < 3 * n_eval; ++m)
        if (!std::isfinite(eval_pts[m])) return set_error(ctx, BEMB200_EINVAL, "evaluation point " + std::to_string(m / 3) + " is not finite");
    if (!sm) return set_error(nullptr, BEMB200_EINVAL, "NULL staged mesh");
    if (on_device && (!device_ptr_on(ctx->device, surface_pressure) || (surface_velocity && !device_ptr_on(ctx->device, surface_velocity))))
        return set_error(ctx, BEMB200_EINVAL, "surface values are not device memory of the staged mesh's device");
    std::lock_guard<std::mutex> lk(ctx->mu);
    BEMB_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint32_t n = sm->dm.n, ne = (uint32_t)n_eval;
    const double wavruim = phys->wave_number * phys->harmonic_factor;
    cudaStream_t s = ctx->stream;
    struct Allocs {  // stream-ordered frees after the last kernel, on every return path
        cudaStream_t s;
        std::vector<void*> p;
        cudaError_t get(void** out, size_t bytes) {
            cudaError_t e = cudaMallocAsync(out, bytes ? bytes : 1, s);
            if (e == cudaSuccess) p.push_back(*out);
            return e;
        }
        ~Allocs() { for (void* q : p) cudaFreeAsync(q, s); }
    } mem{s, {}};
    // The regular pass splits the elements as far_field does (depending on n_eval and n only, so a solution's bits do not
    // depend on nsol).
    const uint32_t pt_blocks = (ne + FE_POINTS - 1) / FE_POINTS, tiles = (n + FF_TILE - 1) / FF_TILE;
    uint32_t nsplit = (1184u + pt_blocks - 1) / pt_blocks;
    nsplit = std::max(1u, std::min({nsplit, 32u, tiles}));
    const uint32_t per_split = std::max(1u, (tiles + nsplit - 1) / nsplit) * FF_TILE;
    nsplit = std::max(1u, (n + per_split - 1) / per_split);
    const size_t nout = (size_t)nsol * ne;
    double *dev = nullptr;
    double4* elem = nullptr;
    uint32_t* counts = nullptr;
    cplx *part = nullptr, *dout = nullptr, *tmp_p = nullptr, *tmp_v = nullptr;
    const cplx *dps = nullptr, *dvs = nullptr;
    cudaError_t e = mem.get((void**)&dev, (size_t)ne * 3 * sizeof(double));
    if (e == cudaSuccess) e = mem.get((void**)&elem, (size_t)n * sizeof(double4));
    if (e == cudaSuccess) e = mem.get((void**)&counts, (size_t)ne * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMemcpyAsync(dev, eval_pts, (size_t)ne * 3 * sizeof(double), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess && n) {
        field_element_kernel<<<(n + 255) / 256, 256, 0, s>>>(sm->dm.coords, sm->dm.etype, n, elem);
        e = cudaGetLastError();
    }
    const unsigned warp_blocks = (unsigned)(((uint64_t)ne * 32 + 255) / 256);
    if (e == cudaSuccess) {
        field_near_count_kernel<<<warp_blocks, 256, 0, s>>>(elem, n, dev, ne, counts);
        e = cudaGetLastError();
    }
    // near list sized exactly: counts -> host prefix sum -> offsets
    std::vector<uint32_t> hcount(ne);
    std::vector<uint64_t> hoff((size_t)ne + 1, 0);
    if (e == cudaSuccess) e = cudaMemcpyAsync(hcount.data(), counts, (size_t)ne * sizeof(uint32_t), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "evaluate_field (near count)");
    for (uint32_t m = 0; m < ne; ++m) hoff[m + 1] = hoff[m] + hcount[m];
    const uint64_t npairs = hoff[ne];
    uint64_t* off = nullptr;
    uint32_t *pair_pt = nullptr, *pair_el = nullptr;
    cplx* ab = nullptr;
    e = mem.get((void**)&off, hoff.size() * sizeof(uint64_t));
    if (e == cudaSuccess) e = mem.get((void**)&pair_pt, npairs * sizeof(uint32_t));
    if (e == cudaSuccess) e = mem.get((void**)&pair_el, npairs * sizeof(uint32_t));
    if (e == cudaSuccess) e = mem.get((void**)&ab, 2 * npairs * sizeof(cplx));
    if (e == cudaSuccess) e = mem.get((void**)&part, nout * nsplit * sizeof(cplx));
    if (e == cudaSuccess) e = mem.get((void**)&dout, nout * sizeof(cplx));
    if (e == cudaSuccess) e = cudaMemcpyAsync(off, hoff.data(), hoff.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess && npairs) {
        field_near_fill_kernel<<<warp_blocks, 256, 0, s>>>(elem, n, dev, ne, off, pair_pt, pair_el);
        e = cudaGetLastError();
        if (e == cudaSuccess) {
            field_near_kernel<<<(unsigned)((npairs * 32 + 255) / 256), 256, 0, s>>>(sm->dm.coords, sm->dm.etype, dev, pair_pt, pair_el,
                                                                                  npairs, wavruim, ab);
            e = cudaGetLastError();
        }
    }
    if (e == cudaSuccess) {
        e = solutions_on_device(surface_pressure, on_device, (size_t)nsol * n, s, &tmp_p, &dps);
        if (tmp_p) mem.p.push_back(tmp_p);
    }
    if (e == cudaSuccess && surface_velocity) {
        e = solutions_on_device(surface_velocity, on_device, (size_t)nsol * n, s, &tmp_v, &dvs);
        if (tmp_v) mem.p.push_back(tmp_v);
    }
    if (e == cudaSuccess) {
        field_regular_kernel<<<dim3(pt_blocks, (nsol + SOL_CHUNK - 1) / SOL_CHUNK, nsplit), 256, 0, s>>>(
            sm->dm.coords, sm->dm.etype, elem, n, per_split, dev, ne, nsol, dps, dvs, wavruim, part);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) {
        field_combine_kernel<<<(unsigned)((nout + 255) / 256), 256, 0, s>>>(part, nsplit, nsol, ne, n, off, pair_el, ab, dps, dvs, dout);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, dout, nout * sizeof(cplx), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "evaluate_field");
    return BEMB200_OK;
}
