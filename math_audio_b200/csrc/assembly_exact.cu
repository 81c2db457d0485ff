// assembly_exact.cu -- prep, near-field (adaptive subdivision) and self-element kernels.
//
// Compiled with -fmad=false: these kernels take the reference's data-dependent
// DECISIONS (the strict `<` of the subdivision ratio test, the for_ka class
// thresholds), so every expression that feeds a decision is evaluated in the
// reference's operation order with IEEE add/mul/div/sqrt and no FMA contraction.
//
// Reference (paths relative to /root/reference/math-bem/src/core/):
//   integration/regular.rs:33-260   regular_integration + compute_parameters
//   integration/singular.rs:123-465 singular_integration(_with_params)
//   integration/singular.rs:497-721 generate_subelements, local_to_global
//   assembly/tbem.rs:273-345        add_free_terms, assemble_tbem
//
// Mapping: one WARP per (collocation row, field element) pair.  The candidate
// sub-elements of one refinement level are tested one per lane; ballots rebuild
// the reference's sequential scan order (including its `ndie > 15` early break
// and the 110-output cap); quadrature points of all accepted sub-elements are
// then spread over the lanes and reduced with warp shuffles.
#include "internal.h"

namespace bemb {

namespace {

constexpr int WARPS_PER_BLOCK = 2;
constexpr int MAX_NSE = 60;
constexpr int MAX_SUB = 110;

__device__ __constant__ double d_CSI6[6] = {0.0, 1.0, 0.0, 0.5, 0.5, 0.0};
__device__ __constant__ double d_ETA6[6] = {0.0, 0.0, 1.0, 0.0, 0.5, 0.5};
__device__ __constant__ double d_CSI8[8] = {1.0, -1.0, -1.0, 1.0, 0.0, -1.0, 0.0, 1.0};
__device__ __constant__ double d_ETA8[8] = {1.0, 1.0, -1.0, -1.0, 1.0, 0.0, -1.0, 0.0};

struct Params {
    double shape[4];
    double jac;
    double nrm[3];
    double pos[3];
};

__device__ __forceinline__ double dot3(const double* a, const double* b) {
    double s = 0.0;
    s = s + a[0] * b[0];
    s = s + a[1] * b[1];
    s = s + a[2] * b[2];
    return s;
}

// regular.rs:193-260 / singular.rs:398-465
__device__ __forceinline__ Params compute_parameters(const double* c, int et, double s, double t) {
    Params p;
    double ds[4], dt[4];
    if (et == 3) {
        p.shape[0] = 1.0 - s - t; p.shape[1] = s; p.shape[2] = t; p.shape[3] = 0.0;
        ds[0] = -1.0; ds[1] = 1.0; ds[2] = 0.0; ds[3] = 0.0;
        dt[0] = -1.0; dt[1] = 0.0; dt[2] = 1.0; dt[3] = 0.0;
    } else {
        double s1 = 0.25 * (s + 1.0), s2 = 0.25 * (s - 1.0), t1 = t + 1.0, t2 = t - 1.0;
        p.shape[0] = s1 * t1; p.shape[1] = -s2 * t1; p.shape[2] = s2 * t2; p.shape[3] = -s1 * t2;
        ds[0] = 0.25 * (t + 1.0); ds[1] = -0.25 * (t + 1.0); ds[2] = 0.25 * (t - 1.0); ds[3] = -0.25 * (t - 1.0);
        dt[0] = 0.25 * (s + 1.0); dt[1] = 0.25 * (1.0 - s); dt[2] = 0.25 * (s - 1.0); dt[3] = -0.25 * (s + 1.0);
    }
    double dxds[3] = {0, 0, 0}, dxdt[3] = {0, 0, 0};
    p.pos[0] = p.pos[1] = p.pos[2] = 0.0;
    for (int i = 0; i < et; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            p.pos[j] += p.shape[i] * c[3 * i + j];
            dxds[j] += ds[i] * c[3 * i + j];
            dxdt[j] += dt[i] * c[3 * i + j];
        }
    double n[3];
    n[0] = dxds[1] * dxdt[2] - dxds[2] * dxdt[1];
    n[1] = dxds[2] * dxdt[0] - dxds[0] * dxdt[2];
    n[2] = dxds[0] * dxdt[1] - dxds[1] * dxdt[0];
    p.jac = sqrt(dot3(n, n));
    if (p.jac > 1e-15) {
        p.nrm[0] = n[0] / p.jac; p.nrm[1] = n[1] / p.jac; p.nrm[2] = n[2] / p.jac;
    } else {
        p.nrm[0] = p.nrm[1] = p.nrm[2] = 0.0;
    }
    return p;
}

// singular.rs:696-721
__device__ __forceinline__ void local_to_global(const double* c, int et, double s, double t, double* out) {
    double fn[4];
    if (et == 3) {
        fn[0] = 1.0 - s - t; fn[1] = s; fn[2] = t; fn[3] = 0.0;
    } else {
        double s1 = 0.25 * (s + 1.0), s2 = 0.25 * (s - 1.0), t1 = t + 1.0, t2 = t - 1.0;
        fn[0] = s1 * t1; fn[1] = -s2 * t1; fn[2] = s2 * t2; fn[3] = -s1 * t2;
    }
    out[0] = out[1] = out[2] = 0.0;
    for (int i = 0; i < et; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) out[j] += fn[i] * c[3 * i + j];
}

__device__ __forceinline__ void quad_point(int et, int q, double& xi, double& eta, double& w) {
    if (et == 3) {
        xi = BEMQ_TR13[q][0]; eta = BEMQ_TR13[q][1]; w = BEMQ_TR13[q][2] * 0.5;  // gauss.rs:67-89
    } else {
        int i = q >> 2, j = q & 3;  // gauss.rs:94-105, i outer
        xi = BEMQ_GL4_X[i]; eta = BEMQ_GL4_X[j]; w = BEMQ_GL4_W[i] * BEMQ_GL4_W[j];
    }
}

struct Acc {
    cplx g, h, ht, e, rhs;
};
__device__ __forceinline__ Acc acc_zero() { return Acc{C(0, 0), C(0, 0), C(0, 0), C(0, 0), C(0, 0)}; }
__device__ __forceinline__ double shfl_xor_d(double v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
__device__ __forceinline__ void warp_reduce(cplx& z) {
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) {
        z.re += shfl_xor_d(z.re, m);
        z.im += shfl_xor_d(z.im, m);
    }
}
__device__ __forceinline__ void warp_reduce(Acc& a) {
    warp_reduce(a.g); warp_reduce(a.h); warp_reduce(a.ht); warp_reduce(a.e); warp_reduce(a.rhs);
}

__device__ __forceinline__ uint64_t below(int i) { return i >= 64 ? ~0ull : ((1ull << i) - 1ull); }

// per-warp scratch for the subdivision
struct WarpScratch {
    double cand[2][MAX_NSE][8];  // [buffer][slot][xi0..3, eta0..3]
    double subs[MAX_SUB][7];     // tri: v0xi,v0eta,v1xi,v1eta,v2xi,v2eta,faclin ; quad: xc,ec,-,-,-,-,faclin
};

// generate_subelements(): singular.rs:497-660, warp-cooperative.  Returns the number
// of accepted sub-elements (stored in ws.subs in the reference's output order).
__device__ int generate_subelements_warp(WarpScratch& ws, const double* src, const double* c, int et, double area,
                                         int lane) {
    const int nv = et;
    if (lane < nv) {
        ws.cand[0][0][lane] = (et == 3) ? d_CSI6[lane] : d_CSI8[lane];
        ws.cand[0][0][4 + lane] = (et == 3) ? d_ETA6[lane] : d_ETA8[lane];
    }
    __syncwarp();
    int nsfl = 1, nres = 0, cur = 0;
    double faclin = 2.0;
    for (int level = 0; level < 80; ++level) {
        faclin *= 0.5;
        const double arels = area * faclin * faclin;
        const double sq = sqrt(arels);
        const int nsel = nsfl;
        bool need[2] = {false, false};
        double scent[2] = {0, 0}, tcent[2] = {0, 0};
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
            int idi = lane + 32 * hh;
            if (idi < nsel) {
                const double* xs = ws.cand[cur][idi];
                double sc = 0.0, tc = 0.0;
                for (int v = 0; v < nv; ++v) sc += xs[v];
                sc = sc / (double)nv;
                for (int v = 0; v < nv; ++v) tc += xs[4 + v];
                tc = tc / (double)nv;
                double crd[3];
                local_to_global(c, et, sc, tc, crd);
                double diff[3] = {crd[0] - src[0], crd[1] - src[1], crd[2] - src[2]};
                double dist = sqrt(dot3(diff, diff));
                double ratdis = dist / sq;
                need[hh] = ratdis < 3.0;  // TOL_F (singular.rs:507,553-556)
                scent[hh] = sc; tcent[hh] = tc;
            }
        }
        const unsigned nm0 = __ballot_sync(0xffffffffu, need[0]);
        const unsigned nm1 = __ballot_sync(0xffffffffu, need[1]);
        const uint64_t needmask = (uint64_t)nm0 | ((uint64_t)nm1 << 32);
        const int ndie_total = __popcll(needmask);
        // `ndie > 15 => break`: the 16th element that needs subdivision and everything
        // after it in scan order are dropped (singular.rs:558-562)
        int cut = nsel;
        if (ndie_total > 15) {
            uint64_t mm = needmask;
            for (int i = 0; i < 15; ++i) mm &= mm - 1;  // clear the 15 lowest set bits
            cut = __ffsll((long long)mm) - 1;
        }
        const uint64_t inrange = below(cut < nsel ? cut : nsel);
        const uint64_t nmask = needmask & inrange;
        const uint64_t amask = (~needmask) & inrange;
        const int nxt = cur ^ 1;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
            int idi = lane + 32 * hh;
            if (idi < nsel && idi < cut) {
                const double* xs = ws.cand[cur][idi];
                if (need[hh]) {
                    int rank = __popcll(nmask & below(idi));
                    int nsf0 = rank * 4;
                    double xisp[8], etsp[8];
                    for (int j = 0; j < nv; ++j) {
                        int j1 = (j + 1) % nv;
                        xisp[j] = xs[j];
                        xisp[j + nv] = (xs[j] + xs[j1]) / 2.0;
                        etsp[j] = xs[4 + j];
                        etsp[j + nv] = (xs[4 + j] + xs[4 + j1]) / 2.0;
                    }
                    for (int j = 0; j < nv; ++j) {
                        double* o = ws.cand[nxt][nsf0 + j];
                        int j1 = j + nv;
                        int j2 = (j1 > nv) ? j1 - 1 : j1 + nv - 1;
                        if (et == 4) {
                            o[0] = xisp[j]; o[1] = xisp[j1]; o[2] = scent[hh]; o[3] = xisp[j2];
                            o[4] = etsp[j]; o[5] = etsp[j1]; o[6] = tcent[hh]; o[7] = etsp[j2];
                        } else {
                            o[0] = xisp[j]; o[1] = xisp[j1]; o[2] = xisp[j2]; o[3] = 0.0;
                            o[4] = etsp[j]; o[5] = etsp[j1]; o[6] = etsp[j2]; o[7] = 0.0;
                        }
                    }
                    if (et == 3) {
                        double* o = ws.cand[nxt][nsf0 + 3];
                        o[0] = xisp[3]; o[1] = xisp[4]; o[2] = xisp[5]; o[3] = 0.0;
                        o[4] = etsp[3]; o[5] = etsp[4]; o[6] = etsp[5]; o[7] = 0.0;
                    }
                } else {
                    int pos = nres + __popcll(amask & below(idi));
                    if (pos < MAX_SUB) {
                        double* o = ws.subs[pos];
                        if (et == 4) {
                            double xc = 0.0, ec = 0.0;
                            for (int v = 0; v < 4; ++v) xc += xs[v];
                            for (int v = 0; v < 4; ++v) ec += xs[4 + v];
                            o[0] = xc / 4.0; o[1] = ec / 4.0;
                        } else {
                            o[0] = xs[0]; o[1] = xs[4]; o[2] = xs[1]; o[3] = xs[5]; o[4] = xs[2]; o[5] = xs[6];
                        }
                        o[6] = faclin;
                    }
                }
            }
        }
        nres += __popcll(amask);
        if (nres >= MAX_SUB) { nres = MAX_SUB; break; }  // singular.rs:648-650
        if (ndie_total == 0) break;
        nsfl = __popcll(nmask) * 4;
        cur = nxt;
        __syncwarp();
    }
    __syncwarp();
    return nres;
}

// regular_integration(): regular.rs:33-182 for one (source, field element) pair.
// All lanes return the reduced result.
__device__ Acc regular_integration_warp(WarpScratch& ws, const double* src, const double* nx, const double* c, int et,
                                        double area, const Phys& ph, const cplx* bc, int bc_len, int bc_type,
                                        bool compute_rhs, int lane) {
    const int nsub = generate_subelements_warp(ws, src, c, et, area, lane);
    const int NQ = (et == 3) ? NQ_TRI : NQ_QUAD;
    Acc a = acc_zero();
    const int total = nsub * NQ;
    // The DECISIONS above are bit-faithful; the integrals below only have to agree with the
    // reference to ~1e-15, so they use the far kernel's arithmetic (explicit fma(), MUFU-seeded
    // rsqrt, Cody-Waite sincos) instead of IEEE divisions and the libm sincos.
    // Tri3: position/normal/Jacobian are affine -> hoisted out of the point loop.
    double e1[3], e2[3], nyc[3] = {0, 0, 0}, jac_c = 0.0;
    if (et == 3) {
#pragma unroll
        for (int d = 0; d < 3; ++d) { e1[d] = c[3 + d] - c[d]; e2[d] = c[6 + d] - c[d]; }
        double nv[3] = {e1[1] * e2[2] - e1[2] * e2[1], e1[2] * e2[0] - e1[0] * e2[2], e1[0] * e2[1] - e1[1] * e2[0]};
        double n2 = dot3(nv, nv);
        jac_c = sqrt(n2);
        if (jac_c > 1e-15) { nyc[0] = nv[0] / jac_c; nyc[1] = nv[1] / jac_c; nyc[2] = nv[2] / jac_c; }
    }
    for (int p = lane; p < total; p += 32) {
        const int is = p / NQ, q = p - is * NQ;
        const double* se = ws.subs[is];
        const double fase = se[6];
        const bool iforie = fabs(fabs(fase) - 1.0) < 1e-10;
        double csi, eta, wei;
        quad_point(et, q, csi, eta, wei);
        double xio, eto, weih2;
        if (iforie) {
            xio = csi; eto = eta; weih2 = wei;
        } else if (et == 3) {
            double l0 = 1.0 - csi - eta;
            xio = se[0] * l0 + se[2] * csi + se[4] * eta;
            eto = se[1] * l0 + se[3] * csi + se[5] * eta;
            double dx1 = se[2] - se[0], dy1 = se[3] - se[1], dx2 = se[4] - se[0], dy2 = se[5] - se[1];
            double det = fabs(dx1 * dy2 - dx2 * dy1);
            weih2 = wei * det;
        } else {
            xio = se[0] + csi * fase; eto = se[1] + eta * fase; weih2 = wei * (fase * fase);
        }
        double pos[3], ny[3], jac, shp[4];
        if (et == 3) {
            shp[0] = 1.0 - xio - eto; shp[1] = xio; shp[2] = eto; shp[3] = 0.0;
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                pos[d] = fma(eto, e2[d], fma(xio, e1[d], c[d]));
                ny[d] = nyc[d];
            }
            jac = jac_c;
        } else {
            const double s1 = 0.25 * (xio + 1.0), s2 = 0.25 * (xio - 1.0), t1 = eto + 1.0, t2 = eto - 1.0;
            shp[0] = s1 * t1; shp[1] = -s2 * t1; shp[2] = s2 * t2; shp[3] = -s1 * t2;
            const double ds[4] = {0.25 * t1, -0.25 * t1, 0.25 * t2, -0.25 * t2};
            const double dt[4] = {s1, -s2, s2, -s1};
            double xs[3], xt[3];
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                pos[d] = fma(shp[3], c[9 + d], fma(shp[2], c[6 + d], fma(shp[1], c[3 + d], shp[0] * c[d])));
                xs[d] = fma(ds[3], c[9 + d], fma(ds[2], c[6 + d], fma(ds[1], c[3 + d], ds[0] * c[d])));
                xt[d] = fma(dt[3], c[9 + d], fma(dt[2], c[6 + d], fma(dt[1], c[3 + d], dt[0] * c[d])));
            }
            double nv[3] = {fma(xs[1], xt[2], -(xs[2] * xt[1])), fma(xs[2], xt[0], -(xs[0] * xt[2])),
                            fma(xs[0], xt[1], -(xs[1] * xt[0]))};
            const double n2 = fma(nv[2], nv[2], fma(nv[1], nv[1], nv[0] * nv[0]));
            if (n2 > 1e-30) {
                const double rn = fast_rsqrt(n2);
                jac = n2 * rn;
                ny[0] = nv[0] * rn; ny[1] = nv[1] * rn; ny[2] = nv[2] * rn;
            } else {
                jac = sqrt(n2);
                ny[0] = ny[1] = ny[2] = 0.0;
            }
        }
        const double dx = pos[0] - src[0], dy = pos[1] - src[1], dz = pos[2] - src[2];
        const double r2 = fma(dz, dz, fma(dy, dy, dx * dx));
        if (!(r2 > 1e-30)) continue;  // `dis_fsp < 1e-15` skip (regular.rs:120)
        const double rho = fast_rsqrt(r2);
        const double dis = r2 * rho;
        double sn, cs;
        fast_sincos(ph.wavruim * dis, sn, cs);
        const double g = (weih2 * jac) * (INV_4PI * rho);
        const cplx zg = C(g * cs, g * sn);
        const cplx zb = C(fma(-zg.re, rho, -(zg.im * ph.wavruim)), fma(zg.re, ph.wavruim, -(zg.im * rho)));  // zg*(-1/r + ik)
        const double re1_h = fma(dz, ny[2], fma(dy, ny[1], dx * ny[0])) * rho;
        const double re2_h = -(fma(dz, nx[2], fma(dy, nx[1], dx * nx[0])) * rho);
        const cplx zhh = C(zb.re * re1_h, zb.im * re1_h);
        const cplx zht = C(zb.re * re2_h, zb.im * re2_h);
        const double rq = re1_h * re2_h;
        const double nxny = fma(nx[2], ny[2], fma(nx[1], ny[1], nx[0] * ny[0]));
        const double rho2 = rho * rho;
        const double t3 = fma(3.0, rq, nxny);
        const double fre = fma(rho2, t3, -(ph.k2 * rq));
        const double fim = -(ph.wavruim * rho) * t3;
        const cplx ze = C(fma(zg.re, fre, -(zg.im * fim)), fma(zg.re, fim, zg.im * fre));
        a.g += zg; a.h += zhh; a.ht += zht; a.e += ze;
        if (compute_rhs) {
            cplx zbg = C(0, 0);
            for (int i = 0; i < et; ++i)
                if (i < bc_len) zbg += bc[i] * shp[i];
            if (bc_type == 0) a.rhs += (zg * ph.gamma * ph.tau + zht * ph.beta_unscaled) * zbg;
            else if (bc_type == 1) a.rhs -= (zhh * ph.gamma * ph.tau + ze * ph.beta_unscaled) * zbg;
        }
    }
    warp_reduce(a);
    return a;
}

// QuadratureParams::for_ka(): singular.rs:48-82
__device__ __forceinline__ void quad_params_for_ka(double ka, int& eo, int& so, int& ns1, int& ns2) {
    if (ka < 0.3) { eo = 3; so = 4; ns1 = 4; ns2 = 2; }
    else if (ka < 1.0) { eo = 4; so = 5; ns1 = 6; ns2 = 2; }
    else if (ka < 2.0) { eo = 5; so = 6; ns1 = 8; ns2 = 3; }
    else { eo = 6; so = 7; ns1 = 10; ns2 = 4; }
}
__device__ __forceinline__ void gl_point(int order, int i, double& x, double& w) {
    switch (order) {  // orders reachable through for_ka(): 3..7
        case 3: x = BEMQ_GL3_X[i]; w = BEMQ_GL3_W[i]; break;
        case 4: x = BEMQ_GL4_X[i]; w = BEMQ_GL4_W[i]; break;
        case 5: x = BEMQ_GL5_X[i]; w = BEMQ_GL5_W[i]; break;
        case 6: x = BEMQ_GL6_X[i]; w = BEMQ_GL6_W[i]; break;
        default: x = BEMQ_GL7_X[i]; w = BEMQ_GL7_W[i]; break;
    }
}

// singular_integration(): singular.rs:123-394 (self element), warp-cooperative.
__device__ Acc singular_integration_warp(const double* src, const double* nx, const double* c, int et, double esize,
                                         const Phys& ph, const cplx* bc, int bc_len, int bc_type, bool compute_rhs,
                                         int lane) {
    int ngpo1, ngs, nsec1, nsec2;
    quad_params_for_ka(ph.k * esize, ngpo1, ngs, nsec1, nsec2);
    const int nn = et;
    Acc a = acc_zero();
    // ---- edge integral of the hypersingular kernel (singular.rs:176-254)
    const int per_edge = nsec1 * ngpo1;
    for (int p = lane; p < nn * per_edge; p += 32) {
        const int ieg = p / per_edge;
        const int rem = p - ieg * per_edge;
        const int isec = rem / ngpo1, ig = rem - isec * ngpo1;
        const int ig1 = (ieg + 1) % nn;
        double diff_poi[3], leneg = 0.0;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            diff_poi[i] = c[3 * ig1 + i] - c[3 * ieg + i];
            leneg += diff_poi[i] * diff_poi[i];
        }
        leneg = sqrt(leneg);
        double poo[3] = {diff_poi[0] / leneg, diff_poi[1] / leneg, diff_poi[2] / leneg};
        double leneg_scaled = leneg / (2.0 * (double)nsec1);
        double delsec = 2.0 / (double)nsec1;
        double secmid = -1.0 - delsec / 2.0;
        for (int s = 0; s <= isec; ++s) secmid += delsec;  // same running sum as the reference
        double gx, gw;
        gl_point(ngpo1, ig, gx, gw);
        double sga = secmid + gx / (double)nsec1;
        double wga = gw * leneg_scaled;
        double diff[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            double crd = c[3 * ieg + i] + diff_poi[i] * (sga + 1.0) / 2.0;
            diff[i] = crd - src[i];
        }
        double dis = sqrt(dot3(diff, diff));
        if (!(dis > 1e-15)) continue;
        double u[3] = {diff[0] / dis, diff[1] / dis, diff[2] / dis};
        double re1 = ph.wavruim * dis;
        double re2 = 4.0 * PI * dis;
        double sn, cs;
        sincos(re1, &sn, &cs);
        cplx zg = C(cs / re2, sn / re2);
        cplx z1 = C(-1.0 / dis, ph.wavruim);
        cplx zgf = zg * z1;
        cplx zd0 = zgf * u[0], zd1 = zgf * u[1], zd2 = zgf * u[2];
        cplx w0 = zd1 * poo[2] - zd2 * poo[1];
        cplx w1 = zd2 * poo[0] - zd0 * poo[2];
        cplx w2 = zd0 * poo[1] - zd1 * poo[0];
        a.e += (w0 * nx[0] + w1 * nx[1] + w2 * nx[2]) * wga;
    }
    // ---- Duffy sub-triangles for G, H, H^T and the k^2 (nx.ny) G part of E (singular.rs:257-375)
    const int per_sec = ngs * ngs;
    const int per_edge2 = nsec2 * per_sec;
    for (int p = lane; p < nn * per_edge2; p += 32) {
        const int ieg = p / per_edge2;
        int rem = p - ieg * per_edge2;
        const int isec = rem / per_sec;
        rem -= isec * per_sec;
        const int i = rem / ngs, j = rem - i * ngs;
        const int ig1 = (ieg + 1) % nn, ig2 = ieg + nn;
        const double* CS = (et == 3) ? d_CSI6 : d_CSI8;
        const double* ET = (et == 3) ? d_ETA6 : d_ETA8;
        double ssub[3], tsub[3], aresub;
        if (et == 3) {
            aresub = 1.0 / 24.0 / (double)nsec2;
            ssub[0] = 1.0 / 3.0; tsub[0] = 1.0 / 3.0;
        } else {
            aresub = 0.25 / (double)nsec2;
            ssub[0] = 0.0; tsub[0] = 0.0;
        }
        if (isec == 0) {
            ssub[1] = CS[ieg]; ssub[2] = CS[ig2]; tsub[1] = ET[ieg]; tsub[2] = ET[ig2];
        } else {  // quirk: every isec >= 1 integrates the SAME second sub-triangle (singular.rs:268-278)
            ssub[1] = CS[ig2]; ssub[2] = CS[ig1]; tsub[1] = ET[ig2]; tsub[2] = ET[ig1];
        }
        double sga, wi, tga, wj;
        gl_point(ngs, i, sga, wi);
        gl_point(ngs, j, tga, wj);
        double wei = wi * wj;
        double sgg = 0.5 * (1.0 - sga) * ssub[0] + 0.25 * (1.0 + sga) * ((1.0 - tga) * ssub[1] + (1.0 + tga) * ssub[2]);
        double tgg = 0.5 * (1.0 - sga) * tsub[0] + 0.25 * (1.0 + sga) * ((1.0 - tga) * tsub[1] + (1.0 + tga) * tsub[2]);
        Params pr = compute_parameters(c, et, sgg, tgg);
        double wga = wei * (1.0 + sga) * aresub * pr.jac;
        double diff[3] = {pr.pos[0] - src[0], pr.pos[1] - src[1], pr.pos[2] - src[2]};
        double dis = sqrt(dot3(diff, diff));
        if (!(dis > 1e-15)) continue;
        double u[3] = {diff[0] / dis, diff[1] / dis, diff[2] / dis};
        double re1 = ph.wavruim * dis;
        double re2 = wga / (4.0 * PI * dis);
        double sn, cs;
        sincos(re1, &sn, &cs);
        cplx zg = C(cs * re2, sn * re2);
        cplx z1 = C(-1.0 / dis, ph.wavruim);
        cplx zb = zg * z1;
        double re1_h = dot3(u, pr.nrm);
        double re2_h = -dot3(u, nx);
        cplx zhh = zb * re1_h;
        cplx zht = zb * re2_h;
        a.g += zg; a.h += zhh; a.ht += zht;
        a.e += zg * ph.k2 * dot3(nx, pr.nrm);
        if (compute_rhs && bc_type == 0) {
            cplx zbg = C(0, 0);
            for (int ii = 0; ii < et; ++ii)
                if (ii < bc_len) zbg += bc[ii] * pr.shape[ii];
            a.rhs += (zg * ph.gamma * ph.tau + zht * ph.beta_unscaled) * zbg;
        }
    }
    warp_reduce(a);
    if (compute_rhs && bc_type == 1) {  // singular.rs:380-391
        cplx zbg = C(0, 0);
        for (int i = 0; i < bc_len; ++i) zbg += bc[i];
        zbg = zbg / (double)bc_len;
        a.rhs = -(a.h * ph.gamma * ph.tau + a.e * ph.beta_unscaled) * zbg;
    }
    return a;
}

// assemble_tbem(): tbem.rs:311-345 (coefficient only)
__device__ __forceinline__ cplx combine(const Acc& a, int field_bc_type, const Phys& ph) {
    cplx gam = C(ph.gamma, 0.0), tau = C(ph.tau, 0.0);
    cplx h = a.h * ph.sign;  // result.dg_dn_integral *= dg_dn_sign (tbem.rs:203)
    if (field_bc_type == 0) return h * gam * tau + a.e * ph.beta;
    if (field_bc_type == 1) return -(a.g * gam * tau + a.ht * ph.beta);
    return C(0, 0);
}

// admittance column (DESIGN.md 4.8): v_j = vbar_j + Y_j p_j moves -Y_j (gamma tau G + beta H^T) to the left-hand side; G and H^T
// are the integrals of this pair (no dg_dn_sign), beta the assembly's
__device__ __forceinline__ cplx admittance_term(const Acc& a, cplx y, const Phys& ph) {
    cplx gam = C(ph.gamma, 0.0), tau = C(ph.tau, 0.0);
    return y * (a.g * gam * tau + a.ht * ph.beta);
}
__device__ __forceinline__ cplx admittance_of(const Phys& ph, uint32_t col) { return ph.adm ? ph.adm[col] : C(0.0, 0.0); }
__device__ __forceinline__ bool nonzero(cplx z) { return z.re != 0.0 || z.im != 0.0; }

__device__ __forceinline__ void atomic_add_cplx(cplx* p, cplx v) {
    atomicAdd(&p->re, v.re);
    atomicAdd(&p->im, v.im);
}

__device__ void do_pair(WarpScratch& ws, const DeviceMesh& m, const Phys& ph, uint32_t row, uint32_t col,
                        uint64_t row_begin, cplx* A, uint64_t lda, cplx* rhs, int lane) {
    double src[3], nx[3], c[12];
#pragma unroll
    for (int i = 0; i < 3; ++i) { src[i] = m.src[8ull * row + i]; nx[i] = m.src[8ull * row + 3 + i]; }
#pragma unroll
    for (int i = 0; i < 12; ++i) c[i] = m.coords[12ull * col + i];
    const int et = m.etype[col];
    const int fbt = m.bc_type[col];
    const int fbl = m.bc_len[col];
    const bool crhs = m.nonzero_bc[col] != 0;
    cplx bc[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) bc[i] = m.bc_val[4ull * col + i];
    Acc a = regular_integration_warp(ws, src, nx, c, et, m.area[col], ph, bc, fbl, fbt, crhs, lane);
    if (lane == 0) {
        cplx coeff = combine(a, fbt, ph);
        const cplx y = admittance_of(ph, col);
        if (nonzero(y)) coeff -= admittance_term(a, y, ph);
        A[(uint64_t)(row - row_begin) * lda + col] = coeff;
        if (crhs) atomic_add_cplx(&rhs[row - row_begin], a.rhs);
    }
}

__global__ void __launch_bounds__(32 * WARPS_PER_BLOCK)
near_list_kernel(DeviceMesh m, Phys ph, uint64_t row_begin, cplx* A, uint64_t lda, cplx* rhs, const uint2* list,
                 unsigned int count) {
    __shared__ WarpScratch ws[WARPS_PER_BLOCK];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (unsigned int idx = blockIdx.x * WARPS_PER_BLOCK + w; idx < count; idx += gridDim.x * WARPS_PER_BLOCK) {
        uint2 e = list[idx];
        do_pair(ws[w], m, ph, e.x, e.y, row_begin, A, lda, rhs, lane);
        __syncwarp();
    }
}

// dense generic path over (row, special column) pairs
__global__ void __launch_bounds__(32 * WARPS_PER_BLOCK)
special_kernel(DeviceMesh m, Phys ph, uint64_t row_begin, uint64_t row_end, cplx* A, uint64_t lda, cplx* rhs) {
    __shared__ WarpScratch ws[WARPS_PER_BLOCK];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint64_t nrows = row_end - row_begin;
    const uint64_t total = nrows * m.n_special;
    for (uint64_t idx = (uint64_t)blockIdx.x * WARPS_PER_BLOCK + w; idx < total;
         idx += (uint64_t)gridDim.x * WARPS_PER_BLOCK) {
        uint32_t row = (uint32_t)(row_begin + idx / m.n_special);
        uint32_t col = m.special_cols[idx % m.n_special];
        if (row != col) do_pair(ws[w], m, ph, row, col, row_begin, A, lda, rhs, lane);
        __syncwarp();
    }
}

// diagonal: free terms (tbem.rs:273-304) + singular self integral
__global__ void __launch_bounds__(32 * WARPS_PER_BLOCK)
self_kernel(DeviceMesh m, Phys ph, uint64_t row_begin, uint64_t row_end, cplx* A, uint64_t lda, cplx* rhs) {
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (uint64_t row = row_begin + (uint64_t)blockIdx.x * WARPS_PER_BLOCK + w; row < row_end;
         row += (uint64_t)gridDim.x * WARPS_PER_BLOCK) {
        double src[3], nx[3], c[12];
#pragma unroll
        for (int i = 0; i < 3; ++i) { src[i] = m.src[8ull * row + i]; nx[i] = m.src[8ull * row + 3 + i]; }
#pragma unroll
        for (int i = 0; i < 12; ++i) c[i] = m.coords[12ull * row + i];
        const int et = m.etype[row];
        const int bt = m.bc_type[row];
        const int bl = m.bc_len[row];
        const bool crhs = m.nonzero_bc[row] != 0;
        cplx bc[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) bc[i] = m.bc_val[4ull * row + i];
        Acc a = singular_integration_warp(src, nx, c, et, m.esize[row], ph, bc, bl, bt, crhs, lane);
        if (lane == 0) {
            cplx gam = C(ph.gamma, 0.0), tau = C(ph.tau, 0.0);
            cplx sum = C(0, 0);
            for (int i = 0; i < bl; ++i) sum += bc[i];
            cplx avg = sum / (double)bl;
            cplx diag = C(0, 0), r0 = C(0, 0);
            if (bt == 0) {
                diag -= gam * 0.5;
                r0 += avg * ph.beta * tau * 0.5;
            } else if (bt == 1) {
                diag -= ph.beta * tau * 0.5;
                r0 += avg * tau * 0.5;
            }
            diag += combine(a, bt, ph);
            const cplx y = admittance_of(ph, (uint32_t)row);
            if (nonzero(y)) {
                diag -= admittance_term(a, y, ph);
                diag -= y * ph.beta * tau * 0.5;
            }
            A[(row - row_begin) * lda + row] = diag;
            if (crhs) r0 += a.rhs;
            atomic_add_cplx(&rhs[row - row_begin], r0);
        }
    }
}

// ---- prep: per-column far-field records -------------------------------------------
// For a flat element (Tri3, parallelogram Quad4) y_q = y_0 + a_q e1 + b_q e2 with
// e1 = dx/ds, e2 = dx/dt constant, so the far kernel only needs y_0, e1, e2, n_y, J and
// kappa_q = |y_q - y_0|^2 (see assembly_far.cu).
__device__ __forceinline__ void tangents(const double* c, int et, double s, double t, double* e1, double* e2) {
    double ds[4], dt[4];
    if (et == 3) {
        ds[0] = -1.0; ds[1] = 1.0; ds[2] = 0.0; ds[3] = 0.0;
        dt[0] = -1.0; dt[1] = 0.0; dt[2] = 1.0; dt[3] = 0.0;
    } else {
        ds[0] = 0.25 * (t + 1.0); ds[1] = -0.25 * (t + 1.0); ds[2] = 0.25 * (t - 1.0); ds[3] = -0.25 * (t - 1.0);
        dt[0] = 0.25 * (s + 1.0); dt[1] = 0.25 * (1.0 - s); dt[2] = 0.25 * (s - 1.0); dt[3] = -0.25 * (s + 1.0);
    }
    for (int d = 0; d < 3; ++d) { e1[d] = 0.0; e2[d] = 0.0; }
    for (int i = 0; i < et; ++i)
        for (int d = 0; d < 3; ++d) { e1[d] += ds[i] * c[3 * i + d]; e2[d] += dt[i] * c[3 * i + d]; }
}

__global__ void prep_kernel(DeviceMesh m) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m.ntiles * TILE) return;
    const uint32_t tile = j / TILE, t = j % TILE;
    double* fk = m.far_k + (uint64_t)tile * NQ_MAX * TILE;
    double* fc = m.far_c + (uint64_t)tile * FAR_NCONST * TILE;
    if (j >= m.n) {  // padding columns of the last tile
        for (int q = 0; q < NQ_MAX; ++q) fk[q * TILE + t] = 0.0;
        for (int s = 0; s < FAR_NCONST; ++s) fc[s * TILE + t] = 0.0;
        fc[FC_Y0X * TILE + t] = 1.0e30;
        m.col_class[j] = COL_NONE;
        return;
    }
    double c[12];
    for (int i = 0; i < 12; ++i) c[i] = m.coords[12ull * j + i];
    const int et = m.etype[j];
    const int NQ = (et == 3) ? NQ_TRI : NQ_QUAD;
    double n0[3] = {0, 0, 0}, j0 = 0.0, y0[3] = {0, 0, 0}, dev = 0.0, devp = 0.0, e1[3], e2[3];
    double xi0 = 0.0, eta0 = 0.0;
    for (int q = 0; q < NQ_MAX; ++q) {
        double kap = 0.0;
        if (q < NQ) {
            double xi, eta, w;
            quad_point(et, q, xi, eta, w);
            Params p = compute_parameters(c, et, xi, eta);
            if (q == 0) {
                for (int d = 0; d < 3; ++d) { n0[d] = p.nrm[d]; y0[d] = p.pos[d]; }
                j0 = p.jac;
                xi0 = xi; eta0 = eta;
                tangents(c, et, xi, eta, e1, e2);
            } else {
                for (int d = 0; d < 3; ++d) dev = fmax(dev, fabs(p.nrm[d] * p.jac - n0[d] * j0));
                // the affine model must reproduce the true quadrature point
                double aq = xi - xi0, bq = eta - eta0;
                for (int d = 0; d < 3; ++d) devp = fmax(devp, fabs(y0[d] + aq * e1[d] + bq * e2[d] - p.pos[d]));
                double dl[3] = {p.pos[0] - y0[0], p.pos[1] - y0[1], p.pos[2] - y0[2]};
                kap = dot3(dl, dl);
            }
        }
        fk[q * TILE + t] = kap;
    }
    fc[FC_NX * TILE + t] = n0[0]; fc[FC_NY * TILE + t] = n0[1]; fc[FC_NZ * TILE + t] = n0[2];
    fc[FC_J4PI * TILE + t] = j0 * INV_4PI;
    fc[FC_Y0X * TILE + t] = y0[0]; fc[FC_Y0Y * TILE + t] = y0[1]; fc[FC_Y0Z * TILE + t] = y0[2];
    // |y_0 - x|^2 < 9*area  <=>  ratdis < 3 up to rounding (y_0 is the table centroid, 3e-16 away
    // from the 1/3-centroid of singular.rs:541-548); the 1e-9 guard band sends every borderline
    // pair to the exact near kernel, which re-takes the decision bit-faithfully
    fc[FC_THR * TILE + t] = 9.0 * m.area[j] * (1.0 + 1e-9);
    fc[FC_E1X * TILE + t] = e1[0]; fc[FC_E1Y * TILE + t] = e1[1]; fc[FC_E1Z * TILE + t] = e1[2];
    fc[FC_E2X * TILE + t] = e2[0]; fc[FC_E2Y * TILE + t] = e2[1]; fc[FC_E2Z * TILE + t] = e2[2];
    // kappa of the ratio-test centre relative to y_0: the centre is y_0 for TR13 (q = 0 is the
    // centroid) but (s,t) = (0,0) for the 4x4 Gauss rule, i.e. y_0 - s_0 e1 - t_0 e2
    {
        double kc = 0.0;
        if (et == 4) {
            double dl[3];
            for (int d = 0; d < 3; ++d) dl[d] = -xi0 * e1[d] - eta0 * e2[d];
            kc = dot3(dl, dl);
        }
        fc[FC_KC * TILE + t] = kc;
    }
    fc[FC_SPARE1 * TILE + t] = 0.0;
    // estimate_element_size(): singular.rs:730-745
    double total = 0.0;
    for (int i = 0; i < et; ++i) {
        int jn = (i + 1) % et;
        double e2s = 0.0;
        for (int k = 0; k < 3; ++k) {
            double d = c[3 * jn + k] - c[3 * i + k];
            e2s += d * d;
        }
        total += sqrt(e2s);
    }
    m.esize[j] = total / (double)et;
    // flat <=> n_y*J constant over the rule (1e-13 relative) and the affine model reproduces the
    // quadrature points to 1e-12 of the element size
    const double len = sqrt(dot3(e1, e1)) + sqrt(dot3(e2, e2));
    // (a non-zero prescribed VELOCITY keeps the column in the far kernel: the entry is that of a rigid element, the
    //  right-hand-side term is added by rhs_far_kernel; pressure / transfer BCs and warped quads take the generic path)
    bool special = (m.bc_type[j] != 0) || !(j0 > 1e-15) || (dev > 1e-13 * j0) ||
                   (devp > 1e-12 * len) || !(m.area[j] > 0.0);
    m.col_class[j] = special ? COL_SPECIAL : (et == 3 ? COL_FLAT_TRI : COL_FLAT_QUAD);
}

}  // namespace

cudaError_t launch_prep(const DeviceMesh& m, cudaStream_t s) {
    const uint32_t total = m.ntiles * TILE;
    prep_kernel<<<(total + 127) / 128, 128, 0, s>>>(m);
    return cudaGetLastError();
}

cudaError_t launch_near_list(const DeviceMesh& m, const Phys& ph, uint64_t row_begin, cplx* A, uint64_t lda, cplx* rhs,
                             const uint2* near_list, unsigned int count, cudaStream_t s) {
    if (count == 0) return cudaSuccess;
    unsigned int blocks = (count + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
    const unsigned int maxb = 148u * 16u * 4u;
    if (blocks > maxb) blocks = maxb;
    near_list_kernel<<<blocks, 32 * WARPS_PER_BLOCK, 0, s>>>(m, ph, row_begin, A, lda, rhs, near_list, count);
    return cudaGetLastError();
}

cudaError_t launch_special(const DeviceMesh& m, const Phys& ph, uint64_t row_begin, uint64_t row_end, cplx* A,
                           uint64_t lda, cplx* rhs, cudaStream_t s) {
    if (m.n_special == 0 || row_end <= row_begin) return cudaSuccess;
    uint64_t total = (row_end - row_begin) * m.n_special;
    uint64_t blocks = (total + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
    const uint64_t maxb = 148ull * 16ull * 4ull;
    if (blocks > maxb) blocks = maxb;
    special_kernel<<<(unsigned int)blocks, 32 * WARPS_PER_BLOCK, 0, s>>>(m, ph, row_begin, row_end, A, lda, rhs);
    return cudaGetLastError();
}

cudaError_t launch_self(const DeviceMesh& m, const Phys& ph, uint64_t row_begin, uint64_t row_end, cplx* A, uint64_t lda,
                        cplx* rhs, cudaStream_t s) {
    if (row_end <= row_begin) return cudaSuccess;
    uint64_t rows = row_end - row_begin;
    uint64_t blocks = (rows + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
    const uint64_t maxb = 148ull * 16ull * 4ull;
    if (blocks > maxb) blocks = maxb;
    self_kernel<<<(unsigned int)blocks, 32 * WARPS_PER_BLOCK, 0, s>>>(m, ph, row_begin, row_end, A, lda, rhs);
    return cudaGetLastError();
}

}  // namespace bemb
