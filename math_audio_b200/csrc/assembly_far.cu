// assembly_far.cu -- the FP64 compute-bound far-field assembly kernel (K1).
//
// Replaces, for every (collocation row i, field element j) pair whose level-0 ratio test
// passes (dist/sqrt(area) >= 3, singular.rs:553-556), the un-subdivided branch of
// regular_integration (regular.rs:67-154) followed by assemble_tbem for a velocity-BC field
// element (tbem.rs:323-331):
//     A[i,j] = sign*gamma*tau * sum_q H_q  +  beta * sum_q E_q
// with the 13-point triangle rule (Tri3) or the 4x4 Gauss rule (flat Quad4).
//
// Mapping (B200): block = 128 threads <-> one tile of 128 consecutive matrix columns.  Per
// column the thread keeps the element's frame in registers -- first quadrature point y_0,
// tangents e1 = dx/ds, e2 = dx/dt, unit normal n_y, J/(4 pi) -- and the tile's table
// kappa_q = |y_q - y_0|^2 (13-16 values per element, SoA) is brought into shared memory by one
// TMA bulk copy (cp.async.bulk + mbarrier).  The block then walks a chunk of collocation rows:
// every warp computes 32 adjacent entries of one row, so the complex128 stores are 512
// contiguous bytes per warp; the source point/normal are block-uniform loads.
//
// Arithmetic per pair (x = source, d0 = y_0 - x):  on a flat element y_q = y_0 + a_q e1 + b_q e2
// (a_q, b_q compile-time constants of the rule), hence
//     r_q^2        = |d0|^2 + a_q (2 d0.e1) + b_q (2 d0.e2) + kappa_q            3 DP ops
//     (y_q-x).n_x  = d0.n_x + a_q (e1.n_x) + b_q (e2.n_x)                       2 DP ops
//     (y_q-x).n_y  = d0.n_y                                   (constant over the element)
// then one MUFU-seeded rsqrt (5), one table-based sincos (pi/256 reduction, 512-entry (cos,sin) table in
// shared memory, degree-4/5 kernels, one rotation: 14) and the kernel algebra
// with H and E folded into ONE complex accumulator:
//     A_ij = sum_q zg_q * [ cH h rho (-rho + ik) + beta (P_q - i Q_q) ],
//     P = rho^2 t - k^2 rq,  Q = k rho t,  t = 3 rq + n_x.n_y,  rq = (h rho)(-m rho)
// (for purely imaginary beta -- the reference's beta = i*scale/k -- the bracket factors as rho (X + iY), see the
// loop) ~41 DP-pipe instructions per quadrature point.  Nothing but the 16-byte result touches HBM.
// Pairs that fail the (guard-banded) ratio test are appended to a compact list for the exact
// near-field kernel, which re-takes the decision bit-faithfully and overwrites the entry.
#include <atomic>
#include <cmath>

#include "internal.h"

namespace bemb {

namespace {

struct RuleConst {
    double w[NQ_MAX];   // weights (0.5*TR13 weight | w_i*w_j)
    double a[NQ_MAX];   // xi_q  - xi_0
    double b[NQ_MAX];   // eta_q - eta_0
    double a2[NQ_MAX];  // 2 a_q
    double b2[NQ_MAX];  // 2 b_q
    double ac, bc;      // ratio-test centre relative to (xi_0, eta_0)
    double ac2, bc2;
    double xi[NQ_MAX];  // absolute local coordinates of the points (shape functions of the BC interpolation)
    double eta[NQ_MAX];
};
__device__ __constant__ RuleConst d_rule_tri;
__device__ __constant__ RuleConst d_rule_quad;
__device__ double2 d_sincos_tab[SINCOS_TAB];  // (cos, sin)(i*pi/1024), filled by upload_tables()

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// resident blocks per SM the far kernel is compiled for (registers <= 128 per thread)
constexpr int FAR_MINB = 4;

// ADM: the instantiation for assemblies with admittance columns (DESIGN.md 4.8).  A tile that holds one accumulates, in the
// same quadrature loop, T_ij = sum_q zg_q (gamma tau + beta (m rho^2 - i k m rho)) = gamma tau G_ij + beta H^T_ij and stores
// A_ij - Y_j T_ij; its Y = 0 columns, and every column of the other tiles, keep the instruction sequence of ADM = false.
template <int NQ, bool BIMAG, bool ADM>
__global__ void __launch_bounds__(TILE, FAR_MINB)
far_kernel(const double* __restrict__ far_k, const double* __restrict__ far_c, const uint8_t* __restrict__ col_class,
           const double* __restrict__ srcdat, uint32_t n, uint64_t row_begin, uint64_t row_end, uint32_t rows_per_block,
           uint32_t nchunks, uint32_t total_items, uint32_t items_per_block,
           double wavruim, CisConst cis, double k2, double cH, double beta_re, double beta_im, cplx* __restrict__ A, uint64_t lda,
           uint2* __restrict__ near_list, unsigned int near_cap, unsigned int* __restrict__ near_count,
           unsigned int* __restrict__ work_counter, const cplx* __restrict__ adm, double gamtau) {
    __shared__ __align__(128) double sm_k[NQ * TILE];  // kappa_q, [q][column]
    __shared__ uint32_t s_item;
    extern __shared__ __align__(16) double2 sm_tab[];  // [SINCOS_TAB] (cos, sin) table: 32 KB, dynamic (static + dynamic > 48 KB)
    __shared__ __align__(8) unsigned long long mbar;

    const uint32_t t = threadIdx.x;
    constexpr uint32_t BYTES = NQ * TILE * sizeof(double);
    constexpr bool QUAD = (NQ == NQ_QUAD);
    const uint8_t want = QUAD ? COL_FLAT_QUAD : COL_FLAT_TRI;
    const RuleConst& rc = QUAD ? d_rule_quad : d_rule_tri;
    const double bk = beta_im * wavruim, bk2 = beta_im * k2, bk3 = 3.0 * bk, b3 = 3.0 * beta_im;

    if (t == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&mbar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (uint32_t i = t; i < SINCOS_TAB; i += TILE) sm_tab[i] = d_sincos_tab[i];
    __syncthreads();

    // Work item = (column tile, row chunk); a block owns a contiguous range of items, ordered so
    // that consecutive items share the tile (one item per block in the normal launch; a
    // "background" launch -- assembly of the next frequency underneath a running solve -- uses a
    // small persistent grid so that it leaves registers and shared memory to the solver's kernels).
    // With a work counter the items are pulled dynamically instead, so that a second launch of this
    // kernel ("boost", once the solver has left the GPU) can join in and finish the same assembly.
    const uint32_t item_first = blockIdx.x * items_per_block;
    const uint32_t item_last = (item_first + items_per_block < total_items) ? item_first + items_per_block : total_items;
    uint32_t cur_tile = 0xffffffffu, loads = 0;
    double nyx = 0, nyy = 0, nyz = 0, j4pi = 0, y0x = 0, y0y = 0, y0z = 0, thr = 0, e1x = 0, e1y = 0, e1z = 0, e2x = 0, e2y = 0,
           e2z = 0, kc = 0;
    bool active = false;
    double yre = 0.0, yim = 0.0;  // ADM: Y of this thread's column
    bool tile_adm = false;        // ADM: some column of the current tile has Y != 0 (block-uniform)
    uint32_t col = 0;
    const double* kq = sm_k + t;

    for (uint32_t it = 0;; ++it) {
    uint32_t item;
    if (work_counter) {
        __syncthreads();
        if (t == 0) s_item = atomicAdd(work_counter, 1u);
        __syncthreads();
        item = s_item;
        if (item >= total_items) break;
    } else {
        item = item_first + it;
        if (item >= item_last) break;
    }
    const uint32_t tile = item / nchunks, chunk = item - tile * nchunks;
    if (tile != cur_tile) {
        cur_tile = tile;
        col = tile * TILE + t;
        __syncthreads();  // everybody is done with the previous tile's kappa table
        // ---- stage the tile's kappa table with one TMA bulk copy ----------------------------
        if (t == 0) {
            const double* gsrc = far_k + (uint64_t)tile * NQ_MAX * TILE;
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&mbar)), "r"(BYTES) : "memory");
            asm volatile(
                "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(sm_k)),
                "l"(gsrc), "r"(BYTES), "r"(smem_u32(&mbar))
                : "memory");
        }
        // per-column frame -> registers (coalesced, overlaps the bulk copy)
        const double* fc = far_c + (uint64_t)tile * FAR_NCONST * TILE + t;
        nyx = fc[FC_NX * TILE]; nyy = fc[FC_NY * TILE]; nyz = fc[FC_NZ * TILE];
        j4pi = fc[FC_J4PI * TILE];
        y0x = fc[FC_Y0X * TILE]; y0y = fc[FC_Y0Y * TILE]; y0z = fc[FC_Y0Z * TILE];
        thr = fc[FC_THR * TILE];
        e1x = fc[FC_E1X * TILE]; e1y = fc[FC_E1Y * TILE]; e1z = fc[FC_E1Z * TILE];
        e2x = fc[FC_E2X * TILE]; e2y = fc[FC_E2Y * TILE]; e2z = fc[FC_E2Z * TILE];
        kc = fc[FC_KC * TILE];
        active = (col < n) && (col_class[col] == want);
        if (ADM) {
            // per-frequency, so not part of the staged far_c record: one coalesced 16-byte load per column
            const cplx y = col < n ? adm[col] : C(0.0, 0.0);
            yre = y.re; yim = y.im;
            tile_adm = __syncthreads_or(active && (yre != 0.0 || yim != 0.0)) != 0;
        }
        {
            const uint32_t parity = loads & 1u;
            uint32_t done = 0;
            while (!done) {
                asm volatile(
                    "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                    : "=r"(done)
                    : "r"(smem_u32(&mbar)), "r"(parity)
                    : "memory");
            }
            ++loads;
        }
    }

    const uint64_t r0 = row_begin + (uint64_t)chunk * rows_per_block;
    const uint64_t r1 = (r0 + rows_per_block < row_end) ? r0 + rows_per_block : row_end;

    for (uint64_t row = r0; row < r1; ++row) {
        const double* sp = srcdat + 8ull * row;  // block-uniform
        const double sx = __ldg(sp + 0), sy = __ldg(sp + 1), sz = __ldg(sp + 2);
        const double nxx = __ldg(sp + 3), nxy = __ldg(sp + 4), nxz = __ldg(sp + 5);
        const double dx = y0x - sx, dy = y0y - sy, dz = y0z - sz;
        const double D = fma(dz, dz, fma(dy, dy, dx * dx));
        const double p1 = fma(dz, e1z, fma(dy, e1y, dx * e1x));  // d0.e1  (the factor 2 lives in a2/b2)
        const double p2 = fma(dz, e2z, fma(dy, e2y, dx * e2x));
        // level-0 ratio test against the element centre, guard-banded (the exact decision is
        // re-taken by the near kernel)
        double d2c = D;
        if (QUAD) d2c = fma(rc.ac2, p1, fma(rc.bc2, p2, D + kc));
        const bool is_near = active && (d2c < thr);
        if (__any_sync(0xffffffffu, is_near)) {
            const unsigned mask = __ballot_sync(0xffffffffu, is_near && (uint64_t)col != row);
            if (mask) {
                unsigned base = 0;
                const int leader = __ffs(mask) - 1;
                if ((int)(t & 31) == leader) base = atomicAdd(near_count, __popc(mask));
                base = __shfl_sync(0xffffffffu, base, leader);
                if (is_near && (uint64_t)col != row) {
                    unsigned pos = base + __popc(mask & ((1u << (t & 31)) - 1u));
                    if (pos < near_cap) near_list[pos] = make_uint2((unsigned)row, col);
                }
            }
        }
        const double h = fma(dz, nyz, fma(dy, nyy, dx * nyx));   // (y_q - x).n_y, same for all q
        const double nn = fma(nxz, nyz, fma(nxy, nyy, nxx * nyx));
        const double M0 = fma(dz, nxz, fma(dy, nxy, dx * nxx));  // d0.n_x
        const double E1 = fma(e1z, nxz, fma(e1y, nxy, e1x * nxx));
        const double E2 = fma(e2z, nxz, fma(e2y, nxy, e2x * nxx));
        // per-pair constants of the folded kernel (see header): with rho = 1/r, m = (y_q-x).n_x
        //   rq = (u.n_y)(-(u.n_x)) = (-h m) rho^2          t = 3 rq + n_x.n_y
        //   H factor  cH (h rho)(-rho + ik)             = (-cH h) rho^2 + i (cH h k) rho
        //   E factor  (rho^2 t - k^2 rq) - i (k rho) t
        const double nh = -h;
        const double nhc = -cH * h;             // A1 = nhc * rho^2
        const double hck = (cH * h) * wavruim;  // A2 = hck * rho
        // purely imaginary beta = i b: with u = rho^2, nm = -h m the bracket factors as rho (X + iY),
        //   X = nhc rho + 3 b k nm u + b k nn,   Y = rho [nm (3 b u - b k^2) + b nn] + hck
        // and the contribution of the point is  w u (cs + i sn)(X + iY)
        const double c3 = bk * nn, c2 = beta_im * nn;
        const double bk3nh = bk3 * nh, b3nh = b3 * nh, bk2nh = bk2 * nh;
        double are = 0.0, aim = 0.0;
        double tre = 0.0, tim = 0.0;  // ADM: gamma tau G + beta H^T (without J / 4 pi)
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            const double r2 = (q == 0) ? D : fma(rc.a2[q], p1, fma(rc.b2[q], p2, D + kq[q * TILE]));
            const double rho = fast_rsqrt(r2);  // 1/r
            const double r = r2 * rho;
            double sn, cs;
            fast_cis_tab(r, cis, sm_tab, sn, cs);
            const double m = (q == 0) ? M0 : fma(rc.a[q], E1, fma(rc.b[q], E2, M0));  // (y_q - x).n_x
            const double rho2 = rho * rho;
            if (BIMAG) {
                // X = nhc rho + (3 b k nh) m rho^2 + c3,  Y = rho [m (3 b nh rho^2 - b k^2 nh) + c2] + hck   (nh = -h folded per pair)
                const double X = fma(bk3nh, m * rho2, fma(nhc, rho, c3));
                const double Z = fma(m, fma(b3nh, rho2, -bk2nh), c2);
                const double Y = fma(rho, Z, hck);
                const double G = rc.w[q] * rho2;  // w / r^2   (J/(4 pi) is applied once per pair)
                are = fma(G, fma(cs, X, -(sn * Y)), are);
                aim = fma(G, fma(cs, Y, sn * X), aim);
            } else {
                const double g = rho * rc.w[q];  // w / r
                const double zgr = g * cs, zgi = g * sn;
                const double rq = (nh * m) * rho2;
                const double t3 = fma(3.0, rq, nn);
                const double A1 = nhc * rho2;
                const double A2 = hck * rho;
                const double P = fma(rho2, t3, -(k2 * rq));
                const double Q = (wavruim * rho) * t3;
                const double fre = fma(beta_re, P, fma(beta_im, Q, A1));
                const double fim = fma(beta_im, P, fma(-beta_re, Q, A2));
                are = fma(zgr, fre, fma(-zgi, fim, are));
                aim = fma(zgr, fim, fma(zgi, fre, aim));
            }
            if (ADM && tile_adm) {
                // zg (gamma tau + beta (m rho^2 - i k m rho)),  zg = w rho (cs + i sn)
                const double mr = m * rho;
                double fr, fi;
                if (BIMAG) {
                    fr = fma(bk, mr, gamtau);  // beta = i b:  gamma tau + b k m rho  +  i b m rho^2
                    fi = beta_im * (mr * rho);
                } else {
                    const double hr = mr * rho, hi = -(wavruim * mr);
                    fr = fma(beta_re, hr, fma(-beta_im, hi, gamtau));
                    fi = fma(beta_re, hi, beta_im * hr);
                }
                const double gw = rc.w[q] * rho;
                tre = fma(gw, fma(cs, fr, -(sn * fi)), tre);
                tim = fma(gw, fma(cs, fi, sn * fr), tim);
            }
        }
        if (active) {
            double2 v = make_double2(are * j4pi, aim * j4pi);
            if (ADM && (yre != 0.0 || yim != 0.0)) {
                const double ur = tre * j4pi, ui = tim * j4pi;
                v.x = v.x - (yre * ur - yim * ui);
                v.y = v.y - (yre * ui + yim * ur);
            }
            __stcs(reinterpret_cast<double2*>(A + (row - row_begin) * lda + col), v);
        }
    }
    }  // work items
}


// Right-hand-side term of the un-subdivided pairs of columns that carry a non-zero prescribed velocity
// (regular.rs:157-177 with bc_type == 0):  rhs_i += sum_q (zg gamma tau + zht beta0) * (sum_n bc_n N_n(xi_q, eta_q)),
// zg = w J e^{ikr} / (4 pi r),  zht = zg (ik - 1/r) (-(y_q - x).n_x / r),  beta0 = physics.burton_miller_beta() -- the UNSCALED
// coupling, whatever beta the matrix was built with.  One warp per row, lanes over the listed columns; the near / far split is
// the far kernel's (pairs inside the guard band belong to the exact near kernel, which adds their term itself).
template <int NQ>
__global__ void __launch_bounds__(256)
rhs_far_kernel(const double* __restrict__ far_k, const double* __restrict__ far_c, const uint32_t* __restrict__ cols, uint32_t ncols,
               const double* __restrict__ srcdat, const cplx* __restrict__ bc_val, const uint8_t* __restrict__ bc_len,
               uint64_t row_begin, uint64_t row_end, double wavruim, double gamtau, cplx beta0, cplx* __restrict__ rhs) {
    constexpr bool QUAD = (NQ == NQ_QUAD);
    const RuleConst& rc = QUAD ? d_rule_quad : d_rule_tri;
    const int lane = threadIdx.x & 31;
    const uint64_t row = row_begin + (((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (row >= row_end) return;
    const double* sp = srcdat + 8ull * row;
    const double sx = sp[0], sy = sp[1], sz = sp[2], nxx = sp[3], nxy = sp[4], nxz = sp[5];
    double accr = 0.0, acci = 0.0;
    for (uint32_t ci = lane; ci < ncols; ci += 32) {
        const uint32_t col = cols[ci];
        if ((uint64_t)col == row) continue;  // the self term belongs to self_kernel
        const uint32_t tile = col / TILE, t = col % TILE;
        const double* fc = far_c + (uint64_t)tile * FAR_NCONST * TILE + t;
        const double* fk = far_k + (uint64_t)tile * NQ_MAX * TILE + t;
        const double dx = fc[FC_Y0X * TILE] - sx, dy = fc[FC_Y0Y * TILE] - sy, dz = fc[FC_Y0Z * TILE] - sz;
        const double e1x = fc[FC_E1X * TILE], e1y = fc[FC_E1Y * TILE], e1z = fc[FC_E1Z * TILE];
        const double e2x = fc[FC_E2X * TILE], e2y = fc[FC_E2Y * TILE], e2z = fc[FC_E2Z * TILE];
        const double D = fma(dz, dz, fma(dy, dy, dx * dx));
        const double p1 = fma(dz, e1z, fma(dy, e1y, dx * e1x));
        const double p2 = fma(dz, e2z, fma(dy, e2y, dx * e2x));
        double d2c = D;
        if (QUAD) d2c = fma(rc.ac2, p1, fma(rc.bc2, p2, D + fc[FC_KC * TILE]));
        if (d2c < fc[FC_THR * TILE]) continue;  // near pair: the exact kernel integrates it (and its right-hand-side term)
        const double M0 = fma(dz, nxz, fma(dy, nxy, dx * nxx));
        const double E1 = fma(e1z, nxz, fma(e1y, nxy, e1x * nxx));
        const double E2 = fma(e2z, nxz, fma(e2y, nxy, e2x * nxx));
        const int bl = bc_len[col];
        cplx bc[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) bc[i] = i < bl ? bc_val[4ull * col + i] : C(0, 0);
        double pr = 0.0, pi = 0.0;
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            const double r2 = (q == 0) ? D : fma(rc.a2[q], p1, fma(rc.b2[q], p2, D + fk[q * TILE]));
            const double rho = fast_rsqrt(r2);
            const double r = r2 * rho;
            double sn, cs;
            fast_sincos(wavruim * r, sn, cs);
            const double m = (q == 0) ? M0 : fma(rc.a[q], E1, fma(rc.b[q], E2, M0));
            // shape functions at the point (only the first bc_len take part: regular.rs:159-164)
            double N[4];
            if (QUAD) {
                const double s1 = 0.25 * (rc.xi[q] + 1.0), s2 = 0.25 * (rc.xi[q] - 1.0), t1 = rc.eta[q] + 1.0, t2 = rc.eta[q] - 1.0;
                N[0] = s1 * t1; N[1] = -s2 * t1; N[2] = s2 * t2; N[3] = -s1 * t2;
            } else {
                N[0] = 1.0 - rc.xi[q] - rc.eta[q]; N[1] = rc.xi[q]; N[2] = rc.eta[q]; N[3] = 0.0;
            }
            double zr = 0.0, zi = 0.0;
#pragma unroll
            for (int i = 0; i < 4; ++i) { zr = fma(bc[i].re, N[i], zr); zi = fma(bc[i].im, N[i], zi); }
            const double g = rc.w[q] * rho;               // w / r   (J / 4 pi applied once per pair)
            const double gr = g * cs, gi = g * sn;        // zg
            // zht = zg (-rho + i k) (-m rho) = zg (m rho^2 - i k m rho)
            const double hr = m * rho * rho, hi = -wavruim * m * rho;
            const double tr = gr * hr - gi * hi, ti = gr * hi + gi * hr;
            // (zg gamma tau + zht beta0) * zbgao
            const double fr = gr * gamtau + (tr * beta0.re - ti * beta0.im), fi = gi * gamtau + (tr * beta0.im + ti * beta0.re);
            pr += fr * zr - fi * zi;
            pi += fr * zi + fi * zr;
        }
        const double j4pi = fc[FC_J4PI * TILE];
        accr = fma(pr, j4pi, accr);
        acci = fma(pi, j4pi, acci);
    }
#pragma unroll
    for (int mm = 16; mm >= 1; mm >>= 1) {
        accr += __shfl_xor_sync(0xffffffffu, accr, mm);
        acci += __shfl_xor_sync(0xffffffffu, acci, mm);
    }
    if (lane == 0) {
        atomicAdd(&rhs[row - row_begin].re, accr);
        atomicAdd(&rhs[row - row_begin].im, acci);
    }
}

bool g_tables_uploaded[64] = {false};

cudaError_t upload_tables() {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 64 && g_tables_uploaded[dev]) return cudaSuccess;
    RuleConst tri = {}, quad = {};
    for (int q = 0; q < NQ_TRI; ++q) {  // gauss.rs:67-89
        tri.w[q] = hosttab::BEMQ_TR13[q][2] * 0.5;
        tri.a[q] = hosttab::BEMQ_TR13[q][0] - hosttab::BEMQ_TR13[0][0];
        tri.b[q] = hosttab::BEMQ_TR13[q][1] - hosttab::BEMQ_TR13[0][1];
        tri.xi[q] = hosttab::BEMQ_TR13[q][0];
        tri.eta[q] = hosttab::BEMQ_TR13[q][1];
    }
    tri.ac = 0.0; tri.bc = 0.0;  // q = 0 of TR13 is the centroid
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j) {  // gauss.rs:94-105, i outer
            const int q = i * 4 + j;
            quad.w[q] = hosttab::BEMQ_GL4_W[i] * hosttab::BEMQ_GL4_W[j];
            quad.a[q] = hosttab::BEMQ_GL4_X[i] - hosttab::BEMQ_GL4_X[0];
            quad.b[q] = hosttab::BEMQ_GL4_X[j] - hosttab::BEMQ_GL4_X[0];
            quad.xi[q] = hosttab::BEMQ_GL4_X[i];
            quad.eta[q] = hosttab::BEMQ_GL4_X[j];
        }
    quad.ac = -hosttab::BEMQ_GL4_X[0]; quad.bc = -hosttab::BEMQ_GL4_X[0];  // centre (0,0) relative to q = 0
    for (RuleConst* r : {&tri, &quad}) {
        for (int q = 0; q < NQ_MAX; ++q) { r->a2[q] = 2.0 * r->a[q]; r->b2[q] = 2.0 * r->b[q]; }
        r->ac2 = 2.0 * r->ac; r->bc2 = 2.0 * r->bc;
    }
    {
        double2 tab[SINCOS_TAB];
        for (int i = 0; i < SINCOS_TAB; ++i) {
            const long double ang = (long double)i * (3.14159265358979323846264338327950288L / (long double)SINCOS_STEPS_PER_PI);
            tab[i] = make_double2((double)cosl(ang), (double)sinl(ang));
        }
        tab[0] = make_double2(1.0, 0.0); tab[SINCOS_TAB / 4] = make_double2(0.0, 1.0);
        tab[SINCOS_TAB / 2] = make_double2(-1.0, 0.0); tab[3 * SINCOS_TAB / 4] = make_double2(0.0, -1.0);
        e = cudaMemcpyToSymbol(d_sincos_tab, tab, sizeof tab);
        if (e != cudaSuccess) return e;
    }
    e = cudaMemcpyToSymbol(d_rule_tri, &tri, sizeof tri);
    if (e != cudaSuccess) return e;
    e = cudaMemcpyToSymbol(d_rule_quad, &quad, sizeof quad);
    if (e != cudaSuccess) return e;
    if (dev < 64) g_tables_uploaded[dev] = true;
    return cudaSuccess;
}

template <int NQ, bool BIMAG, bool ADM>
cudaError_t launch_far_v(const DeviceMesh& m, const Phys& ph, uint64_t row_begin, uint64_t row_end, cplx* A, uint64_t lda,
                         uint2* near_list, unsigned int near_cap, unsigned int* near_count, int background_blocks_per_sm,
                         unsigned int* work_counter, FarRelaunch* relaunch, cudaStream_t s) {
    const uint64_t nrows = row_end - row_begin;
    // enough work items to fill 148 SMs x FAR_MINB resident blocks several times over, but row chunks
    // long enough to amortise the per-block set-up
    uint32_t rpb = 128;
    while (rpb > 8 && (uint64_t)m.ntiles * ((nrows + rpb - 1) / rpb) < 148ull * FAR_MINB * 4ull) rpb >>= 1;
    const uint32_t nchunks = (uint32_t)((nrows + rpb - 1) / rpb);
    const uint32_t total = m.ntiles * nchunks;
    uint32_t grid = total, ipb = 1;
    unsigned int* counter = nullptr;
    if (background_blocks_per_sm > 0 && total > 148u * (uint32_t)background_blocks_per_sm) {
        grid = 148u * (uint32_t)background_blocks_per_sm;  // persistent, polite grid
        ipb = (total + grid - 1) / grid;
        grid = (total + ipb - 1) / ipb;
        counter = work_counter;  // dynamic item distribution (pre-zeroed by the caller) when a boost may join
    }
    const double cH = ph.sign * ph.gamma * ph.tau;
    const double *far_k = m.far_k, *far_c = m.far_c, *src = m.src;
    const uint8_t* col_class = m.col_class;
    const uint32_t n = m.n;
    const double wavruim = ph.wavruim, k2 = ph.k2, bre = ph.beta.re, bim = ph.beta.im;
    const CisConst cis = make_cis_const(ph.wavruim);
    const cplx* adm = ph.adm;
    const double gamtau = ph.gamma * ph.tau;
    constexpr size_t TAB_BYTES = SINCOS_TAB * sizeof(double2);
    {
        static std::atomic<unsigned char> attr_done[64];
        int dev = 0;
        cudaGetDevice(&dev);
        if (dev < 0 || dev >= 64) dev = 63;
        if (!attr_done[dev].load()) {
            cudaError_t ae = cudaFuncSetAttribute(far_kernel<NQ, BIMAG, ADM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TAB_BYTES);
            if (ae != cudaSuccess) return ae;
            attr_done[dev].store(1);
        }
    }
    auto launch = [=](cudaStream_t st, unsigned int g, unsigned int* ctr) -> cudaError_t {
        far_kernel<NQ, BIMAG, ADM><<<g, TILE, TAB_BYTES, st>>>(far_k, far_c, col_class, src, n, row_begin, row_end, rpb, nchunks, total,
                                                       ipb, wavruim, cis, k2, cH, bre, bim, A, lda, near_list, near_cap, near_count, ctr,
                                                       adm, gamtau);
        return cudaGetLastError();
    };
    if (counter && relaunch) {
        // helper launch for bemb200_matrix_boost_assembly: a full-occupancy grid pulling from the same counter
        const unsigned int hg = total < 148u * FAR_MINB ? total : 148u * FAR_MINB;
        relaunch->push_back([=](cudaStream_t st) { return launch(st, hg, counter); });
    }
    return launch(s, grid, counter);
}

template <int NQ>
cudaError_t launch_far_t(const DeviceMesh& m, const Phys& ph, uint64_t row_begin, uint64_t row_end, cplx* A, uint64_t lda,
                         uint2* near_list, unsigned int near_cap, unsigned int* near_count, int bg, unsigned int* work_counter,
                         FarRelaunch* relaunch, cudaStream_t s) {
    const bool bimag = (ph.beta.re == 0.0);
    if (ph.adm) {  // admittance columns: one instantiation per beta form
        if (bimag) return launch_far_v<NQ, true, true>(m, ph, row_begin, row_end, A, lda, near_list, near_cap, near_count, bg, work_counter,
                                                       relaunch, s);
        return launch_far_v<NQ, false, true>(m, ph, row_begin, row_end, A, lda, near_list, near_cap, near_count, bg, work_counter,
                                             relaunch, s);
    }
    if (bimag) return launch_far_v<NQ, true, false>(m, ph, row_begin, row_end, A, lda, near_list, near_cap, near_count, bg, work_counter,
                                                    relaunch, s);
    return launch_far_v<NQ, false, false>(m, ph, row_begin, row_end, A, lda, near_list, near_cap, near_count, bg, work_counter, relaunch, s);
}

}  // namespace

cudaError_t launch_rhs_far(const DeviceMesh& m, const Phys& ph, uint64_t row_begin, uint64_t row_end, cplx* rhs, cudaStream_t s) {
    if (row_end <= row_begin || (m.n_rhs_tri == 0 && m.n_rhs_quad == 0)) return cudaSuccess;
    cudaError_t e = upload_tables();
    if (e != cudaSuccess) return e;
    const uint64_t nrows = row_end - row_begin;
    const unsigned blocks = (unsigned)((nrows * 32 + 255) / 256);
    const double gamtau = ph.gamma * ph.tau;
    if (m.n_rhs_tri)
        rhs_far_kernel<NQ_TRI><<<blocks, 256, 0, s>>>(m.far_k, m.far_c, m.rhs_cols_tri, m.n_rhs_tri, m.src, m.bc_val, m.bc_len, row_begin,
                                                     row_end, ph.wavruim, gamtau, ph.beta_unscaled, rhs);
    if (m.n_rhs_quad)
        rhs_far_kernel<NQ_QUAD><<<blocks, 256, 0, s>>>(m.far_k, m.far_c, m.rhs_cols_quad, m.n_rhs_quad, m.src, m.bc_val, m.bc_len, row_begin,
                                                      row_end, ph.wavruim, gamtau, ph.beta_unscaled, rhs);
    return cudaGetLastError();
}

int far_kernel_launch_count(const DeviceMesh& m) { return (m.n_flat_tri ? 1 : 0) + (m.n_flat_quad ? 1 : 0); }

cudaError_t launch_far(const DeviceMesh& m, const Phys& ph, uint64_t row_begin, uint64_t row_end, cplx* A, uint64_t lda,
                       uint2* near_list, unsigned int near_cap, unsigned int* near_count, int background_blocks_per_sm,
                       unsigned int* work_counters, FarRelaunch* relaunch, cudaStream_t s) {
    if (row_end <= row_begin) return cudaSuccess;
    cudaError_t e = upload_tables();
    if (e != cudaSuccess) return e;
    if (m.n_flat_tri) {
        e = launch_far_t<NQ_TRI>(m, ph, row_begin, row_end, A, lda, near_list, near_cap, near_count, background_blocks_per_sm,
                                 work_counters ? work_counters + 0 : nullptr, relaunch, s);
        if (e != cudaSuccess) return e;
    }
    if (m.n_flat_quad) {
        e = launch_far_t<NQ_QUAD>(m, ph, row_begin, row_end, A, lda, near_list, near_cap, near_count, background_blocks_per_sm,
                                  work_counters ? work_counters + 1 : nullptr, relaunch, s);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

}  // namespace bemb
