// gmres_fused.cu -- the whole restarted GMRES solve (math-solvers/src/iterative/gmres.rs:105-277 and the
// left-preconditioned variant :434-585) as ONE persistent cooperative kernel per rank: streaming ZGEMV,
// row-sharded Gram-Schmidt, Givens / convergence test, solution update and restarts all happen on the
// device; the host launches once and reads one result record.
//
// Layout (P ranks, G CTAs per rank, 512 threads per CTA):
//   * rank p owns rows [p*chunk, (p+1)*chunk) of A and the same slice of every vector (Krylov basis V,
//     x, b); CTA c of the rank owns the contiguous rows [c*S, (c+1)*S) of that slice, S = ceil(chunk/G).
//     Everything element-wise (ZGEMV rows, inner-product partials, the w -= V h update, x += V y) is done
//     by the owning CTA on its own rows: no grid barrier between those steps.
//   * full-length vectors (the matvec input) travel through an exchange buffer in "flag-in-data" form:
//     a complex number is two 16-byte words {lo32, epoch, hi32, epoch}, written with st.volatile (8-byte
//     halves are single-copy atomic), so a consumer that sees the right epoch in all four flags has the
//     value -- no fence, no counter.  Every producer stores its rows into EVERY rank's buffer (NVLink peer
//     memory for the others), consumers poll their local copy: this is the all-gather of the Krylov vector.
//   * ONE reduction round per Arnoldi iteration (north_star: "dot products reduced with all-reduce"): CTA
//     partials -> reducer CTA of the rank (fixed order) -> rank partials to every rank (fixed order) ->
//     every rank's reducer holds bit-identical totals, runs the (j+1)-term forward substitution and the
//     Givens update redundantly, and broadcasts the Hessenberg column / stop decision to its CTAs.
//
// One round per iteration needs the norm of the new basis vector in the SAME reduction as the next
// inner products.  The kernel therefore keeps u_j = (un-normalised) w - V h, runs the matvec on u_j and
// uses linearity: with s = 1/||u_j||, v_j = s u_j, w = A v_j = s (A u_j),
//        a_l = v_l^H w = s (v_l^H A u_j)  (l < j),   a_j = s^2 (u_j^H A u_j),   L_jl = v_j^H v_l = s (u_j^H v_l),
// (I + L) h = a  gives exactly the modified Gram-Schmidt coefficients of gmres.rs:184-188 (same algebra
// as mgs_lowsync_kernel in linalg.cu), and h_{j,j-1} = ||u_j|| completes the previous Hessenberg column.
// The convergence test of column j-1 is therefore taken one matvec late: a solve costs one A-product more
// than the reference's count, the reported iteration/restart numbers are the reference's.
#include <cooperative_groups.h>
#include <atomic>
#include <cstring>

#include "api_internal.h"
#include "gmres_fused.h"

namespace bemb {

namespace {

constexpr int FT = FUSED_THREADS;   // threads per CTA
constexpr int NW = FT / 32;         // warps per CTA
constexpr int KMAX = FUSED_KMAX;    // values per reduction round: 2 (restart + 1) + 2 <= 130

__device__ __forceinline__ unsigned long long gtimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// ---- flag-in-data words -------------------------------------------------------------------------
__device__ __forceinline__ void ll_put(uint4* dst, cplx v, uint32_t flag) {
    const uint32_t rl = (uint32_t)__double2loint(v.re), rh = (uint32_t)__double2hiint(v.re);
    const uint32_t il = (uint32_t)__double2loint(v.im), ih = (uint32_t)__double2hiint(v.im);
    asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "r"(rl), "r"(flag), "r"(rh), "r"(flag) : "memory");
    asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(dst + 1), "r"(il), "r"(flag), "r"(ih), "r"(flag) : "memory");
}
__device__ __forceinline__ bool ll_try(const uint4* q, uint32_t flag, cplx& out) {
    uint4 a, b;
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w) : "l"(q) : "memory");
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "l"(q + 1) : "memory");
    if (a.y == flag && a.w == flag && b.y == flag && b.w == flag) {
        out = C(__hiloint2double((int)a.z, (int)a.x), __hiloint2double((int)b.z, (int)b.x));
        return true;
    }
    return false;
}

struct Ctl {
    volatile int* abort_s;        // shared flag of the CTA: somebody gave up waiting
    unsigned long long timeout_ns;
    FusedResult* result;
};

// wait for N flag-in-data elements (addresses q[e], skipped when !want[e]); all outstanding loads of a pass are issued
// back to back.  Bounded: after timeout_ns the CTA-wide abort flag is raised and the wait returns (values undefined).
template <int N>
__device__ __forceinline__ void ll_wait_many(cplx (&out)[N], const uint4* const (&q)[N], const bool (&want)[N], uint32_t flag, const Ctl& ctl) {
    bool have[N];
#pragma unroll
    for (int e = 0; e < N; ++e) { have[e] = !want[e]; out[e] = C(0, 0); }
    unsigned long long t0 = 0;
    unsigned spins = 0;
    for (;;) {
        bool all = true;
#pragma unroll
        for (int e = 0; e < N; ++e)
            if (!have[e]) { have[e] = ll_try(q[e], flag, out[e]); all = all && have[e]; }
        if (all) return;
        // back off between passes: thousands of threads spinning on L2 would starve the producers they are waiting for
        __nanosleep(spins < 4 ? 40u : (spins < 16 ? 120u : 400u));
        if ((++spins & 255u) == 0) {
            if (*ctl.abort_s) return;
            const unsigned long long t = gtimer();
            if (t0 == 0) t0 = t;
            else if (t - t0 > ctl.timeout_ns) {
                *ctl.abort_s = 1;
                ctl.result->error = 1;
                return;
            }
        }
    }
}
// spin (bounded, with back-off) until ONE element carries `flag`; used by a few probe lanes so that the bulk of the
// consumers touches the buffer only when the data is (almost certainly) there
__device__ __forceinline__ void ll_probe(const uint4* q, uint32_t flag, const Ctl& ctl) {
    cplx dummy;
    unsigned long long t0 = 0;
    unsigned spins = 0;
    while (!ll_try(q, flag, dummy)) {
        __nanosleep(spins < 8 ? 60u : 250u);
        if ((++spins & 255u) == 0) {
            if (*ctl.abort_s) return;
            const unsigned long long t = gtimer();
            if (t0 == 0) t0 = t;
            else if (t - t0 > ctl.timeout_ns) {
                *ctl.abort_s = 1;
                ctl.result->error = 1;
                return;
            }
        }
    }
}
__device__ __forceinline__ cplx ll_wait1(const uint4* q, uint32_t flag, const Ctl& ctl) {
    cplx out[1];
    const uint4* const qq[1] = {q};
    const bool want[1] = {true};
    ll_wait_many<1>(out, qq, want, flag, ctl);
    return out[0];
}

// NV per-lane partial sums -> lane 4*v ends up with the warp total of value v (NV = 8) resp. lane 8*v (NV = 4);
// fixed order, NV - 1 + log2(32 / NV) shuffles instead of 5 NV
template <int NV>
__device__ __forceinline__ double warp_fold(double (&v)[NV], int lane) {
    static_assert(NV == 4 || NV == 8, "fold width");
    int off = 16;
#pragma unroll
    for (int cnt = NV / 2; cnt >= 1; cnt >>= 1, off >>= 1) {
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < cnt; ++i) {
            const double send = upper ? v[i] : v[i + cnt];
            const double keep = upper ? v[i + cnt] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
    }
    double r = v[0];
    for (; off >= 1; off >>= 1) r += __shfl_xor_sync(0xffffffffu, r, off);
    return r;
}

__device__ __forceinline__ cplx ldcg_c(const cplx* p) {
    const double2 v = __ldcg(reinterpret_cast<const double2*>(p));
    return C(v.x, v.y);
}
__device__ __forceinline__ void cfma2(double& are, double& aim, double2 a, cplx x) {
    are = fma(a.x, x.re, are);
    are = fma(-a.y, x.im, are);
    aim = fma(a.x, x.im, aim);
    aim = fma(a.y, x.re, aim);
}

// ---- reference arithmetic of the small dense part (no FMA contraction, num-complex operation order) ----
__device__ __forceinline__ cplx rmul(cplx a, cplx b) {
    return C(__dsub_rn(__dmul_rn(a.re, b.re), __dmul_rn(a.im, b.im)), __dadd_rn(__dmul_rn(a.re, b.im), __dmul_rn(a.im, b.re)));
}
__device__ __forceinline__ cplx radd(cplx a, cplx b) { return C(__dadd_rn(a.re, b.re), __dadd_rn(a.im, b.im)); }
__device__ __forceinline__ cplx rsub(cplx a, cplx b) { return C(__dsub_rn(a.re, b.re), __dsub_rn(a.im, b.im)); }
__device__ __forceinline__ double rnorm_sqr(cplx a) { return __dadd_rn(__dmul_rn(a.re, a.re), __dmul_rn(a.im, a.im)); }
__device__ __forceinline__ double rnorm(cplx a) { return __dsqrt_rn(rnorm_sqr(a)); }

// shared-memory carve-up (dynamic)
struct Smem {
    double* ypart;   // [rblk][NW][2]  matvec partial sums (re, im) per row and warp; P2 aliases it
    cplx* w_s;       // [S]  A z on this CTA's rows
    cplx* u_s;       // [S]  u_j (un-normalised current basis vector) on this CTA's rows
    cplx* part_s;    // [KMAX] this CTA's partials of the round
    cplx* bc_s;      // [KMAX] broadcast payload of the round
    // reducer CTA only
    cplx* red4;      // [strands][Kpad] <= FT entries
    cplx* tot_s;     // [KMAX]
    cplx* Lp;        // packed strictly-lower Gram triangle, column-major: L(k,l), k > l
    cplx* Rp;        // packed upper triangle of the rotated Hessenberg matrix, column-major: R(i,c), i <= c
    cplx* cs;        // [m]
    cplx* sn;        // [m]
    cplx* g;         // [m+1]
    cplx* hprev;     // [m+1] un-rotated column j-1 (h_0 .. h_{j-1})
    cplx* ycoef;     // [m]
};

__device__ __forceinline__ int lp_off(int l, int m1) { return l * m1 - (l * (l + 1)) / 2 - l - 1; }  // + k  (k > l), m1 = m + 1
__device__ __forceinline__ int rp_off(int c) { return (c * (c + 1)) / 2; }                          // + i  (i <= c)

// ---- y = A z on this CTA's rows -------------------------------------------------------------------
// z is read from the local exchange buffer (epoch `ex`).  Warp wq owns columns [sg*SEGW + wq*128, +128) of every
// segment sg: its 4 x-values per lane stay in registers while it walks the CTA's rows two pairs at a time (16
// independent 16-byte streaming loads in flight per lane); per (row pair, warp) partial sums are accumulated in shared
// memory in segment order and added over the warps in warp order: deterministic.
// Boundary rows.  With `units` (p.unit_off) the CTA boundaries sit at (row, segment) granularity -- a row is nseg units,
// so shares are balanced to a fraction of a percent even when a CTA owns only ~17 rows (8 ranks) -- and the row a boundary
// cuts through is computed by TWO CTAs: the upper one (which owns the row: it holds the row's first segments in visiting
// order) and the next CTA, which computes the remaining segments ("head fragment") and hands its partial sum to the owner
// through one flag-in-data slot.  Frag describes that for one CTA.
struct Frag {
    bool has_head;   // this CTA computes the tail segments (visiting positions >= s0) of row rb - 1 for CTA cta - 1
    uint32_t s0;
    uint32_t s1;     // visiting positions < s1 of this CTA's LAST owned row are computed here, the rest by CTA cta + 1
};

template <int RB, int CPL>
__device__ __forceinline__ void matvec_rows(const FusedParams& p, const Smem& sm, uint32_t rb, uint32_t sc, const Frag& fr, uint32_t ex,
                                            const Ctl& ctl) {
    constexpr int WCOLS = 32 * CPL;   // columns per warp and segment
    constexpr int SEGW = NW * WCOLS;  // columns per segment
    static_assert(RB == 2 || RB == 4, "rows per step");
    static_assert(SEGW == FUSED_SEGMENT_WIDTH, "the host sizes the row-balancing units by FUSED_SEGMENT_WIDTH");
    const int tid = threadIdx.x, lane = tid & 31, wq = tid >> 5;
    const uint4* xin = p.xbuf[p.rank] + (size_t)(ex & 1u) * 2 * p.npad;
    const uint32_t n = p.n;
    const uint32_t nseg = (n + SEGW - 1) / SEGW;
    const uint32_t head = fr.has_head ? 1u : 0u;
    // slot 0 of ypart is the head-fragment row (row rb - 1) when there is one; owned row i sits in slot head + i
    for (uint32_t blk = 0; blk < sc + head; blk += p.rblk) {
        const uint32_t nslots = sc + head - blk < p.rblk ? sc + head - blk : p.rblk;
        for (uint32_t e = tid; e < nslots * NW * 2; e += FT) sm.ypart[e] = 0.0;
        __syncthreads();
        // segments are visited starting with the rank's OWN columns (their part of the vector is published locally and
        // is there first); the other ranks' parts cross NVLink while this rank already streams
        const uint32_t sg0 = (uint32_t)(((uint64_t)p.row0 + SEGW / 2) / SEGW) % nseg;
        for (uint32_t si = 0; si < nseg; ++si) {
            const uint32_t sg = si + sg0 < nseg ? si + sg0 : si + sg0 - nseg;
            const uint32_t cbase = sg * SEGW + wq * WCOLS;
            if (cbase >= n) continue;  // warp-uniform: no columns for this warp in this segment
            // slots of this block that take part in this segment: the head row only from position s0 on, the last owned row
            // only before position s1
            uint32_t lo = 0, hi = nslots;
            if (blk == 0 && head && si < fr.s0) lo = 1;
            if (blk + nslots == sc + head && sc > 0 && si >= fr.s1) hi -= 1;
            if (lo >= hi) continue;
            cplx xr[CPL];
            uint32_t col[CPL];
            {
                const uint4* q[CPL];
                bool want[CPL];
#pragma unroll
                for (int c = 0; c < CPL; ++c) {
                    const uint32_t cc = cbase + lane + 32 * c;
                    want[c] = cc < n;
                    col[c] = cc < n ? cc : n - 1;  // clamped address, zero x: contributes nothing
                    q[c] = xin + 2 * (size_t)col[c];
                }
                // two probe lanes per warp wait for the ends of the warp's column slab, then everybody loads
                if ((lane == 0 && want[0]) || (lane == 31 && want[CPL - 1])) ll_probe(lane == 0 ? q[0] : q[CPL - 1], ex, ctl);
                __syncwarp();
                ll_wait_many<CPL>(xr, q, want, ex, ctl);
            }
            const cplx* arow = p.A + ((size_t)rb + blk + lo - head) * p.lda;  // slot s <-> slab row rb - head + blk + s
            for (uint32_t r0 = lo; r0 < hi; r0 += RB, arow += RB * p.lda) {
                const uint32_t nr = hi - r0;  // rows left (warp-uniform); rows beyond it are neither loaded nor stored
                double2 a[RB][CPL];
#pragma unroll
                for (int r = 0; r < RB; ++r) {
                    if ((uint32_t)r < nr) {
#pragma unroll
                        for (int c = 0; c < CPL; ++c) a[r][c] = __ldcs(reinterpret_cast<const double2*>(arow + (size_t)r * p.lda + col[c]));
                    } else {
#pragma unroll
                        for (int c = 0; c < CPL; ++c) a[r][c] = make_double2(0.0, 0.0);
                    }
                }
                double acc[2 * RB];
#pragma unroll
                for (int v = 0; v < 2 * RB; ++v) acc[v] = 0.0;
#pragma unroll
                for (int c = 0; c < CPL; ++c)
#pragma unroll
                    for (int r = 0; r < RB; ++r) cfma2(acc[2 * r], acc[2 * r + 1], a[r][c], xr[c]);
                const double tot = warp_fold<2 * RB>(acc, lane);  // lane (32 / (2 RB)) v holds value v = 2 r + (re | im)
                constexpr int LSH = RB == 4 ? 2 : 3;
                if ((lane & ((1 << LSH) - 1)) == 0) {
                    const int v = lane >> LSH;
                    if ((uint32_t)(v >> 1) < nr) sm.ypart[((size_t)(r0 + (v >> 1)) * NW + wq) * 2 + (v & 1)] += tot;
                }
            }
        }
        __syncthreads();
        for (uint32_t t = tid; t < nslots; t += FT) {
            const double* yp = sm.ypart + (size_t)t * NW * 2;
            double sr = 0.0, si = 0.0;
#pragma unroll
            for (int w = 0; w < NW; ++w) { sr += yp[w * 2]; si += yp[w * 2 + 1]; }
            const uint32_t slot = blk + t;
            if (head && slot == 0) {
                // head fragment: partial sum of row rb - 1 for its owner, CTA cta - 1
                ll_put(p.frag + ((size_t)(ex & 1u) * gridDim.x + blockIdx.x) * 2, C(sr, si), ex);
            } else {
                sm.w_s[slot - head] = C(sr, si);
            }
        }
        __syncthreads();
    }
    if (sc > 0 && fr.s1 < nseg) {
        // the rest of my last row comes from the next CTA
        if (tid == 0) {
            const cplx o = ll_wait1(p.frag + ((size_t)(ex & 1u) * gridDim.x + blockIdx.x + 1) * 2, ex, ctl);
            sm.w_s[sc - 1].re += o.re;
            sm.w_s[sc - 1].im += o.im;
        }
        __syncthreads();
    }
}

// publish `vals[i]` (this CTA's rows) as epoch `ex` of the full vector into every rank's exchange buffer
__device__ __forceinline__ void publish_rows(const FusedParams& p, const cplx* vals, uint32_t rb, uint32_t sc, uint32_t ex) {
    const size_t g0 = (size_t)p.row0 + rb;
    for (uint32_t i = threadIdx.x; i < sc; i += FT) {
        const cplx v = vals[i];
#pragma unroll
        for (int r = 0; r < MAX_PEERS; ++r)
            if (r < p.nranks) ll_put(p.xbuf[r] + ((size_t)(ex & 1u) * p.npad + g0 + i) * 2, v, ex);
    }
}

// One reduction round.  In: part_s[0..K) of every CTA of every rank.  Reducer CTAs: tot_s[0..K) = totals (identical on
// every rank).  Returns after the reducer-side totals are in place (other CTAs return immediately after posting).
__device__ __forceinline__ void round_gather(const FusedParams& p, const Smem& sm, int K, uint32_t er, const Ctl& ctl) {
    const int tid = threadIdx.x;
    const uint32_t cta = blockIdx.x, G = gridDim.x;
    if (tid < K) ll_put(p.cpart + (((size_t)(er & 1u) * G + cta) * KMAX + tid) * 2, sm.part_s[tid], er);
    if (cta != 0) return;
    // ---- reducer: CTA partials in CTA order (FT / Kpad strands of consecutive CTAs, combined in strand order) ----
    const int kpad = (K + 31) & ~31;
    const int nstr = FT / kpad;
    {
        const int k = tid % kpad, q = tid / kpad;
        const uint32_t per = (G + nstr - 1) / nstr;
        const uint32_t c0 = q * per < G ? q * per : G, c1 = (c0 + per < G) ? c0 + per : G;
        cplx t = C(0, 0);
        if (k < K && q < nstr) {
            constexpr int GB = 10;  // partials in flight per thread and pass (148 CTAs in 8 strands: two passes)
            for (uint32_t c = c0; c < c1; c += GB) {
                cplx v[GB];
                const uint4* qq[GB];
                bool want[GB];
#pragma unroll
                for (int e = 0; e < GB; ++e) {
                    want[e] = c + e < c1;
                    qq[e] = p.cpart + (((size_t)(er & 1u) * G + (want[e] ? c + e : c)) * KMAX + k) * 2;
                }
                ll_wait_many<GB>(v, qq, want, er, ctl);
#pragma unroll
                for (int e = 0; e < GB; ++e) { t.re += v[e].re; t.im += v[e].im; }
            }
            sm.red4[q * kpad + k] = t;
        }
    }
    __syncthreads();
    if (tid < K) {
        cplx t = sm.red4[tid];
        for (int q = 1; q < nstr; ++q) { t.re += sm.red4[q * kpad + tid].re; t.im += sm.red4[q * kpad + tid].im; }
        if (p.nranks > 1) {
            // rank partial -> every rank's inbox; totals in rank order
#pragma unroll
            for (int r = 0; r < MAX_PEERS; ++r)
                if (r < p.nranks) ll_put(p.rpart[r] + (((size_t)(er & 1u) * p.nranks + p.rank) * KMAX + tid) * 2, t, er);
            cplx s = C(0, 0);
            for (int r0 = 0; r0 < p.nranks; r0 += 8) {
                cplx v[8];
                const uint4* qq[8];
                bool want[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    want[e] = r0 + e < p.nranks;
                    qq[e] = p.rpart[p.rank] + (((size_t)(er & 1u) * p.nranks + (want[e] ? r0 + e : r0)) * KMAX + tid) * 2;
                }
                ll_wait_many<8>(v, qq, want, er, ctl);
#pragma unroll
                for (int e = 0; e < 8; ++e) { s.re += v[e].re; s.im += v[e].im; }
            }
            t = s;
        }
        sm.tot_s[tid] = t;
    }
    __syncthreads();
}

// reducer: bc_s[0..nb) -> broadcast slots; everybody: wait for the payload of round `er`
__device__ __forceinline__ void round_broadcast(const FusedParams& p, const Smem& sm, int nb, uint32_t er, const Ctl& ctl) {
    const int tid = threadIdx.x;
    if (blockIdx.x == 0) {
        __syncthreads();  // bc_s complete
        if (tid < nb) ll_put(p.hbuf + ((size_t)(er & 1u) * KMAX + tid) * 2, sm.bc_s[tid], er);
    } else if (tid < nb) {
        sm.bc_s[tid] = ll_wait1(p.hbuf + ((size_t)(er & 1u) * KMAX + tid) * 2, er, ctl);  // (ll_wait_many backs off between polls)
    }
    __syncthreads();
}

// payload codes (bc_s[0].re)
constexpr double CODE_CONTINUE = 0.0, CODE_STOP = 1.0, CODE_RESTART = 2.0;

// Givens update of Hessenberg column c (gmres.rs:204-222) by ONE thread: hprev[0..c] un-rotated, sub = h_{c+1,c}
// (real).  Writes the rotated column to Rp, updates cs/sn/g; returns |g_{c+1}|.
__device__ double givens_column(const Smem& sm, int c, double sub) {
    cplx hc = C(0, 0);  // h[i][c] being carried
    cplx hi = sm.hprev[0];
    for (int i = 0; i < c; ++i) {
        const cplx hn = sm.hprev[i + 1];
        const cplx ci = sm.cs[i], si = sm.sn[i];
        const cplx temp = radd(rmul(conj(ci), hi), rmul(conj(si), hn));
        const cplx nxt = radd(rsub(C(0, 0), rmul(si, hi)), rmul(ci, hn));
        sm.Rp[rp_off(c) + i] = temp;
        hi = nxt;
    }
    hc = hi;  // h[c][c] after the previous rotations
    const cplx hs = C(sub, 0.0);
    cplx cc, ss;
    {  // givens_rotation (gmres.rs:589-603)
        const double tol = 1e-30;
        if (rnorm(hs) < tol) { cc = C(1, 0); ss = C(0, 0); }
        else if (rnorm(hc) < tol) { cc = C(0, 0); ss = C(1, 0); }
        else {
            const double r = __dsqrt_rn(__dadd_rn(rnorm_sqr(hc), rnorm_sqr(hs)));
            const double ir = __ddiv_rn(1.0, r);
            cc = rmul(hc, C(ir, 0.0));
            ss = rmul(hs, C(ir, 0.0));
        }
    }
    sm.cs[c] = cc;
    sm.sn[c] = ss;
    sm.Rp[rp_off(c) + c] = radd(rmul(conj(cc), hc), rmul(conj(ss), hs));
    const cplx g0 = sm.g[c], g1 = sm.g[c + 1];
    const cplx temp = radd(rmul(conj(cc), g0), rmul(conj(ss), g1));
    const cplx gn = radd(rsub(C(0, 0), rmul(ss, g0)), rmul(cc, g1));
    sm.g[c] = temp;
    sm.g[c + 1] = gn;
    return rnorm(gn);
}

// solve_upper_triangular (gmres.rs:606-621) on the rotated k x k system, one thread
__device__ void back_substitute(const Smem& sm, int k) {
    for (int i = k - 1; i >= 0; --i) {
        cplx sum = sm.g[i];
        for (int j = i + 1; j < k; ++j) sum = rsub(sum, rmul(sm.Rp[rp_off(j) + i], sm.ycoef[j]));
        const cplx d = sm.Rp[rp_off(i) + i];
        cplx y = C(0, 0);
        if (rnorm(d) > 1e-30) {
            const double ns = rnorm_sqr(d);
            y = rmul(sum, C(__ddiv_rn(d.re, ns), __ddiv_rn(-d.im, ns)));
        }
        sm.ycoef[i] = y;
    }
}

template <int RB, int CPL>
__device__ __forceinline__ void gmres_body(const FusedParams& p) {
    extern __shared__ __align__(16) unsigned char dyn[];
    __shared__ int abort_s;
    const int tid = threadIdx.x, lane = tid & 31, wq = tid >> 5;
    const uint32_t cta = blockIdx.x, G = gridDim.x;
    const int m = (int)p.restart, m1 = m + 1;

    Smem sm;
    {
        unsigned char* q = dyn;
        auto take = [&](size_t bytes) { unsigned char* r = q; q += (bytes + 15) & ~(size_t)15; return r; };
        sm.ypart = reinterpret_cast<double*>(take((size_t)p.rblk * NW * 2 * sizeof(double) > FT * sizeof(cplx)
                                                      ? (size_t)p.rblk * NW * 2 * sizeof(double) : FT * sizeof(cplx)));
        sm.w_s = reinterpret_cast<cplx*>(take((size_t)p.S * sizeof(cplx)));
        sm.u_s = reinterpret_cast<cplx*>(take((size_t)p.S * sizeof(cplx)));
        sm.part_s = reinterpret_cast<cplx*>(take(KMAX * sizeof(cplx)));
        sm.bc_s = reinterpret_cast<cplx*>(take(KMAX * sizeof(cplx)));
        sm.red4 = reinterpret_cast<cplx*>(take((FT + 32) * sizeof(cplx)));
        sm.tot_s = reinterpret_cast<cplx*>(take(KMAX * sizeof(cplx)));
        sm.Lp = reinterpret_cast<cplx*>(take((size_t)(m1 * m / 2 + 1) * sizeof(cplx)));
        sm.Rp = reinterpret_cast<cplx*>(take((size_t)(m1 * m / 2 + 1) * sizeof(cplx)));
        sm.cs = reinterpret_cast<cplx*>(take(m1 * sizeof(cplx)));
        sm.sn = reinterpret_cast<cplx*>(take(m1 * sizeof(cplx)));
        sm.g = reinterpret_cast<cplx*>(take((m1 + 1) * sizeof(cplx)));
        sm.hprev = reinterpret_cast<cplx*>(take((m1 + 1) * sizeof(cplx)));
        sm.ycoef = reinterpret_cast<cplx*>(take(m1 * sizeof(cplx)));
    }
    if (tid == 0) abort_s = 0;
    __syncthreads();
    Ctl ctl{&abort_s, p.timeout_ns, p.result};

    // rows of this CTA inside the rank's slab: equal shares, or the host's table (shares proportional to the measured
    // streaming speed of the SM each CTA sits on: SMs of fuller GPCs get less HBM bandwidth)
    uint32_t rb, sc;
    Frag fr{false, 0u, 0xffffffffu};
    if (p.unit_off) {
        // boundaries in units of (row, segment position); a row is owned by the CTA holding its first position
        const uint32_t nsegu = p.units_per_row;
        const uint32_t U0 = p.unit_off[cta], U1 = p.unit_off[cta + 1];
        rb = (U0 + nsegu - 1) / nsegu;
        const uint32_t own1 = (U1 + nsegu - 1) / nsegu;
        sc = own1 > rb ? own1 - rb : 0;
        fr.s0 = U0 % nsegu;
        fr.has_head = fr.s0 != 0 && U1 > U0;
        fr.s1 = (U1 % nsegu) ? (U1 % nsegu) : nsegu;
        if (sc == 0) fr.s1 = nsegu;
    } else if (p.row_off) {
        rb = p.row_off[cta];
        sc = p.row_off[cta + 1] - rb;
    } else {
        rb = cta * p.S < p.nloc ? cta * p.S : p.nloc;
        const uint32_t re = rb + p.S < p.nloc ? rb + p.S : p.nloc;
        sc = re - rb;
    }
    unsigned smid = 0;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    uint32_t ex = p.ex0, er = p.er0;
    auto next_epoch = [](uint32_t& e) { e += 1; if (e == 0) e = 1; };

    // reducer-side solve state (CTA 0, thread 0)
    unsigned long long total_iterations = 0, restarts = 0, matvecs = 0;
    double b_norm = 0.0;
    unsigned long long t_begin = 0, t_mv = 0, t_round = 0;
    unsigned long long tc_mv = 0, tc_wait = 0, tc_mark = 0;  // per-CTA trace (thread 0): time inside matvec_rows, time from posting partials to payload
    if (cta == 0 && tid == 0) t_begin = gtimer();
    int final_code = 0;       // 1: converged, 0: cycle budget exhausted
    double final_res = 0.0;

#define ABORT_CHECK()                     \
    do {                                  \
        if (abort_s) return;              \
    } while (0)

    // x -> exchange buffer (epoch ex+1) happens at the top of every cycle
    for (uint32_t outer = 0;; ++outer) {
        // ---- r = b - A x on own rows (with M^-1 for the preconditioned variant) -----------------------------
        next_epoch(ex);
        publish_rows(p, p.x + p.row0 + rb, rb, sc, ex);
        unsigned long long tm0 = 0;
        if (cta == 0 && tid == 0) tm0 = gtimer();
        matvec_rows<RB, CPL>(p, sm, rb, sc, fr, ex, ctl);
        ABORT_CHECK();
        if (cta == 0 && tid == 0) { t_mv += gtimer() - tm0; matvecs += 1; }
        double bn2 = 0.0, rn2 = 0.0;
        for (uint32_t i = tid; i < sc; i += FT) {
            const size_t gi = (size_t)p.row0 + rb + i;
            cplx bv = p.b[gi];
            cplx r = C(bv.re - sm.w_s[i].re, bv.im - sm.w_s[i].im);
            if (p.pinv) { const cplx pv = ldcg_c(p.pinv + gi); r = r * pv; bv = bv * pv; }
            sm.u_s[i] = r;
            rn2 = fma(r.re, r.re, fma(r.im, r.im, rn2));
            bn2 = fma(bv.re, bv.re, fma(bv.im, bv.im, bn2));
        }
        __syncthreads();
        const bool last_pass = outer >= p.max_cycles;  // cycle budget exhausted: only the true residual is wanted
        const bool need_bnorm = outer == 0;
        if (last_pass) {
            // ---- final residual round (gmres.rs:264-276) ------------------------------------------------------
            double v4[4] = {rn2, bn2, 0.0, 0.0};
            const double tot = warp_fold<4>(v4, lane);
            __shared__ double fin_s[NW][2];
            if (lane == 0) fin_s[wq][0] = tot;
            if (lane == 8) fin_s[wq][1] = tot;
            __syncthreads();
            if (tid < 2) {
                double t = 0.0;
                for (int w = 0; w < NW; ++w) t += fin_s[w][tid];
                sm.part_s[tid] = C(t, 0.0);
            }
            __syncthreads();
            next_epoch(er);
            round_gather(p, sm, 2, er, ctl);
            ABORT_CHECK();
            if (cta == 0 && tid == 32) {  // thread 32 owns the solve state (norms, counts, decision)
                if (need_bnorm) b_norm = __dsqrt_rn(sm.tot_s[1].re);
                const double rn = __dsqrt_rn(sm.tot_s[0].re);
                final_code = 0;
                if (need_bnorm && b_norm < 1e-15) { final_code = 1; final_res = 0.0; }
                else final_res = __ddiv_rn(rn, b_norm);
                sm.bc_s[0] = C(CODE_STOP, 0.0);
            }
            round_broadcast(p, sm, 1, er, ctl);
            ABORT_CHECK();
            break;
        }
        // ---- u_0 = r: publish, first Arnoldi matvec ---------------------------------------------------------
        bool stop_all = false;
        for (int j = 0;; ++j) {
            // u_j is in u_s (own rows); j == m: no matvec, only the norm that completes column m-1
            const bool norm_only = j == m;
            if (!norm_only) {
                next_epoch(ex);
                publish_rows(p, sm.u_s, rb, sc, ex);
                if (tid == 0) tm0 = gtimer();
                matvec_rows<RB, CPL>(p, sm, rb, sc, fr, ex, ctl);
                ABORT_CHECK();
                if (tid == 0) { const unsigned long long dt = gtimer() - tm0; tc_mv += dt; if (cta == 0) { t_mv += dt; matvecs += 1; } }
                if (p.pinv) {
                    for (uint32_t i = tid; i < sc; i += FT) sm.w_s[i] = sm.w_s[i] * ldcg_c(p.pinv + p.row0 + rb + i);
                    __syncthreads();
                }
            }
            unsigned long long tr0 = 0;
            if (cta == 0 && tid == 0) tr0 = gtimer();
            // ---- partial inner products over own rows: a'_l = v_l^H w' (l < j), a'_j = u^H w', g'_l = u^H v_l, |u|^2 ----
            const int nv = j + 1;                       // vectors 0..j (vector j is u itself)
            const int K = norm_only ? 1 : 2 * nv + (need_bnorm && j == 0 ? 1 : 0);
            if (norm_only) {
                double v4[4] = {0.0, 0.0, 0.0, 0.0};
                for (uint32_t i = tid; i < sc; i += FT) v4[0] = fma(sm.u_s[i].re, sm.u_s[i].re, fma(sm.u_s[i].im, sm.u_s[i].im, v4[0]));
                const double tot = warp_fold<4>(v4, lane);
                __shared__ double nrm_s[NW];
                if (lane == 0) nrm_s[wq] = tot;
                __syncthreads();
                if (tid == 0) {
                    double t = 0.0;
                    for (int w = 0; w < NW; ++w) t += nrm_s[w];
                    sm.part_s[0] = C(t, 0.0);
                }
            } else {
                // warp wq owns the vectors l = wq, wq + 16, wq + 32, wq + 48 (restart <= 63); their rows are loaded together so that
                // the L2 round trips of the (up to four) vectors overlap
                {
                    constexpr int NP = (FUSED_MAX_RESTART + 1 + NW - 1) / NW;  // 4
                    double acc[NP][4];  // a.re, a.im, g.re, g.im per owned vector
#pragma unroll
                    for (int pq = 0; pq < NP; ++pq)
#pragma unroll
                        for (int c = 0; c < 4; ++c) acc[pq][c] = 0.0;
                    for (uint32_t i = lane; i < sc; i += 32) {
                        const cplx u = sm.u_s[i], w = sm.w_s[i];
                        cplx v[NP];
#pragma unroll
                        for (int pq = 0; pq < NP; ++pq) {
                            const int l = wq + pq * NW;
                            v[pq] = l < j ? ldcg_c(p.V + (size_t)l * p.ldv + rb + i) : C(0, 0);
                        }
#pragma unroll
                        for (int pq = 0; pq < NP; ++pq) {
                            const int l = wq + pq * NW;
                            if (l < j) {
                                acc[pq][0] = fma(v[pq].re, w.re, fma(v[pq].im, w.im, acc[pq][0]));
                                acc[pq][1] = fma(v[pq].re, w.im, fma(-v[pq].im, w.re, acc[pq][1]));
                                acc[pq][2] = fma(u.re, v[pq].re, fma(u.im, v[pq].im, acc[pq][2]));
                                acc[pq][3] = fma(u.re, v[pq].im, fma(-u.im, v[pq].re, acc[pq][3]));
                            } else if (l == j) {
                                acc[pq][0] = fma(u.re, w.re, fma(u.im, w.im, acc[pq][0]));
                                acc[pq][1] = fma(u.re, w.im, fma(-u.im, w.re, acc[pq][1]));
                                acc[pq][2] = fma(u.re, u.re, fma(u.im, u.im, acc[pq][2]));  // |u|^2 rides in the g slot of l = j
                            }
                        }
                    }
                    double* dst = reinterpret_cast<double*>(sm.part_s);
#pragma unroll
                    for (int pq = 0; pq < NP; ++pq) {
                        const int l = wq + pq * NW;
                        if (l < nv) {  // warp-uniform
                            const double tot = warp_fold<4>(acc[pq], lane);  // lane 8 v holds value v
                            if (lane == 0) dst[2 * l] = tot;
                            if (lane == 8) dst[2 * l + 1] = tot;
                            if (lane == 16) dst[2 * (nv + l)] = tot;
                            if (lane == 24) dst[2 * (nv + l) + 1] = tot;
                        }
                    }
                }
                if (K > 2 * nv) {  // ||b||^2 (resp. ||M^-1 b||^2) rides along in the very first round
                    __shared__ double bn_s[NW];
                    double v4[4] = {bn2, 0.0, 0.0, 0.0};
                    const double tot = warp_fold<4>(v4, lane);
                    if (lane == 0) bn_s[wq] = tot;
                    __syncthreads();
                    if (tid == 0) {
                        double t = 0.0;
                        for (int w = 0; w < NW; ++w) t += bn_s[w];
                        sm.part_s[2 * nv] = C(t, 0.0);
                    }
                }
            }
            __syncthreads();
            next_epoch(er);
            if (tid == 0) tc_mark = gtimer();
            round_gather(p, sm, K, er, ctl);
            ABORT_CHECK();
            // ---- reducer: norm, scaling, forward substitution, Givens of the previous column, decision ----------
            int nb = norm_only ? 2 + m : 2 + nv;
            if (cta == 0) {
                __shared__ double s_scal;   // s = 1 / ||u_j||
                __shared__ double s_rel;    // relative residual of the column just completed
                __shared__ int s_code;      // 0 continue, 1 stop, 2 restart
                __shared__ int s_k;         // columns in the solution update
                // thread 32 (warp 1): norm, Givens update of the previous column, decision, back substitution;
                // warp 0, at the same time: forward substitution (I + L) h = a for the new column (discarded on a stop)
                if (tid == 32) {
                    const double sigma = norm_only ? sm.tot_s[0].re : sm.tot_s[nv + j].re;
                    const double nrm = __dsqrt_rn(sigma);
                    int code = 0, k = 0;
                    double rel = 0.0;
                    if (j == 0) {
                        if (need_bnorm) b_norm = __dsqrt_rn(sm.tot_s[2 * nv].re);
                        if (need_bnorm && b_norm < 1e-15) { code = 1; k = 0; rel = 0.0; final_code = 1; }
                        else {
                            rel = __ddiv_rn(nrm, b_norm);  // beta / ||b||   (gmres.rs:146-156)
                            if (rel < p.tol) { code = 1; k = 0; final_code = 1; }
                            else {
                                for (int i = 0; i <= m; ++i) sm.g[i] = C(0, 0);
                                sm.g[0] = C(nrm, 0.0);
                            }
                        }
                    } else {
                        // column j-1 is complete: h_{j,j-1} = ||u_j||
                        total_iterations += 1;
                        const double gres = givens_column(sm, j - 1, nrm);
                        rel = __ddiv_rn(gres, b_norm);
                        const bool breakdown = nrm < 1e-14;
                        if (rel < p.tol || breakdown) { code = 1; k = j; final_code = 1; }
                        else if (norm_only) { code = 2; k = m; }
                    }
                    if (code != 0 && k > 0) back_substitute(sm, k);
                    if (code == 2) restarts += 1;
                    s_scal = __ddiv_rn(1.0, nrm);
                    s_rel = rel;
                    s_code = code;
                    s_k = k;
                    if (code == 1) final_res = rel;
                }
                if (wq == 0 && !norm_only) {
                    const double s = __ddiv_rn(1.0, __dsqrt_rn(sm.tot_s[nv + j].re));
                    // new Gram row L(j, l) = s g'_l
                    for (int l = lane; l < j; l += 32) sm.Lp[lp_off(l, m1) + j] = C(sm.tot_s[nv + l].re * s, sm.tot_s[nv + l].im * s);
                    __syncwarp();
                    auto scaled_a = [&](int k) -> cplx {
                        if (k >= nv) return C(0, 0);
                        const double f = k == j ? s * s : s;
                        return C(sm.tot_s[k].re * f, sm.tot_s[k].im * f);
                    };
                    cplx a0 = scaled_a(lane), a1 = scaled_a(lane + 32);
                    for (int l = 0; l < nv; ++l) {
                        const cplx src = l < 32 ? a0 : a1;
                        cplx hl;
                        hl.re = __shfl_sync(0xffffffffu, src.re, l & 31);
                        hl.im = __shfl_sync(0xffffffffu, src.im, l & 31);
                        if (lane > l && lane < nv) {
                            const cplx lk = sm.Lp[lp_off(l, m1) + lane];
                            a0.re -= lk.re * hl.re - lk.im * hl.im;
                            a0.im -= lk.re * hl.im + lk.im * hl.re;
                        }
                        if (lane + 32 > l && lane + 32 < nv) {
                            const cplx lk = sm.Lp[lp_off(l, m1) + lane + 32];
                            a1.re -= lk.re * hl.re - lk.im * hl.im;
                            a1.im -= lk.re * hl.im + lk.im * hl.re;
                        }
                    }
                    // (hprev is read by the Givens thread of THIS round: the new column is parked in red4 and moved below)
                    if (lane < nv) sm.red4[lane] = a0;
                    if (lane + 32 < nv) sm.red4[lane + 32] = a1;
                }
                __syncthreads();
                const int code = s_code;
                if (code == 0) {
                    for (int i = tid; i < nv; i += FT) { sm.hprev[i] = sm.red4[i]; sm.bc_s[2 + i] = sm.red4[i]; }
                } else {
                    for (int i = tid; i < nb - 2; i += FT) sm.bc_s[2 + i] = i < s_k ? sm.ycoef[i] : C(0, 0);
                }
                if (tid == 0) {
                    sm.bc_s[0] = C((double)code, (double)s_k);
                    sm.bc_s[1] = C(s_scal, s_rel);
                }
            }
            round_broadcast(p, sm, nb, er, ctl);
            ABORT_CHECK();
            if (tid == 0) tc_wait += gtimer() - tc_mark;
            if (cta == 0 && tid == 0) t_round += gtimer() - tr0;
            const int code = (int)sm.bc_s[0].re;
            if (code == 0) {
                // ---- v_j = s u_j -> V[j];  u_{j+1} = s w' - sum_{l<=j} h_l v_l  on own rows -------------------------
                const double s = sm.bc_s[1].re;
                const double scm1 = s - 1.0;
                cplx* red2 = reinterpret_cast<cplx*>(sm.ypart);
                for (uint32_t base = 0; base < sc; base += FT) {
                    const uint32_t cnt = sc - base < (uint32_t)FT ? sc - base : (uint32_t)FT;
                    const uint32_t rpad = (cnt + 31u) & ~31u;          // rows of this pass, padded to whole warps
                    const uint32_t ngrp = FT / rpad;                    // vector strands working on the same rows
                    const uint32_t grp = tid / rpad, i = tid - grp * rpad;
                    cplx acc = C(0, 0);
                    if (grp < ngrp && i < cnt) {
                        const cplx* vcol = p.V + rb + base + i;
                        for (int l0 = (int)grp; l0 < j; l0 += 8 * (int)ngrp) {  // 8 independent loads in flight
                            cplx v[8];
#pragma unroll
                            for (int e = 0; e < 8; ++e) {
                                const int l = l0 + e * (int)ngrp;
                                v[e] = l < j ? ldcg_c(vcol + (size_t)l * p.ldv) : C(0, 0);
                            }
#pragma unroll
                            for (int e = 0; e < 8; ++e) {
                                const int l = l0 + e * (int)ngrp;
                                if (l < j) {
                                    const cplx h = sm.bc_s[2 + l];
                                    acc.re = fma(h.re, v[e].re, fma(-h.im, v[e].im, acc.re));
                                    acc.im = fma(h.re, v[e].im, fma(h.im, v[e].re, acc.im));
                                }
                            }
                        }
                    }
                    if (ngrp > 1) {
                        if (grp < ngrp && i < cnt) red2[grp * rpad + i] = acc;
                        __syncthreads();
                    }
                    if (grp == 0 && i < cnt) {
                        for (uint32_t q = 1; q < ngrp; ++q) { acc.re += red2[q * rpad + i].re; acc.im += red2[q * rpad + i].im; }
                        const cplx u = sm.u_s[base + i], w = sm.w_s[base + i];
                        // v_0 = r * (1/beta) (gmres.rs:163); v_{j+1} = w + (1/||w|| - 1) w (gmres.rs:198-201); the preconditioned
                        // variant scales directly (gmres.rs:362)
                        const cplx vj = (j == 0 || p.direct_scale) ? C(u.re * s, u.im * s) : C(u.re + u.re * scm1, u.im + u.im * scm1);
                        p.V[(size_t)j * p.ldv + rb + base + i] = vj;
                        const cplx hj = sm.bc_s[2 + j];
                        cplx un = C(w.re * s - acc.re, w.im * s - acc.im);
                        un.re = fma(-hj.re, vj.re, fma(hj.im, vj.im, un.re));
                        un.im = fma(-hj.re, vj.im, fma(-hj.im, vj.re, un.im));
                        sm.u_s[base + i] = un;
                    }
                    __syncthreads();
                }
                continue;
            }
            // ---- stop or restart: x += sum_{l<k} y_l v_l in the reference's order (gmres.rs:241-243) ------------------
            const int k = (int)sm.bc_s[0].im;
            for (uint32_t i = tid; i < sc; i += FT) {
                cplx xv = p.x[(size_t)p.row0 + rb + i];
                const cplx* vcol = p.V + rb + i;
                for (int l0 = 0; l0 < k; l0 += 8) {
                    cplx v[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) v[e] = l0 + e < k ? ldcg_c(vcol + (size_t)(l0 + e) * p.ldv) : C(0, 0);
#pragma unroll
                    for (int e = 0; e < 8; ++e)
                        if (l0 + e < k) {
                            const cplx y = sm.bc_s[2 + l0 + e];
                            xv.re += y.re * v[e].re - y.im * v[e].im;
                            xv.im += y.re * v[e].im + y.im * v[e].re;
                        }
                }
                p.x[(size_t)p.row0 + rb + i] = xv;
            }
            __syncthreads();
            stop_all = code == 1;
            break;
        }
        if (stop_all) break;
    }
#undef ABORT_CHECK

    // ---- every rank ends with the full solution: own rows -> all exchange buffers -> plain x --------------------
    next_epoch(ex);
    publish_rows(p, p.x + p.row0 + rb, rb, sc, ex);
    {
        const uint4* xin = p.xbuf[p.rank] + (size_t)(ex & 1u) * 2 * p.npad;
        const uint32_t per = (p.n + G - 1) / G;
        const uint32_t e0 = cta * per < p.n ? cta * per : p.n, e1 = e0 + per < p.n ? e0 + per : p.n;
        for (uint32_t e = e0 + tid; e < e1; e += FT) {
            if (e >= p.row0 && e < p.row0 + p.nloc) continue;  // own slice is already in place
            p.x[e] = ll_wait1(xin + 2 * (size_t)e, ex, ctl);
        }
    }
    __syncthreads();
    if (abort_s) return;
    if (p.trace && tid == 0) {
        p.trace[4 * cta + 0] = tc_mv;
        p.trace[4 * cta + 1] = tc_wait;
        p.trace[4 * cta + 2] = p.unit_off ? (unsigned long long)(p.unit_off[cta + 1] - p.unit_off[cta]) : (unsigned long long)sc * 16ull;  // work share
        p.trace[4 * cta + 3] = smid;
    }
    __shared__ int fin_flag;
    if (cta == 0 && tid == 32) {
        FusedResult* r = p.result;
        r->iterations = total_iterations;
        r->restarts = restarts;
        r->residual = final_res;
        r->converged = final_code;
        __threadfence_system();
    }
    if (tid == 0) fin_flag = 1;
    __syncthreads();
    if (cta == 0 && tid == 0 && fin_flag) {
        FusedResult* r = p.result;
        r->matvecs = matvecs;
        r->ex_final = ex;
        r->er_final = er;
        r->t_total_ns = gtimer() - t_begin;
        r->t_matvec_ns = t_mv;
        r->t_round_ns = t_round;
        __threadfence_system();
        r->done = 1;
    }
}

__global__ void __launch_bounds__(FUSED_THREADS, 1) gmres_fused_kernel(const __grid_constant__ FusedParams p) { gmres_body<4, 4>(p); }
// "polite" build: at most 96 registers per thread, so that a background assembly block (128 threads x 128 registers) fits
// beside a solver CTA on every SM (frequency sweeps: assembly of f + 1 underneath the solve of f)
__global__ void __maxnreg__(96) gmres_fused_kernel_polite(const __grid_constant__ FusedParams p) { gmres_body<2, 4>(p); }

}  // namespace

size_t fused_smem_bytes(uint32_t S, uint32_t rblk, uint32_t restart) {
    const size_t m = restart, m1 = m + 1;
    auto al = [](size_t b) { return (b + 15) & ~(size_t)15; };
    size_t yb = (size_t)rblk * NW * 2 * sizeof(double);
    if (yb < FT * sizeof(cplx)) yb = FT * sizeof(cplx);
    size_t t = al(yb) + 2 * al((size_t)S * sizeof(cplx)) + 2 * al(KMAX * sizeof(cplx)) + al((FT + 32) * sizeof(cplx)) + al(KMAX * sizeof(cplx));
    t += 2 * al((m1 * m / 2 + 1) * sizeof(cplx)) + 2 * al(m1 * sizeof(cplx)) + 2 * al((m1 + 1) * sizeof(cplx)) + al(m1 * sizeof(cplx));
    return t;
}

// rows per pass of the matvec inside a CTA: as many as fit 64 KB of partial sums
uint32_t fused_pick_rblk(uint32_t S) {
    const uint32_t cap = 256;
    const uint32_t r = S < cap ? S : cap;
    return r ? r : 1;
}

cudaError_t launch_gmres_fused(const FusedParams& p, int grid, size_t smem, bool polite, cudaStream_t s) {
    static std::atomic<unsigned long long> attr_done[64];
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 63;
    if (attr_done[dev].load() < smem) {
        cudaError_t e = cudaFuncSetAttribute(gmres_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(gmres_fused_kernel_polite, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        attr_done[dev].store(smem);
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid, 1, 1);
    cfg.blockDim = dim3(FUSED_THREADS, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;  // co-residency of all CTAs is required (they wait for each other)
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (polite) return cudaLaunchKernelEx(&cfg, gmres_fused_kernel_polite, p);
    return cudaLaunchKernelEx(&cfg, gmres_fused_kernel, p);
}

}  // namespace bemb
