// linalg.cu -- device kernels of the solve phase.
//
//   zgemv_kernel        K5: y = A x, streaming complex128 GEMV (HBM-bound), replaces
//                       DenseOperator::apply = Array2::dot -> cblas zgemv
//                       (math-bem/src/core/solver/fmm_interface.rs:45-47)
//   zgemv_t_kernel      apply_transpose (fmm_interface.rs:49-51)
//   mgs_cluster_kernel  K7: one Arnoldi step of gmres.rs:184-202 -- modified Gram-Schmidt
//                       of w against v_0..v_j, ||w||, v_{j+1} -- in ONE launch: a thread-block
//                       cluster keeps w in (distributed) shared memory, and the j+1 DEPENDENT
//                       dot products are reduced across the CTAs through DSMEM + cluster
//                       barriers instead of j+1 kernel launches / host round trips.
//   residual / scale / update kernels for gmres.rs:143-172,238-262
#include <cooperative_groups.h>
#include <atomic>

#include "linalg.h"

namespace cg = cooperative_groups;

namespace bemb {

// Function attributes (dynamic shared memory, non-portable cluster size) and "this kernel cannot be
// placed here" demotions are PER DEVICE: a process may hold contexts on several GPUs.
constexpr int MAX_DEVICES = 64;
static inline int cur_dev() {
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess) { cudaGetLastError(); d = 0; }
    return d >= 0 && d < MAX_DEVICES ? d : MAX_DEVICES - 1;
}
struct PerDeviceFlag {
    std::atomic<unsigned char> v[MAX_DEVICES];
    PerDeviceFlag() { for (auto& x : v) x.store(0); }
    bool get() const { return v[cur_dev()].load() != 0; }
    void set() { v[cur_dev()].store(1); }
};
struct PerDeviceInt {  // starts at `init` on every device
    std::atomic<int> v[MAX_DEVICES];
    explicit PerDeviceInt(int init) { for (auto& x : v) x.store(init); }
    int get() const { return v[cur_dev()].load(); }
    void set(int val) { v[cur_dev()].store(val); }
};

namespace {

// ------------------------------------------------------------------------------------------
// ZGEMV: block = 256 threads = 8 warps walks RB rows at once; lane-contiguous 128-bit loads
// (each warp load instruction covers 512 contiguous bytes of one row), x re-used across the
// RB rows from registers, 2x unrolled => RB*2 independent 16-byte loads in flight per thread.
// ------------------------------------------------------------------------------------------
constexpr int GEMV_THREADS = 256;

__device__ __forceinline__ double2 ld_stream(const cplx* p) { return __ldcs(reinterpret_cast<const double2*>(p)); }
__device__ __forceinline__ double2 ld_ro(const cplx* p) { return __ldg(reinterpret_cast<const double2*>(p)); }

__device__ __forceinline__ void cfma(double& are, double& aim, double2 a, double2 x) {
    are = fma(a.x, x.x, are);
    are = fma(-a.y, x.y, are);
    aim = fma(a.x, x.y, aim);
    aim = fma(a.y, x.x, aim);
}

// ---- peer-memory helpers (row-sharded solve) -------------------------------------------------
// The ZGEMV epilogue stores its slab of y straight into every rank's work vector over NVLink in
// "flag-in-data" form: each complex number travels as two 16-byte stores {lo32, epoch, hi32, epoch}
// whose 8-byte halves are written atomically, so the data is its own arrival flag -- no system
// fence, no counter, no separate signal.  The consumer spins per element until all four epochs
// match (bounded by PEER_WAIT_TIMEOUT_NS, failure reported through a mapped host int).
__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void ll_store(uint4* dst, double re, double im, uint32_t flag) {
    const uint32_t rl = (uint32_t)__double2loint(re), rh = (uint32_t)__double2hiint(re);
    const uint32_t il = (uint32_t)__double2loint(im), ih = (uint32_t)__double2hiint(im);
    asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "r"(rl), "r"(flag), "r"(rh), "r"(flag) : "memory");
    asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(dst + 1), "r"(il), "r"(flag), "r"(ih), "r"(flag) : "memory");
}
// loads N elements (element e at src + 2*(first + e*stride), skipped when first + e*stride >= len);
// every pass issues all outstanding loads back to back, then re-polls only what has not arrived
template <int N>
__device__ __forceinline__ void ll_load_many(cplx (&out)[N], const uint4* src, uint64_t first, uint64_t stride, uint64_t len,
                                             uint32_t flag, int* err, unsigned long long timeout_ns) {
    bool have[N];
#pragma unroll
    for (int e = 0; e < N; ++e) {
        have[e] = first + (uint64_t)e * stride >= len;
        out[e] = C(0, 0);
    }
    unsigned long long t0 = 0;
    unsigned int spins = 0;
    for (;;) {
        uint4 a[N], b[N];
#pragma unroll
        for (int e = 0; e < N; ++e) {
            if (!have[e]) {
                const uint4* q = src + 2 * (first + (uint64_t)e * stride);
                asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(a[e].x), "=r"(a[e].y), "=r"(a[e].z), "=r"(a[e].w) : "l"(q) : "memory");
                asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(b[e].x), "=r"(b[e].y), "=r"(b[e].z), "=r"(b[e].w) : "l"(q + 1) : "memory");
            }
        }
        bool all = true;
#pragma unroll
        for (int e = 0; e < N; ++e) {
            if (!have[e]) {
                if (a[e].y == flag && a[e].w == flag && b[e].y == flag && b[e].w == flag) {
                    have[e] = true;
                    out[e] = C(__hiloint2double((int)a[e].z, (int)a[e].x), __hiloint2double((int)b[e].z, (int)b[e].x));
                } else {
                    all = false;
                }
            }
        }
        if (all) break;
        if ((++spins & 63u) == 0) {
            const unsigned long long t = global_timer_ns();
            if (t0 == 0) t0 = t;
            else if (t - t0 > timeout_ns) {
                *reinterpret_cast<volatile int*>(err) = 1;
                break;
            }
        }
    }
}

template <int GEMV_RB, int GEMV_U, bool FUSED>
__global__ void __launch_bounds__(GEMV_THREADS)
zgemv_kernel(const cplx* __restrict__ A, uint64_t lda, uint64_t nrows, uint64_t ncols, const cplx* __restrict__ x,
             cplx* __restrict__ y, PeerOut po) {
    __shared__ double red[GEMV_RB][2][GEMV_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (uint64_t rb = (uint64_t)blockIdx.x * GEMV_RB; rb < nrows; rb += (uint64_t)gridDim.x * GEMV_RB) {
        double are[GEMV_RB], aim[GEMV_RB];
        const cplx* rowp[GEMV_RB];
#pragma unroll
        for (int r = 0; r < GEMV_RB; ++r) {
            are[r] = 0.0; aim[r] = 0.0;
            uint64_t row = rb + r < nrows ? rb + r : nrows - 1;  // clamp: tail rows recompute the last row
            rowp[r] = A + row * lda;
        }
        uint64_t c = tid;
        for (; c + (GEMV_U - 1) * GEMV_THREADS < ncols; c += GEMV_U * GEMV_THREADS) {
            double2 a[GEMV_RB][GEMV_U], xv[GEMV_U];
#pragma unroll
            for (int u = 0; u < GEMV_U; ++u) {
#pragma unroll
                for (int r = 0; r < GEMV_RB; ++r) a[r][u] = ld_stream(rowp[r] + c + u * GEMV_THREADS);
                xv[u] = ld_ro(x + c + u * GEMV_THREADS);
            }
#pragma unroll
            for (int u = 0; u < GEMV_U; ++u)
#pragma unroll
                for (int r = 0; r < GEMV_RB; ++r) cfma(are[r], aim[r], a[r][u], xv[u]);
        }
        for (; c < ncols; c += GEMV_THREADS) {
            const double2 x0 = ld_ro(x + c);
#pragma unroll
            for (int r = 0; r < GEMV_RB; ++r) cfma(are[r], aim[r], ld_stream(rowp[r] + c), x0);
        }
#pragma unroll
        for (int r = 0; r < GEMV_RB; ++r) {
#pragma unroll
            for (int m = 16; m >= 1; m >>= 1) {
                are[r] += __shfl_xor_sync(0xffffffffu, are[r], m);
                aim[r] += __shfl_xor_sync(0xffffffffu, aim[r], m);
            }
            if (lane == 0) { red[r][0][warp] = are[r]; red[r][1][warp] = aim[r]; }
        }
        __syncthreads();
        if (tid < GEMV_RB && rb + tid < nrows) {
            double sr = 0.0, si = 0.0;
#pragma unroll
            for (int w = 0; w < GEMV_THREADS / 32; ++w) { sr += red[tid][0][w]; si += red[tid][1][w]; }
            if (FUSED) {
#pragma unroll
                for (int p = 0; p < MAX_PEERS; ++p)  // constant indices: the pointer table stays in the parameter bank
                    if (p < po.npeers) ll_store(po.ll[p] + 2 * (rb + tid), sr, si, po.epoch);  // NVLink (own rank: local)
            } else {
                y[rb + tid] = C(sr, si);
            }
        }
        __syncthreads();
    }
}

// apply_transpose, deterministic two-pass column reduction: pass 1 writes the partial sum of every row
// chunk to part[chunk][col] (each thread owns its column: coalesced reads of A, no atomics), pass 2 adds the
// chunks of a column in chunk order.  At most GEMVT_MAX_CHUNKS chunks, so the scratch stays 32 n complex numbers.
constexpr int GEMVT_MAX_CHUNKS = 32;
__global__ void __launch_bounds__(256)
zgemv_t_partial_kernel(const cplx* __restrict__ A, uint64_t lda, uint64_t nrows, uint64_t ncols, uint64_t rows_per_chunk,
                       const cplx* __restrict__ x, cplx* __restrict__ part) {
    const uint64_t col = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    const uint64_t r0 = (uint64_t)blockIdx.y * rows_per_chunk;
    const uint64_t r1 = r0 + rows_per_chunk < nrows ? r0 + rows_per_chunk : nrows;
    if (col >= ncols) return;
    double sr = 0.0, si = 0.0;
    for (uint64_t r = r0; r < r1; ++r) cfma(sr, si, ld_stream(A + r * lda + col), ld_ro(x + r));
    part[(uint64_t)blockIdx.y * ncols + col] = C(sr, si);
}
__global__ void __launch_bounds__(256)
zgemv_t_reduce_kernel(const cplx* __restrict__ part, uint64_t ncols, int nchunks, cplx* __restrict__ y) {
    const uint64_t col = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (col >= ncols) return;
    double sr = 0.0, si = 0.0;
    for (int c = 0; c < nchunks; ++c) { sr += part[(uint64_t)c * ncols + col].re; si += part[(uint64_t)c * ncols + col].im; }
    y[col] = C(sr, si);
}

// ------------------------------------------------------------------------------------------
// cluster helpers
// ------------------------------------------------------------------------------------------
constexpr int MAX_CLUSTER = 16;
constexpr int MAX_WARPS = 32;

struct ClusterShared {
    cplx part[2][MAX_CLUSTER * MAX_WARPS];  // [parity][cta * nwarps + warp]
};

// Sum of one complex value over every thread of every CTA of the cluster with ONE cluster
// barrier and no block barrier: warp shuffle -> each warp posts its partial into the slot table
// of every CTA through DSMEM -> barrier.cluster -> every warp adds the nb*nw slots in the same
// fixed order (bit-identical result in all warps of all CTAs).  `parity` must alternate between
// consecutive calls (double-buffered slot table).
__device__ __forceinline__ cplx cluster_allreduce(cplx v, ClusterShared& sh, int parity) {
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned nb = cluster.num_blocks(), me = cluster.block_rank();
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) {
        v.re += __shfl_xor_sync(0xffffffffu, v.re, m);
        v.im += __shfl_xor_sync(0xffffffffu, v.im, m);
    }
    if (lane < nb) {
        ClusterShared* remote = cluster.map_shared_rank(&sh, lane);
        remote->part[parity][me * nw + warp] = v;
    }
    cluster.sync();
    cplx t = C(0, 0);
    const unsigned total = nb * nw;
    for (unsigned sidx = lane; sidx < total; sidx += 32) {
        t.re += sh.part[parity][sidx].re;
        t.im += sh.part[parity][sidx].im;
    }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) {
        t.re += __shfl_xor_sync(0xffffffffu, t.re, m);
        t.im += __shfl_xor_sync(0xffffffffu, t.im, m);
    }
    return t;
}

__device__ __forceinline__ cplx ldg_c(const cplx* p) {
    double2 v = __ldg(reinterpret_cast<const double2*>(p));
    return C(v.x, v.y);
}

// One Arnoldi orthogonalisation step (gmres.rs:184-202), register-resident variant: CTA c owns
// the slice [c*S, (c+1)*S) and thread t its elements t, t+T, ... (EPT per thread) of w in
// registers; v_{i+1} is prefetched while step i's dot product crosses the cluster.
template <int EPT>
__global__ void __launch_bounds__(256)
mgs_cluster_reg_kernel(const cplx* __restrict__ V, uint64_t ldv, const cplx* __restrict__ w, int j, uint64_t n, uint64_t S,
                       cplx* __restrict__ hcol, cplx* __restrict__ vnext, double breakdown_tol,
                       const cplx* __restrict__ pinv, int direct_scale) {
    __shared__ ClusterShared sh;
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned me = cluster.block_rank();
    const uint64_t begin = (uint64_t)me * S;
    const uint64_t end = begin + S < n ? begin + S : n;
    const uint64_t len = end > begin ? end - begin : 0;
    cplx wr[EPT], vc[EPT], vn[EPT];
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
        const uint64_t k = threadIdx.x + (uint64_t)e * blockDim.x;
        wr[e] = k < len ? w[begin + k] : C(0, 0);
        if (pinv && k < len) wr[e] = wr[e] * ldg_c(pinv + begin + k);  // w = M^-1 (A v_j)  (gmres.rs:345-347)
        vc[e] = k < len ? ldg_c(V + begin + k) : C(0, 0);
    }
    int parity = 0;
    for (int i = 0; i <= j; ++i) {
        if (i < j) {
            const cplx* vi1 = V + (uint64_t)(i + 1) * ldv + begin;
#pragma unroll
            for (int e = 0; e < EPT; ++e) {
                const uint64_t k = threadIdx.x + (uint64_t)e * blockDim.x;
                vn[e] = k < len ? ldg_c(vi1 + k) : C(0, 0);
            }
        }
        cplx acc = C(0, 0);
#pragma unroll
        for (int e = 0; e < EPT; ++e) {  // conj(v) * w  (inner_product: blas_helpers.rs:21-33)
            acc.re = fma(vc[e].re, wr[e].re, fma(vc[e].im, wr[e].im, acc.re));
            acc.im = fma(vc[e].re, wr[e].im, fma(-vc[e].im, wr[e].re, acc.im));
        }
        const cplx h = cluster_allreduce(acc, sh, parity);
        parity ^= 1;
        if (me == 0 && threadIdx.x == 0) hcol[i] = h;
#pragma unroll
        for (int e = 0; e < EPT; ++e) {  // axpy(-h, v_i, w)
            wr[e].re = fma(-h.re, vc[e].re, fma(h.im, vc[e].im, wr[e].re));
            wr[e].im = fma(-h.re, vc[e].im, fma(-h.im, vc[e].re, wr[e].im));
            vc[e] = vn[e];
        }
    }
    cplx acc = C(0, 0);
#pragma unroll
    for (int e = 0; e < EPT; ++e) acc.re = fma(wr[e].re, wr[e].re, fma(wr[e].im, wr[e].im, acc.re));
    const cplx nn = cluster_allreduce(acc, sh, parity);
    const double nrm = sqrt(nn.re);
    if (me == 0 && threadIdx.x == 0) hcol[j + 1] = C(nrm, 0.0);
    if (!(nrm < breakdown_tol)) {
        const double inv = 1.0 / nrm;
        const double sc = inv - 1.0;  // new_v = w; axpy(1/||w|| - 1, w, new_v)   (gmres.rs:198-201)
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const uint64_t k = threadIdx.x + (uint64_t)e * blockDim.x;
            if (k < len)
                vnext[begin + k] = direct_scale ? C(wr[e].re * inv, wr[e].im * inv)  // w.mapv(|wi| wi * (1/||w||)) (gmres.rs:362)
                                                : C(wr[e].re + wr[e].re * sc, wr[e].im + wr[e].im * sc);
        }
    }
    cluster.sync();  // no CTA may exit while a peer could still address its shared memory
}

// ------------------------------------------------------------------------------------------
// Low-synchronisation form of the same modified Gram-Schmidt sweep.  With L the strictly lower
// triangle of the Gram matrix of the stored basis, L_kl = v_k^H v_l (k > l; rounding-level numbers,
// the loss of orthogonality of V), the MGS coefficients h_k = v_k^H (w - sum_{l<k} h_l v_l) satisfy
//       (I + L) h = V^H w ,
// so ALL j+1 inner products can be taken in one pass over V and cross the cluster in ONE barrier;
// a (j+1)x(j+1) forward substitution then yields exactly the h of gmres.rs:184-188 (same algebra,
// different rounding), and a second pass applies w -= V h.  Row j of L (v_j^H v_l, l < j) is
// computed in the same first pass, kept in global memory for the later iterations of the cycle.
// 2 cluster barriers per iteration instead of j+2.
// ------------------------------------------------------------------------------------------
constexpr int LS_THREADS = 256;
constexpr int LS_WARPS = LS_THREADS / 32;
constexpr int LS_MAXV = 64;  // max j+1 handled here (restart <= 63), else the one-vector kernels

template <int EPT>
__global__ void __launch_bounds__(LS_THREADS)
mgs_lowsync_kernel(const cplx* __restrict__ V, uint64_t ldv, const cplx* __restrict__ w, int j, uint64_t n, uint64_t S,
                   cplx* __restrict__ Lmat, int ldl, cplx* __restrict__ hcol, cplx* __restrict__ vnext, double breakdown_tol,
                   const cplx* __restrict__ pinv, int direct_scale, cplx* __restrict__ hcol_host, PeerWait pw) {
    extern __shared__ __align__(16) unsigned char dyn[];
    __shared__ ClusterShared sh1;  // single-value all-reduce (norm)
    // dynamic layout: warp_part[LS_WARPS][2*LS_MAXV] | slots[MAX_CLUSTER][2*LS_MAXV] | a[LS_MAXV] | Ls[(j+1)*(j+1)]
    cplx* warp_part = reinterpret_cast<cplx*>(dyn);
    cplx* slots = warp_part + LS_WARPS * 2 * LS_MAXV;
    cplx* avec = slots + MAX_CLUSTER * 2 * LS_MAXV;
    cplx* Ls = avec + LS_MAXV;
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned nb = cluster.num_blocks(), me = cluster.block_rank();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nv = j + 1;
    const uint64_t begin = (uint64_t)me * S;
    const uint64_t end = begin + S < n ? begin + S : n;
    const uint64_t len = end > begin ? end - begin : 0;

    cplx wr[EPT], vj[EPT];
    // row-sharded solve: w arrives from every rank's ZGEMV epilogue in flag-in-data form
    if (pw.ll) ll_load_many<EPT>(wr, pw.ll + 2 * begin, (uint64_t)tid, (uint64_t)LS_THREADS, len, pw.epoch, pw.err, pw.timeout_ns);
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
        const uint64_t k = tid + (uint64_t)e * LS_THREADS;
        if (!pw.ll) wr[e] = k < len ? w[begin + k] : C(0, 0);
        if (pinv && k < len) wr[e] = wr[e] * ldg_c(pinv + begin + k);
        vj[e] = (k < len) ? ldg_c(V + (uint64_t)j * ldv + begin + k) : C(0, 0);
    }
    // previous rows of L (rows 1..j-1) -> shared memory
    for (int idx = tid; idx < nv * nv; idx += LS_THREADS) {
        const int k = idx / nv, l = idx - k * nv;
        Ls[idx] = (l < k && k < j) ? Lmat[k * ldl + l] : C(0, 0);
    }

    // ---- pass 1: a_l = v_l^H w (l <= j) and g_l = v_j^H v_l (l < j), 8 vectors at a time -------
    for (int l0 = 0; l0 < nv; l0 += 8) {
        cplx aa[8], gg[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) { aa[q] = C(0, 0); gg[q] = C(0, 0); }
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const uint64_t k = tid + (uint64_t)e * LS_THREADS;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int l = l0 + q;
                const cplx v = (l < nv && k < len) ? ldg_c(V + (uint64_t)l * ldv + begin + k) : C(0, 0);
                aa[q].re = fma(v.re, wr[e].re, fma(v.im, wr[e].im, aa[q].re));    // conj(v_l) * w
                aa[q].im = fma(v.re, wr[e].im, fma(-v.im, wr[e].re, aa[q].im));
                gg[q].re = fma(vj[e].re, v.re, fma(vj[e].im, v.im, gg[q].re));    // conj(v_j) * v_l
                gg[q].im = fma(vj[e].re, v.im, fma(-vj[e].im, v.re, gg[q].im));
            }
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) {
#pragma unroll
            for (int m = 16; m >= 1; m >>= 1) {
                aa[q].re += __shfl_xor_sync(0xffffffffu, aa[q].re, m);
                aa[q].im += __shfl_xor_sync(0xffffffffu, aa[q].im, m);
                gg[q].re += __shfl_xor_sync(0xffffffffu, gg[q].re, m);
                gg[q].im += __shfl_xor_sync(0xffffffffu, gg[q].im, m);
            }
            if (lane == 0 && l0 + q < nv) {
                warp_part[warp * 2 * LS_MAXV + l0 + q] = aa[q];
                warp_part[warp * 2 * LS_MAXV + LS_MAXV + l0 + q] = gg[q];
            }
        }
    }
    __syncthreads();
    // block partials -> slot `me` of every CTA of the cluster (DSMEM)
    if (tid < 2 * nv) {
        const int idx = tid < nv ? tid : LS_MAXV + (tid - nv);
        cplx t = C(0, 0);
#pragma unroll
        for (int wq = 0; wq < LS_WARPS; ++wq) { t.re += warp_part[wq * 2 * LS_MAXV + idx].re; t.im += warp_part[wq * 2 * LS_MAXV + idx].im; }
        for (unsigned d = 0; d < nb; ++d) {
            cplx* remote = cluster.map_shared_rank(slots, d);
            remote[me * 2 * LS_MAXV + idx] = t;
        }
    }
    cluster.sync();
    // every CTA: totals in fixed CTA order, forward substitution (I + L) h = a
    if (tid < 2 * nv) {
        const int idx = tid < nv ? tid : LS_MAXV + (tid - nv);
        cplx t = C(0, 0);
        for (unsigned d = 0; d < nb; ++d) { t.re += slots[d * 2 * LS_MAXV + idx].re; t.im += slots[d * 2 * LS_MAXV + idx].im; }
        if (tid < nv) {
            avec[tid] = t;
        } else {
            const int l = tid - nv;
            if (l < j) {
                Ls[j * nv + l] = t;                                   // new row j of L
                if (me == 0) Lmat[j * ldl + l] = t;
            }
        }
    }
    __syncthreads();
    if (warp == 0) {
        for (int l = 0; l < nv; ++l) {
            const cplx hl = avec[l];
            for (int k = l + 1 + lane; k < nv; k += 32) {
                const cplx lk = Ls[k * nv + l];
                cplx ak = avec[k];
                ak.re -= lk.re * hl.re - lk.im * hl.im;
                ak.im -= lk.re * hl.im + lk.im * hl.re;
                avec[k] = ak;
            }
            __syncwarp();
        }
        if (me == 0)
            for (int l = lane; l < nv; l += 32) {
                hcol[l] = avec[l];
                if (hcol_host) hcol_host[l] = avec[l];  // mapped pinned memory: the column lands on the host with the kernel
            }
    }
    __syncthreads();
    // ---- pass 2: w -= sum_l h_l v_l ----------------------------------------------------------------
    for (int l0 = 0; l0 < nv; l0 += 8) {
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const uint64_t k = tid + (uint64_t)e * LS_THREADS;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int l = l0 + q;
                if (l < nv && k < len) {
                    const cplx v = ldg_c(V + (uint64_t)l * ldv + begin + k);
                    const cplx h = avec[l];
                    wr[e].re = fma(-h.re, v.re, fma(h.im, v.im, wr[e].re));
                    wr[e].im = fma(-h.re, v.im, fma(-h.im, v.re, wr[e].im));
                }
            }
        }
    }
    cplx acc = C(0, 0);
#pragma unroll
    for (int e = 0; e < EPT; ++e) acc.re = fma(wr[e].re, wr[e].re, fma(wr[e].im, wr[e].im, acc.re));
    const cplx nn = cluster_allreduce(acc, sh1, 0);
    const double nrm = sqrt(nn.re);
    if (me == 0 && tid == 0) {
        hcol[j + 1] = C(nrm, 0.0);
        if (hcol_host) hcol_host[j + 1] = C(nrm, 0.0);
    }
    if (!(nrm < breakdown_tol)) {
        const double inv = 1.0 / nrm;
        const double sc = inv - 1.0;
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const uint64_t k = tid + (uint64_t)e * LS_THREADS;
            if (k < len)
                vnext[begin + k] = direct_scale ? C(wr[e].re * inv, wr[e].im * inv)
                                                : C(wr[e].re + wr[e].re * sc, wr[e].im + wr[e].im * sc);
        }
    }
    cluster.sync();
}

// ------------------------------------------------------------------------------------------
// Whole-GPU form of the low-synchronisation sweep: one CTA per SM (cooperative launch, two
// grid barriers) instead of one 16-CTA cluster, so the two passes over V run at the bandwidth
// of 148 SMs instead of 16.  Same algebra as mgs_lowsync_kernel; partial sums cross the grid
// through a small global scratch and are added in fixed CTA order by every CTA (bit-identical
// on every rank: the grid size depends on n only).
// ------------------------------------------------------------------------------------------
constexpr int GR_MAX_CTAS = 148;

// 32 per-lane partial sums -> lane L ends up with the warp total of value L (31 exchanges
// instead of 32 x 5; fixed order, so deterministic)
__device__ __forceinline__ double warp_reduce32(double (&v)[32], int lane) {
#pragma unroll
    for (int off = 16, cnt = 16; off >= 1; off >>= 1, cnt >>= 1) {
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < cnt; ++i) {
            const double send = upper ? v[i] : v[i + cnt];
            const double keep = upper ? v[i + cnt] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
    }
    return v[0];
}

template <int EPT, int GR_THREADS>
__global__ void __launch_bounds__(GR_THREADS)
mgs_grid_kernel(const cplx* __restrict__ V, uint64_t ldv, const cplx* __restrict__ w, int j, uint64_t n, uint64_t S,
                cplx* __restrict__ Lmat, int ldl, cplx* __restrict__ hcol, cplx* __restrict__ vnext, double breakdown_tol,
                const cplx* __restrict__ pinv, int direct_scale, cplx* __restrict__ part, double* __restrict__ npart,
                cplx* __restrict__ hcol_host, PeerWait pw) {
    constexpr int GR_WARPS = GR_THREADS / 32;
    extern __shared__ __align__(16) unsigned char dyn[];
    // dynamic layout: warp_part[GR_WARPS][2*LS_MAXV] | a[LS_MAXV] | LsT[(j+1)*(j+1)]  (LsT[l*nv + k] = L_kl)
    cplx* warp_part = reinterpret_cast<cplx*>(dyn);
    cplx* avec = warp_part + GR_WARPS * 2 * LS_MAXV;
    cplx* LsT = avec + LS_MAXV;
    __shared__ double nred[GR_WARPS];
    __shared__ double nrm_s;
    cg::grid_group grid = cg::this_grid();
    const unsigned G = gridDim.x, me = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nv = j + 1;
    const uint64_t begin = (uint64_t)me * S;
    const uint64_t end = begin + S < n ? begin + S : n;
    const uint64_t len = end > begin ? end - begin : 0;

    cplx wr[EPT], vj[EPT];
    if (pw.ll) ll_load_many<EPT>(wr, pw.ll + 2 * begin, (uint64_t)tid, (uint64_t)GR_THREADS, len, pw.epoch, pw.err, pw.timeout_ns);
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
        const uint64_t k = tid + (uint64_t)e * GR_THREADS;
        if (!pw.ll) wr[e] = k < len ? w[begin + k] : C(0, 0);
        if (pinv && k < len) wr[e] = wr[e] * ldg_c(pinv + begin + k);
        vj[e] = (k < len) ? ldg_c(V + (uint64_t)j * ldv + begin + k) : C(0, 0);
    }
    for (int idx = tid; idx < nv * nv; idx += GR_THREADS) {
        const int l = idx / nv, k = idx - l * nv;
        LsT[idx] = (l < k && k < j) ? Lmat[k * ldl + l] : C(0, 0);
    }

    // ---- pass 1: a_l = v_l^H w (l <= j), g_l = v_j^H v_l (l < j) over this CTA's rows ----------
    for (int l0 = 0; l0 < nv; l0 += 8) {
        double acc[32];  // [q]: a.re | [8+q]: a.im | [16+q]: g.re | [24+q]: g.im
#pragma unroll
        for (int q = 0; q < 32; ++q) acc[q] = 0.0;
        cplx v[EPT][8];
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const uint64_t k = tid + (uint64_t)e * GR_THREADS;
#pragma unroll
            for (int q = 0; q < 8; ++q) v[e][q] = (l0 + q < nv && k < len) ? ldg_c(V + (uint64_t)(l0 + q) * ldv + begin + k) : C(0, 0);
        }
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                acc[q] = fma(v[e][q].re, wr[e].re, fma(v[e][q].im, wr[e].im, acc[q]));
                acc[8 + q] = fma(v[e][q].re, wr[e].im, fma(-v[e][q].im, wr[e].re, acc[8 + q]));
                acc[16 + q] = fma(vj[e].re, v[e][q].re, fma(vj[e].im, v[e][q].im, acc[16 + q]));
                acc[24 + q] = fma(vj[e].re, v[e][q].im, fma(-vj[e].im, v[e][q].re, acc[24 + q]));
            }
        }
        const double tot = warp_reduce32(acc, lane);  // lane = part*8 + q
        const int q = lane & 7, prt = lane >> 3;
        if (l0 + q < nv) {
            double* dst = reinterpret_cast<double*>(warp_part + warp * 2 * LS_MAXV + (prt >> 1) * LS_MAXV + l0 + q);
            dst[prt & 1] = tot;
        }
    }
    __syncthreads();
    // slot idx: [0, nv) -> a_idx ; [LS_MAXV, LS_MAXV + j) -> g_(idx - LS_MAXV)
    const bool live = tid < nv || (tid >= LS_MAXV && tid < LS_MAXV + j);
    if (live) {
        cplx t = C(0, 0);
#pragma unroll
        for (int wq = 0; wq < GR_WARPS; ++wq) { t.re += warp_part[wq * 2 * LS_MAXV + tid].re; t.im += warp_part[wq * 2 * LS_MAXV + tid].im; }
        part[(size_t)me * 2 * LS_MAXV + tid] = t;
    }
    grid.sync();
    // every CTA: totals in fixed CTA order, then the forward substitution (I + L) h = a
    if (live) {
        cplx t = C(0, 0);
        unsigned d = 0;
        for (; d + 37 <= G; d += 37) {
            double2 pv[37];
#pragma unroll
            for (int u = 0; u < 37; ++u) pv[u] = __ldcg(reinterpret_cast<const double2*>(part + (size_t)(d + u) * 2 * LS_MAXV + tid));
#pragma unroll
            for (int u = 0; u < 37; ++u) { t.re += pv[u].x; t.im += pv[u].y; }
        }
        for (; d < G; ++d) {
            const double2 pv = __ldcg(reinterpret_cast<const double2*>(part + (size_t)d * 2 * LS_MAXV + tid));
            t.re += pv.x;
            t.im += pv.y;
        }
        if (tid < nv) {
            avec[tid] = t;
        } else {
            const int l = tid - LS_MAXV;
            LsT[l * nv + j] = t;
            if (me == 0) Lmat[j * ldl + l] = t;
        }
    }
    __syncthreads();
    if (warp == 0) {
        // lane holds a[lane] and a[lane + 32]; column l of L comes from LsT row l (conflict-free)
        cplx a0 = lane < nv ? avec[lane] : C(0, 0);
        cplx a1 = lane + 32 < nv ? avec[lane + 32] : C(0, 0);
        for (int l = 0; l < nv; ++l) {
            const cplx src = l < 32 ? a0 : a1;
            cplx hl;
            hl.re = __shfl_sync(0xffffffffu, src.re, l & 31);
            hl.im = __shfl_sync(0xffffffffu, src.im, l & 31);
            if (lane > l && lane < nv) {
                const cplx lk = LsT[l * nv + lane];
                a0.re -= lk.re * hl.re - lk.im * hl.im;
                a0.im -= lk.re * hl.im + lk.im * hl.re;
            }
            if (lane + 32 > l && lane + 32 < nv) {
                const cplx lk = LsT[l * nv + lane + 32];
                a1.re -= lk.re * hl.re - lk.im * hl.im;
                a1.im -= lk.re * hl.im + lk.im * hl.re;
            }
        }
        if (lane < nv) avec[lane] = a0;
        if (lane + 32 < nv) avec[lane + 32] = a1;
        if (me == 0) {
            if (lane < nv) hcol[lane] = a0;
            if (lane + 32 < nv) hcol[lane + 32] = a1;
            if (hcol_host) {
                if (lane < nv) hcol_host[lane] = a0;
                if (lane + 32 < nv) hcol_host[lane + 32] = a1;
            }
        }
    }
    __syncthreads();
    // ---- pass 2: w -= sum_l h_l v_l ----------------------------------------------------------------
    for (int l0 = 0; l0 < nv; l0 += 8) {
        cplx v[EPT][8];
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const uint64_t k = tid + (uint64_t)e * GR_THREADS;
#pragma unroll
            for (int q = 0; q < 8; ++q) v[e][q] = (l0 + q < nv && k < len) ? ldg_c(V + (uint64_t)(l0 + q) * ldv + begin + k) : C(0, 0);
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            if (l0 + q < nv) {
                const cplx h = avec[l0 + q];
#pragma unroll
                for (int e = 0; e < EPT; ++e) {
                    wr[e].re = fma(-h.re, v[e][q].re, fma(h.im, v[e][q].im, wr[e].re));
                    wr[e].im = fma(-h.re, v[e][q].im, fma(-h.im, v[e][q].re, wr[e].im));
                }
            }
        }
    }
    double acc = 0.0;
#pragma unroll
    for (int e = 0; e < EPT; ++e) acc = fma(wr[e].re, wr[e].re, fma(wr[e].im, wr[e].im, acc));
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, m);
    if (lane == 0) nred[warp] = acc;
    __syncthreads();
    if (tid == 0) {
        double t = 0.0;
#pragma unroll
        for (int wq = 0; wq < GR_WARPS; ++wq) t += nred[wq];
        npart[me] = t;
    }
    grid.sync();
    if (warp == 0) {
        double t = 0.0;
        for (unsigned d = lane; d < G; d += 32) t += __ldcg(npart + d);
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) t += __shfl_xor_sync(0xffffffffu, t, m);
        if (lane == 0) nrm_s = sqrt(t);
    }
    __syncthreads();
    const double nrm = nrm_s;
    if (me == 0 && tid == 0) {
        hcol[j + 1] = C(nrm, 0.0);
        if (hcol_host) hcol_host[j + 1] = C(nrm, 0.0);
    }
    if (!(nrm < breakdown_tol)) {
        const double inv = 1.0 / nrm;
        const double sc = inv - 1.0;
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const uint64_t k = tid + (uint64_t)e * GR_THREADS;
            if (k < len)
                vnext[begin + k] = direct_scale ? C(wr[e].re * inv, wr[e].im * inv)
                                                : C(wr[e].re + wr[e].re * sc, wr[e].im + wr[e].im * sc);
        }
    }
}

// Same step for long vectors: w slice in shared memory (or global/L2 if even that does not
// fit), v_i streamed from L2.
constexpr int VEC_THREADS = 512;
__global__ void __launch_bounds__(VEC_THREADS)
mgs_cluster_kernel(const cplx* __restrict__ V, uint64_t ldv, cplx* __restrict__ w, int j, uint64_t n, uint64_t S,
                   int w_in_smem, cplx* __restrict__ hcol, cplx* __restrict__ vnext, double breakdown_tol,
                   const cplx* __restrict__ pinv, int direct_scale) {
    extern __shared__ __align__(16) unsigned char dyn[];
    __shared__ ClusterShared sh;
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned me = cluster.block_rank();
    const uint64_t begin = (uint64_t)me * S;
    const uint64_t end = begin + S < n ? begin + S : n;
    const uint64_t len = end > begin ? end - begin : 0;
    cplx* ws = w_in_smem ? reinterpret_cast<cplx*>(dyn) : (w + begin);
    if (w_in_smem || pinv)
        for (uint64_t k = threadIdx.x; k < len; k += blockDim.x) {
            cplx v = w[begin + k];
            if (pinv) v = v * ldg_c(pinv + begin + k);
            ws[k] = v;
        }
    // (each thread only ever touches its own k's of ws: no barrier needed for ws itself)
    int parity = 0;
    for (int i = 0; i <= j; ++i) {
        const cplx* vi = V + (uint64_t)i * ldv + begin;
        cplx acc = C(0, 0);
        for (uint64_t k = threadIdx.x; k < len; k += blockDim.x) {
            const cplx a = ldg_c(vi + k), b = ws[k];
            acc.re = fma(a.re, b.re, fma(a.im, b.im, acc.re));
            acc.im = fma(a.re, b.im, fma(-a.im, b.re, acc.im));
        }
        const cplx h = cluster_allreduce(acc, sh, parity);
        parity ^= 1;
        if (me == 0 && threadIdx.x == 0) hcol[i] = h;
        for (uint64_t k = threadIdx.x; k < len; k += blockDim.x) {
            const cplx a = ldg_c(vi + k);
            cplx b = ws[k];
            b.re = fma(-h.re, a.re, fma(h.im, a.im, b.re));
            b.im = fma(-h.re, a.im, fma(-h.im, a.re, b.im));
            ws[k] = b;
        }
    }
    cplx acc = C(0, 0);
    for (uint64_t k = threadIdx.x; k < len; k += blockDim.x) acc.re = fma(ws[k].re, ws[k].re, fma(ws[k].im, ws[k].im, acc.re));
    const cplx nn = cluster_allreduce(acc, sh, parity);
    const double nrm = sqrt(nn.re);
    if (me == 0 && threadIdx.x == 0) hcol[j + 1] = C(nrm, 0.0);
    if (!(nrm < breakdown_tol)) {
        const double inv = 1.0 / nrm;
        const double sc = inv - 1.0;
        for (uint64_t k = threadIdx.x; k < len; k += blockDim.x) {
            const cplx b = ws[k];
            vnext[begin + k] = direct_scale ? C(b.re * inv, b.im * inv) : C(b.re + b.re * sc, b.im + b.im * sc);
        }
    }
    cluster.sync();
}

// r = b - ax ; out[0] = sum |r|^2  (one cluster)
__global__ void __launch_bounds__(VEC_THREADS)
residual_cluster_kernel(const cplx* __restrict__ b, const cplx* __restrict__ ax, cplx* __restrict__ r, uint64_t n, uint64_t S,
                        double* __restrict__ out, const cplx* __restrict__ pinv) {
    __shared__ ClusterShared sh;
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned me = cluster.block_rank();
    const uint64_t begin = (uint64_t)me * S;
    const uint64_t end = begin + S < n ? begin + S : n;
    cplx acc = C(0, 0);
    for (uint64_t k = begin + threadIdx.x; k < end; k += blockDim.x) {
        cplx v = b[k];
        if (ax) { v.re -= ax[k].re; v.im -= ax[k].im; }
        if (pinv) v = v * pinv[k];  // r = M^-1 (b - A x)
        if (r) r[k] = v;
        acc.re = fma(v.re, v.re, fma(v.im, v.im, acc.re));
    }
    const cplx t = cluster_allreduce(acc, sh, 0);
    if (me == 0 && threadIdx.x == 0) out[0] = t.re;
    cluster.sync();
}

// ------------------------------------------------------------------------------------------
// BiCGSTAB vector kernels (math-solvers/src/iterative/bicgstab.rs:88-190): every update of the
// iteration fused with the inner products that follow it, reduced over an 8-CTA cluster in a
// fixed order (bit-deterministic, identical on every rank of a row-sharded solve).
//   out[0..1] = sum conj(a) b   (inner_product, blas_helpers.rs:21-33)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(VEC_THREADS)
bicg_dot_kernel(const cplx* __restrict__ a, const cplx* __restrict__ b, uint64_t n, uint64_t S, cplx* __restrict__ out) {
    __shared__ ClusterShared sh;
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned me = cluster.block_rank();
    const uint64_t begin = (uint64_t)me * S, end = begin + S < n ? begin + S : n;
    cplx acc = C(0, 0);
    for (uint64_t k = begin + threadIdx.x; k < end; k += blockDim.x) {
        const cplx x = a[k], y = b[k];
        acc.re = fma(x.re, y.re, fma(x.im, y.im, acc.re));
        acc.im = fma(x.re, y.im, fma(-x.im, y.re, acc.im));
    }
    const cplx t = cluster_allreduce(acc, sh, 0);
    if (me == 0 && threadIdx.x == 0) out[0] = t;
    cluster.sync();
}

// p = r + beta (p - omega v)       (bicgstab.rs:111)
__global__ void bicg_p_kernel(const cplx* __restrict__ r, cplx* __restrict__ p, const cplx* __restrict__ v, cplx beta, cplx omega, uint64_t n) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const cplx d = p[k] - v[k] * omega;
    p[k] = r[k] + d * beta;
}

// s = r - alpha v ; out[0].re = ||s||^2        (bicgstab.rs:129-132)
__global__ void __launch_bounds__(VEC_THREADS)
bicg_s_kernel(const cplx* __restrict__ r, const cplx* __restrict__ v, cplx alpha, cplx* __restrict__ s, uint64_t n, uint64_t S,
              cplx* __restrict__ out) {
    __shared__ ClusterShared sh;
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned me = cluster.block_rank();
    const uint64_t begin = (uint64_t)me * S, end = begin + S < n ? begin + S : n;
    cplx acc = C(0, 0);
    for (uint64_t k = begin + threadIdx.x; k < end; k += blockDim.x) {
        const cplx x = r[k] - v[k] * alpha;
        s[k] = x;
        acc.re = fma(x.re, x.re, fma(x.im, x.im, acc.re));
    }
    const cplx t = cluster_allreduce(acc, sh, 0);
    if (me == 0 && threadIdx.x == 0) out[0] = t;
    cluster.sync();
}

// out[0] = (t, t), out[1] = (t, s)          (bicgstab.rs:147-160)
__global__ void __launch_bounds__(VEC_THREADS)
bicg_tt_kernel(const cplx* __restrict__ t, const cplx* __restrict__ s, uint64_t n, uint64_t S, cplx* __restrict__ out) {
    __shared__ ClusterShared sh;
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned me = cluster.block_rank();
    const uint64_t begin = (uint64_t)me * S, end = begin + S < n ? begin + S : n;
    cplx a0 = C(0, 0), a1 = C(0, 0);
    for (uint64_t k = begin + threadIdx.x; k < end; k += blockDim.x) {
        const cplx x = t[k], y = s[k];
        a0.re = fma(x.re, x.re, fma(x.im, x.im, a0.re));
        a1.re = fma(x.re, y.re, fma(x.im, y.im, a1.re));
        a1.im = fma(x.re, y.im, fma(-x.im, y.re, a1.im));
    }
    const cplx r0 = cluster_allreduce(a0, sh, 0);
    const cplx r1 = cluster_allreduce(a1, sh, 1);
    if (me == 0 && threadIdx.x == 0) { out[0] = r0; out[1] = r1; }
    cluster.sync();
}

// x += alpha p + omega s ; r = s - omega t ; out[0].re = ||r||^2 ; out[1] = (r0, r)   (bicgstab.rs:163-166, 94)
__global__ void __launch_bounds__(VEC_THREADS)
bicg_update_kernel(cplx* __restrict__ x, const cplx* __restrict__ p, const cplx* __restrict__ s, const cplx* __restrict__ t,
                   cplx* __restrict__ r, const cplx* __restrict__ r0, cplx alpha, cplx omega, uint64_t n, uint64_t S,
                   cplx* __restrict__ out) {
    __shared__ ClusterShared sh;
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned me = cluster.block_rank();
    const uint64_t begin = (uint64_t)me * S, end = begin + S < n ? begin + S : n;
    cplx a0 = C(0, 0), a1 = C(0, 0);
    for (uint64_t k = begin + threadIdx.x; k < end; k += blockDim.x) {
        x[k] = (x[k] + p[k] * alpha) + s[k] * omega;
        const cplx rr = s[k] - t[k] * omega;
        r[k] = rr;
        const cplx q = r0[k];
        a0.re = fma(rr.re, rr.re, fma(rr.im, rr.im, a0.re));
        a1.re = fma(q.re, rr.re, fma(q.im, rr.im, a1.re));
        a1.im = fma(q.re, rr.im, fma(-q.im, rr.re, a1.im));
    }
    const cplx t0 = cluster_allreduce(a0, sh, 0);
    const cplx t1 = cluster_allreduce(a1, sh, 1);
    if (me == 0 && threadIdx.x == 0) { out[0] = t0; out[1] = t1; }
    cluster.sync();
}

// x += alpha p           (early convergence, bicgstab.rs:135)
__global__ void bicg_axpy_kernel(cplx* __restrict__ x, const cplx* __restrict__ p, cplx alpha, uint64_t n) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) x[k] = x[k] + p[k] * alpha;
}

// ------------------------------------------------------------------------------------------
// CGS vector kernels (math-solvers/src/iterative/cgs.rs:71-140): two element-wise updates and one
// update fused with the two reductions that follow it (same fixed-order cluster reduction as above).
// ------------------------------------------------------------------------------------------
// q = u - alpha v ; uq = u + q       (cgs.rs:89-93)
__global__ void cgs_q_kernel(const cplx* __restrict__ u, const cplx* __restrict__ v, cplx alpha, cplx* __restrict__ q,
                             cplx* __restrict__ uq, uint64_t n) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const cplx uu = u[k];
    const cplx qq = uu - v[k] * alpha;
    q[k] = qq;
    uq[k] = uu + qq;
}

// x += alpha uq ; r -= alpha w ; out[0].re = ||r||^2 ; out[1] = (r0, r)      (cgs.rs:96-102, 121)
__global__ void __launch_bounds__(VEC_THREADS)
cgs_update_kernel(cplx* __restrict__ x, const cplx* __restrict__ uq, const cplx* __restrict__ w, cplx* __restrict__ r,
                  const cplx* __restrict__ r0, cplx alpha, uint64_t n, uint64_t S, cplx* __restrict__ out) {
    __shared__ ClusterShared sh;
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned me = cluster.block_rank();
    const uint64_t begin = (uint64_t)me * S, end = begin + S < n ? begin + S : n;
    cplx a0 = C(0, 0), a1 = C(0, 0);
    for (uint64_t k = begin + threadIdx.x; k < end; k += blockDim.x) {
        x[k] = x[k] + uq[k] * alpha;
        const cplx rr = r[k] - w[k] * alpha;
        r[k] = rr;
        const cplx q = r0[k];
        a0.re = fma(rr.re, rr.re, fma(rr.im, rr.im, a0.re));
        a1.re = fma(q.re, rr.re, fma(q.im, rr.im, a1.re));
        a1.im = fma(q.re, rr.im, fma(-q.im, rr.re, a1.im));
    }
    const cplx t0 = cluster_allreduce(a0, sh, 0);
    const cplx t1 = cluster_allreduce(a1, sh, 1);
    if (me == 0 && threadIdx.x == 0) { out[0] = t0; out[1] = t1; }
    cluster.sync();
}

// u = r + beta q ; p = u + beta (q + beta p)      (cgs.rs:134-139)
__global__ void cgs_p_kernel(const cplx* __restrict__ r, const cplx* __restrict__ q, cplx beta, cplx* __restrict__ u,
                             cplx* __restrict__ p, uint64_t n) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const cplx qq = q[k];
    const cplx uu = r[k] + qq * beta;
    u[k] = uu;
    const cplx qp = qq + p[k] * beta;
    p[k] = uu + qp * beta;
}

// ---- batched (one cluster per right-hand side) MGS step; same algebra as
// mgs_cluster_reg_kernel.  RHS index = blockIdx.y.  w is read from the block-matvec output
// Yblk[k][S]; v_{j+1} is written both to the RHS's own contiguous Krylov basis and to the
// interleaved block Xblk[k][S] that feeds the next block matvec.
template <int EPT>
__global__ void __launch_bounds__(256)
mgs_batched_kernel(const cplx* __restrict__ Vall, uint64_t ldv, uint64_t vstride, const cplx* __restrict__ Yblk, int S_rhs,
                   int j, uint64_t n, uint64_t S, cplx* __restrict__ hcol_all, uint64_t hstride, cplx* __restrict__ Xblk,
                   double breakdown_tol, const unsigned char* __restrict__ active) {
    __shared__ ClusterShared sh;
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned me = cluster.block_rank();
    const int rhs = blockIdx.y;
    if (active && !active[rhs]) return;  // whole cluster leaves together: no barrier is left waiting
    const cplx* V = Vall + (uint64_t)rhs * vstride;
    cplx* hcol = hcol_all + (uint64_t)rhs * hstride;
    const uint64_t begin = (uint64_t)me * S;
    const uint64_t end = begin + S < n ? begin + S : n;
    const uint64_t len = end > begin ? end - begin : 0;
    cplx wr[EPT], vc[EPT], vn[EPT];
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
        const uint64_t k = threadIdx.x + (uint64_t)e * blockDim.x;
        wr[e] = k < len ? ldg_c(Yblk + (begin + k) * S_rhs + rhs) : C(0, 0);
        vc[e] = k < len ? ldg_c(V + begin + k) : C(0, 0);
    }
    int parity = 0;
    for (int i = 0; i <= j; ++i) {
        if (i < j) {
            const cplx* vi1 = V + (uint64_t)(i + 1) * ldv + begin;
#pragma unroll
            for (int e = 0; e < EPT; ++e) {
                const uint64_t k = threadIdx.x + (uint64_t)e * blockDim.x;
                vn[e] = k < len ? ldg_c(vi1 + k) : C(0, 0);
            }
        }
        cplx acc = C(0, 0);
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            acc.re = fma(vc[e].re, wr[e].re, fma(vc[e].im, wr[e].im, acc.re));
            acc.im = fma(vc[e].re, wr[e].im, fma(-vc[e].im, wr[e].re, acc.im));
        }
        const cplx h = cluster_allreduce(acc, sh, parity);
        parity ^= 1;
        if (me == 0 && threadIdx.x == 0) hcol[i] = h;
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            wr[e].re = fma(-h.re, vc[e].re, fma(h.im, vc[e].im, wr[e].re));
            wr[e].im = fma(-h.re, vc[e].im, fma(-h.im, vc[e].re, wr[e].im));
            vc[e] = vn[e];
        }
    }
    cplx acc = C(0, 0);
#pragma unroll
    for (int e = 0; e < EPT; ++e) acc.re = fma(wr[e].re, wr[e].re, fma(wr[e].im, wr[e].im, acc.re));
    const cplx nn = cluster_allreduce(acc, sh, parity);
    const double nrm = sqrt(nn.re);
    if (me == 0 && threadIdx.x == 0) hcol[j + 1] = C(nrm, 0.0);
    if (!(nrm < breakdown_tol)) {
        const double sc = 1.0 / nrm - 1.0;
        cplx* vnext = const_cast<cplx*>(V) + (uint64_t)(j + 1) * ldv;
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const uint64_t k = threadIdx.x + (uint64_t)e * blockDim.x;
            if (k < len) {
                const cplx v = C(wr[e].re + wr[e].re * sc, wr[e].im + wr[e].im * sc);
                vnext[begin + k] = v;
                Xblk[(begin + k) * S_rhs + rhs] = v;
            }
        }
    }
    cluster.sync();
}

// Same step for slices that do not fit the registers (n > 32 768): the CTA keeps its slice of w in SHARED memory (up to
// 12 288 complex numbers = 192 KB per CTA, 16 CTAs per cluster => n <= 196 608) and streams the basis vectors through
// registers; every thread owns the same elements k = tid + 256 e in all passes, so no block barrier is needed between
// them, and the summation order per thread equals the register variant's.
__global__ void __launch_bounds__(256)
mgs_batched_smem_kernel(const cplx* __restrict__ Vall, uint64_t ldv, uint64_t vstride, const cplx* __restrict__ Yblk, int S_rhs,
                        int j, uint64_t n, uint64_t S, cplx* __restrict__ hcol_all, uint64_t hstride, cplx* __restrict__ Xblk,
                        double breakdown_tol, const unsigned char* __restrict__ active) {
    extern __shared__ __align__(16) unsigned char mgs_smem_raw[];
    cplx* w_s = reinterpret_cast<cplx*>(mgs_smem_raw);
    __shared__ ClusterShared sh;
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned me = cluster.block_rank();
    const int rhs = blockIdx.y;
    if (active && !active[rhs]) return;  // whole cluster leaves together
    const cplx* V = Vall + (uint64_t)rhs * vstride;
    cplx* hcol = hcol_all + (uint64_t)rhs * hstride;
    const uint64_t begin = (uint64_t)me * S;
    const uint64_t end = begin + S < n ? begin + S : n;
    const uint64_t len = end > begin ? end - begin : 0;
    for (uint64_t k = threadIdx.x; k < len; k += 256) w_s[k] = ldg_c(Yblk + (begin + k) * S_rhs + rhs);
    int parity = 0;
    for (int i = 0; i <= j; ++i) {
        const cplx* vi = V + (uint64_t)i * ldv + begin;
        cplx acc = C(0, 0);
        for (uint64_t k = threadIdx.x; k < len; k += 256) {
            const cplx v = ldg_c(vi + k), w = w_s[k];
            acc.re = fma(v.re, w.re, fma(v.im, w.im, acc.re));
            acc.im = fma(v.re, w.im, fma(-v.im, w.re, acc.im));
        }
        const cplx h = cluster_allreduce(acc, sh, parity);
        parity ^= 1;
        if (me == 0 && threadIdx.x == 0) hcol[i] = h;
        for (uint64_t k = threadIdx.x; k < len; k += 256) {
            const cplx v = ldg_c(vi + k);
            cplx w = w_s[k];
            w.re = fma(-h.re, v.re, fma(h.im, v.im, w.re));
            w.im = fma(-h.re, v.im, fma(-h.im, v.re, w.im));
            w_s[k] = w;
        }
    }
    cplx acc = C(0, 0);
    for (uint64_t k = threadIdx.x; k < len; k += 256) {
        const cplx w = w_s[k];
        acc.re = fma(w.re, w.re, fma(w.im, w.im, acc.re));
    }
    const cplx nn = cluster_allreduce(acc, sh, parity);
    const double nrm = sqrt(nn.re);
    if (me == 0 && threadIdx.x == 0) hcol[j + 1] = C(nrm, 0.0);
    if (!(nrm < breakdown_tol)) {
        const double sc = 1.0 / nrm - 1.0;
        cplx* vnext = const_cast<cplx*>(V) + (uint64_t)(j + 1) * ldv;
        for (uint64_t k = threadIdx.x; k < len; k += 256) {
            const cplx w = w_s[k];
            const cplx v = C(w.re + w.re * sc, w.im + w.im * sc);
            vnext[begin + k] = v;
            Xblk[(begin + k) * S_rhs + rhs] = v;
        }
    }
    cluster.sync();
}

// per-RHS residual of a block: R[:, s] = B[:, s] - AX[:, s] (interleaved [n][S]); out[s] = sum |R[:, s]|^2.
// One block per RHS (deterministic block reduction).
__global__ void __launch_bounds__(1024)
block_residual_kernel(const cplx* __restrict__ B, const cplx* __restrict__ AX, cplx* __restrict__ R, uint64_t n, int S_rhs,
                      double* __restrict__ out) {
    __shared__ double red[32];
    const int rhs = blockIdx.x;
    double acc = 0.0;
    for (uint64_t k = threadIdx.x; k < n; k += blockDim.x) {
        cplx v = B[k * S_rhs + rhs];
        if (AX) { v.re -= AX[k * S_rhs + rhs].re; v.im -= AX[k * S_rhs + rhs].im; }
        if (R) R[k * S_rhs + rhs] = v;
        acc = fma(v.re, v.re, fma(v.im, v.im, acc));
    }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, m);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
        out[rhs] = t;
    }
}

// v0[:, s] = R[:, s] * scale[s]: written to the RHS's contiguous basis slot 0 and to the interleaved block
__global__ void block_scale_kernel(const cplx* __restrict__ R, const double* __restrict__ scale, cplx* __restrict__ Vall,
                                   uint64_t vstride, cplx* __restrict__ Xblk, uint64_t n, int S_rhs) {
    const uint64_t total = n * (uint64_t)S_rhs;
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t k = e / S_rhs;
        const int s = (int)(e - k * S_rhs);
        const double sc = scale[s];
        const cplx v = C(R[e].re * sc, R[e].im * sc);
        Xblk[e] = v;
        Vall[(uint64_t)s * vstride + k] = v;
    }
}

// X[:, s] += sum_i y[s][i] V_s[i]  for the right-hand sides with cnt[s] > 0 (interleaved X)
__global__ void block_update_x_kernel(cplx* __restrict__ Xsol, const cplx* __restrict__ Vall, uint64_t ldv, uint64_t vstride,
                                      const cplx* __restrict__ ycoef, int ldy, const int* __restrict__ cnt, uint64_t n, int S_rhs) {
    const uint64_t total = n * (uint64_t)S_rhs;
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t k = e / S_rhs;
        const int s = (int)(e - k * S_rhs);
        const int c = cnt[s];
        if (c <= 0) continue;
        cplx v = Xsol[e];
        const cplx* V = Vall + (uint64_t)s * vstride;
        for (int i = 0; i < c; ++i) {
            const cplx a = ycoef[s * ldy + i], b = V[(uint64_t)i * ldv + k];
            v.re += a.re * b.re - a.im * b.im;
            v.im += a.re * b.im + a.im * b.re;
        }
        Xsol[e] = v;
    }
}

__global__ void scale_kernel(const cplx* __restrict__ r, double s, cplx* __restrict__ v, uint64_t n) {
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (uint64_t)gridDim.x * blockDim.x)
        v[k] = C(r[k].re * s, r[k].im * s);
}

// x += sum_i y_i V_i, applied in the reference's order i = 0..cnt-1 (gmres.rs:241-243)
__global__ void update_x_kernel(cplx* __restrict__ x, const cplx* __restrict__ V, uint64_t ldv, const cplx* __restrict__ ycoef,
                                int cnt, uint64_t n) {
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (uint64_t)gridDim.x * blockDim.x) {
        cplx v = x[k];
        for (int i = 0; i < cnt; ++i) {
            const cplx a = ycoef[i], b = V[(uint64_t)i * ldv + k];
            v.re += a.re * b.re - a.im * b.im;
            v.im += a.re * b.im + a.im * b.re;
        }
        x[k] = v;
    }
}

// apply_row_sum_correction (tbem.rs:500-520): one warp per local row
__global__ void row_sum_kernel(cplx* __restrict__ A, uint64_t lda, uint64_t nloc, uint64_t ncols, uint64_t r0,
                               cplx* __restrict__ rowsums) {
    const int lane = threadIdx.x & 31;
    const uint64_t row = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= nloc) return;
    cplx acc = C(0, 0);
    for (uint64_t c = lane; c < ncols; c += 32) { acc.re += A[row * lda + c].re; acc.im += A[row * lda + c].im; }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) {
        acc.re += __shfl_xor_sync(0xffffffffu, acc.re, m);
        acc.im += __shfl_xor_sync(0xffffffffu, acc.im, m);
    }
    if (lane == 0) {
        rowsums[row] = acc;
        A[row * lda + r0 + row].re -= acc.re;
        A[row * lda + r0 + row].im -= acc.im;
    }
}

// ---- measurement kernels ---------------------------------------------------------------------
__global__ void __launch_bounds__(256)
dfma_peak_kernel(double* out, int iters, double a, double b) {
    double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
            x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
        }
    }
    double s = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
    if (s == 123.456) out[0] = s;
}

__device__ __forceinline__ void atomic_max_pos(double* addr, double v) {
    atomicMax(reinterpret_cast<unsigned long long*>(addr), (unsigned long long)__double_as_longlong(v));
}
struct SelftestKappas {
    double kap[8];
    CisConst pos[8], neg[8];
};
__global__ void math_selftest_kernel(uint64_t n, double xmax, double* err, SelftestKappas kk) {
    __shared__ double2 tab[SINCOS_TAB];
    for (int i = threadIdx.x; i < SINCOS_TAB; i += blockDim.x) {
        double sv, cv;
        sincospi((double)i / SINCOS_STEPS_PER_PI, &sv, &cv);
        tab[i] = make_double2(cv, sv);
    }
    __syncthreads();
    double e_sc = 0.0, e_rs = 0.0;
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (uint64_t)gridDim.x * blockDim.x) {
        // low-discrepancy sample of [0, xmax]
        double u = (double)k * 0.6180339887498949;
        u -= floor(u);
        double x = u * xmax;
        double s, c, fs, fc;
        sincos(x, &s, &c);
        fast_sincos(x, fs, fc);
        e_sc = fmax(e_sc, fmax(fabs(fs - s), fabs(fc - c)));
        // the far kernel's variant takes the distance r and has kappa folded into its constants: reference = sin / cos of the
        // EXACT product kappa * r (double-double: p + e), first-order corrected
        const int ki = (int)(k & 7);
        const double kap = kk.kap[ki];
        const double r = x / kap;
        const double p = kap * r, e = fma(kap, r, -p);
        sincos(p, &s, &c);
        const double s_ref = fma(e, c, s), c_ref = fma(-e, s, c);
        fast_cis_tab(r, kk.pos[ki], tab, fs, fc);
        e_sc = fmax(e_sc, fmax(fabs(fs - s_ref), fabs(fc - c_ref)));
        fast_cis_tab(r, kk.neg[ki], tab, fs, fc);  // harmonic_factor = -1
        e_sc = fmax(e_sc, fmax(fabs(fs + s_ref), fabs(fc - c_ref)));
        double a = x * x + 1e-12;
        double ref = 1.0 / sqrt(a);
        e_rs = fmax(e_rs, fabs(fast_rsqrt(a) - ref) / ref);
    }
    atomic_max_pos(&err[0], e_sc);
    atomic_max_pos(&err[1], e_rs);
}

template <class Kern, class... Args>
cudaError_t launch_cluster(Kern kern, int cluster, int threads, size_t smem, cudaStream_t s, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(cluster, 1, 1);
    cfg.blockDim = dim3(threads, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cluster;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, args...);
}

}  // namespace

static cudaError_t launch_zgemv_impl(const cplx* A, uint64_t lda, uint64_t nrows, uint64_t ncols, const cplx* x, cplx* y,
                                     const PeerOut* po, cudaStream_t s) {
    if (nrows == 0 && !po) return cudaSuccess;
    uint64_t blocks = (nrows + 1) / 2;  // 2 rows per block
    const uint64_t maxb = 148ull * 8ull * 8ull;
    if (blocks > maxb) blocks = maxb;
    if (blocks == 0) blocks = 1;  // an empty slab still has to publish its epoch
    if (po) zgemv_kernel<2, 4, true><<<(unsigned)blocks, GEMV_THREADS, 0, s>>>(A, lda, nrows, ncols, x, y, *po);
    else zgemv_kernel<2, 4, false><<<(unsigned)blocks, GEMV_THREADS, 0, s>>>(A, lda, nrows, ncols, x, y, PeerOut{});
    return cudaGetLastError();
}

cudaError_t launch_zgemv(const cplx* A, uint64_t lda, uint64_t nrows, uint64_t ncols, const cplx* x, cplx* y, cudaStream_t s) {
    return launch_zgemv_impl(A, lda, nrows, ncols, x, y, nullptr, s);
}

cudaError_t launch_zgemv_peer(const cplx* A, uint64_t lda, uint64_t nrows, uint64_t ncols, const cplx* x, const PeerOut& po,
                              cudaStream_t s) {
    return launch_zgemv_impl(A, lda, nrows, ncols, x, nullptr, &po, s);
}

cudaError_t launch_zgemv_t(const cplx* A, uint64_t lda, uint64_t nrows, uint64_t ncols, const cplx* x, cplx* y, cudaStream_t s) {
    if (nrows == 0) return cudaMemsetAsync(y, 0, ncols * sizeof(cplx), s);
    const uint64_t rpc = (nrows + GEMVT_MAX_CHUNKS - 1) / GEMVT_MAX_CHUNKS;
    const int nchunks = (int)((nrows + rpc - 1) / rpc);
    cplx* part = nullptr;
    cudaError_t e = cudaMallocAsync((void**)&part, (size_t)nchunks * ncols * sizeof(cplx), s);
    if (e != cudaSuccess) return e;
    dim3 grid((unsigned)((ncols + 255) / 256), (unsigned)nchunks);
    zgemv_t_partial_kernel<<<grid, 256, 0, s>>>(A, lda, nrows, ncols, rpc, x, part);
    zgemv_t_reduce_kernel<<<(unsigned)((ncols + 255) / 256), 256, 0, s>>>(part, ncols, nchunks, y);
    e = cudaGetLastError();
    cudaFreeAsync(part, s);
    return e;
}

// cluster size / slice / where w lives.  `level` 0: preferred (w in shared memory, 16 CTAs if a
// slice would not fit in 8), level 1: conservative fallback (8 CTAs, w in global/L2).
static int pick_cluster(uint64_t n, int level, bool* w_in_smem, size_t* smem_bytes, uint64_t* slice) {
    int cl = n >= 4096 ? 8 : 1;
    uint64_t S = (n + cl - 1) / cl;
    const size_t cap = 200 * 1024;
    if (level == 0 && S * sizeof(cplx) > cap && cl == 8) {
        cl = 16;
        S = (n + cl - 1) / cl;
    }
    bool fits = level == 0 && S * sizeof(cplx) <= cap;
    *w_in_smem = fits;
    *smem_bytes = fits ? S * sizeof(cplx) : 0;
    *slice = S;
    return cl;
}

static PerDeviceInt g_cluster_level(0);

template <int EPT>
static cudaError_t launch_mgs_reg(int cl, const cplx* V, uint64_t ldv, const cplx* w, int j, uint64_t n, uint64_t S, cplx* hcol,
                                  cplx* vnext, const cplx* pinv, int direct_scale, cudaStream_t s) {
    static PerDeviceFlag attr_done;
    if (!attr_done.get()) {
        cudaError_t e = cudaFuncSetAttribute(mgs_cluster_reg_kernel<EPT>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        if (e != cudaSuccess) return e;
        attr_done.set();
    }
    return launch_cluster(mgs_cluster_reg_kernel<EPT>, cl, 256, 0, s, V, ldv, w, j, n, S, hcol, vnext, 1e-14, pinv, direct_scale);
}

template <int EPT>
static cudaError_t launch_mgs_lowsync(int cl, const cplx* V, uint64_t ldv, const cplx* w, int j, uint64_t n, uint64_t S, cplx* Lmat,
                                      int ldl, cplx* hcol, cplx* vnext, const cplx* pinv, int direct_scale, cplx* hcol_host,
                                      const PeerWait& pw, cudaStream_t s) {
    static PerDeviceFlag attr_done;
    const size_t fixed = (size_t)(LS_WARPS * 2 * LS_MAXV + MAX_CLUSTER * 2 * LS_MAXV + LS_MAXV) * sizeof(cplx);
    if (!attr_done.get()) {
        cudaError_t e = cudaFuncSetAttribute(mgs_lowsync_kernel<EPT>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(mgs_lowsync_kernel<EPT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)(fixed + (size_t)LS_MAXV * LS_MAXV * sizeof(cplx)));
        if (e != cudaSuccess) return e;
        attr_done.set();
    }
    const size_t smem = fixed + (size_t)(j + 1) * (j + 1) * sizeof(cplx);
    return launch_cluster(mgs_lowsync_kernel<EPT>, cl, LS_THREADS, smem, s, V, ldv, w, j, n, S, Lmat, ldl, hcol, vnext, 1e-14, pinv,
                          direct_scale, hcol_host, pw);
}

template <int EPT, int GR_THREADS>
static cudaError_t launch_mgs_grid(int G, const cplx* V, uint64_t ldv, const cplx* w, int j, uint64_t n, uint64_t S, cplx* Lmat,
                                   int ldl, cplx* hcol, cplx* vnext, const cplx* pinv, int direct_scale, cplx* scratch,
                                   cplx* hcol_host, const PeerWait& pw, cudaStream_t s) {
    constexpr int GR_WARPS = GR_THREADS / 32;
    static PerDeviceFlag attr_done;
    const size_t fixed = (size_t)(GR_WARPS * 2 * LS_MAXV + LS_MAXV) * sizeof(cplx);
    if (!attr_done.get()) {
        cudaError_t e = cudaFuncSetAttribute(mgs_grid_kernel<EPT, GR_THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)(fixed + (size_t)LS_MAXV * LS_MAXV * sizeof(cplx)));
        if (e != cudaSuccess) return e;
        attr_done.set();
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(G, 1, 1);
    cfg.blockDim = dim3(GR_THREADS, 1, 1);
    cfg.dynamicSmemBytes = fixed + (size_t)(j + 1) * (j + 1) * sizeof(cplx);
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cplx* part = scratch;
    double* npart = reinterpret_cast<double*>(scratch + (size_t)GR_MAX_CTAS * 2 * LS_MAXV);
    const double tol = 1e-14;
    return cudaLaunchKernelEx(&cfg, mgs_grid_kernel<EPT, GR_THREADS>, V, ldv, w, j, n, S, Lmat, ldl, hcol, vnext, tol, pinv, direct_scale,
                              part, npart, hcol_host, pw);
}

size_t mgs_scratch_elems() { return (size_t)GR_MAX_CTAS * 2 * LS_MAXV + GR_MAX_CTAS; }

// 3: whole-GPU cooperative low-sync kernel; 0: the cluster kernels of launch_mgs_cluster_path, for good once this device
// could not place the cooperative grid
static PerDeviceInt g_mgs_mode(3);

bool mgs_peer_wait_capable(uint64_t n, uint32_t restart) {
    if (restart + 1 > (uint32_t)LS_MAXV) return false;
    if (n <= 16ull * LS_THREADS * 8ull) return true;  // cluster low-sync kernel
    return g_mgs_mode.get() == 3 && n <= (uint64_t)GR_MAX_CTAS * 1024ull;
}

// `strict`: the caller is one rank of a row-sharded solve.  Every rank must run the SAME Arnoldi kernel
// (convergence decisions are not all-reduced; they agree because the arithmetic is identical), so a
// kernel that cannot be placed on this device is an error there, never a silent per-rank fallback.
static cudaError_t launch_mgs_cluster_path(const cplx* V, uint64_t ldv, cplx* w, int j, uint64_t n, cplx* hcol,
                                           cplx* vnext, const cplx* pinv, int direct_scale, cplx* Lmat, int ldl, cplx* hcol_host,
                                           bool* wrote_host, const PeerWait& pw, bool strict, cudaStream_t s) {
    *wrote_host = false;
    // 0: low-sync register kernel (16-CTA cluster) when the slice fits, 2: one-vector register kernel, 1: generic kernel;
    // a kernel this device cannot place demotes the mode of THIS device for good
    static PerDeviceInt cluster_mode(0);
    int mode = cluster_mode.get();
    if (mode == 0 && Lmat && j + 1 <= LS_MAXV && n <= 16ull * LS_THREADS * 8ull) {
        const int cl = n >= 2048 ? 16 : (n >= 512 ? 4 : 1);
        const uint64_t S = (n + cl - 1) / cl;
        const uint64_t ept = (S + LS_THREADS - 1) / LS_THREADS;
        cudaError_t e;
        if (ept <= 1) e = launch_mgs_lowsync<1>(cl, V, ldv, w, j, n, S, Lmat, ldl, hcol, vnext, pinv, direct_scale, hcol_host, pw, s);
        else if (ept <= 2) e = launch_mgs_lowsync<2>(cl, V, ldv, w, j, n, S, Lmat, ldl, hcol, vnext, pinv, direct_scale, hcol_host, pw, s);
        else if (ept <= 4) e = launch_mgs_lowsync<4>(cl, V, ldv, w, j, n, S, Lmat, ldl, hcol, vnext, pinv, direct_scale, hcol_host, pw, s);
        else e = launch_mgs_lowsync<8>(cl, V, ldv, w, j, n, S, Lmat, ldl, hcol, vnext, pinv, direct_scale, hcol_host, pw, s);
        if (e == cudaSuccess) { *wrote_host = hcol_host != nullptr; return e; }
        if (strict) return e;
        cudaGetLastError();
        mode = 2;
        cluster_mode.set(mode);
    }
    if (pw.ll) return cudaErrorNotSupported;  // only the two low-sync kernels know how to wait for peer slabs
    if ((mode == 0 || mode == 2) && n <= 16ull * 256ull * 8ull) {
        // register-resident w: 16 CTAs (non-portable cluster size) x 256 threads x <= 8 elements
        const int cl = n >= 2048 ? 16 : (n >= 512 ? 4 : 1);
        const uint64_t S = (n + cl - 1) / cl;
        const uint64_t ept = (S + 255) / 256;
        cudaError_t e;
        if (ept <= 1) e = launch_mgs_reg<1>(cl, V, ldv, w, j, n, S, hcol, vnext, pinv, direct_scale, s);
        else if (ept <= 2) e = launch_mgs_reg<2>(cl, V, ldv, w, j, n, S, hcol, vnext, pinv, direct_scale, s);
        else if (ept <= 4) e = launch_mgs_reg<4>(cl, V, ldv, w, j, n, S, hcol, vnext, pinv, direct_scale, s);
        else e = launch_mgs_reg<8>(cl, V, ldv, w, j, n, S, hcol, vnext, pinv, direct_scale, s);
        if (e == cudaSuccess) return e;
        if (strict) return e;
        cudaGetLastError();  // a 16-CTA cluster this device cannot place: fall back for good
        cluster_mode.set(1);
    }
    static PerDeviceFlag attr_done;
    if (!attr_done.get()) {
        cudaError_t e = cudaFuncSetAttribute(mgs_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(mgs_cluster_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        if (e != cudaSuccess) return e;
        attr_done.set();
    }
    for (;;) {
        bool in_smem;
        size_t smem;
        uint64_t S;
        // a row-sharded solve always uses the conservative placement (8 CTAs, w in global): identical on every rank
        const int level = strict ? 1 : g_cluster_level.get();
        int cl = pick_cluster(n, level, &in_smem, &smem, &S);
        cudaError_t e = launch_cluster(mgs_cluster_kernel, cl, VEC_THREADS, smem, s, V, ldv, w, j, n, S, (int)in_smem, hcol,
                                       vnext, 1e-14, pinv, direct_scale);
        if (e == cudaSuccess || level == 1) return e;
        cudaGetLastError();  // e.g. a 16-CTA / 200 KB cluster that this GPC layout cannot place
        g_cluster_level.set(1);
    }
}

cudaError_t launch_mgs(const cplx* V, uint64_t ldv, cplx* w, int j, uint64_t n, cplx* hcol, cplx* vnext, const cplx* pinv,
                       int direct_scale, cplx* Lmat, int ldl, cplx* scratch, cplx* hcol_host, bool* wrote_host,
                       const PeerWait& pw, bool strict, cudaStream_t s) {
    *wrote_host = false;
    // mode 3: whole-GPU cooperative kernel; the slice per CTA depends on n only.
    // It runs beside a background assembly too: with the counter-driven far kernel at two persistent blocks per SM it measured
    // 100.4 against 104.3 ms per frequency for cluster kernel + one block per SM on the same box (profiles/r02r_*.json); the
    // cluster kernel cannot be placed while two far blocks sit on every SM, the cooperative grid (one small CTA per SM) can.
    if (g_mgs_mode.get() == 3 && Lmat && scratch && j + 1 <= LS_MAXV && n >= 4096 && n <= (uint64_t)GR_MAX_CTAS * 1024ull) {
        const int G = GR_MAX_CTAS;  // fixed (not the SM count of the device): the summation order must not depend on the rank's GPU
        const uint64_t S = (n + G - 1) / G;
        cudaError_t e;
#define GRID_CASE(E, T) e = launch_mgs_grid<E, T>(G, V, ldv, w, j, n, S, Lmat, ldl, hcol, vnext, pinv, direct_scale, scratch, hcol_host, pw, s)
        if (S <= 128) GRID_CASE(1, 128);
        else if (S <= 256) GRID_CASE(2, 128);
        else if (S <= 512) GRID_CASE(2, 256);
        else GRID_CASE(4, 256);
#undef GRID_CASE
        if (e == cudaSuccess) { *wrote_host = hcol_host != nullptr; return e; }
        if (strict) return e;  // e.g. a device with fewer than 148 SMs in a multi-rank job: fail loudly
        cudaGetLastError();  // cooperative launch not placeable on this device: cluster kernels from now on
        g_mgs_mode.set(0);
    }
    // small or very long vectors, or a device that cannot place the cooperative grid: the cluster kernels
    return launch_mgs_cluster_path(V, ldv, w, j, n, hcol, vnext, pinv, direct_scale, Lmat, ldl, hcol_host, wrote_host, pw, strict, s);
}

cudaError_t launch_residual(const cplx* b, const cplx* ax, cplx* r, uint64_t n, double* out, const cplx* pinv, cudaStream_t s) {
    bool in_smem;
    size_t smem;
    uint64_t S;
    int cl = pick_cluster(n, 1, &in_smem, &smem, &S);  // no shared-memory slice needed: 8 CTAs always place
    return launch_cluster(residual_cluster_kernel, cl, VEC_THREADS, 0, s, b, ax, r, n, S, out, pinv);
}

static inline int bicg_cluster(uint64_t n, uint64_t* S) {
    const int cl = n >= 4096 ? 8 : 1;
    *S = (n + cl - 1) / cl;
    return cl;
}
cudaError_t launch_bicg_dot(const cplx* a, const cplx* b, uint64_t n, cplx* out, cudaStream_t s) {
    uint64_t S;
    const int cl = bicg_cluster(n, &S);
    return launch_cluster(bicg_dot_kernel, cl, VEC_THREADS, 0, s, a, b, n, S, out);
}
cudaError_t launch_bicg_p(const cplx* r, cplx* p, const cplx* v, cplx beta, cplx omega, uint64_t n, cudaStream_t s) {
    bicg_p_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(r, p, v, beta, omega, n);
    return cudaGetLastError();
}
cudaError_t launch_bicg_s(const cplx* r, const cplx* v, cplx alpha, cplx* sv, uint64_t n, cplx* out, cudaStream_t s) {
    uint64_t S;
    const int cl = bicg_cluster(n, &S);
    return launch_cluster(bicg_s_kernel, cl, VEC_THREADS, 0, s, r, v, alpha, sv, n, S, out);
}
cudaError_t launch_bicg_tt(const cplx* t, const cplx* sv, uint64_t n, cplx* out, cudaStream_t s) {
    uint64_t S;
    const int cl = bicg_cluster(n, &S);
    return launch_cluster(bicg_tt_kernel, cl, VEC_THREADS, 0, s, t, sv, n, S, out);
}
cudaError_t launch_bicg_update(cplx* x, const cplx* p, const cplx* sv, const cplx* t, cplx* r, const cplx* r0, cplx alpha, cplx omega,
                               uint64_t n, cplx* out, cudaStream_t s) {
    uint64_t S;
    const int cl = bicg_cluster(n, &S);
    return launch_cluster(bicg_update_kernel, cl, VEC_THREADS, 0, s, x, p, sv, t, r, r0, alpha, omega, n, S, out);
}
cudaError_t launch_bicg_axpy(cplx* x, const cplx* p, cplx alpha, uint64_t n, cudaStream_t s) {
    bicg_axpy_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(x, p, alpha, n);
    return cudaGetLastError();
}

cudaError_t launch_cgs_q(const cplx* u, const cplx* v, cplx alpha, cplx* q, cplx* uq, uint64_t n, cudaStream_t s) {
    cgs_q_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(u, v, alpha, q, uq, n);
    return cudaGetLastError();
}
cudaError_t launch_cgs_update(cplx* x, const cplx* uq, const cplx* w, cplx* r, const cplx* r0, cplx alpha, uint64_t n, cplx* out,
                              cudaStream_t s) {
    uint64_t S;
    const int cl = bicg_cluster(n, &S);
    return launch_cluster(cgs_update_kernel, cl, VEC_THREADS, 0, s, x, uq, w, r, r0, alpha, n, S, out);
}
cudaError_t launch_cgs_p(const cplx* r, const cplx* q, cplx beta, cplx* u, cplx* p, uint64_t n, cudaStream_t s) {
    cgs_p_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(r, q, beta, u, p, n);
    return cudaGetLastError();
}

template <int EPT>
static cudaError_t launch_mgs_batched_t(int cl, int nrhs, const cplx* Vall, uint64_t ldv, uint64_t vstride, const cplx* Yblk,
                                        int j, uint64_t n, uint64_t S, cplx* hcol_all, uint64_t hstride, cplx* Xblk,
                                        const unsigned char* active, cudaStream_t s) {
    static PerDeviceFlag attr_done;
    if (!attr_done.get()) {
        cudaError_t e = cudaFuncSetAttribute(mgs_batched_kernel<EPT>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        if (e != cudaSuccess) return e;
        attr_done.set();
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(cl, nrhs, 1);
    cfg.blockDim = dim3(256, 1, 1);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cl;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, mgs_batched_kernel<EPT>, Vall, ldv, vstride, Yblk, nrhs, j, n, S, hcol_all, hstride, Xblk,
                              1e-14, active);
}

cudaError_t launch_mgs_batched(int nrhs, const cplx* Vall, uint64_t ldv, uint64_t vstride, const cplx* Yblk, int j, uint64_t n,
                               cplx* hcol_all, uint64_t hstride, cplx* Xblk, const unsigned char* active, cudaStream_t s) {
    if (n > 16ull * 256ull * 8ull) {  // slices beyond the register-resident variant: w in shared memory
        constexpr uint64_t SMEM_ELEMS = 12288;  // 192 KB per CTA
        const int clb = 16;
        const uint64_t Sb = (n + clb - 1) / clb;
        if (Sb > SMEM_ELEMS) return cudaErrorInvalidValue;  // n > 196 608
        static PerDeviceFlag attr_done_b;
        if (!attr_done_b.get()) {
            cudaError_t e = cudaFuncSetAttribute(mgs_batched_smem_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
            if (e == cudaSuccess)
                e = cudaFuncSetAttribute(mgs_batched_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(SMEM_ELEMS * sizeof(cplx)));
            if (e != cudaSuccess) return e;
            attr_done_b.set();
        }
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(clb, nrhs, 1);
        cfg.blockDim = dim3(256, 1, 1);
        cfg.dynamicSmemBytes = Sb * sizeof(cplx);
        cfg.stream = s;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = clb;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        return cudaLaunchKernelEx(&cfg, mgs_batched_smem_kernel, Vall, ldv, vstride, Yblk, nrhs, j, n, Sb, hcol_all, hstride, Xblk, 1e-14,
                                  active);
    }
    const int cl = n >= 2048 ? 16 : (n >= 512 ? 4 : 1);
    const uint64_t S = (n + cl - 1) / cl;
    const uint64_t ept = (S + 255) / 256;
    if (ept <= 1) return launch_mgs_batched_t<1>(cl, nrhs, Vall, ldv, vstride, Yblk, j, n, S, hcol_all, hstride, Xblk, active, s);
    if (ept <= 2) return launch_mgs_batched_t<2>(cl, nrhs, Vall, ldv, vstride, Yblk, j, n, S, hcol_all, hstride, Xblk, active, s);
    if (ept <= 4) return launch_mgs_batched_t<4>(cl, nrhs, Vall, ldv, vstride, Yblk, j, n, S, hcol_all, hstride, Xblk, active, s);
    return launch_mgs_batched_t<8>(cl, nrhs, Vall, ldv, vstride, Yblk, j, n, S, hcol_all, hstride, Xblk, active, s);
}

__global__ void interleave_kernel(const cplx* __restrict__ src, cplx* __restrict__ dst, uint64_t n, int nsrc, int S_rhs, int to_block) {
    // to_block: src [nsrc][n] -> dst [n][S_rhs] (columns >= nsrc zero);  else: src [n][S_rhs] -> dst [nsrc][n]
    const uint64_t total = n * (uint64_t)S_rhs;
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t k = e / S_rhs;
        const int s2 = (int)(e - k * S_rhs);
        if (to_block) dst[e] = s2 < nsrc ? src[(uint64_t)s2 * n + k] : C(0, 0);
        else if (s2 < nsrc) dst[(uint64_t)s2 * n + k] = src[e];
    }
}

cudaError_t launch_interleave(const cplx* src, cplx* dst, uint64_t n, int nsrc, int nrhs, int to_block, cudaStream_t s) {
    interleave_kernel<<<148 * 4, 256, 0, s>>>(src, dst, n, nsrc, nrhs, to_block);
    return cudaGetLastError();
}

cudaError_t launch_block_residual(const cplx* B, const cplx* AX, cplx* R, uint64_t n, int nrhs, double* out, cudaStream_t s) {
    block_residual_kernel<<<nrhs, 1024, 0, s>>>(B, AX, R, n, nrhs, out);
    return cudaGetLastError();
}

cudaError_t launch_block_scale(const cplx* R, const double* scale, cplx* Vall, uint64_t vstride, cplx* Xblk, uint64_t n, int nrhs,
                               cudaStream_t s) {
    block_scale_kernel<<<148 * 4, 256, 0, s>>>(R, scale, Vall, vstride, Xblk, n, nrhs);
    return cudaGetLastError();
}

cudaError_t launch_block_update_x(cplx* Xsol, const cplx* Vall, uint64_t ldv, uint64_t vstride, const cplx* ycoef, int ldy,
                                  const int* cnt, uint64_t n, int nrhs, cudaStream_t s) {
    block_update_x_kernel<<<148 * 4, 256, 0, s>>>(Xsol, Vall, ldv, vstride, ycoef, ldy, cnt, n, nrhs);
    return cudaGetLastError();
}

cudaError_t launch_scale(const cplx* r, double sc, cplx* v, uint64_t n, cudaStream_t s) {
    unsigned blocks = (unsigned)((n + 255) / 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    scale_kernel<<<blocks, 256, 0, s>>>(r, sc, v, n);
    return cudaGetLastError();
}

cudaError_t launch_update_x(cplx* x, const cplx* V, uint64_t ldv, const cplx* ycoef, int cnt, uint64_t n, cudaStream_t s) {
    unsigned blocks = (unsigned)((n + 255) / 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    update_x_kernel<<<blocks, 256, 0, s>>>(x, V, ldv, ycoef, cnt, n);
    return cudaGetLastError();
}

cudaError_t launch_row_sum(cplx* A, uint64_t lda, uint64_t nloc, uint64_t ncols, uint64_t r0, cplx* rowsums, cudaStream_t s) {
    if (nloc == 0) return cudaSuccess;
    unsigned blocks = (unsigned)((nloc * 32 + 255) / 256);
    row_sum_kernel<<<blocks, 256, 0, s>>>(A, lda, nloc, ncols, r0, rowsums);
    return cudaGetLastError();
}

cudaError_t launch_dfma_peak(double* out, int iters, cudaStream_t s) {
    dfma_peak_kernel<<<148 * 8, 256, 0, s>>>(out, iters, 1.0000001, 1e-9);
    return cudaGetLastError();
}

cudaError_t launch_math_selftest(uint64_t n, double xmax, double* err, cudaStream_t s) {
    SelftestKappas kk;
    const double kaps[8] = {1.0, 2.5, 9.162978572970230, 18.31686157546442, 20.0, 36.63372315092884, 0.3, 146.5348926037154};
    for (int i = 0; i < 8; ++i) {
        kk.kap[i] = kaps[i];
        kk.pos[i] = make_cis_const(kaps[i]);
        kk.neg[i] = make_cis_const(-kaps[i]);
    }
    math_selftest_kernel<<<148 * 4, 256, 0, s>>>(n, xmax, err, kk);
    return cudaGetLastError();
}

}  // namespace bemb
