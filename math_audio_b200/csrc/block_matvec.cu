// block_matvec.cu -- Y = A X for S = 8 ... 32 right-hand sides at once (BASELINE config 5; the reference would loop
// DenseOperator::apply, math-bem/src/core/solver/fmm_interface.rs:44-47, over the right-hand sides).
//
// 8 N^2 S flop on 16 N^2 bytes: 16 flop/byte at S = 32, above the FP64 ridge of the B200 (5.8), so the kernel is bound by
// FP64 issue.  tcgen05 has no f64 kind; what the part offers is measured by tools/fp64_operand_probe.cu
// (profiles/r02h_fp64_operand_probe.log):
//   * DFMA with three register sources issues at 2/3 rate (0.66 of the nominal 37.2 TFLOP/s; 0.99 with two), a register-tiled
//     DFMA GEMM reaches 0.79-0.85 even with nothing else in the loop (a first version of this kernel: 0.686);
//   * mma.sync.m8n8k4.f64 (SASS DMMA.8x8x4; the larger f64 shapes compile to sequences of it) runs at 0.99 of nominal
//     from registers: 256 FMAs per instruction for four 64-bit register reads.
// So the contraction is done by DMMA.8x8x4 -- complex product = 4 real MMAs -- and everything else exists to keep that pipe fed:
//   * CTA tile = 256 rows x S right-hand sides, 8 warps; warp = 32 rows (4 m-blocks of 8) x S (S/8 n-tiles): per 4-k step
//     4 + S/8 shared-memory loads of 16 bytes feed 16 S/8 DMMAs (S = 32: 8 LDS for 64 DMMAs = 1 024 pipe cycles);
//   * A (256 x 8 complex per stage) and X (8 x S) reach shared memory by 16-byte cp.async in a 4-stage ring; 8 consecutive
//     lanes fetch the 128 contiguous bytes of one matrix row segment; both tiles are XOR-swizzled so that the fragment loads
//     (lanes = 8 rows x 4 k for A, 4 k x 8 columns for X) are conflict-free without padding;
//   * stream-K: the grid is one CTA per SM and CTA c owns the contiguous range [c U / G, (c+1) U / G) of the U = tiles x
//     k-chunks work units, so every SM executes the same number of MMAs whatever the row count (20 480 rows are 80 tiles
//     for 148 SMs: a tile-per-CTA grid would idle 46 % of the machine).  A CTA that covers only part of a tile's k range
//     writes a partial tile; block_fixup_kernel adds the partials of a tile in CTA order -- fixed order, bit-deterministic.
#include <algorithm>
#include <cstdlib>
#include <mutex>

#include "linalg.h"

namespace bemb {

namespace {

constexpr int SK_WARPS = 8;
constexpr int SK_THREADS = SK_WARPS * 32;
constexpr int SK_BM = SK_WARPS * 32;  // rows per tile
constexpr int SK_BK = 8;              // k per stage
constexpr int SK_LDA = SK_BK;         // A tile row stride (complex); slot of (r, k) is r * 8 + (k ^ ((r & 1) << 2))
constexpr int SK_STAGES = 4;

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, bool valid) {
    const uint32_t sa = (uint32_t)__cvta_generic_to_shared(smem);
    const int sz = valid ? 16 : 0;  // src-size 0: the 16 bytes are zero-filled
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sa), "l"(gmem), "r"(sz) : "memory");
}

struct SkRange {
    unsigned long long u0, u1;
};
__host__ __device__ inline SkRange sk_range(unsigned c, unsigned G, unsigned long long U) {
    return SkRange{(unsigned long long)c * U / G, (unsigned long long)(c + 1) * U / G};
}

__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// NT = S / 8 n-tiles per warp
template <int NT>
__global__ void __launch_bounds__(SK_THREADS, 1)
zgemm_streamk_kernel(const cplx* __restrict__ A, uint64_t lda, uint64_t nrows, uint64_t ncols, const cplx* __restrict__ X,
                     cplx* __restrict__ Y, cplx* __restrict__ partial, unsigned nk) {
    constexpr int S = 8 * NT;
    constexpr int MR = 4;  // m-blocks (8 rows each) per warp
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cplx* As = reinterpret_cast<cplx*>(smem_raw);                    // [SK_STAGES][SK_BM * SK_LDA]
    cplx* Xs = As + (size_t)SK_STAGES * SK_BM * SK_LDA;              // [SK_STAGES][SK_BK * S]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, kq = lane & 3;  // MMA fragment coordinates: A[g][kq], B[kq][g], C[g][2 kq .. 2 kq + 1]
    const unsigned G = gridDim.x;
    const unsigned long long ntiles = (nrows + SK_BM - 1) / SK_BM;
    const unsigned long long U = ntiles * nk;
    const SkRange mine = sk_range(blockIdx.x, G, U);
    // cp.async roles: 8 consecutive lanes fetch one 128-byte row segment; thread -> (row tid/8 + 32 p, k tid%8)
    const int ld_k = tid & 7, ld_r = tid >> 3;
    constexpr int LD_ROWS = SK_THREADS / 8;

    unsigned long long u = mine.u0;
    while (u < mine.u1) {
        const unsigned long long tile = u / nk;
        const unsigned k0 = (unsigned)(u - tile * nk);
        const unsigned long long kend_l = k0 + (mine.u1 - u);
        const unsigned kend = kend_l < nk ? (unsigned)kend_l : nk;
        const uint64_t row0 = tile * SK_BM;
        // first source row of this thread (rows past the end are clamped: computed and dropped)
        const uint64_t last_row = nrows - 1;

        auto stage = [&](unsigned kc, int slot) {
            cplx* as = As + (size_t)slot * SK_BM * SK_LDA;
            cplx* xs = Xs + (size_t)slot * SK_BK * S;
            const uint64_t k = (uint64_t)kc * SK_BK + ld_k;
            const bool kin = k < ncols;
            const uint64_t ks = kin ? k : 0;
#pragma unroll
            for (int p = 0; p < SK_BM / LD_ROWS; ++p) {
                const int r = ld_r + LD_ROWS * p;
                uint64_t gr = row0 + r;
                if (gr > last_row) gr = last_row;
                cp_async16(as + r * SK_LDA + (ld_k ^ ((r & 1) << 2)), A + gr * lda + ks, kin);
            }
            for (int e = tid; e < SK_BK * S; e += SK_THREADS) {
                const int kk = e / S, n = e - kk * S;
                const uint64_t kx = (uint64_t)kc * SK_BK + kk;
                cp_async16(xs + kk * S + (n ^ ((kk & 3) << 1)), X + (kx < ncols ? kx * S + n : 0), kx < ncols);
            }
        };

        double cre[MR][NT][2], cim[MR][NT][2];
#pragma unroll
        for (int m = 0; m < MR; ++m)
#pragma unroll
            for (int t = 0; t < NT; ++t) cre[m][t][0] = cre[m][t][1] = cim[m][t][0] = cim[m][t][1] = 0.0;

        __syncthreads();  // the previous segment is done with the ring
        // prologue: SK_STAGES - 1 stages in flight (empty commit groups keep the count uniform)
#pragma unroll
        for (int s = 0; s < SK_STAGES - 1; ++s) {
            if (k0 + s < kend) stage(k0 + s, s);
            asm volatile("cp.async.commit_group;" ::: "memory");
        }
        for (unsigned kc = k0; kc < kend; ++kc) {
            const int slot = (int)((kc - k0) % SK_STAGES);
            asm volatile("cp.async.wait_group %0;" ::"n"(SK_STAGES - 2) : "memory");
            __syncthreads();  // stage kc has landed for everybody, and everybody has left stage kc - 1
            {
                const unsigned nxt = kc + SK_STAGES - 1;
                if (nxt < kend) stage(nxt, (int)((nxt - k0) % SK_STAGES));
                asm volatile("cp.async.commit_group;" ::: "memory");
            }
            const cplx* as = As + (size_t)slot * SK_BM * SK_LDA + (warp * 32 + g) * SK_LDA;
            const cplx* xs = Xs + (size_t)slot * SK_BK * S;
#pragma unroll
            for (int k4 = 0; k4 < SK_BK / 4; ++k4) {
                const int k = 4 * k4 + kq;
                double2 a[MR], x[NT];
#pragma unroll
                for (int m = 0; m < MR; ++m)  // row warp*32 + 8 m + g has the parity of g
                    a[m] = *reinterpret_cast<const double2*>(as + 8 * m * SK_LDA + (k ^ ((g & 1) << 2)));
#pragma unroll
                for (int t = 0; t < NT; ++t)
                    x[t] = *reinterpret_cast<const double2*>(xs + k * S + ((8 * t + g) ^ (kq << 1)));
#pragma unroll
                for (int m = 0; m < MR; ++m) {
                    const double naim = -a[m].y;
#pragma unroll
                    for (int t = 0; t < NT; ++t) {
                        dmma884(cre[m][t][0], cre[m][t][1], a[m].x, x[t].x);
                        dmma884(cim[m][t][0], cim[m][t][1], a[m].x, x[t].y);
                        dmma884(cre[m][t][0], cre[m][t][1], naim, x[t].y);
                        dmma884(cim[m][t][0], cim[m][t][1], a[m].y, x[t].x);
                    }
                }
            }
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");

        // ---- epilogue: whole k range -> Y, otherwise a partial tile (slot 0: the segment starts inside the tile) ----
        const bool whole = (k0 == 0 && kend == nk);
        cplx* dst = whole ? Y + row0 * S
                          : partial + ((size_t)blockIdx.x * 2 + (k0 > 0 ? 0 : 1)) * (size_t)SK_BM * S;
#pragma unroll
        for (int m = 0; m < MR; ++m) {
            const int r = warp * 32 + 8 * m + g;
            if (!whole || row0 + r < nrows) {
#pragma unroll
                for (int t = 0; t < NT; ++t)  // D fragment: row g, columns 2 kq and 2 kq + 1 of n-tile t
                    *reinterpret_cast<double4*>(dst + (size_t)r * S + 8 * t + 2 * kq) =
                        make_double4(cre[m][t][0], cim[m][t][0], cre[m][t][1], cim[m][t][1]);
            }
        }
        u += kend - k0;
    }
}

// Y tile = sum of its partial tiles, in CTA order (tiles covered by one CTA were written directly)
template <int S>
__global__ void __launch_bounds__(256)
block_fixup_kernel(uint64_t nrows, unsigned nk, unsigned G, const cplx* __restrict__ partial, cplx* __restrict__ Y) {
    __shared__ unsigned s_cnt;
    __shared__ unsigned s_src[8];  // (cta * 2 + slot) of every contributor, ascending CTA
    const unsigned long long tile = blockIdx.x;
    const unsigned long long ntiles = (nrows + SK_BM - 1) / SK_BM;
    const unsigned long long U = ntiles * nk;
    if (threadIdx.x == 0) {
        const unsigned long long t0 = tile * nk, t1 = t0 + nk;
        // first CTA whose range reaches into the tile, then walk forward
        unsigned long long cg0 = t0 * G / U;
        unsigned c = cg0 < G - 1 ? (unsigned)cg0 : G - 1;
        while (c > 0 && sk_range(c, G, U).u0 > t0) --c;
        while (sk_range(c, G, U).u1 <= t0) ++c;
        unsigned cnt = 0;
        for (; c < G; ++c) {
            const SkRange r = sk_range(c, G, U);
            if (r.u0 >= t1) break;
            const unsigned long long a = r.u0 > t0 ? r.u0 : t0, b = r.u1 < t1 ? r.u1 : t1;
            if (a >= b) continue;
            if (a == t0 && b == t1) { cnt = 0; break; }  // written directly
            if (cnt < 8) s_src[cnt++] = c * 2 + (a > t0 ? 0 : 1);
        }
        s_cnt = cnt;
    }
    __syncthreads();
    const unsigned cnt = s_cnt;
    if (cnt == 0) return;
    const uint64_t row0 = tile * SK_BM;
    for (unsigned e = blockIdx.y * blockDim.x + threadIdx.x; e < SK_BM * S; e += gridDim.y * blockDim.x) {
        const unsigned r = e / S;
        if (row0 + r >= nrows) continue;
        double re = 0.0, im = 0.0;
        for (unsigned q = 0; q < cnt; ++q) {
            const double2 v = *reinterpret_cast<const double2*>(partial + (size_t)s_src[q] * SK_BM * S + e);
            re += v.x; im += v.y;
        }
        *reinterpret_cast<double2*>(Y + row0 * S + e) = make_double2(re, im);
    }
}

struct SkDevice {
    int sms = 0;
    bool attr[8] = {};
};
SkDevice g_sk[64];
std::mutex g_sk_mu;

template <int NT>
cudaError_t launch_streamk_t(const cplx* A, uint64_t lda, uint64_t nrows, uint64_t ncols, const cplx* X, cplx* Y, cudaStream_t s) {
    constexpr int S = 8 * NT;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    const size_t smem = (size_t)SK_STAGES * (SK_BM * SK_LDA + SK_BK * S) * sizeof(cplx);
    unsigned G = 0;
    {
        std::lock_guard<std::mutex> lk(g_sk_mu);
        SkDevice& w = g_sk[dev];
        if (w.sms == 0) {
            e = cudaDeviceGetAttribute(&w.sms, cudaDevAttrMultiProcessorCount, dev);
            if (e != cudaSuccess) return e;
        }
        G = (unsigned)w.sms;
        if (!w.attr[NT]) {
            e = cudaFuncSetAttribute(zgemm_streamk_kernel<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            w.attr[NT] = true;
        }
    }
    const unsigned nk = (unsigned)((ncols + SK_BK - 1) / SK_BK);
    const unsigned long long ntiles = (nrows + SK_BM - 1) / SK_BM;
    if (ntiles * nk < G) G = (unsigned)(ntiles * nk);
    if (6ull * ntiles < G) G = (unsigned)(6ull * ntiles);  // a tile has at most G / ntiles + 2 <= 8 contributors (block_fixup_kernel's table)
    // partial tiles: stream-ordered scratch of THIS launch (two contexts of one device may run block products concurrently)
    cplx* partial = nullptr;
    e = cudaMallocAsync((void**)&partial, (size_t)G * 2 * SK_BM * S * sizeof(cplx), s);
    if (e != cudaSuccess) return e;
    zgemm_streamk_kernel<NT><<<G, SK_THREADS, smem, s>>>(A, lda, nrows, ncols, X, Y, partial, nk);
    e = cudaGetLastError();
    if (e == cudaSuccess) {
        block_fixup_kernel<S><<<dim3((unsigned)ntiles, 4), 256, 0, s>>>(nrows, nk, G, partial, Y);
        e = cudaGetLastError();
    }
    const cudaError_t fe = cudaFreeAsync(partial, s);
    return e != cudaSuccess ? e : fe;
}

}  // namespace

cudaError_t launch_zgemm_block(const cplx* A, uint64_t lda, uint64_t nrows, uint64_t ncols, const cplx* X, cplx* Y, int nrhs,
                               cudaStream_t s) {
    if (nrows == 0) return cudaSuccess;
    if (ncols == 0) return cudaMemsetAsync(Y, 0, nrows * (size_t)nrhs * sizeof(cplx), s);
    switch (nrhs) {
        case 8: return launch_streamk_t<1>(A, lda, nrows, ncols, X, Y, s);
        case 16: return launch_streamk_t<2>(A, lda, nrows, ncols, X, Y, s);
        case 24: return launch_streamk_t<3>(A, lda, nrows, ncols, X, Y, s);
        case 32: return launch_streamk_t<4>(A, lda, nrows, ncols, X, Y, s);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace bemb
