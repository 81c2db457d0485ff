// Persistent fused GMRES kernel (gmres_fused.cu): parameter block and launcher.
#pragma once
#include "linalg.h"

namespace bemb {

constexpr int FUSED_THREADS = 512;
constexpr int FUSED_KMAX = 160;        // complex values per reduction round / broadcast (2 (restart + 1) + 2 <= 130, padded)
constexpr int FUSED_MAX_RESTART = 63;  // larger restarts use the per-iteration kernels of linalg.cu
constexpr uint32_t FUSED_SEGMENT_WIDTH = FUSED_THREADS * 4;  // matrix columns per segment of the matvec (4 per thread, both builds)

struct FusedResult {
    unsigned long long iterations, restarts, matvecs;
    double residual;
    int converged;
    int error;   // a bounded wait timed out (a peer or a CTA never delivered): the solve is void
    int done;
    unsigned int ex_final, er_final;
    unsigned long long t_total_ns, t_matvec_ns, t_round_ns;  // reducer CTA's view: whole solve, inside matvec_rows, post-matvec -> payload received
};

struct FusedParams {
    const cplx* A;       // this rank's slab, row-major
    uint64_t lda;
    uint32_t n;          // unknowns (= columns)
    uint32_t row0;       // first global row of the slab
    uint32_t nloc;       // rows of the slab
    uint32_t npad;       // elements per exchange vector
    int rank, nranks;
    const cplx* b;       // right-hand side, full length
    cplx* x;             // in: initial guess (full length), out: solution (full length)
    cplx* V;             // Krylov basis, own rows only: V[l * ldv + i], i < nloc
    uint64_t ldv;
    const cplx* pinv;    // inverse diagonal (full length) or nullptr
    int direct_scale;    // preconditioned variant: v_{j+1} = w * (1/||w||)
    uint4* xbuf[MAX_PEERS];   // every rank's exchange vectors  [2][npad] flag-in-data elements
    uint4* rpart[MAX_PEERS];  // every rank's inbox of rank partials [2][nranks][FUSED_KMAX]
    uint4* cpart;             // local inbox of CTA partials [2][G][FUSED_KMAX]
    uint4* hbuf;              // local broadcast slots [2][FUSED_KMAX]
    uint32_t restart, max_cycles;
    double tol;
    uint32_t ex0, er0;   // last epochs used on these buffers
    unsigned long long timeout_ns;
    FusedResult* result; // device-visible (mapped pinned) record
    uint32_t S;          // rows per CTA (the largest share when row_off is given)
    uint32_t rblk;       // rows per matvec pass inside a CTA
    const uint32_t* row_off;    // optional [G + 1]: first slab row of every CTA (weighted shares); nullptr: equal shares of S rows
    const uint32_t* unit_off;   // optional [G + 1]: CTA boundaries in units of (row, segment position), units_per_row per row
    uint32_t units_per_row;     // segments per row the unit table was built for (must be the kernel's nseg)
    uint4* frag;                // [2][G] flag-in-data slots: head-fragment partial sums handed to the owning CTA
    unsigned long long* trace;  // optional [G][4]: per CTA ns inside matvec_rows, ns waiting for round payloads, rows owned, SM id
};

size_t fused_smem_bytes(uint32_t S, uint32_t rblk, uint32_t restart);
uint32_t fused_pick_rblk(uint32_t S);
// polite: the 96-register build that leaves room for a background assembly block on every SM
cudaError_t launch_gmres_fused(const FusedParams& p, int grid, size_t smem, bool polite, cudaStream_t s);

}  // namespace bemb
