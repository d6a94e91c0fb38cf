// Argument blocks of the run and pull kernels (host side fills them in spmv.cu).
#pragma once
#include "spmv_common.cuh"

static constexpr int RUN = 256;
// fix-up work item of the run plan: a run that contains a row start, the row still open at its end (its last row start)
// and the last run that row reaches; 16 bytes, so one load gives a thread all three
struct __align__(16) RunFix { uint32_t run, row, last, pad; };
constexpr uint32_t FIX_LANES = 8;             // rows reaching more than this many runs further are folded by 8 lanes, the others by one thread
struct RunArgs {
    const uint32_t *col; const void *aval; const void *uval;
    const uint32_t *headw; const uint16_t *lane_rank; const uint32_t *run_base; const uint32_t *nzrow; const uint32_t *rowptr;
    const RunFix *fix; int64_t fix_long, fix_short;          // fix-up list: the fix_long items that reach > FIX_LANES runs first
    int64_t nruns; int64_t nnz;
    void *tval;
    void *head_val; void *tail_val;                            // per run: partial of the row it starts inside / of the row open at its end
    int add_op, mul_op, flip;                                  // run-time operator codes (kernels instantiated with ADD = MUL = -1)
    const uint8_t *upres;                                      // SPARSE kernels: presence bytes of u ...
    uint8_t *tpres; uint8_t *head_has; uint8_t *tail_has;      // ... and of everything they produce
};

// hot-table run kernel (spmv_run.cuh)
struct Hot2Args {
    const void *u_hot;        // [henc] u at the hottest columns (prep kernel)
    uint32_t henc;            // ids below this are hot ranks
    uint32_t tab_n;           // entries of u_hot kept in shared memory (<= henc)
    const uint8_t *pres_tmpl; // [nrows] the plan's presence template: T's presence bytes (u is dense) ...
    uint8_t *tpres;           // ... copied here by the kernel, which also writes 0 to T's values of the empty rows
    int64_t nrows;
};

// ------------------------------------------------------------------ masked pull with early exit (BFS-shaped calls)
// w<mask> = A (+).(x) u for monoids with a terminal value (LOR, LAND, ANY): one warp per row, rows the mask
// rules out are skipped entirely (their entries are never read), and a row stops as soon as its monoid
// saturates -- the BFS step `A.mxv(q, mask=visited, desc=RC, semiring=LOR_LAND)` of
// /root/reference/tests/test_descriptor.py:13-30 touches only the unvisited rows and, for each, only the
// entries up to the first frontier hit.  Output: T restricted to the rows the mask lets through.
struct PullArgs {
    const uint32_t *rowptr; const uint32_t *col; const void *aval; int64_t nrows;
    const void *uval; const uint8_t *upres;
    const void *mval; const uint8_t *mpres; int mtc; int mask_comp, mask_struct;
    void *tval; uint8_t *tpres;
    int add_op, mul_op, flip;
    int has_long; int64_t long_cap;
    uint32_t *long_rows; int *long_count;                      // work list of the rows left to the CTA-per-row kernel
};
constexpr uint32_t PULL_LONG = 4096;          // rows longer than this go to the CTA-per-row kernel

// ------------------------------------------------------------------ masked push for small frontiers (same three monoids)
// The transpose of the pull: for every present u(k), walk row k of the OTHER orientation's CSR and store into
// T(j) for the columns j the mask lets through.  LOR / LAND / ANY need no atomics: T(j) starts at the monoid's
// identity-like value and every store is idempotent (LOR: "a product was true", LAND: "a product was false",
// ANY: any product).  Work is proportional to the frontier's out-edges; used when those are < nnz / 16.
struct PushArgs {
    const uint32_t *rowptr; const uint32_t *col; const void *aval; int64_t nin;    // CSR whose rows are the input positions k
    const void *uval; const uint8_t *upres;
    const void *mval; const uint8_t *mpres; int mtc; int mask_comp, mask_struct;
    void *tval; uint8_t *tpres; int64_t nout;
    int add_op, mul_op, flip;
    uint32_t *list; int64_t *chunk_scan; unsigned long long *counters;           // frontier list, chunk offsets, {count, edges}
};
GrB_Info spmv_masked_push_try(int xt, int zt, PushArgs &a, int64_t nnz_total, bool *done, std::string *err);
