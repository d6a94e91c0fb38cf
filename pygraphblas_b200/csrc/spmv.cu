// spmv.cu -- GrB_mxv / GrB_vxm on sm_100a:  w<mask> = accum(w, op(A) (+).(x) u)
//
// Replaces the SuiteSparse call behind /root/reference/pygraphblas/matrix.py:2716
// (Matrix.mxv) and /root/reference/pygraphblas/vector.py:961 (Vector.vxm).
//
// Layout in HBM: A is CSR (32-bit row offsets shadow, 32-bit column ids, values of
// the matrix type), vectors are dense value arrays + one presence byte per position
// (no presence array at all when every position is present).
//
// This file: the host logic of both calls (operand casts, kernel choice, write-back) and the tile kernel.
// Kernel choice, in order (DESIGN.md section 3.1):
//   mask + LOR/LAND/ANY monoid  -> masked push (small frontier, spmv_pull.cu) or masked pull with early exit
//   nnz >= 4096                 -> run kernel (spmv_run*.cu): 256-entry runs per warp on a cached run plan,
//                                  compile-time semirings (+ shared-memory hot-column table), run-time
//                                  operator codes, dense or sparse u
//   otherwise                   -> tile kernel below: the nnz range is cut into tiles of SPMV_THREADS * items
//                                  entries, one CTA per tile, item-centric segmented reduction; rows that straddle
//                                  tiles leave head / tail partials that a fix-up kernel combines in a fixed order.
// Every path is nnz-split (R-MAT hub rows cannot serialise a warp) and deterministic for a given matrix.
//
// Algorithmic bytes per call (DESIGN.md): nnz*(4 + sizeof(a)) + (nrows+1)*4
//   + ncols*sizeof(u) + nrows*(sizeof(t) + 1).
#include "spmv_args.cuh"

// build with -DB200GRB_PHASE_TIMERS=1 and run with B200GRB_SPMV_DEBUG=1 to get per-phase cycle counts of the tile kernel
#ifndef B200GRB_PHASE_TIMERS
#define B200GRB_PHASE_TIMERS 0
#endif
static constexpr bool SPMV_PHASE_TIMERS = B200GRB_PHASE_TIMERS != 0;
static constexpr int SPMV_THREADS = 256;
static constexpr int SPMV_WARPS = SPMV_THREADS / 32;

struct SpmvArgs {
    const uint32_t *rowptr; const uint32_t *col; const void *aval;
    const uint32_t *tile_row; int64_t ntiles; int64_t nrows; int64_t nnz;
    const void *uval; const uint8_t *upres;
    void *tval; uint8_t *tpres;
    void *head_val; uint8_t *head_has; void *tail_val; uint8_t *tail_has; int32_t *tail_row;
    int add_op, mul_op;
    int flip;      // 0: z = mul(a, u) (mxv)   1: z = mul(u, a) (vxm)   (run-time-operator kernels only)
    int tile;      // entries per tile = SPMV_THREADS * items per thread
    unsigned long long *dbg;   // optional per-phase cycle counters (B200GRB_SPMV_DEBUG), nullptr in production
};

// ---- plan: tile_row[t] = row holding entry t*tile (tile_row[0] = 0, tile_row[ntiles] = nrows)
__global__ void spmv_plan_kernel(const uint32_t *rowptr, int64_t nrows, int64_t ntiles, int tile, uint32_t *tile_row) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t > ntiles) return;
    if (t == 0) { tile_row[0] = 0; return; }
    if (t == ntiles) { tile_row[t] = (uint32_t)nrows; return; }
    const uint32_t x = (uint32_t)(t * tile);
    int64_t lo = 0, hi = nrows;           // first r in [0, nrows] with rowptr[r] > x
    while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (rowptr[mid] > x) hi = mid; else lo = mid + 1; }
    tile_row[t] = (uint32_t)(lo - 1);
}

static GrB_Info spmv_plan(Csr &c, int tile, std::string *err) {
    if (c.tile_row && c.tile_size == tile) return GrB_SUCCESS;
    if (!c.rowptr32) return gb_fail(GrB_INVALID_VALUE, err, "mxv: matrices with >= 2^32 entries are not supported");
    dfree(c.tile_row); c.tile_row = nullptr;
    c.ntiles = ceil_div(c.nnz, tile); c.tile_size = tile;
    GB_TRY(dalloc(&c.tile_row, (size_t)c.ntiles + 1, err));
    const int64_t n = c.ntiles + 1;
    spmv_plan_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, G.stream>>>(c.rowptr32, c.nrows, c.ntiles, tile, c.tile_row); GB_LAUNCHED();
    CU_TRY(cudaGetLastError(), err);
    return GrB_SUCCESS;
}


// One tile of SPMV_THREADS * IT consecutive entries per CTA:
//
//   1. every thread streams its IT consecutive entries (128-bit loads), issues all its gathers of u
//      back to back and keeps the products in registers;
//   2. the rows of the tile are walked thread-per-row (coalesced rowptr reads): empty rows are
//      written out as "no entry", the others mark their first entry in shared memory;
//   3. item-centric segmented reduction: each thread folds its items between row marks (rows that
//      begin and end inside a thread are final), then a segmented suffix scan over the threads
//      (shuffles inside a warp, 8 aggregates across warps) completes the rows that span threads.
//      Work per thread is constant whatever the row lengths: hub rows and runs of short rows cost
//      the same;
//   4. what sticks out of the tile goes to the per-tile head / tail slots for the fix-up kernel.
//
// ADD/MUL >= 0: compile-time semiring (flip already folded into MUL by the host); -1: run-time codes.
// SPARSE: u has a presence array (entries with absent u(k) do not contribute).
// Everything after the column / value words of a tile are in registers: gather u, mark rows, fold,
// scan, write.  `sync` is the barrier of the 256 threads that share s_head / s_wv / s_wflag.
template <typename XT, typename ZT, int ADD, int MUL, bool SPARSE, int IT, typename Sync>
__device__ __forceinline__ void spmv_tile_finish(const SpmvArgs &p, const uint32_t tile, const int tid, const int tlen, const int nvalid,
                                                 uint32_t (&c)[IT], XT (&a)[IT], int32_t *s_head, ZT *s_wv, int *s_wflag, Sync &&sync) {
    constexpr int TILE = SPMV_THREADS * IT;
    constexpr bool NEED_A = MUL < 0 || mul_reads_x(MUL);
    constexpr bool NEED_U = MUL < 0 || mul_reads_y(MUL);
    const int add = ADD >= 0 ? ADD : p.add_op;
    const int mul = MUL >= 0 ? MUL : p.mul_op;
    const int lane = tid & 31, warp = tid >> 5;
    const int loc0 = tid * IT;
    const int64_t tstart = (int64_t)tile * TILE;
    const XT *uval = static_cast<const XT *>(p.uval);
    ZT *tval = static_cast<ZT *>(p.tval);

    long long t0 = 0, t1 = 0, t2 = 0, t3 = 0;
    if (SPMV_PHASE_TIMERS && p.dbg && tid == 0) t0 = clock64();
    const uint32_t r0 = p.tile_row[tile];
    const uint32_t r1 = (uint32_t)min((int64_t)p.tile_row[tile + 1], p.nrows - 1);
    uint32_t pre_rs = 0, pre_re = 0;                                      // row pointers of this thread's first row
    if (r0 + tid <= r1) { pre_rs = p.rowptr[r0 + tid]; pre_re = p.rowptr[r0 + tid + 1]; }
#pragma unroll
    for (int j = 0; j < IT; j += 4) *reinterpret_cast<int4 *>(&s_head[loc0 + j]) = make_int4(-1, -1, -1, -1);
    if (tid == 0) { p.tail_row[tile] = -1; p.head_has[tile] = 0; p.tail_has[tile] = 0; }
    uint8_t hs[SPARSE ? IT : 1]; XT uv[IT];
    if (SPARSE) {
#pragma unroll
        for (int j = 0; j < IT; ++j) hs[j] = __ldg(p.upres + c[j]);
    }
    if (NEED_U) {
#pragma unroll
        for (int j = 0; j < IT; ++j) {
            uv[j] = gload<XT>(uval + c[j]);
        }
    }
    sync();                                                               // head marks are clear
    if (SPMV_PHASE_TIMERS && p.dbg && tid == 0) t1 = clock64();

    // ---- (2) rows of the tile: empty ones are final, the others mark their first entry
    {
        const uint32_t ts32 = (uint32_t)tstart;                           // nnz < 2^32
        uint32_t rs = pre_rs, re = pre_re;
        for (uint32_t r = r0 + tid; r <= r1; r += SPMV_THREADS) {
            if (r != r0 + tid) { rs = p.rowptr[r]; re = p.rowptr[r + 1]; }
            if (rs == re) { p.tpres[r] = 0; tval[r] = (ZT)0; }
            else if (rs >= ts32 && rs - ts32 < (uint32_t)tlen) s_head[rs - ts32] = (int32_t)(r - r0);
        }
    }
    ZT prod[IT];
#pragma unroll
    for (int j = 0; j < IT; ++j) {
        const XT av = NEED_A ? a[j] : (XT)1;
        const XT uu = NEED_U ? uv[j] : (XT)1;
        if (MUL >= 0) prod[j] = MulApply<XT, ZT>::f(mul, av, uu);
        else prod[j] = p.flip ? MulApply<XT, ZT>::f(mul, uu, av) : MulApply<XT, ZT>::f(mul, av, uu);
    }
    sync();                                                               // head marks are complete
    if (SPMV_PHASE_TIMERS && p.dbg && tid == 0) t2 = clock64();

    // ---- (3a) fold this thread's items between row marks
    int32_t h[IT];
#pragma unroll
    for (int j = 0; j < IT; j += 4) {
        const int4 t4 = *reinterpret_cast<const int4 *>(&s_head[loc0 + j]);
        h[j] = t4.x; h[j + 1] = t4.y; h[j + 2] = t4.z; h[j + 3] = t4.w;
    }
    Part<ZT> acc{(ZT)0, 0}, lead{(ZT)0, 0};
    bool seen = false; int32_t cur = -1;
    if (!SPARSE && nvalid == IT) {
        // every item contributes: presence is structural, no per-item flags
#pragma unroll
        for (int j = 0; j < IT; ++j) {
            if (h[j] >= 0) {
                if (!seen) lead = acc;
                else { tval[r0 + cur] = acc.v; p.tpres[r0 + cur] = 1; }      // row began and ended in this thread
                seen = true; cur = h[j]; acc.v = prod[j]; acc.has = 1;
            } else if (j == 0) { acc.v = prod[0]; acc.has = 1; }
            else acc.v = MulApply<ZT, ZT>::f(add, acc.v, prod[j]);
        }
    } else {
#pragma unroll
        for (int j = 0; j < IT; ++j) {
            if (h[j] >= 0) {
                if (!seen) lead = acc;
                else { tval[r0 + cur] = acc.v; p.tpres[r0 + cur] = (uint8_t)acc.has; }
                seen = true; cur = h[j]; acc.has = 0;
            }
            const Part<ZT> it{prod[j], (j < nvalid && (!SPARSE || hs[SPARSE ? j : 0])) ? 1 : 0};
            acc = part_join<ZT>(add, acc, it);
        }
    }
    if (!seen) { lead = acc; acc.has = 0; }                               // no mark: everything continues an earlier row

    // ---- (3b) segmented suffix scan of the leads: X_t = lead_t (+) (stop_t ? nothing : X_{t+1}); stop = thread has a mark
    Part<ZT> x = lead; int stop = seen ? 1 : 0;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        Part<ZT> y; y.v = shfl_down_t<ZT>(x.v, d); y.has = __shfl_down_sync(0xffffffffu, x.has, d);
        const int ystop = __shfl_down_sync(0xffffffffu, stop, d);
        if (lane + d < 32) { if (!stop) x = part_join<ZT>(add, x, y); stop |= ystop; }
    }
    if (lane == 0) { s_wv[warp] = x.v; s_wflag[warp] = x.has | (stop << 1); }
    sync();
    if (SPMV_PHASE_TIMERS && p.dbg && tid == 0) t3 = clock64();
    Part<ZT> carry{(ZT)0, 0}; int carry_stop = 0;                         // what the following warps add to a row open at this warp's end
    for (int w = SPMV_WARPS - 1; w > warp; --w) {
        Part<ZT> y; y.v = s_wv[w]; const int f = s_wflag[w]; y.has = f & 1;
        if (f >> 1) { carry = y; carry_stop = 1; } else carry = part_join<ZT>(add, y, carry);
    }
    if (!stop) { x = part_join<ZT>(add, x, carry); stop |= carry_stop; }
    Part<ZT> nxt; nxt.v = shfl_down_t<ZT>(x.v, 1); nxt.has = __shfl_down_sync(0xffffffffu, x.has, 1);   // S_t = X_{t+1}
    int nxt_stop = __shfl_down_sync(0xffffffffu, stop, 1);
    if (lane == 31) { nxt = carry; nxt_stop = carry_stop; }

    // ---- (4) rows still open at the end of a thread, and what sticks out of the tile
    if (seen) {
        const Part<ZT> total = part_join<ZT>(add, acc, nxt);
        if (nxt_stop) { tval[r0 + cur] = total.v; p.tpres[r0 + cur] = (uint8_t)total.has; }
        else { static_cast<ZT *>(p.tail_val)[tile] = total.v; p.tail_has[tile] = (uint8_t)total.has; p.tail_row[tile] = (int32_t)(r0 + cur); }
    }
    if (tid == 0 && h[0] < 0) {                                           // the tile starts inside a row of an earlier tile
        static_cast<ZT *>(p.head_val)[tile] = x.v; p.head_has[tile] = (uint8_t)x.has;
    }
    if (SPMV_PHASE_TIMERS && p.dbg && tid == 0) {
        const long long t4 = clock64();
        atomicAdd(&p.dbg[0], (unsigned long long)(t1 - t0)); atomicAdd(&p.dbg[1], (unsigned long long)(t2 - t1));
        atomicAdd(&p.dbg[2], (unsigned long long)(t3 - t2)); atomicAdd(&p.dbg[3], (unsigned long long)(t4 - t3));
        atomicAdd(&p.dbg[4], 1ull);
    }
}

// General path: one CTA per tile, loads straight from global memory into registers.
template <typename XT, typename ZT, int ADD, int MUL, bool SPARSE, int IT>
__global__ void __launch_bounds__(SPMV_THREADS) spmv_tile_kernel(const SpmvArgs p) {
    constexpr int TILE = SPMV_THREADS * IT;
    constexpr bool NEED_A = MUL < 0 || mul_reads_x(MUL);
    __shared__ __align__(16) int32_t s_head[TILE];     // row (relative to the tile's first row) starting at this entry, or -1
    __shared__ ZT s_wv[SPMV_WARPS];
    __shared__ int s_wflag[SPMV_WARPS];
    const int tid = threadIdx.x;
    const uint32_t tile = blockIdx.x;
    const int64_t tstart = (int64_t)tile * TILE;
    const int tlen = (int)min((int64_t)TILE, p.nnz - tstart);            // valid entries in this tile
    const int loc0 = tid * IT;
    const int nvalid = min(max(tlen - loc0, 0), IT);                     // valid entries of this thread
    const uint32_t *colp = p.col + tstart + loc0;
    const XT *avalp = static_cast<const XT *>(p.aval) + tstart + loc0;
    uint32_t c[IT]; XT a[IT];
    if (nvalid == IT) {
#pragma unroll
        for (int g = 0; g < IT / 4; ++g) {
            load4<uint32_t>(colp + g * 4, &c[g * 4]);
            if (NEED_A) load4<XT>(avalp + g * 4, &a[g * 4]);
        }
    } else {
#pragma unroll
        for (int j = 0; j < IT; ++j) {
            c[j] = j < nvalid ? colp[j] : 0u;                            // 0 is always a valid column to gather
            if (NEED_A) a[j] = j < nvalid ? avalp[j] : (XT)1;
        }
    }
    spmv_tile_finish<XT, ZT, ADD, MUL, SPARSE, IT>(p, tile, tid, tlen, nvalid, c, a, s_head, s_wv, s_wflag, [] { __syncthreads(); });
}

// ---- fix-up: rows that straddle tiles = tail partial of the tile they start in
//      (+) head partials of the following tiles, combined by one warp in a fixed order
template <typename ZT, int ADD>
__global__ void __launch_bounds__(256) spmv_fixup_kernel(const SpmvArgs p) {
    const int add = ADD >= 0 ? ADD : p.add_op;
    const int lane = threadIdx.x & 31;
    const int64_t t = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (t >= p.ntiles) return;
    const int32_t r = p.tail_row[t];
    if (r < 0) return;
    const int64_t re = p.rowptr[r + 1];
    const int64_t last_tile = (re - 1) / p.tile;
    Part<ZT> acc{(ZT)0, 0};
    if (lane == 0 && p.tail_has[t]) { acc.v = static_cast<const ZT *>(p.tail_val)[t]; acc.has = 1; }
    for (int64_t tt = t + 1 + lane; tt <= last_tile; tt += 32) if (p.head_has[tt]) {
        const Part<ZT> y{static_cast<const ZT *>(p.head_val)[tt], 1};
        acc = part_join<ZT>(add, acc, y);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        Part<ZT> y; y.v = shfl_xor_t<ZT>(acc.v, o); y.has = __shfl_xor_sync(0xffffffffu, acc.has, o);
        acc = part_join<ZT>(add, acc, y);
    }
    if (lane == 0) { static_cast<ZT *>(p.tval)[r] = acc.v; p.tpres[r] = (uint8_t)(acc.has != 0); }
}

__global__ void clear_presence_kernel(uint8_t *p, int64_t n) {
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) p[k] = 0;
}

static int g_items_fast = 8, g_items_generic = 8;     // entries per thread (tunable: B200GRB_SPMV_ITEMS)

template <typename XT, typename ZT, int ADD, int MUL, bool SPARSE, int IT>
static void spmv_launch(const SpmvArgs &a) {
    spmv_tile_kernel<XT, ZT, ADD, MUL, SPARSE, IT><<<(unsigned)a.ntiles, SPMV_THREADS, 0, G.stream>>>(a); GB_LAUNCHED();
    spmv_fixup_kernel<ZT, ADD><<<(unsigned)ceil_div(a.ntiles * 32, 256), 256, 0, G.stream>>>(a); GB_LAUNCHED();
}

// compile-time specialised semirings (BASELINE.json north_star: PLUS_TIMES, LOR_LAND, MIN_PLUS,
// PLUS_SECOND; plus PLUS_PAIR / ANY_PAIR / PLUS_FIRST / MIN_FIRST / MIN_SECOND which the reference's
// demos use) for dense u; everything else runs the same kernel with run-time operator codes.
template <typename T> static bool spmv_fast(int add, int mul, int items, const SpmvArgs &a) {
#define GB_FAST(A, M) if (add == A && mul == M) { if (items == 16) spmv_launch<T, T, A, M, false, 16>(a); else if (items == 4) spmv_launch<T, T, A, M, false, 4>(a); else spmv_launch<T, T, A, M, false, 8>(a); return true; }
    GB_FAST(OP_PLUS, OP_TIMES) GB_FAST(OP_MIN, OP_PLUS) GB_FAST(OP_PLUS, OP_SECOND) GB_FAST(OP_PLUS, OP_FIRST)
    GB_FAST(OP_PLUS, OP_PAIR) GB_FAST(OP_MIN, OP_FIRST) GB_FAST(OP_MIN, OP_SECOND)
#undef GB_FAST
    return false;
}
static bool spmv_fast_bool(int add, int mul, int items, const SpmvArgs &a) {
#define GB_FAST(A, M) if (add == A && mul == M) { if (items == 16) spmv_launch<bool, bool, A, M, false, 16>(a); else spmv_launch<bool, bool, A, M, false, 8>(a); return true; }
    GB_FAST(OP_LOR, OP_LAND) GB_FAST(OP_ANY, OP_PAIR) GB_FAST(OP_LOR, OP_PAIR) GB_FAST(OP_LOR, OP_SECOND) GB_FAST(OP_LOR, OP_FIRST)
#undef GB_FAST
    return false;
}

// the tile size a call will use (so that the plan can be built first)
static bool spmv_is_fast(int xt, int zt, int add, int mul, bool sparse_u) {
    if (sparse_u || xt != zt) return false;
    const bool num = (add == OP_PLUS && (mul == OP_TIMES || mul == OP_SECOND || mul == OP_FIRST || mul == OP_PAIR)) ||
                     (add == OP_MIN && (mul == OP_PLUS || mul == OP_FIRST || mul == OP_SECOND));
    const bool boo = (add == OP_LOR && (mul == OP_LAND || mul == OP_PAIR || mul == OP_SECOND || mul == OP_FIRST)) || (add == OP_ANY && mul == OP_PAIR);
    switch (xt) {
        case TC_FP32: case TC_FP64: case TC_INT32: case TC_INT64: case TC_UINT32: case TC_UINT64: return num;
        case TC_BOOL: return boo;
        default: return false;
    }
}

static GrB_Info spmv_dispatch(int xt, int zt, int add, int mul, bool sparse_u, const SpmvArgs &a, std::string *err) {
    if (spmv_is_fast(xt, zt, add, mul, sparse_u)) {
        const int items = a.tile / SPMV_THREADS;
        switch (xt) {
            case TC_FP32:  if (spmv_fast<float>(add, mul, items, a)) return GrB_SUCCESS; break;
            case TC_FP64:  if (spmv_fast<double>(add, mul, items, a)) return GrB_SUCCESS; break;
            case TC_INT32: if (spmv_fast<int32_t>(add, mul, items, a)) return GrB_SUCCESS; break;
            case TC_INT64: if (spmv_fast<int64_t>(add, mul, items, a)) return GrB_SUCCESS; break;
            case TC_UINT32: if (spmv_fast<uint32_t>(add, mul, items, a)) return GrB_SUCCESS; break;
            case TC_UINT64: if (spmv_fast<uint64_t>(add, mul, items, a)) return GrB_SUCCESS; break;
            case TC_BOOL:  if (spmv_fast_bool(add, mul, items, a)) return GrB_SUCCESS; break;
            default: break;
        }
        return gb_fail(GrB_PANIC, err, "mxv: internal dispatch error");
    }
#define GB_GEN2(XT_, ZT_) do { if (sparse_u) spmv_launch<XT_, ZT_, -1, -1, true, 8>(a); else spmv_launch<XT_, ZT_, -1, -1, false, 8>(a); return GrB_SUCCESS; } while (0)
    if (xt == zt) {
        switch (xt) {
#define GB_GEN(TC, T) case TC: GB_GEN2(T, T);
            GB_GEN(TC_BOOL, bool) GB_GEN(TC_INT8, int8_t) GB_GEN(TC_INT16, int16_t) GB_GEN(TC_INT32, int32_t) GB_GEN(TC_INT64, int64_t)
            GB_GEN(TC_UINT8, uint8_t) GB_GEN(TC_UINT16, uint16_t) GB_GEN(TC_UINT32, uint32_t) GB_GEN(TC_UINT64, uint64_t)
            GB_GEN(TC_FP32, float) GB_GEN(TC_FP64, double)
#undef GB_GEN
        }
    } else if (zt == TC_BOOL) {
        switch (xt) {
#define GB_GEN(TC, T) case TC: GB_GEN2(T, bool);
            GB_GEN(TC_INT8, int8_t) GB_GEN(TC_INT16, int16_t) GB_GEN(TC_INT32, int32_t) GB_GEN(TC_INT64, int64_t)
            GB_GEN(TC_UINT8, uint8_t) GB_GEN(TC_UINT16, uint16_t) GB_GEN(TC_UINT32, uint32_t) GB_GEN(TC_UINT64, uint64_t)
            GB_GEN(TC_FP32, float) GB_GEN(TC_FP64, double)
#undef GB_GEN
        }
    }
#undef GB_GEN2
    return gb_fail(GrB_DOMAIN_MISMATCH, err, "mxv: unsupported semiring domains (x=%d, z=%d)", xt, zt);
}

static inline int grid_for(int64_t n, int threads = 256) {
    return (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div(n, threads), (int64_t)G.num_sms * 16));
}

static bool op_uses_x(int op) { return !(op == OP_SECOND || op == OP_PAIR); }
static bool op_uses_y(int op) { return !(op == OP_FIRST || op == OP_PAIR || op == OP_ANY); }

// w<mask> = accum(w, A' (+).(x) u) with `flip` selecting mul(u,a) (vxm) and `use_transpose`
// selecting the cached CSR of A' (so that the kernel always pulls along CSR rows).
static GrB_Info mxv_core(GrB_Vector w, const GrB_Vector mask, const GrB_BinaryOp accum, const GrB_Semiring s,
                         const GrB_Matrix A, const GrB_Vector u, const DescFlags &f, bool use_transpose, bool flip,
                         const char *fn) {
    std::string *err = &w->err;
    // ---- domain / dimension checks (host, synchronous)
    const GrB_BinaryOp mulop = s->mul; const GrB_BinaryOp addop = s->add->op;
    if (mulop->opcode == OP_USER || addop->opcode == OP_USER || (accum && accum->opcode == OP_USER))
        return gb_fail(GrB_INVALID_VALUE, err, "%s: user-defined operators are host function pointers and cannot run on the GPU (no CPU fallback)", fn);
    const uint64_t out_n = use_transpose ? A->ncols : A->nrows, in_n = use_transpose ? A->nrows : A->ncols;
    if (u->n != in_n || w->n != out_n || (mask && mask->n != out_n))
        return gb_fail(GrB_DIMENSION_MISMATCH, err, "%s: dimensions do not match (A is %llux%llu%s, u %llu, w %llu)", fn,
                       (unsigned long long)A->nrows, (unsigned long long)A->ncols, use_transpose ? " transposed" : "",
                       (unsigned long long)u->n, (unsigned long long)w->n);
    if (!G.have_device) return gb_fail(GrB_PANIC, err, "%s: no CUDA device: libb200grb computes only on the GPU (no CPU fallback)", fn);
    const int xt = mulop->xtype->code, zt = addop->ztype->code;
    const int add = addop->opcode, mul = mulop->opcode;
    if (!mask && f.mask_comp)      // w<!NULL>: nothing is let through, no product needed (vector_write clears w under REPLACE)
        return vector_write(w, nullptr, accum, f, nullptr, nullptr, zt, false, nullptr, true);

    // ---- operands in HBM
    if (use_transpose) GB_TRY(matrix_ensure_transpose(A)); else GB_TRY(matrix_ensure_device(A));
    Csr &c = use_transpose ? A->devT : A->dev;
    GB_TRY(vector_ensure_device(u));
    if (mask) GB_TRY(vector_ensure_device(mask));
    const bool need_final = mask != nullptr || accum != nullptr;
    const bool w_empty = w->host_valid && w->hi.empty() && w->pi.empty();   // nothing to merge with
    if (need_final && !w_empty) GB_TRY(vector_ensure_device(w));
    // the multiply sees (x = matrix entry, y = u entry) for mxv and the reverse for vxm; for the
    // operators that ignore one side the flip folds into the operator itself
    int kmul = mul; bool kflip = flip;
    if (flip && (mul == OP_FIRST || mul == OP_SECOND)) { kmul = mul == OP_FIRST ? OP_SECOND : OP_FIRST; kflip = false; }
    if (flip && (mul == OP_TIMES || mul == OP_PLUS || mul == OP_MIN || mul == OP_MAX || mul == OP_PAIR || mul == OP_LAND || mul == OP_LOR ||
                 mul == OP_LXOR || mul == OP_EQ || mul == OP_NE || mul == OP_ISEQ || mul == OP_ISNE)) kflip = false;     // commutative
    const bool need_a = kflip ? op_uses_y(kmul) : op_uses_x(kmul);
    const bool need_u = kflip ? op_uses_x(kmul) : op_uses_y(kmul);
    const bool sparse_u = u->dpres != nullptr;
    const bool fast_sr = !kflip && spmv_is_fast(xt, zt, add, kmul, false);      // a compile-time specialised semiring
    const bool fast = fast_sr && !sparse_u;
    const Tunables &tn = tunables();
    GbBurble burble(fn);
    g_items_fast = (tn.spmv_items == 16 || tn.spmv_items == 4) ? tn.spmv_items : 8;
    const int tile = SPMV_THREADS * (fast ? g_items_fast : g_items_generic);
    GB_TRY(spmv_plan(c, tile, err));

    void *a_cast = nullptr, *u_cast = nullptr;
    const void *aval = c.val, *uval = u->dval;
    if (need_a && A->type->code != xt) { GB_TRY(dev_cast_values(&a_cast, xt, c.val, A->type->code, c.nnz, err)); aval = a_cast; }
    if (need_u && u->type->code != xt) { GB_TRY(dev_cast_values(&u_cast, xt, u->dval, u->type->code, (int64_t)u->n, err)); uval = u_cast; }
    // run-time-operator kernels always read both operands: give them something readable of the right type
    if (!fast && !need_a && A->type->code != xt) { GB_TRY(dev_cast_values(&a_cast, xt, c.val, A->type->code, c.nnz, err)); aval = a_cast; }
    if (!fast && !need_u && u->type->code != xt) { GB_TRY(dev_cast_values(&u_cast, xt, u->dval, u->type->code, (int64_t)u->n, err)); uval = u_cast; }

    const int64_t n = (int64_t)out_n;
    const size_t zsz = (size_t)tc_size(zt);
    // T's buffers become w (no mask, no accumulator: w<-T).  When w already owns device buffers of the right shape and is not an
    // operand of this call, T is formed in place -- the iterated call `A.mxv(u, out=w)` then allocates nothing.
    void *tval = nullptr; uint8_t *tpres = nullptr;
    const bool w_reusable = !need_final && w != u && w->dev_valid && w->dval && w->dpres && w->type->code == zt && !w->borrowed &&
                            a_cast != w->dval && u_cast != w->dval;
    const bool in_place = w_reusable && (tn.mxv_inplace == 2 || (tn.mxv_inplace == 1 && !w->h2d_pending && !w->d2h_pending));
    if (in_place && tn.mxv_inplace == 2) {      // whatever the flags say: the kernels below start after w's last overlapped copies
        if (w->ev_h2d) { cudaStreamWaitEvent(G.stream, w->ev_h2d, 0); cudaStreamWaitEvent(G.stream, w->ev_d2h, 0); }
        w->h2d_pending = false; w->d2h_pending = false;
    }
    if (in_place) { tval = w->dval; tpres = w->dpres; }
    else {
        GB_TRY(dmalloc(&tval, (size_t)n * zsz + 16, err));
        GB_TRY(dmalloc((void **)&tpres, (size_t)n + 16, err));
    }

    // mask + saturating monoid (BFS-shaped): skip masked-out rows, stop rows at the first hit
    const bool use_pull = mask != nullptr && (add == OP_LOR || add == OP_LAND || add == OP_ANY) && c.nnz > 0 && !tn.no_pull;
    if (use_pull) {
        // the run-time-operator kernel reads both operands: make sure both are of the operand type
        if (aval == c.val && A->type->code != xt) { GB_TRY(dev_cast_values(&a_cast, xt, c.val, A->type->code, c.nnz, err)); aval = a_cast; }
        if (uval == u->dval && u->type->code != xt) { GB_TRY(dev_cast_values(&u_cast, xt, u->dval, u->type->code, (int64_t)u->n, err)); uval = u_cast; }
        // few frontier edges: push along the rows of the other orientation (already in HBM) instead of pulling every row
        bool pushed = false;
        const Csr &o = use_transpose ? A->dev : A->devT;
        if (sparse_u && o.valid && o.rowptr32 && o.nnz == c.nnz && A->type->code == xt && !tn.no_push) {
            PushArgs ps{};
            ps.rowptr = o.rowptr32; ps.col = o.col; ps.aval = o.val; ps.nin = o.nrows; ps.uval = uval; ps.upres = u->dpres;
            ps.mval = mask->dval; ps.mpres = mask->dpres; ps.mtc = mask->type->code; ps.mask_comp = f.mask_comp; ps.mask_struct = f.mask_struct;
            ps.tval = tval; ps.tpres = tpres; ps.nout = n; ps.add_op = add; ps.mul_op = kmul; ps.flip = kflip;
            GB_TRY(spmv_masked_push_try(xt, zt, ps, c.nnz, &pushed, err));
        }
        PullArgs pa{};
        pa.rowptr = c.rowptr32; pa.col = c.col; pa.aval = aval; pa.nrows = c.nrows; pa.uval = uval; pa.upres = u->dpres;
        pa.mval = mask->dval; pa.mpres = mask->dpres; pa.mtc = mask->type->code; pa.mask_comp = f.mask_comp; pa.mask_struct = f.mask_struct;
        pa.tval = tval; pa.tpres = tpres; pa.add_op = add; pa.mul_op = kmul; pa.flip = kflip;
        // rows longer than PULL_LONG: at most nnz / PULL_LONG of them
        pa.long_cap = c.nnz / (int64_t)PULL_LONG + 1; pa.has_long = c.nnz > (int64_t)PULL_LONG;
        GB_TRY(dalloc(&pa.long_rows, (size_t)pa.long_cap + 1, err));
        GB_TRY(dalloc(&pa.long_count, 4, err));
        CU_TRY(cudaMemsetAsync(pa.long_count, 0, sizeof(int), G.stream), err);
        GrB_Info r = pushed ? GrB_SUCCESS : spmv_masked_pull_dispatch(xt, zt, pa, err);
        dfree(pa.long_rows); dfree(pa.long_count);
        if (r != GrB_SUCCESS) { if (!in_place) { dfree(tval); dfree(tpres); } dfree(a_cast); dfree(u_cast); return r; }
    }
    // dense u + specialised semiring: warp-independent run kernel on the cached run plan
    const bool run_ok = !use_pull && (fast_sr || xt == zt || zt == TC_BOOL);     // specialised or run-time operators; dense or sparse u
    bool use_run = run_ok && c.nnz >= 4096;
    if (tn.spmv_run >= 0) use_run = run_ok && c.nnz > 0 && tn.spmv_run != 0;
    const char *kernel_name = "pull";
    if (use_pull) {
        // done above
    } else if (use_run) {
        GB_TRY(spmv_run_plan(c, err));
        RunArgs ra{};
        ra.col = c.col; ra.aval = aval; ra.uval = uval; ra.headw = c.run_headw; ra.lane_rank = c.run_lane; ra.run_base = c.run_base;
        ra.nzrow = c.nzrow; ra.rowptr = c.rowptr32; ra.nruns = c.nruns; ra.nnz = c.nnz; ra.tval = tval;
        ra.fix = c.run_fix; ra.fix_long = c.run_fix_long; ra.fix_short = c.run_fix_short;
        ra.add_op = add; ra.mul_op = kmul; ra.flip = kflip;
        ra.head_val = c.ws_head; ra.tail_val = c.ws_tail;            // scratch kept with the plan (the library serialises calls)
        if (sparse_u) { ra.upres = u->dpres; ra.tpres = tpres; ra.head_has = c.ws_head_has; ra.tail_has = c.ws_tail_has; }
        // hot-column table: on by default for large matrices whose gathers are concentrated (R-MAT-like);
        // B200GRB_SPMV_HOT=0 disables it, =<KB> caps the table size (and forces the kernel whatever the coverage)
        int hot_kb = tn.spmv_hot_kb >= 0 ? tn.spmv_hot_kb : 128;     // stage + table stay inside the 196 KB carve-out: the 228 KB one leaves no L1 and is 40 % slower
        if (fast && need_u && hot_kb > 0 && c.nnz >= ((int64_t)1 << 20) && c.ncols >= (1 << 16)) {
            GB_TRY(spmv_hot_plan(c, err));
            if (!c.hcol || (tn.spmv_hot_kb < 0 && c.hot_cover < 0.25)) hot_kb = 0;
        } else hot_kb = 0;
        Hot2Args hot{};
        if (hot_kb > 0) {
            // u at the hot columns; the kernel writes T's presence and the values of the empty rows itself
            spmv_hot2_prep(c, uval, tc_size(xt));
            ra.col = c.hcol; hot.u_hot = c.ws_uhot; hot.henc = c.henc; hot.tab_n = 0;
            hot.pres_tmpl = c.pres_tmpl; hot.tpres = tpres; hot.nrows = n;
            kernel_name = "run+hot-table (TMA-staged)";
        } else {
            CU_TRY(cudaMemsetAsync(tval, 0, (size_t)n * zsz, G.stream), err);
            if (sparse_u) CU_TRY(cudaMemsetAsync(tpres, 0, (size_t)n, G.stream), err);     // presence follows u: written row by row
            else CU_TRY(cudaMemcpyAsync(tpres, c.pres_tmpl, (size_t)n, cudaMemcpyDeviceToDevice, G.stream), err);
            kernel_name = sparse_u ? "run (sparse u)" : "run";
        }
        const bool ok = fast_sr ? spmv_run_dispatch(xt, add, kmul, ra, hot_kb > 0 ? &hot : nullptr, (size_t)hot_kb << 10) : spmv_run_generic(xt, zt, ra);
        if (!ok) { if (!in_place) { dfree(tval); dfree(tpres); } dfree(a_cast); dfree(u_cast); return gb_fail(GrB_PANIC, err, "mxv: internal dispatch error"); }
    } else if (c.nnz == 0) {
        clear_presence_kernel<<<grid_for(n), 256, 0, G.stream>>>(tpres, n); GB_LAUNCHED();
        kernel_name = "empty";
    } else {
        kernel_name = "tile";
        SpmvArgs a{};
        a.rowptr = c.rowptr32; a.col = c.col; a.aval = aval; a.tile_row = c.tile_row; a.ntiles = c.ntiles;
        a.nrows = c.nrows; a.nnz = c.nnz; a.uval = uval; a.upres = u->dpres; a.tval = tval; a.tpres = tpres;
        a.add_op = add; a.mul_op = kmul; a.flip = kflip; a.tile = tile;
        GB_TRY(dmalloc(&a.head_val, (size_t)c.ntiles * zsz + 16, err));
        GB_TRY(dmalloc(&a.tail_val, (size_t)c.ntiles * zsz + 16, err));
        GB_TRY(dmalloc((void **)&a.head_has, (size_t)c.ntiles + 16, err));
        GB_TRY(dmalloc((void **)&a.tail_has, (size_t)c.ntiles + 16, err));
        GB_TRY(dalloc(&a.tail_row, (size_t)c.ntiles, err));
        if (SPMV_PHASE_TIMERS && tn.spmv_debug) { GB_TRY(dalloc(&a.dbg, 8, err)); CU_TRY(cudaMemsetAsync(a.dbg, 0, 64, G.stream), err); }
        GrB_Info r = spmv_dispatch(xt, zt, add, kmul, sparse_u, a, err);
        if (a.dbg) {
            unsigned long long h[5];
            cudaMemcpyAsync(h, a.dbg, 40, cudaMemcpyDeviceToHost, G.stream); cudaStreamSynchronize(G.stream);
            if (h[4]) fprintf(stderr, "[spmv phases, avg cycles per tile] load+issue %.0f | rows+gather %.0f | fold+scan %.0f | carry+store %.0f | tiles %llu\n",
                              (double)h[0] / h[4], (double)h[1] / h[4], (double)h[2] / h[4], (double)h[3] / h[4], h[4]);
            dfree(a.dbg);
        }
        dfree(a.head_val); dfree(a.tail_val); dfree(a.head_has); dfree(a.tail_has); dfree(a.tail_row);
        if (r != GrB_SUCCESS) { if (!in_place) { dfree(tval); dfree(tpres); } dfree(a_cast); dfree(u_cast); return r; }
    }
    if (burble.on) burble.note(kernel_name, (double)c.nnz * (4.0 + (need_a ? tc_size(xt) : 0)) + (double)(c.nrows + 1) * 4 + (double)c.ncols * (need_u ? tc_size(xt) : 0) + (double)n * (zsz + 1));
    dfree(a_cast); dfree(u_cast);
    vector_mark_used(u); if (mask) vector_mark_used(mask);          // an overlapped import into u may start as soon as these kernels are done

    if (in_place) {                    // T was formed in w's own buffers: only the bookkeeping changes
        w->dev_nvals = -1; w->host_valid = false; w->hi.clear(); w->hx.clear(); w->pi.clear(); w->px.clear();
        CU_TRY(cudaGetLastError(), err);
        return GrB_SUCCESS;
    }
    // ---- w<mask> = accum(w, t)   (vector_ops.cu)
    return vector_write(w, mask, accum, f, tval, tpres, zt, /*t_scalar=*/false, /*region=*/nullptr, /*own_t=*/true);
}

static GrB_Info mxv_check(GrB_Vector w, const GrB_Vector mask, const GrB_Semiring s, const GrB_Matrix A, const GrB_Vector u, const char *fn) {
    if (!w || !s || !A || !u) return gb_fail(GrB_NULL_POINTER, nullptr, "%s: NULL argument", fn);
    if (!gb_valid_vector(w) || !gb_valid_vector(u) || !gb_valid_matrix(A) || (mask && !gb_valid_vector(mask)) || s->magic != GB_MAGIC)
        return gb_fail(GrB_UNINITIALIZED_OBJECT, nullptr, "%s: invalid object", fn);
    return GrB_SUCCESS;
}

extern "C" GrB_Info GrB_mxv(GrB_Vector w, const GrB_Vector mask, const GrB_BinaryOp accum, const GrB_Semiring semiring,
                            const GrB_Matrix A, const GrB_Vector u, const GrB_Descriptor desc) {
    GB_LOCK; GB_CHECK_INIT;
    GB_TRY(mxv_check(w, mask, semiring, A, u, "GrB_mxv"));
    if (gb_hyper_matrix(A) || gb_hyper_vector(u) || gb_hyper_vector(w)) return hyper_mxv(w, mask, accum, semiring, A, u, desc, false);
    const DescFlags f = desc_flags(desc);
    return mxv_core(w, mask, accum, semiring, A, u, f, /*use_transpose=*/f.tran0, /*flip=*/false, "GrB_mxv");
}

extern "C" GrB_Info GrB_vxm(GrB_Vector w, const GrB_Vector mask, const GrB_BinaryOp accum, const GrB_Semiring semiring,
                            const GrB_Vector u, const GrB_Matrix A, const GrB_Descriptor desc) {
    GB_LOCK; GB_CHECK_INIT;
    GB_TRY(mxv_check(w, mask, semiring, A, u, "GrB_vxm"));
    if (gb_hyper_matrix(A) || gb_hyper_vector(u) || gb_hyper_vector(w)) return hyper_mxv(w, mask, accum, semiring, A, u, desc, true);
    const DescFlags f = desc_flags(desc);
    // w' = u'A  <=>  w = A'u: pull along the rows of A' (INP1 = TRAN cancels the transpose)
    return mxv_core(w, mask, accum, semiring, A, u, f, /*use_transpose=*/!f.tran1, /*flip=*/true, "GrB_vxm");
}

