// The run kernels and their launcher, as templates; instantiated by spmv_run.cu (FP32 / FP64 semirings),
// spmv_run_int.cu (integer / BOOL semirings) and spmv_run_generic.cu (run-time operator codes).
#pragma once
#include "spmv_args.cuh"

// ==================================================================================================
// Dense-u kernel for the specialised semirings: warp-independent RUNS.
//
// The entries are cut into runs of 256 (one warp, 8 consecutive entries per lane).  A cached plan gives
// every lane what the tile kernel has to discover with shared-memory marks, a row pass and barriers:
//   run_headw   one bit per entry: "this entry starts a row"
//   run_base    number of row starts before the run;  run_lane: row starts inside the run before the lane
//   nzrow       ids of the non-empty rows (row start rank -> row id);  pres_tmpl: the output's presence
// so a warp needs no shared memory and no barrier: stream 8 entries, gather, fold between the row-start
// bits (rows inside a lane are final), one segmented suffix scan over the 32 lanes, and the two partial
// rows sticking out of the run go to per-run slots that spmv_run_fixup_kernel combines in a fixed order
// (deterministic).  ~3.5x fewer instructions per entry than the tile kernel.
// HOT: persistent CTAs, hot_n most referenced entries of the (relabelled) u in a shared-memory table.


// A lane's share of a run in flight: its 8 matrix values, the 8 values of u it gathered (presence bytes for a sparse u),
// its row-start bits and the rank of its first row start.
template <typename XT> struct RunLane { XT a[8]; XT uv[8]; uint8_t up[8]; uint32_t hb; uint32_t rank; int nvalid; };

// Part 1: everything that ISSUES loads -- the plan words of the lane and the gathers of u.
// `gather(c)` returns u's value for an (encoded) column id of a dense u; SPARSE kernels read p.uval / p.upres directly.
template <typename XT, int MUL_C, bool SPARSE, typename Gather>
__device__ __forceinline__ void spmv_run_gather(const RunArgs &p, const int64_t run, const int lane, const int nvalid,
                                                const uint32_t (&c)[8], RunLane<XT> &L, Gather &&gather) {
    constexpr bool NEED_U = MUL_C < 0 || mul_reads_y(MUL_C);
    const int64_t q = run * RUN + lane * 8;
    const XT *uval = static_cast<const XT *>(p.uval);
    const uint32_t hw = nvalid > 0 ? __ldg(p.headw + (q >> 5)) : 0u;
    L.hb = (hw >> ((lane & 3) * 8)) & 0xffu;                               // this lane's 8 row-start bits
    L.rank = __ldg(p.run_base + run) + __ldg(p.lane_rank + run * 32 + lane);   // row starts before this lane's first entry
    L.nvalid = nvalid;
    if (SPARSE) {
        // u has holes: a product exists only where u(col) does; the values are fetched only for those
#pragma unroll
        for (int j = 0; j < 8; ++j) L.up[j] = j < nvalid ? __ldg(p.upres + c[j]) : (uint8_t)0;
#pragma unroll
        for (int j = 0; j < 8; ++j) L.uv[j] = (NEED_U && L.up[j]) ? gload<XT>(uval + c[j]) : (XT)0;
    } else if (NEED_U) {
#pragma unroll
        for (int j = 0; j < 8; ++j) L.uv[j] = gather(c[j]);
    }
}

// Part 2: multiply, fold between the row-start bits, segmented scan over the lanes, stores.
template <typename XT, typename ZT, int ADD_C, int MUL_C, bool SPARSE>
__device__ __forceinline__ void spmv_run_fold(const RunArgs &p, const int64_t run, const int lane, const RunLane<XT> &L) {
    // ADD_C / MUL_C >= 0: compile-time semiring; -1: run-time operator codes (both operands are read)
    constexpr bool NEED_A = MUL_C < 0 || mul_reads_x(MUL_C);
    constexpr bool NEED_U = MUL_C < 0 || mul_reads_y(MUL_C);
    const int ADD = ADD_C >= 0 ? ADD_C : p.add_op;
    const int MUL = MUL_C >= 0 ? MUL_C : p.mul_op;
    ZT *tval = static_cast<ZT *>(p.tval);
    const int nvalid = L.nvalid;
    const uint32_t hb = L.hb; uint32_t rank = L.rank;
    const uint8_t (&up)[8] = L.up;
    ZT prod[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const XT av = NEED_A ? L.a[j] : (XT)1, uu = NEED_U ? L.uv[j] : (XT)1;
        prod[j] = (MUL_C < 0 && p.flip) ? MulApply<XT, ZT>::f(MUL, uu, av) : MulApply<XT, ZT>::f(MUL, av, uu);
    }

    // ---- fold between row starts
    Part<ZT> acc{(ZT)0, 0}, lead{(ZT)0, 0};
    bool seen = false; uint32_t cur = 0;
    if (nvalid == 8 && !SPARSE) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if ((hb >> j) & 1u) {
                if (!seen) lead = acc;
                else tval[__ldg(p.nzrow + cur)] = acc.v;                    // row began and ended inside this lane
                seen = true; cur = rank++; acc.v = prod[j]; acc.has = 1;
            } else if (j == 0) { acc.v = prod[0]; acc.has = 1; }
            else acc.v = MulApply<ZT, ZT>::f(ADD, acc.v, prod[j]);
        }
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (j < nvalid) {
                if ((hb >> j) & 1u) {
                    if (!seen) lead = acc;
                    else { const uint32_t row = __ldg(p.nzrow + cur); tval[row] = acc.v; if (SPARSE) p.tpres[row] = (uint8_t)acc.has; }
                    seen = true; cur = rank++; acc.has = 0;
                }
                const Part<ZT> it{prod[j], SPARSE ? (int)up[j] : 1};
                acc = part_join<ZT>(ADD, acc, it);
            }
        }
    }
    if (!seen) { lead = acc; acc.has = 0; }

    // ---- segmented suffix scan of the leads over the 32 lanes
    Part<ZT> x = lead; int stop = seen ? 1 : 0;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        Part<ZT> y; y.v = shfl_down_t<ZT>(x.v, d);
        const int yf = __shfl_down_sync(0xffffffffu, x.has | (stop << 1), d);
        y.has = yf & 1;
        if (lane + d < 32) { if (!stop) x = part_join<ZT>(ADD, x, y); stop |= yf >> 1; }
    }
    Part<ZT> nxt; nxt.v = shfl_down_t<ZT>(x.v, 1);
    const int nf = __shfl_down_sync(0xffffffffu, x.has | (stop << 1), 1);
    nxt.has = nf & 1; int nxt_stop = nf >> 1;
    if (lane == 31) { nxt.has = 0; nxt_stop = 0; }

    // the lane holding the last row start of the run owns the row that is still open at the run's end
    // (which row that is, and where it ends, is structural: the plan's fix-up list)
    if (seen) {
        const Part<ZT> total = part_join<ZT>(ADD, acc, nxt);
        if (nxt_stop) { const uint32_t row = __ldg(p.nzrow + cur); tval[row] = total.v; if (SPARSE) p.tpres[row] = (uint8_t)total.has; }
        else { static_cast<ZT *>(p.tail_val)[run] = total.v; if (SPARSE) p.tail_has[run] = (uint8_t)total.has; }
    }
    if (lane == 0 && !(hb & 1u) && nvalid > 0) {                                            // the run starts inside a row of an earlier run
        static_cast<ZT *>(p.head_val)[run] = x.v; if (SPARSE) p.head_has[run] = (uint8_t)x.has;
    }
}

// ---- plain run kernel: 8 warps per CTA, each warp streams its run straight from global memory into registers
template <typename XT, typename ZT, int MUL_C>
__device__ __forceinline__ int spmv_run_load_global(const RunArgs &p, const int64_t run, const int lane, uint32_t (&c)[8], XT (&a)[8]) {
    constexpr bool NEED_A = MUL_C < 0 || mul_reads_x(MUL_C);
    const int64_t q = run * RUN + lane * 8;
    const int nvalid = (int)min((int64_t)8, max((int64_t)0, p.nnz - q));
    if (nvalid == 8) {
        load4<uint32_t>(p.col + q, &c[0]); load4<uint32_t>(p.col + q + 4, &c[4]);
        if (NEED_A) { load4<XT>(static_cast<const XT *>(p.aval) + q, &a[0]); load4<XT>(static_cast<const XT *>(p.aval) + q + 4, &a[4]); }
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            c[j] = j < nvalid ? p.col[q + j] : 0u;
            if (NEED_A) a[j] = j < nvalid ? static_cast<const XT *>(p.aval)[q + j] : (XT)1;
        }
    }
    return nvalid;
}

template <typename XT, typename ZT, int ADD, int MUL, bool SPARSE>
__global__ void __launch_bounds__(256) spmv_run_kernel(const RunArgs p) {
    const int64_t run = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (run >= p.nruns) return;
    const int lane = threadIdx.x & 31;
    uint32_t c[8]; RunLane<XT> L;
    const int nvalid = spmv_run_load_global<XT, ZT, MUL>(p, run, lane, c, L.a);
    const XT *uval = static_cast<const XT *>(p.uval);
    spmv_run_gather<XT, MUL, SPARSE>(p, run, lane, nvalid, c, L, [uval](uint32_t col) { return gload<XT>(uval + col); });
    spmv_run_fold<XT, ZT, ADD, MUL, SPARSE>(p, run, lane, L);
}

// ==================================================================================================
// Hot-table run kernel (dense u, specialised semirings, large skewed matrices) -- the benchmarked kernel.
//
// One persistent 1024-thread CTA per SM.  Shared memory holds
//   * the HOT TABLE: u at the tab_n most referenced columns (a scattered 4-byte gather costs one L1 wavefront
//     per lane; a shared-memory lookup a few bank-conflict cycles per warp), filled once per CTA by bulk TMA
//     copies (cp.async.bulk -> SASS UBLKCP) from the gathered copy u_hot that the prep kernel writes;
//   * one STAGE per warp: the column ids and values of the warp's NEXT run, brought in by two bulk TMA copies
//     issued by lane 0 and completed on the warp's own mbarrier, so the DRAM stream of run r+1 is in flight
//     while the warp gathers and folds run r (registers are the second buffer: a run is copied out of the
//     stage before the next copy is issued).  A warp is its own producer and consumer: no CTA barrier after
//     the table is in.
// Column ids are ENCODED by the cached plan: id < henc -> rank among the hottest columns (table if < tab_n,
// else u_hot in L2); id >= henc -> original column + henc, gathered from u itself.  u needs no permutation.

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile("{\n\t.reg .pred p;\n\tWAIT_%=:\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
                 "@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

// Programmatic dependent launch: a kernel launched with launch_pdl may start while the kernel before it on the stream is
// still running; pdl_wait() returns once that kernel has completed and its writes are visible (a no-op without PDL), and
// pdl_trigger() lets the next one be launched before this one ends.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
template <typename... KA, typename... A> static inline void launch_pdl(void (*kernel)(KA...), unsigned grid, unsigned block, size_t smem, A &&...args) {
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = smem; cfg.stream = G.stream; cfg.attrs = attr; cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, kernel, std::forward<A>(args)...);
}

template <typename XT> __host__ __device__ constexpr int hot2_stage_bytes(bool need_a) { return RUN * 4 + (need_a ? RUN * (int)sizeof(XT) : 0); }
constexpr int HOT2_WARPS = 32;

template <typename XT, typename ZT, int ADD, int MUL, bool PIPE>
__global__ void __launch_bounds__(HOT2_WARPS * 32, 1) spmv_run_hot2_kernel(const RunArgs p, const Hot2Args h) {
    constexpr bool NEED_A = mul_reads_x(MUL);
    constexpr int STAGE = hot2_stage_bytes<XT>(NEED_A);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // layout: [warp stages][mbarriers][hot table]
    unsigned char *s_stage = smem_raw;
    uint64_t *s_bar = reinterpret_cast<uint64_t *>(smem_raw + HOT2_WARPS * STAGE);        // [HOT2_WARPS] per warp + [1] table
    XT *s_hot = reinterpret_cast<XT *>(smem_raw + HOT2_WARPS * STAGE + (HOT2_WARPS + 1) * 8 + 8);   // 16-byte aligned
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint64_t *bar = s_bar + warp;
    unsigned char *stage = s_stage + warp * STAGE;
    const int64_t stride = (int64_t)gridDim.x * HOT2_WARPS;
    int64_t run = (int64_t)blockIdx.x * HOT2_WARPS + warp;

    auto issue = [&](int64_t r) {             // lane 0: the bulk copies of run r into this warp's stage
        const int64_t q = r * RUN;
        const int64_t left = p.nnz - q;
        const uint32_t cnt = (uint32_t)(left < RUN ? left : RUN);
        const uint32_t cb = (cnt * 4u + 15u) & ~15u;                                      // arrays are padded by >= 16 bytes
        const uint32_t ab = NEED_A ? ((cnt * (uint32_t)sizeof(XT) + 15u) & ~15u) : 0u;
        mbar_expect_tx(bar, cb + ab);
        tma_bulk_g2s(stage, p.col + q, cb, bar);
        if (NEED_A) tma_bulk_g2s(stage + RUN * 4, static_cast<const XT *>(p.aval) + q, ab, bar);
    };

    if (lane == 0) mbar_init(bar, 1);
    if (threadIdx.x == 0) mbar_init(s_bar + HOT2_WARPS, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();
    if (threadIdx.x == 0 && h.tab_n) {        // the table: bulk copies of <= 16 KB of u_hot, once the prep kernel has written it
        pdl_wait();
        const uint32_t total = h.tab_n * (uint32_t)sizeof(XT);
        mbar_expect_tx(s_bar + HOT2_WARPS, total);
        for (uint32_t off = 0; off < total; off += 16384u)
            tma_bulk_g2s(reinterpret_cast<unsigned char *>(s_hot) + off, static_cast<const unsigned char *>(h.u_hot) + off,
                         min(16384u, total - off), s_bar + HOT2_WARPS);
    }
    if (lane == 0 && run < p.nruns) issue(run);

    // While the table and the first run are in flight: this warp's fixed slice of T's rows gets its presence byte from the
    // plan's template and, where the row is empty, the value 0.  The non-empty rows are written by spmv_run_fold and the
    // fix-up only, so these stores never meet theirs and need no ordering.  The 16-byte padding of both arrays is covered
    // too (presence: template bytes; values: 0), as a 16-byte-granular clear and copy would.
    {
        const int64_t rows_p = (h.nrows + 15) & ~(int64_t)15;
        const int64_t rows_v = ((h.nrows * (int64_t)sizeof(ZT) + 15) & ~(int64_t)15) / (int64_t)sizeof(ZT);
        const int64_t rows = rows_p > rows_v ? rows_p : rows_v;
        const int64_t nwarps = (int64_t)gridDim.x * HOT2_WARPS;
        const int64_t slice = (ceil_div(rows, nwarps) + 31) & ~(int64_t)31;
        const int64_t r0 = ((int64_t)blockIdx.x * HOT2_WARPS + warp) * slice;
        const int64_t r1 = r0 + slice < rows ? r0 + slice : rows;
        ZT *tval = static_cast<ZT *>(p.tval);
        for (int64_t b = r0; b < r1; b += 4 * 32) {
            uint8_t t[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) { const int64_t r = b + k * 32 + lane; t[k] = r < r1 ? __ldg(h.pres_tmpl + r) : (uint8_t)0; }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int64_t r = b + k * 32 + lane;
                if (r < r1) {
                    if (r < rows_p) h.tpres[r] = t[k];
                    if (r < rows_v && (r >= h.nrows || t[k] == 0)) tval[r] = (ZT)0;
                }
            }
        }
    }
    pdl_wait();                               // every thread: the gathers below read u_hot beyond the table
    pdl_trigger();                            // the fix-up may be launched; it waits for this kernel to complete
    if (h.tab_n) mbar_wait(s_bar + HOT2_WARPS, 0);

    const XT *uval = static_cast<const XT *>(p.uval);
    const XT *uhot = static_cast<const XT *>(h.u_hot);
    const uint32_t tab_n = h.tab_n, henc = h.henc;
    auto gather = [=](uint32_t col) -> XT {
        if (col < tab_n) return s_hot[col];
        if (col < henc) return gload<XT>(uhot + col);
        return gload<XT>(uval + (col - henc));
    };
    // Software pipeline over the warp's runs: the words of run r+1 are copied out of the stage and its gathers of u
    // are ISSUED before run r is multiplied, folded and stored, so the gather latency sits under a run's worth of
    // arithmetic instead of in front of it (and the bulk copy of run r+2 is in flight under both).
    uint32_t parity = 0;
    RunLane<XT> cur, nxt;
    int64_t cur_run = -1;
    auto fetch = [&](int64_t r, RunLane<XT> &L) {
        mbar_wait(bar, parity); parity ^= 1u;
        const int64_t q = r * RUN + lane * 8;
        const int nvalid = (int)min((int64_t)8, max((int64_t)0, p.nnz - q));
        uint32_t c[8];
        if (NEED_A) {
            const XT *sa = reinterpret_cast<const XT *>(stage + RUN * 4) + lane * 8;
            if constexpr (sizeof(XT) == 4) {
                const uint4 a0 = reinterpret_cast<const uint4 *>(sa)[0], a1 = reinterpret_cast<const uint4 *>(sa)[1];
                const uint32_t w[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
                for (int j = 0; j < 8; ++j) L.a[j] = reinterpret_cast<const XT &>(w[j]);
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j) L.a[j] = sa[j];
            }
        }
        const uint4 *sc = reinterpret_cast<const uint4 *>(stage) + lane * 2;
        const uint4 c0 = sc[0], c1 = sc[1];
        c[0] = c0.x; c[1] = c0.y; c[2] = c0.z; c[3] = c0.w; c[4] = c1.x; c[5] = c1.y; c[6] = c1.z; c[7] = c1.w;
        // WAR guard of the stage.  The bulk copy of the next run writes this stage through the async proxy; nothing orders it
        // after generic-proxy loads that were only ISSUED (a __syncwarp does not wait for their data), and under load a
        // shared-memory load can sit in the LSU queue longer than an L2-hit bulk copy takes -- a lane then folds words of the
        // NEXT run into this run's rows (seen as one wrong hub-row sum in ~1 % of the launches of the overlapped e2e loop).  A vote
        // that READS the first and last loaded word of every lane cannot issue before the warp's loads have written their
        // registers; its predicate is never true (encoded ids stay below 2^32 - 1: spmv_hot_plan), so the copy is always issued.
        uint32_t guard = c[0] & c[7];
        if (NEED_A) {                                                       // the value loads take part too (first and last word of the lane)
            uint32_t w0, w7;
            if constexpr (sizeof(XT) >= 4) { memcpy(&w0, &L.a[0], 4); memcpy(&w7, &L.a[7], 4); }
            else { w0 = (uint32_t)L.a[0]; w7 = (uint32_t)L.a[7]; }             // 1-byte values (BOOL)
            guard &= (w0 | 0x80000000u) & (w7 | 0x80000000u);
        }
        const unsigned never = __ballot_sync(0xffffffffu, guard == 0xFFFFFFFFu);
        if (nvalid < 8) {                                                   // tail of the last run: what lies past nnz is not data
#pragma unroll
            for (int j = 0; j < 8; ++j) { if (j >= nvalid) { c[j] = henc; if (NEED_A) L.a[j] = (XT)1; } }
        }
        if (lane == 0 && never == 0u && r + stride < p.nruns) issue(r + stride);
        spmv_run_gather<XT, MUL, false>(p, r, lane, nvalid, c, L, gather);
    };
    if constexpr (sizeof(XT) > 4 || !PIPE) {
        // one run at a time (8-byte values: two runs in flight do not fit in 64 registers per thread)
        for (; run < p.nruns; run += stride) { fetch(run, cur); spmv_run_fold<XT, ZT, ADD, MUL, false>(p, run, lane, cur); }
        (void)nxt; (void)cur_run;
    } else {
        if (run < p.nruns) { fetch(run, cur); cur_run = run; run += stride; }
        while (cur_run >= 0) {
            const bool more = run < p.nruns;
            if (more) fetch(run, nxt);
            spmv_run_fold<XT, ZT, ADD, MUL, false>(p, cur_run, lane, cur);
            if (more) { cur = nxt; cur_run = run; run += stride; } else cur_run = -1;
        }
    }
}

// The row open at the end of a run: its tail partial (+) the head partials of the following runs up to the last run it
// reaches (every one of those starts inside the row, so its head partial exists).  One item of the plan's fix-up list each.
// The association order is fixed whatever the row's length: lane s of 8 folds head[run+1+s], head[run+9+s], ... (lane 0
// starts with the tail), then lanes combine by the xor butterfly 4, 2, 1.  Items reaching <= FIX_LANES runs have at most one
// head per lane: one thread evaluates the same tree.  The long items come first in the list and take 8 lanes each.
template <typename ZT, int ADD_C, bool SPARSE>
__global__ void __launch_bounds__(256) spmv_run_fixup_kernel(const RunArgs p) {
    pdl_wait();                               // the partials of the run kernel
    const int ADD = ADD_C >= 0 ? ADD_C : p.add_op;
    const ZT *head = static_cast<const ZT *>(p.head_val);
    const int64_t long_threads = p.fix_long * FIX_LANES;
    const int64_t long_ctas = ceil_div(long_threads, 256);
    if ((int64_t)blockIdx.x < long_ctas) {
        const int64_t tid = (int64_t)blockIdx.x * 256 + threadIdx.x;
        const int sub = threadIdx.x & (FIX_LANES - 1);
        const bool ok = tid < long_threads;
        RunFix f{0u, 0u, 0u, 0u};
        if (ok) { const uint4 w = __ldg(reinterpret_cast<const uint4 *>(p.fix + tid / FIX_LANES)); f = RunFix{w.x, w.y, w.z, w.w}; }
        Part<ZT> acc{(ZT)0, 0};
        if (ok) {
            if (sub == 0) { acc.v = static_cast<const ZT *>(p.tail_val)[f.run]; acc.has = SPARSE ? (int)p.tail_has[f.run] : 1; }
            for (int64_t t = (int64_t)f.run + 1 + sub; t <= (int64_t)f.last; t += FIX_LANES) {
                const Part<ZT> y{head[t], SPARSE ? (int)p.head_has[t] : 1};
                acc = part_join<ZT>(ADD, acc, y);
            }
        }
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) {
            Part<ZT> y; y.v = shfl_xor_t<ZT>(acc.v, o); y.has = __shfl_xor_sync(0xffffffffu, acc.has, o);
            acc = part_join<ZT>(ADD, acc, y);
        }
        if (ok && sub == 0) { static_cast<ZT *>(p.tval)[f.row] = acc.v; if (SPARSE) p.tpres[f.row] = (uint8_t)acc.has; }
        return;
    }
    const int64_t i = ((int64_t)blockIdx.x - long_ctas) * 256 + threadIdx.x;
    if (i >= p.fix_short) return;
    const uint4 w = __ldg(reinterpret_cast<const uint4 *>(p.fix + p.fix_long + i));
    const uint32_t run = w.x, row = w.y, n = w.z - w.x;                 // heads run+1 .. run+n, n <= FIX_LANES
    Part<ZT> l[FIX_LANES];                                               // l[s]: what lane s of the 8-lane form holds
#pragma unroll
    for (int s = 0; s < (int)FIX_LANES; ++s) {
        l[s].has = (uint32_t)s < n ? (SPARSE ? (int)p.head_has[run + 1 + s] : 1) : 0;
        l[s].v = (uint32_t)s < n ? head[run + 1 + s] : (ZT)0;
    }
    const Part<ZT> tail{static_cast<const ZT *>(p.tail_val)[run], SPARSE ? (int)p.tail_has[run] : 1};
    l[0] = part_join<ZT>(ADD, tail, l[0]);
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) {
#pragma unroll
        for (int s = 0; s < o; ++s) l[s] = part_join<ZT>(ADD, l[s], l[s + o]);
    }
    static_cast<ZT *>(p.tval)[row] = l[0].v;
    if (SPARSE) p.tpres[row] = (uint8_t)l[0].has;
}

// nnz > 0: the first row start makes at least one item
template <typename ZT, int ADD, bool SPARSE> static void spmv_run_fixup(const RunArgs &a) {
    const int64_t ctas = ceil_div(a.fix_long * FIX_LANES, 256) + ceil_div(a.fix_short, 256);
    launch_pdl(spmv_run_fixup_kernel<ZT, ADD, SPARSE>, (unsigned)ctas, 256, 0, a); GB_LAUNCHED();
}

// shared memory the hot-table kernel can use for its table, after the warp stages and barriers
template <typename XT> static inline uint32_t hot2_table_entries(bool need_a, uint32_t henc, size_t limit_bytes) {
    static int max_optin = 0;                   // one device per process: ask once
    if (!max_optin) cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, G.device);
    const size_t fixed = (size_t)HOT2_WARPS * hot2_stage_bytes<XT>(need_a) + (HOT2_WARPS + 1) * 8 + 8;
    size_t avail = (size_t)max_optin > fixed + 256 ? (size_t)max_optin - fixed - 256 : 0;
    avail = std::min(avail, limit_bytes);
    return (uint32_t)std::min<size_t>(henc, avail / sizeof(XT)) & ~15u;
}

template <typename XT, typename ZT, int ADD, int MUL>
static void spmv_run_launch(const RunArgs &a, const Hot2Args *hot, size_t table_limit) {
    if constexpr (ADD >= 0) {
        if (hot && !a.upres) {
            constexpr bool NEED_A = mul_reads_x(MUL);
            Hot2Args h = *hot;
            h.tab_n = hot2_table_entries<XT>(NEED_A, h.henc, table_limit);
            const size_t smem = (size_t)HOT2_WARPS * hot2_stage_bytes<XT>(NEED_A) + (HOT2_WARPS + 1) * 8 + 8 + (size_t)h.tab_n * sizeof(XT);
            const int ctas = (int)std::min<int64_t>(G.num_sms, ceil_div(a.nruns, HOT2_WARPS));
            // the dynamic shared-memory limit of a kernel is raised once per size (a driver call per launch is host time the
            // multi-GPU step cannot hide: its kernels take tens of microseconds)
            if (sizeof(XT) <= 4 && tunables().spmv_pipe) {
                auto kernel = spmv_run_hot2_kernel<XT, ZT, ADD, MUL, true>;
                static size_t set_for = 0;
                if (set_for != smem) { cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); set_for = smem; }
                launch_pdl(kernel, (unsigned)ctas, HOT2_WARPS * 32, smem, a, h); GB_LAUNCHED();
            } else {
                auto kernel = spmv_run_hot2_kernel<XT, ZT, ADD, MUL, false>;
                static size_t set_for = 0;
                if (set_for != smem) { cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); set_for = smem; }
                launch_pdl(kernel, (unsigned)ctas, HOT2_WARPS * 32, smem, a, h); GB_LAUNCHED();
            }
            spmv_run_fixup<ZT, ADD, false>(a);
            return;
        }
    }
    if (a.upres) {
        spmv_run_kernel<XT, ZT, ADD, MUL, true><<<(unsigned)ceil_div(a.nruns, 8), 256, 0, G.stream>>>(a); GB_LAUNCHED();
        spmv_run_fixup<ZT, ADD, true>(a);
        return;
    }
    spmv_run_kernel<XT, ZT, ADD, MUL, false><<<(unsigned)ceil_div(a.nruns, 8), 256, 0, G.stream>>>(a); GB_LAUNCHED();
    spmv_run_fixup<ZT, ADD, false>(a);
}
