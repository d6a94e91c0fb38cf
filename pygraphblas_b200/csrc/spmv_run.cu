// Run plan, hot-column plan, and the FP32 / FP64 instantiations of the run kernels.
#include "spmv_run.cuh"
#include <cub/device/device_radix_sort.cuh>

// ---- run plan (cached per CSR)
__global__ void plan_nonempty_kernel(const uint32_t *rowptr, int64_t nrows, int64_t *flag, uint8_t *pres) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < nrows; r += (int64_t)gridDim.x * blockDim.x) {
        const int ne = rowptr[r + 1] > rowptr[r];
        flag[r] = ne; pres[r] = (uint8_t)ne;
    }
}
__global__ void plan_rows_kernel(const uint32_t *rowptr, const int64_t *rank, int64_t nrows, uint32_t *nzrow, uint32_t *headw) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < nrows; r += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t rs = rowptr[r];
        if (rowptr[r + 1] > rs) { nzrow[rank[r]] = (uint32_t)r; atomicOr(&headw[rs >> 5], 1u << (rs & 31)); }
    }
}
__global__ void plan_runs_kernel(const uint32_t *headw, int64_t nruns, int64_t nwords, uint16_t *lane_rank, int64_t *run_cnt) {
    const int lane = threadIdx.x & 31;
    const int64_t run = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (run >= nruns) return;
    const int64_t w = run * 8 + (lane >> 2);
    const uint32_t hw = w < nwords ? headw[w] : 0u;
    const int pc = __popc((hw >> ((lane & 3) * 8)) & 0xffu);
    int inc = pc;
    for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += y; }
    lane_rank[run * 32 + lane] = (uint16_t)(inc - pc);
    if (lane == 31) run_cnt[run] = inc;
}
__global__ void plan_base_kernel(const int64_t *scan, int64_t nruns, uint32_t *run_base) {
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k <= nruns; k += (int64_t)gridDim.x * blockDim.x) run_base[k] = (uint32_t)scan[k];
}
// the row that starts last inside a run always holds the run's last entry: it is the run's "open" row (possibly ending
// exactly at the run's end), completed by the fix-up kernel.  One fix-up item per run that holds a row start.
__device__ __forceinline__ bool plan_fix_item(const uint32_t *run_base, const uint32_t *nzrow, const uint32_t *rowptr, int64_t k, RunFix &f) {
    if (run_base[k + 1] == run_base[k]) return false;
    const uint32_t r = nzrow[run_base[k + 1] - 1];
    f = RunFix{(uint32_t)k, r, (rowptr[r + 1] - 1) / RUN, 0u};
    return true;
}
// is_long[k] / is_short[k]: run k has an item whose row reaches more / at most FIX_LANES runs further
__global__ void plan_fix_count_kernel(const uint32_t *run_base, const uint32_t *nzrow, const uint32_t *rowptr, int64_t nruns,
                                      int64_t *is_long, int64_t *is_short) {
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nruns; k += (int64_t)gridDim.x * blockDim.x) {
        RunFix f;
        const bool has = plan_fix_item(run_base, nzrow, rowptr, k, f);
        const bool lg = has && f.last - f.run > FIX_LANES;
        is_long[k] = lg; is_short[k] = has && !lg;
    }
}
// the list in run order, the long items first (their exclusive scans give the slots)
__global__ void plan_fix_list_kernel(const uint32_t *run_base, const uint32_t *nzrow, const uint32_t *rowptr, int64_t nruns,
                                     const int64_t *long_at, const int64_t *short_at, int64_t nlong, RunFix *list) {
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nruns; k += (int64_t)gridDim.x * blockDim.x) {
        RunFix f;
        if (plan_fix_item(run_base, nzrow, rowptr, k, f)) list[f.last - f.run > FIX_LANES ? long_at[k] : nlong + short_at[k]] = f;
    }
}
static inline int rgrid(int64_t n) { return (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div(n, 256), (int64_t)G.num_sms * 16)); }

GrB_Info spmv_run_plan(Csr &c, std::string *err) {
    if (c.run_headw) return GrB_SUCCESS;
    if (!c.rowptr32) return gb_fail(GrB_INVALID_VALUE, err, "mxv: matrices with >= 2^32 entries are not supported");
    const int64_t nwords = ceil_div(c.nnz, 32);
    c.nruns = ceil_div(c.nnz, RUN);
    int64_t *flag = nullptr, *cnt = nullptr;
    GB_TRY(dalloc(&flag, (size_t)c.nrows + 1, err));
    GB_TRY(dalloc(&cnt, (size_t)c.nruns + 1, err));
    GB_TRY(dalloc(&c.pres_tmpl, (size_t)c.nrows, err));
    GB_TRY(dalloc(&c.run_headw, (size_t)nwords + 8, err));
    GB_TRY(dalloc(&c.run_lane, (size_t)c.nruns * 32, err));
    GB_TRY(dalloc(&c.run_base, (size_t)c.nruns + 1, err));
    CU_TRY(cudaMemsetAsync(c.run_headw, 0, ((size_t)nwords + 8) * 4, G.stream), err);
    CU_TRY(cudaMemsetAsync(flag + c.nrows, 0, 8, G.stream), err);
    plan_nonempty_kernel<<<rgrid(c.nrows), 256, 0, G.stream>>>(c.rowptr32, c.nrows, flag, c.pres_tmpl); GB_LAUNCHED();
    GB_TRY(dev_exclusive_scan(flag, c.nrows + 1, err));
    int64_t nz = 0;
    CU_TRY(cudaMemcpyAsync(&nz, flag + c.nrows, 8, cudaMemcpyDeviceToHost, G.stream), err);
    CU_TRY(cudaStreamSynchronize(G.stream), err);
    c.nnzrows = nz;
    GB_TRY(dalloc(&c.nzrow, (size_t)nz, err));
    plan_rows_kernel<<<rgrid(c.nrows), 256, 0, G.stream>>>(c.rowptr32, flag, c.nrows, c.nzrow, c.run_headw); GB_LAUNCHED();
    CU_TRY(cudaMemsetAsync(cnt + c.nruns, 0, 8, G.stream), err);
    plan_runs_kernel<<<(unsigned)ceil_div(c.nruns * 32, 256), 256, 0, G.stream>>>(c.run_headw, c.nruns, nwords, c.run_lane, cnt); GB_LAUNCHED();
    GB_TRY(dev_exclusive_scan(cnt, c.nruns + 1, err));
    plan_base_kernel<<<rgrid(c.nruns + 1), 256, 0, G.stream>>>(cnt, c.nruns, c.run_base); GB_LAUNCHED();
    // fix-up list: flag the runs by kind into the two halves of `flag2`, scan each, scatter
    int64_t *flag2 = nullptr;
    GB_TRY(dalloc(&flag2, 2 * ((size_t)c.nruns + 1), err));
    int64_t *is_long = flag2, *is_short = flag2 + c.nruns + 1;
    CU_TRY(cudaMemsetAsync(is_long + c.nruns, 0, 8, G.stream), err);
    CU_TRY(cudaMemsetAsync(is_short + c.nruns, 0, 8, G.stream), err);
    plan_fix_count_kernel<<<rgrid(c.nruns), 256, 0, G.stream>>>(c.run_base, c.nzrow, c.rowptr32, c.nruns, is_long, is_short); GB_LAUNCHED();
    GB_TRY(dev_exclusive_scan(is_long, c.nruns + 1, err));
    GB_TRY(dev_exclusive_scan(is_short, c.nruns + 1, err));
    int64_t nfix[2] = {0, 0};
    CU_TRY(cudaMemcpyAsync(&nfix[0], is_long + c.nruns, 8, cudaMemcpyDeviceToHost, G.stream), err);
    CU_TRY(cudaMemcpyAsync(&nfix[1], is_short + c.nruns, 8, cudaMemcpyDeviceToHost, G.stream), err);
    CU_TRY(cudaStreamSynchronize(G.stream), err);
    c.run_fix_long = nfix[0]; c.run_fix_short = nfix[1];
    GB_TRY(dalloc(&c.run_fix, (size_t)(nfix[0] + nfix[1]), err));
    plan_fix_list_kernel<<<rgrid(c.nruns), 256, 0, G.stream>>>(c.run_base, c.nzrow, c.rowptr32, c.nruns, is_long, is_short, nfix[0], c.run_fix); GB_LAUNCHED();
    dfree(flag); dfree(cnt); dfree(flag2);
    // per-call scratch lives with the plan: partials of the rows that straddle runs (8 bytes covers every type)
    GB_TRY(dmalloc(&c.ws_head, (size_t)c.nruns * 8 + 16, err));
    GB_TRY(dmalloc(&c.ws_tail, (size_t)c.nruns * 8 + 16, err));
    GB_TRY(dmalloc((void **)&c.ws_head_has, (size_t)c.nruns + 16, err));
    GB_TRY(dmalloc((void **)&c.ws_tail_has, (size_t)c.nruns + 16, err));
    CU_TRY(cudaGetLastError(), err);
    return GrB_SUCCESS;
}

// ---- hot-column plan (cached per CSR): the HOT_ENC most referenced columns are renamed to their rank, every other
//      column c to c + henc, so the kernel tells a table lookup from a gather of u by one compare and u itself is
//      read in place (no permuted copy per call)
constexpr uint32_t HOT_ENC = 40960;
__global__ void hot_count_kernel(const uint32_t *col, int64_t nnz, uint32_t *deg) {
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nnz; k += (int64_t)gridDim.x * blockDim.x) atomicAdd(&deg[col[k]], 1u);
}
__global__ void hot_iota_kernel(uint32_t *a, int64_t n) {
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) a[k] = (uint32_t)k;
}
// inv[col] = rank for the first k ranks whose degree is non-zero; sum of their degrees; how many there are
__global__ void hot_invert_kernel(const uint32_t *perm, const uint32_t *deg_sorted, int64_t k, uint32_t *inv, unsigned long long *stats) {
    unsigned long long c = 0, d = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < k; i += (int64_t)gridDim.x * blockDim.x) {
        if (deg_sorted[i] != 0) { inv[perm[i]] = (uint32_t)i; c += 1; d += deg_sorted[i]; }
    }
    for (int o = 16; o > 0; o >>= 1) { c += __shfl_xor_sync(0xffffffffu, c, o); d += __shfl_xor_sync(0xffffffffu, d, o); }
    if ((threadIdx.x & 31) == 0 && c) { atomicAdd(stats, c); atomicAdd(stats + 1, d); }
}
__global__ void hot_encode_kernel(const uint32_t *col, const uint32_t *inv, int64_t nnz, uint32_t henc, uint32_t *out) {
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nnz; k += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t c = col[k], r = inv[c];
        out[k] = r < henc ? r : c + henc;
    }
}

GrB_Info spmv_hot_plan(Csr &c, std::string *err) {
    if (c.hot_planned) return GrB_SUCCESS;
    const int64_t n = c.ncols;
    if (n + (int64_t)HOT_ENC >= ((int64_t)1 << 32)) { c.hot_planned = true; return GrB_SUCCESS; }
    uint32_t *deg = nullptr, *deg_sorted = nullptr, *ids = nullptr, *inv = nullptr, *perm = nullptr; unsigned long long *stats = nullptr;
    GB_TRY(dalloc(&deg, (size_t)n, err)); GB_TRY(dalloc(&deg_sorted, (size_t)n, err)); GB_TRY(dalloc(&ids, (size_t)n, err));
    GB_TRY(dalloc(&inv, (size_t)n, err)); GB_TRY(dalloc(&perm, (size_t)n, err)); GB_TRY(dalloc(&stats, 2, err));
    CU_TRY(cudaMemsetAsync(deg, 0, (size_t)n * 4, G.stream), err);
    CU_TRY(cudaMemsetAsync(inv, 0xff, (size_t)n * 4, G.stream), err);
    CU_TRY(cudaMemsetAsync(stats, 0, 16, G.stream), err);
    hot_count_kernel<<<hgrid(c.nnz), 256, 0, G.stream>>>(c.col, c.nnz, deg); GB_LAUNCHED();
    hot_iota_kernel<<<hgrid(n), 256, 0, G.stream>>>(ids, n); GB_LAUNCHED();
    size_t tmp_bytes = 0;     // stable sort: equal degrees keep ascending column order (deterministic plan)
    CU_TRY(cub::DeviceRadixSort::SortPairsDescending(nullptr, tmp_bytes, deg, deg_sorted, ids, perm, n, 0, 32, G.stream), err);
    void *tmp = nullptr; GB_TRY(dmalloc(&tmp, tmp_bytes, err));
    CU_TRY(cub::DeviceRadixSort::SortPairsDescending(tmp, tmp_bytes, deg, deg_sorted, ids, perm, n, 0, 32, G.stream), err);
    G.launches += 8;
    const int64_t topk = std::min<int64_t>(n, HOT_ENC);
    hot_invert_kernel<<<hgrid(topk), 256, 0, G.stream>>>(perm, deg_sorted, topk, inv, stats); GB_LAUNCHED();
    unsigned long long h[2] = {0, 0};
    CU_TRY(cudaMemcpyAsync(h, stats, 16, cudaMemcpyDeviceToHost, G.stream), err);
    CU_TRY(cudaStreamSynchronize(G.stream), err);
    c.hot_cover = c.nnz ? (double)h[1] / (double)c.nnz : 0.0;
    c.hot_planned = true;
    if (h[0] >= 16) {
        c.henc = (uint32_t)h[0];
        GB_TRY(dalloc(&c.hperm, (size_t)c.henc, err));
        GB_TRY(dalloc(&c.hcol, (size_t)c.nnz, err));
        GB_TRY(dmalloc(&c.ws_uhot, (size_t)c.henc * 8 + 16, err));
        CU_TRY(cudaMemcpyAsync(c.hperm, perm, (size_t)c.henc * 4, cudaMemcpyDeviceToDevice, G.stream), err);
        hot_encode_kernel<<<hgrid(c.nnz), 256, 0, G.stream>>>(c.col, inv, c.nnz, c.henc, c.hcol); GB_LAUNCHED();
    }
    dfree(tmp); dfree(deg); dfree(deg_sorted); dfree(ids); dfree(inv); dfree(perm); dfree(stats);
    CU_TRY(cudaGetLastError(), err);
    return GrB_SUCCESS;
}

// prep for the hot-table kernel: u_hot[i] = u[hperm[i]] for the henc hottest columns (the kernel fills T itself)
__global__ void __launch_bounds__(256) spmv_hot2_prep_kernel(const uint32_t *hperm, const uint8_t *u, uint8_t *u_hot, int vsize, uint32_t henc) {
    pdl_trigger();                            // the hot-table kernel's prologue needs nothing from here
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= henc) return;
    const uint32_t col = hperm[i];
    switch (vsize) {
        case 1: u_hot[i] = u[col]; break;
        case 4: ((uint32_t *)u_hot)[i] = ((const uint32_t *)u)[col]; break;
        default: ((uint64_t *)u_hot)[i] = ((const uint64_t *)u)[col]; break;
    }
}

void spmv_hot2_prep(const Csr &c, const void *u, int vsize) {
    spmv_hot2_prep_kernel<<<(unsigned)ceil_div(c.henc, 256), 256, 0, G.stream>>>(c.hperm, (const uint8_t *)u, (uint8_t *)c.ws_uhot, vsize, c.henc);
    GB_LAUNCHED();
}

template <typename T> static bool spmv_run_fast(int add, int mul, const RunArgs &a, const Hot2Args *hot, size_t table_limit) {
#define GB_FAST(A, M) if (add == A && mul == M) { spmv_run_launch<T, T, A, M>(a, hot, table_limit); return true; }
    GB_FAST(OP_PLUS, OP_TIMES) GB_FAST(OP_MIN, OP_PLUS) GB_FAST(OP_PLUS, OP_SECOND) GB_FAST(OP_PLUS, OP_FIRST)
    GB_FAST(OP_PLUS, OP_PAIR) GB_FAST(OP_MIN, OP_FIRST) GB_FAST(OP_MIN, OP_SECOND)
#undef GB_FAST
    return false;
}
bool spmv_run_fast_int(int xt, int add, int mul, const RunArgs &a, const Hot2Args *hot, size_t table_limit);
bool spmv_run_dispatch(int xt, int add, int mul, const RunArgs &a, const Hot2Args *hot, size_t table_limit) {
    switch (xt) {
        case TC_FP32: return spmv_run_fast<float>(add, mul, a, hot, table_limit);
        case TC_FP64: return spmv_run_fast<double>(add, mul, a, hot, table_limit);
        case TC_INT32:
        case TC_INT64:
        case TC_UINT32:
        case TC_UINT64:
        case TC_BOOL: return spmv_run_fast_int(xt, add, mul, a, hot, table_limit);
        default: return false;
    }
}
