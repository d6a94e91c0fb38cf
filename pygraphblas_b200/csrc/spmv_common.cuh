// Shared by the SpMV translation units (spmv.cu: tile kernel + host logic; spmv_run*.cu: run kernels;
// spmv_pull.cu: masked pull kernels).  Split only to keep nvcc's per-file time down.
#pragma once
#include "common.cuh"
#include <algorithm>
#include <type_traits>

GrB_Info dev_exclusive_scan(int64_t *data, int64_t n, std::string *err);

// ---- 128-bit streaming loads of four consecutive entries (no L1 allocation: L1 is kept for u)
__device__ __forceinline__ uint4 ldg_stream128(const void *p) {
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
template <typename T> __device__ __forceinline__ void load4(const T *p, T *out) {
    if constexpr (sizeof(T) == 4) {
        const uint4 v = ldg_stream128(p);
        out[0] = reinterpret_cast<const T &>(v.x); out[1] = reinterpret_cast<const T &>(v.y);
        out[2] = reinterpret_cast<const T &>(v.z); out[3] = reinterpret_cast<const T &>(v.w);
    } else if constexpr (sizeof(T) == 8) {
        const uint4 v0 = ldg_stream128(p);
        const uint4 v1 = ldg_stream128(reinterpret_cast<const uint4 *>(p) + 1);
        uint64_t q[4] = {((uint64_t)v0.y << 32) | v0.x, ((uint64_t)v0.w << 32) | v0.z,
                         ((uint64_t)v1.y << 32) | v1.x, ((uint64_t)v1.w << 32) | v1.z};
        for (int k = 0; k < 4; ++k) out[k] = reinterpret_cast<const T &>(q[k]);
    } else if constexpr (sizeof(T) == 2) {
        const uint2 v = __ldg(reinterpret_cast<const uint2 *>(p));
        uint16_t q[4] = {(uint16_t)(v.x & 0xffff), (uint16_t)(v.x >> 16), (uint16_t)(v.y & 0xffff), (uint16_t)(v.y >> 16)};
        for (int k = 0; k < 4; ++k) out[k] = reinterpret_cast<const T &>(q[k]);
    } else {
        const uint32_t v = __ldg(reinterpret_cast<const uint32_t *>(p));
        uint8_t q[4] = {(uint8_t)(v & 0xff), (uint8_t)((v >> 8) & 0xff), (uint8_t)((v >> 16) & 0xff), (uint8_t)(v >> 24)};
        for (int k = 0; k < 4; ++k) out[k] = reinterpret_cast<const T &>(q[k]);
    }
}

template <typename T> __device__ __forceinline__ T gload(const T *p) {
    if constexpr (sizeof(T) == 1) { const unsigned char v = __ldg(reinterpret_cast<const unsigned char *>(p)); return reinterpret_cast<const T &>(v); }
    else return __ldg(p);
}

template <typename T> __device__ __forceinline__ T shfl_xor_t(T v, int o) {
    if constexpr (sizeof(T) == 8) { long long x = reinterpret_cast<long long &>(v); x = __shfl_xor_sync(0xffffffffu, x, o); return reinterpret_cast<T &>(x); }
    else if constexpr (sizeof(T) == 4) { int x = reinterpret_cast<int &>(v); x = __shfl_xor_sync(0xffffffffu, x, o); return reinterpret_cast<T &>(x); }
    else { int x = (int)v; x = __shfl_xor_sync(0xffffffffu, x, o); return (T)x; }
}
template <typename T> __device__ __forceinline__ T shfl_down_t(T v, int d) {
    if constexpr (sizeof(T) == 8) { long long x = reinterpret_cast<long long &>(v); x = __shfl_down_sync(0xffffffffu, x, d); return reinterpret_cast<T &>(x); }
    else if constexpr (sizeof(T) == 4) { int x = reinterpret_cast<int &>(v); x = __shfl_down_sync(0xffffffffu, x, d); return reinterpret_cast<T &>(x); }
    else { int x = (int)v; x = __shfl_down_sync(0xffffffffu, x, d); return (T)x; }
}

// A partial monoid value: `has` says whether anything was folded in yet (identity-free, so that
// ANY and "no entry" need no special cases).
template <typename ZT> struct Part { ZT v; int has; };
template <typename ZT> __device__ __forceinline__ Part<ZT> part_join(int add, Part<ZT> a, Part<ZT> b) {
    Part<ZT> r;
    r.has = a.has | b.has;
    r.v = a.has ? (b.has ? MulApply<ZT, ZT>::f(add, a.v, b.v) : a.v) : b.v;
    return r;
}

// which operands a multiply reads (compile-time for the specialised semirings)
__host__ __device__ constexpr bool mul_reads_x(int op) { return !(op == OP_SECOND || op == OP_PAIR); }
__host__ __device__ constexpr bool mul_reads_y(int op) { return !(op == OP_FIRST || op == OP_PAIR || op == OP_ANY); }

template <typename T> __device__ __forceinline__ T shfl_idx_t(T v, int src) {
    if constexpr (sizeof(T) == 8) { long long x = reinterpret_cast<long long &>(v); x = __shfl_sync(0xffffffffu, x, src); return reinterpret_cast<T &>(x); }
    else if constexpr (sizeof(T) == 4) { int x = reinterpret_cast<int &>(v); x = __shfl_sync(0xffffffffu, x, src); return reinterpret_cast<T &>(x); }
    else { int x = (int)v; x = __shfl_sync(0xffffffffu, x, src); return (T)x; }
}
static inline int hgrid(int64_t n) { return (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div(n, 256), (int64_t)G.num_sms * 32)); }

// ---- run kernels (spmv_run.cuh, spmv_run*.cu)
struct RunArgs;
GrB_Info spmv_run_plan(Csr &c, std::string *err);
GrB_Info spmv_hot_plan(Csr &c, std::string *err);
struct Hot2Args;
void spmv_hot2_prep(const Csr &c, const void *u, int vsize);
bool spmv_run_dispatch(int xt, int add, int mul, const RunArgs &a, const Hot2Args *hot, size_t table_limit);
bool spmv_run_generic(int xt, int zt, const RunArgs &a);

// ---- masked pull kernels (spmv_pull.cu)
struct PullArgs;
GrB_Info spmv_masked_pull_dispatch(int xt, int zt, const PullArgs &a, std::string *err);
