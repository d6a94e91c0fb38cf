// common.cuh -- internal declarations of libb200grb (not part of the C ABI).
//
// Object model behind the opaque GraphBLAS handles of include/b200grb.h, the
// scalar "carrier" used wherever a value's type is only known at run time
// (typecasts, accumulators, dup operators), and the typed operator templates
// that the sm_100a kernels instantiate.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <math.h>
#include <float.h>
#include <limits.h>
#include <string>
#include <vector>
#include <mutex>
#include "../../include/b200grb.h"

#define GB_MAGIC 0x42323030  /* "B200" */
#define GB_FREED 0x0DEAD000

// ---------------------------------------------------------------- type codes
enum TypeCode : int {
    TC_BOOL = 0, TC_INT8, TC_INT16, TC_INT32, TC_INT64,
    TC_UINT8, TC_UINT16, TC_UINT32, TC_UINT64, TC_FP32, TC_FP64, TC_COUNT
};

// ---------------------------------------------------------------- operator codes
enum OpCode : int {
    OP_FIRST = 0, OP_SECOND, OP_PAIR, OP_ANY, OP_MIN, OP_MAX, OP_PLUS, OP_MINUS, OP_RMINUS,
    OP_TIMES, OP_DIV, OP_RDIV, OP_POW, OP_ISEQ, OP_ISNE, OP_ISGT, OP_ISLT, OP_ISGE, OP_ISLE,
    OP_LOR, OP_LAND, OP_LXOR, OP_BOR, OP_BAND, OP_BXOR, OP_BXNOR,
    OP_EQ, OP_NE, OP_GT, OP_LT, OP_GE, OP_LE,   // z = BOOL
    OP_USER, OP_COUNT
};
static inline bool op_is_cmp(int op) { return op >= OP_EQ && op <= OP_LE; }

// ---------------------------------------------------------------- opaque objects
struct GB_Type_opaque { int magic; int code; size_t size; const char *name; };
struct GB_BinaryOp_opaque {
    int magic; int opcode; GrB_Type xtype, ytype, ztype; const char *name; void *user_fn;
};
struct GB_Monoid_opaque { int magic; GrB_BinaryOp op; const char *name; bool builtin; };
struct GB_Semiring_opaque { int magic; GrB_Monoid add; GrB_BinaryOp mul; const char *name; bool builtin; };
struct GB_Descriptor_opaque {
    int magic; int outp, mask, inp0, inp1; int axb; int nthreads; double chunk; int sort;
    bool builtin; const char *name;
};
struct GB_UnaryOp_opaque { int magic; int opcode; GrB_Type xtype, ztype; const char *name; };
enum UnaryCode : int {
    UOP_IDENTITY = 0, UOP_AINV, UOP_MINV, UOP_LNOT, UOP_ONE, UOP_ABS, UOP_BNOT,
    // floating point only
    UOP_SQRT, UOP_LOG, UOP_EXP, UOP_LOG2, UOP_SIN, UOP_COS, UOP_TAN, UOP_ACOS, UOP_ASIN, UOP_ATAN, UOP_SINH, UOP_COSH,
    UOP_TANH, UOP_ACOSH, UOP_ASINH, UOP_ATANH, UOP_SIGNUM, UOP_CEIL, UOP_FLOOR, UOP_ROUND, UOP_TRUNC, UOP_EXP2,
    UOP_EXPM1, UOP_LOG10, UOP_LOG1P, UOP_LGAMMA, UOP_TGAMMA, UOP_ERF, UOP_ERFC,
    UOP_ISINF, UOP_ISNAN, UOP_ISFINITE,      // z = BOOL
    UOP_COUNT
};

struct RunFix;
// Device CSR panel: rows sorted, columns sorted inside each row.
struct Csr {
    int64_t nrows = 0, ncols = 0, nnz = 0;
    int64_t *rowptr = nullptr;     // [nrows+1] 64-bit offsets (canonical)
    uint32_t *rowptr32 = nullptr;  // [nrows+1] 32-bit shadow, built when nnz < 2^32
    uint32_t *col = nullptr;       // [nnz]
    void *val = nullptr;           // [nnz] of the matrix type
    // SpMV plan: first row of every TILE-sized slice of the nnz range (spmv.cu)
    uint32_t *tile_row = nullptr;
    int64_t ntiles = 0;
    int tile_size = 0;
    // run plan (spmv.cu, dense-u kernel): entries cut into warp-sized runs of 256
    uint32_t *run_headw = nullptr;   // [ceil(nnz/32)] bit q = entry q starts a row
    uint16_t *run_lane = nullptr;    // [nruns*32] row starts inside the run before the lane's first entry
    uint32_t *run_base = nullptr;    // [nruns+1] row starts before the run (= rank of its first row start)
    RunFix *run_fix = nullptr;       // [run_fix_long + run_fix_short] fix-up items (spmv_args.cuh), the long ones first
    int64_t run_fix_long = 0, run_fix_short = 0;
    uint32_t *nzrow = nullptr;       // [nnzrows] ids of the non-empty rows, ascending
    uint8_t *pres_tmpl = nullptr;    // [nrows] 1 where the row is non-empty
    int64_t nruns = 0, nnzrows = 0;
    // hot-column plan (spmv_run.cu): the henc most referenced columns get their rank as id, the others col + henc
    uint32_t *hperm = nullptr;     // [henc] hot rank -> original column
    uint32_t *hcol = nullptr;      // [nnz] encoded column ids
    uint32_t henc = 0;             // ids below this are hot ranks
    bool hot_planned = false;      // the plan was attempted (hcol stays NULL when the gathers are not concentrated)
    double hot_cover = 0.0;        // share of the entries whose column is among the henc most referenced
    // per-call scratch of the run kernels, kept with the plan (no allocation on the call path)
    void *ws_head = nullptr, *ws_tail = nullptr;   // [nruns] x 8 bytes: partials of the rows a run starts / ends inside
    uint8_t *ws_head_has = nullptr, *ws_tail_has = nullptr;
    void *ws_uhot = nullptr;       // [henc] x 8 bytes: u at the hot columns
    bool valid = false;
};

// per-object storage hints of SuiteSparse's GxB_*_Option_set/get: recorded and reported back, without effect on the HBM
// layout (always CSR by row / dense + presence) -- the API is format-agnostic, results do not depend on them
struct GBObjOpts { double hyper = 0.0625; int format = 0 /* GxB_BY_ROW */; int sparsity = 15 /* GxB_AUTO_SPARSITY */; };

struct GB_Matrix_opaque {
    int magic; GrB_Type type; uint64_t nrows, ncols;
    GBObjOpts opts;
    // host form: row-major sorted unique COO
    std::vector<uint64_t> hi, hj; std::vector<uint8_t> hx; bool host_valid;
    // pending setElement tuples (in call order; later wins)
    std::vector<uint64_t> pi, pj; std::vector<uint8_t> px;
    // device form (+ cached transpose)
    Csr dev, devT;
    std::string err;
};

struct GB_Vector_opaque {
    int magic; GrB_Type type; uint64_t n;
    GBObjOpts opts;
    // host form: sorted unique (index, value)
    std::vector<uint64_t> hi; std::vector<uint8_t> hx; bool host_valid;
    std::vector<uint64_t> pi; std::vector<uint8_t> px;
    // device form: dense values + presence bytes (present == nullptr: all present)
    void *dval = nullptr; uint8_t *dpres = nullptr; bool dev_valid = false; int64_t dev_nvals = -1;
    bool borrowed = false;     // dval / dpres belong to a communicator (dist.cu): never freed through the vector
    // overlapped host copies (B200_Vector_set_dense / export_dense with where = 2): the copy streams' hand-shakes with the compute stream
    cudaEvent_t ev_h2d = nullptr, ev_d2h = nullptr, ev_use = nullptr;
    bool h2d_pending = false, d2h_pending = false, use_recorded = false;
    std::string err;
};

// ---------------------------------------------------------------- globals (objects.cu)
struct GBGlobal {
    bool initialized = false;
    bool have_device = false;
    int device = 0;
    int num_sms = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t h2d = nullptr, d2h = nullptr;     // copy streams of the overlapped import / export (where = 2)
    uint64_t launches = 0;
    uint64_t last_flops = 0, last_nnz_out = 0;
    int burble = 0;
    cudaEvent_t burble_e0 = nullptr, burble_e1 = nullptr;
    std::recursive_mutex mu;
};
extern GBGlobal G;
extern thread_local std::string tl_error;

GrB_Info gb_fail(GrB_Info code, std::string *where, const char *fmt, ...);

// every entry point: take the library lock and make the library's device current for the calling host thread
// (the reference drives `lib` from a ThreadPool, /root/reference/demo/dnn/challenge.py:48-51; a new thread starts on device 0)
static inline void gb_thread_enter() {
    // the embedding application (torch, another library) may have switched this thread to another GPU since the last call:
    // ask, do not cache
    if (G.have_device) { int cur = -1; if (cudaGetDevice(&cur) != cudaSuccess || cur != G.device) cudaSetDevice(G.device); }
    tl_error.clear();                      // GrB_*_error / B200_last_error report the failure of the LAST call of this thread
}
#define GB_LOCK std::lock_guard<std::recursive_mutex> _lk(G.mu); gb_thread_enter()
#define GB_CHECK_INIT  do { if (!G.initialized) return gb_fail(GrB_PANIC, nullptr, "GrB_init not called"); } while (0)
#define GB_TRY(expr) do { GrB_Info _i = (expr); if (_i != GrB_SUCCESS) return _i; } while (0)
#define CU_TRY(expr, errstr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) \
    return gb_fail(_e == cudaErrorMemoryAllocation ? GrB_OUT_OF_MEMORY : GrB_PANIC, errstr, \
                   "CUDA error %s at %s:%d", cudaGetErrorString(_e), __FILE__, __LINE__); } while (0)

// kernel-choice switches read from the environment ONCE (GrB_init) and again only on B200_reload_tunables()
// (tests flip them between calls); nothing on a call path touches getenv
struct Tunables {
    int spmv_items = 8;        // B200GRB_SPMV_ITEMS   entries per thread of the tile kernel (4 / 8 / 16)
    int spmv_run = -1;         // B200GRB_SPMV_RUN     -1 default choice, 0 never, 1 always the run kernel
    int spmv_hot_kb = -1;      // B200GRB_SPMV_HOT     -1 default (on when the gathers are concentrated), 0 off, >0 table cap in KB
    bool no_pull = false, no_push = false, force_push = false, spmv_debug = false;
    bool spmv_pipe = false;    // B200GRB_SPMV_PIPE    software-pipeline two runs per warp in the hot-table kernel (4-byte types)
    bool spgemm_trace = false; // B200GRB_SPGEMM_TRACE phase times of GrB_mxm (masked) on stderr
    int stream_blk_log2 = 7;   // B200GRB_STREAM_BLK   log2 of the block of a long B row one warp takes (masked SpGEMM)
    int spgemm_v = 0;          // B200GRB_SPGEMM_V     masked SpGEMM kernel generation (0 = default)
    bool spgemm_esc = true;    // B200GRB_SPGEMM_ESC   0: the shared-memory bins of the unmasked numeric pass use the hash kernels instead of expand-sort-compress
    int mxv_inplace = 1;       // B200GRB_MXV_INPLACE  0: mxv / vxm never form T in w's own buffers; 1: when w has no copy in flight;
                               //                      2: always, the compute stream first joins w's last overlapped copies
};
const Tunables &tunables();

// GxB_BURBLE (/root/reference/pygraphblas/base.py:84-86): when on, every compute entry point prints which kernel it
// chose, the algorithmic bytes of the call and its device time; every entry point is also an NVTX range
struct GbBurble {
    bool on; const char *fn; const char *kernel = ""; double bytes = 0.0;
    explicit GbBurble(const char *fn);
    void note(const char *k, double b) { kernel = k; bytes = b; }
    ~GbBurble();
};

// device memory (stream-ordered pool on G.stream)
GrB_Info dmalloc(void **p, size_t bytes, std::string *err);
void dfree(void *p);
template <typename T> static inline GrB_Info dalloc(T **p, size_t count, std::string *err) {
    return dmalloc((void **)p, count * sizeof(T) + 16, err);   // +16: bulk copies may over-read a tail
}
void csr_free(Csr &c);
void csr_drop_plans(Csr &c);
// Persistent scratch of the compute calls: slot k keeps its buffer between calls and only grows (calls are serialised on one
// stream, so a slot is never in use twice).  Large transient cudaMallocAsync / cudaFreeAsync pairs were measured to cost
// 10-70 ms per call when the pool has to map fresh memory (masked GrB_mxm: 620 MB of column maps) -- these buffers never leave.
enum WsSlot : int { WS_WORDS = 0, WS_FOUND, WS_FLOPS, WS_TOTAL, WS_CS, WS_CM, WS_CL, WS_C1, WS_SROW, WS_SIDX, WS_SCNT, WS_MROW, WS_MIDX, WS_MCNT,
                    WS_LROW, WS_LIDX, WS_LCNT, WS_WROWS, WS_QUEUES, WS_SPA_SLOT, WS_COUNT };
GrB_Info ws_get(int slot, void **p, size_t bytes, std::string *err, bool *fresh = nullptr);
template <typename T> static inline GrB_Info ws_array(int slot, T **p, size_t count, std::string *err, bool *fresh = nullptr) {
    return ws_get(slot, (void **)p, count * sizeof(T) + 16, err, fresh);
}

// host <-> device sync of containers (objects.cu)
GrB_Info matrix_flush_pending(GrB_Matrix A);
GrB_Info matrix_ensure_host(GrB_Matrix A);
GrB_Info matrix_ensure_device(GrB_Matrix A);
GrB_Info matrix_ensure_transpose(GrB_Matrix A);     // builds A->devT on the device
void matrix_invalidate_device(GrB_Matrix A);
void matrix_adopt_device(GrB_Matrix A, Csr &c);     // A takes ownership of c, host form dropped
GrB_Info vector_ensure_host(GrB_Vector v);
GrB_Info vector_ensure_device(GrB_Vector v);
void vector_invalidate_device(GrB_Vector v);
void vector_adopt_device(GrB_Vector v, void *vals, uint8_t *pres);
void vector_mark_used(GrB_Vector v);               // after the kernels reading v were enqueued (lets the next overlapped import of v start early)
bool gb_valid_matrix(const GrB_Matrix A);
bool gb_valid_vector(const GrB_Vector v);

struct DescFlags { bool replace, mask_comp, mask_struct, tran0, tran1; int axb; };
// hypersparse operands (dimension beyond 2^31-1): computed on in their compact index space (hyper.cu)
bool gb_hyper_matrix(const GrB_Matrix A);
bool gb_hyper_vector(const GrB_Vector v);
GrB_Info hyper_mxv(GrB_Vector w, const GrB_Vector mask, const GrB_BinaryOp accum, const GrB_Semiring s, const GrB_Matrix A, const GrB_Vector u,
                   const GrB_Descriptor desc, bool vxm);
GrB_Info hyper_mxm(GrB_Matrix C, const GrB_Matrix Mask, const GrB_BinaryOp accum, const GrB_Semiring s, const GrB_Matrix A, const GrB_Matrix B,
                   const GrB_Descriptor desc);
DescFlags desc_flags(const GrB_Descriptor d);

// w<mask> = accum(w, T) on the device (vector_ops.cu).  T = (tval, tpres) of type ttc over w->n positions
// (tpres NULL: every position present; t_scalar: tval is ONE value standing for all positions).  region
// (NULL = everything) limits the write to the positions it flags, GrB_assign style.  own_t: T's buffers are
// released here.
struct Sc;
// C<Mask> = accum(C, T) for a CSR T of type ttc (spgemm.cu); consumes T
GrB_Info matrix_writeback(GrB_Matrix C, const GrB_Matrix Mask, const GrB_BinaryOp accum, const DescFlags &f,
                          Csr &T, int ttc, bool t_already_masked, std::string *err);
// fold of n values (presence bytes optional) with a builtin monoid operator on the device (vector_ops.cu)
GrB_Info dev_reduce_values(const void *val, const uint8_t *pres, int vtc, int64_t n, int op, int mtc, Sc *out, bool *has, std::string *err);
GrB_Info vector_write(GrB_Vector w, const GrB_Vector mask, const GrB_BinaryOp accum, const DescFlags &f,
                      void *tval, uint8_t *tpres, int ttc, bool t_scalar, const uint8_t *region, bool own_t);

// kernels (device_ops.cu / spmv.cu / spgemm.cu)
GrB_Info dev_build_rowptr32(Csr &c, std::string *err);
GrB_Info dev_exclusive_scan(int64_t *data, int64_t n, std::string *err);
GrB_Info dev_transpose(const Csr &a, size_t vsize, Csr &t, std::string *err);
GrB_Info dev_cast_values(void **out, int to_code, const void *in, int from_code, int64_t n, std::string *err);
GrB_Info dev_count_present(const uint8_t *pres, int64_t n, int64_t *count, std::string *err);

// ---------------------------------------------------------------- scalar carrier
// A value of any builtin type held in 64 bits: BOOL/UINT* in .u, INT* in .i, FP* in .d
// (a float is held as the exactly-equal double).
struct Sc { union { int64_t i; uint64_t u; double d; }; };
struct GB_Scalar_opaque { int magic; GrB_Type type; bool has; Sc v; };     // GxB_Scalar (compat.cu)
enum SelectCode : int { SEL_TRIL = 0, SEL_TRIU, SEL_DIAG, SEL_OFFDIAG, SEL_NONZERO, SEL_EQ_ZERO, SEL_GT_ZERO, SEL_GE_ZERO, SEL_LT_ZERO, SEL_LE_ZERO,
                        SEL_NE_THUNK, SEL_EQ_THUNK, SEL_GT_THUNK, SEL_GE_THUNK, SEL_LT_THUNK, SEL_LE_THUNK };
struct GB_SelectOp_opaque { int magic; const char *name; int code; };

__host__ __device__ static inline int tc_size(int tc) {
    switch (tc) {
        case TC_BOOL: case TC_INT8: case TC_UINT8: return 1;
        case TC_INT16: case TC_UINT16: return 2;
        case TC_INT32: case TC_UINT32: case TC_FP32: return 4;
        default: return 8;
    }
}
__host__ __device__ static inline bool tc_is_float(int tc) { return tc == TC_FP32 || tc == TC_FP64; }
__host__ __device__ static inline bool tc_is_signed(int tc) { return tc >= TC_INT8 && tc <= TC_INT64; }

__host__ __device__ static inline Sc sc_load(int tc, const void *p, size_t k) {
    Sc s; s.u = 0;
    switch (tc) {
        case TC_BOOL:   s.u = ((const uint8_t *)p)[k] != 0; break;
        case TC_INT8:   s.i = ((const int8_t *)p)[k]; break;
        case TC_INT16:  s.i = ((const int16_t *)p)[k]; break;
        case TC_INT32:  s.i = ((const int32_t *)p)[k]; break;
        case TC_INT64:  s.i = ((const int64_t *)p)[k]; break;
        case TC_UINT8:  s.u = ((const uint8_t *)p)[k]; break;
        case TC_UINT16: s.u = ((const uint16_t *)p)[k]; break;
        case TC_UINT32: s.u = ((const uint32_t *)p)[k]; break;
        case TC_UINT64: s.u = ((const uint64_t *)p)[k]; break;
        case TC_FP32:   s.d = (double)((const float *)p)[k]; break;
        case TC_FP64:   s.d = ((const double *)p)[k]; break;
    }
    return s;
}
__host__ __device__ static inline void sc_store(int tc, void *p, size_t k, Sc s) {
    switch (tc) {
        case TC_BOOL:   ((uint8_t *)p)[k] = (uint8_t)(s.u != 0); break;
        case TC_INT8:   ((int8_t *)p)[k] = (int8_t)s.i; break;
        case TC_INT16:  ((int16_t *)p)[k] = (int16_t)s.i; break;
        case TC_INT32:  ((int32_t *)p)[k] = (int32_t)s.i; break;
        case TC_INT64:  ((int64_t *)p)[k] = s.i; break;
        case TC_UINT8:  ((uint8_t *)p)[k] = (uint8_t)s.u; break;
        case TC_UINT16: ((uint16_t *)p)[k] = (uint16_t)s.u; break;
        case TC_UINT32: ((uint32_t *)p)[k] = (uint32_t)s.u; break;
        case TC_UINT64: ((uint64_t *)p)[k] = s.u; break;
        case TC_FP32:   ((float *)p)[k] = (float)s.d; break;
        case TC_FP64:   ((double *)p)[k] = s.d; break;
    }
}

// float -> integer conversion as GraphBLAS defines it (NaN -> 0, saturate, truncate).
__host__ __device__ static inline int64_t sat_i64(double d, int64_t lo, int64_t hi) {
    if (d != d) return 0;
    if (d <= (double)lo) return lo;
    if (d >= (double)hi) return hi;
    return (int64_t)d;
}
__host__ __device__ static inline uint64_t sat_u64(double d, uint64_t hi) {
    if (d != d) return 0;
    if (d <= 0.0) return 0;
    if (d >= (double)hi) return hi;
    return (uint64_t)d;
}

// C-style typecast between builtin types, on the carrier.
__host__ __device__ static inline Sc sc_cast(Sc x, int from, int to) {
    if (from == to) return x;
    Sc r; r.u = 0;
    const bool ff = tc_is_float(from), fs = tc_is_signed(from);
    if (to == TC_BOOL) { r.u = ff ? (x.d != 0.0) : (x.u != 0); return r; }
    if (to == TC_FP64) { r.d = ff ? x.d : (fs ? (double)x.i : (double)x.u); return r; }
    if (to == TC_FP32) { r.d = ff ? (double)(float)x.d : (fs ? (double)(float)x.i : (double)(float)x.u); return r; }
    if (ff) {
        switch (to) {
            case TC_INT8:   r.i = sat_i64(x.d, INT8_MIN, INT8_MAX); break;
            case TC_INT16:  r.i = sat_i64(x.d, INT16_MIN, INT16_MAX); break;
            case TC_INT32:  r.i = sat_i64(x.d, INT32_MIN, INT32_MAX); break;
            case TC_INT64:  r.i = sat_i64(x.d, INT64_MIN, INT64_MAX); break;
            case TC_UINT8:  r.u = sat_u64(x.d, UINT8_MAX); break;
            case TC_UINT16: r.u = sat_u64(x.d, UINT16_MAX); break;
            case TC_UINT32: r.u = sat_u64(x.d, UINT32_MAX); break;
            case TC_UINT64: r.u = sat_u64(x.d, UINT64_MAX); break;
        }
        return r;
    }
    // integer/bool -> integer: modular truncation, then sign- or zero-extension
    switch (to) {
        case TC_INT8:   r.i = (int8_t)x.u; break;
        case TC_INT16:  r.i = (int16_t)x.u; break;
        case TC_INT32:  r.i = (int32_t)x.u; break;
        case TC_INT64:  r.i = (int64_t)x.u; break;
        case TC_UINT8:  r.u = (uint8_t)x.u; break;
        case TC_UINT16: r.u = (uint16_t)x.u; break;
        case TC_UINT32: r.u = (uint32_t)x.u; break;
        case TC_UINT64: r.u = x.u; break;
    }
    return r;
}

// ---------------------------------------------------------------- typed operators
template <typename T> struct TypeOf;
template <> struct TypeOf<bool>     { static constexpr int code = TC_BOOL; };
template <> struct TypeOf<int8_t>   { static constexpr int code = TC_INT8; };
template <> struct TypeOf<int16_t>  { static constexpr int code = TC_INT16; };
template <> struct TypeOf<int32_t>  { static constexpr int code = TC_INT32; };
template <> struct TypeOf<int64_t>  { static constexpr int code = TC_INT64; };
template <> struct TypeOf<uint8_t>  { static constexpr int code = TC_UINT8; };
template <> struct TypeOf<uint16_t> { static constexpr int code = TC_UINT16; };
template <> struct TypeOf<uint32_t> { static constexpr int code = TC_UINT32; };
template <> struct TypeOf<uint64_t> { static constexpr int code = TC_UINT64; };
template <> struct TypeOf<float>    { static constexpr int code = TC_FP32; };
template <> struct TypeOf<double>   { static constexpr int code = TC_FP64; };

template <typename T> struct NumTraits {
    static constexpr bool is_float = false;
    static constexpr bool is_signed = ((T)-1) < (T)0;
    __host__ __device__ static inline T maxv() {
        return is_signed ? (T)((((uint64_t)1) << (sizeof(T) * 8 - 1)) - 1) : (T)~(T)0;
    }
    __host__ __device__ static inline T minv() {
        return is_signed ? (T)(((uint64_t)1) << (sizeof(T) * 8 - 1)) : (T)0;
    }
};
template <> struct NumTraits<float> {
    static constexpr bool is_float = true; static constexpr bool is_signed = true;
    __host__ __device__ static inline float maxv() { return INFINITY; }
    __host__ __device__ static inline float minv() { return -INFINITY; }
};
template <> struct NumTraits<double> {
    static constexpr bool is_float = true; static constexpr bool is_signed = true;
    __host__ __device__ static inline double maxv() { return (double)INFINITY; }
    __host__ __device__ static inline double minv() { return -(double)INFINITY; }
};

template <typename T> struct UnsignedOf { typedef T type; };
template <> struct UnsignedOf<int8_t>  { typedef uint8_t type; };
template <> struct UnsignedOf<int16_t> { typedef uint16_t type; };
template <> struct UnsignedOf<int32_t> { typedef uint32_t type; };
template <> struct UnsignedOf<int64_t> { typedef uint64_t type; };

template <typename T> __host__ __device__ static inline T t_from_double(double d) {
    if (NumTraits<T>::is_float) return (T)d;
    if (NumTraits<T>::is_signed) return (T)sat_i64(d, (int64_t)NumTraits<T>::minv(), (int64_t)NumTraits<T>::maxv());
    return (T)sat_u64(d, (uint64_t)NumTraits<T>::maxv());
}

// integer division with GraphBLAS' defined results for x/0 and INT_MIN/-1
template <typename T> __host__ __device__ static inline T int_div(T x, T y) {
    if constexpr (NumTraits<T>::is_signed) {
        if (y == (T)-1) return (T)(0 - (typename UnsignedOf<T>::type)x);
        if (y == 0) return x == 0 ? (T)0 : (x < 0 ? NumTraits<T>::minv() : NumTraits<T>::maxv());
        return (T)(x / y);
    } else {
        if (y == 0) return x == 0 ? (T)0 : NumTraits<T>::maxv();
        return (T)(x / y);
    }
}

// z = op(x, y) with z of the operand type T (arithmetic, logical and IS* operators).
template <typename T> __host__ __device__ __forceinline__ T op_apply(int op, T x, T y) {
    typedef typename UnsignedOf<T>::type U;
    constexpr bool F = NumTraits<T>::is_float;
    switch (op) {
        case OP_FIRST:  return x;
        case OP_SECOND: return y;
        case OP_ANY:    return y;
        case OP_PAIR:   return (T)1;
        case OP_MIN:    if (F) return (T)fmin((double)x, (double)y); return x < y ? x : y;
        case OP_MAX:    if (F) return (T)fmax((double)x, (double)y); return x > y ? x : y;
        case OP_PLUS:   if (F) return x + y; return (T)((U)x + (U)y);
        case OP_MINUS:  if (F) return x - y; return (T)((U)x - (U)y);
        case OP_RMINUS: if (F) return y - x; return (T)((U)y - (U)x);
        case OP_TIMES:  if (F) return x * y; return (T)((U)x * (U)y);
        case OP_DIV:    if constexpr (F) return x / y; else return int_div<T>(x, y);
        case OP_RDIV:   if constexpr (F) return y / x; else return int_div<T>(y, x);
        case OP_POW:    return t_from_double<T>(pow((double)x, (double)y));
        case OP_ISEQ:   return (T)(x == y);
        case OP_ISNE:   return (T)(x != y);
        case OP_ISGT:   return (T)(x > y);
        case OP_ISLT:   return (T)(x < y);
        case OP_ISGE:   return (T)(x >= y);
        case OP_ISLE:   return (T)(x <= y);
        case OP_LOR:    return (T)((x != 0) || (y != 0));
        case OP_LAND:   return (T)((x != 0) && (y != 0));
        case OP_LXOR:   return (T)((x != 0) != (y != 0));
        case OP_BOR:    if constexpr (F) return x; else return (T)((U)x | (U)y);
        case OP_BAND:   if constexpr (F) return x; else return (T)((U)x & (U)y);
        case OP_BXOR:   if constexpr (F) return x; else return (T)((U)x ^ (U)y);
        case OP_BXNOR:  if constexpr (F) return x; else return (T)~((U)x ^ (U)y);
        default:        return x;
    }
}
template <> __host__ __device__ __forceinline__ float op_apply<float>(int op, float x, float y) {
    switch (op) {
        case OP_FIRST: return x;
        case OP_SECOND: case OP_ANY: return y;
        case OP_PAIR:   return 1.0f;
        case OP_MIN:    return fminf(x, y);
        case OP_MAX:    return fmaxf(x, y);
        case OP_PLUS:   return x + y;
        case OP_MINUS:  return x - y;
        case OP_RMINUS: return y - x;
        case OP_TIMES:  return x * y;
        case OP_DIV:    return x / y;
        case OP_RDIV:   return y / x;
        case OP_POW:    return powf(x, y);
        case OP_ISEQ:   return (float)(x == y);
        case OP_ISNE:   return (float)(x != y);
        case OP_ISGT:   return (float)(x > y);
        case OP_ISLT:   return (float)(x < y);
        case OP_ISGE:   return (float)(x >= y);
        case OP_ISLE:   return (float)(x <= y);
        case OP_LOR:    return (float)((x != 0) || (y != 0));
        case OP_LAND:   return (float)((x != 0) && (y != 0));
        case OP_LXOR:   return (float)((x != 0) != (y != 0));
        default:        return x;
    }
}
// BOOL: arithmetic names alias logical ones (PLUS=LOR, TIMES=LAND, MIN=LAND, MAX=LOR, MINUS=LXOR, DIV=FIRST ...)
template <> __host__ __device__ __forceinline__ bool op_apply<bool>(int op, bool x, bool y) {
    switch (op) {
        case OP_FIRST: case OP_DIV: return x;
        case OP_SECOND: case OP_RDIV: case OP_ANY: return y;
        case OP_PAIR:   return true;
        case OP_MIN: case OP_TIMES: case OP_LAND: return x && y;
        case OP_MAX: case OP_PLUS: case OP_LOR: return x || y;
        case OP_MINUS: case OP_RMINUS: case OP_LXOR: case OP_ISNE: return x != y;
        case OP_POW:    return x || !y;
        case OP_ISEQ:   return x == y;
        case OP_ISGT:   return x && !y;
        case OP_ISLT:   return !x && y;
        case OP_ISGE:   return x || !y;
        case OP_ISLE:   return !x || y;
        default:        return x;
    }
}
// z = cmp(x, y), z BOOL
template <typename T> __host__ __device__ __forceinline__ bool cmp_apply(int op, T x, T y) {
    switch (op) {
        case OP_EQ: return x == y;
        case OP_NE: return x != y;
        case OP_GT: return x > y;
        case OP_LT: return x < y;
        case OP_GE: return x >= y;
        case OP_LE: return x <= y;
        default:    return false;
    }
}
// multiply of a semiring: ZT == XT for arithmetic operators, ZT == bool for comparisons
template <typename XT, typename ZT> struct MulApply {
    __host__ __device__ static __forceinline__ ZT f(int op, XT a, XT b) { return (ZT)cmp_apply<XT>(op, a, b); }
};
template <typename T> struct MulApply<T, T> {
    __host__ __device__ static __forceinline__ T f(int op, T a, T b) {
        if (op >= OP_EQ && op <= OP_LE) return (T)cmp_apply<T>(op, a, b);
        return op_apply<T>(op, a, b);
    }
};

// identity / terminal value of a monoid operator on type T
template <typename T> __host__ __device__ static inline T monoid_identity(int op) {
    switch (op) {
        case OP_MIN:   return NumTraits<T>::maxv();
        case OP_MAX:   return NumTraits<T>::minv();
        case OP_TIMES: return (T)1;
        case OP_LAND:  return (T)1;
        case OP_EQ:    return (T)1;
        case OP_BAND: case OP_BXNOR: return (T)~(uint64_t)0;
        default:       return (T)0;   // PLUS, LOR, LXOR, ANY, BOR, BXOR
    }
}
template <> __host__ __device__ inline bool monoid_identity<bool>(int op) {
    switch (op) {
        case OP_MIN: case OP_TIMES: case OP_LAND: case OP_EQ: return true;
        default: return false;
    }
}
template <> __host__ __device__ inline float monoid_identity<float>(int op) {
    switch (op) { case OP_MIN: return INFINITY; case OP_MAX: return -INFINITY;
                  case OP_TIMES: case OP_LAND: case OP_EQ: return 1.0f; default: return 0.0f; }
}
template <> __host__ __device__ inline double monoid_identity<double>(int op) {
    switch (op) { case OP_MIN: return (double)INFINITY; case OP_MAX: return -(double)INFINITY;
                  case OP_TIMES: case OP_LAND: case OP_EQ: return 1.0; default: return 0.0; }
}

// carrier-level operator: x, y, z all of the operator's type `tc` (z BOOL for comparisons)
__host__ __device__ static inline Sc sc_binop(int op, int tc, Sc x, Sc y) {
    Sc r; r.u = 0;
#define GB_CASE(TC, T, FIELD) case TC: { T a = (T)x.FIELD, b = (T)y.FIELD; \
        if (op >= OP_EQ && op <= OP_LE) r.u = cmp_apply<T>(op, a, b); \
        else { T z = op_apply<T>(op, a, b); Sc t; t.u = 0; t.FIELD = z; r = t; } } break;
    switch (tc) {
        case TC_BOOL: { bool a = x.u != 0, b = y.u != 0;
            if (op >= OP_EQ && op <= OP_LE) r.u = cmp_apply<bool>(op, a, b); else r.u = op_apply<bool>(op, a, b); } break;
        GB_CASE(TC_INT8, int8_t, i) GB_CASE(TC_INT16, int16_t, i) GB_CASE(TC_INT32, int32_t, i) GB_CASE(TC_INT64, int64_t, i)
        GB_CASE(TC_UINT8, uint8_t, u) GB_CASE(TC_UINT16, uint16_t, u) GB_CASE(TC_UINT32, uint32_t, u) GB_CASE(TC_UINT64, uint64_t, u)
        case TC_FP32: { float a = (float)x.d, b = (float)y.d;
            if (op >= OP_EQ && op <= OP_LE) r.u = cmp_apply<float>(op, a, b); else r.d = (double)op_apply<float>(op, a, b); } break;
        case TC_FP64: { double a = x.d, b = y.d;
            if (op >= OP_EQ && op <= OP_LE) r.u = cmp_apply<double>(op, a, b); else r.d = op_apply<double>(op, a, b); } break;
    }
#undef GB_CASE
    return r;
}

// carrier-level unary operator: x of type `tc`; z of type `tc` (BOOL for ISINF / ISNAN / ISFINITE)
template <typename T> __host__ __device__ static inline T uop_apply(int op, T x) {
    typedef typename UnsignedOf<T>::type U;
    constexpr bool F = NumTraits<T>::is_float;
    switch (op) {
        case UOP_IDENTITY: return x;
        case UOP_AINV: if (F) return -x; return (T)((U)0 - (U)x);
        case UOP_MINV: if constexpr (F) return (T)1 / x; else return int_div<T>((T)1, x);
        case UOP_LNOT: return (T)!(x != (T)0);
        case UOP_ONE:  return (T)1;
        case UOP_ABS:  if constexpr (F) return (T)fabs((double)x); else if constexpr (NumTraits<T>::is_signed) return x < 0 ? (T)((U)0 - (U)x) : x; else return x;
        case UOP_BNOT: if constexpr (F) return x; else return (T)~(U)x;
        default: break;
    }
    if constexpr (F) {
        const double d = (double)x;
        switch (op) {
            case UOP_SQRT: return (T)sqrt(d);   case UOP_LOG: return (T)log(d);     case UOP_EXP: return (T)exp(d);
            case UOP_LOG2: return (T)log2(d);   case UOP_SIN: return (T)sin(d);     case UOP_COS: return (T)cos(d);
            case UOP_TAN: return (T)tan(d);     case UOP_ACOS: return (T)acos(d);   case UOP_ASIN: return (T)asin(d);
            case UOP_ATAN: return (T)atan(d);   case UOP_SINH: return (T)sinh(d);   case UOP_COSH: return (T)cosh(d);
            case UOP_TANH: return (T)tanh(d);   case UOP_ACOSH: return (T)acosh(d); case UOP_ASINH: return (T)asinh(d);
            case UOP_ATANH: return (T)atanh(d); case UOP_SIGNUM: return (T)(d != d ? d : (d > 0) - (d < 0));
            case UOP_CEIL: return (T)ceil(d);   case UOP_FLOOR: return (T)floor(d); case UOP_ROUND: return (T)round(d);
            case UOP_TRUNC: return (T)trunc(d); case UOP_EXP2: return (T)exp2(d);   case UOP_EXPM1: return (T)expm1(d);
            case UOP_LOG10: return (T)log10(d); case UOP_LOG1P: return (T)log1p(d); case UOP_LGAMMA: return (T)lgamma(d);
            case UOP_TGAMMA: return (T)tgamma(d); case UOP_ERF: return (T)erf(d);   case UOP_ERFC: return (T)erfc(d);
            default: break;
        }
    }
    return x;
}
__host__ __device__ static inline Sc sc_unop(int op, int tc, Sc x) {
    Sc r; r.u = 0;
    if (op >= UOP_ISINF && op <= UOP_ISFINITE) {
        const double d = tc == TC_FP32 ? (double)(float)x.d : x.d;
        const bool inf = d == (double)INFINITY || d == -(double)INFINITY, nan = d != d;
        r.u = op == UOP_ISINF ? inf : (op == UOP_ISNAN ? nan : (!inf && !nan));
        return r;
    }
#define GB_CASE(TC, T, FIELD) case TC: { Sc t; t.u = 0; t.FIELD = uop_apply<T>(op, (T)x.FIELD); r = t; } break;
    switch (tc) {
        case TC_BOOL: r.u = uop_apply<bool>(op, x.u != 0); break;
        GB_CASE(TC_INT8, int8_t, i) GB_CASE(TC_INT16, int16_t, i) GB_CASE(TC_INT32, int32_t, i) GB_CASE(TC_INT64, int64_t, i)
        GB_CASE(TC_UINT8, uint8_t, u) GB_CASE(TC_UINT16, uint16_t, u) GB_CASE(TC_UINT32, uint32_t, u) GB_CASE(TC_UINT64, uint64_t, u)
        case TC_FP32: r.d = (double)uop_apply<float>(op, (float)x.d); break;
        case TC_FP64: r.d = uop_apply<double>(op, x.d); break;
    }
#undef GB_CASE
    return r;
}
// identity of a builtin monoid operator, on the carrier (same table the kernels use)
__host__ __device__ static inline Sc sc_monoid_identity(int op, int tc) {
    Sc acc; acc.u = 0;
    switch (tc) {
#define GB_ID(TC, T, F) case TC: { Sc t; t.u = 0; t.F = monoid_identity<T>(op); acc = t; } break;
        case TC_BOOL: acc.u = monoid_identity<bool>(op); break;
        GB_ID(TC_INT8, int8_t, i) GB_ID(TC_INT16, int16_t, i) GB_ID(TC_INT32, int32_t, i) GB_ID(TC_INT64, int64_t, i)
        GB_ID(TC_UINT8, uint8_t, u) GB_ID(TC_UINT16, uint16_t, u) GB_ID(TC_UINT32, uint32_t, u) GB_ID(TC_UINT64, uint64_t, u)
        case TC_FP32: acc.d = (double)monoid_identity<float>(op); break;
        case TC_FP64: acc.d = monoid_identity<double>(op); break;
#undef GB_ID
    }
    return acc;
}

// value of a mask entry as a truth value (any builtin type), without the carrier
__host__ __device__ static inline bool mask_value_true(int mtc, const void *mval, int64_t i) {
    switch (mtc) {
        case TC_FP32: return ((const float *)mval)[i] != 0.0f;
        case TC_FP64: return ((const double *)mval)[i] != 0.0;
        default: break;
    }
    switch (tc_size(mtc)) {
        case 1: return ((const uint8_t *)mval)[i] != 0;
        case 2: return ((const uint16_t *)mval)[i] != 0;
        case 4: return ((const uint32_t *)mval)[i] != 0;
        default: return ((const uint64_t *)mval)[i] != 0;
    }
}

// ---------------------------------------------------------------- launch helpers
__host__ __device__ static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
#define GB_LAUNCHED() (G.launches++)
