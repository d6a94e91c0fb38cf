// objects.cu -- host side of libb200grb: lifecycle, types, operator tables,
// descriptors, and the Matrix / Vector containers with their host<->HBM duality.
//
// Containers keep two interchangeable forms:
//   host   sorted unique tuples (+ a list of pending setElement calls), the form
//          the element-wise plumbing of the reference works on
//          (/root/reference/pygraphblas/matrix.py:3279-3282 setElement loop,
//           matrix.py:1467-1492 extractTuples);
//   HBM    CSR with 32-bit column indices (matrices) / dense values + presence
//          bytes (vectors): what the sm_100a kernels consume and produce.
// Either may be stale; *_ensure_host / *_ensure_device bring one up to date.
#include "common.cuh"
#include <stdarg.h>
#include <string.h>
#include <stdlib.h>
#include <algorithm>
#include <numeric>
#include <unordered_map>
#include <nvtx3/nvToolsExt.h>

GBGlobal G;
thread_local std::string tl_error;

GrB_Info gb_fail(GrB_Info code, std::string *where, const char *fmt, ...) {
    char buf[1024];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    tl_error = buf;
    if (where) *where = buf;
    return code;
}

extern "C" const char *B200_last_error(void) { return tl_error.c_str(); }

// ------------------------------------------------------------------ tunables, burble, NVTX
static Tunables g_tun; static bool g_tun_loaded = false;
static void tunables_load() {
    Tunables t;
    auto geti = [](const char *k, int d) { const char *e = getenv(k); return e ? atoi(e) : d; };
    t.spmv_items = geti("B200GRB_SPMV_ITEMS", 8);
    t.spmv_run = geti("B200GRB_SPMV_RUN", -1);
    t.spmv_hot_kb = geti("B200GRB_SPMV_HOT", -1);
    t.no_pull = getenv("B200GRB_NO_PULL") != nullptr; t.no_push = getenv("B200GRB_NO_PUSH") != nullptr;
    t.force_push = getenv("B200GRB_FORCE_PUSH") != nullptr; t.spmv_debug = getenv("B200GRB_SPMV_DEBUG") != nullptr;
    t.spmv_pipe = geti("B200GRB_SPMV_PIPE", 0) != 0;
    t.spgemm_trace = getenv("B200GRB_SPGEMM_TRACE") != nullptr;
    t.stream_blk_log2 = std::min(12, std::max(7, geti("B200GRB_STREAM_BLK", 7)));
    t.spgemm_v = geti("B200GRB_SPGEMM_V", 0);
    t.mxv_inplace = geti("B200GRB_MXV_INPLACE", 1);
    t.spgemm_esc = geti("B200GRB_SPGEMM_ESC", 1) != 0;
    g_tun = t; g_tun_loaded = true;
}
const Tunables &tunables() { if (!g_tun_loaded) tunables_load(); return g_tun; }
extern "C" GrB_Info B200_reload_tunables(void) { GB_LOCK; tunables_load(); return GrB_SUCCESS; }

GbBurble::GbBurble(const char *f) : on(G.burble != 0 && G.have_device), fn(f) {
    nvtxRangePushA(f);
    if (on) {
        if (!G.burble_e0) { cudaEventCreate(&G.burble_e0); cudaEventCreate(&G.burble_e1); }
        cudaEventRecord(G.burble_e0, G.stream);
    }
}
GbBurble::~GbBurble() {
    if (on) {
        cudaEventRecord(G.burble_e1, G.stream);
        float ms = 0.f;
        if (cudaEventSynchronize(G.burble_e1) == cudaSuccess && cudaEventElapsedTime(&ms, G.burble_e0, G.burble_e1) == cudaSuccess) {
            const double us = ms * 1e3;
            printf(" [ B200 %s: kernel %s, %.3f MB algorithmic, %.1f us on the device", fn, kernel, bytes / 1e6, us);
            if (us > 0 && bytes > 0) printf(", %.1f GB/s", bytes / (us * 1e-6) / 1e9);
            printf(" ]\n"); fflush(stdout);
        }
    }
    nvtxRangePop();
}
extern "C" void B200_set_burble(int on) { G.burble = on; }
extern "C" int B200_get_burble(void) { return G.burble; }

// ------------------------------------------------------------------ types
static GB_Type_opaque type_BOOL   = {GB_MAGIC, TC_BOOL, 1, "BOOL"};
static GB_Type_opaque type_INT8   = {GB_MAGIC, TC_INT8, 1, "INT8"};
static GB_Type_opaque type_INT16  = {GB_MAGIC, TC_INT16, 2, "INT16"};
static GB_Type_opaque type_INT32  = {GB_MAGIC, TC_INT32, 4, "INT32"};
static GB_Type_opaque type_INT64  = {GB_MAGIC, TC_INT64, 8, "INT64"};
static GB_Type_opaque type_UINT8  = {GB_MAGIC, TC_UINT8, 1, "UINT8"};
static GB_Type_opaque type_UINT16 = {GB_MAGIC, TC_UINT16, 2, "UINT16"};
static GB_Type_opaque type_UINT32 = {GB_MAGIC, TC_UINT32, 4, "UINT32"};
static GB_Type_opaque type_UINT64 = {GB_MAGIC, TC_UINT64, 8, "UINT64"};
static GB_Type_opaque type_FP32   = {GB_MAGIC, TC_FP32, 4, "FP32"};
static GB_Type_opaque type_FP64   = {GB_MAGIC, TC_FP64, 8, "FP64"};

extern "C" {
GrB_Type GrB_BOOL = &type_BOOL, GrB_INT8 = &type_INT8, GrB_INT16 = &type_INT16, GrB_INT32 = &type_INT32,
         GrB_INT64 = &type_INT64, GrB_UINT8 = &type_UINT8, GrB_UINT16 = &type_UINT16,
         GrB_UINT32 = &type_UINT32, GrB_UINT64 = &type_UINT64, GrB_FP32 = &type_FP32, GrB_FP64 = &type_FP64;

#include "ops_table.inc"
}

static inline bool valid_type(GrB_Type t) { return t && t->magic == GB_MAGIC; }

extern "C" GrB_Info GxB_Type_size(size_t *size, GrB_Type type) {
    if (!size || !type) return gb_fail(GrB_NULL_POINTER, nullptr, "GxB_Type_size: NULL argument");
    *size = type->size; return GrB_SUCCESS;
}
extern "C" GrB_Info B200_Type_info(const char **name, int *code, GrB_Type type) {
    if (!valid_type(type)) return gb_fail(GrB_NULL_POINTER, nullptr, "B200_Type_info: invalid type");
    if (name) *name = type->name;
    if (code) *code = type->code;
    return GrB_SUCCESS;
}

// ------------------------------------------------------------------ lifecycle
extern "C" int B200_have_device(void) { return G.have_device ? 1 : 0; }
extern "C" uint64_t B200_kernel_launches(void) { return G.launches; }
extern "C" GrB_Info B200_last_mxm_stats(uint64_t *flops, uint64_t *nnz_out) {
    if (flops) *flops = G.last_flops;
    if (nnz_out) *nnz_out = G.last_nnz_out;
    return GrB_SUCCESS;
}

extern "C" GrB_Info GrB_init(GrB_Mode mode) {
    GB_LOCK;
    (void)mode;
    if (G.initialized) return GrB_SUCCESS;   // tolerate re-init (the reference guards with is_initialized)
    G.initialized = true;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) { cudaGetLastError(); G.have_device = false; return GrB_SUCCESS; }
    int dev = 0;
    const char *env = getenv("B200GRB_DEVICE");
    const char *lr = getenv("LOCAL_RANK");
    if (env) dev = atoi(env); else if (lr) dev = atoi(lr) % ndev;
    if (cudaSetDevice(dev) != cudaSuccess) { cudaGetLastError(); G.have_device = false; return GrB_SUCCESS; }
    G.device = dev;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) { cudaGetLastError(); return GrB_SUCCESS; }
    G.num_sms = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&G.stream, cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); return GrB_SUCCESS; }
    // keep freed blocks in the stream-ordered pool instead of returning them to the driver
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        uint64_t thr = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    G.have_device = true;
    tunables_load();
    return GrB_SUCCESS;
}

extern "C" GrB_Info GrB_finalize(void) {
    GB_LOCK;
    if (G.have_device && G.stream) { cudaStreamSynchronize(G.stream); }
    return GrB_SUCCESS;
}

extern "C" GrB_Info B200_get_stream(void **stream) {
    if (!stream) return gb_fail(GrB_NULL_POINTER, nullptr, "B200_get_stream: NULL");
    *stream = (void *)G.stream; return GrB_SUCCESS;
}
extern "C" GrB_Info B200_device_synchronize(void) {
    GB_LOCK;
    if (!G.have_device) return GrB_SUCCESS;
    CU_TRY(cudaStreamSynchronize(G.stream), nullptr);
    if (G.h2d) { CU_TRY(cudaStreamSynchronize(G.h2d), nullptr); CU_TRY(cudaStreamSynchronize(G.d2h), nullptr); }
    return GrB_SUCCESS;
}

GrB_Info dmalloc(void **p, size_t bytes, std::string *err) {
    *p = nullptr;
    if (!G.have_device) return gb_fail(GrB_PANIC, err, "no CUDA device: libb200grb computes only on the GPU (no CPU fallback)");
    if (bytes == 0) bytes = 16;
    bytes = (bytes + 255) & ~(size_t)255;
    CU_TRY(cudaMallocAsync(p, bytes, G.stream), err);
    return GrB_SUCCESS;
}
void dfree(void *p) { if (p && G.have_device) cudaFreeAsync(p, G.stream); }

static void *g_ws[WS_COUNT]; static size_t g_ws_cap[WS_COUNT];
GrB_Info ws_get(int slot, void **p, size_t bytes, std::string *err, bool *fresh) {
    if (fresh) *fresh = false;
    if (g_ws_cap[slot] < bytes) {
        dfree(g_ws[slot]); g_ws[slot] = nullptr; g_ws_cap[slot] = 0;
        const size_t cap = bytes + bytes / 4 + 256;
        GB_TRY(dmalloc(&g_ws[slot], cap, err));
        g_ws_cap[slot] = cap;
        if (fresh) *fresh = true;
    }
    *p = g_ws[slot];
    return GrB_SUCCESS;
}

// the cached SpMV plans and scratch of a CSR (dropped whenever its structure changes)
void csr_drop_plans(Csr &c) {
    dfree(c.tile_row); c.tile_row = nullptr; c.ntiles = 0; c.tile_size = 0;
    dfree(c.hperm); dfree(c.hcol); c.hperm = nullptr; c.hcol = nullptr; c.henc = 0; c.hot_planned = false; c.hot_cover = 0.0;
    dfree(c.run_headw); dfree(c.run_lane); dfree(c.run_base); dfree(c.run_fix); dfree(c.nzrow); dfree(c.pres_tmpl);
    c.run_headw = nullptr; c.run_lane = nullptr; c.run_base = nullptr; c.run_fix = nullptr; c.run_fix_long = c.run_fix_short = 0; c.nzrow = nullptr; c.pres_tmpl = nullptr;
    c.nruns = 0; c.nnzrows = 0;
    dfree(c.ws_head); dfree(c.ws_tail); dfree(c.ws_head_has); dfree(c.ws_tail_has); dfree(c.ws_uhot);
    c.ws_head = c.ws_tail = c.ws_uhot = nullptr; c.ws_head_has = c.ws_tail_has = nullptr;
}
void csr_free(Csr &c) {
    csr_drop_plans(c);
    dfree(c.rowptr); dfree(c.rowptr32); dfree(c.col); dfree(c.val);
    c = Csr();
}

// ------------------------------------------------------------------ operators
static inline bool valid_binop(GrB_BinaryOp o) { return o && o->magic == GB_MAGIC; }
static inline bool valid_monoid(GrB_Monoid o) { return o && o->magic == GB_MAGIC; }
static inline bool valid_semiring(GrB_Semiring o) { return o && o->magic == GB_MAGIC; }

extern "C" GrB_Info GrB_BinaryOp_new(GrB_BinaryOp *op, GxB_binary_function fn, GrB_Type z, GrB_Type x, GrB_Type y) {
    if (!op || !fn) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_BinaryOp_new: NULL argument");
    if (!valid_type(z) || !valid_type(x) || !valid_type(y)) return gb_fail(GrB_UNINITIALIZED_OBJECT, nullptr, "GrB_BinaryOp_new: bad type");
    // The object can be created, but a host function pointer cannot run inside a GPU
    // kernel: any operation given this operator is refused (no CPU fallback).
    GB_BinaryOp_opaque *o = new GB_BinaryOp_opaque{GB_MAGIC, OP_USER, x, y, z, "user_binaryop", (void *)fn};
    *op = o; return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_BinaryOp_free(GrB_BinaryOp *op) {
    if (!op || !*op) return GrB_SUCCESS;
    if ((*op)->opcode == OP_USER && (*op)->magic == GB_MAGIC) { (*op)->magic = GB_FREED; delete *op; }
    *op = nullptr; return GrB_SUCCESS;
}
extern "C" GrB_Info GxB_BinaryOp_ztype(GrB_Type *t, GrB_BinaryOp op) {
    if (!t) return gb_fail(GrB_NULL_POINTER, nullptr, "NULL"); if (!valid_binop(op)) return gb_fail(GrB_UNINITIALIZED_OBJECT, nullptr, "bad binaryop");
    *t = op->ztype; return GrB_SUCCESS;
}
extern "C" GrB_Info GxB_BinaryOp_xtype(GrB_Type *t, GrB_BinaryOp op) {
    if (!t) return gb_fail(GrB_NULL_POINTER, nullptr, "NULL"); if (!valid_binop(op)) return gb_fail(GrB_UNINITIALIZED_OBJECT, nullptr, "bad binaryop");
    *t = op->xtype; return GrB_SUCCESS;
}
extern "C" GrB_Info GxB_BinaryOp_ytype(GrB_Type *t, GrB_BinaryOp op) {
    if (!t) return gb_fail(GrB_NULL_POINTER, nullptr, "NULL"); if (!valid_binop(op)) return gb_fail(GrB_UNINITIALIZED_OBJECT, nullptr, "bad binaryop");
    *t = op->ytype; return GrB_SUCCESS;
}
// A monoid over a builtin operator must be one the kernels know the identity of: the associative, commutative builtin operators.
// The identity the caller passes has to be that identity (the kernels initialise accumulators from the operator, not from the object).
static bool op_is_monoid(int opcode, int tc) {
    switch (opcode) {
        case OP_MIN: case OP_MAX: case OP_PLUS: case OP_TIMES: case OP_ANY: return true;
        case OP_LOR: case OP_LAND: case OP_LXOR: case OP_EQ: return tc == TC_BOOL;
        case OP_BOR: case OP_BAND: case OP_BXOR: case OP_BXNOR: return tc >= TC_UINT8 && tc <= TC_UINT64;
        default: return false;
    }
}
static GrB_Info monoid_new(GrB_Monoid *m, GrB_BinaryOp op, Sc identity) {
    if (!m) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Monoid_new: NULL");
    if (!valid_binop(op)) return gb_fail(GrB_UNINITIALIZED_OBJECT, nullptr, "GrB_Monoid_new: bad operator");
    if (op->xtype != op->ztype || op->ytype != op->ztype) return gb_fail(GrB_DOMAIN_MISMATCH, nullptr, "GrB_Monoid_new: operator domains must all match");
    if (op->opcode != OP_USER) {
        const int tc = op->ztype->code;
        if (!op_is_monoid(op->opcode, tc)) return gb_fail(GrB_DOMAIN_MISMATCH, nullptr, "GrB_Monoid_new: %s is not an associative, commutative builtin operator with an identity", op->name);
        if (op->opcode != OP_ANY) {
            const Sc want = sc_monoid_identity(op->opcode, tc);
            const bool same = tc_is_float(tc) ? (want.d == identity.d) : (want.u == identity.u);
            if (!same) return gb_fail(GrB_INVALID_VALUE, nullptr, "GrB_Monoid_new: the identity passed is not the identity of %s", op->name);
        }
    }
    *m = new GB_Monoid_opaque{GB_MAGIC, op, "user_monoid", false};
    return GrB_SUCCESS;
}
#define GB_MONOID_NEW(TN, CT, FIELD) extern "C" GrB_Info GrB_Monoid_new_##TN(GrB_Monoid *m, GrB_BinaryOp op, CT identity) { \
    Sc s; s.u = 0; s.FIELD = identity; return monoid_new(m, op, s); }
GB_MONOID_NEW(BOOL, bool, u) GB_MONOID_NEW(INT8, int8_t, i) GB_MONOID_NEW(INT16, int16_t, i) GB_MONOID_NEW(INT32, int32_t, i)
GB_MONOID_NEW(INT64, int64_t, i) GB_MONOID_NEW(UINT8, uint8_t, u) GB_MONOID_NEW(UINT16, uint16_t, u) GB_MONOID_NEW(UINT32, uint32_t, u)
GB_MONOID_NEW(UINT64, uint64_t, u) GB_MONOID_NEW(FP32, float, d) GB_MONOID_NEW(FP64, double, d)

extern "C" GrB_Info GrB_Monoid_free(GrB_Monoid *m) {
    if (!m || !*m) return GrB_SUCCESS;
    if (!(*m)->builtin && (*m)->magic == GB_MAGIC) { (*m)->magic = GB_FREED; delete *m; }
    *m = nullptr; return GrB_SUCCESS;
}
extern "C" GrB_Info GxB_Monoid_operator(GrB_BinaryOp *op, GrB_Monoid m) {
    if (!op) return gb_fail(GrB_NULL_POINTER, nullptr, "NULL"); if (!valid_monoid(m)) return gb_fail(GrB_UNINITIALIZED_OBJECT, nullptr, "bad monoid");
    *op = m->op; return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Semiring_new(GrB_Semiring *s, GrB_Monoid add, GrB_BinaryOp mul) {
    if (!s) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Semiring_new: NULL");
    if (!valid_monoid(add) || !valid_binop(mul)) return gb_fail(GrB_UNINITIALIZED_OBJECT, nullptr, "GrB_Semiring_new: bad operator");
    if (mul->ztype != add->op->ztype) return gb_fail(GrB_DOMAIN_MISMATCH, nullptr, "GrB_Semiring_new: multiply output type must match the monoid type");
    *s = new GB_Semiring_opaque{GB_MAGIC, add, mul, "user_semiring", false};
    return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Semiring_free(GrB_Semiring *s) {
    if (!s || !*s) return GrB_SUCCESS;
    if (!(*s)->builtin && (*s)->magic == GB_MAGIC) { (*s)->magic = GB_FREED; delete *s; }
    *s = nullptr; return GrB_SUCCESS;
}
extern "C" GrB_Info GxB_Semiring_add(GrB_Monoid *add, GrB_Semiring s) {
    if (!add) return gb_fail(GrB_NULL_POINTER, nullptr, "NULL"); if (!valid_semiring(s)) return gb_fail(GrB_UNINITIALIZED_OBJECT, nullptr, "bad semiring");
    *add = s->add; return GrB_SUCCESS;
}
extern "C" GrB_Info GxB_Semiring_multiply(GrB_BinaryOp *mul, GrB_Semiring s) {
    if (!mul) return gb_fail(GrB_NULL_POINTER, nullptr, "NULL"); if (!valid_semiring(s)) return gb_fail(GrB_UNINITIALIZED_OBJECT, nullptr, "bad semiring");
    *mul = s->mul; return GrB_SUCCESS;
}
extern "C" GrB_Info GxB_BinaryOp_fprint(GrB_BinaryOp op, const char *name, int pr, FILE *f) {
    if (!valid_binop(op)) return gb_fail(GrB_UNINITIALIZED_OBJECT, nullptr, "bad binaryop");
    if (pr > 0) fprintf(f ? f : stdout, "\n    B200 GraphBLAS BinaryOp: %s z=%s(x,y) : %s(%s,%s)\n", name ? name : "",
                        op->name, op->ztype->name, op->xtype->name, op->ytype->name);
    return GrB_SUCCESS;
}
extern "C" GrB_Info GxB_Monoid_fprint(GrB_Monoid m, const char *name, int pr, FILE *f) {
    if (!valid_monoid(m)) return gb_fail(GrB_UNINITIALIZED_OBJECT, nullptr, "bad monoid");
    if (pr > 0) fprintf(f ? f : stdout, "\n    B200 GraphBLAS Monoid: %s %s over %s\n", name ? name : "", m->name, m->op->ztype->name);
    return GrB_SUCCESS;
}
extern "C" GrB_Info GxB_Semiring_fprint(GrB_Semiring s, const char *name, int pr, FILE *f) {
    if (!valid_semiring(s)) return gb_fail(GrB_UNINITIALIZED_OBJECT, nullptr, "bad semiring");
    if (pr > 0) fprintf(f ? f : stdout, "\n    B200 GraphBLAS Semiring: %s %s  add: %s  multiply: %s\n", name ? name : "",
                        s->name, s->add->op->name, s->mul->name);
    return GrB_SUCCESS;
}
extern "C" GrB_Info B200_lookup(void **obj, int kind, const char *name) {
    if (!obj || !name) return gb_fail(GrB_NULL_POINTER, nullptr, "B200_lookup: NULL");
    static std::unordered_map<std::string, const GB_named *> index;
    {
        GB_LOCK;
        if (index.empty()) for (const GB_named *p = gb_named_objects; p->name; ++p) index[std::string(p->name) + "#" + std::to_string(p->kind)] = p;
    }
    auto it = index.find(std::string(name) + "#" + std::to_string(kind));
    if (it == index.end()) { *obj = nullptr; return gb_fail(GrB_INVALID_VALUE, nullptr, "B200_lookup: no builtin operator named %s", name); }
    *obj = it->second->obj; return GrB_SUCCESS;
}
extern "C" GrB_Info B200_object_name(const char **name, int kind, const void *obj) {
    if (!name || !obj) return gb_fail(GrB_NULL_POINTER, nullptr, "B200_object_name: NULL");
    switch (kind) {
        case 0: *name = ((const GB_BinaryOp_opaque *)obj)->name; break;
        case 1: *name = ((const GB_Monoid_opaque *)obj)->name; break;
        case 2: *name = ((const GB_Semiring_opaque *)obj)->name; break;
        default: return gb_fail(GrB_INVALID_VALUE, nullptr, "B200_object_name: bad kind");
    }
    return GrB_SUCCESS;
}

// ------------------------------------------------------------------ descriptors
#define D_(NAME, OUTP, MASK, I0, I1) \
    static GB_Descriptor_opaque desc_##NAME = {GB_MAGIC, OUTP, MASK, I0, I1, 0, 0, 0.0, 0, true, #NAME}; \
    extern "C" { GrB_Descriptor GrB_DESC_##NAME = &desc_##NAME; }
#define D4_(P, OUTP, MASK) D_(P##T1, OUTP, MASK, 0, GrB_TRAN) D_(P##T0, OUTP, MASK, GrB_TRAN, 0) D_(P##T0T1, OUTP, MASK, GrB_TRAN, GrB_TRAN)
D4_(, 0, 0)
D_(C, 0, GrB_COMP, 0, 0)                      D4_(C, 0, GrB_COMP)
D_(S, 0, GrB_STRUCTURE, 0, 0)                 D4_(S, 0, GrB_STRUCTURE)
D_(SC, 0, GrB_COMP + GrB_STRUCTURE, 0, 0)     D4_(SC, 0, GrB_COMP + GrB_STRUCTURE)
D_(R, GrB_REPLACE, 0, 0, 0)                   D4_(R, GrB_REPLACE, 0)
D_(RC, GrB_REPLACE, GrB_COMP, 0, 0)           D4_(RC, GrB_REPLACE, GrB_COMP)
D_(RS, GrB_REPLACE, GrB_STRUCTURE, 0, 0)      D4_(RS, GrB_REPLACE, GrB_STRUCTURE)
D_(RSC, GrB_REPLACE, GrB_COMP + GrB_STRUCTURE, 0, 0) D4_(RSC, GrB_REPLACE, GrB_COMP + GrB_STRUCTURE)

extern "C" GrB_Info GrB_Descriptor_new(GrB_Descriptor *d) {
    if (!d) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Descriptor_new: NULL");
    *d = new GB_Descriptor_opaque{GB_MAGIC, 0, 0, 0, 0, 0, 0, 0.0, 0, false, "user"};
    return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Descriptor_free(GrB_Descriptor *d) {
    // called by the reference on builtin descriptors and on a NULL one
    // (/root/reference/pygraphblas/descriptor.py:76-78,148): both are no-ops.
    if (!d || !*d) return GrB_SUCCESS;
    if (!(*d)->builtin && (*d)->magic == GB_MAGIC) { (*d)->magic = GB_FREED; delete *d; *d = nullptr; }
    return GrB_SUCCESS;
}
static GrB_Info desc_set(GrB_Descriptor d, int field, int value) {
    if (!d || d->magic != GB_MAGIC) return gb_fail(GrB_UNINITIALIZED_OBJECT, nullptr, "GrB_Descriptor_set: bad descriptor");
    if (d->builtin) return gb_fail(GrB_INVALID_VALUE, nullptr, "GrB_Descriptor_set: builtin descriptors are read-only");
    switch (field) {
        case GrB_OUTP:
            if (value != GxB_DEFAULT && value != GrB_REPLACE) return gb_fail(GrB_INVALID_VALUE, nullptr, "GrB_OUTP must be GxB_DEFAULT or GrB_REPLACE");
            d->outp = value; break;
        case GrB_MASK:
            if (value == GxB_DEFAULT) d->mask = 0;
            else if (value == GrB_COMP || value == GrB_STRUCTURE || value == GrB_COMP + GrB_STRUCTURE) d->mask |= value;
            else return gb_fail(GrB_INVALID_VALUE, nullptr, "GrB_MASK must be GxB_DEFAULT, GrB_COMP, GrB_STRUCTURE or both");
            break;
        case GrB_INP0:
            if (value != GxB_DEFAULT && value != GrB_TRAN) return gb_fail(GrB_INVALID_VALUE, nullptr, "GrB_INP0 must be GxB_DEFAULT or GrB_TRAN");
            d->inp0 = value; break;
        case GrB_INP1:
            if (value != GxB_DEFAULT && value != GrB_TRAN) return gb_fail(GrB_INVALID_VALUE, nullptr, "GrB_INP1 must be GxB_DEFAULT or GrB_TRAN");
            d->inp1 = value; break;
        case GxB_AxB_METHOD: d->axb = value; break;
        case GxB_DESCRIPTOR_NTHREADS: d->nthreads = value; break;
        case GxB_SORT: d->sort = value; break;
        case GxB_DESCRIPTOR_CHUNK: d->chunk = (double)value; break;
        default: return gb_fail(GrB_INVALID_VALUE, nullptr, "GrB_Descriptor_set: unknown field %d", field);
    }
    return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Descriptor_set(GrB_Descriptor d, GrB_Desc_Field field, GrB_Desc_Value value) { return desc_set(d, (int)field, (int)value); }
extern "C" GrB_Info GxB_Desc_set(GrB_Descriptor d, GrB_Desc_Field field, ...) {
    va_list ap; va_start(ap, field);
    GrB_Info r;
    if (field == GxB_DESCRIPTOR_CHUNK) { double c = va_arg(ap, double); r = GrB_SUCCESS; if (d && !d->builtin) d->chunk = c; }
    else { int v = va_arg(ap, int); r = desc_set(d, (int)field, v); }
    va_end(ap); return r;
}
extern "C" GrB_Info GxB_Desc_get(GrB_Descriptor d, GrB_Desc_Field field, ...) {
    va_list ap; va_start(ap, field);
    GrB_Info r = GrB_SUCCESS;
    if (field == GxB_DESCRIPTOR_CHUNK) {
        // the reference reads every field through a GrB_Desc_Value* (descriptor.py:106-109)
        int *out = va_arg(ap, int *);
        if (!out) r = gb_fail(GrB_NULL_POINTER, nullptr, "GxB_Desc_get: NULL"); else *out = d ? (int)d->chunk : 0;
    } else {
        int *out = va_arg(ap, int *);
        if (!out) r = gb_fail(GrB_NULL_POINTER, nullptr, "GxB_Desc_get: NULL");
        else if (!d) *out = GxB_DEFAULT;   // NULL descriptor: all defaults
        else switch (field) {
            case GrB_OUTP: *out = d->outp; break;
            case GrB_MASK: *out = d->mask; break;
            case GrB_INP0: *out = d->inp0; break;
            case GrB_INP1: *out = d->inp1; break;
            case GxB_AxB_METHOD: *out = d->axb; break;
            case GxB_DESCRIPTOR_NTHREADS: *out = d->nthreads; break;
            case GxB_SORT: *out = d->sort; break;
            default: r = gb_fail(GrB_INVALID_VALUE, nullptr, "GxB_Desc_get: unknown field %d", (int)field);
        }
    }
    va_end(ap); return r;
}
DescFlags desc_flags(const GrB_Descriptor d) {
    DescFlags f{false, false, false, false, false, 0};
    if (d && d->magic == GB_MAGIC) {
        f.replace = d->outp == GrB_REPLACE;
        f.mask_comp = (d->mask & GrB_COMP) != 0;
        f.mask_struct = (d->mask & GrB_STRUCTURE) != 0;
        f.tran0 = d->inp0 == GrB_TRAN;
        f.tran1 = d->inp1 == GrB_TRAN;
        f.axb = d->axb;
    }
    return f;
}

// ------------------------------------------------------------------ container helpers
bool gb_valid_matrix(const GrB_Matrix A) { return A && A->magic == GB_MAGIC; }
bool gb_valid_vector(const GrB_Vector v) { return v && v->magic == GB_MAGIC; }
static const uint64_t DEV_DIM_MAX = ((uint64_t)1 << 31) - 1;   // 32-bit column / row ids in HBM

void matrix_invalidate_device(GrB_Matrix A) { csr_free(A->dev); csr_free(A->devT); }
// copies still running on the copy streams must finish before the compute stream frees (or overwrites) the buffers
static void vector_join_copies(GrB_Vector v) {
    if (v->h2d_pending) { cudaStreamWaitEvent(G.stream, v->ev_h2d, 0); v->h2d_pending = false; }
    if (v->d2h_pending) { cudaStreamWaitEvent(G.stream, v->ev_d2h, 0); v->d2h_pending = false; }
}
void vector_mark_used(GrB_Vector v) {
    if (v && v->ev_use) { cudaEventRecord(v->ev_use, G.stream); v->use_recorded = true; }
}
void vector_invalidate_device(GrB_Vector v) {
    vector_join_copies(v);
    if (!v->borrowed) { dfree(v->dval); dfree(v->dpres); }       // a borrowed view (B200_Comm_result) does not own its buffers
    v->borrowed = false; v->dval = nullptr; v->dpres = nullptr; v->dev_valid = false; v->dev_nvals = -1;
}
void matrix_adopt_device(GrB_Matrix A, Csr &c) {
    matrix_invalidate_device(A);
    A->dev = c; A->dev.valid = true; c = Csr();
    A->hi.clear(); A->hj.clear(); A->hx.clear(); A->hi.shrink_to_fit(); A->hj.shrink_to_fit(); A->hx.shrink_to_fit();
    A->pi.clear(); A->pj.clear(); A->px.clear();
    A->host_valid = false;
}
void vector_adopt_device(GrB_Vector v, void *vals, uint8_t *pres) {
    vector_invalidate_device(v);
    v->dval = vals; v->dpres = pres; v->dev_valid = true; v->dev_nvals = pres ? -1 : (int64_t)v->n;
    v->hi.clear(); v->hx.clear(); v->pi.clear(); v->px.clear(); v->host_valid = false;
}

// merge the pending list into the sorted host form; later pending entries win
GrB_Info matrix_flush_pending(GrB_Matrix A) {
    const size_t np = A->pi.size();
    if (np == 0) return GrB_SUCCESS;
    const size_t sz = A->type->size;
    std::vector<size_t> ord(np);
    std::iota(ord.begin(), ord.end(), 0);
    std::stable_sort(ord.begin(), ord.end(), [&](size_t a, size_t b) {
        return A->pi[a] != A->pi[b] ? A->pi[a] < A->pi[b] : A->pj[a] < A->pj[b]; });
    std::vector<uint64_t> ni, nj; std::vector<uint8_t> nx;
    const size_t nh = A->hi.size();
    ni.reserve(nh + np); nj.reserve(nh + np); nx.reserve((nh + np) * sz);
    size_t h = 0, p = 0;
    auto push = [&](uint64_t i, uint64_t j, const uint8_t *x) { ni.push_back(i); nj.push_back(j); nx.insert(nx.end(), x, x + sz); };
    while (h < nh || p < np) {
        if (p < np) {   // advance p to the last pending entry of its (i,j) group
            size_t q = p;
            while (q + 1 < np && A->pi[ord[q + 1]] == A->pi[ord[p]] && A->pj[ord[q + 1]] == A->pj[ord[p]]) ++q;
            const uint64_t i = A->pi[ord[q]], j = A->pj[ord[q]];
            if (h < nh && (A->hi[h] < i || (A->hi[h] == i && A->hj[h] < j))) { push(A->hi[h], A->hj[h], &A->hx[h * sz]); ++h; continue; }
            if (h < nh && A->hi[h] == i && A->hj[h] == j) ++h;   // overwritten
            push(i, j, &A->px[ord[q] * sz]);
            p = q + 1;
        } else { push(A->hi[h], A->hj[h], &A->hx[h * sz]); ++h; }
    }
    A->hi.swap(ni); A->hj.swap(nj); A->hx.swap(nx);
    A->pi.clear(); A->pj.clear(); A->px.clear();
    return GrB_SUCCESS;
}

static GrB_Info vector_flush_pending(GrB_Vector v) {
    const size_t np = v->pi.size();
    if (np == 0) return GrB_SUCCESS;
    const size_t sz = v->type->size;
    std::vector<size_t> ord(np);
    std::iota(ord.begin(), ord.end(), 0);
    std::stable_sort(ord.begin(), ord.end(), [&](size_t a, size_t b) { return v->pi[a] < v->pi[b]; });
    std::vector<uint64_t> ni; std::vector<uint8_t> nx;
    const size_t nh = v->hi.size();
    size_t h = 0, p = 0;
    auto push = [&](uint64_t i, const uint8_t *x) { ni.push_back(i); nx.insert(nx.end(), x, x + sz); };
    while (h < nh || p < np) {
        if (p < np) {
            size_t q = p;
            while (q + 1 < np && v->pi[ord[q + 1]] == v->pi[ord[p]]) ++q;
            const uint64_t i = v->pi[ord[q]];
            if (h < nh && v->hi[h] < i) { push(v->hi[h], &v->hx[h * sz]); ++h; continue; }
            if (h < nh && v->hi[h] == i) ++h;
            push(i, &v->px[ord[q] * sz]);
            p = q + 1;
        } else { push(v->hi[h], &v->hx[h * sz]); ++h; }
    }
    v->hi.swap(ni); v->hx.swap(nx); v->pi.clear(); v->px.clear();
    return GrB_SUCCESS;
}

GrB_Info matrix_ensure_host(GrB_Matrix A) {
    if (A->host_valid) return matrix_flush_pending(A);
    // HBM CSR -> host COO
    const Csr &c = A->dev;
    if (!c.valid) { A->host_valid = true; return GrB_SUCCESS; }
    const size_t sz = A->type->size;
    std::vector<int64_t> rp((size_t)c.nrows + 1);
    std::vector<uint32_t> cj((size_t)c.nnz);
    A->hx.assign((size_t)c.nnz * sz, 0);
    CU_TRY(cudaMemcpyAsync(rp.data(), c.rowptr, rp.size() * 8, cudaMemcpyDeviceToHost, G.stream), &A->err);
    if (c.nnz) {
        CU_TRY(cudaMemcpyAsync(cj.data(), c.col, cj.size() * 4, cudaMemcpyDeviceToHost, G.stream), &A->err);
        CU_TRY(cudaMemcpyAsync(A->hx.data(), c.val, A->hx.size(), cudaMemcpyDeviceToHost, G.stream), &A->err);
    }
    CU_TRY(cudaStreamSynchronize(G.stream), &A->err);
    A->hi.resize((size_t)c.nnz); A->hj.resize((size_t)c.nnz);
    for (int64_t r = 0; r < c.nrows; ++r)
        for (int64_t k = rp[r]; k < rp[r + 1]; ++k) { A->hi[k] = (uint64_t)r; A->hj[k] = cj[k]; }
    A->host_valid = true;
    return GrB_SUCCESS;
}

GrB_Info matrix_ensure_device(GrB_Matrix A) {
    if (!G.have_device) return gb_fail(GrB_PANIC, &A->err, "no CUDA device: libb200grb computes only on the GPU (no CPU fallback)");
    if (A->host_valid) GB_TRY(matrix_flush_pending(A));
    if (A->dev.valid) return GrB_SUCCESS;
    if (A->nrows > DEV_DIM_MAX || A->ncols > DEV_DIM_MAX)
        return gb_fail(GrB_INVALID_VALUE, &A->err, "matrix dimensions %llu x %llu exceed the 2^31-1 limit of the HBM CSR layout",
                       (unsigned long long)A->nrows, (unsigned long long)A->ncols);
    const size_t sz = A->type->size;
    const int64_t nnz = (int64_t)A->hi.size();
    Csr c; c.nrows = (int64_t)A->nrows; c.ncols = (int64_t)A->ncols; c.nnz = nnz;
    std::vector<int64_t> rp((size_t)c.nrows + 1, 0);
    for (int64_t k = 0; k < nnz; ++k) rp[A->hi[k] + 1]++;
    for (int64_t r = 0; r < c.nrows; ++r) rp[r + 1] += rp[r];
    std::vector<uint32_t> cj((size_t)nnz);
    for (int64_t k = 0; k < nnz; ++k) cj[k] = (uint32_t)A->hj[k];
    GB_TRY(dalloc(&c.rowptr, rp.size(), &A->err));
    GB_TRY(dalloc(&c.col, (size_t)nnz, &A->err));
    GB_TRY(dmalloc(&c.val, (size_t)nnz * sz + 16, &A->err));
    CU_TRY(cudaMemcpyAsync(c.rowptr, rp.data(), rp.size() * 8, cudaMemcpyHostToDevice, G.stream), &A->err);
    if (nnz) {
        CU_TRY(cudaMemcpyAsync(c.col, cj.data(), cj.size() * 4, cudaMemcpyHostToDevice, G.stream), &A->err);
        CU_TRY(cudaMemcpyAsync(c.val, A->hx.data(), (size_t)nnz * sz, cudaMemcpyHostToDevice, G.stream), &A->err);
    }
    CU_TRY(cudaStreamSynchronize(G.stream), &A->err);   // host staging vectors go out of scope
    GB_TRY(dev_build_rowptr32(c, &A->err));
    c.valid = true;
    A->dev = c;
    return GrB_SUCCESS;
}

GrB_Info matrix_ensure_transpose(GrB_Matrix A) {
    GB_TRY(matrix_ensure_device(A));
    if (A->devT.valid) return GrB_SUCCESS;
    Csr t;
    GB_TRY(dev_transpose(A->dev, A->type->size, t, &A->err));
    t.valid = true; A->devT = t;
    return GrB_SUCCESS;
}

GrB_Info vector_ensure_host(GrB_Vector v) {
    if (v->host_valid) return vector_flush_pending(v);
    if (!v->dev_valid) { v->host_valid = true; return GrB_SUCCESS; }
    const size_t sz = v->type->size, n = (size_t)v->n;
    std::vector<uint8_t> vals(n * sz), pres;
    CU_TRY(cudaMemcpyAsync(vals.data(), v->dval, n * sz, cudaMemcpyDeviceToHost, G.stream), &v->err);
    if (v->dpres) { pres.resize(n); CU_TRY(cudaMemcpyAsync(pres.data(), v->dpres, n, cudaMemcpyDeviceToHost, G.stream), &v->err); }
    CU_TRY(cudaStreamSynchronize(G.stream), &v->err);
    v->hi.clear(); v->hx.clear();
    for (size_t i = 0; i < n; ++i)
        if (!v->dpres || pres[i]) { v->hi.push_back(i); v->hx.insert(v->hx.end(), &vals[i * sz], &vals[i * sz] + sz); }
    v->host_valid = true;
    return GrB_SUCCESS;
}

__global__ void vec_scatter_kernel(const uint64_t *idx, const uint8_t *x, uint8_t *val, uint8_t *pres, int sz, int64_t k) {
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < k; q += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t i = idx[q];
        for (int b = 0; b < sz; ++b) val[i * sz + b] = x[q * sz + b];
        pres[i] = 1;
    }
}
GrB_Info vector_ensure_device(GrB_Vector v) {
    if (!G.have_device) return gb_fail(GrB_PANIC, &v->err, "no CUDA device: libb200grb computes only on the GPU (no CPU fallback)");
    if (v->host_valid) GB_TRY(vector_flush_pending(v));
    if (v->h2d_pending) { cudaStreamWaitEvent(G.stream, v->ev_h2d, 0); v->h2d_pending = false; }     // an overlapped import is in flight
    if (v->dev_valid) return GrB_SUCCESS;
    if (v->n > DEV_DIM_MAX) return gb_fail(GrB_INVALID_VALUE, &v->err, "vector size %llu exceeds the 2^31-1 limit of the HBM layout", (unsigned long long)v->n);
    const size_t sz = v->type->size, n = (size_t)v->n, k = v->hi.size();
    GB_TRY(dmalloc(&v->dval, n * sz + 16, &v->err));
    const bool full = k == n && n > 0;
    if (!full) GB_TRY(dmalloc((void **)&v->dpres, n + 16, &v->err));
    if (n && k < n / 8) {
        // few entries (a BFS source, a seed set): ship the tuples and scatter them in HBM rather than two dense arrays
        CU_TRY(cudaMemsetAsync(v->dval, 0, n * sz, G.stream), &v->err);
        CU_TRY(cudaMemsetAsync(v->dpres, 0, n, G.stream), &v->err);
        if (k) {
            uint64_t *di = nullptr; void *dx = nullptr;
            GB_TRY(dmalloc((void **)&di, k * sizeof(uint64_t), &v->err));
            GB_TRY(dmalloc(&dx, k * sz, &v->err));
            CU_TRY(cudaMemcpyAsync(di, v->hi.data(), k * sizeof(uint64_t), cudaMemcpyHostToDevice, G.stream), &v->err);
            CU_TRY(cudaMemcpyAsync(dx, v->hx.data(), k * sz, cudaMemcpyHostToDevice, G.stream), &v->err);
            const int grid = (int)std::min<size_t>((k + 255) / 256, 4096);
            vec_scatter_kernel<<<grid, 256, 0, G.stream>>>(di, (const uint8_t *)dx, (uint8_t *)v->dval, v->dpres, (int)sz, (int64_t)k);
            G.launches++;
            CU_TRY(cudaGetLastError(), &v->err);
            dfree(di); dfree(dx);
        }
    } else if (n) {
        std::vector<uint8_t> vals(n * sz, 0), pres(full ? 0 : n, 0);
        for (size_t q = 0; q < k; ++q) { memcpy(&vals[v->hi[q] * sz], &v->hx[q * sz], sz); if (!full) pres[v->hi[q]] = 1; }
        CU_TRY(cudaMemcpyAsync(v->dval, vals.data(), n * sz, cudaMemcpyHostToDevice, G.stream), &v->err);
        if (!full) CU_TRY(cudaMemcpyAsync(v->dpres, pres.data(), n, cudaMemcpyHostToDevice, G.stream), &v->err);
        CU_TRY(cudaStreamSynchronize(G.stream), &v->err);      // the staging vectors die here
    }
    CU_TRY(cudaStreamSynchronize(G.stream), &v->err);
    v->dev_valid = true; v->dev_nvals = (int64_t)v->hi.size();
    return GrB_SUCCESS;
}

// ------------------------------------------------------------------ Matrix API
extern "C" GrB_Info GrB_Matrix_new(GrB_Matrix *A, GrB_Type type, GrB_Index nrows, GrB_Index ncols) {
    GB_LOCK; GB_CHECK_INIT;
    if (!A) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Matrix_new: NULL handle");
    *A = nullptr;
    if (!valid_type(type)) return gb_fail(GrB_UNINITIALIZED_OBJECT, nullptr, "GrB_Matrix_new: bad type");
    if (type->code >= TC_COUNT) return gb_fail(GrB_DOMAIN_MISMATCH, nullptr, "GrB_Matrix_new: complex and user-defined types are out of scope");
    // 0 x n objects are legal in SuiteSparse 5 (an empty slice, /root/reference/tests/test_vector.py:522 `len(v[1:9:-3]) == 0`)
    if (nrows > ((uint64_t)1 << 60) || ncols > ((uint64_t)1 << 60))
        return gb_fail(GrB_INVALID_VALUE, nullptr, "GrB_Matrix_new: dimensions must be in 0..2^60");
    GB_Matrix_opaque *m = new GB_Matrix_opaque();
    m->magic = GB_MAGIC; m->type = type; m->nrows = nrows; m->ncols = ncols; m->host_valid = true;
    *A = m; return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Matrix_free(GrB_Matrix *A) {
    GB_LOCK;
    if (!A || !*A) return GrB_SUCCESS;
    if ((*A)->magic == GB_MAGIC) { matrix_invalidate_device(*A); (*A)->magic = GB_FREED; delete *A; }
    *A = nullptr; return GrB_SUCCESS;
}
#define GB_MATRIX_OK(A, fn) do { if (!(A)) return gb_fail(GrB_NULL_POINTER, nullptr, fn ": NULL matrix"); \
    if (!gb_valid_matrix(A)) return gb_fail(GrB_UNINITIALIZED_OBJECT, nullptr, fn ": invalid matrix handle"); } while (0)
#define GB_VECTOR_OK(v, fn) do { if (!(v)) return gb_fail(GrB_NULL_POINTER, nullptr, fn ": NULL vector"); \
    if (!gb_valid_vector(v)) return gb_fail(GrB_UNINITIALIZED_OBJECT, nullptr, fn ": invalid vector handle"); } while (0)

static GrB_Info csr_clone(const Csr &a, size_t vsize, Csr &c, std::string *err) {
    c = Csr(); c.nrows = a.nrows; c.ncols = a.ncols; c.nnz = a.nnz;
    GB_TRY(dalloc(&c.rowptr, (size_t)a.nrows + 1, err));
    GB_TRY(dalloc(&c.col, (size_t)a.nnz, err));
    GB_TRY(dmalloc(&c.val, (size_t)a.nnz * vsize + 16, err));
    CU_TRY(cudaMemcpyAsync(c.rowptr, a.rowptr, ((size_t)a.nrows + 1) * 8, cudaMemcpyDeviceToDevice, G.stream), err);
    if (a.nnz) {
        CU_TRY(cudaMemcpyAsync(c.col, a.col, (size_t)a.nnz * 4, cudaMemcpyDeviceToDevice, G.stream), err);
        CU_TRY(cudaMemcpyAsync(c.val, a.val, (size_t)a.nnz * vsize, cudaMemcpyDeviceToDevice, G.stream), err);
    }
    GB_TRY(dev_build_rowptr32(c, err));
    c.valid = true;
    return GrB_SUCCESS;
}

extern "C" GrB_Info GrB_Matrix_dup(GrB_Matrix *C, const GrB_Matrix A) {
    GB_LOCK; GB_CHECK_INIT;
    if (!C) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Matrix_dup: NULL handle");
    GB_MATRIX_OK(A, "GrB_Matrix_dup");
    GB_Matrix_opaque *m = new GB_Matrix_opaque();
    m->magic = GB_MAGIC; m->type = A->type; m->nrows = A->nrows; m->ncols = A->ncols;
    if (A->host_valid) {
        GrB_Info r = matrix_flush_pending(A);
        if (r != GrB_SUCCESS) { delete m; return r; }
        m->hi = A->hi; m->hj = A->hj; m->hx = A->hx; m->host_valid = true;
    } else {
        m->host_valid = false;
        GrB_Info r = csr_clone(A->dev, A->type->size, m->dev, &A->err);
        if (r != GrB_SUCCESS) { delete m; return r; }
    }
    *C = m; return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Matrix_clear(GrB_Matrix A) {
    GB_LOCK; GB_MATRIX_OK(A, "GrB_Matrix_clear");
    matrix_invalidate_device(A);
    A->hi.clear(); A->hj.clear(); A->hx.clear(); A->pi.clear(); A->pj.clear(); A->px.clear(); A->host_valid = true;
    return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Matrix_nrows(GrB_Index *n, const GrB_Matrix A) {
    if (!n) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Matrix_nrows: NULL"); GB_MATRIX_OK(A, "GrB_Matrix_nrows");
    *n = A->nrows; return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Matrix_ncols(GrB_Index *n, const GrB_Matrix A) {
    if (!n) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Matrix_ncols: NULL"); GB_MATRIX_OK(A, "GrB_Matrix_ncols");
    *n = A->ncols; return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Matrix_nvals(GrB_Index *n, const GrB_Matrix A) {
    GB_LOCK;
    if (!n) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Matrix_nvals: NULL"); GB_MATRIX_OK(A, "GrB_Matrix_nvals");
    if (A->host_valid) { GB_TRY(matrix_flush_pending(A)); *n = A->hi.size(); }
    else { if (G.have_device) CU_TRY(cudaStreamSynchronize(G.stream), &A->err); *n = (GrB_Index)A->dev.nnz; }
    return GrB_SUCCESS;
}
extern "C" GrB_Info GxB_Matrix_type(GrB_Type *t, const GrB_Matrix A) {
    if (!t) return gb_fail(GrB_NULL_POINTER, nullptr, "GxB_Matrix_type: NULL"); GB_MATRIX_OK(A, "GxB_Matrix_type");
    *t = A->type; return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Matrix_wait(GrB_Matrix *A) {
    GB_LOCK;
    if (!A) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Matrix_wait: NULL"); GB_MATRIX_OK(*A, "GrB_Matrix_wait");
    if ((*A)->host_valid) GB_TRY(matrix_flush_pending(*A));
    if (G.have_device) CU_TRY(cudaStreamSynchronize(G.stream), &(*A)->err);
    return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Matrix_error(const char **error, const GrB_Matrix A) {
    if (!error) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Matrix_error: NULL");
    // the reference asks right after a failing call (matrix.py:43-51): report the latest error of this thread
    if (!gb_valid_matrix(A) || !tl_error.empty()) { *error = tl_error.c_str(); return GrB_SUCCESS; }
    *error = A->err.c_str(); return GrB_SUCCESS;
}

static GrB_Info matrix_host_writable(GrB_Matrix A) {
    GB_TRY(matrix_ensure_host(A));
    if (A->dev.valid || A->devT.valid) matrix_invalidate_device(A);
    return GrB_SUCCESS;
}

static GrB_Info matrix_set_element(GrB_Matrix C, int src_tc, const void *x, GrB_Index i, GrB_Index j) {
    GB_LOCK; GB_MATRIX_OK(C, "GrB_Matrix_setElement");
    if (i >= C->nrows || j >= C->ncols) return gb_fail(GrB_INVALID_INDEX, &C->err, "GrB_Matrix_setElement: index (%llu,%llu) out of bounds", (unsigned long long)i, (unsigned long long)j);
    GB_TRY(matrix_host_writable(C));
    const size_t sz = C->type->size;
    Sc s = sc_cast(sc_load(src_tc, x, 0), src_tc, C->type->code);
    C->pi.push_back(i); C->pj.push_back(j);
    C->px.resize(C->px.size() + sz);
    sc_store(C->type->code, C->px.data() + C->px.size() - sz, 0, s);
    return GrB_SUCCESS;
}
static int64_t matrix_find(GrB_Matrix A, GrB_Index i, GrB_Index j) {
    size_t lo = 0, hi = A->hi.size();
    while (lo < hi) {
        size_t mid = (lo + hi) / 2;
        if (A->hi[mid] < i || (A->hi[mid] == i && A->hj[mid] < j)) lo = mid + 1; else hi = mid;
    }
    return (lo < A->hi.size() && A->hi[lo] == i && A->hj[lo] == j) ? (int64_t)lo : -1;
}
static GrB_Info matrix_extract_element(void *x, int dst_tc, const GrB_Matrix A, GrB_Index i, GrB_Index j) {
    GB_LOCK; GB_MATRIX_OK(A, "GrB_Matrix_extractElement");
    if (!x) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Matrix_extractElement: NULL");
    if (i >= A->nrows || j >= A->ncols) return gb_fail(GrB_INVALID_INDEX, &A->err, "GrB_Matrix_extractElement: index out of bounds");
    GB_TRY(matrix_ensure_host(A));
    int64_t k = matrix_find(A, i, j);
    if (k < 0) return GrB_NO_VALUE;
    sc_store(dst_tc, x, 0, sc_cast(sc_load(A->type->code, A->hx.data(), (size_t)k), A->type->code, dst_tc));
    return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Matrix_removeElement(GrB_Matrix C, GrB_Index i, GrB_Index j) {
    GB_LOCK; GB_MATRIX_OK(C, "GrB_Matrix_removeElement");
    if (i >= C->nrows || j >= C->ncols) return gb_fail(GrB_INVALID_INDEX, &C->err, "GrB_Matrix_removeElement: index out of bounds");
    GB_TRY(matrix_host_writable(C));
    int64_t k = matrix_find(C, i, j);
    if (k < 0) return GrB_SUCCESS;
    const size_t sz = C->type->size;
    C->hi.erase(C->hi.begin() + k); C->hj.erase(C->hj.begin() + k);
    C->hx.erase(C->hx.begin() + k * sz, C->hx.begin() + (k + 1) * sz);
    return GrB_SUCCESS;
}
static GrB_Info matrix_extract_tuples(GrB_Index *I, GrB_Index *J, void *X, int dst_tc, GrB_Index *nvals, const GrB_Matrix A) {
    GB_LOCK; GB_MATRIX_OK(A, "GrB_Matrix_extractTuples");
    if (!nvals) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Matrix_extractTuples: NULL nvals");
    GB_TRY(matrix_ensure_host(A));
    const size_t n = A->hi.size();
    if (*nvals < n) return gb_fail(GrB_INSUFFICIENT_SPACE, &A->err, "GrB_Matrix_extractTuples: output arrays hold %llu < %llu entries", (unsigned long long)*nvals, (unsigned long long)n);
    if (I) memcpy(I, A->hi.data(), n * 8);
    if (J) memcpy(J, A->hj.data(), n * 8);
    if (X) {
        const int tc = A->type->code;
        if (tc == dst_tc) memcpy(X, A->hx.data(), n * A->type->size);
        else for (size_t k = 0; k < n; ++k) sc_store(dst_tc, X, k, sc_cast(sc_load(tc, A->hx.data(), k), tc, dst_tc));
    }
    *nvals = n; return GrB_SUCCESS;
}

// fold duplicates of a sorted run with `dup` (left to right, in input order); NULL dup: last wins
static GrB_Info check_dup_op(GrB_BinaryOp dup, std::string *err) {
    if (!dup) return GrB_SUCCESS;
    if (!valid_binop(dup)) return gb_fail(GrB_UNINITIALIZED_OBJECT, err, "build: bad dup operator");
    if (dup->opcode == OP_USER) return gb_fail(GrB_INVALID_VALUE, err, "build: user-defined dup operators (host function pointers) are not supported");
    if (op_is_cmp(dup->opcode) && dup->xtype->code != TC_BOOL) return gb_fail(GrB_DOMAIN_MISMATCH, err, "build: dup operator must have one domain");
    return GrB_SUCCESS;
}
static GrB_Info matrix_build(GrB_Matrix C, const GrB_Index *I, const GrB_Index *J, const void *X, int src_tc, GrB_Index nvals, GrB_BinaryOp dup) {
    GB_LOCK; GB_MATRIX_OK(C, "GrB_Matrix_build");
    if ((!I || !J || !X) && nvals) return gb_fail(GrB_NULL_POINTER, &C->err, "GrB_Matrix_build: NULL array");
    GB_TRY(check_dup_op(dup, &C->err));
    GrB_Index cur = 0; GB_TRY(GrB_Matrix_nvals(&cur, C));
    if (cur != 0) return gb_fail(GrB_OUTPUT_NOT_EMPTY, &C->err, "GrB_Matrix_build: output already has entries");
    for (GrB_Index k = 0; k < nvals; ++k)
        if (I[k] >= C->nrows || J[k] >= C->ncols) return gb_fail(GrB_INDEX_OUT_OF_BOUNDS, &C->err, "GrB_Matrix_build: tuple %llu out of bounds", (unsigned long long)k);
    GB_TRY(matrix_host_writable(C));
    const int tc = C->type->code; const size_t sz = C->type->size;
    std::vector<size_t> ord(nvals);
    std::iota(ord.begin(), ord.end(), 0);
    std::stable_sort(ord.begin(), ord.end(), [&](size_t a, size_t b) { return I[a] != I[b] ? I[a] < I[b] : J[a] < J[b]; });
    C->hi.clear(); C->hj.clear(); C->hx.clear();
    C->hi.reserve(nvals); C->hj.reserve(nvals); C->hx.reserve(nvals * sz);
    const int dtc = dup ? dup->xtype->code : tc;
    for (size_t p = 0; p < nvals;) {
        size_t q = p;
        Sc acc = sc_cast(sc_load(src_tc, X, ord[p]), src_tc, dtc);
        while (q + 1 < nvals && I[ord[q + 1]] == I[ord[p]] && J[ord[q + 1]] == J[ord[p]]) {
            ++q;
            Sc nxt = sc_cast(sc_load(src_tc, X, ord[q]), src_tc, dtc);
            acc = dup ? sc_binop(dup->opcode, dtc, acc, nxt) : nxt;
        }
        C->hi.push_back(I[ord[p]]); C->hj.push_back(J[ord[p]]);
        C->hx.resize(C->hx.size() + sz);
        sc_store(tc, C->hx.data(), C->hi.size() - 1, sc_cast(acc, dup ? dup->ztype->code : dtc, tc));
        p = q + 1;
    }
    return GrB_SUCCESS;
}

// ------------------------------------------------------------------ Vector API
extern "C" GrB_Info GrB_Vector_new(GrB_Vector *v, GrB_Type type, GrB_Index n) {
    GB_LOCK; GB_CHECK_INIT;
    if (!v) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Vector_new: NULL handle");
    *v = nullptr;
    if (!valid_type(type)) return gb_fail(GrB_UNINITIALIZED_OBJECT, nullptr, "GrB_Vector_new: bad type");
    if (type->code >= TC_COUNT) return gb_fail(GrB_DOMAIN_MISMATCH, nullptr, "GrB_Vector_new: complex and user-defined types are out of scope");
    if (n > ((uint64_t)1 << 60)) return gb_fail(GrB_INVALID_VALUE, nullptr, "GrB_Vector_new: size must be in 0..2^60");
    GB_Vector_opaque *o = new GB_Vector_opaque();
    o->magic = GB_MAGIC; o->type = type; o->n = n; o->host_valid = true;
    *v = o; return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Vector_free(GrB_Vector *v) {
    GB_LOCK;
    if (!v || !*v) return GrB_SUCCESS;
    if ((*v)->magic == GB_MAGIC) {
        vector_invalidate_device(*v);
        if ((*v)->ev_h2d) { cudaEventDestroy((*v)->ev_h2d); cudaEventDestroy((*v)->ev_d2h); cudaEventDestroy((*v)->ev_use); }
        (*v)->magic = GB_FREED; delete *v;
    }
    *v = nullptr; return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Vector_dup(GrB_Vector *w, const GrB_Vector u) {
    GB_LOCK; GB_CHECK_INIT;
    if (!w) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Vector_dup: NULL handle");
    GB_VECTOR_OK(u, "GrB_Vector_dup");
    GB_Vector_opaque *o = new GB_Vector_opaque();
    o->magic = GB_MAGIC; o->type = u->type; o->n = u->n;
    if (u->host_valid) {
        vector_flush_pending(u);
        o->hi = u->hi; o->hx = u->hx; o->host_valid = true;
    } else {
        o->host_valid = false;
        const size_t sz = u->type->size, n = (size_t)u->n;
        GrB_Info r = dmalloc(&o->dval, n * sz + 16, &u->err);
        if (r == GrB_SUCCESS && u->dpres) r = dmalloc((void **)&o->dpres, n + 16, &u->err);
        if (r != GrB_SUCCESS) { dfree(o->dval); delete o; return r; }
        cudaMemcpyAsync(o->dval, u->dval, n * sz, cudaMemcpyDeviceToDevice, G.stream);
        if (u->dpres) cudaMemcpyAsync(o->dpres, u->dpres, n, cudaMemcpyDeviceToDevice, G.stream);
        o->dev_valid = true; o->dev_nvals = u->dev_nvals;
    }
    *w = o; return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Vector_clear(GrB_Vector v) {
    GB_LOCK; GB_VECTOR_OK(v, "GrB_Vector_clear");
    vector_invalidate_device(v);
    v->hi.clear(); v->hx.clear(); v->pi.clear(); v->px.clear(); v->host_valid = true;
    return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Vector_size(GrB_Index *n, const GrB_Vector v) {
    if (!n) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Vector_size: NULL"); GB_VECTOR_OK(v, "GrB_Vector_size");
    *n = v->n; return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Vector_nvals(GrB_Index *n, const GrB_Vector v) {
    GB_LOCK;
    if (!n) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Vector_nvals: NULL"); GB_VECTOR_OK(v, "GrB_Vector_nvals");
    if (v->host_valid) { GB_TRY(vector_flush_pending(v)); *n = v->hi.size(); return GrB_SUCCESS; }
    if (v->dev_nvals < 0) {
        if (!v->dpres) v->dev_nvals = (int64_t)v->n;
        else GB_TRY(dev_count_present(v->dpres, (int64_t)v->n, &v->dev_nvals, &v->err));
    }
    *n = (GrB_Index)v->dev_nvals; return GrB_SUCCESS;
}
extern "C" GrB_Info GxB_Vector_type(GrB_Type *t, const GrB_Vector v) {
    if (!t) return gb_fail(GrB_NULL_POINTER, nullptr, "GxB_Vector_type: NULL"); GB_VECTOR_OK(v, "GxB_Vector_type");
    *t = v->type; return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Vector_wait(GrB_Vector *v) {
    GB_LOCK;
    if (!v) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Vector_wait: NULL"); GB_VECTOR_OK(*v, "GrB_Vector_wait");
    if ((*v)->host_valid) GB_TRY(vector_flush_pending(*v));
    if (G.have_device) {
        if ((*v)->d2h_pending) {
            // an overlapped export of v is in flight: its completion implies that of every kernel that produced v, and it is all this
            // vector is waiting for -- the compute stream itself (later, unrelated steps) is left running
            CU_TRY(cudaEventSynchronize((*v)->ev_d2h), &(*v)->err);
            (*v)->d2h_pending = false;
        } else {
            CU_TRY(cudaStreamSynchronize(G.stream), &(*v)->err);
            if ((*v)->h2d_pending) { CU_TRY(cudaEventSynchronize((*v)->ev_h2d), &(*v)->err); (*v)->h2d_pending = false; }
        }
    }
    return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Vector_error(const char **error, const GrB_Vector v) {
    if (!error) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Vector_error: NULL");
    if (!gb_valid_vector(v) || !tl_error.empty()) { *error = tl_error.c_str(); return GrB_SUCCESS; }
    *error = v->err.c_str(); return GrB_SUCCESS;
}
static GrB_Info vector_host_writable(GrB_Vector v) {
    GB_TRY(vector_ensure_host(v));
    if (v->dev_valid) vector_invalidate_device(v);
    return GrB_SUCCESS;
}
static GrB_Info vector_set_element(GrB_Vector w, int src_tc, const void *x, GrB_Index i) {
    GB_LOCK; GB_VECTOR_OK(w, "GrB_Vector_setElement");
    if (i >= w->n) return gb_fail(GrB_INVALID_INDEX, &w->err, "GrB_Vector_setElement: index %llu out of bounds", (unsigned long long)i);
    GB_TRY(vector_host_writable(w));
    const size_t sz = w->type->size;
    w->pi.push_back(i); w->px.resize(w->px.size() + sz);
    sc_store(w->type->code, w->px.data() + w->px.size() - sz, 0, sc_cast(sc_load(src_tc, x, 0), src_tc, w->type->code));
    return GrB_SUCCESS;
}
static int64_t vector_find(GrB_Vector v, GrB_Index i) {
    auto it = std::lower_bound(v->hi.begin(), v->hi.end(), i);
    return (it != v->hi.end() && *it == i) ? (int64_t)(it - v->hi.begin()) : -1;
}
static GrB_Info vector_extract_element(void *x, int dst_tc, const GrB_Vector v, GrB_Index i) {
    GB_LOCK; GB_VECTOR_OK(v, "GrB_Vector_extractElement");
    if (!x) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Vector_extractElement: NULL");
    if (i >= v->n) return gb_fail(GrB_INVALID_INDEX, &v->err, "GrB_Vector_extractElement: index out of bounds");
    GB_TRY(vector_ensure_host(v));
    int64_t k = vector_find(v, i);
    if (k < 0) return GrB_NO_VALUE;
    sc_store(dst_tc, x, 0, sc_cast(sc_load(v->type->code, v->hx.data(), (size_t)k), v->type->code, dst_tc));
    return GrB_SUCCESS;
}
extern "C" GrB_Info GrB_Vector_removeElement(GrB_Vector v, GrB_Index i) {
    GB_LOCK; GB_VECTOR_OK(v, "GrB_Vector_removeElement");
    if (i >= v->n) return gb_fail(GrB_INVALID_INDEX, &v->err, "GrB_Vector_removeElement: index out of bounds");
    GB_TRY(vector_host_writable(v));
    int64_t k = vector_find(v, i);
    if (k < 0) return GrB_SUCCESS;
    const size_t sz = v->type->size;
    v->hi.erase(v->hi.begin() + k); v->hx.erase(v->hx.begin() + k * sz, v->hx.begin() + (k + 1) * sz);
    return GrB_SUCCESS;
}
static GrB_Info vector_extract_tuples(GrB_Index *I, void *X, int dst_tc, GrB_Index *nvals, const GrB_Vector v) {
    GB_LOCK; GB_VECTOR_OK(v, "GrB_Vector_extractTuples");
    if (!nvals) return gb_fail(GrB_NULL_POINTER, nullptr, "GrB_Vector_extractTuples: NULL nvals");
    GB_TRY(vector_ensure_host(v));
    const size_t n = v->hi.size();
    if (*nvals < n) return gb_fail(GrB_INSUFFICIENT_SPACE, &v->err, "GrB_Vector_extractTuples: output arrays too small");
    if (I) memcpy(I, v->hi.data(), n * 8);
    if (X) {
        const int tc = v->type->code;
        if (tc == dst_tc) memcpy(X, v->hx.data(), n * v->type->size);
        else for (size_t k = 0; k < n; ++k) sc_store(dst_tc, X, k, sc_cast(sc_load(tc, v->hx.data(), k), tc, dst_tc));
    }
    *nvals = n; return GrB_SUCCESS;
}
static GrB_Info vector_build(GrB_Vector w, const GrB_Index *I, const void *X, int src_tc, GrB_Index nvals, GrB_BinaryOp dup) {
    GB_LOCK; GB_VECTOR_OK(w, "GrB_Vector_build");
    if ((!I || !X) && nvals) return gb_fail(GrB_NULL_POINTER, &w->err, "GrB_Vector_build: NULL array");
    GB_TRY(check_dup_op(dup, &w->err));
    GrB_Index cur = 0; GB_TRY(GrB_Vector_nvals(&cur, w));
    if (cur != 0) return gb_fail(GrB_OUTPUT_NOT_EMPTY, &w->err, "GrB_Vector_build: output already has entries");
    for (GrB_Index k = 0; k < nvals; ++k)
        if (I[k] >= w->n) return gb_fail(GrB_INDEX_OUT_OF_BOUNDS, &w->err, "GrB_Vector_build: tuple %llu out of bounds", (unsigned long long)k);
    GB_TRY(vector_host_writable(w));
    const int tc = w->type->code; const size_t sz = w->type->size;
    std::vector<size_t> ord(nvals);
    std::iota(ord.begin(), ord.end(), 0);
    std::stable_sort(ord.begin(), ord.end(), [&](size_t a, size_t b) { return I[a] < I[b]; });
    w->hi.clear(); w->hx.clear();
    const int dtc = dup ? dup->xtype->code : tc;
    for (size_t p = 0; p < nvals;) {
        size_t q = p;
        Sc acc = sc_cast(sc_load(src_tc, X, ord[p]), src_tc, dtc);
        while (q + 1 < nvals && I[ord[q + 1]] == I[ord[p]]) {
            ++q;
            Sc nxt = sc_cast(sc_load(src_tc, X, ord[q]), src_tc, dtc);
            acc = dup ? sc_binop(dup->opcode, dtc, acc, nxt) : nxt;
        }
        w->hi.push_back(I[ord[p]]);
        w->hx.resize(w->hx.size() + sz);
        sc_store(tc, w->hx.data(), w->hi.size() - 1, sc_cast(acc, dup ? dup->ztype->code : dtc, tc));
        p = q + 1;
    }
    return GrB_SUCCESS;
}

// typed entry points
#define GB_TYPED(TN, CT, TC) \
    extern "C" GrB_Info GrB_Matrix_setElement_##TN(GrB_Matrix C, CT x, GrB_Index i, GrB_Index j) { return matrix_set_element(C, TC, &x, i, j); } \
    extern "C" GrB_Info GrB_Matrix_extractElement_##TN(CT *x, const GrB_Matrix A, GrB_Index i, GrB_Index j) { return matrix_extract_element(x, TC, A, i, j); } \
    extern "C" GrB_Info GrB_Matrix_extractTuples_##TN(GrB_Index *I, GrB_Index *J, CT *X, GrB_Index *nvals, const GrB_Matrix A) { return matrix_extract_tuples(I, J, X, TC, nvals, A); } \
    extern "C" GrB_Info GrB_Matrix_build_##TN(GrB_Matrix C, const GrB_Index *I, const GrB_Index *J, const CT *X, GrB_Index nvals, const GrB_BinaryOp dup) { return matrix_build(C, I, J, X, TC, nvals, dup); } \
    extern "C" GrB_Info GrB_Vector_setElement_##TN(GrB_Vector w, CT x, GrB_Index i) { return vector_set_element(w, TC, &x, i); } \
    extern "C" GrB_Info GrB_Vector_extractElement_##TN(CT *x, const GrB_Vector v, GrB_Index i) { return vector_extract_element(x, TC, v, i); } \
    extern "C" GrB_Info GrB_Vector_extractTuples_##TN(GrB_Index *I, CT *X, GrB_Index *nvals, const GrB_Vector v) { return vector_extract_tuples(I, X, TC, nvals, v); } \
    extern "C" GrB_Info GrB_Vector_build_##TN(GrB_Vector w, const GrB_Index *I, const CT *X, GrB_Index nvals, const GrB_BinaryOp dup) { return vector_build(w, I, X, TC, nvals, dup); }
GB_TYPED(BOOL, bool, TC_BOOL) GB_TYPED(INT8, int8_t, TC_INT8) GB_TYPED(INT16, int16_t, TC_INT16) GB_TYPED(INT32, int32_t, TC_INT32)
GB_TYPED(INT64, int64_t, TC_INT64) GB_TYPED(UINT8, uint8_t, TC_UINT8) GB_TYPED(UINT16, uint16_t, TC_UINT16)
GB_TYPED(UINT32, uint32_t, TC_UINT32) GB_TYPED(UINT64, uint64_t, TC_UINT64) GB_TYPED(FP32, float, TC_FP32) GB_TYPED(FP64, double, TC_FP64)

// ------------------------------------------------------------------ printing
extern "C" GrB_Info GxB_Matrix_fprint(GrB_Matrix A, const char *name, int pr, FILE *f) {
    GB_LOCK; GB_MATRIX_OK(A, "GxB_Matrix_fprint");
    if (pr <= 0) return GrB_SUCCESS;
    GrB_Index nv = 0; GB_TRY(GrB_Matrix_nvals(&nv, A));
    fprintf(f ? f : stdout, "\n  %llux%llu B200 GraphBLAS %s matrix %s, CSR by row: %llu entries\n",
            (unsigned long long)A->nrows, (unsigned long long)A->ncols, A->type->name, name ? name : "", (unsigned long long)nv);
    return GrB_SUCCESS;
}
extern "C" GrB_Info GxB_Vector_fprint(GrB_Vector v, const char *name, int pr, FILE *f) {
    GB_LOCK; GB_VECTOR_OK(v, "GxB_Vector_fprint");
    if (pr <= 0) return GrB_SUCCESS;
    GrB_Index nv = 0; GB_TRY(GrB_Vector_nvals(&nv, v));
    fprintf(f ? f : stdout, "\n  %llu B200 GraphBLAS %s vector %s: %llu entries\n",
            (unsigned long long)v->n, v->type->name, name ? name : "", (unsigned long long)nv);
    return GrB_SUCCESS;
}

// ------------------------------------------------------------------ bulk import / export (B200 extensions)
// first overlapped copy of a vector: the copy streams and the vector's events
static GrB_Info vector_async_setup(GrB_Vector v) {
    if (!G.h2d) {
        CU_TRY(cudaStreamCreateWithFlags(&G.h2d, cudaStreamNonBlocking), &v->err);
        CU_TRY(cudaStreamCreateWithFlags(&G.d2h, cudaStreamNonBlocking), &v->err);
    }
    if (!v->ev_h2d) {
        CU_TRY(cudaEventCreateWithFlags(&v->ev_h2d, cudaEventDisableTiming), &v->err);
        CU_TRY(cudaEventCreateWithFlags(&v->ev_d2h, cudaEventDisableTiming), &v->err);
        CU_TRY(cudaEventCreateWithFlags(&v->ev_use, cudaEventDisableTiming), &v->err);
    }
    return GrB_SUCCESS;
}
static GrB_Info copy_in(void *dst, const void *src, size_t bytes, int where, std::string *err) {
    if (!bytes) return GrB_SUCCESS;
    CU_TRY(cudaMemcpyAsync(dst, src, bytes, where ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, G.stream), err);
    return GrB_SUCCESS;
}
static GrB_Info copy_out(void *dst, const void *src, size_t bytes, int where, std::string *err) {
    if (!bytes) return GrB_SUCCESS;
    CU_TRY(cudaMemcpyAsync(dst, src, bytes, where ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, G.stream), err);
    return GrB_SUCCESS;
}

extern "C" GrB_Info B200_Matrix_import_CSR(GrB_Matrix *A, GrB_Type type, GrB_Index nrows, GrB_Index ncols,
                                            const int64_t *Ap, const uint32_t *Aj, const void *Ax, GrB_Index nvals, int where) {
    GB_LOCK; GB_CHECK_INIT;
    if (!A || !Ap || (nvals && !Aj)) return gb_fail(GrB_NULL_POINTER, nullptr, "B200_Matrix_import_CSR: NULL argument");
    if (!G.have_device) return gb_fail(GrB_PANIC, nullptr, "no CUDA device: libb200grb computes only on the GPU (no CPU fallback)");
    if (nrows > DEV_DIM_MAX || ncols > DEV_DIM_MAX) return gb_fail(GrB_INVALID_VALUE, nullptr, "B200_Matrix_import_CSR: dimensions exceed 2^31-1");
    GB_TRY(GrB_Matrix_new(A, type, nrows, ncols));
    GrB_Matrix m = *A;
    Csr c; c.nrows = (int64_t)nrows; c.ncols = (int64_t)ncols; c.nnz = (int64_t)nvals;
    const size_t sz = type->size;
    GrB_Info r = dalloc(&c.rowptr, (size_t)nrows + 1, &m->err);
    if (r == GrB_SUCCESS) r = dalloc(&c.col, (size_t)nvals, &m->err);
    if (r == GrB_SUCCESS) r = dmalloc(&c.val, (size_t)nvals * sz + 16, &m->err);
    if (r == GrB_SUCCESS) r = copy_in(c.rowptr, Ap, ((size_t)nrows + 1) * 8, where, &m->err);
    if (r == GrB_SUCCESS) r = copy_in(c.col, Aj, (size_t)nvals * 4, where, &m->err);
    if (r == GrB_SUCCESS) {
        if (Ax) r = copy_in(c.val, Ax, (size_t)nvals * sz, where, &m->err);
        else {  // pattern-only import: every value is 1
            std::vector<uint8_t> ones((size_t)nvals * sz);
            Sc one; one.u = 0; if (tc_is_float(type->code)) one.d = 1.0; else one.u = 1;
            for (size_t k = 0; k < (size_t)nvals; ++k) sc_store(type->code, ones.data(), k, one);
            r = copy_in(c.val, ones.data(), ones.size(), 0, &m->err);
            if (r == GrB_SUCCESS && cudaStreamSynchronize(G.stream) != cudaSuccess) r = GrB_PANIC;
        }
    }
    if (r == GrB_SUCCESS && !where && cudaStreamSynchronize(G.stream) != cudaSuccess) r = GrB_PANIC;
    if (r == GrB_SUCCESS) r = dev_build_rowptr32(c, &m->err);
    if (r != GrB_SUCCESS) { csr_free(c); GrB_Matrix_free(A); return r; }
    matrix_adopt_device(m, c);
    return GrB_SUCCESS;
}

extern "C" GrB_Info B200_Matrix_export_CSR(const GrB_Matrix A, int64_t *Ap, uint32_t *Aj, void *Ax, int where) {
    GB_LOCK; GB_MATRIX_OK(A, "B200_Matrix_export_CSR");
    GB_TRY(matrix_ensure_device(A));
    const Csr &c = A->dev;
    if (Ap) GB_TRY(copy_out(Ap, c.rowptr, ((size_t)c.nrows + 1) * 8, where, &A->err));
    if (Aj) GB_TRY(copy_out(Aj, c.col, (size_t)c.nnz * 4, where, &A->err));
    if (Ax) GB_TRY(copy_out(Ax, c.val, (size_t)c.nnz * A->type->size, where, &A->err));
    CU_TRY(cudaStreamSynchronize(G.stream), &A->err);
    return GrB_SUCCESS;
}

extern "C" GrB_Info B200_Vector_set_dense(GrB_Vector v, const void *x, const uint8_t *present, int where) {
    GB_LOCK; GB_VECTOR_OK(v, "B200_Vector_set_dense");
    if (!x) return gb_fail(GrB_NULL_POINTER, &v->err, "B200_Vector_set_dense: NULL values");
    if (!G.have_device) return gb_fail(GrB_PANIC, &v->err, "no CUDA device: libb200grb computes only on the GPU (no CPU fallback)");
    if (v->n > DEV_DIM_MAX) return gb_fail(GrB_INVALID_VALUE, &v->err, "vector size exceeds 2^31-1");
    const size_t sz = v->type->size, n = (size_t)v->n;
    if (where == 2) GB_TRY(vector_async_setup(v));
    const bool fresh = !v->dev_valid || !v->dval || (present && !v->dpres) || (!present && v->dpres);
    if (!v->dev_valid || !v->dval) { vector_invalidate_device(v); GB_TRY(dmalloc(&v->dval, n * sz + 16, &v->err)); }
    if (present && !v->dpres) GB_TRY(dmalloc((void **)&v->dpres, n + 16, &v->err));
    if (!present && v->dpres) { vector_join_copies(v); dfree(v->dpres); v->dpres = nullptr; }
    if (where == 2) {
        // pinned host memory, copied on the import stream so that it overlaps kernels already enqueued on the compute stream.
        // The copy may start once the last kernels that READ this vector are done (their event, recorded by the call that
        // used it) -- or, when the buffers are new or the use was not recorded, once everything enqueued so far is done.
        if (v->use_recorded && !fresh) cudaStreamWaitEvent(G.h2d, v->ev_use, 0);
        else { cudaEventRecord(v->ev_use, G.stream); cudaStreamWaitEvent(G.h2d, v->ev_use, 0); }
        v->use_recorded = false;
        if (v->d2h_pending) cudaStreamWaitEvent(G.h2d, v->ev_d2h, 0);
        CU_TRY(cudaMemcpyAsync(v->dval, x, n * sz, cudaMemcpyHostToDevice, G.h2d), &v->err);
        if (present) CU_TRY(cudaMemcpyAsync(v->dpres, present, n, cudaMemcpyHostToDevice, G.h2d), &v->err);
        CU_TRY(cudaEventRecord(v->ev_h2d, G.h2d), &v->err);
        v->h2d_pending = true;
    } else {
        vector_join_copies(v);
        GB_TRY(copy_in(v->dval, x, n * sz, where, &v->err));
        if (present) GB_TRY(copy_in(v->dpres, present, n, where, &v->err));
    }
    v->dev_valid = true; v->dev_nvals = present ? -1 : (int64_t)n;
    v->hi.clear(); v->hx.clear(); v->pi.clear(); v->px.clear(); v->host_valid = false;
    return GrB_SUCCESS;
}
extern "C" GrB_Info B200_Vector_import_dense(GrB_Vector *v, GrB_Type type, GrB_Index n, const void *x, const uint8_t *present, int where) {
    GB_LOCK; GB_CHECK_INIT;
    if (!v) return gb_fail(GrB_NULL_POINTER, nullptr, "B200_Vector_import_dense: NULL handle");
    GB_TRY(GrB_Vector_new(v, type, n));
    GrB_Info r = B200_Vector_set_dense(*v, x, present, where);
    if (r != GrB_SUCCESS) GrB_Vector_free(v);
    return r;
}
extern "C" GrB_Info B200_Vector_export_dense(const GrB_Vector v, void *x, uint8_t *present, int where) {
    GB_LOCK; GB_VECTOR_OK(v, "B200_Vector_export_dense");
    GB_TRY(vector_ensure_device(v));
    const size_t sz = v->type->size, n = (size_t)v->n;
    if (where == 2) {
        // pinned host memory, copied on the export stream once everything enqueued so far on the compute stream is done; the data
        // is in host memory after GrB_Vector_wait(v) / B200_device_synchronize (GraphBLAS non-blocking mode)
        GB_TRY(vector_async_setup(v));
        if (v->d2h_pending) cudaStreamWaitEvent(G.d2h, v->ev_d2h, 0);
        CU_TRY(cudaEventRecord(v->ev_d2h, G.stream), &v->err);
        CU_TRY(cudaStreamWaitEvent(G.d2h, v->ev_d2h, 0), &v->err);
        if (x) CU_TRY(cudaMemcpyAsync(x, v->dval, n * sz, cudaMemcpyDeviceToHost, G.d2h), &v->err);
        if (present) {
            if (v->dpres) CU_TRY(cudaMemcpyAsync(present, v->dpres, n, cudaMemcpyDeviceToHost, G.d2h), &v->err);
            else memset(present, 1, n);
        }
        CU_TRY(cudaEventRecord(v->ev_d2h, G.d2h), &v->err);
        v->d2h_pending = true;
        return GrB_SUCCESS;
    }
    if (x) GB_TRY(copy_out(x, v->dval, n * sz, where, &v->err));
    if (present) {
        if (v->dpres) GB_TRY(copy_out(present, v->dpres, n, where, &v->err));
        else if (where) CU_TRY(cudaMemsetAsync(present, 1, n, G.stream), &v->err);
        else memset(present, 1, n);
    }
    CU_TRY(cudaStreamSynchronize(G.stream), &v->err);
    return GrB_SUCCESS;
}
extern "C" GrB_Info B200_Vector_device_ptrs(GrB_Vector v, void **values, uint8_t **present) {
    GB_LOCK; GB_VECTOR_OK(v, "B200_Vector_device_ptrs");
    GB_TRY(vector_ensure_device(v));
    if (values) *values = v->dval;
    if (present) *present = v->dpres;
    // the caller may write through these pointers: the host form is no longer authoritative
    v->hi.clear(); v->hx.clear(); v->host_valid = false; if (v->dpres) v->dev_nvals = -1;
    return GrB_SUCCESS;
}
