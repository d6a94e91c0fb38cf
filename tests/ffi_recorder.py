"""Recorder of the C calls a GraphBLAS package makes (used by tests/test_reference_dropin.py and
tests/golden/make_dropin_goldens.py, each in a subprocess of its own).  The library's compute entry points are
replaced by a recorder BEFORE the package under test (the mirror, or the reference over the binding stub) is
imported, so it captures the recorder; every call is normalised at record time (operator handle -> name, descriptor
-> field values, vector / matrix -> type, shape, nvals, index list -> its values) and nothing computes.
`run(fn, pkg)` returns what `pkg` passes to the C ABI for the user-level expression `fn(pkg)`."""
import os
import importlib.util, sys
_spec = importlib.util.spec_from_file_location("pygraphblas_b200._ffi", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "pygraphblas_b200", "_ffi.py"))
_ffi = importlib.util.module_from_spec(_spec); sys.modules["pygraphblas_b200._ffi"] = _ffi; _spec.loader.exec_module(_ffi)

NAMES = ("eWiseAdd", "eWiseMult", "_apply", "_assign", "_extract", "_select", "_reduce", "GrB_mxm", "GrB_mxv", "GrB_vxm", "GrB_transpose")
_real = _ffi.lib
CALLS = []


class Recorder:
    def __dir__(self):
        return dir(_real)

    def __getattr__(self, name):
        real = getattr(_real, name)
        if name.startswith(("GrB_", "GxB_")) and any(k in name for k in NAMES) and callable(real):
            def rec(*args):
                CALLS.append(_row(name, args))      # normalised now: the operands may be temporaries
                return 0
            rec.__name__ = name
            return rec
        return real


_ffi.lib = Recorder()
import pygraphblas_b200 as gb          # noqa: E402
ffi = gb.ffi
KIND = {"struct GB_BinaryOp_opaque *": 0, "struct GB_Monoid_opaque *": 1, "struct GB_Semiring_opaque *": 2, "struct GB_UnaryOp_opaque *": 3}


def norm(a):
    if isinstance(a, (bool, int, float)):
        return ("py", type(a).__name__, a)
    if isinstance(a, (list, tuple)):
        return ("idx", [int(x) for x in a])
    try:
        c = ffi.typeof(a).cname
    except Exception:
        return ("obj", type(a).__name__)
    if c.endswith("*") and a == ffi.NULL:
        return "NULL"
    if c == "struct GB_UnaryOp_opaque *":
        for name, u in gb.ops.unaryops.items():
            if u.unaryop == a:
                return "unary:" + name
        return "unary:?"
    if c in KIND:
        p = ffi.new("char**")
        assert _real.B200_object_name(ffi.cast("const char**", p), KIND[c], ffi.cast("void*", a)) == 0, c
        return ffi.string(ffi.cast("char*", p[0])).decode()
    if c == "struct GB_Descriptor_opaque *":
        out = []
        for f in (_real.GrB_OUTP, _real.GrB_MASK, _real.GrB_INP0, _real.GrB_INP1):
            v = ffi.new("GrB_Desc_Value*"); _real.GxB_Desc_get(a, f, v); out.append(int(v[0]))
        return ("desc", tuple(out))
    if c == "struct GB_Vector_opaque *":
        t = ffi.new("GrB_Type*"); n = ffi.new("GrB_Index*")
        _real.GxB_Vector_type(t, a); _real.GrB_Vector_size(n, a)
        nv = ffi.new("GrB_Index*"); _real.GrB_Vector_nvals(nv, a)
        return ("vec", gb.types.from_handle(t[0]).name, int(n[0]), "nvals=%d" % nv[0])
    if c == "struct GB_Matrix_opaque *":
        t = ffi.new("GrB_Type*"); n = ffi.new("GrB_Index*"); m = ffi.new("GrB_Index*")
        _real.GxB_Matrix_type(t, a); _real.GrB_Matrix_nrows(n, a); _real.GrB_Matrix_ncols(m, a)
        nv = ffi.new("GrB_Index*"); _real.GrB_Matrix_nvals(nv, a)
        return ("mat", gb.types.from_handle(t[0]).name, int(n[0]), int(m[0]), "nvals=%d" % nv[0])
    if c == "struct GB_Scalar_opaque *":
        x = ffi.new("double*"); _real.GxB_Scalar_extractElement_FP64(x, a)
        t = ffi.new("GrB_Type*"); _real.GxB_Scalar_type(t, a)
        return ("scalar", gb.types.from_handle(t[0]).name, x[0])
    if c == "struct GB_SelectOp_opaque *":
        return ("selop", _selname(a))
    if "uint64_t" in c and (c.endswith("*") or "[" in c):
        if a == _real.GrB_ALL:
            return "GrB_ALL"
        return ("idx",)
    if c.endswith("*") or "[" in c:
        return ("ptr", c.replace("_Bool", "bool").split("[")[0].rstrip(" *"))
    return ("c", c)


_SEL = ["TRIL", "TRIU", "DIAG", "OFFDIAG", "NONZERO", "EQ_ZERO", "GT_ZERO", "GE_ZERO", "LT_ZERO", "LE_ZERO", "NE_THUNK", "EQ_THUNK", "GT_THUNK", "GE_THUNK", "LT_THUNK", "LE_THUNK"]


def _selname(a):
    for n in _SEL:
        if getattr(_real, "GxB_" + n) == a:
            return n
    return "?"


def _row(name, args):
    row = [name]
    for k, a in enumerate(args):
        v = norm(a)
        if isinstance(v, tuple) and v[:1] == ("idx",) and len(v) == 2:
            pass
        elif v == ("idx",):                       # index list: expand with the following ni argument
            ni = int(args[k + 1])
            if ni in (int(_real.GxB_RANGE), int(_real.GxB_STRIDE), int(_real.GxB_BACKWARDS)):
                v = ("idx", [int(a[q]) for q in range(2 if ni == int(_real.GxB_RANGE) else 3)])
            else:
                v = ("idx", [int(a[q]) for q in range(ni)])
        row.append(v)
    return tuple(row)


def run(fn, pkg):
    n0 = len(CALLS)
    try:
        fn(pkg)
    except Exception as e:
        return ("EXC", type(e).__name__, str(e)[:60])
    return tuple(CALLS[n0:])
