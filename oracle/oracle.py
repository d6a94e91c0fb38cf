"""ctypes wrapper around oracle/grb_oracle.c (+ grb_fast.c) -- TEST INFRASTRUCTURE ONLY.

The C files restate the GraphBLAS C API 1.3 semantics of the three calls the reference
makes on its hot path (/root/reference/pygraphblas/matrix.py:2574, :2716, vector.py:961);
see the header of grb_oracle.c for the step-by-step citation.  This module compiles them
with gcc into oracle/_build/liboracle.so and exposes

    mxm(C, M, accum, semiring, A, B, desc) -> SpMat
    mxv(w, mask, accum, semiring, A, u, desc) -> SpVec
    vxm(w, mask, accum, semiring, u, A, desc) -> SpVec

on plain numpy COO containers.  Operators are named the way the reference names them:
semiring = ("PLUS", "TIMES", "INT64")  (add, multiply, operand type of the multiply --
semiring.py:29-44 `pls`, `mul`, `type`), accum = ("MIN", "INT64") or None, desc = a string of
descriptor letters as in /root/reference/pygraphblas/descriptor.py:150-182 ("", "T0", "RC", "RSCT0T1").
"""
import ctypes
import os
import subprocess
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
def _cpu_tag():
    """Builds are keyed by the host CPU's feature flags: a -march=native library must not be
    carried to a different machine (the GPU box) and executed there."""
    import hashlib
    try:
        with open("/proc/cpuinfo") as f:
            flags = next((ln for ln in f if ln.startswith("flags")), "")
    except OSError:
        flags = ""
    return hashlib.sha1(flags.encode()).hexdigest()[:10]


_BUILD = os.path.join(_HERE, "_build", _cpu_tag())
_LIB = os.path.join(_BUILD, "liboracle.so")
_SOURCES = [os.path.join(_HERE, "grb_oracle.c"), os.path.join(_HERE, "grb_fast.c")]

TYPES = ["BOOL", "INT8", "INT16", "INT32", "INT64", "UINT8", "UINT16", "UINT32", "UINT64", "FP32", "FP64"]
DTYPES = {"BOOL": np.bool_, "INT8": np.int8, "INT16": np.int16, "INT32": np.int32, "INT64": np.int64,
          "UINT8": np.uint8, "UINT16": np.uint16, "UINT32": np.uint32, "UINT64": np.uint64,
          "FP32": np.float32, "FP64": np.float64}
OPS = ["FIRST", "SECOND", "PAIR", "ANY", "MIN", "MAX", "PLUS", "MINUS", "RMINUS", "TIMES", "DIV", "RDIV",
       "POW", "ISEQ", "ISNE", "ISGT", "ISLT", "ISGE", "ISLE", "LOR", "LAND", "LXOR", "BOR", "BAND", "BXOR",
       "BXNOR", "EQ", "NE", "GT", "LT", "GE", "LE"]
CMP_OPS = {"EQ", "NE", "GT", "LT", "GE", "LE"}


def build(force=False):
    global _BUILD, _LIB
    srcs = [s for s in _SOURCES if os.path.exists(s)]
    if (not force and os.path.exists(_LIB)
            and all(os.path.getmtime(_LIB) >= os.path.getmtime(s) for s in srcs)):
        return _LIB
    try:
        os.makedirs(_BUILD, exist_ok=True)
        writable = os.access(_BUILD, os.W_OK)
    except OSError:
        writable = False
    if not writable:                 # a read-only checkout: build per process in a temporary directory
        import tempfile
        _BUILD = tempfile.mkdtemp(prefix="b200grb_oracle_")
        _LIB = os.path.join(_BUILD, "liboracle.so")
    cmd = ["gcc", "-O3", "-march=native", "-fopenmp", "-fPIC", "-shared", "-std=gnu11", "-o", _LIB] + srcs + ["-lm"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        # -march=native objects would not travel between different hosts anyway: retry portable
        cmd.remove("-march=native")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("oracle build failed:\n" + r.stderr)
    return _LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        try:
            _lib = ctypes.CDLL(build())
        except OSError:       # e.g. built with -march=native on another CPU
            _lib = ctypes.CDLL(build(force=True))
    return _lib


class _Res(ctypes.Structure):
    _fields_ = [("nvals", ctypes.c_int64), ("I", ctypes.POINTER(ctypes.c_uint64)),
                ("J", ctypes.POINTER(ctypes.c_uint64)), ("X", ctypes.c_void_p)]


class _Desc(ctypes.Structure):
    _fields_ = [("replace", ctypes.c_int), ("mask_comp", ctypes.c_int), ("mask_struct", ctypes.c_int),
                ("tran0", ctypes.c_int), ("tran1", ctypes.c_int)]


class SpMat:
    """Row-major sorted COO matrix with a GraphBLAS type name."""

    def __init__(self, typ, nrows, ncols, I=(), J=(), X=()):
        self.type = typ
        self.nrows, self.ncols = int(nrows), int(ncols)
        I = np.asarray(I, dtype=np.uint64).reshape(-1)
        J = np.asarray(J, dtype=np.uint64).reshape(-1)
        X = np.asarray(X, dtype=DTYPES[typ]).reshape(-1)
        order = np.lexsort((J, I))
        self.I, self.J, self.X = (np.ascontiguousarray(I[order]), np.ascontiguousarray(J[order]),
                                  np.ascontiguousarray(X[order]))

    @property
    def nvals(self):
        return len(self.I)

    def todict(self):
        return {(int(i), int(j)): x.item() for i, j, x in zip(self.I, self.J, self.X)}

    def __repr__(self):
        return f"SpMat({self.type}, {self.nrows}x{self.ncols}, {self.todict()})"


class SpVec:
    """Sorted sparse vector with a GraphBLAS type name."""

    def __init__(self, typ, size, I=(), X=()):
        self.type = typ
        self.size = int(size)
        I = np.asarray(I, dtype=np.uint64).reshape(-1)
        X = np.asarray(X, dtype=DTYPES[typ]).reshape(-1)
        order = np.argsort(I, kind="stable")
        self.I, self.X = np.ascontiguousarray(I[order]), np.ascontiguousarray(X[order])

    @property
    def nvals(self):
        return len(self.I)

    def todict(self):
        return {int(i): x.item() for i, x in zip(self.I, self.X)}

    def as_col(self):
        return SpMat(self.type, self.size, 1, self.I, np.zeros(len(self.I), np.uint64), self.X)

    def as_row(self):
        return SpMat(self.type, 1, self.size, np.zeros(len(self.I), np.uint64), self.I, self.X)

    def __repr__(self):
        return f"SpVec({self.type}, {self.size}, {self.todict()})"


def parse_desc(desc):
    """'RSCT0T1'-style string -> flags (descriptor.py:150-182 names)."""
    d = desc or ""
    t0 = "T0" in d
    t1 = "T1" in d
    rest = d.replace("T0", "").replace("T1", "")
    return dict(replace="R" in rest, mask_comp="C" in rest, mask_struct="S" in rest, tran0=t0, tran1=t1)


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def mxm(C, M, accum, semiring, A, B, desc=""):
    add, mul, mtype = semiring
    f = parse_desc(desc)
    d = _Desc(int(f["replace"]), int(f["mask_comp"]), int(f["mask_struct"]), int(f["tran0"]), int(f["tran1"]))
    res = _Res()
    L = lib()
    empty_i = np.zeros(0, np.uint64)
    empty_x = np.zeros(0, np.uint8)
    args = [ctypes.byref(res),
            TYPES.index(C.type), ctypes.c_int64(C.nrows), ctypes.c_int64(C.ncols), ctypes.c_int64(C.nvals), _ptr(C.I), _ptr(C.J), _ptr(C.X)]
    if M is not None:
        args += [1, TYPES.index(M.type), ctypes.c_int64(M.nvals), _ptr(M.I), _ptr(M.J), _ptr(M.X)]
    else:
        args += [0, 0, ctypes.c_int64(0), _ptr(empty_i), _ptr(empty_i), _ptr(empty_x)]
    if accum is not None:
        args += [1, OPS.index(accum[0]), TYPES.index(accum[1])]
    else:
        args += [0, 0, 0]
    args += [OPS.index(add), OPS.index(mul), TYPES.index(mtype)]
    for X in (A, B):
        args += [TYPES.index(X.type), ctypes.c_int64(X.nrows), ctypes.c_int64(X.ncols), ctypes.c_int64(X.nvals), _ptr(X.I), _ptr(X.J), _ptr(X.X)]
    args.append(ctypes.byref(d))
    L.oracle_mxm.restype = ctypes.c_int
    rc = L.oracle_mxm(*args)
    if rc == -2:
        raise ValueError("oracle_mxm: dimension mismatch")
    if rc != 0:
        raise MemoryError("oracle_mxm failed")
    n = res.nvals
    I = np.ctypeslib.as_array(res.I, shape=(max(n, 1),))[:n].copy()
    J = np.ctypeslib.as_array(res.J, shape=(max(n, 1),))[:n].copy()
    dt = np.dtype(DTYPES[C.type])
    buf = (ctypes.c_char * (max(n, 1) * dt.itemsize)).from_address(res.X)
    X = np.frombuffer(buf, dtype=dt, count=n).copy()
    L.oracle_free_result(ctypes.byref(res))
    out = SpMat.__new__(SpMat)
    out.type, out.nrows, out.ncols, out.I, out.J, out.X = C.type, C.nrows, C.ncols, I, J, X
    return out


def mxv(w, mask, accum, semiring, A, u, desc=""):
    """w<mask> = accum(w, op(A) (+).(x) u); INP1 does not apply (matrix.py:2586-2726)."""
    d = (desc or "").replace("T1", "")
    r = mxm(w.as_col(), None if mask is None else mask.as_col(), accum, semiring, A, u.as_col(), d)
    return SpVec(w.type, w.size, r.I, r.X)


def vxm(w, mask, accum, semiring, u, A, desc=""):
    """w'<mask'> = accum(w', u' (+).(x) op(A)); INP0 is ignored for the vector (vector.py:922-926)."""
    d = (desc or "").replace("T0", "")
    r = mxm(w.as_row(), None if mask is None else mask.as_row(), accum, semiring, u.as_row(), A, d)
    return SpVec(w.type, w.size, r.J, r.X)


def semiring_ztype(semiring):
    """Type of the semiring's monoid (types.py:442-461): BOOL for comparison multiplies."""
    return "BOOL" if semiring[1] in CMP_OPS else semiring[2]
