"""The drop-in boundary, pinned to what the UNMODIFIED reference package (Graphegon/pygraphblas) does.
`suitesparse_graphblas/` at the repository root is the binding stub of INTEGRATION.md: with it ahead on PYTHONPATH
the reference imports and runs on libb200grb.so.  What the reference decides on the host -- the binding names it
reads, its index encoding of slices, its type promotion and default operators, the output it infers for the hot calls
and the C calls its user-level expressions make -- was recorded by running it over the stub
(tests/golden/make_dropin_goldens.py) into tests/golden/reference_dropin.json.  These tests hold the stub and the
host-side mirror (pygraphblas_b200) to that record; none of them needs the reference tree or a GPU."""
import itertools
import json
import os
import subprocess
import sys
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TESTS = os.path.join(ROOT, "tests")
NAMES = ["BOOL", "INT8", "INT16", "INT32", "INT64", "UINT8", "UINT16", "UINT32", "UINT64", "FP32", "FP64"]


@pytest.fixture(scope="module")
def golden():
    with open(os.path.join(TESTS, "golden", "reference_dropin.json")) as f:
        return json.load(f)


def run_snippet(code, pkg, pythonpath=ROOT):
    """Run `code` with PKG = the package under test in a fresh interpreter; its last stdout line is JSON."""
    env = dict(os.environ, PYTHONPATH=pythonpath)
    prelude = f"PKG = {pkg!r}\nTESTS = {TESTS!r}\n"
    r = subprocess.run([sys.executable, "-c", prelude + textwrap.dedent(code)], capture_output=True, text=True, env=env,
                       cwd=TESTS, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_unmodified_reference_imports_and_plumbing_works(golden):
    """Every name the reference reads from suitesparse_graphblas.lib while it imports and does the handle plumbing
    below is present in the stub, the plumbing gives the reference's results through the mirror, and without a GPU
    every call that computes refuses with Panic ("no CPU fallback") -- never computes on the host."""
    import suitesparse_graphblas
    import pygraphblas_b200 as gb
    from pygraphblas_b200 import Matrix, Vector, Scalar, INT64, BOOL, descriptor, lib
    ref = golden["binding"]
    assert len(ref["names"]) > 100, len(ref["names"])
    missing = [n for n in ref["names"] if not hasattr(suitesparse_graphblas.lib, n)]
    assert not missing, missing
    m = Matrix.from_lists([0, 1, 2], [1, 2, 0], [1, 2, 3])       # tests/test_matrix.py:250
    v = Vector.from_lists([0, 1, 2], [2, 3, 4])
    got = {"implementation_major": int(suitesparse_graphblas.lib.GxB_IMPLEMENTATION_MAJOR),
           "shape": [m.nrows, m.ncols, m.nvals], "type": m.type.name,
           "to_lists": m.to_lists(), "dup": m.dup().to_lists(), "vdup": v.dup().to_lists(),
           "ztypes": [INT64.PLUS_TIMES.ztype.name, BOOL.LOR_LAND.ztype.name], "min_plus_alias": INT64.min_plus is INT64.MIN_PLUS,
           "ct1": [descriptor.T1 in descriptor.CT1, descriptor.CT1 == (descriptor.C & descriptor.T1)],
           "scalar": Scalar.from_value(3)[0], "sparse_nrows": Matrix.sparse(INT64).nrows}
    assert json.loads(json.dumps(got)) == ref["plumbing"]
    # the reference's m.iseq(m.dup()) is an eWiseMult with EQ (matrix.py:1451-1453); the mirror's compares on the host
    for call in (lambda: m.mxv(v), lambda: v.vxm(m), lambda: m.mxm(m), lambda: m @ m,
                 lambda: m.emult(m.dup(), INT64.EQ), lambda: m.reduce_int(), lambda: v + v, lambda: m.tril(), lambda: v.apply(INT64.AINV)):
        try:
            call()
            assert lib.B200_have_device()
        except gb.base.Panic as e:
            assert not lib.B200_have_device() and "no CPU fallback" in str(e)


def test_slice_to_index_list_matches_the_reference(golden):
    """Vector._index (the mirror) against the reference's own base._build_range (base.py:216-252) on a grid of
    slices and lists: same GrB_ALL / GxB_RANGE / GxB_STRIDE / GxB_BACKWARDS encoding, same result length."""
    import pygraphblas_b200 as gb
    v = gb.Vector.sparse(gb.INT64, 10)
    vals = [None, 0, 1, 3, 8, 9]
    steps = [None, 1, 2, 3, -1, -2, -3]
    ref = golden["slices"]
    assert len(ref["grid"]) == len(vals) ** 2 * len(steps)
    n = 0
    for (a, b, c), exp in zip(itertools.product(vals, vals, steps), ref["grid"]):
        sl = slice(a, b, c)
        I1, ni1, sz1 = v._index(sl, 10)
        if exp == "ALL":
            assert I1 == gb.lib.GrB_ALL and sz1 == 10, (sl,)
            continue
        ni0, I0, sz0 = exp
        assert ni0 == int(ni1), (sl, ni0, ni1)
        assert I0 == [int(I1[q]) for q in range(len(I0))], sl
        assert sz0 == sz1, (sl, sz0, sz1)
        n += 1
    assert n > 0
    I1, ni1, sz1 = v._index([2, 3, 5, 7], 10)
    ni0, I0, sz0 = ref["list"]
    assert (ni0, sz0) == (ni1, sz1) == (4, 4) and [int(I1[q]) for q in range(4)] == I0


def test_type_promotion_and_default_operators_match_the_reference(golden):
    """types.promote (types.py:484-500), the default semiring / add / mult operators per type (types.py:156-160)
    and every semiring's ztype, mirror against the reference's own objects."""
    import pygraphblas_b200 as gb
    ref = golden["types"]
    for a in NAMES:
        for b in NAMES:
            assert ref["promote"][a][b] == gb.types.promote(getattr(gb, a), getattr(gb, b)).name, (a, b)
        ga = getattr(gb, a)
        assert ref["defaults"][a] == [ga._default_semiring().name, ga._default_addop().name, ga._default_multop().name], a
    n = 0
    for name, ztype in ref["semiring_ztypes"].items():
        assert gb.ops.semirings[name].ztype.name == ztype, name
        n += 1
    assert n > 1000, n


INFERENCE = """
    import importlib, itertools, json
    import pygraphblas_b200 as gb
    pkg = importlib.import_module(PKG)
    importlib.import_module(PKG + ".matrix"); importlib.import_module(PKG + ".vector")

    class Recorder:
        def __init__(self, real, pkg):
            self._real, self._pkg, self.calls = real, pkg, []
        def __getattr__(self, name):
            if name in ("GrB_mxm", "GrB_mxv", "GrB_vxm"):
                def rec(out, mask, accum, semiring, a, b, desc):
                    self.calls.append((name, out, mask != self._real_null(), accum, semiring, desc))
                    return 0
                return rec
            return getattr(self._real, name)
        def _real_null(self):
            return self._pkg.base.NULL if hasattr(self._pkg, "base") else None

    rec = Recorder(pkg.lib, pkg)
    pkg.matrix.lib = rec; pkg.vector.lib = rec

    def name_of(pkg, kind, handle):
        ffi = pkg.ffi if hasattr(pkg, "ffi") else pkg.base.ffi
        if handle == ffi.NULL:
            return None
        p = ffi.new("char**")
        k = {"binop": 0, "semiring": 2}[kind]
        assert gb.lib.B200_object_name(gb.ffi.cast("const char**", p), k, gb.ffi.cast("void*", handle)) == 0
        return gb.ffi.string(gb.ffi.cast("char*", p[0])).decode()

    def desc_bits(pkg, d):
        ffi = pkg.ffi if hasattr(pkg, "ffi") else pkg.base.ffi
        if d == ffi.NULL:
            return (0, 0, 0, 0)
        out = []
        for f in (gb.lib.GrB_OUTP, gb.lib.GrB_MASK, gb.lib.GrB_INP0, gb.lib.GrB_INP1):
            v = gb.ffi.new("GrB_Desc_Value*")
            assert gb.lib.GxB_Desc_get(gb.ffi.cast("GrB_Descriptor", d), f, v) == 0
            out.append(int(v[0]))
        return tuple(out)

    def summarize(pkg, rec, result):
        name, out, has_mask, accum, semiring, desc = rec.calls[-1]
        typ = result.type.__name__ if hasattr(result.type, "__name__") else result.type.name
        shape = result.shape if hasattr(result, "nrows") else (result.size,)
        return (name, typ, tuple(int(x) for x in shape), has_mask, name_of(pkg, "binop", accum), name_of(pkg, "semiring", semiring), desc_bits(pkg, desc))

    types_ = ["BOOL", "INT8", "INT64", "UINT16", "FP32", "FP64"]
    res = []
    for ta, tb in itertools.product(types_, types_):
        for variant in range(8):
            A = pkg.Matrix.sparse(getattr(pkg, ta), 3, 5)
            B = pkg.Matrix.sparse(getattr(pkg, tb), 5, 4)
            Bt = pkg.Matrix.sparse(getattr(pkg, tb), 4, 5)
            At = pkg.Matrix.sparse(getattr(pkg, ta), 5, 3)
            u = pkg.Vector.sparse(getattr(pkg, tb), 5)
            u3 = pkg.Vector.sparse(getattr(pkg, tb), 3)
            T = getattr(pkg, ta)
            d = pkg.descriptor
            if variant == 0:
                out = A.mxm(B)
            elif variant == 1:
                out = A.mxm(Bt, desc=d.T1, semiring=T.MIN_PLUS if ta != "BOOL" else T.LOR_LAND)
            elif variant == 2:
                out = A.mxv(u, cast=pkg.FP64)
            elif variant == 3:
                # square operand: with a descriptor that does NOT transpose, the reference sizes the implicit output
                # by ncols (its Descriptor.__contains__ always answers True, descriptor.py:126-142) and then fails in
                # GrB_mxv on a non-square A; the mirror sizes it correctly -- the one deliberate deviation
                S = pkg.Matrix.sparse(getattr(pkg, ta), 5, 5)
                out = S.mxv(u, accum=pkg.INT64.MIN, mask=pkg.Vector.sparse(pkg.BOOL, 5), desc=d.RC)
            elif variant == 4:
                out = u3.vxm(A)
            elif variant == 5:
                with (T.PLUS_PLUS if ta != "BOOL" else T.LOR_LOR), pkg.Accum(pkg.FP32.PLUS):
                    out = A @ B
            elif variant == 6:
                out = u.vxm(A, desc=d.T1, semiring=pkg.INT64.PLUS_PAIR)
            else:
                with d.S:
                    out = A.mxm(B, mask=pkg.Matrix.sparse(pkg.BOOL, 3, 4), cast=pkg.UINT8)
            res.append([ta, tb, variant, summarize(pkg, rec, out)])
    print(json.dumps(res))
"""


def test_output_inference_of_the_hot_calls_matches_the_reference(golden):
    """Rows a1-a4: what Matrix.mxm / Matrix.mxv / Vector.vxm decide on the host before the FFI call -- type and
    shape of an implicit output, the semiring actually passed, accumulator / descriptor from the context managers
    (matrix.py:2553-2584, 2693-2726, vector.py:942-971, matrix.py:2380-2399).  The mirror runs with the three hot
    entry points replaced by a recorder, so nothing computes; its recorded calls must agree with the reference's."""
    ref = golden["inference"]
    got = run_snippet(INFERENCE, "pygraphblas_b200")
    assert len(ref) == len(got) == 6 * 6 * 8
    bad = [(r, g) for r, g in zip(ref, got) if r != g]
    assert not bad, bad[:5]


FFI_CASES = r'''
MASKS={}
v=lambda p,t="INT64": p.Vector.from_lists([0,2,5],[1,2,3],8,getattr(p,t))
w=lambda p,t="INT64": p.Vector.from_lists([0,1,2,6],[1,2,3,4],8,getattr(p,t))
m=lambda p,t="INT64": p.Matrix.from_lists([0,1,2],[1,2,0],[1,2,3],4,4,getattr(p,t))
m2=lambda p,t="INT64": p.Matrix.from_lists([0,1,2,3,3],[1,2,0,0,3],[1,2,3,4,5],4,4,getattr(p,t))
bmask=lambda p: p.Vector.from_lists([0,2],[True,False],8,p.BOOL)
cases={
 "eadd": lambda p: v(p).eadd(w(p)), "eadd_max": lambda p: v(p).eadd(w(p), p.INT64.MAX), "eadd_mon": lambda p: v(p).eadd(w(p), p.INT64.PLUS_MONOID),
 "or": lambda p: v(p) | w(p), "add": lambda p: v(p) + w(p), "sub": lambda p: v(p) - w(p), "mul": lambda p: v(p) * w(p), "div": lambda p: v(p) / w(p),
 "and": lambda p: v(p) & w(p), "emult": lambda p: v(p).emult(w(p)), "emult_mixed": lambda p: v(p,"FP32").emult(v(p,"INT8")),
 "apply": lambda p: v(p).apply(p.INT64.AINV), "neg": lambda p: -v(p), "abs": lambda p: abs(v(p)), "inv": lambda p: ~v(p,"FP64"),
 "first": lambda p: v(p).apply_first(2, p.INT64.PLUS), "second": lambda p: v(p).apply_second(p.INT64.MINUS, 2),
 "add3": lambda p: v(p) + 3, "radd3": lambda p: 3 + v(p), "rsub": lambda p: 3 - v(p), "sub3": lambda p: v(p) - 3, "mul3": lambda p: v(p) * 3, "rmul": lambda p: 3 * v(p),
 "div3": lambda p: v(p) / 3, "rdiv": lambda p: 15 / v(p), "mulf": lambda p: v(p,"FP64") * 2.5,
 "iadd": lambda p: v(p).__iadd__(3), "iaddv": lambda p: v(p).__iadd__(w(p)), "isub": lambda p: v(p).__isub__(3), "isubv": lambda p: v(p).__isub__(w(p)),
 "imul": lambda p: v(p).__imul__(3), "imulv": lambda p: v(p).__imul__(w(p)), "idiv": lambda p: v(p).__itruediv__(3), "idivv": lambda p: v(p).__itruediv__(w(p)),
 "ior": lambda p: v(p).__ior__(w(p)), "iand": lambda p: v(p).__iand__(w(p)),
 "assign_scalar": lambda p: v(p).assign_scalar(3), "assign_scalar_f": lambda p: v(p).assign_scalar(2.5), "assign_scalar_mask": lambda p: v(p,"UINT8").assign_scalar(2, mask=MASKS.setdefault(p.__name__, bmask(p))),
 "setall": lambda p: v(p).__setitem__(slice(None), 3), "setslice": lambda p: v(p).__setitem__(slice(2,7), 1), "setmask": lambda p: v(p).__setitem__(MASKS.setdefault(p.__name__, bmask(p)), 4),
 "setvec": lambda p: v(p).__setitem__(slice(None), w(p)), "assign": lambda p: v(p).assign(w(p)), "getslice": lambda p: v(p)[1:5], "getstride": lambda p: v(p)[7:1:-2], "getlist": lambda p: v(p)[[2,3,5]],
 "reduce_int": lambda p: v(p).reduce_int(), "reduce_bool": lambda p: p.Vector.from_lists([0,2],[True,False],8,p.BOOL).reduce_bool(), "reduce_float": lambda p: v(p,"FP64").reduce_float(), "reduce_int_mon": lambda p: v(p).reduce_int(p.INT64.MAX_MONOID),
 "pattern": lambda p: v(p).pattern(), "pattern8": lambda p: v(p).pattern(p.INT8),
 "nonzero": lambda p: v(p).nonzero(), "select_gt": lambda p: v(p).select(">", 1),
 "m_tril": lambda p: m(p).tril(), "m_triu1": lambda p: m(p).triu(1), "m_offdiag": lambda p: m(p).offdiag(), "m_nonzero": lambda p: m(p).nonzero(),
 "m_select_gt": lambda p: m(p).select(">", 2), "m_select_op": lambda p: m(p).select(p.lib.GxB_TRIL, -1),
 "m_apply": lambda p: m(p).apply(p.INT64.ABS), "m_neg": lambda p: -m(p), "m_first": lambda p: m(p).apply_first(2, p.INT64.PLUS), "m_second": lambda p: m(p).apply_second(p.INT64.TIMES, 3),
 "m_reduce_int": lambda p: m(p).reduce_int(), "m_reduce_float": lambda p: m(p,"FP64").reduce_float(), "m_reduce_bool": lambda p: p.Matrix.from_lists([0,1],[1,0],[True,False],4,4,p.BOOL).reduce_bool(), "m_reduce_vector": lambda p: m(p).reduce_vector(),
 "m_reduce_vector_T0": lambda p: m(p).reduce_vector(desc=p.descriptor.T0),
 "m_eadd": lambda p: m(p).eadd(m2(p)), "m_add": lambda p: m(p) + m2(p), "m_sub": lambda p: m(p) - m2(p), "m_emult": lambda p: m(p).emult(m2(p)), "m_mul": lambda p: m(p) * m2(p), "m_div": lambda p: m(p) / m2(p),
 "m_or": lambda p: m(p) | m2(p), "m_and": lambda p: m(p) & m2(p), "m_pattern": lambda p: m(p).pattern(), "m_add3": lambda p: m(p) + 3, "m_mul3": lambda p: m(p) * 3,
 "m_iadd": lambda p: m(p).__iadd__(m2(p)), "m_isub": lambda p: m(p).__isub__(m2(p)), "m_imul": lambda p: m(p).__imul__(m2(p)), "m_idiv": lambda p: m(p).__itruediv__(m2(p)), "m_ior": lambda p: m(p).__ior__(m2(p)), "m_iand": lambda p: m(p).__iand__(m2(p)), "m_iadd3": lambda p: m(p).__iadd__(3), "m_isub3": lambda p: m(p).__isub__(3), "m_imul3": lambda p: m(p).__imul__(3), "m_idiv3": lambda p: m(p).__itruediv__(3), "m_radd": lambda p: 3 + m(p), "m_rsub": lambda p: 3 - m(p), "m_rmul": lambda p: 3 * m(p), "m_rdiv": lambda p: 12 / m(p), "m_inv": lambda p: ~m(p,"FP64"), "m_abs": lambda p: abs(m(p)),
 "m_transpose": lambda p: m(p).transpose(), "m_T": lambda p: m(p).T,
}

cases.update({
 # operators taken from context managers, string operators, Scalar operands, masks / accumulators / descriptors
 "ctx_binop": lambda p: _with(p.INT64.MAX, lambda: v(p) | w(p)), "ctx_binop_m": lambda p: _with(p.INT64.MIN, lambda: m(p) + m2(p)),
 "ctx_monoid": lambda p: _with(p.INT64.TIMES_MONOID, lambda: v(p).reduce_int()), "ctx_monoid_m": lambda p: _with(p.FP64.MAX_MONOID, lambda: m(p, "FP64").reduce_float()),
 "ctx_accum": lambda p: _with(p.Accum(p.INT64.MIN), lambda: v(p).eadd(w(p), out=v(p))),
 "str_op": lambda p: v(p).emult(w(p), "+"), "str_op2": lambda p: m(p).emult(m2(p), ">="),
 "scalar_first": lambda p: v(p).apply_first(MASKS.setdefault(p.__name__ + "s", p.Scalar.from_value(2)), p.INT8.PLUS),
 "scalar_second": lambda p: m(p).apply_second(p.INT8.MINUS, MASKS.setdefault(p.__name__ + "s", p.Scalar.from_value(2))),
 "eadd_full": lambda p: v(p).eadd(w(p), p.INT64.MIN, out=w(p), mask=MASKS.setdefault(p.__name__ + "2", bmask(p)), accum=p.INT64.PLUS, desc=p.descriptor.RSC),
 "m_eadd_T": lambda p: m(p).eadd(m2(p), p.INT64.MAX, desc=p.descriptor.T0T1), "m_select_desc": lambda p: m(p).select("<", 3, desc=p.descriptor.T0),
 "cast": lambda p: v(p).eadd(w(p), cast=p.FP32), "m_cast": lambda p: m(p).emult(m2(p, "FP32"), cast=p.FP64),
})
'''


FFI = """
    import importlib, json, sys
    sys.path.insert(0, TESTS)
    from ffi_recorder import run      # replaces the library's compute entry points before PKG binds them
    pkg = importlib.import_module(PKG)
    def _with(cm, fn):
        with cm:
            return fn()
    exec(FFI_CASES)
    print(json.dumps({k: run(fn, pkg) for k, fn in cases.items()}))
"""


def test_every_operation_makes_the_same_ffi_call_as_the_reference(golden):
    """Rows (f)1 / (f)3 host logic: for ~110 user-level expressions on vectors and matrices (eadd / emult / apply /
    assign / extract / reduce / select / pattern / transpose, every arithmetic operator incl. the reflected and in-place
    forms, operators from `with` contexts and strings, Scalar operands, masks, accumulators, descriptors, casts) the
    mirror hands the C ABI the same function, operator handles, operands (in the same order), scalars, index lists and
    descriptor as the unmodified reference does.  Nothing computes: the mirror runs on the recorder of tests/ffi_recorder.py."""
    ref = golden["ffi_calls"]
    got = run_snippet(f"FFI_CASES = {FFI_CASES!r}\n" + textwrap.dedent(FFI), "pygraphblas_b200")
    assert sorted(ref) == sorted(got)
    bad = []
    for k in ref:
        a, b = ref[k], got[k]
        if a != b:
            bad.append((k, a, b))
        elif a[:1] == ["EXC"] and k != "m_inv":
            bad.append((k, "raises in both", a))
    assert not bad, bad
