#!/usr/bin/env python
"""Record what the reference package decides on the host, for tests/test_reference_dropin.py.

    python tests/golden/make_dropin_goldens.py PATH_TO_PYGRAPHBLAS_CHECKOUT

Runs the UNMODIFIED reference (Graphegon/pygraphblas, the directory that holds its `pygraphblas/` package) over the
binding stub `suitesparse_graphblas/` of this repository, on a build of libb200grb.so (no GPU needed: nothing here
computes), and writes tests/golden/reference_dropin.json:

    binding     every name the reference reads from suitesparse_graphblas.lib while it imports and does basic handle
                plumbing, and the results of that plumbing
    slices      its index encoding of slices and index lists (base._build_range)
    types       its type promotion, default operators per type and the ztype of every semiring the mirror defines
    inference   type / shape / operators / descriptor of the implicit outputs of mxm / mxv / vxm
    ffi_calls   the C calls its user-level expressions make

The last two run the same code as the tests do (INFERENCE and FFI of tests/test_reference_dropin.py).
"""
import importlib.util
import json
import os
import sys
import textwrap

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))

BINDING = """
    import importlib.util, json, os, sys
    spec = importlib.util.spec_from_file_location("pygraphblas_b200._ffi", os.path.join(%r, "pygraphblas_b200", "_ffi.py"))
    _ffi = importlib.util.module_from_spec(spec); sys.modules["pygraphblas_b200._ffi"] = _ffi; spec.loader.exec_module(_ffi)
    real, seen = _ffi.lib, set()

    class Names:
        def __dir__(self):
            return dir(real)
        def __getattr__(self, name):
            seen.add(name)
            return getattr(real, name)

    _ffi.lib = Names()                 # before the reference binds suitesparse_graphblas.lib
    import pygraphblas as gb
    from pygraphblas import Matrix, Vector, Scalar, INT64, BOOL, descriptor, lib
    assert os.path.realpath(gb.__file__).startswith(os.path.realpath(REF)), gb.__file__
    m = Matrix.from_lists([0, 1, 2], [1, 2, 0], [1, 2, 3])
    v = Vector.from_lists([0, 1, 2], [2, 3, 4])
    plumbing = {"implementation_major": int(lib.GxB_IMPLEMENTATION_MAJOR),
                "shape": [m.nrows, m.ncols, m.nvals], "type": m.type.__name__,
                "to_lists": m.to_lists(), "dup": m.dup().to_lists(), "vdup": v.dup().to_lists(),
                "ztypes": [INT64.PLUS_TIMES.ztype.__name__, BOOL.LOR_LAND.ztype.__name__], "min_plus_alias": INT64.min_plus is INT64.MIN_PLUS,
                "ct1": [descriptor.T1 in descriptor.CT1, descriptor.CT1 == (descriptor.C & descriptor.T1)],
                "scalar": Scalar.from_value(3)[0], "sparse_nrows": Matrix.sparse(INT64).nrows}
    for call in (lambda: m.mxv(v), lambda: v.vxm(m), lambda: m.mxm(m), lambda: m @ m,
                 lambda: m.iseq(m.dup()), lambda: m.reduce_int(), lambda: v + v, lambda: m.tril(), lambda: v.apply(INT64.AINV)):
        try:
            call()
        except gb.base.Panic:
            pass
    print(json.dumps({"names": sorted(n for n in seen if hasattr(real, n)), "plumbing": plumbing}))
"""

SLICES = """
    import itertools, json
    from pygraphblas.base import _build_range, lib as rlib
    vals = [None, 0, 1, 3, 8, 9]
    steps = [None, 1, 2, 3, -1, -2, -3]
    grid = []
    for a, b, c in itertools.product(vals, vals, steps):
        I0, ni0, sz0 = _build_range(slice(a, b, c), 9)
        if I0 == rlib.GrB_ALL:
            grid.append("ALL")
            continue
        k = 2 if int(ni0) == int(rlib.GxB_RANGE) else 3
        grid.append([int(ni0), [int(I0[q]) for q in range(k)], int(sz0)])
    I0, ni0, sz0 = _build_range([2, 3, 5, 7], 9)
    print(json.dumps({"grid": grid, "list": [int(ni0), [int(x) for x in I0], int(sz0)]}))
"""

TYPES = """
    import json
    import pygraphblas as ref
    import pygraphblas_b200 as gb
    names = ["BOOL", "INT8", "INT16", "INT32", "INT64", "UINT8", "UINT16", "UINT32", "UINT64", "FP32", "FP64"]
    promote = {a: {b: ref.types.promote(getattr(ref, a), getattr(ref, b)).__name__ for b in names} for a in names}
    defaults = {}
    for a in names:
        ra = getattr(ref, a)
        defaults[a] = [ra._default_semiring().name, ra._default_addop().name, ra._default_multop().name]
    ztypes = {}
    for name, sr in gb.ops.semirings.items():
        rs = getattr(getattr(ref, sr.type), f"{sr.pls}_{sr.mul}", None)
        if rs is not None:
            ztypes[name] = rs.ztype.__name__
    print(json.dumps({"promote": promote, "defaults": defaults, "semiring_ztypes": ztypes}))
"""


def main(ref_dir):
    ref_dir = os.path.abspath(ref_dir)
    if not os.path.isdir(os.path.join(ref_dir, "pygraphblas")):
        raise SystemExit(f"{ref_dir} has no pygraphblas/ package")
    spec = importlib.util.spec_from_file_location("_dropin_tests", os.path.join(ROOT, "tests", "test_reference_dropin.py"))
    t = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(t)
    path = f"{ROOT}:{ref_dir}"
    run = lambda code: t.run_snippet(f"REF = {ref_dir!r}\n" + textwrap.dedent(code), "pygraphblas", pythonpath=path)
    out = {"reference": "Graphegon/pygraphblas @ 2d89301",
           "binding": run(BINDING % ROOT),
           "slices": run(SLICES),
           "types": run(TYPES),
           "inference": run(t.INFERENCE),
           "ffi_calls": run(f"FFI_CASES = {t.FFI_CASES!r}\n" + textwrap.dedent(t.FFI))}
    with open(os.path.join(HERE, "reference_dropin.json"), "w") as f:
        json.dump(out, f, separators=(",", ":"))
        f.write("\n")
    print(f"wrote {len(out['binding']['names'])} binding names, {len(out['slices']['grid'])} slices, "
          f"{len(out['types']['semiring_ztypes'])} semirings, {len(out['inference'])} inferred outputs, {len(out['ffi_calls'])} expressions")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
