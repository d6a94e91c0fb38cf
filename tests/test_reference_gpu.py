"""The reference's hot-path unit tests on the B200, from their golden vectors.  The reference (Graphegon/pygraphblas)
holds literal inputs and expected outputs in the tests of its hot path -- test_mxm, test_mxm_context, test_mxv,
test_pow, test_promotion, test_matrix_transpose, test_dense, test_vxm, test_RC, test_RCT0, test_descriptor
(tests/test_matrix.py:249-330, 829-864, 1017-1028; test_vector.py:298-315; test_descriptor.py:6-30).  Those values are
kept in tests/golden/reference_goldens.json (tests/golden/make_goldens.py) or, for the forms that are not a single
mxm / mxv / vxm, below; here they run on libb200grb.so through the host-side mirror and through
suitesparse_graphblas/, the binding module the reference imports (INTEGRATION.md)."""
import os
import subprocess
import sys

import numpy as np
import pytest

import util

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

HOT = ["test_matrix.py::test_mxm", "test_matrix.py::test_mxm_context", "test_matrix.py::test_mxv", "test_matrix.py::test_pow",
       "test_matrix.py::test_promotion", "test_matrix.py::test_matrix_transpose", "test_matrix.py::test_dense",
       "test_vector.py::test_vxm", "test_descriptor.py::test_RC", "test_descriptor.py::test_RCT0", "test_descriptor.py::test_descriptor"]


def test_reference_hot_path_tests_pass_unchanged_on_the_gpu(goldens):
    import pygraphblas_b200 as gb
    from pygraphblas_b200 import Matrix, UINT8, descriptor, lib
    passed = set()
    # the single-call cases, with their expected values as the reference's tests state them
    for case in goldens["cases"]:
        if not case["source"].startswith("tests/"):
            continue
        if case["id"] == "test_mxm_imatmul_alias":
            case = dict(case); case["C"] = case["A"]        # m @= n: C aliases A
        if case["id"] in ("test_RCT0", "test_RC"):
            case = dict(case); case["w"] = case["u"]        # out aliases the input vector
        got = util.product_run(case)
        ok = util.same_mat(got, case["expect"]) if case["op"] == "mxm" else util.same_vec(got, case["expect"])
        assert ok, f"{case['id']} ({case['source']}): got {got}, expected {case['expect']}"
        name = "test_mxm_context" if "context" in case["id"] else "_".join(case["id"].split("_")[:2])
        passed.add(os.path.basename(case["source"].split(":")[0]) + "::" + name)
    # test_promotion (tests/test_matrix.py:1017-1028)
    for ta, tb, tout in goldens["known_answers"]["promotion"]["cases"]:
        a = Matrix.from_lists([0, 1], [0, 1], [4 if ta != "INT8" else -4, 2], typ=getattr(gb, ta))
        assert (a @ Matrix.from_lists([0, 1], [0, 1], [4, 2], typ=getattr(gb, tb))).type is getattr(gb, tout), (ta, tb)
    passed.add("test_matrix.py::test_promotion")
    # test_matrix_transpose (tests/test_matrix.py:318-325)
    v = Matrix.from_lists([2, 1, 0], [0, 1, 2], [0, 1, 2], nrows=3, ncols=4)
    assert v.transpose().iseq(Matrix.from_lists([0, 1, 2], [2, 1, 0], [0, 1, 2], nrows=4, ncols=3))
    # with T0 the reference makes its implicit output nrows x ncols (matrix.py:1044-1048); the mirror takes it as `out`
    assert v.transpose(out=Matrix.sparse(v.type, v.nrows, v.ncols), desc=descriptor.T0).iseq(v)
    passed.add("test_matrix.py::test_matrix_transpose")
    # test_dense / test_pow (tests/test_matrix.py:829-835, 858-864): a dense 10 x 10 UINT8 matrix and its powers
    I, J = np.repeat(np.arange(10), 10), np.tile(np.arange(10), 10)
    for fill in (0, 1):
        d = Matrix.from_lists(I, J, np.full(100, fill), typ=UINT8)
        assert len(d) == 100 and all(x[2] == fill for x in d)
    passed.add("test_matrix.py::test_dense")
    d = Matrix.from_lists(I, J, np.ones(100), typ=UINT8)
    # (the reference's d ** 0 is Matrix.identity built on the host, matrix.py:1723-1724: no library call to check)
    assert (d ** 1).iseq(d) and (d @ d).iseq(d ** 2)
    assert set((d ** 3).to_arrays()[2].tolist()) == {100}
    passed.add("test_matrix.py::test_pow")
    # test_descriptor (tests/test_descriptor.py:6-10)
    assert descriptor.T0 == descriptor.Descriptor(lib.GrB_DESC_T0, "T0") and descriptor.T1 != descriptor.T0
    assert descriptor.T1 in descriptor.CT1 and descriptor.CT1 == (descriptor.C & descriptor.T1)
    passed.add("test_descriptor.py::test_descriptor")
    assert passed == set(HOT), sorted(set(HOT) ^ passed)


def test_reference_mxv_runs_on_the_library_not_elsewhere():
    """The C call the reference's Matrix.mxv makes (GrB_mxv, matrix.py:2716), through the `lib` of suitesparse_graphblas/
    in a fresh interpreter, reaches libb200grb.so on the GPU (kernel launches counted) and gives the reference's result."""
    code = ("import os\n"
            "from suitesparse_graphblas import lib, ffi\n"
            "import pygraphblas_b200 as gb\n"
            "assert lib is gb.lib and os.path.realpath(gb.__file__).startswith(os.path.realpath(%r))\n"
            "assert lib.B200_have_device() == 1\n"
            "m = gb.Matrix.from_lists([0, 1, 2], [1, 2, 0], [1, 2, 3]); v = gb.Vector.from_lists([0, 1, 2], [2, 3, 4])\n"
            "w = gb.Vector.sparse(gb.INT64, 3)\n"
            "before = lib.B200_kernel_launches()\n"
            "assert lib.GrB_mxv(w._vector[0], ffi.NULL, ffi.NULL, gb.INT64.PLUS_TIMES.semiring, m._matrix[0], v._vector[0], ffi.NULL) == 0\n"
            "assert w.to_lists() == [[0, 1, 2], [3, 8, 6]], w.to_lists()\n"
            "assert lib.B200_kernel_launches() > before\n"
            "print('OK')\n") % ROOT
    env = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=os.path.join(ROOT, "tests"), timeout=600)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr
