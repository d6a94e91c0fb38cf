"""The benchmarked SpMV step (prep -> hot-table run kernel -> fix-up list) against the plain run kernel, bit for bit.

Both paths fold the entries of a run in the same order and combine the rows that cross runs with the same fix-up, so on
float data their results must be identical to the last bit; the hot kernel also writes T's presence bytes and the
values of the empty rows itself, which the stale in-place test checks on the raw dense export."""
import functools
import os

import numpy as np
import pytest

import pygraphblas_b200 as gb
from pygraphblas_b200 import Matrix, Vector, FP32, FP64, INT64, BOOL, descriptor
from pygraphblas_b200.generators import rmat_csr

pytestmark = pytest.mark.gpu
RUN = 256


def _with_hot(value):
    """Run a body with B200GRB_SPMV_HOT set (None: unset), restoring the caller's setting."""
    def deco(fn):
        @functools.wraps(fn)
        def wrapped(*a, **k):
            old = os.environ.get("B200GRB_SPMV_HOT")
            if value is None:
                os.environ.pop("B200GRB_SPMV_HOT", None)
            else:
                os.environ["B200GRB_SPMV_HOT"] = value
            gb.lib.B200_reload_tunables()
            try:
                return fn(*a, **k)
            finally:
                if old is None:
                    os.environ.pop("B200GRB_SPMV_HOT", None)
                else:
                    os.environ["B200GRB_SPMV_HOT"] = old
                gb.lib.B200_reload_tunables()
        return wrapped
    return deco


def _csr_from_pairs(nrows, ncols, r, c):
    key = np.unique(r.astype(np.int64) * ncols + c)
    r, c = key // ncols, (key % ncols).astype(np.uint32)
    indptr = np.zeros(nrows + 1, np.int64)
    np.cumsum(np.bincount(r, minlength=nrows), out=indptr[1:])
    return indptr, c


def _skewed_cols(rng, k, ncols):
    # a few columns take most of the references (as in R-MAT), so the hot-column plan has something to rank
    return np.minimum((rng.pareto(1.2, k) * 50).astype(np.int64), ncols - 1)


@functools.lru_cache(maxsize=None)
def _matrix(kind):
    """(nrows, ncols, indptr, indices) of the R-MAT s17 graph or of a crafted matrix; all have >= 2^20 entries and
    >= 2^16 rows and columns, so both orientations can take the hot-table kernel."""
    rng = np.random.default_rng(23)
    if kind == "rmat17":
        n, indptr, indices = rmat_csr(17, 16, 1)
        return n, n, np.asarray(indptr, np.int64), np.asarray(indices, np.uint32)
    if kind == "empty_ends":
        # rows 0..2999 and the last 4000 rows are empty (rowptr == nnz at the end), scattered empty rows in between
        nrows, ncols = 150_000, 100_000
        deg = rng.integers(0, 21, nrows)
        deg[:3000] = 0
        deg[-4000:] = 0
        r = np.repeat(np.arange(nrows), deg)
        indptr, indices = _csr_from_pairs(nrows, ncols, r, _skewed_cols(rng, len(r), ncols))
    elif kind == "long_row":
        # row 5 holds 2000 runs and a bit more, among short rows
        nrows, ncols = 70_000, 600_000
        deg = rng.integers(0, 21, nrows)
        r = np.repeat(np.arange(nrows), deg)
        c = _skewed_cols(rng, len(r), ncols)
        long_c = rng.choice(ncols, 2000 * RUN + 100, replace=False)
        indptr, indices = _csr_from_pairs(nrows, ncols, np.concatenate([r, np.full(len(long_c), 5)]), np.concatenate([c, long_c]))
        assert indptr[6] - indptr[5] >= 2000 * RUN
    elif kind == "run_aligned":
        # many rows end exactly on a run boundary: 256-long rows, (100, 156) pairs and 512-long rows from offset 0
        nrows, ncols = 80_000, 80_000
        deg = np.concatenate([np.full(2000, 256), np.tile([100, 156], 1000), np.full(500, 512), rng.integers(0, 9, nrows - 4500)])
        indptr = np.zeros(nrows + 1, np.int64)
        np.cumsum(deg, out=indptr[1:])
        indices = np.concatenate([np.sort(rng.choice(ncols, d, replace=False)) for d in deg]).astype(np.uint32)
        assert np.count_nonzero(indptr[1:4501] % RUN == 0) >= 3000
    else:
        raise ValueError(kind)
    if indptr[-1] % RUN == 0:                  # keep a partial last run
        indptr = indptr.copy()
        indptr[-1] -= 1
        indices = indices[:-1]
    assert indptr[-1] % RUN != 0 and indptr[-1] >= 1 << 20
    return nrows, ncols, indptr, indices


CASES = {
    "fp32_plus_times": (FP32, "PLUS_TIMES", None),
    "fp32_min_plus_t0": (FP32, "MIN_PLUS", "T0"),
    "fp64_plus_times": (FP64, "PLUS_TIMES", None),
    "int64_plus_times": (INT64, "PLUS_TIMES", None),
    "bool_lor_land": (BOOL, "LOR_LAND", None),
}


def _operands(kind, case):
    nrows, ncols, indptr, indices = _matrix(kind)
    typ, sr, desc = CASES[case]
    rng = np.random.default_rng(7)
    nnz = len(indices)
    if typ is BOOL:
        vals, u = rng.random(nnz) < 0.7, rng.random(nrows if desc else ncols) < 0.5
    elif typ is INT64:
        vals, u = rng.integers(-1000, 1000, nnz), rng.integers(-1000, 1000, nrows if desc else ncols)
    else:                                      # full-mantissa floats: a different association order shows in the last bits
        vals, u = rng.standard_normal(nnz), rng.standard_normal(nrows if desc else ncols)
    A = Matrix.from_csr(indptr, indices, vals.astype(typ.dtype), nrows, ncols, typ)
    return A, u.astype(typ.dtype), getattr(typ, sr), getattr(descriptor, desc) if desc else None


def _step(A, u, semiring, desc):
    """the second of two calls (the first builds the plans): result and kernel launches of the call"""
    A.mxv(Vector.from_numpy(u), semiring=semiring, desc=desc)
    uv = Vector.from_numpy(u)
    before = gb.lib.B200_kernel_launches()
    w = A.mxv(uv, semiring=semiring, desc=desc)
    x, p = w.to_numpy()
    return x, p, gb.lib.B200_kernel_launches() - before


@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("kind", ["rmat17", "empty_ends", "long_row", "run_aligned"])
def test_hot_step_equals_plain_run_kernel_bitwise(kind, case):
    A, u, semiring, desc = _operands(kind, case)
    x_hot, p_hot, n_hot = _with_hot("64")(_step)(A, u, semiring, desc)
    x_run, p_run, n_run = _with_hot("0")(_step)(A, u, semiring, desc)
    assert n_hot == n_run + 1                  # prep + hot-table kernel + fix-up against run kernel + fix-up
    assert np.array_equal(p_hot, p_run)
    assert x_hot.tobytes() == x_run.tobytes()
    nrows, ncols, indptr, _ = _matrix(kind)
    if desc is None:                           # presence is structural (u is dense): the non-empty rows
        assert np.array_equal(p_hot != 0, np.diff(indptr) > 0)
    assert not np.any(x_hot[p_hot == 0])


@_with_hot("64")
def test_stale_in_place_w_is_cleared_on_empty_rows():
    nrows, ncols, indptr, indices = _matrix("empty_ends")
    rng = np.random.default_rng(5)
    A = Matrix.from_csr(indptr, indices, rng.standard_normal(len(indices)).astype(np.float32), nrows, ncols, FP32)
    # another matrix with every row non-empty and positive entries: w starts fully present with non-zero values
    bcols = ((np.arange(nrows) * 8) % (ncols - 8))[:, None] + np.arange(8)
    B = Matrix.from_csr(np.arange(nrows + 1, dtype=np.int64) * 8, bcols.ravel().astype(np.uint32),
                        np.ones(nrows * 8, np.float32), nrows, ncols, FP32)
    u = Vector.from_numpy((rng.random(ncols) + 0.5).astype(np.float32))
    w = B.mxv(u, semiring=FP32.PLUS_TIMES)
    x, p = w.to_numpy()
    assert np.all(p == 1) and np.all(x != 0)
    A.mxv(u, semiring=FP32.PLUS_TIMES, out=w)
    x, p = w.to_numpy()
    empty = np.diff(indptr) == 0
    assert np.all(p[empty] == 0) and np.all(x[empty] == 0)
    assert np.all(p[~empty] == 1)
    ref = _with_hot("0")(lambda: A.mxv(u, semiring=FP32.PLUS_TIMES).to_numpy())()
    assert x.tobytes() == ref[0].tobytes() and np.array_equal(p, ref[1])


@_with_hot("64")
def test_hot_step_is_deterministic():
    A, u, semiring, desc = _operands("rmat17", "fp32_plus_times")
    uv = Vector.from_numpy(u)
    first = None
    for _ in range(20):
        x, p = A.mxv(uv, semiring=semiring).to_numpy()
        if first is None:
            first = (x.tobytes(), p.tobytes())
        assert (x.tobytes(), p.tobytes()) == first
