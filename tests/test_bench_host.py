"""Host-side logic of bench.py that needs no GPU: the row-panel plan and the closed-form checksum of the streamed unmasked
SpGEMM (bench_spgemm_unmasked_streamed), checked against scipy at a small scale; the workload dict both arms must share."""
import os
import sys

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import bench


def _graph(scale=10):
    n, indptr, indices = bench._generators().rmat_csr(scale, 8, seed=3)
    vals = (np.random.default_rng(5).integers(1, 5, len(indices)) / 4.0).astype(np.float32)
    return n, indptr, indices, vals


def test_streamed_plan_covers_every_row_and_respects_the_cap():
    n, indptr, indices, vals = _graph()
    rowlen = np.diff(indptr)
    fl = np.add.reduceat(np.concatenate((rowlen[indices], [0])), np.minimum(indptr[:-1], len(indices))) * (rowlen > 0)
    for cap in (1.0, 500.0, 2e4, 1e12):
        cuts, total, _ = bench.streamed_plan(n, indptr, indices, vals, cap)
        assert cuts[0] == 0 and cuts[-1] == n and all(b > a for a, b in zip(cuts, cuts[1:]))
        assert total == int(fl.sum())
        for a, b in zip(cuts, cuts[1:]):
            assert fl[a:b].sum() <= cap or b == a + 1          # a single row may exceed the cap, a longer panel may not
    assert len(bench.streamed_plan(n, indptr, indices, vals, 1e12)[0]) == 2


def test_streamed_closed_form_is_the_sum_of_the_product():
    n, indptr, indices, vals = _graph()
    A = sp.csr_matrix((vals, indices, indptr), shape=(n, n))
    P = sp.csr_matrix((np.ones(len(indices), np.float32), indices, indptr), shape=(n, n))
    C = (P @ A).tocsr()                                        # PLUS_SECOND: sum over k in A(i,:) of A(k,j)
    _, total, expect = bench.streamed_plan(n, indptr, indices, vals, 1e9)
    assert expect == float(C.data.astype(np.float64).sum())
    assert total == int((P @ sp.csr_matrix((np.ones(len(indices)), indices, indptr), shape=(n, n))).sum())


def test_streamed_sample_is_a_row_subset_of_the_parent():
    n, indptr, indices, vals = _graph()
    S, ptr, take = bench.streamed_sample(n, indptr)
    assert len(S) >= 1 and ptr[0] == 0 and ptr[-1] == len(take) and np.all(np.diff(S) > 0)
    A = sp.csr_matrix((vals, indices, indptr), shape=(n, n))
    As = sp.csr_matrix((vals[take], indices[take], ptr), shape=(len(S), n))
    assert (As != A[S]).nnz == 0


def test_both_arms_share_one_workload_dict():
    a = bench.workload_config(22, 1 << 22, 65242949)
    assert a == bench.workload_config(22, 1 << 22, 65242949) and "workload" in a and "model" not in a


def test_dump_outputs_writes_the_result_vector_within_the_size_limit(tmp_path):
    rng = np.random.default_rng(1)
    x, present = rng.random(1000, dtype=np.float32), (rng.random(1000) < 0.5).astype(np.uint8)
    bench.dump_outputs(str(tmp_path / "full"), x, present)
    w, p = np.load(tmp_path / "full" / "w_values.npy"), np.load(tmp_path / "full" / "w_present.npy")
    assert w.dtype == p.dtype == np.float32 and not os.path.exists(tmp_path / "full" / "w_rows.npy")
    assert np.array_equal(p, present.astype(np.float32)) and np.array_equal(w, np.where(present != 0, x, 0))
    # above the limit: the same seeded sample of rows every time
    n = bench.DUMP_BYTES // 8 + 1000
    x, present = np.arange(n, dtype=np.float32), np.ones(n, np.uint8)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), x, present)
    sizes = sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a"))
    assert sizes <= bench.DUMP_BYTES
    rows = np.load(tmp_path / "a" / "w_rows.npy")
    assert rows.dtype == np.float64 and np.array_equal(rows, np.load(tmp_path / "b" / "w_rows.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "w_values.npy"), rows.astype(np.float32))
