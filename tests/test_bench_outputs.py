"""CPU: bench.py --dump-outputs helpers.  The Hessian written as COO triplets must be the device CSR's
entries (rows rebuilt from crow_indices, empty rows included), a seeded sample of them when they do not
fit, and the files together stay within bench.DUMP_BYTES."""
import os

import numpy as np
import scipy.sparse
import torch

import bench
import bench_ef


class _Model(object):
    def __init__(self, D):
        self.D = D

    def kl_tensor(self):
        return torch.tensor(1.25, dtype=torch.float64)

    def grad_tensor(self):
        return torch.arange(self.D, dtype=torch.float64)


class _CSR(object):
    """The accessors of GLMM.DeviceCSR over host tensors."""

    def __init__(self, m):
        self.crow_indices = torch.from_numpy(m.indptr.astype(np.int32))
        self.col_indices = torch.from_numpy(m.indices.astype(np.int32))
        self.values = torch.from_numpy(m.data)


def _matrix(D=400):
    m = scipy.sparse.random(D, D, density=0.03, random_state=4, format="lil")
    m[7, :] = 0                     # empty rows, the first and the last among them
    m[0, :] = 0
    m[D - 1, :] = 0
    m = m.tocsr()
    m.eliminate_zeros()
    m.sort_indices()
    return m


def _dump(tmp_path, m, budget, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", budget)
    out = bench.last_step_outputs(torch, _Model(m.shape[0]), _CSR(m))
    bench.write_outputs(str(tmp_path), out)
    files = sorted(os.listdir(tmp_path))
    assert files == sorted(n + ".npy" for n in ("kl", "grad", "hessian_row", "hessian_col", "hessian_value"))
    assert sum(os.path.getsize(os.path.join(tmp_path, f)) for f in files) <= budget
    r = {f[:-4]: np.load(os.path.join(tmp_path, f)) for f in files}
    assert all(a.dtype == np.float64 for a in r.values())
    return r


def test_dump_writes_every_hessian_entry_in_csr_order(tmp_path, monkeypatch):
    m = _matrix()
    r = _dump(tmp_path, m, bench.DUMP_BYTES, monkeypatch)
    coo = m.tocoo()
    assert np.array_equal(r["hessian_row"], coo.row) and np.array_equal(r["hessian_col"], coo.col)
    assert np.array_equal(r["hessian_value"], coo.data)
    assert r["kl"].tolist() == [1.25] and np.array_equal(r["grad"], np.arange(m.shape[0]))


def test_dump_samples_the_hessian_within_the_budget(tmp_path, monkeypatch):
    m = _matrix()
    budget = 8 * (m.shape[0] + 1) + 4096 + 24 * (m.nnz // 4)
    r = _dump(tmp_path, m, budget, monkeypatch)
    n = r["hessian_value"].size
    assert 0 < n < m.nnz
    rows, cols = r["hessian_row"].astype(np.int64), r["hessian_col"].astype(np.int64)
    assert np.all(np.diff(rows * m.shape[1] + cols) > 0)          # distinct entries in CSR order
    assert np.array_equal(m.toarray()[rows, cols], r["hessian_value"])
    again = bench.last_step_outputs(torch, _Model(m.shape[0]), _CSR(m))
    assert np.array_equal(again["hessian_row"], r["hessian_row"])  # same positions from run to run


def test_ef_factor_sample_is_fixed_and_fits():
    a, b = bench_ef.sample_factors(10), bench_ef.sample_factors(10)
    assert np.array_equal(a, b)
    assert np.all(np.diff(a) > 0) and a[0] >= 0 and a[-1] < bench_ef.M
    assert 8 * 10 * a.size + 4096 <= bench.DUMP_BYTES
