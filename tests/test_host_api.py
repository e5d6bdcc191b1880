"""CPU: host-side mirror of the reference interface (packing, sparse helpers, CG helpers) and the
C-ABI boundary (library loads, exports every declared symbol, fails loudly without a GPU).
Follows the reference's own tests: test_variational_bayes.py:74-106, 282-310, 529-639, 839-883;
test_objectives.py:480-554."""
import os
import re

import numpy as np
import pytest
import scipy.sparse

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cabi_library_loads_and_exports_every_declared_symbol(vb):
    import subprocess
    import sys
    from lrvb_b200 import _native as nat
    lib = nat.load()
    header = open(os.path.join(ROOT, "include", "lrvb_b200.h")).read()
    declared = set(re.findall(r"\b(lrvb_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 30
    assert declared == set(nat.SIGNATURES), declared ^ set(nat.SIGNATURES)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.lrvb_version() >= 100
    # nothing launched: the launch counter is per process and GPU tests of this session may already have
    # launched kernels here, so the library is loaded and queried again in a fresh interpreter
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from lrvb_b200 import _native as nat\n"
            "lib = nat.load(); lib.lrvb_version(); print(lib.lrvb_launch_count())" % ROOT)
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable] + flags + ["-c", code], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.split()[-1] == "0", r.stdout


def test_no_cpu_fallback(vb):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    X = np.zeros((4, 2)); y = np.zeros(4); g = np.array([0, 0, 1, 1])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        vb.LogisticGLMM(X, y, g)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        vb.ExponentialFamilies.gamma_entropy(np.ones(3), np.ones(3))
    with pytest.raises(TypeError, match="device models only"):
        vb.Objective(vb.ModelParamsDict("p"), lambda: 0.0)


def test_transforms_against_reference_golden(vb):
    f = np.load(os.path.join(GOLD, "forward.npz"))
    fv = f["con_free"]
    grid = [(-np.inf, np.inf), (0.0, np.inf), (-1.5, np.inf), (-np.inf, 2.0), (-1.0, 3.0)]
    for i, (lb, ub) in enumerate(grid):
        c = vb.constrain(fv, lb, ub)
        np.testing.assert_allclose(c, f["con%d" % i], rtol=1e-15)
        np.testing.assert_allclose(vb.unconstrain(c, lb, ub), f["unc%d" % i], rtol=1e-13, atol=1e-15)
        np.testing.assert_allclose(vb.unconstrain(c, lb, ub), fv, rtol=1e-9, atol=1e-12)
    with pytest.raises(ValueError):
        vb.constrain(fv, 1.0, 1.0)


def build_par(vb, K, G, lb):
    par = vb.ModelParamsDict("glmm_par")
    par.push_param(vb.UVNParam("mu", min_info=lb))
    par.push_param(vb.GammaParam("tau", min_shape=lb, min_rate=lb))
    par.push_param(vb.UVNParamVector("beta", K, min_info=lb))
    par.push_param(vb.UVNParamVector("u", G, min_info=lb))
    return par


def test_model_params_dict_layout_against_reference_golden(vb):
    f = np.load(os.path.join(GOLD, "forward.npz"))
    par = build_par(vb, 3, 4, 0.25)
    x = f["pack_free"]
    par.set_free(x)
    np.testing.assert_allclose(par.get_vector(), f["pack_vector"], rtol=1e-15)
    np.testing.assert_allclose(par.get_free(), f["pack_free_back"], rtol=1e-12, atol=1e-14)
    assert [str(s) for s in par.names()] == [str(s) for s in f["pack_names"]]
    idx = np.array([[r.start, r.stop] for r in par.free_indices_dict.values()])
    np.testing.assert_array_equal(idx, f["pack_free_index"])
    np.testing.assert_allclose(par["u"].var(), f["pack_u_var"], rtol=1e-15)
    assert par.free_size() == par.vector_size() == 4 + 2 * 3 + 2 * 4
    with pytest.raises(ValueError, match="Wrong size"):
        par.set_free(np.zeros(3))
    with pytest.raises(ValueError, match="Wrong size"):
        par.set_vector(np.zeros(3))
    assert par.values["beta"]["mean"].size == 3 if hasattr(par.values["beta"], "__getitem__") else True
    assert set(par.dictval()) == {"mu", "tau", "beta", "u"}


def execute_required_methods(par):
    """The parameter protocol of test_variational_bayes.py:74-106."""
    par.names()
    par.dictval()
    par.set(par.get()) if hasattr(par, "set") else None
    free = par.get_free()
    par.set_free(free)
    vec = par.get_vector()
    par.set_vector(vec)
    assert free.size == par.free_size() and vec.size == par.vector_size()
    np.testing.assert_allclose(par.free_to_vector(free), vec)
    jac = par.free_to_vector_jac(free)
    hess = par.free_to_vector_hess(free)
    assert jac.shape == (par.vector_size(), par.free_size()) and len(hess) == par.vector_size()
    str(par)


def test_parameter_protocol_and_sparse_transforms(vb):
    rng = np.random.default_rng(42)
    pars = [vb.ScalarParam("s", lb=0.5, val=1.5), vb.ScalarParam("t"),
            vb.VectorParam("v", 4, lb=-1.0, ub=2.0), vb.VectorParam("w", 3, ub=0.0),
            vb.ArrayParam("a", shape=(2, 3), lb=0.1), build_par(vb, 2, 3, 0.1)]
    for par in pars:
        execute_required_methods(par)
        free = rng.normal(0, 0.5, par.free_size())
        jac = scipy.sparse.csr_matrix(par.free_to_vector_jac(free)).toarray()
        h = 1e-6
        for j in range(par.free_size()):
            e = np.zeros(par.free_size()); e[j] = h
            fd = (np.ravel(par.free_to_vector(free + e)) - np.ravel(par.free_to_vector(free - e))) / (2 * h)
            np.testing.assert_allclose(jac[:, j], fd, rtol=1e-6, atol=1e-8)
        hess = par.free_to_vector_hess(free)
        for i, hi in enumerate(hess):
            hi = scipy.sparse.csr_matrix(hi).toarray()
            assert hi.shape == (par.free_size(), par.free_size())
            for j in range(par.free_size()):
                e = np.zeros(par.free_size()); e[j] = h
                ja = scipy.sparse.csr_matrix(par.free_to_vector_jac(free + e)).toarray()[i]
                jb = scipy.sparse.csr_matrix(par.free_to_vector_jac(free - e)).toarray()[i]
                np.testing.assert_allclose(hi[:, j], (ja - jb) / (2 * h), rtol=1e-5, atol=1e-7)


def test_convert_vector_to_free_hessian(vb):
    """H_free = J^T H_vec J + sum_i g_i d2vec_i (Parameters.py:397-424) on a quadratic in vec."""
    par = build_par(vb, 2, 2, 0.2)
    rng = np.random.default_rng(1)
    n = par.vector_size()
    A = rng.standard_normal((n, n)); A = A @ A.T
    b = rng.standard_normal(n)
    free = rng.normal(0, 0.3, n)

    def f_free(x):
        v = par.free_to_vector(x)
        return 0.5 * v @ A @ v + b @ v
    vec = par.free_to_vector(free)
    Hf = vb.convert_vector_to_free_hessian(par, free, A @ vec + b, A)
    h = 1e-4
    fd = np.zeros((n, n))
    for i in range(n):
        for j in range(n):
            ei = np.zeros(n); ej = np.zeros(n); ei[i] = h; ej[j] = h
            fd[i, j] = (f_free(free + ei + ej) - f_free(free + ei - ej)
                        - f_free(free - ei + ej) + f_free(free - ei - ej)) / (4 * h * h)
    np.testing.assert_allclose(np.asarray(Hf), fd, rtol=1e-4, atol=1e-4 * np.abs(fd).max())
    Hs = vb.convert_vector_to_free_hessian(par, free, A @ vec + b, scipy.sparse.csr_matrix(A))
    assert scipy.sparse.issparse(Hs)
    np.testing.assert_allclose(Hs.toarray(), np.asarray(Hf), rtol=1e-12)


def test_sparse_sub_matrix_semantics(vb):
    sub = np.array([[1.0, 0.0, 2.0], [0.0, 0.0, 3.0]])
    m = vb.get_sparse_sub_matrix(sub, [3, 1], [4, 0, 2], 5, 6)
    assert m.nnz == 3                                   # exact zeros dropped (:613)
    assert m.indices.dtype == np.int32 and m.indptr.dtype == np.int32
    dense = np.zeros((5, 6)); dense[3, 4] = 1; dense[3, 2] = 2; dense[1, 2] = 3
    np.testing.assert_array_equal(m.toarray(), dense)
    d = vb.get_sparse_sub_matrix(np.array([[1.0, 2.0]]), [0], [1, 1], 2, 2)
    assert d.nnz == 1 and d[0, 1] == 3.0                # duplicates sum
    h = vb.get_sparse_sub_hessian(np.array([[1.0, 2.0], [2.0, 5.0]]), [2, 0], 3)
    np.testing.assert_array_equal(h.toarray(), [[5, 0, 2], [0, 0, 0], [2, 0, 1]])
    packed = vb.pack_csr_matrix(h)                      # test_objectives.py:480-491
    back = vb.unpack_csr_matrix(packed)
    assert (back != h).nnz == 0
    par = build_par(vb, 2, 3, 0.0)
    ip = vb.make_index_param(par)                       # test_objectives.py:494-509
    np.testing.assert_array_equal(ip.get_vector(), np.arange(par.vector_size()))
    np.testing.assert_array_equal(ip["u"]["info"].get(), [11, 12, 13])


def test_cg_mask_helpers_and_generic_solver(vb):
    cg = vb.ConjugateGradient
    masks = cg.get_masks(23, 5)                         # test_objectives.py:513-522
    assert np.all(np.sum(masks, axis=0) == 1) and len(masks) == 5
    a, b = cg.split_vector(np.array([True, False, True, True, False, True, True]))
    assert a.sum() == 2 and b.sum() == 3 and not np.any(a & b)
    res = cg.recursive_split(np.full(37, True), terminate_len=10)
    assert np.all(np.sum(res, axis=0) == 1) and max(m.sum() for m in res) <= 10
    # K = 50 SPD quadratic, masks of 10, |cg - cholesky| < 1e-8 (test_objectives.py:524-554)
    rng = np.random.default_rng(3)
    K = 50
    M = rng.standard_normal((K, K)); H = M @ M.T + K * np.eye(K)
    solver = vb.ConjugateGradientSolver(lambda x0, v: H @ v, np.zeros(K))
    vec = rng.standard_normal(K)
    solver.get_hinv_vec_subsets(vec, cg.get_masks(K, 10))
    for mask, hv, info in zip(solver.masks, solver.hinv_vecs, solver.cg_infos):
        vm = np.zeros(K); vm[mask] = vec[mask]
        assert info == 0
        assert np.max(np.abs(hv - np.linalg.solve(H, vm))) < 1e-8
    assert len(solver.times) == 5


def test_json_csr_wire_format_round_trip(vb):
    """SparseObjectives.py:639-657: the JSON dictionary of a CSR matrix survives json.dumps /
    loads bit-exactly and carries the json_tricks array layout the reference writes."""
    import json
    import scipy.sparse
    rng = np.random.default_rng(9)
    dense = rng.standard_normal((7, 5)) * (rng.random((7, 5)) < 0.4)
    m = scipy.sparse.csr_matrix(dense)
    packed = vb.json_pack_csr_matrix(m)
    assert packed["type"] == "csr_matrix"
    arr = json.loads(packed["data"])
    assert set(arr) >= {"__ndarray__", "dtype", "shape"} and arr["dtype"] == "float64"
    back = vb.json_unpack_csr_matrix(json.loads(json.dumps(packed)))
    assert back.shape == m.shape
    np.testing.assert_array_equal(back.indptr, m.indptr)
    np.testing.assert_array_equal(back.indices, m.indices)
    np.testing.assert_array_equal(back.data, m.data)
    assert back.indices.dtype == m.indices.dtype


def test_point_key_identity_semantics():
    """Evaluation points are remembered by value for numpy input and by identity + torch's in-place
    version counter for tensors (no device read-back): an in-place update must invalidate the key."""
    import torch
    from lrvb_b200._tensors import PointKey
    x = np.arange(5.0)
    k = PointKey(x)
    assert k.matches(x) and k.matches(x.copy())
    x[2] = 7.0
    assert not k.matches(x)              # the key holds its own copy
    t = torch.arange(5.0, dtype=torch.float64)
    kt = PointKey(t)
    assert kt.matches(t) and kt.matches(t.view(5))       # same storage, same version
    assert not kt.matches(t.clone())                     # equal values, another tensor: evaluated again
    assert not kt.matches(x)                             # kinds do not mix
    t.add_(1.0)
    assert not kt.matches(t)                             # in-place update bumps the version
    assert not PointKey(x).matches(t)


def test_ef_numeric_integration_helpers_host():
    """ExponentialFamilies.py:123-221 (Gauss-Hermite expectations of functions of normals, natural-parameter
    update, small priors): pure host arithmetic, checked against direct quadrature / closed forms as
    test_exponential_families.py:122-172 does."""
    import scipy.integrate
    import scipy.stats
    from lrvb_b200 import ExponentialFamilies as ef
    gx, gw = np.polynomial.hermite.hermgauss(40)
    means, infos = np.array([0.3, -1.2, 2.0]), np.array([2.0, 0.7, 5.0])
    got = ef.get_e_logitnormal(means, infos, gx, gw)
    el, el1 = ef.get_e_log_logitnormal(means, infos, gx, gw)
    for k in range(3):
        pdf = scipy.stats.norm(means[k], 1 / np.sqrt(infos[k])).pdf
        ref = scipy.integrate.quad(lambda x: pdf(x) / (1 + np.exp(-x)), -30, 30)[0]
        assert abs(got[k] - ref) < 1e-9
        ref_l = scipy.integrate.quad(lambda x: pdf(x) * -np.log1p(np.exp(-x)), -30, 30)[0]
        assert abs(el[k] - ref_l) < 1e-8
        assert abs(el1[k] - (ref_l - means[k])) < 1e-8
    sq = ef.get_e_fun_normal(means, infos, gx, gw, lambda x: x ** 2)
    np.testing.assert_allclose(sq, means ** 2 + 1 / infos, rtol=1e-12)
    m, i = ef.get_uvn_from_natural_parameters(1.5, -2.0)
    assert (m, i) == (1.5 / 4.0, 4.0)
    assert ef.exponential_prior(2.0, 3.0) == -6.0
    assert abs(ef.dirichlet_prior(np.array([2.0, 3.0]), np.array([-1.0, -0.5])) - (-1.0 - 1.0)) < 1e-15
    dp = ef.get_e_dp_prior_logitnorm_approx(3.0, means, infos, gx, gw)
    np.testing.assert_allclose(dp, 2.0 * el1)


def test_gram_wide_plan_covers_every_packed_tile_once(tmp_path):
    """The host planner of k_gram_wide (csrc/gram_wide.cuh): for every K it can serve (96 .. 256, K % 8 == 0)
    each tile (i <= j) of the packed [x | s] triangle belongs to exactly one warp job, the staged column
    offsets of a job point at blocks with the right X columns / class, the weight row follows the classes,
    and every job group fits its shared-memory budget.  Host-only: the checker is compiled with nvcc here and
    launches nothing."""
    import shutil
    import subprocess
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "gwplan")
    subprocess.run([nvcc, "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe,
                    os.path.join(root, "tools", "gram_wide_plan_check.cu")], check=True, capture_output=True)
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout[-2000:]
    assert "plan ok" in out.stdout
    assert "K=200 T2=50 groups= 7 ctas=148 live=1275" in out.stdout


def _k_ranges(ks):
    """[53, 54, 55, 64] -> '53..55, 64'"""
    ks, out = sorted(ks), []
    lo = hi = ks[0]
    for k in ks[1:] + [None]:
        if k == hi + 1:
            hi = k
            continue
        out.append(str(lo) if lo == hi else "%d..%d" % (lo, hi))
        lo = hi = k
    return ", ".join(out)


def test_dispatch_cases_reach_every_kernel_class(tmp_path):
    """The parity cases (CASES of test_gpu_glmm_parity.py) run every kernel an evaluation can pick: every
    compiled instantiation of k_fused_eval and k_gram_mid, every k_gram_big plan (job groups, rows per stage,
    straddle tile) and K = kMaxK, both column-chunk counts of k_obs_fused, k_obs with a single tile buffer
    beside k_gram_wide and beside k_gram_big, Q = 1 and Q = kMaxQ on each observation kernel, and a Q that
    runs all three node loops (U at a time, 2, 1) of both fused kernels.  What each K runs comes from
    tools/dispatch_table.cu, which calls the planner's own functions; host-only, it launches nothing."""
    import shutil
    import subprocess
    from test_gpu_glmm_parity import CASES
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "dispatch")
    subprocess.run([nvcc, "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe,
                    os.path.join(root, "tools", "dispatch_table.cu")], check=True, capture_output=True)
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout[-2000:]
    lines = out.stdout.splitlines()
    consts = {k: int(v) for k, v in (t.split("=") for t in lines[-1].split())}
    table = {}
    for line in lines[:-1]:
        row = dict(t.split("=") for t in line.split())
        table[int(row.pop("K"))] = row
    max_k, max_q = consts["kMaxK"], consts["kMaxQ"]
    assert sorted(table) == list(range(1, max_k + 1))
    assert len({r["id"] for r in table.values() if r["gram"] == "fused"}) == consts["fused_ids"] > 0
    assert len({r["id"] for r in table.values() if r["gram"] == "mid"}) == consts["mid_ids"] > 0

    def nbuf(row, Q):
        """k_obs tile buffers at Q; the rule only drops to one buffer as Q grows, so it is known wherever the
        buffer counts at Q = 1 and Q = kMaxQ agree"""
        at = dict(zip((1, 8, max_q), (int(b) for b in row["nbuf"].split(","))))
        return at.get(Q, at[1] if at[1] == at[max_q] else None)

    def all_loops(Q, U):
        return Q >= U and Q % U >= 2 and Q % U % 2 == 1

    def classes(K, Q):
        """the classes a case with K columns and Q nodes reaches (Q = None: the structural ones alone)"""
        row, c = table[K], set()
        obs = []
        if row["gram"] == "fused":
            c.add("k_fused_eval id %s" % row["id"])
            obs.append(("k_fused_eval", consts["kFuUnroll"]))
        elif row["gram"] == "mid":
            c.add("k_gram_mid id %s" % row["id"])
        elif row["gram"] == "big":
            c.add("k_gram_big plan %s (n_groups/TN/straddle)" % row["plan"])
        if K == max_k:
            c.add("K = kMaxK")
        if row["chunks"] != "-":
            c.add("k_obs_fused with %s column chunk(s)" % row["chunks"])
            obs.append(("k_obs_fused", consts["kOfUnroll"]))
        else:
            obs.append(("k_obs", None))
            if row["gram"] in ("wide", "big") and nbuf(row, max_q if Q is None else Q) == 1:
                c.add("k_obs with one tile buffer beside k_gram_%s" % row["gram"])
        for name, U in obs:
            for q in (1, max_q):
                if Q is None or Q == q:
                    c.add("Q = %d on %s" % (q, name))
            if U is not None and (Q is None or all_loops(Q, U)):
                c.add("Q running all node loops of %s, e.g. Q = %d" % (name, U + 3))
        return c

    where = {}
    for K in table:
        for cls in classes(K, None):
            where.setdefault(cls, []).append(K)
    reached = set()
    for case in CASES.values():
        reached |= classes(case["K"], case["Q"])
    assert reached <= set(where)
    missing = sorted(set(where) - reached)
    assert not missing, "no parity case reaches: " + "; ".join(
        "%s (K = %s)" % (cls, _k_ranges(where[cls])) for cls in missing)
