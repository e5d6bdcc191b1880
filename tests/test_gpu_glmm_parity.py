"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle on identical seeded
inputs.  Tolerance 1e-9 relative / 1e-12 absolute (BASELINE.json north_star); sparsity pattern
(indptr / indices) bit-exact."""
import numpy as np
import pytest

from helpers import assert_close, make_case, make_model, make_oracle

pytestmark = pytest.mark.gpu

CASES = {
    # C1 of BASELINE.json: N=5000, K=5, G=100, Q=4
    "c1": dict(N=5000, K=5, G=100, Q=4, seed=1001),
    "c1_weights_bounds": dict(N=5000, K=5, G=100, Q=4, seed=1002, weights=True, bounds=0.05),
    "ragged_shuffled": dict(N=3001, K=7, G=64, Q=8, seed=7, ragged=True, shuffle=True),
    "empty_groups": dict(N=1203, K=3, G=50, Q=5, seed=8, ragged=True, empty_groups=9),
    "k1": dict(N=777, K=1, G=10, Q=6, seed=9),
    "k8_intercept": dict(N=2048, K=8, G=32, Q=8, seed=10, intercept=True),
    "k20": dict(N=20000, K=20, G=200, Q=8, seed=2001),
    "k33_multi_rect": dict(N=4100, K=33, G=41, Q=8, seed=11, weights=True),
    "k50": dict(N=6000, K=50, G=60, Q=8, seed=3001),
    "k70_job_groups": dict(N=1500, K=70, G=15, Q=8, seed=12),
    "one_group": dict(N=900, K=4, G=1, Q=8, seed=13),
    "tiny": dict(N=3, K=2, G=2, Q=3, seed=14),
    # fused observation+group kernel: groups that straddle many warps' row ranges, several
    # stages per warp, ragged last stage, weights
    "big_groups_multistage": dict(N=200003, K=12, G=37, Q=6, seed=15, ragged=True, weights=True),
    # (almost) one observation per group, many empty groups: a flush per row
    "many_tiny_groups": dict(N=40000, K=6, G=30000, Q=4, seed=16, ragged=True),
    # column-chunk boundaries of the fused kernel (K + 1 columns in 32-lane chunks) and the
    # hand-over to the separate observation / group kernels above K = 62
    "k31": dict(N=2500, K=31, G=25, Q=8, seed=17),
    "k32": dict(N=2500, K=32, G=25, Q=8, seed=18, weights=True),
    "k62": dict(N=2500, K=62, G=25, Q=8, seed=19),
    "k63": dict(N=2500, K=63, G=25, Q=8, seed=20),
    # packed-Gram tile shapes: no straddle tile (K = 16), straddle in tile 0 (K = 3)
    "k16": dict(N=3000, K=16, G=30, Q=8, seed=21),
    "k3": dict(N=3000, K=3, G=30, Q=8, seed=22, intercept=True),
    # several job groups of the rectangle Gram kernel, 16-row stages; zero weights among the rest
    "k130_job_groups": dict(N=1100, K=130, G=11, Q=4, seed=23),
    "k21_odd_rows_not_tma": dict(N=2100, K=21, G=20, Q=8, seed=24, weights=True),
    # k_gram_mid: every tile-grid size of the two-warp teams (T2 = 9 .. 13, with and without a straddle
    # tile), ragged last stage (N not a multiple of the 32-row stage), and enough rows that a team's 3-slot ring wraps
    # (148 SMs x 4 teams x 32 rows x 3 slots = 57k rows) with the producer one stage ahead of its partner
    "k36_team": dict(N=2501, K=36, G=25, Q=8, seed=25),
    "k37_team": dict(N=2500, K=37, G=25, Q=6, seed=26, weights=True),
    "k40_team": dict(N=2503, K=40, G=20, Q=8, seed=27),
    "k44_team_ragged": dict(N=3011, K=44, G=30, Q=8, seed=28, ragged=True),
    "k47_team": dict(N=2005, K=47, G=20, Q=4, seed=29),
    "k48_team": dict(N=2000, K=48, G=20, Q=4, seed=30, weights=True),
    "k52_team": dict(N=1999, K=52, G=20, Q=4, seed=31),
    "k50_team_ring_wrap": dict(N=70003, K=50, G=70, Q=4, seed=32, weights=True),
    "k28_ring_wrap": dict(N=120011, K=28, G=120, Q=4, seed=33),
    # teams of four (T2 14..18) and eight (T2 19..26) warps with tile-range roles
    "k56_team4": dict(N=1503, K=56, G=15, Q=4, seed=34),
    "k72_team4": dict(N=1200, K=72, G=12, Q=4, seed=35, weights=True),
    "k77_team8": dict(N=1101, K=77, G=11, Q=4, seed=36),
    "k104_team8_ring_wrap": dict(N=30011, K=104, G=30, Q=4, seed=37),
    "k72_team4_ring_wrap": dict(N=40009, K=72, G=40, Q=4, seed=46, weights=True),
    # k_gram_wide (K = 176 .. 240, K % 8 == 0): blocks of 5,5,4,4,4 tiles (K = 176: mixed 5x4 / 4x5 / 4x4 jobs),
    # of 5 only (K = 200, 240); ragged last stage; enough rows that every CTA's 3-slot ring wraps:
    # gram_wide_plan(192) deals 7 job groups of 28 - 60-row stages to 19 - 24 CTAs each, at most 19 CTAs x 60
    # rows = 1140 rows per round of stages, so N = 12007 gives every CTA >= 10 stages
    "k176_wide": dict(N=2503, K=176, G=20, Q=4, seed=38, weights=True),
    "k240_wide": dict(N=2003, K=240, G=20, Q=4, seed=39),
    "k192_wide_ring_wrap": dict(N=12007, K=192, G=40, Q=4, seed=40),
    "k200_wide_ragged": dict(N=3010, K=200, G=30, Q=4, seed=41, ragged=True, weights=True),
    "k184_wide_default": dict(N=2400, K=184, G=24, Q=4, seed=42),
    # wide-model observation kernel (K > 62): node slots with unequal node counts (Q = 6: 2, 2, 1, 1), an empty
    # slot (Q = 3), more than two nodes per slot (Q = 13); ragged tiles, weights
    "k80_q6": dict(N=1003, K=80, G=10, Q=6, seed=43, weights=True),
    "k65_q3": dict(N=700, K=65, G=7, Q=3, seed=44),
    "k96_q13": dict(N=1500, K=96, G=15, Q=13, seed=45, ragged=True),
}


@pytest.fixture(scope="module", params=sorted(CASES))
def setup(request, vb):
    case = make_case(**CASES[request.param])
    oracle = make_oracle(case)
    model = make_model(vb, case)
    obj = vb.Objective(model.glmm_par, model)
    return case, oracle, model, obj


def test_value_and_gradient(setup):
    case, oracle, model, obj = setup
    x = case["free"]
    kl = obj.fun_free(x)
    assert isinstance(kl, float)
    assert_close(kl, oracle.kl(x), what="KL")
    g = obj.fun_free_grad(x)
    ge = oracle.kl_grad(x)
    assert_close(g, ge, scale=np.abs(ge).max() * 1e-3, what="grad")
    # par holds plain numeric values equal to the evaluation point (SparseObjectives.py:142-150)
    assert_close(model.glmm_par.get_free(), x, what="par.get_free")


def test_hessian_csr_bit_exact_pattern_and_values(setup):
    case, oracle, model, obj = setup
    x = case["free"]
    H = obj.fun_free_hessian(x)
    He = oracle.kl_hessian_csr(x)
    assert H.shape == He.shape
    assert H.indptr.dtype == np.int32 and H.indices.dtype == np.int32
    np.testing.assert_array_equal(H.indptr, He.indptr)
    np.testing.assert_array_equal(H.indices, He.indices)
    assert_close(H.data, He.data, scale=np.abs(He.data).max() * 1e-6, what="hessian data")
    D = H.shape[0]
    if D <= 600:
        Hd = H.toarray()
        assert np.array_equal(Hd, Hd.T), "device Hessian must be exactly symmetric"


def test_structural_nnz_formula(setup):
    case, oracle, model, obj = setup
    # SURVEY A.3: nnz = 4K^2 + 14 + G(8K + 14) when every group is non-empty and no X column
    # is identically zero
    counts = np.bincount(case["g"], minlength=case["G"])
    if (counts > 0).all():
        K, G = case["K"], case["G"]
        H = obj.fun_free_hessian(case["free"])
        assert H.nnz == 4 * K * K + 14 + G * (8 * K + 14)


def test_hvp(setup):
    case, oracle, model, obj = setup
    x = case["free"]
    rng = np.random.default_rng(5)
    v = rng.standard_normal(x.size)
    hv = obj.fun_free_hvp(x, v)
    hve = oracle.kl_hvp(x, v)
    assert_close(hv, hve, scale=np.abs(hve).max() * 1e-3, what="hvp")


def test_vector_coordinates(setup):
    case, oracle, model, obj = setup
    vec = oracle.free_to_vector(case["free"])
    kl, gv, blk = oracle.vector_derivs(vec, hessian=True)
    assert_close(obj.fun_vector(vec), kl, what="KL(vector)")
    g = obj.fun_vector_grad(vec)
    assert_close(g, gv, scale=np.abs(gv).max() * 1e-3, what="grad(vector)")
    if case["free"].size <= 600:
        Hd = obj.fun_vector_hessian(vec).toarray()
        He = oracle.blocks_to_dense(oracle.lay, blk)
        assert_close(Hd, He, scale=np.abs(He).max() * 1e-6, what="hessian(vector)")
    # back to free coordinates: the cache must not leak across coordinate systems
    assert_close(obj.fun_free(case["free"]), oracle.kl(case["free"]), what="KL after vector")


def test_cg_and_direct_solve(setup, vb):
    case, oracle, model, obj = setup
    x = case["free"]
    D = x.size
    if D > 1200:
        pytest.skip("dense reference solve only for small D")
    Hd = oracle.kl_hessian_dense(x)
    if np.linalg.eigvalsh(Hd).min() <= 0:
        pytest.skip("Hessian not PD at this (non-optimal) point")
    rng = np.random.default_rng(6)
    b = rng.standard_normal(D)
    xe = np.linalg.solve(Hd, b)
    solver = vb.ConjugateGradientSolver(obj.fun_free_hvp, x)
    solver.tol = 1e-10
    for pre in (None, "block_jacobi"):
        solver.preconditioner = pre
        xs, info = solver.get_hinv_vec(b)
        assert info == 0
        # contract of test_objectives.py:552-554: agreement with the direct solve to 1e-8
        assert np.max(np.abs(xs - xe)) < 1e-8 * max(1.0, np.abs(xe).max())
    lr = vb.LinearResponseCovariances(obj, x)
    Hinv = np.linalg.inv(Hd)
    Dg = model.Dg
    cov_g = lr.get_global_covariance()
    assert_close(cov_g, Hinv[:Dg, :Dg], rtol=1e-8, scale=np.abs(Hinv[:Dg, :Dg]).max() * 1e-3,
                 what="global covariance")
    xd = lr.hinv(b).cpu().numpy()
    assert_close(xd, xe, rtol=1e-8, scale=np.abs(xe).max() * 1e-3, what="direct solve")
    G = model.G
    if G > 0:
        um, ui = np.arange(Dg, Dg + G), np.arange(Dg + G, Dg + 2 * G)
        loc = lr.get_local_covariances()
        ref = np.stack([Hinv[um, um], Hinv[um, ui], Hinv[ui, ui]], axis=1)
        assert_close(loc, ref, rtol=1e-8, scale=np.abs(ref).max() * 1e-3, what="local covariances")
    J = model.moment_jacobian(x)
    cov_m = lr.get_lr_covariance()
    ref = J @ Hinv @ J.T
    assert_close(cov_m, ref, rtol=1e-8, scale=np.abs(ref).max() * 1e-3, what="moment covariance")


def test_cg_general_preconditioner(vb):
    """scipy's M= (ConjugateGradient.py:84) on the device path: a sparse matrix, a dense array, the
    block-Jacobi and Schur strings must all reach the dense solution; the exact inverse converges at once."""
    import scipy.sparse
    case = make_case(N=3000, K=4, G=25, Q=8, seed=77, bounds=0.05)
    oracle, model = make_oracle(case), make_model(vb, case)
    obj = vb.Objective(model.glmm_par, model)
    xo, res = vb.OptimizationUtils.minimize_objective_newton(obj, case["free"], maxiter=50, gtol=1e-8)
    assert res.success
    Hd = oracle.kl_hessian_dense(xo)
    b = np.random.default_rng(3).standard_normal(model.D)
    xe = np.linalg.solve(Hd, b)
    solver = vb.ConjugateGradientSolver(obj.fun_free_hvp, xo)
    solver.tol = 1e-11
    iters = {}
    diag = scipy.sparse.diags(1.0 / np.diag(Hd)).tocsr()
    for name, M in (("none", None), ("diag_csr", diag), ("dense_inv", np.linalg.inv(Hd)),
                    ("block_jacobi", "block_jacobi"), ("schur", "schur")):
        solver.preconditioner = M
        xs, info = solver.get_hinv_vec(b)
        assert info == 0, name
        assert np.max(np.abs(xs - xe)) < 1e-8 * max(1.0, np.abs(xe).max()), name
        iters[name] = solver.last_iterations
    assert iters["schur"] <= 3 and iters["dense_inv"] <= 3, iters
    assert iters["diag_csr"] < iters["none"], iters
    solver.preconditioner = lambda v: v
    with pytest.raises(ValueError):
        solver.get_hinv_vec(b)


@pytest.mark.parametrize("N,G", [(4000, 40), (30000, 3000)])    # the second: the conditional export walks its roles with a grid stride
def test_csr_refill_follows_pattern_changes(vb, N, G):
    """The CSR export after the first one rewrites the values for the cached pattern and checks the zero
    mask on the device; when an entry becomes exactly zero (or stops being zero) the conditional full
    export must take over -- without any help from the host -- and later refills use the new pattern."""
    import scipy.sparse
    case = make_case(N=N, K=6, G=G, Q=8, seed=91, ragged=True, empty_groups=3)
    oracle, model = make_oracle(case), make_model(vb, case)
    model._csr_refill_min = 0                # the refill path whatever the size
    x = case["free"]

    def dense_from_blocks():
        A, B, L = [t.cpu().numpy() for t in model.blocks()]
        return oracle.blocks_to_dense(oracle.lay, dict(A=A, B=B, L=L))

    def check(H):
        ref = scipy.sparse.csr_matrix(dense_from_blocks())
        ref.sort_indices()
        Hs = H.to_scipy()
        np.testing.assert_array_equal(Hs.indptr, ref.indptr)
        np.testing.assert_array_equal(Hs.indices, ref.indices)
        np.testing.assert_array_equal(Hs.data, ref.data)

    model.evaluate(x, 2)
    H1 = model.hessian_csr()                 # full export
    check(H1)
    H2 = model.hessian_csr()                 # refill, same pattern
    assert H2._pending is not None
    check(H2)
    assert H2._pattern is H1._pattern        # shared index arrays
    A = model.blocks()[0].clone()
    A2 = A.clone()
    A2[5, 7] = A2[7, 5] = 0.0
    A2[0, 0] = 0.0
    model.set_global_block(A2)
    H3 = model.hessian_csr()                 # refill sees a different zero mask -> conditional export ran
    check(H3)
    assert H3.nnz == H1.nnz - 3
    H4 = model.hessian_csr()                 # refill against the NEW pattern
    check(H4)
    assert H4._pattern is H3._pattern and H4._pattern is not H1._pattern
    model.set_global_block(A)
    H5 = model.hessian_csr()                 # and back
    check(H5)
    assert H5.nnz == H1.nnz
    # a new evaluation point through the objective (host matrices share the pattern's index arrays)
    obj = vb.Objective(model.glmm_par, model)
    x2 = x + 0.05 * np.random.default_rng(2).standard_normal(x.size)
    Ha, Hb = obj.fun_free_hessian(x), obj.fun_free_hessian(x2)
    He = oracle.kl_hessian_csr(x2)
    np.testing.assert_array_equal(Hb.indices, He.indices)
    assert_close(Hb.data, He.data, scale=np.abs(He.data).max() * 1e-6, what="hessian data after refill")
    assert Ha.indices is Hb.indices or np.shares_memory(Ha.indices, Hb.indices)
    with pytest.raises(ValueError):
        Hb.indices[0] = 3                    # shared index arrays are read-only


def test_no_observations(vb):
    """N = 0 (a rank that owns no group in a sharded job, or priors only): the data kernels are
    skipped, the non-data terms and the Hessian pattern must still match the oracle."""
    from oracle import glmm_oracle as go
    K, G, Q = 3, 4, 5
    gh_x, gh_w = np.polynomial.hermite.hermgauss(Q)
    X, y, g = np.zeros((0, K)), np.zeros(0), np.zeros(0, np.int64)
    oracle = go.GLMMOracle(X, y, g, gh_x, gh_w, G=G)
    model = vb.LogisticGLMM(X, y, g, gh_x=gh_x, gh_w=gh_w, num_groups=G)
    obj = vb.Objective(model.glmm_par, model)
    x = go.make_free(model.D, 41)
    assert_close(obj.fun_free(x), oracle.kl(x), what="KL")
    ge = oracle.kl_grad(x)
    assert_close(obj.fun_free_grad(x), ge, scale=np.abs(ge).max() * 1e-3, what="grad")
    H, He = obj.fun_free_hessian(x), oracle.kl_hessian_csr(x)
    np.testing.assert_array_equal(H.indptr, He.indptr)
    np.testing.assert_array_equal(H.indices, He.indices)
    assert_close(H.data, He.data, scale=np.abs(He.data).max() * 1e-6, what="hessian data")
    assert np.all(model.weight_cross_matvec(np.zeros(0)).cpu().numpy() == 0.0)


def test_par_follows_a_device_point_lazily(vb):
    """For CUDA-tensor input the evaluation point stays on the device; ``objective.par`` is filled in when
    it is read (the reference contract -- par equals the last evaluation point, SparseObjectives.py:142-150
    -- holds at every read)."""
    import torch
    case = make_case(**CASES["c1"])
    model = make_model(vb, case)
    obj = vb.Objective(model.glmm_par, model)
    x = case["free"]
    xt = torch.from_numpy(x).cuda()
    obj.fun_free_grad(xt)
    assert obj._pending is not None                      # nothing was copied to the host yet
    assert_close(obj.par.get_free(), x, what="par.get_free after a device evaluation")
    assert obj._pending is None
    x2 = x + 0.01
    obj.fun_free(x2)                                     # host input: par is set immediately
    assert_close(model.glmm_par.get_free(), x2, what="par.get_free after a host evaluation")
