"""lrvb_spd_inverse (the role of cho_solve(cho_factor(H), .) in ModelSensitivity.py:594-602) against
numpy.linalg.inv for both kernels: register-resident (n <= 104) and blocked multi-CTA sweeps (n > 104, ragged
and full tiles up to the largest n the library accepts).  Tolerance: 1e-9 relative to the largest entry (the
covariance tolerance of the north star).  The blocked sweeps are also held to 1e-10 of a Gauss-Jordan inverse
in extended precision (np.longdouble, a 64-bit mantissa on x86-64), whose residual |R S - I| stays near 1e-17
on these matrices.  `info` = first non-positive leading minor, as a Cholesky factorisation reports it."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _inverse(S):
    import torch
    from lrvb_b200 import _native as nat
    lib = nat.load()
    Sd = torch.as_tensor(S, dtype=torch.float64, device="cuda").clone()
    info = ctypes.c_int32(-1)
    nat.check(lib.lrvb_spd_inverse(nat.ptr(Sd), S.shape[0], ctypes.byref(info), nat.stream_ptr()))
    return Sd.cpu().numpy(), info.value


def _spd(n, seed, cond=1e3):
    rng = np.random.default_rng(seed)
    Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    ev = np.exp(rng.uniform(0.0, np.log(cond), n))
    return (Q * ev) @ Q.T


@pytest.mark.parametrize("n", [1, 7, 44, 64, 65, 96, 97, 104, 128, 129, 160, 204, 234, 235, 300, 404, 516])
def test_inverse_matches_numpy(n):
    S = _spd(n, n)
    S = 0.5 * (S + S.T)
    got, info = _inverse(S)
    assert info == 0
    want = np.linalg.inv(S)
    assert np.abs(got - want).max() <= 1e-9 * np.abs(want).max()
    if n > 104:
        assert np.array_equal(got, got.T)       # the blocked path symmetrises exactly
    else:
        assert np.abs(got - got.T).max() <= 1e-13 * np.abs(want).max()


def _inverse_longdouble(S):
    """In-place Gauss-Jordan sweeps without pivoting (S is SPD) in np.longdouble."""
    M = S.astype(np.longdouble)
    for k in range(M.shape[0]):
        p = 1 / M[k, k]
        r = M[k] * p
        c = M[:, k].copy()
        M -= np.outer(c, r)
        M[k] = r
        M[:, k] = -c * p
        M[k, k] = p
    return M


@pytest.mark.parametrize("n", [128, 204, 404])
def test_blocked_matches_longdouble_reference(n):
    S = _spd(n, 3 * n)
    S = 0.5 * (S + S.T)
    got, info = _inverse(S)
    assert info == 0
    ref = _inverse_longdouble(S)
    assert np.abs(got - ref).max() <= 1e-10 * np.abs(ref).max()


@pytest.mark.parametrize("n,k", [(40, 17), (100, 1), (130, 33), (130, 70), (300, 290), (404, 129)])
def test_info_is_first_nonpositive_leading_minor(n, k):
    S = _spd(n, 7 * n + k)
    S = 0.5 * (S + S.T)
    # make the leading minor of order k the first one that is not positive: push the Schur complement of the
    # (k-1) x (k-1) corner in S[k-1, k-1] below zero
    kk = k - 1
    if kk > 0:
        s = S[kk, kk] - S[kk, :kk] @ np.linalg.solve(S[:kk, :kk], S[:kk, kk])
    else:
        s = S[0, 0]
    S[kk, kk] -= 2.0 * s
    _, info = _inverse(S)
    assert info == k
