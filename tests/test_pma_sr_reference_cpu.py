"""CPU: the extended-precision reference that tests/test_pma_sr_numerics_gpu.py holds PMA's update_sr kernels to
(helpers.ref_inverse / ref_stationary), checked against mpmath at 40 significant digits, and its matrix generators.

The reference has to be far more accurate than the gates it supports: its error may be at most 1/1000 of the
kernel gates (16 eps kappa max|R| for SR, 8 S eps for the stationary vector, eps = fp64's)."""
import mpmath
import numpy as np
import pytest

from helpers import (EPS64, LD, band_T, decoupled_T, dense_T, kappa_inf, reducible_T, ref_inverse,
                     ref_stationary)

DPS = 40


def mp_inverse(M):
    with mpmath.workdps(DPS):
        R = mpmath.matrix([[mpmath.mpf(float(v)) for v in row] for row in M]) ** -1
        return np.array([[LD(mpmath.nstr(R[i, j], 30)) for j in range(R.cols)] for i in range(R.rows)])


def mp_stationary(T):
    """x^T Q = 0, sum x = 1, by an mpmath LU solve (the last equation replaced by the normalisation), then
    |x| / ||x||_2.  Q is the generator of the chain's off-diagonal transitions (Q[i][i] = -sum_{j != i} T[i][j],
    summed exactly): GTH never reads the diagonal of T, and the fp64 rows of T sum to 1 only up to rounding, which a
    nearly decoupled chain would amplify by its condition number."""
    S = T.shape[0]
    with mpmath.workdps(DPS):
        A = mpmath.matrix(S, S)
        for i in range(S):
            for j in range(S):
                if i != j:
                    A[i, j] = -mpmath.mpf(float(T[j, i]))
        for i in range(S):
            A[i, i] = mpmath.fsum(mpmath.mpf(float(T[i, j])) for j in range(S) if j != i)
        b = mpmath.matrix(S, 1)
        for j in range(S):
            A[S - 1, j] = 1
        b[S - 1] = 1
        x = mpmath.lu_solve(A, b)
        n = mpmath.sqrt(sum(x[i] ** 2 for i in range(S)))
        return np.array([LD(mpmath.nstr(abs(x[i]) / n, 30)) for i in range(S)])


def _matrices():
    out = []
    for S in (1, 2, 5, 12):
        out.append(('dense%d' % S, dense_T(S, 100 + S)))
    out += [('band12_bw3', band_T(12, 3, 7)), ('band9_bw1', band_T(9, 1, 8)), ('decoupled12', decoupled_T(12, 9)),
            ('decoupled2', decoupled_T(2, 10))]
    return out


MATS = _matrices()


def test_longdouble_is_extended():
    assert np.finfo(LD).eps <= 1.1e-19


@pytest.mark.parametrize('gamma', [0.0, 0.5, 0.9, 0.99, 0.999])
@pytest.mark.parametrize('name, T', MATS, ids=[m[0] for m in MATS])
def test_ref_inverse_matches_mpmath(name, T, gamma):
    S = T.shape[0]
    M = np.eye(S) - gamma * T
    X = ref_inverse(M)
    R = mp_inverse(M)
    kappa = kappa_inf(M, R)
    err = float(np.abs(X - R).max())
    gate = 1e-3 * 16 * EPS64 * kappa * float(np.abs(R).max())
    assert err <= gate, '%s gamma=%g: |ref - mpmath| = %.3g, 1/1000 of the kernel gate = %.3g' % (name, gamma, err, gate)
    # M X = I to 1e-17, relative to the size of the products that form it (at gamma = 0.999 the entries of X reach
    # hundreds, and forming M X in longdouble alone rounds at 1e-19 of that)
    Ml = np.asarray(M, dtype=LD)
    res = float(np.abs(np.eye(S, dtype=LD) - Ml @ X).max() / (np.abs(Ml) @ np.abs(X)).max())
    assert res <= 1e-17, '%s gamma=%g: max|I - M X| / max(|M| |X|) = %.3g' % (name, gamma, res)


@pytest.mark.parametrize('name, T', MATS, ids=[m[0] for m in MATS])
def test_ref_stationary_matches_mpmath(name, T):
    S = T.shape[0]
    x = ref_stationary(T)
    r = mp_stationary(T)
    assert np.all(r > 0)
    rel = float((np.abs(x - r) / r).max())
    assert rel <= 1e-3 * 8 * S * EPS64, '%s: max relative error %.3g' % (name, rel)


def test_generators():
    for S, bw in ((12, 3), (40, 7), (93, 31), (5, 1)):
        T = band_T(S, bw, 1)
        i, j = np.indices(T.shape)
        inside = np.abs(i - j) <= bw
        assert np.all(T[inside] > 0) and np.all(T[~inside] == 0), 'every offset in [-bw, bw] is non-zero'
        assert np.allclose(T.sum(axis=1), 1.0, rtol=0, atol=1e-15)
        if S >= 40:
            assert T[inside].min() / T[inside].max() < 1e-6, 'entries spread over many orders of magnitude'
    T = decoupled_T(12, 9)
    x = ref_stationary(T)
    assert float(x.max() / x.min()) > 1e8, 'the decoupled chain spans more than 8 orders of magnitude'
    assert np.allclose(T.sum(axis=1), 1.0, rtol=0, atol=1e-15)
    for T in (reducible_T(12, 3), reducible_T(30, 3, bw=4)):
        m = T.shape[0] // 2
        assert np.all(T[:m, m:] == 0) and np.all(T[m:, :m] == 0)
        assert np.allclose(T.sum(axis=1), 1.0, rtol=0, atol=1e-15)
