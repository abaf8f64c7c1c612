"""Bures-Wasserstein / Gaussian 2-Wasserstein distances without a GPU: the C ABI codes against the
Python constants, the public names, the float64 reference, and a numpy model of the kernel's
formulation (Cholesky factors, A = L_i^T L_j, its singular vectors Y and Z, the sigma coefficients)
against central differences."""

import os
import re

import numpy as np
import pytest
import scipy.linalg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_macros():
    text = open(os.path.join(ROOT, "include", "sqfa_b200.h")).read()
    return {m.group(1): int(m.group(2)) for m in re.finditer(r"#define (SQFA_DIST_\w+) (\d+)", text)}


def test_header_codes_match_ops_and_public_names():
    from sqfa_b200 import _ops, distances, model

    macros = _header_macros()
    assert macros["SQFA_DIST_BURES_WASSERSTEIN"] == _ops.DIST_BW == 3
    assert macros["SQFA_DIST_WASSERSTEIN_GAUSSIAN"] == _ops.DIST_W2 == 4
    for name in ("bures_wasserstein_sq", "bures_wasserstein", "wasserstein_sq", "wasserstein"):
        assert name in distances.__all__
        assert "not reference API" in " ".join(getattr(distances, name).__doc__.split())
    assert model._TENSOR_DISTANCES[distances.bures_wasserstein] == _ops.DIST_BW
    assert model._TENSOR_DISTANCES[distances.bures_wasserstein_sq] == _ops.DIST_BW | _ops.SQUARED
    assert model._DICT_DISTANCES[distances.wasserstein] == _ops.DIST_W2
    assert model._DICT_DISTANCES[distances.wasserstein_sq] == _ops.DIST_W2 | _ops.SQUARED


def spd(rng, m, shift=0.3):
    X = rng.standard_normal((m, m))
    return X @ X.T / m + shift * np.eye(m)


def bw_sq_reference(A, B):
    """float64 reference: tr A + tr B - 2 tr((B^1/2 A B^1/2)^1/2), eigendecompositions only."""
    lam, V = np.linalg.eigh(B)
    R = (V * np.sqrt(lam)) @ V.T
    inner = np.clip(np.linalg.eigvalsh(R @ A @ R), 0, None)
    return max(np.trace(A) + np.trace(B) - 2 * np.sqrt(inner).sum(), 0.0)


@pytest.mark.parametrize("m", [1, 2, 5, 9, 17])
def test_reference_matches_scipy_sqrtm(m):
    rng = np.random.default_rng(m)
    for _ in range(3):
        A, B = spd(rng, m), spd(rng, m)
        R = np.real(scipy.linalg.sqrtm(B))
        fid = np.trace(np.real(scipy.linalg.sqrtm(R @ A @ R)))
        want = np.trace(A) + np.trace(B) - 2 * fid
        assert abs(bw_sq_reference(A, B) - want) <= 1e-10 * (np.trace(A) + np.trace(B))
    assert bw_sq_reference(A, A) <= 1e-12 * np.trace(A)


def kernel_model(Ei, Ej, pad):
    """What the column-pair kernel computes for one pair: A = L_i^T L_j (one zero padding column when
    `pad`, as for odd m), orthogonalised columns A_f = A U, sigma = column norms with the padding
    column masked out, d^2 from the factors' Frobenius norms, and G_i = I - sum sigma^-1 y y^T,
    G_j = I - sum sigma^-3 z z^T with Y = L_i^-T A_f and Z = L_i A_f."""
    Li, Lj = np.linalg.cholesky(Ei), np.linalg.cholesky(Ej)
    m = Ei.shape[0]
    A = Li.T @ Lj
    if pad:
        A = np.concatenate([A, np.zeros((m, 1))], axis=1)
    _, _, Vt = np.linalg.svd(A)  # right singular vectors: the rotation the Jacobi converges to
    Af = A @ Vt.T
    n2 = (Af * Af).sum(axis=0)
    real = np.ones(Af.shape[1], bool)
    if pad:
        real[np.argmin(n2)] = False  # the padding column keeps norm 0
        assert n2[~real][0] < 1e-20
    sig = np.where(real, np.sqrt(np.where(real, n2, 1.0)), 0.0)
    d2 = (Li * Li).sum() + (Lj * Lj).sum() - 2 * sig.sum()
    ci = np.where(real, -1.0 / np.where(real, sig, 1.0), 0.0)
    cj = np.where(real, -1.0 / np.where(real, sig * n2, 1.0), 0.0)
    Y = np.linalg.solve(Li.T, Af)
    Z = Li @ Af
    Gi = np.eye(m) + (Y * ci) @ Y.T
    Gj = np.eye(m) + (Z * cj) @ Z.T
    return max(d2, 0.0), Gi, Gj


def central_difference(f, E, h=1e-6):
    m = E.shape[0]
    g = np.zeros((m, m))
    for a in range(m):
        for b in range(m):
            D = np.zeros((m, m))
            D[a, b] += h / 2
            D[b, a] += h / 2
            g[a, b] = (f(E + D) - f(E - D)) / (2 * h)
    return g


@pytest.mark.parametrize("m,pad", [(2, False), (3, True), (6, False), (7, True), (9, True)])
def test_kernel_formulation_matches_central_differences(m, pad):
    rng = np.random.default_rng(100 + m)
    Ei, Ej = spd(rng, m), spd(rng, m)
    d2, Gi, Gj = kernel_model(Ei, Ej, pad)
    scale = np.trace(Ei) + np.trace(Ej)
    assert abs(d2 - bw_sq_reference(Ei, Ej)) <= 1e-12 * scale
    gi = central_difference(lambda E: bw_sq_reference(E, Ej), Ei)
    gj = central_difference(lambda E: bw_sq_reference(Ei, E), Ej)
    assert np.abs(Gi - gi).max() <= 1e-6 * np.abs(gi).max()
    assert np.abs(Gj - gj).max() <= 1e-6 * np.abs(gj).max()
    # I - G_i is the optimal-transport map T from E_i to E_j: T E_i T = E_j
    T = np.eye(m) - Gi
    assert np.abs(T @ Ei @ T - Ej).max() <= 1e-10 * np.abs(Ej).max()


def test_repeated_eigenvalues_have_finite_gradients():
    """The formulation has no 1/(sigma_a - sigma_b) terms: identical matrices, scalar multiples and the
    identity (all singular values repeated) give finite gradients, and d(E, E) has zero gradient."""
    rng = np.random.default_rng(7)
    E = spd(rng, 5)
    for Ei, Ej in ((E, 4.0 * E), (np.eye(5), 2.0 * np.eye(5)), (E, np.eye(5))):
        _, Gi, Gj = kernel_model(Ei, Ej, False)
        assert np.isfinite(Gi).all() and np.isfinite(Gj).all()
    _, Gi, Gj = kernel_model(2.0 * np.eye(5), 8.0 * np.eye(5), False)
    assert np.allclose(Gi, (1 - 2.0) * np.eye(5)) and np.allclose(Gj, (1 - 0.5) * np.eye(5))
    d2, Gi, Gj = kernel_model(E, E, False)
    assert d2 <= 1e-12 * np.trace(E)
    assert np.abs(Gi).max() <= 1e-6 and np.abs(Gj).max() <= 1e-6
