"""The fitting closure of the mean-covariance distances without a GPU: the C ABI codes against the Python
constants, the model's distance map, a float64 numpy model of the kernel formulation (one shared
Sigma-partial per pair, the +/- mean partials, the class logdet term and the map's derivative) against
central differences and the oracle's autograd gradient, the reason fisher_rao_same_cov stays unmapped,
and the closure workspace."""

import os
import re

import numpy as np
import pytest
import torch

from oracle import sqfa_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = 1e-6
NAMES = ("mahalanobis", "mahalanobis_sq", "bhattacharyya", "hellinger")


def _header_macros():
    text = open(os.path.join(ROOT, "include", "sqfa_b200.h")).read()
    return {m.group(1): int(m.group(2)) for m in re.finditer(r"#define (SQFA_DIST_\w+) (\d+)", text)}


def test_header_codes_match_ops():
    from sqfa_b200 import _ops

    macros = _header_macros()
    assert macros["SQFA_DIST_MAHALANOBIS"] == _ops.DIST_MAHA == 5
    assert macros["SQFA_DIST_BHATTACHARYYA"] == _ops.DIST_BHATT == 6
    assert macros["SQFA_DIST_HELLINGER"] == _ops.DIST_HELL == 7


def test_model_map_holds_the_four_distances():
    from sqfa_b200 import _ops, distances, model

    want = {distances.mahalanobis: _ops.DIST_MAHA, distances.mahalanobis_sq: _ops.DIST_MAHA | _ops.SQUARED,
            distances.bhattacharyya: _ops.DIST_BHATT, distances.hellinger: _ops.DIST_HELL}
    for fun, code in want.items():
        assert model._DICT_DISTANCES[fun] == code
    assert distances.fisher_rao_same_cov not in model._DICT_DISTANCES
    assert distances.fisher_rao_same_cov not in model._TENSOR_DISTANCES
    new = {f for f, c in model._DICT_DISTANCES.items() if 5 <= (c & 15) <= 7}
    assert new == set(want)


def closure_model(Psi, mu, name):
    """What the closure computes for classes (Psi_c, mu_c): loss = -mean_{i>j} d_ij and its gradient w.r.t.
    Psi and mu, pair by pair as the kernels do: M = (Psi_i + Psi_j) / 2, u = M^-1 d, x = d^T u; one Sigma-partial
    g (-c_m / 2 u u^T + c_l / 2 M^-1) shared by i and j, mean partials +-2 c_m g u, and per class the logdet
    term -1/4 Psi_c^-1 sum_o g."""
    C, k = mu.shape
    P = C * (C - 1) // 2
    weight = -1.0 / P
    bhat = name in ("bhattacharyya", "hellinger")
    cm, cl = (0.125, 0.5) if bhat else (1.0, 0.0)
    logdet = np.array([np.linalg.slogdet(p)[1] for p in Psi])
    gPsi, gmu, gsum = np.zeros_like(Psi), np.zeros_like(mu), np.zeros(C)
    loss = 0.0
    for i in range(C):
        for j in range(i):
            M = 0.5 * (Psi[i] + Psi[j])
            Minv = np.linalg.inv(M)
            d = mu[i] - mu[j]
            u = Minv @ d
            x = d @ u
            pre = 0.125 * x + 0.5 * (np.linalg.slogdet(M)[1] - 0.5 * (logdet[i] + logdet[j])) if bhat else x
            if name == "mahalanobis":
                dval = np.sqrt(pre + EPS)
                dmap = 0.5 / dval
            elif name == "hellinger":
                e = np.exp(-pre)
                dval = np.sqrt(1 - e + EPS)
                dmap = 0.5 * e / dval
            else:
                dval, dmap = pre, 1.0
            loss += weight * dval
            g = weight * dmap
            G = g * (-0.5 * cm * np.outer(u, u) + 0.5 * cl * Minv)
            gPsi[i] += G
            gPsi[j] += G
            gmu[i] += 2 * cm * g * u
            gmu[j] -= 2 * cm * g * u
            gsum[i] += g
            gsum[j] += g
    if bhat:
        gPsi -= 0.25 * gsum[:, None, None] * np.linalg.inv(Psi)
    return loss, gPsi, gmu


def _classes(C, k, seed):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((C, k, k))
    Psi = X @ X.transpose(0, 2, 1) / k + 0.3 * np.eye(k)
    mu = rng.standard_normal((C, k))
    return Psi, mu


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("name", NAMES)
def test_kernel_formulation_matches_central_differences_and_oracle(name, k):
    C = 4
    Psi, mu = _classes(C, k, seed=10 * k + len(name))
    loss, gPsi, gmu = closure_model(Psi, mu, name)
    f = lambda P_, m_: closure_model(P_, m_, name)[0]  # noqa: E731
    h = 1e-6
    for c in range(C):
        for a in range(k):
            dm = np.zeros_like(mu)
            dm[c, a] = h
            num = (f(Psi, mu + dm) - f(Psi, mu - dm)) / (2 * h)
            assert abs(num - gmu[c, a]) <= 1e-6 * (np.abs(gmu).max() + 1e-12)
            for b in range(k):
                D = np.zeros_like(Psi)
                D[c, a, b] += h / 2
                D[c, b, a] += h / 2
                num = (f(Psi + D, mu) - f(Psi - D, mu)) / (2 * h)
                assert abs(num - gPsi[c, a, b]) <= 1e-6 * np.abs(gPsi).max()
    # the oracle: its distance function and -mean(tril), differentiated by autograd
    P_t = torch.tensor(Psi, requires_grad=True)
    m_t = torch.tensor(mu, requires_grad=True)
    stats = {"means": m_t, "covariances": P_t}
    d = getattr(O, name)(stats, stats)
    ref_loss = O.closure_loss(d)
    ref_loss.backward()
    assert abs(float(ref_loss.detach()) - loss) <= 1e-12 * max(abs(loss), 1.0)
    sym = 0.5 * (P_t.grad + P_t.grad.transpose(1, 2)).numpy()
    assert np.abs(sym - gPsi).max() <= 1e-10 * np.abs(gPsi).max()
    assert np.abs(m_t.grad.numpy() - gmu).max() <= 1e-10 * (np.abs(gmu).max() + 1e-12)


def test_fisher_rao_same_cov_closure_gradient_is_nan():
    """Why fisher_rao_same_cov has no native closure: the reference's closure evaluates all C^2 pairs, and
    acosh' at the diagonal's x = 0 is infinite, so the gradient of -mean(tril) is 0 * inf = NaN."""
    g = torch.Generator().manual_seed(0)
    C, D, k = 5, 12, 3
    A = torch.randn(C, D, D, generator=g, dtype=torch.float64)
    stats = {"means": torch.randn(C, D, generator=g, dtype=torch.float64),
             "covariances": A @ A.transpose(1, 2) / D + 0.1 * torch.eye(D, dtype=torch.float64)}
    F = torch.randn(k, D, generator=g, dtype=torch.float64)
    loss, grad, _ = O.loss_and_grad("full", stats, F, noise=0.01, distance=O.fisher_rao_same_cov)
    assert torch.isfinite(loss)
    assert torch.isnan(grad).any()


def test_workspace_at_most_affine_invariant_plus_class_terms():
    from sqfa_b200 import _lib, _ops

    lib = _lib.load()
    C, D, k = 1000, 512, 32
    P = C * (C - 1) // 2
    ai = lib.sqfa_fused_loss_workspace_bytes(C, D, k, _ops.DIST_AI, 0, P)
    for code in (_ops.DIST_MAHA, _ops.DIST_MAHA | _ops.SQUARED, _ops.DIST_BHATT, _ops.DIST_HELL):
        got = lib.sqfa_fused_loss_workspace_bytes(C, D, k, code, 0, P)
        assert 0 < got <= ai + 4 * (2 * C * k * k + 2 * C) + 4096
