"""CPU: the float64 closure's C ABI (prototypes, workspace query, argument validation before any launch) and a
float64 numpy model of its pair stage -- the one-sided Jacobi with the kernel's ordering, rotation and stopping
constants (closure64.cu), and the closed-form gradient -- against scipy and central differences."""

import ctypes
import os
import re

import numpy as np
import pytest
import scipy.linalg as sl

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# closure64.cu
J64_TOL = 1e-14
J64_LAST = 1e-8
J64_MAX_SWEEPS = 30
DIST_EPS = 1e-6
AI, FR, SQUARED = 0, 1, 16


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge

    ge.build()
    from sqfa_b200 import _lib

    return _lib.load()


def test_constants_match_the_kernel_source():
    src = open(os.path.join(ROOT, "sqfa_b200", "csrc", "closure64.cu")).read()
    assert float(re.search(r"J64_TOL = ([0-9.e-]+);", src).group(1)) == J64_TOL
    assert float(re.search(r"J64_LAST = ([0-9.e-]+);", src).group(1)) == J64_LAST
    assert int(re.search(r"J64_MAX_SWEEPS = (\d+);", src).group(1)) == J64_MAX_SWEEPS


def test_prototypes_are_bound(lib):
    from sqfa_b200 import _lib

    for name in ("sqfa_fused_loss_workspace_bytes_f64", "sqfa_closure_eval_f64"):
        assert name in _lib.SIGNATURES
        assert hasattr(lib, name)
    assert len(_lib.SIGNATURES["sqfa_closure_eval_f64"][1]) == 18
    assert "sqfa_fused_loss_workspace_bytes_f64" not in lib.sqfa_missing_symbols


def test_workspace_query(lib):
    C, D, k = 19, 104, 8
    P = C * (C - 1) // 2
    for dist in (AI, FR, AI | SQUARED, FR | SQUARED):
        assert lib.sqfa_fused_loss_workspace_bytes_f64(C, D, k, dist, 0, P) > 0
        assert lib.sqfa_fused_loss_workspace_bytes_f64(C, D, 32, dist, 0, P) > 0
        assert lib.sqfa_fused_loss_workspace_bytes_f64(C, D, 33, dist, 0, P) == 0
    for dist in (2, 3, 4, 5, 6, 7, 2 | SQUARED, 5 | SQUARED, 32, -1):
        assert lib.sqfa_fused_loss_workspace_bytes_f64(C, D, k, dist, 0, P) == 0, dist
    assert lib.sqfa_fused_loss_workspace_bytes_f64(C, D, k, FR, 0, P + 1) == 0
    assert 0 < lib.sqfa_fused_loss_workspace_bytes_f64(C, D, k, FR, 0, P // 2) <= \
        lib.sqfa_fused_loss_workspace_bytes_f64(C, D, k, FR, 0, P)


def test_c4_workspace_is_at_most_twice_float32(lib):
    C, D, k = 1000, 512, 16
    P = C * (C - 1) // 2
    w64 = lib.sqfa_fused_loss_workspace_bytes_f64(C, D, k, FR, 0, P)
    w32 = lib.sqfa_fused_loss_workspace_bytes(C, D, k, FR, 0, P)
    assert 0 < w64 <= 2 * w32, (w64, w32)


def test_argument_validation_without_a_launch(lib):
    """Every rejection happens before anything touches the device (the pointers below are not device memory)."""
    fake = ctypes.c_void_p(4096)
    C, D, k = 4, 16, 3
    P = C * (C - 1) // 2

    def call(S=fake, M=fake, W=fake, C=C, D=D, k=k, noise=fake, dist=FR, constraint=1, n_fixed=0, p0=0, p1=P,
             out=fake, grad=fake, ws=fake, ws_bytes=0):
        return lib.sqfa_closure_eval_f64(S, M, W, C, D, k, noise, dist, constraint, n_fixed, p0, p1, out, None, grad,
                                         ws, ws_bytes, None)

    assert call(dist=2) == -3 and b"SQFA_DIST_AFFINE_INVARIANT" in lib.sqfa_last_error()
    assert call(dist=3) == -3
    assert call(dist=6) == -3
    assert call(constraint=2) == -1
    assert call(k=33) == -3 and b"n_filters" in lib.sqfa_last_error()
    assert call(M=None) == -1  # Fisher-Rao needs the means
    assert call(noise=None) == -1
    assert call(S=None) == -1
    assert call(n_fixed=4) == -1
    assert call(p1=P + 1) == -1 and b"pair range" in lib.sqfa_last_error()
    assert call(ws=ctypes.c_void_p(4104)) == -1  # misaligned workspace
    assert call() == -2 and b"workspace" in lib.sqfa_last_error()
    assert call(dist=AI, M=None) == -2  # affine-invariant takes no means; stops at the workspace check


# ------------------------------------------------------------------------------------------------ numpy model
def round_robin(mp):
    """Column pairs of each round of the circle method, as the lanes of jacobi64 take them."""
    n1, rounds = mp - 1, []
    for r in range(n1):
        pairs = []
        for lane in range(mp // 2):
            p, q = (n1, r) if lane == 0 else ((r + lane) % n1, (r - lane) % n1)
            pairs.append((min(p, q), max(p, q)))
        rounds.append(np.array(pairs))
    return rounds


def jacobi64(A):
    """One-sided Jacobi of jacobi64 (closure64.cu): returns A_f = A V and the number of sweeps."""
    m = A.shape[0]
    mp = m + (m & 1)
    X = np.zeros((m, mp))
    X[:, :m] = A
    rounds = round_robin(mp)
    for sweep in range(1, J64_MAX_SWEEPS + 1):
        big = False
        for pr in rounds:
            lo, hi = pr[:, 0], pr[:, 1]
            x, y = X[:, lo], X[:, hi]
            al, be, ga = (x * x).sum(0), (y * y).sum(0), (x * y).sum(0)
            rot = (al > 0) & (be > 0) & (ga * ga > J64_TOL**2 * al * be)
            big |= bool(np.any(rot & (ga * ga > J64_LAST**2 * al * be)))
            zeta = (be - al) / (2 * np.where(rot, ga, 1.0))
            t = np.copysign(1.0 / (np.abs(zeta) + np.sqrt(zeta * zeta + 1)), zeta)
            c = np.where(rot, 1 / np.sqrt(t * t + 1), 1.0)
            s = np.where(rot, c * t, 0.0)
            X[:, lo], X[:, hi] = c * x - s * y, s * x + c * y
        if not big:
            return X[:, :m], sweep
    return X[:, :m], J64_MAX_SWEEPS + 1


def pair_model(Ei, Ej, fr=False, squared=False):
    """Distance and (dd/dE_i, dd/dE_j) as the pair stage forms them."""
    Li, Lj = np.linalg.cholesky(Ei), np.linalg.cholesky(Ej)
    A = (sl.solve_triangular(Lj, np.eye(len(Ei)), lower=True) @ Li).T
    Af, sweeps = jacobi64(A)
    lam = (Af * Af).sum(0)
    ll = np.log(lam)
    cfac = 0.5 if fr else 1.0
    d2 = (ll * ll).sum()
    if squared:
        d, dd = cfac * d2, cfac
    else:
        d = np.sqrt(cfac * d2 + DIST_EPS)
        dd = cfac / (2 * d)
    Y = sl.solve_triangular(Li.T, Af, lower=False)
    Gi = dd * (Y * (2 * ll / lam)) @ Y.T
    Gj = dd * (Y * (-2 * ll)) @ Y.T
    return d, Gi, Gj, lam, sweeps, A, Af


def spd(m, cond, rng):
    Q, _ = np.linalg.qr(rng.standard_normal((m, m)))
    return (Q * np.logspace(0, np.log10(cond), m)) @ Q.T


def pair_cases(rng):
    """(E_i, E_j) with condition numbers up to 1e8: random pairs, and pairs with repeated and clustered
    generalized eigenvalues (E_i = L_j Q diag(ev) Q^T L_j^T)."""
    for m in (1, 2, 3, 4, 9, 16, 17, 32, 33):
        for cond in (1e2, 1e5, 1e8):
            Ej = spd(m, cond, rng)
            L = np.linalg.cholesky(Ej)
            Q, _ = np.linalg.qr(rng.standard_normal((m, m)))
            rep = np.where(np.arange(m) < m // 2, 3.0, 0.5)
            clus = (1 + 1e-9 * rng.standard_normal(m)) * np.where(np.arange(m) % 3 == 0, 7.0, 1.0)
            yield m, cond, "random", spd(m, cond, rng), Ej
            for name, ev in (("repeated", rep), ("clustered", clus)):
                Ei = L @ (Q * ev) @ Q.T @ L.T
                yield m, cond, name, (Ei + Ei.T) / 2, Ej


def sv2_extended(A):
    """Squared singular values of A by a cyclic one-sided Jacobi in long double, run to convergence."""
    X = A.astype(np.longdouble)
    m = X.shape[1]
    for _ in range(60):
        off = 0.0
        for p in range(m):
            for q in range(p + 1, m):
                a, b, g = (X[:, p] ** 2).sum(), (X[:, q] ** 2).sum(), (X[:, p] * X[:, q]).sum()
                if g == 0:
                    continue
                off = max(off, abs(g) / np.sqrt(a * b))
                z = (b - a) / (2 * g)
                t = np.copysign(1 / (abs(z) + np.sqrt(1 + z * z)), z)
                c = 1 / np.sqrt(1 + t * t)
                x, y = X[:, p].copy(), X[:, q].copy()
                X[:, p], X[:, q] = c * x - c * t * y, c * t * x + c * y
        if off < 1e-18:
            break
    return np.sort((X * X).sum(0).astype(np.float64))


def test_jacobi_constants_reach_full_accuracy_within_the_sweep_cap():
    """The stopping constants leave no error of their own: the eigenvalues agree with an extended-precision SVD of
    the same A to 1e-13 relative, eigenvalue by eigenvalue, well within the sweep cap. Against
    scipy.linalg.eigh(E_i, E_j) -- the same problem through a different double-precision reduction -- they agree
    to 1e-13 of the largest eigenvalue where the matrices are well conditioned (cond <= 1e2). At condition
    numbers up to 1e8 the two reductions differ by what the conditioning of the pair allows (up to 3e-9 of the
    largest eigenvalue here; a random pair whose eigenvalues span 15 decades has its smallest one off by 1e-2
    relative between the two), not by the Jacobi."""
    rng = np.random.default_rng(0)
    max_sweeps = 0
    for m, cond, name, Ei, Ej in pair_cases(rng):
        _, _, _, lam, sweeps, A, _ = pair_model(Ei, Ej)
        max_sweeps = max(max_sweeps, sweeps)
        assert sweeps <= J64_MAX_SWEEPS, (m, cond, name)
        lam = np.sort(lam)
        ref = sv2_extended(A)
        err = np.max(np.abs(lam - ref) / ref)
        assert err <= 1e-13, (m, cond, name, err)
        ref_gen = np.sort(sl.eigh(Ei, Ej, eigvals_only=True))
        assert np.max(np.abs(lam - ref_gen)) <= 1e-13 * max(1.0, cond / 1e2) * ref_gen[-1], (m, cond, name)
    assert max_sweeps <= J64_MAX_SWEEPS // 2  # the cap is twice what these cases need


@pytest.mark.parametrize("fr,squared", [(False, False), (False, True), (True, False), (True, True)])
@pytest.mark.parametrize("m", [1, 4, 7])
def test_closed_form_gradient_matches_central_differences(m, fr, squared):
    rng = np.random.default_rng(m + 10 * fr + 20 * squared)
    Ei, Ej = spd(m, 30.0, rng), spd(m, 50.0, rng)
    if m >= 4:  # a repeated generalized eigenvalue: the closed form has no 1 / (lambda_a - lambda_b) term
        L = np.linalg.cholesky(Ej)
        Q, _ = np.linalg.qr(rng.standard_normal((m, m)))
        ev = np.array([2.0, 2.0] + list(np.linspace(0.3, 5.0, m - 2)))
        Ei = L @ (Q * ev) @ Q.T @ L.T
        Ei = (Ei + Ei.T) / 2
    d, Gi, Gj, _, _, _, _ = pair_model(Ei, Ej, fr, squared)
    h = 1e-6
    for E, G, which in ((Ei, Gi, 0), (Ej, Gj, 1)):
        num = np.zeros((m, m))
        for r in range(m):
            for s in range(r, m):
                P = np.zeros((m, m))
                P[r, s] = P[s, r] = h
                args_p = (E + P, Ej) if which == 0 else (Ei, E + P)
                args_m = (E - P, Ej) if which == 0 else (Ei, E - P)
                num[r, s] = num[s, r] = (pair_model(*args_p, fr, squared)[0] - pair_model(*args_m, fr, squared)[0]) / (2 * h)
        ana = G + G.T - np.diag(np.diag(G))  # a symmetric perturbation of (r, s) moves both entries
        assert np.allclose(ana, num, rtol=1e-6, atol=1e-8 * max(1.0, abs(d))), (which, np.abs(ana - num).max())
