"""CPU: the float64 closure of the mean-covariance distances (Mahalanobis, Bhattacharyya, Hellinger) -- its C ABI
(prototypes, workspace query, argument validation before any launch) and a numpy model of the pair stage's
Gauss-Jordan schedule, identity padding included, in float64 against the same schedule in extended precision."""

import ctypes

import numpy as np
import pytest

MAHA, BHATT, HELL, SQUARED = 5, 6, 7, 16
AI, FR = 0, 1


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge

    ge.build()
    from sqfa_b200 import _lib

    return _lib.load()


def test_prototypes_are_bound(lib):
    from sqfa_b200 import _lib
    from test_abi import header_prototypes

    for name in ("sqfa_gauss_closure_workspace_bytes_f64", "sqfa_gauss_closure_eval_f64"):
        assert name in _lib.SIGNATURES
        assert hasattr(lib, name)
        assert name not in lib.sqfa_missing_symbols
    assert len(_lib.SIGNATURES["sqfa_gauss_closure_eval_f64"][1]) == 18
    assert len(header_prototypes()["sqfa_gauss_closure_eval_f64"][1]) == 18


def test_workspace_query(lib):
    C, D = 19, 104
    P = C * (C - 1) // 2
    query = lib.sqfa_gauss_closure_workspace_bytes_f64
    for dist in (MAHA, MAHA | SQUARED, BHATT, HELL):
        for k in (1, 8, 32):
            assert query(C, D, k, dist, 0, P) > 0, (dist, k)
        assert query(C, D, 33, dist, 0, P) == 0
        assert query(C, D, 8, dist, 0, P + 1) == 0
        assert 0 < query(C, D, 8, dist, 0, P // 2) <= query(C, D, 8, dist, 0, P)
    for dist in (0, 1, 2, 3, 4, BHATT | SQUARED, HELL | SQUARED, 32, -1):
        assert query(C, D, 8, dist, 0, P) == 0, dist


def test_workspace_against_float32(lib):
    """At c4 the float64 workspace is at most twice the float32 closure's, as for the affine-invariant /
    Fisher-Rao float64 closure. At the c5 shape the float64 projection splits its rows differently, so the ratio
    is only reported."""
    for name, (C, D, k) in (("c4", (1000, 512, 16)), ("c5", (100, 1024, 32))):
        P = C * (C - 1) // 2
        for dist in (MAHA, BHATT, HELL):
            w64 = lib.sqfa_gauss_closure_workspace_bytes_f64(C, D, k, dist, 0, P)
            w32 = lib.sqfa_fused_loss_workspace_bytes(C, D, k, dist, 0, P)
            print(f"{name} dist {dist}: float64 / float32 workspace = {w64 / w32:.2f}")
            if name == "c4":
                assert 0 < w64 <= 2 * w32, (w64, w32)


def test_argument_validation_without_a_launch(lib):
    """Every rejection happens before anything touches the device (the pointers below are not device memory)."""
    fake = ctypes.c_void_p(4096)
    C, D, k = 4, 16, 3
    P = C * (C - 1) // 2

    def call(S=fake, M=fake, W=fake, C=C, D=D, k=k, noise=fake, dist=HELL, constraint=1, n_fixed=0, p0=0, p1=P,
             out=fake, grad=fake, ws=fake, ws_bytes=0):
        return lib.sqfa_gauss_closure_eval_f64(S, M, W, C, D, k, noise, dist, constraint, n_fixed, p0, p1, out, None,
                                               grad, ws, ws_bytes, None)

    assert call(M=None) == -1
    assert call(noise=None) == -1
    assert call(S=None) == -1
    assert call(constraint=2) == -1
    assert call(n_fixed=4) == -1
    assert call(p1=P + 1) == -1 and b"pair range" in lib.sqfa_last_error()
    assert call(dist=AI) == -3 and b"take sqfa_closure_eval_f64" in lib.sqfa_last_error()
    assert call(dist=FR) == -3 and b"take sqfa_closure_eval_f64" in lib.sqfa_last_error()
    for dist in (2, BHATT | SQUARED):
        assert call(dist=dist) == -3
        msg = lib.sqfa_last_error()
        assert msg.startswith(b"sqfa_gauss_closure_eval_f64:") and b"SQFA_DIST_MAHALANOBIS" in msg, msg
    assert call(k=33) == -3 and b"n_filters" in lib.sqfa_last_error()
    for dist in (MAHA, MAHA | SQUARED, BHATT, HELL):
        assert call(dist=dist) == -2 and b"workspace" in lib.sqfa_last_error()
    # the affine-invariant / Fisher-Rao entry keeps rejecting these codes, and points to the new one
    assert lib.sqfa_closure_eval_f64(fake, fake, fake, C, D, k, fake, HELL, 1, 0, 0, P, fake, None, fake, fake, 0,
                                     None) == -3
    msg = lib.sqfa_last_error()
    assert b"SQFA_DIST_AFFINE_INVARIANT" in msg and b"sqfa_gauss_closure_eval_f64" in msg


# ------------------------------------------------------------------------------------------------ numpy model
def group_width(k):
    G = 2
    while G < k:
        G *= 2
    return G


def gauss_jordan(M, d, dtype):
    """The pair stage's schedule (gauss.cu, gauss_closure_pair_kernel) on M padded with the identity to G x G:
    an in-place Gauss-Jordan sweep without pivoting whose pivot row is broadcast, then u = M^-1 d accumulated in
    column order, x = d^T u and logdet M = sum log(pivots). Returns (x, logdet, u)."""
    k = M.shape[0]
    G = group_width(k)
    A = np.eye(G, dtype=dtype)
    A[:k, :k] = M.astype(dtype)
    dv = np.zeros(G, dtype=dtype)
    dv[:k] = d.astype(dtype)
    piv = np.ones(G, dtype=dtype)
    for p in range(G):
        pv = A[p, p]
        pinv = dtype(1) / pv
        f = A[:, p].copy()
        prow = A[p, :] * pinv
        A = A - f[:, None] * prow[None, :]
        A[:, p] = -f * pinv
        A[p, :] = prow
        A[p, p] = pinv
        piv[p] = pv
    u = np.zeros(G, dtype=dtype)
    for l in range(G):
        u = u + A[:, l] * dv[l]
    x = np.sum(dv * u)
    return x, np.sum(np.log(piv)), u[:k]


def spd(k, cond, rng):
    Q, _ = np.linalg.qr(rng.standard_normal((k, k)))
    ev = np.logspace(0, -np.log10(cond), k) if k > 1 else np.ones(1)
    rng.shuffle(ev)
    return (Q * ev) @ Q.T


@pytest.mark.parametrize("k", [1, 2, 3, 5, 8, 16, 17, 32])
def test_gauss_jordan_schedule_in_float64(k):
    """float64 against the same schedule in extended precision, on SPD matrices with condition numbers up to
    1e8: x = d^T M^-1 d to 1e-13 max(1, kappa / 100) relative, logdet M to 1e-14 kappa absolute, u to 1e-14 kappa
    relative. (Against a different algorithm, such as LU with pivoting, the logdet alone differs by about
    kappa 2^-53 at kappa = 1e8, so the reference is the same schedule.)"""
    rng = np.random.default_rng(100 + k)
    worst = np.zeros(3)
    for cond in (1.0, 1e2, 1e4, 1e6, 1e8):
        for _ in range(10):
            M = spd(k, cond, rng)
            M = (M + M.T) / 2
            kappa = np.linalg.cond(M)
            d = rng.standard_normal(k)
            x, ld, u = gauss_jordan(M, d, np.float64)
            xe, lde, ue = gauss_jordan(M, d, np.longdouble)
            ex = float(abs(x - xe) / abs(xe))
            el = float(abs(ld - lde))
            eu = float(np.linalg.norm((u - ue).astype(np.float64)) / np.linalg.norm(ue.astype(np.float64)))
            assert ex <= 1e-13 * max(1.0, kappa / 100), (cond, ex)
            assert el <= 1e-14 * kappa, (cond, el)
            assert eu <= 1e-14 * kappa, (cond, eu)
            worst = np.maximum(worst, [ex / max(1.0, kappa / 100), el / kappa, eu / kappa])
    print(f"k = {k}: worst x {worst[0]:.1e} max(1, kappa/100), logdet {worst[1]:.1e} kappa, u {worst[2]:.1e} kappa")


def test_gauss_jordan_schedule_is_the_inverse():
    """The model itself: the sweep leaves M^-1 and the pivots multiply to det M."""
    rng = np.random.default_rng(1)
    M = spd(5, 10.0, rng)
    x, ld, u = gauss_jordan(M, np.arange(5.0), np.float64)
    assert np.allclose(u, np.linalg.solve(M, np.arange(5.0)), rtol=1e-12, atol=0)
    assert abs(ld - np.linalg.slogdet(M)[1]) <= 1e-12
