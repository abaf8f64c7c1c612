"""CPU: the C ABI of the class- and pair-sharded float64 closure -- its prototypes, the geometry of the two exchange
spans inside the workspace, and every rejection (code and message) before anything touches the device."""

import ctypes

import pytest

AI, FR, LE, BW, W2, MAHA, BHATT, HELL, SQUARED = 0, 1, 2, 3, 4, 5, 6, 7, 16
CODES = (AI, AI | SQUARED, FR, FR | SQUARED, MAHA, MAHA | SQUARED, BHATT, HELL)


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge

    ge.build()
    from sqfa_b200 import _lib

    return _lib.load()


def _al(n):
    """n doubles rounded up to whole 256-byte granules, as the workspace layout places them."""
    return (n + 31) // 32 * 32


def _workspace_bytes(lib, C, D, k, dist, p0, p1):
    gauss = (dist & 15) in (MAHA, BHATT, HELL)
    query = lib.sqfa_gauss_closure_workspace_bytes_f64 if gauss else lib.sqfa_fused_loss_workspace_bytes_f64
    return query(C, D, k, dist, p0, p1)


def _span(lib, C, D, k, dist, p0, p1, which):
    off, nb = ctypes.c_size_t(0), ctypes.c_size_t(0)
    rc = lib.sqfa_fused_loss_exchange_span_f64(C, D, k, dist, p0, p1, which, ctypes.byref(off), ctypes.byref(nb))
    assert rc == 0, lib.sqfa_last_error()
    return off.value, nb.value


def test_prototypes_are_bound(lib):
    from sqfa_b200 import _lib
    from test_abi import header_prototypes

    protos = header_prototypes()
    for name in ("sqfa_fused_loss_exchange_span_f64", "sqfa_fused_loss_sharded_f64"):
        assert name in _lib.SIGNATURES and name in protos
        assert hasattr(lib, name) and name not in lib.sqfa_missing_symbols
    # the float32 prototypes with double pointers and the noise as a device pointer
    f32 = _lib.SIGNATURES["sqfa_fused_loss_sharded"][1]
    f64 = _lib.SIGNATURES["sqfa_fused_loss_sharded_f64"][1]
    assert len(f64) == len(f32) == 17
    assert [a for i, a in enumerate(f64) if i != 7] == [a for i, a in enumerate(f32) if i != 7]
    assert f64[7] is ctypes.c_void_p
    assert _lib.SIGNATURES["sqfa_fused_loss_exchange_span_f64"] == _lib.SIGNATURES["sqfa_fused_loss_exchange_span"]


@pytest.mark.parametrize("dist", CODES)
@pytest.mark.parametrize("C,D,k", [(1000, 512, 16), (100, 1024, 32), (37, 40, 5), (2, 16, 1)])
def test_span_geometry(lib, dist, C, D, k):
    """Both spans lie inside the workspace of every rank's pair range, 16-byte aligned and disjoint. Span 0 is
    exactly the per-chunk partials of Psi and mu' (64 columns per chunk); span 1 is [gPsi | gMu | 64 doubles]."""
    P = C * (C - 1) // 2
    nchunk = (D + 63) // 64
    for p0, p1 in ((0, P), (0, P // 3), (P // 3, P), (P, P)):
        ws = _workspace_bytes(lib, C, D, k, dist, p0, p1)
        assert ws > 0
        s0 = _span(lib, C, D, k, dist, p0, p1, 0)
        s1 = _span(lib, C, D, k, dist, p0, p1, 1)
        for off, nb in (s0, s1):
            assert off % 16 == 0 and nb % 8 == 0 and nb > 0
            assert off + nb <= ws
        assert s0[0] + s0[1] <= s1[0] or s1[0] + s1[1] <= s0[0]
        assert s0[1] == 8 * (_al(C * nchunk * k * k) + _al(C * nchunk * k))
        assert s1[1] == 8 * (_al(C * k * k) + _al(C * k) + 64)


def test_argument_validation_without_a_launch(lib):
    """Every rejection happens before anything touches the device (the pointers below are not device memory)."""
    fake = ctypes.c_void_p(4096)
    C, D, k = 5, 16, 3
    P = C * (C - 1) // 2

    def call(phase=0, S=fake, M=fake, F=fake, C=C, D=D, k=k, noise=fake, dist=FR, c0=0, c1=C, p0=0, p1=P, dF=fake,
             ws=fake, ws_bytes=0):
        return lib.sqfa_fused_loss_sharded_f64(phase, S, M, F, C, D, k, noise, dist, c0, c1, p0, p1, dF, ws, ws_bytes,
                                               None)

    def invalid(**kw):
        assert call(**kw) == -1, kw
        assert lib.sqfa_last_error().startswith(b"sqfa_fused_loss_sharded_f64:"), lib.sqfa_last_error()

    for phase in (-1, 3):
        invalid(phase=phase)
    for c0, c1 in ((-1, 2), (3, 2), (0, C + 1)):
        invalid(c0=c0, c1=c1)
    invalid(S=None)
    invalid(F=None)
    invalid(ws=None)
    invalid(noise=None)
    invalid(ws=ctypes.c_void_p(4104))
    invalid(phase=2, dF=None)
    for dist in (FR, MAHA, MAHA | SQUARED, BHATT, HELL):
        invalid(dist=dist, M=None)
    for p0, p1 in ((-1, P), (0, P + 1), (3, 2)):
        invalid(p0=p0, p1=p1)
        assert b"pair range" in lib.sqfa_last_error()
    for dist in (BHATT | SQUARED, HELL | SQUARED, 32, -1):
        invalid(dist=dist)
    # known codes without a native float64 closure, and k > 32
    for dist in (LE, LE | SQUARED, BW, BW | SQUARED, W2, W2 | SQUARED):
        assert call(dist=dist) == -3, dist
        msg = lib.sqfa_last_error()
        assert b"SQFA_DIST_AFFINE_INVARIANT" in msg and b"SQFA_DIST_HELLINGER" in msg, msg
    assert call(k=33) == -3 and b"n_filters" in lib.sqfa_last_error()
    # the affine-invariant distance reads no means; phases 0 and 1 take no dF
    for dist in CODES:
        M = None if dist & 15 == AI else fake
        for phase in (0, 1, 2):
            dF = fake if phase == 2 else None
            assert call(phase=phase, dist=dist, M=M, dF=dF) == -2, (dist, phase)
            assert b"workspace" in lib.sqfa_last_error()
            need = _workspace_bytes(lib, C, D, k, dist, 0, P)
            assert call(phase=phase, dist=dist, M=M, dF=dF, ws_bytes=need - 1) == -2
    # a rank's pair range takes the workspace of that range
    p1 = P // 2
    need = _workspace_bytes(lib, C, D, k, FR, 0, p1)
    assert need < _workspace_bytes(lib, C, D, k, FR, 0, P)
    assert call(p1=p1, ws_bytes=need - 1) == -2


def test_exchange_span_validation(lib):
    C, D, k = 5, 16, 3
    P = C * (C - 1) // 2
    off, nb = ctypes.c_size_t(0), ctypes.c_size_t(0)
    span = lib.sqfa_fused_loss_exchange_span_f64
    assert span(C, D, k, FR, 0, P, 2, ctypes.byref(off), ctypes.byref(nb)) == -1
    assert span(C, D, k, FR, 0, P, 0, None, ctypes.byref(nb)) == -1
    assert span(0, D, k, FR, 0, 0, 0, ctypes.byref(off), ctypes.byref(nb)) == -1
    assert span(C, D, k, FR, 0, P + 1, 0, ctypes.byref(off), ctypes.byref(nb)) == -1
    assert span(C, D, k, LE, 0, P, 0, ctypes.byref(off), ctypes.byref(nb)) == -3
    assert span(C, D, 33, FR, 0, P, 0, ctypes.byref(off), ctypes.byref(nb)) == -3


def test_single_device_entries_keep_their_codes(lib):
    """The single-device float64 entries accept and reject what they did: each still refuses the other's codes."""
    fake = ctypes.c_void_p(4096)
    C, D, k = 4, 16, 3
    P = C * (C - 1) // 2
    for fn, other in ((lib.sqfa_closure_eval_f64, (MAHA, BHATT, HELL)), (lib.sqfa_gauss_closure_eval_f64, (AI, FR))):
        for dist in other + (LE, BW, W2):
            assert fn(fake, fake, fake, C, D, k, fake, dist, 1, 0, 0, P, fake, None, fake, fake, 0, None) == -3
