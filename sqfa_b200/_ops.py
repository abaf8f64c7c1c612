"""Host-side glue between torch tensors and the HP2 entry points of libsqfa_b200.so.

Raw wrappers (`*_raw`) take CUDA float32 tensors and call the C ABI; the `torch.autograd.Function`s
below give the kernels analytic backward passes so that filter constraints (parametrizations) and
`torch.optim.LBFGS` stay ordinary torch code above this boundary.
"""

import ctypes

import torch

from . import _lib

DIST_AI = 0  # SQFA_DIST_AFFINE_INVARIANT
DIST_FR = 1  # SQFA_DIST_FISHER_RAO_LB
DIST_LE = 2  # SQFA_DIST_LOG_EUCLIDEAN
DIST_BW = 3  # SQFA_DIST_BURES_WASSERSTEIN
DIST_W2 = 4  # SQFA_DIST_WASSERSTEIN_GAUSSIAN
DIST_MAHA = 5  # SQFA_DIST_MAHALANOBIS (closures only)
DIST_BHATT = 6  # SQFA_DIST_BHATTACHARYYA (closures only)
DIST_HELL = 7  # SQFA_DIST_HELLINGER (closures only)
SQUARED = 16  # SQFA_DIST_SQUARED
MAX_M = 64
MAX_M_BW = 34  # Bures-Wasserstein: column-pair kernel only
MAX_FILTERS = 32


def f32c(t, dev):
    """float32, contiguous, on `dev` (no copy when already so)."""
    return t.detach().to(device=dev, dtype=torch.float32).contiguous()


def _ws(nbytes, dev):
    return torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=dev)


# ------------------------------------------------------------------------------------------------
# raw kernel wrappers
# ------------------------------------------------------------------------------------------------
def project_fwd_raw(S, M, F):
    """T = F S_c, Psi = T F^T, Mu = F m_c for every class (one pass over S)."""
    lib = _lib.load()
    dev = S.device
    C, D, _ = S.shape
    k = F.shape[0]
    T = torch.empty(C, k, D, dtype=torch.float32, device=dev)
    Psi = torch.empty(C, k, k, dtype=torch.float32, device=dev)
    Mu = torch.empty(C, k, dtype=torch.float32, device=dev) if M is not None else None
    nbytes = lib.sqfa_project_workspace_bytes(C, D, k)
    ws = _ws(nbytes, dev)
    _lib.check(
        lib.sqfa_project_fwd(
            _lib.ptr(S), _lib.ptr(M), _lib.ptr(F), C, D, k, _lib.ptr(T), _lib.ptr(Psi), _lib.ptr(Mu), _lib.ptr(ws),
            nbytes, _lib.stream_ptr(dev),
        ),
        "sqfa_project_fwd",
    )
    return T, Psi, Mu


def project_bwd_raw(gPsi, gMu, T, M):
    lib = _lib.load()
    dev = T.device
    C, k, D = T.shape
    dF = torch.empty(k, D, dtype=torch.float32, device=dev)
    nbytes = lib.sqfa_project_workspace_bytes(C, D, k)
    ws = _ws(nbytes, dev)
    _lib.check(
        lib.sqfa_project_bwd(
            _lib.ptr(gPsi), _lib.ptr(gMu), _lib.ptr(T), _lib.ptr(M if gMu is not None else None), C, D, k,
            _lib.ptr(dF), _lib.ptr(ws), nbytes, _lib.stream_ptr(dev),
        ),
        "sqfa_project_bwd",
    )
    return dF


def transform_raw(X, F):
    lib = _lib.load()
    dev = X.device
    n, D = X.shape
    k = F.shape[0]
    Z = torch.empty(n, k, dtype=torch.float32, device=dev)
    if X.dtype in _lib.ELEM_CODES:  # bf16 / fp16 points, float32 filters and Z
        _lib.check(
            lib.sqfa_transform_h(_lib.ptr(X), X.stride(0), _lib.ELEM_CODES[X.dtype], _lib.ptr(F), n, D, k, _lib.ptr(Z),
                                 _lib.stream_ptr(dev)),
            "sqfa_transform_h",
        )
        return Z
    _lib.check(
        lib.sqfa_transform(_lib.ptr(X), X.stride(0), _lib.ptr(F), n, D, k, _lib.ptr(Z), _lib.stream_ptr(dev)),
        "sqfa_transform",
    )
    return Z


def embed_fwd_raw(Psi, Mu, noise, dist):
    lib = _lib.load()
    dev = Psi.device
    C, k, _ = Psi.shape
    m = k + 1 if (dist & 15) == DIST_FR else k
    E = torch.empty(C, m, m, dtype=torch.float32, device=dev)
    _lib.check(
        lib.sqfa_embed_fwd(_lib.ptr(Psi), _lib.ptr(Mu), float(noise), C, k, dist, _lib.ptr(E), _lib.stream_ptr(dev)),
        "sqfa_embed_fwd",
    )
    return E


def embed_bwd_raw(gE, Mu, k, dist):
    lib = _lib.load()
    dev = gE.device
    C = gE.shape[0]
    fr = (dist & 15) == DIST_FR
    gPsi = torch.empty(C, k, k, dtype=torch.float32, device=dev)
    gMu = torch.empty(C, k, dtype=torch.float32, device=dev) if fr else None
    _lib.check(
        lib.sqfa_embed_bwd(_lib.ptr(gE), _lib.ptr(Mu), C, k, dist, _lib.ptr(gPsi), _lib.ptr(gMu), _lib.stream_ptr(dev)),
        "sqfa_embed_bwd",
    )
    return gPsi, gMu


def class_factor_raw(E, dist):
    """Per-class Cholesky (+inverse) or, for log-Euclidean, eigendecomposition + matrix log."""
    lib = _lib.load()
    dev = E.device
    C, m, _ = E.shape
    if m > MAX_M:
        raise ValueError(f"SPD matrices larger than {MAX_M}x{MAX_M} are not supported by the pair kernels")
    W = torch.empty(C, lib.sqfa_class_factor_floats(m, dist), dtype=torch.float32, device=dev)
    flag = torch.empty(1, dtype=torch.int32, device=dev)
    _lib.check(
        lib.sqfa_class_factor(_lib.ptr(E), C, m, dist, _lib.ptr(W), _lib.ptr(flag), _lib.stream_ptr(dev)),
        "sqfa_class_factor",
    )
    return W, flag


def pair_raw(Wa, Wb, n_a, n_b, m, dist, tri, weight=1.0, gD=None, dist_out=None, loss=None, gEa=None, gEb=None,
             pair_range=None, eig_out=None):
    lib = _lib.load()
    total = n_a * (n_a - 1) // 2 if tri else n_a * n_b
    p0, p1 = (0, total) if pair_range is None else pair_range
    ws, nbytes = None, 0
    if loss is not None or gEa is not None:  # per-tile partial sums, reduced in a fixed order
        nbytes = lib.sqfa_pair_distances_workspace_bytes(n_a, n_b, m, dist, 1 if tri else 0, p0, p1)
        ws = _ws(nbytes, Wa.device)
    _lib.check(
        lib.sqfa_pair_distances(
            _lib.ptr(Wa), _lib.ptr(Wb), n_a, n_b, m, dist, 1 if tri else 0, p0, p1, float(weight), _lib.ptr(gD),
            _lib.ptr(dist_out), _lib.ptr(loss), _lib.ptr(gEa), _lib.ptr(gEb), _lib.ptr(eig_out), _lib.ptr(ws), nbytes,
            _lib.stream_ptr(Wa.device),
        ),
        "sqfa_pair_distances",
    )


def class_factor_bwd_raw(W, gLog, m, dist, gE):
    lib = _lib.load()
    _lib.check(
        lib.sqfa_class_factor_bwd(
            _lib.ptr(W), _lib.ptr(gLog), W.shape[0], m, dist, _lib.ptr(gE), _lib.stream_ptr(W.device)
        ),
        "sqfa_class_factor_bwd",
    )


# ------------------------------------------------------------------------------------------------
# autograd functions
# ------------------------------------------------------------------------------------------------
class Project(torch.autograd.Function):
    """(Psi, Mu) = (F S F^T, F m) for class scatters S (symmetric) and means m.

    Forward: conjugate_matrix(S, F) (reference linalg.py:41) + transform(means) (model.py:236).
    Backward w.r.t. F is analytic from the saved T = F S; gradients w.r.t. S / m (rarely needed,
    they are data) are plain torch ops on the device.
    """

    @staticmethod
    def forward(ctx, F, S, M):
        Fc = f32c(F, S.device)
        T, Psi, Mu = project_fwd_raw(S, M, Fc)
        ctx.save_for_backward(Fc, T, M if M is not None else torch.empty(0, device=S.device))
        ctx.has_means = M is not None
        if M is None:
            return Psi, Psi.new_zeros(())
        return Psi, Mu

    @staticmethod
    def backward(ctx, gPsi, gMu):
        Fc, T, M = ctx.saved_tensors
        gPsi = gPsi.contiguous().float()
        gMu_c = gMu.contiguous().float() if ctx.has_means else None
        dF = dS = dM = None
        if ctx.needs_input_grad[0]:
            dF = project_bwd_raw(gPsi, gMu_c, T, M if ctx.has_means else None)
        if ctx.needs_input_grad[1]:
            dS = torch.einsum("fi,cfg,gj->cij", Fc, gPsi, Fc)
        if ctx.has_means and ctx.needs_input_grad[2]:
            dM = gMu_c @ Fc
        return dF, dS, dM


class Embed(torch.autograd.Function):
    """Feature noise + (for Fisher-Rao) the Calvo-Oller embedding (reference distances.py:141-174)."""

    @staticmethod
    def forward(ctx, Psi, Mu, noise, dist):
        fr = (dist & 15) == DIST_FR
        Psi_c = Psi.contiguous().float()
        Mu_c = Mu.contiguous().float() if fr else None
        ctx.k, ctx.dist = Psi_c.shape[-1], dist
        ctx.save_for_backward(Mu_c if fr else torch.empty(0, device=Psi.device))
        return embed_fwd_raw(Psi_c, Mu_c, noise, dist)

    @staticmethod
    def backward(ctx, gE):
        (Mu,) = ctx.saved_tensors
        fr = (ctx.dist & 15) == DIST_FR
        gPsi, gMu = embed_bwd_raw(gE.contiguous().float(), Mu if fr else None, ctx.k, ctx.dist)
        return gPsi, gMu, None, None


class PairDistance(torch.autograd.Function):
    """Pairwise SPD distances D[a, b] = d(A_a, B_b) (AI / FR lower bound on embedded matrices /
    log-Euclidean; squared or not). `same=True` evaluates only the strict lower triangle and
    mirrors it. The backward re-runs the pair kernel with the upstream gradient as pair weights."""

    @staticmethod
    def forward(ctx, A, B, dist, same):
        A_c = A.contiguous().float()
        n_a, m, _ = A_c.shape
        Wa, _ = class_factor_raw(A_c, dist)
        if same:
            Wb, n_b = Wa, n_a
        else:
            B_c = B.contiguous().float()
            n_b = B_c.shape[0]
            Wb, _ = class_factor_raw(B_c, dist)
        D = torch.empty(n_a, n_b, dtype=torch.float32, device=A_c.device)
        pair_raw(Wa, Wb, n_a, n_b, m, dist, same, dist_out=D)
        ctx.save_for_backward(Wa, Wb)
        ctx.meta = (n_a, n_b, m, dist, same)
        return D

    @staticmethod
    def backward(ctx, gD):
        Wa, Wb = ctx.saved_tensors
        n_a, n_b, m, dist, same = ctx.meta
        dev = Wa.device
        gD = gD.contiguous().float()
        ga = torch.zeros(n_a, m, m, dtype=torch.float32, device=dev)
        gb = ga if same else torch.zeros(n_b, m, m, dtype=torch.float32, device=dev)
        pair_raw(Wa, Wb, n_a, n_b, m, dist, same, weight=1.0, gD=gD, gEa=ga, gEb=gb)
        if (dist & 15) == DIST_LE:  # ga / gb are gradients w.r.t. the matrix logs
            la, ga = ga, torch.zeros_like(ga)
            class_factor_bwd_raw(Wa, la, m, dist, ga)
            if same:
                gb = ga
            else:
                lb, gb = gb, torch.zeros_like(gb)
                class_factor_bwd_raw(Wb, lb, m, dist, gb)
        if same:
            return ga, None, None, None
        return ga, gb, None, None


GAUSS_MAHA_SQ = 0  # SQFA_GAUSS_MAHALANOBIS_SQ
GAUSS_BHATT = 1  # SQFA_GAUSS_BHATTACHARYYA


def gauss_pairs_raw(mu_a, sig_a, mu_b, sig_b, mode, gD=None):
    """Mean-covariance distances between Gaussians (Mahalanobis^2 / Bhattacharyya), all n_a x n_b pairs.
    Forward (gD None): returns D (n_a, n_b). Backward: returns (g_sig_a, g_mu_a, g_sig_b, g_mu_b)."""
    lib = _lib.load()
    dev = mu_a.device
    n_a, k = mu_a.shape
    n_b = mu_b.shape[0]
    grad = gD is not None
    nbytes = lib.sqfa_gauss_pair_workspace_bytes(n_a, n_b, k, 1 if grad else 0)
    ws = _ws(nbytes, dev)
    if grad:
        out = (torch.empty(n_a, k, k, dtype=torch.float32, device=dev), torch.empty(n_a, k, dtype=torch.float32, device=dev),
               torch.empty(n_b, k, k, dtype=torch.float32, device=dev), torch.empty(n_b, k, dtype=torch.float32, device=dev))
        D = None
    else:
        out = (None, None, None, None)
        D = torch.empty(n_a, n_b, dtype=torch.float32, device=dev)
    _lib.check(
        lib.sqfa_gauss_pair_distances(
            _lib.ptr(mu_a), _lib.ptr(sig_a), _lib.ptr(mu_b), _lib.ptr(sig_b), n_a, n_b, k, mode, _lib.ptr(gD), _lib.ptr(D),
            _lib.ptr(out[0]), _lib.ptr(out[1]), _lib.ptr(out[2]), _lib.ptr(out[3]), _lib.ptr(ws), nbytes, None,
            _lib.stream_ptr(dev),
        ),
        "sqfa_gauss_pair_distances",
    )
    return out if grad else D


class GaussPairDistance(torch.autograd.Function):
    """D[a, b] = mahalanobis_sq or bhattacharyya between the Gaussians (mu_a, Sigma_a) and (mu_b, Sigma_b)
    (reference distances.py:240-330), one warp per pair, analytic backward (second launch)."""

    @staticmethod
    def forward(ctx, mu_a, sig_a, mu_b, sig_b, mode):
        args = [t.contiguous().float() for t in (mu_a, sig_a, mu_b, sig_b)]
        ctx.save_for_backward(*args)
        ctx.mode = mode
        return gauss_pairs_raw(*args, mode)

    @staticmethod
    def backward(ctx, gD):
        mu_a, sig_a, mu_b, sig_b = ctx.saved_tensors
        g_sig_a, g_mu_a, g_sig_b, g_mu_b = gauss_pairs_raw(mu_a, sig_a, mu_b, sig_b, ctx.mode, gD.contiguous().float())
        return g_mu_a, g_sig_a, g_mu_b, g_sig_b, None


N_OUT = 3  # [loss, number of non-finite pair distances, max |gradient|]


def shard_pairs(n_pairs, n_classes, rank, world):
    """Slice [begin, end) of the linearised lower-triangle pair list (p = i (i - 1) / 2 + j) owned by
    `rank`: whole rows i, cut where the pair count is balanced and at multiples of 4 rows (a tile of the
    pair kernel that straddles a cut is evaluated by both ranks, each masking the other's pairs)."""
    if world <= 1:
        return 0, n_pairs

    def cut(r):
        if r <= 0:
            return 0
        if r >= world:
            return n_pairs
        target = n_pairs * r / world
        i = int((1 + (1 + 8 * target) ** 0.5) / 2)  # row whose first pair is nearest to the target
        i = min(max(4 * round(i / 4), 0), n_classes)
        return i * (i - 1) // 2

    return cut(rank), cut(rank + 1)


def _closure_workspace(lib, C, D, k, dist, p0, p1, dev, ws):
    nbytes = lib.sqfa_fused_loss_workspace_bytes(C, D, k, dist, p0, p1)
    if ws is None or ws.numel() < nbytes or ws.device != dev:
        ws = _ws(nbytes, dev)
    return ws


def fused_loss_raw(F, S, M, noise, dist, group=None, ws=None):
    """One native evaluation of the closure body at the (constrained) filters F: returns the packed
    device vector [loss, #non-finite pair distances, max|dF|, dLoss/dF (k*D)]. With a process group the
    pair list is split across ranks and the vector is all-reduced (entry 2 is then meaningless)."""
    lib = _lib.load()
    dev = S.device
    Fc = f32c(F, dev)
    C, D, _ = S.shape
    k = Fc.shape[0]
    P = C * (C - 1) // 2
    rank, world = 0, 1
    if group is not None:
        import torch.distributed as dist_mod

        rank, world = dist_mod.get_rank(group), dist_mod.get_world_size(group)
    p0, p1 = shard_pairs(P, C, rank, world)
    ws = _closure_workspace(lib, C, D, k, dist, p0, p1, dev, ws)
    # [loss, #non-finite, max|dF|, pad, dF...] in one buffer: one all-reduce when the pair list is sharded
    packed = torch.empty(4 + k * D, dtype=torch.float32, device=dev)
    _lib.check(
        lib.sqfa_fused_loss(
            _lib.ptr(S), _lib.ptr(M), _lib.ptr(Fc), C, D, k, float(noise), dist, p0, p1, _lib.ptr(packed),
            ctypes.c_void_p(packed.data_ptr() + 16), _lib.ptr(ws), ws.numel(), _lib.stream_ptr(dev),
        ),
        "sqfa_fused_loss",
    )
    if world > 1:
        import torch.distributed as dist_mod

        dist_mod.all_reduce(packed, group=group)
    return packed


def _exchange_spans(fn, C, D, k, dist, p0, p1, ws, dtype):
    """The two exchange spans of a sharded closure's workspace, as views of `dtype`."""
    lib = _lib.load()
    spans = []
    for which in (0, 1):
        off, nbytes = ctypes.c_size_t(0), ctypes.c_size_t(0)
        _lib.check(getattr(lib, fn)(C, D, k, dist, p0, p1, which, ctypes.byref(off), ctypes.byref(nbytes)), fn)
        spans.append(ws[off.value : off.value + nbytes.value].view(dtype))
    return spans


def fused_loss_sharded_raw(F, S, M, noise, dist, group, ws=None):
    """`fused_loss_raw` with the classes AND the pairs sharded over the ranks of `group` (AI / FR): every
    rank projects only its share of the classes (the part that reads C D^2 floats) and evaluates only its
    share of the pairs; three small all-reduces -- the per-chunk partials of (Psi, mu') [assembles all classes
    on every rank], the partial (gPsi, gMu, loss, flag), and dF. Returns the same packed vector."""
    import torch.distributed as dist_mod

    from ._stats_driver import class_share

    lib = _lib.load()
    dev = S.device
    Fc = f32c(F, dev)
    C, D, _ = S.shape
    k = Fc.shape[0]
    P = C * (C - 1) // 2
    rank, world = dist_mod.get_rank(group), dist_mod.get_world_size(group)
    p0, p1 = shard_pairs(P, C, rank, world)
    c0, c1 = class_share(C, rank, world)
    ws = _closure_workspace(lib, C, D, k, dist, p0, p1, dev, ws)
    spans = _exchange_spans("sqfa_fused_loss_exchange_span", C, D, k, dist, p0, p1, ws, torch.float32)
    packed = torch.empty(4 + k * D, dtype=torch.float32, device=dev)
    dF = ctypes.c_void_p(packed.data_ptr() + 16)

    def phase(i):
        _lib.check(
            lib.sqfa_fused_loss_sharded(i, _lib.ptr(S), _lib.ptr(M), _lib.ptr(Fc), C, D, k, float(noise), dist, c0, c1, p0,
                                        p1, dF, _lib.ptr(ws), ws.numel(), _lib.stream_ptr(dev)),
            "sqfa_fused_loss_sharded",
        )

    phase(0)
    dist_mod.all_reduce(spans[0], group=group)
    phase(1)
    dist_mod.all_reduce(spans[1], group=group)
    phase(2)
    dist_mod.all_reduce(packed[4:], group=group)
    packed[:4] = spans[1][-64:-60]  # {loss, #non-finite, -, -} summed over the ranks
    return packed


def closure_eval_raw(W, S, M, noise, dist, sphere, n_fixed, out, grad, ws, out_host=None):
    """One closure evaluation of the fitting loop at the RAW filter parameter W, constraint included:
    out <- [loss, #non-finite pair distances, max|grad|], grad <- dLoss/dW. Everything preallocated by
    the caller (the call is capturable in a CUDA graph). `out_host`: pinned host tensor [3] that the last
    kernel fills with a copy of `out` (pinned memory is mapped into the device's address space)."""
    lib = _lib.load()
    C, D, _ = S.shape
    k = W.shape[0]
    P = C * (C - 1) // 2
    _lib.check(
        lib.sqfa_closure_eval(
            _lib.ptr(S), _lib.ptr(M), _lib.ptr(W), C, D, k, float(noise), dist, 1 if sphere else 0, int(n_fixed), 0, P,
            _lib.ptr(out), _lib.ptr(out_host), _lib.ptr(grad), _lib.ptr(ws), ws.numel(), _lib.stream_ptr(S.device),
        ),
        "sqfa_closure_eval",
    )


def _closure_eval_f64(fn, W, S, M, noise, dist, sphere, n_fixed, out, grad, ws, out_host):
    lib = _lib.load()
    C, D, _ = S.shape
    k = W.shape[0]
    P = C * (C - 1) // 2
    _lib.check(
        getattr(lib, fn)(
            _lib.ptr(S), _lib.ptr(M), _lib.ptr(W), C, D, k, _lib.ptr(noise), dist, 1 if sphere else 0, int(n_fixed), 0,
            P, _lib.ptr(out), _lib.ptr(out_host), _lib.ptr(grad), _lib.ptr(ws), ws.numel(), _lib.stream_ptr(S.device),
        ),
        fn,
    )


def closure_eval_f64_raw(W, S, M, noise, dist, sphere, n_fixed, out, grad, ws, out_host=None):
    """`closure_eval_raw` in float64 (affine-invariant / Fisher-Rao lower bound): every tensor is float64 and
    `noise` is a one-element float64 device tensor, read by the kernels."""
    _closure_eval_f64("sqfa_closure_eval_f64", W, S, M, noise, dist, sphere, n_fixed, out, grad, ws, out_host)


def gauss_closure_eval_f64_raw(W, S, M, noise, dist, sphere, n_fixed, out, grad, ws, out_host=None):
    """`closure_eval_f64_raw` for the mean-covariance distances (Mahalanobis, Bhattacharyya, Hellinger); M, the
    class means, is required."""
    _closure_eval_f64("sqfa_gauss_closure_eval_f64", W, S, M, noise, dist, sphere, n_fixed, out, grad, ws, out_host)


def closure_workspace_bytes_f64(C, D, k, dist, p0, p1):
    """Workspace of the float64 closure of `dist` over pairs [p0, p1): the mean-covariance query for Mahalanobis,
    Bhattacharyya and Hellinger, the affine-invariant / Fisher-Rao one otherwise (0 for codes neither takes)."""
    lib = _lib.load()
    gauss = (dist & 15) in (DIST_MAHA, DIST_BHATT, DIST_HELL)
    query = lib.sqfa_gauss_closure_workspace_bytes_f64 if gauss else lib.sqfa_fused_loss_workspace_bytes_f64
    return int(query(C, D, k, dist, p0, p1))


def _group_rank(group):
    import torch.distributed as dist_mod

    return dist_mod.get_rank(group), dist_mod.get_world_size(group)


def fused_loss_f64_raw(F, S, M, noise, dist, group, ws):
    """`fused_loss_raw` in float64 with the pair list sharded over the ranks of `group`: every rank runs the
    single-device float64 closure (no constraint) at the constrained filters F on its `shard_pairs` range -- the
    losses and gradients of disjoint ranges add up -- and ONE all-reduce sums [loss, #non-finite, -, -, dF].
    `noise` is a one-element float64 device tensor. Returns the packed float64 vector (entry 2 is meaningless)."""
    import torch.distributed as dist_mod

    lib = _lib.load()
    C, D, _ = S.shape
    k = F.shape[0]
    rank, world = _group_rank(group)
    p0, p1 = shard_pairs(C * (C - 1) // 2, C, rank, world)
    gauss = (dist & 15) in (DIST_MAHA, DIST_BHATT, DIST_HELL)
    fn = "sqfa_gauss_closure_eval_f64" if gauss else "sqfa_closure_eval_f64"
    packed = torch.empty(4 + k * D, dtype=torch.float64, device=S.device)
    _lib.check(
        getattr(lib, fn)(
            _lib.ptr(S), _lib.ptr(M), _lib.ptr(F), C, D, k, _lib.ptr(noise), dist, 0, 0, p0, p1, _lib.ptr(packed),
            None, ctypes.c_void_p(packed.data_ptr() + 32), _lib.ptr(ws), ws.numel(), _lib.stream_ptr(S.device),
        ),
        fn,
    )
    dist_mod.all_reduce(packed, group=group)
    return packed


def fused_loss_sharded_f64_raw(F, S, M, noise, dist, group, ws):
    """`fused_loss_sharded_raw` in float64 (affine-invariant, Fisher-Rao, Mahalanobis, Bhattacharyya, Hellinger): the
    three phases of sqfa_fused_loss_sharded_f64 with the same three all-reduces, on float64 spans. `noise` is a
    one-element float64 device tensor. Returns the packed float64 vector [loss, #non-finite, -, -, dF]."""
    import torch.distributed as dist_mod

    from ._stats_driver import class_share

    lib = _lib.load()
    dev = S.device
    C, D, _ = S.shape
    k = F.shape[0]
    rank, world = _group_rank(group)
    p0, p1 = shard_pairs(C * (C - 1) // 2, C, rank, world)
    c0, c1 = class_share(C, rank, world)
    spans = _exchange_spans("sqfa_fused_loss_exchange_span_f64", C, D, k, dist, p0, p1, ws, torch.float64)
    packed = torch.empty(4 + k * D, dtype=torch.float64, device=dev)
    dF = ctypes.c_void_p(packed.data_ptr() + 32)

    def phase(i):
        _lib.check(
            lib.sqfa_fused_loss_sharded_f64(i, _lib.ptr(S), _lib.ptr(M), _lib.ptr(F), C, D, k, _lib.ptr(noise), dist,
                                            c0, c1, p0, p1, dF, _lib.ptr(ws), ws.numel(), _lib.stream_ptr(dev)),
            "sqfa_fused_loss_sharded_f64",
        )

    phase(0)
    dist_mod.all_reduce(spans[0], group=group)
    phase(1)
    dist_mod.all_reduce(spans[1], group=group)
    phase(2)
    dist_mod.all_reduce(packed[4:], group=group)
    packed[:4] = spans[1][-64:-60]  # {loss, #non-finite, -, -} summed over the ranks
    return packed


class FusedLoss(torch.autograd.Function):
    """The whole closure body of the reference's fitting loop (_optim.py:90-96) at fixed filters:

        loss = -mean_{i>j} d(E_i, E_j),   E_c from F S_c F^T (+ noise, + Fisher-Rao embedding)

    Forward runs projection -> embedding -> factorisation -> pair kernel (which also accumulates
    dLoss/dE) -> embedding adjoint -> projection adjoint, so the gradient w.r.t. F exists when the
    forward returns; backward just scales it. Returns a 2-vector [loss, #non-finite distances]
    (the NaN/inf guard of _optim.py:16-30 is applied by the caller after its one host read).
    With a process group, the pair list is split across ranks and [loss, flag, dF] is all-reduced.
    """

    @staticmethod
    def forward(ctx, F, S, M, noise, dist, group, ws=None):
        packed = fused_loss_raw(F, S, M, noise, dist, group, ws)
        k, D = F.shape[0], S.shape[1]
        ctx.save_for_backward(packed[4:].view(k, D))
        return packed[:2]

    @staticmethod
    def backward(ctx, g):
        (dF,) = ctx.saved_tensors
        return g[0] * dF, None, None, None, None, None, None
