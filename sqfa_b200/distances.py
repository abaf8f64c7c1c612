"""Distances between Symmetric Positive Definite matrices -- B200-native drop-in for
`sqfa.distances`.

The three distance families SQFA optimises (affine-invariant, its Calvo-Oller / Fisher-Rao
lower-bound use on embedded Gaussians, log-Euclidean; reference distances.py:46-237) run in the
warp-per-pair Jacobi kernels and are differentiable through analytic backward passes. The other
distances of the reference (Bhattacharyya, Mahalanobis, Hellinger, Fisher-Rao with shared
covariance; alternative `distance_fun` plug-ins, SURVEY.md section 8(f) row 4) run in a warp-per-pair
Cholesky kernel with an analytic backward. float64 inputs and matrices above 64 x 64 take the
reference's own composition with device-side library calls, in the dtype of the inputs. As `distance_fun`
of `SQFA`, `mahalanobis`, `mahalanobis_sq`, `bhattacharyya` and `hellinger` also fit through the models'
single-call native closure (up to 32 filters), in float32 and, for a `.double()` model on one device, in
float64; `fisher_rao_same_cov` keeps the generic path. The per-matrix functions stay composed in float64.

Extension (not reference API): the Bures-Wasserstein distance between SPD matrices and the
2-Wasserstein distance between Gaussians run in the same Jacobi pair kernel (up to 34 x 34) and
can be used as `distance_fun` of the models' native fitting closure.
"""

import torch

from . import _lib, _ops

__all__ = [
    "affine_invariant_sq",
    "affine_invariant",
    "log_euclidean_sq",
    "log_euclidean",
    "fisher_rao_lower_bound",
    "fisher_rao_lower_bound_sq",
    "bhattacharyya",
    "mahalanobis_sq",
    "mahalanobis",
    "hellinger",
    "fisher_rao_same_cov",
    "bures_wasserstein_sq",
    "bures_wasserstein",
    "wasserstein_sq",
    "wasserstein",
]


def __dir__():
    return __all__


EPSILON = 1e-6  # Value added inside of square roots


def _batch3(A):
    return A.unsqueeze(0) if A.dim() == 2 else A


def _unsq_mean(x):
    return x.unsqueeze(0) if x.dim() == 1 else x


def _pairwise_composed(a3, b3, dist):
    """The reference's own composition (distances.py:46-138) with device-side library calls, in the
    dtype of the inputs: for what the pair kernels do not take (float64, matrices above 64 x 64)."""
    from . import linalg

    if (dist & 15) == _ops.DIST_LE:
        diff = linalg.spd_log(a3)[:, None] - linalg.spd_log(b3)[None]
        d2 = (diff * diff).sum(dim=(-2, -1))
    elif (dist & 15) == _ops.DIST_BW:
        R = linalg.spd_sqrt(b3)
        inner = torch.linalg.eigvalsh(R[None] @ a3[:, None] @ R[None]).clamp_min(0)
        tr_a = torch.diagonal(a3, dim1=-2, dim2=-1).sum(-1)
        tr_b = torch.diagonal(b3, dim1=-2, dim2=-1).sum(-1)
        d2 = (tr_a[:, None] + tr_b[None] - 2 * torch.sqrt(inner).sum(dim=-1)).clamp_min(0)
    else:
        W = linalg.spd_inv_sqrt(b3)
        conj = W[None] @ a3[:, None] @ W.transpose(-2, -1)[None]
        d2 = (torch.log(torch.linalg.eigvalsh(conj)) ** 2).sum(dim=-1)
        if (dist & 15) == _ops.DIST_FR:
            d2 = d2 / 2
    return d2 if dist & _ops.SQUARED else torch.sqrt(d2 + EPSILON)


def _pairwise(A, B, dist):
    """D[a, b] = d(A_a, B_b) through the native pair kernels; squeezes like the reference."""
    same = A is B
    a3, b3 = _batch3(A), _batch3(B)
    if a3.shape[-1] != a3.shape[-2] or b3.shape[-1] != a3.shape[-1]:
        raise ValueError("expected SPD matrices of equal size, shapes (n, m, m)")
    dev = _lib.compute_device(A, B)
    with torch.cuda.device(dev):
        max_m = _ops.MAX_M_BW if (dist & 15) == _ops.DIST_BW else _ops.MAX_M
        if a3.dtype == torch.float32 and b3.dtype == torch.float32 and a3.shape[-1] <= max_m:
            D = _ops.PairDistance.apply(a3.to(dev), None if same else b3.to(dev), dist, same)
        else:
            D = _pairwise_composed(a3.to(dev), b3.to(dev), dist)
    return torch.squeeze(D).to(device=A.device, dtype=A.dtype)


def affine_invariant_sq(A, B):
    """Squared affine invariant distance between SPD matrices, shape (n_batch_A, n_batch_B)
    (reference distances.py:46-67): sum of squared logs of the generalized eigenvalues."""
    return _pairwise(A, B, _ops.DIST_AI | _ops.SQUARED)


def affine_invariant(A, B):
    """Affine invariant distance, sqrt(d^2 + 1e-6) (reference distances.py:70-89)."""
    return _pairwise(A, B, _ops.DIST_AI)


def log_euclidean_sq(A, B):
    """Squared log-Euclidean distance ||log A - log B||_F^2 (reference distances.py:92-116)."""
    return _pairwise(A, B, _ops.DIST_LE | _ops.SQUARED)


def log_euclidean(A, B):
    """Log-Euclidean distance, sqrt(d^2 + 1e-6) (reference distances.py:119-138)."""
    return _pairwise(A, B, _ops.DIST_LE)


def bures_wasserstein_sq(A, B):
    """Squared Bures-Wasserstein distance between SPD matrices, shape (n_batch_A, n_batch_B), squeezed
    like `affine_invariant_sq`: tr A + tr B - 2 tr((B^1/2 A B^1/2)^1/2), clamped at 0.

    Extension, not reference API (the reference's tutorial writes it as a custom `distance_fun`).
    float32 matrices up to 34 x 34 run in the native pair kernel with an analytic backward; float64
    and larger matrices take a composition of device-side library calls in the input dtype."""
    return _pairwise(A, B, _ops.DIST_BW | _ops.SQUARED)


def bures_wasserstein(A, B):
    """Bures-Wasserstein distance, sqrt(d^2 + 1e-6) (extension, not reference API; see
    `bures_wasserstein_sq`)."""
    return _pairwise(A, B, _ops.DIST_BW)


def _wasserstein_sq(statistics_A, statistics_B):
    mu_a, mu_b = _unsq_mean(statistics_A["means"]), _unsq_mean(statistics_B["means"])
    cov_a = statistics_A["covariances"]
    cov_b = cov_a if statistics_B is statistics_A else statistics_B["covariances"]
    bw = bures_wasserstein_sq(cov_a, cov_b)
    diff = mu_a[:, None] - mu_b.to(mu_a.device)[None]
    return torch.squeeze((diff * diff).sum(dim=-1)).to(bw.device) + bw


def wasserstein_sq(statistics_A, statistics_B):
    """Squared 2-Wasserstein distance between Gaussians given as dicts with "means" (n, k) and
    "covariances" (n, k, k): |mu_A - mu_B|^2 + `bures_wasserstein_sq` of the covariances, shape
    (n_A, n_B), squeezed. Extension, not reference API."""
    return _wasserstein_sq(statistics_A, statistics_B)


def wasserstein(statistics_A, statistics_B):
    """2-Wasserstein distance between Gaussians, sqrt(max(d^2, 0) + 1e-6) (extension, not reference
    API; see `wasserstein_sq`)."""
    return torch.sqrt(_wasserstein_sq(statistics_A, statistics_B).clamp_min(0) + EPSILON)


def _embed_gaussian(statistics):
    """Calvo-Oller embedding [[cov + mu mu^T, mu], [mu^T, 1]] of Gaussians into SPD(k+1)
    (reference distances.py:141-174), native kernel with an analytic adjoint."""
    means = statistics["means"]
    covariances = statistics["covariances"]
    if means.dim() == 1:
        means = means.unsqueeze(0)
    covariances = _batch3(covariances)
    dev = _lib.compute_device(means, covariances)
    with torch.cuda.device(dev):
        return _ops.Embed.apply(covariances.to(dev), means.to(dev), 0.0, _ops.DIST_FR)


def _embed_gaussian_composed(statistics):
    """distances.py:141-174 with torch ops (any dtype / size)."""
    means = _unsq_mean(statistics["means"])
    covariances = _batch3(statistics["covariances"])
    second = covariances + means.unsqueeze(-1) * means.unsqueeze(-2)
    top = torch.cat([second, means.unsqueeze(-1)], dim=-1)
    one = torch.ones(means.shape[0], 1, 1, dtype=means.dtype, device=means.device)
    bottom = torch.cat([means.unsqueeze(-2), one], dim=-1)
    return torch.cat([top, bottom], dim=-2)


def _fisher_rao(statistics_A, statistics_B, dist):
    ref = statistics_A["means"]
    cov = statistics_A["covariances"]
    if ref.dtype != torch.float32 or cov.dtype != torch.float32 or cov.shape[-1] + 1 > _ops.MAX_M:
        dev = _lib.compute_device(ref, cov)
        with torch.cuda.device(dev):
            EA = _embed_gaussian_composed({k: v.to(dev) for k, v in statistics_A.items()})
            EB = EA if statistics_B is statistics_A else _embed_gaussian_composed(
                {k: v.to(dev) for k, v in statistics_B.items()})
            D = _pairwise_composed(EA, EB, dist)
        return torch.squeeze(D).to(device=ref.device, dtype=ref.dtype)
    EA = _embed_gaussian(statistics_A)
    EB = EA if statistics_B is statistics_A else _embed_gaussian(statistics_B)
    with torch.cuda.device(EA.device):
        D = _ops.PairDistance.apply(EA, None if EB is EA else EB, dist, EB is EA)
    return torch.squeeze(D).to(device=ref.device, dtype=ref.dtype)


def fisher_rao_lower_bound_sq(statistics_A, statistics_B):
    """Calvo & Oller lower bound of the squared Fisher-Rao distance between Gaussians given as
    dicts with "means" (n, k) and "covariances" (n, k, k) (reference distances.py:177-207)."""
    return _fisher_rao(statistics_A, statistics_B, _ops.DIST_FR | _ops.SQUARED)


def fisher_rao_lower_bound(statistics_A, statistics_B):
    """sqrt(lower bound^2 + 1e-6) (reference distances.py:210-237)."""
    return _fisher_rao(statistics_A, statistics_B, _ops.DIST_FR)


# ------------------------------------------------------------------------------------------------
# The reference's other distance_fun plug-ins (distances.py:240-432): distances between Gaussians under
# the MEAN covariance of the pair. Native: one warp per pair (Cholesky of the mean covariance), analytic
# backward; mahalanobis, hellinger and fisher_rao_same_cov are scalar maps of the two kernels' outputs.
# In a fit, all but fisher_rao_same_cov run the closure of gauss.cu instead (strict lower triangle only, the
# scalar map and its derivative inside the pair stage; DESIGN.md section 17).
# ------------------------------------------------------------------------------------------------
def _gauss_pairs(statistics_A, statistics_B, mode):
    """(n_a, n_b) matrix of mahalanobis_sq / bhattacharyya values (not squeezed)."""
    mu_a, mu_b = _unsq_mean(statistics_A["means"]), _unsq_mean(statistics_B["means"])
    cov_a, cov_b = _batch3(statistics_A["covariances"]), _batch3(statistics_B["covariances"])
    ref = statistics_A["means"]
    dev = _lib.compute_device(mu_a, cov_a, mu_b, cov_b)
    native = all(t.dtype == torch.float32 for t in (mu_a, mu_b, cov_a, cov_b)) and cov_a.shape[-1] <= _ops.MAX_M
    with torch.cuda.device(dev):
        mu_a, mu_b, cov_a, cov_b = (t.to(dev) for t in (mu_a, mu_b, cov_a, cov_b))
        if native:
            D = _ops.GaussPairDistance.apply(mu_a, cov_a, mu_b, cov_b, mode)
        else:  # float64 / large matrices: the reference's composition with device-side library calls
            mean_cov = 0.5 * (cov_a[:, None] + cov_b[None])
            diff = mu_a[:, None] - mu_b[None]
            D = torch.einsum("abi,abij,abj->ab", diff, torch.linalg.inv(mean_cov), diff)
            if mode == _ops.GAUSS_BHATT:
                logdet = torch.logdet(mean_cov) - 0.5 * (torch.logdet(cov_a)[:, None] + torch.logdet(cov_b)[None])
                D = 0.125 * D + 0.5 * logdet
    return D.to(device=ref.device, dtype=ref.dtype)


def bhattacharyya(statistics_A, statistics_B):
    """Bhattacharyya distance between Gaussians (reference distances.py:240-280)."""
    return torch.squeeze(_gauss_pairs(statistics_A, statistics_B, _ops.GAUSS_BHATT))


def mahalanobis_sq(statistics_A, statistics_B):
    """Squared Mahalanobis distance under the pairwise mean covariance, shape (n_a, n_b) (reference
    distances.py:283-330; not squeezed, like the reference)."""
    return _gauss_pairs(statistics_A, statistics_B, _ops.GAUSS_MAHA_SQ)


def mahalanobis(statistics_A, statistics_B):
    """Mahalanobis distance (reference distances.py:333-361)."""
    return torch.sqrt(mahalanobis_sq(statistics_A, statistics_B) + EPSILON)


def hellinger(statistics_A, statistics_B):
    """Hellinger distance between Gaussians (reference distances.py:364-393)."""
    return torch.sqrt(1 - torch.exp(-bhattacharyya(statistics_A, statistics_B)) + EPSILON)


def fisher_rao_same_cov(statistics_A, statistics_B):
    """Fisher-Rao distance between Gaussians assumed to share a covariance (reference
    distances.py:396-432)."""
    m_sq = mahalanobis_sq(statistics_A, statistics_B)
    return 2.0**0.5 * torch.acosh(1 + m_sq / 4)
