"""Routine to fit SQFA filters with L-BFGS -- drop-in for `sqfa._optim`.

The optimiser driver, stopping rule and progress reporting are host code with the semantics of the
reference (/root/reference/src/sqfa/_optim.py:33-145). The closure body -- the hot loop -- runs
natively: for the built-in distances the whole `get_class_distances -> check -> -mean(tril) ->
backward` sequence is ONE fused native evaluation (`_ops.FusedLoss`), for any other
`distance_fun` the projection is native and the user's function runs on device tensors.
"""

import os
import time

import torch
from torch import optim  # noqa: F401  (kept: the reference module exposes it)
from tqdm import tqdm

from ._lbfgs import LBFGS

__all__ = ["fitting_loop"]


def __dir__():
    return __all__


_NAN_MSG = "Some distances between classes are NaN. Try using float64 or a different regularization parameter."
_INF_MSG = "Some distances between classes are inf. Try using float64 or a different regularization parameter."


def check_distances_valid(distances):
    """
    Check if off-diagonal distances are valid. Raise an error if they are not
    (reference _optim.py:16-30; only the strict lower triangle is inspected).
    """
    n_classes = distances.shape[0]
    i, j = torch.tril_indices(n_classes, n_classes, offset=-1, device=distances.device)
    tril = distances[i, j]
    if torch.isnan(tril).any():
        raise ValueError(_NAN_MSG)
    if torch.isinf(tril).any():
        raise ValueError(_INF_MSG)


class _PlateauStop:
    """The reference's stopping rule (_optim.py:111-133) as one object: the loss of an epoch is compared
    with the loss of the epoch before (0.0 before the first), and training stops once the change
    has stayed below `atol` for `patience` epochs in a row."""

    def __init__(self, atol, patience=3):
        self.atol, self.patience = atol, patience
        self.last, self.run = 0.0, 0

    def observe(self, loss_value):
        self.run = self.run + 1 if abs(self.last - loss_value) < self.atol else 0
        self.last = loss_value

    @property
    def met(self):
        return self.run >= self.patience


class _EpochHistory:
    """Loss and wall-clock time since the start of the fit, one entry per epoch."""

    def __init__(self):
        self.t0 = time.time()
        self.losses, self.seconds = [], []

    def add(self, loss_value):
        self.seconds.append(time.time() - self.t0)
        self.losses.append(loss_value)

    @property
    def epochs(self):
        return len(self.losses)


def fitting_loop(
    model,
    data_statistics,
    max_epochs=200,
    lr=0.1,
    atol=1e-6,
    show_progress=True,
    return_loss=False,
    **kwargs,
):
    """
    Learn SQFA filters using the LBFGS optimizer.

    Same contract as the reference `fitting_loop` (_optim.py:33-145): `model.parameters()` are
    optimised with `torch.optim.LBFGS(lr=lr, **kwargs)`, one epoch is one `optimizer.step`, training
    stops after 3 consecutive epochs whose loss change is below `atol`. Returns
    `(loss per epoch, elapsed time per epoch)` tensors when `return_loss` is True, else None.
    """
    optimizer = LBFGS(model.parameters(), lr=lr, **kwargs)  # torch.optim.LBFGS, direction update on the device

    if isinstance(data_statistics, dict):
        n_classes = data_statistics["means"].shape[0]
    else:
        n_classes = data_statistics.shape[0]

    fused = model._fused_loss_plan(data_statistics) if hasattr(model, "_fused_loss_plan") else None
    direct = model._fused_direct_plan(data_statistics) if hasattr(model, "_fused_direct_plan") else None
    tril_ind = None
    evaluations = 0

    def closure():
        nonlocal tril_ind, evaluations
        evaluations += 1
        if direct is not None:
            # native loss + gradient, gradient written to .grad without an autograd graph; ONE host
            # read per evaluation, which also carries max|grad| for the optimiser's first stopping test
            loss_value, bad, grad_absmax = direct().tolist()
            if bad != 0 or loss_value != loss_value:
                raise ValueError(_NAN_MSG if loss_value != loss_value else _INF_MSG)
            optimizer._last_grad_absmax = grad_absmax
            if getattr(direct, "dtype", None) == torch.float64:
                # a float64 fit keeps its loss in float64, as on the composed path
                return torch.tensor(loss_value, dtype=torch.float64)
            return torch.tensor(loss_value)
        optimizer.zero_grad()
        if fused is not None:
            out = fused()  # [loss, #non-finite pair distances] -- one native evaluation
            loss_value, bad = out.detach().tolist()  # the single host read of this evaluation
            if bad != 0 or loss_value != loss_value:
                raise ValueError(_NAN_MSG if loss_value != loss_value else _INF_MSG)
            epoch_loss = out[0]
            epoch_loss.backward()
            # hand LBFGS a host scalar so its float(loss) does not synchronise again
            return torch.tensor(loss_value)
        distances = model.get_class_distances(data_statistics, regularized=True)
        check_distances_valid(distances)
        if tril_ind is None:
            tril_ind = torch.tril_indices(n_classes, n_classes, offset=-1, device=distances.device)
        epoch_loss = -torch.mean(distances[tril_ind[0], tril_ind[1]])
        epoch_loss.backward()
        return epoch_loss

    if (direct is not None and getattr(direct, "enqueue", None) is not None
            and os.environ.get("SQFA_LBFGS_PIPELINE", "1") == "1"):
        # the two halves of an evaluation for an optimiser that pipelines them (sqfa_b200._lbfgs.LBFGS)
        def collect():
            nonlocal evaluations
            evaluations += 1
            loss_value, bad, grad_absmax = direct.host_out.tolist()
            if bad != 0 or loss_value != loss_value:
                raise ValueError(_NAN_MSG if loss_value != loss_value else _INF_MSG)
            optimizer._last_grad_absmax = grad_absmax
            return loss_value

        closure.launch, closure.collect = direct.enqueue, collect

    stop_rule = _PlateauStop(atol)
    history = _EpochHistory()
    with tqdm(total=max_epochs, desc="Epochs", unit="epoch", disable=not show_progress) as bar:
        while history.epochs < max_epochs and not stop_rule.met:
            epoch_loss = optimizer.step(closure)
            history.add(epoch_loss.item() if isinstance(epoch_loss, torch.Tensor) else float(epoch_loss))
            stop_rule.observe(history.losses[-1])
            bar.update(1)
    if stop_rule.met:
        tqdm.write(
            f"Loss change below {atol} for 3 consecutive epochs. "
            f"Stopping training at epoch {history.epochs}/{max_epochs}."
        )
    else:
        print(
            f"Reached max_epochs ({max_epochs}) without meeting stopping criteria."
            + "Consider increasing max_epochs, changing initialization or using dtype=torch.float64."
        )

    # closure evaluations of this fit (benchmarks extrapolate the CPU fit time from it); summed over
    # the stages of a pairwise curriculum
    model._last_fit_evaluations = getattr(model, "_last_fit_evaluations", 0) + evaluations
    if return_loss:
        return torch.tensor(history.losses), torch.tensor(history.seconds)
    return None
