"""L-BFGS with the direction update on the device (SURVEY.md section 8(f), rank 1).

`LBFGS` is `torch.optim.LBFGS` -- the optimiser the reference's `fitting_loop` uses
(reference _optim.py:78-79) -- with one change: when there is a single float32 or float64 CUDA parameter
and no line search (the reference's configuration), the "update memory + two-loop recursion" block of
`step` -- and the fixed step `x += t d` that follows it -- runs as ONE kernel (`sqfa_lbfgs_direction`,
`sqfa_lbfgs_direction_f64` for float64) instead of 4 tiny torch kernels and 2 implicit host
synchronisations per history entry; a closure that can be launched without a host wait is enqueued right
behind it (one host wait per iteration). Same algorithm, same update rule and stopping tests, same
order of floating-point operations up to the summation order inside each dot product. Every other
configuration -- line search, several parameters, a CPU parameter, more elements than the kernel holds
(`sqfa_lbfgs_max_n()` floats, `sqfa_lbfgs_max_n_f64()` doubles) or a longer history -- falls through to
`torch.optim.LBFGS.step` unchanged.
"""

import ctypes

import torch

from . import _lib

__all__ = ["LBFGS"]


class LBFGS(torch.optim.LBFGS):
    def _native_state(self):
        """Device buffers of the history, or None when this configuration is not handled natively."""
        group = self.param_groups[0]
        if group["line_search_fn"] is not None or len(self._params) != 1:
            return None
        p = self._params[0]
        if not (p.is_cuda and p.dtype in (torch.float32, torch.float64) and p.is_contiguous()):
            return None
        lib = _lib.load()
        n, hist = p.numel(), int(group["history_size"])
        max_n = lib.sqfa_lbfgs_max_n() if p.dtype == torch.float32 else lib.sqfa_lbfgs_max_n_f64()
        if n > max_n or hist > lib.sqfa_lbfgs_max_history() or hist < 1:
            return None
        state = self.state[p]
        nat = state.get("sqfa_native")
        if nat is None:
            dev, dt = p.device, p.dtype
            nat = {
                "prev_g": torch.zeros(n, dtype=dt, device=dev),
                "d": torch.zeros(n, dtype=dt, device=dev),
                "S": torch.empty(hist + 1, n, dtype=dt, device=dev),
                "Y": torch.empty(hist + 1, n, dtype=dt, device=dev),
                "ro": torch.zeros(hist + 1, dtype=dt, device=dev),
                "hdiag": torch.ones(1, dtype=dt, device=dev),
                "meta": torch.zeros(2, dtype=torch.int32, device=dev),
                "out": torch.zeros(8, dtype=dt).pin_memory(),  # written by the kernel (mapped)
                "t": 0.0,
            }
            state["sqfa_native"] = nat
        return nat

    def _direction(self, nat, g, history, first, param, lr, tolerance_change, then=None):
        """Launch the update AND the optimiser's fixed step on `param` (skipped by the kernel when the
        directional derivative is above -tolerance_change), then `then()` -- the next loss / gradient
        evaluation, enqueued behind it --, and wait once. Returns (ys, g.d, max|d|, sum|g|, pairs held, t,
        step applied) as Python numbers."""
        lib, dev = _lib.load(), g.device
        bufs = (_lib.ptr(g), _lib.ptr(nat["prev_g"]), _lib.ptr(nat["d"]), _lib.ptr(nat["S"]), _lib.ptr(nat["Y"]),
                 _lib.ptr(nat["ro"]), _lib.ptr(nat["hdiag"]), _lib.ptr(nat["meta"]), g.numel(), history)
        if g.dtype == torch.float64:
            # the float64 entry takes its three host scalars by pointer (the C ABI passes no double by value)
            scalars = (ctypes.c_double * 3)(float(nat["t"]), float(lr), float(tolerance_change))
            code = lib.sqfa_lbfgs_direction_f64(*bufs, scalars, 1 if first else 0, _lib.ptr(param),
                                                _lib.ptr(nat["out"]), _lib.stream_ptr(dev))
            _lib.check(code, "sqfa_lbfgs_direction_f64")
        else:
            code = lib.sqfa_lbfgs_direction(*bufs, float(nat["t"]), 1 if first else 0, _lib.ptr(param), float(lr),
                                            float(tolerance_change), _lib.ptr(nat["out"]), _lib.stream_ptr(dev))
            _lib.check(code, "sqfa_lbfgs_direction")
        if then is not None:
            then()
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(dev))
        ev.synchronize()  # the kernels stored their scalars in pinned host memory themselves: no copy
        return nat["out"][:7].tolist()

    def _grad_and_absmax(self, p):
        """Flat gradient (a view when possible: the kernel copies what it keeps) and max|grad|; a
        closure that already read that scalar with its loss leaves it in `_last_grad_absmax`."""
        g = p.grad
        flat = g.view(-1) if (g is not None and g.is_contiguous() and not g.is_sparse) else self._gather_flat_grad()
        absmax = self.__dict__.pop("_last_grad_absmax", None)
        if absmax is None:
            absmax = float(flat.abs().max())
        return flat, absmax

    @torch.no_grad()
    def step(self, closure):  # noqa: C901  (mirrors the control flow of torch.optim.LBFGS.step)
        nat = self._native_state()
        if nat is None:
            return super().step(closure)

        # A closure may offer its evaluation in two halves, `launch()` (enqueue, no host wait) and `collect()`
        # (read the result once the stream has been waited for): the evaluation at the new iterate is then
        # enqueued right behind the direction kernel and ONE host wait per iteration serves both.
        launch_eval, collect_eval = getattr(closure, "launch", None), getattr(closure, "collect", None)
        pipelined = launch_eval is not None and collect_eval is not None
        closure = torch.enable_grad()(closure)
        group = self.param_groups[0]
        lr = float(group["lr"])
        max_iter, max_eval = group["max_iter"], group["max_eval"]
        tolerance_grad, tolerance_change = group["tolerance_grad"], group["tolerance_change"]
        history = int(group["history_size"])
        p = self._params[0]
        state = self.state[p]
        state.setdefault("func_evals", 0)
        state.setdefault("n_iter", 0)

        orig_loss = closure()
        loss = float(orig_loss)
        current_evals = 1
        state["func_evals"] += 1
        with torch.cuda.device(p.device):
            flat_grad, grad_absmax = self._grad_and_absmax(p)
            if grad_absmax <= tolerance_grad:
                return orig_loss

            prev_loss = state.get("prev_loss")
            n_iter = 0
            while n_iter < max_iter:
                n_iter += 1
                state["n_iter"] += 1
                first = state["n_iter"] == 1
                evaluate = n_iter != max_iter
                # direction + fixed step (no line search) in one launch; the evaluation at the new point
                # right behind it. If the kernel finds the directional derivative above -tolerance_change it
                # leaves the parameter alone (torch.optim.LBFGS stops before stepping) and the evaluation
                # that was enqueued is not collected.
                _ys, _gtd, dmax, _g_l1, _held, t, stepped = self._direction(
                    nat, flat_grad, history, first, p, lr, tolerance_change,
                    then=launch_eval if (pipelined and evaluate) else None)
                prev_loss = loss
                nat["t"] = t
                if not stepped:  # directional derivative is below tolerance
                    break
                ls_func_evals = 0
                opt_cond = False
                if evaluate:
                    loss = float(collect_eval()) if pipelined else float(closure())
                    flat_grad, grad_absmax = self._grad_and_absmax(p)
                    opt_cond = grad_absmax <= tolerance_grad
                    ls_func_evals = 1
                current_evals += ls_func_evals
                state["func_evals"] += ls_func_evals
                if n_iter == max_iter or current_evals >= max_eval or opt_cond:
                    break
                if dmax * t <= tolerance_change:  # lack of progress
                    break
                if abs(loss - prev_loss) < tolerance_change:
                    break
        state["prev_loss"] = prev_loss
        return orig_loss
