"""Solver plug-in for the reference's own registry seam.

The reference's front end (torchdiffeq/_impl/odeint.py:92-97) does

    solver = SOLVERS[method](func=func, y0=y0, rtol=rtol, atol=atol, **options)
    solution = solver.integrate(t)                       # or solver.integrate_until_event(t[0], event_fn)

after misc._check_inputs (misc.py:200-345) has flattened tuple states, made time ascending, wrapped func in
_PerturbFunc(_ReverseFunc(_TupleFunc(user func))) and put a norm into options['norm']; it also asks the class for
valid_callbacks() (misc.py:341).  adjoint.py:4 imports the SAME dict, so a registration also serves every backward
solve of odeint_adjoint.  The classes below honour exactly that contract on top of libtdq's engines, so that

    import torchdiffeq, torchdiffeq_b200.plugin
    torchdiffeq_b200.plugin.register()                   # patches torchdiffeq's SOLVERS in place

keeps the reference's front end (its input checks, tuple plumbing, event wrappers, adjoint) and replaces what runs
between the constructor and the returned solution for CUDA tensors; CPU tensors keep the reference's own solver.

Through this seam func's call count and order are observable (SURVEY.md 8(b) "Ownership"), so the default is the
reference's exact call sequence (lock step: 2 + S*attempts evaluations, callbacks in order).  Pass
options={'graph': True} (or register(graph=True)) for the captured step body inside the device-side loop.

What the seam cannot express: for tuple states and for every adjoint backward solve the reference hands the solver an
anonymous closure as `norm` (misc.py:251-254 around adjoint.py:247-271), which cannot be recognised; those solves take
the compatibility path -- err/tol is materialised by tdq_error_norm_commit(err_over_tol_out=...), the closure is
evaluated with torch ops and its scalar goes to tdq_controller(ratio_dev=...).  Only torchdiffeq_b200's own front end
can turn those norms into fused segments.
"""
import importlib
import warnings

import torch

from . import _lib
from ._engine import AdaptiveEngine, on_solver_stream
from ._fixed import FixedGridEngine, grid_from_step_size

ADAPTIVE = ("dopri5", "dopri8", "tsit5", "bosh3", "fehlberg2", "adaptive_heun")
FIXED = ("euler", "midpoint", "heun2", "heun3", "rk4")
ADAMS = {"explicit_adams": False, "implicit_adams": True, "fixed_adams": True}
_CB = ("callback_step", "callback_accept_step", "callback_reject_step")
_ADAPTIVE_KEYS = ("min_step", "max_step", "first_step", "step_t", "jump_t", "safety", "ifactor", "dfactor", "max_num_steps")
_OUR_KEYS = ("graph", "run_ahead", "device_loop")


def _is_default_rms(norm):
    """misc._rms_norm, recognised the only way the seam allows: by identity of the function object's origin."""
    return (getattr(norm, "__name__", "") == "_rms_norm"
            and getattr(norm, "__module__", "").rsplit(".", 1)[-1] in ("misc", "odeint", "seam_frontend"))


def _is_null_callback(cb):
    """misc._null_callback (misc.py:11), the placeholder _check_inputs sets for callbacks func does not define."""
    return (getattr(cb, "__name__", "") == "<lambda>"
            and getattr(cb, "__module__", "").rsplit(".", 1)[-1] in ("misc", "seam_frontend")
            and getattr(cb, "__qualname__", "") == "<lambda>")


def _unwrap_perturb(func):
    """The reference wraps func in _PerturbFunc (misc.py:174-197), which casts t to the state's real dtype through a
    full y.abs() pass and applies nextafter for Perturb.PREV/NEXT.  libtdq's controller already hands func stage times
    in the state dtype, perturbed where the reference perturbs them, so the wrapper is peeled off (it would be an
    N-element pass per evaluation that changes nothing)."""
    if type(func).__name__ == "_PerturbFunc" and hasattr(func, "base_func"):
        return func.base_func
    return func


def _callbacks_of(func, names):
    out = {}
    for n in names:
        cb = getattr(func, n, None)
        if cb is not None and not _is_null_callback(cb):
            out[n] = cb
    return out


def _tol(tol, device):
    """rtol/atol as the seam delivers them: a Python/0-dim scalar, or (tuple tolerances, misc.py:115-123) one value
    per element of the flat state."""
    if torch.is_tensor(tol) and tol.ndim > 0:
        return None, tol.detach().to(device=device, dtype=torch.float64).reshape(-1).contiguous()
    return float(tol), None


def make_adaptive(method, **defaults):
    """Class with the interface of RKAdaptiveStepsizeODESolver (rk_common.py:161-264) for one tableau."""

    class B200AdaptiveSolver:
        name = method

        def __init__(self, func, y0, rtol, atol, norm=None, dtype=torch.float64, **options):
            if not y0.is_cuda:
                raise _lib.TdqError("torchdiffeq_b200.plugin solvers take CUDA tensors (got %s)" % y0.device)
            if dtype != torch.float64:
                raise NotImplementedError("time dtype other than float64 (options['dtype']) is not implemented")
            self.func, self.y0, self.shape = func, y0, y0.shape
            self.base = _unwrap_perturb(func)
            opts = dict(defaults)
            opts.update(options)
            unused = {k: v for k, v in opts.items() if k not in _ADAPTIVE_KEYS + _OUR_KEYS}
            if unused:                                                         # misc.py:13-15
                warnings.warn('{}: Unexpected arguments {}'.format(self.__class__.__name__, unused))
            self.opts = opts
            self.rtol, self.rtol_vec = _tol(rtol, y0.device)
            self.atol, self.atol_vec = _tol(atol, y0.device)
            if (self.rtol_vec is None) != (self.atol_vec is None):
                if self.rtol_vec is None:
                    self.rtol_vec = torch.full_like(self.atol_vec, self.rtol)
                else:
                    self.atol_vec = torch.full_like(self.rtol_vec, self.atol)
            self.norm = None if (norm is None or _is_default_rms(norm)) else norm
            self.callbacks = _callbacks_of(func, _CB)
            self.engine = None

        @classmethod
        def valid_callbacks(cls):                                              # rk_common.py:207-211
            return set(_CB)

        def _engine(self, keep_interp):
            o, dev, shape = self.opts, self.y0.device, self.shape
            base = self.base

            def tvals(v):                                                      # rk_common.py:372-375 happens on the device
                return None if v is None else torch.as_tensor(v, dtype=torch.float64).to(dev)
            step_t, jump_t = tvals(o.get("step_t")), tvals(o.get("jump_t"))
            t0 = self._t0
            if step_t is not None:
                step_t = torch.sort(step_t[step_t >= t0]).values
            if jump_t is not None:
                jump_t = torch.sort(jump_t[jump_t >= t0]).values
            both = torch.cat([x for x in (step_t, jump_t) if x is not None]) if (step_t is not None or jump_t is not None) \
                else None
            if both is not None and (both.unique(return_counts=True)[1] > 1).any():        # rk_common.py:233-236
                raise ValueError("`step_t` and `jump_t` must not have any repeated elements between them.")
            lock = "graph" not in o and "run_ahead" not in o                   # default: the reference's call sequence
            return AdaptiveEngine(
                lambda t_, yf: base(t_, yf.view(shape)), self.y0.numel(), self.y0.dtype, dev, method,
                rtol=self.rtol, atol=self.atol, rtol_vec=self.rtol_vec, atol_vec=self.atol_vec,
                min_step=o.get("min_step", 0), max_step=o.get("max_step", float("inf")), first_step=o.get("first_step"),
                step_t=step_t, jump_t=jump_t, safety=o.get("safety", 0.9), ifactor=o.get("ifactor", 10.0),
                dfactor=o.get("dfactor", 0.2), max_num_steps=o.get("max_num_steps", 2 ** 31 - 1),
                norm_fn=self.norm, q_view=(lambda q: q.view(shape)) if self.norm is not None else None,
                graph=False if lock else o.get("graph", False), run_ahead=0 if lock else o.get("run_ahead", 2),
                device_loop=o.get("device_loop", "auto"), callbacks=self.callbacks, keep_interp=keep_interp)

        def integrate(self, t):                                                # solvers.py:28-35
            t_cpu = t.detach().to("cpu", torch.float64)
            self._t0 = float(t_cpu[0])
            with torch.no_grad(), on_solver_stream(self.y0.device) as ss:
                self.engine = eng = self._engine(False)
                sol = eng.solve(self.y0.detach().reshape(-1), t_cpu.to(self.y0.device), t_start=self._t0)
                sol = sol.view(len(t), *self.shape).clone()
                ss.publish(sol)
            return sol

        def integrate_until_event(self, t0, event_fn):                         # solvers.py:41-49, rk_common.py:252-264
            self._t0 = float(t0)
            shape = self.shape
            tol = self.atol if self.atol is not None else float(self.atol_vec.min())
            with torch.no_grad(), on_solver_stream(self.y0.device) as ss:
                self.engine = eng = self._engine(True)
                ev = lambda t_, yf: event_fn(t_, yf.view(shape))
                event_t, y1 = eng.solve_until_event(self.y0.detach().reshape(-1), self._t0, ev, tol)
                sol = torch.stack([self.y0.detach(), y1.view(shape)], dim=0)
                ss.publish(sol)
            return torch.tensor(event_t, dtype=torch.float64, device=self.y0.device), sol

    B200AdaptiveSolver.__name__ = B200AdaptiveSolver.__qualname__ = "B200_" + method
    return B200AdaptiveSolver


def make_fixed(method, **defaults):
    """Class with the interface of FixedGridODESolver (solvers.py:52-128) for one explicit fixed-step method, or of
    AdamsBashforth / AdamsBashforthMoulton (fixed_adams.py:164-228) for the Adams names."""
    adams = method in ADAMS

    class B200FixedSolver:
        name = method

        def __init__(self, func, y0, step_size=None, grid_constructor=None, interp="linear", perturb=False,
                     **unused_kwargs):
            if not y0.is_cuda:
                raise _lib.TdqError("torchdiffeq_b200.plugin solvers take CUDA tensors (got %s)" % y0.device)
            self.atol = unused_kwargs.pop("atol", None)                        # solvers.py:58-61
            self.rtol = unused_kwargs.pop("rtol", None)
            self.adams_kw = {k: unused_kwargs.pop(k) for k in ("max_iters", "max_order") if adams and k in unused_kwargs}
            unused_kwargs.pop("norm", None)
            self.our = {k: unused_kwargs.pop(k) for k in _OUR_KEYS if k in unused_kwargs}
            for k, v in defaults.items():
                self.our.setdefault(k, v)
            if unused_kwargs:
                warnings.warn('{}: Unexpected arguments {}'.format(self.__class__.__name__, unused_kwargs))
            self.func, self.y0, self.shape = func, y0, y0.shape
            self.base = _unwrap_perturb(func)
            self.step_size, self.interp, self.perturb = step_size, interp, perturb
            if step_size is None:                                              # solvers.py:70-79
                self.grid_constructor = grid_constructor if grid_constructor is not None else (lambda f, y0, t: t)
            else:
                if grid_constructor is not None:
                    raise ValueError("step_size and grid_constructor are mutually exclusive arguments.")
                self.grid_constructor = grid_from_step_size(step_size)
            self.callbacks = _callbacks_of(func, ("callback_step",))

        @classmethod
        def valid_callbacks(cls):                                              # solvers.py:81-83
            return {"callback_step"}

        def _make_engine(self, interp, graph):
            shape, base = self.shape, self.base
            fn = lambda t_, yf: base(t_, yf.view(shape))
            if adams:
                from ._adams import AdamsEngine
                return AdamsEngine(fn, self.y0.numel(), self.y0.dtype, self.y0.device, implicit=ADAMS[method],
                                   rtol=self.rtol if self.rtol is not None else 1e-3,
                                   atol=self.atol if self.atol is not None else 1e-4, perturb=self.perturb,
                                   callbacks=self.callbacks, interp=interp, **self.adams_kw)
            return FixedGridEngine(fn, self.y0.numel(), self.y0.dtype, self.y0.device, method=method, perturb=self.perturb,
                                   graph=graph, callbacks=self.callbacks, interp=interp)

        def integrate(self, t):                                                # solvers.py:102-128
            from .odeint import _cubic_or_linear
            interp = _cubic_or_linear(self.interp)
            shape = self.shape
            t_cpu = t.detach().to("cpu")
            grid = self.grid_constructor(self.func, self.y0, t_cpu).detach().to("cpu")
            assert grid[0] == t_cpu[0] and grid[-1] == t_cpu[-1]
            lock = "graph" not in self.our
            with torch.no_grad(), on_solver_stream(self.y0.device) as ss:
                eng = self._make_engine(interp, False if lock else self.our.get("graph", False))
                sol = eng.solve(self.y0.detach().reshape(-1), grid, t_cpu).view(len(t), *shape)
                ss.publish(sol)
            return sol

        def integrate_until_event(self, t0, event_fn):                         # solvers.py:130-164
            from .odeint import _cubic_or_linear, fixed_event_solve
            assert self.step_size is not None, ("Event handling for fixed step solvers currently requires `step_size` "
                                                "to be provided in options.")
            shape = self.shape
            with torch.no_grad(), on_solver_stream(self.y0.device) as ss:
                eng = self._make_engine(_cubic_or_linear(self.interp), False)
                ev = lambda t_, yf: event_fn(t_, yf.view(shape))
                event_t, y1 = fixed_event_solve(eng, self.y0.detach().reshape(-1), t0, self.step_size, ev, float(self.atol))
                sol = torch.stack([self.y0.detach(), y1.view(shape)], dim=0)
                ss.publish(sol)
            return event_t, sol

    B200FixedSolver.__name__ = B200FixedSolver.__qualname__ = "B200_" + method
    return B200FixedSolver


_STATE_DTYPES = (torch.float32, torch.float64, torch.complex64, torch.complex128)


class _Dispatch:
    """What goes into SOLVERS[name]: callable like a solver class, routes CUDA states to libtdq and everything else
    to the class that was registered before."""

    def __init__(self, name, gpu_cls, cpu_cls):
        self.name, self.gpu_cls, self.cpu_cls = name, gpu_cls, cpu_cls

    def __call__(self, func, y0, **kwargs):
        cls = self.gpu_cls if (torch.is_tensor(y0) and y0.is_cuda and y0.dtype in _STATE_DTYPES) else self.cpu_cls
        if cls is None:
            raise _lib.TdqError("no solver registered for %s on %s" % (self.name, y0.device))
        return cls(func=func, y0=y0, **kwargs)

    def valid_callbacks(self):
        return self.gpu_cls.valid_callbacks()


def register(solvers=None, methods=ADAPTIVE + FIXED + tuple(ADAMS), **defaults):
    """Put the libtdq-backed solvers into a SOLVERS dict (default: the reference's, found through
    importlib.import_module('torchdiffeq._impl.odeint') -- the attribute torchdiffeq._impl.odeint is shadowed by the
    function of the same name).  In place, so torchdiffeq._impl.adjoint sees it too.  Returns the dict of replaced
    entries for unregister()."""
    if solvers is None:
        solvers = importlib.import_module("torchdiffeq._impl.odeint").SOLVERS
    replaced = {}
    for name in methods:
        prev = solvers.get(name)
        if isinstance(prev, _Dispatch):
            prev = prev.cpu_cls
        replaced[name] = prev
        gpu = make_adaptive(name, **defaults) if name in ADAPTIVE else make_fixed(name, **defaults)
        solvers[name] = _Dispatch(name, gpu, prev)
    return replaced


def unregister(replaced, solvers=None):
    if solvers is None:
        solvers = importlib.import_module("torchdiffeq._impl.odeint").SOLVERS
    for name, cls in replaced.items():
        if cls is None:
            solvers.pop(name, None)
        else:
            solvers[name] = cls
