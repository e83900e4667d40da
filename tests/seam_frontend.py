"""Stand-in for the CALLER side of the reference's solver-registry seam, used by the plug-in tests so that they
do not need the reference package installed.

It restates only what reaches a solver through the seam (misc.py:200-345 _check_inputs and odeint.py:90-108):
tuple states flattened with torch.cat, tuple tolerances expanded to one value per element, time made ascending with
a sign-flipping wrapper, the perturb= wrapper, the callback attributes (with a null lambda for absent ones),
options['norm'] always set (the module-level _rms_norm for tensor states, an anonymous closure for tuple states) and
the SOLVERS[method](func=..., y0=..., rtol=..., atol=..., **options).integrate(t) / .integrate_until_event(t0,
event_fn) calls.  odeint_adjoint restates what the reference's adjoint (adjoint.py) hands the same seam in its
backward pass: one solve per output interval, backwards in time, of the tuple state (t, y, adj_y, *adj_params) with
an anonymous norm closure.  Test infrastructure, not product."""
import torch

_all_callback_names = ['callback_step', 'callback_accept_step', 'callback_reject_step']
_null_callback = lambda *args, **kwargs: None
SOLVERS = {}


def _rms_norm(tensor):
    return tensor.abs().pow(2).mean().sqrt()


def _mixed_norm(tensor_tuple):
    return max([_rms_norm(tensor) for tensor in tensor_tuple])


def _flat_to_shape(tensor, length, shapes):
    out, total = [], 0
    for shape in shapes:
        nxt = total + shape.numel()
        out.append(tensor[..., total:nxt].view((*length, *shape)))
        total = nxt
    return tuple(out)


def _tuple_tol(tol, shapes):
    """A tolerance given per tuple element becomes one value per element of the flat state (misc.py:115-123)."""
    if not isinstance(tol, (tuple, list)):
        return tol
    assert len(tol) == len(shapes), "a tuple tolerance needs one value per tuple element"
    return torch.cat([torch.as_tensor(v).expand(shape.numel()) for v, shape in zip(tol, shapes)])


class _TupleFunc(torch.nn.Module):
    def __init__(self, base_func, shapes):
        super().__init__()
        self.base_func, self.shapes = base_func, shapes

    def forward(self, t, y):
        f = self.base_func(t, _flat_to_shape(y, (), self.shapes))
        return torch.cat([f_.reshape(-1) for f_ in f])


class _ReverseFunc(torch.nn.Module):
    def __init__(self, base_func, mul=1.0):
        super().__init__()
        self.base_func, self.mul = base_func, mul

    def forward(self, t, y):
        return self.mul * self.base_func(-t, y)


class _PerturbFunc(torch.nn.Module):
    def __init__(self, base_func):
        super().__init__()
        self.base_func = base_func

    def forward(self, t, y, *, perturb=None):
        return self.base_func(t.to(y.abs().dtype), y)


def odeint(func, y0, t, *, rtol=1e-7, atol=1e-9, method=None, options=None, event_fn=None):
    original_func = func
    shapes = None
    if not isinstance(y0, torch.Tensor):
        shapes = [y_.shape for y_ in y0]
        y0 = torch.cat([y_.reshape(-1) for y_ in y0])
        func = _TupleFunc(func, shapes)
        rtol, atol = _tuple_tol(rtol, shapes), _tuple_tol(atol, shapes)
        if event_fn is not None:
            ev_user = event_fn
            event_fn = lambda t_, y_: ev_user(t_, _flat_to_shape(y_, (), shapes))
    options = {} if options is None else options.copy()
    method = method or 'dopri5'
    if shapes is not None:
        norm = options.get('norm', _mixed_norm)

        def _norm(tensor):
            return norm(_flat_to_shape(tensor, (), shapes))
        options['norm'] = _norm
    elif 'norm' not in options:
        options['norm'] = _rms_norm
    t_is_reversed = len(t) > 1 and bool(t[0] > t[1])
    if t_is_reversed:
        t = -t
        func = _ReverseFunc(func, mul=-1.0)
        if event_fn is not None:
            event_fn = _ReverseFunc(event_fn)
        for name in ('step_t', 'jump_t'):
            if name in options:
                options[name] = -options[name]
    func = _PerturbFunc(func)
    for name in _all_callback_names:
        cb = getattr(original_func, name, None)
        if cb is None:
            setattr(func, name, _null_callback)
        else:
            if shapes is not None:
                cb = (lambda t0, y_, dt, _cb=cb: _cb(t0, _flat_to_shape(y_, (), shapes), dt))
            if t_is_reversed:
                cb = (lambda t0, y_, dt, _cb=cb: _cb(-t0, y_, dt))
            setattr(func, name, cb)
    SOLVERS[method].valid_callbacks()
    solver = SOLVERS[method](func=func, y0=y0, rtol=rtol, atol=atol, **options)
    if event_fn is None:
        solution = solver.integrate(t)
    else:
        event_t, solution = solver.integrate_until_event(t[0], event_fn)
        event_t = event_t.to(t)
        if t_is_reversed:
            event_t = -event_t
    if shapes is not None:
        solution = _flat_to_shape(solution, (len(t),), shapes)
    return solution if event_fn is None else (event_t, solution)


class _Adjoint(torch.autograd.Function):
    @staticmethod
    def forward(ctx, func, t, rtol, atol, method, options, adjoint_options, y0, *params):
        with torch.no_grad():
            y = odeint(func, y0, t, rtol=rtol, atol=atol, method=method, options=options)
        ctx.func, ctx.solve_kw = func, dict(rtol=rtol, atol=atol, method=method, options=adjoint_options)
        ctx.save_for_backward(t, y, *params)
        return y

    @staticmethod
    def backward(ctx, grad_y):
        func = ctx.func
        t, y, *params = ctx.saved_tensors

        def augmented(t_, state):
            # d/dt (t, y, adj_y, adj_params) = (-adj_y . df/dt, f, -adj_y . df/dy, -adj_y . df/dparams)
            with torch.enable_grad():
                tg, yg = t_.detach().requires_grad_(True), state[1].detach().requires_grad_(True)
                f = func(tg, yg)
                vjps = torch.autograd.grad(f, (tg, yg, *params), -state[2], allow_unused=True)
            vjps = [torch.zeros_like(x) if v is None else v for x, v in zip((tg, yg, *params), vjps)]
            return (vjps[0], f.detach(), *vjps[1:])

        with torch.no_grad():
            state = [torch.zeros((), dtype=y.dtype, device=y.device), y[-1], grad_y[-1]] + [torch.zeros_like(p) for p in params]
            for i in range(len(t) - 1, 0, -1):
                sol = odeint(augmented, tuple(state), t[i - 1:i + 1].flip(0), **ctx.solve_kw)
                state = [s[1] for s in sol]
                state[1] = y[i - 1]                    # restart from the forward solution, not the backward estimate
                state[2] = state[2] + grad_y[i - 1]
        return (None,) * 7 + (state[2], *state[3:])


def odeint_adjoint(func, y0, t, *, rtol=1e-7, atol=1e-9, method=None, options=None, adjoint_options=None):
    """Gradients w.r.t. y0 and func.parameters() by solving the adjoint system backwards through SOLVERS[method],
    with adjoint tolerances and method equal to the forward ones.  adjoint_options={'norm': 'seminorm'} leaves the
    parameter adjoints out of the error norm; otherwise the norm takes the max of the RMS norms of all parts."""
    params = tuple(p for p in func.parameters() if p.requires_grad)
    adjoint_options = {} if adjoint_options is None else dict(adjoint_options)
    seminorm = adjoint_options.pop("norm", None) == "seminorm"
    state_norm = (options or {}).get("norm", _rms_norm)

    def adjoint_norm(state):
        t_, y_, adj_y = state[:3]
        parts = [t_.abs(), state_norm(y_), state_norm(adj_y)]
        return max(parts if seminorm else parts + [_mixed_norm(state[3:])])
    adjoint_options["norm"] = adjoint_norm
    return _Adjoint.apply(func, t, rtol, atol, method, options, adjoint_options, y0, *params)
