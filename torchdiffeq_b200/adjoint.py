"""odeint_adjoint -- the reference's adjoint sensitivity entry point
(torchdiffeq/_impl/adjoint.py:8-223) on the B200 path.

Forward: the same device-resident solve as odeint, under no_grad (adjoint.py:23-24).
Backward: for every output interval, right to left, the augmented system
    d/dt (vjp_t, y, adj_y, adj_theta) = (-a.df/dt, f, -a.df/dy, -a.df/dtheta)      (adjoint.py:72-105)
is integrated backwards in time by the same adaptive engine on ONE flat, 16-byte aligned vector

    [ vjp_t | y | adj_y | theta_1 | theta_2 | ... ]

Unpacking is views; packing the pieces func/autograd return (the reference's torch.cat, misc.py:145),
the minus of `-adj_y` (adjoint.py:96) and the *(-1) of reverse time (misc.py:165) are one
tdq_pack_segments launch per evaluation.  The default adjoint norm
max(|t|, rms(y), rms(adj_y), max_i rms(theta_i)) (adjoint.py:247-250) and 'seminorm' (:267-271) are
segments of the fused error-norm kernel.  One engine (and one captured graph) serves all intervals.
"""
import warnings

import torch
import torch.nn as nn

from . import _lib
from ._engine import Layout, on_solver_stream
from ._fixed import FixedGridEngine
from .odeint import (ADAPTIVE_METHODS, FIXED_METHODS, _ADJOINT_CALLBACK_NAMES, _CALLBACK_NAMES, _cache_drop, _cache_get,
                     _cache_key, _cache_put, _make_adaptive_engine, _mixed_norm, _rms_norm, _solve, _solve_event, _unflatten,
                     fixed_grid, normalise, Problem)


def find_parameters(module):
    """adjoint.py:226-240."""
    assert isinstance(module, nn.Module)
    if getattr(module, '_is_replica', False):
        def find_tensor_attributes(module):
            return [(k, v) for k, v in module.__dict__.items() if torch.is_tensor(v) and v.requires_grad]
        gen = module._named_members(get_members_fn=find_tensor_attributes)
        return [param for _, param in gen]
    return list(module.parameters())


class _BackwardSolver:
    """The backward half of adjoint.py:36-153: augmented layout, dynamics, norm and one adaptive engine
    shared by every output interval.  Built (and, in graph mode, captured) during the forward call."""

    def __init__(self, p, adjoint_params, adjoint_rtol, adjoint_atol, adjoint_method, adjoint_options,
                 t_requires_grad):
        self.p = p
        self.params = adjoint_params = tuple(adjoint_params)
        self.t_requires_grad = t_requires_grad
        dev, T, n = p.device, p.dtype, p.n
        # ---- augmented layout: [vjp_t | y | adj_y | params...]   (adjoint.py:64-65) ----------
        self.lay = lay = Layout([(1,), (n,), (n,)] + [q.shape for q in adjoint_params], T)
        self.o_t, self.o_y, self.o_a = o_t, o_y, o_a = lay.offsets[0], lay.offsets[1], lay.offsets[2]
        base_fn, fwd_layout = p.fn, p.layout
        self.base_fn, self.fwd_layout = base_fn, fwd_layout

        # ---- augmented dynamics (adjoint.py:72-105), returning RAW pieces ------------------
        def aug_fn(t_, aug_flat):
            y_ = aug_flat[o_y:o_y + n]
            adj = aug_flat[o_a:o_a + n]
            with torch.enable_grad():
                tt = t_.detach()
                if t_requires_grad:
                    tt = tt.clone().requires_grad_(True)
                yy = y_.detach().requires_grad_(True)
                f = base_fn(tt, yy)                                  # Tensor, or tuple of pieces (tuple state)
                if isinstance(f, tuple):
                    outs = [f_.reshape(-1) for f_ in f]
                    gouts = [adj[o:o + l] for o, l in zip(fwd_layout.offsets, fwd_layout.lens)]
                else:
                    outs = [f.reshape(-1)]
                    gouts = [adj]
                keep = [(o_, g_) for o_, g_ in zip(outs, gouts) if o_.requires_grad]
                inputs = ((tt,) if t_requires_grad else ()) + (yy,) + adjoint_params
                if keep:
                    grads = torch.autograd.grad([o_ for o_, _ in keep], inputs, [g_ for _, g_ in keep],
                                                allow_unused=True)   # +adj: the minus sits in the pack scale
                else:
                    grads = (None,) * len(inputs)
            if t_requires_grad:
                vjp_t, vjp_y, *vjp_params = grads
            else:
                vjp_t = None
                vjp_y, *vjp_params = grads
            if isinstance(f, tuple):
                return (vjp_t, *[f_.detach() for f_ in f], vjp_y, *vjp_params)
            return (vjp_t, f.detach(), vjp_y, *vjp_params)

        # Pieces and their scales.  Reference: k_ref = mul * (vjp_t, f, vjp_y, vjp_p) with
        # vjp = grad(f, ., -adj); the backward solve runs against the forward time direction, so after
        # misc.py:273-279 either mul = -1 (forward ascending) or mul = +1 with the roles of the signs
        # swapped -- in both cases the RAW slot (before the engine's t_sign) must hold
        # (-g_t, +f, -g_y, -g_p) with g = grad(f, ., +adj).
        if p.is_tuple:
            f_offs = [o_y + o for o in fwd_layout.offsets]
            f_lens = list(fwd_layout.lens)
        else:
            f_offs, f_lens = [o_y], [n]
        offs = [o_t] + f_offs + [o_a] + list(lay.offsets[3:])
        lens = [1] + f_lens + [n] + list(lay.lens[3:])
        scales = [-1.0] + [1.0] * len(f_offs) + [-1.0] + [-1.0] * len(adjoint_params)
        pieces = (offs, lens, scales)

        # ---- adjoint norm (adjoint.py:243-288) -------------------------------------------
        opts = dict(adjoint_options)
        y_segs = [(o_y + o, l) for o, l in zip(fwd_layout.offsets, fwd_layout.lens)] if p.is_tuple else [(o_y, n)]
        a_segs = [(o_a + o, l) for o, l in zip(fwd_layout.offsets, fwd_layout.lens)] if p.is_tuple else [(o_a, n)]
        p_segs = [(o, l) for o, l in zip(lay.offsets[3:], lay.lens[3:]) if l > 0]
        norm_fn, q_view, segs = None, None, None
        adj_norm = opts.pop("norm", None)

        def views_of(q):
            yq, aq = q[o_y:o_y + n], q[o_a:o_a + n]
            if p.is_tuple:
                yq, aq = fwd_layout.views(yq), fwd_layout.views(aq)
            else:
                yq, aq = yq.view(p.shape), aq.view(p.shape)
            return q[o_t:o_t + 1].view(()), yq, aq, [q[o:o + l].view(s) for o, l, s in
                                                     zip(lay.offsets[3:], lay.lens[3:], lay.shapes[3:])]
        self.views_of = views_of
        if adj_norm is None or adj_norm == "seminorm":
            segs = [(o_t, 1)] + y_segs + a_segs + ([] if adj_norm == "seminorm" else p_segs)
            if p.norm_fn is not None:          # any number of segments stays on the fused path (device chunk table)
                state_norm = p.norm_fn if p.norm_fn is not None else (_mixed_norm if p.is_tuple else _rms_norm)
                semi = adj_norm == "seminorm"

                def norm_fn(parts):                                  # adjoint.py:247-250 / :267-271
                    tq, yq, aq, pq = parts
                    vals = [tq.abs(), state_norm(yq), state_norm(aq)]
                    if not semi:
                        vals.append(_mixed_norm(pq))
                    return max(vals)
                q_view, segs = views_of, None
        else:
            # user callable: gets (t, y, adj_y, *adj_params), y/adj_y expanded for tuple states (:273-288)
            def norm_fn(parts):
                tq, yq, aq, pq = parts
                if p.is_tuple:
                    return adj_norm((tq, *yq, *aq, *pq))
                return adj_norm((tq, yq, aq, *pq))
            q_view = views_of

        # adjoint callbacks (adjoint.py:107-114)
        callbacks = {}
        for name, adj_name in zip(_CALLBACK_NAMES, _ADJOINT_CALLBACK_NAMES):
            cb = getattr(p.original_func, adj_name, None)
            if cb is not None:
                def _cb(t0, y_flat, dt, _cb_=cb):
                    tq, yq, aq, pq = views_of(y_flat)
                    state = (tq, *yq, *aq, *pq) if p.is_tuple else (tq, yq, aq, *pq)
                    return _cb_(t0 * self.bsign, state, dt)               # misc.py:330-331
                callbacks[name] = _cb

        # The backward solve always runs against the forward time direction (adjoint.py:136
        # t[i-1:i+1].flip(0)).  The engine integrates ascending s = bsign * t, bsign = -fwd_sign.
        fwd_sign = -1.0 if p.t_reversed else 1.0
        self.bsign = -fwd_sign
        bp = Problem()                       # the backward problem as the engine factory sees it
        bp.t_sign, bp.device, bp.dtype, bp.n, bp.fn = self.bsign, dev, T, lay.n, aug_fn
        bp.original_func = p.original_func          # decides graph='auto' (only nn.Module funcs are captured)
        bp.t_cpu = (p.t_cpu.to(torch.float64) * fwd_sign * self.bsign).flip(0)
        self.fixed = adjoint_method in FIXED_METHODS
        if self.fixed and opts.get("process_group") is not None:
            raise NotImplementedError("sharded adjoint with a fixed-grid adjoint_method is not implemented")
        if self.fixed:
            # fixed-grid backward (adjoint.py:134-138 with a FixedGridODESolver): the same step kernels; the grid of
            # every interval comes from adjoint_options (step_size / grid_constructor), solvers.py:85-104
            self.fixed_opts = {k: v for k, v in opts.items() if k not in ("graph", "run_ahead", "cache", "exchange",
                                                                           "process_group")}
            self.aug_fn = aug_fn
            valid = {k: v for k, v in callbacks.items() if k == "callback_step"}
            if set(callbacks) - set(valid):
                warnings.warn("Solver '{}' does not support callbacks {}".format(adjoint_method, set(callbacks) - set(valid)))
            # never capture inside autograd's backward (see AdaptiveEngine.prime): eager launches
            self.eng = FixedGridEngine(aug_fn, lay.n, T, dev, method=adjoint_method, t_sign=self.bsign,
                                       perturb=opts.get("perturb", False), graph=False, callbacks=valid, pieces=pieces)
            return
        # ---- batch-sharded backward solve (SURVEY.md section 8(e)) -------------------------------------------------
        # y and adj_y are this rank's rows; vjp_t and the parameter gradients every evaluation produces are PARTIAL
        # sums over the local rows.  They are all-reduced right after the pack (two contiguous ranges of the slot:
        # vjp_t at the front, the parameter block at the tail), so every rank integrates the same GLOBAL adj_theta --
        # which is what the default adjoint norm needs (rms of each global gradient tensor, adjoint.py:250), and what
        # leaves the gradients complete on every rank at the end, with no extra reduction.
        replicated, post_fn = (), None
        pg = opts.get("process_group")
        if pg is not None:
            import torch.distributed as dist
            group = None if pg is True else pg
            if norm_fn is not None:
                raise NotImplementedError("sharded adjoint: custom norm callables are not supported (replicas only)")
            o_p = lay.offsets[3] if len(lay.offsets) > 3 else lay.n
            n_lay = lay.n

            def post_fn(buf):
                dist.all_reduce(buf[o_t:o_t + 1], group=group)
                if o_p < n_lay:
                    dist.all_reduce(buf[o_p:n_lay], group=group)
            n_state_segs = len(y_segs) + len(a_segs)
            replicated = (0,) + tuple(range(1 + n_state_segs, len(segs)))
        self.dist_group = None if pg is None else (None if pg is True else pg)
        self.sharded = pg is not None
        rtol_s, rtol_v = _adj_tol(adjoint_rtol, lay, dev)
        atol_s, atol_v = _adj_tol(adjoint_atol, lay, dev)
        if (rtol_v is None) != (atol_v is None):
            if rtol_v is None:
                rtol_v = torch.full_like(atol_v, rtol_s)
            else:
                atol_v = torch.full_like(rtol_v, atol_s)
        self.eng = _make_adaptive_engine(bp, adjoint_method, rtol_s, atol_s, rtol_v, atol_v, opts, fn=aug_fn,
                                         n=lay.n, segs=segs, pieces=pieces, norm_fn=norm_fn, q_view=q_view,
                                         callbacks=callbacks, solver_name=adjoint_method, replicated=replicated,
                                         post_fn=post_fn)
        # solves run inside autograd's backward: never capture there (see AdaptiveEngine.prime)
        self.eng.capture_in_solve = False

    def prime(self, t, y_last):
        """Capture the backward step graph now (forward call, main thread) on stand-in data."""
        if self.fixed:
            return False
        lay, n = self.lay, self.p.n
        aug = torch.zeros(lay.n, dtype=self.p.dtype, device=self.p.device)
        aug[self.o_y:self.o_y + n] = y_last
        s_cpu = t.detach().to("cpu", torch.float64) * self.bsign         # engine time of the backward solve
        pair = torch.stack([s_cpu[-1], s_cpu[-2]]).to(self.p.device)
        return self.eng.prime(aug, pair, t_start=float(s_cpu[-1]))

    def run(self, t, y, grad_sol):
        """adjoint.py:116-153."""
        p, lay, eng, n = self.p, self.lay, self.eng, self.p.n
        o_t, o_y, o_a = self.o_t, self.o_y, self.o_a
        dev, T = p.device, p.dtype
        aug = torch.zeros(lay.n, dtype=T, device=dev)
        aug[o_y:o_y + n] = y[-1]
        aug[o_a:o_a + n] = grad_sol[-1]
        # interval end points in the engine's ascending time, on the host (start times, no per-interval sync) and
        # on the device (row i-1 = the output times of interval i)
        s_cpu = t.detach().to("cpu", torch.float64) * self.bsign
        s_dev = s_cpu.to(dev)
        pairs = torch.stack([s_dev[1:], s_dev[:-1]], dim=1).contiguous() if len(t) > 1 else None
        time_vjps = torch.empty(len(t), dtype=t.dtype, device=t.device) if self.t_requires_grad else None
        for i in range(len(t) - 1, 0, -1):                            # adjoint.py:124-141
            if self.t_requires_grad:
                fe = self.base_fn(t[i].to(T.to_real()), y[i])
                if isinstance(fe, tuple):
                    fe = self.fwd_layout.flatten([f_.detach() for f_ in fe])
                dLd_cur_t = fe.reshape(-1).dot(grad_sol[i].reshape(-1))
                if getattr(self, "sharded", False):                  # a sum over ALL rows of the batch
                    import torch.distributed as dist
                    dist.all_reduce(dLd_cur_t, group=self.dist_group)
                aug[o_t] -= dLd_cur_t
                time_vjps[i] = dLd_cur_t
            if self.fixed:
                pair = (t[i - 1:i + 1].detach().flip(0) * self.bsign).to("cpu")      # ascending engine time, t's own dtype
                opts = dict(self.fixed_opts)
                if "grid_constructor" in opts:                       # the user sees the true times (misc.py:283-289)
                    gc, sgn = opts["grid_constructor"], self.bsign
                    opts["grid_constructor"] = lambda f_, y_, t_: sgn * gc(f_, y_, sgn * t_)
                grid = fixed_grid(eng.method, opts, self.aug_fn, aug, pair)
                sol = eng.solve(aug, grid, pair)
            else:
                sol = eng.solve(aug, pairs[i - 1], t_start=float(s_cpu[i]))   # ascending for the engine
            aug.copy_(sol[1])
            aug[o_y:o_y + n] = y[i - 1]                               # adjoint.py:140
            aug[o_a:o_a + n] += grad_sol[i - 1]                       # adjoint.py:141
        if self.t_requires_grad:
            time_vjps[0] = aug[o_t]
        adj_y = aug[o_a:o_a + n].clone()
        adj_params = [aug[o:o + l].view(s).clone() for o, l, s in zip(lay.offsets[3:], lay.lens[3:], lay.shapes[3:])]
        return time_vjps, adj_y, adj_params


def _backward_key(p, adjoint_params, bargs):
    adjoint_rtol, adjoint_atol, adjoint_method, adjoint_options, t_requires_grad = bargs
    fkey = _cache_key(p)
    if fkey is None:
        return None
    items = []
    for k, v in sorted(adjoint_options.items()):
        if isinstance(v, torch.Tensor) or callable(v):
            return None
        items.append((k, v))
    try:
        key = ("adjoint", fkey, tuple(q.data_ptr() for q in adjoint_params), float(adjoint_rtol), float(adjoint_atol),
               adjoint_method, tuple(items), t_requires_grad)
        hash(key)
    except (TypeError, ValueError):
        return None
    return key


class _AdjointFunction(torch.autograd.Function):
    """adjoint.py:8-153 OdeintAdjointMethod."""

    @staticmethod
    def forward(ctx, p, adjoint_rtol, adjoint_atol, adjoint_method, adjoint_options, t_requires_grad, t, y0_flat,
                *adjoint_params):
        ctx.p = p
        ctx.bargs = (adjoint_rtol, adjoint_atol, adjoint_method, adjoint_options, t_requires_grad)
        ctx.bsolver, ctx.bkey = None, None
        ctx.event_mode = p.event_fn is not None                          # adjoint.py:21
        with torch.no_grad():
            if ctx.event_mode:                                           # adjoint.py:30-31
                ev, sol, _ = _solve_event(p)
                event_t = torch.tensor(ev, dtype=t.dtype, device=t.device)
                ctx.save_for_backward(t, sol, event_t, *adjoint_params)
                return event_t, sol
            sol, _ = _solve(p)                                          # adjoint.py:23-24
            graph_opt = adjoint_options.get("graph", "auto")
            if any(ctx.needs_input_grad) and len(t) > 1 and graph_opt in (True, "auto") \
                    and int(adjoint_options.get("run_ahead", 2)) > 0:
                try:
                    bkey = ctx.bkey = _backward_key(p, adjoint_params, ctx.bargs)
                    hit = _cache_get(bkey, "backward")
                    if hit is not None:
                        bs = hit[0]
                    else:
                        bs = _BackwardSolver(p, adjoint_params, *ctx.bargs)
                        bs.prime(t, sol[-1])
                        _cache_put(bkey, (bs, p.original_func), "backward")
                    ctx.bsolver = bs
                except Exception as e:
                    if graph_opt is True:
                        raise
                    warnings.warn("torchdiffeq_b200: could not prepare the captured backward step (%s: %s); the "
                                  "backward pass will use eager launches" % (type(e).__name__, e))
        ctx.save_for_backward(t, sol, *adjoint_params)                   # adjoint.py:28
        return sol

    @staticmethod
    def backward(ctx, *grads):
        p = ctx.p
        if ctx.event_mode:
            # backprop as if integrating up to the event time; not through the event time itself (adjoint.py:46-53)
            t_all, y, event_t, *adjoint_params = ctx.saved_tensors
            t = torch.cat([t_all[0].reshape(-1), event_t.reshape(-1).to(t_all)])
            grad_sol = grads[1]
        else:
            t, y, *adjoint_params = ctx.saved_tensors
            grad_sol = grads[0]
        grad_sol = grad_sol.contiguous()
        with torch.no_grad():
            bs = ctx.bsolver
            if bs is None:
                bs = _BackwardSolver(p, adjoint_params, *ctx.bargs)
            try:
                time_vjps, adj_y, adj_params = bs.run(t, y, grad_sol)
            except BaseException:
                _cache_drop(ctx.bkey, "backward")         # a half-finished backward engine is never reused
                raise
            if ctx.event_mode and time_vjps is not None:                 # adjoint.py:146-148
                time_vjps = torch.cat([time_vjps[0].reshape(-1), torch.zeros_like(t_all[1:])])
        ctx.bsolver = None
        return (None, None, None, None, None, None, time_vjps, adj_y, *adj_params)


def _adj_tol(tol, lay, device):
    if isinstance(tol, torch.Tensor) and tol.ndim == 0:
        return float(tol), None
    try:
        iter(tol)
    except TypeError:
        return float(tol), None
    tol = tuple(tol)
    assert len(tol) == len(lay.shapes), "If using tupled adjoint tolerances they must match (t, y, adj_y, *params)"
    vec = torch.ones(lay.n, dtype=torch.float64, device=device)
    for tol_, o, l in zip(tol, lay.offsets, lay.lens):
        vec[o:o + l] = float(torch.as_tensor(tol_).to(torch.float32)) if not torch.is_tensor(tol_) or tol_.ndim == 0 \
            else torch.as_tensor(tol_).to(device).reshape(-1).to(torch.float64)
    return None, vec


def odeint_adjoint(func, y0, t, *, rtol=1e-7, atol=1e-9, method=None, options=None, event_fn=None,
                   adjoint_rtol=None, adjoint_atol=None, adjoint_method=None, adjoint_options=None,
                   adjoint_params=None):
    """adjoint.py:156-223, same signature and defaults."""
    if adjoint_params is None and not isinstance(func, nn.Module):                     # adjoint.py:161-164
        raise ValueError('func must be an instance of nn.Module to specify the adjoint parameters; alternatively they '
                         'can be specified explicitly via the `adjoint_params` argument. If there are no parameters '
                         'then it is allowable to set `adjoint_params=()`.')
    if adjoint_rtol is None:                                                           # adjoint.py:167-172
        adjoint_rtol = rtol
    if adjoint_atol is None:
        adjoint_atol = atol
    if adjoint_method is None:
        adjoint_method = method
    if adjoint_method != method and options is not None and adjoint_options is None:   # adjoint.py:174-176
        raise ValueError("If `adjoint_method != method` then we cannot infer `adjoint_options` from `options`. So as "
                         "`options` has been passed then `adjoint_options` must be passed as well.")
    if adjoint_options is None:                                                        # adjoint.py:178-182
        adjoint_options = {k: v for k, v in options.items() if k != "norm"} if options is not None else {}
    else:
        adjoint_options = adjoint_options.copy()
    if adjoint_params is None:                                                         # adjoint.py:184-187
        adjoint_params = tuple(find_parameters(func))
    else:
        adjoint_params = tuple(adjoint_params)
    oldlen_ = len(adjoint_params)                                                      # adjoint.py:190-197
    adjoint_params = tuple(q for q in adjoint_params if q.requires_grad)
    if len(adjoint_params) != oldlen_:
        if 'norm' in adjoint_options and callable(adjoint_options['norm']):
            warnings.warn("An adjoint parameter was passed without requiring gradient. For efficiency this will be "
                          "excluded from the adjoint pass, and will not appear as a tensor in the adjoint norm.")

    p = normalise(func, y0, t, rtol, atol, method, options, event_fn)
    if p.dtype.is_complex and not all(q.is_complex() for q in adjoint_params):
        # the augmented state [vjp_t | y | adj_y | theta...] is one complex vector, so a real parameter would receive a
        # complex gradient (the reference fails inside autograd here)
        raise TypeError("odeint_adjoint with a complex state needs complex adjoint parameters; got real ones: %s"
                        % [tuple(q.shape) for q in adjoint_params if not q.is_complex()])
    if adjoint_method is None:
        adjoint_method = 'dopri5'
    if adjoint_method not in ADAPTIVE_METHODS + FIXED_METHODS:
        raise NotImplementedError('adjoint_method "{}" is not implemented on the B200 path; implemented: {}'
                                  .format(adjoint_method, ADAPTIVE_METHODS + FIXED_METHODS))
    if p.is_tuple:
        y0_flat = p.layout.flatten(list(y0))          # differentiable wrt every piece (copy_ into zeros)
    else:
        y0_flat = y0.reshape(-1)
    # The autograd node is created on the solver stream, so that its backward -- and every gradient edge
    # into the parameters -- lives on the stream the backward step graph is captured and replayed on.
    with on_solver_stream(p.device) as ss:
        ans = _AdjointFunction.apply(p, adjoint_rtol, adjoint_atol, adjoint_method, adjoint_options, t.requires_grad,
                                     t, y0_flat, *adjoint_params)
        if p.event_fn is not None:                                                     # adjoint.py:209-223
            event_t, sol = ans
            ss.publish(sol, event_t)
            return event_t, _unflatten(p, sol)
        sol = ans
        ss.publish(sol)
    return _unflatten(p, sol)
