"""odeint -- the reference's public entry point (torchdiffeq/_impl/odeint.py:49-108) on the B200 path.

Same signature, argument meaning, output layout and error behaviour; the work between input
normalisation and the returned tensor runs as libtdq kernels.  Input normalisation restates
misc.py:200-345 (_check_inputs) with two differences that are not observable in results:
  * tuple states are laid out with 16-byte aligned pieces instead of back-to-back (misc.py:220);
  * reverse-time integration does not wrap func in a multiply-by-minus-one (misc.py:158-165):
    the sign is folded into the Runge-Kutta coefficients on the device.
"""
import collections
import warnings

import torch

from . import _lib
from ._engine import AdaptiveEngine, Layout, on_solver_stream
from ._fixed import FixedGridEngine, grid_from_step_size

ADAPTIVE_METHODS = ("dopri5", "dopri8", "tsit5", "bosh3", "fehlberg2", "adaptive_heun")
FIXED_METHODS = ("euler", "midpoint", "heun2", "heun3", "rk4")
ADAMS_METHODS = {"explicit_adams": False, "implicit_adams": True, "fixed_adams": True}     # name -> implicit (odeint.py:31-42)
# Every name the reference registers (odeint.py:19-46); the ones outside SURVEY.md section 8 are
# recognised and rejected explicitly rather than reported as "invalid".
REFERENCE_METHODS = (
    "dopri8", "dopri5", "tsit5", "bosh3", "fehlberg2", "adaptive_heun", "euler", "midpoint", "heun2", "heun3",
    "rk4", "explicit_adams", "implicit_adams", "implicit_euler", "implicit_midpoint", "trapezoid", "radauIIA3",
    "gl4", "radauIIA5", "gl6", "sdirk2", "trbdf2", "fixed_adams", "scipy_solver")

_CALLBACK_NAMES = ["callback_step", "callback_accept_step", "callback_reject_step"]   # misc.py:9
_ADJOINT_CALLBACK_NAMES = [name + "_adjoint" for name in _CALLBACK_NAMES]             # misc.py:10
_ADAPTIVE_OPTIONS = {"min_step", "max_step", "first_step", "step_t", "jump_t", "safety", "ifactor", "dfactor",
                     "max_num_steps", "dtype", "norm"}
_FIXED_OPTIONS = {"step_size", "grid_constructor", "interp", "perturb", "norm"}
_ADAMS_OPTIONS = _FIXED_OPTIONS | {"max_iters", "max_order"}
_OUR_OPTIONS = {"graph", "run_ahead", "process_group", "cache", "exchange", "device_loop", "fused_linear", "fused_attempt", "fused_controller"}


def _rms_norm(tensor):
    """misc.py:22-23; recognised by identity so the default norm stays fused."""
    return tensor.abs().pow(2).mean().sqrt()


def _mixed_norm(tensor_tuple):
    """misc.py:30-33."""
    if len(tensor_tuple) == 0:
        return 0.
    return max([_rms_norm(tensor) for tensor in tensor_tuple])


class Problem:
    """Normalised inputs of one solve (what misc.py:200-345 returns as a 10-tuple)."""
    pass


def _combine_event_functions(event_fn, t0, y0):
    """event_handling.py:23-35: make every component initially positive and take the minimum."""
    with torch.no_grad():
        initial_signs = torch.sign(event_fn(t0, y0))

    def combined_event_fn(t, y):
        c = event_fn(t, y)
        return torch.min(c * initial_signs)
    return combined_event_fn


def _check_timelike(name, timelike, can_grad, values=None):                            # misc.py:367-374
    """`values`: a host copy of the tensor, so that the monotonicity test costs no device synchronisation."""
    assert isinstance(timelike, torch.Tensor), '{} must be a torch.Tensor'.format(name)
    if not torch.is_floating_point(timelike):                                          # misc.py:110-112
        raise TypeError('`{}` must be a floating point Tensor but is a {}'.format(name, timelike.type()))
    assert timelike.ndimension() == 1, "{} must be one dimensional".format(name)
    if not can_grad:
        assert not timelike.requires_grad, "{} cannot require gradient".format(name)
    v = timelike if values is None else values
    diff = v[1:] > v[:-1]
    assert diff.all() or (~diff).all(), '{} must be strictly increasing or decreasing'.format(name)


def _tol_vector(name, tol, layout, shape, device):
    """Scalar tolerance -> (float, None).  Tuple of tolerances for a tuple state (misc.py:115-123
    _tuple_tol) or a tensor broadcastable to a tensor state -> (None, per-element float64 vector), the
    dtype the solver casts tolerances to (rk_common.py:186-187)."""
    if isinstance(tol, torch.Tensor):
        if tol.ndim == 0:
            return float(tol), None
        if layout is None:
            return None, tol.detach().to(device=device, dtype=torch.float64).expand(shape).reshape(-1).contiguous()
    else:
        try:
            iter(tol)
        except TypeError:
            return float(tol), None
    assert layout is not None, "tupled {} needs a tuple y0".format(name)
    tol = tuple(tol)
    assert len(tol) == len(layout.shapes), \
        "If using tupled {} it must have the same length as the tuple y0".format(name)
    vec = torch.ones(layout.n, dtype=torch.float64, device=device)   # padding: any finite non-zero value
    for tol_, o, l, shp in zip(tol, layout.offsets, layout.lens, layout.shapes):
        # torch.as_tensor(python float) is float32 in the reference before the float64 cast: keep that rounding
        v = torch.as_tensor(tol_).to(device)
        vec[o:o + l] = v.expand(shp).reshape(-1).to(torch.float64)
    return None, vec


def normalise(func, y0, t, rtol, atol, method, options, event_fn, adjoint=False):
    """Restatement of misc.py:200-345 for our engines."""
    if event_fn is not None:
        if len(t) != 2:                                                                # misc.py:203-204
            raise ValueError(f"We require len(t) == 2 when in event handling mode, but got len(t)={len(t)}.")
        event_fn = _combine_event_functions(event_fn, t[0], y0)                        # misc.py:207
    p = Problem()
    p.original_func = func
    p.is_tuple = not isinstance(y0, torch.Tensor)
    if p.is_tuple:
        assert isinstance(y0, tuple), 'y0 must be either a torch.Tensor or a tuple'   # misc.py:216
        p.dtype = y0[0].dtype
        if any(y_.dtype.is_complex for y_ in y0):
            # the reference's torch.cat promotes a tuple with a complex piece: every piece integrates (and comes back)
            # in the common complex dtype
            for y_ in y0[1:]:
                p.dtype = torch.promote_types(p.dtype, y_.dtype)
        p.layout = Layout([y_.shape for y_ in y0], p.dtype)
        p.device = y0[0].device
    else:
        p.layout = None
        p.device = y0.device
        p.dtype = y0.dtype
    if torch.complex32 in ([y_.dtype for y_ in y0] if p.is_tuple else [p.dtype]):
        raise _lib.TdqError("unsupported state dtype torch.complex32 (float32, float64, complex64 and complex128 are "
                            "implemented)")
    options = {} if options is None else options.copy()                               # misc.py:226-229
    if method is None:
        method = 'dopri5'
    if method not in REFERENCE_METHODS:                                               # misc.py:232-234
        raise ValueError('Invalid method "{}". Must be one of {}'.format(
            method, '{"' + '", "'.join(REFERENCE_METHODS) + '"}.'))
    if method not in ADAPTIVE_METHODS + FIXED_METHODS + tuple(ADAMS_METHODS):
        raise NotImplementedError('method "{}" is not part of the B200 hot path; implemented: {}'.format(
            method, ADAPTIVE_METHODS + FIXED_METHODS + tuple(ADAMS_METHODS)))
    p.method, p.options = method, options
    if p.dtype.is_complex and options.get("process_group") is not None:
        raise NotImplementedError("batch-sharded solves (options['process_group']) of a complex state are not "
                                  "implemented")
    if p.device.type != "cuda":
        raise _lib.TdqError("torchdiffeq_b200 runs on CUDA devices only (got %s); there is no CPU path" % p.device)
    _lib.load()                                   # fail loudly, before any work, if libtdq.so is missing

    t_cpu = t.detach().to("cpu") if isinstance(t, torch.Tensor) else t                 # the one host read of t
    _check_timelike('t', t, True, values=t_cpu)
    p.t_reversed = bool(len(t_cpu) > 1 and t_cpu[0] > t_cpu[1])                        # misc.py:270-271
    p.t_sign = -1.0 if p.t_reversed else 1.0
    p.t_cpu = -t_cpu if p.t_reversed else t_cpu                                        # ascending from here on
    if p.t_reversed:
        for name in ("step_t", "jump_t"):                                              # misc.py:292-293
            if isinstance(options.get(name), torch.Tensor):
                options[name] = -options[name]
        if "grid_constructor" in options:                                             # misc.py:283-289
            _gc = options["grid_constructor"]
            options["grid_constructor"] = lambda func, y0, t: -_gc(func, y0, -t)
    assert (p.t_cpu[1:] > p.t_cpu[:-1]).all(), 't must be strictly increasing or decreasing'   # misc.py:296

    if torch.is_tensor(rtol):                                                          # misc.py:299-302
        assert not rtol.requires_grad, "rtol cannot require gradient"
    if torch.is_tensor(atol):
        assert not atol.requires_grad, "atol cannot require gradient"
    if t.device != p.device:                                                           # misc.py:305-307
        warnings.warn("t is not on the same device as y0. Coercing to y0.device.")

    shape_ = None if p.is_tuple else y0.shape
    p.rtol, p.rtol_vec = _tol_vector('rtol', rtol, p.layout, shape_, p.device)
    p.atol, p.atol_vec = _tol_vector('atol', atol, p.layout, shape_, p.device)
    if (p.rtol_vec is None) != (p.atol_vec is None):                                   # mixed scalar/vector
        if p.rtol_vec is None:
            p.rtol_vec = torch.full_like(p.atol_vec, p.rtol)
        else:
            p.atol_vec = torch.full_like(p.rtol_vec, p.atol)

    # callbacks (misc.py:313-343)
    p.callbacks = {}
    for name in _CALLBACK_NAMES:
        cb = getattr(func, name, None)
        if cb is not None:
            p.callbacks[name] = cb
    valid = set(_CALLBACK_NAMES) if method in ADAPTIVE_METHODS else {"callback_step"}     # solvers.py:81-83
    invalid = set(p.callbacks) - valid
    if invalid:
        warnings.warn("Solver '{}' does not support callbacks {}".format(method, invalid))
        for name in invalid:
            del p.callbacks[name]
    if p.callbacks:
        layout, sign = p.layout, p.t_sign
        def _wrap(cb):
            def _cb(t0, y0_flat, dt):
                y_ = layout.views(y0_flat) if layout is not None else y0_flat.view(p.shape)
                return cb(t0 * sign, y_, dt)                                           # misc.py:326-331
            return _cb
        p.callbacks = {k: _wrap(v) for k, v in p.callbacks.items()}

    # flat state + flat func
    if p.is_tuple:
        p.shape = None
        p.y0_flat = p.layout.flatten([y_.detach() for y_ in y0])
        p.n = p.layout.n
        layout = p.layout
        def fn(t_, y_flat):
            f = func(t_, layout.views(y_flat))                                         # misc.py:143-145
            return tuple(f)
        p.fn = fn
        p.pieces = (list(layout.offsets), list(layout.lens), [1.0] * len(layout.lens))
        p.segs = list(zip(layout.offsets, layout.lens))                                # misc.py:247 _mixed_norm
    else:
        p.shape = y0.shape
        p.y0_flat = y0.detach().reshape(-1)
        p.n = p.y0_flat.numel()
        shape = p.shape
        p.fn = lambda t_, y_flat: func(t_, y_flat.view(shape))
        p.pieces = None
        p.segs = None

    # event function on the flat state, in the solver's ascending time (misc.py:224-225, :281-282)
    p.event_fn = None
    if event_fn is not None:
        unflat = (lambda yf: p.layout.views(yf)) if p.is_tuple else (lambda yf: yf.view(p.shape))
        sign_ = p.t_sign
        p.event_fn = lambda t_, y_flat: event_fn(t_ * sign_, unflat(y_flat))

    # norm (misc.py:237-266): the defaults stay fused; a user callable takes the compatibility path
    p.norm_fn = None
    p.q_view = None
    user_norm = options.get("norm", None)
    if user_norm is not None and user_norm is not _rms_norm and not (p.is_tuple and user_norm is _mixed_norm):
        p.norm_fn = user_norm
        if p.is_tuple:
            p.q_view = lambda q: layout.views(q)
        else:
            p.q_view = lambda q: q.view(shape)
    return p


def _warn_unused(solver_name, options, known):                                        # misc.py:13-15
    unused = {k: v for k, v in options.items() if k not in known and k not in _OUR_OPTIONS}
    if unused:
        warnings.warn('{}: Unexpected arguments {}'.format(solver_name, unused))


def _resolve_graph(graph, func):
    """'auto' captures the step body only for nn.Module funcs.  Capturing runs func's Python ONCE and replays its
    kernels afterwards, which silently freezes Python side effects (NFE counters, schedules, Python RNG) and
    data-dependent branches; for a Module that is the documented contract (README "Graph mode"), for an arbitrary
    callable it is not assumed -- pass options={'graph': True} to opt in."""
    if graph == "auto" and not isinstance(func, torch.nn.Module):
        return False
    return graph


def _make_adaptive_engine(p, method, rtol, atol, rtol_vec, atol_vec, options, fn=None, n=None, segs=None,
                          pieces=None, norm_fn=None, q_view=None, callbacks=None, solver_name=None,
                          keep_interp=False, replicated=(), post_fn=None):
    o = options
    _warn_unused(solver_name or method, o, _ADAPTIVE_OPTIONS)
    graph = _resolve_graph(o.get("graph", "auto"), getattr(p, "original_func", None))
    if o.get("dtype", torch.float64) != torch.float64:
        raise NotImplementedError("time dtype other than float64 (options['dtype']) is not implemented")
    def _tvals(v):                                                                     # rk_common.py:372-375
        v = torch.as_tensor(v, dtype=torch.float64).to("cpu")
        return torch.sort(v[v >= p.t_cpu[0].double()]).values
    step_t, jump_t = o.get("step_t"), o.get("jump_t")
    st = _tvals(step_t) if step_t is not None else torch.tensor([], dtype=torch.float64)
    jt = _tvals(jump_t) if jump_t is not None else torch.tensor([], dtype=torch.float64)
    if (torch.cat([st, jt]).unique(return_counts=True)[1] > 1).any():                  # :233-236
        raise ValueError("`step_t` and `jump_t` must not have any repeated elements between them.")
    step_t = st.to(p.device) if step_t is not None else None
    jump_t = jt.to(p.device) if jump_t is not None else None
    reduce_fn, n_global, seg_counts_global, agree_fn, exchange = None, None, None, None, None
    pg = o.get("process_group")
    if pg is not None:
        from .dist import make_agree, make_reduce
        if norm_fn is not None:
            raise NotImplementedError("a custom norm callable cannot be evaluated on a batch-sharded state "
                                      "(SURVEY.md section 8(e): replicas only); use the default norm or 'seminorm'")
        reduce_fn, n_global, seg_counts_global = make_reduce(pg, segs if segs is not None else
                                                             [(0, n if n is not None else p.n)], p.device,
                                                             replicated=replicated)
        agree_fn = make_agree(pg)
        if o.get("exchange", "peer") == "peer" and norm_fn is None:
            try:
                from .dist import PeerExchange
                n_seg_ = len(segs) if segs is not None else 1
                if n_seg_ > _lib.TDQ_MAX_SEGS:
                    raise _lib.TdqError("more than %d norm segments" % _lib.TDQ_MAX_SEGS)
                exchange = PeerExchange(pg, p.device)
            except Exception as e:      # e.g. CUDA IPC not permitted in this container: keep the NCCL all-reduce
                warnings.warn("torchdiffeq_b200: NVLink peer exchange unavailable (%s: %s); using the process "
                              "group's all-reduce" % (type(e).__name__, e))
    eng = AdaptiveEngine(
        fn if fn is not None else p.fn, n if n is not None else p.n, p.dtype, p.device, method,
        rtol=rtol, atol=atol, rtol_vec=rtol_vec, atol_vec=atol_vec,
        segs=segs, t_sign=p.t_sign, pieces=pieces,
        min_step=o.get("min_step", 0), max_step=o.get("max_step", float("inf")),
        first_step=o.get("first_step"), step_t=step_t, jump_t=jump_t,
        safety=o.get("safety", 0.9), ifactor=o.get("ifactor", 10.0), dfactor=o.get("dfactor", 0.2),
        max_num_steps=o.get("max_num_steps", 2 ** 31 - 1),
        norm_fn=norm_fn, q_view=q_view, graph=graph, run_ahead=o.get("run_ahead", 2),
        reduce_fn=reduce_fn, n_global=n_global, seg_counts_global=seg_counts_global, agree_fn=agree_fn,
        exchange=exchange, callbacks=callbacks, keep_interp=keep_interp, device_loop=o.get("device_loop", "auto"),
        post_fn=post_fn)
    if fn is None and not p.is_tuple and o.get("fused_linear", True):
        # func is a torchdiffeq_b200.LinearField on a float32 [..., 128] state: stages run as one tcgen05 kernel each
        from .fields import fusable
        w = fusable(getattr(p, "original_func", None), tuple(p.shape), p.dtype, p.device, eng.lib)
        if w is not None:
            eng.set_linear(w, whole_attempt=o.get("fused_attempt", True), fused_controller=o.get("fused_controller", True))
    return eng


# ---- engine cache -------------------------------------------------------------------------------
# An engine owns ~10 state-sized buffers and, in graph mode, a captured step graph with its private
# memory pool; building and tearing that down costs far more than a solve of the benchmark size.
# Engines are therefore kept (LRU) and reused when the same func is integrated again with the same
# shapes and options -- the normal situation in a training or serving loop.
#
# A captured graph bakes in everything func did while it was captured, so reuse is restricted to what can be
# keyed reliably (ADVICE r1): func must be an nn.Module, and the key holds the module object, every
# parameter / buffer / tensor attribute (address, shape, dtype, requires_grad; also inside list / tuple / dict
# attributes), every plain Python attribute (int, float, bool, str, None) and the `training` flag of every
# submodule.  Plain functions, closures, partials and bound methods are NOT cached (their globals, defaults and
# cells cannot be enumerated safely): they get a fresh engine per call unless the caller passes
# options={'cache': True} and thereby promises that func is a pure function of (t, y) between calls.
# Anything unhashable (tensor options, callbacks, vector tolerances, custom norms) disables caching;
# options={'cache': False} opts out; torchdiffeq_b200.clear_cache() drops the engines and their memory.
# What no key can see -- data-dependent Python branches inside forward(), state mutated in place through
# channels other than attributes -- is the caller's contract (README "Graph mode").
_ENGINE_CACHE = collections.OrderedDict()          # forward engines
_BACKWARD_CACHE = collections.OrderedDict()        # adjoint backward solvers (their own LRU: no thrashing)
_CACHE_MAX = {"forward": 4, "backward": 4}


def clear_cache():
    _ENGINE_CACHE.clear()
    _BACKWARD_CACHE.clear()


def set_cache_size(forward=4, backward=4):
    """Number of engines kept per cache (each holds ~10 state-sized buffers plus its graph's memory pool)."""
    _CACHE_MAX["forward"], _CACHE_MAX["backward"] = int(forward), int(backward)
    for which, c in (("forward", _ENGINE_CACHE), ("backward", _BACKWARD_CACHE)):
        while len(c) > _CACHE_MAX[which]:
            c.popitem(last=False)


def _tensor_sig(x):
    return (x.data_ptr(), tuple(x.shape), x.dtype, x.requires_grad)


_PLAIN = (int, float, bool, str, type(None), complex)


def _attr_sig(name, v):
    """Key contribution of one attribute of a module (None: nothing to add)."""
    if isinstance(v, torch.Tensor):
        return (name,) + _tensor_sig(v)
    if isinstance(v, _PLAIN):
        return (name, v)
    if isinstance(v, (list, tuple)):
        items = tuple(_attr_sig(i, x) for i, x in enumerate(v) if isinstance(x, (torch.Tensor,) + _PLAIN))
        return (name, type(v).__name__, len(v), items)
    if isinstance(v, dict):
        items = tuple(_attr_sig(str(k), x) for k, x in v.items() if isinstance(x, (torch.Tensor,) + _PLAIN))
        return (name, "dict", len(v), items)
    return None


_SKIP_ATTRS = {"_parameters", "_buffers", "_modules", "_non_persistent_buffers_set", "_backward_hooks",
               "_backward_pre_hooks", "_forward_hooks", "_forward_pre_hooks", "_forward_hooks_with_kwargs",
               "_forward_pre_hooks_with_kwargs", "_forward_hooks_always_called", "_state_dict_hooks",
               "_state_dict_pre_hooks", "_load_state_dict_pre_hooks", "_load_state_dict_post_hooks",
               "_is_full_backward_hook", "_compiled_call_impl", "training"}


def _func_signature(func, explicit=False):
    """Identity of everything a captured step graph bakes in about func, or None when it cannot be established
    (func is not an nn.Module and the caller did not opt in)."""
    if isinstance(func, torch.nn.Module):
        sig = [id(func)]
        for name, m in func.named_modules():
            sig.append((name, type(m).__name__, m.training))
            sig.extend((name,) + _tensor_sig(q) for q in m.parameters(recurse=False))
            sig.extend((name,) + _tensor_sig(b) for b in m.buffers(recurse=False))
            for k, v in vars(m).items():
                if k in _SKIP_ATTRS:
                    continue
                a = _attr_sig(k, v)
                if a is not None:
                    sig.append((name,) + a)
        return tuple(sig)
    if explicit:
        return (id(func),)
    return None


def _cache_key(p, extra=()):
    o = p.options
    if o.get("cache", True) is False or p.callbacks or p.norm_fn is not None or p.rtol_vec is not None:
        return None
    fsig = _func_signature(p.original_func, explicit=o.get("cache", None) is True)
    if fsig is None:
        return None
    items = []
    for k, v in sorted(o.items()):
        if k == "process_group":
            v = id(v)
        elif isinstance(v, torch.Tensor) or callable(v):
            return None
        items.append((k, v))
    shapes = tuple(tuple(s_) for s_ in p.layout.shapes) if p.is_tuple else tuple(p.shape)
    try:
        key = (fsig, p.method, p.dtype, str(p.device), p.is_tuple, shapes, p.rtol, p.atol,
               p.t_sign, tuple(items), torch.is_autocast_enabled(), extra)
        hash(key)
    except TypeError:
        return None
    return key


def _cache_get(key, which="forward"):
    c = _ENGINE_CACHE if which == "forward" else _BACKWARD_CACHE
    if key is None or key not in c:
        return None
    c.move_to_end(key)
    return c[key]


def _cache_put(key, value, which="forward"):
    if key is None:
        return
    c = _ENGINE_CACHE if which == "forward" else _BACKWARD_CACHE
    c[key] = value
    while len(c) > _CACHE_MAX[which]:
        c.popitem(last=False)


def _cache_drop(key, which="forward"):
    c = _ENGINE_CACHE if which == "forward" else _BACKWARD_CACHE
    if key is not None:
        c.pop(key, None)


# The last solve's counters: func runs once at capture and is replayed afterwards in graph mode, so Python-side
# NFE counters inside func do not advance; this is the supported way to read them (torchdiffeq_b200.last_stats()).
_LAST_STATS = {}


def last_stats():
    """{'nfe', 'n_accept', 'n_reject', 'attempts', 'launches'} of the most recent odeint call in this process."""
    return dict(_LAST_STATS)


def _solve(p):
    """Run the normalised problem; returns the flat solution [len(t), n] and the engine."""
    if p.method in ADAPTIVE_METHODS:
        key = _cache_key(p)
        hit = _cache_get(key)
        if hit is not None:
            eng = hit[0]
        else:
            eng = _make_adaptive_engine(p, p.method, p.rtol, p.atol, p.rtol_vec, p.atol_vec, p.options,
                                        segs=p.segs, pieces=p.pieces, norm_fn=p.norm_fn, q_view=p.q_view,
                                        callbacks=p.callbacks)
            _cache_put(key, (eng, p.original_func))     # the func reference keeps id(func) from being recycled
        t64 = p.t_cpu.to(torch.float64).to(p.device)                                   # solvers.py:31
        try:
            sol = eng.solve(p.y0_flat, t64, t_start=float(p.t_cpu[0]))
        except BaseException:
            _cache_drop(key)                            # a half-finished engine is never reused
            raise
        if key is not None:
            sol = sol.clone()                           # the engine reuses its solution buffer
        return sol, eng
    # fixed grid: euler / midpoint / heun2 / heun3 / rk4 (solvers.py:55-128, fixed_grid.py:6-60)
    o = p.options
    y0_view = p.layout.views(p.y0_flat) if p.is_tuple else p.y0_flat.view(p.shape)
    grid = fixed_grid(p.method, o, p.original_func, y0_view, p.t_cpu)
    eng = _fixed_engine(p)
    sol = eng.solve(p.y0_flat, grid, p.t_cpu)
    return sol, eng


def _cubic_or_linear(interp):
    if interp not in ("linear", "cubic"):                                              # solvers.py:125
        raise ValueError(f"Unknown interpolation method {interp}")
    return interp


def fixed_event_solve(eng, y0_flat, t0, step_size, event_fn, atol):
    """solvers.py:130-164 on a FixedGridEngine: (event_t, y(event_t))."""
    return eng.solve_until_event(y0_flat, t0, step_size, event_fn, atol)


_FIXED_NAMES = {"euler": "Euler", "midpoint": "Midpoint", "heun2": "Heun2", "heun3": "Heun3", "rk4": "RK4",
                "explicit_adams": "AdamsBashforth", "implicit_adams": "AdamsBashforthMoulton",
                "fixed_adams": "AdamsBashforthMoulton"}


def _fixed_engine(p, graph=None, interp=None):
    """The fixed-grid engine of a normalised problem: explicit RK step kernels, or the Adams multistep driver."""
    o = p.options
    interp = _cubic_or_linear(o.get("interp", "linear")) if interp is None else interp
    if p.method in ADAMS_METHODS:
        from ._adams import AdamsEngine
        if p.rtol is None or p.atol is None:
            raise NotImplementedError("per-element tolerances are not implemented for the Adams methods")
        return AdamsEngine(p.fn, p.n, p.dtype, p.device, implicit=ADAMS_METHODS[p.method], rtol=p.rtol, atol=p.atol,
                           max_iters=o.get("max_iters", 4), max_order=o.get("max_order", 12), t_sign=p.t_sign,
                           perturb=o.get("perturb", False), callbacks=p.callbacks, pieces=p.pieces, interp=interp)
    g = _resolve_graph(o.get("graph", "auto"), p.original_func) if graph is None else graph
    return FixedGridEngine(p.fn, p.n, p.dtype, p.device, method=p.method, t_sign=p.t_sign,
                           perturb=o.get("perturb", False), graph=g, callbacks=p.callbacks, pieces=p.pieces, interp=interp)


def fixed_grid(method, o, func, y0_view, t_cpu, keep_graph=False):
    """Option handling and time grid of FixedGridODESolver (solvers.py:55-79, :85-96, :103-104) for an
    ascending CPU `t_cpu`; the caller has already wrapped a user grid_constructor for reversed time."""
    _warn_unused(_FIXED_NAMES[method], o, _ADAMS_OPTIONS if method in ADAMS_METHODS else _FIXED_OPTIONS)
    step_size, gc = o.get("step_size"), o.get("grid_constructor")
    if step_size is None:
        grid_constructor = gc if gc is not None else (lambda f, y0, t: t)
    else:
        if gc is not None:
            raise ValueError("step_size and grid_constructor are mutually exclusive arguments.")   # solvers.py:79
        grid_constructor = grid_from_step_size(step_size)
    _cubic_or_linear(o.get("interp", "linear"))
    grid = grid_constructor(func, y0_view, t_cpu)
    grid = grid.to("cpu") if keep_graph else grid.detach().to("cpu")
    assert grid[0] == t_cpu[0] and grid[-1] == t_cpu[-1]                               # solvers.py:104
    return grid


def _solve_event(p):
    """odeint.py:97-100 + solvers.py:41-49: integrate until the event; returns (event_t tensor like t, [2, n])."""
    if p.method in FIXED_METHODS or p.method in ADAMS_METHODS:                         # solvers.py:130-164
        o = p.options
        _warn_unused(_FIXED_NAMES[p.method], o, _ADAMS_OPTIONS if p.method in ADAMS_METHODS else _FIXED_OPTIONS)
        if o.get("step_size") is None:
            raise AssertionError("Event handling for fixed step solvers currently requires `step_size` to be provided "
                                 "in options.")
        if o.get("grid_constructor") is not None:
            raise ValueError("step_size and grid_constructor are mutually exclusive arguments.")
        eng = _fixed_engine(p, graph=False)
        tol = p.atol if p.atol is not None else float(p.atol_vec.min())
        event_t, y_event = fixed_event_solve(eng, p.y0_flat, p.t_cpu[0], o["step_size"], p.event_fn, tol)
        sol = torch.stack([p.y0_flat.to(p.dtype), y_event], dim=0)
        return float(event_t) * p.t_sign, sol, eng
    eng = _make_adaptive_engine(p, p.method, p.rtol, p.atol, p.rtol_vec, p.atol_vec,
                                dict(p.options, run_ahead=0, graph=False), segs=p.segs, pieces=p.pieces,
                                norm_fn=p.norm_fn, q_view=p.q_view, callbacks=p.callbacks, keep_interp=True)
    tol = p.atol if p.atol is not None else float(p.atol_vec.min())
    event_t, y_event = eng.solve_until_event(p.y0_flat, float(p.t_cpu[0]), p.event_fn, tol)
    sol = torch.stack([p.y0_flat.to(p.dtype), y_event], dim=0)                         # solvers.py:48
    return event_t * p.t_sign, sol, eng                                                # odeint.py:99-100


def _unflatten(p, sol):
    if p.is_tuple:
        return p.layout.views(sol, (sol.shape[0],))                                    # odeint.py:102-103
    return sol.view(sol.shape[0], *p.shape)


class _ImplicitFnGradientRerouting(torch.autograd.Function):
    """odeint.py:197-231: gradient of the event time and of the state at the event through the implicit function
    theorem, event_fn(t*, y(t*)) = 0  =>  dt*/dy = -(dc/dy) / (dc/dt + dc/dy . f)."""

    @staticmethod
    def forward(ctx, func, event_fn, event_t, state_t):
        ctx.func, ctx.event_fn = func, event_fn
        ctx.save_for_backward(event_t, state_t)
        return event_t.detach(), state_t.detach()

    @staticmethod
    def backward(ctx, grad_t, grad_state):
        func, event_fn = ctx.func, ctx.event_fn
        event_t, state_t = ctx.saved_tensors
        event_t = event_t.detach().clone().requires_grad_(True)
        state_t = state_t.detach().clone().requires_grad_(True)
        f_val = func(event_t, state_t)
        with torch.enable_grad():
            c, (par_dt, dstate) = torch.autograd.functional.vjp(event_fn, (event_t, state_t))
        dcdt = par_dt + torch.sum(dstate * f_val)                  # total derivative of the event function along the flow
        grad_t = grad_t + torch.sum(grad_state * f_val)
        dstate = dstate * (-grad_t / (dcdt + 1e-12)).reshape_as(c)
        return None, None, None, grad_state + dstate


def odeint_event(func, y0, t0, *, event_fn, reverse_time=False, odeint_interface=None, **kwargs):
    """odeint.py:160-194: solve until event_fn crosses zero and link up the gradient of the event time.
    Pass odeint_interface=odeint_adjoint for gradients with respect to func's parameters and y0."""
    if odeint_interface is None:
        odeint_interface = odeint
    if reverse_time:
        t = torch.cat([t0.reshape(-1), t0.reshape(-1).detach() - 1.0])
    else:
        t = torch.cat([t0.reshape(-1), t0.reshape(-1).detach() + 1.0])
    event_t, solution = odeint_interface(func, y0, t, event_fn=event_fn, **kwargs)
    p = normalise(func, y0, t, 0.0, 0.0, kwargs.get("method"), None, event_fn)        # flat func / event_fn, :172
    sign_ = p.t_sign
    flat_func = lambda t_, y_flat: _as_flat(p, p.fn(t_ * sign_, y_flat)) * sign_       # ascending-time dynamics
    if p.is_tuple:
        state_t = p.layout.flatten([s_[-1] for s_ in solution])
    else:
        state_t = solution[-1].reshape(-1)
    if reverse_time:
        event_t = -event_t
    event_t, state_t = _ImplicitFnGradientRerouting.apply(flat_func, p.event_fn, event_t, state_t)
    if reverse_time:
        event_t = -event_t
    if p.is_tuple:
        pieces = p.layout.views(state_t)
        solution = tuple(torch.cat([s_[:-1], s_t[None]], dim=0) for s_, s_t in zip(solution, pieces))
    else:
        solution = torch.cat([solution[:-1], state_t.view(p.shape)[None]], dim=0)
    return event_t, solution


def _as_flat(p, f):
    if isinstance(f, tuple):
        return p.layout.flatten(list(f))
    return f.reshape(-1)


def odeint_dense(func, y0, t0, t1, *, rtol=1e-7, atol=1e-9, method=None, options=None):
    """odeint.py:111-157: solve from t0 to t1 with dopri5 and return a function that evaluates the solution at any
    time in between from the stored per-step interpolants (on the device, tdq_poly_eval)."""
    import bisect
    import ctypes as C
    from ._engine import _stream
    assert torch.is_tensor(y0)
    t0_, t1_ = torch.as_tensor(t0), torch.as_tensor(t1)
    t = torch.stack([t0_.reshape(()), t1_.reshape(()).to(t0_)]).to(t0_)
    p = normalise(func, y0, t, rtol, atol, method, options, None)
    assert p.method == "dopri5"                                                        # odeint.py:119
    with torch.no_grad(), on_solver_stream(p.device) as ss:
        eng = _make_adaptive_engine(p, p.method, p.rtol, p.atol, p.rtol_vec, p.atol_vec,
                                    dict(p.options, run_ahead=0, graph=False), segs=p.segs, pieces=p.pieces,
                                    norm_fn=p.norm_fn, q_view=p.q_view, callbacks=p.callbacks, keep_interp=True)
        t64 = p.t_cpu.to(torch.float64).to(p.device)
        _, times, coeffs = eng.solve_dense(p.y0_flat, t64)
    lib, dc, n, sign_, shape, dtype, dev = eng.lib, eng.dt_code, p.n, p.t_sign, p.shape, p.dtype, p.device
    ptrs = [_lib.ptr_array([c.data_ptr() for c in cs]) for cs in coeffs]

    def dense_output_fn(t_eval):
        te = float(t_eval) * sign_                                                     # solver (ascending) time
        idx = bisect.bisect_right(times, te)                                           # searchsorted(..., side="right")
        idx = min(max(idx, 1), len(times) - 1)
        lo, hi = times[idx - 1], times[idx]
        assert lo <= te <= hi, 'invalid interpolation, fails `t0 <= t <= t1`: {}, {}, {}'.format(lo, te, hi)
        out = torch.empty(n, dtype=dtype, device=dev)
        with on_solver_stream(dev) as ss2:
            _lib.check(lib.tdq_poly_eval(dc, ptrs[idx - 1], (te - lo) / (hi - lo), out.data_ptr(), n, _stream()))
            ss2.publish(out)
        return out.view(shape)
    dense_output_fn._keep = (coeffs, ptrs)
    return dense_output_fn


def _odeint_backprop(p, func, y0, t, params, _stats):
    """Plain odeint under autograd: gradients of the discrete solve w.r.t. y0, t and every parameter func reaches
    (odeint.py:49-108 differentiated as the reference's recorded graph would be; see backprop.py)."""
    from .backprop import _BackpropFunction, adaptive_tableau
    if p.dtype.is_complex:
        raise NotImplementedError("gradients of the discrete solve of a complex state are not implemented; use "
                                  "odeint_adjoint, or call odeint under torch.no_grad()")
    if p.is_tuple:
        y0_flat = p.layout.flatten(list(y0))          # differentiable w.r.t. every piece
    else:
        y0_flat = y0.reshape(-1)
    holder = {}

    def run():
        if p.method in ADAPTIVE_METHODS:
            eng = _make_adaptive_engine(p, p.method, p.rtol, p.atol, p.rtol_vec, p.atol_vec,
                                        dict(p.options, run_ahead=0, graph=False), segs=p.segs, pieces=p.pieces,
                                        norm_fn=p.norm_fn, q_view=p.q_view, callbacks=p.callbacks)
            t64 = p.t_cpu.to(torch.float64).to(p.device)
            sol, tape = eng.solve_taped(p.y0_flat, t64, t_start=float(p.t_cpu[0]))
            holder["eng"] = eng
            return sol.clone(), {"kind": "adaptive", "tape": tape, "tab": adaptive_tableau(p.method)}
        o = p.options
        if p.method in ADAMS_METHODS:
            raise NotImplementedError("gradients of the discrete solve are implemented for the explicit Runge-Kutta "
                                      "methods; use odeint_adjoint with the Adams methods")
        if o.get("interp", "linear") != "linear":
            raise NotImplementedError("gradients through interp='cubic' are not implemented (use the default linear "
                                      "interpolation, or odeint_adjoint)")
        y0_view = p.layout.views(p.y0_flat) if p.is_tuple else p.y0_flat.view(p.shape)
        with torch.enable_grad():                     # the grid as a differentiable function of the output times
            t_req = p.t_cpu.detach().clone().requires_grad_(True)
            grid_req = fixed_grid(p.method, o, p.original_func, y0_view, t_req, keep_graph=True)
        grid = grid_req.detach()
        eng = FixedGridEngine(p.fn, p.n, p.dtype, p.device, method=p.method, t_sign=p.t_sign,
                              perturb=o.get("perturb", False), graph=False, callbacks=p.callbacks, pieces=p.pieces)
        sol, tape = eng.solve_taped(p.y0_flat, grid, p.t_cpu)
        holder["eng"] = eng
        return sol, {"kind": "fixed", "tape": tape, "grid": grid, "grid_req": grid_req, "t_req": t_req}
    with on_solver_stream(p.device) as ss:
        sol = _BackpropFunction.apply(p, run, t, y0_flat, *params)
        ss.publish(sol)
    eng = holder.get("eng")
    if eng is not None:
        _LAST_STATS.clear()
        _LAST_STATS.update(nfe=eng.nfe, launches=getattr(eng, "launches", 0), attempts=getattr(eng, "n_attempts", None),
                           n_accept=getattr(eng, "n_accept", None), n_reject=getattr(eng, "n_reject", None),
                       fused_linear=getattr(eng, "linear", None) is not None,
                       fused_attempt=bool((getattr(eng, "linear", None) or {}).get("whole")))
        if _stats is not None:
            _stats.update(_LAST_STATS)
    return _unflatten(p, sol)


def odeint(func, y0, t, *, rtol=1e-7, atol=1e-9, method=None, options=None, event_fn=None, _stats=None):
    """Integrate dy/dt = func(t, y), y(t[0]) = y0 and return y at every t (odeint.py:49-108).

    Arguments, defaults, output shape/dtype and errors are the reference's.  `options` additionally
    accepts `graph` (True/False/'auto'), `run_ahead` (int; 0 reproduces the reference's exact func
    call sequence) and `process_group` (batch-sharded solve with a common step size).
    Under autograd the result carries the gradient of the discrete solve w.r.t. y0, t and func's parameters
    (backprop.py); odeint_adjoint gives the continuous adjoint instead.
    """
    p = normalise(func, y0, t, rtol, atol, method, options, event_fn)
    if torch.is_grad_enabled():
        from .backprop import discover_params
        y_req = any(y_.requires_grad for y_ in y0) if p.is_tuple else y0.requires_grad
        params = discover_params(func)
        if y_req or t.requires_grad or params:
            if p.event_fn is not None:
                # gradients through an event solve: the reference backpropagates through the solver up to the event
                # and through the bisection's interpolant; here the adjoint method serves that case
                if isinstance(func, torch.nn.Module):
                    warnings.warn("torchdiffeq_b200.odeint(event_fn=...): gradients are computed with the adjoint method",
                                  stacklevel=2)
                    from .adjoint import odeint_adjoint
                    return odeint_adjoint(func, y0, t, rtol=rtol, atol=atol, method=method, options=options,
                                          event_fn=event_fn)
                raise NotImplementedError("gradients through odeint(event_fn=...) need an nn.Module func (they are "
                                          "computed by odeint_adjoint)")
            return _odeint_backprop(p, func, y0, t, params, _stats)
    with torch.no_grad(), on_solver_stream(p.device) as ss:
        if p.event_fn is not None:
            event_t, sol, eng = _solve_event(p)
            ss.publish(sol)
            return torch.tensor(event_t, dtype=t.dtype, device=t.device), _unflatten(p, sol)     # odeint.py:98, :105-108
        sol, eng = _solve(p)
        ss.publish(sol)
    _LAST_STATS.clear()
    _LAST_STATS.update(nfe=eng.nfe, launches=getattr(eng, "launches", 0), attempts=getattr(eng, "n_attempts", None),
                       n_accept=getattr(eng, "n_accept", None), n_reject=getattr(eng, "n_reject", None),
                       fused_linear=getattr(eng, "linear", None) is not None,
                       fused_attempt=bool((getattr(eng, "linear", None) or {}).get("whole")))
    if _stats is not None:               # private: solver counters for bench.py and the tests
        _stats["nfe"] = eng.nfe
        _stats["launches"] = _stats.get("launches", 0) + getattr(eng, "launches", 0)
        _stats["attempts"] = getattr(eng, "n_attempts", None)
        _stats["n_accept"], _stats["n_reject"] = getattr(eng, "n_accept", None), getattr(eng, "n_reject", None)
        _stats["fused_linear"], _stats["fused_attempt"] = _LAST_STATS["fused_linear"], _LAST_STATS["fused_attempt"]
    return _unflatten(p, sol)
