"""CPU tests of the host-side logic that needs no GPU: state layout, tolerance vectors, the fixed-grid
step tables (checked against the reference's loop semantics, solvers.py:102-128), the engine-cache key."""
import pytest
import torch

from torchdiffeq_b200._engine import Layout
from torchdiffeq_b200._fixed import FixedGridEngine, grid_from_step_size
from torchdiffeq_b200.odeint import _func_signature, _tol_vector


def test_layout_alignment_and_views():
    lay = Layout([(5, 6), (3,), (), (2, 2)], torch.float32)
    assert all(o % 4 == 0 for o in lay.offsets)                   # 16-byte aligned float32 pieces
    assert lay.lens == [30, 3, 1, 4] and lay.n == 32 + 4 + 4 + 4
    parts = [torch.arange(30.).view(5, 6), torch.tensor([1., 2., 3.]), torch.tensor(7.), torch.ones(2, 2)]
    flat = lay.flatten(parts)
    back = lay.views(flat)
    for a, b in zip(parts, back):
        assert torch.equal(a, b)
    pad = torch.ones(lay.n, dtype=torch.bool)
    for o, l in zip(lay.offsets, lay.lens):
        pad[o:o + l] = False
    assert (flat[pad] == 0).all()                                  # padding is zero
    sol = flat.repeat(3, 1)
    assert lay.views(sol, (3,))[0].shape == (3, 5, 6)              # misc.py:126-134 with a leading time dimension
    lay64 = Layout([(3,), (3,)], torch.float64)
    assert lay64.offsets == [0, 4]                                 # 16 bytes = 2 doubles


def test_tol_vector():
    lay = Layout([(2, 3), (3,)], torch.float64)
    s, v = _tol_vector("rtol", 1e-6, lay, None, torch.device("cpu"))
    assert s == 1e-6 and v is None
    s, v = _tol_vector("rtol", (1e-6, 1e-4), lay, None, torch.device("cpu"))
    assert s is None and v.dtype == torch.float64 and v.numel() == lay.n
    # the reference builds these through float32 (torch.as_tensor of a Python float), misc.py:122
    assert v[0] == float(torch.tensor(1e-6)) and v[lay.offsets[1]] == float(torch.tensor(1e-4))
    with pytest.raises(AssertionError):
        _tol_vector("rtol", (1e-6,), lay, None, torch.device("cpu"))
    s, v = _tol_vector("atol", torch.tensor([1e-3, 1e-6]), None, (4, 2), torch.device("cpu"))
    assert v.shape == (8,) and v[1] == float(torch.tensor(1e-6))   # float32 tensor -> float64, like rk_common.py:186


def _reference_fixed_loop(grid, t):
    """solvers.py:108-126 as written: which output index is produced in which step, and how."""
    recs, j = [], 1
    for s, (t0, t1) in enumerate(zip(grid[:-1], grid[1:])):
        while j < len(t) and t1 >= t[j]:
            if t[j] == t0:
                recs.append((s, j, 0, 0.0))
            elif t[j] == t1:
                recs.append((s, j, 1, 0.0))
            else:
                recs.append((s, j, 2, float((t[j] - t0) / (t1 - t0))))
            j += 1
    return recs


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("case", ["grid_is_t", "step_size", "coarse_t"])
def test_fixed_grid_tables(case, dtype):
    if case == "grid_is_t":
        t = torch.linspace(0., 25., 50, dtype=dtype)
        grid = t
    elif case == "step_size":
        t = torch.linspace(0., 5., 7, dtype=dtype)
        grid = grid_from_step_size(0.03)(None, None, t)
    else:
        t = torch.tensor([0., 0.3, 0.31, 2.0], dtype=dtype)
        grid = torch.linspace(0., 2., 5, dtype=dtype)
    eng = FixedGridEngine.__new__(FixedGridEngine)
    eng.dtype, eng.perturb, eng.t_sign, eng.method = torch.float32, False, 1.0, "rk4"
    ts, dtT, rec_begin, out_idx, mode, slope, n_steps = eng._tabulate(grid, t)
    want = _reference_fixed_loop(grid, t)
    got = []
    for s in range(n_steps):
        for r in range(int(rec_begin[s]), int(rec_begin[s + 1])):
            got.append((s, int(out_idx[r]), int(mode[r]), float(slope[r]) if int(mode[r]) == 2 else 0.0))
    assert [g[:3] for g in got] == [w[:3] for w in want]
    for g, w in zip(got, want):
        assert g[3] == pytest.approx(float(torch.tensor(w[3], dtype=dtype).to(torch.float32)), abs=0)
    assert torch.equal(dtT, (grid[1:] - grid[:-1]).to(torch.float32))
    assert torch.equal(ts[:, 0], grid[:-1].to(torch.float32)) and torch.equal(ts[:, 3], grid[1:].to(torch.float32))
    # perturb: first time moved up one ulp, last time down (misc.py:188-193)
    eng.perturb = True
    tsp = eng._tabulate(grid, t)[0]
    assert (tsp[:, 0] > ts[:, 0]).all() and (tsp[:, 3] < ts[:, 3]).all()
    # reverse time: sign folded into the func times and into dt
    eng.perturb, eng.t_sign = False, -1.0
    tsr, dtr = eng._tabulate(grid, t)[:2]
    assert torch.equal(tsr, -ts) and torch.equal(dtr, -dtT)


def test_cache_signature_tracks_reachable_tensors():
    # plain callables are never cached on their own (globals, defaults and cells cannot be enumerated safely, ADVICE r1):
    # no signature unless the caller opts in with options={'cache': True}
    A = torch.randn(3, 3)
    f = lambda t, y: y @ A
    assert _func_signature(f) is None
    assert _func_signature(f, explicit=True) == (id(f),)

    class M(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.lin = torch.nn.Linear(2, 2)
            self.c = torch.ones(2)

        def forward(self, t, y):
            return self.lin(y) * self.c
    m = M()
    k = _func_signature(m)
    m.c = torch.ones(2)                      # plain tensor attribute rebound
    assert _func_signature(m) != k
    k = _func_signature(m)
    m.eval()
    assert _func_signature(m) != k
    k = _func_signature(m)
    with torch.no_grad():
        m.lin.weight.add_(1.0)               # in-place update keeps the storage: same key
    assert _func_signature(m) == k
    m.lin.weight = torch.nn.Parameter(torch.zeros(2, 2))
    assert _func_signature(m) != k
    k = _func_signature(m)
    m.scale = 2.0                            # plain Python attributes a captured graph would have baked in
    assert _func_signature(m) != k
    k = _func_signature(m)
    m.scale = 3.0
    assert _func_signature(m) != k
    k = _func_signature(m)
    m.extra = [torch.zeros(2), 1.5]          # tensors inside containers
    k2 = _func_signature(m)
    assert k2 != k
    m.extra[0] = torch.zeros(2)
    assert _func_signature(m) != k2
    k = _func_signature(m)
    m.lin.training = True                    # a submodule's flag (m.eval() above cleared it)
    assert _func_signature(m) != k
    hash(_func_signature(m))


def test_plugin_registration_and_seam_identification(monkeypatch):
    """torchdiffeq_b200.plugin on the CPU: registration is in place and reversible, CPU states keep the previous
    solver class, and the two identity tests the seam forces on us (default RMS norm, null callback) recognise the
    reference's actual objects, as recorded from it in tests/golden/seam_objects.json."""
    import json
    import os
    import sys
    import types
    from torchdiffeq_b200 import plugin

    class Prev:
        def __init__(self, func, y0, **kw):
            self.kw = kw

        @classmethod
        def valid_callbacks(cls):
            return set()
    solvers = {"dopri5": Prev, "rk4": Prev}
    replaced = plugin.register(solvers, methods=("dopri5", "rk4", "tsit5"))
    assert replaced == {"dopri5": Prev, "rk4": Prev, "tsit5": None}
    assert solvers["dopri5"].valid_callbacks() == {"callback_step", "callback_accept_step", "callback_reject_step"}
    assert solvers["rk4"].valid_callbacks() == {"callback_step"}
    s = solvers["dopri5"](func=lambda t, y: y, y0=torch.zeros(3), rtol=1e-3, atol=1e-4, norm=None)
    assert isinstance(s, Prev) and s.kw["rtol"] == 1e-3             # CPU tensors: the reference's own class
    plugin.register(solvers, methods=("dopri5",))                   # registering twice does not nest dispatchers
    assert solvers["dopri5"].cpu_cls is Prev
    plugin.unregister(replaced, solvers)
    assert solvers == {"dopri5": Prev, "rk4": Prev}

    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "seam_objects.json")) as f:
        ref = json.load(f)

    def like(ident):                                                 # a function that carries a recorded identity
        fn = lambda *a, **k: None
        fn.__name__, fn.__module__, fn.__qualname__ = ident["name"], ident["module"], ident["qualname"]
        return fn
    assert plugin._is_default_rms(like(ref["_rms_norm"])) and not plugin._is_default_rms(like(ref["_mixed_norm"]))
    assert plugin._is_null_callback(like(ref["_null_callback"])) and not plugin._is_null_callback(lambda *a: None)
    assert ref["_PerturbFunc"]["base_func_attr"]
    wrapper = type(ref["_PerturbFunc"]["class"], (torch.nn.Module,), {})()
    wrapper.base_func = abs
    assert plugin._unwrap_perturb(wrapper) is abs
    # register() without a dict patches the registry module of the reference in place; every registered method
    # has a solver of that name there
    assert ref["registry"]["shared_with_adjoint"]
    registry = types.ModuleType(ref["registry"]["module"])
    registry.SOLVERS = {name: Prev for name in ref["registry"]["methods"]}
    monkeypatch.setitem(sys.modules, ref["registry"]["module"], registry)
    rep = plugin.register()
    assert set(rep) <= set(ref["registry"]["methods"]) and all(cls is Prev for cls in rep.values())
    assert isinstance(registry.SOLVERS["dopri5"], plugin._Dispatch)
    plugin.unregister(rep)
    assert registry.SOLVERS == {name: Prev for name in ref["registry"]["methods"]}


def test_fused_linear_options_and_eligibility():
    """The switches of the fused linear paths are options of this package (no 'Unexpected arguments' warning, misc.py:13-15),
    and `fusable` (fields.py) only accepts an unmodified LinearField on a float32 [..., 128] state."""
    import warnings
    import torch
    import torchdiffeq_b200 as tdq
    from torchdiffeq_b200 import _lib
    import importlib
    O_ = importlib.import_module("torchdiffeq_b200.odeint")
    from torchdiffeq_b200.fields import fusable

    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        O_._warn_unused("dopri5", {"fused_linear": False, "fused_attempt": False, "fused_controller": False, "run_ahead": 0}, set())
        assert not w
        O_._warn_unused("dopri5", {"not_an_option": 1}, set())
        assert len(w) == 1 and "not_an_option" in str(w[0].message)

    lib = _lib.load()
    cpu = torch.device("cpu")
    f = tdq.LinearField(torch.eye(128))
    assert fusable(f, (7, 128), torch.float32, cpu, lib) is f.weight
    assert fusable(f, (7, 128), torch.float64, cpu, lib) is None              # state dtype
    assert fusable(f, (7, 64), torch.float32, cpu, lib) is None               # width
    assert fusable(tdq.LinearField(torch.eye(64)), (7, 64), torch.float32, cpu, lib) is None   # no kernel for that width
    assert fusable(lambda t, y: y, (7, 128), torch.float32, cpu, lib) is None

    class Sub(tdq.LinearField):
        def forward(self, t, y):
            return super().forward(t, y) * 2.0

    assert fusable(Sub(torch.eye(128)), (7, 128), torch.float32, cpu, lib) is None   # an overridden forward is never fused
