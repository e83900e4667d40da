"""Generate the golden vectors under tests/golden/ from the UNMODIFIED reference.

Run in the build container, where the reference lives at /root/reference (it does not exist on the GPU
box, so nothing else may import it):

    python tests/golden/make_golden.py

Outputs (committed):
    tableaus.json         float64 coefficients of the reference's own tableau tensors
    zoo.pt                reference solutions + NFE for the analytic problem zoo (tests/problems.py)
    linear_batch.pt       C2-shaped batched linear ODE at a small batch: solution, dt sequence, accept flags
    spiral_rk4.pt         C1: rk4 on the cubic spiral, B=1024, selected output rows
    adjoint_mlp.pt        odeint_adjoint gradients for a small MLP field
    detest.pt             all 25 DETEST problems: NFE, end states and RMS error vs dopri5@1e-12 for dopri5/dopri8 at
                          rtol=atol in {1e-3, 1e-6, 1e-9} (+ dopri8 at 1e-12)
    options.pt            step_t / min_step / max_step / first_step / tuple-state / vector-tol cases
    fixed_extra.pt        interp='cubic' and event handling for the fixed-grid methods
    adjoint_many.pt       odeint_adjoint on a field with 80 parameter tensors (default norm: 83 segments)
    adams.json, adams.pt  Adams-Bashforth(-Moulton) weight tables and explicit_adams / implicit_adams solutions, events
    backprop.pt           gradients of plain odeint (autograd through the reference's solver operations)
    seam_objects.json     identities of the objects the reference hands a registered solver (default norm, null
                          callback, perturb wrapper) and where its SOLVERS registry lives
"""
import json
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, "/root/reference")
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torchdiffeq                                   # noqa: E402  (the reference)
from torchdiffeq._impl import adaptive_heun, bosh3, dopri5, dopri8, fehlberg2, tsit5   # noqa: E402
import problems as P                                 # noqa: E402

assert torchdiffeq.__file__.startswith("/root/reference"), torchdiffeq.__file__
torch.set_num_threads(8)


class Rec(torch.nn.Module):
    """Counts NFE and records the accepted/rejected dt sequence through the reference's callbacks."""

    def __init__(self, f):
        super().__init__()
        self.f, self.nfe, self.dts, self.acc = f, 0, [], []

    def forward(self, t, y):
        self.nfe += 1
        return self.f(t, y)

    def callback_accept_step(self, t0, y0, dt):
        self.dts.append(float(dt)); self.acc.append(True)

    def callback_reject_step(self, t0, y0, dt):
        self.dts.append(float(dt)); self.acc.append(False)


def dump_tableaus():
    out = {}
    for name, cls in [("dopri5", dopri5.Dopri5Solver), ("dopri8", dopri8.Dopri8Solver), ("bosh3", bosh3.Bosh3Solver),
                      ("fehlberg2", fehlberg2.Fehlberg2), ("adaptive_heun", adaptive_heun.AdaptiveHeunSolver),
                      ("tsit5", tsit5.Tsit5Solver)]:
        tab = cls.tableau
        fsal = bool(tab.c_sol[-1] == 0 and (tab.c_sol[:-1] == tab.beta[-1]).all())     # rk_common.py:83
        out[name] = {"alpha": tab.alpha.tolist(), "beta": [b.tolist() for b in tab.beta], "c_sol": tab.c_sol.tolist(),
                     "c_err": tab.c_error.tolist(), "c_mid": cls.mid.tolist(), "order": cls.order, "fsal": fsal,
                     "n_stages": len(tab.alpha)}
    with open(os.path.join(HERE, "tableaus.json"), "w") as f:
        json.dump(out, f, indent=1)


def seam_objects():
    """What torchdiffeq_b200.plugin has to recognise in the reference's objects, by name only (misc.py:11, :18-33,
    :174-197; odeint.py:19-46; adjoint.py:4)."""
    import importlib
    misc = importlib.import_module("torchdiffeq._impl.misc")
    odeint_mod = importlib.import_module("torchdiffeq._impl.odeint")
    ident = lambda fn: {"name": fn.__name__, "module": fn.__module__, "qualname": fn.__qualname__}
    wrapped = misc._PerturbFunc(abs)
    out = {"_rms_norm": ident(misc._rms_norm), "_mixed_norm": ident(misc._mixed_norm),
           "_null_callback": ident(misc._null_callback),
           "_PerturbFunc": {"class": type(wrapped).__name__, "base_func_attr": wrapped.base_func is abs},
           "registry": {"module": odeint_mod.__name__, "methods": sorted(odeint_mod.SOLVERS),
                        "shared_with_adjoint": importlib.import_module("torchdiffeq._impl.adjoint").SOLVERS is odeint_mod.SOLVERS}}
    with open(os.path.join(HERE, "seam_objects.json"), "w") as f:
        json.dump(out, f, indent=1)


def zoo():
    # the matrix construction must agree with the reference's LinearODE (problems.py:35-38)
    sys.path.insert(0, "/root/reference/tests")
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_problems", "/root/reference/tests/problems.py")
    refp = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(refp)
    assert torch.equal(refp.LinearODE().A.detach(), P.LinearODE().A.detach())
    cases = {}
    for ode in ("constant", "sine", "linear", "exp"):
        for method in ("dopri5", "dopri8", "tsit5", "bosh3", "fehlberg2", "adaptive_heun", "rk4", "euler", "midpoint",
                       "heun2", "heun3"):
            for dtype in (torch.float32, torch.float64):
                for reverse in (False, True):
                    if method in ("rk4", "euler", "midpoint", "heun2", "heun3") and ode != "constant":
                        continue                                   # odeint_tests.py:42
                    f, y0, t, sol = P.construct_problem("cpu", ode=ode, reverse=reverse, dtype=dtype)
                    if method == "dopri8":                         # odeint_tests.py:29-32
                        kw = dict(rtol=1e-12, atol=1e-14) if dtype == torch.float64 else dict(rtol=1e-7, atol=1e-7)
                    else:
                        kw = {}
                    rec = Rec(f)
                    with torch.no_grad():
                        y = torchdiffeq.odeint(rec, y0, t, method=method, **kw)
                    key = "%s/%s/%s/%s" % (ode, method, str(dtype).split(".")[1], "rev" if reverse else "fwd")
                    cases[key] = {"y": y, "nfe": rec.nfe, "kw": kw, "exact": sol}
    torch.save(cases, os.path.join(HERE, "zoo.pt"))


def linear_batch():
    out = {}
    for dtype in (torch.float32, torch.float64):
        f = P.BatchedLinear(128, dtype)
        g = torch.Generator().manual_seed(1)
        y0 = torch.randn(64, 128, generator=g).to(dtype)
        for name, t in (("span", torch.tensor([0., 2.])), ("dense", torch.linspace(0, 2, 9))):
            rec = Rec(f)
            with torch.no_grad():
                y = torchdiffeq.odeint(rec, y0, t, method="dopri5", rtol=1e-5, atol=1e-7)
            out["%s/%s" % (name, str(dtype).split(".")[1])] = {"y": y, "nfe": rec.nfe, "dts": rec.dts, "acc": rec.acc,
                                                              "t": t}
    torch.save(out, os.path.join(HERE, "linear_batch.pt"))


def spiral_rk4():
    f = P.Spiral()
    g = torch.Generator().manual_seed(0)
    y0 = torch.tensor([[2., 0.]]) * (1 + 0.1 * torch.rand(1024, 1, generator=g))
    t = torch.linspace(0., 25., 1000)
    with torch.no_grad():
        y = torchdiffeq.odeint(f, y0, t, method="rk4")
        # a coarser output grid on a fine step_size grid exercises the linear interpolation
        t2 = torch.linspace(0., 5., 7)
        y2 = torchdiffeq.odeint(f, y0[:16], t2, method="rk4", options={"step_size": 0.03})
    rows = [0, 1, 2, 10, 100, 500, 998, 999]
    fixed = {}
    for method in ("euler", "midpoint", "heun2", "heun3", "rk4"):
        for perturb in (False, True):
            with torch.no_grad():
                fixed["%s/%d" % (method, perturb)] = torchdiffeq.odeint(
                    f, y0[:16], t2, method=method, options={"step_size": 0.03, "perturb": perturb})
    torch.save({"y0": y0, "rows": rows, "y_rows": y[rows].clone(), "t2": t2, "y2": y2, "fixed": fixed},
               os.path.join(HERE, "spiral_rk4.pt"))


def adjoint_mlp():
    out = {}
    for dtype in (torch.float32, torch.float64):
        f = P.MLPField(dim=8, hidden=16, seed=0, dtype=dtype)
        g = torch.Generator().manual_seed(1)
        y0 = torch.randn(32, 8, generator=g).to(dtype).requires_grad_(True)
        for name, t in (("span", torch.tensor([0., 1.])), ("multi", torch.tensor([0., 0.4, 1.0]))):
            for norm in ("default", "seminorm"):
                f.zero_grad()
                y0.grad = None
                ao = {"norm": "seminorm"} if norm == "seminorm" else None
                y = torchdiffeq.odeint_adjoint(f, y0, t, method="dopri5", rtol=1e-6, atol=1e-8, adjoint_options=ao)
                loss = y[-1].pow(2).mean() + (y[1].sum() * 0.01 if len(t) > 2 else 0)
                loss.backward()
                out["%s/%s/%s" % (name, norm, str(dtype).split(".")[1])] = {
                    "y": y.detach().clone(), "gy0": y0.grad.clone(), "gp": [q.grad.clone() for q in f.parameters()],
                    "t": t}
    torch.save(out, os.path.join(HERE, "adjoint_mlp.pt"))


def detest():
    """All 25 DETEST problems (tests/DETEST/detest.py:8-315) through the UNMODIFIED reference, using the reference's OWN
    problem definitions (so the goldens also pin tests/problems.py's restatement of them): NFE and end state for dopri5
    and dopri8 at rtol = atol in {1e-3, 1e-6, 1e-9}, dopri8 at 1e-12, and the dopri5 @ 1e-12 solution run.py:37-41 uses as
    ground truth with the RMS error run.py:47 reports against it."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_detest", "/root/reference/tests/DETEST/detest.py")
    rd = importlib.util.module_from_spec(spec)
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)                       # run.py:8
    try:
        spec.loader.exec_module(rd)
        out = {}
        for name in P.DETEST_NAMES:
            f, init, _ = getattr(rd, name)()
            t0, y0 = init()
            mine, my0, mt0 = P.detest(name)
            assert torch.equal(y0, my0) and float(t0) == mt0, name
            probe = y0 + 0.125
            assert torch.equal(f(torch.tensor(0.5), probe.clone()), mine(torch.tensor(0.5), probe.clone())), name
            t = torch.stack([t0, torch.tensor(20.)])
            with torch.no_grad():
                truth = torchdiffeq.odeint(f, y0, t, atol=1e-12, rtol=1e-12, method="dopri5")[1]
            out["%s/truth" % name] = {"y": truth.clone()}
            for method, tols in (("dopri5", (1e-3, 1e-6, 1e-9)), ("dopri8", (1e-3, 1e-6, 1e-9, 1e-12))):
                for tol in tols:
                    rec = Rec(f)
                    with torch.no_grad():
                        y = torchdiffeq.odeint(rec, y0, t, method=method, rtol=tol, atol=tol)
                    err = torch.sqrt(torch.mean((truth - y[1]) ** 2))
                    out["%s/%s/%g" % (name, method, tol)] = {"y": y[-1].clone(), "nfe": rec.nfe, "err": float(err)}
                    print(name, method, tol, rec.nfe, float(err), flush=True)
    finally:
        torch.set_default_dtype(old)
    torch.save(out, os.path.join(HERE, "detest.pt"))


def options_cases():
    out = {}
    f, y0, t, _ = P.construct_problem("cpu", ode="linear", dtype=torch.float64)
    for key, opts in (("min_step", {"min_step": 2}), ("max_step", {"max_step": 0.05}), ("first_step", {"first_step": 0.01}),
                      ("step_t", {"step_t": torch.tensor([1.5, 2.25, 6.0])}), ("factors", {"safety": 0.8, "ifactor": 5.0, "dfactor": 0.3})):
        rec = Rec(f)
        with torch.no_grad():
            y = torchdiffeq.odeint(rec, y0, t, method="dopri5", options=dict(opts))
        out[key] = {"y": y, "nfe": rec.nfe, "dts": rec.dts, "acc": rec.acc, "opts": opts}
    # tuple state with per-piece tolerances (misc.py:115-123) and the mixed norm (misc.py:30-33)
    A = P.skew_matrix(6, torch.float64)
    def tf(t_, state):
        a, b = state
        return (a @ A.t(), -0.5 * b + a[:, :2].sum())
    g = torch.Generator().manual_seed(3)
    ya, yb = torch.randn(5, 6, generator=g, dtype=torch.float64), torch.randn(3, generator=g, dtype=torch.float64)
    tt = torch.linspace(0, 2, 5, dtype=torch.float64)
    with torch.no_grad():
        sol = torchdiffeq.odeint(tf, (ya, yb), tt, method="dopri5", rtol=1e-6, atol=1e-8)
        sol_v = torchdiffeq.odeint(tf, (ya, yb), tt, method="dopri5", rtol=(1e-6, 1e-4), atol=(1e-8, 1e-7))
    out["tuple"] = {"ya": ya, "yb": yb, "t": tt, "sol": [s.clone() for s in sol], "sol_vtol": [s.clone() for s in sol_v]}
    # jump_t (rk_common.py:302-308, :346-351; odeint_tests.py:126-161)
    for method in ("dopri5", "tsit5", "bosh3"):
        for dtype in (torch.float32, torch.float64):
            x0 = torch.tensor([1.0, 2.0], dtype=dtype)
            tj = torch.tensor([0., 1.0])
            plain, better = P.JumpField(), P.JumpField()
            with torch.no_grad():
                y_plain = torchdiffeq.odeint(plain, x0, tj, atol=1e-6, method=method)
                y_jump = torchdiffeq.odeint(better, x0, tj, rtol=1e-6, atol=1e-6, method=method,
                                            options={"jump_t": torch.tensor([0.5])})
            out["jump/%s/%s" % (method, str(dtype).split(".")[1])] = {
                "y_plain": y_plain, "nfe_plain": plain.nfe, "y_jump": y_jump, "nfe_jump": better.nfe}
    torch.save(out, os.path.join(HERE, "options.pt"))


def events():
    """event_tests.py:14-49 (forward) and :51-64 (adjoint)."""
    out = {}
    for ode in ("constant", "sine"):
        for method in ("dopri5", "dopri8", "tsit5", "bosh3"):
            for dtype in (torch.float32, torch.float64):
                for reverse in (False, True):
                    f, y0, t, sol = P.construct_problem("cpu", ode=ode, reverse=reverse, dtype=dtype)
                    target = sol[2]
                    rec = Rec(f)
                    with torch.no_grad():
                        et, ys = torchdiffeq.odeint(rec, y0, t[0:2], event_fn=lambda t_, y_: torch.sum(y_ - target).real,
                                                    method=method)
                    out["%s/%s/%s/%s" % (ode, method, str(dtype).split(".")[1], "rev" if reverse else "fwd")] = {
                        "event_t": et, "y": ys, "nfe": rec.nfe, "t2": t[2], "target": target}
    f, y0, t, sol = P.construct_problem("cpu", ode="constant")
    y0 = y0.requires_grad_(True)
    target = sol[-1]
    et, ys = torchdiffeq.odeint_adjoint(f, y0, t[0:2], event_fn=lambda t_, y_: torch.sum(y_ - target), method="dopri5")
    ys[-1].sum().backward()
    out["adjoint/constant"] = {"event_t": et.detach(), "y": ys.detach(), "gy0": y0.grad.clone(),
                               "gp": [q.grad.clone() for q in f.parameters()], "t_last": t[-1]}
    # odeint_event with the implicit-function gradient (odeint.py:160-231): time at which y' = -y + b hits a level
    class Decay(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.b = torch.nn.Parameter(torch.tensor(0.3, dtype=torch.float64))

        def forward(self, t_, y_):
            return -y_ + self.b
    fd = Decay()
    yd = torch.tensor([2.0, 3.0], dtype=torch.float64, requires_grad=True)
    t0 = torch.tensor(0.5, dtype=torch.float64, requires_grad=True)
    et, ys = torchdiffeq.odeint_event(fd, yd, t0, event_fn=lambda t_, y_: y_[0] - 1.0, odeint_interface=torchdiffeq.odeint_adjoint,
                                      method="dopri5", rtol=1e-9, atol=1e-11)
    (et + ys[-1].sum()).backward()
    out["odeint_event/decay"] = {"event_t": et.detach(), "y": ys.detach(), "gy0": yd.grad.clone(), "gt0": t0.grad.clone(),
                                 "gb": fd.b.grad.clone()}
    torch.save(out, os.path.join(HERE, "events.pt"))


def fixed_extra():
    """interp='cubic' (solvers.py:120-125, :166-173) and event handling with the fixed-grid methods (solvers.py:130-164;
    event_tests.py:14-49 runs every fixed method with {"step_size": 0.01, "interp": "cubic"})."""
    out = {}
    f = P.Spiral()
    g = torch.Generator().manual_seed(0)
    y0 = torch.tensor([[2., 0.]]) * (1 + 0.1 * torch.rand(1024, 1, generator=g))
    t2 = torch.linspace(0., 5., 7)
    for method in ("euler", "midpoint", "heun2", "heun3", "rk4"):
        for perturb in (False, True):
            rec = Rec(f)
            with torch.no_grad():
                y = torchdiffeq.odeint(rec, y0[:16], t2, method=method,
                                       options={"step_size": 0.03, "interp": "cubic", "perturb": perturb})
            out["cubic/%s/%d" % (method, perturb)] = {"y": y, "nfe": rec.nfe}
    # cubic on the output grid itself, both directions and dtypes (constant problem: exact solution known)
    for dtype in (torch.float32, torch.float64):
        for reverse in (False, True):
            fc, yc, tc, sol = P.construct_problem("cpu", ode="constant", reverse=reverse, dtype=dtype)
            rec = Rec(fc)
            with torch.no_grad():
                y = torchdiffeq.odeint(rec, yc, tc, method="rk4", options={"step_size": 0.1, "interp": "cubic"})
            out["cubic_grid/%s/%s" % (str(dtype).split(".")[1], "rev" if reverse else "fwd")] = {"y": y, "nfe": rec.nfe}
    for ode in ("constant", "sine"):
        for method in ("euler", "midpoint", "heun2", "heun3", "rk4"):
            for dtype in (torch.float32, torch.float64):
                for reverse in (False, True):
                    for interp in ("cubic", "linear"):
                        fe, ye, te, sol = P.construct_problem("cpu", ode=ode, reverse=reverse, dtype=dtype)
                        target = sol[2]
                        rec = Rec(fe)
                        with torch.no_grad():
                            et, ys = torchdiffeq.odeint(rec, ye, te[0:2], event_fn=lambda t_, y_: torch.sum(y_ - target).real,
                                                        method=method, options={"step_size": 0.01, "interp": interp})
                        out["event/%s/%s/%s/%s/%s" % (ode, method, str(dtype).split(".")[1], "rev" if reverse else "fwd",
                                                    interp)] = {"event_t": et, "y": ys, "nfe": rec.nfe, "t2": te[2],
                                                                "target": target}
    torch.save(out, os.path.join(HERE, "fixed_extra.pt"))


def backprop():
    """Plain odeint differentiated by autograd through the solver's own operations (rk_common.py:31-90,
    gradient_tests.py:13-23, api_tests.py:28-39): gradients w.r.t. y0, t and the parameters of func."""
    out = {}
    for dtype in (torch.float32, torch.float64):
        dn = str(dtype).split(".")[1]
        for name, tv in (("span", [0., 1.]), ("multi", [0., 0.4, 1.0]), ("rev", [1.0, 0.3, 0.])):
            for method in ("dopri5", "tsit5", "bosh3", "rk4", "midpoint", "euler"):
                f = P.MLPField(dim=8, hidden=16, seed=0, dtype=dtype)
                g = torch.Generator().manual_seed(1)
                y0 = torch.randn(32, 8, generator=g).to(dtype).requires_grad_(True)
                t = torch.tensor(tv, dtype=torch.float64).requires_grad_(True)
                tols = dict(rtol=1e-6, atol=1e-8) if dtype == torch.float64 else dict(rtol=1e-4, atol=1e-6)
                kw = tols if method in ("dopri5", "tsit5", "bosh3") else {}
                opts = {"step_size": 0.05} if method in ("rk4", "midpoint", "euler") and name != "multi" else None
                y = torchdiffeq.odeint(f, y0, t, method=method, options=opts, **kw)
                loss = y[-1].pow(2).mean() + (y[1].sum() * 0.01 if len(tv) > 2 else 0)
                loss.backward()
                out["mlp/%s/%s/%s" % (name, method, dn)] = {
                    "y": y.detach().clone(), "gy0": y0.grad.clone(), "gt": t.grad.clone(),
                    "gp": [q.grad.clone() for q in f.parameters()], "t": t.detach().clone(), "opts": opts, "kw": kw}
    # a time-dependent field with parameters: the constant problem (problems.py:7-17), all outputs weighted
    for method in ("dopri5", "dopri8", "adaptive_heun", "fehlberg2", "rk4", "heun3", "heun2"):
        f, y0, t, _ = P.construct_problem("cpu", ode="constant", dtype=torch.float64)
        y0 = y0.requires_grad_(True)
        t = t.detach().clone().requires_grad_(True)
        y = torchdiffeq.odeint(f, y0, t, method=method)
        torch.manual_seed(0)
        w = torch.rand_like(y)
        y.backward(w)
        out["constant/%s" % method] = {"y": y.detach().clone(), "w": w, "gy0": y0.grad.clone(), "gt": t.grad.clone(),
                                       "gp": [q.grad.clone() for q in f.parameters()]}
    # tuple state (api_tests.py:28-39)
    f, y0, t, _ = P.construct_problem("cpu", ode="constant", dtype=torch.float64)
    y0 = y0.requires_grad_(True)
    t = t.detach().clone().requires_grad_(True)
    tuple_f = lambda t_, y_: (f(t_, y_[0]), f(t_, y_[1]))
    ys = torchdiffeq.odeint(tuple_f, (y0, y0 + 0.1), t, method="dopri5")
    (ys[0].sum() + 2 * ys[1][-1].sum()).backward()
    out["tuple/dopri5"] = {"gy0": y0.grad.clone(), "gt": t.grad.clone(), "gp": [q.grad.clone() for q in f.parameters()]}
    torch.save(out, os.path.join(HERE, "backprop.pt"))


def adjoint_many():
    """odeint_adjoint with the default adjoint norm on a field with 80 parameter tensors (83 norm segments)."""
    out = {}
    for norm in ("default", "seminorm"):
        f = P.DeepField(dim=6, depth=40, seed=0)
        y0 = torch.randn(16, 6, generator=torch.Generator().manual_seed(1), dtype=torch.float64).requires_grad_(True)
        t = torch.tensor([0., 0.5, 1.0], dtype=torch.float64)
        ao = {"norm": "seminorm"} if norm == "seminorm" else None
        y = torchdiffeq.odeint_adjoint(f, y0, t, method="dopri5", rtol=1e-6, atol=1e-8, adjoint_options=ao)
        (y[-1].pow(2).mean() + 0.01 * y[1].sum()).backward()
        out[norm] = {"y": y.detach().clone(), "gy0": y0.grad.clone(), "gp": [q.grad.clone() for q in f.parameters()], "t": t}
    torch.save(out, os.path.join(HERE, "adjoint_many.pt"))


def adams():
    """explicit_adams / implicit_adams (fixed_adams.py:164-228): weight tables and solutions."""
    from torchdiffeq._impl import fixed_adams as fa
    with open(os.path.join(HERE, "adams.json"), "w") as f:
        json.dump({"bashforth": [b.tolist() for b in fa._BASHFORTH_DIVISOR[:13]],
                   "moulton": [m.tolist() for m in fa._MOULTON_DIVISOR[:13]]}, f)
    out = {}
    for ode in ("constant", "sine", "linear"):
        for method in ("explicit_adams", "implicit_adams"):
            for dtype in (torch.float32, torch.float64):
                for reverse in (False, True):
                    f, y0, t, sol = P.construct_problem("cpu", ode=ode, reverse=reverse, dtype=dtype)
                    for name, opts in (("grid", None), ("step", {"step_size": 0.02}), ("cubic", {"step_size": 0.05, "interp": "cubic"})):
                        rec = Rec(f)
                        with torch.no_grad(), warnings_off():
                            y = torchdiffeq.odeint(rec, y0, t, method=method, options=opts)
                        out["%s/%s/%s/%s/%s" % (ode, method, str(dtype).split(".")[1], "rev" if reverse else "fwd", name)] = {
                            "y": y, "nfe": rec.nfe, "opts": opts, "exact": sol}
    # batched: the spiral, loose tolerances of the corrector exercised through odeint's rtol/atol
    fs = P.Spiral()
    g = torch.Generator().manual_seed(0)
    y0 = (torch.tensor([[2., 0.]]) * (1 + 0.1 * torch.rand(64, 1, generator=g)))
    t2 = torch.linspace(0., 5., 7)
    for method in ("explicit_adams", "implicit_adams"):
        for kw in ({}, {"rtol": 1e-3, "atol": 1e-4}):
            rec = Rec(fs)
            with torch.no_grad(), warnings_off():
                y = torchdiffeq.odeint(rec, y0, t2, method=method, options={"step_size": 0.01, "max_order": 6}, **kw)
            out["spiral/%s/%s" % (method, "loose" if kw else "tight")] = {"y": y, "nfe": rec.nfe, "kw": kw}
    # event handling (event_tests.py:14-49: every fixed method with step_size 0.01 and cubic interpolation)
    for ode in ("constant", "sine"):
        for method in ("explicit_adams", "implicit_adams"):
            for reverse in (False, True):
                fe, ye, te, sol = P.construct_problem("cpu", ode=ode, reverse=reverse, dtype=torch.float64)
                target = sol[2]
                rec = Rec(fe)
                with torch.no_grad(), warnings_off():
                    et, ys = torchdiffeq.odeint(rec, ye, te[0:2], event_fn=lambda t_, y_: torch.sum(y_ - target).real,
                                                method=method, options={"step_size": 0.01, "interp": "cubic"})
                out["event/%s/%s/%s" % (ode, method, "rev" if reverse else "fwd")] = {"event_t": et, "y": ys, "nfe": rec.nfe}
    torch.save(out, os.path.join(HERE, "adams.pt"))


class warnings_off:
    def __enter__(self):
        import warnings
        self.c = warnings.catch_warnings()
        self.c.__enter__()
        warnings.simplefilter("ignore")

    def __exit__(self, *a):
        return self.c.__exit__(*a)


def dense():
    """odeint_dense (odeint.py:111-157): the dense-output closure of a dopri5 solve."""
    out = {}
    for ode in ("constant", "sine", "linear"):
        for dtype in (torch.float32, torch.float64):
            f, y0, t, sol = P.construct_problem("cpu", ode=ode, dtype=dtype)
            with torch.no_grad():
                fn = torchdiffeq.odeint_dense(f, y0, t[0], t[-1], rtol=1e-6, atol=1e-8)
                qs = torch.linspace(1.0, 7.99, 23, dtype=torch.float64)
                out["%s/%s" % (ode, str(dtype).split(".")[1])] = {"q": qs, "y": torch.stack([fn(q) for q in qs])}
    torch.save(out, os.path.join(HERE, "dense.pt"))


if __name__ == "__main__":
    only = sys.argv[1:]
    if only:
        for name in only:
            globals()[name]()
        sys.exit(0)
    dump_tableaus()
    zoo()
    linear_batch()
    spiral_rk4()
    adjoint_mlp()
    detest()
    options_cases()
    events()
    dense()
    fixed_extra()
    backprop()
    adjoint_many()
    adams()
    seam_objects()
    for fn in sorted(os.listdir(HERE)):
        print(fn, os.path.getsize(os.path.join(HERE, fn)))
