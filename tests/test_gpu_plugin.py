"""The registry-seam plug-in (torchdiffeq_b200/plugin.py) driven through the caller side of the reference's seam:
the plug-in replaces only SOLVERS[method] (odeint.py:19-46, :92-97; adjoint.py:4 shares the dict) and the front end
keeps its odeint / odeint_adjoint, _check_inputs, tuple plumbing, event wrappers and adjoint.  That front end is
tests/seam_frontend.py, a stand-in that hands the solver exactly what the reference's does.  Mirrors the
reference's tests/odeint_tests.py, api_tests.py, norm_tests.py, event_tests.py and gradient_tests.py on CUDA tensors,
against the reference's CPU goldens."""
import os

import pytest
import torch

import problems as P

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
G = os.path.join(HERE, "golden")
ld = lambda name: torch.load(os.path.join(G, name), weights_only=False)
DEV = "cuda:0"


@pytest.fixture(scope="module")
def front():
    """(odeint, odeint_adjoint) of the seam's caller side with the plug-in registered for the duration of the module."""
    import seam_frontend as sf
    from torchdiffeq_b200 import plugin
    replaced = plugin.register(sf.SOLVERS)
    yield sf.odeint, sf.odeint_adjoint
    plugin.unregister(replaced, sf.SOLVERS)


class Counted(torch.nn.Module):
    def __init__(self, f):
        super().__init__()
        self.f, self.nfe = f, 0

    def forward(self, t, y):
        self.nfe += 1
        return self.f(t, y)


ZOO = ld("zoo.pt")
FIXED = ("rk4", "euler", "midpoint", "heun2", "heun3")
STAGES = {"dopri5": 6, "dopri8": 13, "tsit5": 6, "bosh3": 3, "fehlberg2": 2, "adaptive_heun": 1}


@pytest.mark.parametrize("key", sorted(ZOO))
def test_seam_zoo(front, key):
    """tests/odeint_tests.py:17-58 through the seam: every registered method, both dtypes, both directions; the
    default is the reference's exact call sequence, so func's own NFE counter equals 2 + S*attempts."""
    odeint, _ = front
    ode, method, dt, direction = key.split("/")
    dtype = getattr(torch, dt)
    case = ZOO[key]
    f, y0, t, sol = P.construct_problem(DEV, ode=ode, reverse=direction == "rev", dtype=dtype)
    cf = Counted(f)
    with torch.no_grad():
        y = odeint(cf, y0, t, method=method, **case["kw"])
    assert y.shape == sol.shape and y.dtype == dtype and y.is_cuda
    eps = {"constant": 3e-4, "sine": 3e-4, "linear": 2e-3, "exp": 5e-2}[ode]
    if method in ("adaptive_heun", "fehlberg2", "bosh3"):
        eps = {"constant": 1e-3, "sine": 5e-3, "linear": 2e-3, "exp": 5e-2}[ode]
    if method in FIXED:
        eps = 1e-5
    assert ((sol - y) / sol).abs().max() < eps
    tol = 5e-4 if dtype == torch.float32 else 1e-6
    assert torch.allclose(y.cpu(), case["y"], rtol=tol, atol=tol * 1e-2)
    if method in FIXED:
        assert cf.nfe == case["nfe"]
    else:
        assert (cf.nfe - 2) % STAGES[method] == 0
        assert abs(cf.nfe - case["nfe"]) <= max(4 * STAGES[method], case["nfe"] // 4) or dtype == torch.float32


def test_seam_tuple_state_and_options(front):
    """api_tests.py:12-26 (tuple == tensor), tuple tolerances (misc.py:115-123) and the anonymous norm closure the
    seam hands over for tuple states (compatibility path), against the reference's CPU goldens."""
    odeint, _ = front
    case = ld("options.pt")["tuple"]
    A = P.skew_matrix(6, torch.float64).to(DEV)

    def tf(t_, state):
        a, b = state
        return (a @ A.t(), -0.5 * b + a[:, :2].sum())
    ya, yb, tt = case["ya"].to(DEV), case["yb"].to(DEV), case["t"].to(DEV)
    with torch.no_grad():
        sol = odeint(tf, (ya, yb), tt, method="dopri5", rtol=1e-6, atol=1e-8)
        sol_v = odeint(tf, (ya, yb), tt, method="dopri5", rtol=(1e-6, 1e-4), atol=(1e-8, 1e-7))
    for got, want in zip(sol, case["sol"]):
        assert torch.allclose(got.cpu(), want, rtol=1e-5, atol=1e-7)
    for got, want in zip(sol_v, case["sol_vtol"]):
        assert torch.allclose(got.cpu(), want, rtol=1e-4, atol=1e-6)
    # step_t / min_step known answers of odeint_tests.py:251-268 through the seam
    for key in ("min_step", "max_step", "step_t", "first_step", "factors"):
        c = ld("options.pt")[key]
        f, y0, t, _ = P.construct_problem(DEV, ode="linear", dtype=torch.float64)
        with torch.no_grad():
            y = odeint(f, y0, t, method="dopri5", options=dict(c["opts"]))
        assert torch.allclose(y.cpu(), c["y"], rtol=1e-6, atol=1e-8), key
        if key in ("min_step", "max_step", "step_t"):
            assert f.nfe == c["nfe"], key


def test_seam_custom_norm_and_callbacks(front):
    """norm_tests.py style: a user norm reaches the solver through options['norm']; callbacks arrive as attributes
    of the wrapped func (misc.py:311-332) and fire in the reference's order and number."""
    odeint, _ = front
    f, y0, t, _ = P.construct_problem(DEV, ode="linear", dtype=torch.float64)
    calls = {"n": 0}

    def norm(x):
        calls["n"] += 1
        return x.abs().max()
    with torch.no_grad():
        y_inf = odeint(f, y0, t, method="dopri5", options={"norm": norm})
        f2, _, _, sol = P.construct_problem(DEV, ode="linear", dtype=torch.float64)
        y_rms = odeint(f2, y0, t, method="dopri5")
    assert calls["n"] > 0 and f.nfe > f2.nfe                      # the max norm is stricter than the RMS norm
    assert torch.allclose(y_inf, y_rms, rtol=1e-5, atol=1e-7)

    class CB(torch.nn.Module):
        def __init__(self, g):
            super().__init__()
            self.g, self.steps, self.acc, self.rej = g, 0, 0, 0

        def forward(self, t_, y_):
            return self.g(t_, y_)

        def callback_step(self, t0, y0_, dt):
            self.steps += 1

        def callback_accept_step(self, t0, y0_, dt):
            self.acc += 1

        def callback_reject_step(self, t0, y0_, dt):
            self.rej += 1
    f3, _, _, _ = P.construct_problem(DEV, ode="linear", dtype=torch.float64)
    cb = CB(f3)
    with torch.no_grad():
        odeint(cb, y0, t, method="dopri5")
    assert cb.steps == cb.acc + cb.rej and 2 + 6 * cb.steps == f3.nfe          # odeint_tests.py:376-386


EV = ld("events.pt")


@pytest.mark.parametrize("key", sorted(k for k in EV if k.count("/") == 3 and k.split("/")[1] in ("dopri5", "bosh3")))
def test_seam_events(front, key):
    """event_tests.py:14-49 through solver.integrate_until_event (odeint.py:97)."""
    odeint, _ = front
    ode, method, dt, direction = key.split("/")
    dtype = getattr(torch, dt)
    case = EV[key]
    f, y0, t, sol = P.construct_problem(DEV, ode=ode, reverse=direction == "rev", dtype=dtype)
    target = sol[2]
    with torch.no_grad():
        et, ys = odeint(f, y0, t[0:2], event_fn=lambda t_, y_: torch.sum(y_ - target).real, method=method)
    assert ((sol[2] - ys[-1]) / sol[2]).abs().max() < 1e-4 and abs((t[2] - et) / t[2]) < 1e-4
    assert torch.allclose(ys.cpu(), case["y"], rtol=1e-4, atol=1e-6)
    fx = ld("fixed_extra.pt")["event/%s/rk4/%s/%s/cubic" % (ode, dt, direction)]
    f, y0, t, sol = P.construct_problem(DEV, ode=ode, reverse=direction == "rev", dtype=dtype)
    with torch.no_grad():
        et, ys = odeint(f, y0, t[0:2], event_fn=lambda t_, y_: torch.sum(y_ - target).real, method="rk4",
                        options={"step_size": 0.01, "interp": "cubic"})
    assert torch.allclose(ys.cpu(), fx["y"], rtol=2e-5, atol=1e-6)
    assert abs(float(et) - float(fx["event_t"])) <= 2e-5 * abs(float(fx["event_t"]))


@pytest.mark.parametrize("key", sorted(ld("adjoint_mlp.pt")))
def test_seam_adjoint_gradients(front, key):
    """gradient_tests.py:34-86 style: odeint_adjoint with our solver registered -- its backward
    instantiates SOLVERS[method] once per output interval with the augmented flat state and an anonymous norm
    closure (adjoint.py:134-138, :247-288); gradients against the CPU reference's to 1e-4 relative."""
    _, odeint_adjoint = front
    case = ld("adjoint_mlp.pt")[key]
    name, norm, dt = key.split("/")
    dtype = getattr(torch, dt)
    f = P.MLPField(dim=8, hidden=16, seed=0, dtype=dtype).to(DEV)
    y0 = torch.randn(32, 8, generator=torch.Generator().manual_seed(1)).to(dtype).to(DEV).requires_grad_(True)
    t = case["t"].to(DEV)
    ao = {"norm": "seminorm"} if norm == "seminorm" else None
    y = odeint_adjoint(f, y0, t, method="dopri5", rtol=1e-6, atol=1e-8, adjoint_options=ao)
    loss = y[-1].pow(2).mean() + (y[1].sum() * 0.01 if len(t) > 2 else 0)
    loss.backward()
    tol = 1e-4
    assert torch.allclose(y.detach().cpu(), case["y"], rtol=1e-4, atol=1e-6)
    want = case["gy0"]
    assert (y0.grad.cpu() - want).abs().max() <= tol * want.abs().max()
    for q, w in zip(f.parameters(), case["gp"]):
        assert (q.grad.cpu() - w).abs().max() <= tol * max(w.abs().max(), 1e-6)


def test_seam_graph_mode_opt_in(front):
    """options={'graph': True} through the seam: captured step body inside the device loop, same result."""
    odeint, _ = front
    f = P.BatchedLinear(128).to(DEV)
    y0 = torch.randn(512, 128, generator=torch.Generator().manual_seed(1)).to(DEV)
    t = torch.linspace(0, 2, 5).to(DEV)
    with torch.no_grad():
        a = odeint(f, y0, t, method="dopri5", rtol=1e-5, atol=1e-7)
        b = odeint(f, y0, t, method="dopri5", rtol=1e-5, atol=1e-7, options={"graph": True})
    assert torch.equal(a, b)


@pytest.mark.parametrize("method", ["explicit_adams", "implicit_adams"])
def test_seam_adams(front, method):
    """The Adams methods through the seam (odeint.py:31-42 registers AdamsBashforth / AdamsBashforthMoulton; the
    constructor receives odeint's rtol/atol, fixed_adams.py:167-175)."""
    odeint, _ = front
    AD = ld("adams.pt")
    for direction in ("fwd", "rev"):
        case = AD["linear/%s/float64/%s/step" % (method, direction)]
        f, y0, t, _ = P.construct_problem(DEV, ode="linear", reverse=direction == "rev", dtype=torch.float64)
        with torch.no_grad():
            y = odeint(f, y0, t, method=method, options=case["opts"])
        want = case["y"]
        if float(want.abs().max()) < 1e3:                    # the explicit method is unstable in reverse on this problem
            assert torch.allclose(y.cpu(), want, rtol=1e-9, atol=1e-9)
        else:
            assert bool(torch.isfinite(y).all()) == bool(torch.isfinite(want).all())
            assert torch.allclose(y[:2].cpu(), want[:2], rtol=1e-9, atol=1e-9)
        assert f.nfe == case["nfe"]
