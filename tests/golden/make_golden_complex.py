"""Generate tests/golden/complex.pt -- complex64 / complex128 states -- from the UNMODIFIED reference.

It is kept apart from tests/golden/make_golden.py, which writes every other golden file: running this script regenerates
complex.pt and nothing else.  The reference must be importable as `torchdiffeq`,
or its checkout named by TORCHDIFFEQ_REFERENCE:

    TORCHDIFFEQ_REFERENCE=/path/to/torchdiffeq python tests/golden/make_golden_complex.py

The problems are those of tests/complex_problems.py.  Cases:
    schrodinger     y' = -i H y, H Hermitian 4x4: reference solution and the matrix-exponential exact solution (both dtypes)
    damped          y' = W y, W complex, y [256, 16] complex64, dopri5: solution, dt sequence, accept flags, NFE
    zoo             all 14 methods x {complex64, complex128} x {forward, reverse}: solution and NFE
    tuple           a complex tuple state with per-piece tolerances; a mixed real / complex tuple
    options         step_t, jump_t, first_step, max_step
    dense           odeint_dense
    event           odeint_event on |y|^2 = c (dopri5), and with a fixed step (rk4)
    cubic           rk4 with interp='cubic'
    adjoint         odeint_adjoint gradients (y0, complex parameters, t), default norm and 'seminorm'
"""
import os
import sys
import warnings

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REFERENCE = os.environ.get("TORCHDIFFEQ_REFERENCE")
if REFERENCE:
    sys.path.insert(0, REFERENCE)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torchdiffeq                                   # noqa: E402  (the reference)
import complex_problems as CP                        # noqa: E402

assert not REFERENCE or torchdiffeq.__file__.startswith(REFERENCE), torchdiffeq.__file__
torch.set_num_threads(8)


def complex_cases():
    out = {}
    # ---- Schrodinger ----------------------------------------------------------------------------------------------
    for dt in CP.CDTYPES:
        f = CP.Schrodinger(CP.hermitian(4, 1, dt))
        y0 = CP.crandn(3, 4, seed=2, dtype=dt)
        y0 = y0 / y0.abs().pow(2).sum(-1, keepdim=True).sqrt()
        t = torch.linspace(0., 2., 9, dtype=torch.float64)
        kw = dict(rtol=1e-6, atol=1e-8) if dt == torch.complex64 else dict(rtol=1e-10, atol=1e-12)
        r = CP.Rec(f)
        sol = torchdiffeq.odeint(r, y0, t, method="dopri5", **kw)
        out[("schrodinger", str(dt))] = dict(y0=y0, t=t, sol=sol, exact=f.exact(y0.to(torch.complex128), t), kw=kw,
                                             nfe=r.nfe)
    # ---- damped batched linear field, with the dt sequence -----------------------------------------------------
    f = CP.ComplexLinear(CP.damped_weight(16, 7, torch.complex64))
    y0 = CP.crandn(256, 16, seed=8, dtype=torch.complex64)
    t = torch.linspace(0., 2., 5, dtype=torch.float64)
    r = CP.Rec(f)
    with torch.no_grad():
        sol = torchdiffeq.odeint(r, y0, t, method="dopri5", rtol=1e-5, atol=1e-7)
    out["damped"] = dict(W=f.W.detach().clone(), y0=y0, t=t, sol=sol, dts=torch.tensor(r.dts), acc=torch.tensor(r.acc),
                         nfe=r.nfe)
    # ---- every method, both dtypes, both directions ----------------------------------------------------------
    for m in CP.METHODS:
        for dt in CP.CDTYPES:
            for rev in (False, True):
                f, y0, t = CP.zoo_problem(dt, rev)
                r = CP.Rec(f)
                with torch.no_grad():
                    sol = torchdiffeq.odeint(r, y0, t, method=m, **CP.zoo_kwargs(m, dt))
                out[("zoo", m, str(dt), rev)] = dict(sol=sol, nfe=r.nfe)
    # ---- tuple states ----------------------------------------------------------------------------------------------
    for dt in CP.CDTYPES:
        f = CP.TupleField(dt)
        y0 = (CP.crandn(2, 3, seed=20, dtype=dt), CP.crandn(2, 2, seed=21, dtype=dt))
        t = torch.linspace(0., 1., 4, dtype=torch.float64)
        kw = dict(rtol=(1e-5, 1e-6), atol=(1e-7, 1e-8))
        with torch.no_grad():
            sol = torchdiffeq.odeint(f, y0, t, method="dopri5", **kw)
        out[("tuple", str(dt))] = dict(y0=y0, t=t, sol=sol, kw=kw)
    y0 = (torch.tensor([0.5, -1.0, 0.25], dtype=torch.float64), CP.crandn(2, seed=22, dtype=torch.complex128))
    t = torch.linspace(0., 1., 4, dtype=torch.float64)
    with torch.no_grad():
        sol = torchdiffeq.odeint(CP.MixedField(), y0, t, method="dopri5", rtol=1e-8, atol=1e-10)
    out["mixed"] = dict(y0=y0, t=t, sol=sol)
    # ---- step_t / jump_t / first_step / max_step ---------------------------------------------------------------
    f, y0, t = CP.zoo_problem(torch.complex128, False)
    opts = {"step_t": dict(step_t=torch.tensor([0.1, 0.33, 0.7], dtype=torch.float64)),
            "jump_t": dict(jump_t=torch.tensor([0.25, 0.6], dtype=torch.float64)),
            "first_step": dict(first_step=0.01),
            "max_step": dict(max_step=0.05)}
    for name, o in opts.items():
        r = CP.Rec(f)
        with torch.no_grad():
            sol = torchdiffeq.odeint(r, y0, t, method="dopri5", rtol=1e-8, atol=1e-10, options=o)
        out[("options", name)] = dict(sol=sol, nfe=r.nfe, options=o)
    # ---- dense output ----------------------------------------------------------------------------------------------
    with torch.no_grad():
        fn = torchdiffeq.odeint_dense(f, y0, torch.tensor(0., dtype=torch.float64), torch.tensor(1., dtype=torch.float64),
                                      rtol=1e-8, atol=1e-10)
        te = torch.tensor([0.0, 0.13, 0.5, 0.77, 1.0], dtype=torch.float64)
        out["dense"] = dict(te=te, vals=torch.stack([fn(x) for x in te]))
    # ---- events ----------------------------------------------------------------------------------------------------
    c = float((y0.abs() ** 2).sum()) * 0.5
    with torch.no_grad():
        ev_t, sol = torchdiffeq.odeint_event(f, y0, torch.tensor(0., dtype=torch.float64), event_fn=CP.event_fn_norm(c),
                                             method="dopri5", rtol=1e-8, atol=1e-10)
        out["event"] = dict(c=c, event_t=ev_t, sol=sol)
        ev_t, sol = torchdiffeq.odeint_event(f, y0, torch.tensor(0., dtype=torch.float64), event_fn=CP.event_fn_norm(c),
                                             method="rk4", options=dict(step_size=0.05), atol=1e-9)
        out["event_fixed"] = dict(c=c, event_t=ev_t, sol=sol)
    # ---- cubic interpolation -----------------------------------------------------------------------------------
    with torch.no_grad():
        sol = torchdiffeq.odeint(f, y0, torch.tensor([0., 0.123, 0.5, 0.91], dtype=torch.float64), method="rk4",
                                 options=dict(step_size=0.1, interp="cubic"))
    out["cubic"] = dict(t=torch.tensor([0., 0.123, 0.5, 0.91], dtype=torch.float64), sol=sol)
    # ---- adjoint ---------------------------------------------------------------------------------------------------
    for norm in ("default", "seminorm"):
        f = CP.ComplexLinear(CP.damped_weight(4, 3, torch.complex128), bias=True)
        y0 = CP.crandn(8, 4, seed=5, dtype=torch.complex128).requires_grad_(True)
        t = torch.linspace(0., 1., 4, dtype=torch.float64).requires_grad_(True)
        ao = {} if norm == "default" else dict(norm="seminorm")
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            sol = torchdiffeq.odeint_adjoint(f, y0, t, method="dopri5", rtol=1e-9, atol=1e-11, adjoint_options=ao)
            loss = (sol.abs() ** 2).sum()
            loss.backward()
        out[("adjoint", norm)] = dict(sol=sol.detach(), y0_grad=y0.grad.clone(), t_grad=t.grad.clone(),
                                      W_grad=f.W.grad.clone(), b_grad=f.b.grad.clone())
    return out


def main():
    out = complex_cases()
    path = os.path.join(HERE, "complex.pt")
    torch.save(out, path)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
