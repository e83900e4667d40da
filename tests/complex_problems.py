"""Seeded complex-valued test problems, shared by tests/golden/make_golden_complex.py (which runs them through the
reference) and the complex-state tests (which run them through torchdiffeq_b200 and the oracle)."""
import torch

CDTYPES = (torch.complex64, torch.complex128)


def hermitian(n, seed, dtype=torch.complex128):
    g = torch.Generator().manual_seed(seed)
    a = torch.randn(n, n, 2, generator=g, dtype=torch.float64)
    a = torch.view_as_complex(a)
    return ((a + a.mH) / 2).to(dtype)


def crandn(*shape, seed, dtype=torch.complex128):
    g = torch.Generator().manual_seed(seed)
    return torch.view_as_complex(torch.randn(*shape, 2, generator=g, dtype=torch.float64)).to(dtype)


class Schrodinger(torch.nn.Module):
    """y' = -i H y for a Hermitian H (rows of y are states): the norm |y| is conserved and y(t) = exp(-i H t) y0."""

    def __init__(self, H):
        super().__init__()
        self.register_buffer("H", H)

    def forward(self, t, y):
        return -1j * (y @ self.H.T)

    def exact(self, y0, t):
        H = self.H.to(y0.dtype)
        return torch.stack([y0 @ torch.linalg.matrix_exp(-1j * H * float(ti)).T for ti in t])


def damped_weight(d, seed, dtype=torch.complex128, damping=0.5):
    """W = -i H - damping I: oscillatory and decaying."""
    H = hermitian(d, seed, torch.complex128) / d ** 0.5
    return (-1j * H - damping * torch.eye(d, dtype=torch.complex128)).to(dtype)


class ComplexLinear(torch.nn.Module):
    """func = y @ W^T with a complex parameter W (and an optional complex bias), so that odeint_adjoint has complex
    parameters to differentiate."""

    def __init__(self, W, bias=False):
        super().__init__()
        self.W = torch.nn.Parameter(W.clone())
        self.b = torch.nn.Parameter(torch.full((W.shape[0],), 0.1 + 0.05j, dtype=W.dtype)) if bias else None

    def forward(self, t, y):
        out = y @ self.W.T
        if self.b is not None:
            out = out + self.b * torch.cos(t)
        return out


class TupleField(torch.nn.Module):
    """A tuple state (a, b): a' = W a + 0.1 b[..., :1], b' = -i b * (1 + t) - 0.2 a[..., :2] (two pieces of different
    shapes, coupled; t enters so that a wrong time argument shows)."""

    def __init__(self, dtype):
        super().__init__()
        self.register_buffer("W", damped_weight(3, 11, dtype))

    def forward(self, t, y):
        a, b = y
        return a @ self.W.T + 0.1 * b[..., :1], -1j * b * (1 + t) - 0.2 * a[..., :2]


class MixedField(torch.nn.Module):
    """A tuple whose first piece is REAL and second complex: x' = -x + Re(z[..., :1]), z' = (-0.3 - 2i) z + x[..., :1]."""

    def forward(self, t, y):
        x, z = y
        return -x + z[..., :1].real, (-0.3 - 2j) * z + x[..., :1]


class Rec(torch.nn.Module):
    """Counts NFE and records the accepted / rejected dt sequence through the solver callbacks."""

    def __init__(self, f):
        super().__init__()
        self.f, self.nfe, self.dts, self.acc = f, 0, [], []

    def forward(self, t, y):
        self.nfe += 1
        return self.f(t, y)

    def callback_accept_step(self, t0, y0, dt):
        self.dts.append(float(dt))
        self.acc.append(True)

    def callback_reject_step(self, t0, y0, dt):
        self.dts.append(float(dt))
        self.acc.append(False)


ADAPTIVE = ("dopri5", "dopri8", "tsit5", "bosh3", "fehlberg2", "adaptive_heun")
FIXED = ("rk4", "euler", "midpoint", "heun2", "heun3")
ADAMS = ("explicit_adams", "implicit_adams", "fixed_adams")
METHODS = ADAPTIVE + FIXED + ADAMS


def zoo_problem(dtype, reverse):
    """The per-method case: a [8, 4] damped complex linear field over 5 output times."""
    f = ComplexLinear(damped_weight(4, 3, dtype))
    y0 = crandn(8, 4, seed=5, dtype=dtype)
    t = torch.linspace(0., 1., 5, dtype=torch.float64)
    if reverse:
        t = t.flip(0)
    return f, y0, t


def zoo_kwargs(method, dtype):
    if method in ADAPTIVE:
        return dict(rtol=1e-6, atol=1e-8) if dtype == torch.complex64 else dict(rtol=1e-9, atol=1e-11)
    if method == "explicit_adams":
        # The order-12 Adams-Bashforth predictor is not stable on this problem at h = 0.05: it amplifies rounding so
        # that a one-ulp change of func's output moves the reference's own complex64 result by ~1e-3, and no
        # implementation could reproduce that golden.  At order 4 a one-ulp change moves it by ~2e-7.
        return dict(options=dict(step_size=0.05, max_order=4))
    return dict(options=dict(step_size=0.05))


def event_fn_norm(c):
    """|y|^2 = c (sum over the whole state)."""
    def ev(t, y):
        return (y.abs() ** 2).sum() - c
    return ev
