"""Complex64 / complex128 states on the GPU: the complex element rule of the error-norm kernel against torch on the same
device, whole solves of every method against the reference's complex goldens (tests/golden/complex.pt), every interface
a complex state flows through, and the explicit errors of what is not implemented."""
import ctypes as C
import os
import warnings

import pytest
import torch

import complex_problems as CP
from oracle import ode_oracle as O

pytestmark = pytest.mark.gpu

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DEV = "cuda:0"
TOL = {torch.complex64: dict(rtol=1e-4, atol=1e-6), torch.complex128: dict(rtol=1e-5, atol=1e-7)}


def tdq():
    import torchdiffeq_b200
    return torchdiffeq_b200


@pytest.fixture(scope="module")
def gold():
    return torch.load(os.path.join(G, "complex.pt"), weights_only=False)


def cu(x):
    if isinstance(x, tuple):
        return tuple(cu(v) for v in x)
    return x.to(DEV)


def close(got, want, dtype, scale=1.0):
    tol = TOL[dtype]
    if isinstance(want, tuple):
        for g, w in zip(got, want):
            torch.testing.assert_close(g.cpu(), w, rtol=tol["rtol"] * scale, atol=tol["atol"] * scale)
        return
    torch.testing.assert_close(got.cpu(), want, rtol=tol["rtol"] * scale, atol=tol["atol"] * scale)


# ---- kernel level ------------------------------------------------------------------------------------------------------
def _engine(dtype, n, segs=None, method="dopri5", vtol=False, dt=0.0371, t0=0.5, rtol=1e-3, atol=1e-6):
    from torchdiffeq_b200 import _lib
    from torchdiffeq_b200._engine import AdaptiveEngine, _stream
    dev = torch.device(DEV)
    kw = {}
    if vtol:
        g = torch.Generator().manual_seed(77)
        kw = dict(rtol_vec=(torch.rand(n, generator=g, dtype=torch.float64) * 1e-3 + 1e-4).to(dev),
                  atol_vec=(torch.rand(n, generator=g, dtype=torch.float64) * 1e-6 + 1e-7).to(dev))
    eng = AdaptiveEngine(lambda t, y: y, n, dtype, dev, method, rtol=rtol, atol=atol, first_step=dt, segs=segs, **kw)
    eng.t_out = torch.tensor([t0, 100.0], dtype=torch.float64, device=dev)
    eng.solution = torch.zeros(2, n, dtype=dtype, device=dev)
    _lib.check(eng.lib.tdq_ctrl_init(eng.ctrl.data_ptr(), C.byref(eng.tab), C.byref(eng.opt), eng.t_out.data_ptr(),
                                     t0, 2, eng.mbox_dev, _stream()))
    _lib.check(eng.lib.tdq_set_first_step(eng.ctrl.data_ptr(), float(dt), _stream()))
    _lib.check(eng.lib.tdq_prepare_attempt(eng.ctrl.data_ptr(), eng.rt_code, None, _stream()))
    return eng, _lib, _stream


def _norm_commit(eng, _lib, _stream, errp, k_last, y0, y1, q_out=None):
    _lib.check(eng.lib.tdq_error_norm_commit(
        eng.ctrl.data_ptr(), eng.dt_code, errp.data_ptr(), k_last.data_ptr(), y0.data_ptr(), y1.data_ptr(),
        eng.rtol_vec.data_ptr() if eng.rtol_vec is not None else None,
        eng.atol_vec.data_ptr() if eng.atol_vec is not None else None,
        eng.norm_table.data_ptr() if eng.norm_table is not None else None, eng.n_chunks, eng.table_aligned, eng.n_seg,
        eng.n, eng.partials.data_ptr(), eng.norm_out.data_ptr(), q_out.data_ptr() if q_out is not None else None,
        _stream()))


def _inputs(dtype, n, seed):
    err, k, y0, y1 = (CP.crandn(n, seed=seed + i, dtype=dtype).to(DEV) for i in range(4))
    return err * 1e-4, k, y0, y1


def _torch_q(eng, dtype, errp, k_last, y0, y1, method="dopri5", dt=0.0371):
    """misc.py:80-82 in torch ops on the GPU: err = err_pre + k_S * fl(dt * e_S) (FSAL tableau), q = err / tol."""
    R = dtype.to_real()
    ct = O._cast_tableau(O.tableau(method), R)
    dtT = torch.tensor(dt, dtype=torch.float64).to(R)
    eS = (dtT * ct["c_err"])[-1].to(DEV)
    err = errp + k_last * eS
    if eng.rtol_vec is not None:
        tol = eng.atol_vec + eng.rtol_vec * torch.max(y0.abs(), y1.abs())
    else:
        tol = eng.opt.atol + eng.opt.rtol * torch.max(y0.abs(), y1.abs())
    return err / tol


def _ulps(a, b):
    """Largest distance in units in the last place between the components of two complex tensors."""
    ra, rb = torch.view_as_real(a).reshape(-1), torch.view_as_real(b).reshape(-1)
    same = ra == rb
    it = torch.int32 if ra.dtype == torch.float32 else torch.int64
    ia, ib = ra.view(it).to(torch.int64), rb.view(it).to(torch.int64)
    d = (ia - ib).abs()
    d[same] = 0
    return int(d.max())


@pytest.mark.parametrize("dtype", CP.CDTYPES, ids=str)
@pytest.mark.parametrize("vtol", [False, True])
def test_writeq_matches_torch(dtype, vtol):
    """err/tol of the WRITEQ path against torch's `err / tol` on the same device and inputs."""
    n = 4099
    eng, _lib, _stream = _engine(dtype, n, vtol=vtol)
    errp, k, y0, y1 = _inputs(dtype, n, 3)
    qdt = torch.complex128 if vtol else dtype
    q = torch.zeros(n, dtype=qdt, device=DEV)
    _norm_commit(eng, _lib, _stream, errp, k, y0, y1, q_out=q)
    want = _torch_q(eng, dtype, errp, k, y0, y1)
    assert want.dtype == qdt
    u = _ulps(q, want)
    print("\nWRITEQ %s vtol=%s: max ulp difference vs torch err/tol = %d" % (dtype, vtol, u))
    assert u <= 1
    m = want.abs()
    ref = (m * m).double().sum()
    torch.testing.assert_close(eng.norm_out[0], ref, rtol=1e-12, atol=0)
    assert float(eng.norm_out[1]) == 0.0


@pytest.mark.parametrize("dtype", CP.CDTYPES, ids=str)
@pytest.mark.parametrize("layout", ["single", "multi"])
@pytest.mark.parametrize("vtol", [False, True])
def test_norm_modes_against_float64(dtype, layout, vtol):
    """MODE 0 (error ratio + commit), MODE 1 (x/scale) and MODE 2 ((x - x2)/scale) sums for one segment and for a chunk
    table, against a float64 evaluation; reproducible bit for bit; the commit writes the candidate pair; non-finite
    elements counted once per complex element."""
    n = 9001
    segs = None if layout == "single" else [(0, 3), (4, 2500), (2600, 6000), (8700, 250)]
    eng, _lib, _stream = _engine(dtype, n, segs=segs, vtol=vtol)
    segs = segs or [(0, n)]
    errp, k, y0, y1 = _inputs(dtype, n, 11)
    y1[17] = complex(float("inf"), 0.0)
    y1[18] = complex(0.0, float("nan"))
    _norm_commit(eng, _lib, _stream, errp, k, y0, y1)
    out0 = eng.norm_out.clone()
    torch.cuda.synchronize()
    bits = lambda z: torch.view_as_real(z).view(torch.int32 if dtype == torch.complex64 else torch.int64)
    assert torch.equal(bits(eng.ybuf[1]), bits(y1)) and torch.equal(bits(eng.kbuf[1]), bits(k))   # candidate commit
    assert float(out0[-1]) == 2.0                                                  # two non-finite complex elements
    q = _torch_q(eng, dtype, errp, k, y0, y1)
    m = q.abs()
    sq = (m * m).double()
    for s, (o, l) in enumerate(segs):
        want = sq[o:o + l].sum()
        if torch.isfinite(want):
            torch.testing.assert_close(out0[s], want, rtol=1e-12, atol=0)
    _norm_commit(eng, _lib, _stream, errp, k, y0, y1)
    assert torch.equal(eng.norm_out.view(torch.int64), out0.view(torch.int64))   # deterministic, bit for bit
    # MODE 1 / MODE 2 (misc.py:55-58, :69)
    x, x2 = CP.crandn(n, seed=50, dtype=dtype).to(DEV), CP.crandn(n, seed=51, dtype=dtype).to(DEV)
    if eng.rtol_vec is not None:
        scale = eng.atol_vec + y0.abs() * eng.rtol_vec
    else:
        scale = eng.opt.atol + y0.abs() * eng.opt.rtol
    for xx, want_q in ((None, x / scale), (x2, (x - x2) / scale)):
        out = torch.zeros(eng.n_seg + 1, dtype=torch.float64, device=DEV)
        _lib.check(eng.lib.tdq_scaled_sumsq(
            eng.ctrl.data_ptr(), eng.dt_code, x.data_ptr(), xx.data_ptr() if xx is not None else None, y0.data_ptr(),
            eng.rtol_vec.data_ptr() if eng.rtol_vec is not None else None,
            eng.atol_vec.data_ptr() if eng.atol_vec is not None else None,
            eng.norm_table.data_ptr() if eng.norm_table is not None else None, eng.n_chunks, eng.table_aligned,
            eng.n_seg, n, eng.partials.data_ptr(), out.data_ptr(), _stream()))
        m = want_q.abs()
        sq = (m * m).double()
        for s, (o, l) in enumerate(segs):
            torch.testing.assert_close(out[s], sq[o:o + l].sum(), rtol=1e-12, atol=0)


# ---- whole solves ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("dtype", CP.CDTYPES, ids=str)
@pytest.mark.parametrize("method", CP.METHODS)
def test_every_method_against_golden(gold, method, dtype, reverse):
    f, y0, t = CP.zoo_problem(dtype, reverse)
    r = CP.Rec(f).to(DEV)
    with torch.no_grad(), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        y = tdq().odeint(r, cu(y0), cu(t), method=method, **CP.zoo_kwargs(method, dtype))
    case = gold[("zoo", method, str(dtype), reverse)]
    assert y.dtype == dtype and y.shape == case["sol"].shape
    close(y, case["sol"], dtype)
    if method in CP.ADAPTIVE:
        return
    nfe = tdq().last_stats()["nfe"]                               # func evaluations issued, graph replays included
    if dtype == torch.complex64 and method in ("implicit_adams", "fixed_adams"):
        # The corrector stops when max |dy_old - dy| / (atol + rtol max(|dy_old|, |dy|)) < 1 with odeint's default
        # rtol = 1e-7, about one float32 ulp: whether an iteration more is taken is decided by rounding, and func (a
        # complex64 matmul) rounds differently on the GPU than in the reference's CPU run.  The solution is checked above;
        # test_complex64_corrector_follows_func_rounding checks the iteration count against the oracle run on the GPU.
        print("\n%s %s reverse=%s: NFE %d, reference %d" % (method, dtype, reverse, nfe, case["nfe"]))
        assert abs(nfe - case["nfe"]) <= 2
    else:
        assert nfe == case["nfe"]


@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("method", ["implicit_adams", "fixed_adams"])
def test_complex64_corrector_follows_func_rounding(method, reverse):
    """The oracle (the reference's operation order in torch ops) run with func on the GPU takes the same corrector
    iterations and reaches the same solution as the engine: an NFE difference to the CPU golden comes from func's rounding."""
    dtype = torch.complex64
    f, y0, t = CP.zoo_problem(dtype, reverse)
    f = f.to(DEV)
    with torch.no_grad(), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        y = tdq().odeint(f, cu(y0), cu(t), method=method, **CP.zoo_kwargs(method, dtype))
        nfe = tdq().last_stats()["nfe"]
        r = CP.Rec(f)
        sgn = -1.0 if reverse else 1.0
        grid = torch.arange(0, 21, dtype=torch.float64) * 0.05 + t[0] * sgn        # solvers.py:85-96, ascending time
        grid[-1] = t[-1] * sgn
        want = O.odeint_adams(r, cu(y0), t, implicit=True, grid=grid * sgn)
    print("\n%s reverse=%s: engine NFE %d, oracle-on-GPU NFE %d" % (method, reverse, nfe, r.nfe))
    assert nfe == r.nfe
    torch.testing.assert_close(y.cpu(), want.cpu(), rtol=1e-5, atol=1e-6)


def test_damped_batch_dt_sequence(gold):
    """The [256, 16] complex64 case: solution, and where the step sequence matches the reference's, the NFE too."""
    case = gold["damped"]
    f = CP.Rec(CP.ComplexLinear(case["W"])).to(DEV)
    with torch.no_grad():
        y = tdq().odeint(f, cu(case["y0"]), cu(case["t"]), method="dopri5", rtol=1e-5, atol=1e-7)
    close(y, case["sol"], torch.complex64)
    # func (a complex64 matmul) rounds differently on the GPU, and at rtol=1e-5 the complex64 error estimate is partly
    # rounding noise, so the step sequence may differ; where it is the same, so is the number of evaluations
    dts = torch.tensor(f.dts, dtype=torch.float64)
    want = case["dts"].to(torch.float64)
    assert abs(len(dts) - len(want)) <= 2
    same = len(dts) == len(want) and torch.allclose(dts, want, rtol=1e-6, atol=0)
    print("\ndamped complex64: %d attempts (reference %d), step sequence %s, NFE %d (reference %d)"
          % (len(dts), len(want), "the same: flags and NFE compared" if same else "different: flags and NFE not compared",
             f.nfe, case["nfe"]))
    if same:
        assert torch.equal(torch.tensor(f.acc), case["acc"])
        assert f.nfe == case["nfe"]


@pytest.mark.parametrize("dtype", CP.CDTYPES, ids=str)
def test_schrodinger_norm_and_matrix_exp(gold, dtype):
    case = gold[("schrodinger", str(dtype))]
    f = CP.Schrodinger(CP.hermitian(4, 1, dtype)).to(DEV)
    with torch.no_grad():
        y = tdq().odeint(f, cu(case["y0"]), cu(case["t"]), method="dopri5", **case["kw"])
    close(y, case["sol"], dtype)
    norms = y.abs().pow(2).sum(-1).double().cpu()
    drift = (norms - 1).abs().max().item()
    assert drift < (1e-4 if dtype == torch.complex64 else 1e-8), drift
    exact = case["exact"]
    err = (y.cpu().to(torch.complex128) - exact).abs().max().item()
    assert err < (1e-4 if dtype == torch.complex64 else 1e-8), err


@pytest.mark.parametrize("dtype", CP.CDTYPES, ids=str)
def test_execution_modes_bitwise(dtype):
    """Lock step, run ahead and the captured graph inside the device-side loop give the same bits."""
    f, y0, t = CP.zoo_problem(dtype, False)
    f = f.to(DEV)
    y0 = cu(CP.crandn(512, 4, seed=9, dtype=dtype))
    outs = {}
    for name, o in {"lockstep": dict(run_ahead=0, graph=False), "eager": dict(run_ahead=2, graph=False),
                    "loop": dict(run_ahead=2, graph=True, device_loop=True, cache=False)}.items():
        with torch.no_grad():
            outs[name] = tdq().odeint(f, y0, cu(t), method="dopri5", rtol=1e-6, atol=1e-8, options=o).clone()
    assert torch.equal(outs["lockstep"], outs["eager"])
    assert torch.equal(outs["lockstep"], outs["loop"])


# ---- interfaces --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", CP.CDTYPES, ids=str)
def test_tuple_state_per_piece_tol(gold, dtype):
    case = gold[("tuple", str(dtype))]
    with torch.no_grad():
        y = tdq().odeint(CP.TupleField(dtype).to(DEV), cu(case["y0"]), cu(case["t"]), method="dopri5", **case["kw"])
    assert all(p.dtype == dtype for p in y)
    close(y, case["sol"], dtype)


def test_mixed_tuple_is_promoted(gold):
    case = gold["mixed"]
    with torch.no_grad():
        y = tdq().odeint(CP.MixedField(), cu(case["y0"]), cu(case["t"]), method="dopri5", rtol=1e-8, atol=1e-10)
    assert [p.dtype for p in y] == [torch.complex128, torch.complex128]
    assert [p.dtype for p in case["sol"]] == [torch.complex128, torch.complex128]
    close(y, case["sol"], torch.complex128)


def test_vector_tolerances_per_complex_element():
    """A per-element tolerance tensor equal to the scalar everywhere gives the scalar solve's result."""
    f, y0, t = CP.zoo_problem(torch.complex128, False)
    f, y0, t = f.to(DEV), cu(y0), cu(t)
    with torch.no_grad():
        a = tdq().odeint(f, y0, t, method="dopri5", rtol=1e-7, atol=1e-9)
        b = tdq().odeint(f, y0, t, method="dopri5", rtol=torch.full(y0.shape, 1e-7, dtype=torch.float64, device=DEV),
                         atol=torch.full(y0.shape, 1e-9, dtype=torch.float64, device=DEV))
    close(b, a.cpu(), torch.complex128, scale=1e-3)


@pytest.mark.parametrize("name", ["step_t", "jump_t", "first_step", "max_step"])
def test_options_against_golden(gold, name):
    case = gold[("options", name)]
    f, y0, t = CP.zoo_problem(torch.complex128, False)
    r = CP.Rec(f).to(DEV)
    o = {k: (cu(v) if torch.is_tensor(v) else v) for k, v in case["options"].items()}
    with torch.no_grad():
        y = tdq().odeint(r, cu(y0), cu(t), method="dopri5", rtol=1e-8, atol=1e-10, options=o)
    close(y, case["sol"], torch.complex128)


def test_callbacks_see_complex_state():
    f, y0, t = CP.zoo_problem(torch.complex64, False)
    seen = []

    class F(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.f = f

        def forward(self, t_, y):
            assert t_.dtype == torch.float32
            return self.f(t_, y)

        def callback_step(self, t0, y, dt):
            seen.append((y.dtype, tuple(y.shape)))

    with torch.no_grad():
        tdq().odeint(F().to(DEV), cu(y0), cu(t), method="dopri5", rtol=1e-5, atol=1e-7)
    assert seen and all(s == (torch.complex64, (8, 4)) for s in seen)


def test_dense_output(gold):
    case = gold["dense"]
    f, y0, _ = CP.zoo_problem(torch.complex128, False)
    with torch.no_grad():
        fn = tdq().odeint_dense(f.to(DEV), cu(y0), torch.tensor(0., dtype=torch.float64, device=DEV),
                                torch.tensor(1., dtype=torch.float64, device=DEV), rtol=1e-8, atol=1e-10)
        vals = torch.stack([fn(x) for x in case["te"]])
    close(vals, case["vals"], torch.complex128)


@pytest.mark.parametrize("kind", ["event", "event_fixed"])
def test_events_on_modulus(gold, kind):
    case = gold[kind]
    f, y0, _ = CP.zoo_problem(torch.complex128, False)
    kw = dict(method="dopri5", rtol=1e-8, atol=1e-10) if kind == "event" else \
        dict(method="rk4", options=dict(step_size=0.05), atol=1e-9)
    with torch.no_grad():
        ev_t, sol = tdq().odeint_event(f.to(DEV), cu(y0), torch.tensor(0., dtype=torch.float64, device=DEV),
                                       event_fn=CP.event_fn_norm(case["c"]), **kw)
    torch.testing.assert_close(ev_t.cpu(), case["event_t"], rtol=1e-6, atol=1e-8)
    close(sol, case["sol"], torch.complex128, scale=10)


def test_cubic_output(gold):
    case = gold["cubic"]
    f, y0, _ = CP.zoo_problem(torch.complex128, False)
    with torch.no_grad():
        y = tdq().odeint(f.to(DEV), cu(y0), cu(case["t"]), method="rk4", options=dict(step_size=0.1, interp="cubic"))
    close(y, case["sol"], torch.complex128)


@pytest.mark.parametrize("norm", ["default", "seminorm"])
def test_adjoint_against_golden(gold, norm):
    case = gold[("adjoint", norm)]
    f = CP.ComplexLinear(CP.damped_weight(4, 3, torch.complex128), bias=True).to(DEV)
    y0 = cu(CP.crandn(8, 4, seed=5, dtype=torch.complex128)).requires_grad_(True)
    t = torch.linspace(0., 1., 4, dtype=torch.float64, device=DEV).requires_grad_(True)
    ao = {} if norm == "default" else dict(norm="seminorm")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        sol = tdq().odeint_adjoint(f, y0, t, method="dopri5", rtol=1e-9, atol=1e-11, adjoint_options=ao)
        (sol.abs() ** 2).sum().backward()
    close(sol.detach(), case["sol"], torch.complex128)
    assert t.grad.dtype == torch.float64
    for got, want in ((y0.grad, case["y0_grad"]), (f.W.grad, case["W_grad"]), (f.b.grad, case["b_grad"]),
                      (t.grad, case["t_grad"])):
        torch.testing.assert_close(got.cpu(), want, rtol=1e-4, atol=1e-6)


def test_custom_norm_gets_complex_q():
    f, y0, t = CP.zoo_problem(torch.complex128, False)
    seen = []

    def norm(q):
        seen.append(q.dtype)
        return q.abs().pow(2).mean().sqrt()

    with torch.no_grad():
        a = tdq().odeint(f.to(DEV), cu(y0), cu(t), method="dopri5", rtol=1e-8, atol=1e-10, options=dict(norm=norm))
        b = tdq().odeint(f.to(DEV), cu(y0), cu(t), method="dopri5", rtol=1e-8, atol=1e-10)
    assert seen and all(s == torch.complex128 for s in seen)
    close(a, b.cpu(), torch.complex128, scale=1e-2)


def test_plugin_routes_complex(gold):
    import seam_frontend as sf
    from torchdiffeq_b200 import plugin
    replaced = plugin.register(sf.SOLVERS)
    try:
        for dtype in CP.CDTYPES:
            f, y0, t = CP.zoo_problem(dtype, False)
            with torch.no_grad():
                y = sf.odeint(f.to(DEV), cu(y0), cu(t), method="dopri5", **CP.zoo_kwargs("dopri5", dtype))
            assert tdq().last_stats()["nfe"] > 0                     # the solve went through libtdq
            close(y, gold[("zoo", "dopri5", str(dtype), False)]["sol"], dtype)
    finally:
        plugin.unregister(replaced, sf.SOLVERS)


# ---- explicit errors ---------------------------------------------------------------------------------------------------
def test_adjoint_real_params_refused():
    f = CP.ComplexLinear(CP.damped_weight(4, 3, torch.complex64)).to(DEV)
    f.r = torch.nn.Parameter(torch.ones(3, device=DEV))
    y0 = cu(CP.crandn(8, 4, seed=5, dtype=torch.complex64))
    with pytest.raises(TypeError, match="complex adjoint parameters"):
        tdq().odeint_adjoint(f, y0, torch.tensor([0., 1.], device=DEV))


def test_backprop_through_complex_refused():
    f = CP.ComplexLinear(CP.damped_weight(4, 3, torch.complex64)).to(DEV)
    y0 = cu(CP.crandn(8, 4, seed=5, dtype=torch.complex64))
    with pytest.raises(NotImplementedError, match="odeint_adjoint"):
        tdq().odeint(f, y0, torch.tensor([0., 1.], device=DEV))


def test_complex32_and_sharded_refused():
    from torchdiffeq_b200._lib import TdqError
    with pytest.raises(TdqError, match="complex32"):
        tdq().odeint(lambda t, y: y, torch.zeros(4, dtype=torch.complex32, device=DEV), torch.tensor([0., 1.], device=DEV))
    with pytest.raises(NotImplementedError, match="complex"):
        tdq().odeint(lambda t, y: y, torch.zeros(4, dtype=torch.complex64, device=DEV), torch.tensor([0., 1.], device=DEV),
                     options=dict(process_group=object()))


# ---- full size ---------------------------------------------------------------------------------------------------------
def test_full_size_complex64_against_complex128():
    B, D = 65536, 64
    W = CP.damped_weight(D, 13, torch.complex128).to(DEV)
    y0 = CP.crandn(B, D, seed=14, dtype=torch.complex128).to(DEV)
    t = torch.linspace(0., 1., 3, device=DEV)
    with torch.no_grad():
        a = tdq().odeint(CP.ComplexLinear(W.to(torch.complex64)), y0.to(torch.complex64), t, method="dopri5",
                         rtol=1e-5, atol=1e-7)
        b = tdq().odeint(CP.ComplexLinear(W), y0, t, method="dopri5", rtol=1e-5, atol=1e-7)
    err = (a.to(torch.complex128) - b).abs().max().item()
    assert a.dtype == torch.complex64 and err < 1e-4, err
