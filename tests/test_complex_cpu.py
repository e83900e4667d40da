"""Complex states without a GPU: the oracle against the reference's complex goldens, the claim every complex launcher of
libtdq rests on (a real-coefficient combination of complex states is the same combination of their interleaved real
components), and the host side of the C ABI for the complex dtype codes."""
import ctypes as C
import os
import warnings

import pytest
import torch

import complex_problems as CP
from oracle import ode_oracle as O

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOL = {torch.complex64: dict(rtol=1e-4, atol=1e-6), torch.complex128: dict(rtol=1e-5, atol=1e-7)}


@pytest.fixture(scope="module")
def gold():
    return torch.load(os.path.join(G, "complex.pt"), weights_only=False)


@pytest.mark.parametrize("dtype", CP.CDTYPES, ids=str)
@pytest.mark.parametrize("method", CP.ADAPTIVE)
@pytest.mark.parametrize("reverse", [False, True])
def test_oracle_adaptive_against_complex_golden(gold, method, dtype, reverse):
    f, y0, t = CP.zoo_problem(dtype, reverse)
    with torch.no_grad():
        y = O.odeint_adaptive(f, y0, t, method, **CP.zoo_kwargs(method, dtype))
    want = gold[("zoo", method, str(dtype), reverse)]["sol"]
    assert y.dtype == dtype
    torch.testing.assert_close(y, want, **TOL[dtype])


@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("dtype", CP.CDTYPES, ids=str)
@pytest.mark.parametrize("method", CP.FIXED + CP.ADAMS)
def test_oracle_fixed_and_adams_against_complex_golden(gold, method, dtype, reverse):
    """The fixed-grid and Adams methods: solution and number of func evaluations against the reference."""
    f, y0, t = CP.zoo_problem(dtype, reverse)
    opts = CP.zoo_kwargs(method, dtype)["options"]
    # solvers.py:85-96 in the solver's ascending time (misc.py:273-279 negates a descending t), then back
    sgn = -1.0 if reverse else 1.0
    ts = t * sgn
    grid = torch.arange(0, 21, dtype=torch.float64) * opts["step_size"] + ts[0]
    grid[-1] = ts[-1]
    grid = grid * sgn
    r = CP.Rec(f)
    with torch.no_grad():
        if method in CP.ADAMS:
            y = O.odeint_adams(r, y0, t, implicit=method != "explicit_adams", grid=grid,
                               max_order=opts.get("max_order", 12))
        else:
            y = O.odeint_rk4(r, y0, t, grid=grid, method=method)
    case = gold[("zoo", method, str(dtype), reverse)]
    tol = TOL[dtype] if dtype == torch.complex64 else dict(rtol=1e-12, atol=1e-14)
    torch.testing.assert_close(y, case["sol"], **tol)
    assert r.nfe == case["nfe"]


def test_oracle_schrodinger_golden(gold):
    case = gold[("schrodinger", "torch.complex128")]
    f = CP.Schrodinger(CP.hermitian(4, 1, torch.complex128))
    with torch.no_grad():
        y = O.odeint_adaptive(f, case["y0"], case["t"], "dopri5", **case["kw"])
    torch.testing.assert_close(y, case["sol"], rtol=1e-9, atol=1e-11)
    torch.testing.assert_close(case["sol"], case["exact"], rtol=1e-7, atol=1e-8)     # the golden itself is right


@pytest.mark.parametrize("dtype", CP.CDTYPES, ids=str)
@pytest.mark.parametrize("method", ["dopri5", "dopri8", "tsit5"])
def test_complex_combine_is_real_view_combine(dtype, method):
    """Stage combines and the interpolant: the oracle on complex states equals, bit for bit, the oracle on their
    view_as_real components -- what lets libtdq run its real kernels on 2n components."""
    ct = O._cast_tableau(O.tableau(method), dtype.to_real())
    ks = [CP.crandn(64, seed=30 + j, dtype=dtype) for j in range(len(ct["beta"]) + 1)]
    y0 = CP.crandn(64, seed=29, dtype=dtype)
    dt = torch.tensor(0.0371, dtype=dtype.to_real())
    rv = torch.view_as_real
    for b in ct["beta"]:
        zc = y0 + O._weighted(ks, b * dt)
        zr = rv(y0) + O._weighted([rv(k) for k in ks], b * dt)
        assert torch.equal(rv(zc), zr)
    y1 = y0 + O._weighted(ks, dt * ct["c_sol"])
    cc = O.interp_fit(y0, y1, ks, dt, ct)
    cr = O.interp_fit(rv(y0), rv(y1), [rv(k) for k in ks], dt, ct)
    for a, b in zip(cc, cr):
        assert torch.equal(rv(a), b)
    t0, t1 = torch.tensor(0.5, dtype=torch.float64), torch.tensor(0.5371, dtype=torch.float64)
    for te in (0.5, 0.51, 0.53, 0.5371):
        te = torch.tensor(te, dtype=torch.float64)
        assert torch.equal(rv(O.interp_eval(cc, t0, t1, te)), O.interp_eval(cr, t0, t1, te))


def test_complex_error_ratio_rule():
    """The complex rule of the error norm as torch evaluates it: one real tolerance per complex element from the modulus,
    err/tol == err * fl(1/tol) componentwise, and |err/tol|^2 summed once per complex element (misc.py:22-23, :80-82)."""
    for dtype in CP.CDTYPES:
        err, y0, y1 = (CP.crandn(4096, seed=s, dtype=dtype) * 1e-3 for s in (40, 41, 42))
        tol = 1e-6 + 1e-3 * torch.max(y0.abs(), y1.abs())
        assert tol.dtype == dtype.to_real()
        q = err / tol
        assert torch.equal(torch.view_as_real(q), torch.view_as_real(err) * (1 / tol)[:, None])
        ratio = O.rms(q)
        want = torch.view_as_real(q).to(torch.float64).pow(2).sum(-1).mean().sqrt()
        torch.testing.assert_close(ratio.to(torch.float64), want, rtol=1e-5 if dtype == torch.complex64 else 1e-12, atol=0)


# ---- host side of the C ABI ------------------------------------------------------------------------------------------
def _lib():
    from torchdiffeq_b200 import _lib
    return _lib, _lib.load()


CODES_OK = (0, 1, 2, 3)            # float32, float64, complex64, complex128
CODES_BAD = (4, 5, -1)             # complex32 has no code; nothing else is a dtype


def test_abi_complex_codes():
    _l, lib = _lib()
    assert (_l.TDQ_C64, _l.TDQ_C128) == (2, 3)
    assert lib.tdq_abi_version() == 2


def test_abi_validation_accepts_complex_codes():
    """Every launcher that moves or combines the state takes the complex codes; unknown codes (complex32 among them)
    are refused.  The calls below return before they touch the device (n = 0 / empty segments)."""
    _l, lib = _lib()
    bad = C.c_void_p(16)                                   # never dereferenced
    tab = _l.tableau("dopri5")
    k = _l.ptr_array([None] + [16] * 7)
    co = _l.ptr_array([16] * 5)
    one = _l.i64_array([0])
    calls = {
        "stage_combine": lambda c: lib.tdq_stage_combine(bad, C.byref(tab), c, 0, bad, None, k, 0, None),
        "stage_combine_final": lambda c: lib.tdq_stage_combine_final(bad, C.byref(tab), c, bad, bad, None, k, 0, None),
        "probe": lambda c: lib.tdq_initial_step_probe(bad, c, bad, None, None, 0, None),
        "commit": lambda c: lib.tdq_commit_candidates(bad, c, bad, bad, 0, None),
        "fit": lambda c: lib.tdq_interp_fit_eval(bad, C.byref(tab), c, bad, k, None, bad, 0, None),
        "eval_at": lambda c: lib.tdq_interp_eval_at(bad, c, co, bad, bad, 0, None),
        "poly": lambda c: lib.tdq_poly_eval(c, co, 0.5, bad, 0, None),
        "rk4": lambda c: lib.tdq_rk4_stage(c, 1, bad, bad, bad, None, None, None, bad, None, 0, None),
        "lincomb": lambda c: lib.tdq_lincomb(c, bad, None, _l.ptr_array([16]), _l.dbl_array([1.0]), 1, 0, None),
        "cubic": lambda c: lib.tdq_fixed_emit_cubic(c, bad, bad, bad, bad, bad, bad, bad, 0, 1, 0, None),
        "pack": lambda c: lib.tdq_pack_segments(c, bad, _l.ptr_array([None]), one, one, _l.dbl_array([1.0]), 1, None),
        "sumsq": lambda c: lib.tdq_scaled_sumsq(bad, c, bad, None, bad, None, None, None, 0, 0, 1, 0, bad, bad, None),
        "norm_commit": lambda c: lib.tdq_error_norm_commit(bad, c, bad, bad, bad, bad, None, None, None, 0, 0, 1, 0, bad,
                                                           bad, None, None),
    }
    for name, call in calls.items():
        for c in CODES_OK:
            assert call(c) == 0, (name, c, lib.tdq_last_error())
        for c in CODES_BAD:
            assert call(c) == 1, (name, c)                # TDQ_ERR_INVALID


def test_abi_control_block_stays_real():
    """The control block is typed by the component dtype: tdq_ctrl_init refuses the complex codes."""
    _l, lib = _lib()
    tab = _l.tableau("dopri5")
    for c in (2, 3, 4):
        opt = _l.Options(dtype=c, rtol=1e-6, atol=1e-8)
        assert lib.tdq_ctrl_init(C.c_void_p(16), C.byref(tab), C.byref(opt), C.c_void_p(16), 0.0, 2, None, None) == 1


def test_abi_linear_kernels_refuse_complex():
    _l, lib = _lib()
    for m in ("dopri5", "bosh3"):
        tab = _l.tableau(m)
        for c in (2, 3):
            assert lib.tdq_linear_attempt_supported(C.byref(tab), c, 128) == 0
            assert lib.tdq_linear_supported(c, 128) == 0
    from torchdiffeq_b200.fields import fusable
    assert fusable(None, (4, 128), torch.complex64, torch.device("cpu"), lib) is None


@pytest.mark.parametrize("segs,n,want", [
    ([(0, 5000), (5000, 3000)], 8000, {0: 5, 1: 5, 2: 8, 3: 8}),
    ([(0, 1)], 1, {0: 1, 1: 1, 2: 1, 3: 1}),
    ([(1, 4095), (4100, 10)], 4200, {0: 7, 1: 6, 2: 8, 3: 8}),
])
def test_norm_table_complex_chunks(segs, n, want):
    """A chunk holds at most 2048 components: 2048 real or 1024 complex elements.  Complex offsets count complex
    elements, and 16-byte alignment is 2 complex64 / 1 complex128 elements."""
    _l, lib = _lib()
    for code, nch in want.items():
        words = _l.norm_table(segs, n, code)
        assert words[1] == nch, (code, words[:4])
        assert words[2] == (2048 if code < 2 else 1024)
    assert _l.norm_table([(1, 10)], 11, 3)[3] == 1          # complex128: every element is 16-byte aligned
    assert _l.norm_table([(1, 10)], 11, 2)[3] == 0
    for code in CODES_BAD:
        with pytest.raises(Exception):
            _l.norm_table(segs, n, code)


# ---- explicit errors that need no device -------------------------------------------------------------------------------
def test_complex32_is_refused():
    import torchdiffeq_b200 as tdq
    from torchdiffeq_b200._lib import TdqError
    y0 = torch.zeros(4, dtype=torch.complex32)
    with pytest.raises(TdqError, match="complex32"):
        tdq.odeint(lambda t, y: y, y0, torch.tensor([0., 1.]))
    with pytest.raises(TdqError, match="complex32"):
        tdq.odeint(lambda t, y: y, (y0.to(torch.complex64), y0), torch.tensor([0., 1.]))


def test_complex_sharded_is_refused():
    import torchdiffeq_b200 as tdq
    with pytest.raises(NotImplementedError, match="complex"):
        tdq.odeint(lambda t, y: y, torch.zeros(4, dtype=torch.complex64), torch.tensor([0., 1.]),
                   options=dict(process_group=object()))

