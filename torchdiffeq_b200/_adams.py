"""Fixed-step Adams-Bashforth(-Moulton) on the fixed-grid engine: 'explicit_adams', 'implicit_adams', 'fixed_adams'
(torchdiffeq/_impl/fixed_adams.py:164-228; SURVEY.md section 8(f) item 4, last entry).

A multistep method: the step is a linear combination of up to 11 stored derivative evaluations, with a variable order
that grows from an RK4 bootstrap (fixed_adams.py:196-197) and, for the implicit variant, a functional iteration whose
stopping test is a host decision in the reference too (fixed_adams.py:204-213).  So the stepping is host driven (no
captured graph); all state-sized arithmetic is libtdq: the RK4 bootstrap stages, the predictor / corrector sums
(tdq_lincomb), the outputs and the commit (tdq_fixed_emit, tdq_fixed_emit_cubic).

Coefficients: the reference tabulates integer numerators and divisors (fixed_adams.py:10-140) and divides in float64.  They
are the classical Adams-Bashforth / Adams-Moulton weights, generated here as exact rationals
    AB_k:  b_j = (-1)^j / (j! (k-1-j)!) * integral_0^1 prod_{i != j, i < k} (u + i) du          (weights of f_n, f_{n-1}, ...)
    AM_k:  m_j = (-1)^j / (j! (k-1-j)!) * integral_0^1 prod_{i != j, i < k} (u + i - 1) du      (weights of f_{n+1}, f_n, ...)
and converted with one correctly rounded division, which gives the reference's float64 values bit for bit
(tests/test_host_logic.py checks them against tests/golden/adams.json, dumped from the reference)."""
import collections
import warnings
from fractions import Fraction
from math import factorial

import torch

from . import _lib
from ._engine import _stream
from ._fixed import FixedGridEngine, _RetryWithCopies

_MIN_ORDER, _MAX_ORDER, _MAX_ITERS = 4, 12, 4            # fixed_adams.py:143-145


def _poly_mul(p, q):
    r = [Fraction(0)] * (len(p) + len(q) - 1)
    for i, a in enumerate(p):
        for j, b in enumerate(q):
            r[i + j] += a * b
    return r


def _adams_weights(k, shift):
    """k weights; shift = 0: Adams-Bashforth, shift = 1: Adams-Moulton."""
    out = []
    for j in range(k):
        poly = [Fraction(1)]
        for i in range(k):
            if i != j:
                poly = _poly_mul(poly, [Fraction(i - shift), Fraction(1)])      # (u + i - shift)
        integral = sum(c / (n + 1) for n, c in enumerate(poly))
        w = Fraction((-1) ** j, factorial(j) * factorial(k - 1 - j)) * integral
        out.append(w.numerator / w.denominator)                               # one correctly rounded division
    return out


_BASHFORTH = {k: _adams_weights(k, 0) for k in range(1, _MAX_ORDER + 1)}
_MOULTON = {k: _adams_weights(k, 1) for k in range(1, _MAX_ORDER + 1)}


class AdamsEngine(FixedGridEngine):
    """AdamsBashforthMoulton._step_func (fixed_adams.py:193-222) as the step of the fixed-grid engine."""

    def __init__(self, fn, n, dtype, device, *, implicit, rtol, atol, max_iters=_MAX_ITERS, max_order=_MAX_ORDER,
                 t_sign=1.0, perturb=False, callbacks=None, pieces=None, interp="linear"):
        assert max_order <= _MAX_ORDER, "max_order must be at most {}".format(_MAX_ORDER)          # fixed_adams.py:170
        if max_order < _MIN_ORDER:
            warnings.warn("max_order is below {}, so the solver reduces to `rk4`.".format(_MIN_ORDER))
        super().__init__(fn, n, dtype, device, method="rk4", t_sign=t_sign, perturb=perturb, graph=False,
                         callbacks=callbacks, pieces=pieces, interp=interp)
        self.implicit, self.max_iters, self.max_order = bool(implicit), int(max_iters), int(max_order)
        # fixed_adams.py:174-175: tolerances of the corrector's stopping test, in the state dtype (its real part for a
        # complex state: the imaginary part is zero)
        self.rtol = float(torch.as_tensor(rtol, dtype=torch.float64).to(self.rdtype))
        self.atol = float(torch.as_tensor(atol, dtype=torch.float64).to(self.rdtype))
        self.prev_f = collections.deque(maxlen=self.max_order - 1)
        self.prev_t = None
        self.graph_opt = False
        self._grid_cpu, self._event_step = None, None

    FUSE_FINAL = False                     # the step is not a single final expression

    # ---- history (fixed_adams.py:183-186) ----------------------------------------------------------------------------
    def _update_history(self, t, f):
        if self.prev_t is None or bool(self.prev_t != t):
            self.prev_f.appendleft(f)
            self.prev_t = t

    def _lincomb(self, out, base, terms):
        xs = _lib.ptr_array([x.data_ptr() for x, _ in terms])
        cs = _lib.dbl_array([float(c) for _, c in terms])
        _lib.check(self.lib.tdq_lincomb(self.dc, out.data_ptr(), base.data_ptr() if base is not None else None, xs, cs,
                                        len(terms), self.n, _stream()))
        self.launches += 1

    def _solve_impl(self, y0_flat, grid_cpu, t_cpu):
        self._grid_cpu, self._step_index, self._event_step = grid_cpu, 0, None
        self.prev_f.clear()
        self.prev_t = None
        return super()._solve_impl(y0_flat, grid_cpu, t_cpu)

    def solve_until_event(self, y0_flat, t0, step_size, event_fn, atol, max_itrs=20000):
        self.prev_f.clear()
        self.prev_t = None
        try:
            return super().solve_until_event(y0_flat, t0, step_size, event_fn, atol, max_itrs)
        finally:
            self._event_step = None

    def _one_step_tables(self, t0c, dt, t1c):
        super()._one_step_tables(t0c, dt, t1c)
        self._event_step = (t0c, dt, t1c)

    def _stages(self, fuse_final=False):
        """One Adams step: y1 into self.y1; returns [f0] (what _step_func returns besides dy)."""
        T, dev = self.dtype, self.device
        if getattr(self, "_event_step", None) is not None:                      # event stepping: explicit (t0, dt, t1)
            t0, dt, t1 = self._event_step
            dt64 = float(torch.as_tensor(dt, dtype=torch.float64)) if not torch.is_tensor(dt) else float(dt.double())
            dt_T = float(torch.as_tensor(dt64, dtype=torch.float64).to(self.rdtype)) if not torch.is_tensor(dt) \
                else float(dt.to(self.rdtype))
        else:
            k = self._step_index
            t0, t1 = self._grid_cpu[k], self._grid_cpu[k + 1]
            dtt = t1 - t0                                                        # t's dtype (solvers.py:112)
            dt64, dt_T = float(dtt.double()), float(dtt.to(self.rdtype))
            self._step_index += 1
        sgn = self.t_sign
        # func outputs of earlier steps are kept: a func that reuses one output buffer must be copied
        self._taken = {h.data_ptr() for h in self.prev_f}
        # ... and the entry the deque drops in this step stays allocated until the next one: a recycled address would
        # look like a func that reuses its output buffer (_call_fn's aliasing test), also to the cubic emit's f1
        self._hist_alive = list(self.prev_f)
        f0 = self._call_fn(self.tcur[0], self.y0w, None)                         # fixed_adams.py:194 (Perturb.NEXT in tcur)
        self._update_history(t0, f0)
        order = min(len(self.prev_f), self.max_order - 1)
        if order < _MIN_ORDER - 1:                                               # :196-198 RK4 with k1 = prev_f[0]
            lib, dc, n, st = self.lib, self.dc, self.n, _stream()
            y0, ya, y1 = self.y0w.data_ptr(), self.ytmp.data_ptr(), self.y1.data_ptr()
            dtp, stp = self.dt_dev.data_ptr(), self.step_dev.data_ptr()
            k1 = self.prev_f[0]

            def stage(which, out, *ks):
                p = [x.data_ptr() if x is not None else None for x in ks] + [None] * (4 - len(ks))
                _lib.check(lib.tdq_rk4_stage(dc, which, out, y0, p[0], p[1], p[2], p[3], dtp, stp, n, st))
                self.launches += 1
            stage(1, ya, k1)
            k2 = self._call_fn(self.tcur[1], self.ytmp, None)
            stage(2, y1, k1, k2)
            k3 = self._call_fn(self.tcur[2], self.y1, None)
            stage(3, ya, k1, k2, k3)
            k4 = self._call_fn(self.tcur[3], self.ytmp, None)
            stage(4, y1, k1, k2, k3, k4)
            return [f0, k2, k3, k4]
        # Adams-Bashforth predictor (:200-201): dy = sum_m f_{n-m} * T(dt * b_m); the reverse-time sign of the raw
        # func outputs goes into the coefficient (exact)
        hist = list(self.prev_f)[:order]
        bash = _BASHFORTH[order]
        dy = torch.empty(self.n, dtype=T, device=dev)
        self._lincomb(dy, None, [(f, sgn * (dt64 * b)) for f, b in zip(hist, bash)])
        if self.implicit:                                                        # :204-215 Adams-Moulton corrector
            moul = _MOULTON[order + 1]
            S = torch.empty(self.n, dtype=T, device=dev)
            self._lincomb(S, None, [(f, sgn * m) for f, m in zip(hist, moul[1:])])
            delta = torch.empty(self.n, dtype=T, device=dev)
            self._lincomb(delta, None, [(S, dt_T)])                              # dt * (...) with dt cast to T
            converged = False
            c0 = sgn * (dt64 * moul[0])
            alive = []           # keep every output of this step allocated: a recycled address would look like aliasing
            for _ in range(self.max_iters):
                dy_old = dy
                self._lincomb(self.ytmp, self.y0w, [(dy, 1.0)])                  # y0 + dy
                f = self._call_fn(self.tcur[3], self.ytmp, None)                 # t1 (Perturb.PREV in tcur)
                alive.append(f)
                dy = torch.empty(self.n, dtype=T, device=dev)
                self._lincomb(dy, delta, [(f, c0)])                              # (dt*m0*f) + delta
                # fixed_adams.py:188-191: max |(|dy_old - dy|) / (atol + rtol*max(|dy_old|, |dy|))| < 1 -- a host decision
                err = torch.abs(dy_old - dy)
                tol = self.atol + self.rtol * torch.max(dy_old.abs(), dy.abs())
                if T.is_complex:                     # the reference's tolerances are complex there: err/(tol + 0i)
                    tol = tol.to(T)
                converged = bool((err / tol).abs().max() < 1)
                if converged:
                    break
            if not converged:
                warnings.warn('Functional iteration did not converge. Solution may be incorrect.')
                self.prev_f.pop()
            self._update_history(t0, f)                                          # a no-op: prev_t == t0 (as in the reference)
        self._lincomb(self.y1, self.y0w, [(dy, 1.0)])                            # y1 = y0 + dy (solvers.py:115)
        return [f0]

    def _step_once(self, step=None):
        try:
            return super()._step_once(step)
        except _RetryWithCopies:
            # the history was extended before the retry was requested: undo, then let _step() retry
            if self.prev_f and self.prev_t is not None:
                self.prev_f.popleft()
                self.prev_t = None
            if getattr(self, "_event_step", None) is None:
                self._step_index -= 1
            raise
