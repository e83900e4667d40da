"""Host side of the fixed-grid RK4 path (solvers.py:52-128 FixedGridODESolver.integrate,
fixed_grid.py:24-29 RK4, rk_common.py:110-118 rk4_alt_step_func).

The grid is known before the first step, so everything the reference decides per step on the host
(step sizes, stage times, which outputs fall into which step, interpolation slopes) is tabulated
once with the reference's own dtype rules and uploaded; one captured step graph then serves every
grid interval, indexed by a device step counter."""
import torch

from . import _lib
from ._engine import _RetryWithCopies, _stream, pack_pieces, solver_stream, state_codes

_ONE_THIRD = 1 / 3      # rk_common.py:94-96
_TWO_THIRDS = 2 / 3


def grid_from_step_size(step_size):
    """solvers.py:85-96 _grid_constructor_from_step_size."""
    def _grid_constructor(func, y0, t):
        start_time = t[0]
        end_time = t[-1]
        niters = torch.ceil((end_time - start_time) / step_size + 1).item()
        t_infer = torch.arange(0, niters, dtype=t.dtype, device=t.device) * step_size + start_time
        t_infer[-1] = t[-1]
        return t_infer
    return _grid_constructor


FIXED_METHODS = ("euler", "midpoint", "heun2", "heun3", "rk4")


class FixedGridEngine:
    """Explicit fixed-step methods of fixed_grid.py:6-60 on one captured step graph."""
    FUSE_FINAL = True       # last expression of a step fused with the emit/commit kernel (tdq_fixed_final_emit)

    def __init__(self, fn, n, dtype, device, *, method="rk4", t_sign=1.0, perturb=False, graph="auto",
                 callbacks=None, pieces=None, interp="linear"):
        if method not in FIXED_METHODS:
            raise ValueError("unknown fixed-grid method %r" % method)
        self.method = method
        if device.type != "cuda":
            raise _lib.TdqError("torchdiffeq_b200 runs on CUDA devices only (got %s); there is no CPU path" % device)
        self.dc = state_codes(dtype)[0]
        self.lib = _lib.load()
        self.fn, self.n, self.dtype, self.device = fn, int(n), dtype, device
        self.t_sign = float(t_sign)
        self.perturb = bool(perturb)
        self.callbacks = callbacks or {}
        if interp not in ("linear", "cubic"):
            raise ValueError(f"Unknown interpolation method {interp}")           # solvers.py:125
        self.interp = interp
        # cubic Hermite outputs need f(t1, y1) on the steps that contain an output time (solvers.py:120-122): the
        # host knows which steps those are, so they are stepped eagerly instead of through one captured graph
        self.graph_opt = False if (self.callbacks or interp == "cubic") else graph
        self._always_copy = False
        self.pieces = pieces            # fn returns a tuple of pieces (tuple states, the adjoint's augmented state)
        self.nfe = 0
        self.launches = 0

    @property
    def rdtype(self):
        """dtype of func's time argument, step sizes and interpolation weights: the component dtype of the state."""
        return self.dtype.to_real()

    # ---- tables ---------------------------------------------------------------------------
    def _tabulate(self, grid, t):
        """grid, t: ascending CPU tensors of t's dtype.  Returns per-step and per-output tables."""
        T = self.rdtype
        if grid.dtype != t.dtype:                  # a grid_constructor may return another float dtype: compare in
            common = torch.promote_types(grid.dtype, t.dtype)      # the promoted one, like the reference's mixed ops
            t = t.to(common)
        t0, t1 = grid[:-1], grid[1:]
        dt = t1 - t0                                                   # solvers.py:112
        # func times of the four evaluations, then _PerturbFunc's cast to the state dtype (misc.py:187)
        z = torch.zeros_like(t0)
        m = self.method
        if m == "rk4":                                                 # rk_common.py:110-118
            cols, prev_col = [t0, t0 + dt * _ONE_THIRD, t0 + dt * _TWO_THIRDS, t1], 3
        elif m == "euler":                                             # fixed_grid.py:9-11
            cols, prev_col = [t0, z, z, z], None
        elif m == "midpoint":                                          # fixed_grid.py:17-21
            cols, prev_col = [t0, t0 + 0.5 * dt, z, z], None
        elif m == "heun2":                                             # fixed_grid.py:51-60, rk_common.py:141-158
            cols, prev_col = [t0, t0 + dt * 1.0, z, z], 1
        else:                                                          # heun3: fixed_grid.py:35-45, rk_common.py:121-139
            cols, prev_col = [t0, t0 + dt * (1 / 3), t0 + dt * (2 / 3), z], None
        ts = torch.stack(cols, dim=1).to(T)
        if self.perturb:                                               # Perturb.NEXT / PREV, misc.py:188-193
            ts[:, 0] = torch.nextafter(ts[:, 0], ts[:, 0] + 1)
            if prev_col is not None:
                ts[:, prev_col] = torch.nextafter(ts[:, prev_col], ts[:, prev_col] - 1)
        ts = ts * self.t_sign
        dtT = dt.to(T) * self.t_sign           # sign of _ReverseFunc folded into dt (exact)
        # outputs: step s emits every t[j] with t1_s >= t[j] not emitted before (solvers.py:117)
        n_steps = grid.numel() - 1
        step_of = torch.searchsorted(t1.to(t.dtype).contiguous(), t[1:].contiguous(), right=False)
        if step_of.numel() and int(step_of.max()) >= n_steps:
            raise AssertionError("output time beyond the end of the grid")
        g0, g1, tj = t0[step_of], t1[step_of], t[1:]
        mode = torch.full_like(step_of, 2, dtype=torch.int32)
        mode[tj == g1] = 1
        mode[tj == g0] = 0                                             # solvers.py:176-179
        slope = ((tj - g0) / (g1 - g0)).to(T)                          # :180
        counts = torch.bincount(step_of, minlength=n_steps)
        rec_begin = torch.zeros(n_steps + 1, dtype=torch.int32)
        rec_begin[1:] = torch.cumsum(counts, 0).to(torch.int32)
        out_idx = torch.arange(1, t.numel(), dtype=torch.int32)
        # cubic Hermite weights (solvers.py:166-173), evaluated in t's dtype like the reference's 0-dim tensors and
        # cast to the state dtype where they meet a state tensor; dt*f carries _ReverseFunc's sign
        h = (tj - g0) / (g1 - g0)
        dtj = (g1 - g0)
        h00 = (1 + 2 * h) * (1 - h) * (1 - h)
        h10 = h * (1 - h) * (1 - h)
        h01 = h * h * (3 - 2 * h)
        h11 = h * h * (h - 1)
        self._cubic = torch.stack([h00.to(T), (h10 * dtj).to(T) * self.t_sign, h01.to(T), (h11 * dtj).to(T) * self.t_sign],
                                  dim=1).contiguous() if tj.numel() else torch.zeros(1, 4, dtype=T)
        self._t1_T = (t1.to(T) * self.t_sign).contiguous()          # time of the extra evaluation f(t1, y1), as func sees it
        return ts.contiguous(), dtT.contiguous(), rec_begin, out_idx, mode.contiguous(), slope.contiguous(), n_steps

    # ---- one step -----------------------------------------------------------------------------
    def _call_fn(self, t, y, own):
        self.nfe += 1
        f = self.fn(t, y)
        if not isinstance(f, torch.Tensor):
            buf = torch.zeros(self.n, dtype=self.dtype, device=self.device)
            self.launches += pack_pieces(self.lib, self.dc, self.dtype, buf, f, self.pieces)
            return buf
        if f.dtype != self.dtype:
            f = f.to(self.dtype)
        f = f.reshape(-1)
        if f.numel() != self.n:
            raise ValueError("func returned %d elements for a state of %d" % (f.numel(), self.n))
        if f.data_ptr() in self._taken and not self._always_copy:
            self._always_copy = True                       # func reuses one output buffer: redo the step with copies
            raise _RetryWithCopies()
        if (self._always_copy or (not f.is_contiguous()) or f.untyped_storage().data_ptr() in self._own
                or f.data_ptr() in self._taken):
            f = f.clone(memory_format=torch.contiguous_format)
        self._taken.add(f.data_ptr())
        return f

    def _step(self, step=None):
        if getattr(self, "_taping", None) is not None:
            self._taping.append({"y0": self.y0w.clone()})
        try:
            return self._step_once(step)
        except _RetryWithCopies:                           # nothing of the step has been committed yet
            return self._step_once(step)

    def _stages(self, fuse_final=False):
        """The method's stage values and y1 (in self.y1); returns the tensors func returned (k1 first).
        fuse_final: the last expression (y1 = y0 + dy) is fused with the emit/commit (tdq_fixed_final_emit): one launch
        less per step and y1 never stored on its own -- for plain stepping with linear interpolation."""
        lib, dc, n, st = self.lib, self.dc, self.n, _stream()
        y0, ya, y1 = self.y0w.data_ptr(), self.ytmp.data_ptr(), self.y1.data_ptr()
        dtp, stp = self.dt_dev.data_ptr(), self.step_dev.data_ptr()

        def stage(which, out, k1=None, k2=None, k3=None, k4=None):
            p = lambda k: k.data_ptr() if k is not None else None
            if fuse_final and out == y1 and which in (4, 5, 7, 9):
                _lib.check(lib.tdq_fixed_final_emit(
                    dc, which, y0, p(k1), p(k2), p(k3), p(k4), dtp, self.solution.data_ptr(), self.rec_begin.data_ptr(),
                    self.out_idx.data_ptr(), self.mode.data_ptr(), self.slope.data_ptr(), stp, self.ts_all.data_ptr(),
                    self.tcur.data_ptr(), self.n_steps, n, st))
            else:
                _lib.check(lib.tdq_rk4_stage(dc, which, out, y0, p(k1), p(k2), p(k3), p(k4), dtp, stp, n, st))
            self.launches += 1
        m = self.method
        self._taken = set()                                # stage outputs of this step (a func may reuse one buffer)
        k1 = self._call_fn(self.tcur[0], self.y0w, None)
        keep = [k1]
        if m == "rk4":
            stage(1, ya, k1)
            k2 = self._call_fn(self.tcur[1], self.ytmp, None)
            stage(2, y1, k1, k2)
            k3 = self._call_fn(self.tcur[2], self.y1, None)
            stage(3, ya, k1, k2, k3)
            k4 = self._call_fn(self.tcur[3], self.ytmp, None)
            stage(4, y1, k1, k2, k3, k4)
            keep += [k2, k3, k4]
        elif m == "euler":
            stage(5, y1, k1)                                   # dt * f0
        elif m == "midpoint":
            stage(6, ya, k1)                                   # y_mid = y0 + f0 * half_dt
            k2 = self._call_fn(self.tcur[1], self.ytmp, None)
            stage(5, y1, k2)                                   # dt * func(t0 + half_dt, y_mid)
            keep.append(k2)
        elif m == "heun2":
            stage(5, ya, k1)                                   # y0 + dt * k1 * 1.0
            k2 = self._call_fn(self.tcur[1], self.ytmp, None)
            stage(7, y1, k1, k2)
            keep.append(k2)
        else:                                                  # heun3
            stage(1, ya, k1)                                   # y0 + dt * k1 * (1/3)
            k2 = self._call_fn(self.tcur[1], self.ytmp, None)
            stage(8, y1, None, k2)                             # y0 + dt * (k1*0 + k2*(2/3))
            k3 = self._call_fn(self.tcur[2], self.y1, None)
            stage(9, y1, k1, None, k3)                         # y0 + dt * (k1/4 + k2*0 + 3*k3/4)
            keep += [k2, k3]
        return keep

    def _emit(self):
        """Outputs of the step by linear interpolation, y0 <- y1, step counter and func times of the next step."""
        _lib.check(self.lib.tdq_fixed_emit(self.dc, self.y0w.data_ptr(), self.y1.data_ptr(), self.solution.data_ptr(),
                                           self.rec_begin.data_ptr(), self.out_idx.data_ptr(), self.mode.data_ptr(),
                                           self.slope.data_ptr(), self.step_dev.data_ptr(), self.ts_all.data_ptr(),
                                           self.tcur.data_ptr(), self.n_steps, self.n, _stream()))
        self.launches += 1

    def _emit_cubic(self, step, k1):
        """solvers.py:120-122: f1 = func(t1, y1), then the cubic Hermite outputs of this step (one launch).  The
        reference re-evaluates f1 for EVERY output time of the step; the call count is reproduced."""
        lo, hi = int(self._rec_begin_cpu[step]), int(self._rec_begin_cpu[step + 1])
        if hi <= lo:
            return
        alive = []               # keep the evaluations allocated until the step is over (see _call_fn's aliasing test)
        for _ in range(hi - lo):
            f1 = self._call_fn(self.t1_dev[step], self.y1, None)
            alive.append(f1)
        _lib.check(self.lib.tdq_fixed_emit_cubic(self.dc, self.y0w.data_ptr(), self.y1.data_ptr(), k1.data_ptr(),
                                                 f1.data_ptr(), self.solution.data_ptr(), self.out_idx.data_ptr(),
                                                 self.cubic_dev.data_ptr(), lo, hi, self.n, _stream()))
        self.launches += 1

    def _step_once(self, step=None):
        if self.interp == "linear" and self.FUSE_FINAL:
            return self._stages(fuse_final=True)
        keep = self._stages()
        if self.interp == "cubic" and step is not None:
            self._emit_cubic(step, keep[0])
        self._emit()
        return keep

    def solve(self, y0_flat, grid_cpu, t_cpu):
        self._taping = None
        return self._solve_impl(y0_flat, grid_cpu, t_cpu)

    def _solve_impl(self, y0_flat, grid_cpu, t_cpu):
        dev, T = self.device, self.dtype
        ts, dtT, rec_begin, out_idx, mode, slope, n_steps = self._tabulate(grid_cpu, t_cpu)
        self.n_steps = n_steps
        self.ts_all = ts.to(dev)
        self.dt_dev = dtT.to(dev)
        self.rec_begin, self.out_idx = rec_begin.to(dev), out_idx.to(dev)
        self._rec_begin_cpu = rec_begin
        if self.interp == "cubic":
            # every record is written by tdq_fixed_emit_cubic; the linear emit only commits y0 <- y1 and advances
            self.cubic_dev, self.t1_dev = self._cubic.to(dev), self._t1_T.to(dev)
            self.rec_begin = torch.zeros_like(self.rec_begin)
        self.mode = mode.to(dev)
        self.slope = slope.to(dev) if slope.numel() else torch.zeros(1, dtype=self.rdtype, device=dev)
        if self.out_idx.numel() == 0:
            self.out_idx = torch.zeros(1, dtype=torch.int32, device=dev)
            self.mode = torch.zeros(1, dtype=torch.int32, device=dev)
        self.step_dev = torch.zeros(2, dtype=torch.int64, device=dev)     # [0] step counter, [1] ticket of the emit kernel
        self.tcur = self.ts_all[0].clone() if n_steps > 0 else torch.zeros(4, dtype=self.rdtype, device=dev)
        kw = dict(dtype=T, device=dev)
        self.solution = torch.empty(t_cpu.numel(), self.n, **kw)
        self.solution[0].copy_(y0_flat)
        self.y0w = y0_flat.detach().clone()
        self.ytmp = torch.empty(self.n, **kw)
        self.y1 = torch.empty(self.n, **kw)
        self._own = {x.untyped_storage().data_ptr() for x in (self.y0w, self.ytmp, self.y1, self.solution)}
        if n_steps == 0:
            return self.solution
        cb = self.callbacks.get("callback_step")
        if cb is not None:                                            # solvers.py:113, host in the loop
            t0s, dts = grid_cpu[:-1], grid_cpu[1:] - grid_cpu[:-1]
            for s in range(n_steps):
                cb(t0s[s].to(dev), self.y0w, dts[s].to(dev))
                self._step(s)
            torch.cuda.current_stream().synchronize()
            return self.solution
        done = 0
        self._step(0)                                                 # eager first step = warm-up for capture
        done += 1
        graph = None
        if self.graph_opt in (True, "auto") and n_steps > 2:
            try:
                graph = torch.cuda.CUDAGraph()
                nfe, launches = self.nfe, self.launches
                with torch.cuda.graph(graph, stream=solver_stream(self.device)):
                    keep = self._step()
                self._evals, self._graph_launches = self.nfe - nfe, self.launches - launches
                self.nfe, self.launches = nfe, launches
            except Exception as e:
                graph = None
                if self.graph_opt is True:
                    raise
                import warnings
                warnings.warn("torchdiffeq_b200: CUDA graph capture of the RK4 step failed (%s: %s); "
                              "continuing with eager launches" % (type(e).__name__, e))
        while done < n_steps:
            if graph is not None:
                graph.replay()
                self.nfe += self._evals
                self.launches += self._graph_launches
            else:
                self._step(done)
            done += 1
        torch.cuda.current_stream().synchronize()
        del graph
        return self.solution

    # ---- taped solve for the differentiable (non-adjoint) odeint (torchdiffeq_b200/backprop.py) ------------------
    def solve_taped(self, y0_flat, grid_cpu, t_cpu):
        """Eager solve that keeps the state every step started from and the output records it produced."""
        graph_opt, self.graph_opt = self.graph_opt, False
        ts, dtT, rec_begin, out_idx, mode, slope, n_steps = self._tabulate(grid_cpu, t_cpu)
        self._taping = tape = []
        try:
            sol = self._solve_impl(y0_flat, grid_cpu, t_cpu)
        finally:
            self.graph_opt, self._taping = graph_opt, None
        for k, st in enumerate(tape):
            st["k"], st["perturb"] = k, self.perturb
            st["outs"] = [(int(out_idx[r]), int(mode[r]), float(slope[r]))
                          for r in range(int(rec_begin[k]), int(rec_begin[k + 1]))]
        return sol, tape

    # ---- event handling with a fixed step (solvers.py:130-164) ------------------------------------------------
    def solve_until_event(self, y0_flat, t0, step_size, event_fn, atol, max_itrs=20000):
        """Step with dt = step_size from t0 until event_fn(t, y) changes sign, then bisect on the step's interpolant
        (event_handling.py:5-20).  event_fn takes a 0-dim tensor of the state dtype (solver time, ascending) and the
        flat state.  Host driven by nature: one sign test per step.  Returns (event_t tensor, y(event_t))."""
        import math
        dev, T = self.device, self.dtype
        kw = dict(dtype=T, device=dev)
        t0c = torch.as_tensor(t0).detach().to("cpu").to(self.rdtype).reshape(())    # t0.type_as(y0.abs())
        dt = step_size.detach().to("cpu") if torch.is_tensor(step_size) else step_size
        self.solution = torch.empty(1, self.n, **kw)                                # nothing is emitted
        self.y0w = y0_flat.detach().clone()
        self.ytmp, self.y1 = torch.empty(self.n, **kw), torch.empty(self.n, **kw)
        self._own = {x.untyped_storage().data_ptr() for x in (self.y0w, self.ytmp, self.y1, self.solution)}
        z32 = torch.zeros(2, dtype=torch.int32, device=dev)
        self.rec_begin, self.out_idx, self.mode = z32, z32, z32
        self.slope = torch.zeros(1, dtype=self.rdtype, device=dev)
        self.n_steps = 1
        sign0 = torch.sign(event_fn(t0c.to(dev), self.y0w))
        itr = 0
        while True:
            itr += 1
            t1c = t0c + dt                                                         # solvers.py:143
            self._one_step_tables(t0c, dt, t1c)
            keep = self._stages_retry()
            sign1 = torch.sign(event_fn(t1c.to(dev), self.y1))
            if bool(sign0 != sign1):
                break
            self._emit()                                                           # y0 <- y1
            t0c = t1c
            if itr >= max_itrs:
                raise RuntimeError(f"Reached maximum number of iterations {max_itrs}.")
        # the interpolant of the last step on the device, evaluated with torch ops at a handful of bisection points
        y0, y1 = self.y0w, self.y1
        if self.interp == "cubic":
            f0 = keep[0] * self.t_sign
            f1 = self._call_fn((t1c.to(self.rdtype) * self.t_sign).to(dev), self.y1, None) * self.t_sign

            def interp_fn(t):                                                      # solvers.py:166-173
                h = (t - t0c) / (t1c - t0c)
                h00 = (1 + 2 * h) * (1 - h) * (1 - h)
                h10 = h * (1 - h) * (1 - h)
                h01 = h * h * (3 - 2 * h)
                h11 = h * h * (h - 1)
                d = (t1c - t0c)
                return float(h00) * y0 + float(h10 * d) * f0 + float(h01) * y1 + float(h11 * d) * f1
        else:
            def interp_fn(t):                                                      # solvers.py:175-181
                if t == t0c:
                    return y0
                if t == t1c:
                    return y1
                slope = (t - t0c) / (t1c - t0c)
                return y0 + float(slope) * (y1 - y0)
        lo, hi = t0c, t1c                                                          # event_handling.py:5-20
        nitrs = torch.ceil(torch.log((hi - lo) / atol) / math.log(2.0))
        for _ in range(int(nitrs.long())):
            t_mid = (hi + lo) / 2.0
            same = bool(sign0 == torch.sign(event_fn(t_mid.to(dev), interp_fn(t_mid))))
            if same:
                lo = t_mid
            else:
                hi = t_mid
        event_t = (lo + hi) / 2.0
        y_ev = interp_fn(event_t).clone()
        torch.cuda.current_stream().synchronize()
        return event_t.to(dev), y_ev

    def _stages_retry(self):
        try:
            return self._stages()
        except _RetryWithCopies:
            return self._stages()

    def _one_step_tables(self, t0c, dt, t1c):
        """Func times and dt of ONE step taken with an explicit dt (solvers.py:143-145 calls _step_func with
        dt = step_size, not t1 - t0), evaluated like the reference's 0-dim expressions."""
        T, dev, m = self.rdtype, self.device, self.method
        z = torch.zeros((), dtype=T)
        if m == "rk4":
            cols, prev_col = [t0c, t0c + dt * _ONE_THIRD, t0c + dt * _TWO_THIRDS, t1c], 3
        elif m == "euler":
            cols, prev_col = [t0c, z, z, z], None
        elif m == "midpoint":
            cols, prev_col = [t0c, t0c + 0.5 * dt, z, z], None
        elif m == "heun2":
            cols, prev_col = [t0c, t0c + dt * 1.0, z, z], 1
        else:
            cols, prev_col = [t0c, t0c + dt * (1 / 3), t0c + dt * (2 / 3), z], None
        ts = torch.stack([c.to(T).reshape(()) for c in cols]).reshape(1, 4)
        if self.perturb:
            ts[:, 0] = torch.nextafter(ts[:, 0], ts[:, 0] + 1)
            if prev_col is not None:
                ts[:, prev_col] = torch.nextafter(ts[:, prev_col], ts[:, prev_col] - 1)
        ts = ts * self.t_sign
        dt_t = dt if torch.is_tensor(dt) else torch.tensor(dt, dtype=torch.float64)   # a Python float is a double
        dtT = (dt_t.to(T).reshape(1)) * self.t_sign
        self.ts_all = torch.cat([ts, ts]).to(dev)              # row 1: what tdq_fixed_emit stages for a next step
        self.dt_dev = dtT.to(dev)
        self.step_dev = torch.zeros(2, dtype=torch.int64, device=dev)
        self.tcur = self.ts_all[0].clone()
        self.n_steps = 2


FixedRK4Engine = FixedGridEngine      # r1 name
