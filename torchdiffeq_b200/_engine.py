"""Device-resident adaptive Runge-Kutta engine: the host side of libtdq's adaptive path.

What the reference does per attempt in ~570 ATen calls and 15-20 host syncs
(rk_common.py:266-361) is here a fixed launch sequence

    S x (tdq_stage_combine ; func) ; tdq_error_norm_commit ; [all-reduce] ; tdq_controller ;
    tdq_interp_fit_eval

(the last combine is tdq_stage_combine_final, which also emits the prefix of the error estimate) whose
every scalar decision (accept/reject, next dt, output cursor, termination, failure status) is taken on
the device.  The sequence is the same for every attempt, so it is captured once in a CUDA graph; the
graph then becomes the body of a device-side WHILE (tdq_loop_create) and a whole solve is one graph
launch.  Where that is not possible the graph is replayed by the host, which reads a mapped-memory
mailbox to learn when to stop.

State buffers: the accepted state y0 and f0 = k_0 live in ybuf[par] / kbuf[par]; the error-norm kernel
writes each attempt's candidate (y1, k_S) into the other pair and the controller accepts by flipping
`par` -- there is no commit copy, and the interpolant is fitted only for steps that contain an output
time (or when the caller keeps dense output).

Execution modes (options of our path only, SURVEY.md section 5 "config"):
    graph      True/False/'auto'  capture the attempt body in a CUDA graph.
    run_ahead  D >= 0             attempts the host may queue beyond the last one it has seen finish.
                                  0 = lock step: func is called exactly 2 + S*attempts times in the
                                  reference's order (needed for callbacks / NFE counters).
    device_loop True/False/'auto' run the captured attempt inside the device-side while loop.
"""
import ctypes as C
import time

import torch

from . import _lib

_DTYPES = {torch.float32: _lib.TDQ_F32, torch.float64: _lib.TDQ_F64,
           torch.complex64: _lib.TDQ_C64, torch.complex128: _lib.TDQ_C128}


def state_codes(dtype):
    """(libtdq code of the state dtype, code of its real component dtype).  Launchers that move or combine the state
    take the first; the control block and everything scalar (time, step size, error ratio) take the second."""
    if dtype not in _DTYPES:
        raise _lib.TdqError("unsupported state dtype %s (float32, float64, complex64 and complex128 are implemented)"
                            % dtype)
    return _DTYPES[dtype], _DTYPES[dtype.to_real()]


def _stream():
    return torch.cuda.current_stream().cuda_stream


_SOLVER_STREAMS = {}


def solver_stream(device):
    """The dedicated (non-default, non-blocking) stream every solve of a device runs on."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    st = _SOLVER_STREAMS.get(idx)
    if st is None:
        st = _SOLVER_STREAMS[idx] = torch.cuda.Stream(device=idx)
    return st


class on_solver_stream:
    """Run a solve on the device's solver stream, ordered after the caller's stream on entry and before
    it on exit.  Reasons: (1) CUDA graphs cannot be captured on the legacy default stream, and torch's
    capture recipe wants the warm-up on the same kind of stream; (2) when func differentiates inside the
    step (the adjoint's augmented dynamics), autograd synchronises every gradient's producer stream with
    the stream its consumer node was CREATED on -- if that is the legacy stream the capture is
    invalidated ("would make the legacy stream depend on a capturing stream").  Creating the
    odeint_adjoint node, warming up, capturing and replaying all on this one stream removes that edge."""

    def __init__(self, device):
        self.device = device

    def __enter__(self):
        self.cur = torch.cuda.current_stream(self.device)
        self.s = solver_stream(self.device)
        if self.cur == self.s:
            self.ctx = None
            return self
        self.s.wait_stream(self.cur)
        self.ctx = torch.cuda.stream(self.s)
        self.ctx.__enter__()
        return self

    def __exit__(self, *exc):
        if self.ctx is not None:
            self.ctx.__exit__(*exc)
            self.cur.wait_stream(self.s)
        return False

    def publish(self, *tensors):
        """Tensors allocated on the solver stream and handed to the caller's stream."""
        if self.ctx is not None:
            for t in tensors:
                if isinstance(t, torch.Tensor) and t.is_cuda:
                    t.record_stream(self.cur)


class _RetryWithCopies(Exception):
    """func handed back a buffer it had already returned for an earlier stage of the same attempt."""


class SolverFailure(AssertionError):
    """Raised for the reference's in-loop assertions (rk_common.py:247, :286, :287)."""


class Layout:
    """Flat layout of a (possibly tupled) state: pieces at 16-byte aligned offsets.

    The reference concatenates tuple states back to back (misc.py:214-223); we pad each piece so
    that 128-bit accesses stay aligned.  Padding elements are zero in every buffer and belong to no
    norm segment, so they never influence a result."""

    def __init__(self, shapes, dtype):
        self.shapes = [torch.Size(s) for s in shapes]
        self.dtype = dtype
        vec = 16 // torch.empty((), dtype=dtype).element_size()
        self.offsets, self.lens = [], []
        off = 0
        for s in self.shapes:
            n = s.numel()
            self.offsets.append(off)
            self.lens.append(n)
            off += (n + vec - 1) // vec * vec
        self.n = off
        self.n_real = sum(self.lens)

    def flatten(self, tensors, out=None):
        flat = out if out is not None else torch.zeros(self.n, dtype=self.dtype, device=tensors[0].device)
        for t, o, l in zip(tensors, self.offsets, self.lens):
            flat[o:o + l].copy_(t.reshape(-1))
        return flat

    def views(self, flat, lead=()):
        """Unflatten [..., n] -> tuple of [..., *shape] views (misc.py:126-134)."""
        return tuple(flat[..., o:o + l].view((*lead, *s)) for o, l, s in zip(self.offsets, self.lens, self.shapes))


def pack_pieces(lib, dt_code, dtype, buf, f, pieces):
    """Write the pieces func returned (a tuple; None = zeros) into the flat buffer `buf` at their offsets with
    their scales: one tdq_pack_segments launch per 64 pieces (misc.py:145 torch.cat, misc.py:165 the reverse-
    time factor, adjoint.py:96 the unary minus).  Returns the number of launches."""
    offs, lens, scales = pieces
    srcs, keep = [], []
    for p_, l in zip(f, lens):
        if p_ is None:
            srcs.append(None)
            continue
        if p_.dtype != dtype:
            p_ = p_.to(dtype)
        p_ = p_.reshape(-1)
        if not p_.is_contiguous():
            p_ = p_.contiguous()
        if p_.numel() != l:
            raise ValueError("func returned a piece of %d elements, expected %d" % (p_.numel(), l))
        keep.append(p_)
        srcs.append(p_.data_ptr())
    n_launch = 0
    for lo in range(0, len(srcs), _lib.TDQ_MAX_SEGS):
        hi = min(lo + _lib.TDQ_MAX_SEGS, len(srcs))
        _lib.check(lib.tdq_pack_segments(
            dt_code, buf.data_ptr(), _lib.ptr_array(srcs[lo:hi]), _lib.i64_array(offs[lo:hi]),
            _lib.i64_array(lens[lo:hi]), _lib.dbl_array(scales[lo:hi]), hi - lo, _stream()))
        n_launch += 1
    return n_launch


class AdaptiveEngine:
    """One adaptive explicit-RK solve on a flat state vector, all state on the device.

    fn(t, y_flat) -> Tensor (numel n) or tuple of piece tensors matching `pieces` (offsets, lens,
    scales); t is a 0-dim tensor of the state dtype that aliases the control block.
    """

    def __init__(self, fn, n, dtype, device, method, *, rtol, atol, segs=None, t_sign=1.0,
                 pieces=None, min_step=0.0, max_step=float("inf"), first_step=None, step_t=None, jump_t=None,
                 safety=0.9, ifactor=10.0, dfactor=0.2, max_num_steps=2 ** 31 - 1,
                 rtol_vec=None, atol_vec=None, norm_fn=None, q_view=None,
                 graph="auto", run_ahead=2, reduce_fn=None, n_global=None, seg_counts_global=None,
                 agree_fn=None, exchange=None, callbacks=None, keep_interp=False, device_loop="auto", post_fn=None):
        if device.type != "cuda":
            raise _lib.TdqError("torchdiffeq_b200 runs on CUDA devices only (got %s); there is no CPU path" % device)
        self.dt_code, self.rt_code = state_codes(dtype)
        self.lib = _lib.load()
        self.fn = fn
        self.n = int(n)
        self.dtype = dtype
        self.rdtype = dtype.to_real()   # dtype of time, step size and ratio (the component dtype of a complex state)
        self.device = device
        self.tab = _lib.tableau(method)
        self.S = self.tab.n_stages
        self.fsal = bool(self.tab.fsal)
        self.pieces = pieces
        self.first_step = first_step
        self.norm_fn = norm_fn          # custom norm callable on err/tol (compatibility path)
        self.q_view = q_view            # how to present err/tol to norm_fn
        self.reduce_fn = reduce_fn
        self.agree_fn = agree_fn        # sharded solves: host-side max over ranks of the attempts queued
        self.exchange = exchange        # sharded solves: per-attempt all-reduce fused into tdq_controller
        self.post_fn = post_fn          # sharded adjoint: all-reduce of the rank-partial pieces of every func result
        if exchange is not None and post_fn is None:
            self.agree_fn = None        # no collective launch inside an attempt: trailing no-ops need no agreement
        self.callbacks = callbacks or {}
        self.graph_opt = graph
        self.run_ahead = int(run_ahead)
        self.device_loop = device_loop
        self.keep_interp = bool(keep_interp)   # dense output / events: store the interpolant of every accepted step
        self.jump_t = jump_t
        if self.callbacks or (jump_t is not None and jump_t.numel() > 0):
            # both need the host between attempts: callbacks by definition, jump_t because f is re-evaluated on
            # the far side of the discontinuity after the step that lands on it (rk_common.py:346-351)
            self.graph_opt = False
            self.run_ahead = 0

        segs = segs if segs is not None else [(0, self.n)]
        self.n_seg = len(segs)
        n_real = sum(int(l) for _, l in segs)
        counts = seg_counts_global if seg_counts_global is not None else [int(l) for _, l in segs]
        self.seg_counts = torch.tensor(counts, dtype=torch.int64, device=device)
        # one segment covering everything needs no table; anything else (tuple states, the adjoint's augmented
        # state with one segment per parameter tensor -- any number of them) gets a chunk table on the device
        if len(segs) == 1 and int(segs[0][0]) == 0 and int(segs[0][1]) == self.n:
            self.norm_table, self.n_chunks, self.table_aligned = None, 0, 0
        else:
            words = _lib.norm_table(segs, self.n, _DTYPES[dtype])
            self.norm_table = torch.tensor(words, dtype=torch.int64, device=device)
            self.n_chunks, self.table_aligned = int(words[1]), int(words[3])

        self.rtol_vec = rtol_vec
        self.atol_vec = atol_vec
        vtol = rtol_vec is not None
        self.ratio_f64 = vtol or self.rdtype == torch.float64
        self.opt = _lib.Options(
            dtype=self.rt_code, ratio_f64=1 if vtol else 0,
            rtol=float(rtol) if not vtol else 0.0, atol=float(atol) if not vtol else 0.0,
            min_step=float(min_step), max_step=float(max_step), safety=float(safety),
            ifactor=float(ifactor), dfactor=float(dfactor), t_sign=float(t_sign),
            max_num_steps=int(max_num_steps), n_global=int(n_global if n_global is not None else n_real))
        self.step_t = step_t

        kw = dict(dtype=dtype, device=device)
        self.ctrl = torch.zeros(self.lib.tdq_ctrl_size(), dtype=torch.uint8, device=device)
        o = self.lib.tdq_ctrl_tstage_offset()
        self.tstage = self.ctrl[o:o + 8 * _lib.TDQ_MAX_K].view(self.rdtype)
        o = self.lib.tdq_ctrl_taux_offset()
        self.taux = self.ctrl[o:o + 32].view(self.rdtype)
        self.ybuf = [torch.zeros(self.n, **kw) for _ in range(2)]      # pointer table: accepted state ...
        self.kbuf = [torch.zeros(self.n, **kw) for _ in range(2)]      # ... and its derivative f0 = k_0
        self.opt.ybuf[0], self.opt.ybuf[1] = self.ybuf[0].data_ptr(), self.ybuf[1].data_ptr()
        self.opt.kbuf[0], self.opt.kbuf[1] = self.kbuf[0].data_ptr(), self.kbuf[1].data_ptr()
        self.opt.always_fit = 1 if self.keep_interp else 0
        self.ytmp = torch.zeros(self.n, **kw)
        self.y1 = torch.zeros(self.n, **kw)
        self.errp = torch.zeros(self.n, **kw)                          # prefix of the error estimate
        if self.keep_interp:
            self.coeff = [torch.zeros(self.n, **kw) for _ in range(5)]
            self.coeff_ptrs = _lib.ptr_array([c.data_ptr() for c in self.coeff])
        else:
            self.coeff, self.coeff_ptrs = [], None
        self.partials = torch.zeros(self.lib.tdq_norm_partials_len(self.n, self.n_chunks), dtype=torch.float64,
                                    device=device)
        self.norm_out = torch.zeros(self.n_seg + 1, dtype=torch.float64, device=device)
        self.dsum = [torch.zeros(self.n_seg + 1, dtype=torch.float64, device=device) for _ in range(3)]
        self.kslots = {}                 # engine-owned stage slots (pieces path / aliasing outputs)
        self.qbuf = None
        self.ratio_buf = None
        if norm_fn is not None:
            qdt = dtype if not vtol else (torch.complex128 if dtype.is_complex else torch.float64)
            self.qbuf = torch.zeros(self.n, dtype=qdt, device=device)
            self.ratio_buf = torch.zeros((), dtype=torch.float64 if self.ratio_f64 else self.rdtype, device=device)
        self._own_ptrs = None
        self.mbox_host = C.POINTER(_lib.Mailbox)()
        mdev = C.c_void_p()
        _lib.check(self.lib.tdq_mailbox_create(C.byref(self.mbox_host), C.byref(mdev)))
        self.mbox_dev = mdev.value
        self.solution = None
        self._graph = None
        self._graph_failed = False
        self._graph_keep = None
        self._loop = None                # tdq_loop handle: the captured attempt inside a device-side while
        self._loop_handle = 0
        self._loop_failed = False
        self._always_copy = False        # set when func is seen to reuse its output buffer (see _call_fn)
        self.linear = None               # set_linear(): every stage fused with a linear field (csrc/tdq_linear.cu)
        self.capture_in_solve = True     # False: only a prime()d graph is used (solves run inside autograd backward)
        self.n_attempts = 0              # attempts that did work (from the mailbox counters)
        self.nfe = 0                     # func evaluations issued by the host
        self.nfe_total = 0
        self.launches = 0                # libtdq kernel launches issued (graph replays count their nodes)
        self._graph_launches = 0

    def __del__(self):
        try:
            if self.mbox_host:
                torch.cuda.synchronize(self.device)
                self._drop_graph()
                self.lib.tdq_mailbox_destroy(self.mbox_host)
                self.mbox_host = None
        except Exception:
            pass

    # ---------------------------------------------------------------------------------------
    def _call_fn(self, t, y, slot, taken=(), dst=None):
        """Evaluate func and return a tensor holding the flat result that is safe to keep as stage
        slot `slot` (rk_common.py:80-81 writes it into k[..., slot]): the reference COPIES f into k, so an
        output that aliases the solver's buffers, func's input, or an earlier stage's output (a func that
        returns y itself, or reuses one result buffer) must be copied here too."""
        self.nfe += 1
        f = self.fn(t, y)
        if isinstance(f, torch.Tensor):
            if f.dtype != self.dtype:
                f = f.to(self.dtype)
            f = f.reshape(-1)
            if f.numel() != self.n:
                raise ValueError("func returned %d elements for a state of %d" % (f.numel(), self.n))
            if f.data_ptr() in taken and not self._always_copy:
                # func reuses ONE output buffer: the earlier stage's values are already gone.  Nothing of this
                # attempt has been committed yet, so switch to copying every output and redo the attempt.
                self._always_copy = True
                raise _RetryWithCopies()
            if (self._always_copy or not f.is_contiguous() or (f.data_ptr() % 16) != 0 or self._aliases(f)
                    or f.data_ptr() in taken):
                buf = self._slot(slot)
                buf.copy_(f)
                f = buf
            return f
        # tuple of pieces -> one pack launch into an engine-owned slot
        buf = dst if dst is not None else self._slot(slot)
        self.launches += pack_pieces(self.lib, self.dt_code, self.dtype, buf, f, self.pieces)
        if self.post_fn is not None:
            self.post_fn(buf)
        return buf

    def set_linear(self, weight, whole_attempt=True, fused_controller=True):
        """Fuse the stage combination with func = y @ weight^T (torchdiffeq_b200.LinearField): tdq_linear_stage replaces
        tdq_stage_combine + the torch call for every row (rk_common.py:79-81 in one launch; csrc/tdq_linear.cu).
        For dopri5 / bosh3 the whole attempt -- every stage, the error norm, the candidate commit -- is ONE launch
        (tdq_linear_attempt, csrc/tdq_attempt.cu) unless whole_attempt=False.
        Returns False (and changes nothing) if a row of the tableau has more terms than the fused kernel takes."""
        width, S = int(weight.shape[0]), self.S
        if self.pieces is not None or self.post_fn is not None or self.n % width:
            return False
        beta, c_err = self.tab.beta, self.tab.c_err
        for i in range(S):
            used = {j for j in range(i + 1) if beta[i][j] != 0.0}
            if self.fsal and i == S - 1:
                used |= {j for j in range(S) if c_err[j] != 0.0}
            if not 1 <= len(used) <= 8:
                return False
        planes = torch.empty(int(self.lib.tdq_linear_weights_bytes(width)), dtype=torch.uint8, device=self.device)
        # the whole attempt in ONE launch (csrc/tdq_attempt.cu: all stages, error norm, candidate commit; FSAL tableaus of
        # at most 7 stages); the squared norm is folded in when it is the plain one (one segment, scalar tolerances)
        whole = bool(whole_attempt) and bool(self.lib.tdq_linear_attempt_supported(C.byref(self.tab), self.dt_code, width))
        fold = (whole and self.norm_table is None and self.n_seg == 1 and self.rtol_vec is None and self.norm_fn is None)
        self.linear = dict(weight=weight, width=width, planes=planes, whole=whole, fold=fold, ctrl=bool(fused_controller),
                           k=[torch.zeros(self.n, dtype=self.dtype, device=self.device) for _ in range(S)])
        self._drop_graph()
        return True

    def _eval(self, t, y, slot, dst=None):
        """func(t, y) before the first attempt (f0, the initial step's probe): the fused field's own kernel when there is
        one, so that a solve uses one arithmetic for every evaluation."""
        if self.linear is None:
            return self._call_fn(t, y, slot, dst=dst)
        self.nfe += 1
        out = dst if dst is not None else self._slot(slot)
        L = self.linear
        self._launch(self.lib.tdq_linear_apply(self.dt_code, y.data_ptr(), L["planes"].data_ptr(), L["width"],
                                               self.n // L["width"], out.data_ptr(), _stream()))
        return out

    @property
    def y0w(self):
        """The accepted state (valid between attempts in lock step, and after a solve)."""
        return self.ybuf[self.mbox_host.contents.par & 1]

    @property
    def k0(self):
        return self.kbuf[self.mbox_host.contents.par & 1]

    def _drop_graph(self):
        if self._loop is not None:
            try:
                self.lib.tdq_loop_destroy(self._loop)
            except Exception:
                pass
        self._loop, self._loop_handle = None, 0
        self._graph, self._graph_keep = None, None

    def _launch(self, rc):
        _lib.check(rc)
        self.launches += 1

    def _slot(self, i):
        if i not in self.kslots:
            self.kslots[i] = torch.zeros(self.n, dtype=self.dtype, device=self.device)
        return self.kslots[i]

    def _aliases(self, f):
        if self._own_ptrs is None:
            own = self.ybuf + self.kbuf + [self.ytmp, self.y1, self.errp, self.solution] + self.coeff
            self._own_ptrs = {t.untyped_storage().data_ptr() for t in own}
        return f.untyped_storage().data_ptr() in self._own_ptrs

    def _reduce(self, buf):
        if self.reduce_fn is not None:
            self.reduce_fn(buf)

    def _sumsq(self, x, x2, out):
        self._launch(self.lib.tdq_scaled_sumsq(
            self.ctrl.data_ptr(), self.dt_code, x.data_ptr(), x2.data_ptr() if x2 is not None else None,
            None,                                                     # y0: the control block's current pair
            self.rtol_vec.data_ptr() if self.rtol_vec is not None else None,
            self.atol_vec.data_ptr() if self.atol_vec is not None else None,
            self.norm_table.data_ptr() if self.norm_table is not None else None, self.n_chunks, self.table_aligned,
            self.n_seg, self.n, self.partials.data_ptr(), out.data_ptr(), _stream()))
        self._reduce(out)

    # ---------------------------------------------------------------------------------------
    def _attempt_front(self):
        """Stages, error norm, controller: everything up to the accept decision."""
        try:
            return self._attempt_front_once()
        except _RetryWithCopies:
            return self._attempt_front_once()

    def _attempt_front_once(self):
        lib, ctrl, tab, dc, st = self.lib, self.ctrl.data_ptr(), C.byref(self.tab), self.dt_code, _stream()
        S = self.S
        k = [None] * (S + 1)             # k[0] = NULL: the kernels read k_0 (and y0) through the pointer table
        keep = []
        folded = False
        if self.linear is not None and self.linear["whole"]:
            # the whole attempt in one tcgen05 launch (csrc/tdq_attempt.cu): the stages, y1 and the error prefix reach
            # memory only when an output time can fall into the attempt (or every step is kept)
            L = self.linear
            for i in range(S):
                k[i + 1] = L["k"][i].data_ptr()
            folded = L["fold"]
            # ... and the controller step too (the last block to finish runs it), unless a host-launched collective has to
            # reduce the norm sums between the two (NCCL / gloo exchange) or the caller asked for separate launches
            with_ctrl = folded and L["ctrl"] and (self.reduce_fn is None or self.exchange is not None)
            self._launch(lib.tdq_linear_attempt(ctrl, tab, dc, _lib.ptr_array(k), self.y1.data_ptr(), self.errp.data_ptr(),
                                                None, None, L["planes"].data_ptr(), L["width"], self.n,
                                                self.partials.data_ptr() if folded else None,
                                                self.norm_out.data_ptr() if folded else None,
                                                self.seg_counts.data_ptr() if with_ctrl else None,
                                                0 if folded else 1, st))
            self.nfe += S
            if with_ctrl:
                return k, _lib.ptr_array(k), keep
        elif self.linear is not None:
            # combination + evaluation of every row in one tcgen05 launch (csrc/tdq_linear.cu); the FSAL row also writes
            # y1 and the error-sum prefix exactly as tdq_stage_combine_final does
            L = self.linear
            for i in range(S):
                last = i == S - 1 and self.fsal
                out = L["k"][i]
                self._launch(lib.tdq_linear_stage(ctrl, tab, dc, i, out.data_ptr(),
                                                  self.y1.data_ptr() if last else None,
                                                  self.errp.data_ptr() if last else None, None, _lib.ptr_array(k),
                                                  L["planes"].data_ptr(), L["width"], self.n, st))
                self.nfe += 1
                k[i + 1] = out.data_ptr()
        for i in range(S if self.linear is None else 0):
            if i == S - 1 and self.fsal:
                # the row that yields y1, fused with the available prefix of the error estimate (rk_common.py:83-89)
                out = self.y1
                self._launch(lib.tdq_stage_combine_final(ctrl, tab, dc, out.data_ptr(), self.errp.data_ptr(), None,
                                                         _lib.ptr_array(k), self.n, st))
            else:
                out = self.ytmp
                self._launch(lib.tdq_stage_combine(ctrl, tab, dc, i, out.data_ptr(), None, _lib.ptr_array(k), self.n,
                                                   st))
            f = self._call_fn(self.tstage[i], out, i + 1, taken=k)
            keep.append(f)
            k[i + 1] = f.data_ptr()
        if not self.fsal:
            self._launch(lib.tdq_stage_combine_final(ctrl, tab, dc, self.y1.data_ptr(), self.errp.data_ptr(), None,
                                                     _lib.ptr_array(k), self.n, st))
        kp = _lib.ptr_array(k)
        # error ratio + candidate commit (y1 -> ybuf[par^1], k_S -> kbuf[par^1]) in one pass
        if not folded:
            self._launch(lib.tdq_error_norm_commit(
                ctrl, dc, self.errp.data_ptr(), k[S], None, self.y1.data_ptr(),
                self.rtol_vec.data_ptr() if self.rtol_vec is not None else None,
                self.atol_vec.data_ptr() if self.atol_vec is not None else None,
                self.norm_table.data_ptr() if self.norm_table is not None else None, self.n_chunks, self.table_aligned,
                self.n_seg, self.n, self.partials.data_ptr(), self.norm_out.data_ptr(),
                self.qbuf.data_ptr() if self.qbuf is not None else None, st))
        ratio_ptr = None
        if self.norm_fn is not None:
            r = self.norm_fn(self.q_view(self.qbuf))
            r = torch.as_tensor(r, device=self.device)
            self.ratio_buf.copy_(r.to(self.ratio_buf.dtype).reshape(()))
            ratio_ptr = self.ratio_buf.data_ptr()
        elif self.exchange is None:
            self._reduce(self.norm_out)
        self._launch(lib.tdq_controller(ctrl, self.rt_code, self.norm_out.data_ptr(), self.seg_counts.data_ptr(), self.n_seg,
                                      ratio_ptr, st))
        return k, kp, keep

    def _attempt_back(self, kp):
        """Dense output of the step just accepted -- a no-op on the device unless an output time fell into it (or
        the caller keeps the interpolant of every step)."""
        self._launch(self.lib.tdq_interp_fit_eval(self.ctrl.data_ptr(), C.byref(self.tab), self.dt_code,
                                                  self.y1.data_ptr(), kp, self.coeff_ptrs, self.solution.data_ptr(),
                                                  self.n, _stream()))

    def _attempt(self):
        k, kp, keep = self._attempt_front()
        self._attempt_back(kp)
        return keep

    # ---------------------------------------------------------------------------------------
    def _wait_seq(self, target):
        mb = self.mbox_host.contents
        spins = 0
        while mb.seq < target:
            spins += 1
            if spins > 2000:
                time.sleep(0)            # let other Python threads run; the GPU work is independent
                if spins % 20000 == 0 and torch.cuda.current_stream().query() and mb.seq < target:
                    # everything that was queued has run and the attempt never reported: fail instead of spinning forever
                    raise _lib.TdqError("the device finished the queued attempts without reporting attempt %d (mailbox at %d)"
                                        % (target, mb.seq))
        return mb

    def _raise_if_failed(self, mb):
        s = mb.status
        if s == _lib.RUN_OK:
            return
        torch.cuda.current_stream().synchronize()
        if s == _lib.RUN_DT_UNDERFLOW:
            raise SolverFailure("underflow in dt {}".format(mb.next_dt))
        if s == _lib.RUN_NONFINITE:
            raise SolverFailure("non-finite values in state `y`: {}".format(self.y0w))
        if s == _lib.RUN_EXCHANGE_TIMEOUT:
            raise _lib.TdqError("a peer rank did not deliver its norm partials within 10 s (sharded solve)")
        if s == _lib.RUN_MAX_STEPS:
            raise SolverFailure("max_num_steps exceeded ({}>={})".format(self.opt.max_num_steps, self.opt.max_num_steps))
        raise SolverFailure("solver failed with status %d" % s)

    def _lockstep_mode(self):
        return bool(self.callbacks) or self.run_ahead == 0

    def _use_loop(self):
        """Run this solve inside the device-side while loop?  Needs the captured attempt and a body without
        collectives launched by the host between attempts."""
        return (self._loop is not None and not self._lockstep_mode() and self.agree_fn is None
                and self.norm_fn is None)

    def solve(self, y0_flat, t64, t_start=None):
        """Integrate from t64[0] through t64[-1] (ascending float64 device tensor); returns
        solution [len(t), n] (solvers.py:28-35).  The returned tensor is owned by the engine and is
        overwritten by the next solve() with the same number of output times."""
        try:
            n_out = self._begin(y0_flat, t64, t_start, loop=self._use_loop())
            if n_out > 1:
                if self._lockstep_mode():
                    self._loop_lockstep()
                else:
                    self._loop_run_ahead()
        except BaseException:
            # attempts may still be queued: let them drain before anybody resets the mailbox, and do not let a
            # half-finished engine be reused (the caller evicts it from the cache)
            self.poisoned = True
            try:
                torch.cuda.current_stream().synchronize()
            except Exception:
                pass
            raise
        mb = self.mbox_host.contents
        self.n_accept, self.n_reject = int(mb.n_accept), int(mb.n_reject)
        self.n_attempts = self.n_accept + self.n_reject
        return self.solution

    def prime(self, y0_flat, t64, t_start=None):
        """Warm up and capture the attempt graph ahead of time on representative inputs (one eager
        attempt, then capture).  Used by odeint_adjoint to capture the backward step body during the
        FORWARD call: capturing inside autograd's backward is unsafe (a re-entrant engine call may run
        unrelated nodes of the outer graph on the legacy stream in the middle of the capture)."""
        if self.graph_opt not in (True, "auto") or self._lockstep_mode():
            return False
        n_out = self._begin(y0_flat, t64, t_start)
        if n_out <= 1:
            return False
        self._warm_attempt()
        self._capture()
        torch.cuda.current_stream().synchronize()
        return self._graph is not None

    def _begin(self, y0_flat, t64, t_start=None, loop=False):
        """Everything of a solve that precedes the first attempt (rk_common.py:166-241)."""
        lib = self.lib
        self.nfe_total += self.nfe
        self.nfe, self.launches = 0, 0                  # per-solve counters (engines are reused)
        n_out = int(t64.numel())
        self.t_out = t64.contiguous()
        if getattr(self, "solution", None) is None or self.solution.shape[0] != n_out:
            # a captured graph holds this buffer's address: a new shape invalidates it
            self.solution = torch.empty(n_out, self.n, dtype=self.dtype, device=self.device)
            self._drop_graph()
            self._own_ptrs = None
            loop = False
        self.solution[0].copy_(y0_flat)
        self.ybuf[0].copy_(y0_flat)
        st = _stream()
        mb = self.mbox_host.contents
        mb.seq, mb.status, mb.done, mb.par, mb.accept = 0, 0, 0, 0, 0
        mb.n_accept, mb.n_reject = 0, 0
        if t_start is None:
            t_start = float(t64[0])                                   # callers pass it whenever they hold t on the host
        self.opt.loop_handle = self._loop_handle if loop else 0
        _lib.check(lib.tdq_ctrl_init(self.ctrl.data_ptr(), C.byref(self.tab), C.byref(self.opt),
                                     self.t_out.data_ptr(), float(t_start), n_out, self.mbox_dev, st))
        if self.exchange is not None:
            self.exchange.arm(self.ctrl.data_ptr(), st)
        if self.jump_t is not None and self.jump_t.numel() > 0:
            self._launch(lib.tdq_ctrl_set_jump_t(self.ctrl.data_ptr(), self.jump_t.data_ptr(),
                                                 int(self.jump_t.numel()), st))
        if self.step_t is not None and self.step_t.numel() > 0:
            self._launch(lib.tdq_ctrl_set_step_t(self.ctrl.data_ptr(), self.step_t.data_ptr(),
                                               int(self.step_t.numel()), st))
        dc, ctrl = self.dt_code, self.ctrl.data_ptr()
        if self.linear is not None:                                   # the weight may have changed since the last solve
            L = self.linear
            self._launch(lib.tdq_linear_prepare(dc, L["weight"].data_ptr(), L["width"], L["planes"].data_ptr(), st))

        # _before_integrate: f0 and the initial step (rk_common.py:213-221, misc.py:36-77)
        f0 = self._eval(self.taux[0], self.ybuf[0], 0, dst=self.kbuf[0])
        if f0.data_ptr() != self.kbuf[0].data_ptr():
            self.kbuf[0].copy_(f0)
        del f0
        # d0's pass over y0 also counts its non-finite elements: rk_common.py:287 for the first attempt is then
        # checked on the device by tdq_prepare_attempt, where the reference asserts it (no host sync here)
        self._sumsq(self.ybuf[0], None, self.dsum[0])
        if self.first_step is None:
            if self.norm_fn is not None:
                self._initial_step_custom_norm()
            else:
                self._sumsq(self.kbuf[0], None, self.dsum[1])
                self._launch(lib.tdq_initial_step_h0(ctrl, self.rt_code, self.dsum[0].data_ptr(), self.dsum[1].data_ptr(),
                                                   self.seg_counts.data_ptr(), self.n_seg, st))
                self._launch(lib.tdq_initial_step_probe(ctrl, dc, self.ytmp.data_ptr(), None, None, self.n, st))
                f1 = self._eval(self.taux[1], self.ytmp, 1)
                self._sumsq(f1, self.kbuf[0], self.dsum[2])
                del f1
                self._launch(lib.tdq_initial_step_finish(ctrl, self.rt_code, self.dsum[2].data_ptr(),
                                                       self.seg_counts.data_ptr(), self.n_seg, st))
        else:
            self._launch(lib.tdq_set_first_step(ctrl, float(self.first_step), st))
        bad_ptr = self.dsum[0].data_ptr() + 8 * self.n_seg if n_out > 1 else None
        self._launch(lib.tdq_prepare_attempt(ctrl, self.rt_code, bad_ptr, st))
        return n_out

    # ---- lock step: the reference's exact call sequence --------------------------------------
    def _lockstep_attempt(self, issued, mb):
        """One attempt in the reference's exact call order (rk_common.py:266-361): callbacks, stages, the
        accept decision read from the mailbox, accepted-step work, the f re-evaluation after a jump."""
        cb = self.callbacks
        if cb.get("callback_step") is not None:             # rk_common.py:272
            cb["callback_step"](*self._with_y(mb.next_t0, mb.next_dt))
        k, kp, keep = self._attempt_front()
        issued += 1
        mb = self._wait_seq(issued)
        self._raise_if_failed(mb)
        if cb:
            name = "callback_accept_step" if mb.accept else "callback_reject_step"   # :339, :354
            if cb.get(name) is not None:
                cb[name](*self._with_y(mb.att_t0, mb.att_dt))
        jumped = bool(mb.accept) and bool(mb.on_jump_t)
        self._attempt_back(kp)
        del k, kp, keep
        if jumped:                                          # rk_common.py:346-351: f on the far side of the jump
            k0 = self.k0
            f = self._call_fn(self.taux[2], self.y0w, 0, dst=k0)
            if f.data_ptr() != k0.data_ptr():
                k0.copy_(f)
            del f
        return issued, mb

    def _loop_lockstep(self):
        issued = 0
        torch.cuda.current_stream().synchronize()          # first attempt's (t0, dt) and status are in the mailbox
        mb = self.mbox_host.contents
        self._raise_if_failed(mb)
        while True:
            issued, mb = self._lockstep_attempt(issued, mb)
            if mb.done:
                break
        torch.cuda.current_stream().synchronize()

    # ---- dense output (odeint.py:111-157) ------------------------------------------------------------
    def solve_dense(self, y0_flat, t64):
        """Lock-step solve that keeps the interpolant of EVERY accepted step: returns (solution, times, coeffs)
        with times[i], times[i+1] bounding accepted step i and coeffs[i] its five coefficient arrays."""
        n_out = self._begin(y0_flat, t64)
        torch.cuda.current_stream().synchronize()
        mb = self.mbox_host.contents
        self._raise_if_failed(mb)
        times, coeffs, issued = [float(t64[0])], [], 0
        while n_out > 1:
            issued, mb = self._lockstep_attempt(issued, mb)
            if mb.accept:                                                   # odeint.py:141-145
                times.append(float(mb.t1))
                coeffs.append([c.clone() for c in self.coeff])
            if mb.done:
                break
        torch.cuda.current_stream().synchronize()
        return self.solution, times, coeffs

    # ---- taped solve for the differentiable (non-adjoint) odeint (torchdiffeq_b200/backprop.py) ------------------
    def solve_taped(self, y0_flat, t64, t_start=None):
        """Lock-step solve that records every ACCEPTED step: start time, step size, the (y0, k_0) pair it started from
        (clones: 2 n elements per step), the output rows it produced and whether it followed a jump_t re-evaluation.
        Returns (solution, tape)."""
        n_out = self._begin(y0_flat, t64, t_start)
        torch.cuda.current_stream().synchronize()
        mb = self.mbox_host.contents
        self._raise_if_failed(mb)
        tape, issued, cursor, first, jumped = [], 0, 1, True, None
        while n_out > 1:
            issued, mb = self._lockstep_attempt(issued, mb)
            if mb.accept:
                prev = (mb.par ^ 1) & 1                                     # the pair the accepted step started from
                k0 = self.kbuf[prev]
                tape.append(dict(t0=float(mb.att_t0), dt=float(mb.att_dt), y0=self.ybuf[prev].clone(), k0=k0.clone(),
                                 out_lo=cursor, out_hi=int(mb.out_cursor), first=first, jumped_into=jumped))
                cursor, first = int(mb.out_cursor), False
                jumped = True if mb.on_jump_t else None
            if mb.done:
                break
        torch.cuda.current_stream().synchronize()
        self.n_accept, self.n_reject = int(mb.n_accept), int(mb.n_reject)
        self.n_attempts = self.n_accept + self.n_reject
        return self.solution, tape

    # ---- event handling (solvers.py:38-49, rk_common.py:252-264, event_handling.py:5-20) ----------------
    def solve_until_event(self, y0_flat, t0, event_fn, tol):
        """Integrate from t0 until event_fn(t, y) changes sign, then bisect on the dense output of the last
        step.  event_fn takes a 0-dim float64 device tensor (ascending solver time) and the flat state.
        Host driven by nature (a sign test per step); returns (event_t as float, y(event_t) tensor)."""
        t64 = torch.tensor([float(t0), float("inf")], dtype=torch.float64, device=self.device)
        self._begin(y0_flat, t64, float(t0))
        torch.cuda.current_stream().synchronize()
        mb = self.mbox_host.contents
        self._raise_if_failed(mb)
        tt = lambda v: torch.tensor(v, dtype=torch.float64, device=self.device)
        t_cur = float(t0)
        if bool(event_fn(tt(t_cur), self.y0w) == 0):                         # rk_common.py:254-255
            return t_cur, self.y0w.clone()
        sign0 = torch.sign(event_fn(tt(t_cur), self.y0w))
        issued = 0
        while bool(sign0 == torch.sign(event_fn(tt(t_cur), self.y0w))):      # :259
            issued, mb = self._lockstep_attempt(issued, mb)
            t_cur = mb.t1
        torch.cuda.current_stream().synchronize()
        self.n_accept, self.n_reject = int(mb.n_accept), int(mb.n_reject)
        self.n_attempts = self.n_accept + self.n_reject
        # find_event (event_handling.py:5-20): bisection on [t0, t1] of the last accepted step
        lo, hi = float(mb.t0), float(mb.t1)
        import math
        nitrs = int(math.ceil(math.log((hi - lo) / float(tol)) / math.log(2.0)))
        y_mid = torch.empty(self.n, dtype=self.dtype, device=self.device)

        def interp(t_eval):
            self._launch(self.lib.tdq_interp_eval_at(self.ctrl.data_ptr(), self.dt_code, self.coeff_ptrs,
                                                     tt(t_eval).data_ptr(), y_mid.data_ptr(), self.n, _stream()))
            return y_mid
        for _ in range(max(nitrs, 0)):
            t_mid = (hi + lo) / 2.0
            same = bool(sign0 == torch.sign(event_fn(tt(t_mid), interp(t_mid))))
            if same:
                lo = t_mid
            else:
                hi = t_mid
        event_t = (lo + hi) / 2.0
        return event_t, interp(event_t).clone()

    def _with_y(self, t0, dt):
        t0, dt = self._scalars(t0, dt)
        return t0, self.y0w, dt

    def _scalars(self, t0, dt):
        """0-dim float64 device tensors, as the reference passes (t0, dt) to callbacks."""
        kw = dict(dtype=torch.float64, device=self.device)
        return torch.tensor(t0, **kw), torch.tensor(dt, **kw)

    # ---- bounded run-ahead: no host sync, optional CUDA graph -----------------------------------
    def _loop_run_ahead(self):
        D = max(1, self.run_ahead)
        mb = self.mbox_host.contents
        issued = 0
        use_graph = self.graph_opt in (True, "auto") and not self._graph_failed and self.capture_in_solve
        if self._use_loop() and self.opt.loop_handle != 0:
            # the whole adaptive loop is ONE graph launch: a conditional WHILE node around the captured attempt,
            # re-armed by k_controller until the solve has finished or failed
            self._launch_loop()
            return
        # attempt 1 runs eagerly: it is a real attempt and doubles as the warm-up torch wants before capture
        if self._graph is None:
            if use_graph:
                self._warm_attempt()
                self._capture()
            else:
                self._attempt()
            issued += 1
            if self._use_loop():
                # hand the rest of this solve to the loop (if the first attempt already finished it, the loop's
                # single iteration is a no-op on the device)
                _lib.check(self.lib.tdq_ctrl_set_loop(self.ctrl.data_ptr(), self._loop_handle, _stream()))
                self._launch_loop(first=1)
                return
        while True:
            seen = mb.seq
            if mb.status != _lib.RUN_OK or mb.done:
                break
            if issued - seen > D:
                time.sleep(0)                              # the device is >D attempts behind: yield the GIL
                continue
            if self._graph is not None:
                self._graph.replay()
                self.nfe += self.S
                self.launches += self._graph_launches
            else:
                self._attempt()
            issued += 1
        if self.agree_fn is not None:
            # every attempt holds a collective: all ranks must have queued the same number before anyone
            # waits for its stream (trailing attempts are no-ops on the device)
            target = self.agree_fn(issued)
            while issued < target:
                if self._graph is not None:
                    self._graph.replay()
                    self.nfe += self.S
                    self.launches += self._graph_launches
                else:
                    self._attempt()
                issued += 1
        mb = self._wait_seq(issued)
        self._raise_if_failed(mb)
        torch.cuda.current_stream().synchronize()

    def _launch_loop(self, first=0):
        _lib.check(self.lib.tdq_loop_launch(self._loop, _stream()))
        torch.cuda.current_stream().synchronize()
        mb = self.mbox_host.contents
        ran = int(mb.seq) - first
        self.nfe += self.S * ran
        self.launches += self._graph_launches * ran
        self._raise_if_failed(mb)

    def _warm_attempt(self):
        """The first attempt of a solve that is about to be captured: a real attempt that doubles as the
        warm-up torch wants before capture (we are already on the solver stream, never the legacy one)."""
        self._attempt()

    def _capture(self):
        """Capture one attempt.  A first capture that involves autograd (the adjoint's augmented dynamics)
        can be invalidated by one-time initialisation inside autograd's worker thread that no eager
        warm-up reaches; nothing has executed at that point and the engine state is untouched, so the
        capture is simply retried once before giving up."""
        last = None
        for _try in range(2):
            try:
                want_loop = (self.device_loop in (True, "auto") and not self._loop_failed and self.agree_fn is None
                             and self.norm_fn is None)
                g = torch.cuda.CUDAGraph(keep_graph=True) if want_loop else torch.cuda.CUDAGraph()
                nfe, launches = self.nfe, self.launches
                try:
                    with torch.cuda.graph(g, stream=solver_stream(self.device)):
                        keep = self._attempt()
                finally:
                    self._graph_launches = self.launches - launches
                    self.nfe, self.launches = nfe, launches     # capture runs no kernels
                self._graph, self._graph_keep = g, keep
                if want_loop:
                    self._make_loop(g)
                return
            except Exception as e:                              # func is not capturable: stay eager
                last = e
                self._graph = None
                torch.cuda.synchronize(self.device)
        self._graph_failed = True
        if self.graph_opt is True:
            raise last
        import warnings
        warnings.warn("torchdiffeq_b200: CUDA graph capture of the step body failed (%s: %s); "
                      "continuing with eager launches" % (type(last).__name__, last))

    def _make_loop(self, g):
        """Wrap the captured attempt into a device-side while loop (tdq_loop_create).  The body is a clone of
        torch's graph; torch's CUDAGraph object stays alive because it owns the memory pool the body uses."""
        loop, handle = C.c_void_p(), C.c_uint64()
        try:
            _lib.check(self.lib.tdq_loop_create(C.c_void_p(g.raw_cuda_graph()), C.byref(loop), C.byref(handle)))
            self._loop, self._loop_handle = loop.value, int(handle.value)
        except Exception as e:
            self._loop, self._loop_handle, self._loop_failed = None, 0, True
            if self.device_loop is True:
                raise
            import warnings
            warnings.warn("torchdiffeq_b200: the captured step could not be wrapped into a device-side loop "
                          "(%s: %s); the host replays it instead" % (type(e).__name__, e))

    def _initial_step_custom_norm(self):
        """misc.py:36-77 with a user norm callable: torch ops + one host read (compatibility path)."""
        T = self.rdtype
        y0, f0 = self.ybuf[0], self.kbuf[0] * self.opt.t_sign
        if self.rtol_vec is not None:
            scale = self.atol_vec + torch.abs(y0) * self.rtol_vec
        else:
            scale = float(self.opt.atol) + torch.abs(y0) * float(self.opt.rtol)
        nf = lambda v: torch.as_tensor(self.norm_fn(self.q_view(v)), device=self.device).abs()
        d0, d1 = nf(y0 / scale), nf(f0 / scale)
        if d0 < 1e-5 or d1 < 1e-5:
            h0 = torch.tensor(1e-6, dtype=T, device=self.device)
        else:
            h0 = 0.01 * d0 / d1
        h0 = h0.abs()
        self.ytmp.copy_(y0 + h0 * f0)
        t0 = float(self.t_out[0])
        self.taux[1] = (torch.tensor(t0, dtype=torch.float64, device=self.device) + h0.double()).to(T) * self.opt.t_sign
        f1 = self._call_fn(self.taux[1], self.ytmp, 1) * self.opt.t_sign
        d2 = torch.abs(nf((f1 - f0) / scale) / h0)
        order = self.tab.order - 1
        if d1 <= 1e-15 and d2 <= 1e-15:
            h1 = torch.max(torch.tensor(1e-6, dtype=T, device=self.device), h0 * 1e-3)
        else:
            h1 = (0.01 / max(d1, d2)) ** (1. / float(order + 1))
        h1 = h1.abs()
        dt = float(torch.min(100 * h0, h1).to(torch.float64))
        self._launch(self.lib.tdq_set_first_step(self.ctrl.data_ptr(), dt, _stream()))
