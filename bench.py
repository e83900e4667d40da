#!/usr/bin/env python
"""bench.py -- trajectories/sec of the dopri5 hot path on BASELINE.json's configs[1]
(dopri5 adaptive, batch=65536 dim=128 linear ODE y' = A y, float32, rtol=1e-5, atol=1e-7, t in [0, 10]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one complete odeint solve of the batch (about 74 step attempts, 446 func evaluations).
N > 1 (torchrun, one rank per GPU): every rank integrates its own 65536 trajectories (weak scaling,
configs[4] at N=8) and the ranks share one scalar all-reduce per attempt so that all take the common
dt of the unsharded problem.

The vector field is `torchdiffeq_b200.LinearField(A)` -- an nn.Module with forward(t, y) = y @ A^T that the reference runs
unchanged -- so every Runge-Kutta stage (combination + field evaluation) is ONE tcgen05 kernel (csrc/tdq_linear.cu).
`--generic` keeps func an opaque torch module (the path any other func takes: k_combine + the user's kernels); the default
run times that path too and reports it as `generic_path`.

Prints ONE JSON line (rank 0).  `value` is measured with inputs resident in HBM; `e2e` goes through the
public API with pinned HOST buffers (H2D of y0 and D2H of y(t_end) inside the timed region);
`roofline` is the dominant kernel group's algorithmic bytes / its CUDA-event time against the measured
HBM peak; `cpu_baseline` is the unmodified reference (baseline/_ref; the CPU oracle only if it did not travel) on a bounded
sample.  --impl reference times that CPU implementation alone on the host cores.

--dump-outputs DIR writes the solution the last timed step returned as DIR/solution.npy (float32, the rows of a
fixed seeded sample of the trajectories, see dump_outputs), so that two builds can be compared output for output:
the inputs are the same in every run with the same arguments.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

B_PER_GPU, DIM = 65536, 128
T_SPAN = (0.0, 10.0)
RTOL, ATOL = 1e-5, 1e-7
METRIC = "trajectories/sec (dopri5, batch=65536 dim=128)"


def make_problem(device, batch, rank=0, world=1, fused=False):
    """The workload: ONE seeded batch of `batch * world` trajectories (SURVEY.md 8(d) C2/C5: y0 = randn, generator
    seed 1); rank r owns rows [r*batch, (r+1)*batch).  Returns (func, this rank's rows, t, the whole batch).
    fused: func is torchdiffeq_b200.LinearField(A) (same matrix, same mathematics: y @ A^T) instead of the plain module."""
    import problems as P
    if fused:
        import torchdiffeq_b200 as tdq
        f = tdq.LinearField(P.skew_matrix(DIM, torch.float32).to(device))
    else:
        f = P.BatchedLinear(DIM, torch.float32).to(device)
    g = torch.Generator().manual_seed(1)
    y_all = torch.randn(batch * world, DIM, generator=g)
    y0 = y_all[rank * batch:(rank + 1) * batch].contiguous()
    t = torch.tensor(T_SPAN)
    return f, y0, t, y_all


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_tensor_peak():
    """Dense bf16 TFLOP/s: the burst figure (the probe times the kernel alone, a few milliseconds)."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            v = json.load(f).get("bf16_tflops")
        if v:
            return float(v), "measured (MEASURED_PEAKS.json bf16_tflops, burst)"
    return 1700.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 6 for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# DRAM traffic of the six stage-combine launches of one attempt, from the committed ncu capture; a literal, labelled as such
TRAFFIC_STATIC = {"bytes": 928.4e6, "source": "static: dram__bytes_read+write of the six launches from ncu --set full captures "
                                                "(profiles/r2_ncu_full_summary.csv for k_combine<5> 209.3 MB and k_combine_final 216.5 MB, "
                                                "profiles/r1_ncu_full_summary.csv for rows NK=1..4); not measured by this run"}
# the six fused launches (k_linear_stage) of one attempt: filled from the ncu --set full capture under profiles/ (see there)
TRAFFIC_FUSED = {"bytes": 946.1e6, "source": "static: dram__bytes_read+write of the six k_linear_stage launches of one attempt, ncu --set full "
                                               "(profiles/r2_ncu_full_fused_rows_summary.csv: reads 873 MB = the algorithmic reads, writes 73 MB -- most "
                                               "of the 268 MB written is still in L2 when a kernel ends); not measured by this run"}
# the whole-attempt launch (k_linear_attempt): from the ncu --set full capture under profiles/
TRAFFIC_ATTEMPT = {"bytes": 82.8e6, "source": "static: dram__bytes_read.sum 67.4 MB (= y0 + k_0, the algorithmic reads) + dram__bytes_write.sum "
                                                  "15.4 MB of one k_linear_attempt launch, ncu --set full (profiles/r2_ncu_full_k_linear_attempt_raw.csv): "
                                                  "most of the 67 MB of candidates it writes is still in L2 when the launch ends; not measured by this run"}
DUMP_ROWS = 32768          # trajectories kept by --dump-outputs: [len(t), 32768, 128] float32 = 33.5 MB
FULL_ATTEMPTS = 74         # step attempts of the full workload (reference, oracle and CUDA path agree; SURVEY.md section 6)
CPU_SAMPLE_T_END = 1.0     # the CPU sample integrates the FULL batch over t in [0, 1] (9 of the 74 attempts, + the start-up work)
REF_DIR = os.path.join(ROOT, "baseline", "_ref")      # the unmodified reference, `pip install --target` (DESIGN.md section 7)


def cpu_threads():
    """Intra-op threads for the CPU arm.  The reference's path is ~570 small ATen calls per step; on a
    many-core host torch's thread pool stops scaling (and then collapses) well before the core count
    -- measured on the 128-core GPU box: 0.15 s at 8 and 16 threads, 0.28 s at 32, 0.78 s at 64 for a
    B=1024 solve, minutes at 128 -- so the baseline uses the best setting, 16, not the worst."""
    return max(1, min(os.cpu_count() or 1, 16))


def reference_package():
    """The unmodified reference package if it travelled with the repo (baseline/_ref), else None."""
    if os.path.isdir(os.path.join(REF_DIR, "torchdiffeq")):
        if REF_DIR not in sys.path:
            sys.path.insert(0, REF_DIR)
        import torchdiffeq
        return torchdiffeq
    return None


class _Rec(torch.nn.Module):
    """Counts step attempts through the reference's own callbacks (misc.py:311-332)."""

    def __init__(self, f):
        super().__init__()
        self.f, self.n_accept, self.n_reject = f, 0, 0

    def forward(self, t, y):
        return self.f(t, y)

    def callback_accept_step(self, t0, y0, dt):
        self.n_accept += 1

    def callback_reject_step(self, t0, y0, dt):
        self.n_reject += 1


def dump_outputs(path, solution):
    """Writes the solution [len(t), batch, DIM] as path/solution.npy in float32: the rows of DUMP_ROWS trajectories
    drawn once from a generator with a fixed seed (in ascending order), the same rows in every run."""
    import numpy as np
    n = solution.shape[1]
    rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:min(n, DUMP_ROWS)].sort().values
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "solution.npy"), solution.detach().cpu()[:, rows].to(torch.float32).numpy())


def cpu_run(batch, threads, t_end=T_SPAN[1]):
    """One solve of the workload at `batch` rows over t in [0, t_end] on the host cores: the unmodified reference
    when available (kind 'reference'), else the CPU oracle (kind 'port').  Returns (seconds, attempts, kind, solution)."""
    torch.set_num_threads(threads)
    f, y0, _, _ = make_problem("cpu", batch)
    t = torch.tensor([T_SPAN[0], t_end])
    ref = reference_package()
    with torch.no_grad():
        if ref is not None:
            rec = _Rec(f)
            t0 = time.perf_counter()
            sol = ref.odeint(rec, y0, t, method="dopri5", rtol=RTOL, atol=ATOL)
            dt = time.perf_counter() - t0
            return dt, rec.n_accept + rec.n_reject, "reference", sol
        from oracle import ode_oracle as O
        r = {}
        t0 = time.perf_counter()
        sol = O.odeint_adaptive(f, y0, t, "dopri5", rtol=RTOL, atol=ATOL, record=r)
        dt = time.perf_counter() - t0
        return dt, r["n_accept"] + r["n_reject"], "port", sol


def cpu_sample(threads):
    """Bounded CPU sample of the workload: all 65536 rows (so the arrays are as cache-unfriendly as in the real
    job -- a smaller batch fits the host's L3 and runs up to 10x faster per row), but only the first part of the
    time span; the per-attempt cost is constant, so a sample that completes a/74 of every trajectory's attempts in
    s seconds runs at B*(a/74)/s trajectories per second.  Also returns the sample's solution."""
    secs, attempts, kind, sol = cpu_run(B_PER_GPU, threads, CPU_SAMPLE_T_END)
    value = B_PER_GPU * (attempts / FULL_ATTEMPTS) / secs
    desc = ("all %d rows, t in [0,%g]: %d of the %d step attempts per sample, %.2f s per sample; "
            "value = rows x (attempts/74) / seconds" % (B_PER_GPU, CPU_SAMPLE_T_END, attempts, FULL_ATTEMPTS, secs))
    return value, secs, desc, kind, sol


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (baseline/_ref; the oracle port only if the
    package did not travel) on the host cores.  A step = one bounded sample (see cpu_sample); ms_per_step is the
    measured time of a sample, so steps x ms_per_step is the real timed region."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = cpu_threads()
    warm = max(1, min(args.warmup, 2))            # the CPU path has no lazy initialisation beyond its first call
    for _ in range(warm):
        cpu_sample(threads)
    steps = args.steps
    vals, secs = [], []
    for _ in range(steps):
        v, s_, desc, kind, sol = cpu_sample(threads)
        vals.append(v)
        secs.append(s_)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, sol)
    value = sum(vals) / len(vals)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "trajectories/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": 1e3 * sum(secs) / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1]: dopri5 linear ODE batch=65536 dim=128 f32 rtol=1e-5 atol=1e-7 t=[0,10]",
                   "sample": desc, "full_solve_ms_at_this_rate": 1e3 * B_PER_GPU / value,
                   "note": "a step is one bounded sample; ms_per_step is its measured time"},
        "cpu_baseline": {"value": value, "unit": "trajectories/s", "cores": threads, "kind": kind, "sample": desc},
        "e2e": {"value": value, "unit": "trajectories/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def roofline_probe(dev, n_elems, reps=20):
    """CUDA-event time of the stage-combine and error-norm launches of ONE dopri5 attempt at the benchmark's
    size, issued through the C ABI on buffers larger than L2 (9 arrays x 33.5 MB).  Returns per-launch
    (ms per attempt) for the 6 combine rows alone and for combine + error norm."""
    from torchdiffeq_b200 import _lib
    from torchdiffeq_b200._engine import AdaptiveEngine, _stream
    eng = AdaptiveEngine(lambda t, y: y, n_elems, torch.float32, dev, "dopri5", rtol=RTOL, atol=ATOL, first_step=0.05)
    eng.t_out = torch.tensor([0.0, 10.0], dtype=torch.float64, device=dev)
    eng.solution = torch.zeros(2, 4, dtype=torch.float32, device=dev)
    lib = eng.lib
    _lib.check(lib.tdq_ctrl_init(eng.ctrl.data_ptr(), C.byref(eng.tab), C.byref(eng.opt), eng.t_out.data_ptr(), 0.0, 2,
                                 eng.mbox_dev, _stream()))
    _lib.check(lib.tdq_set_first_step(eng.ctrl.data_ptr(), 0.05, _stream()))
    _lib.check(lib.tdq_prepare_attempt(eng.ctrl.data_ptr(), eng.dt_code, None, _stream()))
    ks = [torch.randn(n_elems, device=dev) * 1e-3 for _ in range(7)]
    y0 = torch.randn(n_elems, device=dev)
    outs = [torch.empty(n_elems, device=dev) for _ in range(2)]
    kp = _lib.ptr_array([k.data_ptr() for k in ks])
    ctrl, tab, dc = eng.ctrl.data_ptr(), C.byref(eng.tab), eng.dt_code

    errp = torch.empty(n_elems, device=dev)

    def combine(row):
        if row == 5:       # the row that yields y1, fused with the prefix of the error estimate (one extra N*s write)
            _lib.check(lib.tdq_stage_combine_final(ctrl, tab, dc, outs[1].data_ptr(), errp.data_ptr(), y0.data_ptr(), kp,
                                                   n_elems, _stream()))
        else:
            _lib.check(lib.tdq_stage_combine(ctrl, tab, dc, row, outs[row & 1].data_ptr(), y0.data_ptr(), kp, n_elems,
                                             _stream()))

    def norm():            # error ratio + candidate commit (y1, k_S -> the other pair of the pointer table)
        _lib.check(lib.tdq_error_norm_commit(ctrl, dc, errp.data_ptr(), ks[6].data_ptr(), y0.data_ptr(),
                                             outs[1].data_ptr(), None, None, None, 0, 0, 1, n_elems,
                                             eng.partials.data_ptr(), eng.norm_out.data_ptr(), None, _stream()))
    rows = [lambda r=r: combine(r) for r in range(6)]

    def timed(fns, reps):
        """Back-to-back launches between two events on the launching stream: the queue stays full, so the
        time is device time (a per-launch event pair would add the host's launch latency to every kernel)."""
        for fn in fns:
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            for fn in fns:
                fn()
        b.record()
        b.synchronize()
        return a.elapsed_time(b) / reps

    # every pass over the six rows touches 9 distinct 33.5 MB arrays (>> 126 MB L2), like a real attempt
    comb_ms = timed(rows, reps)
    group_ms = timed(rows + [norm], reps)
    res = {"comb_ms": comb_ms, "group_ms": group_ms}
    if lib.tdq_linear_supported(dc, DIM):
        # the fused rows of one attempt as the engine issues them: row i reads y0, k_0..k_i and writes k_{i+1}
        # (producer -> consumer through memory, 9 + 2 distinct arrays); the last row also writes y1 and the error prefix
        W = torch.randn(DIM, DIM, device=dev) * 0.09
        planes = torch.empty(int(lib.tdq_linear_weights_bytes(DIM)), dtype=torch.uint8, device=dev)
        _lib.check(lib.tdq_linear_prepare(dc, W.data_ptr(), DIM, planes.data_ptr(), _stream()))

        def fused_row(row):
            last = row == 5
            _lib.check(lib.tdq_linear_stage(ctrl, tab, dc, row, ks[row + 1].data_ptr(), outs[1].data_ptr() if last else None,
                                            errp.data_ptr() if last else None, y0.data_ptr(), kp, planes.data_ptr(), DIM,
                                            n_elems, _stream()))
        frows = [lambda r=r: fused_row(r) for r in range(6)]
        res["fused_ms"] = timed(frows, reps)
        res["fused_group_ms"] = timed(frows + [norm], reps)
        if lib.tdq_linear_attempt_supported(tab, dc, DIM):
            # the WHOLE attempt in one launch (csrc/tdq_attempt.cu), as the engine issues it: the squared error norm and the
            # candidate commit folded in, stages not stored.  Three rotating (y0, k_0) input pairs (201 MB) + the 67 MB of
            # candidates it writes: nothing a launch reads is left in L2 by the previous one
            pairs = [(y0, ks[0]), (ks[1], ks[2]), (ks[3], ks[4])]
            kout = _lib.ptr_array([None] + [ks[6].data_ptr()] * 6)

            def attempt(pair):
                _lib.check(lib.tdq_linear_attempt(ctrl, tab, dc, kout, outs[1].data_ptr(), errp.data_ptr(), pair[0].data_ptr(),
                                                  pair[1].data_ptr(), planes.data_ptr(), DIM, n_elems, eng.partials.data_ptr(),
                                                  eng.norm_out.data_ptr(), None, 0, _stream()))
            res["attempt_ms"] = timed([lambda p=p: attempt(p) for p in pairs], reps) / len(pairs)
    return res


def run_ours(args):
    import torch.distributed as dist
    import torchdiffeq_b200 as tdq
    from torchdiffeq_b200 import _lib
    _lib.load()                                       # fail loudly if the CUDA library is missing
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pg = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        pg = True
    strong = args.scaling == "strong"
    if strong:
        assert B_PER_GPU % world == 0
    rows = B_PER_GPU // world if strong else B_PER_GPU      # strong: the 65,536 trajectories are split over the ranks
    fused = not args.generic
    f, y0_host, t, y_all = make_problem(dev, rows, rank, world, fused=fused)
    y0_host = y0_host.pin_memory()
    y0 = y0_host.to(dev)
    t_dev = t.to(dev)
    opts = {"graph": True, "run_ahead": 2, "device_loop": not args.no_device_loop}
    if args.no_fused_controller:
        opts["fused_controller"] = False
    if pg:
        opts["process_group"] = pg
    stats = {}

    def solve(y, func=None, st=None):
        with torch.no_grad():
            return tdq.odeint(func if func is not None else f, y, t_dev, method="dopri5", rtol=RTOL, atol=ATOL,
                              options=dict(opts), _stats=st if st is not None else stats)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    W = max(3, args.warmup)
    for _ in range(W):
        out = solve(y0)
    barrier()
    # ---- device-resident metric ------------------------------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = stats.get("launches", 0)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        out = solve(y0)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)
    launches = stats.get("launches", 0) - launches0
    clocks = sampler.stop() if rank == 0 else None
    # ---- end to end: pinned host y0 -> device -> solve -> y(t_end) back to pinned host -----------------
    res_host = torch.empty(rows, DIM, dtype=torch.float32).pin_memory()
    for _ in range(2):
        res_host.copy_(solve(y0_host.to(dev, non_blocking=True))[-1], non_blocking=True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        res_host.copy_(solve(y0_host.to(dev, non_blocking=True))[-1], non_blocking=True)
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    # ---- the same job with func as an opaque torch module (what any other vector field gets) -------------------------
    ms_gen, gen_stats = None, {}
    if fused:
        f_gen = make_problem(dev, rows, rank, world, fused=False)[0]
        for _ in range(3):
            solve(y0, f_gen, gen_stats)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(args.steps):
            solve(y0, f_gen, gen_stats)
        g1.record()
        barrier()
        ms_gen = g0.elapsed_time(g1)
    if world > 1:
        tm = torch.tensor([ms, ms_e2e, ms_gen if ms_gen is not None else 0.0], device=dev, dtype=torch.float64)
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        ms, ms_e2e = float(tm[0]), float(tm[1])
        ms_gen = float(tm[2]) if ms_gen is not None else None
    # sanity of the result (norm preservation of the skew field) -- a wrong answer must not be timed silently
    n0, n1 = y0.norm(dim=1), out[-1].norm(dim=1)
    drift = float(((n1 - n0).abs() / n0).max())
    assert drift < 5e-3, "solution drifted: %g" % drift
    # N > 1: the sharded rows must be the rows of the UNSHARDED solve of the same seeded batch (global RMS norm =>
    # same dt sequence): rank 0 solves the whole batch alone (outside the timed region) and compares its own rows
    check = {"max_rel_norm_drift": drift}
    if world > 1:
        n_acc, n_rej = stats.get("n_accept"), stats.get("n_reject")
        if rank == 0:
            st1 = {}
            with torch.no_grad():
                full = tdq.odeint(f, y_all.to(dev), t_dev, method="dopri5", rtol=RTOL, atol=ATOL,
                                  options={"graph": True, "run_ahead": 2, "cache": False}, _stats=st1)
            mine = full[-1][:rows]
            check.update({"unsharded_rows": int(y_all.shape[0]), "max_abs_diff_vs_unsharded": float((out[-1] - mine).abs().max()),
                          "bitwise_equal": bool(torch.equal(out[-1], mine)),
                          "steps_sharded": [n_acc, n_rej], "steps_unsharded": [st1.get("n_accept"), st1.get("n_reject")],
                          "same_step_sequence_counts": [n_acc, n_rej] == [st1.get("n_accept"), st1.get("n_reject")]})
            del full, mine
            torch.cuda.empty_cache()
        dist.barrier()

    if rank == 0:
        n_elems = B_PER_GPU * DIM
        peak, peak_src = measured_peaks()
        probe = roofline_probe(dev, n_elems)
        comb_ms, group_ms = probe["comb_ms"], probe["group_ms"]
        nnz = [1, 2, 3, 4, 5, 5]                          # non-zero beta entries per dopri5 row (SURVEY.md 8(a) A1)
        comb_bytes = sum((k + 2) * n_elems * 4 for k in nnz)          # 32*N*s
        norm_bytes = 8 * n_elems * 4
        achieved = comb_bytes / (comb_ms * 1e-3) / 1e9
        group = (comb_bytes + norm_bytes) / (group_ms * 1e-3) / 1e9
        threads = cpu_threads()
        cpu_val, _cpu_s, cpu_desc, cpu_kind, _ = cpu_sample(threads) if args.cpu_baseline and world == 1 else (None,) * 5
        total_traj = rows * world * args.steps
        line = {
            "metric": METRIC, "value": total_traj / (ms * 1e-3), "unit": "trajectories/s", "n_gpus": world,
            "steps": args.steps, "warmup": W, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[1]: dopri5 adaptive, batch=65536 dim=128 linear ODE y'=Ay, f32, rtol=1e-5 "
                                   "atol=1e-7, t=[0,10]" + ((" split over %d ranks (strong scaling)" % world) if strong and world > 1
                                                            else (" x %d ranks (configs[4] layout)" % world if world > 1 else "")),
                       "batch_per_gpu": rows, "dim": DIM,
                       "exec": ("cuda-graph step body inside a device-side while loop (one launch per solve)"
                                if not args.no_device_loop else "cuda-graph step body replayed by the host, run_ahead=2"),
                       "func": ("torchdiffeq_b200.LinearField(A): forward(t, y) = y @ A^T; a whole attempt (6 stage combinations, 6 field "
                                "evaluations, error norm, candidate commit) is ONE tcgen05 kernel, split-bf16 float32-grade products "
                                "(tdq_attempt.cu)" if fused else
                                "plain nn.Module y @ A^T (cuBLAS fp32 SIMT SGEMM, 6 per attempt, ~60 % of a step)"),
                       "attempts_per_solve": stats.get("attempts"), "nfe_per_solve": stats.get("nfe"),
                       "l2": "working set 20 arrays x 33.5 MB >> 126 MB L2 (no flush needed)",
                       "parallelism": "batch-sharded, 1 all-reduce(3 x f64)/attempt" if world > 1 else "single GPU"},
            "e2e": {"value": total_traj / (ms_e2e * 1e-3), "unit": "trajectories/s",
                    "h2d_bytes_per_step": y0_host.numel() * 4 * world, "d2h_bytes_per_step": res_host.numel() * 4 * world},
            "gpu_launches": launches,
            "clocks": clocks,
        }
        k_combine_roof = {"kernel": "k_combine (6 launches per attempt; the stage combination when func is an opaque module)",
                          "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                          # STATIC: dram__bytes_read + dram__bytes_write of the six launches of one attempt from the
                          # committed ncu --set full capture (not re-measured by this run)
                          "traffic": TRAFFIC_STATIC["bytes"], "traffic_source": TRAFFIC_STATIC["source"],
                          "algorithmic_bytes_per_attempt": comb_bytes,
                          # what the six launches really move: the sixth (k_combine_final) also writes the prefix of the
                          # error estimate (+1 N*s); the norm launch reads 4 and writes 2 arrays (the candidate commit)
                          "moved_bytes_per_attempt": comb_bytes + n_elems * 4,
                          "ms_per_attempt": comb_ms, "launches_per_attempt": 6,
                          "combine_plus_error_norm": {"achieved": group, "frac": group / peak,
                                                      "bytes": comb_bytes + norm_bytes, "ms": group_ms,
                                                      "moved_bytes": comb_bytes + n_elems * 4 + 6 * n_elems * 4,
                                                      "target": "BASELINE.md: >= 0.70 of the HBM roofline"}}
        if fused and "fused_ms" in probe:
            # six fused rows: reads y0 + the row's k_j, writes k_i; the last row also writes y1 and the error prefix
            fused_bytes = comb_bytes + 2 * n_elems * 4                        # 34*N*s: y_i is never written or re-read
            fms, fgms = probe["fused_ms"], probe["fused_group_ms"]
            flops = 6 * 6 * 2.0 * B_PER_GPU * DIM * DIM                       # six bf16 products per float32 product
            stage_roof = {
                "bound": "hbm", "kernel": "k_linear_stage (6 launches per attempt: stage combination + linear field, tcgen05)",
                "achieved": fused_bytes / (fms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                "frac": fused_bytes / (fms * 1e-3) / 1e9 / peak, "peak_source": peak_src,
                "traffic": TRAFFIC_FUSED["bytes"], "traffic_source": TRAFFIC_FUSED["source"],
                "algorithmic_bytes_per_attempt": fused_bytes, "ms_per_attempt": fms, "launches_per_attempt": 6,
                "tensor": {"bf16_flop_per_attempt": flops, "achieved_tflops": flops / (fms * 1e-3) / 1e12,
                           "note": "6 bf16 MMA passes per float32 product; the kernel is HBM bound, the tensor pipe is ~20 % busy"},
                "stage_plus_error_norm": {"achieved": (fused_bytes + norm_bytes) / (fgms * 1e-3) / 1e9,
                                          "frac": (fused_bytes + norm_bytes) / (fgms * 1e-3) / 1e9 / peak,
                                          "bytes": fused_bytes + norm_bytes, "ms": fgms}}
            if "attempt_ms" in probe and stats.get("fused_attempt"):
                # ONE launch per attempt: y0, k_0 in, the candidate pair out (4*N*s), everything else on chip -- the kernel
                # is bound by the tensor pipe (6 bf16 products per float32 product, S stages) and the CUDA cores that
                # form, split and store the stage values, not by HBM
                ams = probe["attempt_ms"]
                tpeak, tsrc = measured_tensor_peak()
                att_bytes = 4 * n_elems * 4
                line["roofline"] = {
                    "bound": "tensor",
                    "kernel": "k_linear_attempt (1 launch per attempt: 6 stage combinations + 6 field evaluations + error norm + "
                              "candidate commit, tcgen05 with the stage values resident on chip; csrc/tdq_attempt.cu)",
                    "achieved": flops / (ams * 1e-3) / 1e12, "peak": tpeak, "unit": "TFLOP/s",
                    "frac": flops / (ams * 1e-3) / 1e12 / tpeak, "peak_source": tsrc,
                    "flop_per_launch": flops,
                    "flop_counted": "bf16 tensor flops issued: 2 x 65536 x 128 x 128 per product, six bf16 products per float32 "
                                    "product (hi/mid/lo split, float32-grade result), six stages",
                    "float32_equivalent_tflops": flops / 6 / (ams * 1e-3) / 1e12,
                    "traffic": TRAFFIC_ATTEMPT["bytes"], "traffic_source": TRAFFIC_ATTEMPT["source"],
                    "ms_per_attempt": ams, "launches_per_attempt": 1,
                    "hbm": {"algorithmic_bytes_per_attempt": att_bytes, "achieved_gbs": att_bytes / (ams * 1e-3) / 1e9,
                            "frac_of_hbm_peak": att_bytes / (ams * 1e-3) / 1e9 / peak,
                            "note": "2 reads + 2 writes per element: the six launches it replaces moved 34 + 6 per element"},
                    # SURVEY.md 8(d)'s algorithmic bytes of the stage combinations + error norm (40*N*s per attempt, what any
                    # formulation that passes the stage values through memory must move) over this launch's time: above the
                    # HBM peak, because the launch does not move them
                    "vs_unfused_hbm_roofline": {"survey_algorithmic_bytes_per_attempt": comb_bytes + norm_bytes,
                                                "effective_gbs": (comb_bytes + norm_bytes) / (ams * 1e-3) / 1e9,
                                                "x_of_hbm_peak": (comb_bytes + norm_bytes) / (ams * 1e-3) / 1e9 / peak},
                    "replaces": {"launches": 7, "ms": fgms, "speedup": fgms / ams},
                    "stage_kernels": stage_roof, "generic_path_kernel": k_combine_roof}
            else:
                stage_roof["generic_path_kernel"] = k_combine_roof
                line["roofline"] = stage_roof
        else:
            k_combine_roof.update({"bound": "hbm", "peak_source": peak_src})
            line["roofline"] = k_combine_roof
        if ms_gen is not None:
            line["generic_path"] = {"value": total_traj / (ms_gen * 1e-3), "unit": "trajectories/s",
                                    "ms_per_step": ms_gen / args.steps,
                                    "func": "plain nn.Module y @ A^T (cuBLAS fp32 SIMT SGEMM): k_combine + the user's kernels",
                                    "attempts_per_solve": gen_stats.get("attempts")}
        line.update({
            "result_check": check,
        })
        if cpu_val is not None:
            line["cpu_baseline"] = {"value": cpu_val, "unit": "trajectories/s", "cores": threads, "kind": cpu_kind,
                                    "sample": cpu_desc}
        print(json.dumps(line), flush=True)
    if world > 1:
        # captured step graphs hold NCCL kernels: drop them before tearing the communicator down
        tdq.clear_cache()
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()


def positive_int(v):
    n = int(v)
    if n < 1:
        raise argparse.ArgumentTypeError("must be at least 1, got %s" % v)
    return n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=10, help="timed steps (one complete solve each)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the solution of the last one as DIR/solution.npy (rank 0's rows)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: weak = 65536 trajectories per rank (configs[4]); strong = 65536 split over the ranks")
    ap.add_argument("--generic", action="store_true",
                    help="func as an opaque torch module (k_combine + cuBLAS SGEMM per stage) instead of LinearField")
    ap.add_argument("--no-fused-controller", action="store_true",
                    help="keep the controller step a launch of its own instead of running it in the last block of the "
                         "whole-attempt kernel (needed under ncu: a kernel with a device-runtime call is not profiled)")
    ap.add_argument("--no-device-loop", action="store_true",
                    help="replay the step graph from the host instead of the device-side while loop (needed under ncu: "
                         "kernels inside a conditional graph node are not visible to its kernel-level profiling)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
