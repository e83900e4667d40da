"""Cost of complex states on the GPU.

    python scripts/bench_complex.py [--out FILE]

(a) tdq_error_norm_commit on complex64 (n = 4,194,304 complex elements) next to float32 (n = 8,388,608): the same
    33.5 MB per array, so the same bytes moved -- 4 reads (err prefix, k_S, y0, y1) and 2 writes (the candidate pair)
    per element, 6 * N * s in all.  CUDA events around many launches that rotate through 4 input sets (4 x 134 MB,
    more than the 126 MB L2 holds), so every launch streams from HBM.
(b) A whole dopri5 solve at B = 65,536 x 64 complex64 with func = y @ W^T (an nn.Module with a complex W), next to
    the float32 generic-path solve at B = 65,536 x 128 (the same bytes per state).

Prints one JSON object with the GPU's name and power limit, read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except Exception as e:                     # the number is still worth reporting without it
        info["power_limit_and_max_sm_clock"] = "unavailable (%s)" % type(e).__name__
    return info


def bench_norm(dtype, n, sets=4, launches=400):
    from torchdiffeq_b200 import _lib
    from torchdiffeq_b200._engine import AdaptiveEngine, _stream
    dev = torch.device("cuda:0")
    eng = AdaptiveEngine(lambda t, y: y, n, dtype, dev, "dopri5", rtol=1e-5, atol=1e-7, first_step=0.01)
    t_out = torch.tensor([0.0, 1.0], dtype=torch.float64, device=dev)
    _lib.check(eng.lib.tdq_ctrl_init(eng.ctrl.data_ptr(), C.byref(eng.tab), C.byref(eng.opt), t_out.data_ptr(), 0.0, 2,
                                     eng.mbox_dev, _stream()))
    _lib.check(eng.lib.tdq_set_first_step(eng.ctrl.data_ptr(), 0.01, _stream()))
    _lib.check(eng.lib.tdq_prepare_attempt(eng.ctrl.data_ptr(), eng.rt_code, None, _stream()))
    g = torch.Generator(device=dev).manual_seed(0)
    data = [[torch.randn(n, dtype=dtype, device=dev, generator=g) for _ in range(4)] for _ in range(sets)]

    def launch(i):
        e, k, y0, y1 = data[i % sets]
        _lib.check(eng.lib.tdq_error_norm_commit(eng.ctrl.data_ptr(), eng.dt_code, e.data_ptr(), k.data_ptr(),
                                                 y0.data_ptr(), y1.data_ptr(), None, None, None, 0, 0, 1, n,
                                                 eng.partials.data_ptr(), eng.norm_out.data_ptr(), None, _stream()))
    for i in range(2 * sets):
        launch(i)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(launches):
        launch(i)
    b.record()
    torch.cuda.synchronize()
    us = a.elapsed_time(b) * 1e3 / launches
    nbytes = 6 * n * torch.empty((), dtype=dtype).element_size()
    return {"dtype": str(dtype), "n": n, "array_MB": n * torch.empty((), dtype=dtype).element_size() / 1e6,
            "input_sets": sets, "launches": launches, "us_per_launch": round(us, 2),
            "GB_per_s_of_6Ns": round(nbytes / us / 1e3, 1)}


class Linear(torch.nn.Module):
    def __init__(self, W):
        super().__init__()
        self.W = torch.nn.Parameter(W, requires_grad=False)

    def forward(self, t, y):
        return y @ self.W.T


def bench_solve(dtype, B, D, reps=3):
    import torchdiffeq_b200 as tdq
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(1)
    H = torch.randn(D, D, generator=g, dtype=torch.float64)
    if dtype.is_complex:
        Hi = torch.randn(D, D, generator=g, dtype=torch.float64)
        H = torch.complex(H, Hi)
        H = (H + H.mH) / 2 / D ** 0.5
        W = -1j * H - 0.5 * torch.eye(D, dtype=torch.complex128)
    else:
        W = (H - H.T) / 2 / D ** 0.5 - 0.5 * torch.eye(D, dtype=torch.float64)
    f = Linear(W.to(dtype)).to(dev)
    y0 = torch.randn(B, D, generator=g, dtype=torch.float64)
    y0 = (torch.complex(y0, torch.randn(B, D, generator=g, dtype=torch.float64)) if dtype.is_complex else y0).to(dtype)
    y0 = y0.to(dev)
    t = torch.tensor([0.0, 1.0], device=dev)
    opts = dict(fused_linear=False)
    with torch.no_grad():
        tdq.odeint(f, y0, t, method="dopri5", rtol=1e-5, atol=1e-7, options=opts)            # warm-up + capture
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            tdq.odeint(f, y0, t, method="dopri5", rtol=1e-5, atol=1e-7, options=opts)
        b.record()
        torch.cuda.synchronize()
    ms = a.elapsed_time(b) / reps
    st = tdq.last_stats()
    return {"dtype": str(dtype), "B": B, "D": D, "ms_per_solve": round(ms, 3), "trajectories_per_s": round(B / ms * 1e3),
            "attempts": st.get("attempts"), "n_accept": st.get("n_accept"), "n_reject": st.get("n_reject"),
            "fused_linear": st.get("fused_linear")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_complex.py measures on a CUDA device"
    res = gpu_info()
    res["norm"] = [bench_norm(torch.complex64, 4194304), bench_norm(torch.float32, 8388608),
                   bench_norm(torch.complex64, 4194304), bench_norm(torch.float32, 8388608)]
    c, r = res["norm"][2], res["norm"][3]
    res["norm_complex64_over_float32"] = round(c["us_per_launch"] / r["us_per_launch"], 3)
    res["solve"] = [bench_solve(torch.complex64, 65536, 64), bench_solve(torch.float32, 65536, 128)]
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
