"""Times the interior-point Newton step of the kino-dynamic NLP (landing_kino_step_batch) on device-resident SoA buffers,
after warm-up, with CUDA events, at 16384 scenarios (every input exceeds the 126 MB L2).  The iterate is the one a first
iteration sees: x random at landing magnitudes, the bounds of random drops (landing_kino_setup_batch), s = g pushed
inside its bounds (IPOPT's bound_push = bound_frac = 0.01), z = mu / distance, small random y, mu = 0.1.
Algorithmic counts, from the shapes: bytes = 8 * (inputs read + outputs written) per scenario -- g, jac, hess, grad_f
and the six m-vectors s, y, zL, zU, lbg, ubg, plus mu and dw_last; dx and the four m-vectors ds, dy, dzL, dzU, plus the
scalars; FLOP per factorisation = 2 * (the multiply-adds of the stage assembly, of M + A'PA, of the Cholesky of the
control block, of Y = L^-1 M_u,xi and of P = M_xi,xi - Y'Y) over the N - 1 stages.
   usage: python tools/bench_kino_step.py [N ...]   (default 21 50; one JSON line per N, with the card and power limit)"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
DT_VAL = [0.05] + [0.02] * 15 + [0.05, 0.05, 0.1, 0.2]


def counts(N, nnzJ, nnzH, nx, m, pair_terms):
    """(bytes read, bytes written, FLOP of one factorisation) of one scenario."""
    read = 8 * (m + nnzJ + nnzH + nx + 6 * m + 2)
    written = 8 * (nx + 4 * m + 3) + 2 * 4
    K = N - 1
    fma = pair_terms + (K * (24 * 60 * 12 + 1830 * 12 + 36 ** 3 // 6 + 25 * 36 * 36 // 2 + 300 * 36))
    return read, written, 2 * fma


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except Exception as e:  # (reported, not guessed)
        return "unknown (%s)" % e


def measure(N, B=16384, reps=5):
    import numpy as np
    import torch
    import landing_controller_b200 as lc
    s = lc.LandingSolver(N=N, device=0)
    d = s.kino_dims()
    nnzH = len(s.kino_hess_sparsity()[1])
    pb = s.kino_problem(np.array(DT_VAL) if N == 21 else np.full(N - 1, 0.6 / (N - 1)))
    dev = torch.device("cuda", 0)
    f = dict(dtype=torch.float64, device=dev)
    gen = torch.Generator(device=dev).manual_seed(0)
    x = (torch.rand(d["nx"], B, generator=gen, **f) - 0.5)
    drops = torch.zeros(B, 12, **f)
    drops[:, 2] = 0.3 + 0.2 * torch.rand(B, generator=gen, **f)
    drops[:, 9:12] = torch.rand(B, 3, generator=gen, **f) - 0.5
    lbg, ubg = torch.zeros(d["m"], B, **f), torch.zeros(d["m"], B, **f)
    s.kino_setup_device(drops.T.contiguous(), lbg=lbg, ubg=ubg, layout=lc.SOA)
    g, jac = torch.zeros(d["m"], B, **f), torch.zeros(d["nnzJ"], B, **f)
    s.kino_eval_device(x, pb, g=g, jac=jac)
    y = 0.01 * torch.randn(d["m"], B, generator=gen, **f)
    hess = torch.zeros(nnzH, B, **f)
    s.kino_hess_device(x, pb, hess, lam_f=torch.ones(B, **f), lam_g=y)
    gf = torch.zeros(d["nx"], B, **f)
    ks = s.kino_setup_data()
    s._check(s.lib.landing_kino_cost_batch(s.ctx, B, lc.DEVICE, lc.SOA, __import__("ctypes").byref(ks),
                                           lc.api._ptr(x), None, lc.api._ptr(gf)), "landing_kino_cost_batch")
    s.synchronize()
    inf = float("inf")
    pL = torch.minimum(0.01 * torch.clamp(lbg.abs(), min=1.0), 0.01 * (ubg - lbg))
    pU = torch.minimum(0.01 * torch.clamp(ubg.abs(), min=1.0), 0.01 * (ubg - lbg))
    lo = torch.where(torch.isfinite(lbg), lbg + pL, torch.full_like(lbg, -inf))
    hi = torch.where(torch.isfinite(ubg), ubg - pU, torch.full_like(ubg, inf))
    sl = torch.maximum(torch.minimum(g, hi), lo)
    mu = torch.full((B,), 0.1, **f)
    zL = torch.where(torch.isfinite(lbg), 0.1 / (sl - lbg), torch.zeros_like(sl))
    zU = torch.where(torch.isfinite(ubg), 0.1 / (ubg - sl), torch.zeros_like(sl))
    inp = dict(g=g, jac=jac, hess=hess, grad_f=gf, s=sl, y=y, zL=zL, zU=zU, lbg=lbg, ubg=ubg, mu=mu,
               dw_last=torch.zeros(B, **f))
    out = {"dx": torch.zeros(d["nx"], B, **f)}
    for k in ("ds", "dy", "dzL", "dzU"):
        out[k] = torch.zeros(d["m"], B, **f)
    out.update(delta_w=torch.zeros(B, **f), alpha_pr=torch.zeros(B, **f), alpha_du=torch.zeros(B, **f),
               n_factor=torch.zeros(B, dtype=torch.int32, device=dev), status=torch.zeros(B, dtype=torch.int32, device=dev))
    torch.cuda.synchronize()
    call = lambda: s.kino_step_device(inp, out, tau=0.99)  # noqa: E731
    for _ in range(2):
        call()
    s.synchronize()
    st = torch.cuda.ExternalStream(s.stream_ptr, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(st):
        e0.record()
    for _ in range(reps):
        call()
    with torch.cuda.stream(st):
        e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    status = out["status"].cpu().numpy()
    nf = out["n_factor"].cpu().numpy()
    # pair terms of the stage assembly: sum over inequality rows of n (n + 1) / 2, from the Jacobian pattern
    sp = s.lib.landing_kino_sparsity(N)
    nx = sp[1]
    colind = np.ctypeslib.as_array(sp, shape=(2 + nx + 1,))[2:]
    row = np.ctypeslib.as_array(sp, shape=(2 + nx + 1 + int(colind[-1]),))[2 + nx + 1:]
    per = np.bincount(row, minlength=d["m"])
    r = np.arange(d["m"])
    ineq = (r >= 24) & ~((r >= 48) & ((r - 48) % 141 < 12))
    pairs = int((per[ineq] * (per[ineq] + 1) // 2).sum()) + nnzH
    rd, wr, flop = counts(N, d["nnzJ"], nnzH, d["nx"], d["m"], pairs)
    return {"function": "kino_step", "N": N, "B": B, "layout": "SOA", "ms_per_call": round(ms, 3),
            "status0_fraction": float((status == 0).mean()), "mean_n_factor": round(float(nf.mean()), 3),
            "bytes_read_per_scenario": rd, "bytes_written_per_scenario": wr, "flop_per_factorisation": flop,
            "achieved_GBps": round((rd + wr) * B / (ms * 1e-3) / 1e9, 1),
            "achieved_GFLOPs": round(flop * float(nf.mean()) * B / (ms * 1e-3) / 1e9, 1),
            "card": card()}


if __name__ == "__main__":
    for N in [int(a) for a in sys.argv[1:]] or [21, 50]:
        print(json.dumps(measure(N)), flush=True)
