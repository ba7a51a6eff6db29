"""Times the kino-dynamic evaluation kernels (g, CCS Jacobian, upper-triangle Lagrangian Hessian, Lagrangian gradient and
KKT residuals; SURVEY 8 f-2) on device-resident SoA buffers: algorithmic bytes = 8 * (inputs read + outputs written) per
scenario -- n_x + m for g, n_x + nnzJ for the Jacobian, n_x + m + nnzH (+ lam_f) for the Hessian, n_x + m + 1 + n_x for
grad_x alone, and for all four KKT outputs that plus the bounds (2 m), the g the call computes (m) and the three scalars
-- against the HBM copy bandwidth measured in the same run.  At N = 21 and 16384 scenarios every input exceeds the
126 MB L2.
   usage: python tools/bench_kino.py [N] [B]        (prints one JSON line per function, with the card's name and power limit)"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

DT_VAL = [0.05] + [0.02] * 15 + [0.05, 0.05, 0.1, 0.2]  # generate_landingCtrller_KNITRO.m (the sweep callers' dt_val, N = 21)


def copy_bandwidth(dev, nbytes=2 << 30, reps=10):
    """Device-to-device copy bandwidth (bytes read + written per second) measured with CUDA events."""
    import torch
    a = torch.empty(nbytes // 8, dtype=torch.float64, device=dev).fill_(1.0)
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    gbs = 2.0 * nbytes * reps / (e0.elapsed_time(e1) * 1e-3) / 1e9
    del a, b
    return gbs


def measure_kino(N=21, B=16384, reps=10, solver=None, device=0, hess=False):
    """g and Jacobian against the HBM peak of bench_eval.hbm_peak; hess: also the Lagrangian Hessian, and every function
    against the copy bandwidth measured in this run instead."""
    import numpy as np
    import torch
    import landing_controller_b200 as lc
    s = solver or lc.LandingSolver(N=N, device=device, lib_path=os.environ.get("LANDING_LIB", lc.api.LIB_PATH))
    d = s.kino_dims()
    pb = s.kino_problem(np.array(DT_VAL) if N == 21 else np.full(N - 1, 0.6 / (N - 1)))
    dev = torch.device("cuda", device)
    x = torch.rand(d["nx"], B, dtype=torch.float64, device=dev) - 0.5
    g = torch.zeros(d["m"], B, dtype=torch.float64, device=dev)
    jac = torch.zeros(d["nnzJ"], B, dtype=torch.float64, device=dev)
    nnzH = H = lam_f = lam_g = lbg = ubg = gx = sc = 0
    if hess:
        nnzH = len(s.kino_hess_sparsity()[1])
        lam_f = torch.ones(B, dtype=torch.float64, device=dev)
        lam_g = torch.randn(d["m"], B, dtype=torch.float64, device=dev)
        H = torch.zeros(nnzH, B, dtype=torch.float64, device=dev)
        lbg = -torch.rand(d["m"], B, dtype=torch.float64, device=dev)
        ubg = torch.rand(d["m"], B, dtype=torch.float64, device=dev)
        gx = torch.zeros(d["nx"], B, dtype=torch.float64, device=dev)
        sc = torch.zeros(3, B, dtype=torch.float64, device=dev)
    st = torch.cuda.ExternalStream(s.stream_ptr, device=dev)
    torch.cuda.synchronize()
    if hess:
        peak, peak_src = copy_bandwidth(dev), "device-to-device copy, measured in this run"
    else:
        from bench_eval import hbm_peak
        peak, peak_src = hbm_peak()
    out = []
    calls = (("kino_g", lambda: s.kino_eval_device(x, pb, g=g), d["nx"] + d["m"]),
             ("kino_jac_g", lambda: s.kino_eval_device(x, pb, jac=jac), d["nx"] + d["nnzJ"]),
             ("kino_hess_l", lambda: s.kino_hess_device(x, pb, H, lam_f=lam_f, lam_g=lam_g), d["nx"] + d["m"] + nnzH + 1),
             ("kino_grad_x", lambda: s.kino_kkt_device(x, pb, lam_f=lam_f, lam_g=lam_g, grad_x=gx),
              2 * d["nx"] + d["m"] + 1),
             ("kino_kkt", lambda: s.kino_kkt_device(x, pb, lam_f=lam_f, lam_g=lam_g, lbg=lbg, ubg=ubg, grad_x=gx,
                                                    viol=sc[0], dual_inf=sc[1], compl_inf=sc[2]),
              2 * d["nx"] + d["m"] + 1 + 3 * d["m"] + 3))
    for name, call, words in calls[:5 if hess else 2]:
        for _ in range(3):
            call()
        s.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = s.launches
        with torch.cuda.stream(st):
            e0.record()
        for _ in range(reps):
            call()
        with torch.cuda.stream(st):
            e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        gbs = 8.0 * words * B / (ms * 1e-3) / 1e9
        out.append({"function": name, "N": N, "B": B, "layout": "soa", "ms": ms, "launches_per_call": (s.launches - l0) / reps,
                    "algorithmic_bytes_per_scenario": 8 * words, "achieved": gbs, "peak": peak, "unit": "GB/s",
                    "frac": gbs / peak, "peak_source": peak_src, "evals_per_s": B / (ms * 1e-3),
                    "sizes": {"nx": d["nx"], "m": d["m"], "nnzJ": d["nnzJ"]}})
        if hess:
            out[-1]["sizes"]["nnzH"] = nnzH
    return out


if __name__ == "__main__":
    N = int(sys.argv[1]) if len(sys.argv) > 1 else 21
    B = int(sys.argv[2]) if len(sys.argv) > 2 else 16384
    import torch
    p = torch.cuda.get_device_properties(0)
    try:
        import subprocess
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True).stdout.strip()
    except OSError:
        power = "unknown"
    for r in measure_kino(N, B, hess=True):
        r.update(device=p.name, power_limit_max_sm_clock=power)
        print(json.dumps(r))
