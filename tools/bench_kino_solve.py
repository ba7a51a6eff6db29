"""Benchmark of the batched kino-dynamic interior-point solve (landing_kino_solve_batch): grid drops, SRB solve first
(landing_solve_batch, the reference's dt at N = 21), then the kino-dynamic solve from its solutions, device buffers.
Reports converged NLPs/s, the converged fraction, iterations and restarts, the call's rounds, and a per-phase split of
kernel time from torch.profiler (a separate, profiled run; per-kernel device times, grouped by kernel name, because the
phases interleave inside one library call where the caller cannot place events).  Prints one JSON line per configuration.

    python tools/bench_kino_solve.py [--configs 21:16384,40:4096] [--max-iter 3000] [--no-profile]"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

# kernel name -> phase.  k_kino_g runs at the start (once) and at every line-search trial; k_kino_cost gives the cost
# gradient once per outer round and f at every trial, so it has a row of its own.
PHASES = (("hessian", ("k_kino_hess",)), ("jacobian", ("k_kino_jac",)), ("grad_x + KKT measures", ("k_kino_grad", "k_kino_kkt")),
          ("cost (f, grad f)", ("k_kino_cost",)), ("step", ("k_kino_step",)), ("g at trial points", ("k_kino_g",)),
          ("line search: trial + filter", ("k_ks_trial", "k_ks_filter")),
          ("bookkeeping", ("k_ks_measure", "k_ks_ftb", "k_ks_accept", "k_ks_scan", "k_ks_init", "k_ks_load")),
          ("compaction", ("k_ks_output", "k_ks_gather")))


def phase_of(name):
    for ph, keys in PHASES:
        if any(k in name for k in keys):
            return ph
    return "other"


def run(N, B, max_iter, profile):
    import torch
    import kino_ref as kr
    import landing_controller_b200 as lc
    dev = torch.device("cuda:0")
    drops = lc.grid_sweep(B)
    srb = lc.LandingSolver(N=N, device=0)
    if N == 21:
        srb.set_dt(kr.DT_VAL)
    x_srb = srb.solve(drops)["x"]
    srb.close()
    s = lc.LandingSolver(N=N, device=0)
    pbo = kr.default_problem(N)
    pb = s.kino_problem(pbo["dt"], mu=pbo["mu"], mass=pbo["mass"], Ib=pbo["Ib"], Ib_inv=pbo["Ib_inv"])
    s.options.max_iter = max_iter
    d = s.kino_dims()
    dT, xT = torch.tensor(drops, device=dev), torch.tensor(x_srb, device=dev)
    out = dict(x=torch.zeros(B, d["nx"], dtype=torch.float64, device=dev), f=torch.zeros(B, dtype=torch.float64, device=dev),
               status=torch.zeros(B, dtype=torch.int32, device=dev), iters=torch.zeros(B, dtype=torch.int32, device=dev),
               restarts=torch.zeros(B, dtype=torch.int32, device=dev))

    def call():
        return s.kino_solve_device(dT, out["x"], out["f"], out["status"], out["iters"], x_srb=xT,
                                   restarts=out["restarts"], pb=pb)
    call()  # warm-up (modules, plans, scratch)
    s.synchronize()
    torch.cuda.synchronize()
    l0 = s.launches
    t0 = time.perf_counter()
    stats = call()
    s.synchronize()
    wall = time.perf_counter() - t0
    st, it, rs = (out[k].cpu().numpy() for k in ("status", "iters", "restarts"))
    conv = st == 0
    res = dict(N=N, B=B, wall_s=round(wall, 4), converged_per_s=round(float(conv.sum()) / wall, 2),
               converged_fraction=round(float(conv.mean()), 4), statuses=np.bincount(st, minlength=5).tolist(),
               iters_mean=round(float(it.mean()), 2), iters_p99=int(np.percentile(it, 99)), iters_max=int(it.max()),
               restarts_mean=round(float(rs.mean()), 3), restarts_max=int(rs.max()), outer_rounds=int(stats[0]),
               ls_rounds=int(stats[1]), compactions=int(stats[2]), launches=int(s.launches - l0),
               ms_per_outer_round=round(1e3 * wall / max(1, int(stats[0])), 3))
    if profile:
        from torch.profiler import ProfilerActivity, profile as prof
        with prof(activities=[ProfilerActivity.CUDA]) as p:
            call()
            s.synchronize()
        tot = {}
        for e in p.key_averages():
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = e.cuda_time_total
            if t:
                tot[phase_of(e.key)] = tot.get(phase_of(e.key), 0.0) + t / 1e3
        res["kernel_ms_by_phase"] = {k: round(v, 2) for k, v in sorted(tot.items())}
        # copy bandwidth of this device in the same run, for the bookkeeping kernels' share of it
        a = torch.empty(1 << 28, dtype=torch.uint8, device=dev)
        b = torch.empty_like(a)
        for _ in range(3):
            b.copy_(a)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            b.copy_(a)
        e1.record()
        torch.cuda.synchronize()
        res["copy_GBps"] = round(2 * 20 * a.numel() / (e0.elapsed_time(e1) / 1e3) / 1e9, 1)
        # bytes the bookkeeping kernels of the outer rounds move per running scenario: measure 6 m + n_x, ftb 8 m,
        # accept 8 m doubles; a scenario is running in iters + 1 rounds
        m = d["m"]
        by = 8.0 * (22 * m + d["nx"]) * float(it.sum() + B)
        bk = tot.get("bookkeeping", 0.0)
        if bk > 0:
            res["bookkeeping_fraction_of_copy_bw"] = round(by / (bk / 1e3) / (res["copy_GBps"] * 1e9), 3)
    props = torch.cuda.get_device_properties(0)
    res["device"] = props.name
    try:
        import subprocess
        res["power_limit"] = subprocess.check_output(
            ["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], text=True).strip()
    except Exception:
        res["power_limit"] = "unknown"
    s.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="21:16384,40:4096")
    ap.add_argument("--max-iter", type=int, default=3000)
    ap.add_argument("--no-profile", action="store_true")
    a = ap.parse_args()
    for c in a.configs.split(","):
        N, B = (int(v) for v in c.split(":"))
        print(json.dumps(run(N, B, a.max_iter, not a.no_profile)), flush=True)


if __name__ == "__main__":
    main()
