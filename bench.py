#!/usr/bin/env python
"""bench.py -- converged landing NLPs/sec on the BASELINE.json workload.

One "step" = one pass of the hot path over one batch: solve every drop condition of the sweep
(SRB landing sweep on a height x pitch x roll x forward-velocity grid of drop conditions) with the batched
interior-point kernel.  Under torchrun each rank solves its interleaved shard of the sweep (no data-path
collective) and the step ends with ONE NCCL all-gather of the per-scenario result records (x*, f*, status, iters),
in the device-resident arm and in the end-to-end arm alike.

    python bench.py [--gpus N] [--steps K] [--warmup W]        # this repo's CUDA path
    python bench.py --impl reference ...                        # the CPU path on the host cores (same config object)
    one GPU: BASELINE configs[1] (1k grid, N = 30); under torchrun: configs[2], the FIXED 16k x N = 50 sweep strong-scaled
    --dump-outputs DIR: also write the results of the last timed step as DIR/<name>.npy (see dump_outputs)

Prints ONE JSON line (rank 0).  Writes nothing into the checkout, which may be read-only.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True  # (no __pycache__ in the checkout for the modules imported below)
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "converged landing NLPs/sec (FP64, batch)"
UNIT = "NLP/s"

# BASELINE.json configs -> concrete workloads (SURVEY.md 8d).  One GPU runs configs[1]; under torchrun (N > 1) the FIXED
# 16384-drop N = 50 sweep of configs[2] is strong-scaled over the ranks (interleaved shards), which is the workload the
# >= 100 x target is quoted on.  `--config` overrides.
CONFIGS = {
    "1k": dict(knots=30, total=1024, scaling="weak",
               workload="BASELINE configs[1]: SRB landing sweep, 1024 grid drop conditions (height x pitch x roll x v_x, v_z=-3), N=30 knots"),
    "single": dict(knots=30, total=1, scaling="weak", formulation="schedule",
                   workload="BASELINE configs[0]: SRB landing NLP, one drop condition (0.5 m, level, 1 m/s forward), fixed contact "
                            "schedule (quadruped_SRBM_NLP.m; flight until the ballistic fall reaches 0.28 m, then stance), N=30 knots"),
    "16k": dict(knots=50, total=16384, scaling="strong",
                workload="BASELINE configs[2]: SRB landing sweep, 16384 grid drop conditions (height x pitch x roll x v_x, v_z=-3), N=50 knots, strong-scaled over the GPUs"),
}


def pick_config(args, world):
    name = args.config if args.config != "auto" else ("1k" if world == 1 else "16k")
    cfg = dict(CONFIGS[name])
    cfg["name"] = name
    cfg["restart_mu"] = getattr(args, "restart_mu", 0.0)
    if args.knots:
        cfg["knots"] = args.knots
    if args.batch:
        cfg["total"] = args.batch * (world if cfg["scaling"] == "weak" else 1)
    elif cfg["scaling"] == "weak":
        cfg["total"] = cfg["total"] * world
    return cfg


def config_dict(cfg, world):
    """The `config` object of the JSON line: identical in the GPU arm and the reference arm of one (config, N)."""
    return {"workload": cfg["workload"], "knots": cfg["knots"], "global_batch": cfg["total"],
            "batch_per_gpu": cfg["total"] // world,
            "parallelism": "scenario-sharded x%d (interleaved shards of the %d-scenario sweep), one all-gather of the result records"
                           % (world, cfg["total"]),
            "options": "tol 1e-4, constr_viol_tol 1e-3, max_iter 3000 (generate_landingCtrller_IPOPT.m:232-236)"
                       + (", NON-DEFAULT restart_mu %g" % cfg["restart_mu"] if cfg.get("restart_mu", 0.0) > 0.0 else ""),
            "l2": "GPU arm: the per-scenario solver scratch of the 296 resident CTAs (%.2f GB) exceeds the 126 MB L2 and "
                  "every step rewrites all of it; no flush needed" % (1e-9 * scratch_bytes(cfg["knots"], 296))}


def schedule_setup(cfg, solver=None):
    """configs[0]: the fixed-contact-schedule problem.  Returns (pb, opt) for the CPU arm; configures `solver` (GPU)."""
    import landing_controller_b200 as lc
    N, T, z0 = cfg["knots"], 0.6, 0.5
    cs = lc.ballistic_schedule(N, T, z0)
    if solver is not None:
        lc.apply_schedule_parameters(solver.problem)
        solver.problem.T = T
        solver.set_schedule(cs, lc.SCHED_QX)
        return None, None
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_ip import default_options, default_problem
    pb = lc.apply_schedule_parameters(default_problem())
    pb.T = T
    return pb, default_options(run_Qf=lc.SCHED_QF, kin_box=lc.SCHED_KIN_BOX).set_schedule(cs, lc.SCHED_QX)


def workload(cfg, world, rank):
    import landing_controller_b200 as lc
    if cfg.get("formulation") == "schedule":
        return np.repeat(lc.single_drop(), cfg["total"], axis=0)[rank::world].copy()
    allb = lc.grid_sweep(cfg["total"])
    # interleaved shards: the iteration count grows along the axes of the grid, contiguous blocks would give the last
    # rank the hard end of the sweep
    return allb[lc.shard_indices(cfg["total"], world, rank, "interleaved")].copy()


def iter_bytes(N):
    """Algorithmic HBM bytes of one interior-point iteration of one scenario (SURVEY.md 8d-ii):
    read + write the primal-dual iterate once, read p: 8 * (2 (340N - 316) + 13N + 81)."""
    return 8 * (2 * (340 * N - 316) + 13 * N + 81)


def iter_flops(N):
    """Algorithmic FP64 flops of one iteration of one scenario with ONE Riccati factorisation (DESIGN.md 2.3):
    per stage 2 x MACs of  T = Pxx G (12.12.36) + lower triangle of G'T (78 tiles x 9 x 12) + G'Pxc (36.12.12)
    + partial Cholesky of the 48x48 stage matrix, 24 pivots (sum_j (48-j)(49-j)/2) + condensing (576 terms x 2)
    + forward sweep (24.24 + 300 + 12.36 + 12.24), plus evaluation (3.1k flop / knot, SURVEY 8d) and row passes."""
    chol = sum((48 - j) * (49 - j) // 2 for j in range(24))
    macs = 12 * 12 * 36 + 78 * 9 * 12 + 36 * 12 * 12 + chol + 2 * 576 + (24 * 24 + 300 + 12 * 36 + 12 * 24)
    return (2 * macs + 3100 + 3000) * (N - 1)


def scratch_bytes(N, slots):
    K, nx, MR = N - 1, 36 * N - 24, 36 + 104 * (N - 1)
    n = 3 * nx + 12 * MR + K * (388 + 192 + 480) + K * (1152 + 36) + (K + 1) * 312 + 144 + 128
    return 8 * slots * ((n + 31) // 32 * 32)


def ncu_traffic():
    """DRAM bytes per launch of k_solve from the committed ncu --set full capture of this workload, or None."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(path):
        try:
            return json.load(open(path))
        except Exception:
            return None
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def cpu_run(N, drops, threads, cfg=None):
    """The timed CPU arm: oracle/ip_ref.c built -O3 -march=native on this host (the reference builds its C with gcc -O3,
    generate_landingCtrller_IPOPT.m:296), OpenMP over scenarios."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_ip import solve_cpu
    pb, opt = schedule_setup(cfg) if cfg and cfg.get("formulation") == "schedule" else (None, None)
    if cfg and cfg.get("restart_mu", 0.0) > 0.0:
        from oracle_ip import default_options
        opt = opt or default_options()
        opt.restart_mu = cfg["restart_mu"]
    t = time.perf_counter()
    r = solve_cpu(N, drops, opt, pb, threads=threads, fast=True)
    dt = time.perf_counter() - t
    return r, dt


def cpu_sample(cfg, drops, want):
    """Bounded strided sample of a sweep for the CPU arm (about 5-15 s of work on 16 host threads per step)."""
    n = want or (1024 if cfg["knots"] <= 30 else 512)
    n = min(n, len(drops))
    stride = max(1, len(drops) // n)
    return drops[::stride][:n], stride


def cpu_flags():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_ip import fast_build_flags
    return fast_build_flags()


def run_reference(args):
    """The reference's CPU path for the hot path, on the host cores.  IPOPT/MUMPS are not available
    (SURVEY.md 8c), so this is the CPU restatement (oracle/: generated-function restatement +
    interior-point "IPOPT substitute"), OpenMP over scenarios with all host threads, on a bounded strided sample of the
    SAME workload (same config object) as the GPU arm of this --gpus value."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    cfg = pick_config(args, world)
    N = cfg["knots"]
    cores = os.cpu_count() or 1
    drops = workload(cfg, 1, 0)  # the whole sweep
    sub, stride = cpu_sample(cfg, drops, args.cpu_sample)
    flags = cpu_flags()  # (builds the -O3 library before anything is timed)
    for _ in range(min(args.warmup, 1)):
        cpu_run(N, sub[:cores], cores, cfg)
    tot_t, tot_c, tot_it = 0.0, 0, 0
    for _ in range(args.steps):
        r, dt = cpu_run(N, sub, cores, cfg)
        tot_t += dt
        tot_c += int((r["status"] == 0).sum())
        tot_it += int(r["iters"].sum())
    val = tot_c / tot_t
    sample = ("%d of %d scenarios per step (every %d-th), %d steps; IPOPT substitute (oracle/ip_ref.c, %s), OpenMP over scenarios"
              % (len(sub), cfg["total"], stride, args.steps, flags))
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps, "higher_is_better": True,
        "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(cfg, world),
        "kkt_iters_per_s": tot_it / tot_t, "converged_fraction": tot_c / float(len(sub) * args.steps),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def sweep_records(gathered, total, world):
    """All-gathered result records [world, Bmax, nx + 3] (rank-major; each rank's interleaved shard padded to Bmax)
    -> x, f, status, iters of the whole sweep in sweep order."""
    import landing_controller_b200 as lc
    parts = [gathered[r, :len(lc.shard_indices(total, world, r))] for r in range(world)]
    ordered = np.empty((total, gathered.shape[2]))
    ordered[lc.unshard_order(total, world)] = np.concatenate(parts)
    return lc.unpack_records(ordered)


DUMP_LIMIT = 64 << 20  # bytes written by --dump-outputs


def dump_outputs(path, x, f, status, iters):
    """What the timed path returned to its caller in the last step, as float64 arrays <path>/<name>.npy: x [B, nx]
    (x*), f (f*), status, iters, and scenario (the index in the sweep of each row).  The sweep is fixed by the
    arguments, so two builds run with the same arguments can be compared output for output.  When the whole sweep is
    larger than DUMP_LIMIT a fixed, seeded sample of its scenarios is written."""
    B, nx = x.shape
    keep = np.arange(B)
    row_bytes = 8 * (nx + 4)
    if B * row_bytes > DUMP_LIMIT:
        keep = np.sort(np.random.default_rng(0).choice(B, DUMP_LIMIT // row_bytes, replace=False))
    os.makedirs(path, exist_ok=True)
    out = {"x": x[keep], "f": f[keep], "status": status[keep], "iters": iters[keep], "scenario": keep}
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))


def iter_stats(its, st):
    its = np.asarray(its, dtype=np.float64)
    q = lambda f: float(np.percentile(its, f))
    return {"mean": float(its.mean()), "p50": q(50), "p90": q(90), "p99": q(99), "max": float(its.max()),
            "status_counts": {str(k): int(v) for k, v in zip(*np.unique(np.asarray(st), return_counts=True))}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", default="auto", choices=["auto", "single", "1k", "16k"],
                    help="auto: BASELINE configs[1] on one GPU, configs[2] (fixed 16k x N=50 sweep, strong-scaled) under torchrun")
    ap.add_argument("--batch", type=int, default=0, help="override: scenarios per GPU (weak configs) / in total (strong)")
    ap.add_argument("--knots", type=int, default=0, help="override: knots per trajectory")
    ap.add_argument("--cpu-sample", type=int, default=0, help="scenarios in the CPU sample (0 = auto)")
    ap.add_argument("--no-eval-kernels", action="store_true", help="skip the evaluation-kernel roofline lines")
    ap.add_argument("--restart-mu", type=float, default=0.0,
                    help="NOT the default: landing_options.restart_mu for both arms (DESIGN.md 3); 0 = mu_init")
    ap.add_argument("--no-one-gpu-base", action="store_true",
                    help="N > 1: skip the 1-GPU solve of the same fixed workload on rank 0 (strong-scaling base)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step (x*, f*, status, iters per scenario) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path, not of --impl reference")
    if args.impl == "reference":
        run_reference(args)
        return

    import ctypes
    import torch
    import torch.distributed as dist
    import landing_controller_b200 as lc

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this library has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = pick_config(args, world)
    N = cfg["knots"]
    solver = lc.LandingSolver(N=N, device=local_rank)
    if cfg.get("restart_mu", 0.0) > 0.0:
        solver.options.restart_mu = cfg["restart_mu"]
    if cfg.get("formulation") == "schedule":
        schedule_setup(cfg, solver)
    nx = solver.dims["nx"]
    drops_h = workload(cfg, world, rank)
    B = len(drops_h)
    Bmax = -(-cfg["total"] // world)  # shards differ by at most one scenario: records are padded for the all-gather

    # device-resident arm: inputs already in HBM when the timed region starts
    drops_d = torch.tensor(drops_h, device=dev)
    rec = torch.zeros(Bmax, nx + 3, dtype=torch.float64, device=dev)  # result record [x*, f*, status, iters]
    x_d = torch.zeros(B, nx, dtype=torch.float64, device=dev)
    f_d = torch.zeros(B, dtype=torch.float64, device=dev)
    st_d = torch.zeros(B, dtype=torch.int32, device=dev)
    it_d = torch.zeros(B, dtype=torch.int32, device=dev)
    gathered = torch.zeros(world * Bmax, nx + 3, dtype=torch.float64, device=dev) if world > 1 else None
    lib_stream = torch.cuda.ExternalStream(solver.stream_ptr, device=dev)

    def gather():
        # ONE NCCL all-gather of the per-scenario result records, on the solver's stream (north_star; SURVEY 8e)
        with torch.cuda.stream(lib_stream):
            rec[:B, :nx] = x_d
            rec[:B, nx] = f_d
            rec[:B, nx + 1] = st_d.double()
            rec[:B, nx + 2] = it_d.double()
            dist.all_gather_into_tensor(gathered, rec)

    def step_device():
        solver.solve_device(drops_d, x_d, f_d, st_d, it_d, order_streams=False)
        if world > 1:
            gather()

    # end-to-end arm: HOST buffers (pinned), host<->device copies inside the timed region.
    #   one GPU : the reference-facing C-ABI call landing_solve_batch(LANDING_HOST) does the copies itself
    #   N GPUs  : drops host -> device, solve, all-gather, the WHOLE sweep's records device -> host on every rank
    pin = lambda *sh, dt=torch.float64: torch.empty(*sh, dtype=dt).pin_memory()
    drops_p = pin(B, 12)
    drops_p.copy_(torch.from_numpy(drops_h))
    x_p, f_p, v_p = pin(B, nx), pin(B), pin(B)
    st_p, it_p = pin(B, dt=torch.int32), pin(B, dt=torch.int32)
    io = lc.api.SolveIO(lc.api._ptr(drops_p), None, lc.api._ptr(x_p), lc.api._ptr(f_p), None, lc.api._ptr(v_p),
                        lc.api._ptr(st_p, lc.api._ip), lc.api._ptr(it_p, lc.api._ip))
    gathered_p = pin(world * Bmax, nx + 3) if world > 1 else None
    drops_e = torch.zeros(B, 12, dtype=torch.float64, device=dev)

    def step_e2e():
        if world == 1:
            rc = solver.lib.landing_solve_batch(solver.ctx, B, lc.HOST, ctypes.byref(solver.problem),
                                                ctypes.byref(solver.options), ctypes.byref(io))
            assert rc == 0, solver.lib.landing_last_error()
        else:
            with torch.cuda.stream(lib_stream):
                drops_e.copy_(drops_p, non_blocking=True)
            solver.solve_device(drops_e, x_d, f_d, st_d, it_d, order_streams=False)
            gather()
            with torch.cuda.stream(lib_stream):
                gathered_p.copy_(gathered, non_blocking=True)
            solver.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(lib_stream):
            ev0.record()
        for _ in range(steps):
            fn()
        with torch.cuda.stream(lib_stream):
            ev1.record()
        barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for _ in range(args.warmup):
        step_device()
    l0 = solver.launches
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms = timed(step_device, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    launches = solver.launches - l0
    st = st_d.cpu().numpy()
    its = it_d.cpu().numpy()
    stats = torch.tensor([float((st == 0).sum()), float(its.sum())], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(stats)
    conv_per_step, iters_per_step = float(stats[0].item()), float(stats[1].item())
    value = conv_per_step * args.steps / (ms * 1e-3)
    if world > 1:
        g = gathered.cpu().numpy().reshape(world, Bmax, nx + 3)
        all_its = np.concatenate([g[r, :len(lc.shard_indices(cfg["total"], world, r)), nx + 2] for r in range(world)])
        all_st = np.concatenate([g[r, :len(lc.shard_indices(cfg["total"], world, r)), nx + 1] for r in range(world)])
    else:
        all_its, all_st = its, st
    last = None
    if args.dump_outputs and rank == 0:  # (the end-to-end arm below overwrites the device buffers when N > 1)
        if world > 1:
            last = sweep_records(g, cfg["total"], world)
        else:
            last = dict(x=x_d.cpu().numpy(), f=f_d.cpu().numpy(), status=st, iters=its)

    for _ in range(min(args.warmup, 1)):
        step_e2e()
    ms_e2e = timed(step_e2e, args.steps)
    if world == 1:
        conv_e = float((st_p.numpy() == 0).sum())
        h2d, d2h = B * 12 * 8, B * (nx + 2) * 8 + B * 8
    else:
        ge = gathered_p.numpy().reshape(world, Bmax, nx + 3)
        conv_e = float(sum((ge[r, :len(lc.shard_indices(cfg["total"], world, r)), nx + 1] == 0).sum() for r in range(world)))
        h2d, d2h = B * 12 * 8, world * Bmax * (nx + 3) * 8
    e2e_value = conv_e * args.steps / (ms_e2e * 1e-3)

    # strong-scaling base: the same fixed workload solved by ONE GPU (rank 0) in the same run
    one_gpu = None
    if world > 1 and not args.no_one_gpu_base:
        if rank == 0:
            full = torch.tensor(workload(cfg, 1, 0), device=dev)
            Bf = full.shape[0]
            xf = torch.zeros(Bf, nx, dtype=torch.float64, device=dev)
            ff = torch.zeros(Bf, dtype=torch.float64, device=dev)
            sf = torch.zeros(Bf, dtype=torch.int32, device=dev)
            itf = torch.zeros(Bf, dtype=torch.int32, device=dev)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(lib_stream):
                e0.record()
            solver.solve_device(full, xf, ff, sf, itf, order_streams=False)
            with torch.cuda.stream(lib_stream):
                e1.record()
            torch.cuda.synchronize()
            t1 = e0.elapsed_time(e1)
            one_gpu = {"n_gpus": 1, "value": float((sf == 0).sum().item()) / (t1 * 1e-3), "unit": UNIT, "ms_per_step": t1,
                       "note": "the whole %d-scenario sweep on rank 0's GPU alone, one step, same run" % Bf}
        dist.barrier()

    if rank == 0:
        hbm_peak, peak_src = measured_peaks()
        kernel_ms = ms / args.steps  # one k_solve launch per step; the all-gather (N>1) rides on the same stream
        local_iters = float(its.sum())
        hbm_ach = iter_bytes(N) * local_iters / (kernel_ms * 1e-3) / 1e9
        fp64_peak = solver.fp64_peak_tflops()
        fp64_ach = iter_flops(N) * local_iters / (kernel_ms * 1e-3) / 1e12
        tr = ncu_traffic()
        tr_ok = tr and tr.get("knots") == N and tr.get("batch") == B
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": config_dict(cfg, world),
            "converged_per_step": conv_per_step, "scenarios_per_step": cfg["total"],
            "kkt_iters_per_s": iters_per_step * args.steps / (ms * 1e-3),
            "iters": iter_stats(all_its, all_st),
            "gpu_launches": int(launches),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps,
                    "path": ("landing_solve_batch(LANDING_HOST): pinned host buffers through the C ABI" if world == 1 else
                             "per rank: drops host->device, landing_solve_batch(LANDING_DEVICE), NCCL all-gather of the "
                             "records, whole sweep device->host")},
            # the interior-point kernel is FP64-pipe bound by design (SURVEY 8d-ii): the binding line leads
            "roofline": {"bound": "fp64", "achieved": fp64_ach, "peak": fp64_peak, "unit": "TFLOP/s",
                         "frac": fp64_ach / fp64_peak if fp64_peak else None,
                         "peak_source": "measured in this run (landing_fp64_peak: DFMA micro-kernel, CUDA events; "
                                        "MEASURED_PEAKS.json has no FP64 entry)",
                         "traffic": (tr or {}).get("dram_bytes_per_launch") if tr_ok else None,
                         "traffic_source": (tr or {}).get("source") if tr_ok else None,
                         "kernel": "k_solve", "units_per_launch": local_iters,
                         "flops_per_unit": iter_flops(N), "bytes_per_unit": iter_bytes(N),
                         "hbm": {"bound": "hbm", "achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": hbm_ach / hbm_peak, "peak_source": peak_src},
                         "note": "one launch per step = all interior-point iterations of the rank's scenarios; unit = one "
                                 "KKT iteration of one scenario; achieved = algorithmic flops (one factorisation per "
                                 "iteration, DESIGN.md 2.3) / CUDA-event time; the hbm line uses the algorithmic bytes of "
                                 "SURVEY 8d-ii"},
        }
        if one_gpu:
            line["one_gpu_same_workload"] = one_gpu
            line["strong_scaling_efficiency_vs_one_gpu"] = value / (world * one_gpu["value"])
        if world == 1 and not args.no_eval_kernels and cfg.get("formulation") != "schedule":
            # the evaluation kernels (HBM-bound rows a-3..a-6 of SURVEY 8): 16k scenarios, SoA, a few milliseconds
            try:
                sys.path.insert(0, os.path.join(ROOT, "tools"))
                from bench_eval import cpu_reference, dropin_latency, measure
                keys = ("function", "N", "B", "layout", "ms", "achieved", "peak", "unit", "frac", "evals_per_s")
                line["roofline"]["eval_kernels"] = [
                    {k: r[k] for k in keys} for r in measure(N, 16384, 10, "soa", solver=solver, device=local_rank)]
                # the size the reference ships generated C for (N = 21), with the reference's own compiled functions
                # timed on the host cores beside it (oracle/_ref, kind "reference")
                ref = cpu_reference()
                s21 = lc.LandingSolver(N=21, device=local_rank)
                rows = [{k: r[k] for k in keys} for r in measure(21, 16384, 10, "soa", solver=s21, device=local_rank)]
                # the kino-dynamic functions (SURVEY 8 f-2; the KNITRO variant's N = 21 problem)
                from bench_kino import measure_kino
                line["roofline"]["kino_kernels_n21"] = [{k: r[k] for k in keys} for r in measure_kino(21, 16384, 10, solver=s21, device=local_rank)]
                s21.close()
                for r in rows:
                    r["cpu_baseline"] = ref.get(r["function"]) if ref else None
                line["roofline"]["eval_kernels_n21"] = rows
                # one scenario per call through the CasADi symbols of the drop-in (what the unmodified reference would do)
                line["roofline"]["dropin_call_latency"] = dropin_latency()
            except Exception as e:  # reported, never hidden
                line["roofline"]["eval_kernels"] = {"error": repr(e)}
        if world == 1:
            # CPU baseline on the host cores (bounded sample of the same workload; rank 0 at N = 1 only)
            cores = os.cpu_count() or 1
            sub, stride = cpu_sample(cfg, drops_h, args.cpu_sample)
            cpu_run(N, sub[:cores], cores, cfg)  # (builds the -O3 library, warms the threads)
            r, dt = cpu_run(N, sub, cores, cfg)
            line["cpu_baseline"] = {
                "value": float((r["status"] == 0).sum()) / dt, "unit": UNIT, "cores": cores, "kind": "port",
                "kkt_iters_per_s": float(r["iters"].sum()) / dt,
                "sample": "%d of %d scenarios (every %d-th), %.1f s; IPOPT substitute oracle/ip_ref.c (%s), OpenMP over scenarios"
                          % (len(sub), B, stride, dt, cpu_flags())}
        if last is not None:
            dump_outputs(args.dump_outputs, last["x"], last["f"], last["status"], last["iters"])
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
