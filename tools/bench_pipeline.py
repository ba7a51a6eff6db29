"""The reference's two-stage pipeline on one GPU, the nearest thing to BASELINE configs[3] ("full-body" landing NLP, 4k drop
conditions, N=40): SRB solve of every drop (k_solve) -> bounds and initial guess of the kino-dynamic NLP from the SRB
solutions (k_kino_setup; generate_landingCtrller_KNITRO.m:300-327) -> one evaluation of the kino-dynamic constraint
function and CCS Jacobian at that guess (the hand-over check below) -> the kino-dynamic interior-point solve of every drop
from its SRB solution (landing_kino_solve_batch; DESIGN.md 3.2).  All buffers stay in HBM; times are CUDA events on the
library stream.
   usage: python tools/bench_pipeline.py [N] [B]"""
import json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import landing_controller_b200 as lc

N = int(sys.argv[1]) if len(sys.argv) > 1 else 40
B = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
dev = torch.device("cuda:0")
s = lc.LandingSolver(N=N)
lc.apply_sweep_parameters(s.problem)            # the sweep callers' parameter set (f_max, leg length, weights)
dt = np.full(N - 1, 0.6 / (N - 1))
drops = lc.grid_sweep(B)
d = torch.tensor(drops, device=dev)
kd = s.kino_dims()
pb = s.kino_problem(dt)
nx = s.dims["nx"]
x = torch.zeros(B, nx, dtype=torch.float64, device=dev); f = torch.zeros(B, dtype=torch.float64, device=dev)
st = torch.zeros(B, dtype=torch.int32, device=dev); it = torch.zeros(B, dtype=torch.int32, device=dev)
lb = torch.zeros(B, kd["m"], dtype=torch.float64, device=dev); ub = torch.zeros_like(lb)
x0 = torch.zeros(B, kd["nx"], dtype=torch.float64, device=dev)
g = torch.zeros(B, kd["m"], dtype=torch.float64, device=dev)
jac = torch.zeros(B, kd["nnzJ"], dtype=torch.float64, device=dev)
stream = torch.cuda.ExternalStream(s.stream_ptr, device=dev)
xk = torch.zeros(B, kd["nx"], dtype=torch.float64, device=dev); fk = torch.zeros(B, dtype=torch.float64, device=dev)
stk = torch.zeros(B, dtype=torch.int32, device=dev); itk = torch.zeros(B, dtype=torch.int32, device=dev)
ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]


def run():
    with torch.cuda.stream(stream):
        ev[0].record()
    s.solve_device(d, x, f, st, it)
    with torch.cuda.stream(stream):
        ev[1].record()
    s.kino_setup_device(d, x_srb=x, lbg=lb, ubg=ub, x0=x0)
    with torch.cuda.stream(stream):
        ev[2].record()
    s.kino_eval_device(x0, pb, g=g, jac=jac, layout=lc.AOS)
    with torch.cuda.stream(stream):
        ev[3].record()
    s.kino_solve_device(d, xk, fk, stk, itk, x_srb=x, pb=pb)
    with torch.cuda.stream(stream):
        ev[4].record()
    torch.cuda.synchronize()
    return [ev[i].elapsed_time(ev[i + 1]) for i in range(4)]


run()
t = run()
sth, ith = st.cpu().numpy(), it.cpu().numpy()
viol = torch.clamp(torch.maximum(lb - g, g - ub), min=0.0)
conv = torch.tensor(sth == 0, device=dev)
vmax = viol[conv].max(dim=1).values.cpu().numpy()
# rows that are the same equations in both stages (v+ - v - rddot dt, r+ - r - v dt): the SRB solution must satisfy them to
# the SRB solver's constraint tolerance -- a check that the hand-over (variable order, mass, dt) is consistent
rows = torch.tensor([48 + 141 * k + i for k in range(N - 1) for i in (0, 1, 2, 6, 7, 8)], device=dev)
dyn = g[conv][:, rows].abs().max().item()
stk_h, itk_h = stk.cpu().numpy(), itk.cpu().numpy()
conv_k = int((stk_h == 0).sum())
print(json.dumps({"workload": "%d grid drops, N=%d, sweep callers' parameters: SRB solve -> kino-dynamic set-up -> g and Jacobian at the guess -> kino-dynamic solve" % (B, N),
                  "device": torch.cuda.get_device_name(0), "end_to_end_ms": sum(t),
                  "kino_solve_ms": t[3], "kino_converged": conv_k, "kino_statuses": np.bincount(stk_h, minlength=5).tolist(),
                  "kino_iters_mean": float(itk_h.mean()), "pipeline_converged_per_s": conv_k / (sum(t) * 1e-3),
                  "srb_solve_ms": t[0], "srb_converged": int((sth == 0).sum()), "srb_nlp_per_s": float((sth == 0).sum()) / (t[0] * 1e-3),
                  "srb_kkt_iters": int(ith.sum()), "kino_setup_ms": t[1], "kino_g_jac_ms": t[2],
                  "kino_sizes": kd, "kino_bytes_moved_GB": 8e-9 * B * (2 * kd["m"] + 2 * kd["nx"] + nx + 12 + kd["m"] + kd["nnzJ"]),
                  "kino_row_violation_at_the_guess": {"median_of_max": float(np.median(vmax)), "max": float(vmax.max()),
                                                      "translational_dynamics_rows_max": dyn,
                                                      "note": "translational dynamics are the same equations in both stages (consistency of the hand-over); the SRB stage uses the ZYX, the kino-dynamic NLP the XYZ rotation convention and the guess has constant joint angles, so the other rows are violated at the guess, as in the reference"}}))
s.close()
