#!/usr/bin/env python
"""Matrix-free Jacobian products (tolcuda_jac_vec / tolcuda_jac_tvec) next to the F+G evaluation they replace
when G itself is not wanted, and the Hessian-of-the-Lagrangian product (tolcuda_lag_hess_vec) next to the central
difference of two tolcuda_jac_tvec launches it replaces: device-resident, CUDA events on the launching stream.  Then
the goal-table arm: y, z and w with a table of B distinct goals (tolcuda_*_goals) against the same products with the
context's goal, and w for 256 goals x 64 trajectories as one tolcuda_lag_hess_vec_goals launch against 256 per-goal
contexts launched one after another.  The first line names the card and its power limit, read in the same run.

    python tools/opbench.py [--workload S10_tempest_ts200] [--batch 65536] [--steps 20]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import tol_b200 as T  # noqa: E402
from tol_b200.evaluator import padded_ld  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--workload", default="S10_tempest_ts200")
ap.add_argument("--batch", type=int, default=65536)
ap.add_argument("--steps", type=int, default=20)
args = ap.parse_args()
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
print(json.dumps({"gpu": smi, "library": T.LIB_PATH}))
g = np.load(os.path.join(ROOT, "tests", "golden", args.workload + ".npz"))
ev = T.Evaluator.from_golden(g)
B, n, neF, neG, ts = args.batch, ev.n, ev.neF, ev.neG, int(g["ts"])
ldx, ldF, ldG = padded_ld(n), padded_ld(neF), padded_ld(neG)
U = min(B, 512)
Xu = torch.zeros(U, ldx, dtype=torch.float64)
T.synth.batch(g["x"][0], 1, 0, U, out=Xu.numpy())
idx = torch.arange(B, device="cuda") % U
Xd = Xu.cuda()[idx].contiguous()
D = (torch.rand(B, ldx, dtype=torch.float64, device="cuda") * 2 - 1)
Lam = (torch.rand(B, ldF, dtype=torch.float64, device="cuda") * 2 - 1)
Y, Z = torch.empty(B, ldF, dtype=torch.float64, device="cuda"), torch.empty(B, ldx, dtype=torch.float64, device="cuda")
W, Zh = torch.empty(B, ldx, dtype=torch.float64, device="cuda"), torch.empty(B, ldx, dtype=torch.float64, device="cuda")
Xp, Xm = torch.empty_like(Xd), torch.empty_like(Xd)
h = 1e-6


def central_difference():
    # the pair of jac_tvec launches at x +- h d and the two shifted copies of x that lag_hess_vec replaces
    torch.add(Xd, D, alpha=h, out=Xp)
    torch.add(Xd, D, alpha=-h, out=Xm)
    ev.jac_tvec(Xp, Lam, Z, sync=False)
    ev.jac_tvec(Xm, Lam, W, sync=False)
    torch.sub(Z, W, out=W).mul_(0.5 / h)


Fd, Gd = torch.empty(B, ldF, dtype=torch.float64, device="cuda"), torch.empty(B, ldG, dtype=torch.float64, device="cuda")
st = torch.cuda.Stream()
ev.set_stream(st.cuda_stream)


def timed(fn):
    with torch.cuda.stream(st):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(args.steps):
            fn()
        e1.record(st)
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) / args.steps


for label, fn, by in (
        ("F+G (G written)", lambda: ev.eval_batch_device(Xd, Fd, Gd, sync=False), 8.0 * B * (n + neF + neG)),
        ("y = J d", lambda: ev.jac_vec(Xd, D, Y, sync=False), 8.0 * B * (2 * n + neF)),
        ("z = J^T lambda", lambda: ev.jac_tvec(Xd, Lam, Z, sync=False), 8.0 * B * (2 * n + neF)),
        ("w = H d", lambda: ev.lag_hess_vec(Xd, Lam, D, W, sync=False), 8.0 * B * (4 * n + neF)),
        ("w = H d + z = J^T lambda", lambda: ev.lag_hess_vec(Xd, Lam, D, W, Zh, sync=False), 8.0 * B * (5 * n + neF)),
        ("central difference: 2 shifted x + 2 x J^T lambda", central_difference, 8.0 * B * (2 * (2 * n + neF) + 9 * n))):
    ms = timed(fn)
    print(json.dumps({"workload": args.workload, "B": B, "op": label, "ms": ms, "node_evals_per_s": B * ts / (ms * 1e-3),
                      "algorithmic_GB": by / 1e9, "GBps": by / ms / 1e6, "frac_of_6544": by / ms / 1e6 / 6544.0}))

# goal-table arm: every trajectory its own goal, against the context's goal (the rows above)
mission = str(g["mission"])
ev.set_goals(T.synth.goals(mission, 0, B))
for label, fn in (("y = J d, goal table", lambda: ev.jac_vec(Xd, D, Y, sync=False, row0=0)),
                  ("z = J^T lambda, goal table", lambda: ev.jac_tvec(Xd, Lam, Z, sync=False, row0=0)),
                  ("w = H d, goal table", lambda: ev.lag_hess_vec(Xd, Lam, D, W, sync=False, row0=0))):
    print(json.dumps({"workload": args.workload, "B": B, "op": label, "goals": B, "ms": timed(fn)}))

# 256 missions x 64 trajectories: one launch with a goal table against one context (and one launch) per mission
K, R = 256, 64
if B >= K * R:
    goals = T.synth.goals(mission, 0, K)
    ev.set_goals(np.repeat(goals, R, axis=0))
    Xs, Ls, Ds, Ws = Xd[:K * R], Lam[:K * R], D[:K * R], W[:K * R]
    print(json.dumps({"workload": args.workload, "op": "w = H d, one launch, %d goals x %d" % (K, R),
                      "ms": timed(lambda: ev.lag_hess_vec(Xs, Ls, Ds, Ws, sync=False, row0=0))}))
    ctxs = [T.Evaluator(mission, ts, g["ac"], g["gn"], goals[k], int(g["wind_model"])) for k in range(K)]
    for e in ctxs:
        e.set_stream(st.cuda_stream)

    def per_goal_contexts():
        for k, e in enumerate(ctxs):
            s = slice(k * R, (k + 1) * R)
            e.lag_hess_vec(Xs[s], Ls[s], Ds[s], Ws[s], sync=False)
    print(json.dumps({"workload": args.workload, "op": "w = H d, %d per-goal contexts x %d" % (K, R),
                      "ms": timed(per_goal_contexts)}))
    for e in ctxs:
        e.close()
ev.close()
