#!/usr/bin/env python
"""Kernel-only timing helper (device-resident, CUDA events on the launching stream): used to compare
kernel variants and as the short command that is run under ncu.  Not the bench contract -- bench.py is.

    python tools/kbench.py --workload S10_tempest_ts200 --batch 16384 --steps 10"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ap = argparse.ArgumentParser()
ap.add_argument("--workload", default="S10_tempest_ts200")
ap.add_argument("--batch", type=int, default=16384)
ap.add_argument("--steps", type=int, default=10)
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--kernel", type=int, default=0)
ap.add_argument("--per", type=int, default=0)
ap.add_argument("--tail-x4", type=int, default=-1)
ap.add_argument("--overlap", type=int, default=0, help="1: TOLCUDA_OVERLAP, 2: TOLCUDA_OVERLAP_DISJOINT (two result buffer sets)")
ap.add_argument("--goff", type=int, default=0, help="shift the G buffer by this many doubles (alignment experiments)")
ap.add_argument("--need", default="FG", help="F, FG, or S (the per-trajectory summary alone)")
ap.add_argument("--distinct", type=int, default=512, help="distinct synthetic trajectories (tiled)")
ap.add_argument("--ts", type=int, default=0, help="override the number of windows (x0 = the restated InitialCond for that ts)")
args = ap.parse_args()
import tol_b200 as T  # noqa: E402
from tol_b200.evaluator import padded_ld  # noqa: E402

g = np.load(os.path.join(ROOT, "tests", "golden", args.workload + ".npz"))
if args.ts:
    lm = g["lm"]
    cfg = T.make_config(str(g["mission"]), args.ts, g["ac"], g["gn"], g["goal_ned"],
                        limits=[lm[0], lm[1], lm[5], lm[2], lm[6], lm[3], lm[7], lm[4]])
    x0 = T.initial_guess(cfg)
    ev = T.Evaluator(str(g["mission"]), args.ts, g["ac"], g["gn"], g["goal_ned"])
else:
    x0 = g["x"][0]
    ev = T.Evaluator.from_golden(g)
B, n, neF, neG, ts = args.batch, ev.n, ev.neF, ev.neG, args.ts or int(g["ts"])
ldx, ldF, ldG = padded_ld(n), padded_ld(neF), padded_ld(neG)
seed0 = T.synth.SEED_S10 if str(g["mission"]) == "S10" else T.synth.SEED_G7
U = min(B, args.distinct)
Xu = torch.zeros(U, ldx, dtype=torch.float64)
T.synth.batch(x0, seed0, 0, U, out=Xu.numpy())
Xd = Xu.cuda()[torch.arange(B, device="cuda") % U].contiguous()
ev.set_option("kernel", args.kernel)
ev.set_option("per", args.per)
if args.tail_x4 >= 0:
    ev.set_option("tail_x4", args.tail_x4)
nset = 2 if args.overlap == 2 else 1
Fs = [torch.empty(B, ldF, dtype=torch.float64, device="cuda") for _ in range(nset)]
Gs = [torch.empty(B * ldG + 64, dtype=torch.float64, device="cuda")[args.goff:args.goff + B * ldG].view(B, ldG) for _ in range(nset)]
st = torch.cuda.Stream()
ev.set_stream(st.cuda_stream)
needF, needG = "F" in args.need, "G" in args.need
with torch.cuda.stream(st):
    for i in range(args.warmup):
        ev.eval_batch_device(Xd, Fs[i % nset], Gs[i % nset], needF, needG, sync=False, overlap=args.overlap)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for i in range(args.steps):
        ev.eval_batch_device(Xd, Fs[i % nset], Gs[i % nset], needF, needG, sync=False, overlap=args.overlap)
    e1.record(st)
    torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / args.steps
if args.need == "S":  # screening: only the per-trajectory summary is produced (tolcuda_eval_batch_summary, F = G = NULL)
    Sd = torch.empty(B, 4, dtype=torch.float64, device="cuda")
    fl = T.evaluator.DEVICE_PTRS | T.evaluator.NO_SYNC
    def summ():
        T.lib.check(ev.L.tolcuda_eval_batch_summary(ev.h, B, Xd.data_ptr(), Xd.stride(0), None, 0, None, 0, Sd.data_ptr(), 4, fl))
    with torch.cuda.stream(st):
        for _ in range(args.warmup):
            summ()
        torch.cuda.synchronize()
        e0.record(st)
        for _ in range(args.steps):
            summ()
        e1.record(st)
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    needF = needG = False
by = 8.0 * B * (n + (neF if needF else 0) + (neG if needG else 0) + (4 if args.need == "S" else 0))
print(json.dumps({"workload": args.workload, "B": B, "kernel": args.kernel, "per": args.per, "tail_x4": args.tail_x4, "overlap": args.overlap, "goff": args.goff, "need": args.need, "ms": ms,
                  "node_evals_per_s": B * ts / (ms * 1e-3), "GBps": by / ms / 1e6,
                  "frac_of_6544": by / ms / 1e6 / 6544.0}))
