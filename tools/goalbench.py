"""Per-trajectory goals against the context's goal on one GPU (tolcuda_eval_batch_goals vs tolcuda_eval_batch).

  (a) same bytes, per-row goals: S10 ts=200 B=65,536 (bench.py's batch) and G7 ts=100 B=4,096; F+G, F only and summary
      only; the context's goal against a table of B distinct goals (synth.goals).  Both arms run in the same process,
      alternating in blocks of 50 launches (CUDA events around each block, after warm-up), every launch
      TOLCUDA_OVERLAP_DISJOINT into one of two result-buffer sets as bench.py enqueues its steps.
  (b) many missions: 256 goals x 64 trajectories (S10 ts=200, device pointers) -- one tolcuda_eval_batch_goals launch
      against 256 contexts, one per goal, launched one after another on the same stream; end to end (events around
      the whole enqueue, synchronised), alternating blocks.
  (c) host-pointer path: one end-to-end step of the bench batch (pinned host x -> host F, G rows), both arms, host
      clock around the synchronous call, alternating.
Before timing, a table holding B copies of the context's goal must give the same bits as the homogeneous launch.
Roofline: algorithmic bytes 8*(n + neF + neG) per trajectory (F only: n + neF; summary only: n + 4; the goal table's
64 bytes per row are not counted) over launch time, against 6544 GB/s.

usage: python tools/goalbench.py [--out FILE] [--blocks N]"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PEAK_GBS = 6544.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--blocks", type=int, default=6, help="timed blocks per arm")
    args = ap.parse_args()
    import torch
    import tol_b200 as T
    EV = T.evaluator
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    say("device: %s (nvidia-smi name, power.limit); torch sees %s" % (smi[0] if smi else "?", torch.cuda.get_device_name(0)))
    stream = torch.cuda.current_stream()

    def golden(name):
        return np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))

    def blocks_ms(fn_a, fn_b, per_block, nblocks):
        """alternating timed blocks of `per_block` calls of each arm; returns (median ms per call of a, of b)"""
        ta, tb = [], []
        for fn, out in ((fn_a, None), (fn_b, None)):  # warm-up
            for _ in range(5):
                fn()
        torch.cuda.synchronize()
        for _ in range(nblocks):
            for fn, out in ((fn_a, ta), (fn_b, tb)):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(per_block):
                    fn()
                e1.record(stream)
                torch.cuda.synchronize()
                out.append(e0.elapsed_time(e1) / per_block)
        return float(np.median(ta)), float(np.median(tb)), ta, tb

    def bits(t):
        return t.view(torch.int64)

    # ---- (a) -------------------------------------------------------------------------------------------------------
    say("\n(a) same bytes: context goal vs a table of B distinct goals; %d alternating blocks of 50 launches per arm, "
        "TOLCUDA_OVERLAP_DISJOINT into two buffer sets" % args.blocks)
    for fixture, seed0, B in (("S10_tempest_ts200", T.synth.SEED_S10, 65536), ("G7_skywalker_ts100", T.synth.SEED_G7, 4096)):
        g = golden(fixture)
        mission, ts = str(g["mission"]), int(g["ts"])
        ev = T.Evaluator.from_golden(g)
        ev.set_stream(stream.cuda_stream)
        X = torch.from_numpy(T.synth.batch(g["x"][0], seed0, 0, B)).cuda()
        ev.set_goals(np.repeat(np.asarray(g["goal_ned"], dtype=np.float64)[None, :], B, axis=0))
        F = [torch.empty(B, ev.neF, dtype=torch.float64, device="cuda") for _ in range(2)]
        G = [torch.empty(B, ev.neG, dtype=torch.float64, device="cuda") for _ in range(2)]
        S = [torch.empty(B, 4, dtype=torch.float64, device="cuda") for _ in range(2)]
        # sanity: B copies of the context's goal give the homogeneous launch's bits (F+G and summary)
        ev.eval_batch_device(X, F[0], G[0])
        ev.eval_batch_goals(X, F[1], G[1])
        T.lib.check(ev.L.tolcuda_eval_batch_summary(ev.h, B, X.data_ptr(), X.stride(0), None, 0, None, 0, S[0].data_ptr(), 4,
                                                    EV.DEVICE_PTRS))
        ev.eval_batch_goals(X, None, None, summary=S[1], needF=False, needG=False)
        assert torch.equal(bits(F[0]), bits(F[1])) and torch.equal(bits(G[0]), bits(G[1])), "goal table of copies differs"
        assert torch.equal(bits(S[0]), bits(S[1])), "goal table of copies differs (summary)"
        ev.set_goals(T.synth.goals(mission, 0, B))
        fl = EV.DEVICE_PTRS | EV.NO_SYNC | EV.OVERLAP_DISJOINT
        by = {"F+G": 8.0 * (ev.n + ev.neF + ev.neG) * B, "F only": 8.0 * (ev.n + ev.neF) * B, "summary only": 8.0 * (ev.n + 4) * B}
        for flav in ("F+G", "F only", "summary only"):
            k = [0]

            def args_of():
                i = k[0] = k[0] ^ 1
                if flav == "F+G":
                    return (F[i].data_ptr(), F[i].stride(0), G[i].data_ptr(), G[i].stride(0), None, 0, fl | EV.NEED_F | EV.NEED_G)
                if flav == "F only":
                    return (F[i].data_ptr(), F[i].stride(0), None, 0, None, 0, fl | EV.NEED_F)
                return (None, 0, None, 0, S[i].data_ptr(), 4, fl)

            def ctx():
                T.lib.check(ev.L.tolcuda_eval_batch_summary(ev.h, B, X.data_ptr(), X.stride(0), *args_of()))

            def tab():
                T.lib.check(ev.L.tolcuda_eval_batch_goals(ev.h, 0, B, X.data_ptr(), X.stride(0), *args_of()))
            ma, mb, ta, tb = blocks_ms(ctx, tab, 50, args.blocks)
            say("  %s ts=%d B=%d %-12s context goal %.4f ms (%.4g node-evals/s, %.3f of roofline) | goal table %.4f ms "
                "(%.4g node-evals/s, %.3f of roofline) | table/context throughput %.4f   [blocks ctx %s | table %s]"
                % (mission, ts, B, flav, ma, B * ts / ma * 1e3, by[flav] / ma / 1e6 / PEAK_GBS, mb, B * ts / mb * 1e3,
                   by[flav] / mb / 1e6 / PEAK_GBS, ma / mb, " ".join("%.4f" % t for t in ta), " ".join("%.4f" % t for t in tb)))
        ev.close()
        del X, F, G, S
        torch.cuda.empty_cache()

    # ---- (b) -------------------------------------------------------------------------------------------------------
    g = golden("S10_tempest_ts200")
    K, R = 256, 64
    B = K * R
    say("\n(b) many missions: %d goals x %d trajectories, S10 ts=200, device pointers; one launch with a goal table vs "
        "%d contexts launched one after another on one stream" % (K, R, K))
    goals = T.synth.goals("S10", 0, K)
    X = torch.from_numpy(T.synth.batch(g["x"][0], T.synth.SEED_S10, 0, B)).cuda()  # rows [k*R, (k+1)*R): goal k
    ev = T.Evaluator.from_golden(g)
    ev.set_stream(stream.cuda_stream)
    ev.set_goals(np.repeat(goals, R, axis=0))
    ctxs = []
    for k in range(K):
        e = T.Evaluator("S10", 200, g["ac"], g["gn"], goals[k], 1)
        e.set_stream(stream.cuda_stream)
        ctxs.append(e)
    F = [torch.empty(B, ev.neF, dtype=torch.float64, device="cuda") for _ in range(2)]
    G = [torch.empty(B, ev.neG, dtype=torch.float64, device="cuda") for _ in range(2)]
    ev.eval_batch_goals(X, F[0], G[0])
    for k, e in enumerate(ctxs):
        e.eval_batch_device(X[k * R:(k + 1) * R], F[1][k * R:(k + 1) * R], G[1][k * R:(k + 1) * R])
    assert torch.equal(bits(F[0]), bits(F[1])) and torch.equal(bits(G[0]), bits(G[1])), "(b): one launch != 256 contexts"

    def one():
        ev.eval_batch_goals(X, F[0], G[0], sync=False)

    def many():
        for k, e in enumerate(ctxs):
            e.eval_batch_device(X[k * R:(k + 1) * R], F[1][k * R:(k + 1) * R], G[1][k * R:(k + 1) * R], sync=False)
    ma, mb, ta, tb = blocks_ms(one, many, 10, args.blocks)
    say("  one launch %.4f ms | %d launches %.4f ms | ratio %.2f   [blocks one %s | many %s]"
        % (ma, K, mb, mb / ma, " ".join("%.4f" % t for t in ta), " ".join("%.4f" % t for t in tb)))
    for e in ctxs:
        e.close()
    ev.close()
    del X, F, G
    torch.cuda.empty_cache()

    # ---- (c) -------------------------------------------------------------------------------------------------------
    B = 65536
    say("\n(c) host-pointer path: one end-to-end step of S10 ts=200 B=%d (pinned host x -> host F, G rows), host clock "
        "around the synchronous call, %d alternating steps per arm" % (B, args.blocks))
    ev = T.Evaluator.from_golden(g)
    ev.set_goals(T.synth.goals("S10", 0, B))
    Xh = torch.zeros(B, ev.n, dtype=torch.float64, pin_memory=True)
    T.synth.batch(g["x"][0], T.synth.SEED_S10, 0, B, out=Xh.numpy())
    Fh = torch.empty(B, ev.neF, dtype=torch.float64, pin_memory=True)
    Gh = torch.empty(B, ev.neG, dtype=torch.float64, pin_memory=True)
    arms = {"context goal": lambda: ev.eval_batch_host(Xh.numpy(), Fh.numpy(), Gh.numpy()),
            "goal table": lambda: ev.eval_batch_goals(Xh.numpy(), Fh.numpy(), Gh.numpy())}
    res = {k: [] for k in arms}
    for k, fn in arms.items():
        fn()
    for _ in range(args.blocks):
        for k, fn in arms.items():
            t0 = time.perf_counter()
            fn()
            res[k].append((time.perf_counter() - t0) * 1e3)
    for k, v in res.items():
        say("  %-12s median %.3f ms (%.4g node-evals/s end to end)   [steps %s]"
            % (k, np.median(v), B * 200 / np.median(v) * 1e3, " ".join("%.3f" % t for t in v)))
    ev.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
