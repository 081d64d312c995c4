#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Metric: FP64 F+G node-evals/s = trajectories x collocation windows evaluated per second.
Workload: S10 / tempest, 65,536 trajectories x ts = 200 windows (BASELINE.json configs[3], the configuration the
metric's 60 %-of-HBM target and its 1/2/4/8-GPU scaling are quoted on; 13.2 GB, fits one B200), synthetic inputs per
SURVEY.md section 8d.  The batch is SHARDED by trajectory index over the N ranks (STRONG scaling: 65,536 rows on 1
GPU, 8,192 per GPU on 8; BASELINE.md: 1.656 GB / GPU at 8) -- no collective on the data path.  One "step" = one F+G
pass over the whole batch = one kernel launch per rank.

  value     device-resident: x, F, G live in HBM; K launches per rank timed with CUDA events on the launching
            stream, max over ranks.  Consecutive steps are independent batches, so they are enqueued with
            TOLCUDA_OVERLAP_DISJOINT (programmatic dependent launch: the next grid's CTAs move into the SMs the
            previous grid's tail has left) and write two result-buffer sets alternately; run.launch_ms_serial is
            the same loop with plain, serialised launches.  Every step touches far more than the 126 MB L2
            (13.2 GB on 1 GPU, 1.66 GB per GPU on 8), so no L2 flush is needed.
  e2e       the same pass through tolcuda_eval_batch with HOST (pinned) x, F, G: chunked H2D -> kernel -> D2H inside
            the timed region; full F and G rows are in host memory at the end of every step.  e2e.ceiling is what
            the box's host side could deliver at best for those bytes (tools/exp/hostceil: concurrent pinned copies
            on the N GPUs + non-temporal fills on the host threads, measured in this run), e2e.frac = value/ceiling.
  roofline  algorithmic bytes 8*(n+neF+neG) per trajectory x this rank's rows / average launch duration / HBM peak.
  cpu_baseline (N=1)  the reference's own CPU path (oracle/_ref, unmodified sources, -O2): all host cores as
            independent processes on a bounded sample of the same batch, plus the two single-core variants of
            BASELINE.md section 4 (callback as shipped with its dump files; arithmetic only).
  secondary (N=1)  BASELINE.json configs[2] (G7, 4,096 x 100) and the single-trajectory callback latency.
  gather (N>1)  the shards' rows gathered on GPU 0: fused evaluate+gather over NVLink peer memory against the NCCL
            gather, with a bit-identity flag.

--impl reference runs only the CPU arm (same config dict, bounded sample of the same rows) with "impl": "reference".

--dump-outputs DIR writes what the last timed step left in HBM, for a fixed, seeded sample of the batch's trajectories
(the same rows on any number of GPUs, at most 64 MB in all): DIR/F.npy [k, neF] and DIR/G.npy [k, neG], float64, the
rows a caller of tolcuda_eval_batch receives.  The inputs depend only on the arguments, so two builds run with the
same arguments can be compared output for output."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "fp64_FG_node_evals_per_s"
UNIT = "node-evals/s"
WORKLOADS = {
    # name: (fixture with x0 + parameters, seed0, trajectories of the whole batch)
    "S10_tempest_ts200_B65536": ("S10_tempest_ts200", 20270000, 65536),
    "G7_skywalker_ts100_B4096": ("G7_skywalker_ts100", 20260000, 4096),
}
RTOL, ATOL = 1e-12, 1e-14  # north_star tolerance
DUMP_BYTES = 64 * 10**6 - 4096  # --dump-outputs: both .npy files together, headers included
DUMP_SEED = 20261020


def golden(name):
    return np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))


def config_of(wl_name, B_total):
    """identical in both arms: what is evaluated, not how"""
    fixture, seed0, _ = WORKLOADS[wl_name]
    g = golden(fixture)
    mission, ts = str(g["mission"]), int(g["ts"])
    n = 1 + 11 * (ts + 1)
    neF = 1 + 8 * ts + (11 if mission == "S10" else 12)
    neG = 107 * ts + 37 if mission == "S10" else 105 * ts + 48
    return {"workload": wl_name, "mission": mission, "aircraft": str(g["aircraft"]), "ts": ts,
            "trajectories_total": B_total, "n": n, "neF": neF, "neG": neG,
            "inputs": "x0*(1+0.05u)+0.01u', PCG64(seed0+b), seed0=%d (SURVEY.md 8d)" % seed0,
            "parallelism": "rows sharded by trajectory index over the ranks, no collective",
            "l2": "every step touches >= 1.6 GB per GPU, far more than the 126 MB L2; no flush needed"}


def close(a, b):
    return bool((np.abs(a - b) <= ATOL + RTOL * np.abs(b)).all())


# ------------------------------------------------------------------------------ CPU reference arm

_W = {}
CPU_BLOCK = 128  # trajectories a worker evaluates per call (its F/G rows are reused, as the reference reuses its arrays)


def _make_problem(fixture, use_ref, null_io=True):
    g = golden(fixture)
    if use_ref:
        import refclient as R
        ts = int(g["ts"])
        return R.RefProblem(str(g["mission"]), str(g["aircraft"]), tuple(g["enu"]), tuple(g["goal_enu"]),
                            ts=None if ts == 100 else ts, null_io=null_io)
    import portclient as P
    return P.PortProblem(str(g["mission"]), int(g["ts"]), g["ac"], g["gn"], g["goal_ned"], int(g["wind_model"]))


def _worker_init(fixture, use_ref):
    """one reference (or port) problem object per process: the reference is not thread-safe
    (process-global `prob`, member scratch; SURVEY.md section 2)"""
    _W["g"] = golden(fixture)
    _W["p"] = _make_problem(fixture, use_ref)


def _worker_run(args):
    seed0, b0, count = args
    import tol_b200.synth as synth
    p, g = _W["p"], _W["g"]
    key = (seed0, b0, count)
    if _W.get("key") != key:  # inputs are prepared once, outside the timed step
        _W["key"] = key
        _W["X"] = synth.batch(g["x"][0], seed0, b0, b0 + count)
        _W["F"] = np.empty((CPU_BLOCK, p.neF))
        _W["G"] = np.empty((CPU_BLOCK, p.neG))
    X, F, G = _W["X"], _W["F"], _W["G"]
    t0 = time.perf_counter()
    acc = 0.0
    for a in range(0, count, CPU_BLOCK):
        e = min(count, a + CPU_BLOCK)
        p.eval_many(X[a:e], F[:e - a], G[:e - a])
        acc += float(F[:e - a, 0].sum())
    return time.perf_counter() - t0, acc


class CpuArm:
    """the reference's CPU implementation of the path on all usable host cores"""

    def __init__(self, fixture, seed0, B_total):
        import multiprocessing as mp
        import portclient as P
        import refclient as R
        self.fixture, self.seed0, self.B_total = fixture, seed0, B_total
        self.use_ref = R.available()
        if not self.use_ref and not P.available():
            subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "port"])
        self.cores = max(1, min(len(os.sched_getaffinity(0)), 128))
        self.kind = "reference" if self.use_ref else "port"
        self.pool = mp.get_context("fork").Pool(self.cores, _worker_init, (fixture, self.use_ref))
        self.ts = int(golden(fixture)["ts"])
        self.rows = 0

    def set_rows(self, rows):
        """rows [0, rows) of the batch per step, split evenly over the processes"""
        per = max(1, min(rows, self.B_total) // self.cores)
        self.rows = per * self.cores
        self.per = per

    def step(self):
        jobs = [(self.seed0, w * self.per, self.per) for w in range(self.cores)]
        t0 = time.perf_counter()
        self.pool.map(_worker_run, jobs, chunksize=1)
        wall = time.perf_counter() - t0
        return self.rows * self.ts / wall, wall

    def what(self):
        return ("unmodified reference modelWind+computeF+computeG (oracle/_ref, g++ -O2, debug dumps to /dev/null)"
                if self.use_ref else "oracle/fg_oracle.c port (non-redundant restatement, gcc -O2)")

    def sample(self):
        return "rows [0, %d) of the %d-trajectory batch per step (sample_of: %d), %d processes x %d trajectories x %d windows; %s" % (
            self.rows, self.B_total, self.B_total, self.cores, self.per, self.ts, self.what())

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_single_core(fixture, seed0, seconds=4.0):
    """BASELINE.md section 4 (i) the callback as shipped (DEFINEGusrfg_ with its four dump files, here written into
    a scratch directory) and (ii) arithmetic only (modelWind+computeF+computeG, dumps to /dev/null), one core each"""
    import shutil
    import tempfile
    import refclient as R
    import tol_b200.synth as synth
    if not R.available():
        return None
    g = golden(fixture)
    ts = int(g["ts"])
    out = {}
    X = synth.batch(g["x"][0], seed0, 0, 64)
    cwd = os.getcwd()
    for key, null_io, full in (("arith_1core", True, False), ("as_shipped_1core", False, True)):
        tmp = tempfile.mkdtemp(prefix="tolref_cwd_")
        try:
            os.chdir(tmp)
            p = _make_problem(fixture, True, null_io=null_io)
            F, G = np.empty((1, p.neF)), np.empty((1, p.neG))
            p.eval_many(X[:1], F, G, full_callback=full)
            calls, t0 = 0, time.perf_counter()
            while time.perf_counter() - t0 < seconds and calls < X.shape[0] * 50:
                p.eval_many(X[calls % 64:calls % 64 + 1], F, G, full_callback=full)
                calls += 1
            dt = time.perf_counter() - t0
            out[key] = {"value": calls * ts / dt, "unit": UNIT, "cores": 1, "ms_per_call": 1e3 * dt / calls, "calls": calls,
                        "what": ("DEFINEGusrfg_ as shipped: Xoutput/Woutput/Foutput/Goutput.txt rewritten on every call "
                                 "(reference src/DefineFG.cpp:16-46)" if full else
                                 "modelWind+computeF+computeG, the dump files sent to /dev/null")}
            p.close()
        finally:
            os.chdir(cwd)
            R.lib().tolref_set_null_io(1)
            shutil.rmtree(tmp, ignore_errors=True)
    return out


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return None


def port_single_core(fixture, seed0, seconds=2.0):
    """for context (BASELINE.md section 4, item 4): the repo's own non-redundant CPU restatement, oracle/fg_oracle.c, one core"""
    import portclient as P
    import tol_b200.synth as synth
    if not P.available():
        return None
    g = golden(fixture)
    p = _make_problem(fixture, False)
    X = synth.batch(g["x"][0], seed0, 0, 64)
    F, G = np.empty((64, p.neF)), np.empty((64, p.neG))
    p.eval_many(X, F, G)
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        p.eval_many(X, F, G)
        n += 64
    dt = time.perf_counter() - t0
    return {"value": n * int(g["ts"]) / dt, "unit": UNIT, "cores": 1, "ms_per_call": 1e3 * dt / n,
            "what": "oracle/fg_oracle.c (plain-C restatement, every sub-expression once per node), not the baseline"}


def run_reference_arm(args, wl_name):
    fixture, seed0, B_total = WORKLOADS[wl_name]
    B_total = args.batch or B_total
    if int(os.environ.get("RANK", "0")) != 0:
        return
    arm = CpuArm(fixture, seed0, B_total)
    # size the step from a probe so that warm-up + K steps end within --cpu-budget seconds (all of the batch if it fits)
    arm.set_rows(arm.cores * 64)
    rate, _ = arm.step()
    nsteps = args.steps + max(1, min(args.warmup, 2))
    rows = int(rate / arm.ts * args.cpu_budget / nsteps)
    arm.set_rows(max(arm.cores * 32, min(B_total, rows)))
    for _ in range(max(1, min(args.warmup, 2))):
        arm.step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        arm.step()
    wall = time.perf_counter() - t0
    value = arm.rows * arm.ts * args.steps / wall
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": config_of(wl_name, B_total),
        "sample": {"sample_of": B_total, "rows_per_step": arm.rows, "what": arm.sample()},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.cores, "kind": arm.kind, "sample": arm.sample(),
                         "cpu_model": cpu_model()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    arm.close()
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------- GPU arm

class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append((time.perf_counter(), ln.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], 0, set()
        for t, ln in self.rows:
            if not (t0 <= t <= t1 + 0.2):
                continue
            f = [s.strip() for s in ln.split(",")]
            try:
                sm.append(float(f[0]))
                smax = max(smax, float(f[1]))
            except (ValueError, IndexError):
                continue
            for nm, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": smax or None, "reasons": sorted(reasons), "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy)"
        except (KeyError, ValueError):
            pass
    return 6650.0, "fallback (B200_PROFILING.md, 6.65 TB/s)"


def kernel_sass_hash(mission, wind, ts):
    """sha256 (16 hex digits) of the bench kernel's SASS in the library this run loaded: ties the stored ncu traffic
    ratio to a kernel binary.  None when cuobjdump is not at hand."""
    from tol_b200.sass import bench_kernel_pattern, kernel_sass_hash as h
    return h(bench_kernel_pattern(mission, wind, ts))


def ncu_traffic(wl_name, alg_bytes, sass_hash):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from an `ncu --set full`
    capture under profiles/ (never measured during a bench run), as a ratio to the algorithmic bytes of the captured
    launch.  The record carries the hash of the kernel's SASS at capture time; a different kernel binary voids it."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        t = json.load(open(p)).get(wl_name)
    except (OSError, ValueError):
        return None, "no record", None
    if not t:
        return None, "no record for this workload", None
    if sass_hash is None:
        return None, "cuobjdump unavailable: the record (kernel %s) cannot be tied to the loaded kernel" % t.get("kernel_sass_sha256_16"), None
    if t.get("kernel_sass_sha256_16") != sass_hash:
        return None, "stale: record was captured for kernel %s, this library's kernel is %s" % (t.get("kernel_sass_sha256_16"), sass_hash), None
    ncu = {k: t[k] for k in ("fp64_pipe_pct", "issue_active_pct", "dram_cycles_active_pct", "duration_under_ncu_ms", "captured_B") if k in t}
    if ncu:  # secondary bound: FP64 pipe utilisation of the same capture, and the DFMA peak measured with tools/exp/fp64peak.cu
        ncu["fp64_dfma_peak_tflops"] = {"measured": 33.9, "nominal": 37.2, "source": "tools/exp/fp64peak.cu, profiles/r1_history.md"}
    return t["ratio"] * alg_bytes, "profiles/roofline_traffic.json (%s; ratio to algorithmic bytes applied; kernel SASS %s)" % (t.get("source"), sass_hash), ncu


def host_ceiling(world, threads_total):
    """tools/exp/hostceil on this box, now (rank 0 only; the other ranks idle at a barrier)"""
    exe = os.path.join(ROOT, "tools", "exp", "hostceil")
    if not os.path.exists(exe):
        return None
    try:
        out = subprocess.run([exe, "--gpus", str(world), "--threads", str(threads_total), "--mb", "1024", "--reps", "2"],
                             capture_output=True, text=True, timeout=180)
        return json.loads(out.stdout.strip().splitlines()[-1])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        return None


def e2e_ceilings(hc, h2d, d2h_c, d2h_f, fill, staged, share):
    """Seconds per step the host side needs AT LEAST -- for the compact path, the full-row path and the mix that was
    timed (`share` of the rows as full rows) -- as the slowest of three resources (rates from tools/exp/hostceil in this
    run; bytes of the whole job per step):
      pcie_h2d    x over PCIe, all GPUs concurrently
      dma_ingest  what the GPUs' copy engines write into host memory (F + compact G, or F + G), all GPUs concurrently
      host_dram   the bytes the step cannot avoid moving through host DRAM -- read by DMA (x), written by DMA, and for
                  compact rows the rows stored by the expansion threads -- at the best TOTAL rate the tool saw on this
                  box (non-temporal fill, memcpy read+write, or DMA + fill together).  The read-back of the staging
                  blocks is left out: it can be served by the last-level cache (it is, on some boxes), so this is a
                  true lower bound of the time; host_dram_with_staging_reads adds it."""
    dram = max(hc["fill_nt_GBps"], hc["memcpy_rw_GBps"], hc["mix_d2h_GBps"] + hc["mix_fill_GBps"]) * 1e9
    out = {"dram_GBps": dram / 1e9,
           "model": "slowest of: x over PCIe; DMA ingest; unavoidable host-DRAM traffic (x read, DMA-written bytes, rows stored by "
                    "the threads; the staging read-back may hit the last-level cache and is listed separately) at the best total "
                    "rate the tool saw"}
    for name, p in (("compact_rows", 0.0), ("full_rows", 1.0), ("chosen", share)):
        d2h, stores, back = p * d2h_f + (1 - p) * d2h_c, (1 - p) * fill, (1 - p) * staged
        parts = {"pcie_h2d": h2d / (hc["h2d_GBps"] * 1e9), "dma_ingest": d2h / (hc["d2h_GBps"] * 1e9),
                 "host_dram": (h2d + d2h + stores) / dram}
        ms = {k: 1e3 * v for k, v in parts.items()}
        if back:
            ms["host_dram_with_staging_reads"] = 1e3 * (h2d + d2h + stores + back) / dram
        out[name] = {"seconds": max(parts.values()), "bound_by": max(parts, key=parts.get), "ms": ms}
    return out


def time_launches(torch, ev, stream, X, outs, steps, overlap):
    """K launches back to back on `stream`, CUDA events around them; returns ms"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(steps):
        F, G = outs[i % len(outs)]
        ev.eval_batch_device(X, F, G, sync=False, overlap=overlap)
    e1.record(stream)
    return e0, e1


def dump_outputs(directory, torch, dist, F, G, neF, neG, B_total, rank, world):
    """--dump-outputs: rows of F and G (this rank's device buffers, rows = its shard) for a seeded sample of the global
    trajectory indices, gathered on rank 0 and written as directory/F.npy and directory/G.npy"""
    import tol_b200.synth as synth
    k = min(B_total, DUMP_BYTES // (8 * (neF + neG)))
    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(B_total, k, replace=False))
    b0, b1 = synth.shard_range(B_total, rank, world)
    sel = np.flatnonzero((rows >= b0) & (rows < b1))
    dev = F.device
    src, dst = torch.from_numpy(rows[sel] - b0).to(dev), torch.from_numpy(sel).to(dev)
    out = torch.zeros(k, neF + neG, dtype=torch.float64, device=dev)
    out[dst, :neF] = F[src, :neF]
    out[dst, neF:] = G[src, :neG]
    if world > 1:  # every rank holds the sampled rows of its shard; take each row from its owner
        parts = [torch.empty_like(out) for _ in range(world)]
        dist.all_gather(parts, out)
        owner = torch.from_numpy(rows // -(-B_total // world)).to(dev)
        out = torch.stack(parts)[owner, torch.arange(k, device=dev)]
    if rank == 0:
        os.makedirs(directory, exist_ok=True)
        out = out.cpu().numpy()
        np.save(os.path.join(directory, "F.npy"), np.ascontiguousarray(out[:, :neF]))
        np.save(os.path.join(directory, "G.npy"), np.ascontiguousarray(out[:, neF:]))


def run_ours(args, wl_name):
    import torch
    import torch.distributed as dist
    import tol_b200 as T
    from tol_b200.evaluator import padded_ld

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; libtolcuda has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    fixture, seed0, Bdef = WORKLOADS[wl_name]
    B_total = args.batch or Bdef
    g = golden(fixture)
    ev = T.Evaluator.from_golden(g, device=local)
    ts, n, neF, neG = int(g["ts"]), ev.n, ev.neF, ev.neG
    ldx, ldF, ldG = padded_ld(n), padded_ld(neF), padded_ld(neG)
    b0, b1 = T.synth.shard_range(B_total, rank, world)
    B = b1 - b0  # this rank's rows: global trajectory indices [b0, b1)

    Xh = torch.zeros(B, ldx, dtype=torch.float64, pin_memory=True)
    T.synth.batch(g["x"][0], seed0, b0, b1, out=Xh.numpy())
    Xd = Xh.cuda()
    outs = [(torch.empty(B, ldF, dtype=torch.float64, device="cuda"), torch.empty(B, ldG, dtype=torch.float64, device="cuda"))
            for _ in range(2)]
    stream = torch.cuda.Stream()  # kernels and the timing events share this stream
    torch.cuda.set_stream(stream)
    ev.set_stream(stream.cuda_stream)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(vals):
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def gather_all(val):
        t = torch.tensor([val], dtype=torch.float64, device="cuda")
        if world > 1:
            parts = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(parts, t)
            return [float(p[0]) for p in parts]
        return [float(val)]

    # ---- device-resident, the headline `value`: K launches per rank, consecutive (independent) steps overlapped
    for i in range(args.warmup):
        ev.eval_batch_device(Xd, outs[i & 1][0], outs[i & 1][1], sync=False, overlap=2)
    barrier()
    sampler = ClockSampler(local)
    time.sleep(0.3)
    l0 = ev.launches
    tw0 = time.perf_counter()
    e0, e1 = time_launches(torch, ev, stream, Xd, outs, args.steps, 2)
    barrier()
    tw1 = time.perf_counter()
    ms_dev_local = e0.elapsed_time(e1)
    launches = ev.launches - l0
    clocks = sampler.stop(tw0, tw1)
    if args.dump_outputs:  # before the serial loop below rewrites result set 0
        F_, G_ = outs[(args.steps - 1) % len(outs)]
        dump_outputs(args.dump_outputs, torch, dist, F_, G_, neF, neG, B_total, rank, world)
    # the same loop with plain launches (each waits for the previous grid's last CTA): secondary
    ser_steps = max(3, min(args.steps, 20))
    e0, e1 = time_launches(torch, ev, stream, Xd, outs[:1], ser_steps, 0)
    barrier()
    ms_serial_local = e0.elapsed_time(e1) / ser_steps

    # ---- parity of what the timed launches left in HBM: EVERY rank checks rows of its own shard against the port
    import portclient as P
    if not P.available():
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "port"])
    port = P.PortProblem(str(g["mission"]), ts, g["ac"], g["gn"], g["goal_ned"], int(g["wind_model"]))
    rows = np.unique(np.linspace(0, B - 1, 12).astype(int))
    Xs = np.ascontiguousarray(Xh.numpy()[rows, :n])
    Fr, Gr = np.empty((rows.size, neF)), np.empty((rows.size, neG))
    port.eval_many(Xs, Fr, Gr)
    idx = torch.from_numpy(rows).cuda()
    ok = True
    for F_, G_ in outs:  # both result-buffer sets of the overlapped loop (set 0 was rewritten by the serial loop)
        ok = ok and close(F_[idx, :neF].cpu().numpy(), Fr) and close(G_[idx, :neG].cpu().numpy(), Gr)

    # ---- end to end: host (pinned) buffers through tolcuda_eval_batch, copies inside the timed region
    del outs
    torch.cuda.empty_cache()
    ev.use_own_stream()
    cores = len(os.sched_getaffinity(0))
    local_world = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
    host_threads = args.host_threads or max(1, min(16, cores // local_world))
    ev.set_host_threads(host_threads)
    Fh = torch.empty(B, ldF, dtype=torch.float64, pin_memory=True)
    Gh = torch.empty(B, ldG, dtype=torch.float64, pin_memory=True)
    e2e_steps = max(1, min(args.steps, args.e2e_steps))

    def e2e_run(steps, full_copy):
        for _ in range(2):
            ev.eval_batch_host(Xh.numpy(), Fh.numpy(), Gh.numpy(), full_copy=full_copy)
        barrier()
        l0_ = ev.launches
        t0_ = time.perf_counter()
        for _ in range(steps):
            ev.eval_batch_host(Xh.numpy(), Fh.numpy(), Gh.numpy(), full_copy=full_copy)
        torch.cuda.synchronize()
        t_ = time.perf_counter() - t0_
        barrier()
        return t_, ev.launches - l0_

    # Two ways for G to reach the caller's rows: compact rows across PCIe + expansion by host threads (the library's
    # default), or every G value across PCIe (option compact_host = 0 / TOLCUDA_FULL_G_COPY).  Which one is faster is a
    # property of the HOST (its DMA ingest rate against its cores' store rate, and how many GPUs share it), so the
    # caller calibrates: one untimed step of each with all ranks active, the decision all-reduced, then the timed
    # steps on the chosen path through the plain call.  The other path is reported next to it.
    def cal(full_copy):
        t_, _ = e2e_run(1, full_copy)
        ok_ = close(Fh.numpy()[rows, :neF], Fr) and close(Gh.numpy()[rows, :neG], Gr)
        return reduce_max([t_])[0], ok_
    cands = {}
    cands[0], ok_c = cal(False)     # all chunks as compact rows
    cands[100], ok_f = cal(True)    # all chunks as full rows
    ok = ok and ok_c and ok_f
    # mixed: the copy engines carry a share of the chunks as full rows while the cores expand the others; the share that
    # would equalise the two if they did not disturb each other, and half of it
    p_star = int(round(100.0 * cands[0] / (cands[0] + cands[100])))
    for pct in sorted({p_star, p_star // 2} - {0, 100}):
        ev.set_option("full_rows_pct", pct)
        cands[pct], ok_p = cal(False)
        ok = ok and ok_p
    best = min(cands, key=cands.get)
    if cands[best] > 0.97 * cands[0]:
        best = 0  # compact rows unless something else is clearly faster on this box
    ev.set_option("compact_host", 0 if best == 100 else 1)
    ev.set_option("full_rows_pct", 0 if best == 100 else best)
    t_e2e, e2e_launches = e2e_run(e2e_steps, False)  # the plain call: the context's options decide
    ok = ok and close(Fh.numpy()[rows, :neF], Fr) and close(Gh.numpy()[rows, :neG], Gr)
    ev.set_option("compact_host", 1)
    ev.set_option("full_rows_pct", 0)
    del Fh, Gh
    hc = None
    if rank == 0 and not args.no_ceiling:
        hc = host_ceiling(world, host_threads * world)
    barrier()

    ms_dev, ms_serial, t_e2e, bad = reduce_max([ms_dev_local, ms_serial_local, t_e2e, 0.0 if ok else 1.0])
    per_rank_ms = gather_all(ms_dev_local / args.steps)
    rows_checked = int(sum(gather_all(float(rows.size))))

    units_step = B_total * ts
    value = units_step * args.steps / (ms_dev * 1e-3)
    e2e_value = units_step * e2e_steps / t_e2e
    alg_bytes = 8.0 * (n + neF + neG) * B  # per launch (this rank; the shards differ by at most one row)
    launch_ms = ms_dev / args.steps
    peak, peak_src = measured_peak()
    achieved = alg_bytes / (launch_ms * 1e-3) / 1e9
    sass_hash = kernel_sass_hash(str(g["mission"]), int(g["wind_model"]), ts) if rank == 0 else None
    traffic, traffic_src, ncu_rec = ncu_traffic(wl_name, alg_bytes, sass_hash) if rank == 0 else (None, None, None)
    clen = padded_ld(ev.compact_len)
    h2d, fill = 8.0 * n * B_total, 8.0 * neG * B_total
    d2h_c, d2h_f = 8.0 * (neF + clen) * B_total, 8.0 * (neF + neG) * B_total
    share = best / 100.0
    what = ("every G value crosses PCIe, straight into the caller's rows" if best == 100 else
            "G crosses PCIe as compact rows (x-dependent values only) and host threads write the rows in coordinate order, "
            "structural constants as literals" + ("" if best == 0 else "; %d %% of the chunks cross as full rows instead, so "
                                                  "that copy engines and cores work side by side" % best))
    e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
           "d2h_bytes_per_step": int(share * d2h_f + (1.0 - share) * d2h_c),
           "steps": e2e_steps, "ms_per_step": 1e3 * t_e2e / e2e_steps, "gpu_launches": e2e_launches,
           "api": "tolcuda_eval_batch(TOLCUDA_HOST_PTRS), pinned host x/F/G; full F and G rows in host memory at the end of "
                  "every step; " + what,
           "path": {"full_rows_pct": best, "compact_rows_pct": 100 - best},
           "path_calibration": {"ms_per_step_by_full_rows_pct": {str(k): 1e3 * v for k, v in sorted(cands.items())},
                                "rule": "one untimed step per candidate with all ranks active (all compact, all full, the share "
                                        "t_c/(t_c+t_f) and half of it); the fastest, compact unless something is more than 3 % "
                                        "faster; then tolcuda_set_option(compact_host / full_rows_pct)"},
           "host_threads_per_rank": host_threads,
           "compact_rows_only": {"value": units_step / cands[0], "unit": UNIT, "ms_per_step": 1e3 * cands[0], "steps": 1},
           "full_rows_only": {"value": units_step / cands[100], "unit": UNIT, "ms_per_step": 1e3 * cands[100], "steps": 1,
                              "d2h_bytes_per_step": int(d2h_f)}}
    if hc:
        c = e2e_ceilings(hc, h2d, d2h_c, d2h_f, fill, 8.0 * clen * B_total, share)
        e2e["ceiling"] = units_step / c["chosen"]["seconds"]
        e2e["frac"] = e2e_value / e2e["ceiling"]
        e2e["ceiling_bound_by"] = c["chosen"]["bound_by"]
        e2e["ceiling_ms"] = c["chosen"]["ms"]
        e2e["compact_rows_only"]["ceiling"] = units_step / c["compact_rows"]["seconds"]
        e2e["full_rows_only"]["ceiling"] = units_step / c["full_rows"]["seconds"]
        e2e["ceiling_source"] = {"tool": "tools/exp/hostceil (this run, this box)", **hc, "host_dram_GBps_used": c["dram_GBps"],
                                 "model": c["model"]}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": launch_ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_of(wl_name, B_total),
        "run": {"trajectories_per_gpu": B, "per_rank_launch_ms": {"min": min(per_rank_ms), "max": max(per_rank_ms), "all": per_rank_ms},
                "launch_ms_serial": ms_serial, "value_serial": units_step / (ms_serial * 1e-3),
                "launches": "TOLCUDA_OVERLAP_DISJOINT: consecutive steps are independent batches writing two result-buffer "
                            "sets alternately; the next grid's CTAs start in the SMs the previous grid's tail has left",
                "parity_spot_check": bad == 0.0, "parity_rows_checked": rows_checked,
                "parity": "every rank: rows of its own shard in both device result sets and in the host rows of both e2e "
                          "paths, against the oracle port, |d| <= 1e-14 + 1e-12*|ref|; all-reduced over the ranks"},
        "e2e": e2e,
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "kernel": "fg_cta_kernel<%s, wind %d, PLAIN, runs of 2 trajectories per CTA + single-trajectory tail>" % (str(g["mission"]), int(g["wind_model"])),
                     "kernel_sass_sha256_16": sass_hash, "algorithmic_bytes_per_launch": alg_bytes, "launch_ms": launch_ms,
                     "frac_serial": alg_bytes / (ms_serial * 1e-3) / 1e9 / peak, "frac_of_nominal_8000_GBps": achieved / 8000.0,
                     "ncu": ncu_rec},
        "clocks": clocks,
    }

    # ---- N > 1: weak-scaling secondary and the device-side gather of the shards on GPU 0
    watchdog = None
    if world > 1:
        def bail():
            line["gather"] = {"error": "timed out after %d s" % args.gather_timeout}
            if rank == 0:
                print(json.dumps(line), flush=True)
            os._exit(0)
        watchdog = threading.Timer(args.gather_timeout, bail)
        watchdog.daemon = True
        watchdog.start()
        try:
            line["gather"] = gather_record(torch, dist, T, ev, g, Xd, B_total, rank, world, stream)
        except Exception as exc:  # the gather is a secondary record: never lose the line over it
            line["gather"] = {"error": "%s: %s" % (type(exc).__name__, exc)}
        try:
            line["run"]["weak"] = weak_record(torch, T, ev, g, seed0, rank, world, stream, Bdef, ts, reduce_max, barrier)
        except Exception as exc:
            line["run"]["weak"] = {"error": "%s: %s" % (type(exc).__name__, exc)}
        watchdog.cancel()
    del Xd
    ev.close()

    # ---- N = 1: the small configurations and the CPU baselines
    if world == 1:
        try:
            line["secondary"] = secondary_records(torch, T, stream, peak)
        except Exception as exc:
            line["secondary"] = {"error": "%s: %s" % (type(exc).__name__, exc)}
        if not args.no_cpu_baseline:
            torch.cuda.empty_cache()
            arm = CpuArm(fixture, seed0, B_total)
            arm.set_rows(arm.cores * args.cpu_sample)
            arm.step()
            v, wall = arm.step()
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": arm.cores, "kind": arm.kind,
                                    "sample": arm.sample(), "seconds": wall, "cpu_model": cpu_model()}
            arm.close()
            single = cpu_single_core(fixture, seed0)
            if single:
                line["cpu_baseline"].update(single)
            line["cpu_baseline"]["port_1core"] = port_single_core(fixture, seed0)
    if world > 1:
        dist.barrier()
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def gather_record(torch, dist, T, ev, g, Xd, B_total, rank, world, stream):
    """F and G rows of ALL shards on GPU 0: the fused evaluate+gather (every rank's kernel stores its rows straight
    into GPU 0's buffer over NVLink peer memory; G as compact rows, expanded by the owner chunk by chunk as the
    flags arrive) against evaluate -> NCCL gather of compact rows -> expansion.  Timed on the device-side clock of
    the gathering rank's host (perf_counter around synchronised calls, max over ranks); bit-identity of the two
    results is checked on the full arrays."""
    import tol_b200.dist as D
    torch.cuda.set_stream(torch.cuda.default_stream())
    ev.follow_torch_stream()  # the gathers allocate and fill through torch: one stream orders everything
    reps = 5
    buf = D.open_peer_buffer(ev, B_total, 0, True)
    out = {}
    res = {}
    for name, fn in (("fused_peer", lambda: D.eval_and_gather_peer(ev, Xd, B_total, dst=0, out=buf, compact=True, chunks=4)[:2]),
                     ("nccl", lambda: D.eval_and_gather_device(ev, Xd, B_total, dst=0))):
        best = 1e30
        for r in range(reps + 1):
            torch.cuda.synchronize()
            dist.barrier()
            t0 = time.perf_counter()
            F, G = fn()
            torch.cuda.synchronize()
            dist.barrier()
            dt = time.perf_counter() - t0
            if r > 0:
                best = min(best, dt)
        t = torch.tensor([best], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out[name + "_ms"] = 1e3 * float(t[0])
        if rank == 0:
            res[name] = (F[:, :ev.neF].clone() if name == "fused_peer" else F, G[:, :ev.neG] if name == "fused_peer" else G)
    if rank == 0:
        Ff, Gf = res["fused_peer"]
        Fn, Gn = res["nccl"]
        same = bool(torch.equal(Ff.view(torch.int64), Fn.contiguous().view(torch.int64)))
        # G in slabs: a whole-array comparison would need another 11 GB
        for a in range(0, B_total, 4096):
            same = same and bool(torch.equal(Gf[a:a + 4096].contiguous().view(torch.int64), Gn[a:a + 4096].contiguous().view(torch.int64)))
        out["bit_identical"] = same
        out["rows"] = B_total
        out["bytes_on_gpu0"] = int(8 * B_total * (ev.neF + ev.neG))
        out["what"] = ("all %d rows of F and G on GPU 0; fused_peer = tol_b200.dist.eval_and_gather_peer (4 chunks per "
                       "peer), nccl = eval_and_gather_device; best of %d, barrier to barrier, max over ranks" % (B_total, reps))
    del res
    dist.barrier()
    buf.close()
    ev.set_stream(stream.cuda_stream)
    torch.cuda.set_stream(stream)
    return out


def weak_record(torch, T, ev, g, seed0, rank, world, stream, Bw, ts, reduce_max, barrier):
    """round 1's protocol: every rank evaluates its OWN Bw trajectories (the full batch size per GPU)"""
    from tol_b200.evaluator import padded_ld
    ldx, ldF, ldG = padded_ld(ev.n), padded_ld(ev.neF), padded_ld(ev.neG)
    U = 2048  # distinct rows, tiled (timing only)
    Xu = torch.zeros(U, ldx, dtype=torch.float64)
    T.synth.batch(g["x"][0], seed0, rank * Bw, rank * Bw + U, out=Xu.numpy())
    X = Xu.cuda()[torch.arange(Bw, device="cuda") % U].contiguous()
    outs = [(torch.empty(Bw, ldF, dtype=torch.float64, device="cuda"), torch.empty(Bw, ldG, dtype=torch.float64, device="cuda"))
            for _ in range(2)]
    steps = 10
    for i in range(3):
        ev.eval_batch_device(X, outs[i & 1][0], outs[i & 1][1], sync=False, overlap=2)
    barrier()
    e0, e1 = time_launches(torch, ev, stream, X, outs, steps, 2)
    barrier()
    ms = reduce_max([e0.elapsed_time(e1)])[0]
    return {"scaling": "weak", "trajectories_per_gpu": Bw, "steps": steps, "ms_per_step": ms / steps,
            "value": world * Bw * ts * steps / (ms * 1e-3), "unit": UNIT}


def secondary_records(torch, T, stream, peak):
    """BASELINE.json configs[2] (G7, 4,096 x 100, one B200) and the drop-in use itself: the single-trajectory snOptA
    callback's latency"""
    from tol_b200.evaluator import padded_ld
    import ctypes as C
    sec = {}
    fixture, seed0, B = WORKLOADS["G7_skywalker_ts100_B4096"]
    g = golden(fixture)
    ev = T.Evaluator.from_golden(g)
    ev.set_stream(stream.cuda_stream)
    ts = int(g["ts"])
    ldx, ldF, ldG = padded_ld(ev.n), padded_ld(ev.neF), padded_ld(ev.neG)
    Xh = torch.zeros(B, ldx, dtype=torch.float64)
    T.synth.batch(g["x"][0], seed0, 0, B, out=Xh.numpy())
    X = Xh.cuda()
    outs = [(torch.empty(B, ldF, dtype=torch.float64, device="cuda"), torch.empty(B, ldG, dtype=torch.float64, device="cuda"))
            for _ in range(2)]
    by = 8.0 * (ev.n + ev.neF + ev.neG) * B
    rec = {"workload": "G7_skywalker_ts100_B4096", "trajectories": B, "ts": ts, "algorithmic_bytes_per_launch": by,
           "l2": "two result sets of 0.4 GB written alternately: 0.8 GB between two uses of a line, > 126 MB L2"}
    for key, ov, sets in (("overlapped", 2, outs), ("serial", 0, outs)):
        for i in range(20):
            ev.eval_batch_device(X, sets[i & 1][0], sets[i & 1][1], sync=False, overlap=ov)
        torch.cuda.synchronize()
        steps = 400
        e0, e1 = time_launches(torch, ev, stream, X, sets, steps, ov)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        rec[key] = {"launch_us": 1e3 * ms, "value": B * ts / (ms * 1e-3), "unit": UNIT, "GBps": by / ms / 1e6,
                    "frac": by / ms / 1e6 / peak, "steps": steps}
    import portclient as P
    port = P.PortProblem(str(g["mission"]), ts, g["ac"], g["gn"], g["goal_ned"], int(g["wind_model"]))
    rows = np.linspace(0, B - 1, 8).astype(int)
    Fr, Gr = np.empty((8, ev.neF)), np.empty((8, ev.neG))
    port.eval_many(np.ascontiguousarray(Xh.numpy()[rows, :ev.n]), Fr, Gr)
    idx = torch.from_numpy(rows).cuda()
    rec["parity_spot_check"] = all(close(F_[idx, :ev.neF].cpu().numpy(), Fr) and close(G_[idx, :ev.neG].cpu().numpy(), Gr)
                                   for F_, G_ in outs)
    sec["config3"] = rec
    ev.close()
    del X, outs

    # F alone (needG = 0: SNOPT's line-search evaluations) and the summary alone (screening) on the bench's own batch:
    # the 64-register flavours of the kernel (MODE_FONLY / MODE_FSUMM)
    fixture, seed0, B = WORKLOADS["S10_tempest_ts200_B65536"]
    g = golden(fixture)
    ev = T.Evaluator.from_golden(g)
    ev.set_stream(stream.cuda_stream)
    ts = int(g["ts"])
    ldx, ldF = padded_ld(ev.n), padded_ld(ev.neF)
    U = 2048  # distinct rows, tiled (timing only; F of the first rows is checked against the oracle port)
    Xu = torch.zeros(U, ldx, dtype=torch.float64)
    T.synth.batch(g["x"][0], seed0, 0, U, out=Xu.numpy())
    X = Xu.cuda()[torch.arange(B, device="cuda") % U].contiguous()
    Fd = torch.empty(B, ldF, dtype=torch.float64, device="cuda")
    Sd = torch.empty(B, 4, dtype=torch.float64, device="cuda")
    Gnone = torch.empty(0, 1, dtype=torch.float64, device="cuda")
    fl = T.evaluator.DEVICE_PTRS | T.evaluator.NO_SYNC

    def f_only():
        ev.eval_batch_device(X, Fd, Gnone, needF=True, needG=False, sync=False)

    def s_only():
        T.lib.check(ev.L.tolcuda_eval_batch_summary(ev.h, B, X.data_ptr(), X.stride(0), None, 0, None, 0, Sd.data_ptr(), 4, fl))
    for key, fn, by in (("f_only", f_only, 8.0 * (ev.n + ev.neF) * B), ("summary_only", s_only, 8.0 * (ev.n + 4) * B)):
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
        steps = 100
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        sec[key] = {"workload": "S10_tempest_ts200_B65536", "launch_ms": ms, "value": B * ts / (ms * 1e-3), "unit": UNIT,
                    "bytes_per_launch": by, "GBps": by / ms / 1e6, "frac_of_own_bytes": by / ms / 1e6 / peak, "steps": steps}
    port = P.PortProblem(str(g["mission"]), ts, g["ac"], g["gn"], g["goal_ned"], int(g["wind_model"]))
    Fr, Gr = np.empty((8, ev.neF)), np.empty((8, ev.neG))
    port.eval_many(np.ascontiguousarray(Xu.numpy()[:8, :ev.n]), Fr, Gr)
    Sh = Sd[:8].cpu().numpy()
    sec["f_only"]["parity_spot_check"] = close(Fd[:8, :ev.neF].cpu().numpy(), Fr)
    sec["summary_only"]["parity_spot_check"] = bool(close(Sh[:, 0], Fr[:, 0]) and
                                                    close(Sh[:, 1], np.abs(Fr[:, 1:1 + 8 * ts]).max(axis=1)))
    ev.close()
    del X, Fd, Sd

    # DEFINEGusrfg_ exactly as SNOPT calls it, on the reference's own initial guess; timed from Python through ctypes
    # with pre-built argument objects (about a microsecond of marshalling per call is included)
    cb = {}
    for fx in ("S10_tempest_ts100", "S10_tempest_ts200"):
        g = golden(fx)
        ev = T.Evaluator.from_golden(g)
        L = ev.L
        L.tolcuda_bind_global(ev.h)
        x = np.ascontiguousarray(g["x"][0])
        F, G = np.empty(ev.neF), np.empty(ev.neG)
        dp = C.POINTER(C.c_double)
        xs, Fs, Gs = x.ctypes.data_as(dp), F.ctypes.data_as(dp), G.ctypes.data_as(dp)
        st, n_, neF_, neG_, z = C.c_int(0), C.c_int(ev.n), C.c_int(ev.neF), C.c_int(ev.neG), C.c_int(0)
        for label, nf, ng in (("FG", 1, 1), ("F", 1, 0)):
            nF, nG = C.c_int(nf), C.c_int(ng)
            a = (C.byref(st), C.byref(n_), xs, C.byref(nF), C.byref(neF_), Fs, C.byref(nG), C.byref(neG_), Gs, None,
                 C.byref(z), None, C.byref(z), None, C.byref(z))
            fn = L.DEFINEGusrfg_
            for _ in range(300):
                fn(*a)
            reps = 3000
            t0 = time.perf_counter()
            for _ in range(reps):
                fn(*a)
            cb["ts%d_%s" % (int(g["ts"]), label)] = 1e6 * (time.perf_counter() - t0) / reps
        assert st.value == 0
        Fr, Gr = port_eval(g, x)
        cb["ts%d_parity" % int(g["ts"])] = close(F, g["F"][0]) and close(G, Gr)
        L.tolcuda_bind_global(None)
        ev.close()
    cb["what"] = "microseconds per DEFINEGusrfg_ call (snOptA argument list, host x/F/G), S10 tempest, reference x0"
    sec["callback_us"] = cb
    return sec


def port_eval(g, x):
    import portclient as P
    port = P.PortProblem(str(g["mission"]), int(g["ts"]), g["ac"], g["gn"], g["goal_ned"], int(g["wind_model"]))
    return port.eval(x)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="S10_tempest_ts200_B65536", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="override the trajectories of the whole batch (experiments)")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--host-threads", type=int, default=0, help="expansion threads per rank on the e2e path (0: cores / ranks, at most 16)")
    ap.add_argument("--cpu-sample", type=int, default=1000, help="ours arm: trajectories per CPU process for cpu_baseline")
    ap.add_argument("--cpu-budget", type=float, default=150.0, help="reference arm: seconds for warm-up + K steps")
    ap.add_argument("--gather-timeout", type=int, default=240)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ceiling", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write F and G of a seeded sample of the last timed step's rows as DIR/F.npy, DIR/G.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours: the reference arm keeps no output rows")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args, args.workload)
    else:
        run_ours(args, args.workload)


if __name__ == "__main__":
    main()
