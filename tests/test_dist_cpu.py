"""CPU, world_size 2, gloo: the host-side logic of the multi-GPU path -- shard ranges by trajectory index,
per-index input seeding, host-side gather of per-trajectory rows, max-over-ranks timing.  The evaluator
here is the oracle port (tests may use it); on GPUs the same code wraps tolcuda_eval_batch (bench.py)."""
import os
import socket

import numpy as np
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import load_golden, port_from_golden


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, B, out_path):
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for p in (root, os.path.join(root, "oracle"), os.path.join(root, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import tol_b200.dist as D
    import tol_b200.synth as synth
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    g = load_golden("S10_skywalker_ts7_gains")
    p = port_from_golden(g)
    b0, b1 = D.my_shard(B)
    X = synth.batch(g["x"][0], 4242, b0, b1)
    F, G = np.empty((b1 - b0, p.neF)), np.empty((b1 - b0, p.neG))
    if b1 > b0:
        p.eval_many(X, F, G)
    fullF = D.gather_rows(F, B)
    fullG = D.gather_rows(G, B)
    tmax = D.max_over_ranks(1.0 + rank)
    if rank == 0:
        np.savez(out_path, F=fullF, G=fullG, tmax=tmax)
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_shard_and_gather_equals_single_process(tmp_path, oracle_built):
    B = 13  # odd on purpose: ranks own 7 and 6 trajectories
    out = str(tmp_path / "gathered.npz")
    mp.spawn(_worker, args=(2, _free_port(), B, out), nprocs=2, join=True)
    got = np.load(out)
    import tol_b200.synth as synth
    g = load_golden("S10_skywalker_ts7_gains")
    p = port_from_golden(g)
    X = synth.batch(g["x"][0], 4242, 0, B)
    F, G = np.empty((B, p.neF)), np.empty((B, p.neG))
    p.eval_many(X, F, G)
    assert np.array_equal(got["F"], F) and np.array_equal(got["G"], G)
    assert float(got["tmax"]) == 2.0


def test_shard_ranges_cover_the_batch_exactly():
    import tol_b200.synth as synth
    for B in (1, 2, 7, 64, 65536, 65537):
        for w in (1, 2, 4, 8):
            r = [synth.shard_range(B, q, w) for q in range(w)]
            assert r[0][0] == 0 and r[-1][1] == B
            assert all(r[i][1] == r[i + 1][0] for i in range(w - 1))
            assert all(b1 >= b0 for b0, b1 in r)


def test_bench_reference_arm_prints_the_same_config_as_the_gpu_arm(oracle_built):
    """bench.py --impl reference (CPU only: the reference's own path on the host cores, a bounded sample of the same
    batch) prints the line of the contract -- same metric, unit and CONFIG as the GPU arm, impl = reference, a
    cpu_baseline describing the run, e2e with zero copies -- and, launched as ranks 0 and 1, only rank 0 works."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1",
           "--cpu-budget", "4", "--batch", "2048"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, RANK="0", WORLD_SIZE="2"))
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == bench.METRIC and line["unit"] == bench.UNIT
    assert line["config"] == bench.config_of("S10_tempest_ts200_B65536", 2048)  # what run_ours prints as `config`
    assert line["higher_is_better"] is True and line["scaling"] == "strong" and line["n_gpus"] == 2 and line["dtype"] == "f64"
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"] > 0
    assert line["sample"]["sample_of"] == 2048 and 0 < line["sample"]["rows_per_step"] <= 2048
    assert line["e2e"] == {"value": line["value"], "unit": bench.UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=60, env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_bench_dump_outputs_writes_a_fixed_sample_of_the_rows(tmp_path):
    """bench.py --dump-outputs: the same seeded rows of F and G on every run, each row the caller's row of that
    trajectory (padding left out), float64, the two files within 64 MB together; all rows when the batch fits"""
    import sys
    import torch
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    neF, neG = 1612, 21437  # S10 ts = 200, the bench workload
    for B in (400, 5):  # 347 rows of 400 fit the budget
        F = torch.arange(B, dtype=torch.float64)[:, None] * 1e5 + torch.arange(neF + 3, dtype=torch.float64)
        G = -torch.arange(B, dtype=torch.float64)[:, None] * 1e5 - torch.arange(neG + 5, dtype=torch.float64)
        got = []
        for run in range(2):
            d = tmp_path / ("B%d_%d" % (B, run))
            bench.dump_outputs(str(d), torch, None, F, G, neF, neG, B, 0, 1)
            Fd, Gd = np.load(d / "F.npy"), np.load(d / "G.npy")
            assert Fd.dtype == Gd.dtype == np.float64 and Fd.shape[1] == neF and Gd.shape[1] == neG
            assert (d / "F.npy").stat().st_size + (d / "G.npy").stat().st_size <= 64 * 10**6
            rows = (Fd[:, 0] / 1e5).astype(np.int64)
            assert np.array_equal(Fd, F.numpy()[rows, :neF]) and np.array_equal(Gd, G.numpy()[rows, :neG])
            got.append(rows)
        assert np.array_equal(got[0], got[1]) and (np.diff(got[0]) > 0).all()
        assert got[0].size == min(B, 347)


def test_bench_dump_outputs_takes_each_row_from_the_rank_that_owns_it(tmp_path):
    """bench.py --dump-outputs with the batch sharded over 3 ranks: each rank contributes the sampled rows of its own
    shard, and rank 0 writes the same files one rank holding the whole batch writes"""
    import sys
    import torch
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    import tol_b200.synth as synth
    neF, neG, B, world = 1612, 21437, 1003, 3
    F = torch.arange(B, dtype=torch.float64)[:, None] * 1e5 + torch.arange(neF, dtype=torch.float64)
    G = -torch.arange(B, dtype=torch.float64)[:, None] * 1e5 - torch.arange(neG, dtype=torch.float64)
    bench.dump_outputs(str(tmp_path / "one"), torch, None, F, G, neF, neG, B, 0, 1)
    sent = {}

    class Dist:  # all_gather of a stand-in process group: every rank's tensor, collected as the ranks call in
        def __init__(self, rank):
            self.rank = rank

        def all_gather(self, parts, t):
            sent[self.rank] = t.clone()
            if len(sent) == world:
                for q in range(world):
                    parts[q].copy_(sent[q])
    for rank in (2, 1, 0):  # rank 0, which writes, comes last so that its all_gather sees every shard
        b0, b1 = synth.shard_range(B, rank, world)
        bench.dump_outputs(str(tmp_path / "three"), torch, Dist(rank), F[b0:b1], G[b0:b1], neF, neG, B, rank, world)
    for name in ("F.npy", "G.npy"):
        assert np.array_equal(np.load(tmp_path / "three" / name), np.load(tmp_path / "one" / name))


def test_bench_ceiling_is_the_slowest_resource():
    """bench.py's e2e lower bound (host side of the box): per path the slowest of PCIe in, DMA ingest and unavoidable
    host-DRAM traffic; the staging read-back only in the separate figure; full rows have no thread stores; a mix lies
    between the two paths in DMA bytes"""
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    B, n, neF, neG, clen = 65536, 2212, 1612, 21437, 6848
    h2d, d2h_c, d2h_f, fill, staged = 8.0 * n * B, 8.0 * (neF + clen) * B, 8.0 * (neF + neG) * B, 8.0 * neG * B, 8.0 * clen * B
    hc = {"d2h_GBps": 90.0, "h2d_GBps": 186.0, "fill_nt_GBps": 200.0, "memcpy_rw_GBps": 185.0, "mix_d2h_GBps": 52.0, "mix_fill_GBps": 52.0}
    c = bench.e2e_ceilings(hc, h2d, d2h_c, d2h_f, fill, staged, 0.25)
    assert c["dram_GBps"] == 200.0
    cr, fr, mx = c["compact_rows"], c["full_rows"], c["chosen"]
    assert cr["bound_by"] == "host_dram" and abs(cr["seconds"] - (h2d + d2h_c + fill) / 200e9) < 1e-12
    assert abs(cr["ms"]["host_dram_with_staging_reads"] - 1e3 * (h2d + d2h_c + fill + staged) / 200e9) < 1e-9
    assert fr["bound_by"] == "dma_ingest" and abs(fr["seconds"] - d2h_f / 90e9) < 1e-12 and "host_dram_with_staging_reads" not in fr["ms"]
    assert cr["ms"]["dma_ingest"] < mx["ms"]["dma_ingest"] < fr["ms"]["dma_ingest"]
    assert fr["ms"]["host_dram"] < mx["ms"]["host_dram"] < cr["ms"]["host_dram"]
    # a host whose copy engines ingest faster than its cores store: full rows become the better bound
    hc2 = dict(hc, d2h_GBps=175.0)
    c2 = bench.e2e_ceilings(hc2, h2d, d2h_c, d2h_f, fill, staged, 0.0)
    assert c2["full_rows"]["seconds"] < c2["compact_rows"]["seconds"]
    assert bench.config_of("S10_tempest_ts200_B65536", 65536)["neG"] == neG
