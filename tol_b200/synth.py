"""Synthetic batched decision vectors, SURVEY.md section 8d: trajectory b is
x0[i]*(1+0.05*u) + 0.01*u' with (u, u') drawn interleaved per i from
numpy.random.Generator(PCG64(seed0 + b)).uniform(-1, 1, 2n).  The seed is the GLOBAL trajectory
index, so a shard [b0, b1) of a batch is the same on any number of GPUs."""
import numpy as np

SEED_G7 = 20260000
SEED_S10 = 20270000


def perturb(x0, seed):
    r = np.random.Generator(np.random.PCG64(seed)).uniform(-1.0, 1.0, size=2 * x0.size)
    return x0 * (1.0 + 0.05 * r[0::2]) + 0.01 * r[1::2]


def batch(x0, seed0, b0, b1, out=None, ld=None):
    """rows b0..b1-1 of the synthetic batch, into `out` [b1-b0, ld] (allocated if None)"""
    n = x0.size
    if out is None:
        out = np.zeros((b1 - b0, ld or n))
    for b in range(b0, b1):
        out[b - b0, :n] = perturb(x0, seed0 + b)
    return out


SEED_GOALS = 20280000


def goals(mission, lo, hi, seed=SEED_GOALS):
    """goals (xg, yg, zg, rg in NED) of trajectories lo..hi-1 of a batch with per-trajectory goals, [hi-lo, 4].  Row b
    comes from numpy.random.Generator(PCG64(seed + b)) alone, so any sharding of the batch gives the same table.
    The goal lies 300..3000 m from the origin (where the reference puts the aircraft's initial position) at 50..150 m
    altitude, S10 loiter radii 50..400 m.  G7 (whose boundary rows depend on chi_d = atan2(yg, xg)): the even rows sit
    within 1e-9 rad of the +x, +y, -x, -y axis in turn (b mod 8 = 0, 2, 4, 6; the -x axis on both sides of the branch
    cut of atan2), the odd rows at uniform bearings, so the table covers all four quadrants of chi_d and each axis."""
    out = np.empty((hi - lo, 4))
    for b in range(lo, hi):
        r = np.random.Generator(np.random.PCG64(seed + b)).uniform(0.0, 1.0, size=5)
        chi = -np.pi + 2.0 * np.pi * r[0]
        if mission in ("G7", 7) and b % 2 == 0:
            chi = (b % 8) // 2 * (np.pi / 2) + (r[0] - 0.5) * 2e-9
        dist = 300.0 + 2700.0 * r[1]
        out[b - lo] = (dist * np.cos(chi), dist * np.sin(chi), -(50.0 + 100.0 * r[2]), 50.0 + 350.0 * r[3])
    return out


def shard_range(B, rank, world):
    """contiguous block of trajectory indices owned by `rank` (SURVEY.md section 8e)"""
    per = (B + world - 1) // world
    b0 = min(B, rank * per)
    return b0, min(B, b0 + per)
