#!/usr/bin/env python
"""Six coverage/identity threshold sets: one imsame_gpu_align_sweep against six imsame_gpu_align calls, on one GPU.

Workloads (seeded synthetic reads, identities 0.70 .. 0.95 in steps of 0.05 at coverage 0.5):
  cfg5   BASELINE.json configs[4] at cfg1 sizes: 10 k x 150-base query reads (divergence 0.15) vs 100 k database reads
  cfg2   a user-sized run: 1 M x 250-base query reads (divergence 0.10) vs 10 M database reads
The two arms alternate inside one invocation after a warm-up of each, --reps times.  Wall time is a host clock around
the synchronous calls; ms_k2, ms_k3 and n_pairs_dp come from the stats (the separate arm: summed over its six calls).
Every repetition checks that each set's records of the sweep equal those of its separate call.  The card's name and
power limit are printed first.  usage: python tools/sweep_bench.py [--reps 3] [--workloads cfg5,cfg2]"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from imsame_b200 import api, hostlib as H  # noqa: E402

IDENTITIES = (0.70, 0.75, 0.80, 0.85, 0.90, 0.95)
WORKLOADS = {  # name: (pool seed, genomes, genome length, read length, database reads, query reads, divergence)
    "cfg5": (5005, 20, 500_000, 150, 100_000, 10_000, 0.15),
    "cfg2": (2001, 1000, 1_000_000, 250, 10_000_000, 1_000_000, 0.10),
}
FIELDS = ("accepted", "db_seq", "qpos_end", "db_pos", "length", "identities")


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else "nvidia-smi unavailable"


def log(*a):
    print(*a, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--workloads", default="cfg5,cfg2")
    a = ap.parse_args()
    ctx = api.Imsame(0)  # raises without an sm_100 device: this tool never runs on the CPU
    log(f"card: {card()}")
    ps = [api.make_params(n_threads=4, min_coverage=0.5, min_identity=i) for i in IDENTITIES]
    for name in a.workloads.split(","):
        seed, g, glen, L, nd, nq, div = WORKLOADS[name]
        pool = H.SynthPool(seed, g, glen)
        db, q = pool.db_reads(0, nd, L), pool.query_reads(0, nq, L, div)
        pool.close()
        ds, qs = np.arange(nd + 1, dtype=np.uint64) * L, np.arange(nq + 1, dtype=np.uint64) * L
        log(f"\n== {name}: {nq} x {L}-base query reads (divergence {div}) vs {nd} database reads, coverage 0.5, "
            f"identities {', '.join(f'{i:.2f}' for i in IDENTITIES)}")
        ctx.align_sweep((db, ds), (q, qs), ps)  # warm-up of both arms: allocations, pinned buffers, module load
        ctx.align((db, ds), (q, qs), ps[0])
        wall = {"sweep": [], "separate": []}
        for rep in range(a.reps):
            for arm in ("sweep", "separate"):
                t0 = time.perf_counter()
                if arm == "sweep":
                    outs, codes, st = ctx.align_sweep((db, ds), (q, qs), ps)
                    assert codes == [0] * len(ps)
                    k2, k3, dp = st["ms_k2"], st["ms_k3"], st["n_pairs_dp"]
                else:
                    sep = [ctx.align((db, ds), (q, qs), p) for p in ps]
                    k2, k3 = sum(s["ms_k2"] for _, s in sep), sum(s["ms_k3"] for _, s in sep)
                    dp = sum(s["n_pairs_dp"] for _, s in sep)
                wall[arm].append(time.perf_counter() - t0)
                log(f"  rep {rep} {arm:8s} wall {1e3 * wall[arm][-1]:9.1f} ms  ms_k2 {k2:8.1f}  ms_k3 {k3:8.1f}  "
                    f"n_pairs_dp {dp}")
            for t in range(len(ps)):
                assert all(np.array_equal(outs[t][f], sep[t][0][f]) for f in FIELDS), (name, t)
            acc = [int(o["accepted"].sum()) for o in outs]
            log(f"  rep {rep}: records of every set equal the separate calls' (accepted per set: {acc})")
        med = {k: float(np.median(v)) for k, v in wall.items()}
        log(f"  median wall over {a.reps}: one sweep {1e3 * med['sweep']:.1f} ms, six separate calls "
            f"{1e3 * med['separate']:.1f} ms ({med['separate'] / med['sweep']:.2f}x)")
    ctx.close()


if __name__ == "__main__":
    main()
