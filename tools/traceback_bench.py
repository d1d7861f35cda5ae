#!/usr/bin/env python
"""What the alignment of the accepted hits adds (imsame_gpu_align_traceback, IMSAME -cigar), on one GPU.

Workload: 250-base reads, a database of --nd reads drawn from a synthetic pool, --nq query reads of which a fraction
(the acceptance rates of --rates) are noisy copies from that pool (divergence 0.05) and the rest random reads, which
the database does not hold.  Per rate: the alignment (imsame_gpu_align), then the CIGAR traceback of its records,
--reps times after a warm-up of both; wall time is a host clock around the synchronous calls.  Printed per rate: the
accepted records, median align ms, median traceback ms, traceback microseconds per accepted hit, and the traceback's
share of align + traceback.  The winners' text traceback (imsame_gpu_traceback, which the .align records need
anyway) is timed beside it for comparison.  The card's name and power limit are printed first.
usage: python tools/traceback_bench.py [--reps 5] [--nd 1000000] [--nq 100000] [--rates 0.1,0.5,0.9]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from imsame_b200 import api, hostlib as H  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else "nvidia-smi unavailable"


def timed(f):
    t = time.perf_counter()
    r = f()
    return r, 1e3 * (time.perf_counter() - t)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--nd", type=int, default=1_000_000)
    ap.add_argument("--nq", type=int, default=100_000)
    ap.add_argument("--rates", default="0.1,0.5,0.9")
    a = ap.parse_args()
    print("card:", card(), flush=True)
    L = 250
    pool = H.SynthPool(2001, 100, 1_000_000)
    db = pool.db_reads(0, a.nd, L)
    present = pool.query_reads(0, a.nq, L, 0.05)
    pool.close()
    ds = np.arange(a.nd + 1, dtype=np.uint64) * L
    qs = np.arange(a.nq + 1, dtype=np.uint64) * L
    rng = np.random.default_rng(7)
    absent = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=a.nq * L)]
    ctx = api.Imsame(0)
    p = api.make_params()
    for rate in (float(v) for v in a.rates.split(",")):
        take = rng.random(a.nq) < rate
        q = np.where(np.repeat(take, L), present, absent).astype(np.uint8)
        out, _ = ctx.align((db, ds), (q, qs), p)  # warm-up of every shape
        ctx.align_traceback((db, ds), (q, qs), out, p)
        ctx.traceback((db, ds), (q, qs), out, p)
        t_al, t_cg, t_tb = [], [], []
        for _ in range(a.reps):
            out2, ms = timed(lambda: ctx.align((db, ds), (q, qs), p)[0])
            t_al.append(ms)
            assert np.array_equal(out, out2)
            _, ms = timed(lambda: ctx.align_traceback((db, ds), (q, qs), out, p))
            t_cg.append(ms)
            _, ms = timed(lambda: ctx.traceback((db, ds), (q, qs), out, p))
            t_tb.append(ms)
        acc = int(out["accepted"].sum())
        al, cg, tb = (float(np.median(t)) for t in (t_al, t_cg, t_tb))
        print(json.dumps({"query_fraction_present": rate, "nd": a.nd, "nq": a.nq, "accepted": acc,
                          "align_ms": round(al, 2), "cigar_traceback_ms": round(cg, 2),
                          "us_per_accepted_hit": round(1e3 * cg / max(acc, 1), 3),
                          "share_of_align_plus_cigar": round(cg / (al + cg), 4),
                          "text_traceback_ms": round(tb, 2), "reps": a.reps}), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
