#!/usr/bin/env python
"""Five seed lengths: one imsame_gpu_align_kmers against five set_kmer + imsame_gpu_align calls, and one
`IMSAME -kmers 8,10,14,16` process against five `IMSAME -kmer k` processes, on one GPU.

Workload: BASELINE.json configs[4] (the low-identity sweep) at cfg1 sizes, seeded synthetic reads: 10 k x 150-base
query reads against 100 k database reads, query divergence 0.10 and 0.25, seed lengths 8, 10, 12, 14, 16 (k = 16 builds
a 34 GB word table).  The library arms alternate inside one invocation after a warm-up of each, --reps times; wall time
is a host clock around the synchronous calls.  Per entry: K3 ms, candidate pairs (n_pairs) and pairs run through NW
(n_pairs_dp) of both arms; their ratio is the share of NW work the pair-result cache leaves.  Every repetition checks
that each entry's records equal its separate call's; the command-line arm checks that every <out>.k<K> file equals the
separate process's -out file.  The card's name and power limit are printed first.
usage: python tools/kmers_bench.py [--reps 3] [--divergence 0.10,0.25] [--no-cli]"""
import argparse
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from imsame_b200 import api, hostlib as H  # noqa: E402

KS = (8, 10, 12, 14, 16)
SIZES = (5005, 20, 500_000, 150, 100_000, 10_000)  # pool seed, genomes, genome length, read length, db reads, queries
FIELDS = ("accepted", "db_seq", "qpos_end", "db_pos", "length", "identities")
EXE = os.path.join(ROOT, "bin", "IMSAME")


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else "nvidia-smi unavailable"


def log(*a):
    print(*a, flush=True)


def separate(ctx, db, q, p):
    res = []
    try:
        for k in KS:
            ctx.set_kmer(k)
            res.append(ctx.align(db, q, p))
    finally:
        ctx.set_kmer(12)
    return res


def write_fasta(path, seq, start):
    with open(path, "wb") as f:
        for i in range(len(start) - 1):
            f.write(b">r%d\n" % i + bytes(seq[int(start[i]):int(start[i + 1])]) + b"\n")


def cli_arm(db, ds, q, qs):
    with tempfile.TemporaryDirectory() as d:
        dbf, qf = os.path.join(d, "db.fa"), os.path.join(d, "q.fa")
        write_fasta(dbf, db, ds)
        write_fasta(qf, q, qs)
        common = [EXE, "-query", qf, "-db", dbf]
        t0 = time.perf_counter()
        subprocess.run(common + ["-out", os.path.join(d, "f.align"), "-kmers", "8,10,14,16"], check=True,
                       capture_output=True)
        one = time.perf_counter() - t0
        t0 = time.perf_counter()
        for k in KS:
            subprocess.run(common + ["-kmer", str(k), "-out", os.path.join(d, f"g{k}.align")], check=True,
                           capture_output=True)
        five = time.perf_counter() - t0
        for k in KS:
            f = os.path.join(d, "f.align" if k == 12 else f"f.align.k{k}")
            assert open(f, "rb").read() == open(os.path.join(d, f"g{k}.align"), "rb").read(), k
        log(f"  command line: one -kmers process {one:.2f} s, five -kmer processes {five:.2f} s ({five / one:.2f}x); "
            f"every file equals its separate run's")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--divergence", default="0.10,0.25")
    ap.add_argument("--no-cli", action="store_true")
    a = ap.parse_args()
    ctx = api.Imsame(0)  # raises without an sm_100 device: this tool never runs on the CPU
    log(f"card: {card()}")
    p = api.make_params(n_threads=4)
    seed, g, glen, L, nd, nq = SIZES
    for div in (float(x) for x in a.divergence.split(",")):
        pool = H.SynthPool(seed, g, glen)
        db, q = pool.db_reads(0, nd, L), pool.query_reads(0, nq, L, div)
        pool.close()
        ds, qs = np.arange(nd + 1, dtype=np.uint64) * L, np.arange(nq + 1, dtype=np.uint64) * L
        log(f"\n== {nq} x {L}-base query reads (divergence {div}) vs {nd} database reads, seed lengths {KS}")
        ctx.align_kmers((db, ds), (q, qs), KS, p)  # warm-up of both arms: allocations, pinned buffers, module load
        separate(ctx, (db, ds), (q, qs), p)
        wall = {"kmers": [], "separate": []}
        for rep in range(a.reps):
            for arm in ("kmers", "separate"):
                t0 = time.perf_counter()
                if arm == "kmers":
                    outs, codes, sts = ctx.align_kmers((db, ds), (q, qs), KS, p)
                    assert codes == [0] * len(KS)
                else:
                    sep = separate(ctx, (db, ds), (q, qs), p)
                wall[arm].append(time.perf_counter() - t0)
            for t, k in enumerate(KS):
                assert all(np.array_equal(outs[t][f], sep[t][0][f]) for f in FIELDS), (div, k)
            log(f"  rep {rep}: one call {1e3 * wall['kmers'][-1]:9.1f} ms, five calls {1e3 * wall['separate'][-1]:9.1f} ms; "
                f"records of every entry equal the separate calls'")
        for t, k in enumerate(KS):
            s, r = sts[t], sep[t][1]
            log(f"  k={k:2d}  accepted {s['n_accepted']:6d}  n_pairs {s['n_pairs']:9d}  n_pairs_dp {s['n_pairs_dp']:9d} "
                f"(separate {r['n_pairs_dp']:9d})  ms_k3 {s['ms_k3']:8.2f} (separate {r['ms_k3']:8.2f})  "
                f"ms_k1 {s['ms_k1']:7.2f}  ms_k2 {s['ms_k2']:7.2f}")
        dp1, dp5 = sum(s["n_pairs_dp"] for s in sts), sum(r[1]["n_pairs_dp"] for r in sep)
        k31, k35 = sum(s["ms_k3"] for s in sts), sum(r[1]["ms_k3"] for r in sep)
        med = {k: float(np.median(v)) for k, v in wall.items()}
        log(f"  pairs through NW: {dp1} of {dp5} ({dp1 / max(dp5, 1):.3f}); K3 {k31:.1f} ms of {k35:.1f} ms")
        log(f"  median wall over {a.reps}: one call {1e3 * med['kmers']:.1f} ms, five calls {1e3 * med['separate']:.1f} ms "
            f"({med['separate'] / med['kmers']:.2f}x)")
        if not a.no_cli:
            cli_arm(db, ds, q, qs)
    ctx.close()


if __name__ == "__main__":
    main()
