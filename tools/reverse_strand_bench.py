#!/usr/bin/env python
"""The reverse strand of a resident database against the second process of the reference workflow, on one GPU.

On the same seeded cfg2-shaped inputs (1 M x 250-base query reads, 10 M x 250-base database reads, scaled by --scale):
  fwd        imsame_gpu_align: the forward strand (upload, K1, run)
  mirror     imsame_gpu_db_revcomp alone (CUDA events)
  rev_dev    imsame_gpu_align_revcomp: the reverse strand on the resident database (mirror + run)
  rev_host   imsame_gpu_align on the host parse of the reverse complement: the second process's library work
             (upload, K1, run)
and the wall clock of `IMSAME -out_rev r` against `IMSAME; revComp db db.r; IMSAME -db db.r -out r2`.
Workloads: cfg2 as generated (forward strand only: the reverse strand accepts almost nothing), and cfg2 with every
second database read reverse complemented.  Every run checks that both reverse paths give identical records, that
the two command lines write identical files, and 1 024 sampled reads of the reverse strand against the index-free
oracle.  usage: python tools/reverse_strand_bench.py [--scale 1.0] [--reps 2] [--no-cli] [--workloads cfg2,cfg2_mixed]"""
import argparse
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from imsame_b200 import api, hostlib as H  # noqa: E402

COMP = np.arange(256, dtype=np.uint8)
for _a, _b in zip(b"ACGT", b"TGCA"):
    COMP[_a] = _b


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else "nvidia-smi unavailable"


def log(*a):
    print(*a, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--no-cli", action="store_true")
    ap.add_argument("--workloads", default="cfg2,cfg2_mixed")
    a = ap.parse_args()
    import torch
    import helpers as hp
    L = 250
    nd, nq, g = int(10_000_000 * a.scale), int(1_000_000 * a.scale), max(2, int(1000 * a.scale))
    log(f"card: {card()}  (torch: {torch.cuda.get_device_name(0)})")
    log(f"inputs: {nq} query reads x {nd} database reads, {L} bases, seeded (SynthPool 2001)")
    pool = H.SynthPool(2001, g, 1_000_000)
    fwd_db = pool.db_reads(0, nd, L)
    q = pool.query_reads(0, nq, L, 0.03)
    pool.close()
    ds = np.arange(nd + 1, dtype=np.uint64) * L
    qs = np.arange(nq + 1, dtype=np.uint64) * L
    ctx = api.Imsame(0)
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    p = api.make_params(n_threads=4)
    for name in a.workloads.split(","):
        db = fwd_db
        if name == "cfg2_mixed":  # every second read reverse complemented
            db = fwd_db.copy().reshape(nd, L)
            db[1::2] = COMP[db[1::2, ::-1]]
            db = db.reshape(-1)
        rdb = COMP[db[::-1]]  # the reverse parse (fixed-length reads: offsets unchanged)
        log(f"\n== {name}")
        ctx.align((db, ds), (q, qs), p)  # warm-up: allocations, pinned bounce buffers, module load
        t = {"fwd": [], "rev_dev": [], "rev_host": [], "mirror_ms": []}
        acc = {}
        for rep in range(a.reps):
            for what in ("fwd", "rev_dev", "rev_host"):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                if what == "fwd":
                    out, st = ctx.align((db, ds), (q, qs), p)
                elif what == "rev_dev":
                    out, st = ctx.align_revcomp()
                    rev_dev = out
                else:
                    out, st = ctx.align((rdb, ds), (q, qs), p)
                    rev_host = out
                t[what].append(time.perf_counter() - t0)
                acc[what] = int(out["accepted"].sum())
                log(f"  rep {rep} {what:8s} wall {1e3 * t[what][-1]:8.1f} ms  device {st['ms_total']:8.1f} ms  "
                    f"(pack_db {st['ms_pack_db']:.1f}, k1 {st['ms_k1']:.1f}, k2 {st['ms_k2']:.1f}, k3 {st['ms_k3']:.1f}, "
                    f"h2d {st['h2d_bytes'] / 1e9:.2f} GB, passes {st['scan_passes']})  accepted {acc[what]}")
            assert np.array_equal(rev_dev, rev_host), "the two reverse paths differ"
        # the mirror alone: the resident (reverse) database mirrored twice per sample, CUDA events on the context's stream
        ctx.align_revcomp()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(5):
            e0.record()
            ctx.db_revcomp()
            e1.record()
            torch.cuda.synchronize()
            t["mirror_ms"].append(e0.elapsed_time(e1))
        packed_bytes = 2 * (len(db) // 4)  # packed database read once and written once
        m = min(t["mirror_ms"])
        log(f"  db_revcomp alone: min {m:.3f} ms, median {np.median(t['mirror_ms']):.3f} ms over 5 "
            f"({packed_bytes / 1e9:.2f} GB of packed bases read + written: {packed_bytes / m / 1e6:.0f} GB/s)")
        log(f"  records of align_revcomp == align(host reverse parse): True ({acc['rev_dev']} accepted)")
        reads = np.sort(np.random.default_rng(5).choice(nq, 1024, replace=False))
        want, _ = hp.oracle_align_sampled(hp.OracleSeqs(seq=rdb, start=ds), hp.OracleSeqs(seq=q, start=qs),
                                          hp.default_params(n_threads=4), reads)
        got = {int(r): (int(rev_dev[r]["db_seq"]), int(rev_dev[r]["qpos_end"]), int(rev_dev[r]["db_pos"]),
                        int(rev_dev[r]["length"]), int(rev_dev[r]["identities"])) for r in reads if rev_dev[r]["accepted"]}
        assert got == want
        log(f"  1024 sampled reads of the reverse strand == index-free oracle: True ({len(want)} accepted among them)")
        med = {k: float(np.median(v)) for k, v in t.items() if k != "mirror_ms"}
        log(f"  median wall: fwd {1e3 * med['fwd']:.1f} ms, reverse on the resident database {1e3 * med['rev_dev']:.1f} ms, "
            f"reverse from the host parse {1e3 * med['rev_host']:.1f} ms: saved {1e3 * (med['rev_host'] - med['rev_dev']):.1f} ms per run")
        if not a.no_cli:
            cli(name, db, q, nd, nq, L, a.reps)
        del rdb
    ctx.close()


def cli(name, db, q, nd, nq, L, reps):
    exe, rc = os.path.join(ROOT, "bin", "IMSAME"), os.path.join(ROOT, "bin", "revComp")
    with tempfile.TemporaryDirectory(prefix="imsame_rev_") as d:
        dbf, qf, dr, r1, r2 = (os.path.join(d, n) for n in ("db.fa", "q.fa", "db.r.fa", "r1.align", "r2.align"))
        H.write_fasta(dbf, np.ascontiguousarray(db), nd, L, "d")
        H.write_fasta(qf, q, nq, L, "q")

        def run(args):
            r = subprocess.run(args, capture_output=True, text=True)
            assert r.returncode == 0, r.stdout[-2000:]

        walls = {"one process (-out_rev)": [], "revComp + two processes": []}
        for rep in range(reps):  # alternating, the page cache warm after the first
            for how in walls:
                for f_ in ((r1,) if how.startswith("one") else (dr, r2)):
                    if os.path.exists(f_):
                        os.remove(f_)
                t0 = time.perf_counter()
                if how.startswith("one"):
                    run([exe, "-query", qf, "-db", dbf, "-out_rev", r1])
                else:
                    run([exe, "-query", qf, "-db", dbf])
                    run([rc, dbf, dr])
                    run([exe, "-query", qf, "-db", dr, "-out", r2])
                walls[how].append(time.perf_counter() - t0)
                log(f"  CLI rep {rep} {how}: {walls[how][-1]:.2f} s")
        same = open(r1, "rb").read() == open(r2, "rb").read()
        log(f"  CLI reverse-strand files identical: {same} ({os.path.getsize(r1) / 1e6:.1f} MB)")
        med = {k: float(np.median(v)) for k, v in walls.items()}
        log(f"  CLI median wall: one process {med['one process (-out_rev)']:.2f} s, revComp + two processes "
            f"{med['revComp + two processes']:.2f} s")


if __name__ == "__main__":
    main()
