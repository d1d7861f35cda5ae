#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native IMSAME hot path.

  python bench.py --gpus N --steps K --warmup W            (our arm; torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K --warmup W   (reference CPU arm)
  python bench.py ... --dump-outputs DIR          (also write the records of the last timed step, DIR/<field>.npy)

Workload (BASELINE.json): configs[1] = 1 M x 250 bp Illumina-like query reads against a 10 M-read synthetic
metagenome on one B200.  For N > 1 the database grows to N x 10 M reads (configs[2] at N = 8: 80 M reads), sharded
by contiguous read ranges, one shard per GPU, the query replicated (weak scaling: per-GPU work fixed); the
reductions -- ncclAllReduce(ncclUint64, ncclMin) of the packed best-hit keys between k-mer-end bands, ncclMax of the
owner's payload -- run INSIDE the library (imsame_gpu_run_sharded); torch.distributed only hands the communicator id
around and does the barriers.  The N > 1 lines also carry `strong_cfg3`: configs[2] as stated, the FIXED 80 M-read
database cut over the N GPUs (`--cfg3` measures that as the main line, at any N incl. 1).

A "step" = one pass of the hot path (database scan + extension + NW + filter + selection [+ reductions]) over the
resident shard.  `value` counts (query read x 10 M-read shard) alignments per second, i.e. plain query reads/s at
N = 1; `query_reads_per_s` is always the plain figure.  `e2e` times the public C-ABI call imsame_gpu_align with pinned
HOST buffers: H2D of both read sets (one database segment ahead of the scan), 2-bit packing, query table build, scan,
NW, D2H of the records.

After the timed region (never inside it):
  sampled_parity  1024 seeded random query reads re-derived by the index-free CPU oracle (oracle/imsame_sampled.c)
                  against this run's full-size database (per shard + min-key merge at N > 1), all record fields equal;
                  its `cpu_port_same_database` is the port's reads/s on that sample (the one CPU figure at full database size)
  sharded_check   N > 1: the library's band-stepped NCCL run == independent shard runs reduced through torch.distributed
  same_config     N = 1: configs[0] at full size through the unmodified reference binary (whole process and alignment
                  phase, all host threads) and through imsame_gpu_align, record sets compared
  cpu_baseline    the reference binary on a bounded sample of the workload (its index cannot hold configs[1])
  k3_by_read_len  N = 1: cell rate of the packed-word and the generic NW kernel on explicit random pairs of 250 and of
                  300 bases (2 x 300 sequencing: the wide packed-word kernel), results compared
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# INT32 lane-operations one NW cell needs (DESIGN.md section 4/6):
#   generic kernel (nw_core.cuh): the SURVEY.md 8(d) accounting, 24 ops per cell
#   packed-word kernel (nwp_core.cuh): 16 -- 2 compares, 4 selects (2 of them fused with a logic op /
#   add as predicated instructions), one 3-input maximum (2 instructions), 3 logic ops, 5 adds
#   (one fused into the maximum); = the instructions per cell in the SASS of the unrolled row body
OPS_PER_CELL_GENERIC = 24
OPS_PER_CELL_PACKED = 16


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the workload (debug only; <1 is not a valid bench)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--nw-mode", type=int, default=0, help="0: packed-word K3 where eligible (default); 1: generic K3 (A/B only)")
    ap.add_argument("--cpu-sample-queries", type=int, default=2000)
    ap.add_argument("--cpu-sample-db", type=int, default=100000)
    ap.add_argument("--no-same-config", action="store_true", help="skip the cfg1 full-size GPU/reference pair")
    ap.add_argument("--no-strong", action="store_true", help="N > 1: skip the fixed-80M-read-database (cfg3) record")
    ap.add_argument("--cfg3", action="store_true",
                    help="measure BASELINE.json configs[2] itself: the FIXED 80M-read database cut over N GPUs (strong scaling, "
                         "N = 1 allowed); default: configs[1] at N = 1 and N x 10M reads (weak) at N > 1")
    ap.add_argument("--parity-sample", type=int, default=1024,
                    help="query reads checked against the index-free oracle after the timed region (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the records of the last step as DIR/<field>.npy (see dump_records)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the GPU arm's records: not with --impl reference")
    return a


def workload(scale, cfg3=False, world=1):
    w = dict(name="cfg2: 1M x 250bp Illumina-like reads vs 10M-read synthetic metagenome (default flags)",
             seed=2001, genomes_per_shard=1000, genome_len=1_000_000, L=250, nd_per_gpu=10_000_000,
             nq=1_000_000, divergence=0.03, genomes_total=1000 * world, cfg3=False)
    if cfg3:
        w.update(name="cfg3: 1M x 250bp query reads vs the FIXED 80M-read synthetic metagenome (8000 genomes), sharded over N GPUs",
                 nd_per_gpu=80_000_000 // world, genomes_total=8000, cfg3=True)
    if scale != 1.0:
        w["nd_per_gpu"] = max(1000, int(w["nd_per_gpu"] * scale))
        w["nq"] = max(100, int(w["nq"] * scale))
        w["genomes_per_shard"] = max(2, int(w["genomes_per_shard"] * scale))
        w["genomes_total"] = max(2, int(w["genomes_total"] * scale))
        w["name"] += f" [SCALED x{scale}: not a valid bench]"
    return w


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)"""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def int32_peak_gops():
    """measured INT32 lane-op rate (tools/int_peak.cu); ALU-pipe figure = imnmx line"""
    exe = os.path.join(ROOT, "tools", "int_peak")
    out = {}
    try:
        txt = subprocess.run([exe], capture_output=True, text=True, timeout=120).stdout
        for line in txt.splitlines():
            d = json.loads(line)
            if "op" in d:
                out[d["op"]] = d["gops"]
    except Exception as e:  # noqa: BLE001
        out["error"] = str(e)
    return out


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


# ------------------------------------------------------------------------------------------
def reference_cpu_run(args, w, steps, warmup):
    """Times the reference's own CPU implementation (oracle/_ref/IMSAME, compiled unmodified from
    /root/reference/src) on a bounded sample of the workload, all host threads."""
    from imsame_b200 import hostlib as H
    ref = os.path.join(ROOT, "oracle", "_ref", "IMSAME")
    if not os.path.exists(ref):
        return None, "oracle/_ref/IMSAME missing"
    cores = os.cpu_count() or 1
    nq, nd, L = args.cpu_sample_queries, args.cpu_sample_db, w["L"]
    g = max(2, int(w["genomes_per_shard"] * nd / w["nd_per_gpu"]))  # same coverage as the full workload
    pool = H.SynthPool(w["seed"], g, w["genome_len"])
    db = pool.db_reads(0, nd, L)
    q = pool.query_reads(0, nq, L, w["divergence"])
    pool.close()
    tmp = tempfile.mkdtemp(prefix="imsame_ref_")
    dbf, qf, outf = (os.path.join(tmp, n) for n in ("db.fa", "q.fa", "out.align"))
    H.write_fasta(dbf, db, nd, L, "d")
    H.write_fasta(qf, q, nq, L, "q")
    walls, aligns, builds = [], [], []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        txt = subprocess.run([ref, "-query", qf, "-db", dbf, "-out", outf, "-n_threads", str(cores)],
                             capture_output=True, text=True, check=True).stdout
        wall = time.perf_counter() - t0
        # the load phases are single-threaded, so the reference's clock() prints are wall time there
        # (src/IMSAME.c:102,295,407); alignment-phase wall = process wall - those
        ph = {"Initialization took": 0.0, "Hash table building took": 0.0, "Took": 0.0}
        for line in txt.splitlines():
            for key in ph:
                if key in line:
                    try:
                        ph[key] += float(line.split(key)[1].split()[0])
                    except Exception:
                        pass
        if it >= warmup:
            walls.append(wall)
            aligns.append(max(wall - sum(ph.values()), 1e-9))
            builds.append(ph["Hash table building took"])
    import shutil
    shutil.rmtree(tmp, ignore_errors=True)
    wall = sum(walls) / len(walls)
    al = sum(aligns) / len(aligns)
    bl = sum(builds) / len(builds)
    sample = (f"{nq} x {L}bp query reads vs {nd}-read database drawn from {g} genomes (same generator, seeds and "
              f"coverage as the workload, database down-scaled {w['nd_per_gpu'] // nd}x because the reference's "
              f"index needs 24 B per database base, so its per-read cost here is a LOWER bound of the full-size cost); "
              f"whole-process wall {wall:.2f}s, database load + index build {bl:.2f}s (single thread), "
              f"alignment phase {al:.2f}s on {cores} threads")
    return {"reads_per_s_process": nq / wall, "reads_per_s_align_phase": nq / al,
            "reads_per_s_index_plus_align": nq / (al + bl), "cores": cores, "sample": sample,
            "ms_align_phase": al * 1e3, "ms_process": wall * 1e3}, None


def cfg1_inputs(H, np):
    """BASELINE.json configs[0] at full size: 10k x 150bp query reads vs a 100k-read database (seed 1001, 20 genomes)"""
    L, nd, nq = 150, 100_000, 10_000
    pool = H.SynthPool(1001, 20, 500_000)
    db = pool.db_reads(0, nd, L)
    q = pool.query_reads(0, nq, L, 0.03)
    pool.close()
    return db, np.arange(nd + 1, dtype=np.uint64) * L, q, np.arange(nq + 1, dtype=np.uint64) * L, L, nd, nq


def reference_cfg1(H, np, keep_out=None):
    """the unmodified reference binary on configs[0] at full size, all host threads, best of 2: whole process and
    alignment phase (process wall - its single-threaded load / index phases, whose clock() prints are wall time)"""
    import shutil
    ref = os.path.join(ROOT, "oracle", "_ref", "IMSAME")
    if not os.path.exists(ref):
        return None
    cores = os.cpu_count() or 1
    db, ds, q, qs, L, nd, nq = cfg1_inputs(H, np)
    tmp = tempfile.mkdtemp(prefix="imsame_cfg1_")
    dbf, qf, outf = (os.path.join(tmp, n) for n in ("db.fa", "q.fa", "ref.align"))
    H.write_fasta(dbf, db, nd, L, "d")
    H.write_fasta(qf, q, nq, L, "q")
    runs = []
    for _ in range(2):
        t0 = time.perf_counter()
        txt = subprocess.run([ref, "-query", qf, "-db", dbf, "-out", outf, "-n_threads", str(cores)],
                             capture_output=True, text=True, check=True).stdout
        wall = time.perf_counter() - t0
        load = 0.0
        for line in txt.splitlines():
            for key in ("Initialization took", "Hash table building took", "Took"):
                if key in line:
                    try:
                        load += float(line.split(key)[1].split()[0])
                    except Exception:
                        pass
        runs.append((wall, max(wall - load, 1e-9)))
    wall, al = min(r[0] for r in runs), min(r[1] for r in runs)
    headers = None
    if keep_out is not None:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import helpers as hp
        headers = hp.parse_align_headers(outf)
    shutil.rmtree(tmp, ignore_errors=True)
    return {"workload": "cfg1 at full size: 10k x 150bp query reads vs 100k-read database, defaults, -n_threads = host cores",
            "cores": cores, "reference_whole_process_reads_per_s": nq / wall, "reference_whole_process_s": wall,
            "reference_align_phase_reads_per_s": nq / al, "reference_align_phase_s": al,
            "reference_what": "oracle/_ref/IMSAME (unmodified reference) on FASTA files, best of 2; alignment phase = process wall "
                              "- its single-threaded load/index phases", "_headers": headers}


def same_config_cfg1(ctx, api, H, np):
    """BASELINE.json configs[0] at FULL size -- the one configuration the reference itself can run -- through both
    implementations on this box: the unmodified reference binary on all host threads (whole process and alignment
    phase) and imsame_gpu_align() from host buffers.  The two record sets must be identical."""
    r = reference_cfg1(H, np, keep_out=True)
    if r is None:
        return {"unavailable": "oracle/_ref/IMSAME missing"}
    want = r.pop("_headers")
    db, ds, q, qs, L, nd, nq = cfg1_inputs(H, np)
    params = api.make_params(n_threads=r["cores"])
    ctx.align((db, ds), (q, qs), params)
    ts = []
    for _ in range(3):
        t0 = time.perf_counter()
        out, st = ctx.align((db, ds), (q, qs), params)
        ts.append(time.perf_counter() - t0)
    got = sorted(api.header_fields(i, o, L) for i, o in enumerate(out) if o["accepted"])
    t = min(ts)
    r.update({"records": len(want), "records_identical_to_reference": got == want,
              "gpu_e2e_reads_per_s": nq / t, "gpu_e2e_ms": t * 1e3,
              "gpu_what": "imsame_gpu_align() from pageable host buffers: H2D, packing, query table, scan, NW, D2H (best of 3)",
              "speedup_vs_align_phase": (nq / t) / r["reference_align_phase_reads_per_s"],
              "speedup_vs_whole_process": (nq / t) / r["reference_whole_process_reads_per_s"]})
    return r


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = workload(args.scale)
    r, err = reference_cpu_run(args, w, max(1, args.steps), max(0, args.warmup))
    if r is None:
        OUT.emit(json.dumps({"impl": "reference", "unavailable": err}))
        return
    v = r["reads_per_s_align_phase"]
    line = {"impl": "reference", "metric": "query reads aligned/sec", "value": v, "unit": "reads/s",
            # a step = the alignment phase of one run of the reference binary on the sample: value = sample reads / that
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_align_phase"],
            "ms_per_step_whole_process": r["ms_process"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": w["name"], "sample": r["sample"]},
            "cpu_baseline": {"value": v, "unit": "reads/s", "cores": r["cores"], "kind": "reference",
                             "sample": r["sample"], "reads_per_s_whole_process": r["reads_per_s_process"]},
            # the contract: the reference arm's e2e repeats the line's own value.  It is the alignment phase alone
            # (src/IMSAME.c:409-467), the figure that flatters the reference: on this down-scaled sample its
            # single-threaded index build (:232-281, part of what imsame_gpu_align replaces) costs 10x the phase
            "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                    "what": "alignment phase of the reference (src/IMSAME.c:409-467) on all host threads",
                    "reads_per_s_index_plus_align": r["reads_per_s_index_plus_align"]}}
    if not args.no_same_config:
        # the one configuration the reference can run at FULL size, for a same-config pair with our arm's `same_config`
        import numpy as np
        c1 = reference_cfg1(H_mod(), np)
        if c1:
            c1.pop("_headers", None)
            line["same_config"] = c1
    OUT.emit(json.dumps(line))


def k3_by_read_len(ctx, np, lens=(250, 300), pairs_at_250=60000):
    """cell rate of the two NW kernels on explicit random pairs (imsame_gpu_nw_batch, kernel time = the library's CUDA
    events), per read length: 250 = the bench's own, 300 = 2 x 300 sequencing (NW class 10, the wide packed-word
    kernel with 19 columns per lane); one pair in 50 is a noisy copy (an accepted pair).  Outside the timed region."""
    rng = np.random.default_rng(1)
    B = np.frombuffer(b"ACGT", dtype=np.uint8)
    rows = []
    for L in lens:
        n = int(pairs_at_250 * (250.0 / L) ** 2)
        X = B[rng.integers(0, 4, size=(n, L))]
        Y = B[rng.integers(0, 4, size=(n, L))]
        for i in range(0, n, 50):
            Y[i] = X[i]
            hit = rng.random(L) < 0.03
            Y[i, hit] = B[rng.integers(0, 4, size=int(hit.sum()))]
        xs, ys = [X[i] for i in range(n)], [Y[i] for i in range(n)]
        cells = float(n) * (L - 1) * (L - 1)
        row = {"read_len": L, "pairs": n}
        res = {}
        for mode, name in ((0, "packed"), (1, "generic")):
            ctx.set_nw_mode(mode)
            best = None
            for _ in range(2):
                got, ms = ctx.nw_batch(xs, ys)
                best = ms if best is None or ms < best else best
            res[name] = np.asarray(got)
            row[name + "_gcups"] = round(cells / best / 1e6, 1)
        ctx.set_nw_mode(0)
        row["identical"] = bool(np.array_equal(res["packed"], res["generic"]))
        rows.append(row)
    return rows


def H_mod():
    from imsame_b200 import hostlib as H
    return H


DUMP_BYTES_MAX = 60_000_000  # array bytes of one --dump-outputs directory: with the .npy headers under 64 MB
DUMP_FIELDS = (("accepted", "float32"), ("db_seq", "float64"), ("qpos_end", "float64"), ("db_pos", "float64"),
               ("length", "float32"), ("identities", "float32"))


def dump_records(d, rec, np):
    """The records a caller of the timed path receives (imsame_gpu_fetch: one per query read), one file per field,
    plus read.npy with the query read each row belongs to.  Read numbers and positions are float64 (exact below
    2^53), lengths, identities and the accepted flag float32.  Above DUMP_BYTES_MAX, a fixed seeded sample of reads."""
    per_read = 8 + sum(np.dtype(t).itemsize for _, t in DUMP_FIELDS)
    reads = np.arange(len(rec))
    if len(rec) * per_read > DUMP_BYTES_MAX:
        reads = np.sort(np.random.default_rng(20261020).choice(len(rec), DUMP_BYTES_MAX // per_read, replace=False))
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "read.npy"), reads.astype(np.float64))
    for name, t in DUMP_FIELDS:
        np.save(os.path.join(d, name + ".npy"), rec[name][reads].astype(t))


# ------------------------------------------------------------------------------------------
def sampled_parity(n_sample, rec, db, ds, q, qs, db_total_global, rank, world, nd, L, dist, torch, np):
    """AFTER the timed region, checker only: a seeded random sample of query reads (accepted and unaccepted)
    is re-derived by the index-free CPU oracle (oracle/imsame_sampled.c: hash the sample's words, stream this
    rank's database shard once, replay every e-value-passing hit in the reference's scan order through its NW
    and filter until the first acceptance) and compared field by field with the records the GPU run produced.
    Shards: each rank checks its own shard in global coordinates, the oracle's per-shard winners are reduced
    like the reference's order demands (smallest k-mer end, then largest database position)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers as hp
    nq = len(qs) - 1
    n_sample = min(n_sample, nq)
    reads = np.sort(np.random.default_rng(20261018).choice(nq, n_sample, replace=False)).astype(np.uint64)
    hp.oracle_set_threads(max(1, (os.cpu_count() or 1) // max(1, world)))
    t0 = time.perf_counter()
    p = hp.default_params(n_threads=4, db_total_len_global=db_total_global)
    got, st = hp.oracle_align_sampled(hp.OracleSeqs(seq=db, start=ds), hp.OracleSeqs(seq=q, start=qs), p, reads,
                                      db_pos_base=rank * nd * L, db_seq_base=rank * nd)
    t_oracle = time.perf_counter() - t0
    # oracle winners of this shard -> the same (key, payload) words the product reduces
    from imsame_b200 import sharding
    ok = np.full(n_sample, sharding.KEY_NONE, dtype=np.int64)
    op = np.zeros(n_sample, dtype=np.int64)
    for i, r in enumerate(reads):
        v = got.get(int(r))
        if v is not None:
            ok[i] = sharding.make_key(v[1] - int(qs[int(r)]) + 1, v[2])
            op[i] = sharding.make_payload(v[0], v[3], v[4])
    if world > 1:
        tk, tp = torch.from_numpy(ok).cuda(), torch.from_numpy(op).cuda()
        local = tk.clone()
        dist.all_reduce(tk, op=dist.ReduceOp.MIN)
        tp[(tk != local) | (tk == sharding.KEY_NONE)] = 0
        dist.all_reduce(tp, op=dist.ReduceOp.MAX)
        ok, op = tk.cpu().numpy(), tp.cpu().numpy()
    want = sharding.decode(ok, op, qs[reads.astype(np.int64)])
    mism = 0
    n_acc = 0
    first_bad = None
    for i, r in enumerate(reads):
        o = rec[int(r)]
        g = ((int(o["db_seq"]), int(o["qpos_end"]), int(o["db_pos"]), int(o["length"]), int(o["identities"]))
             if o["accepted"] else None)
        w = want.get(i)
        n_acc += w is not None
        if g != w:
            mism += 1
            if first_bad is None:
                first_bad = {"read": int(r), "gpu": g, "oracle": w}
    out = {"reads": int(n_sample), "mismatches": int(mism), "oracle_accepted": int(n_acc),
           "fields": "accepted, db_seq, qpos_end, db_pos, length, identities",
           "oracle": "oracle/imsame_sampled.c (index-free scan-order replay), per shard + min-key merge",
           "oracle_hits_this_rank": int(st.hits), "oracle_nw_calls_this_rank": int(st.nw_calls),
           "seconds": round(time.perf_counter() - t0, 1),
           # the only CPU execution of the reference's algorithm against the FULL database of the workload (the reference's
           # own index cannot hold it): per-read cost of the port on this rank's shard.  It extends every seed hit of the
           # sampled reads (the reference skips the later words of an accepted read) and runs exactly the reference's NW calls.
           "cpu_port_same_database": {"reads_per_s": round(n_sample / max(t_oracle, 1e-9), 1), "seconds": round(t_oracle, 2),
                                      "threads": max(1, (os.cpu_count() or 1) // max(1, world)), "kind": "port",
                                      "what": "oracle/imsame_sampled.c, %d sampled query reads vs this rank's %d-read shard" % (n_sample, nd)}}
    if first_bad:
        out["first_mismatch"] = first_bad
    return out


def run_ours(args):
    import numpy as np
    import torch
    from imsame_b200 import api, hostlib as H

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # torchrun pins OMP_NUM_THREADS=1; the synthetic generator (host/synth.c) is OpenMP
    H.set_synth_threads(max(1, (os.cpu_count() or 1) // max(1, world)))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    w = workload(args.scale, args.cfg3, world)
    L, nq, nd = w["L"], w["nq"], w["nd_per_gpu"]
    n_genomes = w["genomes_total"]
    t0 = time.perf_counter()
    pool = H.SynthPool(w["seed"], n_genomes, w["genome_len"])
    db_pin = api.PinnedArray(nd * L)
    q_pin = api.PinnedArray(nq * L)
    pool.db_reads(rank * nd, nd, L, out=db_pin.array)                    # this rank's shard of the database
    pool.query_reads(0, nq, L, w["divergence"], n_genomes_used=w["genomes_per_shard"], out=q_pin.array)
    pool.close()
    t_gen = time.perf_counter() - t0
    ds = np.arange(nd + 1, dtype=np.uint64) * L
    qs = np.arange(nq + 1, dtype=np.uint64) * L
    db_total_global = nd * L * world
    params = api.make_params(n_threads=4, db_total_len_global=db_total_global, db_pos_base=rank * nd * L,
                             db_seq_base=rank * nd)

    ctx = api.Imsame(local)
    ctx.set_nw_mode(args.nw_mode)
    # one real (non-default) stream for everything: the library's kernels, torch ops and the NCCL reductions
    # issued through torch are ordered on it, and stream attributes (the scan's L2 window) can be set on it
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    keys = torch.empty(nq, dtype=torch.int64, device="cuda")
    payload = torch.empty(nq, dtype=torch.int64, device="cuda")

    ctx.set_query((q_pin.array, qs), params)
    ctx.set_db((db_pin.array, ds))
    torch.cuda.synchronize()

    if world > 1:
        # the reductions are the library's own (imsame_gpu_run_sharded: ncclAllReduce(ncclUint64, ncclMin) of the keys
        # between k-mer-end bands, ncclMax of the owner's payload); torch.distributed only hands the communicator id around
        box = [api.comm_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        ctx.comm_init(box[0], world, rank)

    def step():
        if world == 1:
            return ctx.run(params, keys.data_ptr(), payload.data_ptr())
        # shards exchange the per-read keys between k-mer-end bands, so an accepted early hit in one
        # shard prunes the later candidates of that read in every shard (the reference's early exit)
        return ctx.run_sharded(params, keys.data_ptr(), payload.data_ptr())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stats_steps = []
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        stats_steps.append(step())
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    tmax = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_total = float(tmax.item())
    clocks = sampler.stop() if rank == 0 else None
    rec = ctx.fetch(keys.data_ptr(), payload.data_ptr())
    if args.dump_outputs and rank == 0:  # every rank holds the reduced records
        dump_records(args.dump_outputs, rec, np)
    n_accepted = int(rec["accepted"].sum())
    # self-check of the sharded reduction (N > 1): the band-stepped run with key exchanges must give the
    # same records as independent shard runs followed by one min/max reduction
    sharded_check = None
    if world > 1:
        from imsame_b200 import sharding
        k2, p2 = torch.empty_like(keys), torch.empty_like(payload)
        ctx.run(params, k2.data_ptr(), p2.data_ptr())
        sharding.reduce_best(k2, p2, dist, lambda kr, kl, pl: ctx.mask_payload(kr.data_ptr(), kl.data_ptr(), pl.data_ptr()))
        same = bool(torch.equal(k2, keys)) and bool(torch.equal(p2, payload))
        flag = torch.tensor([1 if same else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        sharded_check = ("library NCCL band-stepped run == independent shard runs reduced through torch.distributed" if int(flag.item()) == 1
                         else "MISMATCH between the band-stepped library run and the unstepped torch-reduced run")

    parity = None
    if args.parity_sample > 0:
        parity = sampled_parity(args.parity_sample, rec, db_pin.array, ds, q_pin.array, qs, db_total_global, rank,
                                world, nd, L, dist, torch, np)

    # per-kernel device times of the timed steps (CUDA events on the launching stream, inside the library)
    def avg(k):
        return sum(s[k] for s in stats_steps) / len(stats_steps)
    cells = avg("n_cells")
    ms_k3, ms_k2 = avg("ms_k3"), avg("ms_k2")
    agg = torch.tensor([cells, ms_k3, ms_k2, avg("n_hits"), avg("n_pairs_dp"), avg("n_db_kmers"),
                        avg("n_evalue_pass")], dtype=torch.float64, device="cuda")
    agg_max = agg.clone()
    if world > 1:
        dist.all_reduce(agg, op=dist.ReduceOp.SUM)
        dist.all_reduce(agg_max, op=dist.ReduceOp.MAX)

    # ---- end to end through the public C-ABI call with host buffers -------------------------
    e2e = None
    if args.e2e_steps > 0:
        ctx2 = ctx
        barrier()
        t_e2e = []
        h2d = d2h = 0
        for it in range(args.e2e_steps + 1):
            barrier()
            t0 = time.perf_counter()
            if world == 1:
                out, st = ctx2.align((db_pin.array, ds), (q_pin.array, qs), params)
            else:
                # the same public calls a sharded caller makes: upload + pack + query table, upload + pack
                # of the shard, band-stepped run with the key exchange, owner's payload, records to the host
                st = ctx2.align_shard((db_pin.array, ds), (q_pin.array, qs), params, keys.data_ptr(), payload.data_ptr())
                out = ctx2.fetch(keys.data_ptr(), payload.data_ptr())
                st["h2d_bytes"] = int(nd * L + nq * L)
                st["d2h_bytes"] = int(16 * nq)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if it > 0:
                t_e2e.append(dt)
                h2d, d2h = st["h2d_bytes"], st["d2h_bytes"]
                e2e_phases = {k: round(float(st[k]), 2) for k in ("ms_h2d", "ms_pack_query", "ms_k1", "ms_pack_db", "ms_k2",
                                                                  "ms_k2b", "ms_k3", "ms_select", "ms_d2h", "ms_total")}
        te = torch.tensor([sum(t_e2e) / len(t_e2e)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e = {"value": (1 if args.cfg3 else world) * nq / float(te.item()), "unit": "reads/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "ms_per_step": float(te.item()) * 1e3,
               "what": ("imsame_gpu_align(): pinned host ASCII reads -> H2D -> pack -> query table -> scan -> NW -> D2H records"
                        if world == 1 else
                        "per rank: imsame_gpu_align_shard (pinned host ASCII reads -> H2D one segment ahead of the scan -> pack -> query "
                        "table -> band-stepped run, ncclMin key reductions and the owner's payload inside the library) -> D2H records"),
               "device_phases_ms": e2e_phases}

    # ---- cfg3 as BASELINE.json states it: the SAME 80 M-read database cut over N GPUs (strong scaling) --------
    strong = None
    if world > 1 and not args.no_strong and args.scale == 1.0 and not args.cfg3:
        nd_total = 80_000_000
        if world * nd == nd_total:
            # N = 8: this run's database already is cfg3 (8 x 10 M reads over the 8 000 genomes)
            strong = {"ms_per_step": ms_total / args.steps, "steps": args.steps, "same_run_as_main_line": True}
        else:
            nd_s = nd_total // world
            db_pin.free()
            db_pin = api.PinnedArray(nd_s * L)
            pool = H.SynthPool(w["seed"], 8000, w["genome_len"])
            pool.db_reads(rank * nd_s, nd_s, L, out=db_pin.array)
            pool.close()
            ds_s = np.arange(nd_s + 1, dtype=np.uint64) * L
            p_s = api.make_params(n_threads=4, db_total_len_global=nd_total * L, db_pos_base=rank * nd_s * L,
                                  db_seq_base=rank * nd_s)
            ctx.set_db((db_pin.array, ds_s))
            ctx.run_sharded(p_s, keys.data_ptr(), payload.data_ptr())  # warm-up (pair table and candidate buffers grow)
            barrier()
            n_s = max(1, min(args.steps, 3))
            e0.record(stream)
            for _ in range(n_s):
                st_s = ctx.run_sharded(p_s, keys.data_ptr(), payload.data_ptr())
            e1.record(stream)
            barrier()
            t_s = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
            dist.all_reduce(t_s, op=dist.ReduceOp.MAX)
            strong = {"ms_per_step": float(t_s.item()) / n_s, "steps": n_s, "same_run_as_main_line": False,
                      "accepted_reads": int((keys != api.KEY_NONE).sum().item()),
                      "ms_k2_rank0": st_s["ms_k2"], "ms_k3_rank0": st_s["ms_k3"], "ms_comm_rank0": st_s["ms_comm"]}
        strong.update({"workload": "cfg3: 1M x 250bp query reads vs the fixed 80M-read database (8000 genomes), sharded by contiguous "
                                   "read ranges over N GPUs, imsame_gpu_run_sharded", "scaling": "strong", "n_gpus": world,
                       "db_reads_total": nd_total, "query_reads_per_s": nq / (strong["ms_per_step"] * 1e-3),
                       "efficiency": "T_2 * 2 / (N * T_N) from the N = 2, 4, 8 lines (an 80M-read database is not the N = 1 workload)"})

    if rank == 0:
        peaks, which = measured_peaks()
        ipk = int32_peak_gops()
        ms_step = ms_total / args.steps
        cells_all, ms_k3_max, ms_k2_max = float(agg[0].item()), float(agg_max[1].item()), float(agg_max[2].item())
        gcups = cells_all / world / (ms_k3_max * 1e-3) / 1e9 if ms_k3_max > 0 else 0.0   # per GPU
        packed = all(s.get("k3_packed_launches", 0) == s.get("k3_launches", -1) for s in stats_steps)
        ops_per_cell = OPS_PER_CELL_PACKED if packed else OPS_PER_CELL_GENERIC
        # INT32 peak = the measured full-chip rate of independent 32-bit adds (ptxas spreads them over the
        # ALU and the FMA pipe: 2 x 64 lanes/clk/SM); the ALU pipe alone (compare/select/min/max/logic) is half
        int_peak = ipk.get("iadd") or 0.0
        alu_peak = ipk.get("imnmx") or 0.0
        achieved = gcups * ops_per_cell
        # K2 algorithmic bytes (SURVEY 8(d)): Nd/4 + 8 per db word + 4 per hit + 16 per passing hit
        k2_bytes = nd * L / 4 + 8 * float(agg[5].item()) / world + 4 * float(agg[3].item()) / world + 16 * float(agg[6].item()) / world
        k2_gbs = k2_bytes / (ms_k2_max * 1e-3) / 1e9 if ms_k2_max > 0 else 0.0
        # what this design streams by construction: every hit reads its 24-byte table entry (qtable.cuh) instead of a 4-byte position
        k2_bytes_design = k2_bytes + 20 * float(agg[3].item()) / world
        k2_gbs_design = k2_bytes_design / (ms_k2_max * 1e-3) / 1e9 if ms_k2_max > 0 else 0.0
        try:  # per-launch DRAM traffic of the two hot kernels out of committed `ncu --set full` captures (tools/ncu_traffic.py)
            _tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        except Exception:
            _tr = {}
        k3_traffic = (_tr.get("nwp_kernel") or _tr.get("nwp_kernel_scale005") or {}) if packed else {}
        k2_traffic = _tr.get("scan_kernel") or {}
        line = {
            "metric": "query reads aligned/sec", "value": (1 if args.cfg3 else world) * nq / (ms_step * 1e-3), "unit": "reads/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "strong" if args.cfg3 else "weak", "vs_baseline": None, "dtype": "int32",
            "data": "synthetic",
            "config": {"workload": w["name"], "query_reads": nq, "db_reads_per_gpu": nd, "db_reads_total": nd * world,
                       "read_len": L, "kmer": 12, "flags": "defaults (evalue 1e-20, coverage 0.5, identity 0.5, igap 5, egap 2, n_threads 4)",
                       "sharding": f"db{world}" if world > 1 else "none",
                       "value_counts": ("query reads/s" if (world == 1 or args.cfg3) else
                                        "WEAK scaling: the database grows with N (N x 10M reads), so `value` counts query-read x "
                                        "10M-read-shard alignments per second; `query_reads_per_s` is the plain figure against the "
                                        "N x 10M-read database, `strong_cfg3` the fixed 80M-read database of configs[2]"),
                       "l2": "inputs (625 MB packed shard + 5.8 GB query table) exceed the 126 MB L2"},
            "query_reads_per_s": nq / (ms_step * 1e-3),
            "dp_gcups_per_gpu": gcups, "dp_gcups_total": gcups * world,
            "accepted_reads": n_accepted, "sharded_check": sharded_check, "sampled_parity": parity, "strong_cfg3": strong,
            "work": {"hits": float(agg[3].item()), "evalue_pass": float(agg[6].item()), "nw_pairs": float(agg[4].item()),
                     "cells": cells_all, "ms_k2": ms_k2_max, "ms_k3": ms_k3_max,
                     "ms_other": max(0.0, ms_step - ms_k2_max - ms_k3_max)},
            "roofline": {"kernel": ("nwp_kernel (K3p, packed-word NW wavefront, 16 lanes per pair)" if packed
                                    else "nw_kernel (K3, per-pair NW wavefront)"),
                         "bound": "int32-issue",
                         "achieved": achieved, "peak": int_peak, "unit": "Gop/s",
                         "frac": (achieved / int_peak) if int_peak else None,
                         # independent of any per-cell op count: thread-instructions the kernel actually executed per second in the
                         # committed `ncu --set full` capture (smsp__inst_executed x average active threads / duration) / issue peak
                         "frac_issue": ((k3_traffic.get("thread_inst_per_s_under_ncu") or 0) / (int_peak * 1e9)) if int_peak and k3_traffic.get("thread_inst_per_s_under_ncu") else None,
                         "issue_active_pct_ncu": k3_traffic.get("issue_active_pct"), "alu_pipe_pct_ncu": k3_traffic.get("alu_pipe_pct"),
                         "traffic": k3_traffic.get("dram_bytes_per_launch"),
                         "traffic_note": "dram__bytes_read + dram__bytes_write of one `ncu --set full` launch (profiles/ncu_traffic.json: "
                                         + str(k3_traffic.get("report")) + ", " + str(k3_traffic.get("note")) + "); the kernel is register/"
                                         "shared-memory resident, HBM is not its bound",
                         "ops_per_cell": ops_per_cell, "gcups": gcups,
                         "gcups_roofline": (int_peak / ops_per_cell) if ops_per_cell else None,
                         "frac_survey24": (gcups * OPS_PER_CELL_GENERIC / int_peak) if int_peak else None,
                         "alu_pipe_peak": alu_peak,
                         "frac_of_alu_pipe_at_24": (gcups * OPS_PER_CELL_GENERIC / alu_peak) if alu_peak else None,
                         "peak_source": "tools/int_peak.cu run on this GPU just now: `iadd` = independent 32-bit adds over both "
                                        "integer pipes (128 lanes/clk/SM); MEASURED_PEAKS.json has no INT32 figure",
                         "int_peak_table": ipk},
            "roofline_k2": {"kernel": "scan_kernel (K2, db scan + extension)", "bound": "hbm", "achieved": k2_gbs,
                            "peak": peaks.get("hbm_gbs"), "unit": "GB/s",
                            "frac": k2_gbs / peaks["hbm_gbs"] if peaks.get("hbm_gbs") else None,
                            "bytes_per_step_survey_8d": k2_bytes,
                            "achieved_design_bytes": k2_gbs_design, "bytes_per_step_design": k2_bytes_design,
                            "frac_design_bytes": k2_gbs_design / peaks["hbm_gbs"] if peaks.get("hbm_gbs") else None,
                            "design_note": "SURVEY 8(d) counts 4 B per hit (a word position); this design reads a 24-byte table entry per hit "
                                           "(both query windows inline) so that a hit needs no dependent gathers; the kernel is bound by the "
                                           "shared-memory pipe (walk-table lookups) and instruction issue, not by HBM",
                            "l1_data_pipe_pct_ncu": k2_traffic.get("l1_data_pipe_pct"), "issue_active_pct_ncu": k2_traffic.get("issue_active_pct"),
                            "traffic": k2_traffic.get("dram_bytes_per_launch"),
                            "traffic_note": "per launch = one database segment of <= 0.5 Gbase (profiles/ncu_traffic.json: "
                                            + str(k2_traffic.get("report")) + "); the algorithmic bytes of `achieved` are per step",
                            "peak_source": which},
            "e2e": e2e, "gpu_launches": int(sum(s["total_launches"] for s in stats_steps)),
            "clocks": clocks, "gen_seconds": t_gen,
        }
        if not args.no_same_config and world == 1 and args.scale == 1.0 and not args.cfg3:
            line["same_config"] = same_config_cfg1(ctx, api, H, np)
        if world == 1 and not args.cfg3 and args.nw_mode == 0:
            line["k3_by_read_len"] = k3_by_read_len(ctx, np)
        if not args.no_cpu_baseline and world == 1:
            r, err = reference_cpu_run(args, w, 1, 0)
            if r:
                line["cpu_baseline"] = {"value": r["reads_per_s_align_phase"], "unit": "reads/s", "cores": r["cores"],
                                        "kind": "reference", "sample": r["sample"],
                                        "reads_per_s_whole_process": r["reads_per_s_process"],
                                        "reads_per_s_index_plus_align": r["reads_per_s_index_plus_align"]}
            else:
                line["cpu_baseline"] = {"unavailable": err}
        OUT.emit(json.dumps(line))
    ctx.close()
    db_pin.free()
    q_pin.free()
    if world > 1:
        dist.destroy_process_group()


class StdoutToStderr:
    """stdout carries exactly ONE line (the JSON): everything libraries print on fd 1 meanwhile (NCCL's
    version banner, torchrun notes) is sent to stderr; `emit` writes to the real stdout."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, text):
        sys.stdout.flush()
        os.write(self.real, (text + "\n").encode())


OUT = None


if __name__ == "__main__":
    a = parse()
    OUT = StdoutToStderr()
    if a.impl == "reference":
        run_reference_arm(a)
    else:
        run_ours(a)
