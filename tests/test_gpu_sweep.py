"""GPU: several coverage/identity threshold sets in one run (imsame_gpu_align_sweep, IMSAME -sweep).  Every set's
records must equal, field by field, a separate imsame_gpu_align with that set's parameters, and the oracle where the
size allows; the command line's files and summary lines must equal those of separate runs."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import helpers as hp
import synth_cases as sc

pytestmark = pytest.mark.gpu
EXE = os.path.join(hp.ROOT, "bin", "IMSAME")
FIELDS = ("accepted", "db_seq", "qpos_end", "db_pos", "length", "identities", "reserved")
CFG5_SETS = [(0.5, i) for i in (0.70, 0.75, 0.80, 0.85, 0.90, 0.95)]


def records(out):
    return {int(r): (int(o["db_seq"]), int(o["qpos_end"]), int(o["db_pos"]), int(o["length"]), int(o["identities"]))
            for r, o in enumerate(out) if o["accepted"]}


def same(a, b):
    return all(np.array_equal(a[f], b[f]) for f in FIELDS)


def sweep_vs_separate(gpu, db, ds, q, qs, sets, n_threads=4, breaks=None, oracle=False, k=12, passes=(None,)):
    """the sweep against separate align() runs of every set (each at every passes mode listed; None = the current
    one) and, with oracle, against the oracle; returns (records per set, sweep stats, separate stats)"""
    from imsame_b200 import api
    ps = [api.make_params(n_threads=n_threads, min_coverage=c, min_identity=i) for c, i in sets]
    outs, codes, st = gpu.align_sweep((db, ds), (q, qs), ps, db_breaks=breaks)
    assert codes == [0] * len(sets)
    seps = []
    for t, p in enumerate(ps):
        for mode in passes:
            if mode is not None:
                gpu.set_passes(mode)
            want, st_t = gpu.align((db, ds), (q, qs), p, db_breaks=breaks)
            assert same(outs[t], want), (t, sets[t], mode)
            seps.append(st_t)
    if oracle:
        odb, oq = hp.OracleSeqs(seq=db, start=ds, brk=breaks), hp.OracleSeqs(seq=q, start=qs)
        for t, (c, i) in enumerate(sets):
            best, _ = hp.oracle_align(odb, oq, hp.default_params(n_threads=n_threads, coverage=c, identity=i, k=k))
            assert records(outs[t]) == hp.best_to_records(best, len(qs) - 1), (t, sets[t])
    assert st["n_accepted"] == int(outs[0]["accepted"].sum())
    return outs, st, seps


@pytest.mark.parametrize("divergence", [0.05, 0.15, 0.25, 0.30])
def test_cfg5_identity_sweep_in_one_run(gpu, divergence):
    """BASELINE.json configs[4] (test_cfg5_low_identity_sweep's inputs) as one six-set sweep: identities 70-95 %,
    coverage 50 %; fewer pairs run through NW than in the six separate runs together"""
    db, ds, q, qs = sc.fixed_case(5005, 4, 100000, 150, 20000, 1500, divergence)
    outs, st, seps = sweep_vs_separate(gpu, db, ds, q, qs, CFG5_SETS, oracle=True)
    acc = [int(o["accepted"].sum()) for o in outs]
    assert acc == sorted(acc, reverse=True) and acc[0] > (10 if divergence >= 0.25 else 300)
    assert st["n_pairs_dp"] < sum(s["n_pairs_dp"] for s in seps)
    assert st["n_db_kmers"] == seps[0]["n_db_kmers"] and st["n_pairs"] >= max(s["n_pairs"] for s in seps)


def test_coverage_sets_unsorted_with_duplicates_and_sizes_1_and_16(gpu):
    db, ds, q, qs = sc.ragged_case(611, 3, 40000, 3000, 500, 0.08, lo=30, hi=300)
    outs, _, _ = sweep_vs_separate(gpu, db, ds, q, qs, [(0.8, 0.5), (0.3, 0.5), (1.0, 0.5), (0.5, 0.5), (0.3, 0.5)],
                                   oracle=True)
    assert same(outs[1], outs[4]) and len({int(o["accepted"].sum()) for o in outs}) >= 3
    sweep_vs_separate(gpu, db, ds, q, qs, [(0.5, 0.5)])
    sixteen = [(c, i) for c in (0.3, 0.5, 0.8, 1.0) for i in (0.95, 0.6, 0.85, 0.5)]
    sweep_vs_separate(gpu, db, ds, q, qs, sixteen)


def test_ragged_reads_share_the_bins_between_both_nw_kernels(gpu):
    """query reads of 30-400 bases: the packed-word and the generic kernel share the bins pair by pair"""
    db, ds, q, qs = sc.ragged_case(808, 3, 60000, 6000, 900, 0.06, lo=30, hi=400)
    _, st, _ = sweep_vs_separate(gpu, db, ds, q, qs, [(0.5, 0.9), (0.3, 0.6), (0.9, 0.8)], oracle=True)
    assert 0 < st["k3_packed_launches"] < st["k3_launches"]


def test_forced_two_pass_run_and_wide_reads(gpu):
    """300-base reads (the wide packed classes) in a forced two-pass run, against separate runs at passes 1 and 2"""
    db, ds, q, qs = sc.fixed_case(3001, 3, 60000, 300, 5000, 800, 0.05)
    try:
        gpu.set_passes(2)
        _, st, seps = sweep_vs_separate(gpu, db, ds, q, qs, [(0.5, 0.95), (0.5, 0.6), (0.7, 0.85)], oracle=True, passes=(2, 1))
        assert st["scan_passes"] == 2 and [s["scan_passes"] for s in seps] == [2, 1] * 3
    finally:
        gpu.set_passes(0)


@pytest.mark.parametrize("k,n_threads", [(10, 4), (14, 4), (12, 3)])
def test_seed_length_and_phantom_words(gpu, k, n_threads):
    db, ds, q, qs = sc.ragged_case(900 + k, 3, 40000, 3000, 400, 0.06, lo=30, hi=300)
    try:
        gpu.set_kmer(k)
        sweep_vs_separate(gpu, db, ds, q, qs, [(0.5, 0.9), (0.5, 0.5), (0.8, 0.7)], n_threads=n_threads, oracle=True, k=k)
    finally:
        gpu.set_kmer(12)


def test_multi_segment_database(gpu):
    """more than one database segment (2^29 bases), shaped like test_multi_segment_database"""
    db, ds, q, qs = sc.ragged_case(4243, 300, 1000000, 3_000_000, 30000, 0.04, lo=30, hi=400)
    assert len(db) > (1 << 29)
    outs, st, _ = sweep_vs_separate(gpu, db, ds, q, qs, [(0.5, 0.95), (0.5, 0.5), (0.8, 0.8)])
    assert st["k2_launches"] >= 2 and outs[1]["accepted"].sum() > 3000


def read_size_case():
    """a database read of 5 000 bases that a query read reaches before any accepted hit under a strict identity, but
    not under a loose one: a mutated copy of the same piece (identity ~0.93) sits later in the database, where the
    scan order reaches it first"""
    db, ds, q, qs = sc.fixed_case(71, 3, 50000, 200, 4000, 300, 0.03)
    rng = np.random.default_rng(3)
    B = np.frombuffer(b"ACGT", dtype=np.uint8)
    contig = B[rng.integers(0, 4, size=5000)]
    cut = 2000 * 200
    db_a = np.concatenate([db[:cut], contig, db[cut:]])
    ds_a = np.concatenate([ds[:2001], ds[2000:] + 5000]).astype(np.uint64)
    piece = contig[1000:1200]
    q_b = q.copy()
    q_b[40 * 200:41 * 200] = piece
    copy = piece.copy()
    lut = {a: b for a, b in zip(b"ACGT", b"CGTA")}
    copy[14::15] = [lut[int(x)] for x in copy[14::15]]
    lo = int(ds_a[3500])
    db_a[lo:lo + 200] = copy
    return db_a, ds_a, q_b, qs


def test_read_size_error_per_set(gpu):
    """set_rc equals each separate align's return code; the other sets' records equal the separate runs'"""
    from imsame_b200 import api
    db_a, ds_a, q_b, qs = read_size_case()
    sets = [(0.5, 0.5), (0.5, 0.95), (0.5, 0.7), (0.5, 0.97)]
    ps = [api.make_params(n_threads=4, min_coverage=c, min_identity=i) for c, i in sets]
    outs, codes, _ = gpu.align_sweep((db_a, ds_a), (q_b, qs), ps)
    want_codes = []
    for t, p in enumerate(ps):
        try:
            want, _ = gpu.align((db_a, ds_a), (q_b, qs), p)
            want_codes.append(0)
            assert same(outs[t], want), t
        except api.ImsameError as e:
            want_codes.append(e.code)
            assert not outs[t]["accepted"].any()
    assert codes == want_codes == [0, -5, 0, -5]
    assert int(outs[0][40]["db_seq"]) == 3500


def test_argument_errors_leave_the_context_usable(gpu):
    from imsame_b200 import api
    db, ds, q, qs = sc.fixed_case(5, 2, 20000, 150, 800, 100, 0.05)
    base = dict(n_threads=4, min_coverage=0.5, min_identity=0.5)
    good, _ = gpu.align((db, ds), (q, qs), api.make_params(**base))
    variants = [dict(min_e_value=1e-10), dict(igap=4), dict(egap=1), dict(n_threads=3), dict(db_total_len_global=len(db) + 10),
                dict(db_pos_base=100), dict(db_seq_base=1)]
    for v in variants:
        a, b = api.make_params(**base), api.make_params(**{**base, **v, "min_identity": 0.9})
        for order in ([a, b], [b, a]):
            with pytest.raises(api.ImsameError) as e:
                gpu.align_sweep((db, ds), (q, qs), order)
            assert e.value.code == -3, v
            out, _ = gpu.align((db, ds), (q, qs), api.make_params(**base))
            assert same(out, good)
    for n in (0, 17):
        with pytest.raises(api.ImsameError) as e:
            gpu.align_sweep((db, ds), (q, qs), [api.make_params(**base)] * n)
        assert e.value.code == -3
    d, k1 = api._seqinfo(db, ds)
    qi, k2 = api._seqinfo(q, qs)
    ps = (api.Params * 2)(api.make_params(**base), api.make_params(**base))
    out = np.zeros(2 * 100, dtype=api.BEST_DTYPE)
    codes = np.zeros(2, dtype=np.int32)
    L = api.lib()
    assert L.imsame_gpu_align_sweep(gpu._h, C.byref(d), C.byref(qi), C.cast(ps, C.c_void_p), 2, None, codes.ctypes.data, None) == -3
    assert L.imsame_gpu_align_sweep(gpu._h, C.byref(d), C.byref(qi), None, 2, out.ctypes.data, codes.ctypes.data, None) == -3
    assert L.imsame_gpu_align_sweep(gpu._h, C.byref(d), C.byref(qi), C.cast(ps, C.c_void_p), 2, out.ctypes.data, None, None) == -3
    out1, _ = gpu.align((db, ds), (q, qs), api.make_params(**base))
    assert same(out1, good) and good["accepted"].sum() > 40
    # after a sweep, the reverse strand has no plain run to repeat
    gpu.align_sweep((db, ds), (q, qs), [api.make_params(**base)])
    with pytest.raises(api.ImsameError) as e:
        gpu.align_revcomp()
    assert e.value.code == -6


# ---- command line -----------------------------------------------------------------------------------
TIMED = re.compile(r"(took|Took|computed in) ")


def untimed(stdout):
    return [l for l in stdout.splitlines() if not TIMED.search(l)]


def run(args, status=0):
    r = subprocess.run([EXE] + args, capture_output=True, text=True)
    assert r.returncode == status, r.stdout[-3000:]
    return r.stdout


def write_fasta(path, seq, start):
    with open(path, "wb") as f:
        for i in range(len(start) - 1):
            f.write(b">r%d\n" % i + bytes(seq[int(start[i]):int(start[i + 1])]) + b"\n")


def summary(stdout):
    found = next(l for l in untimed(stdout) if "from the query were found in the database" in l)
    jac = next(l for l in untimed(stdout) if "The Jaccard-index is" in l)
    return [found, jac]


def check_cli(tmp_path, qf, dbf, entries, n_threads, failing=()):
    """-out and stdout == the run without -sweep plus the entries' lines; <out>.i == a separate run's -out"""
    f, f0 = str(tmp_path / "f.align"), str(tmp_path / "f0.align")
    common = ["-query", qf, "-db", dbf, "-n_threads", str(n_threads), "-coverage", "0.5", "-identity", "0.7"]
    sweep = ",".join(f"{c}:{i}" for c, i in entries)
    both = run(common + ["-out", f, "-sweep", sweep], status=255 if failing else 0)
    plain = run(common + ["-out", f0])
    assert open(f, "rb").read() == open(f0, "rb").read()
    extra = []
    for i, (c, idn) in enumerate(entries, 1):
        extra.append(f"[INFO] Sweep {i} of {len(entries)}: -coverage {c} -identity {idn}")
        g = str(tmp_path / f"g{i}.align")
        if i in failing:
            one = run(["-query", qf, "-db", dbf, "-n_threads", str(n_threads), "-coverage", c, "-identity", idn, "-out", g],
                      status=255)
            assert one.endswith("ERR**** Read size reached for gapped alignment. ****\n")
            extra.append("ERR**** Read size reached for gapped alignment. ****")
            assert os.path.getsize(f"{f}.{i}") == 0
            continue
        one = run(["-query", qf, "-db", dbf, "-n_threads", str(n_threads), "-coverage", c, "-identity", idn, "-out", g])
        assert open(f"{f}.{i}", "rb").read() == open(g, "rb").read(), i
        extra += summary(one)
    want = untimed(plain)
    at = next(i for i, l in enumerate(want) if "The Jaccard-index is" in l) + 1
    assert untimed(both) == want[:at] + extra + want[at:]
    # without -out: the same lines, no file
    d = tmp_path / "noout"
    d.mkdir()
    r = subprocess.run([EXE] + common + ["-sweep", sweep], capture_output=True, text=True, cwd=str(d))
    assert r.returncode == (255 if failing else 0) and untimed(r.stdout) == untimed(both) and os.listdir(d) == []
    return [len(hp.parse_align_headers(f"{f}.{i}")) for i in range(1, len(entries) + 1)]


@pytest.mark.parametrize("n_threads", [1, 4])
def test_cli_sweep_files_equal_separate_runs(gpu, tmp_path, n_threads):
    db, ds, q, qs = sc.ragged_case(1212, 3, 40000, 4000, 600, 0.08, lo=30, hi=300)
    dbf, qf = str(tmp_path / "db.fa"), str(tmp_path / "q.fa")
    write_fasta(dbf, db, ds)
    write_fasta(qf, q, qs)
    n = check_cli(tmp_path, qf, dbf, [("0.5", "0.9"), ("0.3", "0.95"), ("0.8", "0.6"), ("0.5", "0.9"), ("1", "0.5")], n_threads)
    assert n[0] == n[3] and min(n) > 20 and len(set(n)) >= 3


def test_cli_sweep_entry_with_read_size_error(gpu, tmp_path):
    """an entry that stops with the read-size error: its line replaces its summary, its file stays empty, the other
    entries are written, exit status 255 at the end"""
    db, ds, q, qs = read_size_case()
    dbf, qf = str(tmp_path / "db.fa"), str(tmp_path / "q.fa")
    write_fasta(dbf, db, ds)
    write_fasta(qf, q, qs)
    n = check_cli(tmp_path, qf, dbf, [("0.5", "0.95"), ("0.5", "0.5"), ("0.5", "0.97")], 4, failing=(1, 3))
    assert n[1] > 100
