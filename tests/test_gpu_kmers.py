"""GPU: several seed lengths in one call (imsame_gpu_align_kmers, IMSAME -kmers).  Every entry's records must equal, field
by field, a separate set_kmer(k) + align on the same context, and the oracle generalised to FIXED_K = k; the counters
that do not depend on the pair-result cache must equal the separate run's; the command line's entry files and summary
lines must equal those of separate -kmer runs."""
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
SAME_COUNTERS = ("n_query_kmers", "n_db_kmers", "n_hits", "n_evalue_pass", "n_pairs", "n_accepted", "scan_passes")


def records(out):
    return {int(r): (int(o["db_seq"]), int(o["qpos_end"]), int(o["db_pos"]), int(o["length"]), int(o["identities"]))
            for r, o in enumerate(out) if o["accepted"]}


def same(a, b):
    return all(np.array_equal(a[f], b[f]) for f in FIELDS)


def separate(gpu, db, ds, q, qs, k, params, breaks=None):
    """set_kmer(k) + align on the same context: (records, code, stats); the context's seed length is put back"""
    from imsame_b200 import api
    try:
        gpu.set_kmer(k)
        out, st = gpu.align((db, ds), (q, qs), params, db_breaks=breaks)
        return out, 0, st
    except api.ImsameError as e:
        return None, e.code, None
    finally:
        gpu.set_kmer(12)


def kmers_vs_separate(gpu, db, ds, q, qs, ks, n_threads=4, breaks=None, oracle_ks=(), **pkw):
    """align_kmers against separate runs at every k (records, codes, counters) and, for oracle_ks, the oracle;
    returns (outs, codes, kmers stats, separate stats)"""
    from imsame_b200 import api
    p = api.make_params(n_threads=n_threads, **pkw)
    outs, codes, sts = gpu.align_kmers((db, ds), (q, qs), ks, p, db_breaks=breaks)
    seps = []
    for t, k in enumerate(ks):
        want, code, st = separate(gpu, db, ds, q, qs, k, p, breaks)
        assert codes[t] == code, (k, codes)
        if code:
            assert not outs[t]["accepted"].any() and sts[t]["n_pairs"] == 0, k
        else:
            assert same(outs[t], want), k
            for c in SAME_COUNTERS:
                assert sts[t][c] == st[c], (k, c, sts[t][c], st[c])
        seps.append(st)
    for k in oracle_ks:
        t = list(ks).index(k)
        best, _ = hp.oracle_align(hp.OracleSeqs(seq=db, start=ds, brk=breaks), hp.OracleSeqs(seq=q, start=qs),
                                  hp.default_params(n_threads=n_threads, k=k, evalue=pkw.get("min_e_value")))
        assert records(outs[t]) == hp.best_to_records(best, len(qs) - 1), k
    return outs, codes, sts, seps


def dp_ratio(sts, seps):
    got, want = sum(s["n_pairs_dp"] for s in sts), sum(s["n_pairs_dp"] for s in seps)
    print(f"pairs aligned: one call {got}, separate runs {want}, ratio {got / max(want, 1):.3f}")
    return got, want


@pytest.mark.parametrize("ks", [[8, 10, 12, 14], [14, 12, 10, 8]])
def test_fixed_length_reads_in_both_orders(gpu, ks):
    """cfg5's shape at test size; the seed lengths share most of their pairs: fewer pairs run through NW"""
    db, ds, q, qs = sc.fixed_case(5005, 4, 100000, 150, 20000, 1500, 0.10)
    outs, codes, sts, seps = kmers_vs_separate(gpu, db, ds, q, qs, ks, oracle_ks=(8, 10, 14) if ks[0] == 8 else ())
    assert codes == [0] * len(ks) and min(int(o["accepted"].sum()) for o in outs) > 300
    got, want = dp_ratio(sts, seps)
    assert got < want


def test_ragged_reads_and_both_nw_kernels(gpu):
    """query reads of 30-400 bases: the packed-word and the generic kernel share the bins pair by pair"""
    db, ds, q, qs = sc.ragged_case(808, 3, 60000, 6000, 900, 0.06, lo=30, hi=400)
    _, _, sts, seps = kmers_vs_separate(gpu, db, ds, q, qs, [10, 13, 7, 12])
    assert all(0 < s["k3_packed_launches"] < s["k3_launches"] for s in sts[:1])
    got, want = dp_ratio(sts, seps)
    assert got < want


def test_word_breaks(gpu):
    db, ds, q, qs = sc.ragged_case(4242, 2, 30000, 2500, 400, 0.05, lo=20, hi=300)
    rng = np.random.default_rng(7)
    brk = np.unique(rng.integers(1, len(db), size=500)).astype(np.uint64)
    brk = np.array([b for b in brk if b not in set(ds.tolist())], dtype=np.uint64)
    kmers_vs_separate(gpu, db, ds, q, qs, [12, 9, 11], n_threads=3, breaks=brk, oracle_ks=(9, 11), min_e_value=1e-8)


@pytest.mark.parametrize("passes", [1, 2])
def test_forced_scan_plans(gpu, passes):
    """one pass with every word, and early words first (two scans per entry; the late pass reuses the cache too)"""
    db, ds, q, qs = sc.fixed_case(3001, 3, 60000, 300, 5000, 800, 0.05)
    try:
        gpu.set_passes(passes)
        _, _, sts, seps = kmers_vs_separate(gpu, db, ds, q, qs, [12, 10, 14])
        assert [s["scan_passes"] for s in sts] == [passes] * 3
    finally:
        gpu.set_passes(0)
    dp_ratio(sts, seps)


def test_generic_nw_kernel_only(gpu):
    db, ds, q, qs = sc.ragged_case(611, 3, 40000, 3000, 500, 0.08, lo=30, hi=300)
    try:
        gpu.set_nw_mode(1)
        _, _, sts, _ = kmers_vs_separate(gpu, db, ds, q, qs, [11, 12, 9])
        assert all(s["k3_packed_launches"] == 0 for s in sts)
    finally:
        gpu.set_nw_mode(0)


def test_read_size_stop_per_entry_and_the_largest_seed_length(gpu):
    """query read 40 is a piece of a 5 000-base database read; a copy with every 15th base changed sits later in the
    database, where the scan order reaches it first -- when the seed length finds it at all (runs of 14 equal bases):
    k = 16 stops with the read-size error, the other entries are complete.  The only test with k = 16 (a 34 GB word
    table), on a 300-read query."""
    from test_gpu_sweep import read_size_case
    db, ds, q, qs = read_size_case()
    outs, codes, _, _ = kmers_vs_separate(gpu, db, ds, q, qs, [12, 16, 8])
    assert codes[1] == -5 and codes[0] == codes[2] == 0
    assert int(outs[0][40]["db_seq"]) == 3500


def test_argument_errors_and_context_state(gpu):
    """argument errors leave the context usable with its own seed length; afterwards the reverse strand has no
    plain run to repeat"""
    from imsame_b200 import api
    db, ds, q, qs = sc.fixed_case(5, 2, 20000, 150, 800, 100, 0.05)
    p = api.make_params(n_threads=4)
    try:
        gpu.set_kmer(10)
        want10, _ = gpu.align((db, ds), (q, qs), p)
        assert want10["accepted"].sum() > 40
        for ks in ([], list(range(4, 17)) + [8], [3], [17], [8, 12, 8], [0], [12, 12]):
            with pytest.raises(api.ImsameError) as e:
                gpu.align_kmers((db, ds), (q, qs), ks, p)
            assert e.value.code == -3, ks
            out, _ = gpu.align((db, ds), (q, qs), p)
            assert same(out, want10), ks
        d, k1 = api._seqinfo(db, ds)
        qi, k2 = api._seqinfo(q, qs)
        ks = np.array([8, 12], dtype=np.int32)
        out = np.zeros(2 * 100, dtype=api.BEST_DTYPE)
        codes = np.zeros(2, dtype=np.int32)
        L = api.lib()
        assert L.imsame_gpu_align_kmers(gpu._h, C.byref(d), C.byref(qi), C.byref(p), 2, ks.ctypes.data, None,
                                        codes.ctypes.data, None) == -3
        assert L.imsame_gpu_align_kmers(gpu._h, C.byref(d), C.byref(qi), C.byref(p), 2, ks.ctypes.data, out.ctypes.data,
                                        None, None) == -3
        assert L.imsame_gpu_align_kmers(gpu._h, C.byref(d), C.byref(qi), C.byref(p), 2, None, out.ctypes.data,
                                        codes.ctypes.data, None) == -3
        # every k 4..16 once is the limit (k = 16 itself is left to the read-size test)
        assert L.imsame_gpu_align_kmers(gpu._h, C.byref(d), C.byref(qi), C.byref(p), 14,
                                        np.arange(4, 18, dtype=np.int32).ctypes.data, out.ctypes.data, codes.ctypes.data,
                                        None) == -3
        outs, codes2, _ = gpu.align_kmers((db, ds), (q, qs), [8, 12], p)
        assert codes2 == [0, 0]
        out, _ = gpu.align((db, ds), (q, qs), p)
        assert same(out, want10)
        gpu.align_kmers((db, ds), (q, qs), [10], p)
        with pytest.raises(api.ImsameError) as e:
            gpu.align_revcomp()
        assert e.value.code == -6
    finally:
        gpu.set_kmer(12)


def test_failed_allocations_leave_the_context_usable(gpu, monkeypatch):
    """IMSAME_TEST_FAIL_ALLOC=N makes device allocation N of a new context fail as on a full device: every failure is
    IMSAME_ENOMEM and the same context then returns the right blocks"""
    from imsame_b200 import api
    db, ds, q, qs = sc.fixed_case(1001, 2, 50000, 150, 4000, 500, 0.03)
    ks = [12, 9, 14]
    p = api.make_params(n_threads=4)
    want, _, _ = gpu.align_kmers((db, ds), (q, qs), ks, p)
    failures, quiet = [], 0
    for n in range(1, 200):
        monkeypatch.setenv("IMSAME_TEST_FAIL_ALLOC", str(n))
        ctx = api.Imsame(0)  # reads the hook
        failed = []
        try:
            for name in ("kmers", "kmers again"):
                try:
                    outs, codes, _ = ctx.align_kmers((db, ds), (q, qs), ks, p)
                except api.ImsameError as e:
                    assert e.code == -4, (n, name, e)  # IMSAME_ENOMEM
                    failed.append(name)
                    outs, codes, _ = ctx.align_kmers((db, ds), (q, qs), ks, p)
                assert codes == [0, 0, 0] and all(same(outs[t], want[t]) for t in range(3)), (n, name)
        finally:
            ctx.close()
        failures += [(n, f) for f in failed]
        quiet = 0 if failed else quiet + 1
        if quiet == 5:
            break
    else:
        pytest.fail("allocations up to 199 still failed")
    assert sum(f == "kmers" for _, f in failures) >= 10, failures


def test_cache_growth(gpu, monkeypatch, capfd):
    """a cache that starts at 256 slots overflows, doubles with its entries moved, and every entry still equals its
    separate run"""
    db, ds, q, qs = sc.fixed_case(5005, 4, 100000, 150, 20000, 1500, 0.10)
    capfd.readouterr()
    monkeypatch.setenv("IMSAME_TEST_KCACHE_SLOTS", "256")
    monkeypatch.setenv("IMSAME_TRACE", "1")
    _, codes, _, _ = kmers_vs_separate(gpu, db, ds, q, qs, [12, 10, 14, 8])
    err = capfd.readouterr().err
    moved = [int(m) for m in re.findall(r"pair cache: \d+ slots, (\d+) entries moved", err)]
    assert len(moved) >= 3 and max(moved) > 0, err[-2000:]
    assert codes == [0] * 4


@pytest.mark.parametrize("passes", [1, 2])
def test_several_database_segments(gpu, monkeypatch, passes):
    """a database cut into segments of 400 000 bases (IMSAME_TEST_SEG_BASES): the scan of a later segment prunes with
    the keys of its reads, so no cached result may lower a key before the last scan of the pass -- n_pairs (in the
    counters compared) is the separate run's"""
    db, ds, q, qs = sc.ragged_case(4243, 3, 200000, 16000, 1500, 0.05, lo=30, hi=300)
    monkeypatch.setenv("IMSAME_TEST_SEG_BASES", "400000")
    try:
        gpu.set_passes(passes)
        _, _, sts, seps = kmers_vs_separate(gpu, db, ds, q, qs, [12, 10, 14, 11])
        assert all(s["k2_launches"] >= 5 * passes for s in sts) and [s["scan_passes"] for s in sts] == [passes] * 4
    finally:
        gpu.set_passes(0)
    got, want = dp_ratio(sts, seps)
    assert got < want


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


def check_cli(tmp_path, qf, dbf, ks, n_threads, extra=(), failing=()):
    """-out and stdout == the run without -kmers plus the entries' lines; <out>.k<K> == a separate -kmer K run's -out"""
    f, f0 = str(tmp_path / "f.align"), str(tmp_path / "f0.align")
    common = ["-query", qf, "-db", dbf, "-n_threads", str(n_threads), *extra]
    both = run(common + ["-out", f, "-kmers", ",".join(map(str, ks))], status=255 if failing else 0)
    plain = run(common + ["-out", f0])
    assert open(f, "rb").read() == open(f0, "rb").read()
    lines, sizes = [], []
    for k in ks:
        lines.append(f"[INFO] Seed length {k}")
        g = str(tmp_path / f"g{k}.align")
        if k in failing:
            one = run(common + ["-kmer", str(k), "-out", g], status=255)
            assert one.endswith("ERR**** Read size reached for gapped alignment. ****\n")
            lines.append("ERR**** Read size reached for gapped alignment. ****")
            assert os.path.getsize(f"{f}.k{k}") == 0
            continue
        one = run(common + ["-kmer", str(k), "-out", g])
        assert open(f"{f}.k{k}", "rb").read() == open(g, "rb").read(), k
        lines += summary(one)
        sizes.append(len(hp.parse_align_headers(g)))
    want = untimed(plain)
    at = next(i for i, l in enumerate(want) if "The Jaccard-index is" in l) + 1
    assert untimed(both) == want[:at] + lines + want[at:]
    return sizes


@pytest.mark.parametrize("n_threads,cigar", [(1, False), (4, False), (1, True), (4, True)])
def test_cli_entry_files_equal_separate_runs(gpu, tmp_path, n_threads, cigar):
    db, ds, q, qs = sc.ragged_case(1212, 3, 40000, 4000, 600, 0.08, lo=30, hi=300)
    dbf, qf = str(tmp_path / "db.fa"), str(tmp_path / "q.fa")
    write_fasta(dbf, db, ds)
    write_fasta(qf, q, qs)
    n = check_cli(tmp_path, qf, dbf, [8, 14, 10], n_threads, extra=["-cigar"] if cigar else [])
    assert cigar or min(n) > 20  # (the header parser reads files without the -cigar columns)


def test_cli_entry_with_read_size_error(gpu, tmp_path):
    """an entry that stops with the read-size error: its line replaces its summary, its file stays empty, the other
    entries are written, exit status 255 at the end"""
    from test_gpu_sweep import read_size_case
    db, ds, q, qs = read_size_case()
    dbf, qf = str(tmp_path / "db.fa"), str(tmp_path / "q.fa")
    write_fasta(dbf, db, ds)
    write_fasta(qf, q, qs)
    n = check_cli(tmp_path, qf, dbf, [8, 15, 10], 4, failing=(15,))
    assert min(n) > 100
