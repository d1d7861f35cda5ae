"""GPU: the reverse strand of the resident database (imsame_gpu_db_revcomp, imsame_gpu_align_revcomp, IMSAME -out_rev)
against what the reference workflow computes for it: bin/revComp's text parsed as a database, aligned by the library,
by the oracle and by a second bin/IMSAME process.  The databases hold reads of both strands (every second read
reverse complemented), so that the forward and the reverse records are both plentiful."""
import os
import re
import subprocess

import numpy as np
import pytest

import helpers as hp
import synth_cases as sc

pytestmark = pytest.mark.gpu
G = os.path.join(hp.ROOT, "tests", "golden")
EXE = os.path.join(hp.ROOT, "bin", "IMSAME")
REVCOMP = os.path.join(hp.ROOT, "bin", "revComp")
COMP = np.arange(256, dtype=np.uint8)
for _a, _b in zip(b"ACGT", b"TGCA"):
    COMP[_a] = _b


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def records(out):
    return {int(r): (int(o["db_seq"]), int(o["qpos_end"]), int(o["db_pos"]), int(o["length"]), int(o["identities"]))
            for r, o in enumerate(out) if o["accepted"]}


def mixed_strands(seq, start):
    """every second read reverse complemented (vectorised: 32-bit indices, databases of up to 2^32 bases)"""
    seq = np.asarray(seq, dtype=np.uint8)
    start = np.asarray(start, dtype=np.int64)
    lens = np.diff(start)
    rid = np.repeat(np.arange(len(lens), dtype=np.uint32), lens)
    idx = np.arange(len(seq), dtype=np.uint32)
    flip = (rid & 1) == 1
    s, e = start[:-1].astype(np.uint32), start[1:].astype(np.uint32)
    idx[flip] = s[rid[flip]] + e[rid[flip]] - 1 - idx[flip]
    out = seq[idx]
    out[flip] = COMP[out[flip]]
    return out


def mirror(seq, start, brk=()):
    """what revComp + the loader give when the mirror rule holds: bases reversed and complemented, offsets and breaks
    mirrored (a break at base 0 would mirror onto the end, where none can be)"""
    total = len(seq)
    b = np.asarray(brk, dtype=np.int64)
    return (COMP[np.asarray(seq)[::-1]].copy(), (total - np.asarray(start, dtype=np.int64)[::-1]).astype(np.uint64),
            np.sort(total - b[b > 0]).astype(np.uint64))


def write_reads(path, reads, n_every=0, rng=None):
    """FASTA of byte strings; with n_every, an N run inside every n_every-th read (word breaks, mirror-safe)"""
    with open(path, "wb") as f:
        for i, r in enumerate(reads):
            if n_every and i % n_every == 0 and len(r) > 40:
                at = int(rng.integers(15, len(r) - 15))
                r = r[:at] + b"N" * int(rng.integers(1, 4)) + r[at:]
            f.write(b">d%d\n" % i + r + b"\n")


def fasta_case(tmp_path, seed, ragged, n_every=0, nd=4000, nq=500):
    """(db FASTA, query FASTA, bin/revComp's output for the db): reads of both strands, forward-strand queries"""
    from imsame_b200 import hostlib as H
    if ragged:
        db, ds, q, qs = sc.ragged_case(seed, 3, 40000, nd, nq, 0.05, lo=20, hi=400)
    else:
        db, ds, q, qs = sc.fixed_case(seed, 3, 40000, 250, nd, nq, 0.05)
    db = mixed_strands(db, ds)
    rng = np.random.default_rng(seed)
    dbf, qf, rf = (str(tmp_path / n) for n in ("db.fa", "q.fa", "db.r.fa"))
    write_reads(dbf, [bytes(db[int(ds[i]):int(ds[i + 1])]) for i in range(len(ds) - 1)], n_every, rng)
    write_reads(qf, [bytes(q[int(qs[i]):int(qs[i + 1])]) for i in range(len(qs) - 1)])
    subprocess.check_call([REVCOMP, dbf, rf], stdout=subprocess.DEVNULL)
    assert H.revcomp_is_mirror(open(dbf, "rb").read())
    return dbf, qf, rf


@pytest.mark.parametrize("case", ["fixed250", "ragged_n_breaks", "phantom_t3", "two_pass", "kmer10"])
def test_align_revcomp_equals_the_reverse_text(gpu, case, tmp_path):
    """align(db) then align_revcomp() == align(parse of revComp's text) == the oracle on that text"""
    from imsame_b200 import api, hostlib as H
    ragged = case != "fixed250"
    dbf, qf, rf = fasta_case(tmp_path, {"fixed250": 11, "ragged_n_breaks": 12, "phantom_t3": 13, "two_pass": 14, "kmer10": 15}[case],
                             ragged, n_every=5 if ragged else 0)
    seq, start, brk = H.load_fasta(dbf, True)
    q, qs, _ = H.load_fasta(qf, False)
    rseq, rstart, rbrk = H.load_fasta(rf, True)
    assert len(brk) > 100 or not ragged
    if case == "ragged_n_breaks":
        # breaks at read starts change no word: one at base 0 (the first segment's start, dropped by the mirror) and
        # some at other read starts (mirrored onto read starts)
        brk = np.unique(np.concatenate([brk, [0], start[3:400:9]])).astype(np.uint64)
    n_threads = 3 if case == "phantom_t3" else 4
    k = 10 if case == "kmer10" else 12
    p = api.make_params(n_threads=n_threads)
    try:
        gpu.set_kmer(k)
        gpu.set_passes(2 if case == "two_pass" else 0)
        fwd, st_f = gpu.align((seq, start), (q, qs), p, db_breaks=brk)
        rev, st_r = gpu.align_revcomp()
        assert st_r["h2d_bytes"] == 0  # nothing uploaded: the database was resident
        if case == "two_pass":
            assert st_f["scan_passes"] == 2 and st_r["scan_passes"] == 2
        mseq, mstart, mbrk = mirror(seq, start, brk)
        want, _ = gpu.align((mseq, mstart), (q, qs), p, db_breaks=mbrk)
        assert np.array_equal(rev, want)
        if case != "ragged_n_breaks":
            assert np.array_equal(mseq, rseq) and np.array_equal(mstart, rstart) and np.array_equal(mbrk, rbrk)
        orc, _ = hp.oracle_align(hp.OracleSeqs(rf, True), hp.OracleSeqs(qf, False), hp.default_params(n_threads=n_threads, k=k))
        assert records(rev) == hp.best_to_records(orc, len(qs) - 1)
        nq = len(qs) - 1
        assert rev["accepted"].sum() > nq // 10 and fwd["accepted"].sum() > nq // 10
    finally:
        gpu.set_kmer(12)
        gpu.set_passes(0)


def test_multi_segment_database(gpu):
    """a database of more than one segment (2^29 bases), shaped like test_ragged_multi_segment_sampled_against_oracle:
    records equal align(mirror) in full and the index-free oracle on 1 000 sampled reads"""
    from imsame_b200 import api
    db, ds, q, qs = sc.ragged_case(4243, 300, 1000000, 3_000_000, 30000, 0.04, lo=30, hi=400)
    assert len(db) > (1 << 29)
    db = mixed_strands(db, ds)
    p = api.make_params(n_threads=4)
    gpu.align((db, ds), (q, qs), p)
    rev, st = gpu.align_revcomp()
    assert st["k2_launches"] >= 2
    mseq, mstart, _ = mirror(db, ds)
    del db
    want, _ = gpu.align((mseq, mstart), (q, qs), p)
    assert np.array_equal(rev, want) and rev["accepted"].sum() > 3000
    reads = np.sort(np.random.default_rng(8).choice(len(qs) - 1, 1000, replace=False))
    orc, _ = hp.oracle_align_sampled(hp.OracleSeqs(seq=mseq, start=mstart), hp.OracleSeqs(seq=q, start=qs),
                                     hp.default_params(n_threads=4), reads)
    got = {r: v for r, v in records(rev).items() if r in set(reads.tolist())}
    assert got == orc and len(orc) > 100


def test_staged_db_revcomp_is_an_involution(gpu):
    """set_query, set_db, run, db_revcomp, run, db_revcomp, run: the second run is the reverse strand's, the third
    the first again"""
    from imsame_b200 import api
    db, ds, q, qs = sc.ragged_case(77, 3, 40000, 3000, 400, 0.05, lo=20, hi=400)
    db = mixed_strands(db, ds)
    rng = np.random.default_rng(77)
    brk = np.unique(np.concatenate([rng.integers(1, len(db), size=300), [0], ds[5:300:11]])).astype(np.uint64)
    p = api.make_params(n_threads=4)
    gpu.set_query((q, qs), p)
    gpu.set_db((db, ds), db_breaks=brk)
    gpu.run(p)
    first = gpu.fetch()
    gpu.db_revcomp()
    gpu.run(p)
    second = gpu.fetch()
    gpu.db_revcomp()
    gpu.run(p)
    third = gpu.fetch()
    mseq, mstart, mbrk = mirror(db, ds, brk)
    want, _ = gpu.align((mseq, mstart), (q, qs), p, db_breaks=mbrk)
    assert np.array_equal(second, want) and want["accepted"].sum() > 40
    assert np.array_equal(third, first) and first["accepted"].sum() > 40


def test_error_states(gpu):
    from imsame_b200 import api
    db, ds, q, qs = sc.fixed_case(5, 2, 20000, 150, 800, 100, 0.05)
    fresh = api.Imsame(0)
    try:
        for call in (lambda: fresh.align_revcomp(), lambda: fresh.db_revcomp()):
            with pytest.raises(api.ImsameError) as e:
                call()
            assert e.value.code == -6
        # after align_samples: the database is a sample's
        s_db, s_q = fresh.sample((db, ds)), fresh.sample((q, qs))
        fresh.align_samples(s_db, s_q)
        for call in (lambda: fresh.align_revcomp(), lambda: fresh.db_revcomp()):
            with pytest.raises(api.ImsameError) as e:
                call()
            assert e.value.code == -6
        s_db.free(); s_q.free()
        # after a failed align (an empty query read)
        fresh.align((db, ds), (q, qs))
        fresh.align_revcomp()
        bad = qs.copy()
        bad[1] = bad[0]
        with pytest.raises(api.ImsameError):
            fresh.align((db, ds), (q, bad))
        with pytest.raises(api.ImsameError) as e:
            fresh.align_revcomp()
        assert e.value.code == -6
        # a shard of an unknown whole database
        fresh.align((db, ds), (q, qs), api.make_params(db_pos_base=1000, db_seq_base=10, db_total_len_global=len(db) + 1000))
        with pytest.raises(api.ImsameError) as e:
            fresh.align_revcomp()
        assert e.value.code == -3
    finally:
        fresh.close()


# ---- command line -----------------------------------------------------------------------------------
TIMED = re.compile(r"(took|Took|computed in) ")


def untimed(stdout):
    return [l for l in stdout.splitlines() if not TIMED.search(l)]


def run(args):
    r = subprocess.run([EXE] + args, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:]
    return r.stdout


def check_cli(tmp_path, qf, dbf, flags, n_threads, gpus=1, oracle=False):
    """-out_rev == revComp + a second IMSAME, byte for byte; -out and stdout == the run without the flag + two lines"""
    f, r, f0, r2, dr = (str(tmp_path / n) for n in ("f.align", "r.align", "f0.align", "r2.align", "db.r.fa"))
    common = ["-query", qf, "-n_threads", str(n_threads), "-gpus", str(gpus)] + flags
    both = run(common + ["-db", dbf, "-out", f, "-out_rev", r])
    plain = run(common + ["-db", dbf, "-out", f0])
    subprocess.check_call([REVCOMP, dbf, dr], stdout=subprocess.DEVNULL)
    second = run(common + ["-db", dr, "-out", r2])
    assert open(f, "rb").read() == open(f0, "rb").read()
    assert open(r, "rb").read() == open(r2, "rb").read()
    got, want = untimed(both), untimed(plain)
    at = next(i for i, l in enumerate(want) if "The Jaccard-index is" in l) + 1
    found = next(l for l in untimed(second) if "from the query were found in the database" in l)
    jac = next(l for l in untimed(second) if "The Jaccard-index is" in l)
    extra = [found.replace("found in the database", "found in the reverse complement of the database"),
             jac.replace("The Jaccard-index is", "The Jaccard-index against the reverse complement is")]
    assert got == want[:at] + extra + want[at:]
    if oracle:
        o = str(tmp_path / "orc.align")
        hp.oracle_align(hp.OracleSeqs(dr, True), hp.OracleSeqs(qf, False), hp.default_params(n_threads=1), out_path=o)
        assert open(r, "rb").read() == open(o, "rb").read()
    return len(hp.parse_align_headers(f)), len(hp.parse_align_headers(r))


@pytest.mark.parametrize("n_threads", [1, 4])
def test_cli_out_rev_mirror_safe_database(gpu, tmp_path, n_threads):
    dbf, qf, _ = fasta_case(tmp_path, 21, True, n_every=4, nd=6000, nq=600)
    nf, nr = check_cli(tmp_path, qf, dbf, [], n_threads, oracle=n_threads == 1)
    assert nf > 100 and nr > 100


@pytest.mark.parametrize("which", ["dirty", "s1", "s2"])
def test_cli_out_rev_non_mirror_database(gpu, tmp_path, which):
    """databases whose revComp text is not their mirror image (CRLF multi-line records, gap characters, U): the
    reverse parse is uploaded"""
    from imsame_b200 import hostlib as H
    if which == "dirty":
        qf, dbf = os.path.join(G, "dirty.q.fa"), os.path.join(G, "dirty.db.fa")
        flags = ["-coverage", "0.3", "-identity", "0.6", "-evalue", "1e-10", "-igap", "4", "-egap", "1"]
    else:
        d = tmp_path / "samples"
        d.mkdir()
        sc.write_allvsall_filter_samples(d)
        qf, dbf, flags = str(d / "s0.fasta"), str(d / f"{which}.fasta"), ["-coverage", "0.5", "-identity", "0.5"]
    assert not H.revcomp_is_mirror(open(dbf, "rb").read())
    for t in (1, 4):
        nf, nr = check_cli(tmp_path, qf, dbf, flags, t, oracle=t == 1)
    if which != "dirty":  # (dirty's query has no reverse-strand reads: the file is empty, like the second process's)
        assert nr > 100


# ---- two GPUs -----------------------------------------------------------------------------------------
@pytest.mark.skipif(_n_gpus() < 2, reason="needs two GPUs")
def test_two_gpus_align_revcomp_equals_one(gpu):
    """align_revcomp over 2 contexts (each shard more than one segment) == the single-GPU records"""
    from imsame_b200 import api
    L, nd = 250, 4_400_000
    db, ds, q, qs = sc.fixed_case(91, 200, 1000000, L, nd, 20000, 0.04)
    assert len(db) > 2 * (1 << 29)
    db = mixed_strands(db, ds)
    p = api.make_params(n_threads=4)
    gpu.align((db, ds), (q, qs), p)
    want, _ = gpu.align_revcomp()
    c1 = api.Imsame(1)
    try:
        api.align_sharded([gpu, c1], (db, ds), (q, qs), p)
        assert gpu.n_segments() >= 2 and c1.n_segments() >= 2
        got, st = api.align_revcomp([gpu, c1])
        assert np.array_equal(got, want) and want["accepted"].sum() > 1000
        assert all(s["ms_comm"] > 0 for s in st)
    finally:
        gpu.comm_free()
        c1.close()


@pytest.mark.skipif(_n_gpus() < 2, reason="needs two GPUs")
def test_two_gpus_cli_out_rev(gpu, tmp_path):
    dbf, qf, _ = fasta_case(tmp_path, 31, True, n_every=4, nd=6000, nq=600)
    r1, r2 = str(tmp_path / "r1.align"), str(tmp_path / "r2.align")
    for g, r in ((1, r1), (2, r2)):
        run(["-query", qf, "-db", dbf, "-out", str(tmp_path / "f.align"), "-out_rev", r, "-gpus", str(g), "-n_threads", "1"])
    assert open(r1, "rb").read() == open(r2, "rb").read() and os.path.getsize(r1) > 10000
