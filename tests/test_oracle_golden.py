"""The oracle (CPU restatement) against golden vectors produced by the unmodified reference
(tests/golden/make_golden.py).  Runs anywhere: needs neither /root/reference nor a GPU."""
import os

import pytest

import helpers as hp

G = os.path.join(hp.ROOT, "tests", "golden")
CASES = {
    "synth150": dict(),
    "dirty": dict(coverage=0.3, identity=0.6, evalue=1e-10, igap=4, egap=1),
    # 3 query reads against synth150's database: -n_threads 4 > n_seqs, explicit -evalue 1e-20 (double, not the default's long double)
    "few": dict(evalue=1e-20),
}
DB_OF = {"few": "synth150"}


def db_path(name):
    return os.path.join(G, f"{DB_OF.get(name, name)}.db.fa")


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_t1_bytes_equal_reference(name, tmp_path):
    db = hp.OracleSeqs(db_path(name), True)
    q = hp.OracleSeqs(os.path.join(G, f"{name}.q.fa"), False)
    out = str(tmp_path / "o.align")
    best, st = hp.oracle_align(db, q, hp.default_params(n_threads=1, **CASES[name]), out_path=out)
    assert open(out, "rb").read() == open(os.path.join(G, f"{name}.t1.align"), "rb").read()
    want = open(os.path.join(G, f"{name}.stdout")).read()
    assert f"[INFO] {st.accepted} reads ({q.s.n_seqs}) from the query were found in the database ({db.s.n_seqs})" in want


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_t4_headers_equal_reference(name, tmp_path):
    """-n_threads changes which reads see the cross-read 'phantom' word (SURVEY fact 5)"""
    db = hp.OracleSeqs(db_path(name), True)
    q = hp.OracleSeqs(os.path.join(G, f"{name}.q.fa"), False)
    out = str(tmp_path / "o.align")
    hp.oracle_align(db, q, hp.default_params(n_threads=4, **CASES[name]), out_path=out)
    got = sorted(l for l in open(out, "rb").read().split(b"\n") if hp.HEADER_RE.match(l))
    want = [l for l in open(os.path.join(G, f"{name}.t4.headers"), "rb").read().split(b"\n") if l]
    assert got == want


@pytest.mark.parametrize("name", sorted(CASES))
@pytest.mark.parametrize("n_threads", [1, 3, 4])
def test_bulk_min_key_form_equals_scan_order(name, n_threads):
    """winner(read) = argmin (k-mer end asc, db pos desc) over accepted candidates == first accepted"""
    db = hp.OracleSeqs(db_path(name), True)
    q = hp.OracleSeqs(os.path.join(G, f"{name}.q.fa"), False)
    p = hp.default_params(n_threads=n_threads, **CASES[name])
    a, _ = hp.oracle_align(db, q, p)
    b, _ = hp.oracle_align(db, q, p, bulk=True)
    nq = int(q.s.n_seqs)
    assert hp.best_to_records(a, nq) == hp.best_to_records(b, nq)
    assert len(hp.best_to_records(a, nq)) > (5 if nq > 5 else 1)


LIVE_CASES = [(1001, 0.03, 1), (7, 0.10, 4), (99, 0.20, 8)]


def live_case(seed, div, n_threads, d):
    """seeded inputs of test_oracle_vs_live_reference and the oracle's .align file on them"""
    from imsame_b200 import hostlib as H
    pool = H.SynthPool(seed, 3, 60000)
    nd, nq, L = 6000, 600, 150
    dbf, qf, orc_out = (os.path.join(d, n) for n in ("db.fa", "q.fa", "orc.align"))
    H.write_fasta(dbf, pool.db_reads(0, nd, L), nd, L, "d")
    H.write_fasta(qf, pool.query_reads(0, nq, L, div), nq, L, "q")
    pool.close()
    db, q = hp.OracleSeqs(dbf, True), hp.OracleSeqs(qf, False)
    hp.oracle_align(db, q, hp.default_params(n_threads=n_threads), out_path=orc_out)
    return dbf, qf, orc_out


@pytest.mark.parametrize("seed,div,n_threads", LIVE_CASES)
def test_oracle_vs_live_reference(seed, div, n_threads, tmp_path):
    """fresh seeded inputs through the real reference binary where oracle/_ref is built; its output on them is
    pinned in tests/golden/reference_pins.json"""
    dbf, qf, orc_out = live_case(seed, div, n_threads, str(tmp_path))
    if hp.have_reference():
        ref_out = str(tmp_path / "ref.align")
        hp.run_reference(qf, dbf, ref_out, n_threads=n_threads)
        if n_threads == 1:
            assert open(ref_out, "rb").read() == open(orc_out, "rb").read()
        assert hp.parse_align_headers(ref_out) == hp.parse_align_headers(orc_out)
    got = hp.align_digest(orc_out, whole=n_threads == 1)
    assert got == hp.pins("oracle_vs_live_reference")[f"{seed}/{div}/{n_threads}"]
    assert got["records"] > 100


@pytest.mark.parametrize("k", [8, 10, 14])
def test_generalised_seed_length_forms_agree(k):
    """k != 12 has no reference (FIXED_K is compiled in, src/structs.h:15): the oracle generalised to
    FIXED_K = k is only checked for self-consistency -- scan order with early exit == order-free min-key
    form -- and is pinned to the reference at k = 12 by the tests above"""
    db = hp.OracleSeqs(os.path.join(G, "dirty.db.fa"), True)
    q = hp.OracleSeqs(os.path.join(G, "dirty.q.fa"), False)
    p = hp.default_params(n_threads=3, evalue=1e-10, coverage=0.3, identity=0.6, igap=4, egap=1, k=k)
    seq, st1 = hp.oracle_align(db, q, p)
    bulk, st2 = hp.oracle_align(db, q, p, bulk=True)
    nq = int(q.s.n_seqs)
    assert hp.best_to_records(seq, nq) == hp.best_to_records(bulk, nq)
    assert st2.hits >= st1.hits > 0


@pytest.mark.parametrize("name", sorted(CASES))
@pytest.mark.parametrize("n_threads", [1, 4])
def test_sampled_checker_equals_scan_order(name, n_threads):
    """the index-free per-read checker (oracle/imsame_sampled.c, used on inputs the reference's index cannot
    hold) gives exactly the scan-order result, for every read and for a subset"""
    import numpy as np
    db = hp.OracleSeqs(db_path(name), True)
    q = hp.OracleSeqs(os.path.join(G, f"{name}.q.fa"), False)
    p = hp.default_params(n_threads=n_threads, **CASES[name])
    want = hp.best_to_records(hp.oracle_align(db, q, p)[0], int(q.s.n_seqs))
    nq = int(q.s.n_seqs)
    got, st = hp.oracle_align_sampled(db, q, p, np.arange(nq))
    assert got == want
    sub = np.arange(nq)[::3][::-1]
    got, _ = hp.oracle_align_sampled(db, q, p, sub)
    assert got == {r: v for r, v in want.items() if r in set(int(x) for x in sub)}


def test_sampled_checker_on_shards_reduces_to_whole():
    """per-shard results with global coordinates: the smallest (qpos_end, -db_pos) is the whole-database result"""
    import numpy as np
    import synth_cases as sc
    db, ds, q, qs = sc.ragged_case(77, 3, 40000, 5000, 400, 0.05, lo=40, hi=260)
    nd, nq = len(ds) - 1, len(qs) - 1
    p = hp.default_params(n_threads=4)
    whole = hp.best_to_records(hp.oracle_align(hp.OracleSeqs(seq=db, start=ds), hp.OracleSeqs(seq=q, start=qs), p)[0], nq)
    assert len(whole) > 50
    reads = np.arange(nq)
    merged = {}
    Q = hp.OracleSeqs(seq=q, start=qs)
    for lo, hi in ((0, nd // 3), (nd // 3, nd)):
        b0, b1 = int(ds[lo]), int(ds[hi])
        ps = hp.default_params(n_threads=4, db_total_len_global=len(db))
        got, _ = hp.oracle_align_sampled(hp.OracleSeqs(seq=db[b0:b1], start=ds[lo:hi + 1] - ds[lo]), Q, ps, reads,
                                         db_pos_base=b0, db_seq_base=lo)
        for r, v in got.items():
            if r not in merged or (v[1], -v[2]) < (merged[r][1], -merged[r][2]):
                merged[r] = v
    assert merged == whole
