"""GPU: several coverage/identity threshold sets in one run on read sets resident on the device
(imsame_gpu_align_samples_sweep).  Every set's records must equal, field by field, imsame_gpu_align_samples with that
set's parameters and imsame_gpu_align_sweep from host buffers, and the oracle where the size allows; the context and
both samples stay usable after every error."""
import numpy as np
import pytest

import helpers as hp
import synth_cases as sc
from test_gpu_sweep import CFG5_SETS, read_size_case, records, same

pytestmark = pytest.mark.gpu
SIXTEEN = [(c, i) for c in (0.3, 0.5, 0.8, 1.0) for i in (0.95, 0.6, 0.85, 0.5)]


def _revcomp_reads(seq, start, brk=None):
    """what revComp + the loader give for A/C/G/T-only reads (and what imsame_gpu_sample_revcomp makes): the whole
    concatenated array reversed and complemented, offsets and word breaks mirrored"""
    comp = np.zeros(256, dtype=np.uint8)
    for a, b in zip(b"ACGT", b"TGCA"):
        comp[a] = b
    rstart = (len(seq) - np.asarray(start, dtype=np.int64)[::-1]).astype(np.uint64)
    rbrk = None if brk is None else np.sort(len(seq) - brk.astype(np.int64)).astype(np.uint64)
    return comp[seq[::-1]].copy(), rstart, rbrk


def word_breaks(db, ds, seed, n):
    rng = np.random.default_rng(seed)
    starts = set(int(x) for x in ds)
    return np.array([b for b in np.unique(rng.integers(1, len(db), size=n)) if int(b) not in starts], dtype=np.uint64)


def samples_sweep_vs(gpu, db, ds, q, qs, sets, brk=None, rev=False, oracle=False, k=12, n_threads=4):
    """align_samples_sweep against align_samples of every set and against align_sweep from host buffers (and the
    oracle); rev: the database is the device reverse complement of the sample made from (db, ds, brk)"""
    from imsame_b200 import api
    ps = [api.make_params(n_threads=n_threads, min_coverage=c, min_identity=i) for c, i in sets]
    hdb, hds, hbrk = _revcomp_reads(db, ds, brk) if rev else (db, ds, brk)
    s_fwd, s_q = gpu.sample((db, ds), brk), gpu.sample((q, qs))
    s_db = gpu.sample_revcomp(s_fwd) if rev else s_fwd
    try:
        outs, codes, st = gpu.align_samples_sweep(s_db, s_q, ps)
        assert codes == [0] * len(sets)
        assert st["n_accepted"] == int(outs[0]["accepted"].sum())
        for t, p in enumerate(ps):
            want, _ = gpu.align_samples(s_db, s_q, p)
            assert same(outs[t], want), (t, sets[t])
        host, hcodes, _ = gpu.align_sweep((hdb, hds), (q, qs), ps, db_breaks=hbrk)
        assert hcodes == codes
        for t in range(len(sets)):
            assert same(outs[t], host[t]), (t, sets[t])
        if oracle:
            odb, oq = hp.OracleSeqs(seq=hdb, start=hds, brk=hbrk), hp.OracleSeqs(seq=q, start=qs)
            for t, (c, i) in enumerate(sets):
                best, _ = hp.oracle_align(odb, oq, hp.default_params(n_threads=n_threads, coverage=c, identity=i, k=k))
                assert records(outs[t]) == hp.best_to_records(best, len(qs) - 1), (t, sets[t])
    finally:
        for s_ in {id(s): s for s in (s_fwd, s_q, s_db)}.values():
            s_.free()
    return outs, st


@pytest.mark.parametrize("divergence", [0.05, 0.25])
def test_cfg5_identity_sweep_on_samples(gpu, divergence):
    db, ds, q, qs = sc.fixed_case(5005, 4, 100000, 150, 20000, 1500, divergence)
    outs, _ = samples_sweep_vs(gpu, db, ds, q, qs, CFG5_SETS, oracle=True)
    acc = [int(o["accepted"].sum()) for o in outs]
    assert acc == sorted(acc, reverse=True) and acc[0] > (10 if divergence >= 0.25 else 300) and acc[0] > acc[-1]


def test_ragged_reads_with_word_breaks_in_the_database_sample(gpu):
    db, ds, q, qs = sc.ragged_case(808, 3, 60000, 6000, 900, 0.06, lo=30, hi=400)
    brk = word_breaks(db, ds, 5, 700)
    outs, st = samples_sweep_vs(gpu, db, ds, q, qs, [(0.5, 0.9), (0.3, 0.6), (0.9, 0.8)], brk=brk, oracle=True)
    assert 0 < st["k3_packed_launches"] < st["k3_launches"] and len({int(o["accepted"].sum()) for o in outs}) >= 2


def test_database_made_by_the_device_reverse_complement(gpu):
    db, ds, q, qs = sc.ragged_case(89, 3, 40000, 5000, 500, 0.05, lo=20, hi=300)
    # the query is drawn from the reverse strand so that the reverse database holds its winners
    rq, rqs, _ = _revcomp_reads(q, qs)
    brk = word_breaks(db, ds, 6, 500)
    outs, _ = samples_sweep_vs(gpu, db, ds, rq, rqs, [(0.5, 0.95), (0.5, 0.5), (0.8, 0.8)], brk=brk, rev=True, oracle=True)
    assert int(outs[1]["accepted"].sum()) > 30


def test_unsorted_and_duplicate_sets_and_sizes_1_and_16(gpu):
    db, ds, q, qs = sc.ragged_case(611, 3, 40000, 3000, 500, 0.08, lo=30, hi=300)
    outs, _ = samples_sweep_vs(gpu, db, ds, q, qs, [(0.8, 0.5), (0.3, 0.5), (1.0, 0.5), (0.5, 0.5), (0.3, 0.5)], oracle=True)
    assert same(outs[1], outs[4]) and len({int(o["accepted"].sum()) for o in outs}) >= 3
    samples_sweep_vs(gpu, db, ds, q, qs, [(0.5, 0.5)])
    samples_sweep_vs(gpu, db, ds, q, qs, SIXTEEN)


def test_seed_length_10(gpu):
    db, ds, q, qs = sc.ragged_case(910, 3, 40000, 3000, 400, 0.06, lo=30, hi=300)
    try:
        gpu.set_kmer(10)
        samples_sweep_vs(gpu, db, ds, q, qs, [(0.5, 0.9), (0.5, 0.5), (0.8, 0.7)], oracle=True, k=10)
    finally:
        gpu.set_kmer(12)


def test_read_size_stop_of_one_set(gpu):
    """a database read of 5 000 bases stops the strict set only: that block is zeroed, the others are complete"""
    from imsame_b200 import api
    db_a, ds_a, q_b, qs = read_size_case()
    sets = [(0.5, 0.5), (0.5, 0.95), (0.5, 0.7)]
    ps = [api.make_params(n_threads=4, min_coverage=c, min_identity=i) for c, i in sets]
    s_db, s_q = gpu.sample((db_a, ds_a)), gpu.sample((q_b, qs))
    try:
        outs, codes, _ = gpu.align_samples_sweep(s_db, s_q, ps)
        assert codes == [0, -5, 0]
        assert not outs[1]["accepted"].any() and not outs[1]["db_seq"].any()
        for t in (0, 2):
            want, _ = gpu.align_samples(s_db, s_q, ps[t])
            assert same(outs[t], want), t
        with pytest.raises(api.ImsameError) as e:
            gpu.align_samples(s_db, s_q, ps[1])
        assert e.value.code == -5
        host, hcodes, _ = gpu.align_sweep((db_a, ds_a), (q_b, qs), ps)
        assert hcodes == codes and all(same(outs[t], host[t]) for t in range(3))
        assert int(outs[0][40]["db_seq"]) == 3500
    finally:
        s_db.free()
        s_q.free()


def test_state_after_a_samples_sweep(gpu):
    """a plain align_samples afterwards uploads its own filter tables (equals a fresh context's result); the query
    keeps its word table; the reverse strand has no plain run to repeat"""
    from imsame_b200 import api
    db, ds, q, qs = sc.fixed_case(5, 2, 20000, 150, 800, 100, 0.05)
    p = api.make_params(n_threads=4, min_coverage=0.5, min_identity=0.5)
    fresh = api.Imsame(0)
    try:
        f_db, f_q = fresh.sample((db, ds)), fresh.sample((q, qs))
        want, _ = fresh.align_samples(f_db, f_q, p)
        f_db.free(); f_q.free()
    finally:
        fresh.close()
    s_db, s_q = gpu.sample((db, ds)), gpu.sample((q, qs))
    try:
        strict = [api.make_params(n_threads=4, min_coverage=0.9, min_identity=0.97), p]
        outs, codes, st1 = gpu.align_samples_sweep(s_db, s_q, strict)  # builds the query's word table
        assert codes == [0, 0] and same(outs[1], want) and outs[0]["accepted"].sum() < want["accepted"].sum()
        got, _ = gpu.align_samples(s_db, s_q, p)
        assert same(got, want) and want["accepted"].sum() > 40
        outs2, _, st2 = gpu.align_samples_sweep(s_db, s_q, strict)  # the table kept in the sample: no K1 launches
        assert all(same(a, b) for a, b in zip(outs, outs2)) and st2["total_launches"] < st1["total_launches"]
        with pytest.raises(api.ImsameError) as e:
            gpu.align_revcomp()
        assert e.value.code == -6
    finally:
        s_db.free()
        s_q.free()


def test_argument_errors_leave_the_context_usable(gpu):
    from imsame_b200 import api
    db, ds, q, qs = sc.fixed_case(5, 2, 20000, 150, 800, 100, 0.05)
    base = dict(n_threads=4, min_coverage=0.5, min_identity=0.5)
    s_db, s_q = gpu.sample((db, ds)), gpu.sample((q, qs))
    try:
        good, _ = gpu.align_samples(s_db, s_q, api.make_params(**base))
        for v in (dict(min_e_value=1e-10), dict(igap=4), dict(egap=1), dict(n_threads=3), dict(db_seq_base=1)):
            a, b = api.make_params(**base), api.make_params(**{**base, **v, "min_identity": 0.9})
            for order in ([a, b], [b, a]):
                with pytest.raises(api.ImsameError) as e:
                    gpu.align_samples_sweep(s_db, s_q, order)
                assert e.value.code == -3, v
        for n in (0, 17):
            with pytest.raises(api.ImsameError) as e:
                gpu.align_samples_sweep(s_db, s_q, [api.make_params(**base)] * n)
            assert e.value.code == -3
        out, _ = gpu.align_samples(s_db, s_q, api.make_params(**base))
        outs, _, _ = gpu.align_samples_sweep(s_db, s_q, [api.make_params(**base)])
        assert same(out, good) and same(outs[0], good) and good["accepted"].sum() > 40
    finally:
        s_db.free()
        s_q.free()


def test_failed_allocations_leave_context_and_samples_usable(gpu, monkeypatch):
    """IMSAME_TEST_FAIL_ALLOC=N (N = 1, 2, ...) makes device allocation N of a new context fail as on a full device:
    the samples sweep returns IMSAME_ENOMEM where its own buffers (per-set keys, tables, flags) or the run's fail, and
    the same context and samples then give the right records, through the sweep and through align_samples"""
    from imsame_b200 import api
    db, ds, q, qs = sc.fixed_case(1001, 2, 50000, 150, 4000, 500, 0.03)
    sets = [(0.5, 0.5), (0.5, 0.95), (0.8, 0.7)]
    ps = [api.make_params(n_threads=4, min_coverage=c, min_identity=i) for c, i in sets]
    want, _, _ = gpu.align_sweep((db, ds), (q, qs), ps)
    failures, quiet = [], 0
    for n in range(1, 200):
        monkeypatch.setenv("IMSAME_TEST_FAIL_ALLOC", str(n))
        ctx = api.Imsame(0)  # reads the hook
        failed = []

        def step(name, f):
            try:
                return f()
            except api.ImsameError as e:
                assert e.code == -4, (n, name, e)  # IMSAME_ENOMEM
                failed.append(name)
                return f()
        try:
            sdb = step("sample db", lambda: ctx.sample((db, ds)))
            sq = step("sample query", lambda: ctx.sample((q, qs)))
            for name in ("samples sweep", "samples sweep again"):
                outs, codes, _ = step(name, lambda: ctx.align_samples_sweep(sdb, sq, ps))
                assert codes == [0, 0, 0] and all(same(outs[t], want[t]) for t in range(3)), (n, name)
            got, _ = step("align_samples", lambda: ctx.align_samples(sdb, sq, ps[1]))
            assert same(got, want[1]), n
            sdb.free(); sq.free()
        finally:
            ctx.close()
        failures += [(n, f) for f in failed]
        quiet = 0 if failed else quiet + 1
        if quiet == 5:
            break
    else:
        pytest.fail("allocations up to 199 still failed")
    names = {f for _, f in failures}
    assert {"sample db", "sample query", "samples sweep"} <= names, failures
    assert sum(f == "samples sweep" for _, f in failures) >= 5, failures
