"""GPU: bin/IMSAME_allvsall -sweep.  Every OUT/X-Y[.r].align.i must equal the X-Y[.r].align of a separate run at entry i's
thresholds, the main files those of the run without -sweep, at -jobs 1 and -jobs 3, from resident samples, from host
buffers and under cache eviction; the stdout lines, the resume rule and a per-entry read-size stop are checked too."""
import os
import re
import subprocess
import time

import pytest

import helpers as hp
import synth_cases as sc
from test_gpu_sweep import read_size_case, write_fasta

pytestmark = pytest.mark.gpu
EXE = os.path.join(hp.ROOT, "bin", "IMSAME_allvsall")
ENTRIES = [("0.5", "0.9"), ("0.3", "0.95"), ("0.8", "0.6")]
SWEEP = ",".join(f"{c}:{i}" for c, i in ENTRIES)
UNIT_RE = re.compile(r"^(\[INFO\] \S+ vs \S+(?: \(reverse complement\))?)(: \d+ reads .*); [0-9.]+ s$")


def _run(d, o, cov, idn, *extra, env=None):
    os.makedirs(o, exist_ok=True)
    return subprocess.run([EXE, str(d), cov, idn, "4", "fasta", str(o)] + list(extra), capture_output=True, text=True,
                          env=dict(os.environ, **(env or {})))


def _strip_times(stdout):
    return [re.sub(r"; [0-9.]+ s$", "", re.sub(r" in [0-9.]+ s$", "", l)) for l in stdout.splitlines()]


def _same(a, b):
    return open(a, "rb").read() == open(b, "rb").read()


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    """five samples (the text-filter samples of the all-vs-all tests and a divergent copy of their pool, so that the
    identity thresholds split the records), the run without -sweep and one separate run per entry"""
    from imsame_b200 import hostlib as H
    base = tmp_path_factory.mktemp("allvsall_sweep")
    d = base / "samples"
    d.mkdir()
    sc.write_allvsall_filter_samples(d)
    pool = H.SynthPool(4107, 3, 30000)
    H.write_fasta(str(d / "t.fasta"), pool.query_reads(500, 400, 150, 0.08), 400, 150, "t")
    pool.close()
    plain = _run(d, base / "plain", "0.5", "0.5")
    assert plain.returncode == 0, plain.stdout + plain.stderr
    assert "20 comparisons of 5 samples" in plain.stdout
    seps = []
    for i, (c, idn) in enumerate(ENTRIES, 1):
        r = _run(d, base / f"sep{i}", c, idn)
        assert r.returncode == 0, r.stdout + r.stderr
        seps.append((base / f"sep{i}", r.stdout))
    return d, base / "plain", plain.stdout, seps


def _expected_stdout(plain_out, seps):
    """each unit's line, then per entry that unit's line of the separate run, reworded; the summary line as it is"""
    want = []
    sep_lines = [[l for l in out.splitlines() if UNIT_RE.match(l)] for _, out in seps]
    k = 0
    for line in plain_out.splitlines():
        if not UNIT_RE.match(line):
            want.append(line)
            continue
        want.append(line)
        for i, (c, idn) in enumerate(ENTRIES):
            m = UNIT_RE.match(sep_lines[i][k])
            want.append(f"{m.group(1)} sweep {i + 1} of {len(ENTRIES)} (-coverage {c} -identity {idn}){m.group(2)}")
        k += 1
    assert k == len(sep_lines[0])
    return _strip_times("\n".join(want))


def _check_files(runs, o):
    d, plain, plain_out, seps = runs
    mains = sorted(os.listdir(plain))
    assert len(mains) == 20
    assert sorted(os.listdir(o)) == sorted(mains + [f"{n}.{i}" for n in mains for i in range(1, len(ENTRIES) + 1)])
    for n in mains:
        assert _same(o / n, plain / n), n
        for i, (sep, _) in enumerate(seps, 1):
            assert _same(o / f"{n}.{i}", sep / n), (n, i)


def _check(runs, o, r):
    assert r.returncode == 0, r.stdout + r.stderr[-2000:]
    _check_files(runs, o)
    assert _strip_times(r.stdout) == _expected_stdout(runs[2], runs[3])


@pytest.mark.parametrize("jobs", ["1", "3"])
def test_entry_files_equal_separate_runs(runs, tmp_path, jobs):
    o = tmp_path / "o"
    r = _run(runs[0], o, "0.5", "0.5", "-jobs", jobs, "-sweep", SWEEP)
    _check(runs, o, r)
    # the entries are not vacuous: the thresholds give different records
    names = os.listdir(runs[1])
    sizes = [sum(os.path.getsize(o / (n + sfx)) for n in names) for sfx in ("", ".1", ".2", ".3")]
    assert len(set(sizes)) >= 3 and sizes[0] > 10000, sizes


def test_host_buffers_and_eviction_give_the_same_bytes(runs, tmp_path):
    for name, env in (("host", {"IMSAME_NO_RESIDENT": "1"}), ("evict", {"IMSAME_TEST_SAMPLE_BUDGET": str(100 << 20)}),
                      ("tiny", {"IMSAME_TEST_SAMPLE_BUDGET": "1000"})):
        o = tmp_path / name
        r = _run(runs[0], o, "0.5", "0.5", "-jobs", "3", "-sweep", SWEEP, env={**env, "IMSAME_TRACE": "1"})
        _check(runs, o, r)
        rows = re.findall(r"evictions (\d+), host-path fallbacks (\d+)", r.stderr)
        assert rows, r.stderr[-2000:]
        if name == "evict":
            assert sum(int(e) for e, _ in rows) > 0 and sum(int(f) for _, f in rows) == 0, rows
        if name == "tiny":
            assert sum(int(f) for _, f in rows) == 20, rows


def test_resume_rewrites_only_the_unit_with_a_missing_entry_file(runs, tmp_path):
    o = tmp_path / "o"
    r = _run(runs[0], o, "0.5", "0.5", "-sweep", SWEEP)
    assert r.returncode == 0, r.stdout
    os.remove(o / "s1-t.r.align.2")
    before = {n: os.stat(o / n).st_mtime_ns for n in os.listdir(o)}
    time.sleep(1.1)
    r = _run(runs[0], o, "0.5", "0.5", "-sweep", SWEEP)
    assert r.returncode == 0 and "[INFO] 1 comparisons of 5 samples" in r.stdout, r.stdout
    unit = {"s1-t.r.align"} | {f"s1-t.r.align.{i}" for i in (1, 2, 3)}
    after = {n: os.stat(o / n).st_mtime_ns for n in os.listdir(o)}
    assert set(after) == set(before) | {"s1-t.r.align.2"}
    assert all(after[n] == before[n] for n in before if n not in unit)
    assert all(after[n] > before.get(n, 0) for n in unit)
    _check_files(runs, o)


def test_read_size_stop_of_one_entry(tmp_path):
    """a database read of 5 000 bases that the query reaches before any accepted hit at identity 0.95 only: that entry
    writes no file and prints the reference's error line in place of its line, the other entry and the main file are
    those of separate runs, the run ends with exit status 255 (a separate run at 0.95 stops there)"""
    db, ds, q, qs = read_size_case()
    d = tmp_path / "samples"
    d.mkdir()
    write_fasta(str(d / "a.fasta"), q, qs)
    write_fasta(str(d / "b.fasta"), db, ds)
    entries = [("0.5", "0.95"), ("0.5", "0.7")]

    def out_dir(name):
        # only the unit a-b runs: the others' outputs exist (resume rule); b as a query has a read of 5 000 bases
        o = tmp_path / name
        o.mkdir()
        for n in ("b-a.align", "b-a.r.align", "a-b.r.align"):
            for suffix in [""] + [f".{i}" for i in range(1, len(entries) + 1)]:
                (o / (n + suffix)).write_bytes(b"kept")
        return o

    o = out_dir("sweep")
    r = _run(d, o, "0.5", "0.5", "-sweep", ",".join(f"{c}:{i}" for c, i in entries))
    assert r.returncode == 255, r.stdout + r.stderr
    plain = _run(d, out_dir("plain"), "0.5", "0.5")
    strict = _run(d, out_dir("strict"), *entries[0])
    loose = _run(d, out_dir("loose"), *entries[1])
    assert plain.returncode == 0 and loose.returncode == 0, plain.stdout + loose.stdout
    assert strict.returncode == 255 and strict.stdout.endswith("ERR**** Read size reached for gapped alignment. ****\n")
    assert _same(o / "a-b.align", tmp_path / "plain" / "a-b.align")
    assert _same(o / "a-b.align.2", tmp_path / "loose" / "a-b.align") and os.path.getsize(o / "a-b.align.2") > 1000
    assert not os.path.exists(o / "a-b.align.1")
    m = UNIT_RE.match(next(l for l in loose.stdout.splitlines() if UNIT_RE.match(l)))
    want = [l for l in _strip_times(plain.stdout)]
    at = next(k for k, l in enumerate(want) if l.startswith("[INFO] a vs b:")) + 1
    want[at:at] = ["ERR**** Read size reached for gapped alignment. ****",
                   f"{m.group(1)} sweep 2 of 2 (-coverage 0.5 -identity 0.7){m.group(2)}"]
    assert _strip_times(r.stdout) == want
