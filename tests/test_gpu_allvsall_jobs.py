"""GPU: bin/IMSAME_allvsall with several comparisons in flight (-jobs J, -gpus N) writes the files of the default run byte
for byte, prints its [INFO] lines in the same order, keeps the resume rule and stops on an error exactly like it; the
per-worker device sample cache evicts and falls back to host buffers without changing a byte; a context stays usable
after imsame_gpu_align_samples ran out of device memory."""
import os
import re
import subprocess

import numpy as np
import pytest

import helpers as hp
import synth_cases as sc

pytestmark = pytest.mark.gpu
EXE = os.path.join(hp.ROOT, "bin", "IMSAME_allvsall")
TRACE_RE = re.compile(r"\[imsame_allvsall\] worker (\d+) device (\d+): units (\d+), uploads (\d+), table builds (\d+), "
                      r"evictions (\d+), host-path fallbacks (\d+), busy [0-9.]+ s")


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _write_samples(d):
    """the four samples of test_gpu_cli.test_in_process_all_vs_all_equals_the_script (s3 dirty: lower case, N, multi-line,
    '>' inside headers) and, as f0..f3, sc.write_allvsall_filter_samples (revComp's text is not their mirror image)"""
    from imsame_b200 import hostlib as H
    pool = H.SynthPool(4001, 3, 30000)
    for i in range(3):
        H.write_fasta(str(d / f"s{i}.fasta"), pool.db_reads(i * 1000, 500, 150), 500, 150, "r")
    reads = pool.db_reads(5000, 300, 150)
    pool.close()
    with open(d / "s3.fasta", "wb") as f:
        f.write(b"text before the first header\n")
        for r in range(300):
            b = bytes(reads[r * 150:(r + 1) * 150])
            if r % 3 == 0:
                b = b[:40].lower() + b"N" + b[40:]
            f.write(b">x%d with > inside\n" % r + b[:70] + b"\n" + b[70:] + b"\n")
    t = d / "filter"
    t.mkdir()
    sc.write_allvsall_filter_samples(t)
    for i in range(4):
        os.rename(t / f"s{i}.fasta", d / f"f{i}.fasta")
    t.rmdir()


@pytest.fixture(scope="module")
def reference_run(tmp_path_factory):
    """the default run (one worker) on the eight samples: its directory, outputs and stdout"""
    base = tmp_path_factory.mktemp("allvsall_jobs")
    d, o = base / "samples", base / "out_default"
    d.mkdir(); o.mkdir()
    _write_samples(d)
    r = subprocess.run([EXE, str(d), "0.5", "0.5", "4", "fasta", str(o)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "56 comparisons of 8 samples" in r.stdout
    return d, o, r.stdout


def _run(d, o, *extra, env=None):
    os.makedirs(o, exist_ok=True)
    return subprocess.run([EXE, str(d), "0.5", "0.5", "4", "fasta", str(o)] + list(extra), capture_output=True, text=True,
                          env=dict(os.environ, **(env or {})))


def _strip_times(stdout):
    return [re.sub(r"; [0-9.]+ s$", "", re.sub(r" in [0-9.]+ s$", "", l)) for l in stdout.splitlines()]


def _same_files(o1, o2, names=None):
    names = sorted(os.listdir(o1)) if names is None else names
    assert names and all(os.path.exists(os.path.join(o2, n)) for n in names)
    for n in names:
        assert open(os.path.join(o1, n), "rb").read() == open(os.path.join(o2, n), "rb").read(), n


def _trace(stderr):
    rows = [tuple(int(v) for v in m.groups()) for m in TRACE_RE.finditer(stderr)]
    assert rows, stderr[-2000:]
    return rows


def test_jobs3_equals_the_default_run_and_keeps_the_resume_rule(reference_run, tmp_path):
    d, o1, out1 = reference_run
    o2 = tmp_path / "out"
    r = _run(d, o2, "-jobs", "3")
    assert r.returncode == 0, r.stdout + r.stderr
    assert sorted(os.listdir(o2)) == sorted(os.listdir(o1)) and len(os.listdir(o1)) == 56
    _same_files(o1, o2)
    assert _strip_times(r.stdout) == _strip_times(out1)
    assert os.path.getsize(o2 / "s0-s1.align") > 10000 and os.path.getsize(o2 / "f0-f1.r.align") > 1000
    # resume: existing outputs are kept, only the missing ones are recomputed
    os.remove(o2 / "s1-s3.r.align")
    os.remove(o2 / "f2-s0.align")
    (o2 / "s0-s1.align").write_bytes(b"kept")
    r = _run(d, o2, "-jobs", "3")
    assert r.returncode == 0 and "2 comparisons of 8 samples" in r.stdout
    assert (o2 / "s0-s1.align").read_bytes() == b"kept"
    _same_files(o1, o2, ["s1-s3.r.align", "f2-s0.align"])
    info = [l for l in _strip_times(r.stdout) if " vs " in l]
    assert info == [l for l in _strip_times(out1) if l.startswith("[INFO] f2 vs s0:") or l.startswith("[INFO] s1 vs s3 (")]


def test_sample_budget_evicts_and_falls_back_without_changing_a_byte(reference_run, tmp_path):
    d, o1, out1 = reference_run
    # room for one query word table (4^12 offsets, 67 MB) and the read sets of a unit, not for two tables: a worker that
    # moves to the next query sample while another still aligns against the previous one has to evict
    r = _run(d, tmp_path / "evict", "-jobs", "3", env={"IMSAME_TEST_SAMPLE_BUDGET": str(100 << 20), "IMSAME_TRACE": "1"})
    assert r.returncode == 0, r.stdout + r.stderr[-2000:]
    rows = _trace(r.stderr)
    assert len(rows) == 3 and sum(x[2] for x in rows) == 56
    assert sum(x[5] for x in rows) > 0, rows  # evictions
    assert sum(x[6] for x in rows) == 0, rows  # every unit still resident
    assert sum(x[3] for x in rows) > 0 and sum(x[4] for x in rows) > 0
    _same_files(o1, tmp_path / "evict")
    assert _strip_times(r.stdout) == _strip_times(out1)
    # below one read set: every unit runs from host buffers, nothing is uploaded
    r = _run(d, tmp_path / "host", "-jobs", "3", env={"IMSAME_TEST_SAMPLE_BUDGET": "1000", "IMSAME_TRACE": "1"})
    assert r.returncode == 0, r.stdout + r.stderr[-2000:]
    rows = _trace(r.stderr)
    assert sum(x[6] for x in rows) == 56 and sum(x[3] for x in rows) == 0 and sum(x[4] for x in rows) == 0, rows
    _same_files(o1, tmp_path / "host")
    assert _strip_times(r.stdout) == _strip_times(out1)


def test_read_size_stop_is_the_same_under_jobs3(tmp_path):
    """a read longer than 3 000 bases that a query read reaches stops the run with the reference's message; under -jobs 3
    the same [INFO] lines come first, the units before the failing one are written identically, exit status 255"""
    from imsame_b200 import hostlib as H
    d = tmp_path / "samples"
    d.mkdir()
    pool = H.SynthPool(4001, 3, 30000)
    for k, name in enumerate(("a0", "a1", "d0")):
        H.write_fasta(str(d / f"{name}.fasta"), pool.db_reads(k * 1000, 400, 150), 400, 150, "r")
    extra = pool.db_reads(4000, 100, 150)
    pool.close()
    rng = np.random.default_rng(11)
    s = bytes(np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=3200)])
    with open(d / "b.fasta", "wb") as f:
        f.write(b">long\n" + s + b"\n")
        for r in range(50):
            f.write(b">e%d\n" % r + bytes(extra[r * 150:(r + 1) * 150]) + b"\n")
    with open(d / "c.fasta", "wb") as f:
        for r in range(50, 100):
            f.write(b">e%d\n" % r + bytes(extra[r * 150:(r + 1) * 150]) + b"\n")
        f.write(b">rotated\n" + s[100:] + s[:100] + b"\n")
    r1 = _run(d, tmp_path / "o1")
    r3 = _run(d, tmp_path / "o3", "-jobs", "3")
    assert r1.returncode == 255 and r1.stdout.endswith("ERR**** Read size reached for gapped alignment. ****\n"), r1.stdout
    assert r3.returncode == 255 and _strip_times(r3.stdout) == _strip_times(r1.stdout)
    # canonical order: a0-a1 a0-b a0-c a0-d0 a1-b a1-c a1-d0 b-c ...: b-c.align is the first that fails
    done = [l.split(":")[0] for l in r1.stdout.splitlines() if l.startswith("[INFO]")]
    assert len(done) == 14 and done[-1] == "[INFO] a1 vs d0 (reverse complement)", done
    before = [f"{x}-{y}{r}.align" for x, y in (("a0", "a1"), ("a0", "b"), ("a0", "c"), ("a0", "d0"), ("a1", "b"), ("a1", "c"),
                                               ("a1", "d0")) for r in ("", ".r")]
    _same_files(tmp_path / "o1", tmp_path / "o3", before)
    assert sorted(os.listdir(tmp_path / "o1")) == sorted(before + ["b-c.align"])


def test_two_gpus_equal_the_default_run(reference_run, tmp_path):
    if _n_gpus() < 2:
        pytest.skip("needs >= 2 GPUs")
    d, o1, out1 = reference_run
    r = _run(d, tmp_path / "o", "-gpus", "2", env={"IMSAME_TRACE": "1"})
    assert r.returncode == 0, r.stdout + r.stderr[-2000:]
    _same_files(o1, tmp_path / "o")
    assert _strip_times(r.stdout) == _strip_times(out1)
    assert sorted({x[1] for x in _trace(r.stderr)}) == [0, 1]


def test_forced_out_of_memory_retries_then_falls_back_without_changing_a_byte(reference_run, tmp_path):
    """IMSAME_TEST_FAIL_ALLOC makes chosen device allocations of every worker's context fail as on a full device (an
    impossible cudaMalloc request: nothing outside the process is touched).  One failure: the unit retries with every
    other read set evicted and stays resident.  Two in a row: the retry fails too and the unit runs from host buffers on
    the same context.  Either way the files and [INFO] lines are those of the default run."""
    d, o1, out1 = reference_run
    r = _run(d, tmp_path / "once", "-jobs", "3", env={"IMSAME_TEST_FAIL_ALLOC": "6", "IMSAME_TRACE": "1"})
    assert r.returncode == 0, r.stdout + r.stderr[-2000:]
    rows = _trace(r.stderr)
    assert sum(x[2] for x in rows) == 56 and sum(x[6] for x in rows) == 0, rows
    _same_files(o1, tmp_path / "once")
    assert _strip_times(r.stdout) == _strip_times(out1)
    r = _run(d, tmp_path / "twice", "-jobs", "3", env={"IMSAME_TEST_FAIL_ALLOC": "6,2", "IMSAME_TRACE": "1"})
    assert r.returncode == 0, r.stdout + r.stderr[-2000:]
    rows = _trace(r.stderr)
    assert sum(x[2] for x in rows) == 56 and all(x[6] >= 1 for x in rows), rows  # every worker fell back once
    _same_files(o1, tmp_path / "twice")
    assert _strip_times(r.stdout) == _strip_times(out1)


def test_context_stays_usable_after_every_failed_allocation(gpu, monkeypatch):
    """Each device allocation of a context in turn fails with IMSAME_ENOMEM (IMSAME_TEST_FAIL_ALLOC=N, N = 1, 2, ...):
    sample uploads, the query word table, the run's keys / bins / work buffers and, with a small pair table
    (IMSAME_TEST_PAIR_SLOTS), its growth in the middle of a run.  After the failure the same context and samples give the
    records of a fresh run, through imsame_gpu_align_samples and through the host-buffer path."""
    from imsame_b200 import api
    db, ds, q, qs = sc.fixed_case(1001, 2, 50000, 150, 4000, 500, 0.03)
    p = api.make_params(n_threads=4)
    want, _ = gpu.align((db, ds), (q, qs), p)
    monkeypatch.setenv("IMSAME_TEST_PAIR_SLOTS", "64")
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
                ctx.set_kmer(12)  # what imsame_run_job does first: refused while a failed run is still marked active
                return f()
        try:
            sdb = step("sample db", lambda: ctx.sample((db, ds)))
            sq = step("sample query", lambda: ctx.sample((q, qs)))
            for name in ("align_samples", "align_samples again", "align (host buffers)", "align_samples after align"):
                f = (lambda: ctx.align((db, ds), (q, qs), p)) if "host" in name else (lambda: ctx.align_samples(sdb, sq, p))
                got, _ = step(name, f)
                assert np.array_equal(got, want), (n, name)
            sdb.free(); sq.free()
        finally:
            ctx.close()
        failures += [(n, f) for f in failed]
        # (a failure the allocator absorbs by releasing its cached blocks and asking again shows no error): the
        # sweep is over once several allocation numbers in a row lie past the last allocation
        quiet = 0 if failed else quiet + 1
        if quiet == 5:
            break
    else:
        pytest.fail("allocations up to 199 still failed")
    names = {f for _, f in failures}
    assert len(failures) >= 15 and {"sample db", "sample query", "align_samples", "align (host buffers)"} <= names, failures
