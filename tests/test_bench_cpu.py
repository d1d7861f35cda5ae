"""CPU tests of bench.py's own checkers and of its reference arm (no GPU): a parity self-check that cannot
fail proves nothing, so sampled_parity is fed records that ARE right (made by the scan-order oracle) and
records with one field off, and the `--impl reference` line is checked against the contract in bench.py's
docstring."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers as hp
import synth_cases as sc

REC = [("db_seq", "u8"), ("qpos_end", "u8"), ("db_pos", "u8"), ("length", "u4"), ("identities", "u4"), ("accepted", "u1")]


def _bench():
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(hp.ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _oracle_records(db, ds, q, qs):
    nq = len(qs) - 1
    best, _ = hp.oracle_align(hp.OracleSeqs(seq=db, start=ds), hp.OracleSeqs(seq=q, start=qs), hp.default_params(n_threads=4))
    rec = np.zeros(nq, dtype=REC)
    for r, v in hp.best_to_records(best, nq).items():
        rec[r] = (v[0], v[1], v[2], v[3], v[4], 1)
    return rec


def test_sampled_parity_accepts_right_records_and_sees_every_field(built):
    b = _bench()
    db, ds, q, qs = sc.fixed_case(1001, 2, 5000, 150, 400, 500, 0.03)
    rec = _oracle_records(db, ds, q, qs)
    nq = len(qs) - 1
    args = (db, ds, q, qs, len(db), 0, 1, 5000, 150, None, None, np)
    out = b.sampled_parity(nq, rec, *args)  # every read
    assert out["reads"] == nq and out["mismatches"] == 0 and out["oracle_accepted"] == int(rec["accepted"].sum()) > 50
    assert out["cpu_port_same_database"]["reads_per_s"] > 0 and out["cpu_port_same_database"]["kind"] == "port"
    json.dumps(out)  # goes into the bench's JSON line as is
    acc = np.flatnonzero(rec["accepted"])
    rej = np.flatnonzero(rec["accepted"] == 0)
    for field in ("db_seq", "qpos_end", "db_pos", "length", "identities"):
        bad = rec.copy()
        bad[field][acc[3]] += 1
        o = b.sampled_parity(nq, bad, *args)
        assert o["mismatches"] == 1 and o["first_mismatch"]["read"] == int(acc[3]), field
    bad = rec.copy()
    bad["accepted"][acc[5]] = 0  # a lost record
    assert b.sampled_parity(nq, bad, *args)["mismatches"] == 1
    bad = rec.copy()
    bad[rej[0]] = rec[acc[0]]  # a record for a read that has none
    assert b.sampled_parity(nq, bad, *args)["mismatches"] == 1


def test_dump_records_writes_every_field_exactly_and_samples_above_the_cap(built, tmp_path):
    b = _bench()
    rng = np.random.default_rng(4)
    n = 5000
    rec = np.zeros(n, dtype=REC)
    rec["accepted"] = rng.integers(0, 2, n)
    rec["db_seq"] = rng.integers(0, 80_000_000, n)
    rec["qpos_end"] = rng.integers(0, 250_000_000, n)
    rec["db_pos"] = rng.integers(0, 20_000_000_000, n)
    rec["length"] = rng.integers(0, 3000, n)
    rec["identities"] = rng.integers(0, 3000, n)
    b.dump_records(str(tmp_path / "all"), rec, np)
    got = {f[:-4]: np.load(tmp_path / "all" / f) for f in os.listdir(tmp_path / "all")}
    assert sorted(got) == sorted(["read"] + [f for f, _ in b.DUMP_FIELDS])
    assert all(v.dtype in (np.float32, np.float64) and len(v) == n for v in got.values())
    assert np.array_equal(got["read"], np.arange(n))
    for f, _ in b.DUMP_FIELDS:
        assert np.array_equal(got[f].astype(np.uint64), rec[f].astype(np.uint64)), f
    b.DUMP_BYTES_MAX = 1000 * 44  # 44 bytes per read: a fixed sample of 1000 reads
    for d in ("s1", "s2"):
        b.dump_records(str(tmp_path / d), rec, np)
    assert sum(os.path.getsize(tmp_path / "s1" / f) - 128 for f in os.listdir(tmp_path / "s1")) == b.DUMP_BYTES_MAX
    reads = np.load(tmp_path / "s1" / "read.npy").astype(np.int64)
    assert len(reads) == 1000 and np.array_equal(reads, np.load(tmp_path / "s2" / "read.npy"))
    assert np.array_equal(np.load(tmp_path / "s1" / "db_pos.npy"), rec["db_pos"][reads].astype(np.float64))


def test_zero_timed_steps_is_refused(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(hp.ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=120, cwd=str(tmp_path))
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr and not r.stdout


def test_dump_outputs_is_refused_on_the_reference_arm(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(hp.ROOT, "bench.py"), "--impl", "reference", "--dump-outputs",
                        str(tmp_path / "d")], capture_output=True, text=True, timeout=120, cwd=str(tmp_path))
    assert r.returncode == 2 and "not with --impl reference" in r.stderr and not os.path.exists(tmp_path / "d")


@pytest.mark.skipif(not hp.have_reference(), reason="oracle/_ref not built (needs /root/reference at build time)")
def test_reference_arm_prints_the_contract_line(built, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(hp.ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--cpu-sample-queries", "200", "--cpu-sample-db", "10000"], capture_output=True, text=True, timeout=600,
                       cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["metric"] == "query reads aligned/sec" and line["unit"] == "reads/s"
    assert line["higher_is_better"] is True and line["n_gpus"] == 1 and line["steps"] == 1 and line["warmup"] == 1
    assert line["value"] > 0 and line["ms_per_step"] > 0
    assert line["cpu_baseline"]["kind"] == "reference" and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["value"] == line["value"] and line["cpu_baseline"]["sample"]
    e2e = line["e2e"]
    assert (e2e["value"], e2e["unit"], e2e["h2d_bytes_per_step"], e2e["d2h_bytes_per_step"]) == (line["value"], "reads/s", 0, 0)
    assert line["config"]["workload"].startswith("cfg2")
