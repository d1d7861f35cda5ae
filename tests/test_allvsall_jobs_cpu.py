"""bin/IMSAME_allvsall -gpus N / -jobs J without a GPU: argument errors, and no CPU fallback behind the workers."""
import os
import subprocess

import pytest

import helpers as hp

G = os.path.join(hp.ROOT, "tests", "golden")
EXE = os.path.join(hp.ROOT, "bin", "IMSAME_allvsall")


def _samples(tmp_path):
    d, o = tmp_path / "s", tmp_path / "o"
    d.mkdir(); o.mkdir()
    (d / "a.fasta").write_bytes(open(os.path.join(G, "dirty.q.fa"), "rb").read())
    (d / "b.fasta").write_bytes(open(os.path.join(G, "dirty.db.fa"), "rb").read())
    (d / "c.fasta").write_bytes(open(os.path.join(G, "synth150.q.fa"), "rb").read())
    return d, o


@pytest.mark.parametrize("flag,value", [("-gpus", "0"), ("-gpus", "-2"), ("-gpus", "two"), ("-gpus", "2x"), ("-gpus", ""),
                                        ("-gpus", "99999999999"), ("-gpus", "1025"), ("-jobs", "0"), ("-jobs", "-1"),
                                        ("-jobs", "1.5"), ("-jobs", "4096"), ("-jobs", None)])
def test_bad_gpus_or_jobs_value_is_an_argument_error(built, tmp_path, flag, value):
    """rejected like the other argument errors (terror: message on stdout, status 255), before any sample is read or any
    device is touched: no output file is written"""
    d, o = _samples(tmp_path)
    args = [EXE, str(d), "0.5", "0.5", "2", "fasta", str(o), flag] + ([] if value is None else [value])
    r = subprocess.run(args, capture_output=True, text=True)
    assert r.returncode == 255
    assert r.stdout == f"ERR**** {flag} must be an integer from 1 to 1024 ****\n"
    assert os.listdir(o) == []


def test_gpus_and_jobs_without_a_gpu_fail_like_the_default_run(built, tmp_path):
    """no CPU fallback behind the workers either: -gpus 2 -jobs 4 ends with exactly the default run's error (the earliest
    unit's) and writes no record"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    d, o = _samples(tmp_path)
    base = [EXE, str(d), "0.5", "0.5", "2", "fasta", str(o)]
    want = subprocess.run(base, capture_output=True, text=True)
    assert want.returncode == 255 and want.stdout == "ERR**** no usable GPU: no usable sm_100 CUDA device /  ****\n"
    assert os.listdir(o) == []
    for extra in (["-gpus", "2", "-jobs", "4"], ["-jobs", "3"], ["-device", "1", "-gpus", "2"]):
        r = subprocess.run(base + extra, capture_output=True, text=True)
        assert (r.returncode, r.stdout) == (want.returncode, want.stdout), extra
        assert os.listdir(o) == [], extra
    # every unit from host buffers: the error of imsame_run_job, identical too
    env = dict(os.environ, IMSAME_NO_RESIDENT="1")
    want = subprocess.run(base, capture_output=True, text=True, env=env)
    r = subprocess.run(base + ["-gpus", "2", "-jobs", "4"], capture_output=True, text=True, env=env)
    assert want.returncode == 255 and "ERR**** GPU hot path failed: no usable sm_100 CUDA device" in want.stdout
    assert (r.returncode, r.stdout) == (want.returncode, want.stdout)


def test_nothing_to_do_needs_no_gpu(built, tmp_path):
    """every output exists (resume rule): no worker starts, no device is needed, whatever -jobs says"""
    d, o = _samples(tmp_path)
    for x, y in (("a", "b"), ("a", "c"), ("b", "c")):
        for r in ("", ".r"):
            (o / f"{x}-{y}{r}.align").write_bytes(b"kept")
    r = subprocess.run([EXE, str(d), "0.5", "0.5", "2", "fasta", str(o), "-gpus", "2", "-jobs", "8"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout
    assert r.stdout.startswith("[INFO] 0 comparisons of 3 samples in ")
    assert all((o / n).read_bytes() == b"kept" for n in os.listdir(o))
