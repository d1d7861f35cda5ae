"""bin/IMSAME_allvsall -sweep without a GPU: the argument errors are IMSAME -sweep's (one parser, shared by both command
lines), the samples sweep is exported, and there is no CPU fallback behind it."""
import ctypes as C
import os
import subprocess

import pytest

import helpers as hp

G = os.path.join(hp.ROOT, "tests", "golden")
ALLVSALL = os.path.join(hp.ROOT, "bin", "IMSAME_allvsall")
IMSAME = os.path.join(hp.ROOT, "bin", "IMSAME")
MALFORMED = "-sweep expects a list of coverage:identity pairs, e.g. -sweep 0.5:0.7,0.5:0.9"
CASES = [
    ("0.5", MALFORMED),
    ("0.5:0.7,", MALFORMED),
    ("0.5:0.7,0.5:x", MALFORMED),
    (":0.7", MALFORMED),
    ("0.5:0.7:0.9", MALFORMED),
    ("0.5:" + "1" * 70, MALFORMED),
    (",".join(["0.5:0.5"] * 16), "-sweep takes at most 15 coverage:identity pairs"),
    (",".join(["0.5:0.5"] * 15 + ["x"]), "-sweep takes at most 15 coverage:identity pairs"),
    ("0.5:0.7,0:0.5", "Min-coverage must be larger than zero"),
    ("0.5:0.7,-0.1:0.5", "Min-coverage must be larger than zero"),
    ("0.5:0", "Min-identity must be larger than zero"),
    ("0.5:-2", "Min-identity must be larger than zero"),
]


def _samples(tmp_path):
    d, o = tmp_path / "s", tmp_path / "o"
    d.mkdir(); o.mkdir()
    (d / "a.fasta").write_bytes(open(os.path.join(G, "dirty.q.fa"), "rb").read())
    (d / "b.fasta").write_bytes(open(os.path.join(G, "dirty.db.fa"), "rb").read())
    return d, o


def _imsame(*extra):
    return subprocess.run([IMSAME, "-query", os.path.join(G, "dirty.q.fa"), "-db", os.path.join(G, "dirty.db.fa"), *extra],
                          capture_output=True, text=True)


@pytest.mark.parametrize("value,message", CASES)
def test_sweep_errors_equal_those_of_imsame(built, tmp_path, value, message):
    """the reference's terror form (message on stdout, exit status 255) before any sample is read: no output file"""
    d, o = _samples(tmp_path)
    r = subprocess.run([ALLVSALL, str(d), "0.5", "0.5", "2", "fasta", str(o), "-sweep", value], capture_output=True, text=True)
    want = _imsame("-sweep", value)
    assert (r.returncode, r.stdout) == (want.returncode, want.stdout) == (255, f"ERR**** {message} ****\n")
    assert os.listdir(o) == []


@pytest.mark.parametrize("value", ["0.5:0.7", "1:1,0.25:0.5", ",".join(["0.5:0.5"] * 15), "5e-1:7e-1", " 0.5:0.7"])
def test_valid_lists_pass_the_parser(built, tmp_path, value):
    """a well-formed list gets past the argument checks of both command lines (up to the device: with a GPU the runs
    are tests/test_gpu_allvsall_sweep.py's)"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = _imsame("-sweep", value, "-out", str(tmp_path / "f.align"))
    assert r.returncode == 255 and "ERR**** GPU hot path failed: no usable sm_100 CUDA device" in r.stdout, r.stdout
    assert "-sweep" not in r.stdout
    d, o = _samples(tmp_path)
    r = subprocess.run([ALLVSALL, str(d), "0.5", "0.5", "2", "fasta", str(o), "-sweep", value], capture_output=True, text=True)
    assert r.returncode == 255 and r.stdout == "ERR**** no usable GPU: no usable sm_100 CUDA device /  ****\n", r.stdout


def test_samples_sweep_is_exported(built):
    from imsame_b200 import api
    lib = C.CDLL(api.GPU_SO)
    assert getattr(lib, "imsame_gpu_align_samples_sweep") is not None
    assert "imsame_gpu_align_samples_sweep" in api.SYMBOLS
    hdr = open(os.path.join(hp.ROOT, "include", "imsame_gpu.h")).read()
    assert "int imsame_gpu_align_samples_sweep(" in hdr


def test_sweep_fails_loudly_without_a_gpu(built, tmp_path):
    """no CPU fallback behind -sweep, resident or from host buffers: the default run's error, exit status 255, no
    record and no entry file"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    d, o = _samples(tmp_path)
    base = [ALLVSALL, str(d), "0.5", "0.5", "2", "fasta", str(o)]
    want = subprocess.run(base, capture_output=True, text=True)
    r = subprocess.run(base + ["-sweep", "0.5:0.7,0.5:0.9", "-jobs", "2"], capture_output=True, text=True)
    assert (r.returncode, r.stdout) == (want.returncode, want.stdout)
    assert r.returncode == 255 and "no usable GPU" in r.stdout and os.listdir(o) == []
    env = dict(os.environ, IMSAME_NO_RESIDENT="1")
    want = subprocess.run(base, capture_output=True, text=True, env=env)
    r = subprocess.run(base + ["-sweep", "0.5:0.7,0.5:0.9"], capture_output=True, text=True, env=env)
    assert (r.returncode, r.stdout) == (want.returncode, want.stdout)
    assert r.returncode == 255 and "ERR**** GPU hot path failed: no usable sm_100 CUDA device" in r.stdout
    assert "sweep" not in r.stdout
    # the failed unit leaves its (empty) main file as without -sweep, and no entry file
    assert all(not n.endswith((".1", ".2")) for n in os.listdir(o))
    assert all(os.path.getsize(o / n) == 0 for n in os.listdir(o))
