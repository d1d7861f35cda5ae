"""Several seed lengths in one run without a GPU: the exported entry point, and the command line's -kmers argument
checks, which end the run before any device work."""
import ctypes as C
import os
import subprocess

import pytest

import helpers as hp

G = os.path.join(hp.ROOT, "tests", "golden")
EXE = os.path.join(hp.ROOT, "bin", "IMSAME")


def test_align_kmers_is_exported(built):
    from imsame_b200 import api
    lib = C.CDLL(api.GPU_SO)
    assert getattr(lib, "imsame_gpu_align_kmers") is not None
    assert "imsame_gpu_align_kmers" in api.SYMBOLS
    hdr = open(os.path.join(hp.ROOT, "include", "imsame_gpu.h")).read()
    assert "#define IMSAME_KMERS_MAX 13" in hdr and api.KMERS_MAX == 13


def _run(*extra, cwd=None):
    return subprocess.run([EXE, "-query", os.path.join(G, "dirty.q.fa"), "-db", os.path.join(G, "dirty.db.fa"), *extra],
                          capture_output=True, text=True, cwd=cwd)


MALFORMED = "-kmers expects a list of seed lengths, e.g. -kmers 8,10,14"
RANGE = "The seed length must be between 4 and 16"
REPEAT = "-kmers must not repeat a seed length or give the -kmer one"


@pytest.mark.parametrize("args,message", [
    (["-kmers", ""], MALFORMED),
    (["-kmers", "8,"], MALFORMED),
    (["-kmers", ",8"], MALFORMED),
    (["-kmers", "8,,10"], MALFORMED),
    (["-kmers", "8;10"], MALFORMED),
    (["-kmers", "x"], MALFORMED),
    (["-kmers", "-8"], MALFORMED),
    (["-kmers", "8.5"], MALFORMED),
    (["-kmers", "8 "], MALFORMED),
    (["-kmers", "1000"], MALFORMED),
    (["-kmers", "3"], RANGE),
    (["-kmers", "8,17"], RANGE),
    (["-kmers", "0"], RANGE),
    (["-kmers", "8,10,8"], REPEAT),
    (["-kmers", "12"], REPEAT),
    (["-kmers", "8,10", "-kmer", "10"], REPEAT),
    (["-kmer", "8", "-kmers", "8"], REPEAT),
    (["-kmers", "4,5,6,7,8,9,10,11,13,14,15,16,4"], "-kmers takes at most 12 seed lengths"),
    (["-kmers", "8", "-sweep", "0.5:0.7"], "-kmers cannot be combined with -sweep"),
    (["-kmers", "8", "-gpus", "2"], "-kmers runs on one GPU: it cannot be combined with -gpus above 1"),
    (["-kmers", "8", "-out_rev", "REV"], "-kmers cannot be combined with -out_rev"),
])
def test_refused_before_any_work(built, tmp_path, args, message):
    """the reference's terror form (message on stdout, exit status 255) and nothing else: no [INFO] line, no GPU, no
    file"""
    args = [str(tmp_path / "r.align") if a == "REV" else a for a in args]
    r = _run(*args, "-out", str(tmp_path / "f.align"))
    assert r.returncode == 255 and r.stdout == f"ERR**** {message} ****\n", r.stdout
    assert os.listdir(tmp_path) == []


def test_every_other_seed_length_is_accepted_by_the_parser(built, tmp_path):
    """twelve entries (every length but -kmer's) pass the checks; without a GPU the run then fails in the GPU step"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = _run("-kmers", "4,5,6,7,8,9,10,11,13,14,15,16", cwd=str(tmp_path))
    assert r.returncode == 255 and "ERR**** GPU hot path failed" in r.stdout


def test_fails_loudly_without_a_gpu(built, tmp_path):
    """no CPU fallback behind -kmers: the reference's error form, exit status 255, every file empty"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    f = tmp_path / "f.align"
    r = _run("-kmers", "8,14", "-out", str(f))
    assert r.returncode == 255 and "ERR**** GPU hot path failed: no usable sm_100 CUDA device" in r.stdout
    assert "from the query were found" not in r.stdout and "Seed length" not in r.stdout
    assert sorted(os.listdir(tmp_path)) == ["f.align", "f.align.k14", "f.align.k8"]
    assert all(os.path.getsize(tmp_path / p) == 0 for p in os.listdir(tmp_path))


def test_kmers_is_not_in_the_reference_help_text(built):
    r = subprocess.run([EXE, "--help"], capture_output=True, text=True)
    assert r.returncode == 1 and "-kmers" not in r.stdout
