#!/usr/bin/env python
"""cfg4 (BASELINE.json configs[3]): all-vs-all over 8 synthetic metagenome samples (100 k reads x 150 bp
each, shared 40-genome pool), through the reference workflow script (84 processes) and through the
in-process driver bin/IMSAME_allvsall.  Prints wall times and checks that both produce the same files.
--reference: also the UNMODIFIED reference script with the reference's own binaries (oracle/_ref/, built by
oracle/build_ref.sh) on all host cores -- the same-config CPU baseline of cfg4 -- and an order-insensitive
comparison of every record of every output file with the in-process driver's.
--gpus N / --jobs J: bin/IMSAME_allvsall -jobs 1 against -gpus N -jobs J (default J = N) in the same call, alternating
(--repeats times each), every output file of every run compared with the first -jobs 1 run; prints the card and its
power limit.
usage: python tools/allvsall_bench.py [--samples 8] [--reads 100000] [--skip-script] [--reference]
       python tools/allvsall_bench.py --gpus N [--jobs J] [--repeats 3] [--samples 8] [--reads 100000]"""
import argparse, filecmp, os, shutil, subprocess, sys, tempfile, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from imsame_b200 import hostlib as H  # noqa: E402
ap = argparse.ArgumentParser()
ap.add_argument("--samples", type=int, default=8)
ap.add_argument("--reads", type=int, default=100000)
ap.add_argument("--skip-script", action="store_true")
ap.add_argument("--reference", action="store_true")
ap.add_argument("--threads", type=int, default=os.cpu_count() or 8)
ap.add_argument("--gpus", type=int, default=0)
ap.add_argument("--jobs", type=int, default=0)
ap.add_argument("--repeats", type=int, default=3)
a = ap.parse_args()
if a.jobs and not a.gpus:
    a.gpus = 1
d = tempfile.mkdtemp(prefix="imsame_avall_")
sd, o1, o2 = (os.path.join(d, n) for n in ("samples", "out_script", "out_batch"))
for p in (sd, o1, o2):
    os.makedirs(p)
pool = H.SynthPool(4001, 40, 500_000)
for s in range(a.samples):
    H.write_fasta(os.path.join(sd, f"m{s}.fasta"), pool.db_reads(s * a.reads, a.reads, 150), a.reads, 150, "r")
pool.close()
args = [sd, "0.5", "0.5", str(a.threads), "fasta"]


def same_files(x, y):
    names = sorted(os.listdir(x))
    return names == sorted(os.listdir(y)) and all(filecmp.cmp(os.path.join(x, n), os.path.join(y, n), shallow=False) for n in names)


if a.gpus:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    print("cards (index, name, power limit):")
    print(smi.stdout.strip() or smi.stderr.strip())
    jobs = a.jobs or a.gpus
    arms = [("-jobs 1", []), (f"-gpus {a.gpus} -jobs {jobs}", ["-gpus", str(a.gpus), "-jobs", str(jobs)])]
    print(f"{a.samples} samples x {a.reads} reads x 150 bp, {a.samples * (a.samples - 1)} output files, -n_threads {a.threads}")
    times = {name: [] for name, _ in arms}
    first, ok = None, True
    for rep in range(a.repeats):
        for name, extra in arms:
            o = os.path.join(d, f"out_{len(times[name])}_{'a' if not extra else 'b'}")
            os.makedirs(o)
            t = time.time()
            r = subprocess.run([os.path.join(ROOT, "bin", "IMSAME_allvsall")] + args + [o] + extra, capture_output=True, text=True)
            dt = time.time() - t
            if r.returncode:
                sys.exit(f"{name}: rc {r.returncode}: {r.stdout[-500:]}{r.stderr[-500:]}")
            times[name].append(dt)
            if first is None:
                first = o
                size = sum(os.path.getsize(os.path.join(o, n)) for n in os.listdir(o))
                print(f"outputs: {size / 1e6:.0f} MB")
            else:
                same = same_files(first, o)
                ok &= same
                shutil.rmtree(o)
            print(f"run {rep} {name}: {dt:.2f} s wall ({r.stdout.splitlines()[-1]}){'' if o == first else f'; files identical to the first -jobs 1 run: {same}'}")
            sys.stdout.flush()
    for name, _ in arms:
        v = sorted(times[name])
        print(f"{name}: median {v[len(v) // 2]:.2f} s, min {v[0]:.2f} s, max {v[-1]:.2f} s over {len(v)} runs")
    m1, m2 = (sorted(times[n])[len(times[n]) // 2] for n, _ in arms)
    print(f"speed-up of {arms[1][0]} over -jobs 1 (medians): {m1 / m2:.2f}x; all files identical: {ok}")
    shutil.rmtree(d, ignore_errors=True)
    sys.exit(0 if ok else 1)

t = time.time()
r = subprocess.run([os.path.join(ROOT, "bin", "IMSAME_allvsall")] + args + [o2], capture_output=True, text=True)
t_batch = time.time() - t
print(r.stdout.splitlines()[-1] if r.stdout else r.stderr[-300:])
if os.environ.get("IMSAME_TRACE"):
    print(r.stderr[-6000:])
print(f"in-process driver: {t_batch:.2f} s wall, rc {r.returncode}")
if not a.skip_script:
    t = time.time()
    subprocess.run([os.path.join(ROOT, "bin", "all_vs_all_metagenomes_IMSAME.sh")] + args + [o1], stdout=subprocess.DEVNULL,
                   stderr=subprocess.DEVNULL)
    t_script = time.time() - t
    names = sorted(os.listdir(o1))
    same = names == sorted(os.listdir(o2)) and all(filecmp.cmp(os.path.join(o1, n), os.path.join(o2, n), shallow=False) for n in names)
    print(f"workflow script ({len(names)} outputs, one process per comparison): {t_script:.2f} s wall; identical files: {same}")
    print(f"speed-up of the in-process driver: {t_script / t_batch:.1f}x")
if a.reference:
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers as hp
    ref_script = os.path.join(ROOT, "oracle", "_ref", "all_vs_all_metagenomes_IMSAME.sh")
    o3 = os.path.join(d, "out_reference")
    os.makedirs(o3)
    t = time.time()
    subprocess.run(["bash", ref_script] + args + [o3], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    t_ref = time.time() - t
    names = sorted(os.listdir(o3))
    same_names = names == sorted(os.listdir(o2))
    # The reference's threads write a record with two fprintf calls on one FILE* (src/alignmentFunctions.c:167-168), so with
    # -n_threads > 1 the header of one record can be followed by the text of another: files are compared as (i) the sorted
    # set of header lines `(read, db_seq) : id% cov% ylen` and (ii) the sorted multiset of ALL lines (every fprintf call
    # stays contiguous, so every line survives intact).
    n_rec, bad_hdr, bad_lines = 0, 0, 0
    for n in names:
        f_ref, f_new = os.path.join(o3, n), os.path.join(o2, n)
        h_ref = hp.parse_align_headers(f_ref)
        n_rec += len(h_ref)
        if not os.path.exists(f_new):
            bad_hdr += 1
            bad_lines += 1
            continue
        bad_hdr += h_ref != hp.parse_align_headers(f_new)
        bad_lines += sorted(open(f_ref, "rb").read().split(b"\n")) != sorted(open(f_new, "rb").read().split(b"\n"))
    print(f"reference script + reference binaries ({len(names)} outputs, -n_threads {a.threads}): {t_ref:.2f} s wall; "
          f"same file names: {same_names}; {n_rec} records; files whose header sets differ from the in-process driver's: {bad_hdr}; "
          f"files whose sorted lines differ: {bad_lines}")
    print(f"speed-up of the in-process driver over the reference workflow: {t_ref / t_batch:.1f}x")
shutil.rmtree(d, ignore_errors=True)
