#!/usr/bin/env python3
"""Files -> files with and without a BAM index, in fresh processes, alternating.

    python tools/indexed_files_bench.py [--transcripts 2000] [--coverage 100] [--repeats 3] [--out DIR]

Writes the synthetic exome-slice shape (somatic) and the normal shape at the given size, indexes the BAMs with
tests/golden/bailite.py and runs mph_run_somatic / mph_run_normal, plus the somatic run on every third gene of the GTF.
Prints one JSON line per run: wall time, the driver's stage times, peak RSS of the process, compressed bytes read and blocks
inflated (MPH_IO_TRACE), the GPU's name and power limit, and whether the outputs equal the other arm's."""
import argparse
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import bailite  # noqa: E402

CHILD = r"""
import json, os, resource, sys, time
sys.path.insert(0, %r)
import microphaser_b200 as m
d, out, mode, gtf = sys.argv[1:5]
ctx = m.Context(0)
t0 = time.perf_counter()
args = [os.path.join(d, "reads.bam"), os.path.join(d, "ref.fa"), os.path.join(d, "variants.vcf"), os.path.join(d, gtf),
        os.path.join(out, "out.fa"), os.path.join(out, "out.tsv")]
if mode == "somatic":
    ctx.run_somatic(*args, os.path.join(out, "out.normal.fa"))
else:
    ctx.run_normal(*args)
wall = time.perf_counter() - t0
t = ctx.timing()
ctx.close()
print(json.dumps(dict(wall_s=wall, ingest_ms=t["ingest_ms"], pack_ms=t["pack_ms"], write_ms=t["write_ms"], kernels_ms=t["kernels_ms"],
                      peak_rss_mb=resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1024.0)))
""" % ROOT


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--transcripts", type=int, default=2000)
    ap.add_argument("--coverage", type=float, default=100.0)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None, help="where the inputs go (default: a temporary directory)")
    a = ap.parse_args()
    from microphaser_b200 import build
    build.build_all()
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle")], check=True)
    work = a.out or tempfile.mkdtemp(prefix="mph_idx_bench_")
    try:
        run(a, work)
    finally:
        if not a.out:
            shutil.rmtree(work, ignore_errors=True)


def run(a, work):
    cases = []
    for mode, seed in (("somatic", 0x4D500003), ("normal", 0x4D500005)):
        d = os.path.join(work, mode)
        os.makedirs(d, exist_ok=True)
        subprocess.run([os.path.join(ROOT, "oracle", "_build", "mph_synth_files"), d, str(seed), str(a.transcripts), str(a.coverage), "1", "1", "0", "0"],
                       check=True, stdout=subprocess.DEVNULL)
        cases.append((mode, d, "annotation.gtf"))
    d = cases[0][1]
    keep, g = [], -1
    for line in open(os.path.join(d, "annotation.gtf")):
        if line.split("\t")[2:3] == ["gene"]:
            g += 1
        if g % 3 == 0:
            keep.append(line)
    with open(os.path.join(d, "subset.gtf"), "w") as f:
        f.writelines(keep)
    cases.append(("somatic", d, "subset.gtf"))
    for mode, d, gtf in cases:
        bam = os.path.join(d, "reads.bam")
        if not os.path.exists(bam + ".bai.off"):
            bailite.write(bam, bam + ".bai.off")
        outs = {}
        for rep in range(a.repeats):
            for arm in ("whole_file", "indexed"):
                if arm == "indexed":
                    os.replace(bam + ".bai.off", bam + ".bai")
                out = os.path.join(work, "out_%s_%s_%s" % (mode, gtf, arm))
                os.makedirs(out, exist_ok=True)
                gpu = gpu_info()
                r = subprocess.run([sys.executable, "-c", CHILD, d, out, mode, gtf], capture_output=True, text=True,
                                   env=dict(os.environ, MPH_IO_TRACE="1"))
                if arm == "indexed":
                    os.replace(bam + ".bai", bam + ".bai.off")
                if r.returncode != 0:
                    print(json.dumps(dict(case=mode, gtf=gtf, arm=arm, error=r.stderr[-400:])))
                    sys.exit(1)
                res = json.loads(r.stdout.strip().splitlines()[-1])
                m = re.search(r"\[mph io\] BGZF %s: (\d+) seeks, (\d+) compressed bytes read, (\d+) blocks inflated" % re.escape(bam), r.stderr)
                names = ("out.fa", "out.tsv", "out.normal.fa") if mode == "somatic" else ("out.fa", "out.tsv")
                outs[arm] = [open(os.path.join(out, n), "rb").read() for n in names]
                res.update(case=mode, gtf=gtf, arm=arm, repeat=rep, gpu=gpu, bam_mb=os.path.getsize(bam) / 1e6,
                           seeks=int(m.group(1)) if m else None, compressed_bytes_read=int(m.group(2)) if m else None,
                           blocks_inflated=int(m.group(3)) if m else None,
                           outputs_equal=(outs["whole_file"] == outs["indexed"]) if len(outs) == 2 else None)
                print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
