"""The CUDA file drivers with a BAM index next to the BAM (written by tests/golden/bailite.py): genes are streamed in shards
through the index. Outputs must be the oracle's bytes and those of the same run without the index; host memory must follow
the shard size, not the file size."""
import os
import shutil
import struct
import subprocess
import sys

import pytest

from conftest import CONFIG_SHAPES, GOLDEN, ROOT, materialize_reference, read_outputs, run_cli, run_oracle_on_files

sys.path.insert(0, GOLDEN)
import bailite  # noqa: E402
from test_io_indexed import GOLDEN_BAMS, indexed_copy  # noqa: E402

pytestmark = pytest.mark.gpu

SYNTH = os.path.join(ROOT, "oracle", "_build", "mph_synth_files")


def synth_files(d, shape, n_transcripts=None):
    s = CONFIG_SHAPES[shape]
    os.makedirs(d, exist_ok=True)
    subprocess.run([SYNTH, d, str(s["seed"]), str(n_transcripts or s["n_transcripts"]), str(s["coverage"]), str(s["germline_per_kb"]),
                    str(s["somatic_per_kb"]), str(s["ins_var_frac"]), str(s["del_var_frac"])], check=True, stdout=subprocess.DEVNULL)
    return s["mode"]


def run_files(d, out, mode, n_ctx=1, gtf="annotation.gtf"):
    import microphaser_b200 as m
    os.makedirs(out, exist_ok=True)
    ctxs = [m.Context(0) for _ in range(n_ctx)]
    args = [os.path.join(d, "reads.bam"), os.path.join(d, "ref.fa"), os.path.join(d, "variants.vcf"), os.path.join(d, gtf),
            os.path.join(out, "out.fa"), os.path.join(out, "out.tsv")]
    try:
        if mode == "somatic":
            m.run_somatic_multi(ctxs, *args, os.path.join(out, "out.normal.fa"))
        else:
            m.run_normal_multi(ctxs, *args)
    finally:
        for c in ctxs:
            c.close()
    return read_outputs(out, mode)


@pytest.mark.parametrize("case", GOLDEN_BAMS)
def test_cli_with_index_matches_golden(product, case, tmp_path):
    d = os.path.join(GOLDEN, case)
    w = tmp_path / "in"
    indexed_copy(os.path.join(d, "reads.bam"), str(w))
    for fn in os.listdir(d):
        if fn != "reads.bam" and not os.path.isdir(os.path.join(d, fn)):
            shutil.copy(os.path.join(d, fn), str(w))
    fa = materialize_reference(d, str(tmp_path))
    if case == "unsorted_gtf":
        assert run_cli(product[1], str(w), str(tmp_path), gtf="unsorted.gtf", ref=fa).returncode == 101
        assert run_cli(product[1], str(w), str(tmp_path), gtf="sorted.gtf", ref=fa).returncode == 0
        return
    sub = "normal" if "normal" in case else "somatic"
    r = run_cli(product[1], str(w), str(tmp_path), ref=fa, subcommand=sub)
    assert r.returncode == 0, r.stderr.decode()
    for name in sorted(os.listdir(os.path.join(d, "expected"))):
        assert open(tmp_path / name, "rb").read() == open(os.path.join(d, "expected", name), "rb").read(), name
    if case == "reverse_somatic":  # variants as BCF2
        from conftest import make_bcf
        r = run_cli(product[1], str(w), str(tmp_path), ref=fa, variants=make_bcf(d, str(tmp_path)))
        assert r.returncode == 0, r.stderr.decode()
        for name in sorted(os.listdir(os.path.join(d, "expected"))):
            assert open(tmp_path / name, "rb").read() == open(os.path.join(d, "expected", name), "rb").read(), name


@pytest.mark.parametrize("shape", ["C2_chr22", "C5a_normal"])
def test_streamed_shards_match_oracle_and_whole_file(product, oracle_bin, shape, tmp_path, monkeypatch):
    d = str(tmp_path / "in")
    mode = synth_files(d, shape)
    o = str(tmp_path / "oracle")
    os.makedirs(o)
    assert run_oracle_on_files(oracle_bin, d, o, mode).returncode == 0
    want = read_outputs(o, mode)
    monkeypatch.setenv("MPH_IO_THREADS", "4")
    whole = run_files(d, str(tmp_path / "whole"), mode)
    assert whole == want
    bailite.write(os.path.join(d, "reads.bam"))
    n_reads = len(bailite._records(os.path.join(d, "reads.bam"))[1])
    monkeypatch.setenv("MPH_SHARD_READS", str(max(1, n_reads // 10)))  # at least 8 shards
    for n_ctx in (1, 2):
        for io_threads in ("1", "4"):
            monkeypatch.setenv("MPH_IO_THREADS", io_threads)
            assert run_files(d, str(tmp_path / ("idx%d_%s" % (n_ctx, io_threads))), mode, n_ctx) == want, (n_ctx, io_threads)
    monkeypatch.setenv("MPH_GPU_INFLATE", "1")
    monkeypatch.setenv("MPH_IO_THREADS", "4")
    assert run_files(d, str(tmp_path / "idx_gpu_inflate"), mode) == want


def test_streamed_gtf_subset_matches_oracle(product, oracle_bin, tmp_path, monkeypatch):
    d = str(tmp_path / "in")
    mode = synth_files(d, "C2_chr22")
    keep, g = [], -1
    for line in open(os.path.join(d, "annotation.gtf")):
        if line.split("\t")[2:3] == ["gene"]:
            g += 1
        if g % 3 == 0:
            keep.append(line)
    with open(os.path.join(d, "subset.gtf"), "w") as f:
        f.writelines(keep)
    shutil.copy(os.path.join(d, "subset.gtf"), os.path.join(d, "annotation.gtf"))
    o = str(tmp_path / "oracle")
    os.makedirs(o)
    assert run_oracle_on_files(oracle_bin, d, o, mode).returncode == 0
    bailite.write(os.path.join(d, "reads.bam"))
    monkeypatch.setenv("MPH_SHARD_READS", "20000")
    assert run_files(d, str(tmp_path / "p"), mode) == read_outputs(o, mode)


def inflated_bytes(bam):
    """Sum of the ISIZE fields of the BGZF blocks."""
    data, o, total = open(bam, "rb").read(), 0, 0
    while o < len(data):
        xlen = struct.unpack_from("<H", data, o + 10)[0]
        bsize = struct.unpack_from("<H", data, o + 16)[0] + 1 if xlen >= 6 else None
        total += struct.unpack_from("<I", data, o + bsize - 4)[0]
        o += bsize
    return total


PEAK_RSS = r"""
import resource, subprocess, sys
with open(sys.argv[1]) as gin, open(sys.argv[2], "wb") as fo:
    rc = subprocess.run(sys.argv[3:], stdin=gin, stdout=fo).returncode
print(rc, resource.getrusage(resource.RUSAGE_CHILDREN).ru_maxrss * 1024)
"""


def test_streamed_peak_memory_follows_shard_size(product, tmp_path):
    """A synthetic BAM of over 150 MB through the CLI, each run in a fresh wrapper that reports the child's peak RSS. The
    whole-file loader holds every inflated batch until the run ends, so its peak exceeds the inflated size; the streamed
    run holds at most workers + 1 = 3 shards of 50 000 reads (about 16 MB of inflated records each, plus the batches of 64
    blocks they pin and the read-ahead): far less than half the inflated file, which is the margin asserted."""
    d = str(tmp_path / "in")
    synth_files(d, "C3_exome_slice", n_transcripts=900)
    bam = os.path.join(d, "reads.bam")
    assert os.path.getsize(bam) > 150 << 20
    inflated = inflated_bytes(bam)
    env = dict(os.environ, MPH_PACK_THREADS="2", MPH_SHARD_READS="50000", MPH_IO_THREADS="4")
    peak = {}
    for name in ("whole", "indexed"):
        if name == "indexed":
            bailite.write(bam)
        o = tmp_path / name
        o.mkdir()
        cmd = [product[1], "somatic", bam, "-r", os.path.join(d, "ref.fa"), "-b", os.path.join(d, "variants.vcf"), "-t", str(o / "out.tsv"),
               "-n", str(o / "out.normal.fa")]
        r = subprocess.run([sys.executable, "-c", PEAK_RSS, os.path.join(d, "annotation.gtf"), str(o / "out.fa")] + cmd, env=env,
                           capture_output=True, text=True, check=True)
        rc, rss = (int(x) for x in r.stdout.split())
        assert rc == 0, r.stderr[-500:]
        peak[name] = rss
    print("inflated %.1f MB, peak RSS whole-file %.1f MB, indexed %.1f MB" % (inflated / 1e6, peak["whole"] / 1e6, peak["indexed"] / 1e6))
    assert read_outputs(str(tmp_path / "whole")) == read_outputs(str(tmp_path / "indexed"))
    assert peak["whole"] - peak["indexed"] >= inflated // 2, (peak, inflated)
