"""Reads fetched through the BAM index (csrc/io/bam_index.hpp, the indexed mode of ReadBuffer in host/ingest.hpp) on the CPU.

The indexes are written by tests/golden/bailite.py, which shares nothing with the product's reader. Checked here:
  * the same fetch() sequence through the whole-file and the indexed ReadBuffer gives the same records, and both give what a
    Python restatement of bam::RecordBuffer::fetch computes from tests/golden/bamlite.py's decoding of the file;
  * a GTF subset inflates fewer BGZF blocks through the index than the whole file holds;
  * a malformed index is an error naming the index file, also under AddressSanitizer / UBSan;
  * the emulator CLI (product host code, emulated device side) with an index gives the oracle's bytes."""
import os
import random
import shutil
import struct
import subprocess
import sys

import pytest

from conftest import GOLDEN, ROOT, materialize_reference, read_outputs, run_cli

sys.path.insert(0, GOLDEN)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bailite  # noqa: E402
import bamlite  # noqa: E402
from fuzz_compare import PROFILES  # noqa: E402

from microphaser_b200 import synth  # noqa: E402

GOLDEN_BAMS = sorted(d for d in os.listdir(GOLDEN) if os.path.exists(os.path.join(GOLDEN, d, "reads.bam")))


def _compile(tmp_path_factory, name, extra=()):
    exe = str(tmp_path_factory.mktemp("idx") / name)
    subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-Wall", "-Wno-missing-field-initializers", *extra, "-o", exe,
                    os.path.join(ROOT, "tests", "units", "index_fetch.cpp"), "-lz", "-lpthread"], check=True)
    return exe


@pytest.fixture(scope="module")
def index_fetch(tmp_path_factory):
    return _compile(tmp_path_factory, "index_fetch")


def fnv1a(b):
    h = 1469598103934665603
    for c in b:
        h = ((h ^ c) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return h


def py_fetch(bam, queries):
    """bam::RecordBuffer::fetch as the whole-file buffer states it, over bamlite's records: per query the buffered records."""
    refs, recs = bamlite.read_bam(bam)
    tid_of = {n: i for i, (n, _) in enumerate(refs)}
    by_tid = {}
    for r in recs:
        if 0 <= r.tid < len(refs):
            by_tid.setdefault(r.tid, []).append(r)
    inner, overflow, tid_, cur = [], None, -1, 0
    for chrom, start, end in queries:
        if overflow is not None:
            inner.append(overflow)
            overflow = None
        tid = tid_of[chrom]
        v = by_tid.get(tid, [])
        refetch = not inner or inner[-1].pos < start or inner[0].tid != tid or inner[0].pos > start
        if refetch:
            inner, tid_, cur = [], tid, 0
            while cur < len(v) and v[cur].pos < start and (v[cur].flag & 4 or v[cur].end_pos() <= start):
                cur += 1
        else:
            while inner and inner[0].pos < start:
                inner.pop(0)
        w = by_tid.get(tid_, [])
        while tid_ == tid and cur < len(w):
            r = w[cur]
            cur += 1
            if r.flag & 4:
                continue
            if r.pos >= end:
                overflow = r
                break
            if r.pos >= start or (refetch and r.end_pos() > start):
                inner.append(r)
        yield [(r.pos, r.end_pos(), r.flag, r.mapq, fnv1a(r.qname.encode()),
                fnv1a((r.seq + "|" + "".join("%d%s" % (l, op) for op, l in r.cigar)).encode())) for r in inner]


def check_fetches(exe, bam, queries, threads=((1, 1), (3, 4))):
    want = list(py_fetch(bam, queries))
    text = "".join("%s %d %d\n" % q for q in queries)
    for whole_t, idx_t in threads:
        r = subprocess.run([exe, "fetch", bam, str(whole_t), str(idx_t)], input=text, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout[-500:] + r.stderr[-500:]
        lines = r.stdout.splitlines()
        assert lines[-1].endswith(", 0 differences")
        got, i = [], 0
        while i < len(lines) - 1:
            n = int(lines[i].split()[2])
            got.append([tuple(int(x) for x in ln.split()) for ln in lines[i + 1:i + 1 + n]])
            i += 1 + n
        assert len(got) == len(want)
        for k, (g, w) in enumerate(zip(got, want)):
            assert g == w, (k, queries[k])


def indexed_copy(src_bam, d):
    os.makedirs(d, exist_ok=True)
    bam = os.path.join(d, "reads.bam")
    shutil.copy(src_bam, bam)
    bailite.write(bam)
    return bam


def gtf_queries(gtf):
    out = []
    for line in open(gtf):
        t = line.split("\t")
        if len(t) >= 9 and t[2] == "gene":
            out.append((t[0], int(t[3]) - 1, int(t[4])))
    return out


def add_empty_contig(bam, name="chrEmpty", length=50000):
    """The BAM with one more contig in its header, on which no read lies."""
    raw = bamlite.bgzf_decompress(bam)
    o = 8 + struct.unpack_from("<i", raw, 4)[0]
    n_ref = struct.unpack_from("<i", raw, o)[0]
    p = o + 4
    for _ in range(n_ref):
        p += 8 + struct.unpack_from("<i", raw, p)[0]
    new = raw[:o] + struct.pack("<i", n_ref + 1) + raw[o + 4:p] + struct.pack("<i", len(name) + 1) + name.encode() + b"\0" + \
        struct.pack("<i", length) + raw[p:]
    with open(bam, "wb") as f:
        f.write(synth._bgzf_blocks(new))


@pytest.mark.parametrize("case", GOLDEN_BAMS)
def test_golden_gene_order_fetches_match(index_fetch, case, tmp_path):
    d = os.path.join(GOLDEN, case)
    bam = indexed_copy(os.path.join(d, "reads.bam"), str(tmp_path))
    queries = []
    for fn in sorted(os.listdir(d)):
        if fn.endswith(".gtf"):
            queries += gtf_queries(os.path.join(d, fn))
    check_fetches(index_fetch, bam, queries)


def test_multi_batch_synthetic_bam_gene_order_fetches_match(index_fetch, tmp_path):
    """The 30 MB synthetic BAM of the loader test: many batches, records straddling them, seeks and reads forward."""
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle")], check=True)
    d = str(tmp_path / "sample")
    os.makedirs(d)
    subprocess.run([os.path.join(ROOT, "oracle", "_build", "mph_synth_files"), d, "77", "160", "100", "1", "1", "0.1", "0.1"], check=True,
                   stdout=subprocess.DEVNULL)
    bam = os.path.join(d, "reads.bam")
    bailite.write(bam)
    queries = gtf_queries(os.path.join(d, "annotation.gtf"))
    check_fetches(index_fetch, bam, queries + queries[::3], threads=((1, 1), (4, 4)))


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_random_query_sequences_match(index_fetch, seed, tmp_path):
    """Overlapping, backwards and adjacent queries, contig switches, queries past a contig's end, a contig without reads,
    and reads that reach into a query from the left (spliced reads over short introns)."""
    d = str(tmp_path / "in")
    synth.generate(d, synth.Params(seed=seed, n_contigs=3, n_genes=4, coverage=40.0, intron_len=(20, 400), indel_frac=0.1))
    bam = os.path.join(d, "reads.bam")
    add_empty_contig(bam)
    bailite.write(bam)
    refs, _ = bamlite.read_bam(bam)
    rng = random.Random(seed)
    queries, prev = [], None
    for _ in range(300):
        name, length = refs[rng.randrange(len(refs))] if prev is None or rng.random() < 0.15 else prev[:2]
        kind = rng.random()
        if prev is not None and prev[0] == name and kind < 0.25:
            s = max(0, prev[2] + rng.randrange(-300, 300))      # overlapping the previous query
        elif prev is not None and prev[0] == name and kind < 0.4:
            s = prev[3]                                          # adjacent
        elif kind < 0.5:
            s = length + rng.randrange(0, 500)                   # past the contig's end
        else:
            s = rng.randrange(0, length)                         # anywhere, often backwards
        e = s + rng.choice([1, 50, 400, 3000, 20000])
        queries.append((name, s, e))
        prev = (name, length, s, e)
    check_fetches(index_fetch, bam, queries, threads=((1, 1), (2, 3)))


def _trace_blocks(stderr, bam):
    for line in stderr.splitlines():
        if line.startswith("[mph io] BGZF " + bam + ":"):
            return int(line.split(", ")[-1].split()[0])
    raise AssertionError("no BGZF trace for " + bam + " in " + stderr[-400:])


def test_gtf_subset_inflates_fewer_blocks(emu_bin, oracle_bin, tmp_path):
    """Every third gene of the synthetic chr22 shape: through the index the reads between the genes are never inflated."""
    d = str(tmp_path / "in")
    synth.generate(d, synth.Params(seed=0x4D500002, n_genes=30, exons=(8, 8), exon_len=(90, 250), intron_len=(300, 2000), read_len=150,
                                   coverage=30.0, germline_per_kb=1.0, somatic_per_kb=1.0, lowercase_frac=0.0))
    lines, keep, g = open(os.path.join(d, "annotation.gtf")).read().splitlines(True), [], -1
    for line in lines:
        if line.split("\t")[2:3] == ["gene"]:
            g += 1
        if g % 3 == 0:
            keep.append(line)
    with open(os.path.join(d, "subset.gtf"), "w") as f:
        f.writelines(keep)
    bam = os.path.join(d, "reads.bam")
    env = dict(os.environ, MPH_IO_TRACE="1", MPH_IO_THREADS="1")
    outs = {}
    for name in ("whole", "indexed", "oracle"):
        if name == "indexed":
            bailite.write(bam)
        o = tmp_path / name
        o.mkdir()
        binary = oracle_bin if name == "oracle" else emu_bin
        r = subprocess.run([binary, "somatic", bam, "-r", os.path.join(d, "ref.fa"), "-b", os.path.join(d, "variants.vcf"), "-t", str(o / "out.tsv"),
                            "-n", str(o / "out.normal.fa")], stdin=open(os.path.join(d, "subset.gtf")), stdout=open(o / "out.fa", "wb"),
                           stderr=subprocess.PIPE, env=env, text=True)
        assert r.returncode == 0, r.stderr[-500:]
        outs[name] = (read_outputs(str(o)), r.stderr)
    whole, indexed = _trace_blocks(outs["whole"][1], bam), _trace_blocks(outs["indexed"][1], bam)
    assert indexed < whole * 0.8, (indexed, whole)
    assert outs["indexed"][0] == outs["whole"][0] == outs["oracle"][0]


def _malformed(bam, good):
    """(case, index bytes) with one defect each."""
    n_ref = struct.unpack_from("<i", good, 4)[0]
    size = os.path.getsize(bam)
    chunk_at = lin_at = None
    p = 8
    for _ in range(n_ref):  # the first chunk and the first linear-index entry of any reference
        n_bin = struct.unpack_from("<i", good, p)[0]
        p += 4
        for _ in range(n_bin):
            b, n_chunk = struct.unpack_from("<Ii", good, p)
            if b != 37450 and chunk_at is None:
                chunk_at = p + 8
            p += 8 + 16 * n_chunk
        n_lin = struct.unpack_from("<i", good, p)[0]
        if n_lin > 0 and lin_at is None:
            lin_at = p + 4
        p += 4 + 8 * n_lin
    past = struct.pack("<Q", (size + 4096) << 16)
    yield "truncated", good[:len(good) // 2]
    yield "truncated_header", good[:6]
    yield "bad_magic", b"BAI\x02" + good[4:]
    yield "n_ref_mismatch", good[:4] + struct.pack("<i", n_ref + 1) + good[8:]
    yield "chunk_past_eof", good[:chunk_at] + past + good[chunk_at + 8:]
    yield "linear_past_eof", good[:lin_at] + past + good[lin_at + 8:]
    yield "huge_bin_count", good[:8] + struct.pack("<i", 1 << 30) + good[12:]
    yield "negative_chunk_count", good[:chunk_at - 4] + struct.pack("<i", -5) + good[chunk_at:]


@pytest.mark.parametrize("sanitize", [False, True])
def test_malformed_index_is_an_error(tmp_path_factory, tmp_path, sanitize):
    extra = ("-fsanitize=address,undefined", "-fno-sanitize-recover=all") if sanitize else ()
    exe = _compile(tmp_path_factory, "index_fetch_asan" if sanitize else "index_fetch_plain", extra)
    bam = indexed_copy(os.path.join(GOLDEN, "forward_somatic", "reads.bam"), str(tmp_path))
    good = open(bam + ".bai", "rb").read()
    r = subprocess.run([exe, "load", bam, bam + ".bai"], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.strip() == "ok", r.stdout + r.stderr
    for case, data in _malformed(bam, good):
        bad = str(tmp_path / (case + ".bai"))
        with open(bad, "wb") as f:
            f.write(data)
        r = subprocess.run([exe, "load", bam, bad], capture_output=True, text=True)
        assert r.returncode == 1, (case, r.returncode, r.stdout[-300:], r.stderr[-800:])
        assert r.stdout.startswith("error: malformed BAM index " + bad), (case, r.stdout)


def test_cli_with_malformed_index_fails_with_input_error(emu_bin, tmp_path):
    """A wrong index means wrong reads: the CLI stops with exit status 1 instead of falling back to a scan."""
    d = os.path.join(GOLDEN, "forward_somatic")
    bam = indexed_copy(os.path.join(d, "reads.bam"), str(tmp_path / "in"))
    with open(bam + ".bai", "r+b") as f:
        f.write(b"CSI\x01")
    fa = materialize_reference(d, str(tmp_path))
    cmd = [emu_bin, "somatic", bam, "-r", fa, "-b", os.path.join(d, "variants.vcf"), "-t", str(tmp_path / "o.tsv"), "-n", str(tmp_path / "o.n.fa")]
    r = subprocess.run(cmd, stdin=open(os.path.join(d, "annotation.gtf")), capture_output=True, text=True)
    assert r.returncode == 1 and "malformed BAM index" in r.stderr, r.stderr


@pytest.mark.parametrize("sub", ["somatic", "normal"])
@pytest.mark.parametrize("profile", sorted(PROFILES))
def test_emulator_with_index_matches_oracle(emu_bin, oracle_bin, profile, sub, tmp_path):
    """Differential fuzzing as tests/fuzz_compare.py does it, with a .bai next to the BAM: two seeds per profile."""
    for seed in (31, 32):
        kw = dict(PROFILES[profile])
        kw.update(seed=seed * 7919 + len(profile), n_genes=3, coverage=25.0)
        d = str(tmp_path / ("in%d" % seed))
        synth.generate(d, synth.Params(**kw))
        o, p = tmp_path / ("o%d" % seed), tmp_path / ("p%d" % seed)
        o.mkdir()
        p.mkdir()
        ro = run_cli(oracle_bin, d, str(o), subcommand=sub)
        bailite.write(os.path.join(d, "reads.bam"))
        rp = run_cli(emu_bin, d, str(p), subcommand=sub)
        if rp.returncode == 3:
            continue
        assert ro.returncode == rp.returncode, (ro.stderr.decode()[-300:], rp.stderr.decode()[-300:])
        if ro.returncode == 0:
            assert read_outputs(str(o), sub) == read_outputs(str(p), sub)


def test_golden_cli_runs_with_index_match_expected(emu_bin, tmp_path):
    """Every golden through the emulator CLI with an index next to the BAM: the reference's expected bytes."""
    for case in GOLDEN_BAMS:
        d = os.path.join(GOLDEN, case)
        if not os.path.isdir(os.path.join(d, "expected")):
            continue
        sub = "normal" if "normal" in case else "somatic"
        w = tmp_path / case
        bam = indexed_copy(os.path.join(d, "reads.bam"), str(w / "in"))
        for fn in os.listdir(d):
            if fn != "reads.bam" and not os.path.isdir(os.path.join(d, fn)):
                shutil.copy(os.path.join(d, fn), str(w / "in"))
        fa = materialize_reference(d, str(w))
        r = run_cli(emu_bin, os.path.dirname(bam), str(w), ref=fa, subcommand=sub)
        assert r.returncode == 0, (case, r.stderr.decode()[-300:])
        for name in sorted(os.listdir(os.path.join(d, "expected"))):
            assert open(w / name, "rb").read() == open(os.path.join(d, "expected", name), "rb").read(), (case, name)
