"""Synthetic exome-like inputs of the shapes BASELINE.json names (SURVEY.md §8(d)).

Writes real files — FASTA(+.fai), sorted GTF, VCF with the SOMATIC flag, coordinate-sorted
BAM (BGZF) — so the oracle CLI and the product CLI can be run on identical inputs. Small and
medium scale only (pure Python); the whole-exome bench shape is generated natively by
`mph_synth_batch` in the C-ABI library with the same distributions.

Generator constraints that follow from reference behaviour (BASELINE.md §4): CDS free of in-frame
stop codons (a stop closes the transcript, reference src/microphasing.rs:694-718,1485-1488), sorted
GTF with the mandatory attributes (:1994-2038), VCF sorted in GTF contig order, no ANN header.
"""
import os
import random
import struct
import zlib

_COMP = {"A": "T", "C": "G", "G": "C", "T": "A", "N": "N"}
_STOPS = {"TAA", "TAG", "TGA"}
_CODONS = [a + b + c for a in "ACGT" for b in "ACGT" for c in "ACGT" if a + b + c not in _STOPS]
_SEQ_CODE = {c: i for i, c in enumerate("=ACMGRSVTWYHKDBN")}


def revcomp(s):
    return "".join(_COMP[c] for c in reversed(s))


class Params:
    def __init__(self, **kw):
        self.seed = 1
        self.n_contigs = 1
        self.n_genes = 4
        self.exons = (3, 6)            # exons per transcript (min, max)
        self.exon_len = (60, 250)
        self.intron_len = (300, 1200)
        self.utr3 = 60
        self.read_len = 100
        self.coverage = 30.0
        self.germline_per_kb = 2.0
        self.somatic_per_kb = 2.0
        self.indel_frac = 0.0          # share of variants that are indels (half ins, half del)
        self.multiallelic_frac = 0.0
        self.frameshift_ok = False     # allow indel lengths that are not multiples of 3
        self.lowq_frac = 0.02
        self.softclip_frac = 0.02
        self.noise_indel_frac = 0.02   # reads with a private 1-6 nt I/D not in the VCF
        self.mapq0_frac = 0.01
        self.unmapped_frac = 0.005
        self.dup_mate_frac = 0.01      # pairs sharing qname and start (reverse-strand `contains`)
        self.dup_extra_frac = 0.0      # chance that such a group gets one more copy (repeatedly): groups of three and more
        self.lowercase_frac = 0.1      # genes placed in a soft-masked (lowercase) region
        self.first_frame = False       # sometimes give the first CDS a non-zero frame column
        self.short_exon_frac = 0.0     # share of internal exons shorter than the window
        self.start_loss_frac = 0.0     # put a variant into the start codon
        self.transcripts_per_gene = 1
        self.antisense_frac = 0.0      # chance that an additional transcript of a gene is annotated on the opposite strand
        self.variants_in_introns = True
        self.independent_somatic = False  # each somatic variant gets its own draw per read (else one draw per read for all of them)
        self.hotspot_per_gene = 0         # extra somatic SNVs within one 27-nt stretch of one exon per gene (variant-dense windows)
        for k, v in kw.items():
            if not hasattr(self, k):
                raise TypeError(k)
            setattr(self, k, v)


def _bgzf_blocks(data):
    out = []
    for o in range(0, len(data), 0xFF00):
        chunk = data[o:o + 0xFF00]
        co = zlib.compressobj(1, zlib.DEFLATED, -15)
        comp = co.compress(chunk) + co.flush()
        bsize = len(comp) + 25
        out.append(b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", bsize) + comp +
                   struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk)))
    out.append(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))
    return b"".join(out)


def _bam_record(tid, pos, mapq, flag, qname, cigar, seq, qual):
    ops = "MIDNSHP=X"
    cig = b"".join(struct.pack("<I", (l << 4) | ops.index(op)) for op, l in cigar)
    l_seq = len(seq)
    packed = bytearray((l_seq + 1) // 2)
    for i, c in enumerate(seq):
        packed[i >> 1] |= _SEQ_CODE[c] << (4 if i % 2 == 0 else 0)
    name = qname.encode() + b"\0"
    end = pos + sum(l for op, l in cigar if op in "MDN=X")
    body = struct.pack("<iiBBHHHiiii", tid, pos, len(name), mapq, _reg2bin(pos, max(end, pos + 1)), len(cigar), flag, l_seq, -1, -1, 0)
    body += name + cig + bytes(packed) + bytes(qual)
    return struct.pack("<i", len(body)) + body


def _reg2bin(beg, end):
    end -= 1
    if beg >> 14 == end >> 14:
        return ((1 << 15) - 1) // 7 + (beg >> 14)
    if beg >> 17 == end >> 17:
        return ((1 << 12) - 1) // 7 + (beg >> 17)
    if beg >> 20 == end >> 20:
        return ((1 << 9) - 1) // 7 + (beg >> 20)
    if beg >> 23 == end >> 23:
        return ((1 << 6) - 1) // 7 + (beg >> 23)
    if beg >> 26 == end >> 26:
        return ((1 << 3) - 1) // 7 + (beg >> 26)
    return 0


def generate(outdir, p):
    """Write ref.fa(.fai), annotation.gtf, variants.vcf, reads.bam into outdir. Returns a summary dict."""
    rng = random.Random(p.seed)
    os.makedirs(outdir, exist_ok=True)
    contigs = []
    gtf_lines = []
    vcf_rows = []
    bam_recs = []
    n_tx = 0
    cds_nt = 0
    gid = 0
    for ci in range(p.n_contigs):
        cname = "chrS%d" % (ci + 1)
        genome = []
        pos = 0

        def emit(s):
            nonlocal pos
            genome.append(s)
            pos += len(s)

        emit("".join(rng.choice("ACGT") for _ in range(rng.randint(400, 900))))
        genes = []
        for _ in range(p.n_genes):
            gid += 1
            reverse = rng.random() < 0.5
            lower = rng.random() < p.lowercase_frac
            n_ex = rng.randint(*p.exons)
            lens = []
            for e in range(n_ex):
                if 0 < e < n_ex - 1 and rng.random() < p.short_exon_frac:
                    lens.append(rng.randint(3, 26))
                else:
                    lens.append(rng.randint(*p.exon_len))
            total = sum(lens)
            lens[-1] += (3 - total % 3) % 3
            total = sum(lens)
            coding = "ATG" + "".join(rng.choice(_CODONS) for _ in range(total // 3 - 1))
            stop = rng.choice(sorted(_STOPS))
            utr = "".join(rng.choice("ACGT") for _ in range(p.utr3))
            tail = stop + utr  # follows the CDS in transcript direction
            # genomic layout: exons in genomic order; for reverse genes transcript exon 1 is rightmost
            glens = lens[::-1] if reverse else lens
            introns = [rng.randint(*p.intron_len) for _ in range(n_ex - 1)]
            mrna = coding
            pieces = []  # per transcript-order exon: coding slice
            o = 0
            for l in lens:
                pieces.append(mrna[o:o + l])
                o += l
            gstart = pos
            exon_coords = []  # genomic order
            if not reverse:
                for i, l in enumerate(glens):
                    s = pos
                    emit(pieces[i])
                    if i == n_ex - 1:
                        emit(tail)
                    exon_coords.append((s, s + l))
                    if i < n_ex - 1:
                        emit("".join(rng.choice("ACGT") for _ in range(introns[i])))
            else:
                for i, l in enumerate(glens):
                    tx_i = n_ex - 1 - i  # transcript-order index of this genomic exon
                    if i == 0:
                        emit(revcomp(tail))
                    s = pos
                    emit(revcomp(pieces[tx_i]))
                    exon_coords.append((s, s + l))
                    if i < n_ex - 1:
                        emit("".join(rng.choice("ACGT") for _ in range(introns[i])))
            gend = pos
            if lower:
                # soft-mask the whole gene region
                joined = "".join(genome)
                genome[:] = [joined[:gstart], joined[gstart:gend].lower()]
            genes.append(dict(id=gid, reverse=reverse, start=gstart, end=gend, exons=exon_coords, n_ex=n_ex))
            emit("".join(rng.choice("ACGT") for _ in range(rng.randint(500, 1500))))
            cds_nt += total
        seq = "".join(genome)
        contigs.append((cname, seq))

        # ---- GTF
        for g in genes:
            strand = "-" if g["reverse"] else "+"
            gname = "G%05d" % g["id"]
            ga = 'gene_id "ENSG%08d"; gene_version "1"; gene_name "%s"; gene_source "synth"; gene_biotype "protein_coding";' % (g["id"], gname)
            gtf_lines.append("%s\tsynth\tgene\t%d\t%d\t.\t%s\t.\t%s" % (cname, g["start"] + 1, g["end"], strand, ga))
            gene_reverse, gene_strand = g["reverse"], strand
            g = dict(g)
            for ti in range(p.transcripts_per_gene):
                n_tx += 1
                # an antisense transcript reads the same exons from the other strand (its ORF is whatever the sequence gives)
                flip = ti > 0 and rng.random() < p.antisense_frac
                g["reverse"] = (not gene_reverse) if flip else gene_reverse
                strand = ("+" if gene_strand == "-" else "-") if flip else gene_strand
                ta = ga[:-1] + '; transcript_id "ENST%08d%02d"; transcript_name "%s-2%02d"; transcript_biotype "protein_coding";' % (g["id"], ti, gname, ti)
                gtf_lines.append("%s\tsynth\ttranscript\t%d\t%d\t.\t%s\t.\t%s" % (cname, g["start"] + 1, g["end"], strand, ta))
                ex = g["exons"][::-1] if g["reverse"] else g["exons"]
                # alternative transcripts drop one internal exon whose length is a multiple of 3
                if ti > 0 and len(ex) > 2:
                    cands = [i for i in range(1, len(ex) - 1) if (ex[i][1] - ex[i][0]) % 3 == 0]
                    if cands:
                        drop = rng.choice(cands)
                        ex = ex[:drop] + ex[drop + 1:]
                consumed = 0
                first_frame = rng.randint(1, 2) if (p.first_frame and rng.random() < 0.3) else 0
                for i, (s, e) in enumerate(ex):
                    frame = (3 - consumed % 3) % 3
                    if i == 0:
                        frame = first_frame
                    gtf_lines.append("%s\tsynth\texon\t%d\t%d\t.\t%s\t.\t%s exon_number \"%d\";" % (cname, s + 1, e, strand, ta, i + 1))
                    gtf_lines.append("%s\tsynth\tCDS\t%d\t%d\t.\t%s\t%d\t%s exon_number \"%d\";" % (cname, s + 1, e, strand, frame, ta, i + 1))
                    if i == 0 and first_frame == 0:
                        if g["reverse"]:
                            gtf_lines.append("%s\tsynth\tstart_codon\t%d\t%d\t.\t%s\t0\t%s" % (cname, e - 2, e, strand, ta))
                        else:
                            gtf_lines.append("%s\tsynth\tstart_codon\t%d\t%d\t.\t%s\t0\t%s" % (cname, s + 1, s + 3, strand, ta))
                    consumed += e - s
                ls, le = ex[-1]
                if g["reverse"]:
                    gtf_lines.append("%s\tsynth\tstop_codon\t%d\t%d\t.\t%s\t0\t%s" % (cname, ls - 2, ls, strand, ta))
                    gtf_lines.append("%s\tsynth\tthree_prime_utr\t%d\t%d\t.\t%s\t.\t%s" % (cname, ls - 3 - p.utr3 + 1, ls, strand, ta))
                else:
                    gtf_lines.append("%s\tsynth\tstop_codon\t%d\t%d\t.\t%s\t0\t%s" % (cname, le + 1, le + 3, strand, ta))
                    gtf_lines.append("%s\tsynth\tthree_prime_utr\t%d\t%d\t.\t%s\t.\t%s" % (cname, le + 1, le + 3 + p.utr3, strand, ta))

        # ---- variants
        variants = {}  # pos -> (ref, [alts], somatic, het_hap, vaf)
        for g in genes:
            spans = list(g["exons"])
            if p.variants_in_introns:
                spans.append((g["start"], g["end"]))
            for (s, e) in g["exons"]:
                n_g = _poisson(rng, (e - s) * p.germline_per_kb / 1000.0)
                n_s = _poisson(rng, (e - s) * p.somatic_per_kb / 1000.0)
                for somatic in [False] * n_g + [True] * n_s:
                    vp = rng.randint(s, e - 1)
                    _add_variant(rng, p, seq, variants, vp, somatic)
            if p.hotspot_per_gene:
                wide = [(s, e) for (s, e) in g["exons"] if e - s >= 27] or list(g["exons"])
                s, e = rng.choice(wide)
                b = rng.randint(s, max(s, e - 27))
                for vp in rng.sample(range(b, min(b + 27, e)), min(p.hotspot_per_gene, min(b + 27, e) - b)):
                    _add_variant(rng, p, seq, variants, vp, True, snv_only=True)
            if p.start_loss_frac and rng.random() < p.start_loss_frac:
                ex = g["exons"][-1] if g["reverse"] else g["exons"][0]
                vp = (ex[1] - 1 - rng.randint(0, 2)) if g["reverse"] else ex[0] + rng.randint(0, 2)
                _add_variant(rng, p, seq, variants, vp, rng.random() < 0.5, snv_only=True)
            if p.variants_in_introns:
                for _ in range(_poisson(rng, 1.0)):
                    _add_variant(rng, p, seq, variants, rng.randint(g["start"], g["end"] - 1), rng.random() < 0.5)
        for vp in sorted(variants):
            ref, alts, somatic, _, _ = variants[vp]
            info = "DP=100" + (";SOMATIC" if somatic else "")
            vcf_rows.append("%s\t%d\t.\t%s\t%s\t100\t.\t%s" % (cname, vp + 1, ref.upper(), ",".join(alts), info))

        # ---- reads
        vpos = sorted(variants)
        import bisect
        for g in genes:
            lo = max(0, g["start"] - p.read_len)
            hi = min(len(seq) - p.read_len - 10, g["end"] + 20)
            # cover exons only (exome capture): reads starting within [exon.start - L, exon.end]
            starts = []
            for (s, e) in g["exons"]:
                a, b = max(lo, s - p.read_len), min(hi, e + 5)
                if b <= a:
                    continue
                n = int(round(p.coverage * (b - a) / p.read_len))
                starts.extend(rng.randint(a, b) for _ in range(n))
            for st in starts:
                hap = rng.randint(0, 1)
                take_somatic = rng.random()
                cigar = []
                rs = []
                rp = st
                i0 = bisect.bisect_left(vpos, st)
                vi = i0
                noise = rng.random() < p.noise_indel_frac
                noise_at = rng.randint(10, p.read_len - 10) if noise else -1
                noise_kind = rng.choice("ID")
                noise_len = rng.randint(1, 6)

                def push(op, l):
                    if cigar and cigar[-1][0] == op:
                        cigar[-1] = (op, cigar[-1][1] + l)
                    else:
                        cigar.append((op, l))

                while len(rs) < p.read_len and rp < len(seq) - 1:
                    if len(rs) == noise_at and noise_at > 0:
                        noise_at = -1
                        if noise_kind == "I":
                            ins = "".join(rng.choice("ACGT") for _ in range(noise_len))[:p.read_len - len(rs)]
                            rs.extend(ins)
                            push("I", len(ins))
                            continue
                        else:
                            rp += noise_len
                            push("D", noise_len)
                            continue
                    while vi < len(vpos) and vpos[vi] < rp:
                        vi += 1
                    applied = False
                    if vi < len(vpos) and vpos[vi] == rp:
                        ref, alts, somatic, vhap, vaf = variants[rp]
                        carry = ((rng.random() if p.independent_somatic else take_somatic) < vaf) if somatic else (vhap == 2 or vhap == hap)
                        if carry:
                            alt = alts[(hap + st) % len(alts)]
                            if len(ref) == 1 and len(alt) == 1:
                                rs.append(alt)
                                push("M", 1)
                                rp += 1
                                applied = True
                            elif len(ref) == 1 and len(alt) > 1 and len(rs) + len(alt) <= p.read_len and len(rs) > 0:
                                rs.append(alt[0])
                                push("M", 1)
                                rs.extend(alt[1:])
                                push("I", len(alt) - 1)
                                rp += 1
                                applied = True
                            elif len(ref) > 1 and len(rs) > 0 and len(rs) + 1 < p.read_len:
                                rs.append(ref[0].upper())
                                push("M", 1)
                                push("D", len(ref) - 1)
                                rp += len(ref)
                                applied = True
                    if not applied:
                        rs.append(seq[rp].upper())
                        push("M", 1)
                        rp += 1
                if len(rs) < 30:
                    continue
                # trailing I/D are not valid alignments: trim
                while cigar and cigar[-1][0] in "ID":
                    op, l = cigar.pop()
                    if op == "I":
                        del rs[-l:]
                if not cigar:
                    continue
                pos0 = st
                if rng.random() < p.softclip_frac and cigar[0][0] == "M" and cigar[0][1] > 12:
                    c = rng.randint(1, 10)
                    cigar[0] = ("M", cigar[0][1] - c)
                    cigar.insert(0, ("S", c))
                    pos0 += c
                    for i in range(c):
                        rs[i] = rng.choice("ACGT")
                if rng.random() < p.softclip_frac and cigar[-1][0] == "M" and cigar[-1][1] > 12:
                    c = rng.randint(1, 10)
                    cigar[-1] = ("M", cigar[-1][1] - c)
                    cigar.append(("S", c))
                qual = [rng.randint(30, 40) for _ in rs]
                for i in range(len(qual)):
                    if rng.random() < p.lowq_frac:
                        qual[i] = rng.randint(2, 9)
                flag = 0
                mapq = 60
                if rng.random() < p.mapq0_frac:
                    mapq = rng.randint(0, 4)
                if rng.random() < p.unmapped_frac:
                    flag |= 4
                qn = "r%09d" % len(bam_recs)
                bam_recs.append((ci, pos0, mapq, flag, qn, list(cigar), "".join(rs), qual))
                if rng.random() < p.dup_mate_frac:
                    # mate with the same qname and the same start, slightly different length
                    k = rng.randint(0, 8)
                    if cigar[-1][0] == "M" and cigar[-1][1] > k + 2 and k > 0:
                        cig2 = list(cigar)
                        cig2[-1] = ("M", cig2[-1][1] - k)
                        bam_recs.append((ci, pos0, mapq, flag | 128, qn, cig2, "".join(rs[:-k]), qual[:-k]))
                    else:
                        bam_recs.append((ci, pos0, mapq, flag | 128, qn, list(cigar), "".join(rs), list(qual)))
                    while rng.random() < p.dup_extra_frac:
                        bam_recs.append((ci, pos0, mapq, flag | 256, qn, list(cigar), "".join(rs), list(qual)))

    # ---- write files
    with open(os.path.join(outdir, "ref.fa"), "w") as f, open(os.path.join(outdir, "ref.fa.fai"), "w") as fai:
        off = 0
        for name, seq in contigs:
            hdr = ">%s\n" % name
            f.write(hdr)
            off += len(hdr)
            fai.write("%s\t%d\t%d\t60\t61\n" % (name, len(seq), off))
            for i in range(0, len(seq), 60):
                f.write(seq[i:i + 60] + "\n")
            off += len(seq) + (len(seq) + 59) // 60
    with open(os.path.join(outdir, "annotation.gtf"), "w") as f:
        f.write("\n".join(gtf_lines) + "\n")
    with open(os.path.join(outdir, "variants.vcf"), "w") as f:
        f.write("##fileformat=VCFv4.2\n")
        for name, seq in contigs:
            f.write("##contig=<ID=%s,length=%d>\n" % (name, len(seq)))
        f.write('##INFO=<ID=DP,Number=1,Type=Integer,Description="depth">\n')
        f.write('##INFO=<ID=SOMATIC,Number=0,Type=Flag,Description="Somatic variant">\n')
        f.write("#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n")
        f.write("\n".join(vcf_rows) + ("\n" if vcf_rows else ""))
    bam_recs.sort(key=lambda r: (r[0], r[1]))
    text = "@HD\tVN:1.6\tSO:coordinate\n" + "".join("@SQ\tSN:%s\tLN:%d\n" % (n, len(s)) for n, s in contigs)
    raw = [b"BAM\x01", struct.pack("<i", len(text)), text.encode(), struct.pack("<i", len(contigs))]
    for n, s in contigs:
        raw.append(struct.pack("<i", len(n) + 1) + n.encode() + b"\0" + struct.pack("<i", len(s)))
    for r in bam_recs:
        raw.append(_bam_record(*r))
    with open(os.path.join(outdir, "reads.bam"), "wb") as f:
        f.write(_bgzf_blocks(b"".join(raw)))
    return dict(contigs=len(contigs), transcripts=n_tx, reads=len(bam_recs), variants=len(vcf_rows), cds_nt=cds_nt)


def _poisson(rng, lam):
    import math
    if lam <= 0:
        return 0
    l, k, pr = math.exp(-lam), 0, 1.0
    while True:
        pr *= rng.random()
        if pr <= l:
            return k
        k += 1


def _add_variant(rng, p, seq, variants, vp, somatic, snv_only=False):
    if vp in variants or vp + 12 >= len(seq) or vp < 1:
        return
    ref = seq[vp].upper()
    vhap = rng.choice([0, 1, 2])
    vaf = rng.uniform(0.1, 0.5)
    r = rng.random()
    if not snv_only and r < p.indel_frac:
        l = rng.randint(1, 6) if p.frameshift_ok else rng.choice([3, 6])
        if rng.random() < 0.5:
            alt = ref + "".join(rng.choice("ACGT") for _ in range(l))
            variants[vp] = (ref, [alt], somatic, vhap, vaf)
        else:
            # deletions must not swallow another variant's anchor
            if any((vp + d) in variants for d in range(1, l + 1)):
                return
            variants[vp] = (seq[vp:vp + l + 1].upper(), [ref], somatic, vhap, vaf)
        return
    alts = [rng.choice([b for b in "ACGT" if b != ref])]
    if not snv_only and rng.random() < p.multiallelic_frac:
        alts.append(rng.choice([b for b in "ACGT" if b != ref and b not in alts]))
    variants[vp] = (ref, alts, somatic, vhap, vaf)
