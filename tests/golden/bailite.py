"""Pure-Python BAM index (.bai, SAM specification section 5.2) writer, test infrastructure only.

It shares nothing with the product's reader (csrc/io/bam_index.hpp): its own BGZF block walk, reg2bin, 16 kb linear index,
chunk merging and pseudo-bin counts, so that an index it writes checks the reader from outside.

    python bailite.py reads.bam [out.bai]      # default: reads.bam.bai
"""
import struct
import sys
import zlib


def reg2bin(beg, end):
    """The bin of [beg, end) (SAM specification section 5.3)."""
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


def _blocks(data):
    """(file offset, inflated bytes) of every BGZF block."""
    o = 0
    while o < len(data):
        if data[o:o + 4] != b"\x1f\x8b\x08\x04":
            raise ValueError("not BGZF at %d" % o)
        xlen = struct.unpack_from("<H", data, o + 10)[0]
        e, bsize = o + 12, None
        while e + 4 <= o + 12 + xlen:
            si1, si2, slen = data[e], data[e + 1], struct.unpack_from("<H", data, e + 2)[0]
            if si1 == 66 and si2 == 67:
                bsize = struct.unpack_from("<H", data, e + 4)[0] + 1
            e += 4 + slen
        yield o, zlib.decompress(data[o + 12 + xlen:o + bsize - 8], -15)
        o += bsize


def _records(path):
    """(n_ref, [(tid, beg, end, flag, start voff, end voff)]) in file order."""
    data = open(path, "rb").read()
    stream, starts = bytearray(), []  # starts: (inflated offset, file offset) per block
    for coff, raw in _blocks(data):
        starts.append((len(stream), coff))
        stream += raw
    starts.append((len(stream), len(data)))

    def voff(u):
        lo, hi = 0, len(starts) - 1
        while lo < hi:  # last block starting at or before u whose data is not empty at u
            mid = (lo + hi + 1) // 2
            if starts[mid][0] <= u:
                lo = mid
            else:
                hi = mid - 1
        while lo + 1 < len(starts) and starts[lo + 1][0] == u:
            lo += 1
        return (starts[lo][1] << 16) | (u - starts[lo][0])

    assert stream[:4] == b"BAM\x01"
    o = 8 + struct.unpack_from("<i", stream, 4)[0]
    n_ref = struct.unpack_from("<i", stream, o)[0]
    o += 4
    for _ in range(n_ref):
        o += 8 + struct.unpack_from("<i", stream, o)[0]
    recs = []
    while o < len(stream):
        bs = struct.unpack_from("<i", stream, o)[0]
        tid, pos, l_rn, _mapq, _bin, n_cig, flag = struct.unpack_from("<iiBBHHH", stream, o + 4)
        q = o + 4 + 32 + l_rn
        rlen = 0
        for i in range(n_cig):
            c = struct.unpack_from("<I", stream, q + 4 * i)[0]
            if c & 15 in (0, 2, 3, 7, 8):
                rlen += c >> 4
        end = pos + max(rlen, 1)
        recs.append((tid, pos, end, flag, voff(o), voff(o + 4 + bs)))
        o += 4 + bs
    return n_ref, recs


def build(bam_path):
    """The index of a coordinate-sorted BAM as bytes."""
    n_ref, recs = _records(bam_path)
    refs = [dict(bins={}, lin={}, first=None, last=None, mapped=0, unmapped=0) for _ in range(n_ref)]
    n_no_coor = 0
    prev = None  # (tid, bin) of the previous record: consecutive records of one bin share a chunk
    for tid, beg, end, flag, v0, v1 in recs:
        if tid < 0 or beg < 0:
            n_no_coor += 1
            prev = None
            continue
        r = refs[tid]
        b = reg2bin(beg, end)
        chunks = r["bins"].setdefault(b, [])
        if prev == (tid, b) and chunks and chunks[-1][1] == v0:
            chunks[-1][1] = v1
        else:
            chunks.append([v0, v1])
        prev = (tid, b)
        for w in range(beg >> 14, ((end - 1) >> 14) + 1):
            r["lin"].setdefault(w, v0)
        r["first"] = v0 if r["first"] is None else r["first"]
        r["last"] = v1
        if flag & 4:
            r["unmapped"] += 1
        else:
            r["mapped"] += 1
    out = bytearray(b"BAI\x01" + struct.pack("<i", n_ref))
    for r in refs:
        bins = sorted(r["bins"].items())
        has_meta = r["first"] is not None
        out += struct.pack("<i", len(bins) + (1 if has_meta else 0))
        for b, chunks in bins:
            merged = []
            for c in chunks:  # chunks that meet inside one BGZF block are read as one
                if merged and merged[-1][1] >> 16 == c[0] >> 16:
                    merged[-1][1] = max(merged[-1][1], c[1])
                else:
                    merged.append(list(c))
            out += struct.pack("<Ii", b, len(merged))
            for c in merged:
                out += struct.pack("<QQ", c[0], c[1])
        if has_meta:
            out += struct.pack("<IiQQQQ", 37450, 2, r["first"], r["last"], r["mapped"], r["unmapped"])
        n_lin = (max(r["lin"]) + 1) if r["lin"] else 0
        lin, last = [], 0
        for w in range(n_lin):  # windows no record overlaps take the offset of the window before
            last = r["lin"].get(w, last)
            lin.append(last)
        out += struct.pack("<i", n_lin) + struct.pack("<%dQ" % n_lin, *lin)
    out += struct.pack("<Q", n_no_coor)
    return bytes(out)


def write(bam_path, bai_path=None):
    bai_path = bai_path or bam_path + ".bai"
    with open(bai_path, "wb") as f:
        f.write(build(bam_path))
    return bai_path


if __name__ == "__main__":
    print(write(sys.argv[1], sys.argv[2] if len(sys.argv) > 2 else None))
