"""Minimal writers for unaligned SAM / BAM read files (test inputs for the BAM/SAM ingest, reads.cpp:120-143).
BGZF = gzip members with the 'BC' extra subfield (block size), as samtools' bgzf.c requires."""
from __future__ import annotations

import struct
import zlib

NT16 = "=ACMGRSVTWYHKDBN"


def bgzf_block(data: bytes) -> bytes:
    c = zlib.compressobj(6, zlib.DEFLATED, -15)
    comp = c.compress(data) + c.flush()
    bsize = len(comp) + 25                      # total block size - 1
    head = struct.pack("<BBBBIBBHBBHH", 0x1f, 0x8b, 8, 4, 0, 0, 0xff, 6, ord("B"), ord("C"), 2, bsize)
    return head + comp + struct.pack("<II", zlib.crc32(data) & 0xffffffff, len(data))


def bgzf(data: bytes, block=60000) -> bytes:
    out = b"".join(bgzf_block(data[i:i + block]) for i in range(0, len(data), block))
    return out + bgzf_block(b"")                 # EOF marker


def bam_record(name: str, flag: int, seq: str, qual) -> bytes:
    """unmapped record; qual: str (phred+33) or None"""
    l = len(seq)
    codes = [NT16.index(ch.upper()) if ch.upper() in NT16 else 15 for ch in seq]
    if l & 1:
        codes.append(0)
    packed = bytes((codes[i] << 4) | codes[i + 1] for i in range(0, len(codes), 2))
    q = bytes([0xff] * l) if qual is None else bytes(ord(c) - 33 for c in qual)
    qn = name.encode() + b"\0"
    core = struct.pack("<iiBBHHHiiii", -1, -1, len(qn), 0, 4680, 0, flag, l, -1, -1, 0)
    body = core + qn + packed + q
    return struct.pack("<i", len(body)) + body


def write_bam(path, records, header_text="@HD\tVN:1.0\tSO:unsorted\n"):
    """records: iterable of (name, flag, seq, qual)"""
    raw = b"BAM\1" + struct.pack("<i", len(header_text)) + header_text.encode() + struct.pack("<i", 0)
    raw += b"".join(bam_record(*r) for r in records)
    open(path, "wb").write(bgzf(raw))


def write_sam(path, records):
    """headerless SAM text (the reference's CheckFile takes a leading '@' for FASTQ)"""
    with open(path, "w") as f:
        for name, flag, seq, qual in records:
            f.write("\t".join([name, str(flag), "*", "0", "0", "*", "*", "0", "0", seq or "*", qual if qual is not None else "*"]) + "\n")


def aligned_bam_from_sam(path, sam: str, extra_names=()):
    """SAM text (numeric FLAG, @SQ header; Z and i tags) -> an aligned, unsorted BAM file in the same record order.
    Reference names are the @SQ names, then extra_names (records on names outside the FASTA).  BAM stores no lowercase:
    SEQ is upper-cased; SEQ '*' becomes l_seq 0."""
    names, recs = [], []
    for line in sam.splitlines():
        if line.startswith("@SQ"):
            f = dict(x.split(":", 1) for x in line.split("\t")[1:])
            names.append((f["SN"], int(f["LN"])))
    names += [(n, 1) for n in extra_names]
    rid = {n: i for i, (n, _) in enumerate(names)}
    for line in sam.splitlines():
        if line.startswith("@") or not line:
            continue
        c = line.split("\t")
        seq = "" if c[9] == "*" else c[9]
        l = len(seq)
        codes = [NT16.index(ch.upper()) if ch.upper() in NT16 else 15 for ch in seq] + ([0] if l & 1 else [])
        packed = bytes((codes[i] << 4) | codes[i + 1] for i in range(0, len(codes), 2))
        cig = b"" if c[5] == "*" else struct.pack("<I", int(c[5][:-1]) << 4)
        tags = b""
        for t in c[11:]:
            tg, ty, v = t.split(":", 2)
            tags += tg.encode() + (b"Z" + v.encode() + b"\0" if ty == "Z" else b"i" + struct.pack("<i", int(v)))
        qn = c[0].encode() + b"\0"
        ref = rid[c[2]]
        core = struct.pack("<iiBBHHHiiii", ref, int(c[3]) - 1, len(qn), 255, 4680, len(cig) // 4, int(c[1]), l,
                           ref if c[6] != "*" else -1, int(c[7]) - 1, int(c[8]))
        body = core + qn + cig + packed + bytes([0xff] * l) + tags
        recs.append(struct.pack("<i", len(body)) + body)
    head = "@HD\tVN:1.0\tSO:unsorted\n"
    raw = b"BAM\1" + struct.pack("<i", len(head)) + head.encode() + struct.pack("<i", len(names))
    for n, ln in names:
        raw += struct.pack("<i", len(n) + 1) + n.encode() + b"\0" + struct.pack("<i", ln)
    open(path, "wb").write(bgzf(raw + b"".join(recs)))


def bam_to_sam_text(path) -> str:
    """an aligned BAM file as headerless SAM text (what `samtools view` prints, numeric FLAG; Z / A / integer tags only):
    lets the methratio oracle, which reads text, see the records of a BAM file in the file's own order"""
    import gzip
    raw = gzip.open(path, "rb").read()
    assert raw[:4] == b"BAM\1"
    l_text, = struct.unpack_from("<i", raw, 4)
    o = 8 + l_text
    n_ref, = struct.unpack_from("<i", raw, o); o += 4
    names = []
    for _ in range(n_ref):
        ln, = struct.unpack_from("<i", raw, o)
        names.append(raw[o + 4:o + 4 + ln - 1].decode()); o += 4 + ln + 4
    out = []
    while o + 4 <= len(raw):
        bs, = struct.unpack_from("<i", raw, o)
        b = raw[o + 4:o + 4 + bs]; o += 4 + bs
        ref, pos, l_name, mapq, _bin, n_cig, flag, l_seq, nref, npos, tlen = struct.unpack_from("<iiBBHHHiiii", b, 0)
        x = 32
        qname = b[x:x + l_name - 1].decode(); x += l_name
        cig = "".join("%d%s" % (v >> 4, "MIDNSHP=X"[v & 15]) for v in struct.unpack_from("<%dI" % n_cig, b, x)) or "*"; x += 4 * n_cig
        seq = "".join(NT16[(b[x + (i >> 1)] >> (4 if i % 2 == 0 else 0)) & 15] for i in range(l_seq)) or "*"; x += (l_seq + 1) // 2
        qual = "*" if l_seq == 0 or b[x] == 0xff else "".join(chr(c + 33) for c in b[x:x + l_seq]); x += l_seq
        tags = []
        while x + 3 <= len(b):
            tg, ty = b[x:x + 2].decode(), chr(b[x + 2]); x += 3
            if ty == "Z":
                e = b.index(b"\0", x); tags.append("%s:Z:%s" % (tg, b[x:e].decode())); x = e + 1
            elif ty == "A":
                tags.append("%s:A:%s" % (tg, chr(b[x]))); x += 1
            else:
                fmt = {"c": "<b", "C": "<B", "s": "<h", "S": "<H", "i": "<i", "I": "<I"}[ty]
                tags.append("%s:i:%d" % (tg, struct.unpack_from(fmt, b, x)[0])); x += struct.calcsize(fmt)
        rn = names[ref] if ref >= 0 else "*"
        rnext = "*" if nref < 0 else ("=" if nref == ref else names[nref])
        out.append("\t".join([qname, str(flag), rn, str(pos + 1), str(mapq), cig, rnext, str(npos + 1), str(tlen), seq, qual] + tags))
    return "\n".join(out) + ("\n" if out else "")
