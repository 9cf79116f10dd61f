"""Host ingest (bsx_reads_*) and multi-threaded emit (bsx_emit_*) -- no GPU needed.

The record cutter must load exactly what the reference's ifstream token reader loads
(reads.cpp:83-119); the chunked emit must write the bytes of the unmodified reference (golden files).
"""
from __future__ import annotations

import os

import numpy as np
import pytest

import cases as CS
import runners as R

import bsmap_b200 as B
from bsmap_b200 import lib as BL

pytestmark = pytest.mark.skipif(not os.path.exists(BL.LIB_PATH), reason="library not built")


def load_all(path, want=7, threads=3, token=False, stride=64, max_readlen=144):
    r = B.Reads(path, max_readlen=max_readlen)
    if token:
        r.force_token_reader()
    out = []
    while True:
        n, buf, lens = r.next(want, stride=stride, threads=threads)
        if n == 0:
            break
        for i in range(n):
            name, seq, qual = r.get(i)
            assert bytes(buf[i, :lens[i]]) == seq[:stride]
            assert not buf[i, lens[i]:].any()
            out.append((name, seq, qual))
        if n < want:
            break
    kind = r.kind
    r.close()
    return kind, out


def python_token_reader(data: bytes, fastq: bool, max_readlen=144, zero_qual=ord("!")):
    """reads.cpp:90-113 restated with str.split semantics: `>>` = next whitespace-delimited token"""
    pos, n, out = 0, len(data), []
    WS = b" \t\n\r\f\v"

    def skip_ws():
        nonlocal pos
        while pos < n and data[pos] in WS:
            pos += 1

    def token():
        nonlocal pos
        skip_ws()
        s = pos
        while pos < n and data[pos] not in WS:
            pos += 1
        return data[s:pos] if pos > s else None

    def getline():
        nonlocal pos
        e = data.find(b"\n", pos)
        pos = n if e < 0 else e + 1

    while True:
        skip_ws()
        if pos >= n:
            break
        pos += 1                      # fin >> c
        name = token()
        if name is None:
            break
        getline()
        seq = token() or b""
        if fastq:
            token(); getline()
            qual = token() or b""
        else:
            qual = bytes([zero_qual + 40]) * len(seq)
        if len(seq) > max_readlen:
            seq, qual = seq[:max_readlen], qual[:max_readlen]
        out.append((name, seq, qual))
    return out


REGULAR_FQ = b"".join(b"@r%d extra words\nACGTNACGT%s\n+\nIIIIIIIII%s\n" % (i, b"A" * (i % 5), b"#" * (i % 5)) for i in range(53))
IRREGULAR = {
    "crlf": REGULAR_FQ.replace(b"\n", b"\r\n"),
    "no_final_newline": REGULAR_FQ[:-1],
    "blank_lines": REGULAR_FQ.replace(b"@r7 ", b"\n\n@r7 ").replace(b"@r30 ", b"\n@r30 "),
    "indented_header": REGULAR_FQ.replace(b"@r11 ", b"  @r11 "),
    "space_after_at": REGULAR_FQ.replace(b"@r5 ", b"@ r5 "),
    "trailing_blanks": REGULAR_FQ.replace(b"ACGTNACGTAA\n", b"ACGTNACGTAA  \t\n"),
    "junk_after_seq": REGULAR_FQ.replace(b"ACGTNACGTAAA\n", b"ACGTNACGTAAA junk\n", 1),
    "plus_with_name": REGULAR_FQ.replace(b"\n+\n", b"\n+again here\n"),
    "truncated_record": REGULAR_FQ + b"@tail\nACGT\n",
    "only_header": REGULAR_FQ + b"@tail",
    "long_reads": b"".join(b"@L%d\n%s\n+\n%s\n" % (i, b"ACGT" * 50, b"I" * 200) for i in range(9)),
}
REGULAR_FA = b"".join(b">s%d desc\nACGTTGCA%s\n" % (i, b"C" * (i % 3)) for i in range(41))
IRREGULAR_FA = {
    "fa_regular": REGULAR_FA,
    "fa_blank": REGULAR_FA.replace(b">s9 ", b"\n>s9 "),
    "fa_wrapped": REGULAR_FA.replace(b"ACGTTGCAC\n", b"ACGT\nTGCAC\n", 2),
    "fa_no_newline": REGULAR_FA[:-1],
}


@pytest.mark.parametrize("name", ["regular"] + sorted(IRREGULAR) + sorted(IRREGULAR_FA))
def test_record_cutter_equals_token_reader(tmp_path, name):
    data = REGULAR_FQ if name == "regular" else IRREGULAR.get(name, IRREGULAR_FA.get(name))
    fastq = not name.startswith("fa_")
    path = tmp_path / "reads.txt"
    path.write_bytes(data)
    exp = python_token_reader(data, fastq)
    for want, threads in ((7, 3), (1000, 1), (1, 2), (16, 8)):
        kind, fast = load_all(str(path), want=want, threads=threads)
        assert kind == ("fastq" if fastq else "fasta")
        assert fast == exp, (name, want, threads)
    _, slow = load_all(str(path), token=True)
    assert slow == exp


def test_regular_input_takes_the_line_cutter(tmp_path):
    """the fast path must actually be the one that runs on ordinary files"""
    path = tmp_path / "r.fq"
    path.write_bytes(REGULAR_FQ)
    r = B.Reads(str(path))
    n, buf, lens = r.next(1000, stride=32, threads=4)
    assert n == 53 and lens[0] == 9 and bytes(buf[1, :10]) == b"ACGTNACGTA"
    r.close()


@pytest.mark.parametrize("empty_lines", [False, True])
def test_growing_records_span_several_scan_windows(tmp_path, empty_lines):
    """records that keep getting longer defeat the window estimate: the cutter must come back for more;
    with every other sequence line empty the file is irregular throughout and the two readers interleave"""
    path = tmp_path / "grow.fq"
    n_rec = 60_000
    with open(path, "wb") as f:
        for i in range(n_rec):
            l = 10 + i // 450
            base = b"" if (empty_lines and i % 4 == 1) else b"ACGT"[(i & 3):(i & 3) + 1]
            f.write(b"@g%d\n%s\n+\n%s\n" % (i, base * l, b"F" * l))
    for want in (25_000, n_rec + 1):
        _, fast = load_all(str(path), want=want, threads=8, stride=160)
        _, slow = load_all(str(path), want=want, token=True, stride=160)
        assert fast == slow
        assert empty_lines or len(fast) == n_rec


def test_gzip_input(tmp_path):
    """gzip'ed read and reference files are inflated transparently (extension over the reference)"""
    import gzip
    plain, gz = tmp_path / "r.fq", tmp_path / "r.fq.gz"
    plain.write_bytes(REGULAR_FQ)
    with gzip.open(gz, "wb") as f:
        f.write(REGULAR_FQ)
    assert load_all(str(gz)) == load_all(str(plain))
    fa, fagz = tmp_path / "g.fa", tmp_path / "g.fa.gz"
    fa.write_bytes(b">chr1 x\nACGTACGTNN\nacgt\n>chr2\nGGGG\n")
    with gzip.open(fagz, "wb") as f:
        f.write(fa.read_bytes())
    p = B.make_params()
    a, b = B.Index.text_only_from_fasta(p, str(fa)), B.Index.text_only_from_fasta(p, str(fagz))
    assert a.header() == b.header() and np.array_equal(a.download("refcat"), b.download("refcat"))


def test_bam_input(tmp_path):
    """BAM read files (reads.cpp:120-143): 4-bit bases come back upper-cased / as 'N', qualities + 33, over-long reads
    truncated; file a of an interleaved pair takes every other record and drops a last read without a mate; -B does not skip"""
    import bamio
    recs = [("r%d" % i, 4, s, q) for i, (s, q) in enumerate([("ACGTNacgtn", "IIIIIFFFFF"), ("ACRYKM.xTT", None), ("A" * 200, "#" * 200), ("GGG", "!J~")])]
    bam = str(tmp_path / "r.bam")
    bamio.write_bam(bam, recs)
    r = B.Reads(bam, max_readlen=144)
    assert r.kind == "bam"
    r.skip(2)                                     # reference quirk: no effect on BAM
    n, buf, lens = r.next(10, stride=160)
    got = [r.get(i) for i in range(n)]
    assert got == [(b"r0", b"ACGTNACGTN", b"IIIIIFFFFF"), (b"r1", b"ACRYKMNNTT", b" " * 10), (b"r2", b"A" * 144, b"#" * 144), (b"r3", b"GGG", b"!J~")]
    assert list(lens) == [10, 10, 144, 3] and bytes(buf[1, :10]) == b"ACRYKMNNTT"
    r.close()
    pe = [("p%d/%d" % (i // 2, i % 2 + 1), 0x4d if i % 2 == 0 else 0x8d, "ACGT" * 5, "F" * 20) for i in range(9)]   # 4 pairs + a lone first mate
    bam2 = str(tmp_path / "pe.bam")
    bamio.write_bam(bam2, pe)
    ra, rb = B.Reads(bam2), B.Reads(bam2)
    ra.set_readset(1); rb.set_readset(2)
    na, nb = ra.next(100)[0], rb.next(100)[0]
    assert (na, nb) == (4, 4)
    assert [ra.get(i)[0] for i in range(4)] == [b"p%d/1" % i for i in range(4)] and [rb.get(i)[0] for i in range(4)] == [b"p%d/2" % i for i in range(4)]
    ra.close(); rb.close()


def test_bam_input_is_streamed_over_many_windows(tmp_path):
    """a BAM of ~45 MB inflated (the reader's windows are 16-24 MB): every record comes back, single-end and as the two files
    of an interleaved pair, also through a FIFO"""
    import bamio
    import threading
    rng = np.random.default_rng(8)
    n = 300_000
    seqs = ["".join("ACGT"[c] for c in rng.integers(0, 4, int(L))) for L in rng.integers(60, 145, 2000)]
    recs = [("read_%07d" % i, 0x4d if i % 2 == 0 else 0x8d, seqs[i % 2000], "F" * len(seqs[i % 2000])) for i in range(n)]
    bam = str(tmp_path / "big.bam")
    bamio.write_bam(bam, recs)

    def names_of(path, readset, want):
        r = B.Reads(path)
        r.set_readset(readset)
        out = []
        while True:
            k, buf, lens = r.next(want, stride=160)
            for i in (0, k // 2, k - 1) if k else ():
                nm, sq, ql = r.get(i)
                j = len(out) + i
                src = recs[j] if readset == 0 else recs[2 * j + (readset - 1)]
                assert (nm.decode(), sq.decode(), ql.decode()) == (src[0], src[2], src[3]) and bytes(buf[i, :lens[i]]) == sq
            out += [None] * k
            if k < want:
                break
        r.close()
        return len(out)

    assert names_of(bam, 0, 70_000) == n
    assert names_of(bam, 1, 50_000) == n // 2 and names_of(bam, 2, 50_000) == n // 2
    fifo = str(tmp_path / "fifo.bam")
    os.mkfifo(fifo)
    t = threading.Thread(target=lambda: open(fifo, "wb").write(open(bam, "rb").read()))
    t.start()
    assert names_of(fifo, 0, 65_536) == n
    t.join()


def test_skip_and_errors(tmp_path):
    path = tmp_path / "r.fq"
    path.write_bytes(REGULAR_FQ)
    r = B.Reads(str(path))
    r.skip(50)                                     # -B 51
    n, _, _ = r.next(100)
    assert n == 3 and r.get(0)[0] == b"r50"
    with pytest.raises(B.BsxError):
        r.get(3)
    r.close()
    with pytest.raises(B.BsxError, match="failed to open"):
        B.Reads(str(tmp_path / "missing.fq"))
    bad = tmp_path / "bad.txt"
    bad.write_bytes(b"hello\n")
    with pytest.raises(B.BsxError, match="unrecognizable"):
        B.Reads(str(bad))


def test_reference_fasta_loader(tmp_path):
    """RefSeq::LoadNextSeq (dbseq.cpp:18-54): names = first token, sequence = all non-blank bytes"""
    fa = tmp_path / "g.fa"
    rng = np.random.default_rng(3)
    seqs = [bytes(rng.choice(np.frombuffer(b"ACGTNacgt", dtype=np.uint8), size=n)) for n in (9_000_001, 17, 0, 123_457)]
    names = ["chr%d" % k for k in range(len(seqs))]
    with open(fa, "wb") as f:
        for k, s in enumerate(seqs):
            f.write(b">  chr%d some description\r\n" % k if k == 1 else b">chr%d some >description with a > inside\n" % k)
            for i in range(0, len(s), 60):
                f.write(s[i:i + 60] + (b" \r\n" if k & 1 else b"\n"))
    p = B.make_params()
    got = B.Index.text_only_from_fasta(p, str(fa))
    exp = B.Index.text_only(p, names, seqs)
    assert got.header() == exp.header()
    assert np.array_equal(got.download("refcat"), exp.download("refcat"))
    if BL.load().bsx_device_count() > 0:          # the mapping index, built on the device from the same file
        ix = B.Index.from_fasta(p, str(fa))
        assert ix.header() == exp.header()
        assert np.array_equal(ix.download("refcat"), exp.download("refcat"))
        ix.close()
    else:
        with pytest.raises(B.BsxError, match="no CUDA device"):
            B.Index.from_fasta(p, str(fa))         # the mapping index needs the GPU: no CPU fallback
    with pytest.raises(B.BsxError, match="failed to open"):
        B.Index.text_only_from_fasta(p, str(tmp_path / "missing.fa"))


@pytest.mark.parametrize("case", [c for c in CS.CASES if not c.fasta_reads or not c.paired], ids=lambda c: c.name)
@pytest.mark.parametrize("threads", [1, 5])
def test_emit_reproduces_reference_text(tmp_path, case, threads):
    """read files -> Reads -> oracle records -> bsx_emit_* (threads) == bytes of the unmodified reference"""
    d = case.data()
    got = R.oracle_run(case)
    p = B.make_params(**case.param_kwargs())
    ix = B.Index.text_only(p, d["gnames"], d["gseqs"])
    fa, a, b = CS.write_inputs(case, str(tmp_path))
    L = case.opts.get("L", 144)
    ra = B.Reads(a, max_readlen=L)
    n = len(d["names"])
    assert ra.next(n + 5, threads=threads)[0] == n
    out = tmp_path / "out.txt"
    out2 = tmp_path / "out2.txt"
    head = ix.header() if p.out_sam else b""
    exp_main, exp_un = R.golden_load(case)
    fd = os.open(out, os.O_WRONLY | os.O_CREAT | os.O_TRUNC)
    try:
        if not case.paired:
            w, na = B.emit_se(ix, p, ra, n, got["recs"].astype(BL.REC), got["counts"], fd, threads=threads)
            assert na == got["n_aligned"]
            un = b""
        else:
            rb = B.Reads(b, max_readlen=L)
            assert rb.next(n + 5, threads=threads)[0] == n
            fd2 = os.open(out2, os.O_WRONLY | os.O_CREAT | os.O_TRUNC)
            w, st = B.emit_pe(ix, p, ra, rb, n, got["pr"].astype(BL.PAIR_REC), got["ra"].astype(BL.REC), got["rb"].astype(BL.REC),
                              got["ca"], got["cb"], fd, fd2, threads=threads)
            os.close(fd2)
            assert st == got["n_aligned"]
            un = out2.read_bytes()
            rb.close()
    finally:
        os.close(fd)
    txt = out.read_bytes()
    assert w == len(txt)
    assert head + txt == exp_main, R.first_diff(head + txt, exp_main)
    assert un == exp_un, R.first_diff(un, exp_un)
    ra.close()


def _stream_corpus(n_rec=60_000, seed=9):
    """a FASTQ text of ~15 MB (several stream windows at small batch sizes): regular records with irregular ones sprinkled in
    -- CRLF, blank lines, leading blanks, a long wrapped-looking record -- so that both readers work across window borders"""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n_rec):
        L = int(rng.integers(30, 145))
        seq = bytes(rng.choice(np.frombuffer(b"ACGTN", dtype=np.uint8), size=L))
        qual = bytes(rng.integers(33, 74, size=L).astype(np.uint8)).replace(b"@", b"A")
        k = int(rng.integers(0, 400))
        if k == 0:
            out.append(b"@r%d extra words\r\n%s\r\n+\r\n%s\r\n" % (i, seq, qual))
        elif k == 1:
            out.append(b"\n\n@r%d\n%s\n+\n%s\n" % (i, seq, qual))
        elif k == 2:
            out.append(b"  @r%d\n %s\n+\n%s  \n" % (i, seq, qual))
        else:
            out.append(b"@r%d/1\n%s\n+\n%s\n" % (i, seq, qual))
    return b"".join(out)


@pytest.mark.parametrize("want", [1000, 16384])
def test_streamed_gzip_reads_equal_the_mapped_file(tmp_path, want):
    """gzip'ed read files are inflated a window at a time (bounded memory): same records, batch by batch, as the memory-mapped
    plain file -- over many windows, with irregular records and -B style skips in between"""
    import gzip
    data = _stream_corpus()
    plain, gz = tmp_path / "r.fq", tmp_path / "r.fq.gz"
    plain.write_bytes(data)
    with gzip.open(gz, "wb", compresslevel=1) as f:
        f.write(data)
    a, b = load_all(str(plain), want=want, stride=160), load_all(str(gz), want=want, stride=160)
    assert a[0] == b[0] == "fastq" and len(a[1]) == 60_000
    assert a == b
    assert load_all(str(gz), want=want, stride=160, token=True) == a          # the token reader alone, window after window
    for skip in (1, 12_345):
        ra, rb = B.Reads(str(plain)), B.Reads(str(gz))
        ra.skip(skip); rb.skip(skip)
        na, _, _ = ra.next(500); nb, _, _ = rb.next(500)
        assert na == nb == 500 and [ra.get(i) for i in range(500)] == [rb.get(i) for i in range(500)]
        ra.close(); rb.close()


def test_reads_from_a_pipe_are_streamed(tmp_path):
    """a FIFO (e.g. `zcat x.gz |` or a process substitution): read through the same windows, plain or gzip'ed"""
    import gzip
    import threading
    data = _stream_corpus(20_000, seed=4)
    plain = tmp_path / "r.fq"
    plain.write_bytes(data)
    exp = load_all(str(plain), want=4096, stride=160)
    for payload in (data, gzip.compress(data, 1)):
        fifo = str(tmp_path / "fifo")
        if os.path.exists(fifo):
            os.unlink(fifo)
        os.mkfifo(fifo)

        def feed():
            with open(fifo, "wb") as f:
                f.write(payload)
        t = threading.Thread(target=feed)
        t.start()
        got = load_all(fifo, want=4096, stride=160)
        t.join()
        assert got == exp


def test_truncated_gzip_input_is_reported(tmp_path):
    """a gzip read file cut short (or damaged) still serves the reads before the damage, and says so: the command line then
    exits non-zero instead of writing a silently shorter output"""
    import gzip
    data = _stream_corpus(30_000, seed=5)
    blob = gzip.compress(data, 1)
    good, cut = tmp_path / "ok.fq.gz", tmp_path / "cut.fq.gz"
    good.write_bytes(blob)
    cut.write_bytes(blob[:len(blob) * 2 // 3])
    for path, want_fail in ((good, False), (cut, True)):
        r = B.Reads(str(path))
        n_tot = 0
        while True:
            n, _, _ = r.next(8192, stride=160)
            n_tot += n
            if n < 8192:
                break
        assert r.failed == want_fail, (path, n_tot)
        assert (n_tot == 30_000) == (not want_fail) and n_tot > 10_000
        r.close()


def test_chunked_emit_equals_the_two_call_formatter_on_awkward_records(tmp_path):
    """the chunked emitter grows its buffers ahead of a raw cursor (one bound per record); the C ABI's two-call formatter counts
    into a caller-sized buffer: same bytes for read names of 30 KB, unmapped / filtered / repeat records, SAM and BSP, and
    for a second, smaller batch through the same (reused) buffers"""
    import ctypes as C
    from bsmap_b200.lib import load, strs
    rng = np.random.default_rng(12)
    gnames, gseqs = ["chrA_with_a_long_name_" + "x" * 200, "c2"], [bytes(rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=n)) for n in (50_000, 9_000)]
    for out_sam in (1, 0):
        p = B.make_params(v=5, r=1, R=1)
        p.out_sam = out_sam
        ix = B.Index.text_only(p, gnames, gseqs)
        for n in (3000, 17):
            names = [("read%d_" % i + "n" * int(rng.choice([0, 3, 200, 30_000], p=[0.5, 0.3, 0.19, 0.01]))) for i in range(n)]
            L = rng.integers(20, 145, n)
            seqs = ["".join("ACGTN"[c] for c in rng.integers(0, 5, int(l))) for l in L]
            quals = ["I" * int(l) for l in L]
            fq = tmp_path / ("r%d_%d.fq" % (out_sam, n))
            fq.write_text("".join("@%s\n%s\n+\n%s\n" % t for t in zip(names, seqs, quals)))
            recs = np.zeros(n, dtype=BL.REC)
            recs["chr"] = rng.integers(0, 4, n); recs["loc"] = rng.integers(2, 8_000, n); recs["nhits"] = rng.choice([0, 1, 1, 1, 5], n)
            recs["nm"] = rng.integers(0, 6, n); recs["chain"] = rng.integers(0, 2, n); recs["status"] = rng.random(n) < 0.05; recs["len"] = L
            counts = rng.integers(0, 70000, (n, 16)).astype(np.uint16)
            r = B.Reads(str(fq))
            assert r.next(n + 1)[0] == n
            out = tmp_path / "emit.txt"
            fd = os.open(out, os.O_WRONLY | os.O_CREAT | os.O_TRUNC)
            w, na = B.emit_se(ix, p, r, n, recs, counts, fd, threads=3)
            os.close(fd)
            args = (ix.h, C.byref(p), n, strs([s.encode() for s in names]), strs([s.encode() for s in seqs]), strs([s.encode() for s in quals]), 0,
                    recs.ctypes.data, counts.ctypes.data)
            na2 = C.c_uint32(0)
            need = load().bsx_format_se(*args, None, 0, C.byref(na2))
            buf = C.create_string_buffer(need + 1)
            load().bsx_format_se(*args, buf, need + 1, C.byref(na2))
            assert out.read_bytes() == buf.raw[:need] and w == need and na == na2.value
            r.close()
        ix.close()


@pytest.mark.parametrize("seed", [1, 2])
def test_random_read_files_line_cutter_equals_token_reader(tmp_path, seed):
    """random FASTA / FASTQ texts -- regular records mixed with CRLF, blank lines, leading blanks, trailing tabs, a missing
    final line feed, a truncated tail -- cut with random batch sizes and thread counts: the line cutter (which addresses the
    scanners' line starts in place) and the token reader that restates the reference's stream semantics give the same reads"""
    import random
    rnd = random.Random(seed)

    def rec(i, fastq):
        L = rnd.choice([1, 5, 30, 60, 100, 144, 150])
        seq = "".join(rnd.choice("ACGTN") for _ in range(L)); q = "".join(chr(rnd.randint(35, 73)) for _ in range(L))
        k, h, nl = rnd.random(), "@" if fastq else ">", rnd.choice(["\n", "\n", "\n", "\r\n"])
        if k < 0.85: return f"{h}r{i}{nl}{seq}{nl}" + (f"+{nl}{q}{nl}" if fastq else "")
        if k < 0.90: return f"{nl}{h}r{i} extra{nl}{seq}{nl}" + (f"+r{i}{nl}{q}{nl}" if fastq else "")
        if k < 0.94: return f" {h}r{i}{nl} {seq} {nl}" + (f"+{nl}{q}{nl}" if fastq else "")
        if k < 0.97: return f"{h}r{i}{nl}{seq}{nl}{nl}" + (f"+{nl}{q}{nl}{nl}" if fastq else "")
        return f"{h}r{i}\t{nl}{seq}\t{nl}" + (f"+{nl}{q}{nl}" if fastq else "")

    path = str(tmp_path / "fz.txt")
    checked = 0
    for case in range(120):
        fastq = rnd.random() < 0.7
        n = rnd.choice([0, 1, 2, 3, 7, 50, 400, 3000])
        txt = "".join(rec(i, fastq) for i in range(n))
        if n and rnd.random() < 0.4: txt = txt.rstrip("\r\n")
        if n and rnd.random() < 0.1: txt = txt[:len(txt) - rnd.randint(1, min(40, len(txt) - 1))]
        if not txt.strip():
            continue
        open(path, "w", newline="").write(txt)
        want, threads = rnd.choice([1, 2, 3, 7, 64, 1000, 5000]), rnd.choice([1, 2, 3, 8])
        try:
            a = load_all(path, want=want, threads=threads, stride=160)
            b = load_all(path, want=want, threads=threads, stride=160, token=True)
        except B.BsxError:
            continue
        assert a == b, (case, n, want, threads)
        checked += 1
    assert checked > 80
