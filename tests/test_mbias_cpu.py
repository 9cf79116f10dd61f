"""M-bias and per-cycle exclusion: the numpy restatement (oracle/mbias_oracle.py) tied to the reference script's own
tables (tests/golden/methratio/), and hand-computed known answers on a small genome."""
from __future__ import annotations

import gzip
import os
import sys

import numpy as np
import pytest

import cases as CS
from test_methratio_cpu import GOLD, MANIFEST, alignment_files, opts_kwargs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import mbias_oracle as MB  # noqa: E402

CTX = {"CpG": 0, "CHG": 1, "CHH": 2}


def oracle_files(ent, case, td):
    files = alignment_files(case, td, bam=ent.get("bam", False))
    if ent.get("bam"):                                      # the oracle reads text: the BAM's records, in the BAM's order
        import bamio
        sam = os.path.join(td, "from_bam.sam")
        open(sam, "w").write(bamio.bam_to_sam_text(files[0]))
        files = [sam]
    return files


def mbias_kwargs(opts):
    kw = opts_kwargs(opts)
    kw.pop("meth0", None)
    kw.pop("min_depth", None)
    return kw


def row_context(ref: bytes, pos0: int, strand: str) -> int:
    """the context of a table row, from the reference (the 5-mer column is cut short at sequence starts)"""
    up = ref.upper()
    want, step = (ord("G"), 1) if strand == "+" else (ord("C"), -1)
    def at(k):
        return 0 <= k < len(up) and up[k] == want
    return 0 if at(pos0 + step) else (1 if at(pos0 + 2 * step) else 2)


@pytest.mark.parametrize("key", sorted(k for k in MANIFEST if "-m" not in MANIFEST[k]["opts"] or
                                       MANIFEST[k]["opts"][MANIFEST[k]["opts"].index("-m") + 1] == "1"))
def test_oracle_marginals_equal_the_reference_table(tmp_path, key):
    """summed over reads and cycles, the M-bias is the table: methylated per context == sum of methy_C, and with -z
    (every covered position printed) methylated + unmethylated == sum of total_C"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    files = oracle_files(ent, case, str(tmp_path))
    hist, overflow, _, _ = MB.mbias(d["gnames"], d["gseqs"], files, **mbias_kwargs(ent["opts"]))
    assert overflow == 0
    ref = dict(zip(d["gnames"], d["gseqs"]))
    meth_c, total_c = np.zeros(3, dtype=np.int64), np.zeros(3, dtype=np.int64)
    rows = gzip.open(os.path.join(GOLD, key + ".txt.gz"), "rt").read().splitlines()[1:]
    for line in rows:
        col = line.split("\t")
        c = row_context(ref[col[0]], int(col[1]) - 1, col[2])
        total_c[c] += int(col[5])
        meth_c[c] += int(col[6])
    assert rows
    assert np.array_equal(hist[..., 0].sum(axis=(0, 2)), meth_c)
    if "-z" in ent["opts"]:
        assert np.array_equal(hist.sum(axis=(0, 2, 3)), total_c)


# ---- known answers -------------------------------------------------------------------------------------------------
# chr1  0 G  1 C  2 A  3 C  4 G  5 T  6 T  7 C  8 A  9 G  10 C  11 T  12 C  13 N  14 A  15 C  16 C
#   '+' C: 1 CHH, 3 CpG, 7 CHG, 10 CHH, 12 CHH (next to N), 15 CHH (last but one), 16 CHH (last base)
#   '-' G: 0 CHH (position 0), 4 CpG, 9 CHG
# chr2  0 G  1 G  2 T  3 N  4 G  5 A  6 C  7 G   -- follows chr1's "CC": a C at chr1's end must not see chr2's G, nor the
#   G at chr2's start chr1's C
#   '+' C: 6 CpG      '-' G: 0 CHH, 1 CHH, 4 CHH (next to N), 7 CpG
NAMES, SEQS = ["chr1", "chr2"], [b"GCACGTTCAGCTCNACC", b"GGTNGACG"]


def sam_line(flag, chrom, pos1, seq, zs, tlen=0, pnext=0, rnext="*"):
    return "r\t%d\t%s\t%d\t255\t%dM\t%s\t%d\t%d\t%s\t%s\tNM:i:0\tZS:Z:%s\n" % (flag, chrom, pos1, len(seq), rnext, pnext, tlen, seq, "I" * len(seq), zs)


def sparse(hist):
    """{(read 1/2, context, 1-based cycle, 'm'/'u'): count}"""
    names = ("CpG", "CHG", "CHH")
    return {(int(r) + 1, names[c], int(y) + 1, "mu"[k]): int(hist[r, c, y, k]) for r, c, y, k in zip(*np.nonzero(hist))}


def run(tmp_path, lines, **kw):
    p = tmp_path / "kat.sam"
    p.write_text("@HD\tVN:1.0\n" + "".join(lines))
    return MB.mbias(NAMES, SEQS, [str(p)], **kw)


FWD = sam_line(0, "chr1", 1, "GCATGTTTAG", "++")       # C1 meth (CHH), C3 unmeth (CpG), C7 unmeth (CHG)
FWD_CALLS = {(1, "CHH", 2, "m"): 1, (1, "CpG", 4, "u"): 1, (1, "CHG", 8, "u"): 1}

KATS = {
    "forward": ([FWD], {}, FWD_CALLS),
    # '-+': G calls, SEQ printed reversed -> cycle = 9 - j
    "reversed": ([sam_line(16, "chr1", 1, "GCACATTCAG", "-+")], {}, {(1, "CHH", 10, "m"): 1, (1, "CpG", 6, "u"): 1, (1, "CHG", 1, "m"): 1}),
    "read2": ([sam_line(0x80 | 0x1, "chr1", 1, "GCATGTTTAG", "++")], {}, {(2,) + k[1:]: v for k, v in FWD_CALLS.items()}),
    # '--': seq[2:], pos + 2; not reversed, so the cycle keeps the printed offset
    "fillin_minus_minus": ([sam_line(16, "chr1", 1, "GCACATTCAG", "--")], {}, {(1, "CpG", 5, "u"): 1, (1, "CHG", 10, "m"): 1}),
    # '-+' with TLEN -10: trim 10 - (10 - 2) = 2 from the start; reversed
    "fillin_minus_plus": ([sam_line(16, "chr1", 1, "GCACATTCAG", "-+", tlen=-10)], {}, {(1, "CpG", 6, "u"): 1, (1, "CHG", 1, "m"): 1}),
    # '++' with TLEN 10, mate at 0-based 5: seq[:5] after -t 0
    "sam_overlap": ([sam_line(0x1 | 0x2 | 0x40, "chr1", 1, "GCATGTTTAG", "++", tlen=10, pnext=6, rnext="=")], {"trim_fillin": 0},
                    {(1, "CHH", 2, "m"): 1, (1, "CpG", 4, "u"): 1}),
    # read-through pair, printed at the insert (8): mate a '++' loses all to the overlap with b at the same POS; mate b
    # '+-' (reversed) loses its last 2 printed bases to fill-in trimming
    "readthrough": ([sam_line(0x1 | 0x2 | 0x40, "chr1", 1, "GCATGTTC", "++", tlen=8, pnext=1, rnext="="),
                     sam_line(0x1 | 0x2 | 0x80 | 0x10, "chr1", 1, "GCATGTTC", "+-", tlen=-8, pnext=1, rnext="=")], {},
                    {(2, "CHH", 7, "m"): 1, (2, "CpG", 5, "u"): 1}),
    "chr1_end": ([sam_line(0, "chr1", 11, "CTCNACC", "++")], {},
                 {(1, "CHH", 1, "m"): 1, (1, "CHH", 3, "m"): 1, (1, "CHH", 6, "m"): 1, (1, "CHH", 7, "m"): 1}),
    "chr2_start": ([sam_line(16, "chr2", 1, "GATNGA", "-+")], {}, {(1, "CHH", 6, "m"): 1, (1, "CHH", 5, "u"): 1, (1, "CHH", 2, "m"): 1}),
    "chr2_cpg_both_strands": ([sam_line(0, "chr2", 5, "GATG", "++"), sam_line(16, "chr2", 5, "GACA", "--")], {"trim_fillin": 0},
                              {(1, "CpG", 3, "u"): 1, (1, "CHH", 1, "m"): 1, (1, "CpG", 4, "u"): 1}),
    # exclusion, each bound: FWD (read 1) and the same read as read 2, L = 10
    "ignore_r1_5p": ([FWD], {"ignore": (2, 0, 0, 0)}, {(1, "CpG", 4, "u"): 1, (1, "CHG", 8, "u"): 1}),
    "ignore_r1_3p": ([FWD], {"ignore": (0, 3, 2, 2)}, {(1, "CHH", 2, "m"): 1, (1, "CpG", 4, "u"): 1}),
    "ignore_r2_5p": ([sam_line(0x81, "chr1", 1, "GCATGTTTAG", "++")], {"ignore": (9, 9, 4, 0)}, {(2, "CHG", 8, "u"): 1}),
    "ignore_r2_3p": ([sam_line(0x81, "chr1", 1, "GCATGTTTAG", "++")], {"ignore": (9, 9, 0, 7)}, {(2, "CHH", 2, "m"): 1}),
}


@pytest.mark.parametrize("name", sorted(KATS))
def test_known_answers(tmp_path, name):
    lines, kw, exp = KATS[name]
    hist, overflow, counters, nmap = run(tmp_path, lines, **kw)
    assert sparse(hist) == exp and overflow == 0
    assert nmap == len(lines)
    # the table holds exactly the calls the M-bias holds
    assert sum(int(d.sum()) for _, d in counters.values()) == sum(exp.values())
    assert sum(int(m.sum()) for m, _ in counters.values()) == sum(v for k, v in exp.items() if k[3] == "m")


def test_exclusion_reaches_the_table(tmp_path):
    _, _, full, _ = run(tmp_path, [FWD])
    _, _, cut, _ = run(tmp_path, [FWD], ignore=(2, 3, 0, 0))
    assert full["chr1"][1][[1, 3, 7]].tolist() == [1, 1, 1]
    assert cut["chr1"][1][[1, 3, 7]].tolist() == [0, 1, 0] and cut["chr1"][0][1] == 0


def test_long_seq_overflows(tmp_path):
    g = "ACGT" * 150                                          # 600 nt
    p = tmp_path / "long.sam"
    p.write_text(sam_line(0, "c", 1, g, "++"))
    hist, overflow, counters, _ = MB.mbias(["c"], [g.encode()], [str(p)])
    assert overflow == 600 // 4 - 512 // 4 and int(hist.sum()) == 512 // 4
    assert int(counters["c"][1].sum()) == 150


def test_report_text():
    h = np.zeros((2, 3, MB.CYCLES, 2), dtype=np.int64)
    h[1, 0, 0] = (2, 1)
    h[0, 2, 511] = (0, 3)
    h[0, 0, 4] = (1, 0)
    assert MB.mbias_text(h) == ("context\tread\tcycle\tmethylated\tunmethylated\tratio\n"
                                "CpG\t1\t5\t1\t0\t1.000\nCpG\t2\t1\t2\t1\t0.667\nCHH\t1\t512\t0\t3\t0.000\n")
