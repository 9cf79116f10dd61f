"""4-CpG epialleles: the numpy restatement (oracle/epiallele_oracle.py) tied to pdr_oracle and to the reference script's own
tables, a second, character-by-character implementation, and hand-computed known answers on a small genome."""
from __future__ import annotations

import gzip
import math
import os
import sys

import numpy as np
import pytest

import cases as CS
from test_methratio_cpu import GOLD, MANIFEST
from test_mbias_cpu import mbias_kwargs, oracle_files, row_context, sam_line

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import conversion_oracle as CV  # noqa: E402
import epiallele_oracle as EP  # noqa: E402
import mbias_oracle as MB  # noqa: E402
import methratio_oracle as MO  # noqa: E402
import pdr_oracle as PD  # noqa: E402


def golden_lines(key):
    """{(chrom, 0-based pos): (total_C, methy_C)} of the golden table"""
    out = {}
    for line in gzip.open(os.path.join(GOLD, key + ".txt.gz"), "rt").read().splitlines()[1:]:
        col = line.split("\t")
        out[(col[0], int(col[1]) - 1)] = (int(col[5]), int(col[6]))
    return out


def naive(names, seqs, files, threshold=0, chroms=None, unique=False, pair=False, trim_fillin=2, rm_dup=False, ignore=(0, 0, 0, 0)):
    """the window rule read straight off each read's text, one character at a time: -> ({chrom: {(row, pattern): n}},
    spanning, windows)"""
    ref = {n: (s.decode() if isinstance(s, bytes) else s).upper() for n, s in zip(names, seqs) if not chroms or n in chroms}
    rank = {c: {q: j for j, q in enumerate(q for q in range(len(s) - 1) if s[q] == "C" and s[q + 1] == "G")} for c, s in ref.items()}
    out = {c: {} for c in ref}
    spanning = windows = 0
    seen = set()
    for path in files:
        alns = MO.parse_alignments(path, set(ref), unique, pair)
        r2 = MB._read2_flags(path, set(ref), unique, pair) or [False] * len(alns)
        for (seq, strand, cr, pos, insert, mate_pos, sam), read2 in zip(alns, r2):
            if rm_dup:
                key = (cr, pos + len(seq), 2) if strand in ("+-", "-+") else (cr, pos, 1)
                if key in seen:
                    continue
                seen.add(key)
            tseq, tpos = MO.trim(seq, strand, pos, insert, mate_pos, sam, trim_fillin)
            s = ref[cr]
            if tpos + len(tseq) > len(s):
                continue
            minus = strand[0] == "-"
            lo, hi = (ignore[2], len(seq) - ignore[3]) if read2 else (ignore[0], len(seq) - ignore[1])
            score, sites = 0, []                  # sites: (rank, called, methylated) in read order
            for i, ch in enumerate(tseq):
                q = tpos + i
                j = (tpos - pos) + i
                cyc = len(seq) - 1 - j if strand[0] != strand[1] else j
                inb = lo <= cyc < hi
                if minus:
                    is_site = s[q] == "G" and q >= 1 and s[q - 1] == "C"
                    call_m, call_u, base = "G", "A", "G"
                else:
                    is_site = s[q] == "C" and q + 1 < len(s) and s[q + 1] == "G"
                    call_m, call_u, base = "C", "T", "C"
                if s[q] == base and ch == call_m and inb and not is_site:
                    score += 1
                if is_site:
                    called = inb and ch in (call_m, call_u)
                    sites.append((rank[cr][q - 1 if minus else q], called, called and ch == call_m))
            if threshold and score >= threshold:
                continue
            n_w = 0
            for k in range(len(sites) - 3):
                w = sites[k:k + 4]
                if all(c for _, c, _ in w):
                    pat = 0
                    for _, _, m in w:
                        pat = pat * 2 + int(m)
                    out[cr][(w[0][0], pat)] = out[cr].get((w[0][0], pat), 0) + 1
                    n_w += 1
            spanning += n_w > 0
            windows += n_w
    return out, spanning, windows


def sparse(epi):
    return {c: {(int(j), int(i)): int(e[j, i]) for j, i in zip(*np.nonzero(e))} for c, e in epi.items()}


@pytest.mark.parametrize("key", sorted(MANIFEST))
def test_goldens_bound_and_naive(tmp_path, key):
    """every golden run: with epialleles on, the rest is pdr_oracle's; each window's reads are at most the pooled depth
    of each of its sites, and its methylated-at-k reads at most the pooled methylated count; the naive implementation
    agrees"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    files = oracle_files(ent, case, str(tmp_path))
    kw = mbias_kwargs(ent["opts"])
    res = EP.epialleles(d["gnames"], d["gseqs"], files, **kw)
    pd = PD.pdr(d["gnames"], d["gseqs"], files, **kw)
    for k in ("valid", "dropped", "scores", "mbias_overflow", "informative", "discordant_alignments", "patterns"):
        assert res[k] == pd[k], k
    assert np.array_equal(res["mbias"], pd["mbias"]) and np.array_equal(res["bins"], pd["bins"])
    for c in pd["counters"]:
        for a, b in zip(res["counters"][c], pd["counters"][c]):
            assert np.array_equal(a, b), c
        assert np.array_equal(res["concordant"][c], pd["concordant"][c]) and np.array_equal(res["discordant"][c], pd["discordant"][c])
    assert res["windows"] > 0 and res["windows"] == sum(int(e.sum()) for e in res["epi"].values())

    gold = golden_lines(key)
    opts = ent["opts"]
    combine, m1 = "-g" in opts, "-m" not in opts
    # a position without a line: with -z its depth is 0; without -z (at -m 1) its methylated count is 0
    depth_of = lambda cr, q: gold[(cr, q)][0] if (cr, q) in gold else (0 if "-z" in opts and m1 else None)
    meth_of = lambda cr, q: gold[(cr, q)][1] if (cr, q) in gold else (0 if m1 else None)
    checked = 0
    for cr, e in res["epi"].items():
        st = res["sites"][cr]
        for j in np.nonzero(e.sum(axis=1))[0]:
            n = int(e[j].sum())
            for k in range(EP.CPGS):
                c = int(st[j + k])
                at = [c] if combine else [c, c + 1]
                depth, meth = [depth_of(cr, q) for q in at], [meth_of(cr, q) for q in at]
                m_k = int(sum(e[j, i] for i in range(16) if i >> (EP.CPGS - 1 - k) & 1))
                if None not in depth:
                    assert n <= sum(depth), (cr, c, k)
                    checked += 1
                if None not in meth:
                    assert m_k <= sum(meth), (cr, c, k)
                    checked += 1
    assert checked > 0 or not m1                              # -m 3: every window met a site below the depth

    got, spanning, windows = naive(d["gnames"], d["gseqs"], files, **{k: v for k, v in kw.items() if k != "combine_cpg"})
    assert sparse(res["epi"]) == got
    assert (res["spanning"], res["windows"]) == (spanning, windows)


@pytest.mark.parametrize("key", sorted(MANIFEST)[::5])
@pytest.mark.parametrize("extra", [{"threshold": 2}, {"threshold": 1, "ignore": (3, 2, 4, 1)}])
def test_filters_against_naive(tmp_path, key, extra):
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    files = oracle_files(ent, case, str(tmp_path))
    kw = dict(mbias_kwargs(ent["opts"]), **extra)
    res = EP.epialleles(d["gnames"], d["gseqs"], files, **kw)
    cv = CV.conversion(d["gnames"], d["gseqs"], files, **kw)
    assert res["dropped"] == cv["dropped"] and res["valid"] == cv["valid"]
    got, spanning, windows = naive(d["gnames"], d["gseqs"], files, **{k: v for k, v in kw.items() if k != "combine_cpg"})
    assert sparse(res["epi"]) == got and (res["spanning"], res["windows"]) == (spanning, windows)


# ---- known answers -------------------------------------------------------------------------------------------------
#   chrP: 0 A  1 C  2 G  3 T  4 A  5 C  6 G  7 T  8 A  9 C  10 G  11 T  12 A  13 C  14 G  15 T  16 A  17 C  18 G  19 T
#         20 T  21 T  22 C  23 A  24 G  25 C  26 T  27 T  28 G  29 G  30 C  31 C
#   sites (their C): 1 5 9 13 17 -> rows 0 (1 5 9 13) and 1 (5 9 13 17); chrQ: "CG" * 300 + "AA", sites 0 2 .. 598
NAMES, SEQS = ["chrP", "chrQ"], [b"ACGTACGTACGTACGTACGTTTCAGCTTGGCC", b"CG" * 300 + b"AA"]
R16, R20 = "ACGTACGTACGTACGT", "ACGTACGTACGTACGTACGT"
PE = 0x1 | 0x2 | 0x40


def sub(s, i, c):
    return s[:i] + c + s[i + 1:]


def run(tmp_path, lines, **kw):
    p = tmp_path / "kat.sam"
    p.write_text("@HD\tVN:1.0\n" + "".join(lines))
    return EP.epialleles(NAMES, SEQS, [str(p)], **kw)


# name -> (lines, kwargs, {(chrom, row, pattern): count}, spanning alignments)
KATS = {
    "four_cpgs": ([sam_line(0, "chrP", 1, R16, "++")], {}, {("chrP", 0, 15): 1}, 1),
    "five_cpgs": ([sam_line(0, "chrP", 1, R20, "++")], {}, {("chrP", 0, 15): 1, ("chrP", 1, 15): 1}, 1),
    "three_cpgs": ([sam_line(0, "chrP", 1, R16[:12], "++")], {}, {}, 0),
    "pattern_bits": ([sam_line(0, "chrP", 1, sub(sub(R20, 5, "T"), 17, "T"), "++")], {}, {("chrP", 0, 11): 1, ("chrP", 1, 6): 1}, 1),
    "minus": ([sam_line(16, "chrP", 1, sub(R16, 10, "A"), "-+")], {}, {("chrP", 0, 13): 1}, 1),
    "plus_and_minus_one_row": ([sam_line(0, "chrP", 1, R16, "++"), sam_line(16, "chrP", 1, sub(R16, 10, "A"), "-+")], {},
                               {("chrP", 0, 15): 1, ("chrP", 0, 13): 1}, 2),
    "combine_changes_nothing": ([sam_line(0, "chrP", 1, R16, "++"), sam_line(16, "chrP", 1, sub(R16, 10, "A"), "-+")], {"combine_cpg": True},
                                {("chrP", 0, 15): 1, ("chrP", 0, 13): 1}, 2),
    "read_n": ([sam_line(0, "chrP", 1, sub(R20, 1, "N"), "++")], {}, {("chrP", 1, 15): 1}, 1),
    "mismatch": ([sam_line(0, "chrP", 1, sub(R20, 1, "A"), "++")], {}, {("chrP", 1, 15): 1}, 1),
    "n_in_the_middle": ([sam_line(0, "chrP", 1, sub(R20, 9, "N"), "++")], {}, {}, 0),
    "excluded_cycle": ([sam_line(0, "chrP", 1, R20, "++")], {"ignore": (2, 0, 0, 0)}, {("chrP", 1, 15): 1}, 1),
    "excluded_cycle_read2": ([sam_line(0x81, "chrP", 1, R20, "++")], {"ignore": (2, 0, 0, 0)}, {("chrP", 0, 15): 1, ("chrP", 1, 15): 1}, 1),
    # -t: '+-' loses its last 2 printed bases, C 17 with them
    "fillin": ([sam_line(16, "chrP", 1, R20[:18], "+-")], {}, {("chrP", 0, 15): 1}, 1),
    "fillin_off": ([sam_line(16, "chrP", 1, R20[:18], "+-")], {"trim_fillin": 0}, {("chrP", 0, 15): 1, ("chrP", 1, 15): 1}, 1),
    # mate overlap: mate at 0-based 17 -> seq[:17], C 17 gone
    "overlap": ([sam_line(PE, "chrP", 1, R20, "++", tlen=20, pnext=18, rnext="=")], {"trim_fillin": 0}, {("chrP", 0, 15): 1}, 1),
    # span edges: '+' ends on C 13 (its G outside), '-' starts on G 2 (its C outside)
    "plus_edge": ([sam_line(0, "chrP", 1, R16[:14], "++")], {}, {("chrP", 0, 15): 1}, 1),
    "minus_edge": ([sam_line(16, "chrP", 3, R20[2:19], "-+")], {}, {("chrP", 0, 15): 1, ("chrP", 1, 15): 1}, 1),
    # sequence ends: chrQ's first and last windows, '+' and '-'
    "seq_start": ([sam_line(0, "chrQ", 1, "CG" * 4, "++"), sam_line(16, "chrQ", 1, "CA" * 4, "-+")], {}, {("chrQ", 0, 15): 1, ("chrQ", 0, 0): 1}, 2),
    "seq_end": ([sam_line(0, "chrQ", 593, "CGCGCGCGAA", "++")], {}, {("chrQ", 296, 15): 1}, 1),
    # conversion filter: methylated CHG 22 and CHH 25 score 2
    "conversion_dropped": ([sam_line(0, "chrP", 1, "ACGTACGTACGTACGTACGTTTCAGC", "++")], {"threshold": 2}, {}, 0),
    "conversion_kept": ([sam_line(0, "chrP", 1, "ACGTACGTACGTACGTACGTTTCAGC", "++")], {"threshold": 3},
                        {("chrP", 0, 15): 1, ("chrP", 1, 15): 1}, 1),
    # -r: the duplicate loses and is not scored
    "rm_dup": ([sam_line(0, "chrP", 1, R16, "++"), sam_line(0, "chrP", 1, sub(R16, 13, "T"), "++")], {"rm_dup": True}, {("chrP", 0, 15): 1}, 1),
    "no_rm_dup": ([sam_line(0, "chrP", 1, R16, "++"), sam_line(0, "chrP", 1, sub(R16, 13, "T"), "++")], {},
                  {("chrP", 0, 15): 1, ("chrP", 0, 14): 1}, 2),
}


@pytest.mark.parametrize("name", sorted(KATS))
def test_known_answers(tmp_path, name):
    lines, kw, exp, spanning = KATS[name]
    res = run(tmp_path, lines, **kw)
    got = {(c, j, i): n for c, d in sparse(res["epi"]).items() for (j, i), n in d.items()}
    assert got == exp
    assert res["spanning"] == spanning and res["windows"] == sum(exp.values())
    assert [list(res["sites"]["chrP"]), len(res["sites"]["chrQ"])] == [[1, 5, 9, 13, 17], 300]
    nv = naive(NAMES, SEQS, [str(tmp_path / "kat.sam")], **{k: v for k, v in kw.items() if k != "combine_cpg"})
    assert {(c, j, i): n for c, d in nv[0].items() for (j, i), n in d.items()} == exp


def patterned(pat):
    """R16 with the four sites methylated by the bits of pat (the first site the high bit)"""
    s = R16
    for k, q in enumerate((1, 5, 9, 13)):
        if not (pat >> (3 - k)) & 1:
            s = sub(s, q, "T")
    return sam_line(0, "chrP", 1, s, "++")


def test_line_text(tmp_path):
    one = EP.epiallele_text(run(tmp_path, [patterned(15)]))
    assert one == EP.HEADER + "chrP\t2\t15\t1\t1.0000\t0.0000\t0.0000\t" + ",".join(["0"] * 15 + ["1"]) + "\n"
    two = EP.epiallele_text(run(tmp_path, [patterned(15), patterned(0)]))
    assert two.splitlines()[1] == "chrP\t2\t15\t2\t0.5000\t0.2500\t0.5000\t1," + "0," * 14 + "1"
    every = EP.epiallele_text(run(tmp_path, [patterned(i) for i in range(16)]))
    assert every.splitlines()[1] == "chrP\t2\t15\t16\t0.5000\t1.0000\t0.9375\t" + ",".join(["1"] * 16)
    assert EP.window_stats([3, 1] + [0] * 14)[2] == pytest.approx(-(0.75 * math.log2(0.75) + 0.25 * math.log2(0.25)) / 4)
    five = EP.epiallele_text(run(tmp_path, [sam_line(0, "chrP", 1, R20, "++")]))
    assert [ln.split("\t")[:3] for ln in five.splitlines()[1:]] == [["chrP", "2", "15"], ["chrP", "6", "19"]]


def test_snp_modes_and_min_depth(tmp_path):
    """a '-' read with T over C 1 is SNP evidence at a base of row 0: skip and correct drop the window (correct too,
    although another read confirms the C), no-action keeps it; -m drops a window with fewer reads"""
    lines = [sam_line(0, "chrP", 1, R16, "++"), sam_line(16, "chrP", 1, sub(R16, 1, "T"), "-+"), sam_line(16, "chrP", 1, R16, "-+")]
    res = run(tmp_path, lines)
    assert res["counters"]["chrP"][3][1] == 1 and res["counters"]["chrP"][2][1] == 1
    full = EP.epiallele_text(res)
    assert full.splitlines()[1].split("\t")[:4] == ["chrP", "2", "15", "3"]
    assert EP.epiallele_text(res, ct_snp="no-action") == full
    assert EP.epiallele_text(res, ct_snp="skip") == EP.HEADER
    assert EP.epiallele_text(res, ct_snp="correct") == EP.HEADER
    assert EP.epiallele_text(res, min_depth=3) == full and EP.epiallele_text(res, min_depth=4) == EP.HEADER
    g = run(tmp_path, lines, combine_cpg=True)                # the fold moves the evidence, the window still drops
    assert EP.epiallele_text(g, ct_snp="skip") == EP.HEADER and EP.epiallele_text(g) == full
    assert EP.stderr_line(res) == "epialleles: 3 of 3 valid mappings span a 4-CpG window, 3 window patterns counted"
