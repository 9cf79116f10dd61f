"""Read-level CpG concordance (PDR): the numpy restatement (oracle/pdr_oracle.py) tied to conversion_oracle and to the
reference script's own tables, and hand-computed known answers on a small genome."""
from __future__ import annotations

import gzip
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
import pdr_oracle as PD  # noqa: E402


def golden_cpg_depths(key, ref):
    """{(chrom, 0-based pos): total_C} of the golden table's CpG lines"""
    out = {}
    for line in gzip.open(os.path.join(GOLD, key + ".txt.gz"), "rt").read().splitlines()[1:]:
        col = line.split("\t")
        q = int(col[1]) - 1
        if row_context(ref[col[0]], q, col[2]) == 0:
            out[(col[0], q)] = int(col[5])
    return out


@pytest.mark.parametrize("key", sorted(MANIFEST))
def test_k1_counts_every_cpg_call_of_the_goldens(tmp_path, key):
    """K = 1, no filter: concordant + discordant is the depth the reference script prints at every CpG line (-g included);
    with -z that is every position with CpG calls.  K = 4 counts at most that depth."""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    files = oracle_files(ent, case, str(tmp_path))
    kw = mbias_kwargs(ent["opts"])
    ref = dict(zip(d["gnames"], d["gseqs"]))
    gold = golden_cpg_depths(key, ref)
    assert gold
    r1 = PD.pdr(d["gnames"], d["gseqs"], files, min_cpg=1, **kw)
    r4 = PD.pdr(d["gnames"], d["gseqs"], files, min_cpg=4, **kw)
    for (cr, q), dp in gold.items():
        assert r1["concordant"][cr][q] + r1["discordant"][cr][q] == dp, (cr, q)
        assert r4["concordant"][cr][q] + r4["discordant"][cr][q] <= dp, (cr, q)
    min_depth = int(ent["opts"][ent["opts"].index("-m") + 1]) if "-m" in ent["opts"] else 1
    if "-z" in ent["opts"]:
        n_pos = sum(int(((r1["concordant"][cr] + r1["discordant"][cr]) >= min_depth).sum()) for cr in r1["ref"])
        assert n_pos == len(gold)
    assert r1["informative"] == sum(1 for f in r1["patterns"] for p in f if p is not None and sum(p) >= 1)
    assert r4["informative"] <= r1["informative"] and r4["discordant_alignments"] <= r1["discordant_alignments"]


@pytest.mark.parametrize("key", sorted(MANIFEST)[::4])
@pytest.mark.parametrize("extra", [{}, {"threshold": 3}, {"threshold": 2, "ignore": (3, 2, 4, 1)}])
def test_everything_else_is_conversion_oracles(tmp_path, key, extra):
    """with PDR on, the counters, C/T SNP evidence, M-bias, conversion bins, valid mappings and scores are
    conversion_oracle's"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    files = oracle_files(ent, case, str(tmp_path))
    kw = dict(mbias_kwargs(ent["opts"]), **extra)
    res = PD.pdr(d["gnames"], d["gseqs"], files, min_cpg=3, **kw)
    cv = CV.conversion(d["gnames"], d["gseqs"], files, **kw)
    for k in ("valid", "dropped", "scores", "mbias_overflow"):
        assert res[k] == cv[k], k
    assert np.array_equal(res["mbias"], cv["mbias"]) and np.array_equal(res["bins"], cv["bins"])
    for c in cv["counters"]:
        for a, b in zip(res["counters"][c], cv["counters"][c]):
            assert np.array_equal(a, b), c


# ---- known answers -------------------------------------------------------------------------------------------------
#   0 A  1 C  2 G  3 T  4 A  5 C  6 G  7 T  8 A  9 C  10 G  11 T  12 A  13 C  14 G  15 T  16 A  17 C  18 G  19 T
#   20 T  21 T  22 C  23 A  24 G  25 C  26 T  27 T  28 G  29 G  30 C  31 C
#   '+' CpG C: 1 5 9 13 17; C 22 CHG, 25 CHH, 30 CHH, 31 CHH        '-' CpG G: 2 6 10 14 18; G 24 CHG, 28 CHH, 29 CHH
NAMES, SEQS = ["chrP", "chrQ"], [b"ACGTACGTACGTACGTACGTTTCAGCTTGGCC", b"CG" * 300 + b"AA"]
R16 = "ACGTACGTACGTACGT"                     # chrP[0:16]: four '+' CpGs, four '-' CpGs, every C and G kept
PLUS4 = [1, 5, 9, 13]
MINUS4 = [2, 6, 10, 14]
PE = 0x1 | 0x2 | 0x40


def sub(s, i, c):
    return s[:i] + c + s[i + 1:]


def kat_file(tmp_path, lines, name="kat.sam"):
    p = tmp_path / name
    p.write_text("@HD\tVN:1.0\n" + "".join(lines))
    return str(p)


def run(tmp_path, lines, **kw):
    return PD.pdr(NAMES, SEQS, [kat_file(tmp_path, lines)], **kw)


# name -> (lines, kwargs, {position: (concordant, discordant)} on chrP, informative, discordant alignments)
KATS = {
    "four_methylated": ([sam_line(0, "chrP", 1, R16, "++")], {}, {q: (1, 0) for q in PLUS4}, 1, 0),
    "four_unmethylated": ([sam_line(0, "chrP", 1, "ATGTATGTATGTATGT", "++")], {}, {q: (1, 0) for q in PLUS4}, 1, 0),
    "three_plus_one": ([sam_line(0, "chrP", 1, sub(R16, 13, "T"), "++")], {}, {q: (0, 1) for q in PLUS4}, 1, 1),
    "three_cpgs_at_k4": ([sam_line(0, "chrP", 1, R16[:12], "++")], {}, {}, 0, 0),
    "three_cpgs_at_k3": ([sam_line(0, "chrP", 1, R16[:12], "++")], {"min_cpg": 3}, {q: (1, 0) for q in PLUS4[:3]}, 1, 0),
    "minus": ([sam_line(16, "chrP", 1, sub(R16, 10, "A"), "-+")], {}, {q: (0, 1) for q in MINUS4}, 1, 1),
    "combine_cpg": ([sam_line(0, "chrP", 1, R16, "++"), sam_line(16, "chrP", 1, sub(R16, 10, "A"), "-+")], {"combine_cpg": True},
                    {q: (1, 1) for q in PLUS4}, 2, 1),
    "read_n": ([sam_line(0, "chrP", 1, sub(R16, 13, "N"), "++")], {}, {}, 0, 0),
    "read_lower_case": ([sam_line(0, "chrP", 1, sub(R16, 13, "c"), "++")], {}, {}, 0, 0),
    "read_n_k3": ([sam_line(0, "chrP", 1, sub(R16, 13, "N"), "++")], {"min_cpg": 3}, {q: (1, 0) for q in PLUS4[:3]}, 1, 0),
    # -t: '+-' loses its last 2 printed bases, C 13 with them
    "fillin": ([sam_line(16, "chrP", 1, R16[:15], "+-")], {}, {}, 0, 0),
    "fillin_off": ([sam_line(16, "chrP", 1, R16[:15], "+-")], {"trim_fillin": 0}, {q: (1, 0) for q in PLUS4}, 1, 0),
    # mate overlap: mate at 0-based 13 -> seq[:13]
    "overlap": ([sam_line(PE, "chrP", 1, R16, "++", tlen=16, pnext=14, rnext="=")], {"trim_fillin": 0}, {}, 0, 0),
    "overlap_bsp_rules": ([sam_line(PE, "chrP", 1, R16, "++", tlen=16, pnext=14, rnext="=")], {"trim_fillin": 0, "sam_rules": False},
                          {q: (1, 0) for q in PLUS4}, 1, 0),
    # exclusion: read 1's last three cycles hold C 13; read 2 keeps it
    "ignore": ([sam_line(0, "chrP", 1, R16, "++")], {"ignore": (0, 3, 0, 0)}, {}, 0, 0),
    "ignore_read2": ([sam_line(0x81, "chrP", 1, R16, "++")], {"ignore": (0, 3, 0, 0)}, {q: (1, 0) for q in PLUS4}, 1, 0),
    # conversion filter: methylated CHG 22 and CHH 25 score 2
    "conversion_dropped": ([sam_line(0, "chrP", 1, "ACGTACGTACGTACGTACGTTTCAGC", "++")], {"threshold": 2}, {}, 0, 0),
    "conversion_kept": ([sam_line(0, "chrP", 1, "ACGTACGTACGTACGTACGTTTCAGC", "++")], {"threshold": 3},
                        {q: (1, 0) for q in PLUS4 + [17]}, 1, 0),
    # -r: the duplicate loses and is not scored
    "rm_dup": ([sam_line(0, "chrP", 1, R16, "++"), sam_line(0, "chrP", 1, sub(R16, 13, "T"), "++")], {"rm_dup": True},
               {q: (1, 0) for q in PLUS4}, 1, 0),
    "no_rm_dup": ([sam_line(0, "chrP", 1, R16, "++"), sam_line(0, "chrP", 1, sub(R16, 13, "T"), "++")], {},
                  {q: (1, 1) for q in PLUS4}, 2, 1),
    "k1": ([sam_line(0, "chrP", 1, "ACGT", "++")], {"min_cpg": 1}, {1: (1, 0)}, 1, 0),
    # chrQ: 255 CpG calls make an alignment informative at K = 255, 254 do not
    "k255": ([sam_line(0, "chrQ", 1, "CG" * 255, "++"), sam_line(0, "chrQ", 3, "CG" * 254, "++")], {"min_cpg": 255}, {}, 1, 0),
}


@pytest.mark.parametrize("name", sorted(KATS))
def test_known_answers(tmp_path, name):
    lines, kw, exp, informative, n_disc = KATS[name]
    res = run(tmp_path, lines, **kw)
    c, d = res["concordant"]["chrP"], res["discordant"]["chrP"]
    got = {int(q): (int(c[q]), int(d[q])) for q in np.nonzero(c + d)[0]}
    assert got == exp
    assert res["informative"] == informative and res["discordant_alignments"] == n_disc
    if name == "k255":
        q = res["concordant"]["chrQ"]
        assert int(q.sum()) == 255 and int(res["discordant"]["chrQ"].sum()) == 0


def snp_lines():
    """'+' CpGs 1 5 9 13 concordant; '-' reads over C 1: one T (SNP evidence), one C (confirming); their G calls concordant"""
    return [sam_line(0, "chrP", 1, R16, "++"), sam_line(16, "chrP", 1, sub(R16, 1, "T"), "-+"), sam_line(16, "chrP", 1, R16, "-+")]


def test_pdr_file_and_snp_modes(tmp_path):
    res = run(tmp_path, snp_lines())
    assert res["counters"]["chrP"][3][1] == 1 and res["counters"]["chrP"][2][1] == 1     # snp, confirm at C 1
    full = PD.HEADER + "".join("chrP\t%d\t%s\t%d\t0\t0.000\n" % (q + 1, "+" if q in PLUS4 else "-", 1 if q in PLUS4 else 2)
                               for q in sorted(PLUS4 + MINUS4))
    assert PD.pdr_text(res) == full
    assert PD.pdr_text(res, ct_snp="no-action") == full
    assert PD.pdr_text(res, ct_snp="correct") == full                                     # confirmed: eff > 0
    skip = PD.pdr_text(res, ct_snp="skip")
    assert skip == full.replace("chrP\t2\t+\t1\t0\t0.000\n", "")
    alone = run(tmp_path, snp_lines()[:2])                                                 # no confirming read: correct drops it too
    assert "chrP\t2\t" not in PD.pdr_text(alone, ct_snp="correct")
    assert PD.pdr_text(res, min_depth=2) == PD.HEADER + "".join("chrP\t%d\t-\t2\t0\t0.000\n" % (q + 1) for q in MINUS4)


def test_pdr_value_and_lines(tmp_path):
    res = run(tmp_path, [sam_line(0, "chrP", 1, R16, "++"), sam_line(0, "chrP", 1, sub(R16, 13, "T"), "++"),
                         sam_line(0, "chrP", 1, sub(sub(R16, 13, "T"), 9, "T"), "++")])
    assert PD.pdr_text(res) == PD.HEADER + "".join("chrP\t%d\t+\t1\t2\t0.667\n" % (q + 1) for q in PLUS4)
    assert PD.stderr_line(res, 4) == "PDR: 3 of 3 valid mappings informative (>= 4 CpG calls), 2 discordant"


def test_region_columns(tmp_path):
    res = run(tmp_path, [sam_line(0, "chrP", 1, R16, "++"), sam_line(0, "chrP", 1, sub(R16, 13, "T"), "++")])
    regs = [("chrP", 0, 8), ("chrP", 0, 32), ("chrP", 20, 32), ("chrQ", 0, 10)]
    txt = PD.region_text(res, regs).splitlines()
    assert txt[0] == PD.REGION_HEADER[:-1]
    assert txt[1] == "chrP\t0\t8\tCpG\t4\t2\t4\t4\t1.0000\t2\t2\t0.5000"
    assert txt[2].endswith("\t0\t0\tNA") and txt[3].endswith("\t0\t0\tNA") and txt[2].split("\t")[3] == "CHG"
    assert txt[4].split("\t")[9:] == ["4", "4", "0.5000"]
    assert txt[7].split("\t")[9:] == ["0", "0", "NA"] and txt[10].split("\t")[9:] == ["0", "0", "NA"]
    assert len(txt) == 1 + 3 * len(regs)
    # -m drops lines below it from the sums, as from the file
    assert PD.region_text(res, regs, min_depth=3).splitlines()[4].split("\t")[9:] == ["0", "0", "NA"]
    assert np.array_equal(PD.region_pdr(res, regs, min_depth=2), [[2, 2], [4, 4], [0, 0], [0, 0]])


def test_region_sums_are_the_file_lines(tmp_path):
    """the region sums are the sums of the PDR file's lines in the region, whatever -m and the SNP mode"""
    res = run(tmp_path, snp_lines())
    regs = [("chrP", s, e) for s in range(0, 20, 3) for e in (s, s + 4, s + 11)]
    for mode in (None, "skip", "correct"):
        for m in (1, 2):
            rows = [ln.split("\t") for ln in PD.pdr_text(res, min_depth=m, ct_snp=mode).splitlines()[1:]]
            exp = [[sum(int(r[k]) for r in rows if s < int(r[1]) <= e) for k in (3, 4)] for _, s, e in regs]
            assert np.array_equal(PD.region_pdr(res, regs, min_depth=m, ct_snp=mode), exp), (mode, m)
