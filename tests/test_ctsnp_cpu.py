"""C/T SNP evidence and the SNP-corrected table: the numpy restatement (oracle/ctsnp_oracle.py) tied to the reference
script's own tables in no-action mode (tests/golden/methratio/), and hand-computed known answers on a small genome."""
from __future__ import annotations

import gzip
import os
import sys

import numpy as np
import pytest

import cases as CS
from test_methratio_cpu import GOLD, MANIFEST, opts_kwargs
from test_mbias_cpu import NAMES, SEQS, oracle_files, sam_line

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ctsnp_oracle as CT  # noqa: E402
import mbias_oracle as MB  # noqa: E402


def split_kwargs(opts):
    """methratio options -> (counters() kwargs, table() kwargs)"""
    kw = opts_kwargs(opts)
    tk = {k: kw.pop(k) for k in ("meth0", "min_depth") if k in kw}
    return kw, tk


@pytest.mark.parametrize("key", sorted(MANIFEST))
def test_no_action_projects_to_the_reference_table(tmp_path, key):
    """no-action: the 12-column table, projected onto the plain 9 columns, is the reference script's table, and the
    summary line's numbers are the script's"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    files = oracle_files(ent, case, str(tmp_path))
    kw, tk = split_kwargs(ent["opts"])
    txt, (nmap, nc, nd), _ = CT.methratio_ct_snp(d["gnames"], d["gseqs"], files, "no-action", **kw, **tk)
    gold = gzip.open(os.path.join(GOLD, key + ".txt.gz"), "rt").read()
    assert CT.project_plain(txt) == gold
    assert ent["stdout"] == "total %d valid mappings, %d covered cytosines, average coverage: %.2f fold." % (nmap, nc, nd / nc if nc else 0.0)


@pytest.mark.parametrize("key", ["pe_sam.r", "se_cfg1.g_z", "se_cfg2_bsp.u_t_0", "rrbs_pe.t_0"])
def test_calls_equal_the_mbias_oracle(tmp_path, key):
    """the calls are mbias_oracle's counters (exclusion on), and the golden files carry opposite-strand evidence"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    files = oracle_files(ent, case, str(tmp_path))
    kw, _ = split_kwargs(ent["opts"])
    cnt, nmap, _ = CT.counters(d["gnames"], d["gseqs"], files, ignore=(1, 2, 3, 4), **kw)
    _, _, mb, mb_nmap = MB.mbias(d["gnames"], d["gseqs"], files, ignore=(1, 2, 3, 4), **kw)
    assert nmap == mb_nmap
    for c, (m, dp, conf, snp) in cnt.items():
        assert np.array_equal(m, mb[c][0]) and np.array_equal(dp, mb[c][1])
    assert sum(int(v[2].sum()) for v in cnt.values()) > 0


# ---- known answers -------------------------------------------------------------------------------------------------
# chr1  0 G  1 C  2 A  3 C  4 G  5 T  6 T  7 C  8 A  9 G  10 C  11 T  12 C  13 N  14 A  15 C  16 C   (chr2: GGTNGACG)
# A '+' hit over chr1[0:10] has evidence at the Gs 0, 4, 9; a '-' hit over it at the Cs 1, 3, 7.
REF10 = "GCACGTTCAG"


def kat_file(tmp_path, lines, bsp=False):
    p = tmp_path / ("kat.bsp" if bsp else "kat.sam")
    p.write_text(("" if bsp else "@HD\tVN:1.0\n") + "".join(lines))
    return str(p)


def run(tmp_path, lines, bsp=False, **kw):
    cnt, nmap, ref = CT.counters(NAMES, SEQS, [kat_file(tmp_path, lines, bsp)], **kw)
    return cnt, nmap, ref


def evidence(cnt):
    """{(chrom, 0-based position): (confirm, snp)} where either is non-zero"""
    out = {}
    for c, (_, _, conf, snp) in cnt.items():
        for i in np.nonzero(conf + snp)[0]:
            out[(c, int(i))] = (int(conf[i]), int(snp[i]))
    return out


def bsp_line(seq, chrom, pos1, strand, insert=0):
    return "r\t%s\t%s\tUM\t%s\t%d\t%s\t%d\t%s\t0\t1:0:0:0:0:0\n" % (seq, "I" * len(seq), chrom, pos1, strand, insert, "n" * (len(seq) + 4))


KATS = {
    # '+' hits over reference Gs: G confirms, A is the SNP allele, N counts nothing
    "plus_over_g": ([sam_line(0, "chr1", 1, REF10, "++"), sam_line(0, "chr1", 1, "ACACATTCAA", "++"),
                     sam_line(0, "chr1", 1, "NCACNTTCAN", "++")], {},
                    {("chr1", 0): (1, 1), ("chr1", 4): (1, 1), ("chr1", 9): (1, 1)}),
    # '-' hits over reference Cs: C confirms, T is the SNP allele (SEQ as printed, '-+' unreversed placement)
    "minus_over_c": ([sam_line(16, "chr1", 1, REF10, "-+"), sam_line(16, "chr1", 1, "GTATGTTTAG", "-+")], {},
                     {("chr1", 1): (1, 1), ("chr1", 3): (1, 1), ("chr1", 7): (1, 1)}),
    # lower-case read characters are not upper-cased: they count nothing, as they make no call
    "lower_case": ([sam_line(0, "chr1", 1, "gCACaTTCAG", "++")], {}, {("chr1", 9): (1, 0)}),
    # the same through BSP records
    "bsp": ([bsp_line(REF10, "chr1", 1, "++"), bsp_line("GTATGTTTAG", "chr1", 1, "-+")], {"bsp": True},
            {("chr1", 0): (1, 0), ("chr1", 4): (1, 0), ("chr1", 9): (1, 0), ("chr1", 1): (0, 1), ("chr1", 3): (0, 1), ("chr1", 7): (0, 1)}),
    # -t: '+-' loses its last 2 printed bases, and the G at 9 with them
    "fillin_plus_minus": ([sam_line(16, "chr1", 1, REF10, "+-")], {}, {("chr1", 0): (1, 0), ("chr1", 4): (1, 0)}),
    "fillin_off": ([sam_line(16, "chr1", 1, REF10, "+-")], {"trim_fillin": 0}, {("chr1", 0): (1, 0), ("chr1", 4): (1, 0), ("chr1", 9): (1, 0)}),
    # '--': seq[2:], pos + 2: the C at 1 is gone
    "fillin_minus_minus": ([sam_line(16, "chr1", 1, "GTATGTTTAG", "--")], {}, {("chr1", 3): (0, 1), ("chr1", 7): (0, 1)}),
    # mate-overlap removal: TLEN 10, mate at 0-based 5 -> seq[:5]
    "sam_overlap": ([sam_line(0x1 | 0x2 | 0x40, "chr1", 1, REF10, "++", tlen=10, pnext=6, rnext="=")], {"trim_fillin": 0},
                    {("chr1", 0): (1, 0), ("chr1", 4): (1, 0)}),
    # exclusion: read 1's first cycle and read 2's last cycle
    "ignore_r1_5p": ([sam_line(0, "chr1", 1, REF10, "++")], {"ignore": (1, 0, 0, 0)}, {("chr1", 4): (1, 0), ("chr1", 9): (1, 0)}),
    "ignore_r2_3p": ([sam_line(0x81, "chr1", 1, REF10, "++")], {"ignore": (5, 5, 0, 1)}, {("chr1", 0): (1, 0), ("chr1", 4): (1, 0)}),
    # reversed SEQ ('-+'): cycle 9 - j, so dropping read 1's first 3 cycles removes the C at 7, not at 1
    "ignore_reversed": ([sam_line(16, "chr1", 1, "GTATGTTTAG", "-+")], {"ignore": (3, 0, 0, 0)}, {("chr1", 1): (0, 1), ("chr1", 3): (0, 1)}),
    # -r: the second alignment at the same start and direction does not count
    "rm_dup": ([sam_line(0, "chr1", 1, REF10, "++"), sam_line(0, "chr1", 1, "ACACATTCAA", "++")], {"rm_dup": True},
               {("chr1", 0): (1, 0), ("chr1", 4): (1, 0), ("chr1", 9): (1, 0)}),
    # -g: a CpG's G evidence (from '+' hits) joins its C's (from '-' hits): chr1 3/4, chr2 6/7
    "combine_cpg": ([sam_line(0, "chr1", 1, REF10, "++"), sam_line(16, "chr1", 1, "GTATGTTTAG", "-+"),
                     sam_line(0, "chr2", 5, "GATA", "++"), sam_line(16, "chr2", 5, "GACG", "-+")], {"combine_cpg": True},
                    {("chr1", 0): (1, 0), ("chr1", 3): (1, 1), ("chr1", 9): (1, 0), ("chr1", 1): (0, 1), ("chr1", 7): (0, 1), ("chr2", 4): (1, 0), ("chr2", 6): (1, 1)}),
}


@pytest.mark.parametrize("name", sorted(KATS))
def test_known_evidence(tmp_path, name):
    lines, kw, exp = KATS[name]
    cnt, nmap, _ = run(tmp_path, lines, **kw)
    assert evidence(cnt) == exp
    assert nmap == len(lines) - (1 if kw.get("rm_dup") else 0)


def rows(text):
    """{(chrom, 1-based pos): {column: value}} of a 12-column table"""
    head = text.splitlines()[0].split("\t")
    return {(c[0], int(c[1])): dict(zip(head, c)) for c in (line.split("\t") for line in text.splitlines()[1:])}


# C at chr1:3 (1-based 4): four '+' hits, three show C; two '-' hits, one shows C, one T -> heterozygous
HET = [sam_line(0, "chr1", 1, REF10, "++")] * 3 + [sam_line(0, "chr1", 1, "GCATGTTCAG", "++"),
       sam_line(16, "chr1", 1, REF10, "-+"), sam_line(16, "chr1", 1, "GCATGTTCAG", "-+")]
# C at chr1:7 (1-based 8): one '+' hit shows C; two '-' hits show T -> homozygous C/T
HOM = [sam_line(0, "chr1", 1, REF10, "++"), sam_line(16, "chr1", 1, "GCACGTTTAG", "-+"), sam_line(16, "chr1", 1, "GCACGTTTAG", "-+")]


def table(tmp_path, lines, mode, meth0=False, **kw):
    cnt, _, ref = run(tmp_path, lines, **kw)
    return rows(CT.table(cnt, ref, mode, meth0=meth0)[0])


def test_heterozygous_site(tmp_path):
    r = {m: table(tmp_path, HET, m)[("chr1", 4)] for m in ("no-action", "correct")}
    for m in r:
        assert (r[m]["C_count"], r[m]["CT_count"], r[m]["rev_G_count"], r[m]["rev_GA_count"]) == ("3", "4", "1", "2")
    assert (r["no-action"]["eff_CT_count"], r["no-action"]["ratio"]) == ("4.00", "0.750")
    assert (r["correct"]["eff_CT_count"], r["correct"]["ratio"]) == ("2.00", "1.000")     # min(3, 2) / 2
    assert ("chr1", 4) not in table(tmp_path, HET, "skip")


def test_homozygous_site(tmp_path):
    t = {m: table(tmp_path, HOM, m) for m in CT.MODES}
    assert t["no-action"][("chr1", 8)]["eff_CT_count"] == "1.00" and t["no-action"][("chr1", 8)]["rev_GA_count"] == "2"
    assert ("chr1", 8) not in t["correct"] and ("chr1", 8) not in t["skip"]
    # the '+' C at 1-based 2, confirmed by both '-' hits: kept in every mode
    for m in CT.MODES:
        assert t[m][("chr1", 2)]["eff_CT_count"] == "1.00" and t[m][("chr1", 2)]["rev_G_count"] == "2"


def test_meth0_with_eff(tmp_path):
    """-z: an unmethylated C is printed with its corrected depth; without -z it is not printed"""
    lines = [sam_line(0, "chr1", 1, "GCATGTTCAG", "++"), sam_line(16, "chr1", 1, REF10, "-+"), sam_line(16, "chr1", 1, "GCATGTTCAG", "-+")]
    assert ("chr1", 4) not in table(tmp_path, lines, "correct")
    row = table(tmp_path, lines, "correct", meth0=True)[("chr1", 4)]
    assert (row["ratio"], row["eff_CT_count"], row["C_count"], row["CT_count"]) == ("0.000", "0.50", "0", "1")


def test_summary_is_the_plain_one(tmp_path):
    cnt, _, ref = run(tmp_path, HOM + HET)
    stats = {m: CT.table(cnt, ref, m)[1] for m in CT.MODES}
    assert stats["no-action"] == stats["correct"] == stats["skip"] and stats["skip"][0] > 0


def test_interval_uses_eff(tmp_path):
    """the Wilson interval of a corrected line is the plain formula at depth eff (here 2 with 2 methylated)"""
    row = table(tmp_path, HET, "correct")[("chr1", 4)]
    z, ratio, d = 1.96, 1.0, 2.0
    pmid, sd, nm = ratio + z * z / (2 * d), z * ((ratio * (1 - ratio) / d + z * z / (4 * d * d)) ** 0.5), 1 + z * z / d
    assert (row["CI_lower"], row["CI_upper"]) == ("%.3f" % ((pmid - sd) / nm), "%.3f" % ((pmid + sd) / nm))
