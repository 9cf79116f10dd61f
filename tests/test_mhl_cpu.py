"""Methylation haplotype load: the numpy restatement (oracle/mhl_oracle.py) on hand-computed known answers, its
histogram-plus-clip reduction against direct l-mer enumeration, and its agreement with the epiallele and region
oracles on every golden methratio run."""
from __future__ import annotations

import os
import sys

import numpy as np
import pytest

import cases as CS
from test_methratio_cpu import MANIFEST
from test_mbias_cpu import mbias_kwargs, oracle_files, sam_line
from test_pdr_cpu import kat_file

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import epiallele_oracle as EP  # noqa: E402
import mhl_oracle as MH  # noqa: E402
import region_oracle as RG  # noqa: E402

# CpG sites j = 0..39 at 3 + 4 j (the C of ACGT)
NAMES = ["chrK"]
SEQS = ["TT" + "ACGT" * 40 + "TT"]


def read(n_sites, pattern=None, first=0):
    """a '+' read over sites first .. first + n_sites - 1 (it starts at the A before the first): pattern[k] 'M' keeps
    the C, 'U' converts it, 'N' puts an N there (no call); default all methylated -> (1-based POS, SEQ)"""
    pattern = pattern or "M" * n_sites
    s = list(SEQS[0][2 + 4 * first:2 + 4 * (first + n_sites)])
    for k, c in enumerate(pattern):
        s[4 * k + 1] = {"M": "C", "U": "T", "N": "N"}[c]
    return 3 + 4 * first, "".join(s)


def lines_of(*reads):
    return [sam_line(0, "chrK", pos, seq, "++") for pos, seq in reads]


WHOLE = [("chrK", 0, len(SEQS[0]))]
# name -> (reads, regions, ct_snp, [(L, MHL, uMHL, T, M, U)] per region)
KATS = {
    "clonal": (lines_of(read(4), read(4), read(4, "UUUU"), read(4, "UUUU")), WHOLE, None,
               [(4, "0.5000", "0.5000", [16, 12, 8, 4], [8, 6, 4, 2], [8, 6, 4, 2])]),
    "alternating": (lines_of(read(4, "MUMU"), read(4, "UMUM")), WHOLE, None,
                    [(4, "0.0500", "0.0500", [8, 6, 4, 2], [4, 0, 0, 0], [4, 0, 0, 0])]),
    "gap": (lines_of(read(5, "MMNMM")), WHOLE, None, [(2, "1.0000", "0.0000", [4, 2], [4, 2], [0, 0])]),
    # sites 1, 2 only ([6, 12) holds the Cs at 7 and 11); site 1 only; no site; a start past the end
    "edges": (lines_of(read(4)), [("chrK", 6, 12), ("chrK", 4, 8), ("chrK", 0, 3), ("chrK", 500, 900)], None,
              [(2, "1.0000", "0.0000", [2, 1], [2, 1], [0, 0]), (1, "1.0000", "0.0000", [1], [1], [0]), (0,) * 6, (0,) * 6]),
    "long": (lines_of(read(20)), WHOLE, None,
             [(16, "1.0000", "0.0000", [20 - l + 1 for l in range(1, 17)], [20 - l + 1 for l in range(1, 17)], [0] * 16)]),
}


def _snp_read():
    pos, seq = read(4)
    s = list(seq)
    s[4 * 2 + 2] = "A"                                      # the G of site 2 read as A: C/T SNP evidence on the '+' strand
    return pos, "".join(s)


KATS["snp_skip"] = (lines_of(_snp_read()), WHOLE, "skip", [(2, "1.0000", "0.0000", [3, 1], [3, 1], [0, 0])])
KATS["snp_off"] = (lines_of(_snp_read()), WHOLE, None, [(4, "1.0000", "0.0000", [4, 3, 2, 1], [4, 3, 2, 1], [0, 0, 0, 0])])


def expected_line(reg, ln):
    cr, s, e = reg
    sites = int(np.sum((np.array([3 + 4 * j for j in range(40)]) >= s) & (np.array([3 + 4 * j for j in range(40)]) < min(e, len(SEQS[0])))))
    if ln[0] == 0:
        return "%s\t%d\t%d\t%d\t0\t0\tNA\tNA\tNA\tNA\tNA\n" % (cr, s, e, sites)
    L, hm, hu, T, M, U = ln
    j = lambda v: ",".join(str(x) for x in v)
    return "%s\t%d\t%d\t%d\t%d\t%d\t%s\t%s\t%s\t%s\t%s\n" % (cr, s, e, sites, T[0], L, hm, hu, j(T), j(M), j(U))


@pytest.mark.parametrize("name", sorted(KATS))
def test_known_answers(tmp_path, name):
    lines, regs, ct_snp, exp = KATS[name]
    res = MH.mhl(NAMES, SEQS, [kat_file(tmp_path, lines)], trim_fillin=0)
    assert res["valid"] == len(lines)
    assert MH.mhl_text(res, regs, ct_snp) == MH.HEADER + "".join(expected_line(r, e) for r, e in zip(regs, exp))
    cut = MH.cut_sites(res, "chrK", ct_snp)
    for (cr, s, e) in regs:
        a, b = MH.site_range(res, cr, s, e)
        assert np.array_equal(MH.region_sums(res["counts"][cr], cut, a, b), MH.region_sums_direct(res["haplotypes"][cr], cut, a, b))


def test_stderr_line(tmp_path):
    res = MH.mhl(NAMES, SEQS, [kat_file(tmp_path, lines_of(read(5, "MMNMM"), read(3, "UUU")) + [sam_line(0, "chrK", 1, "TTAA", "++")])],
                 trim_fillin=0)
    assert MH.stderr_line(res) == "MHL: 2 of 3 valid mappings carry a CpG call, 7 CpG calls in haplotypes"


@pytest.mark.parametrize("seed", range(6))
def test_histogram_equals_direct_enumeration(seed):
    """random haplotypes (runs longer than 16, gaps, every start) and random cuts: the reduction over the run counters
    equals counting the l-mers of the haplotypes themselves, for random site ranges"""
    rng = np.random.default_rng(seed)
    n = 80
    for _ in range(50):
        counts = np.zeros((n, 3, MH.MAX_LEN), dtype=np.int64)
        haps = []
        for _ in range(int(rng.integers(1, 12))):
            k = int(rng.integers(1, 40))
            first = int(rng.integers(0, n - k + 1))
            called = rng.random(k) < rng.choice([0.7, 0.95, 1.0])
            meth = rng.random(k) < rng.choice([0.0, 0.5, 0.9, 1.0])
            haps.append((first, called, meth))
            MH.add_runs(counts, first, called, meth)
        cut = rng.random(n) < rng.choice([0.0, 0.05, 0.2])
        a = int(rng.integers(0, n))
        b = int(rng.integers(a, n + 1))
        assert np.array_equal(MH.region_sums(counts, cut, a, b), MH.region_sums_direct(haps, cut, a, b)), (seed, a, b)


def golden(tmp_path, key):
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    files = oracle_files(ent, case, str(tmp_path))
    return ent, d, files, mbias_kwargs(ent["opts"])


def region_list(d, res):
    lengths = {n: len(s) for n, s in res["ref"].items()}
    return RG.tiles(lengths, 60) + RG.tiles(lengths, 1000) + [(n, 0, L) for n, L in lengths.items()]


@pytest.mark.parametrize("key", sorted(MANIFEST))
def test_agrees_with_the_epiallele_and_region_oracles(tmp_path, key):
    """every golden run: the valid count is the epiallele oracle's; T_4, M_4 and U_4 of a region are the sums over the
    4-CpG windows inside it of reads, counts[15] and counts[0]; T_1 and M_1 are the pooled CpG calls (with -g, the
    region report's CpG CT_count and C_count); the reduction equals direct enumeration"""
    ent, d, files, kw = golden(tmp_path, key)
    res = MH.mhl(d["gnames"], d["gseqs"], files, **{k: v for k, v in kw.items() if k != "combine_cpg"})
    ep = EP.epialleles(d["gnames"], d["gseqs"], files, **kw)
    assert res["valid"] == ep["valid"]
    assert res["calls"] > 0
    regs = region_list(d, res)
    sums = MH.regions(res, regs)
    cnt = ep["counters"]
    if not kw.get("combine_cpg"):                         # the region report's CpG lines after -g pool both strands
        cnt = {c: tuple(x.copy() for x in v) for c, v in cnt.items()}
        for c, v in cnt.items():
            st = ep["sites"][c]
            for x in v[:2]:
                x[st] += x[st + 1]
                x[st + 1] = 0
    rr = RG.regions(cnt, ep["ref"], regs, combine_cpg=True)
    for (cr, s, e), (n, t), r in zip(regs, sums, rr):
        st = ep["sites"][cr]
        a, b = MH.site_range(res, cr, s, e)
        assert n == b - a == r[0][0]
        win = ep["epi"][cr][a:max(b - 3, a)]
        assert t[0, 3] == win.sum() and t[1, 3] == win[:, 15].sum() and t[2, 3] == win[:, 0].sum(), (cr, s, e)
        assert t[0, 0] == r[0][3] and t[1, 0] == r[0][2], (cr, s, e)
        assert t[0, 0] == t[1, 0] + t[2, 0]
    cut = np.zeros(0, dtype=bool)
    for cr in res["ref"]:
        cut = MH.cut_sites(res, cr, "skip")
        n = len(res["sites"][cr])
        for a, b in ((0, n), (0, n // 2), (n // 3, n)):
            for c in (cut, np.zeros(n, dtype=bool)):
                assert np.array_equal(MH.region_sums(res["counts"][cr], c, a, b), MH.region_sums_direct(res["haplotypes"][cr], c, a, b))
