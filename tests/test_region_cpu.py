"""The region report: the numpy restatement (oracle/region_oracle.py) tied to the lines of the reference script's own
-z tables, and hand-computed known answers on a small genome."""
from __future__ import annotations

import gzip
import os
import random
import sys
import zlib

import numpy as np
import pytest

import cases as CS
from test_methratio_cpu import GOLD, MANIFEST, opts_kwargs
from test_mbias_cpu import NAMES, SEQS, oracle_files

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ctsnp_oracle as CT  # noqa: E402
import region_oracle as RO  # noqa: E402

# -g, -m 2, -r and -t 3, written by the reference script with -z
Z_KEYS = ["se_cfg1.g_z", "se_cfg2_r0_uR.z_m_2", "se_cfg5.r_z", "se_mixed_A.z", "rrbs_se_A.z", "pe_sam_v5_R.t_3_z"]


def random_regions(lengths, n, seed, chunk=4096):
    """single positions, empty regions, regions across many chunks, regions straddling chunk edges, ends past the
    sequence end, and the whole sequences"""
    rnd = random.Random(seed)
    names = sorted(lengths)
    regs = [(c, 0, lengths[c]) for c in names]
    for i in range(n):
        c = rnd.choice(names)
        L = lengths[c]
        kind = i % 6
        if kind == 0:
            s = rnd.randrange(L); regs.append((c, s, s + 1))
        elif kind == 1:
            s = rnd.randrange(L + 1); regs.append((c, s, s))
        elif kind == 2:
            s = rnd.randrange(L); regs.append((c, s, s + rnd.randrange(1, 3 * chunk)))
        elif kind == 3:
            edge = rnd.randrange(1, max(2, L // chunk + 1)) * chunk
            regs.append((c, max(0, edge - rnd.randrange(1, 40)), edge + rnd.randrange(1, 40)))
        elif kind == 4:
            s = rnd.randrange(L); regs.append((c, s, L + rnd.randrange(0, 100)))
        else:
            s = rnd.randrange(L); regs.append((c, s, min(L, s + rnd.randrange(1, 400))))
    return regs


@pytest.mark.parametrize("key", Z_KEYS)
def test_oracle_equals_the_reference_table_lines(tmp_path, key):
    """covered, C and CT are the count and sums of the reference script's -z table lines in the region, by context"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    files = oracle_files(ent, case, str(tmp_path))
    kw = opts_kwargs(ent["opts"])
    ckw = {k: v for k, v in kw.items() if k not in ("meth0", "min_depth")}
    cnt, _, ref = CT.counters(d["gnames"], d["gseqs"], files, **ckw)
    lengths = {c: len(s) for c, s in ref.items()}
    regs = random_regions(lengths, 300, seed=zlib.crc32(key.encode()))
    got = RO.regions(cnt, ref, regs, combine_cpg=kw.get("combine_cpg", False), min_depth=kw.get("min_depth", 1))
    table = gzip.open(os.path.join(GOLD, key + ".txt.gz"), "rt").read()
    exp = RO.table_line_sums(table, ref, regs)
    assert np.array_equal(got[:, :, 1:], exp)
    assert (got[:, :, 0] >= got[:, :, 1]).all()
    whole = got[:len(lengths)].sum(axis=0)
    assert whole[:, 1].sum() == len(table.splitlines()) - 1 > 0      # every line lies in one whole-sequence region


# ---- known answers -------------------------------------------------------------------------------------------------
# chr1  0 G  1 C  2 A  3 C  4 G  5 T  6 T  7 C  8 A  9 G  10 C  11 T  12 C  13 N  14 A  15 C  16 C
#   '+' C: 1 CHH, 3 CpG, 7 CHG, 10 CHH, 12 CHH (next to N), 15 CHH, 16 CHH (last base)
#   '-' G: 0 CHH (position 0), 4 CpG (after the C at 3: no site with -g), 9 CHG
# chr2  0 G  1 G  2 T  3 N  4 G  5 A  6 C  7 G        '+' C: 6 CpG      '-' G: 0 CHH, 1 CHH, 4 CHH (next to N), 7 CpG
REF = {n: s.decode() for n, s in zip(NAMES, SEQS)}


def sites(regs, combine_cpg=False, ref=REF):
    cnt = {c: (np.zeros(len(s), np.int64), np.zeros(len(s), np.int64)) for c, s in ref.items()}
    return RO.regions(cnt, ref, regs, combine_cpg=combine_cpg)[:, :, 0].tolist()


SITES = [
    (("chr1", 0, 17), False, [2, 2, 6]),
    (("chr1", 0, 17), True, [1, 2, 6]),
    (("chr1", 0, 1), False, [0, 0, 1]),          # G at the sequence start: q-1, q-2 are off the sequence
    (("chr1", 16, 17), False, [0, 0, 1]),        # C at the sequence end
    (("chr1", 15, 1000), False, [0, 0, 2]),      # clipped
    (("chr1", 12, 14), False, [0, 0, 1]),        # C next to N; N is no site
    (("chr1", 4, 5), False, [1, 0, 0]),
    (("chr1", 4, 5), True, [0, 0, 0]),           # -g: the CpG's G is no site
    (("chr1", 3, 5), True, [1, 0, 0]),
    (("chr1", 5, 5), False, [0, 0, 0]),          # empty
    (("chr1", 17, 30), False, [0, 0, 0]),        # past the end
    (("chr2", 0, 8), False, [2, 0, 3]),
    (("chr2", 0, 8), True, [1, 0, 3]),
    (("chr2", 4, 5), False, [0, 0, 1]),          # G after N
]


@pytest.mark.parametrize("reg,g,exp", SITES)
def test_known_sites(reg, g, exp):
    assert sites([reg], g) == [exp]
    low = {c: s.lower() for c, s in REF.items()}
    assert sites([reg], g, ref=low) == [exp]                     # lower case reads as upper case


def counters():
    """chr1: the CpG C at 3 depth 2 / meth 1; the CHG C at 7 depth 1 / meth 0; CHH C at 10 depth 5 / meth 5 with SNP
    evidence only (confirm 0, snp 1); CHH C at 12 depth 3 / meth 2 with both (confirm 2, snp 1)"""
    z = lambda c: np.zeros(len(REF[c]), np.int64)
    cnt = {c: (z(c), z(c), z(c), z(c)) for c in REF}
    m, d, cf, sn = cnt["chr1"]
    for q, dd, mm, c, s in ((3, 2, 1, 0, 0), (7, 1, 0, 0, 0), (10, 5, 5, 0, 1), (12, 3, 2, 2, 1)):
        d[q], m[q], cf[q], sn[q] = dd, mm, c, s
    return cnt


# (min_depth, ct_snp) -> [context][sites, covered, C, CT] of chr1 as a whole
COVERED = [
    ((1, None), [[2, 1, 1, 2], [2, 1, 0, 1], [6, 2, 7, 8]]),
    ((0, None), [[2, 1, 1, 2], [2, 1, 0, 1], [6, 2, 7, 8]]),    # -m 0 still needs depth > 0
    ((2, None), [[2, 1, 1, 2], [2, 0, 0, 0], [6, 2, 7, 8]]),
    ((3, None), [[2, 0, 0, 0], [2, 0, 0, 0], [6, 2, 7, 8]]),
    ((1, "no-action"), [[2, 1, 1, 2], [2, 1, 0, 1], [6, 2, 7, 8]]),
    ((1, "skip"), [[2, 1, 1, 2], [2, 1, 0, 1], [6, 0, 0, 0]]),  # any SNP evidence drops the line
    ((1, "correct"), [[2, 1, 1, 2], [2, 1, 0, 1], [6, 1, 2, 3]]),   # eff = 5 * 0 / 1 == 0 drops 10; 12 keeps raw CT 3
]


@pytest.mark.parametrize("opt,exp", COVERED)
def test_known_covered_and_sums(opt, exp):
    min_depth, mode = opt
    cnt = counters()
    regs = [("chr1", 0, 17)]
    got = RO.regions(cnt, REF, regs, min_depth=min_depth, ct_snp=mode)
    assert got[0].tolist() == exp
    # the same numbers from the lines of the -z table those counters print
    txt, _ = CT.table(cnt, {c: s.upper() for c, s in REF.items()}, mode or "no-action", meth0=True, min_depth=min_depth)
    assert RO.table_line_sums(txt, REF, regs)[0].tolist() == [row[1:] for row in exp]


def test_overlapping_and_repeated_regions():
    cnt = counters()
    regs = [("chr1", 0, 17), ("chr1", 0, 17), ("chr1", 0, 11), ("chr1", 5, 17), ("chr2", 0, 8), ("chr1", 0, 17)]
    got = RO.regions(cnt, REF, regs)
    assert np.array_equal(got[0], got[1]) and np.array_equal(got[0], got[5])
    overlap = RO.regions(cnt, REF, [("chr1", 5, 11)])[0]
    assert np.array_equal(got[2] + got[3] - overlap, got[0])


def test_tiles_that_do_not_divide_the_length():
    lengths = {c: len(s) for c, s in REF.items()}
    t = RO.tiles(lengths, 5)
    assert t == [("chr1", 0, 5), ("chr1", 5, 10), ("chr1", 10, 15), ("chr1", 15, 17), ("chr2", 0, 5), ("chr2", 5, 8)]
    assert RO.tiles({"b": 3, "a": 2}, 10) == [("a", 0, 2), ("b", 0, 3)]            # sorted by name, as the table
    cnt = counters()
    per = RO.regions(cnt, REF, t)
    whole = RO.regions(cnt, REF, [("chr1", 0, 17), ("chr2", 0, 8)])
    assert np.array_equal(per[:4].sum(axis=0), whole[0]) and np.array_equal(per[4:].sum(axis=0), whole[1])


def test_report_text():
    regs = [("chr1", 0, 17), ("chr2", 0, 1000)]
    txt = RO.report_text(regs, RO.regions(counters(), REF, regs))
    assert txt == RO.HEADER + ("chr1\t0\t17\tCpG\t2\t1\t1\t2\t0.5000\n"
                               "chr1\t0\t17\tCHG\t2\t1\t0\t1\t0.0000\n"
                               "chr1\t0\t17\tCHH\t6\t2\t7\t8\t0.8750\n"
                               "chr2\t0\t1000\tCpG\t2\t0\t0\t0\tNA\n"
                               "chr2\t0\t1000\tCHG\t0\t0\t0\t0\tNA\n"
                               "chr2\t0\t1000\tCHH\t3\t0\t0\t0\tNA\n")


def test_parse_bed():
    text = ("# comment\ntrack name=x\nbrowser position chr1:1-10\n\n \t\nchr1\t3\t9\tname\t0\t+\r\n"
            "chrX\t0\t5\nchr2\t0\t100\nchr1\t4\t4\n")
    regs, skipped = RO.parse_bed(text, {"chr1", "chr2"})
    assert regs == [("chr1", 3, 9), ("chr2", 0, 100), ("chr1", 4, 4)] and skipped == 1
    assert RO.skip_line(1, 4) == "regions: 1 of 4 skipped (sequence not in the reference or not selected)"
    for bad, msg in (("chr1\t3\n", "line 2: fewer than 3 columns"), ("chr1\tx\t5\n", "line 2: start and end"),
                     ("chr1\t-1\t5\n", "line 2: start and end"), ("chr1\t9\t5\n", "line 2: start 9 > end 5")):
        with pytest.raises(ValueError, match=msg):
            RO.parse_bed("#\n" + bad, {"chr1"})
