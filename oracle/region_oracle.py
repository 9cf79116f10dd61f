"""oracle/region_oracle.py -- CPU restatement of the region report (TEST INFRASTRUCTURE ONLY).

Only tests/ may import this module; the product path (bsmap_b200/csrc/bsx_meth.cu) never does.  It takes the counters
of methratio_oracle / ctsnp_oracle / conversion_oracle, {chrom: (meth, depth[, confirm, snp])} after -g combining;
tests/test_region_cpu.py ties its sums to the lines of the reference script's own -z tables.

  region   (chrom, start, end), 0-based and half-open as in BED; start == end is empty; an end past the sequence end is
           clipped when counting and printed as given.  Reported for the contexts CpG, CHG, CHH, in that order.
  site     a reference C (strand '+') or G (strand '-') at q, start <= q < end.  Context: '+' CpG if ref[q+1] == G, else
           CHG if ref[q+2] == G, else CHH; '-' the same with ref[q-1], ref[q-2] and C; non-ACGT bases and positions off
           the sequence count as H (mbias_oracle's rule).  With -g a G that follows a C is not a site: its counts sit on
           the C, and the CpG is one site.
  sites    the number of sites
  covered  the sites whose line the table would print with -z: depth >= max(-m, 1), and with --ct-snp `skip` no SNP
           evidence (snp == 0), with `correct` an eff that is not 0 (snp == 0 or confirm > 0)
  C, CT    over the covered sites: sum of meth (methy_C / C_count) and of depth (total_C / the raw CT_count)
  -z       ignored; `correct`'s scaled eff_CT_count is not summed (the sums stay exact integers)

  report   header "chr start end context sites covered C_count CT_count level", three lines per region in region
           order, level = %.4f of C / CT or NA when CT == 0
  BED      columns 1-3 (tab-separated), further columns ignored; '#', track and browser lines and blank lines skipped;
           CRLF accepted; fewer than 3 columns, a coordinate that is not a non-negative integer or start > end is an
           error naming the line; a region on a sequence not in the reference (or not selected) is skipped and counted
  tiles    [i*W, min((i+1)*W, len)) over every selected sequence, sequences sorted by name (the table's order)
"""
from __future__ import annotations

import numpy as np

CONTEXTS = ("CpG", "CHG", "CHH")
HEADER = "chr\tstart\tend\tcontext\tsites\tcovered\tC_count\tCT_count\tlevel\n"


def site_context(ref: str, combine_cpg=False):
    """-> (site bool[len], context int[len] 0/1/2) of one sequence"""
    r = np.frombuffer(ref.upper().encode(), dtype=np.uint8)
    pad = np.concatenate([np.zeros(2, np.uint8), r, np.zeros(2, np.uint8)])   # off the sequence: neither C nor G
    C, G = ord("C"), ord("G")
    n = len(r)
    at = lambda k: pad[2 + k:2 + k + n]
    plus, minus = r == C, r == G
    ctx_plus = np.where(at(1) == G, 0, np.where(at(2) == G, 1, 2))
    ctx_minus = np.where(at(-1) == C, 0, np.where(at(-2) == C, 1, 2))
    site = plus | minus
    if combine_cpg:
        site &= ~(minus & (at(-1) == C))
    return site, np.where(plus, ctx_plus, ctx_minus)


def prefix_sums(cnt, ref, combine_cpg=False, min_depth=1, ct_snp=None):
    """-> {chrom: int64 [len + 1][3 contexts][sites, covered, C, CT]}, the running sums over positions"""
    out = {}
    for cr, c in cnt.items():
        meth, depth = (np.asarray(x, dtype=np.int64) for x in c[:2])
        site, ctx = site_context(ref[cr], combine_cpg)
        cov = site & (depth >= max(min_depth, 1))
        if ct_snp in ("skip", "correct"):
            confirm, snp = (np.asarray(x, dtype=np.int64) for x in c[2:4])
            cov &= (snp == 0) if ct_snp == "skip" else ((snp == 0) | (confirm > 0))
        per = np.zeros((len(depth) + 1, 3, 4), dtype=np.int64)
        for k in range(3):
            in_k = ctx == k
            per[1:, k, 0] = site & in_k
            per[1:, k, 1] = cov & in_k
            per[1:, k, 2] = np.where(cov & in_k, meth, 0)
            per[1:, k, 3] = np.where(cov & in_k, depth, 0)
        out[cr] = np.cumsum(per, axis=0)
    return out


def regions(cnt, ref, regs, combine_cpg=False, min_depth=1, ct_snp=None):
    """-> int64 [n][3][4] (sites, covered, C, CT) of the regions [(chrom, start, end)]; cnt as in the module doc,
    ref {chrom: sequence}; ct_snp None / "no-action" / "correct" / "skip" """
    ps = prefix_sums(cnt, ref, combine_cpg, min_depth, ct_snp)
    out = np.zeros((len(regs), 3, 4), dtype=np.int64)
    for i, (cr, s, e) in enumerate(regs):
        assert 0 <= s <= e
        n = len(ps[cr]) - 1
        out[i] = ps[cr][min(e, n)] - ps[cr][min(s, n)]
    return out


def report_text(regs, sums) -> str:
    lines = [HEADER]
    for (cr, s, e), v in zip(regs, sums):
        for k, name in enumerate(CONTEXTS):
            sites, cov, c, ct = (int(x) for x in v[k])
            lines.append("%s\t%d\t%d\t%s\t%d\t%d\t%d\t%d\t%s\n" % (cr, s, e, name, sites, cov, c, ct, "%.4f" % (c / ct) if ct else "NA"))
    return "".join(lines)


def parse_bed(text: str, known):
    """-> (regions [(chrom, start, end)] on the sequences in `known`, in file order, skipped regions); ValueError naming
    the line for a malformed one"""
    regs, skipped = [], 0
    for no, line in enumerate(text.split("\n"), 1):
        if line.endswith("\r"):
            line = line[:-1]
        if not line.strip(" \t"):
            continue
        head = line.split(" ")[0].split("\t")[0]
        if line.startswith("#") or head in ("track", "browser"):
            continue
        col = line.split("\t")
        if len(col) < 3:
            raise ValueError("line %d: fewer than 3 columns" % no)
        if not (col[1].isdigit() and col[2].isdigit() and col[1].isascii() and col[2].isascii()):
            raise ValueError("line %d: start and end must be non-negative integers" % no)
        s, e = int(col[1]), int(col[2])
        if s > e:
            raise ValueError("line %d: start %d > end %d" % (no, s, e))
        if col[0] in known:
            regs.append((col[0], s, e))
        else:
            skipped += 1
    return regs, skipped


def tiles(lengths, width):
    """lengths {chrom: length} of the selected sequences -> [(chrom, start, end)] in the table's order"""
    assert width >= 1
    return [(cr, s, min(s + width, lengths[cr])) for cr in sorted(lengths) for s in range(0, lengths[cr], width)]


def skip_line(skipped, total) -> str:
    return "regions: %d of %d skipped (sequence not in the reference or not selected)" % (skipped, total)


def table_line_sums(text, ref, regs):
    """the contract from text alone: per region and context, (lines, sum of the methylated count, sum of the depth)
    of a -z table (plain 9 columns or the 12-column C/T SNP one) whose position lies in the region"""
    cols = None
    rows = {}
    for line in text.splitlines()[1:]:
        c = line.split("\t")
        if cols is None:
            cols = (6, 5) if len(c) == 9 else (6, 7)               # (methy_C, total_C) / (C_count, CT_count)
        q = int(c[1]) - 1
        s = ref[c[0]].upper()
        want, step = ("G", 1) if c[2] == "+" else ("C", -1)
        at = lambda k: 0 <= k < len(s) and s[k] == want
        k = 0 if at(q + step) else (1 if at(q + 2 * step) else 2)
        rows.setdefault(c[0], []).append((q, k, int(c[cols[0]]), int(c[cols[1]])))
    ps = {}
    for cr, rr in rows.items():
        per = np.zeros((len(ref[cr]) + 1, 3, 3), dtype=np.int64)
        for q, k, m, d in rr:
            per[q + 1, k] += (1, m, d)
        ps[cr] = np.cumsum(per, axis=0)
    out = np.zeros((len(regs), 3, 3), dtype=np.int64)
    for i, (cr, s, e) in enumerate(regs):
        if cr in ps:
            n = len(ps[cr]) - 1
            out[i] = ps[cr][min(e, n)] - ps[cr][min(s, n)]
    return out
