"""oracle/ctsnp_oracle.py -- CPU restatement of the C/T SNP evidence and the SNP-corrected table (TEST INFRASTRUCTURE ONLY).

Only tests/ may import this module; the product path (bsmap_b200/csrc/bsx_meth.cu) never does.  It takes its alignments
from methratio_oracle.parse_alignments and trim, and the read number and cycle rule from mbias_oracle, so its calls are
exactly the counters of those two; tests/test_ctsnp_cpu.py ties its no-action table to the reference script's own tables.

  evidence  every base of an alignment that survives the filters, -r, fill-in trimming, mate-overlap removal, the bounds
            test and the per-cycle exclusion (the calls' cycle rule).  q = its reference position.
              '+' hit (first ZS character '+'), ref[q] == G: read G -> confirm[q] += 1, read A -> snp[q] += 1
              '-' hit,                          ref[q] == C: read C -> confirm[q] += 1, read T -> snp[q] += 1
            other read characters, and other reference bases (N included), count nothing
  -g        confirm and snp combine like meth and depth: the CpG's G adds to its C, then is zeroed
  table     chr pos strand context ratio eff_CT_count C_count CT_count rev_G_count rev_GA_count CI_lower CI_upper over the
            lines the plain table prints (CT >= min_depth, CT > 0, C > 0 unless -z); rev_G = confirm, rev_GA = confirm + snp
              no-action  eff = CT
              correct    eff = CT if rev_GA == 0 else float(CT) * rev_G / rev_GA; dropped when eff == 0
              skip       dropped when rev_G < rev_GA, else eff = CT
            ratio = min(C, eff) / eff, the Wilson interval with eff for the depth, eff as %.2f; the summary counts come
            from the raw depth, as the plain table's do
"""
from __future__ import annotations

import numpy as np

import mbias_oracle as MB
import methratio_oracle as MO

MODES = ("no-action", "correct", "skip")
HEADER = "chr\tpos\tstrand\tcontext\tratio\teff_CT_count\tC_count\tCT_count\trev_G_count\trev_GA_count\tCI_lower\tCI_upper\n"


def counters(names, seqs, files, chroms=None, unique=False, pair=False, trim_fillin=2, combine_cpg=False, rm_dup=False,
             ignore=(0, 0, 0, 0), sam_rules=None):
    """-> ({chrom: (meth, depth, confirm, snp)} after the exclusion and -g, valid mappings, {chrom: reference upper case}).
    sam_rules as in mbias_oracle.mbias."""
    ref = {}
    for n, s in zip(names, seqs):
        s = s.decode() if isinstance(s, bytes) else s
        if not chroms or n in chroms:
            ref[n] = s.upper()
    chroms = set(ref)
    cnt = {c: tuple(np.zeros(len(s), dtype=np.int64) for _ in range(4)) for c, s in ref.items()}
    refarr = {c: np.frombuffer(s.encode(), dtype=np.uint8) for c, s in ref.items()}
    coverage = {c: np.zeros(len(s), dtype=np.uint8) for c, s in ref.items()} if rm_dup else None
    nmap = 0
    C, G, A, T = (ord(x) for x in "CGAT")
    for path in files:
        alns = MO.parse_alignments(path, chroms, unique, pair)
        r2 = MB._read2_flags(path, chroms, unique, pair) or [False] * len(alns)
        assert len(r2) == len(alns)
        for (seq, strand, cr, pos, insert, mate_pos, sam), read2 in zip(alns, r2):
            if rm_dup:                                       # methratio.py:52-55
                frag_end, direction = (pos + len(seq), 2) if strand in ("+-", "-+") else (pos, 1)
                if coverage[cr][frag_end] & direction:
                    continue
                coverage[cr][frag_end] |= direction
            L = len(seq)
            tseq, tpos = MO.trim(seq, strand, pos, insert, mate_pos, sam if sam_rules is None else sam_rules, trim_fillin)
            if tpos + len(tseq) > len(ref[cr]):
                continue
            nmap += 1
            if not tseq:
                continue
            start = tpos - pos
            minus = strand[0] == "-"
            match, convert, opp, opp_snp = (G, A, C, T) if minus else (C, T, G, A)
            r = refarr[cr][tpos:tpos + len(tseq)]
            q = np.frombuffer(tseq.encode(), dtype=np.uint8)
            j = start + np.arange(len(tseq))
            cyc = L - 1 - j if strand[0] != strand[1] else j
            lo, hi = (ignore[2], L - ignore[3]) if read2 else (ignore[0], L - ignore[1])
            keep = (cyc >= lo) & (cyc < hi)
            meth, depth, confirm, snp = cnt[cr]
            call = keep & (r == match)
            np.add.at(depth, tpos + np.nonzero(call & ((q == match) | (q == convert)))[0], 1)
            np.add.at(meth, tpos + np.nonzero(call & (q == match))[0], 1)
            ev = keep & (r == opp)
            np.add.at(confirm, tpos + np.nonzero(ev & (q == opp))[0], 1)
            np.add.at(snp, tpos + np.nonzero(ev & (q == opp_snp))[0], 1)
    if combine_cpg:
        for cr in cnt:
            r = refarr[cr]
            cg = np.nonzero((r[:-1] == C) & (r[1:] == G))[0]
            for a in cnt[cr]:
                a[cg] += a[cg + 1]
                a[cg + 1] = 0
    return cnt, nmap, ref


def table(cnt, ref, mode, meth0=False, min_depth=1):
    """-> (12-column table text, (covered cytosines, their summed depth))"""
    assert mode in MODES
    z95, z95sq = 1.96, 1.96 * 1.96
    lines = [HEADER]
    nc = nd = 0
    ss = {"C": "+", "G": "-"}
    for cr in sorted(cnt):
        m_all, d_all, c_all, s_all = cnt[cr]
        refcr = ref[cr]
        for i in np.nonzero((d_all >= min_depth) & (d_all > 0))[0]:
            i = int(i)
            d, m = int(d_all[i]), int(m_all[i])
            nc += 1
            nd += d
            if m == 0 and not meth0:
                continue
            rg = int(c_all[i])
            rga = rg + int(s_all[i])
            eff = d
            if mode == "correct":
                eff = d if rga == 0 else float(d) * rg / rga
                if eff == 0:
                    continue
            elif mode == "skip" and rg < rga:
                continue
            eff = float(eff)
            ratio = min(m, eff) / eff
            pmid = ratio + z95sq / (2 * eff)
            sd = z95 * ((ratio * (1 - ratio) / eff + z95sq / (4 * eff * eff)) ** 0.5)
            nm = 1 + z95sq / eff
            lines.append("%s\t%d\t%c\t%s\t%.3f\t%.2f\t%d\t%d\t%d\t%d\t%.3f\t%.3f\n" % (
                cr, i + 1, ss[refcr[i]], refcr[i - 2:i + 3], ratio, eff, m, d, rg, rga, (pmid - sd) / nm, (pmid + sd) / nm))
    return "".join(lines), (nc, nd)


def methratio_ct_snp(names, seqs, files, mode, meth0=False, min_depth=1, **kw):
    """-> (table text, (valid mappings, covered cytosines, summed depth), counters); kw as for counters()"""
    cnt, nmap, ref = counters(names, seqs, files, **kw)
    txt, (nc, nd) = table(cnt, ref, mode, meth0=meth0, min_depth=min_depth)
    return txt, (nmap, nc, nd), cnt


def project_plain(text):
    """the 12-column table (no-action) as the plain 9-column one: ratio, CT, C and the interval, plain header"""
    out = ["chr\tpos\tstrand\tcontext\tratio\ttotal_C\tmethy_C\tCI_lower\tCI_upper\n"]
    for line in text.splitlines()[1:]:
        c = line.split("\t")
        out.append("\t".join(c[:5] + [c[7], c[6], c[10], c[11]]) + "\n")
    return "".join(out)
