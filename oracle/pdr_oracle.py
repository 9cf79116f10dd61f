"""oracle/pdr_oracle.py -- CPU restatement of read-level CpG concordance, the proportion of discordant reads (TEST
INFRASTRUCTURE ONLY).

Only tests/ may import this module; the product path (bsmap_b200/csrc/bsx_meth.cu) never does.  It restates
conversion_oracle's per-alignment loop (alignments from methratio_oracle.parse_alignments and trim; read number, cycle
and context rules from mbias_oracle; the conversion filter and the C/T SNP evidence) and adds the CpG pattern of each
alignment, so one call returns everything conversion_oracle.conversion returns and the concordance counters;
tests/test_pdr_cpu.py ties the two together and to the reference script's own tables.

  call         one increment of the counters: after the filters, -r, fill-in trimming, mate-overlap removal, the bounds
               test and the per-cycle exclusion
  context      '+': CpG if ref[q+1] == G; '-': CpG if ref[q-1] == C (positions off the sequence are not)
  pattern      m = the alignment's methylated CpG calls, u = its unmethylated ones; each mate on its own calls
  informative  m + u >= K (1..255); concordant when m == 0 or u == 0, else discordant
  counters     each CpG call of an informative alignment adds 1 to concordant[q] or discordant[q] by the alignment's
               class; -g adds a CpG's G counts to its C and zeroes the G
  other rules  an alignment dropped by the conversion filter and a -r loser are not scored
  file         header "chr pos strand concordant discordant PDR"; a line per position with concordant + discordant >=
               max(-m, 1) that the C/T SNP mode would not drop (skip: snp > 0; correct: snp > 0 and confirm == 0); sequences
               sorted by name; strand from the reference base; PDR = discordant / (concordant + discordant) as %.3f
  regions      the region report with "concordant discordant PDR" on every line: on the CpG line the sums over the PDR
               file's lines in the region and PDR %.4f (NA at 0), on the CHG and CHH lines 0 0 NA
"""
from __future__ import annotations

import numpy as np

import conversion_oracle as CV
import mbias_oracle as MB
import methratio_oracle as MO
import region_oracle as RG

HEADER = "chr\tpos\tstrand\tconcordant\tdiscordant\tPDR\n"
REGION_HEADER = RG.HEADER[:-1] + "\tconcordant\tdiscordant\tPDR\n"


def pdr(names, seqs, files, min_cpg=4, threshold=0, chroms=None, unique=False, pair=False, trim_fillin=2, combine_cpg=False,
        rm_dup=False, ignore=(0, 0, 0, 0), sam_rules=None):
    """-> conversion_oracle.conversion's dict (counters, mbias, mbias_overflow, bins, dropped, valid, scores, ref) plus
         concordant, discordant  {chrom: int64 [len]} after -g
         informative             the informative alignments; discordant_alignments: the discordant ones
         patterns                per file, one entry per alignment parse_alignments keeps: (m, u) of a scored alignment,
                                 None when it is no valid mapping or was dropped by the conversion filter
    threshold: the conversion filter's (0 = none dropped)."""
    assert 1 <= min_cpg <= 255 and 0 <= threshold < CV.BINS
    ref = {}
    for n, s in zip(names, seqs):
        s = s.decode() if isinstance(s, bytes) else s
        if not chroms or n in chroms:
            ref[n] = s.upper()
    chroms = set(ref)
    cnt = {c: tuple(np.zeros(len(s), dtype=np.int64) for _ in range(4)) for c, s in ref.items()}
    conc = {c: np.zeros(len(s), dtype=np.int64) for c, s in ref.items()}
    disc = {c: np.zeros(len(s), dtype=np.int64) for c, s in ref.items()}
    refarr = {c: np.frombuffer(s.encode(), dtype=np.uint8) for c, s in ref.items()}
    coverage = {c: np.zeros(len(s), dtype=np.uint8) for c, s in ref.items()} if rm_dup else None
    hist = np.zeros((2, 3, MB.CYCLES, 2), dtype=np.int64)
    bins = np.zeros(CV.BINS, dtype=np.int64)
    overflow = nmap = dropped = informative = n_disc = 0
    scores, patterns = [], []
    C, G, A, T = (ord(x) for x in "CGAT")
    for path in files:
        alns = MO.parse_alignments(path, chroms, unique, pair)
        r2 = MB._read2_flags(path, chroms, unique, pair) or [False] * len(alns)
        assert len(r2) == len(alns)
        fs, fp = [], []
        scores.append(fs)
        patterns.append(fp)
        for (seq, strand, cr, pos, insert, mate_pos, sam), read2 in zip(alns, r2):
            if rm_dup:                                       # methratio.py:52-55, before the filter
                frag_end, direction = (pos + len(seq), 2) if strand in ("+-", "-+") else (pos, 1)
                if coverage[cr][frag_end] & direction:
                    fs.append(None)
                    fp.append(None)
                    continue
                coverage[cr][frag_end] |= direction
            L = len(seq)
            tseq, tpos = MO.trim(seq, strand, pos, insert, mate_pos, sam if sam_rules is None else sam_rules, trim_fillin)
            if tpos + len(tseq) > len(ref[cr]):
                fs.append(None)
                fp.append(None)
                continue
            nmap += 1
            start = tpos - pos
            minus = strand[0] == "-"
            match, convert, opp, opp_snp = (G, A, C, T) if minus else (C, T, G, A)
            r = refarr[cr]
            q = np.frombuffer(tseq.encode(), dtype=np.uint8)
            rr = r[tpos:tpos + len(tseq)]
            jj = start + np.arange(len(tseq))
            cyc_all = L - 1 - jj if strand[0] != strand[1] else jj
            lo, hi = (ignore[2], L - ignore[3]) if read2 else (ignore[0], L - ignore[1])
            keep = (cyc_all >= lo) & (cyc_all < hi)
            i = np.nonzero(keep & (rr == match) & ((q == match) | (q == convert)))[0]
            is_m, cyc, p = q[i] == match, cyc_all[i], tpos + i
            want, step = (C, -1) if minus else (G, 1)

            def at(k):
                ok = (k >= 0) & (k < len(r))
                return ok & (r[np.clip(k, 0, len(r) - 1)] == want)
            ctx = np.where(at(p + step), 0, np.where(at(p + 2 * step), 1, 2))
            score = int((is_m & (ctx != 0)).sum())
            fs.append(score)
            bins[min(score, CV.BINS - 1)] += 1
            if threshold and score >= threshold:
                dropped += 1
                fp.append(None)
                continue
            cpg = ctx == 0
            m, u = int((is_m & cpg).sum()), int((~is_m & cpg).sum())
            fp.append((m, u))
            if m + u >= min_cpg:                             # informative: every CpG call counts by the class
                informative += 1
                is_disc = m > 0 and u > 0
                n_disc += is_disc
                np.add.at(disc[cr] if is_disc else conc[cr], p[cpg], 1)
            meth, depth, confirm, snp = cnt[cr]
            np.add.at(depth, p, 1)
            np.add.at(meth, p[is_m], 1)
            inr = cyc < MB.CYCLES
            overflow += int((~inr).sum())
            np.add.at(hist, (int(read2), ctx[inr], cyc[inr], np.where(is_m[inr], 0, 1)), 1)
            ev = keep & (rr == opp)
            np.add.at(confirm, tpos + np.nonzero(ev & (q == opp))[0], 1)
            np.add.at(snp, tpos + np.nonzero(ev & (q == opp_snp))[0], 1)
    if combine_cpg:
        for cr in cnt:
            r = refarr[cr]
            cg = np.nonzero((r[:-1] == C) & (r[1:] == G))[0]
            for a in cnt[cr] + (conc[cr], disc[cr]):
                a[cg] += a[cg + 1]
                a[cg + 1] = 0
    return {"counters": cnt, "mbias": hist, "mbias_overflow": overflow, "bins": bins, "dropped": dropped, "valid": nmap,
            "scores": scores, "ref": ref, "concordant": conc, "discordant": disc, "informative": informative,
            "discordant_alignments": n_disc, "patterns": patterns}


def shown(res, cr, min_depth=1, ct_snp=None):
    """bool [len]: the positions of sequence cr that the PDR file prints"""
    c, d = res["concordant"][cr], res["discordant"][cr]
    keep = c + d >= max(min_depth, 1)
    if ct_snp in ("skip", "correct"):
        confirm, snp = res["counters"][cr][2:4]
        keep &= (snp == 0) if ct_snp == "skip" else ((snp == 0) | (confirm > 0))
    return keep


def pdr_text(res, min_depth=1, ct_snp=None) -> str:
    lines = [HEADER]
    for cr in sorted(res["ref"]):
        s = res["ref"][cr]
        c, d = res["concordant"][cr], res["discordant"][cr]
        for q in np.nonzero(shown(res, cr, min_depth, ct_snp))[0]:
            x, y = int(c[q]), int(d[q])
            lines.append("%s\t%d\t%s\t%d\t%d\t%.3f\n" % (cr, q + 1, "+" if s[q] == "C" else "-", x, y, y / (x + y)))
    return "".join(lines)


def stderr_line(res, min_cpg) -> str:
    return "PDR: %d of %d valid mappings informative (>= %d CpG calls), %d discordant" % (
        res["informative"], res["valid"], min_cpg, res["discordant_alignments"])


def region_pdr(res, regs, min_depth=1, ct_snp=None):
    """-> int64 [n][concordant, discordant]: the sums over the PDR file's lines in each region (chrom, start, end)"""
    ps = {}
    for cr in res["ref"]:
        keep = shown(res, cr, min_depth, ct_snp)
        per = np.zeros((len(keep) + 1, 2), dtype=np.int64)
        per[1:, 0] = np.where(keep, res["concordant"][cr], 0)
        per[1:, 1] = np.where(keep, res["discordant"][cr], 0)
        ps[cr] = np.cumsum(per, axis=0)
    out = np.zeros((len(regs), 2), dtype=np.int64)
    for i, (cr, s, e) in enumerate(regs):
        n = len(ps[cr]) - 1
        out[i] = ps[cr][min(e, n)] - ps[cr][min(s, n)]
    return out


def region_text(res, regs, combine_cpg=False, min_depth=1, ct_snp=None) -> str:
    """the region report with the PDR columns"""
    sums = RG.regions(res["counters"], res["ref"], regs, combine_cpg=combine_cpg, min_depth=min_depth, ct_snp=ct_snp)
    pd = region_pdr(res, regs, min_depth, ct_snp)
    base = RG.report_text(regs, sums).splitlines(keepends=True)[1:]
    lines = [REGION_HEADER]
    for i in range(len(regs)):
        x, y = (int(v) for v in pd[i])
        for k in range(3):
            ext = ("%d\t%d\t%s" % (x, y, "%.4f" % (y / (x + y)) if x + y else "NA")) if k == 0 else "0\t0\tNA"
            lines.append(base[3 * i + k][:-1] + "\t" + ext + "\n")
    return "".join(lines)
