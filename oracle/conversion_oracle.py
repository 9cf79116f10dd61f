"""oracle/conversion_oracle.py -- CPU restatement of the conversion filter (TEST INFRASTRUCTURE ONLY).

Only tests/ may import this module; the product path (bsmap_b200/csrc/bsx_meth.cu) never does.  It takes its alignments
from methratio_oracle.parse_alignments and trim, and the read number, cycle rule and context rule from mbias_oracle, so
with threshold 0 its counters are exactly mbias_oracle's; tests/test_conversion_cpu.py ties them to the reference
script's own tables.

  call      one increment of the counters: after the filters, -r, fill-in trimming, mate-overlap removal, the bounds
            test and the per-cycle exclusion (excluded cycles, trimmed bases and the mate overlap hold no call)
  context   '+': CpG if ref[q+1] == G, else CHG if ref[q+2] == G, else CHH; '-': the same with ref[q-1], ref[q-2] and C;
            non-ACGT bases and positions off the sequence count as H
  score     the alignment's methylated calls (read C on '+', read G on '-') in CHG or CHH context
  filter    threshold N in 1..255: an alignment with score >= N adds nothing (meth, depth, M-bias, C/T SNP evidence) but
            is still a valid mapping; N = 0 drops nothing
  -r        decided before the filter: a dropped alignment still holds its (fragment end, direction)
  report    bins[min(score, 255)] += 1 for every valid mapping; dropped = sum of bins[N:] (0 when N = 0)
"""
from __future__ import annotations

import numpy as np

import ctsnp_oracle as CT
import mbias_oracle as MB
import methratio_oracle as MO

BINS = 256
HEADER = "methylated_nonCpG_calls\talignments\tdropped\n"


def records(path, chroms, unique=False, pair=False):
    """(0-based line number, QNAME / read id) of each alignment parse_alignments keeps, in its order"""
    sam = path[-4:].upper() == ".SAM"
    out = []
    for ln, line in enumerate(open(path)):
        if sam and line.startswith("@"):
            continue
        col = line.rstrip("\n").split("\t")
        if sam:
            f = int(col[1])
            if f & 0x4 or (unique and f & 0x100) or (pair and not f & 0x2) or col[2] not in chroms:
                continue
        else:
            flag = col[3][:2]
            if flag in ("NM", "QC") or (unique and flag != "UM") or (pair and col[7] == "0") or col[4] not in chroms:
                continue
        out.append((ln, col[0]))
    return out


def conversion(names, seqs, files, threshold=0, chroms=None, unique=False, pair=False, trim_fillin=2, combine_cpg=False,
               rm_dup=False, ignore=(0, 0, 0, 0), sam_rules=None):
    """-> dict with
         counters  {chrom: (meth, depth, confirm, snp)} of the kept alignments, after the exclusion and -g
         mbias     int64 [read][context][cycle][methylated, unmethylated] of the kept calls; mbias_overflow
         bins      int64 [BINS], the valid mappings by score; dropped; valid (the valid mappings)
         scores    per file, one entry per alignment parse_alignments keeps, in file order: its score, or None when it
                   is no valid mapping (-r loser, or past the sequence end)
    sam_rules as in mbias_oracle.mbias."""
    assert 0 <= threshold < BINS
    ref = {}
    for n, s in zip(names, seqs):
        s = s.decode() if isinstance(s, bytes) else s
        if not chroms or n in chroms:
            ref[n] = s.upper()
    chroms = set(ref)
    cnt = {c: tuple(np.zeros(len(s), dtype=np.int64) for _ in range(4)) for c, s in ref.items()}
    refarr = {c: np.frombuffer(s.encode(), dtype=np.uint8) for c, s in ref.items()}
    coverage = {c: np.zeros(len(s), dtype=np.uint8) for c, s in ref.items()} if rm_dup else None
    hist = np.zeros((2, 3, MB.CYCLES, 2), dtype=np.int64)
    bins = np.zeros(BINS, dtype=np.int64)
    overflow = nmap = dropped = 0
    scores = []
    C, G, A, T = (ord(x) for x in "CGAT")
    for path in files:
        alns = MO.parse_alignments(path, chroms, unique, pair)
        r2 = MB._read2_flags(path, chroms, unique, pair) or [False] * len(alns)
        assert len(r2) == len(alns)
        fs = []
        scores.append(fs)
        for (seq, strand, cr, pos, insert, mate_pos, sam), read2 in zip(alns, r2):
            if rm_dup:                                       # methratio.py:52-55, before the filter
                frag_end, direction = (pos + len(seq), 2) if strand in ("+-", "-+") else (pos, 1)
                if coverage[cr][frag_end] & direction:
                    fs.append(None)
                    continue
                coverage[cr][frag_end] |= direction
            L = len(seq)
            tseq, tpos = MO.trim(seq, strand, pos, insert, mate_pos, sam if sam_rules is None else sam_rules, trim_fillin)
            if tpos + len(tseq) > len(ref[cr]):
                fs.append(None)
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
            bins[min(score, BINS - 1)] += 1
            if threshold and score >= threshold:
                dropped += 1
                continue
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
            for a in cnt[cr]:
                a[cg] += a[cg + 1]
                a[cg + 1] = 0
    return {"counters": cnt, "mbias": hist, "mbias_overflow": overflow, "bins": bins, "dropped": dropped, "valid": nmap,
            "scores": scores, "ref": ref}


def report_text(bins, threshold) -> str:
    """the report: one row per non-empty bin, the last labelled 255+; dropped 1 / 0 per bin"""
    lines = [HEADER]
    for b in range(BINS):
        if bins[b]:
            lines.append("%s\t%d\t%d\n" % ("%d+" % b if b == BINS - 1 else str(b), int(bins[b]), 1 if threshold and b >= threshold else 0))
    return "".join(lines)


def stderr_line(res, threshold) -> str:
    if threshold:
        return "conversion filter: %d of %d valid mappings dropped (>= %d methylated non-CpG calls)" % (res["dropped"], res["valid"], threshold)
    return "conversion filter: 0 of %d valid mappings dropped (report only)" % res["valid"]


def table(res, meth0=False, min_depth=1, ct_snp=None):
    """the methratio table of the kept alignments -> (text, (covered cytosines, summed depth)): ctsnp_oracle's 12-column
    table in mode ct_snp, or without it, that table in no-action mode projected onto the plain 9 columns"""
    txt, stats = CT.table(res["counters"], res["ref"], ct_snp or "no-action", meth0=meth0, min_depth=min_depth)
    return (txt if ct_snp else CT.project_plain(txt)), stats
