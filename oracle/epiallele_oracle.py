"""oracle/epiallele_oracle.py -- CPU restatement of 4-CpG epialleles: the methylation patterns of reads over windows of
four consecutive CpG sites, with methylation entropy and epipolymorphism (TEST INFRASTRUCTURE ONLY).

Only tests/ may import this module; the product path (bsmap_b200/csrc/bsx_meth.cu) never does.  It restates
pdr_oracle's per-alignment loop (and so conversion_oracle's: alignments from methratio_oracle.parse_alignments and trim,
read number, cycle and context rules from mbias_oracle, the conversion filter and the C/T SNP evidence) and adds the
window rule, so one call returns everything pdr_oracle.pdr returns and the pattern counters; tests/test_epiallele_cpu.py
ties the two together and to the reference script's own tables.

  site         a position c with ref[c] == C and ref[c+1] == G (upper-cased; N and other letters are neither), numbered
               per sequence in reference order; a '+' CpG call at q belongs to site q, a '-' CpG call at q to site q - 1
  call         the PDR call: after the filters, -r, fill-in trimming, mate-overlap removal, the bounds test and the
               per-cycle exclusion; only CpG calls matter
  read's sites the sites whose call position (the C on '+', the G on '-') lies in the trimmed span; one without a call
               breaks every window through it
  window       sites s..s+3; an alignment with a call at all four adds 1 to counts[s][i], i = sum m_k 2^(3-k), k = 0
               for site s, m_k = 1 when methylated; each mate on its own calls; strands pooled, -g changes nothing
  other rules  an alignment dropped by the conversion filter and a -r loser are not scored
  file         header "chr start end reads level entropy EPM patterns"; a line per window with reads >= max(-m, 1);
               skip and correct drop a window with snp > 0 at any of its eight bases; sequences sorted by name;
               start = first C + 1, end = fourth G + 1 (1-based); level = methylated / (4 reads); entropy =
               -(1/4) sum p log2 p; EPM = 1 - sum p^2 (ascending i, in double; %.4f); patterns = 16 counts, i = 0 first
"""
from __future__ import annotations

import math

import numpy as np

import conversion_oracle as CV
import mbias_oracle as MB
import methratio_oracle as MO

CPGS = 4
HEADER = "chr\tstart\tend\treads\tlevel\tentropy\tEPM\tpatterns\n"


def cpg_sites(s: str) -> np.ndarray:
    """0-based positions of the CpG sites (their C) of an upper-cased sequence"""
    r = np.frombuffer(s.encode(), dtype=np.uint8)
    return np.nonzero((r[:-1] == ord("C")) & (r[1:] == ord("G")))[0]


def epialleles(names, seqs, files, min_cpg=4, threshold=0, chroms=None, unique=False, pair=False, trim_fillin=2, combine_cpg=False,
               rm_dup=False, ignore=(0, 0, 0, 0), sam_rules=None):
    """-> pdr_oracle.pdr's dict (counters, mbias, mbias_overflow, bins, dropped, valid, scores, ref, concordant, discordant,
         informative, discordant_alignments, patterns) plus
         sites        {chrom: int64 [n]} the CpG sites' positions
         epi          {chrom: int64 [n, 16]} the pattern counters, row j = the window starting at site j
         spanning     the alignments with at least one window; windows: the windows counted
    min_cpg is PDR's K (pdr's counters come along); threshold the conversion filter's (0 = none dropped)."""
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
    sites = {c: cpg_sites(s) for c, s in ref.items()}
    epi = {c: np.zeros((len(sites[c]), 16), dtype=np.int64) for c in ref}
    refarr = {c: np.frombuffer(s.encode(), dtype=np.uint8) for c, s in ref.items()}
    coverage = {c: np.zeros(len(s), dtype=np.uint8) for c, s in ref.items()} if rm_dup else None
    hist = np.zeros((2, 3, MB.CYCLES, 2), dtype=np.int64)
    bins = np.zeros(CV.BINS, dtype=np.int64)
    overflow = nmap = dropped = informative = n_disc = spanning = windows = 0
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
            if m + u >= min_cpg:                             # PDR: informative, every CpG call counts by the class
                informative += 1
                is_disc = m > 0 and u > 0
                n_disc += is_disc
                np.add.at(disc[cr] if is_disc else conc[cr], p[cpg], 1)
            if m + u >= CPGS:                                # windows: the read's sites in order, called or not
                st = sites[cr]
                shift = 1 if minus else 0                    # the call position of site c: c, or c + 1 on '-'
                a, b = np.searchsorted(st + shift, tpos), np.searchsorted(st + shift, tpos + len(tseq))
                called = np.zeros(b - a, dtype=bool)
                meth = np.zeros(b - a, dtype=np.int64)
                k = np.searchsorted(st, p[cpg] - shift) - a
                called[k] = True
                meth[k] = is_m[cpg]
                run = np.convolve(called.astype(np.int64), np.ones(CPGS, dtype=np.int64), "valid") == CPGS if b - a >= CPGS else np.zeros(0, bool)
                w = np.nonzero(run)[0]
                if len(w):
                    pat = sum(meth[w + t] << (CPGS - 1 - t) for t in range(CPGS))
                    np.add.at(epi[cr], (a + w, pat), 1)
                    spanning += 1
                    windows += len(w)
            meth_, depth, confirm, snp = cnt[cr]
            np.add.at(depth, p, 1)
            np.add.at(meth_, p[is_m], 1)
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
            "discordant_alignments": n_disc, "patterns": patterns, "sites": sites, "epi": epi, "spanning": spanning,
            "windows": windows}


def window_stats(c):
    """(reads, level, entropy, EPM) of one window's 16 counts, computed as the device's writer does"""
    n = int(sum(int(x) for x in c))
    meth = sum(int(x) * bin(i).count("1") for i, x in enumerate(c))
    h = sq = 0.0
    for x in c:
        x = int(x)
        if x:
            p = x / n
            h += p * math.log2(p)
            sq += p * p
    return n, meth / (4 * n), (0.0 - h) / 4.0, 1.0 - sq


def line(cr, pos, c):
    n, level, ent, epm = window_stats(c)
    return "%s\t%d\t%d\t%d\t%.4f\t%.4f\t%.4f\t%s\n" % (cr, pos[0] + 1, pos[CPGS - 1] + 2, n, level, ent, epm, ",".join(str(int(x)) for x in c))


def epiallele_text(res, min_depth=1, ct_snp=None) -> str:
    lines = [HEADER]
    for cr in sorted(res["ref"]):
        st, e = res["sites"][cr], res["epi"][cr]
        snp = res["counters"][cr][3]
        for j in range(len(st) - CPGS + 1):
            if e[j].sum() < max(min_depth, 1):
                continue
            win = st[j:j + CPGS]
            if ct_snp in ("skip", "correct") and (snp[win] > 0).any() | (snp[win + 1] > 0).any():
                continue
            lines.append(line(cr, win, e[j]))
    return "".join(lines)


def stderr_line(res) -> str:
    return "epialleles: %d of %d valid mappings span a %d-CpG window, %d window patterns counted" % (
        res["spanning"], res["valid"], CPGS, res["windows"])
