"""oracle/mhl_oracle.py -- CPU restatement of the methylation haplotype load (MHL, uMHL; Guo et al., Nat Genet 2017) over
regions, from the runs of consecutive CpG calls of each alignment (TEST INFRASTRUCTURE ONLY).

Only tests/ may import this module; the product path (bsmap_b200/csrc/bsx_meth.cu) never does.  It restates
epiallele_oracle's per-alignment loop (alignments, trimming, -r, bounds test, cycle exclusion, the conversion filter and
the C/T SNP evidence) for the calls, and keeps each scored alignment's haplotype; the rules are those of
include/bsmap_b200.h:

  site, call   as for epialleles: a '+' CpG call at q belongs to site q, a '-' one to site q - 1; strands pooled; each
               mate on its own calls; conversion-filter drops and -r losers not scored; -g changes nothing
  haplotype    the alignment's sites in order (call position inside the trimmed span); a site without a call breaks it
  counters     counts[s][f][min(run, 16) - 1] += 1 for each called site s, f = 0 (the run of called sites ending at s)
               and f = 1 or 2 (the run of methylated / unmethylated sites ending at s)
  region       (seq, start, end) clipped to the sequence; its sites [a, b) those whose C lies in [start, end)
  cuts         skip / correct: a site with snp > 0 at its C or G is not counted, nor any haplotype through it
  reduction    T_l, M_l, U_l = sum over s in [a, b) with l <= s - a + 1 and no cut in [s - l + 1, s] of sum_{r >= l}
               counts[s][f][r - 1]; region_sums_direct enumerates the l-mers of the haplotypes instead
  file         "chr start end sites calls L MHL uMHL haplotypes methylated unmethylated"; MHL = (sum over ascending l of
               float(l M_l) / float(T_l)) / (L (L + 1) / 2), %.4f; NA when L = 0
"""
from __future__ import annotations

import numpy as np

import mbias_oracle as MB
import methratio_oracle as MO

MAX_LEN = 16
HEADER = "chr\tstart\tend\tsites\tcalls\tL\tMHL\tuMHL\thaplotypes\tmethylated\tunmethylated\n"


def cpg_sites(s: str) -> np.ndarray:
    r = np.frombuffer(s.encode(), dtype=np.uint8)
    return np.nonzero((r[:-1] == ord("C")) & (r[1:] == ord("G")))[0]


def mhl(names, seqs, files, threshold=0, chroms=None, unique=False, pair=False, trim_fillin=2, rm_dup=False, ignore=(0, 0, 0, 0),
        sam_rules=None):
    """-> dict: ref {chrom: upper-cased sequence}, sites {chrom: int64 [n]}, counts {chrom: int64 [n, 3, 16]},
    snp {chrom: int64 [len]} (the C/T SNP evidence, uncombined), valid, alignments (with a CpG call), calls, and
    haplotypes {chrom: [(first site index, called bool [k], methylated bool [k])]} for direct enumeration"""
    ref = {}
    for n, s in zip(names, seqs):
        s = s.decode() if isinstance(s, bytes) else s
        if not chroms or n in chroms:
            ref[n] = s.upper()
    chroms = set(ref)
    sites = {c: cpg_sites(s) for c, s in ref.items()}
    counts = {c: np.zeros((len(sites[c]), 3, MAX_LEN), dtype=np.int64) for c in ref}
    snp = {c: np.zeros(len(s), dtype=np.int64) for c, s in ref.items()}
    haps = {c: [] for c in ref}
    refarr = {c: np.frombuffer(s.encode(), dtype=np.uint8) for c, s in ref.items()}
    coverage = {c: np.zeros(len(s), dtype=np.uint8) for c, s in ref.items()} if rm_dup else None
    nmap = n_aln = n_calls = 0
    C, G, A, T = (ord(x) for x in "CGAT")
    for path in files:
        alns = MO.parse_alignments(path, chroms, unique, pair)
        r2 = MB._read2_flags(path, chroms, unique, pair) or [False] * len(alns)
        assert len(r2) == len(alns)
        for (seq, strand, cr, pos, insert, mate_pos, sam), read2 in zip(alns, r2):
            if rm_dup:
                frag_end, direction = (pos + len(seq), 2) if strand in ("+-", "-+") else (pos, 1)
                if coverage[cr][frag_end] & direction:
                    continue
                coverage[cr][frag_end] |= direction
            L = len(seq)
            tseq, tpos = MO.trim(seq, strand, pos, insert, mate_pos, sam if sam_rules is None else sam_rules, trim_fillin)
            if tpos + len(tseq) > len(ref[cr]):
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
            ev = keep & (rr == opp)
            i = np.nonzero(keep & (rr == match) & ((q == match) | (q == convert)))[0]
            is_m, p = q[i] == match, tpos + i
            want, step = (C, -1) if minus else (G, 1)

            def at(k):
                ok = (k >= 0) & (k < len(r))
                return ok & (r[np.clip(k, 0, len(r) - 1)] == want)
            ctx = np.where(at(p + step), 0, np.where(at(p + 2 * step), 1, 2))
            score = int((is_m & (ctx != 0)).sum())
            if threshold and score >= threshold:
                continue
            np.add.at(snp[cr], tpos + np.nonzero(ev & (q == opp_snp))[0], 1)
            cpg = ctx == 0
            if not cpg.any():
                continue
            n_aln += 1
            n_calls += int(cpg.sum())
            st = sites[cr]
            shift = 1 if minus else 0                        # the call position of site c: c, or c + 1 on '-'
            a, b = np.searchsorted(st + shift, tpos), np.searchsorted(st + shift, tpos + len(tseq))
            called = np.zeros(b - a, dtype=bool)
            meth = np.zeros(b - a, dtype=bool)
            k = np.searchsorted(st, p[cpg] - shift) - a
            called[k] = True
            meth[k] = is_m[cpg]
            haps[cr].append((int(a), called, meth))
            add_runs(counts[cr], int(a), called, meth)
    return {"ref": ref, "sites": sites, "counts": counts, "snp": snp, "valid": nmap, "alignments": n_aln, "calls": n_calls,
            "haplotypes": haps}


def add_runs(counts, first, called, meth):
    """one haplotype (sites first, first + 1, ...; called / methylated bool arrays) into the run counters [n, 3, 16]"""
    run = [0, 0, 0]
    for j in range(len(called)):
        run[0] = run[0] + 1 if called[j] else 0
        run[1] = run[1] + 1 if called[j] and meth[j] else 0
        run[2] = run[2] + 1 if called[j] and not meth[j] else 0
        if called[j]:
            counts[first + j, 0, min(run[0], MAX_LEN) - 1] += 1
            f = 1 if meth[j] else 2
            counts[first + j, f, min(run[f], MAX_LEN) - 1] += 1


def cut_sites(res, cr, ct_snp=None) -> np.ndarray:
    """bool [n]: the sites the SNP mode cuts (skip / correct: snp > 0 at the C or the G)"""
    st = res["sites"][cr]
    if ct_snp not in ("skip", "correct"):
        return np.zeros(len(st), dtype=bool)
    s = res["snp"][cr]
    return (s[st] > 0) | (s[st + 1] > 0)


def site_range(res, cr, start, end):
    n = len(res["ref"][cr])
    st = res["sites"][cr]
    return int(np.searchsorted(st, min(start, n))), int(np.searchsorted(st, min(end, n)))


def region_sums(counts, cut, a, b) -> np.ndarray:
    """int64 [3, 16]: T_l, M_l, U_l of sites [a, b) from the run counters (the histogram-plus-clip form)"""
    out = np.zeros((3, MAX_LEN), dtype=np.int64)
    lim = 0
    for s in range(a, b):
        lim = 0 if cut[s] else min(lim + 1, MAX_LEN)
        if lim:
            suffix = counts[s][:, ::-1].cumsum(axis=1)[:, ::-1]
            out[:, :lim] += suffix[:, :lim]
    return out


def region_sums_direct(haps, cut, a, b) -> np.ndarray:
    """the same by enumerating every l consecutive called sites of every haplotype inside [a, b) and free of cuts"""
    out = np.zeros((3, MAX_LEN), dtype=np.int64)
    for first, called, meth in haps:
        for j in range(len(called)):
            for l in range(1, MAX_LEN + 1):
                if j + l > len(called):
                    break
                s0 = first + j
                if s0 < a or s0 + l > b or not called[j:j + l].all() or cut[s0:s0 + l].any():
                    continue
                m = meth[j:j + l]
                out[0, l - 1] += 1
                out[1, l - 1] += bool(m.all())
                out[2, l - 1] += bool((~m).all())
    return out


def load_stats(sums):
    """(L, MHL, uMHL) of a region's [3, 16] sums; MHL None when L = 0"""
    T, M, U = (list(int(x) for x in sums[f]) for f in range(3))
    L = max((l for l in range(1, MAX_LEN + 1) if T[l - 1] > 0), default=0)
    if not L:
        return 0, None, None
    hm = hu = 0.0
    for l in range(1, L + 1):
        hm += float(l * M[l - 1]) / float(T[l - 1])
        hu += float(l * U[l - 1]) / float(T[l - 1])
    w = float(L * (L + 1) // 2)
    return L, hm / w, hu / w


def regions(res, regs, ct_snp=None):
    """-> [(sites, int64 [3, 16])] for regs = [(chrom, start, end)]"""
    out = []
    cuts = {}
    for cr, s, e in regs:
        if cr not in cuts:
            cuts[cr] = cut_sites(res, cr, ct_snp)
        a, b = site_range(res, cr, s, e)
        out.append((b - a, region_sums(res["counts"][cr], cuts[cr], a, b)))
    return out


def mhl_text(res, regs, ct_snp=None) -> str:
    lines = [HEADER]
    for (cr, s, e), (n, sums) in zip(regs, regions(res, regs, ct_snp)):
        L, hm, hu = load_stats(sums)
        head = "%s\t%d\t%d\t%d\t%d\t%d\t" % (cr, s, e, n, sums[0, 0], L)
        if not L:
            lines.append(head + "NA\tNA\tNA\tNA\tNA\n")
            continue
        lists = "\t".join(",".join(str(int(x)) for x in sums[f, :L]) for f in range(3))
        lines.append(head + "%.4f\t%.4f\t%s\n" % (hm, hu, lists))
    return "".join(lines)


def tiles(res, width):
    """the regions of --tiles W: every selected sequence in name order, W bases a tile"""
    return [(cr, s, min(s + width, len(res["ref"][cr]))) for cr in sorted(res["ref"]) for s in range(0, len(res["ref"][cr]), width)]


def stderr_line(res) -> str:
    return "MHL: %d of %d valid mappings carry a CpG call, %d CpG calls in haplotypes" % (res["alignments"], res["valid"], res["calls"])
