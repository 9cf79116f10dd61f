"""oracle/mbias_oracle.py -- CPU restatement of the M-bias report and per-cycle exclusion (TEST INFRASTRUCTURE ONLY).

Only tests/ may import this module; the product path (bsmap_b200/csrc/bsx_meth.cu) never does.  It takes its
alignments from methratio_oracle.parse_alignments and trim, so a call here is exactly one increment of methratio.py's
counters (methratio.py:95-118); tests/test_mbias_cpu.py ties its sums to the reference script's own tables.

  call      a reference C under a '+' hit / G under a '-' hit where the read shows C or T / G or A, after the filters,
            -r, fill-in trimming, mate-overlap removal and the bounds test
  cycle     j, the call's 0-based offset in SEQ as printed (before trimming), or L-1-j when SEQ is printed reversed
            (the two ZS characters differ); L = printed length
  read      2 when FLAG has 0x80 (SAM), else 1; BSP records are read 1
  context   '+': CpG if ref[q+1] == G, else CHG if ref[q+2] == G, else CHH; '-': the same with ref[q-1], ref[q-2] and C;
            positions off the sequence count as H
  ignore    (r1_5p, r1_3p, r2_5p, r2_3p): a call of read r is dropped, from the counters too, when cycle < r_5p or
            cycle >= L - r_3p
"""
from __future__ import annotations

import numpy as np

import methratio_oracle as MO

CYCLES = 512
CONTEXTS = ("CpG", "CHG", "CHH")


def _read2_flags(path, chroms, unique, pair):
    """FLAG 0x80 of each alignment parse_alignments keeps, in its order"""
    if path[-4:].upper() != ".SAM":
        return None                                    # BSP: no read number
    out = []
    for line in open(path):
        if line.startswith("@"):
            continue
        col = line.rstrip("\n").split("\t")
        f = int(col[1])
        if f & 0x4 or (unique and f & 0x100) or (pair and not f & 0x2) or col[2] not in chroms:
            continue
        out.append(bool(f & 0x80))
    return out


def mbias(names, seqs, files, chroms=None, unique=False, pair=False, trim_fillin=2, combine_cpg=False, rm_dup=False,
          ignore=(0, 0, 0, 0), sam_rules=None):
    """-> (hist int64 [read][context][cycle][methylated, unmethylated], overflow, {chrom: (meth, depth)} with the
    exclusion applied (and -g combining when asked), valid mappings).  sam_rules: None = by file suffix as the script
    does; False / True force the BSP / SAM branch (mate-overlap removal) for SAM text that stands in for BSP output."""
    ref = {}
    for n, s in zip(names, seqs):
        s = s.decode() if isinstance(s, bytes) else s
        if not chroms or n in chroms:
            ref[n] = s.upper()
    chroms = set(ref)
    meth = {c: np.zeros(len(s), dtype=np.int64) for c, s in ref.items()}
    depth = {c: np.zeros(len(s), dtype=np.int64) for c, s in ref.items()}
    refarr = {c: np.frombuffer(s.encode(), dtype=np.uint8) for c, s in ref.items()}
    coverage = {c: np.zeros(len(s), dtype=np.uint8) for c, s in ref.items()} if rm_dup else None
    hist = np.zeros((2, 3, CYCLES, 2), dtype=np.int64)
    overflow = nmap = 0
    C, G = ord("C"), ord("G")
    for path in files:
        alns = MO.parse_alignments(path, chroms, unique, pair)
        r2 = _read2_flags(path, chroms, unique, pair) or [False] * len(alns)
        assert len(r2) == len(alns)
        for (seq, strand, cr, pos, insert, mate_pos, sam), read2 in zip(alns, r2):
            if rm_dup:                                       # methratio.py:52-55, as in methratio_oracle.methratio
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
            start = tpos - pos                               # '--' / '-+' trimming drops this many printed characters
            minus = strand[0] == "-"
            match, convert = (G, ord("A")) if minus else (C, ord("T"))
            r = refarr[cr]
            q = np.frombuffer(tseq.encode(), dtype=np.uint8)
            i = np.nonzero((r[tpos:tpos + len(tseq)] == match) & ((q == match) | (q == convert)))[0]
            is_m = q[i] == match
            j = start + i
            cyc = L - 1 - j if strand[0] != strand[1] else j
            lo, hi = (ignore[2], L - ignore[3]) if read2 else (ignore[0], L - ignore[1])
            keep = (cyc >= lo) & (cyc < hi)
            i, is_m, cyc = i[keep], is_m[keep], cyc[keep]
            p = tpos + i
            np.add.at(depth[cr], p, 1)
            np.add.at(meth[cr], p[is_m], 1)
            want, step = (C, -1) if minus else (G, 1)

            def at(k):
                ok = (k >= 0) & (k < len(r))
                return ok & (r[np.clip(k, 0, len(r) - 1)] == want)
            ctx = np.where(at(p + step), 0, np.where(at(p + 2 * step), 1, 2))
            inr = cyc < CYCLES
            overflow += int((~inr).sum())
            np.add.at(hist, (int(read2), ctx[inr], cyc[inr], np.where(is_m[inr], 0, 1)), 1)
    if combine_cpg:
        for cr in depth:
            r = refarr[cr]
            cg = np.nonzero((r[:-1] == C) & (r[1:] == G))[0]
            for a in (depth[cr], meth[cr]):
                a[cg] += a[cg + 1]
                a[cg + 1] = 0
    return hist, overflow, {c: (meth[c], depth[c]) for c in ref}, nmap


def mbias_text(hist) -> str:
    """the report: per context, per read, per 1-based cycle with calls; ratio %.3f"""
    lines = ["context\tread\tcycle\tmethylated\tunmethylated\tratio\n"]
    for c, name in enumerate(CONTEXTS):
        for rd in range(2):
            for y in range(hist.shape[2]):
                m, u = int(hist[rd, c, y, 0]), int(hist[rd, c, y, 1])
                if m + u:
                    lines.append("%s\t%d\t%d\t%d\t%d\t%.3f\n" % (name, rd + 1, y + 1, m, u, m / (m + u)))
    return "".join(lines)
